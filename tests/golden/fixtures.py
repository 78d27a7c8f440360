"""Deterministic inputs/weights shared by make_goldens.py (which feeds them to the real reference)
and by the tests (which feed them to the oracle and to the CUDA path).  Everything is derived from
integer seeds with torch's CPU generator, so fixtures only need to store outputs plus checksums."""
import json
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def gen(seed):
    return torch.Generator().manual_seed(int(seed))


def randn(seed, *shape, scale=1.0):
    return torch.randn(*shape, generator=gen(seed)) * scale


def seeded_state_dict(shapes, seed):
    """shapes: {param name: shape tuple}.  Non-degenerate values: non-zero biases, LayerNorm gains
    around 1, weights with unit-ish fan-in gain so predictor scores are well spread (no near-ties)."""
    g = gen(seed)
    sd = {}
    for name in sorted(shapes):
        shape = tuple(shapes[name])
        if name.endswith("num_batches_tracked"):
            sd[name] = torch.zeros(shape, dtype=torch.long)
        elif name.endswith("running_var"):
            sd[name] = torch.rand(shape, generator=g) + 0.5
        elif name.endswith("running_mean"):
            sd[name] = torch.randn(shape, generator=g) * 0.1
        elif name in ("cls_token", "pos_embed"):
            sd[name] = torch.randn(shape, generator=g) * 0.2
        elif len(shape) == 1 and name.endswith("weight"):
            sd[name] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        elif len(shape) == 1:
            sd[name] = 0.05 * torch.randn(shape, generator=g)
        else:
            fan_in = int(np.prod(shape[1:]))
            sd[name] = torch.randn(shape, generator=g) / (fan_in ** 0.5)
    return sd


def checksum(t):
    t = t.detach().double()
    return [float(t.sum()), float(t.abs().sum())]


def sd_checksum(sd):
    s = a = 0.0
    for k in sorted(sd):
        if sd[k].is_floating_point():
            c = checksum(sd[k])
            s += c[0]
            a += c[1]
    return [s, a]


# A golden tensor of more than SAMPLE_ABOVE elements is stored as SAMPLE_N of its elements (flat indices from sample_index),
# with its shape and its largest magnitude in meta["sampled"]: every golden file stays under 1 MB.
SAMPLE_ABOVE, SAMPLE_N = 16384, 8192


def sample_index(numel):
    """Sorted flat indices of the stored elements of a sampled golden tensor.  numpy's legacy RandomState keeps its stream
    fixed across numpy versions, so the indices are a pure function of `numel`."""
    return torch.from_numpy(np.sort(np.random.RandomState(numel).choice(numel, SAMPLE_N, replace=False)))


def sample_arrays(arrays, meta):
    """Replace every tensor above SAMPLE_ABOVE elements by its sample; record what golden_view needs in meta["sampled"].
    Used for the model goldens (save_npz(..., sample=True)), the only ones that would exceed 1 MB whole."""
    out = dict(arrays)
    for k, v in arrays.items():
        if torch.is_tensor(v) and v.numel() > SAMPLE_ABOVE:
            out[k] = v.reshape(-1)[sample_index(v.numel())]
            meta.setdefault("sampled", {})[k] = dict(shape=list(v.shape), absmax=float(v.abs().max()))
    return out


def golden_view(arrays, meta, key, t):
    """(t, golden, max |golden|) for comparing a computed tensor `t` with golden `key`: a sampled golden is compared on the
    same elements of t, against the largest magnitude of the whole golden tensor."""
    s = meta.get("sampled", {}).get(key)
    if s is None:
        ref = arrays[key]
        return t, ref, float(ref.abs().max())
    assert list(t.shape) == s["shape"], (key, tuple(t.shape), s["shape"])
    return t.reshape(-1)[sample_index(t.numel()).to(t.device)], arrays[key], s["absmax"]


def save_npz(name, arrays, meta, sample=False):
    if sample:
        arrays = sample_arrays(arrays, meta)
    out = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()}
    out["__meta__"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, name), **out)


def load_npz(name):
    z = np.load(os.path.join(HERE, name))
    meta = json.loads(bytes(z["__meta__"]).decode())
    arrays = {k: torch.from_numpy(z[k]) for k in z.files if k != "__meta__"}
    return arrays, meta


# small model used for the model-level goldens (N=196 is hard-coded by the reference: 224/16 squared)
SMALL_CFG = dict(embed_dim=128, depth=4, num_heads=2, patch_size=16, num_classes=16)


def loss_inputs(seed, B=4, N=196, L=4, H=3, C=32, ratios=(0.7, 0.49), classes=16):
    """Seeded stand-ins for what train.py:40-46 feeds the losses (shapes of a 2-stage Dense2Sparse student)."""
    K = [int(N * r) for r in ratios]
    n_in = [N] + K[:-1]
    g = gen(seed)
    cls_attn = torch.softmax(torch.randn(B, L, H, N + 1, generator=g) * 2.0, dim=-1)
    pred_logits = [torch.randn(B, n, generator=g) for n in n_in]
    kept = [torch.stack([torch.sort(torch.randperm(n, generator=g)[:k])[0] for _ in range(B)]) for n, k in zip(n_in, K)]
    logits_s, logits_t = torch.randn(B, classes, generator=g), torch.randn(B, classes, generator=g)
    token_s, token_t = torch.randn(B, K[-1], C, generator=g), torch.randn(B, N, C, generator=g)
    labels = torch.randint(0, classes, (B,), generator=g)
    soft = torch.softmax(torch.randn(B, classes, generator=g), dim=-1)
    return dict(cls_attn=cls_attn, pred_logits=pred_logits, kept=kept, logits_s=logits_s, logits_t=logits_t, token_s=token_s,
                token_t=token_t, labels=labels, soft=soft, ratios=list(ratios))
