"""Attention forward beyond 256 tokens (d2s_attn_long_fwd, ops.attention_long): the key-blocked tcgen05 kernel against a float64
restatement of the reference formula, against the T <= 256 kernel where both run, at the edges of the exponent range, in its
variable-length form, in guard zones, and inside whole DeiT-S models at 384 and 512 pixels."""
import ctypes

import pytest
import torch

import fixtures as fx

DEIT_S = dict(patch_size=16, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, qkv_bias=True)
LOCS, RATIOS = [3, 6, 9], [0.7, 0.7 ** 2, 0.7 ** 3]
VARLEN_LENS = [577, 513, 512, 385, 257, 129, 2, 1]     # Tmax = 577: every 128-row / 128-key block boundary is crossed


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ref(qkv, H, policy=None, eps=1e-6, scale=0.125):
    """Attention.forward's core in float64 on the same bf16 qkv (dynamic_vit.py:195-214 softmax_with_policy, :218-234):
    (out (B,T,H*64), cls_row (B,H,T))."""
    B, T, _ = qkv.shape
    q, k, v = qkv.double().view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4).unbind(0)
    s = (q @ k.transpose(-1, -2)) * scale
    if policy is None:
        p = torch.softmax(s, dim=-1)
    else:
        pol = policy.double().view(B, 1, 1, T)
        eye = torch.eye(T, dtype=torch.float64, device=qkv.device).view(1, 1, T, T)
        mask = pol + (1.0 - pol) * eye
        e = (s - s.amax(-1, keepdim=True)).exp() * mask
        p = (e + eps / T) / (e.sum(-1, keepdim=True) + eps)
    return (p @ v).transpose(1, 2).reshape(B, T, H * 64), p[:, :, 0, :]


def _policy(B, T, g, frac=0.5):
    pol = (torch.rand(B, T, device="cuda", generator=g) > frac).float()     # many zeros
    pol[:, 0] = 1
    return pol


# ----------------------------------------------------------------------------------------------------------------- host / CPU
def test_long_attention_argument_errors_precede_any_launch(d2s):
    lib = d2s._lib.load()
    before = d2s._lib.launch_count()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    f = lib.d2s_attn_long_fwd
    assert f(None, None, None, 2, 577, 6, 64, 0.125, 1e-6, p, None, None) == 1 and b"null" in lib.d2s_last_error()
    assert f(p, None, None, 2, 577, 6, 64, 0.125, 1e-6, None, None, None) == 1 and b"null" in lib.d2s_last_error()
    assert f(p, None, None, 2, 577, 6, 48, 0.125, 1e-6, p, None, None) == 1 and b"head dim" in lib.d2s_last_error()
    assert f(p, None, None, 2, 0, 6, 64, 0.125, 1e-6, p, None, None) == 1 and b"T=0" in lib.d2s_last_error()
    assert f(p, None, None, 2, 2049, 6, 64, 0.125, 1e-6, p, None, None) == 1 and b"T=2049" in lib.d2s_last_error()
    assert f(p, p, p, 2, 577, 6, 64, 0.125, 1e-6, p, None, None) == 1 and b"exclusive" in lib.d2s_last_error()
    assert f(p, None, None, 2, 577, 6, 64, 0.0, 1e-6, p, None, None) == 1 and b"scale" in lib.d2s_last_error()
    assert f(p + 4, None, None, 2, 577, 6, 64, 0.125, 1e-6, p, None, None) == 2
    assert f(p, None, None, 2, 577, 6, 64, 0.125, 1e-6, p + 8, None, None) == 2
    assert d2s._lib.launch_count() == before
    assert f(p, None, None, 0, 577, 6, 64, 0.125, 1e-6, p, None, None) == 0        # an empty batch is a no-op
    # the T <= 256 entry points keep their limits
    assert lib.d2s_attn_policy_fwd(p, None, 1, 1, 300, 6, 64, 0.125, 1e-6, p, None, None, None) == 1
    assert b"T=300 exceeds 256" in lib.d2s_last_error()
    assert d2s._lib.launch_count() == before


def test_engine_routes_long_bf16_attention_behind_its_switch(d2s, monkeypatch):
    """The fused path takes bf16, head dim 64, 256 < T <= 2048 unless engine._LONG_ATTN is False; fp32 above 256 keeps the torch path."""
    ok = d2s.engine._attn_kernel_ok
    bf = torch.empty(1, 577, 3 * 6 * 64, dtype=torch.bfloat16)
    assert ok(bf, 6) and ok(torch.empty(1, 2048, 3 * 6 * 64, dtype=torch.bfloat16), 6)
    assert not ok(torch.empty(1, 2049, 3 * 6 * 64, dtype=torch.bfloat16), 6)
    assert not ok(torch.empty(1, 577, 3 * 6 * 64, dtype=torch.float32), 6)
    assert not ok(torch.empty(1, 577, 3 * 6 * 48, dtype=torch.bfloat16), 6)
    assert ok(torch.empty(1, 197, 3 * 6 * 64, dtype=torch.bfloat16), 6)
    monkeypatch.setattr(d2s.engine, "_LONG_ATTN", False)
    assert not ok(bf, 6) and ok(torch.empty(1, 256, 3 * 6 * 64, dtype=torch.bfloat16), 6)


# ----------------------------------------------------------------------------------------------------------------- kernel
@pytest.mark.gpu
@pytest.mark.parametrize("T", [257, 300, 577, 785, 1025, 2048])
@pytest.mark.parametrize("H", [6, 12])
@pytest.mark.parametrize("with_policy", [False, True])
def test_long_attention_matches_float64_reference(d2s, cuda_dev, T, H, with_policy):
    ops = d2s.ops
    B = 2
    g = torch.Generator(device="cuda").manual_seed(1000 + T + H)
    qkv = torch.randn(B, T, 3 * H * 64, device="cuda", generator=g).bfloat16()
    pol = _policy(B, T, g) if with_policy else None
    n0 = d2s._lib.launch_count()
    out, cls = ops.attention_long(qkv, H, policy=pol, want_cls_row=True)
    assert d2s._lib.launch_count() == n0 + 1
    ro, rc = _ref(qkv, H, pol)
    # the tolerances of the T <= 256 bf16 attention tests (test_gpu_parity.py: bf16 operands and probabilities, fp32 accumulate)
    torch.testing.assert_close(out.double(), ro, rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(cls.double(), rc, rtol=1e-2, atol=2e-4)
    if not with_policy:
        torch.testing.assert_close(cls.sum(-1), torch.ones(B, H, device="cuda"), rtol=1e-3, atol=1e-3)
    # attention_core hands T > 256 in bf16 to the same kernel
    o2, c2 = ops.attention_core(qkv, H, policy=pol, want_cls_row=True)
    assert torch.equal(out, o2) and torch.equal(cls, c2)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 17, 128, 129, 197, 256])
@pytest.mark.parametrize("with_policy", [False, True])
def test_long_attention_agrees_with_the_one_block_kernel(d2s, cuda_dev, T, with_policy):
    """Where both run, the key-blocked kernel and d2s_attn_policy_fwd compute the same thing: the same exponent reference and
    exponentials, a different summation order (bf16 rounding of the output, fp32 rounding of the CLS row)."""
    ops = d2s.ops
    B, H = 3, 6
    g = torch.Generator(device="cuda").manual_seed(2000 + T)
    qkv = torch.randn(B, T, 3 * H * 64, device="cuda", generator=g).bfloat16()
    pol = _policy(B, T, g, 0.3) if with_policy else None
    o1, c1 = ops.attention_long(qkv, H, policy=pol, want_cls_row=True)
    o2, c2 = ops.attention_core(qkv, H, policy=pol, want_cls_row=True)
    torch.testing.assert_close(o1.float(), o2.float(), rtol=1.6e-2, atol=1e-3)     # one bf16 ulp of the output
    torch.testing.assert_close(c1, c2, rtol=2e-3, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("with_policy", [False, True])
def test_long_attention_logits_far_above_the_row_reference(d2s, cuda_dev, with_policy):
    """T = 577: every second query row holds logits of ~200 nats at a key of the last key block and at a key that image 0's
    policy masks, and ~50 nats inside the reference columns (the first 16 keys): ~216 binades above the reference, so those
    rows overflow and are redone from global memory.  The result must equal the float64 reference: no inf, no NaN, no clamp."""
    ops = d2s.ops
    B, T, H, hd = 2, 577, 6, 64
    g = fx.gen(140)
    qkv = torch.randn(B, T, 3, H, hd, generator=g) * 0.5
    u = torch.nn.functional.normalize(torch.randn(hd, generator=g), dim=0)
    j_last, j_mask = T - 13, 300
    qkv[:, 0::2, 0] += 40.0 * u
    qkv[:, j_last, 1] = 40.0 * u
    qkv[:, j_mask, 1] = 40.2 * u
    qkv[:, 5, 1] = 10.0 * u
    qkv = qkv.reshape(B, T, 3 * H * hd).bfloat16().cuda()
    pol = None
    if with_policy:
        pol = (torch.rand(B, T, generator=g) > 0.3).float().cuda()
        pol[:, 0] = 1
        pol[0, j_last], pol[0, j_mask] = 1, 0        # image 0: the row maximum itself is masked out (the eps terms follow it)
        pol[1, j_last], pol[1, j_mask] = 1, 1
    out, cls = ops.attention_long(qkv, H, policy=pol, want_cls_row=True)
    ro, rc = _ref(qkv, H, pol)
    s = torch.einsum("bihd,bjhd->bhij", qkv.float().view(B, T, 3, H, hd)[:, :, 0], qkv.float().view(B, T, 3, H, hd)[:, :, 1]) / 8
    assert float((s[:, :, 0::2].amax(-1) - s[:, :, 0::2, :16].amax(-1)).min()) > 100       # the case is really exercised
    assert bool(torch.isfinite(out).all()) and bool(torch.isfinite(cls).all())
    torch.testing.assert_close(out.double(), ro, rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(cls.double(), rc, rtol=1e-2, atol=2e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [2, 6])
def test_long_attention_varlen_matches_each_image_alone(d2s, cuda_dev, H):
    ops = d2s.ops
    lens = VARLEN_LENS
    B, T = len(lens), max(lens)
    g = torch.Generator(device="cuda").manual_seed(3000 + H)
    qkv = (torch.randn(B, T, 3 * H * 64, device="cuda", generator=g) * 0.8).bfloat16()
    n = torch.tensor(lens, dtype=torch.int32, device="cuda")
    out, cls = ops.attention_long(qkv, H, want_cls_row=True, lengths=n)
    for b, L in enumerate(lens):
        o1, c1 = ops.attention_long(qkv[b:b + 1, :L].contiguous(), H, want_cls_row=True)
        assert torch.equal(out[b, :L], o1[0]), (b, L)           # same blocks, same chunks, same order: bit for bit
        assert torch.equal(cls[b, :, :L], c1[0]), (b, L)
        assert not out[b, L:].any() and not cls[b, :, L:].any(), (b, L)      # pad rows / columns are zeros
    # pad rows take no part: other finite values there change nothing
    q2 = qkv.clone()
    for b, L in enumerate(lens):
        q2[b, L:] = (torch.randn(q2[b, L:].shape, device="cuda", generator=g) * 3).bfloat16()
    out2, cls2 = ops.attention_long(q2, H, want_cls_row=True, lengths=n)
    assert torch.equal(out, out2) and torch.equal(cls, cls2)
    # attention_core's variable-length form takes T > 256 to the same kernel
    o3, c3 = ops.attention_core(qkv, H, want_cls_row=True, lengths=n)
    assert torch.equal(out, o3) and torch.equal(cls, c3)


class _Guarded:
    """A tensor inside a larger byte buffer whose guard zones hold a sentinel (outputs) or NaN (behind inputs)."""
    GUARD, SENT = 4096, 0x5A

    def __init__(self, shape, dtype, fill=None, poison_after=False):
        n = 1
        for s in shape:
            n *= s
        es = torch.empty(0, dtype=dtype).element_size()
        gb = self.GUARD * es
        self.raw = torch.full((gb + n * es + gb,), self.SENT, dtype=torch.uint8, device="cuda")
        self.t = self.raw[gb:gb + n * es].view(dtype).view(shape)
        if fill is not None:
            self.t.copy_(fill)
        else:
            self.t.fill_(float("nan") if dtype.is_floating_point else -1)
        self.gb = gb
        self.tail = None
        if poison_after:
            self.raw[gb + n * es:].view(torch.int16).fill_(-1)       # 0xFFFF: NaN as bf16, NaN pairs as fp32
            self.tail = self.raw[gb + n * es:].clone()

    def ok(self):
        head = bool((self.raw[:self.gb] == self.SENT).all())
        tail = self.raw[self.raw.numel() - self.gb:]
        return head and (bool((tail == self.SENT).all()) if self.tail is None else bool(torch.equal(tail, self.tail)))


@pytest.mark.gpu
@pytest.mark.parametrize("T", [577, 1025])
@pytest.mark.parametrize("form", ["dense", "policy", "varlen"])
def test_long_attention_stays_in_bounds(d2s, cuda_dev, T, form):
    lib = d2s._lib
    B, H = 3, 6
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(T)
    qkv = _Guarded((B, T, 3 * D), torch.bfloat16, (torch.randn(B, T, 3 * D, device="cuda", generator=g) * 0.7).bfloat16(), poison_after=True)
    pol = _Guarded((B, T), torch.float32, _policy(B, T, g, 0.3), poison_after=True) if form == "policy" else None
    lens = _Guarded((B,), torch.int32, torch.tensor([T, T // 2 + 1, 129], dtype=torch.int32), poison_after=True) if form == "varlen" else None
    results = []
    for _ in range(2):
        out, cls = _Guarded((B, T, D), torch.bfloat16), _Guarded((B, H, T), torch.float32)
        lib.call("d2s_attn_long_fwd", qkv.t.data_ptr(), pol.t.data_ptr() if pol else None, lens.t.data_ptr() if lens else None, B, T, H, 64,
                 0.125, 1e-6, out.t.data_ptr(), cls.t.data_ptr(), _stream())
        torch.cuda.synchronize()
        for name, gd in (("out", out), ("cls_row", cls), ("qkv", qkv), ("policy", pol), ("lens", lens)):
            if gd is not None:
                assert gd.ok(), f"{name}: guard zone overwritten"
        for name, gd in (("out", out), ("cls_row", cls)):
            assert bool(torch.isfinite(gd.t.float()).all()), f"{name}: element left unwritten or fed by an out-of-bounds read"
        results.append((out.t.clone(), cls.t.clone()))
    assert torch.equal(results[0][0], results[1][0]) and torch.equal(results[0][1], results[1][1])   # run to run: bit for bit


# ----------------------------------------------------------------------------------------------------------------- models
def _model(d2s, kind, img_size, ratios=RATIOS, seed=171):
    if kind == "teacher":
        m = d2s.variant_a.DefaultVisionTransformerTeacher(img_size=img_size, num_classes=1000, **DEIT_S)
    elif kind == "a":
        m = d2s.variant_a.DefaultVisionTransformerDiffPruning(img_size=img_size, pruning_loc=LOCS, token_ratio=ratios, distill=True,
                                                              num_classes=1000, **DEIT_S)
    else:
        m = d2s.variant_b.VisionTransformerDiffPruning(img_size=img_size, pruning_loc=LOCS, token_ratio=ratios, distill=True,
                                                       topk_selection=True, predictor_loss_type="kl_div", num_classes=1000, **DEIT_S)
    sd = fx.seeded_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, seed)
    m.load_state_dict({k: (v.bfloat16().float() if v.is_floating_point() else v) for k, v in sd.items()})   # bf16-representable
    return m


def _outputs(kind, out, model):
    """(logits, stage-1 kept set (B,K) or None, CLS attention of blocks 0-2 (before any pruning) or None) of one eval forward."""
    if kind == "teacher":
        return out[0], None, None
    if kind == "a":
        return out, model.kept_token_indices[0].clone(), None
    return out[0], out[3][0].clone(), torch.stack([c.float() for c in out[1][:3]])


KEEP_ALL = [576 / 196 + 1e-4] * 3      # int(196 r) = 576: every token of a 384-px image stays (the reference counts from 196)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,ratios", [("teacher", None), ("a", KEEP_ALL), ("a", RATIOS), ("b", RATIOS)])
def test_models_at_384_pixels_bf16_graph(d2s, cuda_dev, monkeypatch, kind, ratios):
    """DeiT-S/16 at 384 px (T = 577) in bf16 through the CUDA-graph runner, B = 64, with the key-blocked attention kernel and with
    engine._LONG_ATTN off (torch matmuls around the policy softmax), each against the fp32 GPU path on identical (bf16-representable)
    weights and images -- the rule of test_bench_config_bf16_graph_at_batch_1024:
      * no token can change sides (the teacher; Variant A keeping all 576 tokens): logits within 1e-2 relative (L2), largest
        deviation 3e-2 of max |logit|;
      * real ratios (int(196 r) of 576 tokens, as the reference counts): the stage-1 kept set equals the fp32 one wherever the fp32
        score margin at the cut exceeds bf16 noise, only tokens within that noise of the cut change sides, and no more of them with
        the kernel than with the torch path it replaces; logits loosely bounded;
      * Variant B: the CLS attention of blocks 0-2 (before any pruning, T = 577) within 1e-2 relative (L2) on every image."""
    B = 64
    x = torch.randn(B, 3, 384, 384, device=cuda_dev, generator=torch.Generator(device=cuda_dev).manual_seed(173)).bfloat16()
    m32 = _model(d2s, kind, 384, ratios).to(cuda_dev).eval()
    with torch.no_grad():
        o32 = m32(x.float())
        l32, k32, c32 = _outputs(kind, o32, m32)
        l32 = l32.float().clone()
        s32 = None                                               # fp32 stage-1 scores (the kept set is their top K): margins at the cut
        if kind == "b":
            s32 = o32[2][0].float().clone()
        elif kind == "a" and ratios is RATIOS:
            st = d2s.engine._embed_stream(m32, x.float())
            for blk in m32.blocks[:LOCS[0]]:
                st.block(blk)
            s32 = d2s.engine.predictor_a_forward(m32.score_predictor[0], st.value()[:, 1:], torch.ones(B, 576, 1, device=cuda_dev))[:, :, 0]
    calls = {"n": 0}
    attention_long = d2s.ops.attention_long

    def counted(*a, **k):
        calls["n"] += 1
        return attention_long(*a, **k)
    monkeypatch.setattr(d2s.ops, "attention_long", counted)
    mean_flips = {}
    for on in (True, False):
        monkeypatch.setattr(d2s.engine, "_LONG_ATTN", on)
        calls["n"] = 0
        runner = d2s.runner.InferenceRunner(_model(d2s, kind, 384, ratios), B, cuda_dev, dtype=torch.bfloat16, img_shape=(3, 384, 384),
                                            use_graph=True, warmup=1)
        l16, k16, c16 = _outputs(kind, runner(x), runner.model)
        l16 = l16.float().clone()
        torch.cuda.synchronize()
        assert runner.graph is not None
        assert (calls["n"] > 0) == on, calls                     # the new kernel runs exactly when it is switched on
        scale = float(l32.abs().max())
        rel_l2 = float((l16 - l32).norm() / l32.norm())
        if k32 is None or k32.shape[1] == 576:
            assert rel_l2 <= 1e-2, (on, rel_l2)
            assert float((l16 - l32).abs().max()) <= 3e-2 * scale, on
        else:
            K = k32.shape[1]
            a_, b_ = torch.zeros(B, 576, dtype=torch.bool), torch.zeros(B, 576, dtype=torch.bool)
            a_.scatter_(1, k16.cpu(), True)
            b_.scatter_(1, k32.cpu(), True)
            flips = (a_ ^ b_).sum(1)
            srt = torch.sort(s32, dim=-1, descending=True).values
            margin = (srt[:, K - 1] - srt[:, K]).cpu()
            near = ((s32 - srt[:, K - 1:K]).abs() < 0.05).sum(1).cpu()
            print(f"{kind} on={on}: mean flips {float(flips.float().mean()):.3f}, mean near {float(near.float().mean()):.2f}, "
                  f"images with flips {int((flips > 0).sum())}, rel_l2 {rel_l2:.4f}")
            assert bool((flips <= 2 * near).all()), (on, int(flips.max()), int(near.min()))
            assert bool((flips[margin > 0.05] == 0).all()), on
            mean_flips[on] = float(flips.float().mean())
            assert rel_l2 <= 0.25, (on, rel_l2)
        if c32 is not None:
            assert float((c16.float() - c32).norm() / c32.norm()) <= 1e-2, on
        del runner
    if mean_flips:
        # Few tokens change sides.  The budget of the 224-px test (2 % of K over 196 scores) scales with the score density at the
        # cut: 576 scores put 576 / 196 times as many tokens within bf16 noise of it.  And the key-blocked kernel (fp32 scores, bf16
        # probabilities) must not move more tokens than the path it replaces (scores rounded to bf16 before the softmax).
        K = k32.shape[1]
        for on, mf in mean_flips.items():
            assert mf <= 0.02 * K * 576 / 196, (on, mf)
        assert mean_flips[True] <= 1.25 * mean_flips[False] + 0.5, mean_flips


@pytest.mark.gpu
def test_forward_varlen_at_384_pixels_matches_batch_one(d2s, cuda_dev, monkeypatch):
    """Dynamic keep-ratio inference at 384 px: forward_varlen on a batch of 16 against the batch-1 opt-in on each image, as the
    224-px test does, at a threshold that keeps more than 256 tokens per image after the first stage (so the variable-length
    stages run the key-blocked kernel).  Kept sets agree except at near-ties of the cut; the agreeing images' logits meet the
    bf16 bound."""
    m = d2s.variant_b.VisionTransformerDiffPruning(img_size=384, pruning_loc=LOCS, token_ratio=RATIOS, distill=True,
                                                   topk_selection=True, predictor_loss_type="kl_div", patch_score_threshold=0.3,
                                                   num_classes=1000, **DEIT_S)
    sd = fx.seeded_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, 151)
    m.load_state_dict(sd)
    model = m.to(cuda_dev).eval().to(torch.bfloat16)
    B = 16
    img = fx.randn(181, B, 3, 384, 384).to(cuda_dev, torch.bfloat16)
    with torch.no_grad():
        for thr in (0.3, 0.1, 0.03, 0.01, 0.003, 0.001):
            model.patch_score_threshold = thr
            _, _, _, kept = model.forward_varlen(img)
            if int((kept[0] >= 0).sum(1).min()) > 256:
                break
    assert int((kept[0] >= 0).sum(1).min()) > 256, thr
    calls = {"n": 0}
    attention_long = d2s.ops.attention_long

    def counted(*a, **k):
        calls["n"] += k.get("lengths") is not None
        return attention_long(*a, **k)
    monkeypatch.setattr(d2s.ops, "attention_long", counted)
    with torch.no_grad():
        logits, _, pred_logits, kept = model.forward_varlen(img)
    assert calls["n"] > 0                                          # the variable-length stages above 256 tokens ran the new kernel
    counts = [[int((k[b] >= 0).sum()) for b in range(B)] for k in kept]
    model.d2s_threshold_inference = True
    agree = 0
    for b in range(B):
        with torch.no_grad():
            lg1, _, pl1, kept1 = model(img[b:b + 1])
        same = True
        for s in range(3):
            c = counts[s][b]
            if not torch.equal(kept[s][b, :c], kept1[s][0]):
                probs = torch.sort(torch.softmax(pl1[s][0].float(), -1))[0]
                assert float((torch.cumsum(probs, -1) - thr).abs().min()) < 2e-2, (b, s)   # only a near-tie at the cut may flip
                same = False
                break
        if same:
            agree += 1
            d = logits[b].float() - lg1[0].float()
            assert float(d.norm() / lg1.float().norm()) < 1e-2 and float(d.abs().max() / lg1.float().abs().max()) < 2e-2, b
    assert agree >= 3 * B // 4, agree


@pytest.mark.gpu
def test_teacher_at_512_pixels_runs_and_its_first_attention_matches_float64(d2s, cuda_dev):
    """T = 1025: beyond what the torch fallback's softmax kernel takes, so only the new kernel can run this forward.  The teacher
    runs through the CUDA-graph runner, and block 0's attention on the model's own bf16 tokens matches the float64 reference."""
    B = 8
    m = _model(d2s, "teacher", 512)
    runner = d2s.runner.InferenceRunner(m, B, cuda_dev, dtype=torch.bfloat16, img_shape=(3, 512, 512), use_graph=True, warmup=1)
    x = torch.randn(B, 3, 512, 512, device=cuda_dev, generator=torch.Generator(device=cuda_dev).manual_seed(191)).bfloat16()
    logits = runner(x)[0].float().clone()
    torch.cuda.synchronize()
    assert logits.shape == (B, 1000) and bool(torch.isfinite(logits).all())
    model = runner.model
    with torch.no_grad():
        tok = torch.nn.functional.conv2d(x, model.patch_embed.proj.weight, model.patch_embed.proj.bias, stride=16).flatten(2).transpose(1, 2)
        tok = torch.cat([model.cls_token.expand(B, -1, -1), tok], 1) + model.pos_embed
        blk = model.blocks[0]
        qkv = blk.attn.qkv(blk.norm1(tok))
        assert qkv.shape == (B, 1025, 3 * 384) and qkv.dtype == torch.bfloat16
        out, cls = d2s.ops.attention_core(qkv, 6, scale=blk.attn.scale, want_cls_row=True)
    ro, rc = _ref(qkv, 6, scale=blk.attn.scale)
    torch.testing.assert_close(out.double(), ro, rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(cls.double(), rc, rtol=1e-2, atol=2e-4)
    del runner
