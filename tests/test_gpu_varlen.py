"""Variable-length (padded) dynamic keep-ratio inference: the varlen entry points against their dense siblings run on each image
alone, in guard zones, and the whole model (forward_varlen) against the oracle and against the batch-1 opt-in.

Layout under test (include/d2s.h): a stage's tokens are x (B,Tmax,D) plus per-image lengths; rows past an image's length are pad
rows, and no valid output may depend on them."""
import ctypes

import pytest
import torch

import fixtures as fx

LENS = [197, 150, 129, 128, 97, 2, 1, 68]      # Tmax = 197: both sides of 128, a single-token image
LENS_SHORT = [97, 64, 1, 33, 96, 17]           # Tmax = 97 <= 128: the one-tile kernel


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _lens(lens):
    return torch.tensor(lens, dtype=torch.int32, device="cuda")


# ----------------------------------------------------------------------------------------------------------------- host / CPU
def test_varlen_argument_errors_precede_any_launch(d2s):
    lib = d2s._lib.load()
    before = d2s._lib.launch_count()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    assert lib.d2s_attn_varlen_fwd(p, None, 1, 2, 197, 6, 64, 0.125, p, None, None) == 1 and b"null" in lib.d2s_last_error()
    assert lib.d2s_attn_varlen_fwd(p, p, 1, 2, 300, 6, 64, 0.125, p, None, None) == 1 and b"Tmax=300" in lib.d2s_last_error()
    assert lib.d2s_attn_varlen_fwd(p, p, 1, 2, 197, 6, 48, 0.125, p, None, None) == 1 and b"head dim" in lib.d2s_last_error()
    assert lib.d2s_attn_varlen_fwd(p, p, 1, 2, 197, 6, 64, 0.0, p, None, None) == 1 and b"scale" in lib.d2s_last_error()
    assert lib.d2s_attn_varlen_fwd(p + 4, p, 1, 2, 197, 6, 64, 0.125, p, None, None) == 2
    assert lib.d2s_threshold_select_varlen_f32(p, None, 2, 196, 0.3, p, p, p, None) == 1 and b"null" in lib.d2s_last_error()
    assert lib.d2s_threshold_select_varlen_f32(p, p, 2, 2000, 0.3, p, p, p, None) == 1 and b"Nmax=2000" in lib.d2s_last_error()
    assert lib.d2s_score_tail_b_varlen(p, None, 0, 2, 196, 64, None, None, 1e-5, p, None, 0, p, p, None) == 1
    assert b"null" in lib.d2s_last_error()
    assert lib.d2s_score_tail_b_varlen(p, p, 0, 2, 196, 60, None, None, 1e-5, p, None, 0, p, p, None) == 1 and b"C=60" in lib.d2s_last_error()
    assert lib.d2s_score_tail_b_varlen(p, p, 0, 2, 196, 64, p, None, 1e-5, p, None, 0, p, p, None) == 1 and b"ln_w" in lib.d2s_last_error()
    assert lib.d2s_pool_concat_varlen_inplace(p, None, 1, 2, 196, 384, None) == 1 and b"null" in lib.d2s_last_error()
    assert lib.d2s_pool_concat_varlen_inplace(p, p, 1, 2, 196, 100, None) == 1 and b"C=100" in lib.d2s_last_error()
    assert lib.d2s_gather_layernorm_varlen(p, p, None, p, p, 1, 2, 197, 384, 137, 1e-6, p, p, None) == 1
    assert b"null" in lib.d2s_last_error()
    assert lib.d2s_gather_layernorm_varlen(p, p, p, p, p, 1, 2, 197, 384, 197, 1e-6, p, p, None) == 1 and b"Kmax=197" in lib.d2s_last_error()
    assert lib.d2s_gather_layernorm_stats_varlen(p, p, None, 2, 197, 384, 137, 1e-6, p, p, None) == 1 and b"null" in lib.d2s_last_error()
    assert lib.d2s_gather_layernorm_stats_varlen(p, p, p, 2, 197, 380, 137, 1e-6, p, p, None) == 1 and b"D=380" in lib.d2s_last_error()
    assert d2s._lib.launch_count() == before
    # empty batches are a no-op, not an error
    assert lib.d2s_attn_varlen_fwd(p, p, 1, 0, 197, 6, 64, 0.125, p, None, None) == 0
    assert lib.d2s_threshold_select_varlen_f32(p, p, 0, 196, 0.3, p, p, p, None) == 0


def test_forward_varlen_rejects_training_mode_and_a_missing_threshold(d2s):
    C = fx.SMALL_CFG
    common = dict(patch_size=C["patch_size"], embed_dim=C["embed_dim"], depth=C["depth"], num_heads=C["num_heads"],
                  num_classes=C["num_classes"], topk_selection=True, predictor_loss_type="kl_div", small_predictor=True)
    m = d2s.variant_b.VisionTransformerDiffPruning(pruning_loc=[1, 2], token_ratio=[0.7, 0.49], patch_score_threshold=0.3, **common)
    x = torch.zeros(1, 3, 224, 224)
    with pytest.raises(ValueError, match="eval"):
        m.train().forward_varlen(x)
    m2 = d2s.variant_b.VisionTransformerDiffPruning(pruning_loc=[1, 2], token_ratio=[0.7, 0.49], **common).eval()
    with pytest.raises(ValueError, match="patch_score_threshold"):
        m2.forward_varlen(x)


# ----------------------------------------------------------------------------------------------------------------- kernels
def _qkv(lens, H, seed, dtype=torch.bfloat16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    B, T = len(lens), max(lens)
    return (torch.randn(B, T, 3 * H * 64, device="cuda", generator=g) * 0.8).to(dtype)


def _refill_pads(t, lens, seed):
    """t with every pad row (row >= lens[b]) replaced by other finite values."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    t = t.clone()
    for b, n in enumerate(lens):
        t[b, n:] = (torch.randn(t[b, n:].shape, device="cuda", generator=g) * 3).to(t.dtype)
    return t


def _check_attention_against_dense(ops, qkv, lens, H, exact_rows=True):
    Tmax = qkv.shape[1]
    out, cls = ops.attention_core(qkv, H, want_cls_row=True, lengths=_lens(lens))
    for b, n in enumerate(lens):
        o1, c1 = ops.attention_core(qkv[b:b + 1, :n].contiguous(), H, want_cls_row=True)
        if exact_rows and (n > 128) == (Tmax > 128):
            assert torch.equal(out[b, :n], o1[0]), (b, n)
            assert torch.equal(cls[b, :, :n], c1[0]), (b, n)
        else:
            torch.testing.assert_close(out[b, :n].float(), o1[0].float(), rtol=1e-2, atol=1e-2)
            torch.testing.assert_close(cls[b, :, :n], c1[0], rtol=1e-2, atol=2e-4)
        assert not out[b, n:].any() and not cls[b, :, n:].any(), (b, n)      # pad rows / columns are zeros
    return out, cls


@pytest.mark.gpu
@pytest.mark.parametrize("lens,H", [(LENS, 2), (LENS_SHORT, 3)])
def test_attention_varlen_matches_each_image_alone(d2s, lens, H):
    ops = d2s.ops
    qkv = _qkv(lens, H, seed=len(lens))
    out, cls = _check_attention_against_dense(ops, qkv, lens, H)
    # pad rows of qkv take no part: other finite values there change nothing
    out2, cls2 = ops.attention_core(_refill_pads(qkv, lens, 5), H, want_cls_row=True, lengths=_lens(lens))
    assert torch.equal(out, out2) and torch.equal(cls, cls2)


@pytest.mark.gpu
def test_attention_varlen_logits_far_above_the_first_chunk(d2s):
    """Short images of a long batch whose rows hold a logit more than 100 binades above the maximum of their first key chunk:
    the rare path redoes those rows from global qkv with the image's own length (and so never reads a pad row)."""
    ops = d2s.ops
    lens, H = [197, 150, 40], 2
    qkv = _qkv(lens, H, seed=11) * 0.1
    for b, j in ((1, 140), (2, 35)):                    # one key per image, outside chunk 0, for every query row of head 0
        qkv[b, :lens[b], 0:64] = 4.0                    # q (head 0)
        qkv[b, j, H * 64:H * 64 + 64] = 4.0             # k_j (head 0): q . k = 1024, 177 binades at scale 1/8
        qkv[b, lens[b]:, H * 64:H * 64 + 64] = 8.0      # pad keys larger still: must stay masked
    out, cls = _check_attention_against_dense(ops, qkv, lens, H)
    assert torch.isfinite(out).all() and torch.isfinite(cls).all()
    for b, j in ((1, 140), (2, 35)):
        assert float(cls[b, 0, j]) > 0.999            # the CLS row of head 0 puts all its mass on key j


@pytest.mark.gpu
@pytest.mark.parametrize("lens,H", [(LENS, 2), (LENS_SHORT, 1)])
def test_attention_varlen_fp32_simt_against_the_oracle(d2s, lens, H):
    from oracle import ops as oo
    ops = d2s.ops
    qkv = _qkv(lens, H, seed=3, dtype=torch.float32)
    out, cls = ops.attention_core(qkv, H, want_cls_row=True, lengths=_lens(lens))
    for b, n in enumerate(lens):
        ro, rc = oo.attention_core(qkv[b:b + 1, :n].cpu().view(1, n, 3, H, 64), H)
        torch.testing.assert_close(out[b:b + 1, :n].cpu(), ro, rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(cls[b:b + 1, :, :n].cpu(), rc, rtol=1e-4, atol=1e-6)
        assert not out[b, n:].any() and not cls[b, :, n:].any()


def _nan_pads(t, n):
    t = t.clone()
    for b, k in enumerate(n):
        t[b, k:] = float("nan")
    return t


@pytest.mark.gpu
def test_threshold_select_varlen_matches_each_prefix(d2s):
    ops = d2s.ops
    n = [196, 137, 96, 1, 0, 60]
    g = torch.Generator(device="cuda").manual_seed(7)
    raw = torch.rand(len(n), 196, device="cuda", generator=g)
    raw[:, 10:20] = raw[:, 30:40]                                      # ties
    for thr in (0.0, 0.3, 0.9, 2.0):
        score = _nan_pads(raw.softmax(-1), n)                          # NaN behind every prefix: never read
        mask, count, kept = ops.threshold_select(score, thr, want_indices=True, lengths=_lens(n))
        for b, k in enumerate(n):
            if k:
                m1, c1, k1 = ops.threshold_select(score[b:b + 1, :k], thr, want_indices=True)
                assert torch.equal(mask[b, :k], m1[0]) and torch.equal(count[b:b + 1], c1) and torch.equal(kept[b, :k], k1[0])
            else:
                assert int(count[b]) == 0
            assert not mask[b, k:].any() and bool((kept[b, k:] == -1).all())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("prob_mode", [0, 1])
def test_score_tail_b_varlen_matches_each_prefix(d2s, dtype, prob_mode):
    ops = d2s.ops
    n = [196, 137, 96, 1, 60]
    g = torch.Generator(device="cuda").manual_seed(9)
    C = 96
    h = _nan_pads(torch.randn(len(n), 196, C, device="cuda", generator=g).to(dtype), n)
    lw, lb = torch.rand(C, device="cuda", generator=g) + 0.5, torch.randn(C, device="cuda", generator=g) * 0.1
    W, bias = torch.randn(1, C, device="cuda", generator=g) * 0.2, torch.randn(1, device="cuda", generator=g)
    scores, probs = ops.score_tail_b_varlen(h, _lens(n), lw, lb, W, bias, 1e-5, prob_mode)
    for b, k in enumerate(n):
        s1, p1, _, _ = ops.score_tail_b(h[b:b + 1, :k], lw, lb, W, bias, 0, 1e-5, prob_mode, select=False)
        assert torch.equal(scores[b, :k], s1[0]) and torch.equal(probs[b, :k], p1[0]), b
        assert bool((scores[b, k:] == float("-inf")).all()) and not probs[b, k:].any()
    if prob_mode == 0:
        torch.testing.assert_close(probs.sum(-1), torch.ones(len(n), device="cuda"), rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pool_concat_varlen_matches_each_prefix(d2s, dtype):
    ops = d2s.ops
    n = [196, 137, 96, 1, 60]
    g = torch.Generator(device="cuda").manual_seed(13)
    z = _nan_pads(torch.randn(len(n), 196, 384, device="cuda", generator=g).to(dtype), n)
    got = ops.pool_concat_varlen_(z.clone(), _lens(n))
    for b, k in enumerate(n):
        ref = ops.pool_concat_(z[b:b + 1, :k].contiguous())
        assert torch.equal(got[b, :k], ref[0]), b
        assert bool(got[b, k:].isnan().all())                          # pad rows: neither read nor written


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_gather_layernorm_varlen_matches_each_image(d2s, dtype):
    ops = d2s.ops
    counts = [136, 0, 95, 1, 60]
    B, T_in, D, K = len(counts), 197, 384, max(counts)
    g = torch.Generator(device="cuda").manual_seed(17)
    x = torch.randn(B, T_in, D, device="cuda", generator=g).to(dtype)
    kept = torch.full((B, K), -1, dtype=torch.int64, device="cuda")
    for b, c in enumerate(counts):
        kept[b, :c] = torch.sort(torch.randperm(T_in - 1, device="cuda", generator=g)[:c])[0]
    w = (torch.rand(D, device="cuda", generator=g) + 0.5).to(dtype)
    bias = (torch.randn(D, device="cuda", generator=g) * 0.1).to(dtype)
    xs, xn = ops.gather_layernorm(x, kept, w, bias, 1e-6, counts=_lens(counts))
    stats = None
    if dtype == torch.bfloat16:
        xs2, stats = ops.gather_layernorm(x, kept, w, bias, 1e-6, want_stats=True, counts=_lens(counts))
        assert torch.equal(xs, xs2)
        stats = stats.view(B, K + 1, 2)
    for b, c in enumerate(counts):
        s1, n1 = ops.gather_layernorm(x[b:b + 1], kept[b:b + 1, :c].contiguous(), w, bias, 1e-6)
        assert torch.equal(xs[b, :c + 1], s1[0]) and torch.equal(xn[b, :c + 1], n1[0]), b
        assert not xs[b, c + 1:].any() and not xn[b, c + 1:].any()
        if stats is not None:
            _, st1 = ops.gather_layernorm(x[b:b + 1], kept[b:b + 1, :c].contiguous(), w, bias, 1e-6, want_stats=True)
            assert torch.equal(stats[b, :c + 1], st1), b
            pad = stats[b, c + 1:]
            assert not pad[:, 0].any() and bool(torch.isfinite(pad).all())    # a zero row: mean 0, rstd finite


# ----------------------------------------------------------------------------------------------------------------- guard zones
@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["attn_bf16", "attn_f32", "select", "tail", "pool", "gather", "gather_stats"])
def test_varlen_entry_points_stay_in_bounds(d2s, entry):
    """Outputs between sentinel zones and pre-poisoned, inputs with NaN behind them; two runs must agree bit for bit."""
    from test_gpu_guards import Guarded
    lib = d2s._lib
    g = torch.Generator(device="cuda").manual_seed(23)
    lens = [197, 150, 2, 97]
    B, Tmax = len(lens), max(lens)
    ln = Guarded((B,), torch.int32, torch.tensor(lens, dtype=torch.int32, device="cuda"), poison_after=True)
    spatial = Guarded((B,), torch.int32, torch.tensor([n - 1 for n in lens], dtype=torch.int32, device="cuda"), poison_after=True)
    results = []
    for _ in range(2):
        if entry.startswith("attn"):
            H, dt = 2, (torch.bfloat16 if entry == "attn_bf16" else torch.float32)
            qkv = Guarded((B, Tmax, 3 * H * 64), dt, torch.randn(B, Tmax, 3 * H * 64, device="cuda", generator=g.manual_seed(1)).to(dt),
                          poison_after=True)
            out, cls = Guarded((B, Tmax, H * 64), dt), Guarded((B, H, Tmax), torch.float32)
            lib.call("d2s_attn_varlen_fwd", qkv.ptr, ln.ptr, 1 if dt == torch.bfloat16 else 0, B, Tmax, H, 64, 0.125, out.ptr, cls.ptr,
                     _stream())
            outs, ins = [out, cls], [qkv]
        elif entry == "select":
            N = Tmax - 1
            sc = Guarded((B, N), torch.float32, torch.rand(B, N, device="cuda", generator=g.manual_seed(2)).softmax(-1), poison_after=True)
            mask, cnt, kept = Guarded((B, N), torch.uint8), Guarded((B,), torch.int32), Guarded((B, N), torch.int64)
            lib.call("d2s_threshold_select_varlen_f32", sc.ptr, spatial.ptr, B, N, 0.3, mask.ptr, cnt.ptr, kept.ptr, _stream())
            outs, ins = [mask, cnt, kept], [sc]
        elif entry == "tail":
            N, C = Tmax - 1, 64
            h = Guarded((B, N, C), torch.bfloat16, torch.randn(B, N, C, device="cuda", generator=g.manual_seed(3)).bfloat16(),
                        poison_after=True)
            w = Guarded((C,), torch.float32, torch.randn(C, device="cuda", generator=g.manual_seed(4)), poison_after=True)
            sc, pr = Guarded((B, N), torch.float32), Guarded((B, N), torch.float32)
            lib.call("d2s_score_tail_b_varlen", h.ptr, spatial.ptr, 1, B, N, C, w.ptr, w.ptr, 1e-5, w.ptr, None, 0, sc.ptr, pr.ptr,
                     _stream())
            outs, ins = [sc, pr], [h, w]
        elif entry == "pool":
            N, C = Tmax - 1, 384
            z = Guarded((B, N, C), torch.bfloat16, torch.randn(B, N, C, device="cuda", generator=g.manual_seed(5)).bfloat16(),
                        poison_after=True)
            lib.call("d2s_pool_concat_varlen_inplace", z.ptr, spatial.ptr, 1, B, N, C, _stream())
            outs, ins = [z], []
        else:
            D, K = 384, Tmax - 1
            x = Guarded((B, Tmax, D), torch.bfloat16, torch.randn(B, Tmax, D, device="cuda", generator=g.manual_seed(6)).bfloat16(),
                        poison_after=True)
            idx = torch.full((B, K), -1, dtype=torch.int64, device="cuda")
            cnt = [n - 1 for n in lens]
            for b, c in enumerate(cnt):
                idx[b, :c] = torch.arange(c, device="cuda").flip(0)
            kept = Guarded((B, K), torch.int64, idx, poison_after=True)
            gam = Guarded((D,), torch.bfloat16, torch.ones(D, device="cuda").bfloat16(), poison_after=True)
            xs = Guarded((B, K + 1, D), torch.bfloat16)
            if entry == "gather":
                xn = Guarded((B, K + 1, D), torch.bfloat16)
                lib.call("d2s_gather_layernorm_varlen", x.ptr, kept.ptr, spatial.ptr, gam.ptr, gam.ptr, 1, B, Tmax, D, K, 1e-6, xs.ptr,
                         xn.ptr, _stream())
                outs = [xs, xn]
            else:
                st = Guarded((B * (K + 1), 2), torch.float32)
                lib.call("d2s_gather_layernorm_stats_varlen", x.ptr, kept.ptr, spatial.ptr, B, Tmax, D, K, 1e-6, xs.ptr, st.ptr,
                         _stream())
                outs = [xs, st]
            ins = [x, kept, gam]
        torch.cuda.synchronize()
        for gd in outs + ins + [ln, spatial]:
            assert gd.ok(), entry
        results.append([o.t.clone() for o in outs])
    for a, b in zip(*results):
        assert torch.equal(a.view(torch.uint8) if a.dtype.is_floating_point else a,
                           b.view(torch.uint8) if b.dtype.is_floating_point else b), entry
    if entry != "pool":                                    # every output element written (no NaN / -1 poison left on valid rows)
        for o in results[0]:
            if o.dtype.is_floating_point and entry != "tail":
                assert not o.isnan().any(), entry


# ----------------------------------------------------------------------------------------------------------------- models
C = fx.SMALL_CFG
THR = 0.3


def _small_threshold_model(d2s, dev):
    m = d2s.variant_b.VisionTransformerDiffPruning(
        pruning_loc=[1, 2], token_ratio=[0.7, 0.49], distill=True, topk_selection=True, predictor_loss_type="kl_div",
        patch_score_threshold=THR, small_predictor=True, patch_size=C["patch_size"], embed_dim=C["embed_dim"], depth=C["depth"],
        num_heads=C["num_heads"], num_classes=C["num_classes"], mlp_ratio=4, qkv_bias=True)
    sd = fx.seeded_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, 131)
    m.load_state_dict(sd)
    return m.to(dev).eval(), sd


def _oracle_threshold_cls_attns(sd, cfg, img):
    """The oracle's threshold inference (variant_b_threshold_eval_intended) on one image, with the CLS attention rows of the
    blocks that are not pruning stages (what forward / forward_varlen return in that mode)."""
    from oracle import model as om
    from oracle import ops as oo
    x = om.embed(sd, cfg, img)
    rows, p = [], 0
    for i in range(cfg.depth):
        if i in cfg.pruning_loc:
            _, probs = oo.predictor_b(sd, f"score_predictor.{p}", x[:, 1:], cfg.small_predictor, cfg.predictor_bn,
                                      cfg.predictor_loss_type, False)
            kept = torch.nonzero(oo.threshold_keep_mask(probs, cfg.patch_score_threshold)[0]).flatten().unsqueeze(0)
            x = oo.gather_tokens_with_cls(x, kept)
            x = om.block(sd, cfg, i, x)
            p += 1
        else:
            x, ca = om.block(sd, cfg, i, x, want_cls_attn=True)
            rows.append(ca[:, :, 1:])
    return rows


@pytest.mark.gpu
def test_forward_varlen_fp32_matches_the_oracle_per_image(d2s, cuda_dev):
    from oracle import model as om
    model, sd = _small_threshold_model(d2s, cuda_dev)
    img = fx.randn(141, 10, 3, 224, 224)
    with torch.no_grad():
        logits, cls_attns, pred_logits, kept = model.forward_varlen(img.to(cuda_dev))
    counts = [[int((k[b] >= 0).sum()) for b in range(img.shape[0])] for k in kept]
    assert all(len(set(c)) > 1 for c in counts), counts                 # ragged at both stages: the test is not vacuous
    assert model.max_keep_ratio == max(counts[-1]) / 196 and model.min_keep_ratio == min(counts[-1]) / 196
    assert torch.equal((model.keep_ratios.cpu() * 196).round(), torch.tensor(counts[-1], dtype=torch.float32))
    cfg = om.VitCfg(embed_dim=C["embed_dim"], depth=C["depth"], num_heads=C["num_heads"], num_classes=C["num_classes"],
                    pruning_loc=[1, 2], token_ratio=[0.7, 0.49], small_predictor=True, patch_score_threshold=THR)
    for b in range(img.shape[0]):
        ref = om.variant_b_threshold_eval_intended(sd, cfg, img[b:b + 1])
        for s in range(2):
            c = counts[s][b]
            assert torch.equal(kept[s][b, :c].cpu(), ref["kept"][s][0]), (b, s)
            assert bool((kept[s][b, c:] == -1).all())
        torch.testing.assert_close(logits[b:b + 1].cpu(), ref["logits"], rtol=1e-4, atol=2e-5)
        rows = _oracle_threshold_cls_attns(sd, cfg, img[b:b + 1])
        assert len(rows) == len(cls_attns) == C["depth"] - 2
        for ca, rc in zip(cls_attns, rows):
            n = rc.shape[-1]
            torch.testing.assert_close(ca[b:b + 1, :, :n].cpu(), rc, rtol=1e-4, atol=1e-6)
            assert not ca[b, :, n:].any()
    # stage s's predictor logits: -inf exactly on the pad entries
    for s, pl in enumerate(pred_logits):
        nvalid = [196] * img.shape[0] if s == 0 else counts[s - 1]
        for b, n in enumerate(nvalid):
            assert bool(torch.isfinite(pl[b, :n]).all()) and bool((pl[b, n:] == float("-inf")).all())


def _deit_s_threshold_model(d2s, dev, thr):
    m = d2s.variant_b.VisionTransformerDiffPruning(
        pruning_loc=[3, 6, 9], token_ratio=[0.7, 0.49, 0.343], distill=True, topk_selection=True, predictor_loss_type="kl_div",
        patch_score_threshold=thr, num_classes=1000, patch_size=16, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, qkv_bias=True)
    sd = fx.seeded_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, 151)
    m.load_state_dict(sd)
    return m.to(dev).eval().to(torch.bfloat16)


def _cut_margin(probs, thr):
    """Distance of the threshold from the cumulative mass at the cut (sorted ascending, as the select does), in fp32."""
    cs = torch.cumsum(torch.sort(probs.float())[0], dim=-1)
    return float((cs - thr).abs().min())


@pytest.mark.gpu
def test_forward_varlen_bf16_fused_path_matches_batch_one(d2s, cuda_dev, monkeypatch):
    """DeiT-S widths, B = 64: forward_varlen on the batch against the batch-1 opt-in on each image.  Kept sets must agree except
    where the fp32 cumulative mass at an image's cut is within bf16 noise of the threshold (those images are excluded, and
    must be few); logits of the agreeing images meet the bf16 criterion.  The attention and GEMMs run on the d2s kernels."""
    model = _deit_s_threshold_model(d2s, cuda_dev, THR)
    img = fx.randn(161, 64, 3, 224, 224).to(cuda_dev, torch.bfloat16)
    calls = {"attn_varlen": 0, "linear_act": 0}
    attn, lin = d2s.ops.attention_core, d2s.ops.linear_act

    def attn_counted(*a, **k):
        calls["attn_varlen"] += k.get("lengths") is not None
        return attn(*a, **k)

    def lin_counted(*a, **k):
        calls["linear_act"] += 1
        return lin(*a, **k)
    monkeypatch.setattr(d2s.ops, "attention_core", attn_counted)
    monkeypatch.setattr(d2s.ops, "linear_act", lin_counted)
    n0 = d2s._lib.launch_count()
    with torch.no_grad():
        logits, _, pred_logits, kept = model.forward_varlen(img)
    assert calls["attn_varlen"] == 9                   # blocks 3..11 run on the variable-length attention kernel
    assert calls["linear_act"] >= 12                   # qkv projections (and fc1) on the tcgen05 GEMM
    assert d2s._lib.launch_count() - n0 >= 12 * 3      # qkv GEMM, attention, proj + LN, MLP per block
    counts = [[int((k[b] >= 0).sum()) for b in range(64)] for k in kept]
    assert all(len(set(c)) > 1 for c in counts), counts
    model.d2s_threshold_inference = True
    agree = 0
    for b in range(64):
        with torch.no_grad():
            lg1, _, pl1, kept1 = model(img[b:b + 1])
        same = True
        for s in range(3):
            c = counts[s][b]
            if not torch.equal(kept[s][b, :c], kept1[s][0]):
                probs = torch.softmax(pl1[s][0].float(), -1)
                assert _cut_margin(probs, THR) < 2e-2, (b, s)     # only a near-tie at the cut may flip
                same = False
                break
        if same:
            agree += 1
            d = logits[b].float() - lg1[0].float()
            l2, mx = float(d.norm() / lg1.float().norm()), float(d.abs().max() / lg1.float().abs().max())
            assert l2 < 1e-2 and mx < 2e-2, (b, l2, mx)
    assert agree >= 48, agree
