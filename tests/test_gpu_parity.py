"""GPU parity tests: every d2s kernel, called through the C ABI (ctypes via ops.py), against the CPU oracle
on the same seeded inputs, against the committed reference goldens, and - at BASELINE sizes - through
size-independent properties.  Integer/index results are bit-exact; float tolerances are stated per test
(north_star: 1e-4 relative in fp32, 1e-2 in bf16)."""
import pytest
import torch

import fixtures as fx
from oracle import ops as oo

pytestmark = pytest.mark.gpu

OPS, OPS_META = fx.load_npz("golden_ops.npz")
C = OPS_META["cases"]
FP32 = dict(rtol=1e-4, atol=1e-6)
BF16 = dict(rtol=1e-2, atol=1e-2)


@pytest.fixture(scope="module")
def ops(d2s, cuda_dev):
    return d2s.ops


def cu(t):
    return t.cuda()


# ------------------------------------------------------------------------------------------ select
@pytest.mark.parametrize("B,N,K", [(4, 196, 137), (3, 137, 96), (2, 96, 67), (1, 196, 58), (5, 196, 176),
                                   (2, 7, 3), (2, 300, 150), (1, 1024, 512), (3, 196, 0), (3, 196, 196)])
@pytest.mark.parametrize("order", [0, 1])
def test_select_bit_exact(ops, B, N, K, order):
    sc = torch.softmax(fx.randn(1000 + B * N + K, B, N), dim=-1)
    kept, dropped = ops.select_topk(cu(sc), K, order)
    rk, rd = oo.select_topk(sc, K, order)
    assert torch.equal(kept.cpu(), rk)
    if order == 0:
        assert torch.equal(dropped.cpu(), rd)


def test_select_ties_nan_signed_zero(ops):
    sc = torch.tensor([[0.5, 0.7, 0.5, 0.7, 0.1, float("nan"), -0.0, 0.0],
                       [1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0]])
    for order in (0, 1):
        kept, dropped = ops.select_topk(cu(sc), 4, order)
        rk, rd = oo.select_topk(sc, 4, order)
        assert torch.equal(kept.cpu(), rk), (order, kept, rk)
    # heavy ties: bf16-quantised softmax scores (SURVEY hard part 1)
    q = torch.softmax(fx.randn(7, 16, 196) * 0.02, dim=-1).bfloat16().float()
    kept, dropped = ops.select_topk(cu(q), 137, 0)
    rk, rd = oo.select_topk(q, 137, 0)
    assert torch.equal(kept.cpu(), rk) and torch.equal(dropped.cpu(), rd)


def test_select_golden_call_sites(ops):
    c = C["select"]
    sc = torch.softmax(fx.randn(c["seed"], *c["shape"]), dim=-1)
    kept, dropped = ops.select_topk(cu(sc), c["k"], 0)
    assert torch.equal(kept.cpu(), OPS["sel_keptB"]) and torch.equal(dropped.cpu(), OPS["sel_dropB"])
    kept, _ = ops.select_topk(cu(sc), c["k"], 1)
    assert torch.equal(kept.cpu(), OPS["sel_keptA"])


def test_select_full_size_properties(ops):
    B, N, K = 4096, 196, 137
    sc = torch.rand(B, N, generator=fx.gen(5)).cuda()
    kept, dropped = ops.select_topk(sc, K, 0)
    allidx = torch.cat([kept, dropped], dim=1).sort(dim=1).values
    assert torch.equal(allidx, torch.arange(N, device="cuda").expand(B, N))          # a partition of 0..N-1
    assert bool((kept[:, 1:] > kept[:, :-1]).all()) and bool((dropped[:, 1:] > dropped[:, :-1]).all())
    assert bool((sc.gather(1, kept).min(1).values >= sc.gather(1, dropped).max(1).values).all())
    kept_a, _ = ops.select_topk(sc, K, 1)
    va = sc.gather(1, kept_a)
    assert bool((va[:, 1:] <= va[:, :-1]).all())
    assert torch.equal(kept_a.sort(1).values, kept)


# ------------------------------------------------------------------------------------------ gather
@pytest.mark.parametrize("B,N", [(64, 196), (3, 137), (2, 1000), (5, 5), (1, 1)])
def test_threshold_select_bit_exact(ops, B, N):
    """d2s_threshold_select_f32 (the prefix-sum form of the select, dynamic_vit.py:880-890) against the oracle: keep masks,
    per-image counts and the ascending kept-index lists bit-exact, with tied scores and every threshold regime
    (nothing kept ... everything kept)."""
    g = fx.gen(40 + N)
    p = torch.softmax(torch.randn(B, N, generator=g) * 2.0, dim=-1)
    p[:, : N // 4] = p[:, N // 2: N // 2 + N // 4].clone() if N >= 4 else p[:, : N // 4]      # exact ties
    for thr in (-1.0, 0.0, 0.05, 0.3, 0.9, 0.999999, 1.5):
        mask, count, kept = ops.threshold_select(cu(p), thr, want_indices=True)
        ref = oo.threshold_keep_mask(p, thr)
        assert torch.equal(mask.cpu(), ref), thr
        assert torch.equal(count.cpu().long(), ref.sum(1)), thr
        for b in range(B):
            k = int(ref[b].sum())
            assert torch.equal(kept[b, :k].cpu(), torch.nonzero(ref[b]).flatten())
            assert bool((kept[b, k:] == -1).all())
        m2, c2 = ops.threshold_select(cu(p), thr)
        assert torch.equal(m2, mask) and torch.equal(c2, count)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,T,D,K", [(3, 197, 384, 137), (2, 138, 384, 96), (2, 97, 768, 67), (1, 197, 768, 176),
                                     (5, 197, 384, 58), (2, 10, 8, 4), (2, 197, 384, 0), (1, 2, 384, 1)])
def test_gather_scatter_bit_exact(ops, dtype, B, T, D, K):
    x = fx.randn(31 + T + D, B, T, D).to(dtype)
    kept = torch.stack([torch.randperm(T - 1, generator=fx.gen(40 + b))[:K].sort().values for b in range(B)]).long()
    out = ops.gather_tokens(cu(x), cu(kept), prepend_cls=True)
    ref = oo.gather_tokens_with_cls(x, kept)
    assert torch.equal(out.cpu(), ref)
    g = fx.randn(99, B, K + 1, D).to(dtype)
    gx = ops.scatter_tokens_bwd(cu(g), cu(kept), T, prepend_cls=True)
    assert torch.equal(gx.cpu(), oo.scatter_tokens_bwd(g, kept, T))


def test_batch_index_select_contract(ops):
    c = C["bis"]
    x = fx.randn(c["x_seed"], *c["x_shape"])
    assert torch.equal(ops.batch_index_select(cu(x), cu(OPS["bis3_idx"])).cpu(), OPS["bis3_out"])
    x2 = fx.randn(c["x2_seed"], *c["x2_shape"])
    assert torch.equal(ops.batch_index_select(cu(x2), cu(OPS["bis3_idx"])).cpu(), OPS["bis2_out"])
    with pytest.raises(NotImplementedError):
        ops.batch_index_select(torch.zeros(2, 2, 2, 2).cuda(), cu(OPS["bis3_idx"]))
    # prev_decision case: (B,196,1) fp32 goes through the scalar path; unsorted (score-order) indices
    pd = (torch.rand(4, 196, 1, generator=fx.gen(3)) > 0.5).float()
    idx = torch.stack([torch.randperm(196, generator=fx.gen(50 + b))[:137] for b in range(4)])
    assert torch.equal(ops.batch_index_select(cu(pd), cu(idx)).cpu(), oo.batch_index_select(pd, idx))


def test_gather_autograd_matches_torch_gather(ops):
    x = fx.randn(1, 3, 50, 64).cuda().requires_grad_(True)
    kept = torch.stack([torch.randperm(49, generator=fx.gen(60 + b))[:20].sort().values for b in range(3)]).cuda()
    up = fx.randn(2, 3, 21, 64).cuda()
    (ops.gather_tokens(x, kept) * up).sum().backward()
    g1 = x.grad.clone()
    x.grad = None
    rows = torch.cat([torch.zeros(3, 1, dtype=torch.long, device="cuda"), kept + 1], 1)
    (torch.gather(x, 1, rows.unsqueeze(-1).expand(-1, -1, 64)) * up).sum().backward()
    assert torch.equal(g1, x.grad)


def test_gather_full_size_roundtrip(ops):
    B, T, D, K = 1024, 197, 384, 137
    x = torch.randn(B, T, D, device="cuda", dtype=torch.bfloat16)
    sc = torch.rand(B, T - 1, device="cuda")
    kept, dropped = ops.select_topk(sc, K, 0)
    out = ops.gather_tokens(x, kept)
    rows = torch.cat([torch.zeros(B, 1, dtype=torch.long, device="cuda"), kept + 1], 1)
    assert torch.equal(out, torch.gather(x, 1, rows.unsqueeze(-1).expand(-1, -1, D)))
    back = ops.scatter_tokens_bwd(out, kept, T)
    assert torch.equal(ops.gather_tokens(back, kept), out)                       # gather(scatter(g)) == g
    assert float(ops.gather_tokens(back, dropped, prepend_cls=True)[:, 1:].float().abs().sum()) == 0.0


# ------------------------------------------------------------------------------------------ tails / gumbel
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_score_tail_a_eval(ops, dtype):
    B, N, Cc, K = 5, 196, 96, 137
    h = torch.nn.functional.gelu(fx.randn(71, B, N, Cc)).to(dtype)
    W, b = fx.randn(72, 2, Cc, scale=0.3), fx.randn(73, 2, scale=0.1)
    logp, kept = ops.score_tail_a(cu(h), cu(W), cu(b), k=K)
    ref = oo.score_tail_a(h.float(), W, b)
    torch.testing.assert_close(logp.cpu(), ref, rtol=1e-4, atol=1e-5)
    # indices are bit-exact w.r.t. the kernel's own scores (near-ties may legitimately differ from the oracle's)
    rk, _ = oo.select_topk(logp.cpu()[:, :, 0], K, oo.ORDER_SCORE_DESC)
    assert torch.equal(kept.cpu(), rk)


def test_score_tail_a_train_and_gumbel_golden(ops):
    c = C["gumbel"]
    logp = torch.log_softmax(fx.randn(c["logit_seed"], *c["shape"], scale=c["scale"]), dim=-1)
    lg = cu(logp).requires_grad_(True)
    hard = ops.gumbel_keep_decision(lg, cu(OPS["gum_noise"]), cu(OPS["gum_prev"]))
    assert torch.equal(hard.detach().cpu(), OPS["gum_hard"])                     # bit-exact decisions
    (hard * cu(fx.randn(c["up_seed"], 2, 50, 1))).sum().backward()
    torch.testing.assert_close(lg.grad.cpu(), OPS["gum_grad"], rtol=1e-4, atol=1e-7)
    # fused tail, train mode
    B, N, Cc = 3, 196, 96
    h = torch.nn.functional.gelu(fx.randn(74, B, N, Cc))
    W, b = fx.randn(75, 2, Cc, scale=0.3), fx.randn(76, 2, scale=0.1)
    g = -torch.log(-torch.log(torch.rand(B, N, 2, generator=fx.gen(77)).clamp_min(1e-9)))
    prev = (torch.rand(B, N, generator=fx.gen(78)) > 0.2).float()
    lp, dec, ys = ops.score_tail_a(cu(h), cu(W), cu(b), gumbel=cu(g), prev=cu(prev))
    torch.testing.assert_close(lp.cpu(), oo.score_tail_a(h, W, b), rtol=1e-4, atol=1e-5)
    rdec, rys = oo.gumbel_keep_decision(lp.cpu(), g, prev.unsqueeze(-1))
    assert torch.equal(dec.cpu(), rdec[..., 0])
    torch.testing.assert_close(ys.cpu(), rys, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("use_ln", [True, False])
@pytest.mark.parametrize("prob_mode", [0, 1])
def test_score_tail_b(ops, dtype, use_ln, prob_mode):
    B, N, Cc, K = 4, 196, 96, 137
    h = torch.relu(fx.randn(81, B, N, Cc)).to(dtype)
    lw, lb = (1 + 0.1 * fx.randn(82, Cc), 0.1 * fx.randn(83, Cc)) if use_ln else (None, None)
    W, b = fx.randn(84, 1, Cc, scale=0.3), fx.randn(85, 1, scale=0.1)
    scores, probs, kept, dropped = ops.score_tail_b(cu(h), None if lw is None else cu(lw), None if lb is None else cu(lb),
                                                    cu(W), cu(b), K, prob_mode=prob_mode)
    rs, rp = oo.score_tail_b(h.float(), lw, lb, W, b, "kl_div" if prob_mode == 0 else "bce")
    torch.testing.assert_close(scores.cpu(), rs, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(probs.cpu(), rp, rtol=1e-4, atol=1e-7)
    rk, rd = oo.select_topk(probs.cpu(), K, oo.ORDER_INDEX_ASC)
    assert torch.equal(kept.cpu(), rk) and torch.equal(dropped.cpu(), rd)


# ------------------------------------------------------------------------------------------ PerturbedTopK
@pytest.mark.parametrize("tag", ["ptk_small", "ptk_vit"])
def test_perturbed_topk_golden(ops, tag):
    c = C[tag]
    x = torch.softmax(fx.randn(c["x_seed"], c["b"], c["d"]), dim=-1)
    noise = fx.randn(c["noise_seed"], c["b"], c["ns"], c["d"])
    xg = cu(x).requires_grad_(True)
    ind = ops.perturbed_topk(xg, c["k"], c["ns"], c["sigma"], noise=cu(noise))
    assert torch.equal(ind.detach().cpu(), OPS[tag + "_ind"])                    # bit-exact vs the reference
    (ind * cu(fx.randn(c["gout_seed"], c["b"], c["k"], c["d"]))).sum().backward()
    torch.testing.assert_close(xg.grad.cpu(), OPS[tag + "_gx"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("B,N,K,S", [(1, 196, 98, 500), (8, 196, 98, 500), (3, 196, 137, 64), (2, 100, 1, 33),
                                     (2, 64, 64, 20), (70, 196, 98, 40), (300, 196, 58, 16)])
def test_perturbed_topk_vs_oracle(ops, B, N, K, S):
    x = torch.softmax(fx.randn(90, B, N), dim=-1)
    noise = fx.randn(91, B, S, N)
    ind, eg = oo.perturbed_topk_fwd(x, noise, K, 0.05)
    xg = cu(x).requires_grad_(True)
    out = ops.perturbed_topk(xg, K, S, 0.05, noise=cu(noise))
    assert torch.equal(out.detach().cpu(), ind)
    g = fx.randn(92, B, K, N)
    (out * cu(g)).sum().backward()
    torch.testing.assert_close(xg.grad.cpu(), oo.perturbed_topk_bwd(g, eg), rtol=1e-4, atol=1e-4)


def test_perturbed_topk_ties_and_rng(ops):
    # all-equal scores and zero noise: every sample picks the K lowest indices (tie rule)
    x = torch.zeros(2, 196).cuda()
    out = ops.perturbed_topk(x, 98, 10, 0.05, noise=torch.zeros(2, 10, 196).cuda())
    assert torch.equal(out, torch.eye(98, 196, device="cuda").expand(2, 98, 196))
    # in-kernel RNG contract: rows sum to 1, deterministic per seed, close to the injected-noise estimate
    xs = torch.softmax(fx.randn(93, 4, 196), dim=-1).cuda()
    a = ops.perturbed_topk(xs, 98, 500, 0.05, seed=1234)
    b = ops.perturbed_topk(xs, 98, 500, 0.05, seed=1234)
    c2 = ops.perturbed_topk(xs, 98, 500, 0.05, noise=torch.randn(4, 500, 196, device="cuda"))
    assert torch.equal(a, b)
    torch.testing.assert_close(a.sum(-1), torch.ones(4, 98, device="cuda"))
    assert float((a - c2).abs().max()) < 0.12 and float((a - c2).abs().mean()) < 4e-3
    # noise statistics of the Philox/Box-Muller stream, recovered from egrad of a constant score vector
    assert float(a.sum(1).mean()) == pytest.approx(0.5, abs=1e-3)


# ------------------------------------------------------------------------------------------ softmax_with_policy
def test_softmax_with_policy_golden_and_grads(ops):
    c = C["swp"]
    s = fx.randn(c["s_seed"], *c["s_shape"], scale=c["s_scale"])
    torch.testing.assert_close(ops.softmax_with_policy(cu(s), cu(OPS["swp_policy"])).cpu(), OPS["swp_out"], **FP32)
    torch.testing.assert_close(ops.softmax_with_policy(cu(s), cu(OPS["swp_policy_frac"])).cpu(), OPS["swp_out_frac"], **FP32)
    torch.testing.assert_close(ops.softmax_with_policy(cu(s), None).cpu(), torch.softmax(s, -1), **FP32)
    sg = cu(s).requires_grad_(True)
    pg = cu(OPS["swp_policy_frac"]).requires_grad_(True)
    (ops.softmax_with_policy(sg, pg) * cu(fx.randn(c["up_seed"], *c["s_shape"]))).sum().backward()
    torch.testing.assert_close(sg.grad.cpu(), OPS["swp_grad_s"], rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(pg.grad.cpu(), OPS["swp_grad_p"], rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("T", [197, 138, 68, 300])
def test_softmax_with_policy_sizes(ops, dtype, T):
    B, H = 2, 3
    s = (fx.randn(100 + T, B, H, T, T) * 2).to(dtype)
    pol = (torch.rand(B, T, 1, generator=fx.gen(101)) > 0.3).float()
    pol[:, 0] = 1
    out = ops.softmax_with_policy(cu(s), cu(pol))
    ref = oo.softmax_with_policy(s, pol)
    tol = FP32 if dtype == torch.float32 else dict(rtol=2e-2, atol=1e-3)
    torch.testing.assert_close(out.cpu().float(), ref.float(), **tol)
    if dtype == torch.float32:
        sg, pg = cu(s).requires_grad_(True), cu(pol).requires_grad_(True)
        up = fx.randn(102, B, H, T, T)
        (ops.softmax_with_policy(sg, pg) * cu(up)).sum().backward()
        s2, p2 = s.clone().requires_grad_(True), pol.clone().requires_grad_(True)
        (oo.softmax_with_policy(s2, p2) * up).sum().backward()
        torch.testing.assert_close(sg.grad.cpu(), s2.grad, rtol=1e-4, atol=1e-6)
        torch.testing.assert_close(pg.grad.cpu(), p2.grad, rtol=1e-4, atol=1e-5)


# ------------------------------------------------------------------------------------------ fused attention
def _qkv(seed, B, T, H, hd, scale=1.0):
    return fx.randn(seed, B, T, 3 * H * hd, scale=scale)


@pytest.mark.parametrize("T", [197, 138, 97, 68, 21, 1])
@pytest.mark.parametrize("with_policy", [False, True])
def test_attention_fp32_simt(ops, T, with_policy):
    B, H, hd = 2, 6, 64
    qkv = _qkv(110 + T, B, T, H, hd)
    pol = None
    if with_policy:
        pol = (torch.rand(B, T, generator=fx.gen(111)) > 0.3).float()
        pol[:, 0] = 1
    out, cls = ops.attention_core(cu(qkv), H, policy=None if pol is None else cu(pol), want_cls_row=True)
    ro, rc = oo.attention_core(qkv.view(B, T, 3, H, hd), H, policy=pol)
    torch.testing.assert_close(out.cpu(), ro, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(cls.cpu(), rc, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("T", [197, 138, 97, 68, 128, 129, 16, 5])
@pytest.mark.parametrize("with_policy", [False, True])
def test_attention_bf16_tcgen05(ops, T, with_policy):
    B, H, hd = 3, 6, 64
    qkv = _qkv(120 + T, B, T, H, hd).bfloat16()
    pol = None
    if with_policy:
        pol = (torch.rand(B, T, generator=fx.gen(121)) > 0.3).float()
        pol[:, 0] = 1
    out, cls = ops.attention_core(cu(qkv), H, policy=None if pol is None else cu(pol), want_cls_row=True)
    ro, rc = oo.attention_core(qkv.float().view(B, T, 3, H, hd), H, policy=pol)
    # bf16 operands, fp32 accumulate, bf16 probabilities: 1e-2 (north_star tolerance for bf16)
    torch.testing.assert_close(out.cpu().float(), ro, rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(cls.cpu(), rc, rtol=1e-2, atol=2e-4)


def test_attention_bf16_large_scores_and_full_batch(ops):
    # peaked rows (large logits), masked-max rows, and the BASELINE batch: compare with torch SDPA on device
    B, T, H, hd = 1024, 197, 6, 64
    qkv = torch.randn(B, T, 3 * H * hd, device="cuda", dtype=torch.bfloat16) * 2.0
    out, cls = ops.attention_core(qkv, H, want_cls_row=True)
    q, k, v = qkv.view(B, T, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)
    ref = torch.nn.functional.scaled_dot_product_attention(q.float(), k.float(), v.float()).transpose(1, 2).reshape(B, T, H * hd)
    torch.testing.assert_close(out.float(), ref, rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(cls.sum(-1), torch.ones(B, H, device="cuda"), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("T,with_policy", [(197, False), (197, True), (138, True), (97, False), (97, True), (40, True)])
def test_attention_bf16_logits_far_above_the_row_reference(ops, T, with_policy):
    """The single-pass softmax of the tcgen05 kernel takes its exponent reference from 16 columns of the row.  Rows whose
    maximum sits ~300 binades above those columns (logits of ~200 nats at columns 20 and T-27, ~50 nats inside the reference
    columns) must come out like any other row: the kernel raises the reference by whole binades and rescales what it has
    already produced, exactly.  Every second query is such a row, so lanes of one warp take both paths; at T = 197 without a
    policy the two large keys fall into different column halves (two warps per row)."""
    B, H, hd = 2, 6, 64
    g = fx.gen(130 + T)
    qkv = torch.randn(B, T, 3, H, hd, generator=g) * 0.5
    u = torch.nn.functional.normalize(torch.randn(hd, generator=g), dim=0)
    j1, j2 = 20, T - 13
    qkv[:, 0::2, 0] += 40.0 * u
    qkv[:, j1, 1] = 40.0 * u
    qkv[:, j2, 1] = 40.2 * u
    qkv[:, 5, 1] = 10.0 * u
    qkv = qkv.reshape(B, T, 3 * H * hd).bfloat16()
    pol = None
    if with_policy:
        pol = (torch.rand(B, T, generator=g) > 0.3).float()
        pol[:, 0] = 1
        pol[0, j1], pol[0, j2] = 1, 0          # image 0: the row maximum itself is masked out (the eps terms follow the true max)
        pol[1, j1], pol[1, j2] = 1, 1
    out, cls = ops.attention_core(cu(qkv), H, policy=None if pol is None else cu(pol), want_cls_row=True)
    ro, rc = oo.attention_core(qkv.float().view(B, T, 3, H, hd), H, policy=pol)
    s = torch.einsum("bihd,bjhd->bhij", qkv.float().view(B, T, 3, H, hd)[:, :, 0], qkv.float().view(B, T, 3, H, hd)[:, :, 1]) / 8
    assert float((s[:, :, 0::2].amax(-1) - s[:, :, 0::2, :16].amax(-1)).min()) > 100       # the case is really exercised
    assert bool(torch.isfinite(out).all())
    torch.testing.assert_close(out.cpu().float(), ro, rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(cls.cpu(), rc, rtol=1e-2, atol=2e-4)


@pytest.mark.parametrize("T,with_policy", [(197, True), (197, False), (138, True), (97, True), (16, False)])
def test_attention_bf16_row_statistics(d2s, T, with_policy):
    """`stats` of d2s_attn_policy_fwd: (m', 1/den, c/den) per query row reproduce the reference probabilities,
    P_ij = 2^(k2 s_ij - m') m_ij / den + c / den  (what d2s_attn_policy_bwd recomputes P from)."""
    B, H, hd = 2, 3, 64
    qkv = (fx.randn(140 + T, B, T, 3 * H * hd) * 0.8).bfloat16()
    pol = None
    if with_policy:
        pol = (torch.rand(B, T, generator=fx.gen(141 + T)) > 0.3).float()
        pol[:, 0] = 1
    q_d, out = cu(qkv), torch.empty(B, T, H * hd, dtype=torch.bfloat16, device="cuda")
    stats = torch.full((B, H, T, 4), float("nan"), device="cuda")
    pol_d = None if pol is None else cu(pol)
    d2s._lib.call("d2s_attn_policy_fwd", q_d.data_ptr(), None if pol is None else pol_d.data_ptr(), 1, B, T, H, hd, hd ** -0.5, 1e-6,
                  out.data_ptr(), None, stats.data_ptr(), torch.cuda.current_stream().cuda_stream)
    st = stats.cpu()
    assert bool(torch.isfinite(st[..., :3]).all())
    v = qkv.float().view(B, T, 3, H, hd)
    s = torch.einsum("bihd,bjhd->bhij", v[:, :, 0], v[:, :, 1]) * hd ** -0.5
    ref = oo.softmax_with_policy(s, pol.view(B, T, 1)) if pol is not None else torch.softmax(s, -1)
    k2s = s * 1.4426950408889634
    e = torch.exp2(k2s - st[..., 0:1])
    if pol is not None:
        e = e * (pol.view(B, 1, 1, T) + (1 - pol.view(B, 1, 1, T)) * torch.eye(T).view(1, 1, T, T))
    torch.testing.assert_close(e * st[..., 1:2] + st[..., 2:3], ref, rtol=2e-4, atol=1e-7)
    assert bool((st[..., 0] == st[..., 0].round()).all())            # the reference is a whole number of binades
    assert float((k2s.amax(-1) - st[..., 0]).max()) <= 101.0         # and never more than ~100 binades below the row maximum


def test_attention_train_full_batch_against_torch_autograd(ops):
    """BASELINE configs[2] shape (B = 256 per GPU, T = 197, 6 heads): forward + backward of the tcgen05 training attention
    against torch's fp32 autograd of the reference formulas on the same device; d policy sums 256 x 6 x 197 rows."""
    B, T, H, hd = 256, 197, 6, 64
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = (torch.randn(B, T, 3 * H * hd, device="cuda", generator=g) * 0.7).bfloat16()
    pol = (torch.rand(B, T, 1, device="cuda", generator=g) > 0.3).float()
    pol[:, 0] = 1
    go = (torch.randn(B, T, H * hd, device="cuda", generator=g) * 0.5).bfloat16()
    q1, p1 = qkv.clone().requires_grad_(True), pol.clone().requires_grad_(True)
    o1, _ = ops.attention_train(q1, H, policy=p1)
    (o1.float() * go.float()).sum().backward()
    q2, p2 = qkv.float().requires_grad_(True), pol.clone().requires_grad_(True)
    o2, _ = oo.attention_core(q2.view(B, T, 3, H, hd), H, policy=p2)
    (o2 * go.float()).sum().backward()
    torch.testing.assert_close(o1.detach().float(), o2.detach(), rtol=2e-2, atol=2e-2)
    assert float((q1.grad.float() - q2.grad).abs().max()) <= 3e-2 * float(q2.grad.abs().max())
    assert float((q1.grad.float() - q2.grad).norm()) <= 1e-2 * float(q2.grad.norm())
    assert float((p1.grad - p2.grad).abs().max()) <= 1e-2 * float(p2.grad.abs().max())
    assert float((p1.grad - p2.grad).norm()) <= 5e-3 * float(p2.grad.norm())


def test_attention_golden_module(d2s, ops):
    c = C["attn"]
    sd = fx.seeded_state_dict(c["shapes"], c["w_seed"])
    m = d2s.layers.Attention(c["dim"], num_heads=c["heads"], qkv_bias=True)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    x = cu(fx.randn(c["x_seed"], *c["x_shape"]))
    with torch.no_grad():
        o, ca = m(x, None, return_cls_attn=True)
        torch.testing.assert_close(o.cpu(), OPS["attn_out"], **FP32)
        torch.testing.assert_close(ca.cpu(), OPS["attn_cls"], **FP32)
        o, ca = m(x, cu(OPS["attn_policy"]), return_cls_attn=True)
        torch.testing.assert_close(o.cpu(), OPS["attn_out_pol"], **FP32)
        torch.testing.assert_close(ca.cpu(), OPS["attn_cls_pol"], **FP32)
    # autograd path gives the same forward
    o2, ca2 = m(x.requires_grad_(True), cu(OPS["attn_policy"]), return_cls_attn=True)
    torch.testing.assert_close(o2.detach().cpu(), OPS["attn_out_pol"], **FP32)


# ------------------------------------------------------------------------------------------ add + LayerNorm
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,T,D", [(3, 197, 384), (2, 138, 768), (5, 68, 128), (2, 197, 192), (1, 1, 384), (33, 7, 1536)])
@pytest.mark.parametrize("with_y,row0", [(True, 0), (False, 0), (True, 1), (False, 1)])
def test_add_layernorm(ops, dtype, B, T, D, with_y, row0):
    if dtype == torch.float32 and D > 768:
        pytest.skip("fp32 rows are limited to D <= 768")
    if row0 >= T:
        pytest.skip("nothing to normalise")
    x = (fx.randn(130 + D, B, T, D) * 2 + 0.5).to(dtype)
    y = fx.randn(131 + T, B, T, D).to(dtype) if with_y else None
    w, b = (1 + 0.1 * fx.randn(132, D)).to(dtype), (0.1 * fx.randn(133, D)).to(dtype)
    s, h = ops.add_layernorm(cu(x), None if y is None else cu(y), cu(w), cu(b), 1e-6, norm_row0=row0)
    rs, rh = oo.add_layernorm(x, y, w, b, 1e-6, norm_row0=row0)
    assert torch.equal(s.cpu(), rs)                                    # the residual sum is bit-exact
    tol = dict(rtol=1e-5, atol=1e-5) if dtype == torch.float32 else dict(rtol=1.6e-2, atol=1e-2)   # bf16: 1 ulp
    torch.testing.assert_close(h.cpu().float(), rh.float(), **tol)


def test_add_layernorm_strided_view_and_full_size(ops):
    B, T, D = 1024, 197, 384
    x = torch.randn(B, T, D, device="cuda", dtype=torch.bfloat16)
    y = torch.randn(B, T, D, device="cuda", dtype=torch.bfloat16)
    ln = torch.nn.LayerNorm(D, eps=1e-6).cuda().bfloat16()
    torch.nn.init.normal_(ln.weight, 1.0, 0.1)
    torch.nn.init.normal_(ln.bias, 0.0, 0.1)
    s, h = ops.add_layernorm(x, y, ln.weight, ln.bias, ln.eps)
    assert torch.equal(s, x + y)
    torch.testing.assert_close(h.float(), ln(x + y).float(), rtol=1.6e-2, atol=1e-2)
    # token-slice view (the predictors normalise x[:, 1:]) and the CLS-only view used by the eval heads
    _, h1 = ops.add_layernorm(x, y, ln.weight, ln.bias, ln.eps, norm_row0=1)
    assert torch.equal(h1, h[:, 1:])
    _, h0 = ops.add_layernorm(x[:, :1], y[:, :1].contiguous(), ln.weight, ln.bias, ln.eps, want_sum=False)
    assert torch.equal(h0, h[:, :1])
    _, hs = ops.add_layernorm(x[:, 1:], None, ln.weight, ln.bias, ln.eps)
    torch.testing.assert_close(hs.float(), ln(x[:, 1:]).float(), rtol=1.6e-2, atol=1e-2)


@pytest.mark.parametrize("xd,hd", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16)])
@pytest.mark.parametrize("rows,D", [(3 * 197, 384), (1000, 768), (37, 128), (5, 8)])
def test_layer_norm_autograd(ops, xd, hd, rows, D):
    x = (fx.randn(190 + D, rows, D) * 1.5 + 0.3).to(xd)
    w, b = 1 + 0.1 * fx.randn(191, D), 0.1 * fx.randn(192, D)
    up = fx.randn(193, rows, D).to(hd)
    xg, wg, bg = cu(x).requires_grad_(True), cu(w).requires_grad_(True), cu(b).requires_grad_(True)
    h = ops.layer_norm(xg, wg, bg, 1e-6, out_dtype=hd)
    assert h.dtype == hd
    (h.float() * cu(up).float()).sum().backward()
    x2, w2, b2 = x.double().requires_grad_(True), w.double().requires_grad_(True), b.double().requires_grad_(True)
    h2 = torch.nn.functional.layer_norm(x2, (D,), w2, b2, 1e-6)
    (h2 * up.double()).sum().backward()
    lo = hd == torch.bfloat16 or xd == torch.bfloat16
    torch.testing.assert_close(h.detach().cpu().double(), h2.detach(), rtol=1.6e-2 if lo else 1e-5, atol=1e-2 if lo else 1e-5)
    def rel(a, r):
        return float((a.cpu().double() - r).abs().max() / r.abs().max())
    assert rel(xg.grad, x2.grad) < (2e-2 if xd == torch.bfloat16 else 1e-4)
    assert rel(wg.grad, w2.grad) < 1e-4 and rel(bg.grad, b2.grad) < 1e-4


@pytest.mark.parametrize("xd,hd", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16)])
@pytest.mark.parametrize("rows,D", [(3 * 197, 384), (1000, 768), (37, 128)])
def test_add_layer_norm_train_autograd(ops, xd, hd, rows, D):
    """(s, h) = (x + y, LayerNorm(x + y)) as one kernel each way, against torch autograd in float64 on the same inputs:
    s exact (one rounding of the sum), h, and the gradients of x, y (identical), weight, bias with s and h BOTH used downstream."""
    x = (fx.randn(290 + D, rows, D) * 1.5 + 0.3).to(xd)
    y = fx.randn(291 + D, rows, D).to(xd)
    w, b = 1 + 0.1 * fx.randn(292, D), 0.1 * fx.randn(293, D)
    up_h, up_s = fx.randn(294, rows, D).to(hd), fx.randn(295, rows, D).to(xd)
    xg, yg = cu(x).requires_grad_(True), cu(y).requires_grad_(True)
    wg, bg = cu(w).requires_grad_(True), cu(b).requires_grad_(True)
    s, h = ops.add_layer_norm_train(xg, yg, wg, bg, 1e-6, out_dtype=hd)
    assert s.dtype == xd and h.dtype == hd
    assert torch.equal(s.detach().cpu(), x + y)
    ((h.float() * cu(up_h).float()).sum() + (s.float() * cu(up_s).float()).sum()).backward()
    assert torch.equal(xg.grad, yg.grad)
    s2 = (x + y).double().requires_grad_(True)
    w2, b2 = w.double().requires_grad_(True), b.double().requires_grad_(True)
    h2 = torch.nn.functional.layer_norm(s2, (D,), w2, b2, 1e-6)
    ((h2 * up_h.double()).sum() + (s2 * up_s.double()).sum()).backward()
    lo = hd == torch.bfloat16 or xd == torch.bfloat16
    torch.testing.assert_close(h.detach().cpu().double(), h2.detach(), rtol=1.6e-2 if lo else 1e-5, atol=1e-2 if lo else 1e-5)
    def rel(a, r):
        return float((a.cpu().double() - r).abs().max() / r.abs().max())
    assert rel(xg.grad, s2.grad) < (2e-2 if xd == torch.bfloat16 else 1e-4)
    assert rel(wg.grad, w2.grad) < 1e-4 and rel(bg.grad, b2.grad) < 1e-4
    # only s used downstream: the gradient passes straight through
    xg2, yg2 = cu(x).requires_grad_(True), cu(y).requires_grad_(True)
    s3, _ = ops.add_layer_norm_train(xg2, yg2, wg, bg, 1e-6, out_dtype=hd)
    (s3.float() * cu(up_s).float()).sum().backward()
    assert torch.equal(xg2.grad.cpu(), up_s) and torch.equal(yg2.grad.cpu(), up_s)


# ------------------------------------------------------------------------------------------ predictor body, embed
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,N,Cc", [(3, 196, 384), (2, 137, 768), (2, 96, 128), (1, 5, 1536)])
@pytest.mark.parametrize("with_policy", [True, False])
def test_pool_act(ops, dtype, B, N, Cc, with_policy):
    if dtype == torch.float32 and Cc > 1024:
        pytest.skip("fp32 rows are limited to C <= 1024")
    z = (fx.randn(140 + Cc, B, N, Cc) * 1.5).to(dtype)
    pol = (torch.rand(B, N, generator=fx.gen(141)) > 0.3).float() if with_policy else None
    if pol is not None:
        pol[:, 0] = 1
    local, pooled = ops.pool_act(cu(z), None if pol is None else cu(pol), ops.ACT_GELU)
    rl, rp = oo.pool_act(z, pol, "gelu")
    tol = dict(rtol=1e-5, atol=1e-6) if dtype == torch.float32 else dict(rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(local.cpu().float(), rl.float(), **tol)
    torch.testing.assert_close(pooled.cpu().float(), rp.float(), **tol)
    l2, p2 = ops.pool_act(cu(z), None, ops.ACT_RELU)
    rl2, rp2 = oo.pool_act(z, None, "relu")
    assert torch.equal(l2.cpu(), rl2)                                      # ReLU halves are bit-exact
    torch.testing.assert_close(p2.cpu().float(), rp2.float(), **tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,N,Cc", [(3, 196, 384), (2, 137, 768), (1, 5, 64)])
def test_pool_act_pooled_only(ops, dtype, B, N, Cc):
    """want_local=False (an already activated tensor whose local half is read in place by the next kernel): the pooled rows are
    BIT-identical to the two-output call's, nothing else is written."""
    z = (fx.randn(160 + Cc, B, N, Cc) * 1.5).to(dtype)
    pol = (torch.rand(B, N, generator=fx.gen(161)) > 0.3).float()
    pol[:, 0] = 1
    for act in (ops.ACT_NONE, ops.ACT_GELU):
        _, p_both = ops.pool_act(cu(z), cu(pol), act)
        none, p_only = ops.pool_act(cu(z), cu(pol), act, want_local=False)
        assert none is None
        torch.testing.assert_close(p_only, p_both, rtol=2e-3, atol=2e-3)      # (the token groups sum in a different order)
    _, rp = oo.pool_act(z, pol, "gelu")
    tol = dict(rtol=1e-5, atol=1e-6) if dtype == torch.float32 else dict(rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(p_only.cpu().float(), rp.float(), **tol)


def test_predictor_a_tail_reads_a_column_slice_in_place(ops):
    """local given as the first 192 columns of a (B, N, 384) tensor (the Linear + GELU GEMM's output): identical results to the
    dense copy, no copy made (the tensor map carries the row stride)."""
    B, N, K = 5, 196, 137
    local, per_image, w2, w3, b3, w4, b4, prev = _tail_inputs(B, N, 990)
    wide = torch.cat([local, torch.full_like(local, float("nan"))], dim=-1)      # whatever sits in the other half is never read
    wide_c = cu(wide)
    a = ops.predictor_a_tail(wide_c[:, :, :192], cu(per_image), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), K, prev=cu(prev))
    b = ops.predictor_a_tail(cu(local), cu(per_image), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), K, prev=cu(prev))
    assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_bias_act_and_split_linear_identity(ops, dtype):
    B, N, Cc = 4, 196, 192
    u = fx.randn(150, B, N, Cc).to(dtype)
    bias = fx.randn(151, B, Cc).to(dtype)
    out = ops.bias_act_(cu(u).clone(), cu(bias), ops.ACT_GELU)
    tol = dict(rtol=1e-5, atol=1e-6) if dtype == torch.float32 else dict(rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(out.cpu().float(), oo.bias_act(u, bias, "gelu").float(), **tol)
    shared = fx.randn(152, Cc).to(dtype)
    out = ops.bias_act_(cu(u).clone(), cu(shared), ops.ACT_NONE)
    assert torch.equal(out.cpu(), u + shared)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,N,Cc", [(3, 196, 1536), (2, 137, 384), (2, 5, 64)])
def test_pool_concat_inplace(ops, dtype, B, N, Cc):
    if dtype == torch.float32 and Cc > 1024:
        pytest.skip("fp32 rows are limited")
    z = torch.relu(fx.randn(165 + Cc, B, N, Cc)).to(dtype)
    half = Cc // 2
    ref = torch.cat([z[..., :half], z[..., half:].float().mean(dim=1, keepdim=True).to(dtype).expand(B, N, half)], dim=-1)
    out = ops.pool_concat_(cu(z).clone())
    assert torch.equal(out.cpu()[..., :half], ref[..., :half])
    torch.testing.assert_close(out.cpu()[..., half:].float(), ref[..., half:].float(), rtol=1e-2 if dtype == torch.bfloat16 else 1e-5,
                               atol=1e-2 if dtype == torch.bfloat16 else 1e-6)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_assemble_tokens(ops, dtype):
    B, N, D = 5, 196, 384
    pe, cls, pos = fx.randn(160, B, N, D).to(dtype), fx.randn(161, 1, 1, D).to(dtype), fx.randn(162, 1, N + 1, D).to(dtype)
    out = ops.assemble_tokens(cu(pe), cu(cls), cu(pos))
    assert torch.equal(out.cpu(), oo.assemble_tokens(pe, cls, pos))            # one rounding per element: bit-exact


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_patchify_bit_exact(ops, dtype):
    B, Cc, Hh, Ww, p = 3, 3, 224, 224, 16
    img = fx.randn(180, B, Cc, Hh, Ww).to(dtype)
    ref = img.view(B, Cc, Hh // p, p, Ww // p, p).permute(0, 2, 4, 1, 3, 5).reshape(B, (Hh // p) * (Ww // p), Cc * p * p)
    assert torch.equal(ops.patchify(cu(img), p, p).cpu(), ref)
    img2 = fx.randn(181, 2, 1, 32, 64).to(dtype)
    ref2 = img2.view(2, 1, 4, 8, 4, 16).permute(0, 2, 4, 1, 3, 5).reshape(2, 16, 128)
    assert torch.equal(ops.patchify(cu(img2), 8, 16).cpu(), ref2)
    img3 = fx.randn(183, 2, 3, 32, 1024).to(dtype)          # a band wider than 48 KB of shared memory: the one-vector-per-thread kernel
    ref3 = img3.view(2, 3, 2, 16, 64, 16).permute(0, 2, 4, 1, 3, 5).reshape(2, 128, 768)
    assert torch.equal(ops.patchify(cu(img3), 16, 16).cpu(), ref3)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,C,H,W,p", [(3, 3, 224, 224, 16), (2, 1, 32, 64, 8), (1, 3, 48, 32, 16)])
def test_patchify_u8_is_totensor_normalize_im2col_bit_exact(ops, dtype, B, C, H, W, p):
    """Raw uint8 pixels -> normalised patches: bit-identical to torch's x / 255, (x - mean) / std in fp32, cast, im2col."""
    u8 = torch.randint(0, 256, (B, C, H, W), generator=fx.gen(330 + H), dtype=torch.uint8)
    u8[0, 0, 0, :16] = torch.arange(240, 256, dtype=torch.uint8)
    mean, std = torch.tensor([0.485, 0.456, 0.406][:C]), torch.tensor([0.229, 0.224, 0.225][:C])
    out = ops.patchify_u8(cu(u8), p, p, cu(mean), cu(std), out_dtype=dtype)
    x = ((u8.float().div(255.0) - mean.view(1, C, 1, 1)) / std.view(1, C, 1, 1)).to(dtype)
    ref = x.view(B, C, H // p, p, W // p, p).permute(0, 2, 4, 1, 3, 5).reshape(B, (H // p) * (W // p), C * p * p)
    assert torch.equal(out.cpu(), ref)


def test_gelu_inplace_matches_exact_erf(ops):
    u = (fx.randn(182, 64, 197, 1536) * 2.0)
    ref = torch.nn.functional.gelu(u)
    out32 = ops.bias_act_(cu(u).clone(), None, ops.ACT_GELU)
    torch.testing.assert_close(out32.cpu(), ref, rtol=1e-5, atol=5e-6)           # fp32: erff
    ub = u.bfloat16()
    outb = ops.bias_act_(cu(ub).clone(), None, ops.ACT_GELU)
    refb = torch.nn.functional.gelu(ub.float())
    # bf16: erf evaluated to ~1e-6 absolute, result rounded to bf16 -> within one bf16 ulp of the exactly rounded value
    err = (outb.cpu().float() - refb).abs()
    assert bool((err <= refb.abs() * 2 ** -7 + 1e-6).all())
    core = ub.float() > -3.0          # outside the far negative tail (|gelu| < 4e-3) the rounded results are identical
    assert float((outb.cpu().float() != refb.bfloat16().float())[core].float().mean()) < 1e-4


@pytest.mark.parametrize("M,N,K,act", [(1000, 1536, 384, 1), (256, 256, 64, 1), (77, 512, 128, 0), (3 * 197, 1536, 384, 2),
                                       (20000, 1536, 384, 1), (513, 3072, 768, 1), (129, 256, 64, 0), (128, 256, 64, 1),
                                       (1000, 384, 384, 1), (3 * 196 + 5, 384, 384, 1), (257, 192, 64, 0), (20000, 384, 384, 2),
                                       (300, 576, 128, 1)])
def test_linear_act_pair_gemm(ops, M, N, K, act):
    """CTA-pair (cta_group::2) variant of the fc1 GEMM: same contract, ragged row tails in either CTA of the pair."""
    x = (fx.randn(210 + M % 97, M, K) * 1.0).bfloat16()
    w = (fx.randn(211 + N % 89, N, K) / K ** 0.5).bfloat16()
    b = (fx.randn(212, N) * 0.2).bfloat16()
    out = ops.linear_act(cu(x), cu(w), cu(b), act)
    ref = torch.nn.functional.linear(x.float(), w.float(), b.float())
    ref = torch.nn.functional.gelu(ref) if act == 1 else (torch.relu(ref) if act == 2 else ref)
    torch.testing.assert_close(out.cpu().float(), ref, rtol=1e-2, atol=1e-2)
    assert out.shape == (M, N) and out.dtype == torch.bfloat16


@pytest.mark.parametrize("M,N,K", [(1000, 1536, 384), (50432, 1536, 384), (77, 256, 64), (777, 384, 384)])
def test_linear_act_pair_gemm_second_output(ops, M, N, K):
    """Training forward of fc1 -> GELU: the same GEMM also writes the Linear's own output (GELU' needs it)."""
    x = (fx.randn(220 + M % 97, M, K) * 1.0).bfloat16()
    w = (fx.randn(221 + N % 89, N, K) / K ** 0.5).bfloat16()
    b = (fx.randn(222, N) * 0.2).bfloat16()
    out, pre = ops.linear_act(cu(x), cu(w), cu(b), 1, want_pre=True)
    ref = torch.nn.functional.linear(x.float(), w.float(), b.float())
    torch.testing.assert_close(pre.cpu().float(), ref, rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(out.cpu().float(), torch.nn.functional.gelu(ref), rtol=1e-2, atol=1e-2)
    assert torch.equal(out, ops.linear_act(cu(x), cu(w), cu(b), 1))


def test_gelu_epilogue_is_erf_gelu_to_one_bf16_ulp(ops):
    """The epilogue's GELU (erfcx polynomial x one ex2) against float64 erf GELU of the exact pre-activation: identity
    weights make the accumulator exact, so any deviation is the activation's.  <= 1 bf16 ulp down to x = -5.6 (the
    negative tail included: |GELU| ~ 6e-8 there); below that the polynomial's argument is clamped and only |err| < 1e-8 holds."""
    K = N = 256
    xs = torch.linspace(-6.0, 6.0, 512 * K).reshape(512, K).bfloat16()
    w = torch.eye(N, K).bfloat16()
    out = ops.linear_act(cu(xs), cu(w), None, 1).cpu().double()
    x64 = xs.double()
    ref = 0.5 * x64 * torch.special.erfc(-x64 / 2 ** 0.5)
    ulp = torch.maximum(ref.abs(), torch.tensor(1e-30, dtype=torch.float64)) * 2.0 ** -8
    bad = ((out - ref).abs() > 1.001 * ulp) & (x64 >= -5.6)
    assert not bool(bad.any()), (xs[bad][:5], out[bad][:5], ref[bad][:5])
    assert float((out - ref).abs()[x64 < -5.6].max()) < 1e-8


def _residual_ln_reference(a, w, b, x, g, bt, eps):
    y = torch.nn.functional.linear(a.float(), w.float(), None if b is None else b.float()).bfloat16()     # Linear output, bf16
    s = (x.float() + y.float()).bfloat16()                                                              # residual add, bf16
    return s, y


@pytest.mark.parametrize("M,N,K", [(256, 384, 384), (1000, 384, 384), (77, 384, 1536), (3 * 197, 384, 1536), (20000, 384, 384),
                                   (130, 192, 192), (1000, 192, 768), (5 * 138, 384, 64),
                                   (256, 768, 768), (1000, 768, 768), (77, 768, 3072), (3 * 197, 768, 3072), (20000, 768, 768), (5 * 138, 768, 64)])
def test_linear_residual_ln(ops, M, N, K):
    """proj / fc2 + residual + next LayerNorm (dynamic_vit.py:263-283) in one kernel vs the three separate bf16 ops."""
    a = fx.randn(300 + M % 91, M, K).bfloat16()
    w = (fx.randn(301 + K % 83, N, K) / K ** 0.5).bfloat16()
    b = (fx.randn(302, N) * 0.2).bfloat16()
    x = (fx.randn(303 + M % 7, M, N) * 1.5).bfloat16()
    g = (1.0 + 0.3 * fx.randn(304, N)).bfloat16()
    bt = (0.2 * fx.randn(305, N)).bfloat16()
    s, h = ops.linear_residual_ln(cu(a), cu(w), cu(b), cu(x), cu(g), cu(bt), 1e-6)
    s, h = s.cpu(), h.cpu()
    s_ref, _ = _residual_ln_reference(a, w, b, x, g, bt, 1e-6)
    # fp32 accumulation order differs from the CPU matmul: a few results land on the other side of a bf16 rounding boundary
    # (one bf16 ulp of the Linear output y, |y| < 8, survives a cancelling residual add: atol = 2^-5)
    torch.testing.assert_close(s.float(), s_ref.float(), rtol=1e-2, atol=3.2e-2)
    assert float((s == s_ref).float().mean()) > 0.98
    # the LayerNorm is exact on the kernel's own residual sum
    h_ref = torch.nn.functional.layer_norm(s.float(), (N,), g.float(), bt.float(), 1e-6)
    torch.testing.assert_close(h.float(), h_ref, rtol=8e-3, atol=8e-3)
    assert float((h == h_ref.bfloat16()).float().mean()) > 0.97
    s2, none = ops.linear_residual_ln(cu(a), cu(w), cu(b), cu(x), want_norm=False)
    assert none is None and torch.equal(s2.cpu(), s)


@pytest.mark.parametrize("M,HID", [(256, 1536), (1000, 1536), (77, 1536), (3 * 197, 1536), (20000, 1536), (513, 128), (300, 768), (5 * 77, 1536)])
def test_mlp_residual_ln_fused(ops, M, HID):
    """fc1 + GELU + fc2 + residual + next LayerNorm (dynamic_vit.py:159-175, :263-283) in one kernel vs the separate bf16 ops
    (each intermediate rounded to bf16 like the reference's modules)."""
    D = 384
    h = fx.randn(700 + M % 91, M, D).bfloat16()
    w1 = (fx.randn(701, HID, D) / D ** 0.5).bfloat16()
    b1 = (fx.randn(702, HID) * 0.2).bfloat16()
    w2 = (fx.randn(703, D, HID) / HID ** 0.5).bfloat16()
    b2 = (fx.randn(704, D) * 0.2).bfloat16()
    x = (fx.randn(705 + M % 7, M, D) * 1.5).bfloat16()
    g = (1.0 + 0.3 * fx.randn(706, D)).bfloat16()
    bt = (0.2 * fx.randn(707, D)).bfloat16()
    s, hn = ops.mlp_residual_ln(cu(h), cu(w1), cu(b1), cu(w2), cu(b2), cu(x), cu(g), cu(bt), 1e-6)
    s, hn = s.cpu(), hn.cpu()
    u = torch.nn.functional.gelu(torch.nn.functional.linear(h.float(), w1.float(), b1.float())).bfloat16()
    y = torch.nn.functional.linear(u.float(), w2.float(), b2.float()).bfloat16()
    s_ref = (x.float() + y.float()).bfloat16()
    torch.testing.assert_close(s.float(), s_ref.float(), rtol=1e-2, atol=3.2e-2)
    assert float((s == s_ref).float().mean()) > 0.95      # bf16 flips of u (1 ulp) propagate into a few sums
    hn_ref = torch.nn.functional.layer_norm(s.float(), (D,), g.float(), bt.float(), 1e-6)
    torch.testing.assert_close(hn.float(), hn_ref, rtol=8e-3, atol=8e-3)
    s2, none = ops.mlp_residual_ln(cu(h), cu(w1), cu(b1), cu(w2), cu(b2), cu(x), want_norm=False)
    assert none is None and torch.equal(s2.cpu(), s)
    if M % 77 == 0:   # the predictors' norm over x[:, 1:]: images of 77 tokens, CLS rows skipped and the output compacted
        Bn, Tn = M // 77, 77
        s3, h3 = ops.mlp_residual_ln(cu(h).view(Bn, Tn, D), cu(w1), cu(b1), cu(w2), cu(b2), cu(x).view(Bn, Tn, D), cu(g), cu(bt), 1e-6,
                                     norm_row0=1)
        assert h3.shape == (Bn, Tn - 1, D) and torch.equal(s3.cpu().view(M, D), s)
        assert torch.equal(h3.cpu(), hn.view(Bn, Tn, D)[:, 1:])


@pytest.mark.parametrize("B,T,D,K,dtype", [(3, 197, 384, 137, torch.bfloat16), (2, 138, 384, 96, torch.float32), (1, 9, 64, 0, torch.float32),
                                            (2, 197, 768, 196, torch.bfloat16)])
def test_gather_layernorm_fused(ops, B, T, D, K, dtype):
    """Kept-token gather + next LayerNorm in one kernel: the gathered rows bit-exact, the norm as add_layernorm's."""
    x = fx.randn(800 + T, B, T, D).to(dtype)
    kept = torch.stack([torch.sort(torch.randperm(T - 1, generator=fx.gen(801 + b))[:K])[0] for b in range(B)]).long()
    g = (1.0 + 0.3 * fx.randn(802, D)).to(dtype)
    bt = (0.2 * fx.randn(803, D)).to(dtype)
    xg, h = ops.gather_layernorm(cu(x), cu(kept), cu(g), cu(bt), 1e-6)
    ref = oo.gather_tokens_with_cls(x, kept)
    assert torch.equal(xg.cpu(), ref)
    href = torch.nn.functional.layer_norm(ref.float(), (D,), g.float(), bt.float(), 1e-6)
    tol = dict(rtol=1e-2, atol=1e-2) if dtype == torch.bfloat16 else FP32
    torch.testing.assert_close(h.cpu().float(), href, **tol)


def test_score_tail_a_gelu_on_load_and_prev_gather(ops):
    B, N, Cc, K = 4, 196, 96, 137
    raw = fx.randn(170, B, N, Cc)
    W, b = fx.randn(171, 2, Cc, scale=0.3), fx.randn(172, 2, scale=0.1)
    prev = (torch.rand(B, N, generator=fx.gen(173)) > 0.2).float()
    logp, kept, pk = ops.score_tail_a(cu(raw), cu(W), cu(b), k=K, prev=cu(prev), act_input=ops.ACT_GELU, want_prev_kept=True)
    torch.testing.assert_close(logp.cpu(), oo.score_tail_a(torch.nn.functional.gelu(raw), W, b), rtol=1e-4, atol=1e-5)
    rk, _ = oo.select_topk(logp.cpu()[:, :, 0], K, oo.ORDER_SCORE_DESC)
    assert torch.equal(kept.cpu(), rk)
    assert torch.equal(pk.cpu(), oo.batch_index_select(prev, kept.cpu()))
    _, _, pk1 = ops.score_tail_a(cu(raw), cu(W), cu(b), k=K, act_input=ops.ACT_GELU, want_prev_kept=True)
    assert torch.equal(pk1.cpu(), torch.ones(B, K))


def _tail_inputs(B, N, seed, with_prev=True):
    H = 192
    local = (0.6 * fx.randn(seed, B, N, H)).bfloat16()
    per_image = (0.3 * fx.randn(seed + 1, B, H)).bfloat16()
    w2 = fx.randn(seed + 2, H, 2 * H, scale=0.08).bfloat16()
    w3, b3 = fx.randn(seed + 3, H // 2, H, scale=0.1).bfloat16(), fx.randn(seed + 4, H // 2, scale=0.1).bfloat16()
    w4, b4 = fx.randn(seed + 5, 2, H // 2, scale=0.3), fx.randn(seed + 6, 2, scale=0.1)
    prev = (torch.rand(B, N, generator=fx.gen(seed + 7)) > 0.25).float() if with_prev else None
    return local, per_image, w2, w3, b3, w4, b4, prev


def _tail_reference(local, per_image, w2, w3, b3, w4, b4):
    """out_conv of PredictorLG (default_dynamic_vit.py:315-320) on cat(local, pooled.expand) with the first Linear split as
    local @ W[:, :H]^T + per_image, in fp32 from the same bf16 operands."""
    F = torch.nn.functional
    H = local.shape[-1]
    u = F.gelu(local.float() @ w2.float()[:, :H].t() + per_image.float()[:, None, :])
    v = F.gelu(u @ w3.float().t() + b3.float())
    return F.log_softmax(v @ w4.t() + b4, dim=-1)


@pytest.mark.parametrize("B,N,K", [(3, 196, 137), (5, 137, 96), (4, 96, 67), (2, 128, 64), (2, 129, 70), (1, 17, 5), (1, 1, 1),
                                   (2, 256, 200), (3, 200, 0), (2, 64, 64), (300, 196, 137)])
def test_predictor_a_tail_kernel(ops, B, N, K):
    """d2s_predictor_a_tail_bf16 (second / third Linear + GELUs + Linear(., 2) + log-softmax + selection as one tcgen05 kernel)
    against an fp32 evaluation of the same bf16 operands at bf16 tolerance (three chained bf16 roundings: 3e-2 on log-probs of
    magnitude ~1), the kept list bit-exact against the stable descending sort of the kernel's OWN scores, prev gathered exactly."""
    local, per_image, w2, w3, b3, w4, b4, prev = _tail_inputs(B, N, 900 + N)
    logp, kept, pk = ops.predictor_a_tail(cu(local), cu(per_image), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), K, prev=cu(prev))
    ref = _tail_reference(local, per_image, w2, w3, b3, w4, b4)
    assert logp.shape == (B, N, 2) and kept.shape == (B, K) and pk.shape == (B, K)
    torch.testing.assert_close(logp.cpu(), ref, rtol=3e-2, atol=3e-2)
    rk, _ = oo.select_topk(logp.cpu()[:, :, 0], K, oo.ORDER_SCORE_DESC)
    assert torch.equal(kept.cpu(), rk)
    assert torch.equal(pk.cpu(), oo.batch_index_select(prev, kept.cpu()))
    # deterministic, and prev = None gathers ones
    logp2, kept2, pk1 = ops.predictor_a_tail(cu(local), cu(per_image), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), K)
    assert torch.equal(logp2, logp) and torch.equal(kept2, kept)
    assert torch.equal(pk1.cpu(), torch.ones(B, K))


def test_predictor_a_tail_matches_the_unfused_path(d2s, ops):
    """engine.predictor_a_select with the tail kernel against the same call on the library GEMMs + bias_act + score_tail_a: same
    roundings (every Linear / GELU output in bf16), so the log-probs agree to a few bf16 ulps of the hidden activations and the
    kept sets differ only where two scores are closer than that."""
    eng = d2s.engine
    torch.manual_seed(5)
    pred = d2s.variant_a.PredictorLG(384).cuda()
    for p in pred.parameters():
        torch.nn.init.normal_(p, std=0.08 if p.dim() > 1 else 0.05)
    pred = pred.to(torch.bfloat16).eval()
    B, N, K = 6, 196, 137
    normed = cu(fx.randn(77, B, N, 384)).bfloat16()
    prev = cu((torch.rand(B, N, generator=fx.gen(78)) > 0.3).float())
    old = eng._PRED_FUSED
    try:
        with torch.no_grad():
            eng._PRED_FUSED = False
            lp_u, kept_u, pk_u = eng.predictor_a_select(pred, normed, prev, K)
            eng._PRED_FUSED = True
            n0 = d2s._lib.launch_count()
            lp_f, kept_f, pk_f = eng.predictor_a_select(pred, normed, prev, K)
            assert d2s._lib.launch_count() - n0 == 3          # Linear + GELU GEMM, pool_act (pooled only), the tail kernel
    finally:
        eng._PRED_FUSED = old
    torch.testing.assert_close(lp_f, lp_u, rtol=2e-2, atol=2e-2)
    same = sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(kept_u.cpu(), kept_f.cpu()))
    assert same >= 0.98 * B * K
    assert torch.equal(pk_f, torch.gather(prev, 1, kept_f))


def test_predictor_a_tail_rejects_what_it_cannot_take(ops):
    local, per_image, w2, w3, b3, w4, b4, prev = _tail_inputs(2, 50, 950)
    with pytest.raises(RuntimeError):
        ops.predictor_a_tail(cu(local), cu(per_image), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), 51)          # K > N
    with pytest.raises(RuntimeError):
        ops.predictor_a_tail(cu(local), cu(per_image[:1]), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), 10)     # per_image rows
    assert not ops.predictor_a_tail_ok(cu(local).float(), cu(w2), cu(w3), cu(w4))                           # fp32 stays unfused
    assert not ops.predictor_a_tail_ok(cu(local)[:, :, :96], cu(w2), cu(w3), cu(w4))                        # other widths too
    empty = ops.predictor_a_tail(cu(local)[:0], cu(per_image)[:0], cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), 10)
    assert empty[0].shape == (0, 50, 2) and empty[1].shape == (0, 10)


@pytest.mark.parametrize("B,T,H,frac", [(3, 197, 6, False), (2, 138, 6, True), (2, 97, 6, True), (2, 64, 3, False), (1, 8, 2, True),
                                        (2, 208, 3, True), (1, 200, 2, False), (2, 129, 2, True), (2, 128, 2, False), (3, 1, 2, False),
                                        (1, 250, 2, True), (2, 226, 6, True), (1, 256, 2, False)])
def test_attention_train_fwd_bwd_vs_oracle_autograd(ops, B, T, H, frac):
    """bf16 training attention (T <= 208: the tcgen05 flash forward with row statistics + d2s_attn_policy_bwd; beyond: their
    key-blocked forms d2s_attn_long_fwd_stats + d2s_attn_long_bwd) against the fp32 oracle's autograd on the same
    bf16-rounded inputs: output, CLS row, d qkv and d policy at bf16 tolerance."""
    hd = 64
    qkv = (fx.randn(600 + T, B, T, 3 * H * hd) * 0.7).bfloat16()
    pol = torch.rand(B, T, 1, generator=fx.gen(601 + T)) if frac else (torch.rand(B, T, 1, generator=fx.gen(602 + T)) > 0.3).float()
    pol[:, 0] = 1.0
    go = (fx.randn(603 + T, B, T, H * hd) * 0.5).bfloat16()
    gc = fx.randn(604 + T, B, H, T) * 0.5
    q1 = cu(qkv).requires_grad_(True)
    p1 = cu(pol).requires_grad_(True)
    o1, c1 = ops.attention_train(q1, H, policy=p1, want_cls_row=True)
    (o1.float() * cu(go).float()).sum().add((c1.float() * cu(gc)).sum()).backward()
    q2 = qkv.float().requires_grad_(True)
    p2 = pol.clone().requires_grad_(True)
    o2, c2 = oo.attention_core(q2.view(B, T, 3, H, hd), H, policy=p2)
    (o2 * go.float()).sum().add((c2 * gc).sum()).backward()
    tol = dict(rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(o1.detach().cpu().float(), o2.detach(), **tol)
    torch.testing.assert_close(c1.detach().cpu().float(), c2.detach(), rtol=2e-2, atol=2e-3)
    gq1, gq2 = q1.grad.cpu().float(), q2.grad
    assert float((gq1 - gq2).abs().max()) <= 3e-2 * float(gq2.abs().max()) + 1e-3
    gp1, gp2 = p1.grad.cpu().float(), p2.grad
    # d policy is accumulated in fp32 from fp32 scores
    assert float((gp1 - gp2).abs().max()) <= 1e-3 * float(gp2.abs().max()) + 1e-5
    # no policy: plain softmax attention
    q3 = cu(qkv).requires_grad_(True)
    o3, none = ops.attention_train(q3, H)
    (o3.float() * cu(go).float()).sum().backward()
    q4 = qkv.float().requires_grad_(True)
    o4, _ = oo.attention_core(q4.view(B, T, 3, H, hd), H)
    (o4 * go.float()).sum().backward()
    assert none is None
    torch.testing.assert_close(o3.detach().cpu().float(), o4.detach(), **tol)
    assert float((q3.grad.cpu().float() - q4.grad).abs().max()) <= 3e-2 * float(q4.grad.abs().max()) + 1e-3


@pytest.mark.parametrize("M,N", [(50432, 1536), (50432, 384), (197 * 7, 1152), (3, 8), (1, 2048), (0, 384)])
def test_colsum_matches_fp32_sum(ops, M, N):
    """d2s_colsum_bf16: fp32 column sums of a bf16 matrix (a Linear layer's bias gradient)."""
    dy = (fx.randn(820 + N, max(M, 1), N) * 0.5).bfloat16()[:M]
    out = ops.colsum(cu(dy))
    ref = dy.double().sum(0)
    assert out.dtype == torch.float32 and out.shape == (N,)
    assert float((out.cpu().double() - ref).abs().max()) <= 2e-5 * float(dy.double().abs().sum(0).max()) + 1e-6


@pytest.mark.parametrize("M,N", [(50432, 1536), (197 * 3, 384), (5, 8), (0, 64)])
def test_gelu_bwd_colsum_matches_autograd(ops, M, N):
    """du = ga * gelu'(u) (exact-erf GELU) and db = column sums of du, against torch autograd in float64 on the same bf16 inputs."""
    u = (fx.randn(840 + N, max(M, 1), N) * 2.0).bfloat16()[:M]
    ga = (fx.randn(841 + N, max(M, 1), N) * 0.5).bfloat16()[:M]
    du, db = ops.gelu_bwd_colsum(cu(u), cu(ga))
    u64 = u.double().requires_grad_(True)
    (torch.nn.functional.gelu(u64) * ga.double()).sum().backward()
    ref = u64.grad
    if M > 0:
        err = (du.cpu().double() - ref).abs()
        assert bool((err <= ref.abs() * 2 ** -7 + 2e-4).all())                       # one bf16 ulp + the tail's absolute error
        assert float((db.cpu().double() - du.cpu().double().sum(0)).abs().max()) <= 2e-5 * float(du.cpu().double().abs().sum(0).max()) + 1e-6
    else:
        assert du.shape == (0, N) and float(db.abs().max()) == 0
    du2, none = ops.gelu_bwd_colsum(cu(u), cu(ga), want_bias=False)
    assert none is None and torch.equal(du2, du)


def test_linear_gelu_train_matches_modules_under_autocast(ops):
    """ops.linear_gelu_train(fc1, GELU, x) == GELU(fc1(x)) in value and in every gradient (fp32 master weights, bf16 autocast)."""
    lin, lin2 = torch.nn.Linear(384, 1536).cuda(), torch.nn.Linear(384, 1536).cuda()
    lin2.load_state_dict(lin.state_dict())
    act = torch.nn.GELU()
    x1 = cu(fx.randn(850, 4, 197, 384)).requires_grad_(True)
    x2 = x1.detach().clone().requires_grad_(True)
    up = cu(fx.randn(851, 4, 197, 1536))
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y1 = ops.linear_gelu_train(lin, act, x1)
        y2 = act(lin2(x2))
    # the fused forward applies GELU to the fp32 accumulator (torch: to the bf16-rounded Linear output): within one bf16 ulp
    assert y1.dtype == torch.bfloat16
    torch.testing.assert_close(y1.float(), y2.float(), rtol=2 ** -7, atol=2e-3)
    assert float((y1 != y2).float().mean()) < 0.35     # single vs double rounding: a quarter of the results move by one ulp
    (y1.float() * up).sum().backward()
    (y2.float() * up).sum().backward()
    for a, b in ((x1.grad, x2.grad), (lin.weight.grad, lin2.weight.grad), (lin.bias.grad, lin2.bias.grad)):
        assert a.dtype == b.dtype and float((a - b).abs().max()) <= 1e-2 * float(b.abs().max()) + 1e-4
    assert torch.equal(ops.linear_gelu_train(lin, torch.nn.ReLU(), x1.detach()), torch.relu(lin(x1.detach())))   # other activations: unfused


def test_linear_train_matches_module_under_autocast(ops):
    """ops.linear_train(lin, x) == lin(x) in value and in every gradient, fp32 master weights under bf16 autocast."""
    lin = torch.nn.Linear(384, 1152).cuda()
    lin2 = torch.nn.Linear(384, 1152).cuda()
    lin2.load_state_dict(lin.state_dict())
    x1 = cu(fx.randn(810, 4, 197, 384)).requires_grad_(True)
    x2 = x1.detach().clone().requires_grad_(True)
    up = cu(fx.randn(811, 4, 197, 1152))
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y1 = ops.linear_train(lin, x1)
        y2 = lin2(x2)
    assert y1.dtype == torch.bfloat16 and torch.equal(y1, y2)
    (y1.float() * up).sum().backward()
    (y2.float() * up).sum().backward()
    assert lin.weight.grad.dtype == torch.float32 and lin.bias.grad.dtype == torch.float32
    for a, b in ((x1.grad, x2.grad), (lin.weight.grad, lin2.weight.grad), (lin.bias.grad, lin2.bias.grad)):
        assert float((a - b).abs().max()) <= 8e-3 * float(b.abs().max()) + 1e-4
    with torch.no_grad():                                   # no gradient wanted: the module itself
        assert torch.equal(ops.linear_train(lin, x1), lin(x1))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,N,D", [(3, 196, 384), (2, 196, 768), (1, 4, 64)])
def test_assemble_layernorm_equals_assembly_then_layernorm(ops, dtype, B, N, D):
    """Token assembly fused with the first norm1: x bit-identical to assemble_tokens (and to the oracle), h bit-identical to the
    stand-alone LayerNorm kernel on that x."""
    patches = fx.randn(830 + D, B, N, D).to(dtype)
    cls, pos = fx.randn(831, 1, 1, D).to(dtype), (fx.randn(832, 1, N + 1, D) * 0.5).to(dtype)
    w, b = (1 + 0.1 * fx.randn(833, D)).to(dtype), (0.1 * fx.randn(834, D)).to(dtype)
    x, h = ops.assemble_layernorm(cu(patches), cu(cls), cu(pos), cu(w), cu(b), 1e-6)
    x0 = ops.assemble_tokens(cu(patches), cu(cls), cu(pos))
    assert torch.equal(x, x0) and torch.equal(x.cpu(), oo.assemble_tokens(patches, cls, pos))
    _, h0 = ops.add_layernorm(x0, None, cu(w), cu(b), 1e-6)
    assert torch.equal(h, h0)


# ------------------------------------------------------------------------------------------ error behaviour
def test_errors_are_loud(ops):
    with pytest.raises(RuntimeError):
        ops.select_topk(torch.rand(2, 196), 10)                                   # CPU tensor: no fallback
    with pytest.raises(RuntimeError, match="N="):
        ops.select_topk(torch.rand(2, 2000).cuda(), 10)
    with pytest.raises(RuntimeError, match="K="):
        ops.select_topk(torch.rand(2, 196).cuda(), 500)
    with pytest.raises(TypeError):
        ops.gather_tokens(torch.zeros(2, 4, 8, dtype=torch.float64).cuda(), torch.zeros(2, 2, dtype=torch.long).cuda())
    xh = torch.randn(2, 5, 8).half().cuda()                                       # any 2-byte element type is a pure copy
    assert torch.equal(ops.gather_tokens(xh, torch.tensor([[0, 2], [1, 3]]).cuda()), xh[:, [0, 1, 3]][:1].new_tensor(
        torch.stack([xh[0, [0, 1, 3]], xh[1, [0, 2, 4]]]).tolist()))
    with pytest.raises(RuntimeError, match="head dim"):
        ops.attention_core(torch.zeros(1, 8, 3 * 2 * 48, dtype=torch.bfloat16).cuda(), 2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,N,C,with_policy", [(3, 196, 384, True), (2, 137, 384, False), (2, 5, 16, True), (1, 1, 1536, True),
                                                (4, 196, 768, True)])
def test_pool_concat_train_matches_the_torch_composition(ops, B, N, C, with_policy, dtype):
    """d2s_pool_concat_fwd/bwd against the reference's slice / multiply / sum / divide / expand / cat (default_dynamic_vit.py
    :326-329; plain mean: dynamic_vit.py:541-545) under torch autograd in fp32."""
    if dtype == torch.float32 and C // 2 > 384:
        pytest.skip("f32 rows up to C/2 = 384")
    h = fx.randn(900 + N, B, N, C).to(dtype)
    pol = (torch.rand(B, N, 1, generator=fx.gen(901 + N)) > 0.4).float() * (0.5 + torch.rand(B, N, 1, generator=fx.gen(902))) if with_policy else None
    if pol is not None:
        pol[:, 0] = 1.0
    go = fx.randn(903 + N, B, N, C).to(dtype)
    hr = h.float().clone().requires_grad_(True)
    pr = None if pol is None else pol.clone().requires_grad_(True)
    half = C // 2
    if pr is not None:
        pooled = (hr[:, :, half:] * pr).sum(dim=1, keepdim=True) / pr.sum(dim=1, keepdim=True)
    else:
        pooled = hr[:, :, half:].mean(dim=1, keepdim=True)
    ref = torch.cat([hr[:, :, :half], pooled.expand(B, N, half)], dim=-1)
    (ref * go.float()).sum().backward()
    hd = cu(h).requires_grad_(True)
    pd = None if pol is None else cu(pol).requires_grad_(True)
    out = ops.pool_concat_train(hd, pd)
    assert out.dtype == dtype and out.shape == (B, N, C)
    (out.float() * cu(go).float()).sum().backward()
    tol = dict(rtol=1e-5, atol=1e-5) if dtype == torch.float32 else dict(rtol=1e-2, atol=1e-2)
    assert torch.equal(out[:, :, :half].cpu(), h[:, :, :half])                       # the local half is a copy
    torch.testing.assert_close(out.float().cpu(), ref.detach(), **tol)
    assert torch.equal(hd.grad[:, :, :half].cpu(), go[:, :, :half])
    gscale = float(hr.grad.abs().max())
    torch.testing.assert_close(hd.grad.float().cpu(), hr.grad, rtol=tol["rtol"], atol=tol["atol"] * max(1.0, gscale))
    if pol is not None:
        pscale = float(pr.grad.abs().max())
        torch.testing.assert_close(pd.grad.cpu(), pr.grad, rtol=1e-4 if dtype == torch.float32 else 2e-2,
                                   atol=(1e-5 if dtype == torch.float32 else 2e-2) * max(1.0, pscale))


@pytest.mark.parametrize("dtype,out_dtype", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16), (torch.float32, torch.bfloat16)])
@pytest.mark.parametrize("B,T,D,row0", [(3, 197, 384, 1), (2, 9, 64, 1), (2, 10, 768, 2), (1, 2, 8, 1)])
def test_layer_norm_over_a_row_slice_reads_in_place(ops, B, T, D, row0, dtype, out_dtype):
    """ops.layer_norm(x, row0=r) == layer_norm(x[:, r:]) forward and backward (d2s_layernorm_seg_fwd/bwd): the gradient has
    x's full shape with zeros in the skipped rows, dgamma / dbeta as usual."""
    x = fx.randn(910 + T, B, T, D).to(dtype)
    w, b = 1.0 + 0.1 * fx.randn(911, D), 0.1 * fx.randn(912, D)
    go = fx.randn(913 + T, B, T - row0, D).to(out_dtype)
    xr, wr, br = x.float().clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ref = torch.nn.functional.layer_norm(xr[:, row0:], (D,), wr, br, 1e-5)
    (ref * go.float()).sum().backward()
    xd, wd, bd = cu(x).requires_grad_(True), cu(w).requires_grad_(True), cu(b).requires_grad_(True)
    out = ops.layer_norm(xd, wd, bd, 1e-5, out_dtype=out_dtype, row0=row0)
    assert out.shape == (B, T - row0, D) and out.dtype == out_dtype and out.is_contiguous()
    (out.float() * cu(go).float()).sum().backward()
    lo = dtype == torch.bfloat16 or out_dtype == torch.bfloat16
    tol = dict(rtol=2e-2, atol=2e-2) if lo else dict(rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(out.float().cpu(), ref.detach(), **tol)
    assert xd.grad.shape == x.shape and float(xd.grad[:, :row0].abs().max()) == 0.0
    torch.testing.assert_close(xd.grad.float().cpu(), xr.grad, rtol=tol["rtol"], atol=tol["atol"] * max(1.0, float(xr.grad.abs().max())))
    torch.testing.assert_close(wd.grad.cpu(), wr.grad, rtol=tol["rtol"], atol=tol["atol"] * max(1.0, float(wr.grad.abs().max())))
    torch.testing.assert_close(bd.grad.cpu(), br.grad, rtol=tol["rtol"], atol=tol["atol"] * max(1.0, float(br.grad.abs().max())))


@pytest.mark.parametrize("sdt,tdt", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16)])
@pytest.mark.parametrize("B,N,C,sliced", [(3, 196, 384, True), (2, 67, 384, False), (2, 5, 8, True), (1, 3, 1024, False), (2, 9, 768, True)])
def test_token_kl_rows_match_f_kl_div(ops, B, N, C, sliced, sdt, tdt):
    """d2s_token_kl_fwd against F.kl_div(F.log_softmax(s), F.log_softmax(t), log_target=True) (losses.py:220-225), value and
    gradient in s; inputs as x[:, 1:] views (read in place) or dense."""
    full_s = (fx.randn(920 + N, B, N + 1, C) * 2.0).to(sdt)
    full_t = (fx.randn(921 + N, B, N + 1, C) * 2.0).to(tdt)
    w = torch.rand(B * N, generator=fx.gen(922))
    sr = full_s.float().clone().requires_grad_(True)
    ref_rows = torch.nn.functional.kl_div(torch.log_softmax(sr[:, 1:].reshape(-1, C), -1), torch.log_softmax(full_t.float()[:, 1:].reshape(-1, C), -1),
                                          reduction="none", log_target=True).sum(-1)
    (ref_rows * w).sum().backward()
    sd = cu(full_s.detach().clone()).requires_grad_(True)
    td = cu(full_t)
    s_in, t_in = (sd[:, 1:], td[:, 1:]) if sliced else (sd[:, 1:].contiguous(), td[:, 1:].contiguous())
    assert ops.token_kl_ok(s_in, t_in)
    rows = ops.token_kl_rows(s_in, t_in)
    assert rows.shape == (B * N,) and rows.dtype == torch.float32
    (rows * cu(w)).sum().backward()
    torch.testing.assert_close(rows.detach().cpu(), ref_rows.detach(), rtol=1e-5, atol=1e-6)
    g = sd.grad.float().cpu()
    assert float(g[:, 0].abs().max()) == 0.0
    tol = 1e-6 if sdt == torch.float32 else 4e-3 * float(sr.grad.abs().max())
    torch.testing.assert_close(g, sr.grad, rtol=1e-4 if sdt == torch.float32 else 1e-2, atol=tol)


def test_round2_training_ops_take_empty_inputs(ops):
    """B = 0 / empty ranges return without a launch (the C ABI reports shape errors, not empty work)."""
    dev = torch.device("cuda")
    h = torch.zeros(0, 196, 384, device=dev, dtype=torch.bfloat16)
    assert ops.pool_concat_train(h, torch.zeros(0, 196, 1, device=dev)).shape == (0, 196, 384)
    s = torch.zeros(0, 197, 384, device=dev)
    assert ops.token_kl_rows(s[:, 1:], s[:, 1:]).shape == (0,)
    w, b = torch.ones(384, device=dev), torch.zeros(384, device=dev)
    assert ops.layer_norm(torch.zeros(0, 197, 384, device=dev), w, b, 1e-5, row0=1).shape == (0, 196, 384)
    p = torch.ones(16, device=dev)
    g, m, v = torch.ones(16, device=dev), torch.zeros(16, device=dev), torch.zeros(16, device=dev)
    lr, st = torch.full((1,), 1e-3, device=dev), torch.ones(1, device=dev)
    ops.adamw_flat(p, g, m, v, None, 5, 5, lr, st, 0.9, 0.999, 1e-8, 0.0)
    assert torch.equal(p, torch.ones(16, device=dev)) and float(m.abs().max()) == 0.0
    with pytest.raises(RuntimeError):
        ops.adamw_flat(p, g, m, v, None, 0, 17, lr, st, 0.9, 0.999, 1e-8, 0.0)          # range outside the buffers
    with pytest.raises(RuntimeError):
        ops.token_kl_rows(torch.zeros(2, 4, 12, device=dev), torch.zeros(2, 4, 12, device=dev))   # C % 8 != 0
    with pytest.raises(RuntimeError):
        ops.pool_concat_train(torch.zeros(2, 4, 12, device=dev, dtype=torch.float64))


def test_cached_fp32_parameter_copies_follow_the_parameter(ops):
    """ops._f32c_param (fp32 copies of the tail's last Linear, cached across calls): in-place updates, dtype casts of the
    module and a NEW tensor that reuses a dead one's address must all be seen."""
    lin = torch.nn.Linear(96, 2).cuda().to(torch.bfloat16)
    a = ops._f32c_param(lin.weight)
    assert ops._f32c_param(lin.weight) is a                                  # cached
    with torch.no_grad():
        lin.weight.mul_(2.0)
    b = ops._f32c_param(lin.weight)
    assert torch.equal(b, lin.weight.float()) and not torch.equal(a, b)
    for i in range(20):                                                      # same shape, freed and reallocated: never stale
        w = (torch.full((2, 96), float(i), device="cuda")).to(torch.bfloat16)
        assert float(ops._f32c_param(w)[0, 0]) == float(i)
        del w


@pytest.mark.parametrize("B,T,row0", [(3, 197, 0), (2, 138, 1), (7, 97, 0), (1, 1, 0), (5, 68, 0), (40, 197, 1), (300, 97, 0)])
def test_mlp_kernel_applies_its_input_layernorm_from_row_statistics(ops, B, T, row0):
    """proj + residual with per-row (mean, rstd) instead of the normalised copy (d2s_linear_residual_stats_bf16) followed by the
    one-kernel MLP that normalises its input tile in shared memory (d2s_mlp_lnin_residual_ln_bf16): BIT-identical to the pair that
    materialises LayerNorm(x') in between (same arithmetic, same roundings), statistics equal to the fp32 row statistics of x'."""
    D, HID = 384, 1536
    bf = torch.bfloat16
    r = lambda seed, *s, sc=1.0: cu(fx.randn(seed, *s) * sc).to(bf)
    Wp, bp = r(1, D, D, sc=D ** -0.5), r(2, D, sc=0.1)
    W1, b1, W2, b2 = r(3, HID, D, sc=D ** -0.5), r(4, HID, sc=0.1), r(5, D, HID, sc=HID ** -0.5), r(6, D, sc=0.1)
    g2, bt2 = (1 + 0.2 * cu(fx.randn(7, D))).to(bf), r(8, D, sc=0.2)
    g1, bt1 = (1 + 0.2 * cu(fx.randn(9, D))).to(bf), r(10, D, sc=0.2)
    a, x = r(11 + T, B, T, D), r(12 + T, B, T, D, sc=2.0)
    x = x + 3.0 * (torch.arange(D, device="cuda") % 7 == 0).to(bf)            # a few channels with a large mean
    xs0, hn = ops.linear_residual_ln(a, Wp, bp, x, g2, bt2, 1e-6)
    ref = ops.mlp_residual_ln(hn, W1, b1, W2, b2, xs0, g1, bt1, 1e-6, norm_row0=row0)
    xs1, st = ops.linear_residual_ln(a, Wp, bp, x, eps=1e-6, want_norm=False, want_stats=True)
    assert torch.equal(xs1, xs0) and st.shape == (B * T, 2)
    xf = xs1.float().reshape(B * T, D)
    torch.testing.assert_close(st[:, 0], xf.mean(-1), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(st[:, 1], torch.rsqrt(xf.var(-1, unbiased=False) + 1e-6), rtol=1e-4, atol=1e-4)
    out = ops.mlp_residual_ln(None, W1, b1, W2, b2, xs1, g1, bt1, 1e-6, norm_row0=row0, in_stats=st, in_ln_weight=g2, in_ln_bias=bt2)
    assert torch.equal(out[0], ref[0]) and torch.equal(out[1], ref[1])


def test_lazy_norms_are_invisible_at_model_level(d2s, monkeypatch):
    """engine: norm2 handed to the one-kernel MLP and norm1 to the qkv GEMM as row statistics (engine._LAZY_NORM2 / _LAZY_NORM1)
    against the same forward with the normalised copies: identical logits and kept sets (the kernels are bit-identical; the
    CLS-only last MLP normalises its rows itself)."""
    torch.manual_seed(3)
    m = d2s.variant_a.DefaultVisionTransformerDiffPruning(patch_size=16, embed_dim=384, depth=6, num_heads=6, num_classes=32, mlp_ratio=4,
                                                          qkv_bias=True, pruning_loc=[2, 4], token_ratio=[0.7, 0.49], distill=True)
    m = m.cuda().eval().to(torch.bfloat16)
    img = cu(fx.randn(55, 96, 3, 224, 224)).bfloat16()      # enough rows for a last-bit difference anywhere to show up
    outs = []
    with torch.no_grad():
        for n1, n2 in ((True, True), (False, True), (True, False), (False, False)):
            monkeypatch.setattr(d2s.engine, "_LAZY_NORM1", n1)      # norm1 inside the qkv GEMM, from the MLP kernel's row statistics
            monkeypatch.setattr(d2s.engine, "_LAZY_NORM2", n2)      # norm2 inside the MLP kernel, from the proj kernel's
            n0 = d2s._lib.launch_count()
            logits = m(img)
            outs.append((logits, [k.clone() for k in m.kept_token_indices], d2s._lib.launch_count() - n0))
    for logits, kept, _ in outs[1:]:
        assert torch.equal(logits, outs[0][0]) and all(torch.equal(p, q) for p, q in zip(kept, outs[0][1]))
    ns = [n for _, _, n in outs]                                    # same kernels launched, only what they read / write differs
    assert max(ns) - min(ns) <= 1, ns                               # (+ the CLS rows' norm2 in front of the CLS-only last MLP)


@pytest.mark.parametrize("B,T", [(3, 197), (2, 138), (7, 97), (1, 1), (300, 68)])
def test_qkv_gemm_applies_norm1_from_the_mlp_kernels_row_statistics(ops, B, T):
    """d2s_mlp_lnin_residual_ln_bf16 with out_stats -> d2s_linear_lnin_act_pair_bf16 (the next block's qkv projection normalising
    its resident input rows): bit-identical to the chain that materialises LayerNorm(x'') in between."""
    D, HID = 384, 1536
    bf = torch.bfloat16
    r = lambda seed, *s, sc=1.0: cu(fx.randn(seed, *s) * sc).to(bf)
    W1, b1, W2, b2 = r(3, HID, D, sc=D ** -0.5), r(4, HID, sc=0.1), r(5, D, HID, sc=HID ** -0.5), r(6, D, sc=0.1)
    Wq, bq = r(13, 3 * D, D, sc=D ** -0.5), r(14, 3 * D, sc=0.1)
    g2, bt2 = (1 + 0.2 * cu(fx.randn(7, D))).to(bf), r(8, D, sc=0.2)
    g1, bt1 = (1 + 0.2 * cu(fx.randn(9, D))).to(bf), r(10, D, sc=0.2)
    x = r(20 + T, B, T, D, sc=2.0)
    xf = x.float().reshape(B * T, D)
    st = torch.stack([xf.mean(-1), torch.rsqrt(xf.var(-1, unbiased=False) + 1e-6)], -1).contiguous()
    x2, hn = ops.mlp_residual_ln(None, W1, b1, W2, b2, x, g1, bt1, 1e-6, in_stats=st, in_ln_weight=g2, in_ln_bias=bt2)
    ref = ops.linear_act(hn, Wq, bq, ops.ACT_NONE)
    x3, st2 = ops.mlp_residual_ln(None, W1, b1, W2, b2, x, None, None, 1e-6, want_norm=False, in_stats=st, in_ln_weight=g2,
                                  in_ln_bias=bt2, want_stats=True)
    out = ops.linear_act(x3, Wq, bq, ops.ACT_NONE, in_stats=st2, in_ln_weight=g1, in_ln_bias=bt1)
    assert torch.equal(x3, x2) and torch.equal(out, ref)
    torch.testing.assert_close(out.float(), torch.nn.functional.linear(hn.float(), Wq.float(), bq.float()), rtol=2e-2, atol=2e-2)


def test_pool_and_tail_kernels_read_a_row_slice_in_place(ops):
    """x[:, 1:] of a (B, N + 1, 384) tensor (the predictor's Linear + GELU output over every token, CLS row included): the pooled
    rows and the tail kernel's results through the batch stride are identical to those on a dense copy of the slice."""
    B, N, K, C = 5, 196, 137, 384
    local, per_image, w2, w3, b3, w4, b4, prev = _tail_inputs(B, N, 1200)
    wide = cu(torch.cat([fx.randn(1201, B, N + 1, 192).bfloat16(), fx.randn(1202, B, N + 1, 192).bfloat16()], -1))   # (B, N+1, 384)
    view = wide[:, 1:]
    dense = view.contiguous()
    _, p_view = ops.pool_act(view, cu(prev), ops.ACT_NONE, want_local=False)
    _, p_dense = ops.pool_act(dense, cu(prev), ops.ACT_NONE, want_local=False)
    assert torch.equal(p_view, p_dense)
    a = ops.predictor_a_tail(view[:, :, :192], cu(per_image), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), K, prev=cu(prev))
    b = ops.predictor_a_tail(dense[:, :, :192].contiguous(), cu(per_image), cu(w2), cu(w3), cu(b3), cu(w4), cu(b4), K, prev=cu(prev))
    assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("B,T,K", [(3, 197, 137), (2, 138, 96), (5, 97, 1), (1, 8, 0)])
def test_gather_and_assemble_hand_norm1_on_as_row_statistics(ops, B, T, K):
    """d2s_gather_layernorm_stats / d2s_assemble_layernorm_stats: the same summed rows as the forms that also write LayerNorm(x),
    per-row (mean, rstd) equal to the fp32 statistics of those rows, and the qkv GEMM fed with (x, stats) BIT-identical to the qkv
    GEMM fed with the materialised LayerNorm output (both use fma(fma(x, rstd, -mean * rstd), gamma, beta))."""
    D = 384
    bf = torch.bfloat16
    x = cu(fx.randn(1300 + T, B, T, D) * 1.5).to(bf)
    kept = torch.stack([torch.randperm(T - 1, generator=fx.gen(1301 + b))[:K].sort().values for b in range(B)]).cuda()
    g, bt = (1 + 0.2 * cu(fx.randn(1302, D))).to(bf), cu(fx.randn(1303, D) * 0.2).to(bf)
    Wq, bq = cu(fx.randn(1304, 3 * D, D) * D ** -0.5).to(bf), cu(fx.randn(1305, 3 * D) * 0.1).to(bf)
    xg, hn = ops.gather_layernorm(x, kept, g, bt, 1e-6)
    xs, st = ops.gather_layernorm(x, kept, g, bt, 1e-6, want_stats=True)
    assert torch.equal(xs, xg) and st.shape == (B * (K + 1), 2)
    xf = xs.float().reshape(-1, D)
    torch.testing.assert_close(st[:, 0], xf.mean(-1), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(st[:, 1], torch.rsqrt(xf.var(-1, unbiased=False) + 1e-6), rtol=1e-4, atol=1e-5)
    assert torch.equal(ops.linear_act(xs, Wq, bq, ops.ACT_NONE, in_stats=st, in_ln_weight=g, in_ln_bias=bt),
                       ops.linear_act(hn, Wq, bq, ops.ACT_NONE))
    patches = cu(fx.randn(1306, B, T - 1, D)).to(bf) if T > 1 else None
    cls, pos = cu(fx.randn(1307, 1, 1, D)).to(bf), cu(fx.randn(1308, 1, T, D) * 0.5).to(bf)
    xa, ha = ops.assemble_layernorm(patches, cls, pos, g, bt, 1e-6)
    xb, sb = ops.assemble_layernorm(patches, cls, pos, g, bt, 1e-6, want_stats=True)
    assert torch.equal(xa, xb)
    assert torch.equal(ops.linear_act(xb, Wq, bq, ops.ACT_NONE, in_stats=sb, in_ln_weight=g, in_ln_bias=bt),
                       ops.linear_act(ha, Wq, bq, ops.ACT_NONE))
