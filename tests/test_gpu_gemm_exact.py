"""The CTA-pair GEMMs (csrc/d2s_gemm_pair.cu) and the one-kernel MLP (csrc/d2s_mlp_pair.cu) checked bit for bit on exact
operands, every LayerNorm producer checked against float64, and the GEMMs checked on Gaussian operands against a bound derived
from their arithmetic.

Exact operands: every operand is a small integer times a power of two and every partial sum of every output stays within 2^20
units of its grid (four bits below fp32's 24), so each fp32 accumulator holds the exact value whatever the accumulation order,
and also when the tensor cores truncate instead of rounding while aligning addends.  The float64 references are then exact as
well (any cuBLAS order), and the kernels' outputs must equal the exact values rounded to nearest even to bf16: no tolerance.
Values depend on (row, column) through a hash, so a swapped row, column or k-block changes the result.

The CPU tests (rounding helper, generator bound, host dispatch mirror) run without a GPU; the others are marked one by one.
"""
import math

import pytest
import torch

import fixtures as fx

NUM_PAIRS = 74                 # CTA pairs on a B200 (148 SMs): the host's work-unit cost model (d2s_gemm_pair.cu, gp_linear_act)
GRID_BOUND = 2 ** 20           # largest |partial sum| in grid units: 4 bits of headroom below fp32's 24-bit significand
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2
BF = torch.bfloat16


# ============================================================================================ helpers (no GPU needed)
def round_bf16(x):
    """float64 -> the nearest bf16 value (ties to even), returned as float64.  Written out by hand: torch's float64 -> bf16
    conversion rounds through fp32 on the CPU (1 + 2^-8 + 2^-30 becomes 1.0 instead of 1.0078125).  bf16 keeps 8 significant
    bits down to 2^-126 and is subnormal below (quantum 2^-133); |x| >= (2 - 2^-8) 2^127 rounds to infinity."""
    x = x.double()
    a = x.abs()
    _, e = torch.frexp(a)                                   # a = m 2^e, m in [0.5, 1): the 8-bit quantum is 2^(e - 8)
    q = torch.exp2(torch.clamp(e.double() - 8.0, min=-133.0))
    r = torch.round(a / q) * q                              # a / q is exact (power of two); torch.round is half-to-even
    r = torch.where(r >= 2.0 ** 128, torch.full_like(r, math.inf), r)
    r = torch.where(torch.isnan(x), x, r)
    return torch.copysign(r, x)


def ulp_bf16(v):
    """Spacing of the bf16 values at |v| (upwards from the binade's bottom): 2^(floor(log2 |v|) - 7), at least 2^-133."""
    v = v.double().abs()
    _, e = torch.frexp(v)
    u = torch.exp2(torch.clamp(e.double() - 8.0, min=-133.0))
    return torch.where(v == 0, torch.full_like(u, 2.0 ** -133), u)


def hgrid(rows, cols, salt, lo, hi, device="cpu"):
    """(rows, cols) int64 in [lo, hi], a hash of (row, column, salt).  int64 products wrap; only their low 32 bits are kept."""
    r = torch.arange(rows, device=device, dtype=torch.int64)[:, None]
    c = torch.arange(cols, device=device, dtype=torch.int64)[None, :]
    h = (r * 2654435761 + c * 2246822519 + (salt * 3266489917 + 374761393)) & 0xFFFFFFFF
    h = ((h ^ (h >> 15)) * 2246822519) & 0xFFFFFFFF
    h = ((h ^ (h >> 13)) * 3266489917) & 0xFFFFFFFF
    h = h ^ (h >> 16)
    return lo + h % (hi - lo + 1)


def grid_bound(a_int, w_int, b_int=None):
    """An upper bound, in grid units, of every partial sum of a_int @ w_int^T (+ b_int) in any order:
    max_i sum_k |a_ik| * max |w| + max |b|  >=  sum_k |a_ik| |w_jk| + |b_j|  >=  |any partial sum of output (i, j)|."""
    s = int(a_int.abs().sum(1).max()) * int(w_int.abs().max())
    return s + (int(b_int.abs().max()) if b_int is not None else 0)


def exact_gemm_operands(M, N, K, salt, device="cpu", bias=True, a_max=15, w_max=15, w_shift=6, b_max=1024):
    """A (M,K) integers in [-a_max, a_max]; W (N,K) integers in [-w_max, w_max] times 2^-w_shift; bias on W's grid.  All exact
    in bf16 (|integer| <= 256).  Returns (A, W, b) bf16 and the exact float64 A @ W^T + b (or None for the reference)."""
    ai = hgrid(M, K, salt, -a_max, a_max, device)
    wi = hgrid(N, K, salt + 1, -w_max, w_max, device)
    bi = hgrid(1, N, salt + 2, -b_max, b_max, device)[0] if bias else None
    assert grid_bound(ai, wi, bi) <= GRID_BOUND, "operands too wide for an exact fp32 accumulator"
    s = 2.0 ** -w_shift
    A, W = ai.to(BF), (wi.double() * s).to(BF)
    b = None if bi is None else (bi.double() * s).to(BF)
    return A, W, b


def exact_linear(A, W, b):
    """Float64 A @ W^T + b: exact for exact_gemm_operands (products and sums well inside float64's 53 bits)."""
    y = A.double() @ W.double().t()
    return y if b is None else y + b.double()


def gelu64(x):
    return 0.5 * x * torch.special.erfc(-x / math.sqrt(2.0))


def dispatch(M, N, K, lnin=False):
    """Python mirror of gp_linear_act's choices (d2s_gemm_pair.cu): 192- or 256-column tiles, resident A rows, the on-the-fly
    input LayerNorm, and the cost-model split of each row tile's column tiles into `groups` work units.  Shape selection only."""
    t192 = N % 256 != 0
    ares = t192 and K <= 384
    n_tiles = N // (192 if t192 else 256)
    pair_tiles = -(-M // 256)
    groups = 1
    best = ((pair_tiles + NUM_PAIRS - 1) // NUM_PAIRS) * (n_tiles + 0.25)
    for g in range(2, n_tiles + 1):
        if n_tiles % g:
            continue
        r = ((pair_tiles * g + NUM_PAIRS - 1) // NUM_PAIRS) * (n_tiles // g + 0.25)
        if r < best * 0.99:
            best, groups = r, g
    return ("act192" if t192 else "act256", groups, ares, lnin and ares)


def reachable_groups(N, max_pair_tiles=4096):
    """Every `groups` value the cost model picks for width N over 1 .. max_pair_tiles row-tile pairs (M up to ~10^6)."""
    return sorted({dispatch(256 * pt, N, 384)[1] for pt in range(1, max_pair_tiles + 1)})


# ---- shapes
N_T192 = [192, 384, 576, 960, 1152]
N_T256 = [256, 768, 1536, 2304, 3072, 4096]
K_LIST = [64, 384, 448, 768, 3072]                 # one k-block; either side of the resident-A limit (K <= 384); fc2 widths
SMALL_M = [1, 127, 128, 129, 255, 256, 257]
# M that selects each `groups` value (ragged: 5 rows short of whole row-tile pairs); from dispatch(), pinned here so that the
# coverage test below notices a change of either
GROUP_M = {
    384: [251, 9723], 576: [251, 12795], 960: [251, 15355], 1152: [251, 3323, 6395, 12611],
    768: [251, 12795], 1536: [1, 3105, 6209, 12611], 2304: [251, 4347, 14843],
    3072: [251, 1787, 3323, 4859, 6395, 15867], 4096: [251, 1275, 3579, 7163, 16635],
}
BENCH_ROWS = [1024 * t for t in (197, 138, 97, 68)]      # DeiT-S bench batch at each stage's token count
EDGE_M = [NUM_PAIRS * 256 - 1, NUM_PAIRS * 256 + 1]


def _small_cases():
    return [(N, K) for N in N_T192 + N_T256 for K in K_LIST]


def _group_cases():
    out = []
    for N, ms in GROUP_M.items():
        for M in ms:
            out.append((N, M, 384))
            if N % 256:
                out.append((N, M, 448))              # the same split without resident A rows
    out += [(N, M, 384) for N in (1152, 1536) for M in EDGE_M]
    return out


GROUP_CASES = _group_cases()
LNIN_CASES = [(N, M) for N in (384, 1152) for M in (1, 129, 257, 3 * 197, 3323, 6395, 12611, NUM_PAIRS * 256 + 1, 69632)]


def _reached():
    """(mode, groups, ares, lnin) of every linear_act / lnin case of this file."""
    seen = set()
    for N, K in _small_cases():
        for M in SMALL_M:
            seen.add(dispatch(M, N, K))
    for N, M, K in GROUP_CASES:
        seen.add(dispatch(M, N, K))
    for M in BENCH_ROWS:
        seen.add(dispatch(M, 1152, 384))
        seen.add(dispatch(M, 1536, 384))
    for N, M in LNIN_CASES:
        seen.add(dispatch(M, N, 384, lnin=True))
    return seen


# ============================================================================================ CPU tests
def test_round_bf16_ties_neighbours_subnormals_and_signed_zero():
    d = lambda v: torch.tensor(v, dtype=torch.float64)
    cases = [
        (1.0 + 2 ** -8, 1.0),                                  # tie, even neighbour below
        (1.0 + 3 * 2 ** -8, 1.0 + 2 ** -6),                    # tie, even neighbour above
        (1.0 + 2 ** -8 + 2 ** -30, 1.0 + 2 ** -7),             # just above a tie (fp32 would lose the 2^-30)
        (1.0 + 2 ** -8 - 2 ** -40, 1.0),                       # just below a tie
        (257.0, 256.0), (259.0, 260.0), (258.0, 258.0),        # integer ties at grid unit 1
        (-257.0, -256.0), (-(1.0 + 2 ** -8 + 2 ** -30), -(1.0 + 2 ** -7)),
        (2.0 ** -133, 2.0 ** -133),                            # smallest subnormal
        (2.0 ** -134, 0.0),                                    # tie between 0 and the smallest subnormal: even (0)
        (3 * 2.0 ** -134, 2.0 ** -132),                        # subnormal tie, even neighbour above
        (2.0 ** -134 + 2.0 ** -160, 2.0 ** -133),
        (2.0 ** -126 * (1 - 2 ** -9), 2.0 ** -126),            # rounds up into the normal range
        (3.0e38, 2.0 ** 127 * (1 + 98 / 128)),
        (2.0 ** 128 * (1 - 2 ** -9), math.inf),                # halfway to 2^128: overflows
    ]
    for v, want in cases:
        got = float(round_bf16(d(v)))
        assert got == want, (v, got, want)
    z = round_bf16(d([0.0, -0.0, -2.0 ** -140, 2.0 ** -140]))
    assert torch.equal(torch.signbit(z), torch.tensor([False, True, True, False])) and bool((z == 0).all())
    assert bool(torch.isnan(round_bf16(d(math.nan)))) and float(round_bf16(d(-math.inf))) == -math.inf


def test_round_bf16_matches_the_fp32_conversion_where_that_is_exact():
    """On fp32 inputs torch's fp32 -> bf16 conversion is round-to-nearest-even: the helper must agree on every one of them."""
    g = fx.gen(5)
    bits = torch.randint(0, 2 ** 32, (200000,), generator=g, dtype=torch.int64)
    bits = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32)
    f = bits.view(torch.float32)
    f = f[torch.isfinite(f) & (f.abs() < 3.3e38)]
    ties = (torch.arange(-3000, 3000, dtype=torch.float32) + 0.5) * 2.0 ** -7   # exact ties of the 1.x binade and around 0
    for x in (f, ties):
        assert torch.equal(round_bf16(x.double()), x.to(BF).double())


def test_ulp_bf16():
    v = torch.tensor([1.0, 1.5, 2.0, -3.0, 2.0 ** -126, 2.0 ** -130, 0.0], dtype=torch.float64)
    assert ulp_bf16(v).tolist() == [2 ** -7, 2 ** -7, 2 ** -6, 2 ** -6, 2 ** -133, 2 ** -133, 2 ** -133]


def test_exact_operand_generator_bound_and_exactness():
    # the widest case of the file (K = 3072) stays within the bound; a wider one is refused
    ai, wi = hgrid(64, 3072, 7, -15, 15), hgrid(48, 3072, 8, -15, 15)
    assert grid_bound(ai, wi, hgrid(1, 48, 9, -1024, 1024)[0]) <= GRID_BOUND
    with pytest.raises(AssertionError):
        exact_gemm_operands(4, 8, 16384, 1)
    # the bound dominates the true largest partial sum
    assert int((ai.abs() @ wi.abs().t()).max()) <= grid_bound(ai, wi)
    # values depend on row and column: no two rows / columns alike, and the range is used
    assert len({tuple(r) for r in ai[:, :16].tolist()}) == 64 and int(ai.min()) == -15 and int(ai.max()) == 15
    assert not torch.equal(ai[:, :32], ai[:, 32:64]) and not torch.equal(hgrid(8, 8, 1, 0, 99), hgrid(8, 8, 1, 0, 99).t())
    # fp32 accumulation in a random order (and with truncating adds) gives the exact value
    A, W, b = exact_gemm_operands(16, 8, 3072, 11)
    ref = exact_linear(A, W, b)
    prods = (A.float()[:, None, :] * W.float()[None, :, :])                  # (16, 8, K), exact in fp32
    perm = torch.randperm(3072, generator=fx.gen(12))
    acc = torch.zeros(16, 8, dtype=torch.float32)
    for k in perm.tolist():
        acc = acc + prods[:, :, k]
    assert torch.equal((acc + b.float()).double(), ref)
    # and the references contain bf16 ties, so that the rounding mode is pinned
    assert float((round_bf16(ref) != ref).float().mean()) > 0.3
    u = ref.abs() / ulp_bf16(ref)
    assert bool(((u - u.floor()) == 0.5).any())


def test_dispatch_mirror_reaches_every_split_the_cost_model_can_choose():
    want = {1152: [1, 2, 3, 6], 1536: [1, 2, 3, 6], 3072: [1, 2, 3, 4, 6, 12], 4096: [1, 2, 4, 8, 16]}
    for N, gs in want.items():
        assert reachable_groups(N) == gs, (N, reachable_groups(N))
    reached = _reached()
    for N in N_T192 + N_T256:
        mode = "act192" if N % 256 else "act256"
        for g in reachable_groups(N):
            assert (mode, g) in {(m, gg) for m, gg, _, _ in reached if m == mode}, (N, g)
            # every split at the width it was computed for
            assert any(dispatch(M, N, K)[1] == g for NN, M, K in GROUP_CASES if NN == N) or g == 1, (N, g)
    for ares in (False, True):
        for g in (1, 2, 3, 6):
            assert ("act192", g, ares, False) in reached, (g, ares)
    for g in (1, 2, 3, 6):
        assert ("act192", g, True, True) in reached, g


# ============================================================================================ GPU fixtures
@pytest.fixture(scope="module")
def ops(d2s, cuda_dev):
    return d2s.ops


def _first_bad(bad, got, want):
    idx = bad.nonzero()[:4].tolist()
    return [(i, float(got[tuple(i)]), float(want[tuple(i)])) for i in idx]


def assert_bits(got, want64, what):
    """got (bf16) equals want64 rounded to nearest even, element for element."""
    ref = round_bf16(want64)
    bad = got.double() != ref
    assert not bool(bad.any()), (what, int(bad.sum()), _first_bad(bad, got.double(), ref))


GELU_ULP = 0.07        # gelu_erf_pair (d2s_tc.cuh): within 0.07 bf16 ulp of float64 erf GELU for |x| < 5.6


def gelu_clear(ref):
    """Elements whose correct rounding the GELU's own accuracy cannot move: farther than GELU_ULP ulp from a rounding midpoint."""
    d = GELU_ULP * ulp_bf16(ref)
    return round_bf16(ref - d) == round_bf16(ref + d)


def assert_gelu(got, pre64, what, min_exact=0.995):
    """GELU of an exact fp32 pre-activation: <= 1 bf16 ulp from float64 erf-GELU down to x = -5.6 (|err| < 1e-8 below, where
    the epilogue clamps its polynomial), and >= 99.5 % exactly rounded there among the values its accuracy (0.07 ulp) cannot
    round either way (gelu_clear).  A truncating conversion leaves about half of them."""
    ref = gelu64(pre64)
    o = got.double()
    err = (o - ref).abs()
    core = pre64 >= -5.6
    bad = core & (err > ulp_bf16(ref))
    assert not bool(bad.any()), (what, int(bad.sum()), _first_bad(bad, o, ref))
    if bool((~core).any()):
        assert float(err[~core].max()) < 1e-8, what
    if bool(core.any()):
        clear = core & gelu_clear(ref)
        frac = float((o == round_bf16(ref))[clear].double().mean())
        assert frac >= min_exact, (what, frac)


def _act_ref(y, act):
    return torch.relu(y) if act == ACT_RELU else y


def _run_linear_act(ops, M, N, K, act, salt, bias=True, want_pre=False):
    A, W, b = exact_gemm_operands(M, N, K, salt, "cuda", bias=bias)
    y = exact_linear(A, W, b)
    if want_pre:
        out, pre = ops.linear_act(A, W, b, act, want_pre=True)
        assert_bits(pre, y, ("pre", M, N, K))
    else:
        out = ops.linear_act(A, W, b, act)
    assert out.shape == (M, N)
    if act == ACT_GELU:
        assert_gelu(out, y, ("gelu", M, N, K))
    else:
        assert_bits(out, _act_ref(y, act), ("act", act, M, N, K))


# ============================================================================================ 2. bit-exact GEMMs
@pytest.mark.gpu
@pytest.mark.parametrize("N,K", _small_cases())
def test_linear_act_exact_small_m(ops, N, K):
    """d2s_linear_act_pair_bf16 at M in {1, 127, 128, 129, 255, 256, 257}: act none / relu bit-exact, GELU to 1 ulp; the
    pre-activation output (want_pre) bit-exact; bias None covered."""
    for i, M in enumerate(SMALL_M):
        act = (ACT_NONE, ACT_RELU, ACT_GELU)[(i + N // 64 + K // 64) % 3]
        _run_linear_act(ops, M, N, K, act, salt=10 * i + N + K, bias=(i % 4 != 1), want_pre=(i % 2 == 0))


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,K", GROUP_CASES)
def test_linear_act_exact_every_split(ops, N, M, K):
    """Row counts that make the host split each row tile into every `groups` work-unit count it can choose, with and without
    resident A rows, and 74 CTA pairs +- one row."""
    act = (ACT_NONE, ACT_RELU, ACT_GELU)[(M + N) % 3]
    _run_linear_act(ops, M, N, K, act, salt=M + N, want_pre=(M % 2 == 1))


@pytest.mark.gpu
@pytest.mark.parametrize("M", BENCH_ROWS)
def test_linear_act_exact_bench_rows(ops, M):
    """The DeiT-S benchmark's qkv (N 1152) and fc1 (N 1536, GELU) shapes at batch 1024, every stage's token count."""
    _run_linear_act(ops, M, 1152, 384, ACT_NONE, salt=M)
    _run_linear_act(ops, M, 1536, 384, ACT_GELU, salt=M + 1)


def lnin_operands(M, K, salt, device="cuda"):
    """Raw rows x = mean_i + 2^k_i t with integer means, rstd_i = 2^-k_i, t in [-3, 3]; gamma in [1, 2] and beta in [-1, 1]
    per column: the normalised tile (x - mean) rstd gamma + beta = t gamma + beta is an exact small integer in any fp32 order."""
    mean = hgrid(M, 1, salt, -20, 20, device).double()
    k = hgrid(M, 1, salt + 1, 0, 3, device).double()
    t = hgrid(M, K, salt + 2, -3, 3, device).double()
    x = mean + torch.exp2(k) * t
    stats = torch.cat([mean, torch.exp2(-k)], 1).float().contiguous()
    g = hgrid(1, K, salt + 3, 1, 2, device)[0].double()
    bt = hgrid(1, K, salt + 4, -1, 1, device)[0].double()
    h = t * g + bt
    return x.to(BF), stats, g.to(BF), bt.to(BF), h


@pytest.mark.gpu
@pytest.mark.parametrize("N,M", LNIN_CASES)
def test_linear_lnin_act_exact(ops, N, M):
    """d2s_linear_lnin_act_pair_bf16 (the input LayerNorm formed in the resident A tile from per-row statistics): rows with
    different statistics and columns with different gamma / beta, so a wrong row of stats or column of gamma shows."""
    K = 384
    x, st, g, bt, h = lnin_operands(M, K, salt=N + M)
    wi = hgrid(N, K, N + M + 5, -15, 15, "cuda")
    bi = hgrid(1, N, N + M + 6, -1024, 1024, "cuda")[0]
    assert int(h.abs().sum(1).max()) * 15 + 1024 <= GRID_BOUND
    W, b = (wi.double() / 64).to(BF), (bi.double() / 64).to(BF)
    y = h @ W.double().t() + b.double()
    act = (ACT_NONE, ACT_GELU, ACT_RELU)[M % 3]
    out = ops.linear_act(x, W, b, act, in_stats=st, in_ln_weight=g, in_ln_bias=bt)
    if act == ACT_GELU:
        assert_gelu(out, y, ("lnin gelu", N, M))
    else:
        assert_bits(out, _act_ref(y, act), ("lnin", N, M))


# ---------------------------------------------------------------- LayerNorm checks shared by the residual / MLP / producer tests
EPS_STAT = 2.0 ** -17        # rstd, relative
EPS_MEAN = 2.0 ** -16        # mean, in units of the row's rms


def ln_reference(xk, eps):
    """Float64 LayerNorm statistics of exactly the bf16 rows a kernel wrote: (mean, rstd, rms), eps as the kernel's fp32."""
    x = xk.double()
    e = float(torch.tensor(eps, dtype=torch.float32))
    m = x.mean(1, keepdim=True)
    var = ((x - m) ** 2).mean(1, keepdim=True)
    return m, (var + e).rsqrt(), (x * x).mean(1, keepdim=True).sqrt()


def ln_metrics(xk, h, stats, g, bt, eps):
    """Per-row errors of a LayerNorm producer against float64 on its own rows xk (R, D):
    mean_err / rms, |rstd / rstd64 - 1|, |h - h64| in excess of the allowed band, and whether h is exactly rounded."""
    m, r, rms = ln_reference(xk, eps)
    out = {}
    if stats is not None:
        out["mean"] = ((stats[:, :1].double() - m).abs() / torch.clamp(rms, min=1e-30))[:, 0]
        out["rstd"] = ((stats[:, 1:].double() / r - 1).abs())[:, 0]
    if h is not None:
        x = xk.double()
        gg, bb = g.double()[None, :], bt.double()[None, :]
        z = (x - m) * r
        h64 = z * gg + bb
        # deviation any fp32 evaluation within the statistics bound may have before the final rounding (see the test's docstring)
        band = 1.01 * (gg.abs() * ((EPS_STAT + 2.0 ** -24) * z.abs() + (EPS_MEAN + 2.0 ** -24) * r * rms)
                       + 2.0 ** -23 * ((z * gg).abs() + bb.abs()))
        lo, hi = round_bf16(h64 - band), round_bf16(h64 + band)
        o = h.double()
        out["outside"] = ((o < lo) | (o > hi)).any(1)
        out["exact"] = (o == round_bf16(h64))
        # elements whose value fp32 itself pins down: the representation error of the mean, 2^-24 |mean| rstd |gamma|, is
        # under 1/256 of their ulp, so an exactly rounded result is expected unless the arithmetic is wrong
        out["clear"] = (2.0 ** -24 * m.abs() * r * gg.abs() + EPS_STAT * gg.abs() * z.abs()) < ulp_bf16(h64) / 256
        out["ulp"] = ((o - h64).abs() / ulp_bf16(h64))
    return out


def assert_ln(xk, h, stats, g, bt, eps, what):
    """The LayerNorm bound every producer must meet (derivation in test_layernorm_producers_against_float64)."""
    met = ln_metrics(xk, h, stats, g, bt, eps)
    if stats is not None:
        assert float(met["mean"].max()) <= EPS_MEAN, (what, "mean", float(met["mean"].max()))
        assert float(met["rstd"].max()) <= EPS_STAT, (what, "rstd", float(met["rstd"].max()), int(met["rstd"].argmax()))
    if h is not None:
        assert not bool(met["outside"].any()), (what, "h outside band", int(met["outside"].sum()))
        clear = met["clear"]
        if int(clear.sum()) > 1000:
            frac = float(met["exact"][clear].double().mean())
            assert frac >= 0.995, (what, "exactly rounded", frac)
    return met


@pytest.mark.gpu
@pytest.mark.parametrize("N", [192, 384, 768])
@pytest.mark.parametrize("K", [64, 384, 768, 1536, 3072])
def test_linear_residual_ln_exact(ops, N, K):
    """d2s_linear_residual_ln_bf16 / _stats_bf16: x' = bf16(x + bf16(acc + b)) bit-exact at ragged M (tails with fewer than 128
    rows in either CTA, one row, beyond 74 pairs), N = 768 as two 384-column halves; the LayerNorm and statistics to the
    producer bound on the kernel's own x'."""
    Ms = [1, 33, 130, 257, 1000] + ([NUM_PAIRS * 256 + 77] if K <= 768 else [])
    for i, M in enumerate(Ms):
        A, W, b = exact_gemm_operands(M, N, K, salt=M + N + K, device="cuda", bias=(i != 2))
        x = (hgrid(M, N, M + 7, -255, 255, "cuda").double() / 64).to(BF)
        g = (hgrid(1, N, 3, 48, 80, "cuda")[0].double() / 64).to(BF)
        bt = (hgrid(1, N, 4, -32, 32, "cuda")[0].double() / 128).to(BF)
        want = x.double() + round_bf16(exact_linear(A, W, b))
        xs, h = ops.linear_residual_ln(A, W, b, x, g, bt, 1e-6)
        assert_bits(xs, want, ("x'", M, N, K))
        assert_ln(xs, h, None, g, bt, 1e-6, ("h", M, N, K))
        xs2, st = ops.linear_residual_ln(A, W, b, x, eps=1e-5, want_norm=False, want_stats=True)
        assert torch.equal(xs2, xs)
        assert_ln(xs2, None, st, g, bt, 1e-5, ("stats", M, N, K))


def mlp_exact_operands(M, HID, salt, lnin, device="cuda"):
    """fc1 kept in GELU's identity range: h in [-7, 7], four weights in [-2, 2] per hidden unit (spread over the k-blocks), b1
    lifting every pre-activation to an integer in [6, 125], where bf16(GELU(u)) = u; fc2 weights in [-3, 3] 2^-6, so
    HID 125 3 <= 768000 < 2^20 grid units.  lnin: x = mean + 2^k t and h = t gamma + beta from per-row statistics."""
    D = 384
    if lnin:
        mean = hgrid(M, 1, salt, -20, 20, device).double()
        k = hgrid(M, 1, salt + 1, 0, 3, device).double()
        t = hgrid(M, D, salt + 2, -3, 3, device).double()
        xr = mean + torch.exp2(k) * t
        st = torch.cat([mean, torch.exp2(-k)], 1).float().contiguous()
        gi = hgrid(1, D, salt + 3, 1, 2, device)[0].double()
        bi = hgrid(1, D, salt + 4, -1, 1, device)[0].double()
        h64 = t * gi + bi
        extra = dict(in_stats=st, in_ln_weight=gi.to(BF), in_ln_bias=bi.to(BF))
    else:
        h64 = hgrid(M, D, salt, -7, 7, device).double()
        xr = hgrid(M, D, salt + 5, -255, 255, device).double() / 64
        extra = {}
    j = torch.arange(HID, device=device)[:, None]
    kk = torch.arange(D, device=device)[None, :]
    w1i = hgrid(HID, D, salt + 6, -2, 2, device) * ((kk - 7 * j) % 96 == 0)
    b1i = 6 + 7 * w1i.abs().sum(1) + hgrid(1, HID, salt + 7, 0, 7, device)[0]
    w2i = hgrid(D, HID, salt + 8, -3, 3, device)
    b2i = hgrid(1, D, salt + 9, -1024, 1024, device)[0]
    pre = h64 @ w1i.double().t() + b1i.double()
    assert float(pre.min()) >= 6 and float(pre.max()) <= 255
    assert int(pre.max()) * HID * 3 + 1024 <= GRID_BOUND
    W2 = (w2i.double() / 64).to(BF)
    b2 = (b2i.double() / 64).to(BF)
    u = round_bf16(gelu64(pre))                                  # = pre for integers >= 6
    y = round_bf16(u @ W2.double().t() + b2.double())
    x = xr.to(BF)
    return dict(h=h64.to(BF), w1=w1i.to(BF), b1=b1i.to(BF), w2=W2, b2=b2, x=x, want=x.double() + y, extra=extra)


MLP_CASES = [(HID, M) for HID in (128, 256, 768, 1536, 2048) for M in (1, 129, 255, 257, 1000)] + \
            [(1536, NUM_PAIRS * 256 + 1), (2048, NUM_PAIRS * 512 + 129)]


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["plain", "lnin"])
@pytest.mark.parametrize("HID,M", MLP_CASES)
def test_mlp_residual_ln_exact(ops, HID, M, form):
    """d2s_mlp_residual_ln_bf16 / d2s_mlp_lnin_residual_ln_bf16: x' bit-exact (fc1 -> GELU identity range -> fc2 -> residual),
    its LayerNorm and (lnin) its row statistics to the producer bound."""
    D = 384
    o = mlp_exact_operands(M, HID, salt=HID + M, lnin=(form == "lnin"))
    g = (hgrid(1, D, 3, 48, 80, "cuda")[0].double() / 64).to(BF)
    bt = (hgrid(1, D, 4, -32, 32, "cuda")[0].double() / 128).to(BF)
    h = None if form == "lnin" else o["h"]
    xs, hn = ops.mlp_residual_ln(h, o["w1"], o["b1"], o["w2"], o["b2"], o["x"], g, bt, 1e-6, **o["extra"])
    assert_bits(xs, o["want"], ("x'", form, HID, M))
    assert_ln(xs, hn, None, g, bt, 1e-6, ("h", form, HID, M))
    if form == "lnin":
        xs2, st = ops.mlp_residual_ln(None, o["w1"], o["b1"], o["w2"], o["b2"], o["x"], None, None, 1e-5, want_norm=False,
                                      want_stats=True, **o["extra"])
        assert torch.equal(xs2, xs)
        assert_ln(xs2, None, st, g, bt, 1e-5, ("stats", HID, M))


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(5, 197), (13, 77), (300, 2)])
@pytest.mark.parametrize("form", ["plain", "lnin"])
def test_mlp_residual_ln_exact_skipping_the_first_token(ops, B, T, form):
    """norm_row0 = 1 (the predictor's norm over x[:, 1:]): x' bit-exact, the LayerNorm of every token but the first of each image,
    compacted to (B, T - 1, D)."""
    D, HID = 384, 1536
    o = mlp_exact_operands(B * T, HID, salt=T, lnin=(form == "lnin"))
    g = (hgrid(1, D, 5, 48, 80, "cuda")[0].double() / 64).to(BF)
    bt = (hgrid(1, D, 6, -32, 32, "cuda")[0].double() / 128).to(BF)
    h = None if form == "lnin" else o["h"].view(B, T, D)
    xs, hn = ops.mlp_residual_ln(h, o["w1"], o["b1"], o["w2"], o["b2"], o["x"].view(B, T, D), g, bt, 1e-6, norm_row0=1, **o["extra"])
    assert hn.shape == (B, T - 1, D)
    assert_bits(xs.view(-1, D), o["want"], ("x'", B, T))
    assert_ln(xs[:, 1:].reshape(-1, D), hn.reshape(-1, D), None, g, bt, 1e-6, ("h", B, T))


@pytest.mark.gpu
def test_mlp_gelu_probe(ops):
    """The MLP kernel's own GELU, value by value: w1 = w2 = identity (HID = D = 384), x = 0, b = 0, so x' = bf16(GELU(h)) of the
    E1 warps.  <= 1 bf16 ulp from float64 erf-GELU down to h = -5.6 (|err| < 1e-8 below) and >= 99.5 % exactly rounded
    (the criterion of the gemm_pair epilogue test); and the integers 6 .. 255 map to themselves, which the exact MLP tests use."""
    D = 384
    grid = torch.linspace(-6.0, 6.0, 511 * D, device="cuda").to(BF).view(511, D)
    ints = torch.arange(6, 6 + D, device="cuda").clamp(max=255).to(BF).view(1, D)
    h = torch.cat([grid, ints]).contiguous()
    eye = torch.eye(D, device="cuda", dtype=BF)
    x = torch.zeros_like(h)
    xs, _ = ops.mlp_residual_ln(h, eye, None, eye, None, x, want_norm=False)
    assert torch.equal(xs[-1], ints[0])
    assert_gelu(xs[:-1], h[:-1].double(), "mlp gelu")


# ============================================================================================ 3. LayerNorm producers vs float64
LN_GROUPS = ["gauss", "massive", "ratio16", "ratio64", "ratio128", "ratio256", "const", "zero"]
LN_ROWS = 162                   # rows per group (gather: 1 CLS + 161 tokens; assemble: 161 patches + the class token)


def ln_rows(D, salt=0):
    """(8 * 162, D) bf16 rows, 162 per group of LN_GROUPS: Gaussian rows of scale 0.1 .. 10; one massive channel (200 sigma);
    mean / std in {16, 64, 128, 256}; constant rows; all-zero rows."""
    R = LN_ROWS
    g = torch.Generator(device="cuda").manual_seed(1234 + salt)
    z = torch.randn(8, R, D, generator=g, device="cuda", dtype=torch.float64)
    scale = torch.exp(torch.linspace(math.log(0.1), math.log(10.0), R, device="cuda", dtype=torch.float64))[:, None]
    rows = [z[0] * scale]
    m = z[1].clone()
    m[torch.arange(R), torch.arange(R) * 7 % D] = 200.0 * torch.sign(torch.randn(R, generator=g, device="cuda", dtype=torch.float64))
    rows.append(m)
    sgn = torch.where(torch.arange(R, device="cuda") % 2 == 0, 1.0, -1.0).double()[:, None]
    for i, ratio in enumerate((16, 64, 128, 256)):
        rows.append(sgn * ratio * (1 + 0.5 * scale / 10) + z[2 + i])
    const = torch.tensor([3.5, -1.25, 300.0, 0.1, -7.0, 1e-3], device="cuda", dtype=torch.float64)
    rows.append(const[torch.arange(R) % 6][:, None].expand(R, D))
    rows.append(torch.zeros(R, D, device="cuda", dtype=torch.float64))
    return torch.cat(rows).to(BF).contiguous()


def ln_affine(D):
    g = (1 + 0.3 * torch.randn(D, generator=torch.Generator(device="cuda").manual_seed(7), device="cuda")).to(BF)
    bt = (0.2 * torch.randn(D, generator=torch.Generator(device="cuda").manual_seed(8), device="cuda")).to(BF)
    return g, bt


def ln_produce(ops, producer, rows, g, bt, eps):
    """Run one producer on `rows` (R, D) bf16; returns (the rows it wrote, its normalised output or None, its stats or None)."""
    R, D = rows.shape
    dev = rows.device
    if producer == "layer_norm":                  # the standalone two-pass kernel (d2s_layernorm_fwd)
        h = torch.empty_like(rows)
        st = torch.empty(R, 2, dtype=torch.float32, device=dev)
        g32, bt32 = g.float().contiguous(), bt.float().contiguous()      # alive until the kernel has run
        ops._call("d2s_layernorm_fwd", ops._ptr(rows), 1, ops._ptr(g32), ops._ptr(bt32), R, D, float(eps), ops._ptr(h), 1,
                  ops._ptr(st), ops._stream(rows))
        torch.cuda.current_stream().synchronize()
        return rows, h, st
    if producer == "add_layernorm":
        xs, h = ops.add_layernorm(rows.view(1, R, D), torch.zeros(1, R, D, dtype=BF, device=dev), g, bt, eps)
        return xs.view(R, D), h.view(R, D), None
    if producer.startswith("gather"):
        B = R // LN_ROWS
        x = rows.view(B, LN_ROWS, D)                      # token 0 is the CLS row, 161 spatial tokens, 160 kept (permuted)
        kept = torch.stack([torch.randperm(LN_ROWS - 1, generator=fx.gen(40 + b))[:LN_ROWS - 2] for b in range(B)]).to(dev)
        xs, second = ops.gather_layernorm(x, kept, g, bt, eps, want_stats=producer.endswith("stats"))
        xs = xs.reshape(-1, D)
        return (xs, None, second) if producer.endswith("stats") else (xs, second.reshape(-1, D), None)
    if producer.startswith("assemble"):
        B = R // LN_ROWS
        patches = rows.view(B, LN_ROWS, D)[:, 1:].contiguous()
        cls = rows[0].view(1, 1, D)
        pos = torch.zeros(1, LN_ROWS, D, dtype=BF, device=dev)
        xs, second = ops.assemble_layernorm(patches, cls, pos, g, bt, eps, want_stats=producer.endswith("stats"))
        xs = xs.reshape(-1, D)
        return (xs, None, second) if producer.endswith("stats") else (xs, second.reshape(-1, D), None)
    if producer.startswith("linear_residual"):          # W = 0, no bias: x' = x
        a = torch.zeros(R, 64, dtype=BF, device=dev)
        w = torch.zeros(D, 64, dtype=BF, device=dev)
        if producer.endswith("stats"):
            xs, st = ops.linear_residual_ln(a, w, None, rows, eps=eps, want_norm=False, want_stats=True)
            return xs, None, st
        xs, h = ops.linear_residual_ln(a, w, None, rows, g, bt, eps)
        return xs, h, None
    if producer.startswith("mlp"):                      # W1 = W2 = 0, no biases: x' = x
        w1 = torch.zeros(128, D, dtype=BF, device=dev)
        w2 = torch.zeros(D, 128, dtype=BF, device=dev)
        if producer == "mlp":
            xs, h = ops.mlp_residual_ln(torch.zeros_like(rows), w1, None, w2, None, rows, g, bt, eps)
            return xs, h, None
        st_in = torch.cat([torch.zeros(R, 1, device=dev), torch.ones(R, 1, device=dev)], 1).contiguous()
        ones, zeros = torch.ones(D, dtype=BF, device=dev), torch.zeros(D, dtype=BF, device=dev)
        if producer == "mlp_lnin_stats":
            xs, st = ops.mlp_residual_ln(None, w1, None, w2, None, rows, None, None, eps, want_norm=False, in_stats=st_in,
                                         in_ln_weight=ones, in_ln_bias=zeros, want_stats=True)
            return xs, None, st
        xs, h = ops.mlp_residual_ln(None, w1, None, w2, None, rows, g, bt, eps, in_stats=st_in, in_ln_weight=ones, in_ln_bias=zeros)
        return xs, h, None
    raise ValueError(producer)


LN_PRODUCERS = [("layer_norm", 384), ("layer_norm", 768), ("add_layernorm", 384), ("gather", 384), ("gather_stats", 384),
                ("assemble", 384), ("assemble_stats", 384), ("linear_residual", 384), ("linear_residual_stats", 384),
                ("linear_residual", 768), ("linear_residual_stats", 768), ("mlp", 384), ("mlp_lnin", 384), ("mlp_lnin_stats", 384)]


@pytest.mark.gpu
@pytest.mark.parametrize("eps", [1e-6, 1e-5])
@pytest.mark.parametrize("producer,D", LN_PRODUCERS)
def test_layernorm_producers_against_float64(ops, producer, D, eps):
    """Every producer of a LayerNorm (or of the per-row statistics a consumer applies) on the same rows, against float64
    LayerNorm of exactly the bf16 rows it wrote.  Bound, from fp32 arithmetic:

    * statistics: every producer sums its n <= 768 terms in fp32 chains of at most 192 additions followed by a short tree
      (L <= 195 roundings in all).  For the variance the terms are squared deviations from the row's mean, or, in the fused
      kernels on rows with 8 mean^2 <= var, squares, which then add up to at most 1.125 x the squared deviations (a row farther
      off zero gets two-pass statistics there).  A sum of non-negative terms through L additions is off by at most L 2^-24 of
      itself, so the variance is within 1.125 x 195 x 2^-24 < 2^-16.2 relative, rstd within 2^-17.2 + 2^-22 (rsqrtf: 2 ulp)
      < eps_s = 2^-17, and the mean within 195 x 2^-24 mean |x| < eps_m rms(row), eps_m = 2^-16.  The mean's
      own rounding, (2^-24 |mean|)^2, adds below 2^-32 of var + eps here except for constant rows, whose fp32 sums are exact
      and whose mean a correctly rounded division leaves exact.  A one-pass E[x^2] - mean^2 loses log2(1 + mean^2 / var) bits
      and fails this at mean / std >= 16; an unbiased variance (/ (n - 1)) is off by 1.3e-3.
    * normalised output h = fma(fma(x, rstd, -mean rstd), gamma, beta) or fma((x - mean) rstd, gamma, beta): with the
      statistics within these bounds, the value before the final rounding is within
      band = |gamma| ((eps_s + 2^-24) |z| + (eps_m + 2^-24) rstd rms) + 2^-23 (|z gamma| + |beta|), z = (x - mean64) rstd64,
      of h64 (the 2^-24 terms: shift rounding and the two fma roundings), so h must lie between the bf16 roundings of
      h64 -+ band: at most one ulp away, and bit-exact wherever the band does not straddle a rounding midpoint.  Where even the
      mean's representation error is under 1/256 ulp of h, at least 99.5 % must be exactly rounded.
    """
    rows = ln_rows(D)
    g, bt = ln_affine(D)
    xk, h, st = ln_produce(ops, producer, rows, g, bt, eps)
    assert xk.shape[1] == D
    assert_ln(xk, h, st, g, bt, eps, (producer, D, eps))


# ============================================================================================ 4. Gaussian operands
def _acc_bound(a, w, b=None):
    """fp32 accumulation through tcgen05: K / 16 accumulator additions and <= 16 alignments inside an MMA, each off by at most
    one fp32 ulp (2^-23 = 2 x 2^-24: truncation allowed) of a partial sum bounded by sum |a||w| (+ |b|):
    c 2^-24 sum_k |a_k||w_k| with c = 2 (K / 16 + 16 + 1)."""
    K = a.shape[1]
    s = a.double().abs() @ w.double().abs().t()
    if b is not None:
        s = s + b.double().abs()
    return 2.0 * (K / 16 + 17) * 2.0 ** -24 * s


def _check_rounded(got, v64, err, what, min_exact=0.99, count=None):
    """got = bf16 of a value within err of v64: |got - v64| <= err + ulp(|v64| + err) / 2; >= 99 % equal to round(v64) (truncation
    instead of rounding would leave ~50 %).  The residual sums are compared with the chain rounded at the same two points instead."""
    o = got.double()
    lim = err + 0.5 * ulp_bf16(v64.abs() + err)
    bad = (o - v64).abs() > lim
    assert not bool(bad.any()), (what, int(bad.sum()), _first_bad(bad, o, v64))
    eq = o == round_bf16(v64)
    frac = float((eq if count is None else eq[count]).double().mean())
    assert frac >= min_exact, (what, frac)


def _gauss(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, generator=g, device="cuda") * scale).to(BF)


@pytest.mark.gpu
@pytest.mark.parametrize("name,M,N,K,act,lnin", [
    ("qkv DeiT-S lnin", 4 * 197 + 3, 1152, 384, ACT_NONE, True),
    ("qkv DeiT-S", 3 * 197, 1152, 384, ACT_NONE, False),
    ("qkv DeiT-B", 4 * 197 + 3, 2304, 768, ACT_NONE, False),
    ("fc1 DeiT-S", 6209, 1536, 384, ACT_GELU, False),
    ("fc1 DeiT-B", 2 * 197, 3072, 768, ACT_GELU, False),
    ("predictor Linear", 4 * 197, 384, 384, ACT_GELU, True),
])
def test_linear_act_gaussian(ops, name, M, N, K, act, lnin):
    """Realistic weight scales at the engine's shapes, against float64: one bf16 rounding plus the fp32 accumulation bound
    (_acc_bound); GELU adds its slope (<= 1.13) times that and its own error (0.07 ulp; 3.8e-5 absolute below -5.6), and its
    exact-rounding count leaves out what that error may round either way; lnin adds one bf16 ulp of each normalised input
    (h computed in fp32 vs float64) times |w|."""
    w = _gauss((N, K), N + K, K ** -0.5)
    b = _gauss((N,), N, 0.1)
    if lnin:
        x = (_gauss((M, K), M + 1, 1.0).float() * 2 + 0.5).to(BF)
        g = (1 + 0.2 * _gauss((K,), 3).float()).to(BF)
        bt = _gauss((K,), 4, 0.2)
        xf = x.double()
        mean = xf.mean(1, keepdim=True)
        rstd = (((xf - mean) ** 2).mean(1, keepdim=True) + 1e-6).rsqrt()
        st = torch.cat([mean, rstd], 1).float().contiguous()
        h64 = (xf - st[:, :1].double()) * st[:, 1:].double() * g.double() + bt.double()     # with the fp32 statistics supplied
        a64 = round_bf16(h64)
        out = ops.linear_act(x, w, b, act, in_stats=st, in_ln_weight=g, in_ln_bias=bt)
        flip = ulp_bf16(h64).abs() @ w.double().abs().t() + 2.0 ** -20 * (h64.abs() @ w.double().abs().t())
    else:
        x = _gauss((M, K), M, 1.0)
        a64 = x.double()
        out = ops.linear_act(x, w, b, act)
        flip = 0.0
    v = a64 @ w.double().t() + b.double()
    err = _acc_bound(a64, w, b) + flip
    if act == ACT_GELU:
        gv = gelu64(v)
        _check_rounded(out, gv, 1.13 * err + GELU_ULP * ulp_bf16(gv) + 4e-5 * (v < -5.6), name, count=gelu_clear(gv))
    else:
        _check_rounded(out, v, err, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name,M,N,K", [
    ("proj DeiT-S", 4 * 197 + 3, 384, 384), ("fc2 DeiT-S", 3 * 197, 384, 1536),
    ("proj DeiT-B", 2 * 197 + 1, 768, 768), ("fc2 DeiT-B", 2 * 197, 768, 3072),
    ("proj 192", 1000, 192, 384),
])
def test_linear_residual_gaussian(ops, name, M, N, K):
    """x' = bf16(x + bf16(A W^T + b)) against float64: y within the accumulation bound plus one rounding, then one more
    rounding of the residual sum; >= 99 % of x' equal to the float64 chain rounded at the same two points."""
    a = _gauss((M, K), M + K, 1.0)
    w = _gauss((N, K), N + K + 1, K ** -0.5)
    b = _gauss((N,), N + 2, 0.1)
    x = _gauss((M, N), M + 3, 1.5)
    g, bt = ln_affine(N)
    xs, h = ops.linear_residual_ln(a, w, b, x, g, bt, 1e-6)
    y64 = a.double() @ w.double().t() + b.double()
    ey = _acc_bound(a, w, b)
    ey = ey + 0.5 * ulp_bf16(y64.abs() + ey)                       # |bf16(y) - y64|
    _check_rounded(xs, x.double() + y64, ey, name, min_exact=0.0)
    frac = float((xs.double() == round_bf16(x.double() + round_bf16(y64))).double().mean())
    assert frac >= 0.99, (name, frac)
    assert_ln(xs, h, None, g, bt, 1e-6, name)


@pytest.mark.gpu
@pytest.mark.parametrize("M", [3 * 197, 4 * 197 + 3])
def test_mlp_gaussian(ops, M):
    """The MLP kernel at DeiT-S (HID 1536) against the float64 chain u = bf16(GELU(h W1^T + b1)), y = bf16(u W2^T + b2),
    x' = bf16(x + y): the fc2 accumulation bound, plus sum_h |w2| ulp(u_h) for hidden values that land one ulp off (fc1's own
    accumulation error and the GELU's 0.07 ulp move a few percent of the roundings), plus two roundings.  And >= 99 % of x'
    exactly as the chain continued in float64 from the hidden values the pair GEMM computes with the same GELU
    (linear_act, fc1 + GELU epilogue): what is left then is fc2's fp32 accumulation against float64."""
    D, HID = 384, 1536
    h = _gauss((M, D), M, 1.0)
    w1, b1 = _gauss((HID, D), 11, D ** -0.5), _gauss((HID,), 12, 0.1)
    w2, b2 = _gauss((D, HID), 13, HID ** -0.5), _gauss((D,), 14, 0.1)
    x = _gauss((M, D), M + 1, 1.5)
    g, bt = ln_affine(D)
    xs, hn = ops.mlp_residual_ln(h, w1, b1, w2, b2, x, g, bt, 1e-6)
    u = round_bf16(gelu64(h.double() @ w1.double().t() + b1.double()))
    y64 = u @ w2.double().t() + b2.double()
    ey = _acc_bound(u, w2, b2) + ulp_bf16(u) @ w2.double().abs().t()
    ey = ey + 0.5 * ulp_bf16(y64.abs() + ey)
    _check_rounded(xs, x.double() + y64, ey, "mlp", min_exact=0.0)
    uk = ops.linear_act(h, w1, b1, ACT_GELU).double()
    yk = uk @ w2.double().t() + b2.double()
    frac = float((xs.double() == round_bf16(x.double() + round_bf16(yk))).double().mean())
    assert frac >= 0.99, ("mlp", frac)
    assert_ln(xs, hn, None, g, bt, 1e-6, "mlp h")
