"""Training attention beyond 256 tokens: the key-blocked forward with row statistics (d2s_attn_long_fwd_stats) and the key-blocked
backward (d2s_attn_long_bwd), through ops.attention_train and engine.attention_pre_proj.  Against float64 autograd of the reference
formula, against the T <= 208 flash kernels where both run, at the edges of the exponent range, in guard zones, and inside
DeiT-S-width models at 384 and 512 pixels."""
import copy
import ctypes
import types

import pytest
import torch

import fixtures as fx

DEIT_S_W = dict(patch_size=16, embed_dim=384, num_heads=6, mlp_ratio=4, qkv_bias=True)
K2 = 1.4426950408889634


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ref(qkv, H, policy=None, eps=1e-6):
    """Attention.forward's core (dynamic_vit.py:195-214 softmax_with_policy, :218-234) in float64 with scale hd^-0.5, differentiable
    in qkv and policy: (out (B,T,H*hd), cls_row (B,H,T), probabilities (B,H,T,T))."""
    B, T, C3 = qkv.shape
    hd = C3 // 3 // H
    q, k, v = qkv.view(B, T, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)
    s = (q @ k.transpose(-1, -2)) * hd ** -0.5
    if policy is None:
        p = torch.softmax(s, dim=-1)
    else:
        pol = policy.reshape(B, 1, 1, T)
        eye = torch.eye(T, dtype=torch.float64, device=qkv.device).view(1, 1, T, T)
        mask = pol + (1.0 - pol) * eye
        e = (s - s.amax(-1, keepdim=True)).exp() * mask
        p = (e + eps / T) / (e.sum(-1, keepdim=True) + eps)
    return (p @ v).transpose(1, 2).reshape(B, T, H * hd), p[:, :, 0, :], p


def _policy(B, T, g, kind):
    if kind == "none":
        return None
    pol = torch.rand(B, T, device="cuda", generator=g)
    if kind == "binary":
        pol = (pol > 0.3).float()
    pol[:, 0] = 1
    return pol


def _far_logits(B, T, H, seed=140):
    """The construction of test_gpu_long_attn.py: every second query row holds logits ~200 nats above the reference columns (the
    first 16 keys) at a key of the last key block and at key 300, which image 0's policy masks (the reference is raised by whole
    binades there); other rows overflow and are redone in fp32 from global memory."""
    hd = 64
    g = fx.gen(seed)
    qkv = torch.randn(B, T, 3, H, hd, generator=g) * 0.5
    u = torch.nn.functional.normalize(torch.randn(hd, generator=g), dim=0)
    j_last, j_mask = T - 13, 300
    qkv[:, 0::2, 0] += 40.0 * u
    qkv[:, j_last, 1] = 40.0 * u
    qkv[:, j_mask, 1] = 40.2 * u
    qkv[:, 5, 1] = 10.0 * u
    qkv = qkv.reshape(B, T, 3 * H * hd).bfloat16().cuda()
    pol = (torch.rand(B, T, generator=g) > 0.3).float().cuda()
    pol[:, 0] = 1
    pol[0, j_last], pol[0, j_mask] = 1, 0
    pol[1, j_last], pol[1, j_mask] = 1, 1
    return qkv, pol


def _fwd_stats(lib, qkv, H, pol, want_cls=True):
    B, T, _ = qkv.shape
    out = torch.empty(B, T, H * 64, dtype=torch.bfloat16, device="cuda")
    cls = torch.empty(B, H, T, device="cuda") if want_cls else None
    stats = torch.full((B, H, T, 4), float("nan"), device="cuda")
    lib.call("d2s_attn_long_fwd_stats", qkv.data_ptr(), None if pol is None else pol.data_ptr(), B, T, H, 64, 0.125, 1e-6,
             out.data_ptr(), None if cls is None else cls.data_ptr(), stats.data_ptr(), _stream())
    return out, cls, stats


# ----------------------------------------------------------------------------------------------------------------- host / CPU
def test_long_attention_training_argument_errors_precede_any_launch(d2s):
    lib = d2s._lib.load()
    before = d2s._lib.launch_count()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    f = lib.d2s_attn_long_fwd_stats
    assert f(None, None, 2, 577, 6, 64, 0.125, 1e-6, p, None, p, None) == 1 and b"null" in lib.d2s_last_error()
    assert f(p, None, 2, 577, 6, 64, 0.125, 1e-6, p, None, None, None) == 1 and b"null" in lib.d2s_last_error()
    assert f(p, None, 2, 577, 6, 48, 0.125, 1e-6, p, None, p, None) == 1 and b"head dim" in lib.d2s_last_error()
    assert f(p, None, 2, 0, 6, 64, 0.125, 1e-6, p, None, p, None) == 1 and b"T=0" in lib.d2s_last_error()
    assert f(p, None, 2, 2049, 6, 64, 0.125, 1e-6, p, None, p, None) == 1 and b"T=2049" in lib.d2s_last_error()
    assert f(p, None, 2, 577, 6, 64, 0.0, 1e-6, p, None, p, None) == 1 and b"scale" in lib.d2s_last_error()
    assert f(p, None, 2, 577, 6, 64, 0.125, 1e-6, p, None, p + 8, None) == 2
    assert f(p + 4, None, 2, 577, 6, 64, 0.125, 1e-6, p, None, p, None) == 2
    assert f(p, None, 0, 577, 6, 64, 0.125, 1e-6, p, None, p, None) == 0             # an empty batch is a no-op
    b = lib.d2s_attn_long_bwd
    #        qkv pol out gout cls gcls stats B  T   H  hd scale  dqkv gpol ws
    args = [p, None, p, p, None, None, p, 2, 577, 6, 64, 0.125, p, None, p, None]

    def call(**kw):
        a = list(args)
        for i, v in kw.items():
            a[int(i[1:])] = v
        return b(*a)
    for i in (0, 2, 3, 6, 12, 14):                                                   # every required pointer
        assert call(**{f"a{i}": None}) == 1 and b"null" in lib.d2s_last_error(), i
    assert call(a1=p) == 1 and b"policy and gpolicy" in lib.d2s_last_error()
    assert call(a13=p) == 1 and b"policy and gpolicy" in lib.d2s_last_error()
    assert call(a5=p) == 1 and b"cls_row" in lib.d2s_last_error()
    assert call(a10=48) == 1 and b"head dim" in lib.d2s_last_error()
    assert call(a8=0) == 1 and b"T=0" in lib.d2s_last_error()
    assert call(a8=2049) == 1 and b"T=2049" in lib.d2s_last_error()
    assert call(a11=0.0) == 1 and b"scale" in lib.d2s_last_error()
    assert call(a11=-0.125) == 1 and b"scale" in lib.d2s_last_error()
    for i in (0, 2, 3, 6, 12, 14):                                                   # misalignment
        assert call(**{f"a{i}": p + 4}) == 2, i
    assert d2s._lib.launch_count() == before
    assert call(a7=0) == 0                                                            # an empty batch is a no-op
    assert d2s._lib.launch_count() == before


def test_engine_routes_long_bf16_training_attention_behind_its_switch(d2s, monkeypatch):
    """The training branch takes bf16 with head dim 64 and 1 <= T <= 2048 (ops.attention_train_ok: the flash pair up to 208 tokens,
    the key-blocked pair beyond); _LONG_ATTN = False sends everything above 208 tokens back to torch matmuls around the policy
    softmax, as every other dtype, head dim and non-positive scale goes there."""
    train_ok = d2s.ops.attention_train_ok
    bf = lambda T, hd=64: torch.empty(1, T, 3 * 6 * hd, dtype=torch.bfloat16)     # noqa: E731
    assert train_ok(bf(1), 6) and train_ok(bf(197), 6) and train_ok(bf(2048), 6) and train_ok(bf(197), 6, 0.125)
    assert not train_ok(bf(2049), 6) and not train_ok(torch.empty(1, 0, 3 * 6 * 64, dtype=torch.bfloat16), 6)
    assert not train_ok(bf(197, 48), 6) and not train_ok(bf(197, 32), 6) and not train_ok(bf(197), 4)
    assert not train_ok(torch.empty(1, 197, 3 * 6 * 64, dtype=torch.float32), 6)
    assert not train_ok(torch.empty(1, 197, 3 * 6 * 64, dtype=torch.float16), 6)
    assert not train_ok(bf(197), 6, 0.0) and not train_ok(bf(577), 6, -0.125) and not train_ok(bf(197), 6, float("nan"))
    ok = d2s.engine._attn_train_kernel_ok
    assert ok(bf(577), 6) and ok(bf(2048), 6) and ok(bf(197), 6) and ok(bf(208), 6) and ok(bf(209), 6) and ok(bf(256), 6)
    assert ok(bf(257), 6) and ok(bf(197), 6, 0.125)
    assert not ok(bf(2049), 6)
    assert not ok(torch.empty(1, 577, 3 * 6 * 64, dtype=torch.float32), 6)
    assert not ok(torch.empty(1, 197, 3 * 6 * 64, dtype=torch.float32), 6)
    assert not ok(bf(577, 48), 6)
    assert not ok(bf(197, 48), 6)                                                    # head dim 48 goes to torch
    assert not ok(bf(197), 6, 0.0) and not ok(bf(577), 6, -0.125)                    # so does a non-positive scale
    monkeypatch.setattr(d2s.engine, "_LONG_ATTN", False)
    assert not ok(bf(577), 6) and not ok(bf(257), 6) and not ok(bf(256), 6) and not ok(bf(209), 6)
    assert ok(bf(208), 6) and ok(bf(197), 6)


# ----------------------------------------------------------------------------------------------------------------- kernels
@pytest.mark.gpu
@pytest.mark.parametrize("T", [209, 256, 257, 577, 1025])
@pytest.mark.parametrize("with_policy", [False, True])
def test_long_row_statistics(d2s, cuda_dev, T, with_policy):
    """stats of d2s_attn_long_fwd_stats reproduce the float64 probabilities through P = 2^(k2 s - m') m / den + c / den, and out /
    cls_row are bit-identical to d2s_attn_long_fwd's."""
    lib = d2s._lib
    B, H = 2, 3
    g = torch.Generator(device="cuda").manual_seed(5000 + T)
    qkv = (torch.randn(B, T, 3 * H * 64, device="cuda", generator=g) * 0.8).bfloat16()
    pol = _policy(B, T, g, "binary") if with_policy else None
    _check_stats(lib, qkv, H, pol)


@pytest.mark.gpu
def test_long_row_statistics_logits_far_above_the_row_reference(d2s, cuda_dev):
    """Rows redone in fp32 from global memory and rows whose reference was raised by whole binades (image 0, masked key) store
    the m' and den that produced out."""
    qkv, pol = _far_logits(2, 577, 6)
    _check_stats(d2s._lib, qkv, 6, pol)
    _check_stats(d2s._lib, qkv, 6, None)


def _check_stats(lib, qkv, H, pol):
    B, T, _ = qkv.shape
    out, cls, stats = _fwd_stats(lib, qkv, H, pol)
    o0 = torch.empty_like(out)
    c0 = torch.empty_like(cls)
    lib.call("d2s_attn_long_fwd", qkv.data_ptr(), None if pol is None else pol.data_ptr(), None, B, T, H, 64, 0.125, 1e-6, o0.data_ptr(),
             c0.data_ptr(), _stream())
    assert torch.equal(out, o0) and torch.equal(cls, c0)
    st = stats.double()
    assert bool(torch.isfinite(st[..., :3]).all())
    assert bool((st[..., 0] == st[..., 0].round()).all())                      # a whole number of binades
    v = qkv.double().view(B, T, 3, H, 64)
    s = torch.einsum("bihd,bjhd->bhij", v[:, :, 0], v[:, :, 1]) * 0.125
    _, _, ref = _ref(qkv.double(), H, None if pol is None else pol.double())
    e = torch.exp2(s * K2 - st[..., 0:1])
    if pol is not None:
        p = pol.double().view(B, 1, 1, T)
        e = e * (p + (1 - p) * torch.eye(T, dtype=torch.float64, device="cuda").view(1, 1, T, T))
    torch.testing.assert_close(e * st[..., 1:2] + st[..., 2:3], ref, rtol=2e-4, atol=1e-7)


def _train_vs_f64(d2s, qkv, H, pol, seed, attend=None, dpol_tol=1e-3):
    """attend(qkv, H, policy) -> (out, cls_row), ops.attention_train by default: forward + backward (a loss on out and on the CLS
    rows) against float64 autograd of the reference formula on the same bf16 inputs, at the bounds of
    test_gpu_parity.py::test_attention_train_fwd_bwd_vs_oracle_autograd."""
    B, T, C3 = qkv.shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    go = (torch.randn(B, T, C3 // 3, device="cuda", generator=g) * 0.5).bfloat16()
    gc = torch.randn(B, H, T, device="cuda", generator=g) * 0.5
    q1 = qkv.clone().requires_grad_(True)
    p1 = pol.clone().requires_grad_(True) if pol is not None else None
    if attend is None:
        o1, c1 = d2s.ops.attention_train(q1, H, policy=p1, want_cls_row=True)
    else:
        o1, c1 = attend(q1, H, p1)
    (o1.float() * go.float()).sum().add((c1.float() * gc).sum()).backward()
    q2 = qkv.double().requires_grad_(True)
    p2 = pol.double().requires_grad_(True) if pol is not None else None
    o2, c2, _ = _ref(q2, H, p2)
    (o2 * go.double()).sum().add((c2 * gc.double()).sum()).backward()
    assert bool(torch.isfinite(o1).all()) and bool(torch.isfinite(q1.grad).all())
    torch.testing.assert_close(o1.double(), o2.detach(), rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(c1.double(), c2.detach(), rtol=2e-2, atol=2e-3)
    gq1, gq2 = q1.grad.double(), q2.grad
    assert float((gq1 - gq2).abs().max()) <= 3e-2 * float(gq2.abs().max()) + 1e-3
    if pol is not None:
        gp1, gp2 = p1.grad.double(), p2.grad
        assert bool(torch.isfinite(gp1).all())
        assert float((gp1 - gp2).abs().max()) <= dpol_tol * float(gp2.abs().max()) + 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("T", [209, 256, 257, 300, 577, 785, 1025, 2048])
@pytest.mark.parametrize("H", [6, 12])
@pytest.mark.parametrize("pol_kind", ["none", "binary", "fraction"])
def test_long_attention_train_matches_float64_autograd(d2s, cuda_dev, T, H, pol_kind):
    B = 2
    g = torch.Generator(device="cuda").manual_seed(6000 + T + H)
    qkv = (torch.randn(B, T, 3 * H * 64, device="cuda", generator=g) * 0.7).bfloat16()
    n0 = d2s._lib.launch_count()
    _train_vs_f64(d2s, qkv, H, _policy(B, T, g, pol_kind), 6100 + T)
    assert d2s._lib.launch_count() > n0


@pytest.mark.gpu
@pytest.mark.parametrize("hd", [32, 48])
def test_bf16_training_at_other_head_dims_runs_the_torch_branch(d2s, cuda_dev, monkeypatch, hd):
    """bf16 training at a head dim the tcgen05 pairs do not take goes through engine.attention_pre_proj's torch branch (matmuls around
    ops.softmax_with_policy), never ops.attention_train, and matches float64 autograd of the reference formula.  The stand-in
    module's qkv projection returns the packed tensor under test, so its gradient is observed directly; x carries the shape only
    (fp32, so no qkv GEMM takes it).  d policy is held to 3e-2: this branch rounds the scores, the probabilities and dP to bf16."""
    B, T, H = 2, 197, 6
    g = torch.Generator(device="cuda").manual_seed(6500 + hd)
    qkv = (torch.randn(B, T, 3 * H * hd, device="cuda", generator=g) * 0.7).bfloat16()
    x = torch.empty(B, T, H * hd, device="cuda")
    monkeypatch.setattr(d2s.ops, "attention_train", lambda *a, **k: pytest.fail("head dim %d reached ops.attention_train" % hd))

    def attend(q, H, policy):
        m = types.SimpleNamespace(num_heads=H, scale=hd ** -0.5, qkv=lambda _: q)
        return d2s.engine.attention_pre_proj(m, x, policy=policy, return_cls_attn=True)
    _train_vs_f64(d2s, qkv, H, _policy(B, T, g, "fraction"), 6600 + hd, attend=attend, dpol_tol=3e-2)


@pytest.mark.gpu
def test_long_attention_train_logits_far_above_the_row_reference(d2s, cuda_dev):
    qkv, pol = _far_logits(2, 577, 6)
    _train_vs_f64(d2s, qkv, 6, pol, 7000)
    _train_vs_f64(d2s, qkv, 6, None, 7001)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 17, 128, 129, 197, 208])
@pytest.mark.parametrize("with_policy", [False, True])
def test_long_backward_agrees_with_the_flash_kernels(d2s, cuda_dev, T, with_policy):
    """Where both run, the key-blocked entry points and d2s_attn_policy_fwd / d2s_attn_policy_bwd compute the same thing: the
    same exponent reference and exponentials, a different summation order (one bf16 ulp of out and dqkv, fp32 rounding of the
    statistics and of d policy)."""
    lib = d2s._lib
    B, H = 3, 6
    g = torch.Generator(device="cuda").manual_seed(8000 + T)
    qkv = (torch.randn(B, T, 3 * H * 64, device="cuda", generator=g) * 0.8).bfloat16()
    go = (torch.randn(B, T, H * 64, device="cuda", generator=g) * 0.5).bfloat16()
    gc = torch.randn(B, H, T, device="cuda", generator=g) * 0.5
    pol = _policy(B, T, g, "binary") if with_policy else None
    pp = None if pol is None else pol.data_ptr()
    o1, c1, s1 = _fwd_stats(lib, qkv, H, pol)
    o2 = torch.empty_like(o1)
    c2, s2 = torch.empty_like(c1), torch.empty_like(s1)
    lib.call("d2s_attn_policy_fwd", qkv.data_ptr(), pp, 1, B, T, H, 64, 0.125, 1e-6, o2.data_ptr(), c2.data_ptr(), s2.data_ptr(), _stream())
    torch.testing.assert_close(o1.float(), o2.float(), rtol=1.6e-2, atol=1e-3)
    torch.testing.assert_close(c1, c2, rtol=2e-3, atol=1e-6)
    # the exponent reference is a free whole-binade choice (the T > 128 flash kernel takes it per key half); what both must agree on
    # is the normaliser 2^m' den and the offset c/den
    torch.testing.assert_close(s1[..., 0] - torch.log2(s1[..., 1]), s2[..., 0] - torch.log2(s2[..., 1]), rtol=0, atol=1e-5)
    torch.testing.assert_close(s1[..., 2], s2[..., 2], rtol=1e-5, atol=0)
    # both backwards on the flash forward's outputs
    res = []
    for name in ("d2s_attn_long_bwd", "d2s_attn_policy_bwd"):
        st = s2.clone()
        dq = torch.empty_like(qkv)
        gp = torch.zeros(B, T, device="cuda") if pol is not None else None
        ws = [torch.empty(B, H, T, 64, device="cuda").data_ptr()] if name == "d2s_attn_long_bwd" else []
        lib.call(name, qkv.data_ptr(), pp, o2.data_ptr(), go.data_ptr(), c2.data_ptr(), gc.data_ptr(), st.data_ptr(), B, T, H, 64, 0.125,
                 dq.data_ptr(), None if gp is None else gp.data_ptr(), *ws, _stream())
        res.append((dq, gp))
    (d1, g1), (d2, g2) = res
    assert float((d1.float() - d2.float()).abs().max()) <= 8e-3 * float(d2.float().abs().max()) + 1e-6
    if pol is not None:
        assert float((g1 - g2).abs().max()) <= 1e-4 * float(g2.abs().max()) + 1e-7


# ----------------------------------------------------------------------------------------------------------------- guard zones
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

    @property
    def ptr(self):
        return self.t.data_ptr()


@pytest.mark.gpu
@pytest.mark.parametrize("T", [226, 257, 300, 577, 1025])
@pytest.mark.parametrize("H,pol", [(1, True), (6, False), (6, True)])
def test_long_attention_train_stays_in_bounds(d2s, cuda_dev, T, H, pol):
    """Odd B, T with a nearly empty last tile: no write outside any output or the workspace, NaN behind every input never reaches a
    result, every output element is written (outputs and the workspace start as NaN), and out, cls_row, stats and dqkv are bitwise
    equal across two runs."""
    lib = d2s._lib
    B, D = 3, H * 64
    g = torch.Generator(device="cuda").manual_seed(9000 + T + H)
    qkv = _Guarded((B, T, 3 * D), torch.bfloat16, (torch.randn(B, T, 3 * D, device="cuda", generator=g) * 0.7).bfloat16(), poison_after=True)
    go = _Guarded((B, T, D), torch.bfloat16, (torch.randn(B, T, D, device="cuda", generator=g) * 0.5).bfloat16(), poison_after=True)
    gc = _Guarded((B, H, T), torch.float32, torch.randn(B, H, T, device="cuda", generator=g) * 0.5, poison_after=True)
    policy = _Guarded((B, T), torch.float32, _policy(B, T, g, "binary"), poison_after=True) if pol else None
    results = []
    for _ in range(2):
        out, cls, stats = _Guarded((B, T, D), torch.bfloat16), _Guarded((B, H, T), torch.float32), _Guarded((B, H, T, 4), torch.float32)
        dqkv, ws = _Guarded((B, T, 3 * D), torch.bfloat16), _Guarded((B, H, T, 64), torch.float32)
        gpol = _Guarded((B, T), torch.float32, torch.zeros(B, T, device="cuda")) if pol else None
        pp = policy.ptr if pol else None
        lib.call("d2s_attn_long_fwd_stats", qkv.ptr, pp, B, T, H, 64, 0.125, 1e-6, out.ptr, cls.ptr, stats.ptr, _stream())
        torch.cuda.synchronize()
        s_fwd = stats.t.clone()
        lib.call("d2s_attn_long_bwd", qkv.ptr, pp, out.ptr, go.ptr, cls.ptr, gc.ptr, stats.ptr, B, T, H, 64, 0.125, dqkv.ptr,
                 gpol.ptr if pol else None, ws.ptr, _stream())
        torch.cuda.synchronize()
        for name, gd in (("out", out), ("cls_row", cls), ("stats", stats), ("dqkv", dqkv), ("workspace", ws), ("gpolicy", gpol),
                         ("qkv", qkv), ("gout", go), ("g_cls", gc), ("policy", policy)):
            if gd is not None:
                assert gd.ok(), f"{name}: guard zone overwritten"
        for name, t in (("out", out.t), ("cls_row", cls.t), ("stats", s_fwd[..., :3]), ("delta", stats.t[..., 3]), ("dqkv", dqkv.t),
                        ("gpolicy", gpol.t if pol else None)):
            if t is not None:
                assert bool(torch.isfinite(t.float()).all()), f"{name}: element left unwritten or fed by an out-of-bounds read"
        results.append((out.t.clone(), cls.t.clone(), s_fwd, dqkv.t.clone()))
    for a, b in zip(*results):
        assert torch.equal(a, b)


# ----------------------------------------------------------------------------------------------------------------- models
def _seeded(d2s, m, seed):
    sd = fx.seeded_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, seed)
    m.load_state_dict({k: (v.bfloat16().float() if v.is_floating_point() else v) for k, v in sd.items()})
    return m


def _step(d2s, m, x, up):
    m.zero_grad()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = m(x)
    logits = out[0] if isinstance(out, tuple) else out
    (logits.float() * up).sum().backward()
    grads = {k: p.grad.detach().float().clone() for k, p in m.named_parameters() if p.grad is not None}
    return logits.detach().float(), out, grads


def _count_calls(d2s, monkeypatch):
    calls = {"n": 0}
    orig = d2s.ops._call

    def counting(name, *a):
        if name in ("d2s_attn_long_fwd_stats", "d2s_attn_long_bwd"):
            calls["n"] += 1
        return orig(name, *a)
    monkeypatch.setattr(d2s.ops, "_call", counting)
    return calls


def _compare(lf, gf, lp, gp):
    """The bound of test_training_fusions_match_the_unfused_training_path: logits and every parameter gradient within 5e-2 max + 1e-5."""
    assert float((lf - lp).abs().max()) <= 5e-2 * float(lp.abs().max()) + 1e-5
    assert gf.keys() == gp.keys()
    for k in gf:
        a, b = gf[k], gp[k]
        assert bool(torch.isfinite(a).all()), k
        assert float((a - b).abs().max()) <= 5e-2 * float(b.abs().max()) + 1e-5, k


KEEP_ALL = [576 / 196 + 1e-4]      # int(196 r) = 576: every token of a 384-px image stays (the reference counts from 196)


@pytest.mark.gpu
def test_variant_b_topk_training_at_384_pixels(d2s, cuda_dev, monkeypatch):
    """Variant B (top-k) at 384 px, bf16 autocast, forward + backward: blocks at T = 577 return CLS rows that carry a gradient (the
    stage scores from them).  The stage keeps every token, so no top-k cut can move with bf16 noise and the two paths differ only
    by their arithmetic: the long kernels against engine._LONG_ATTN = False (torch matmuls around the policy softmax), logits and
    every parameter gradient within 5e-2 max + 1e-5."""
    m = _seeded(d2s, d2s.variant_b.VisionTransformerDiffPruning(img_size=384, depth=3, pruning_loc=[1], token_ratio=KEEP_ALL, distill=True,
                                                                 topk_selection=True, predictor_loss_type="kl_div", num_classes=16,
                                                                 **DEIT_S_W), 301).to(cuda_dev).train()
    x = fx.randn(302, 2, 3, 384, 384).to(cuda_dev)
    up = fx.randn(303, 2, 16).to(cuda_dev)
    calls = _count_calls(d2s, monkeypatch)
    lf, _, gf = _step(d2s, m, x, up)
    assert calls["n"] >= 2
    monkeypatch.setattr(d2s.engine, "_LONG_ATTN", False)
    n = calls["n"]
    lp, _, gp = _step(d2s, m, x, up)
    assert calls["n"] == n
    _compare(lf, gf, lp, gp)


@pytest.mark.gpu
def test_variant_b_threshold_training_at_384_pixels(d2s, cuda_dev, monkeypatch):
    """Variant B in the dynamic keep-ratio (threshold) mode at 384 px: the blocks after the stage run with a keep policy over all
    577 tokens.  The cut on the cumulative score moves with bf16 noise of the scores, so keep decisions may differ at the cut:
    at most 2 % of the 576 tokens per image (the budget of test_gpu_long_attn.py's 384-px test).  Where the decisions agree, logits
    and gradients meet the bound of the top-k test; otherwise the two steps follow different policies and only finiteness is
    checked."""
    m = _seeded(d2s, d2s.variant_b.VisionTransformerDiffPruning(img_size=384, depth=3, pruning_loc=[1], token_ratio=[0.7], distill=True,
                                                                 topk_selection=True, predictor_loss_type="kl_div", num_classes=16,
                                                                 patch_score_threshold=0.3, **DEIT_S_W), 311).to(cuda_dev).train()
    x = fx.randn(312, 2, 3, 384, 384).to(cuda_dev)
    up = fx.randn(313, 2, 16).to(cuda_dev)
    calls = _count_calls(d2s, monkeypatch)
    lf, of, gf = _step(d2s, m, x, up)
    assert calls["n"] >= 2
    monkeypatch.setattr(d2s.engine, "_LONG_ATTN", False)
    lp, op, gp = _step(d2s, m, x, up)
    flips = (of[3] != op[3]).reshape(of[3].shape[0], -1).sum(1)
    assert bool((flips <= 0.02 * 576).all()), flips
    if int(flips.sum()) == 0:
        _compare(lf, gf, lp, gp)
    else:
        assert bool(torch.isfinite(lf).all()) and all(bool(torch.isfinite(v).all()) for v in gf.values())


@pytest.mark.gpu
def test_training_step_at_512_pixels(d2s, cuda_dev, monkeypatch):
    """A reduced-depth DeiT-S-width training step at 512 px (T = 1025), which had no bf16 path before: it runs, and the first
    block's attention gradient matches float64 autograd of the reference formula at the bounds of the kernel test."""
    m = _seeded(d2s, d2s.variant_a.DefaultVisionTransformerTeacher(img_size=512, depth=2, num_classes=16, **DEIT_S_W), 321)
    m = m.to(cuda_dev).train()
    x = fx.randn(322, 2, 3, 512, 512).to(cuda_dev)
    up = fx.randn(323, 2, 16).to(cuda_dev)
    seen = []
    orig = d2s.ops.attention_train

    def capture(qkv, H, **kw):
        o, c = orig(qkv, H, **kw)
        if not seen:
            qkv.retain_grad()
            o.retain_grad()
            seen.append((qkv, o, kw))
        return o, c
    monkeypatch.setattr(d2s.ops, "attention_train", capture)
    lf, _, gf = _step(d2s, m, x, up)
    assert seen and seen[0][0].shape[1] == 1025
    assert bool(torch.isfinite(lf).all()) and all(bool(torch.isfinite(v).all()) for v in gf.values())
    qkv, o, kw = seen[0]
    assert kw.get("policy") is None
    q2 = qkv.detach().double().requires_grad_(True)
    o2, _, _ = _ref(q2, 6)
    (o2 * o.grad.double()).sum().backward()
    torch.testing.assert_close(o.detach().double(), o2.detach(), rtol=2e-2, atol=2e-2)
    assert float((qkv.grad.double() - q2.grad).abs().max()) <= 3e-2 * float(q2.grad.abs().max()) + 1e-3


@pytest.mark.gpu
def test_graphed_training_step_at_384_pixels_matches_eager(d2s, cuda_dev):
    """runner.TrainStepRunner captures a 384-px training step (the long kernels inside the graph): the loss trajectory over a few
    AdamW steps equals the eager one."""
    base = _seeded(d2s, d2s.variant_a.DefaultVisionTransformerTeacher(img_size=384, depth=2, num_classes=16, **DEIT_S_W), 331)
    base = base.to(cuda_dev)
    x = fx.randn(332, 2, 3, 384, 384).to(cuda_dev)
    y = torch.tensor([1, 5], device=cuda_dev)
    losses = {}
    for mode in ("eager", "graph"):
        m = copy.deepcopy(base).train()
        opt = torch.optim.AdamW(m.parameters(), lr=1e-4, weight_decay=0.05, capturable=True)

        def fwd_loss(xx, yy, m=m):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = m(xx)
                logits = out[0] if isinstance(out, tuple) else out
                return torch.nn.functional.cross_entropy(logits.float(), yy)
        run = d2s.runner.TrainStepRunner(fwd_loss, opt, x, y, warmup=2, use_graph=mode != "eager")
        assert (run.graph is not None) == (mode != "eager")
        losses[mode] = [float(run()) for _ in range(4)]
    for a, b in zip(losses["eager"], losses["graph"]):
        assert abs(a - b) <= 2e-2 * abs(a) + 1e-3, losses
    assert losses["graph"][-1] != losses["graph"][0]          # the replays really update the weights
