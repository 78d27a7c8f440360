"""Operator layer: torch tensors in, hand-written sm_100a kernels underneath (via the C ABI in _lib.py).

Every function here enqueues on torch's current CUDA stream and allocates outputs through torch's
caching allocator; nothing synchronises with the host.  Inputs must be CUDA tensors -- there is no CPU
fallback (the CPU restatement lives in oracle/ and is test infrastructure only).
"""
import os
import weakref

import torch
import torch.nn.functional as F

from . import _lib
from ._lib import (ACT_GELU, ACT_NONE, ACT_RELU, BF16, F32, ORDER_INDEX_ASC, ORDER_SCORE_DESC, PROB_SIGMOID,  # noqa: F401
                   PROB_SOFTMAX)


def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"d2s kernels take float32 or bfloat16 tensors, got {t.dtype}")


def _copy_code(t: torch.Tensor) -> int:
    """dtype code for the pure copy kernels (gather / scatter): only the element size matters."""
    if t.element_size() == 2:
        return BF16
    if t.element_size() == 4:
        return F32
    raise TypeError(f"d2s gather/scatter kernels move 2- and 4-byte elements, got {t.dtype}")


def _as_kernel_float(t):
    """Tensors of other float types (fp16 under autocast) enter the fp32-math tail kernels as fp32."""
    return t if t.dtype in (torch.float32, torch.bfloat16) else t.float()


def _check_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("d2s ops run on CUDA tensors only (no CPU fallback)")


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(t):
    """(device, handle of torch's current stream ON THAT DEVICE) for the tensor a call works on."""
    return t.device, torch.cuda.current_stream(t.device).cuda_stream


def _call(name, *args):
    """One C-ABI call; the last argument comes from _stream(tensor).  The library launches (and sets function attributes, and
    encodes tensor maps) on the CURRENT device: when the tensors live on another one (model.to('cuda:1') without set_device)
    the call is made under a device guard, like torch's own ops."""
    dev, stream = args[-1]
    if dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):
            _lib.call(name, *args[:-1], stream)
    else:
        _lib.call(name, *args[:-1], stream)


def _f32c(t):
    return None if t is None else t.detach().to(torch.float32).contiguous()


# ----------------------------------------------------------------------------------------------
# (1) selection and fused predictor tails
# ----------------------------------------------------------------------------------------------

def select_topk(score: torch.Tensor, k: int, order: int = ORDER_INDEX_ASC, want_dropped: bool = True):
    """Stable top-k over (B,N) fp32 scores -> (kept (B,k) int64, dropped (B,N-k) int64 or None).
    Replaces argsort/sort at vit_models/dynamic_vit.py:858-862 and default_dynamic_vit.py:463."""
    _check_cuda(score)
    s = _f32c(score)
    B, N = s.shape
    if not 0 <= k <= N:
        raise RuntimeError(f"select_topk: K={k} outside [0, N={N}]")
    kept = torch.empty(B, k, dtype=torch.int64, device=s.device)
    dropped = torch.empty(B, N - k, dtype=torch.int64, device=s.device) if want_dropped else None
    _call("d2s_select_topk_f32", _ptr(s), B, N, k, order, _ptr(kept), _ptr(dropped), _stream(s))
    return kept, dropped


def _lengths(lengths, B, what):
    """Per-image valid lengths of a padded (B, n_max, ...) tensor as the int32 device vector the varlen kernels read."""
    _check_cuda(lengths)
    if lengths.dim() != 1 or lengths.shape[0] != B:
        raise ValueError(f"{what}: lengths must be a (B={B},) vector, got shape {tuple(lengths.shape)}")
    return lengths.to(torch.int32).contiguous()


def threshold_select(score, threshold, want_indices=False, lengths=None):
    """Dynamic keep-ratio selection (vit_models/dynamic_vit.py:880-890, :935-945): tokens whose cumulative ascending-sorted
    score mass exceeds `threshold` are kept.  score (B,N) -> (mask (B,N) bool, count (B) int32[, kept (B,N) int64: the kept
    indices in ascending order, then -1 padding]).
    lengths (B) int: image b selects among its first lengths[b] scores only (a padded batch); entries past it are never read,
    their mask is False and their kept entry -1."""
    _check_cuda(score)
    s = _f32c(score)
    B, N = s.shape
    mask = torch.empty(B, N, dtype=torch.bool, device=s.device)
    count = torch.empty(B, dtype=torch.int32, device=s.device)
    kept = torch.empty(B, N, dtype=torch.int64, device=s.device) if want_indices else None
    if lengths is None:
        _call("d2s_threshold_select_f32", _ptr(s), B, N, float(threshold), _ptr(mask), _ptr(count), _ptr(kept), _stream(s))
    else:
        n = _lengths(lengths, B, "threshold_select")
        _call("d2s_threshold_select_varlen_f32", _ptr(s), _ptr(n), B, N, float(threshold), _ptr(mask), _ptr(count), _ptr(kept),
              _stream(s))
    return (mask, count, kept) if want_indices else (mask, count)


def score_tail_b_varlen(hidden, lengths, ln_weight, ln_bias, weight, bias, ln_eps=1e-5, prob_mode=PROB_SOFTMAX):
    """score_tail_b without selection over a padded batch: image b's rows are hidden[b, :lengths[b]].  The softmax runs over
    those rows only; pad rows are never read, their scores are -inf and their probabilities 0.  Returns (scores, probs) (B,N)."""
    _check_cuda(hidden, weight)
    h = _as_kernel_float(hidden.detach()).contiguous()
    B, N, C = h.shape
    n = _lengths(lengths, B, "score_tail_b_varlen")
    lw, lb = _f32c(ln_weight), _f32c(ln_bias)
    w = _f32c(weight).reshape(-1)
    bz = _f32c(bias).reshape(-1) if bias is not None else None
    scores = torch.empty(B, N, dtype=torch.float32, device=h.device)
    probs = torch.empty(B, N, dtype=torch.float32, device=h.device)
    _call("d2s_score_tail_b_varlen", _ptr(h), _ptr(n), _dtype_code(h), B, N, C, _ptr(lw), _ptr(lb), float(ln_eps), _ptr(w),
          _ptr(bz), prob_mode, _ptr(scores), _ptr(probs), _stream(h))
    return scores, probs


def score_tail_a(hidden, weight, bias, k=0, gumbel=None, prev=None, act_input=ACT_NONE, want_prev_kept=False):
    """Variant A predictor tail (Linear(C,2)+LogSoftmax) fused with selection or the Gumbel decision.
    eval  (gumbel None): returns (logp (B,N,2), kept (B,k) int64 in descending-score order[, prev_kept (B,k) f32])
    train (gumbel (B,N,2)): returns (logp, decision (B,N), ysoft (B,N))
    act_input=ACT_GELU: `hidden` is the previous Linear's raw output, the GELU is applied on load."""
    _check_cuda(hidden, weight, bias)
    h = _as_kernel_float(hidden.detach()).contiguous()
    B, N, C = h.shape
    w, b = _f32c_param(weight), _f32c_param(bias)
    logp = torch.empty(B, N, 2, dtype=torch.float32, device=h.device)
    p = _f32c(prev.reshape(B, N)) if prev is not None else None
    if gumbel is None:
        kept = torch.empty(B, k, dtype=torch.int64, device=h.device)
        prev_kept = torch.empty(B, k, dtype=torch.float32, device=h.device) if want_prev_kept else None
        _call("d2s_score_tail_a", _ptr(h), _dtype_code(h), B, N, C, _ptr(w), _ptr(b), k, None, _ptr(p),
                  _ptr(logp), _ptr(kept), None, None, int(act_input), _ptr(prev_kept), _stream(h))
        return (logp, kept, prev_kept) if want_prev_kept else (logp, kept)
    g = _f32c(gumbel)
    decision = torch.empty(B, N, dtype=torch.float32, device=h.device)
    ysoft = torch.empty(B, N, dtype=torch.float32, device=h.device)
    _call("d2s_score_tail_a", _ptr(h), _dtype_code(h), B, N, C, _ptr(w), _ptr(b), 0, _ptr(g), _ptr(p),
              _ptr(logp), None, _ptr(decision), _ptr(ysoft), int(act_input), None, _stream(h))
    return logp, decision, ysoft


def score_tail_b(hidden, ln_weight, ln_bias, weight, bias, k, ln_eps=1e-5, prob_mode=PROB_SOFTMAX, select=True):
    """Variant B predictor tail ([LayerNorm]+Linear(C,1)+softmax|sigmoid) fused with the ascending-index
    top-k.  Returns (scores (B,N), probs (B,N), kept (B,k)|None, dropped (B,N-k)|None)."""
    _check_cuda(hidden, weight)
    h = _as_kernel_float(hidden.detach()).contiguous()
    B, N, C = h.shape
    lw, lb = _f32c(ln_weight), _f32c(ln_bias)
    w = _f32c(weight).reshape(-1)
    bz = _f32c(bias).reshape(-1) if bias is not None else None
    scores = torch.empty(B, N, dtype=torch.float32, device=h.device)
    probs = torch.empty(B, N, dtype=torch.float32, device=h.device)
    kept = torch.empty(B, k, dtype=torch.int64, device=h.device) if select else None
    dropped = torch.empty(B, N - k, dtype=torch.int64, device=h.device) if select else None
    _call("d2s_score_tail_b", _ptr(h), _dtype_code(h), B, N, C, _ptr(lw), _ptr(lb), float(ln_eps), _ptr(w),
              _ptr(bz), prob_mode, k, _ptr(scores), _ptr(probs), _ptr(kept), _ptr(dropped), _stream(h))
    return scores, probs, kept, dropped


class _GumbelKeep(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logp, gumbel, prev):
        lp, g = _f32c(logp), _f32c(gumbel)
        n = lp.numel() // 2
        pv = _f32c(prev.reshape(-1)) if prev is not None else None
        decision = torch.empty(lp.shape[:-1], dtype=torch.float32, device=lp.device)
        _call("d2s_gumbel_decision_f32", _ptr(lp), _ptr(g), _ptr(pv), n, _ptr(decision), None, _stream(lp))
        ctx.save_for_backward(lp, g, pv if pv is not None else torch.empty(0, device=lp.device))
        ctx.has_prev = pv is not None
        ctx.in_dtype = logp.dtype
        ctx.prev_meta = None if prev is None else (prev.shape, prev.dtype)
        return decision.unsqueeze(-1).to(logp.dtype)

    @staticmethod
    def backward(ctx, gout):
        lp, gm, pv = ctx.saved_tensors
        g = _f32c(gout.reshape(-1))
        n = lp.numel() // 2
        glogp = torch.empty_like(lp)
        want_gprev = ctx.has_prev and ctx.needs_input_grad[2]
        gprev = torch.empty(n, dtype=torch.float32, device=lp.device) if want_gprev else None
        _call("d2s_gumbel_decision_bwd_f32", _ptr(g), _ptr(lp), _ptr(gm), _ptr(pv) if ctx.has_prev else None, n,
                  _ptr(glogp), _ptr(gprev), _stream(g))
        if gprev is not None:
            gprev = gprev.reshape(ctx.prev_meta[0]).to(ctx.prev_meta[1])
        return glogp.to(ctx.in_dtype), None, gprev


def gumbel_keep_decision(logp, gumbel, prev=None):
    """hard keep decision (B,N,1) in {0,1} * prev with the straight-through gradient of
    F.gumbel_softmax(hard=True)[..., 0:1] (vit_models/default_dynamic_vit.py:454), noise injected."""
    _check_cuda(logp, gumbel)
    return _GumbelKeep.apply(logp, gumbel, prev)


# ----------------------------------------------------------------------------------------------
# (3) gather / scatter
# ----------------------------------------------------------------------------------------------

class _GatherTokens(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, idx, prepend_cls):
        xc = x.contiguous()
        ic = idx.contiguous()
        B, T, D = xc.shape
        K = ic.shape[1]
        out = torch.empty(B, K + (1 if prepend_cls else 0), D, dtype=xc.dtype, device=xc.device)
        _call("d2s_gather_tokens", _ptr(xc), _copy_code(xc), B, T, D, _ptr(ic), K, int(prepend_cls), _ptr(out), _stream(xc))
        ctx.save_for_backward(ic)
        ctx.shape = (B, T, D, K, bool(prepend_cls))
        return out

    @staticmethod
    def backward(ctx, gout):
        (ic,) = ctx.saved_tensors
        B, T, D, K, prepend_cls = ctx.shape
        g = gout.contiguous()
        gx = torch.empty(B, T, D, dtype=g.dtype, device=g.device)
        _call("d2s_scatter_tokens_bwd", _ptr(g), _copy_code(g), B, T, D, _ptr(ic), K, int(prepend_cls), _ptr(gx), _stream(g))
        return gx, None, None


_CHECK_INDICES = os.environ.get("D2S_CHECK_INDICES", "0") == "1"   # debug: validate gather indices (host sync)


def _validate_indices(kept, n):
    lo, hi = int(kept.min()), int(kept.max())
    if lo < 0 or hi >= n:
        raise IndexError(f"gather_tokens: index range [{lo}, {hi}] outside [0, {n})")
    srt = torch.sort(kept, dim=1).values
    if bool((srt[:, 1:] == srt[:, :-1]).any()):
        raise ValueError("gather_tokens: duplicate indices in a row (the backward keeps one gradient per source row)")


def gather_tokens(x, kept, prepend_cls=True):
    """x (B,T,D) with CLS at row 0, kept (B,K) spatial indices -> (B,K+1,D) = [CLS, x[kept+1]]
    (vit_models/dynamic_vit.py:907-912).  Differentiable in x (backward = scatter + zero fill).
    Contract: the indices of a row are UNIQUE and in range -- what every caller on the hot path passes (kept-token sets from
    the selection kernels).  The backward writes each source row once (no atomics), so with duplicates it would keep one of
    the gradients where torch.gather's backward sums them, and the forward clamps out-of-range indices where torch raises;
    D2S_CHECK_INDICES=1 validates both on every call (with a host synchronisation)."""
    _check_cuda(x, kept)
    if kept.dtype != torch.int64:
        raise TypeError("indices must be int64")
    if _CHECK_INDICES and kept.numel():
        _validate_indices(kept, x.shape[1] - (1 if prepend_cls else 0))
    return _GatherTokens.apply(x, kept, prepend_cls)


def scatter_tokens_bwd(gout, kept, t_in, prepend_cls=True):
    _check_cuda(gout, kept)
    g = gout.contiguous()
    B, _, D = g.shape
    gx = torch.empty(B, t_in, D, dtype=g.dtype, device=g.device)
    _call("d2s_scatter_tokens_bwd", _ptr(g), _copy_code(g), B, t_in, D, _ptr(kept.contiguous()), kept.shape[1],
              int(prepend_cls), _ptr(gx), _stream(g))
    return gx


def batch_index_select(x, idx):
    """Same contract as the reference's batch_index_select (vit_models/default_dynamic_vit.py:37-53)."""
    if x.dim() == 3:
        return gather_tokens(x, idx, prepend_cls=False)
    if x.dim() == 2:
        return gather_tokens(x.unsqueeze(-1), idx, prepend_cls=False).squeeze(-1)
    raise NotImplementedError


# ----------------------------------------------------------------------------------------------
# (2) PerturbedTopK
# ----------------------------------------------------------------------------------------------

class _PerturbedTopK(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, k, num_samples, sigma, noise, seed):
        xc = _f32c(x)
        B, N = xc.shape
        ind = torch.empty(B, k, N, dtype=torch.float32, device=xc.device)
        egrad = torch.empty(B, k, N, dtype=torch.float32, device=xc.device)
        if noise is not None:
            nz = _f32c(noise)
            if tuple(nz.shape) != (B, num_samples, N):
                raise ValueError(f"noise must be {(B, num_samples, N)}, got {tuple(nz.shape)}")
            _call("d2s_ptopk_fwd", _ptr(xc), _ptr(nz), B, N, k, num_samples, float(sigma), _ptr(ind), _ptr(egrad), _stream(xc))
        else:
            _call("d2s_ptopk_fwd_rng", _ptr(xc), int(seed), B, N, k, num_samples, float(sigma), _ptr(ind), _ptr(egrad), _stream(xc))
        ctx.save_for_backward(egrad)
        ctx.in_dtype = x.dtype
        return ind

    @staticmethod
    def backward(ctx, gout):
        (egrad,) = ctx.saved_tensors
        B, K, N = egrad.shape
        g = _f32c(gout)
        gx = torch.empty(B, N, dtype=torch.float32, device=g.device)
        _call("d2s_ptopk_bwd", _ptr(g), _ptr(egrad), B, N, K, _ptr(gx), _stream(g))
        return gx.to(ctx.in_dtype), None, None, None, None, None


def perturbed_topk(x, k, num_samples=500, sigma=0.05, noise=None, seed=None):
    """Differentiable top-k indicators (B,k,N) of vit_models/peturbed_topk.py.  `noise` (B,num_samples,N)
    reproduces the reference bit-for-bit given the same draws; with noise=None the kernel draws its own
    (Philox) from `seed` (default: a fresh seed from torch's generator)."""
    _check_cuda(x, noise)
    if noise is None and seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    return _PerturbedTopK.apply(x, int(k), int(num_samples), float(sigma), noise, seed)


# ----------------------------------------------------------------------------------------------
# (4) policy attention
# ----------------------------------------------------------------------------------------------

class _SoftmaxPolicy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, attn, policy, eps):
        a = attn.contiguous()
        B, H, T, _ = a.shape
        pol = _f32c(policy.reshape(B, T)) if policy is not None else None
        out = torch.empty_like(a)
        stats = torch.empty(B, H, T, 2, dtype=torch.float32, device=a.device)
        _call("d2s_softmax_policy_fwd", _ptr(a), _ptr(pol), _dtype_code(a), B, H, T, float(eps), _ptr(out), _ptr(stats), _stream(a))
        ctx.save_for_backward(a, stats, pol if pol is not None else torch.empty(0, device=a.device))
        ctx.meta = (B, H, T, float(eps), pol is not None, None if policy is None else (policy.shape, policy.dtype))
        return out

    @staticmethod
    def backward(ctx, gout):
        a, stats, pol = ctx.saved_tensors
        B, H, T, eps, has_pol, pol_meta = ctx.meta
        g = gout.contiguous().to(a.dtype)
        gattn = torch.empty_like(a)
        gpol = torch.zeros(B, T, dtype=torch.float32, device=a.device) if has_pol else None
        _call("d2s_softmax_policy_bwd", _ptr(a), _ptr(pol) if has_pol else None, _ptr(g), _ptr(stats), _dtype_code(a),
                  B, H, T, eps, _ptr(gattn), _ptr(gpol), _stream(a))
        if has_pol:
            gpol = gpol.reshape(pol_meta[0]).to(pol_meta[1])
        return gattn, gpol, None


def softmax_with_policy(attn, policy, eps=1e-6):
    """Drop-in for Attention.softmax_with_policy (vit_models/dynamic_vit.py:195-214): attn (B,H,T,T),
    policy (B,T,1) or None (plain softmax).  One kernel forward, one backward, differentiable in both."""
    _check_cuda(attn, policy)
    return _SoftmaxPolicy.apply(attn, policy, eps)


# Test hook: True in use; tests/test_gpu_models.py::test_training_fusions_match_the_unfused_training_path sets it to False to run
# linear_train on torch's own Linear, the reference it compares the fused training path against.
_FUSED_WGRAD = True   # ops.linear_train (d2s bias gradient)


def colsum(dy):
    """Column sums of a bf16 matrix (M,N) in fp32 (`d2s_colsum_bf16`): the bias gradient of a Linear layer."""
    _check_cuda(dy)
    if dy.dtype != torch.bfloat16 or dy.dim() != 2:
        raise RuntimeError("colsum: a 2-D bf16 tensor is expected")
    dy = dy.contiguous()
    if dy.shape[0] == 0:
        return torch.zeros(dy.shape[1], dtype=torch.float32, device=dy.device)
    out = torch.empty(dy.shape[1], dtype=torch.float32, device=dy.device)
    _call("d2s_colsum_bf16", _ptr(dy), dy.shape[0], dy.shape[1], _ptr(out), _stream(dy))
    return out


# ---- gradient slots: parameter gradients written where they live ------------------------------------------------
# autograd hands a parameter gradient to an AccumulateGrad node, which adds it into an existing .grad with one more elementwise
# launch per parameter (~200 launches, ~0.5 ms of a DeiT-S training step, plus a second pass over every weight gradient).  When
# the gradients live in a runner.FlatGrads buffer the training-path nodes below write them there directly -- dW as the output of
# the library GEMM, bias / LayerNorm gradients by kernels that accumulate into the slot -- and return None to autograd (the
# "main_grad" arrangement of large-model trainers).  A slot is fp32, zeroed once per step by FlatGrads.zero(), which also re-arms
# the "first write overwrites" flag of every slot; a parameter used twice in one backward accumulates on its second write.
_GRAD_SLOTS = {}          # id(parameter) -> [weakref(parameter), first_write_pending]


def register_grad_slots(params):
    import weakref
    for p in params:
        _GRAD_SLOTS[id(p)] = [weakref.ref(p), True]


def unregister_grad_slots(params):
    for p in params:
        _GRAD_SLOTS.pop(id(p), None)


def reset_grad_slots(params):
    for p in params:
        e = _GRAD_SLOTS.get(id(p))
        if e is not None:
            e[1] = True


def _grad_slot(p):
    """(slot tensor, entry) when `p`'s gradient is to be written in place, else (None, None)."""
    if p is None:
        return None, None
    e = _GRAD_SLOTS.get(id(p))
    if e is None or e[0]() is not p:
        return None, None
    g = p.grad
    if g is None or g.dtype != torch.float32 or not g.is_contiguous() or not g.is_cuda:
        return None, None
    return g, e


def _wgrad_into(p, dy, x, b_p=None):
    """dW = dy^T x landed in `p`'s gradient slot -- and, when `b_p` has a slot too, its bias gradient (column sums of dy) right
    behind it; returns (weight done, bias done).  False: the caller returns that gradient to autograd."""
    slot, e = _grad_slot(p)
    bslot, be = _grad_slot(b_p) if (b_p is not None and dy.shape[0] > 0) else (None, None)
    w_ok = slot is not None and _MM_OUT
    if not w_ok and bslot is None:
        return False, False
    if w_ok:
        if e[1]:
            torch.mm(dy.t(), x, out_dtype=torch.float32, out=slot)
            e[1] = False
        else:
            slot.add_(torch.mm(dy.t(), x, out_dtype=torch.float32))
    if bslot is not None:
        _call("d2s_colsum_acc_bf16", _ptr(dy), dy.shape[0], dy.shape[1], _ptr(bslot), _stream(dy))
        be[1] = False
    return w_ok, bslot is not None


def adamw_flat(p, g, m, v, shadow, begin, end, lr, step, beta1, beta2, eps, weight_decay, grad_scale=1.0):
    """One AdamW update of elements [begin, end) of the flat fp32 buffers (p, g, m, v) (`d2s_adamw_flat_f32`): lr and step are
    1-element fp32 CUDA tensors; shadow (bf16, same layout) or None receives the updated parameters."""
    _check_cuda(p, g, m, v, lr, step)
    for t in (p, g, m, v, lr, step):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise TypeError("adamw_flat: contiguous fp32 tensors are expected")
    if not (p.numel() == g.numel() == m.numel() == v.numel()) or not 0 <= begin <= end <= p.numel():
        raise RuntimeError("adamw_flat: the flat buffers must have one size and [begin, end) must lie inside it")
    if shadow is not None and (shadow.dtype != torch.bfloat16 or shadow.numel() != p.numel() or not shadow.is_contiguous()):
        raise TypeError("adamw_flat: shadow must be a contiguous bf16 tensor of the parameters' size")
    if begin == end:
        return
    _call("d2s_adamw_flat_f32", _ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(shadow), int(begin), int(end), _ptr(lr), _ptr(step),
          float(beta1), float(beta2), float(eps), float(weight_decay), float(grad_scale), _stream(p))


class BF16WeightCache:
    """bf16 copies of a model's fp32 master parameters, refreshed ONCE per step by one multi-tensor copy instead of one cast
    kernel per Linear weight and bias per forward (141 launches, 0.5 ms of a DeiT-S training step).  The training-path Linear
    ops (linear_train / linear_gelu_train) pick the copy up when one is registered for the parameter; whoever owns the step
    (runner.TrainStepRunner) calls refresh() after every optimizer update -- between refreshes the copies are what the forward
    sees, so a refresh must follow every change of the master weights."""

    _active = {}          # id(parameter) -> bf16 copy

    def __init__(self, params, copies=None):
        """copies: bf16 tensors somebody else keeps current (runner.FlatAdamW's kernel writes them with the update), one per
        parameter; refresh() is then a no-op."""
        params = list(params)
        if copies is not None:
            self.src, self.dst, self.external = params, list(copies), True
        else:
            self.src = [p for p in params if p.dtype == torch.float32 and p.is_cuda]
            self.dst = [torch.empty_like(p, dtype=torch.bfloat16) for p in self.src]
            self.external = False
        for p, d in zip(self.src, self.dst):
            BF16WeightCache._active[id(p)] = (p, d)
        self.refresh()

    def refresh(self):
        if self.external:
            return
        with torch.no_grad():
            torch._foreach_copy_(self.dst, self.src)

    def close(self):
        for p in self.src:
            BF16WeightCache._active.pop(id(p), None)

    @staticmethod
    def lookup(p):
        hit = BF16WeightCache._active.get(id(p))
        return hit[1] if hit is not None and hit[0] is p else None


def _bf16_of(p):
    """The bf16 form of a Linear weight / bias for the forward: the per-step cached copy when one is registered, else a cast."""
    if p is None:
        return None
    c = BF16WeightCache.lookup(p)
    return c if c is not None else p.to(torch.bfloat16)


def _wgrad(dy, x, dtype):
    """dW = dy^T x for bf16 (M,N) x (M,K) operands in the parameter's dtype: with fp32 master weights the library GEMM writes
    its fp32 accumulator out directly (no bf16 rounding of the weight gradient, no separate cast pass)."""
    if dtype == torch.float32 and _MM_OUT_DTYPE:
        return torch.mm(dy.t(), x, out_dtype=torch.float32)
    return (dy.t() @ x).to(dtype)


def _probe_mm_out_dtype():
    try:
        torch.mm(torch.zeros(8, 8, dtype=torch.bfloat16, device="meta"), torch.zeros(8, 8, dtype=torch.bfloat16, device="meta"),
                 out_dtype=torch.float32)
        return True
    except (TypeError, RuntimeError, NotImplementedError):
        return False


_MM_OUT_DTYPE = _probe_mm_out_dtype()


def _probe_mm_out():
    try:
        a = torch.zeros(8, 8, dtype=torch.bfloat16, device="meta")
        torch.mm(a, a, out_dtype=torch.float32, out=torch.zeros(8, 8, dtype=torch.float32, device="meta"))
        return True
    except (TypeError, RuntimeError, NotImplementedError):
        return False


_MM_OUT = _MM_OUT_DTYPE and _probe_mm_out()


class _LinearTrain(torch.autograd.Function):
    """nn.Linear on the bf16 training path (fp32 master weights under bf16 autocast, or a bf16 module).  Forward is the library
    GEMM torch would run on the bf16 casts; backward computes dx and dW with library GEMMs and the bias gradient with the d2s
    column-sum kernel in fp32 -- torch.autograd's own column reduction of dy (61 launches, 3.7 ms of a 34 ms DeiT-S step) and the bf16 -> fp32 round trip of
    the bias gradient disappear."""

    @staticmethod
    def forward(ctx, x, w, b):
        xb, wb = x.to(torch.bfloat16), _bf16_of(w)
        bb = _bf16_of(b)
        ctx.save_for_backward(xb, wb)
        ctx.meta = (x.dtype, w.dtype, None if b is None else b.dtype)
        ctx.params = (w, b)
        return F.linear(xb, wb, bb)

    @staticmethod
    def backward(ctx, gy):
        xb, wb = ctx.saved_tensors
        xd, wd, bd = ctx.meta
        N, K = wb.shape
        gy2 = gy.reshape(-1, N)
        if gy2.dtype != torch.bfloat16 or not gy2.is_contiguous():
            gy2 = gy2.to(torch.bfloat16).contiguous()
        gx = (gy2 @ wb).view(xb.shape).to(xd) if ctx.needs_input_grad[0] else None
        gw = gb = None
        want_b = bd is not None and ctx.needs_input_grad[2]
        w_p, b_p = ctx.params
        w_done, b_done = _wgrad_into(w_p if ctx.needs_input_grad[1] else None, gy2, xb.reshape(-1, K), b_p if want_b else None)
        if ctx.needs_input_grad[1] and not w_done:
            gw = _wgrad(gy2, xb.reshape(-1, K), wd)
        if want_b and not b_done:
            gb = colsum(gy2)
        return gx, gw, None if gb is None else gb.to(bd)


def gelu_bwd_colsum(u, ga, want_bias=True, db_into=None):
    """(du, db) = (ga * gelu'(u), column sums of du in fp32) for 2-D bf16 u, ga: the exact-erf GELU backward fused with the bias
    gradient of the Linear that produced u (`d2s_gelu_bwd_colsum_bf16`)."""
    _check_cuda(u, ga)
    if u.dtype != torch.bfloat16 or ga.dtype != torch.bfloat16 or u.dim() != 2 or u.shape != ga.shape:
        raise RuntimeError("gelu_bwd_colsum: two 2-D bf16 tensors of one shape are expected")
    u, ga = u.contiguous(), ga.contiguous()
    M, N = u.shape
    du = torch.empty_like(u)
    if db_into is not None:           # an fp32 (N,) gradient slot: accumulated into, nothing returned for it
        if M > 0:
            _call("d2s_gelu_bwd_colsum_acc_bf16", _ptr(u), _ptr(ga), M, N, _ptr(du), _ptr(db_into), _stream(u))
        return du, None
    db = torch.zeros(N, dtype=torch.float32, device=u.device) if want_bias else None
    if M > 0:
        _call("d2s_gelu_bwd_colsum_bf16", _ptr(u), _ptr(ga), M, N, _ptr(du), _ptr(db), _stream(u))
    return du, db


class _LinearGeluTrain(torch.autograd.Function):
    """GELU(nn.Linear(x)) on the bf16 training path (Mlp.forward's fc1 -> act, dynamic_vit.py:170-172) as ONE autograd node: the
    backward runs GELU' and the Linear's bias gradient in one pass over (u, dy) and then the two library GEMMs for dx and dW."""

    @staticmethod
    def forward(ctx, x, w, b):
        xb, wb = x.to(torch.bfloat16), _bf16_of(w)
        bb = _bf16_of(b)
        if wb.shape[0] % 256 == 0 and wb.shape[0] <= 4096 and wb.shape[1] % 64 == 0:
            # one tcgen05 GEMM writes both the Linear's output (kept for GELU') and its GELU: torch's separate GELU pass
            # (read + write of the (M, 4D) hidden tensor) disappears
            a, u = linear_act(xb, wb, bb, ACT_GELU, want_pre=True)
        else:
            u = F.linear(xb, wb, bb)
            a = F.gelu(u)
        ctx.save_for_backward(xb, wb, u)
        ctx.meta = (x.dtype, w.dtype, None if b is None else b.dtype)
        ctx.params = (w, b)
        return a

    @staticmethod
    def backward(ctx, ga):
        xb, wb, u = ctx.saved_tensors
        xd, wd, bd = ctx.meta
        N, K = wb.shape
        ga2 = ga.reshape(-1, N)
        if ga2.dtype != torch.bfloat16 or not ga2.is_contiguous():
            ga2 = ga2.to(torch.bfloat16).contiguous()
        want_b = bd is not None and ctx.needs_input_grad[2]
        w_p, b_p = ctx.params
        slot, e = _grad_slot(b_p) if want_b else (None, None)
        du, gb = gelu_bwd_colsum(u.reshape(-1, N), ga2, want_bias=want_b, db_into=slot)
        if e is not None:
            e[1] = False
        gx = (du @ wb).view(xb.shape).to(xd) if ctx.needs_input_grad[0] else None
        gw = None
        if ctx.needs_input_grad[1] and not _wgrad_into(w_p, du, xb.reshape(-1, K))[0]:
            gw = _wgrad(du, xb.reshape(-1, K), wd)
        return gx, gw, None if gb is None else gb.to(bd)


def _linear_train_ok(lin, x):
    bf16 = (torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16) or \
        (x.dtype == torch.bfloat16 and lin.weight.dtype == torch.bfloat16)
    return (_FUSED_WGRAD and isinstance(lin, torch.nn.Linear) and x.is_cuda and bf16 and torch.is_grad_enabled()
            and lin.weight.requires_grad and lin.in_features % 8 == 0 and lin.out_features % 8 == 0
            and x.dtype in (torch.bfloat16, torch.float32))


def linear_gelu_train(lin, act, x):
    """`act(lin(x))` under autograd: one node with the fused GELU-backward + bias-gradient kernel when `act` is the exact-erf
    nn.GELU and the bf16 training path applies, else `act(linear_train(lin, x))`."""
    if (_linear_train_ok(lin, x) and isinstance(act, torch.nn.GELU)
            and getattr(act, "approximate", "none") == "none" and lin.out_features <= 8192):
        return _LinearGeluTrain.apply(x, lin.weight, lin.bias)
    return act(linear_train(lin, x))


def linear_train(lin, x):
    """`lin(x)` for an nn.Linear under autograd: the fused-bias-gradient path when it applies (CUDA, bf16 compute -- a bf16
    module or bf16 autocast --, feature counts multiples of 8), else the module itself."""
    if _linear_train_ok(lin, x):
        return _LinearTrain.apply(x, lin.weight, lin.bias)
    return lin(x)


class _AttentionTrain(torch.autograd.Function):
    """Training attention on the packed qkv tensor, differentiable in qkv and in the keep policy.

    One d2s relayout pass turns the packed (B,T,3,H,hd) tensor into head-major (3,B,H,Tp,hd) with Tp = round_up(T, 8) zero
    padded, so that the six batched GEMMs of forward + backward run over B*H matrices whose every dimension and leading
    dimension is a multiple of 8 (T = 197 otherwise sends cuBLAS to unaligned legacy kernels and torch to permute copies),
    and the d2s policy-softmax kernels move 16-byte vectors.  dq/dk/dv are merged straight into the packed qkv gradient
    (no cat).  Saves q/k/v head-major, the scaled scores, the probabilities and the (row max, denominator) pairs."""

    @staticmethod
    def forward(ctx, qkv, policy, H, scale, eps, want_cls):
        qkv = qkv.contiguous()
        B, T, C3 = qkv.shape
        D = C3 // 3
        hd = D // H
        Tp = (T + 7) // 8 * 8
        dev, dt = qkv.device, qkv.dtype
        qkvh = torch.empty(3, B * H, Tp, hd, dtype=dt, device=dev)
        _call("d2s_split_heads_bf16", _ptr(qkv), B, T, Tp, 3, H, hd, _ptr(qkvh), _stream(qkv))
        S = torch.empty(B * H, Tp, Tp, dtype=dt, device=dev)
        torch.baddbmm(S, qkvh[0], qkvh[1].transpose(1, 2), beta=0, alpha=scale, out=S)
        pol = _f32c(policy.reshape(B, T)) if policy is not None else None
        P = torch.empty_like(S)
        stats = torch.empty(B, H, T, 2, dtype=torch.float32, device=dev)
        _call("d2s_softmax_policy_fwd_ld", _ptr(S), _ptr(pol), B, H, T, Tp, Tp, float(eps), _ptr(P), _ptr(stats), _stream(S))
        Oh = torch.bmm(P, qkvh[2])                                                    # (B*H, Tp, hd)
        O = torch.empty(B, T, D, dtype=dt, device=dev)
        _call("d2s_merge_heads_bf16", _ptr(Oh), B, T, Tp, 1, H, hd, _ptr(O), _stream(Oh))
        cls_attn = P.view(B, H, Tp, Tp)[:, :, 0, :T].clone() if want_cls else None
        ctx.save_for_backward(qkvh, S, P, stats, pol if pol is not None else torch.empty(0, device=dev))
        ctx.meta = (B, T, Tp, H, hd, float(scale), float(eps), pol is not None,
                    None if policy is None else (policy.shape, policy.dtype))
        return O, cls_attn

    @staticmethod
    def backward(ctx, gO, g_cls):
        qkvh, S, P, stats, pol = ctx.saved_tensors
        B, T, Tp, H, hd, scale, eps, has_pol, pol_meta = ctx.meta
        polp = pol if has_pol else None
        dev, dt = S.device, S.dtype
        g = gO.to(dt).contiguous()
        gOh = torch.empty(B * H, Tp, hd, dtype=dt, device=dev)
        _call("d2s_split_heads_bf16", _ptr(g), B, T, Tp, 1, H, hd, _ptr(gOh), _stream(g))
        dqkvh = torch.empty(3, B * H, Tp, hd, dtype=dt, device=dev)
        torch.bmm(P.transpose(1, 2), gOh, out=dqkvh[2])                               # dV = P^T dO
        dP = torch.bmm(gOh, qkvh[2].transpose(1, 2))                                  # dP = dO V^T  (padding rows are zero)
        if g_cls is not None:
            dP.view(B, H, Tp, Tp)[:, :, 0, :T] += g_cls.to(dt)
        gpol = torch.zeros(B, T, dtype=torch.float32, device=dev) if has_pol else None
        _call("d2s_softmax_policy_bwd_ld", _ptr(S), _ptr(polp), _ptr(dP), _ptr(stats), B, H, T, Tp, Tp, eps, _ptr(dP),
                  _ptr(gpol), _stream(S))
        torch.baddbmm(dqkvh[0], dP, qkvh[1], beta=0, alpha=scale, out=dqkvh[0])                    # dQ = scale dS K
        torch.baddbmm(dqkvh[1], dP.transpose(1, 2), qkvh[0], beta=0, alpha=scale, out=dqkvh[1])    # dK = scale dS^T Q
        dqkv = torch.empty(B, T, 3 * H * hd, dtype=dt, device=dev)
        _call("d2s_merge_heads_bf16", _ptr(dqkvh), B, T, Tp, 3, H, hd, _ptr(dqkv), _stream(dqkvh))
        if has_pol:
            gpol = gpol.reshape(pol_meta[0]).to(pol_meta[1])
        return dqkv, gpol, None, None, None, None


class _AttentionFlash(torch.autograd.Function):
    """Training attention as two tcgen05 kernels on the packed qkv tensor, differentiable in qkv and in the keep policy:
    forward = the inference kernel, which also writes per-row softmax statistics (`d2s_attn_policy_fwd` with `stats`);
    backward = `d2s_attn_policy_bwd`, which recomputes scores and probabilities on chip.  Saves qkv, the output and
    (B,H,T,4) floats; no (B,H,T,T) tensor, no head-major copies, no library GEMM."""

    @staticmethod
    def forward(ctx, qkv, policy, H, scale, eps, want_cls):
        qkv = qkv.contiguous()
        B, T, C3 = qkv.shape
        D = C3 // 3
        dev = qkv.device
        pol = _f32c(policy.reshape(B, T)) if policy is not None else None
        out = torch.empty(B, T, D, dtype=qkv.dtype, device=dev)
        cls_row = torch.empty(B, H, T, dtype=torch.float32, device=dev) if want_cls else None
        stats = torch.empty(B, H, T, 4, dtype=torch.float32, device=dev)
        _call("d2s_attn_policy_fwd", _ptr(qkv), _ptr(pol), BF16, B, T, H, D // H, float(scale), float(eps), _ptr(out),
                  _ptr(cls_row), _ptr(stats), _stream(qkv))
        none = torch.empty(0, device=dev)
        ctx.save_for_backward(qkv, out, stats, pol if pol is not None else none, cls_row if want_cls else none)
        ctx.meta = (B, T, H, D // H, float(scale), pol is not None, want_cls,
                    None if policy is None else (policy.shape, policy.dtype))
        return out, (cls_row.to(qkv.dtype) if want_cls else None)

    @staticmethod
    def backward(ctx, gO, g_cls):
        qkv, out, stats, pol, cls_row = ctx.saved_tensors
        B, T, H, hd, scale, has_pol, want_cls, pol_meta = ctx.meta
        g = gO.to(qkv.dtype).contiguous()
        gc = _f32c(g_cls) if (want_cls and g_cls is not None) else None
        dqkv = torch.empty_like(qkv)
        gpol = torch.zeros(B, T, dtype=torch.float32, device=qkv.device) if has_pol else None
        _call("d2s_attn_policy_bwd", _ptr(qkv), _ptr(pol) if has_pol else None, _ptr(out), _ptr(g),
                  _ptr(cls_row) if want_cls else None, _ptr(gc), _ptr(stats), B, T, H, hd, scale, _ptr(dqkv), _ptr(gpol), _stream(qkv))
        if has_pol:
            gpol = gpol.reshape(pol_meta[0]).to(pol_meta[1])
        return dqkv, gpol, None, None, None, None


FLASH_MAX_T = 208


def attention_train(qkv, num_heads, policy=None, scale=None, eps=1e-6, want_cls_row=False):
    """Differentiable attention core of Attention.forward (vit_models/dynamic_vit.py:216-231) on the packed qkv (B,T,3*H*hd):
    returns (out (B,T,H*hd), cls_row (B,H,T) | None).  bf16 CUDA tensors, T <= 256.  hd == 64 and T <= 208 (every DeiT shape
    at 224 px) run the tcgen05 flash kernels; the rest keeps the head-major GEMMs around the padded-row softmax kernels."""
    _check_cuda(qkv, policy)
    if qkv.dtype != torch.bfloat16 or qkv.shape[1] > 256:
        raise RuntimeError("attention_train: bf16 and T <= 256 only (other cases use softmax_with_policy around torch matmuls)")
    hd = qkv.shape[-1] // 3 // num_heads
    scale = hd ** -0.5 if scale is None else scale
    if hd == 64 and qkv.shape[1] <= FLASH_MAX_T and scale > 0:
        return _AttentionFlash.apply(qkv, policy, num_heads, float(scale), float(eps), bool(want_cls_row))
    return _AttentionTrain.apply(qkv, policy, num_heads, float(scale), float(eps), bool(want_cls_row))


def attention_core(qkv, num_heads, policy=None, scale=None, eps=1e-6, want_cls_row=False, lengths=None):
    """Fused inference attention: packed qkv (B,T,3*H*hd) straight from the qkv Linear -> (out (B,T,H*hd),
    cls_row (B,H,T) fp32 | None).  bf16 runs the tcgen05/TMEM kernel, fp32 the SIMT parity kernel.
    No autograd: the training path uses softmax_with_policy around library GEMMs.
    lengths (B) int: a padded batch, image b is its first lengths[b] tokens (keys and queries); out rows and cls_row columns
    past it are zeros.  No policy in that form.
    bf16 inputs with T > 256 run the key-blocked kernel of attention_long."""
    _check_cuda(qkv, policy)
    if qkv.dtype == torch.bfloat16 and qkv.shape[1] > LONG_ATTN_MIN_T:
        return attention_long(qkv, num_heads, policy=policy, scale=scale, eps=eps, want_cls_row=want_cls_row, lengths=lengths)
    q = qkv.detach().contiguous()
    B, T, C3 = q.shape
    D = C3 // 3
    hd = D // num_heads
    scale = hd ** -0.5 if scale is None else scale
    out = torch.empty(B, T, D, dtype=q.dtype, device=q.device)
    cls_row = torch.empty(B, num_heads, T, dtype=torch.float32, device=q.device) if want_cls_row else None
    if lengths is not None:
        if policy is not None:
            raise ValueError("attention_core: the variable-length form takes no policy")
        n = _lengths(lengths, B, "attention_core")
        _call("d2s_attn_varlen_fwd", _ptr(q), _ptr(n), _dtype_code(q), B, T, num_heads, hd, float(scale), _ptr(out), _ptr(cls_row),
              _stream(q))
        return out, cls_row
    pol = _f32c(policy.reshape(B, T)) if policy is not None else None
    _call("d2s_attn_policy_fwd", _ptr(q), _ptr(pol), _dtype_code(q), B, T, num_heads, hd, float(scale), float(eps),
              _ptr(out), _ptr(cls_row), None, _stream(q))
    return out, cls_row


LONG_ATTN_MIN_T = 256     # attention_core hands bf16 sequences longer than this to attention_long
LONG_ATTN_MAX_T = 2048


def attention_long(qkv, num_heads, policy=None, scale=None, eps=1e-6, want_cls_row=False, lengths=None):
    """Fused inference attention for any 1 <= T <= 2048 (384 / 512-pixel inputs): the key-blocked tcgen05 kernel
    (d2s_attn_long_fwd), with the semantics of attention_core -- policy softmax (vit_models/dynamic_vit.py:195-214), CLS row,
    and the variable-length form (lengths (B) int, no policy).  bf16 packed qkv (B,T,3*H*64) -> (out (B,T,H*64) bf16,
    cls_row (B,H,T) fp32 | None).  No autograd."""
    _check_cuda(qkv, policy)
    if qkv.dtype != torch.bfloat16:
        raise TypeError(f"attention_long: bf16 qkv only, got {qkv.dtype}")
    q = qkv.detach().contiguous()
    B, T, C3 = q.shape
    D = C3 // 3
    hd = D // num_heads
    scale = hd ** -0.5 if scale is None else scale
    if lengths is not None and policy is not None:
        raise ValueError("attention_long: the variable-length form takes no policy")
    out = torch.empty(B, T, D, dtype=q.dtype, device=q.device)
    cls_row = torch.empty(B, num_heads, T, dtype=torch.float32, device=q.device) if want_cls_row else None
    n = _lengths(lengths, B, "attention_long") if lengths is not None else None
    pol = _f32c(policy.reshape(B, T)) if policy is not None else None
    _call("d2s_attn_long_fwd", _ptr(q), _ptr(pol), _ptr(n), B, T, num_heads, hd, float(scale), float(eps), _ptr(out),
          _ptr(cls_row), _stream(q))
    return out, cls_row


# ----------------------------------------------------------------------------------------------
# residual add + LayerNorm (inference path of Block.forward and of the predictors' leading LayerNorm)
# ----------------------------------------------------------------------------------------------

def add_layernorm(x, y, weight, bias, eps, norm_row0=0, want_sum=True):
    """s = x + y (y may be None); returns (s or None, LayerNorm(s[:, norm_row0:]) * weight + bias).
    x (B,T,D) may be a strided view with contiguous rows (e.g. a token slice); y contiguous.  No autograd:
    training keeps torch's add + LayerNorm (vit_models/dynamic_vit.py:263-283)."""
    _check_cuda(x, y, weight, bias)
    if x.stride(-1) != 1:
        x = x.contiguous()
    B, T, D = x.shape
    yc = None if y is None else y.detach().contiguous()
    w = weight.detach().to(x.dtype).contiguous()
    b = bias.detach().to(x.dtype).contiguous()
    need_sum = want_sum and (y is not None)
    out_sum = torch.empty(B, T, D, dtype=x.dtype, device=x.device) if need_sum else None
    out_norm = torch.empty(B, T - norm_row0, D, dtype=x.dtype, device=x.device)
    _call("d2s_add_layernorm", _ptr(x), _ptr(yc), _ptr(w), _ptr(b), _dtype_code(x), B, T, D, x.stride(0), x.stride(1),
              float(eps), int(norm_row0), _ptr(out_sum), _ptr(out_norm), _stream(x))
    if want_sum and y is None:
        out_sum = x
    return out_sum, out_norm


def layernorm_from_stats(x, stats, weight, bias, rows_per_image=1):
    """LayerNorm of the first `rows_per_image` rows of every image of x (B,T,D) bf16 from GIVEN per-row (mean, rstd) (stats (B*T, 2)
    f32, as the producers of x write them), with the arithmetic of the GEMM kernels' on-the-fly normalisation.  (B, rows, D)."""
    _check_cuda(x, stats, weight, bias)
    B, T, D = x.shape
    if x.dtype != torch.bfloat16 or rows_per_image != 1 or not x.is_contiguous():
        raise RuntimeError("layernorm_from_stats: contiguous bf16 (B,T,D) input, first row of every image")
    st = stats.detach().contiguous()
    w, b = weight.detach().to(torch.bfloat16).contiguous(), bias.detach().to(torch.bfloat16).contiguous()
    out = torch.empty(B, 1, D, dtype=x.dtype, device=x.device)
    _call("d2s_apply_layernorm_stats_bf16", _ptr(x.detach()), _ptr(st), _ptr(w), _ptr(b), B, D, T * D, T, _ptr(out), _stream(x))
    return out


def gather_layernorm(x, kept, weight, bias, eps, want_stats=False, counts=None):
    """(xg, LayerNorm(xg)) with xg = [CLS, x[:, kept + 1]]: the kept-token gather of the pruning stage fused with the next
    block's norm1 (vit_models/default_dynamic_vit.py:464-468, dynamic_vit.py:907-912 + :263).  Inference only.
    want_stats (bf16): (xg, stats (B*(K+1), 2) f32 = per-row (mean, rstd)) instead; the consumer applies the LayerNorm.
    counts (B) int: a variable-length gather, image b keeps kept[b, :counts[b]] (the rest of the row is padding, never read);
    output rows 1 + counts[b] .. K are zeros (both outputs), their stats those of a zero row."""
    _check_cuda(x, kept, weight, bias, counts)
    if kept.dtype != torch.int64:
        raise TypeError("indices must be int64")
    xc, ic = x.detach().contiguous(), kept.contiguous()
    B, T, D = xc.shape
    K = ic.shape[1]
    n = None if counts is None else _lengths(counts, B, "gather_layernorm")
    if want_stats:
        if xc.dtype != torch.bfloat16:
            raise TypeError("gather_layernorm(want_stats=True) is a bf16 path")
        out_sum = torch.empty(B, K + 1, D, dtype=xc.dtype, device=xc.device)
        stats = torch.empty(B * (K + 1), 2, dtype=torch.float32, device=xc.device)
        if B and n is None:
            _call("d2s_gather_layernorm_stats", _ptr(xc), _ptr(ic), B, T, D, K, float(eps), _ptr(out_sum), _ptr(stats), _stream(xc))
        elif B:
            _call("d2s_gather_layernorm_stats_varlen", _ptr(xc), _ptr(ic), _ptr(n), B, T, D, K, float(eps), _ptr(out_sum), _ptr(stats),
                  _stream(xc))
        return out_sum, stats
    w, b = weight.detach().to(xc.dtype).contiguous(), bias.detach().to(xc.dtype).contiguous()
    out_sum = torch.empty(B, K + 1, D, dtype=xc.dtype, device=xc.device)
    out_norm = torch.empty_like(out_sum)
    if n is None:
        _call("d2s_gather_layernorm", _ptr(xc), _ptr(ic), _ptr(w), _ptr(b), _dtype_code(xc), B, T, D, K, float(eps),
              _ptr(out_sum), _ptr(out_norm), _stream(xc))
    else:
        _call("d2s_gather_layernorm_varlen", _ptr(xc), _ptr(ic), _ptr(n), _ptr(w), _ptr(b), _dtype_code(xc), B, T, D, K, float(eps),
              _ptr(out_sum), _ptr(out_norm), _stream(xc))
    return out_sum, out_norm


# ----------------------------------------------------------------------------------------------
# predictor body (inference)
# ----------------------------------------------------------------------------------------------

def pool_act(z, policy=None, act=ACT_GELU, want_local=True):
    """z (B,N,C) -> (local (B,N,C/2) = act(z[..., :C/2]), pooled (B,C/2) = policy-weighted mean over tokens of
    act(z[..., C/2:])) in one pass (vit_models/default_dynamic_vit.py:325-328; dynamic_vit.py:538-542).
    want_local=False: (None, pooled) -- z is already activated and its local half is consumed in place by the next kernel."""
    _check_cuda(z, policy)
    zd = z.detach()
    B, N, C = zd.shape
    if (not want_local and zd.dtype == torch.bfloat16 and not zd.is_contiguous() and B > 1 and N > 1 and zd.stride(2) == 1
            and zd.stride(1) == C and zd.stride(0) >= N * C and zd.stride(0) % 8 == 0 and zd.data_ptr() % 16 == 0 and C % 16 == 0):
        # a row slice of a wider tensor (x[:, 1:]): pooled in place through the batch stride
        pol = _f32c(policy.reshape(B, N)) if policy is not None else None
        pooled = torch.empty(B, C // 2, dtype=zd.dtype, device=zd.device)
        _call("d2s_pool_strided_bf16", _ptr(zd), _ptr(pol), B, N, C, zd.stride(0), int(act), _ptr(pooled), _stream(zd))
        return None, pooled
    zc = zd.contiguous()
    pol = _f32c(policy.reshape(B, N)) if policy is not None else None
    local = torch.empty(B, N, C // 2, dtype=zc.dtype, device=zc.device) if want_local else None
    pooled = torch.empty(B, C // 2, dtype=zc.dtype, device=zc.device)
    _call("d2s_pool_act", _ptr(zc), _ptr(pol), _dtype_code(zc), B, N, C, int(act), _ptr(local), _ptr(pooled), _stream(zc))
    return local, pooled


def bias_act_(u, bias, act=ACT_GELU):
    """In place: u (..., N, C) = act(u + bias) with a per-image bias (B,C) broadcast over tokens, a shared bias (C,),
    or no bias (None)."""
    _check_cuda(u, bias)
    if not u.is_contiguous():
        raise ValueError("bias_act_ works in place on a contiguous tensor")
    C = u.shape[-1]
    rows = u.numel() // C
    per_image = bias is not None and bias.dim() == 2
    bc = None if bias is None else bias.detach().to(u.dtype).contiguous()
    n = u.shape[-2] if per_image else 0
    _call("d2s_bias_act", _ptr(u), _ptr(bc), _dtype_code(u), rows, n, C, int(act), _stream(u))
    return u


_F32_PARAM_CACHE = {}


def _f32c_param(t):
    """fp32 contiguous copy of a (small) parameter, cached while THIS tensor object, its storage and its version counter stand:
    the tail kernels take their last Linear in fp32, and converting it on every call costs two serialised copy kernels per
    stage.  The entry holds a weak reference to the tensor it was made from: a new tensor that happens to reuse the id, the
    address and the version of a dead one is a miss."""
    if t is None:
        return None
    if t.dtype == torch.float32 and t.is_contiguous():
        return t.detach()
    key = (t.data_ptr(), t._version, t.dtype, tuple(t.shape), t.device)
    hit = _F32_PARAM_CACHE.get(id(t))
    if hit is not None and hit[0]() is t and hit[1] == key:
        return hit[2]
    if len(_F32_PARAM_CACHE) > 256:
        for k in [k for k, v in _F32_PARAM_CACHE.items() if v[0]() is None]:
            del _F32_PARAM_CACHE[k]
        if len(_F32_PARAM_CACHE) > 256:
            _F32_PARAM_CACHE.clear()
    c = t.detach().to(torch.float32).contiguous()
    _F32_PARAM_CACHE[id(t)] = (weakref.ref(t), key, c)
    return c


PRED_TAIL_H = 192
PRED_TAIL_MAX_N = 256


def predictor_a_tail_ok(local, w2, w3, w4):
    """Shapes / dtypes d2s_predictor_a_tail_bf16 takes: bf16, D/2 = 192 with the D -> D/2 -> D/4 -> 2 stack, N <= 256."""
    H = PRED_TAIL_H
    return (local.is_cuda and local.dtype == torch.bfloat16 and local.dim() == 3 and local.shape[-1] == H
            and 1 <= local.shape[1] <= PRED_TAIL_MAX_N
            and all(w.dtype == torch.bfloat16 and w.is_contiguous() for w in (w2, w3))
            and tuple(w2.shape) == (H, 2 * H) and tuple(w3.shape) == (H // 2, H) and tuple(w4.shape) == (2, H // 2))


def predictor_a_tail(local, per_image, w2, w3, b3, w4, b4, k, prev=None, want_prev_kept=True):
    """Second half of Variant A's PredictorLG.forward + the stage's selection (vit_models/default_dynamic_vit.py:329-330,
    :461-467) as ONE tcgen05 kernel: local (B,N,192) bf16 from pool_act, per_image (B,192) = pooled @ W2[:, 192:]^T + b2,
    prev (B,N) f32 keep decisions or None.
    Returns (logp (B,N,2) f32, kept (B,k) int64 in descending-score order[, prev_kept (B,k) f32])."""
    _check_cuda(local, per_image, w2, w3, w4)
    h = local.detach()
    B, N, H = h.shape
    # a column slice of a wider contiguous (B, N, ld) tensor is read in place through the tensor map's row stride
    if not (h.stride(2) == 1 and h.stride(1) % 8 == 0 and h.stride(1) >= H and N > 1 and B > 1 and h.stride(0) >= N * h.stride(1)
            and h.stride(0) % 8 == 0 and h.data_ptr() % 16 == 0):
        h = h.contiguous()
    ld, lb = h.stride(1), h.stride(0)
    pl = per_image.detach().to(torch.bfloat16).contiguous()
    if not 0 <= k <= N:
        raise RuntimeError(f"predictor_a_tail: K={k} outside [0, N={N}]")
    dev = h.device
    logp = torch.empty(B, N, 2, dtype=torch.float32, device=dev)
    kept = torch.empty(B, k, dtype=torch.int64, device=dev)
    prev_kept = torch.empty(B, k, dtype=torch.float32, device=dev) if want_prev_kept else None
    if tuple(pl.shape) != (B, H):
        raise RuntimeError(f"predictor_a_tail: per_image must be ({B}, {H}), got {tuple(pl.shape)}")
    if B == 0:
        return (logp, kept, prev_kept) if want_prev_kept else (logp, kept)
    p = _f32c(prev.reshape(B, N)) if prev is not None else None
    b3c = b3.detach().to(torch.bfloat16).contiguous()
    w4f, b4f = _f32c_param(w4), _f32c_param(b4)
    _call("d2s_predictor_a_tail_bf16", _ptr(h), int(ld), int(lb), _ptr(pl), _ptr(w2.detach()), _ptr(w3.detach()), _ptr(b3c),
          _ptr(w4f), _ptr(b4f), _ptr(p), B, N, H, k, _ptr(logp), _ptr(kept), _ptr(prev_kept), _stream(h))
    return (logp, kept, prev_kept) if want_prev_kept else (logp, kept)


class _PoolConcat(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, policy):
        hc = h.contiguous()
        B, N, C = hc.shape
        pol = None if policy is None else _f32c(policy.reshape(B, N))
        out = torch.empty_like(hc)
        pooled = torch.empty(B, C // 2, dtype=torch.float32, device=hc.device)
        wsum = torch.empty(B, dtype=torch.float32, device=hc.device)
        if B > 0:
            _call("d2s_pool_concat_fwd", _ptr(hc), _ptr(pol), _dtype_code(hc), B, N, C, _ptr(out), _ptr(pooled), _ptr(wsum), _stream(hc))
        ctx.save_for_backward(hc, pooled, wsum, pol if pol is not None else torch.empty(0, device=hc.device))
        ctx.meta = (pol is not None, None if policy is None else (policy.shape, policy.dtype))
        return out

    @staticmethod
    def backward(ctx, gout):
        hc, pooled, wsum, pol = ctx.saved_tensors
        has_pol, pol_meta = ctx.meta
        B, N, C = hc.shape
        g = gout.to(hc.dtype).contiguous()
        dh = torch.empty_like(hc)
        want_dp = has_pol and ctx.needs_input_grad[1]
        dpol = torch.empty(B, N, dtype=torch.float32, device=hc.device) if want_dp else None
        if B > 0:
            _call("d2s_pool_concat_bwd", _ptr(g), _ptr(hc), _ptr(pol if has_pol else None), _ptr(pooled), _ptr(wsum), _dtype_code(hc),
                  B, N, C, _ptr(dh), _ptr(dpol), _stream(g))
        return dh, None if dpol is None else dpol.view(pol_meta[0]).to(pol_meta[1])


def pool_concat_train(h, policy=None):
    """cat(h[..., :C/2], weighted mean over tokens of h[..., C/2:] broadcast to every token) for h (B,N,C) f32|bf16 with
    autograd in h and policy (B,N,1) or None (plain mean): the local / global split of PredictorLG.forward
    (default_dynamic_vit.py:326-329, dynamic_vit.py:541-545) as one kernel forward and one backward."""
    _check_cuda(h, policy)
    if h.dim() != 3 or h.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError("pool_concat_train: a (B,N,C) f32 | bf16 tensor is expected")
    return _PoolConcat.apply(h, policy)


def pool_concat_train_ok(h):
    ve = 8 if h.dtype == torch.bfloat16 else 4
    return (h.is_cuda and h.dim() == 3 and h.dtype in (torch.float32, torch.bfloat16) and h.shape[-1] % (2 * ve) == 0
            and h.shape[-1] // 2 // ve <= 96 and h.shape[1] >= 1)


def _rows_view_ok(t):
    """(B,N,C) f32 | bf16 CUDA tensor whose tokens are dense rows (strides (bs, C, 1)): contiguous, or a row slice x[:, r:]."""
    return (t.dim() == 3 and t.is_cuda and t.dtype in (torch.float32, torch.bfloat16) and t.stride(2) == 1 and t.stride(1) == t.shape[2]
            and t.stride(0) >= t.shape[1] * t.shape[2] and t.stride(0) % 8 == 0 and t.data_ptr() % 16 == 0)


def token_kl_ok(s, t):
    return (_rows_view_ok(s) and _rows_view_ok(t) and s.shape == t.shape and s.shape[2] % 8 == 0 and s.shape[2] <= 1024
            and s.shape[1] >= 1)


class _TokenKL(torch.autograd.Function):
    @staticmethod
    def forward(ctx, s, t):
        B, N, C = s.shape
        kl = torch.empty(B * N, dtype=torch.float32, device=s.device)
        diff = torch.empty(B * N, C, dtype=torch.float32, device=s.device)
        if B > 0:
            _call("d2s_token_kl_fwd", _ptr(s), _dtype_code(s), s.stride(0), _ptr(t), _dtype_code(t), t.stride(0), B, N, C, _ptr(kl),
                  _ptr(diff), _stream(s))
        ctx.save_for_backward(diff)
        ctx.meta = (s.shape, s.dtype)
        return kl

    @staticmethod
    def backward(ctx, g):
        (diff,) = ctx.saved_tensors
        shape, dt = ctx.meta
        return (diff * g.reshape(-1, 1)).view(shape).to(dt), None


def token_kl_rows(s, t):
    """Per-token KL(softmax(t) || softmax(s)) over the channels, (B*N,) f32, differentiable in s (t is a constant target):
    F.kl_div(F.log_softmax(s), F.log_softmax(t), log_target=True, reduction='none').sum(-1) of losses.py:220-225 as one pass
    (`d2s_token_kl_fwd`); s and t may be x[:, 1:] views."""
    _check_cuda(s, t)
    if not token_kl_ok(s, t):
        raise RuntimeError(f"token_kl_rows: (B,N,C) f32 | bf16 row-dense tensors of one shape with C % 8 == 0, C <= 1024 are expected, got "
                           f"{tuple(s.shape)} {s.dtype} strides {s.stride()} and {tuple(t.shape)} {t.dtype} strides {t.stride()}")
    return _TokenKL.apply(s, t.detach())


def pool_concat_(z):
    """In place: z (B,N,C) <- cat(z[..., :C/2], mean over tokens of z[..., C/2:] broadcast) (dynamic_vit.py:539-545)."""
    _check_cuda(z)
    if not z.is_contiguous():
        raise ValueError("pool_concat_ works in place on a contiguous tensor")
    B, N, C = z.shape
    _call("d2s_pool_concat_inplace", _ptr(z), _dtype_code(z), B, N, C, _stream(z))
    return z


def pool_concat_varlen_(z, lengths):
    """pool_concat_ over a padded batch: image b's mean runs over z[b, :lengths[b]] and is written into those rows only; pad
    rows are neither read nor written."""
    _check_cuda(z)
    if not z.is_contiguous():
        raise ValueError("pool_concat_varlen_ works in place on a contiguous tensor")
    B, N, C = z.shape
    n = _lengths(lengths, B, "pool_concat_varlen_")
    _call("d2s_pool_concat_varlen_inplace", _ptr(z), _ptr(n), _dtype_code(z), B, N, C, _stream(z))
    return z


def assemble_tokens(patches, cls_token, pos_embed):
    """cat(cls_token.expand(B,-1,-1), patches) + pos_embed in one pass (vit_models/dynamic_vit.py:820-823)."""
    _check_cuda(patches, cls_token, pos_embed)
    pc = patches.detach().contiguous()
    B, N, D = pc.shape
    cls = cls_token.detach().to(pc.dtype).reshape(D).contiguous()
    pos = pos_embed.detach().to(pc.dtype).reshape(N + 1, D).contiguous()
    out = torch.empty(B, N + 1, D, dtype=pc.dtype, device=pc.device)
    _call("d2s_assemble_tokens", _ptr(pc), _ptr(cls), _ptr(pos), _dtype_code(pc), B, N, D, _ptr(out), _stream(pc))
    return out


def assemble_layernorm(patches, cls_token, pos_embed, weight, bias, eps, want_stats=False):
    """(x, LayerNorm(x)) with x = cat(cls_token, patches) + pos_embed: token assembly fused with the first block's norm1
    (vit_models/dynamic_vit.py:820-823 + :263).  Inference only.
    want_stats (bf16): (x, stats (B*(N+1), 2) f32 = per-row (mean, rstd)) instead; the consumer applies the LayerNorm."""
    _check_cuda(patches, cls_token, pos_embed, weight, bias)
    pc = patches.detach().contiguous()
    B, N, D = pc.shape
    cls = cls_token.detach().to(pc.dtype).reshape(D).contiguous()
    pos = pos_embed.detach().to(pc.dtype).reshape(N + 1, D).contiguous()
    if want_stats:
        if pc.dtype != torch.bfloat16:
            raise TypeError("assemble_layernorm(want_stats=True) is a bf16 path")
        out_sum = torch.empty(B, N + 1, D, dtype=pc.dtype, device=pc.device)
        stats = torch.empty(B * (N + 1), 2, dtype=torch.float32, device=pc.device)
        if B:
            _call("d2s_assemble_layernorm_stats", _ptr(pc), _ptr(cls), _ptr(pos), B, N, D, float(eps), _ptr(out_sum), _ptr(stats),
                  _stream(pc))
        return out_sum, stats
    w, b = weight.detach().to(pc.dtype).contiguous(), bias.detach().to(pc.dtype).contiguous()
    out_sum = torch.empty(B, N + 1, D, dtype=pc.dtype, device=pc.device)
    out_norm = torch.empty_like(out_sum)
    _call("d2s_assemble_layernorm", _ptr(pc), _ptr(cls), _ptr(pos), _ptr(w), _ptr(b), _dtype_code(pc), B, N, D, float(eps),
              _ptr(out_sum), _ptr(out_norm), _stream(pc))
    return out_sum, out_norm


def patchify(img, ph, pw):
    """img (B,C,H,W) -> (B, (H/ph)*(W/pw), C*ph*pw): im2col of non-overlapping patches, k = (c, py, px)."""
    _check_cuda(img)
    x = img.detach().contiguous()
    B, C, Hh, Ww = x.shape
    out = torch.empty(B, (Hh // ph) * (Ww // pw), C * ph * pw, dtype=x.dtype, device=x.device)
    _call("d2s_patchify", _ptr(x), _dtype_code(x), B, C, Hh, Ww, int(ph), int(pw), _ptr(out), _stream(x))
    return out


def patchify_u8(img, ph, pw, mean, std, out_dtype=torch.bfloat16):
    """Raw uint8 images (B,C,H,W) -> normalised patches (B, (H/ph)*(W/pw), C*ph*pw) of `out_dtype`: torchvision's ToTensor +
    Normalize ((x / 255 - mean[c]) / std[c], fp32) and the im2col of PatchEmbed in one pass, bit-identical to doing them with
    torch.  mean, std: per-channel fp32 tensors."""
    _check_cuda(img, mean, std)
    if img.dtype != torch.uint8:
        raise TypeError("patchify_u8 takes uint8 images")
    x = img.detach().contiguous()
    B, C, Hh, Ww = x.shape
    m, s = _f32c(mean).reshape(-1), _f32c(std).reshape(-1)
    if m.numel() != C or s.numel() != C:
        raise ValueError(f"patchify_u8: mean / std must have {C} entries")
    out = torch.empty(B, (Hh // ph) * (Ww // pw), C * ph * pw, dtype=out_dtype, device=x.device)
    _call("d2s_patchify_u8", _ptr(x), _ptr(m), _ptr(s), _dtype_code(out), B, C, Hh, Ww, int(ph), int(pw), _ptr(out), _stream(x))
    return out


# ----------------------------------------------------------------------------------------------
# LayerNorm with autograd (training path)
# ----------------------------------------------------------------------------------------------

def _ln_grad_targets(ctx, D, dev):
    """Where the LayerNorm backward accumulates (dgamma, dbeta): the parameters' gradient slots when both have one (nothing is
    returned to autograd then), else a fresh zeroed pair."""
    weight, bias = ctx.params
    (sw, ew), (sb, eb) = _grad_slot(weight), _grad_slot(bias)
    if sw is not None and sb is not None:
        ew[1] = eb[1] = False
        return sw, sb, True
    dgb = torch.zeros(2, D, dtype=torch.float32, device=dev)
    return dgb[0], dgb[1], False


class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_dtype, row0):
        xc = x.contiguous()
        D = xc.shape[-1]
        w, b = _f32c(weight), _f32c(bias)
        if row0:                                     # LayerNorm(x[:, row0:]) of a (B, T, D) tensor without the slice copy
            B, T = xc.shape[0], xc.shape[1]
            seg = T - row0
            rows = B * seg
            h = torch.empty(B, seg, D, dtype=out_dtype, device=xc.device)
            stats = torch.empty(rows, 2, dtype=torch.float32, device=xc.device)
            if rows:
                _call("d2s_layernorm_seg_fwd", _ptr(xc), _dtype_code(xc), _ptr(w), _ptr(b), rows, D, seg, row0, float(eps), _ptr(h),
                      _dtype_code(h), _ptr(stats), _stream(xc))
        else:
            rows = xc.numel() // D
            seg = 0
            h = torch.empty(xc.shape, dtype=out_dtype, device=xc.device)
            stats = torch.empty(rows, 2, dtype=torch.float32, device=xc.device)
            _call("d2s_layernorm_fwd", _ptr(xc), _dtype_code(xc), _ptr(w), _ptr(b), rows, D, float(eps), _ptr(h),
                      _dtype_code(h), _ptr(stats), _stream(xc))
        ctx.save_for_backward(xc, stats, w)
        ctx.meta = (weight.dtype, bias.dtype, rows, seg, row0)
        ctx.params = (weight, bias)
        return h

    @staticmethod
    def backward(ctx, dh):
        xc, stats, w = ctx.saved_tensors
        _, _, rows, seg, row0 = ctx.meta
        D = xc.shape[-1]
        g = dh.contiguous()
        dx = torch.empty_like(xc)
        dg, db, direct = _ln_grad_targets(ctx, D, xc.device)
        if seg:
            if rows:
                _call("d2s_layernorm_seg_bwd", _ptr(g), _dtype_code(g), _ptr(xc), _dtype_code(xc), _ptr(stats), _ptr(w), rows, D, seg,
                      row0, _ptr(dx), _ptr(dg), _ptr(db), _stream(g))
            else:
                dx.zero_()
        else:
            _call("d2s_layernorm_bwd", _ptr(g), _dtype_code(g), _ptr(xc), _dtype_code(xc), _ptr(stats), _ptr(w), rows, D,
                      _ptr(dx), _ptr(dg), _ptr(db), _stream(g))
        if direct:
            return dx, None, None, None, None, None
        return dx, dg.to(ctx.meta[0]), db.to(ctx.meta[1]), None, None, None


class _AddLayerNorm(torch.autograd.Function):
    """(s, h) = (x + y, LayerNorm(x + y)) as one kernel each way: the forward writes both, the backward adds the gradient
    reaching s directly into the LayerNorm's input gradient and hands the same tensor to x and y."""

    @staticmethod
    def forward(ctx, x, y, weight, bias, eps, out_dtype):
        xc, yc = x.contiguous(), y.contiguous()
        D = xc.shape[-1]
        rows = xc.numel() // D
        w, b = _f32c(weight), _f32c(bias)
        s = torch.empty_like(xc)
        h = torch.empty(xc.shape, dtype=out_dtype, device=xc.device)
        stats = torch.empty(rows, 2, dtype=torch.float32, device=xc.device)
        _call("d2s_add_layernorm_fwd", _ptr(xc), _ptr(yc), _dtype_code(xc), _ptr(w), _ptr(b), rows, D, float(eps), _ptr(s),
                  _ptr(h), _dtype_code(h), _ptr(stats), _stream(xc))
        ctx.save_for_backward(s, stats, w)
        ctx.meta = (weight.dtype, bias.dtype)
        ctx.params = (weight, bias)
        return s, h

    @staticmethod
    def backward(ctx, gs, gh):
        s, stats, w = ctx.saved_tensors
        if gh is None:
            return gs, gs, None, None, None, None
        D = s.shape[-1]
        rows = s.numel() // D
        g = gh.contiguous()
        ga = None if gs is None else gs.to(s.dtype).contiguous()
        dx = torch.empty_like(s)
        dg, db, direct = _ln_grad_targets(ctx, D, s.device)
        _call("d2s_add_layernorm_bwd", _ptr(g), _dtype_code(g), _ptr(s), _dtype_code(s), _ptr(stats), _ptr(w), _ptr(ga), rows, D,
                  _ptr(dx), _ptr(dg), _ptr(db), _stream(g))
        if direct:
            return dx, dx, None, None, None, None
        return dx, dx, dg.to(ctx.meta[0]), db.to(ctx.meta[1]), None, None


def add_layer_norm_train(x, y, weight, bias, eps, out_dtype=None):
    """(x + y, LayerNorm(x + y)) with autograd in x, y, weight and bias: the training-path form of the fused residual add +
    LayerNorm (x and y of one dtype, f32 or bf16; the sum is rounded to that dtype like torch's add)."""
    _check_cuda(x, y, weight, bias)
    if x.dtype != y.dtype or x.shape != y.shape:
        raise RuntimeError(f"add_layer_norm_train: x {tuple(x.shape)} {x.dtype} and y {tuple(y.shape)} {y.dtype} must match")
    if out_dtype is None:
        out_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    return _AddLayerNorm.apply(x, y, weight, bias, eps, out_dtype)


def layer_norm(x, weight, bias, eps, out_dtype=None, row0=0):
    """LayerNorm over the last dim with autograd: x f32|bf16 -> out_dtype (default: bf16 under CUDA autocast, else
    x.dtype), statistics in fp32.  One streaming kernel forward, one backward (dx + dgamma + dbeta).
    row0 > 0: x is (B, T, D) and the result is LayerNorm(x[:, row0:]) (B, T - row0, D) -- the predictors' input norm over the
    patch tokens -- read in place (no slice copy; the backward writes the full (B, T, D) gradient, zeros in the skipped rows)."""
    _check_cuda(x, weight, bias)
    if out_dtype is None:
        out_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    if row0 and (x.dim() != 3 or not 0 < row0 < x.shape[1]):
        raise RuntimeError(f"layer_norm: row0={row0} needs a (B, T, D) input with T > row0, got {tuple(x.shape)}")
    return _LayerNorm.apply(x, weight, bias, eps, out_dtype, int(row0))


def linear_act(x, weight, bias, act=ACT_GELU, want_pre=False, in_stats=None, in_ln_weight=None, in_ln_bias=None):
    """act(x @ weight^T + bias) in one CTA-pair tcgen05 GEMM with the activation in the epilogue (bf16, no autograd).
    x (..., K) contiguous, weight (N, K), N % 256 == 0 or N % 192 == 0 (256- or 192-column tiles), K % 64 == 0.  want_pre: returns (act(u), u) with u the Linear's own
    output as a second result of the same kernel."""
    _check_cuda(x, weight, bias)
    if x.dtype != torch.bfloat16:
        raise TypeError("linear_act is a bf16 kernel")
    xc = x.detach().contiguous()
    w = weight.detach().to(torch.bfloat16).contiguous()
    b = None if bias is None else bias.detach().to(torch.bfloat16).contiguous()
    K = xc.shape[-1]
    M = xc.numel() // K
    N = w.shape[0]
    out = torch.empty(*xc.shape[:-1], N, dtype=torch.bfloat16, device=xc.device)
    if in_stats is not None:
        # x is the raw residual stream: LayerNorm(x) (in_ln_weight / in_ln_bias, statistics from the producer) is formed in the
        # kernel's resident input tile (N % 192 == 0, K <= 384)
        st = in_stats.detach().contiguous()
        if want_pre or st.dtype != torch.float32 or st.numel() != 2 * M:
            raise RuntimeError(f"linear_act: in_stats must be ({M}, 2) float32 (and no second output)")
        gi, bi = (t.detach().to(torch.bfloat16).contiguous() for t in (in_ln_weight, in_ln_bias))
        if M:
            _call("d2s_linear_lnin_act_pair_bf16", _ptr(xc), _ptr(st), _ptr(gi), _ptr(bi), _ptr(w), _ptr(b), M, N, K, int(act),
                  _ptr(out), _stream(xc))
        return out
    pre = torch.empty_like(out) if want_pre else None
    _call("d2s_linear_act_pair_bf16", _ptr(xc), _ptr(w), _ptr(b), M, N, K, int(act), _ptr(out), _ptr(pre), _stream(xc))
    return (out, pre) if want_pre else out


def linear_residual_ln(a, weight, bias, x, ln_weight=None, ln_bias=None, eps=1e-5, want_norm=True, want_stats=False):
    """(x', h) with x' = x + (a @ weight^T + bias) and h = LayerNorm(x') * ln_weight + ln_bias (h None when
    want_norm is False): attn.proj / mlp.fc2 + residual add + the next LayerNorm of Block.forward
    (vit_models/dynamic_vit.py:263-283) in one CTA-pair tcgen05 GEMM.  bf16, inference only; N in {192, 384, 768}.
    want_stats (with want_norm=False): returns (x', stats) with stats (M,2) f32 = per-row (mean, rstd) of x' for `eps`: the
    consumer (mlp_residual_ln(in_stats=...)) applies the LayerNorm itself and the normalised copy is never written."""
    _check_cuda(a, weight, bias, x, ln_weight, ln_bias)
    if a.dtype != torch.bfloat16 or x.dtype != torch.bfloat16:
        raise TypeError("linear_residual_ln is a bf16 kernel")
    ac = a.detach().contiguous()
    xc = x.detach().contiguous()
    w = weight.detach().to(torch.bfloat16).contiguous()
    b = None if bias is None else bias.detach().to(torch.bfloat16).contiguous()
    K = ac.shape[-1]
    M = ac.numel() // K
    N = w.shape[0]
    if xc.numel() != M * N:
        raise RuntimeError(f"linear_residual_ln: residual has {xc.numel()} elements, expected {M}x{N}")
    g = bt = None
    if want_norm:
        g = ln_weight.detach().to(torch.bfloat16).contiguous()
        bt = ln_bias.detach().to(torch.bfloat16).contiguous()
    out_sum = torch.empty_like(xc)
    if want_stats:
        if want_norm:
            raise RuntimeError("linear_residual_ln: want_stats replaces the normalised output (want_norm=False)")
        stats = torch.empty(M, 2, dtype=torch.float32, device=xc.device)
        if M:
            _call("d2s_linear_residual_stats_bf16", _ptr(ac), _ptr(w), _ptr(b), _ptr(xc), float(eps), M, N, K, _ptr(out_sum),
                  _ptr(stats), _stream(ac))
        return out_sum, stats
    out_norm = torch.empty_like(xc) if want_norm else None
    _call("d2s_linear_residual_ln_bf16", _ptr(ac), _ptr(w), _ptr(b), _ptr(xc), _ptr(g), _ptr(bt), float(eps), M, N, K,
              _ptr(out_sum), _ptr(out_norm), _stream(ac))
    return out_sum, out_norm


def mlp_residual_ln(h, w1, b1, w2, b2, x, ln_weight=None, ln_bias=None, eps=1e-5, want_norm=True, norm_row0=0,
                    in_stats=None, in_ln_weight=None, in_ln_bias=None, want_stats=False):
    """(x', hn) with x' = x + fc2(GELU(fc1(h))) and hn = LayerNorm(x') * ln_weight + ln_bias (None when want_norm is False):
    the MLP branch of Block.forward with its residual add and the next LayerNorm (vit_models/dynamic_vit.py:159-175, :263-283)
    in ONE CTA-pair tcgen05 kernel; the hidden activations stay on chip.  bf16, inference only, D == 384.
    norm_row0 > 0 (x of shape (B,T,D)): hn = LayerNorm(x'[:, norm_row0:]) of shape (B, T-norm_row0, D).
    in_stats (M,2) f32 with in_ln_weight / in_ln_bias: h is None and the MLP's input is LayerNorm(x) formed on the fly from the
    per-row (mean, rstd) that linear_residual_ln(want_stats=True) wrote next to x.
    want_stats (with in_stats, want_norm=False): returns (x', stats (M,2) f32 = per-row (mean, rstd) of x' for `eps`) -- the next
    LayerNorm is then applied by its consumer (linear_act(in_stats=...): the next block's qkv projection)."""
    if in_stats is not None:
        h = x
    _check_cuda(h, w1, b1, w2, b2, x, ln_weight, ln_bias, in_stats, in_ln_weight, in_ln_bias)
    if h.dtype != torch.bfloat16 or x.dtype != torch.bfloat16:
        raise TypeError("mlp_residual_ln is a bf16 kernel")
    hc, xc = h.detach().contiguous(), x.detach().contiguous()
    bf = lambda t: None if t is None else t.detach().to(torch.bfloat16).contiguous()
    w1c, w2c = bf(w1), bf(w2)
    D = hc.shape[-1]
    M = hc.numel() // D
    HID = w1c.shape[0]
    if xc.numel() != M * D or tuple(w2c.shape) != (D, HID) or w1c.shape[1] != D:
        raise RuntimeError(f"mlp_residual_ln: inconsistent shapes h{tuple(h.shape)} w1{tuple(w1.shape)} w2{tuple(w2.shape)} x{tuple(x.shape)}")
    g, bt = (bf(ln_weight), bf(ln_bias)) if want_norm else (None, None)
    out_sum = torch.empty_like(xc)
    T = 1
    if norm_row0:
        if xc.dim() != 3:
            raise RuntimeError("mlp_residual_ln: norm_row0 needs x of shape (B, T, D)")
        T = xc.shape[1]
    out_norm = None
    if want_norm:
        out_norm = torch.empty(xc.shape[0], T - norm_row0, D, dtype=xc.dtype, device=xc.device) if norm_row0 else torch.empty_like(xc)
    if in_stats is not None:
        st = in_stats.detach().contiguous()
        if st.dtype != torch.float32 or st.numel() != 2 * M:
            raise RuntimeError(f"mlp_residual_ln: in_stats must be ({M}, 2) float32")
        out_stats = torch.empty(M, 2, dtype=torch.float32, device=xc.device) if want_stats else None
        _call("d2s_mlp_lnin_residual_ln_bf16", _ptr(xc), _ptr(st), _ptr(bf(in_ln_weight)), _ptr(bf(in_ln_bias)), _ptr(w1c),
              _ptr(bf(b1)), _ptr(w2c), _ptr(bf(b2)), _ptr(g), _ptr(bt), float(eps), M, D, HID, T, int(norm_row0), _ptr(out_sum),
              _ptr(out_norm), _ptr(out_stats), _stream(xc))
        return (out_sum, out_stats) if want_stats else (out_sum, out_norm)
    if want_stats:
        raise RuntimeError("mlp_residual_ln: want_stats is an output of the in_stats form of the kernel")
    _call("d2s_mlp_residual_ln_bf16", _ptr(hc), _ptr(w1c), _ptr(bf(b1)), _ptr(w2c), _ptr(bf(b2)), _ptr(xc), _ptr(g), _ptr(bt),
              float(eps), M, D, HID, T, int(norm_row0), _ptr(out_sum), _ptr(out_norm), _stream(hc))
    return out_sum, out_norm
