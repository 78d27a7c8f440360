"""Forward routines of the hot path, written against the reference's attribute names.

Every function takes a module that exposes the same attributes as the corresponding reference class
(`qkv`, `proj`, `num_heads`, `scale`, `in_conv`, `out_conv`, `blocks`, `score_predictor`, ...), so the same
code serves this package's own nn.Modules (modules.py) and, through patch.py, the reference's classes
themselves.  File:line citations point into the reference tree.

Two execution modes, chosen per call:
  * fused    (no gradient needed): qkv Linear -> d2s attention kernel (tcgen05 in bf16) -> proj; predictor
             tail + selection in one kernel; gather kernel.  Dense Linear layers stay on cuBLAS.
  * autograd (a gradient is needed): library GEMMs around the one-pass policy-softmax kernel
             (forward + backward in both arguments), gather/scatter kernels, Gumbel decision kernel.
"""
import copy
import os
import weakref

import torch
import torch.nn.functional as F

from . import ops

# Test hooks.  Each is True in use; a test sets one to False to run the unfused reference path it compares the fused path
# against (tests/test_gpu_models.py::test_fused_block_kernels_at_deit_s_width, ::test_training_fusions_match_the_unfused_training_path,
# ::test_frozen_teacher_under_autocast_runs_on_a_cached_bf16_copy; tests/test_gpu_parity.py::test_predictor_a_tail_matches_the_unfused_path,
# ::test_lazy_norms_are_invisible_at_model_level; the kernel on/off comparisons in tests/test_gpu_long_attn.py).
_FUSED_PAIR = True           # the CTA-pair GEMMs (qkv, fc1 pair; proj/fc2 + add + LN)
_FUSED_MLP = True            # the one-kernel MLP (ops.mlp_residual_ln)
_FUSED_ADD_LN_TRAIN = True   # residual adds folded into LayerNorm fwd/bwd
_FROZEN_BF16 = True          # cached bf16 copy of a frozen teacher under bf16 autocast
_PRED_FUSED = True           # second half of the Variant A predictor + selection as one tcgen05 kernel (inference, D = 384)
_LAZY_NORM1 = True           # norm1 applied inside the qkv GEMM from the MLP kernel's row statistics
_LAZY_NORM2 = True           # norm2 applied inside the one-kernel MLP from per-row statistics (no normalised copy)
_LONG_ATTN = True            # bf16 attention beyond 256 tokens on the key-blocked kernels (inference, and training fwd + bwd)
_THRESHOLD_INFERENCE = os.environ.get("D2S_THRESHOLD_INFERENCE", "0") == "1"   # opt-in: what dynamic_vit.py:935-949 intends
INIT_N = 14 * 14  # the reference hard-codes 196 spatial tokens (dynamic_vit.py:828, default_dynamic_vit.py:446)


def _needs_grad(*ts):
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts)


def _d2s_float(t):
    """The d2s kernels read float32 / bfloat16 and, under autocast, can only stand in for torch when the autocast dtype is bf16
    (fp16 autocast -- the mode ddp_training.py:84-85,130 sets a GradScaler up for -- keeps torch's own modules)."""
    if t.dtype not in (torch.float32, torch.bfloat16):
        return False
    return not torch.is_autocast_enabled("cuda") or torch.get_autocast_dtype("cuda") == torch.bfloat16


def _ln_rows_ok(x):
    """Row widths the LayerNorm-family kernels take: multiples of 8, up to 1536 (bf16) / 768 (fp32)."""
    return x.shape[-1] % 8 == 0 and x.shape[-1] <= (1536 if x.dtype == torch.bfloat16 else 768)


def _attn_kernel_ok(qkv, H):
    """Shapes of the fused attention kernels: bf16 -> tcgen05 kernel (hd 64), fp32 -> SIMT kernel (hd 32 / 64), T <= 256; and bf16,
    hd 64, 256 < T <= 2048 -> the key-blocked tcgen05 kernel (d2s_attn_long_fwd)."""
    hd = qkv.shape[-1] // 3 // H
    if qkv.shape[-1] != 3 * H * hd:
        return False
    if qkv.shape[1] > 256:
        return _LONG_ATTN and qkv.dtype == torch.bfloat16 and hd == 64 and qkv.shape[1] <= ops.LONG_ATTN_MAX_T
    return (qkv.dtype == torch.bfloat16 and hd == 64) or (qkv.dtype == torch.float32 and hd in (32, 64))


def _attn_train_kernel_ok(qkv, H):
    """Shapes the training branch hands to ops.attention_train: bf16 with T <= 256 (tcgen05 flash kernels at hd 64, T <= 208,
    else head-major GEMMs around the padded-row softmax), and bf16, hd 64, 256 < T <= 2048 (the key-blocked forward with row
    statistics + d2s_attn_long_bwd) unless _LONG_ATTN is off."""
    if qkv.dtype != torch.bfloat16:
        return False
    if qkv.shape[1] <= 256:
        return True
    hd = qkv.shape[-1] // 3 // H
    return _LONG_ATTN and qkv.shape[-1] == 3 * H * hd and hd == 64 and qkv.shape[1] <= ops.LONG_ATTN_MAX_T


def _softmax_policy_torch(attn, policy, eps=1e-6):
    """Attention.softmax_with_policy (dynamic_vit.py:195-214) in plain torch, for dtypes / shapes the kernels do not take:
    keep mask p_j off the diagonal and 1 on it, fp32 exponentials of (attn - rowmax), eps/N added to every entry."""
    B, H, N, _ = attn.shape
    p = policy.reshape(B, 1, 1, N).to(torch.float32)
    mask = p + (1.0 - p) * torch.eye(N, dtype=torch.float32, device=attn.device).view(1, 1, N, N)
    e = (attn - attn.amax(dim=-1, keepdim=True)).to(torch.float32).exp() * mask
    return ((e + eps / N) / (e.sum(dim=-1, keepdim=True) + eps)).type_as(attn)


def softmax_with_policy(attn, policy, eps=1e-6):
    """Attention.softmax_with_policy (dynamic_vit.py:195-214): the one-pass d2s kernel pair (forward, backward in both
    arguments) for fp32 / bf16 CUDA tensors; other CUDA float types (fp16 autocast) take the torch restatement."""
    if attn.is_cuda and attn.dtype not in (torch.float32, torch.bfloat16):
        return _softmax_policy_torch(attn, policy, eps) if policy is not None else attn.softmax(dim=-1)
    return ops.softmax_with_policy(attn, policy, eps)


def patch_embed_forward(m, img):
    """Conv2d(kernel=stride=patch) as im2col + GEMM (dynamic_vit.py:286-303).  Avoids cuDNN's TF32 conv path so fp32
    runs stay within 1e-4 of the reference; the im2col is one d2s kernel when no gradient flows into the image."""
    B, C, Hh, Ww = img.shape
    ph, pw = m.patch_size
    assert Hh == m.img_size[0] and Ww == m.img_size[1], \
        f"Input image size ({Hh}*{Ww}) doesn't match model ({m.img_size[0]}*{m.img_size[1]})."
    gh, gw = Hh // ph, Ww // pw
    w = m.proj.weight
    if img.dtype == torch.uint8:
        # raw pixels (runner.InferenceRunner(..., uint8_input=True)): ToTensor + Normalize fused into the im2col kernel
        norm = getattr(m, "d2s_input_norm", None)
        if norm is None:
            raise RuntimeError("uint8 images need the normalisation constants: set patch_embed.d2s_input_norm = (mean, std)")
        if img.is_cuda and w.dtype in (torch.float32, torch.bfloat16) and pw % 8 == 0 and Ww % 16 == 0 and C <= 4:
            patches = ops.patchify_u8(img, ph, pw, norm[0], norm[1], out_dtype=w.dtype)
            return F.linear(patches, w.view(w.shape[0], -1), m.proj.bias)
        mean, std = (t.to(img.device, torch.float32).view(1, C, 1, 1) for t in norm)
        img = (img.to(torch.float32).div(255.0) - mean) / std
    img = img.to(w.dtype)
    if img.is_cuda and not _needs_grad(img) and img.dtype in (torch.float32, torch.bfloat16) and pw % 8 == 0 and Ww % 8 == 0:
        patches = ops.patchify(img, ph, pw)
    else:
        patches = img.view(B, C, gh, ph, gw, pw).permute(0, 2, 4, 1, 3, 5).reshape(B, gh * gw, C * ph * pw)
    return F.linear(patches, w.view(w.shape[0], -1), m.proj.bias)


def _qkv_pair_ok(lin, x):
    """The qkv projection runs on the CTA-pair tcgen05 GEMM with 192-column tiles and resident input rows: inference, bf16, D <= 384."""
    return (_FUSED_PAIR and x.is_cuda and x.dtype == torch.bfloat16 and lin.weight.dtype == torch.bfloat16
            and not _needs_grad(x, lin.weight, lin.bias) and lin.in_features % 64 == 0 and lin.in_features <= 384
            and lin.out_features % 192 == 0 and lin.out_features % 256 != 0)


def attention_pre_proj(m, x, policy=None, return_cls_attn=False, lens=None):
    """Attention.forward up to (not including) the output projection (dynamic_vit.py:216-231): (o (B,T,C), cls_attn).
    lens (B) int32: a padded batch (image b = its first lens[b] tokens), run by the variable-length attention kernel."""
    B, T, C = x.shape
    H = m.num_heads
    lin = m.qkv
    if isinstance(x, _LazyNorm):
        if _qkv_pair_ok(lin, x):
            # norm1 was not materialised: the qkv GEMM normalises its resident input rows from the producer's row statistics
            qkv = ops.linear_act(x.x, lin.weight, lin.bias, ops.ACT_NONE, in_stats=x.stats, in_ln_weight=x.norm.weight,
                                 in_ln_bias=x.norm.bias)
        else:
            x = x.value()
    if isinstance(x, _LazyNorm):
        pass
    elif _qkv_pair_ok(lin, x):
        # inference, D <= 384: the CTA-pair tcgen05 GEMM with 192-column tiles and the row tile's input rows resident in shared
        # memory -- bit-identical to the library GEMM and as fast (both are bound by the 3 x (B,T,D) write stream)
        qkv = ops.linear_act(x, lin.weight, lin.bias, ops.ACT_NONE)
    else:
        qkv = ops.linear_train(lin, x)
    if lens is not None:
        if _needs_grad(qkv) or not qkv.is_cuda or not _attn_kernel_ok(qkv, H) or policy is not None:
            raise RuntimeError("variable-length attention: inference only, no policy, CUDA qkv of a shape the d2s attention kernels "
                               f"take (bf16 with head dim 64 and T <= 2048, or fp32 with head dim 32 / 64 and T <= 256); got {tuple(qkv.shape)} {qkv.dtype}")
        o, cls_attn = ops.attention_core(qkv, H, scale=m.scale, want_cls_row=return_cls_attn, lengths=lens)
        return o, (cls_attn.to(qkv.dtype) if cls_attn is not None else None)
    if _needs_grad(qkv, policy) and qkv.is_cuda and _attn_train_kernel_ok(qkv, H):
        # training, bf16: the tcgen05 flash forward / backward pair on the packed tensor (T <= 208, hd 64; key-blocked beyond 256
        # tokens), else per-head GEMMs on a head-major copy around the padded-row policy softmax
        o, cls_attn = ops.attention_train(qkv, H, policy=policy, scale=m.scale, want_cls_row=return_cls_attn)
    elif _needs_grad(qkv, policy) or not qkv.is_cuda or not _attn_kernel_ok(qkv, H):
        q, k, v = qkv.reshape(B, T, 3, H, C // H).permute(2, 0, 3, 1, 4).unbind(0)
        attn = (q @ k.transpose(-2, -1)) * m.scale
        if qkv.is_cuda:
            attn = softmax_with_policy(attn, policy)
        elif policy is None:
            attn = attn.softmax(dim=-1)
        else:                                  # CPU tensors (module construction / shape tests off the GPU)
            attn = _softmax_policy_torch(attn, policy)
        o = (attn @ v).transpose(1, 2).reshape(B, T, C)
        cls_attn = attn[:, :, 0, :] if return_cls_attn else None
    else:
        o, cls_attn = ops.attention_core(qkv, H, policy=policy, scale=m.scale, want_cls_row=return_cls_attn)
        if cls_attn is not None:
            cls_attn = cls_attn.to(x.dtype)
    return o, cls_attn


def attention_forward(m, x, policy=None, return_cls_attn=False):
    """Attention.forward (dynamic_vit.py:216-236 / default_dynamic_vit.py:201-216)."""
    o, cls_attn = attention_pre_proj(m, x, policy, return_cls_attn)
    o = m.proj_drop(ops.linear_train(m.proj, o))
    return (o, cls_attn) if return_cls_attn else o


def _is_plain_ln(n):
    return isinstance(n, torch.nn.LayerNorm) and n.elementwise_affine and n.bias is not None


def _drop_off(d, training):
    return isinstance(d, torch.nn.Identity) or (isinstance(d, torch.nn.Dropout) and (d.p == 0 or not training))


def _fusable(m, x, *extra):
    """The carried-residual inference path applies when no gradient is needed and the norms are plain LayerNorms."""
    return (not _needs_grad(x, *extra, m.norm1.weight if hasattr(m.norm1, "weight") else None)
            and x.is_cuda and _d2s_float(x) and _ln_rows_ok(x) and _is_plain_ln(m.norm1) and _is_plain_ln(m.norm2)
            and isinstance(m.drop_path, torch.nn.Identity) and _drop_off(m.attn.proj_drop, m.training))


def _train_fusable(m, x, y=None):
    """The training path with fused residual adds applies: CUDA, plain LayerNorms on rows the d2s LayerNorm kernels take, no
    stochastic depth, and a residual stream of one dtype."""
    return (_FUSED_ADD_LN_TRAIN and x.is_cuda and _d2s_float(x) and (y is None or y.dtype == x.dtype)
            and _is_plain_ln(m.norm1) and _is_plain_ln(m.norm2) and x.shape[-1] % 8 == 0 and x.shape[-1] <= 768
            and isinstance(m.drop_path, torch.nn.Identity) and isinstance(m.mlp, torch.nn.Module))


def _mlp_is_plain(m, h):
    return (isinstance(m.act, torch.nn.GELU) and getattr(m.act, "approximate", "none") == "none"
            and isinstance(m.fc1, torch.nn.Linear) and isinstance(m.fc2, torch.nn.Linear)
            and not _needs_grad(h, m.fc1.weight) and _drop_off(m.drop, m.training))


def mlp_hidden(m, h):
    """act(fc1(h)) of Mlp.forward (dynamic_vit.py:159-175) for inference: the tcgen05 GEMM with the exact-erf GELU in its
    epilogue when the shapes allow, else cuBLAS + the in-place d2s GELU kernel."""
    if (_FUSED_PAIR and h.dtype == torch.bfloat16 and m.fc1.weight.dtype == torch.bfloat16 and m.fc1.out_features % 256 == 0
            and m.fc1.out_features <= 4096 and m.fc1.in_features % 64 == 0):
        return ops.linear_act(h, m.fc1.weight, m.fc1.bias, ops.ACT_GELU)
    u = m.fc1(h)
    ops.bias_act_(u, None, ops.ACT_GELU)
    return u


def mlp_forward(m, h):
    """Mlp.forward (dynamic_vit.py:159-175) for inference."""
    if _mlp_is_plain(m, h):
        return m.fc2(mlp_hidden(m, h))
    return m(h)


def _mlp_fused_ok(m, h, x):
    """The one-kernel MLP applies: bf16, D == 384 (whole rows in one CTA's TMEM next to the hidden chunks), 4D hidden."""
    return (_FUSED_MLP and _FUSED_PAIR and h.dtype == torch.bfloat16 and x.dtype == torch.bfloat16
            and m.fc1.weight.dtype == torch.bfloat16 and m.fc1.in_features == 384 and m.fc2.out_features == 384
            and m.fc1.out_features % 128 == 0 and 128 <= m.fc1.out_features <= 2048 and h.shape == x.shape)


def _pair_ok(lin, a, x):
    """The CTA-pair GEMM with residual + LayerNorm epilogue applies: bf16, whole rows stay in one CTA (D in {192, 384}: in its
    TMEM; D = 768, DeiT-B: as two 384-column halves)."""
    return (_FUSED_PAIR and isinstance(lin, torch.nn.Linear) and a.dtype == torch.bfloat16 and x.dtype == torch.bfloat16
            and lin.weight.dtype == torch.bfloat16 and lin.out_features in (192, 384, 768) and lin.in_features % 64 == 0
            and x.shape[-1] == lin.out_features and a.shape[:-1] == x.shape[:-1])


def norm_forward(n, x, row0=0):
    """A model LayerNorm on the training path: the d2s forward/backward pair when it applies (plain LayerNorm on a CUDA
    tensor whose rows are multiples of 8 elements), torch otherwise.  row0: normalise x[:, row0:] (read in place by the kernel)."""
    if _is_plain_ln(n) and x.is_cuda and _d2s_float(x) and x.shape[-1] % 8 == 0 \
            and x.shape[-1] <= 768 and len(n.normalized_shape) == 1:
        return ops.layer_norm(x, n.weight, n.bias, n.eps, row0=row0)
    return n(x[:, row0:] if row0 else x)


def block_forward(m, x, policy=None, return_cls_attn=False):
    """Block.forward (dynamic_vit.py:263-283)."""
    if _fusable(m, x, policy):
        st = _Stream(x)
        cls_attn = st.block(m, policy, return_cls_attn)
        x = st.value()
        return (x, cls_attn) if return_cls_attn else x
    if return_cls_attn:
        y, cls_attn = attention_forward(m.attn, norm_forward(m.norm1, x), policy=policy, return_cls_attn=True)
        x = x + m.drop_path(y)
        x = x + m.drop_path(m.mlp(norm_forward(m.norm2, x)))
        return x, cls_attn
    x = x + m.drop_path(attention_forward(m.attn, norm_forward(m.norm1, x), policy=policy))
    return x + m.drop_path(m.mlp(norm_forward(m.norm2, x)))


class _LazyNorm:
    """norm(x) that has not been materialised: x is the summed residual stream, `stats` (M,2) f32 its per-row (mean, rstd) as the
    kernel that produced x wrote them (ops.linear_residual_ln(want_stats=True)).  The one-kernel MLP applies the LayerNorm to
    its input tile in shared memory (ops.mlp_residual_ln(in_stats=...)): the normalised copy -- a quarter of the proj + residual +
    LayerNorm kernel's traffic -- is never written or read.  Any other consumer materialises what it needs."""

    def __init__(self, x, stats, norm, row0=0):
        # row0 > 0: the norm is taken over x[:, row0:] (the predictors' input norm); stats still cover every row of x
        self.x, self.stats, self.norm, self.row0 = x, stats, norm, row0
        self.dtype, self.shape, self.is_cuda, self.requires_grad = x.dtype, x.shape, x.is_cuda, False

    def value(self):
        n = self.norm
        return ops.add_layernorm(self.x, None, n.weight, n.bias, n.eps, norm_row0=self.row0, want_sum=False)[1]

    def cls_rows(self):
        n = self.norm
        if self.x.dtype == torch.bfloat16 and self.x.is_contiguous() and self.x.dim() == 3:
            return ops.layernorm_from_stats(self.x, self.stats, n.weight, n.bias)     # same bits as the normalised copy would hold
        return ops.add_layernorm(self.x[:, :1], None, n.weight, n.bias, n.eps, want_sum=False)[1]


def _norm_value(h):
    return h.value() if isinstance(h, _LazyNorm) else h


class _Stream:
    """Residual stream of the model-level inference loops: x plus a pending branch (x + branch is the value the reference
    holds in `x`).  The branch is either a tensor y or a deferred Linear `lin = (a, module)` (attn.proj / mlp.fc2), so
    that the next consumer can run it as ONE kernel with the residual add and its LayerNorm (ops.linear_residual_ln).
    Falls back to plain Block.forward when the fused path does not apply.
    Padded batches (threshold inference): `lens` (B) int32 on the device counts each image's valid tokens (CLS included) of the
    stream's T rows, None when every image has all T.  Rows lens[b].. are pad rows: the variable-length gather writes them as zeros,
    later kernels keep them finite and no valid row depends on them (attention masks them; everything else works row by row)."""

    def __init__(self, x, asm=None):
        # asm = (patches, cls_token, pos_embed): the token assembly itself is deferred, so that it runs fused with the first
        # block's norm1 (ops.assemble_layernorm); any other access to .x materialises it with the plain assembly kernel
        self._x, self._asm = x, asm
        self.y, self.lin, self.mlp, self.gidx = None, None, None, None
        self.gcount, self.lens = None, None

    @property
    def x(self):
        if self._asm is not None:
            (patches, cls, pos), self._asm = self._asm, None
            self._x = ops.assemble_tokens(patches, cls, pos)
        return self._x

    @x.setter
    def x(self, value):
        self._x, self._asm = value, None

    def _probe(self):
        """A tensor with the stream's device / dtype / gradient status, without materialising a deferred assembly."""
        return self._asm[0] if self._asm is not None else self._x

    @property
    def shape(self):
        if self._asm is not None:
            B, N, D = self._asm[0].shape
            return torch.Size((B, N + 1, D))
        return self._x.shape

    def gather(self, x, kept, counts=None):
        """The pruning stage's kept-token gather (default_dynamic_vit.py:464-468, dynamic_vit.py:907-912), deferred so that it
        runs fused with the next block's norm1 (ops.gather_layernorm).  counts (B) int32: image b keeps kept[b, :counts[b]] (the
        threshold inference, dynamic_vit.py:954-960); the stream becomes a padded batch of lengths counts + 1."""
        self.x, self.y, self.lin, self.mlp, self.gidx = x, None, None, None, kept
        self.gcount, self.lens = counts, (None if counts is None else counts + 1)

    def _flush_gather(self):
        if self.gidx is not None:
            if self.gcount is not None:
                raise RuntimeError("the variable-length gather runs fused with the next block's norm1 (ops.gather_layernorm): "
                                   "the block after a threshold stage must take the fused inference path")
            self.x, self.gidx = ops.gather_tokens(self.x, self.gidx, prepend_cls=True), None

    def _flush_lin(self):
        self._flush_gather()
        if self.mlp is not None:                       # deferred whole MLP (h, module): its fc2 becomes the deferred Linear
            h, m = self.mlp
            self.lin, self.mlp = (mlp_hidden(m, _norm_value(h)), m.fc2), None
        if self.lin is not None:
            a, lin = self.lin
            self.y, self.lin = lin(a), None

    def value(self):
        self._flush_lin()
        if self.y is not None:
            self.x, self.y = self.x + self.y, None
        return self.x

    def _sum_norm(self, norm, row0=0, lazy=False):
        """(x + branch, norm((x + branch)[:, row0:])); leaves the stream holding the summed x.
        lazy: the caller's only consumer of the norm is the one-kernel MLP; when the branch is a deferred Linear the second result
        is then a _LazyNorm (statistics instead of the normalised tensor)."""
        if self._asm is not None and row0 == 0 and self.y is None and self.lin is None and self.mlp is None and self.gidx is None:
            (patches, cls, pos), self._asm = self._asm, None
            if lazy and patches.dtype == torch.bfloat16:
                self._x, st = ops.assemble_layernorm(patches, cls, pos, norm.weight, norm.bias, norm.eps, want_stats=True)
                return self._x, _LazyNorm(self._x, st, norm)
            self._x, h = ops.assemble_layernorm(patches, cls, pos, norm.weight, norm.bias, norm.eps)
            return self._x, h
        if self.gidx is not None:
            if row0 == 0 and self.x.dtype in (torch.float32, torch.bfloat16):
                (x, kept, counts), self.gidx, self.gcount = (self.x, self.gidx, self.gcount), None, None
                if lazy and x.dtype == torch.bfloat16:
                    self.x, st = ops.gather_layernorm(x, kept, norm.weight, norm.bias, norm.eps, want_stats=True, counts=counts)
                    return self.x, _LazyNorm(self.x, st, norm)
                self.x, h = ops.gather_layernorm(x, kept, norm.weight, norm.bias, norm.eps, counts=counts)
                return self.x, h
            self._flush_gather()
        if self.mlp is not None:
            h, m = self.mlp
            if _mlp_fused_ok(m, h, self.x):
                self.mlp = None
                if isinstance(h, _LazyNorm) and h.x is self.x and lazy:
                    # ... and the NEXT norm handed on as statistics too (its only reader is the qkv GEMM)
                    self.x, st = ops.mlp_residual_ln(None, m.fc1.weight, m.fc1.bias, m.fc2.weight, m.fc2.bias, self.x, eps=norm.eps,
                                                     want_norm=False, in_stats=h.stats, in_ln_weight=h.norm.weight,
                                                     in_ln_bias=h.norm.bias, want_stats=True)
                    return self.x, _LazyNorm(self.x, st, norm, row0)
                if isinstance(h, _LazyNorm) and h.x is self.x:      # norm2 applied inside the kernel, from its statistics
                    self.x, hn = ops.mlp_residual_ln(None, m.fc1.weight, m.fc1.bias, m.fc2.weight, m.fc2.bias, self.x,
                                                     norm.weight, norm.bias, norm.eps, norm_row0=row0, in_stats=h.stats,
                                                     in_ln_weight=h.norm.weight, in_ln_bias=h.norm.bias)
                else:
                    self.x, hn = ops.mlp_residual_ln(_norm_value(h), m.fc1.weight, m.fc1.bias, m.fc2.weight, m.fc2.bias, self.x,
                                                     norm.weight, norm.bias, norm.eps, norm_row0=row0)
                return self.x, hn
            else:
                self.lin, self.mlp = (mlp_hidden(m, _norm_value(h)), m.fc2), None
        if self.lin is not None and _pair_ok(self.lin[1], self.lin[0], self.x):
            (a, lin), self.lin = self.lin, None
            if row0 == 0 and lazy:
                self.x, st = ops.linear_residual_ln(a, lin.weight, lin.bias, self.x, eps=norm.eps, want_norm=False, want_stats=True)
                return self.x, _LazyNorm(self.x, st, norm)
            if row0 == 0:
                self.x, h = ops.linear_residual_ln(a, lin.weight, lin.bias, self.x, norm.weight, norm.bias, norm.eps)
                return self.x, h
            self.x, _ = ops.linear_residual_ln(a, lin.weight, lin.bias, self.x, want_norm=False)
        self._flush_lin()
        self.x, h = ops.add_layernorm(self.x, self.y, norm.weight, norm.bias, norm.eps, norm_row0=row0)
        self.y = None
        return self.x, h

    def _sum_norm_train(self, norm):
        """Training form of _sum_norm: (x + y, norm(x + y)) with autograd; one kernel forward, one backward."""
        self._flush_lin()
        if self.y is None:
            return self.x, norm_forward(norm, self.x)
        self.x, h = ops.add_layer_norm_train(self.x, self.y, norm.weight, norm.bias, norm.eps)
        self.y = None
        return self.x, h

    def _block_train(self, blk, policy, return_cls_attn):
        """Block.forward (dynamic_vit.py:263-283) under autograd with every residual add folded into the LayerNorm that follows
        it (the second add of a block into the NEXT block's norm1 through the pending branch y)."""
        _, h = self._sum_norm_train(blk.norm1)
        o, cls_attn = attention_pre_proj(blk.attn, h, policy, return_cls_attn)
        self.y = blk.attn.proj_drop(ops.linear_train(blk.attn.proj, o))
        _, h = self._sum_norm_train(blk.norm2)
        self.y = blk.mlp(h)
        return cls_attn

    def block(self, blk, policy=None, return_cls_attn=False):
        """Inference form of Block.forward (dynamic_vit.py:263-283): every residual add is folded into the LayerNorm that
        follows it, and the Linear that produced the branch into the same kernel when it can be."""
        if not _fusable(blk, self._probe(), policy):
            self._flush_gather()
        if _fusable(blk, self._probe(), policy):
            # norm1 is only ever read by this block's qkv projection
            lazy1 = (_LAZY_NORM1 and _is_plain_ln(blk.norm1) and blk.norm1.weight.dtype == torch.bfloat16
                     and _qkv_pair_ok(blk.attn.qkv, self._probe()))
            _, h = self._sum_norm(blk.norm1, lazy=lazy1)
            o, cls_attn = attention_pre_proj(blk.attn, h, policy, return_cls_attn, lens=self.lens)
            self.lin = (o, blk.attn.proj)
            # norm2 is only ever read by this block's MLP: when that MLP runs as the one kernel, hand it the statistics
            lazy = (_LAZY_NORM2 and _mlp_is_plain(blk.mlp, o) and _mlp_fused_ok(blk.mlp, o, o) and o.shape[-1] == 384
                    and _is_plain_ln(blk.norm2) and blk.norm2.weight.dtype == torch.bfloat16)
            _, h = self._sum_norm(blk.norm2, lazy=lazy)
            if _mlp_is_plain(blk.mlp, h):
                self.mlp = (h, blk.mlp)                  # deferred: fused with the residual add and the next LayerNorm
            else:
                self.y = blk.mlp(_norm_value(h))
            return cls_attn
        if self.lens is not None:
            raise RuntimeError("a padded (variable-length) batch runs on the fused inference path only: CUDA, float32 / bfloat16, "
                               "plain LayerNorms, no stochastic depth or active dropout")
        if _train_fusable(blk, self.x, self.y):
            return self._block_train(blk, policy, return_cls_attn)
        out = block_forward(blk, self.value(), policy, return_cls_attn)
        if return_cls_attn:
            self.x, cls_attn = out
            return cls_attn
        self.x = out
        return None

    def normed(self, norm, row0=0, rows=None, lazy=False):
        """(x + y, norm((x + y)[:, row0:])) with the add folded in; leaves the stream holding the summed x.
        lazy: the caller can take a _LazyNorm (row statistics; it applies the norm inside its first GEMM)."""
        if (_is_plain_ln(norm) and self.x.is_cuda and _d2s_float(self.x) and _ln_rows_ok(self.x)
                and not _needs_grad(self.x, self.y, norm.weight)):
            return self._sum_norm(norm, row0, lazy=lazy and row0 > 0 and self.mlp is not None)
        x = self.value()
        return x, norm(x[:, row0:])

    def cls_normed(self, norm):
        """norm(x + y)[:, 0]: only the CLS row (what the eval heads consume)."""
        self._flush_gather()
        if (_is_plain_ln(norm) and self.x.is_cuda and _d2s_float(self.x) and _ln_rows_ok(self.x)
                and not _needs_grad(self.x, self.y, norm.weight)):
            if self.mlp is not None:                     # the last MLP is only needed for the CLS rows
                h, m = self.mlp
                h0 = h.cls_rows() if isinstance(h, _LazyNorm) else h[:, :1].contiguous()
                y0 = m.fc2(mlp_hidden(m, h0))
            elif self.lin is not None:                   # the last fc2 is only needed for the CLS rows
                a, lin = self.lin
                y0 = lin(a[:, :1])
            else:
                y0 = None if self.y is None else self.y[:, :1].contiguous()
            _, h = ops.add_layernorm(self.x[:, :1], y0, norm.weight, norm.bias, norm.eps, want_sum=False)
            return h[:, 0]
        return norm(self.value())[:, 0]


def _seq_forward(layers, h, row0=0):
    """A predictor nn.Sequential on the training path: LayerNorms on the d2s forward/backward kernels, Linear layers through
    ops.linear_train (bias gradient by the column-sum kernel, fp32 weight gradient straight from the GEMM) and Linear -> GELU
    pairs as one autograd node (ops.linear_gelu_train).  Each falls back to the module itself when it does not apply.
    row0: the sequence is applied to h[:, row0:]; a leading LayerNorm reads those rows in place instead of a slice copy."""
    layers = list(layers)
    i = 0
    if row0:
        if layers and isinstance(layers[0], torch.nn.LayerNorm):
            h = norm_forward(layers[0], h, row0=row0)
            i = 1
        else:
            h = h[:, row0:]
    while i < len(layers):
        layer = layers[i]
        if isinstance(layer, torch.nn.LayerNorm):
            h = norm_forward(layer, h)
        elif isinstance(layer, torch.nn.Linear) and h.is_cuda:
            nxt = layers[i + 1] if i + 1 < len(layers) else None
            if isinstance(nxt, torch.nn.GELU):
                h = ops.linear_gelu_train(layer, nxt, h)
                i += 1
            else:
                h = ops.linear_train(layer, h)
        else:
            h = layer(h)
        i += 1
    return h


# ---- Variant A predictor (default_dynamic_vit.py:304-330) ------------------------------------------
def predictor_a_hidden(m, x, policy, normed=None, row0=0):
    """`normed`: in_conv's LayerNorm already applied (by the fused add+LayerNorm kernel).  row0: the predictor sees x[:, row0:]."""
    h = _seq_forward(m.in_conv, x, row0=row0) if normed is None else _seq_forward(list(m.in_conv)[1:], normed)
    B, N, C = h.shape
    half = C // 2
    if ops.pool_concat_train_ok(h) and policy is not None and policy.is_cuda:
        h = ops.pool_concat_train(h, policy)          # slice, multiply, sum, divide, expand, cat: one kernel each way
    else:
        pooled = (h[:, :, half:] * policy).sum(dim=1, keepdim=True) / torch.sum(policy, dim=1, keepdim=True)
        h = torch.cat([h[:, :, :half], pooled.expand(B, N, half)], dim=-1)
    return _seq_forward(list(m.out_conv)[:4], h)      # Linear, GELU, Linear, GELU


def _tail_ok(h):
    """Hidden widths the fused tail kernels take (d2s_score_tail_a / _b): multiples of 8 in [8, 1024], on CUDA."""
    return h.is_cuda and h.shape[-1] % 8 == 0 and 8 <= h.shape[-1] <= 1024


def predictor_a_forward(m, x, policy, row0=0):
    h = predictor_a_hidden(m, x, policy, row0=row0)
    lin = m.out_conv[4]
    if _needs_grad(h, lin.weight) or not _tail_ok(h):
        return m.out_conv[5](lin(h))
    logp, _ = ops.score_tail_a(h, lin.weight, lin.bias, k=0)
    return logp.to(x.dtype)


def _predictor_a_fusable(m):
    ic, oc = list(m.in_conv), list(m.out_conv)
    G, L = torch.nn.GELU, torch.nn.Linear
    return (len(ic) == 3 and len(oc) == 6 and _is_plain_ln(ic[0]) and isinstance(ic[1], L) and isinstance(ic[2], G)
            and isinstance(oc[0], L) and isinstance(oc[1], G) and isinstance(oc[2], L) and isinstance(oc[3], G)
            and isinstance(oc[4], L) and getattr(ic[2], "approximate", "none") == "none"
            and oc[0].in_features == ic[1].out_features and ic[1].out_features % 16 == 0
            and oc[4].in_features % 8 == 0 and 8 <= oc[4].in_features <= 1024)


def _predictor_a_gemm_ok(m, x):
    """in_conv's Linear(D,D) + GELU runs on the pair GEMM with its input LayerNorm applied inside (bf16, D = 384)."""
    l1 = m.in_conv[1]
    return (_PRED_FUSED and _FUSED_PAIR and _predictor_a_fusable(m) and x.is_cuda and x.dtype == torch.bfloat16
            and l1.weight.dtype == torch.bfloat16 and l1.in_features == 384 and l1.out_features == 384 and l1.bias is not None
            and m.in_conv[0].weight.dtype == torch.bfloat16)


def predictor_a_select(m, normed, prev, k):
    """Inference form of PredictorLG.forward + selection (default_dynamic_vit.py:324-330, :461-467) without the
    GELU / multiply / reduce / expand / concat passes: `normed` = in_conv's LayerNorm output (from the fused
    add+LayerNorm), `prev` (B,N) fp32 keep decisions of the previous stage or None (all ones).
    Returns (log-probs (B,N,2) fp32, kept (B,k) int64 in descending-score order, prev gathered at kept (B,k) fp32)."""
    l1, l0, l2, lin = m.in_conv[1], m.out_conv[0], m.out_conv[2], m.out_conv[4]
    half = l0.in_features // 2
    tail_ok = _PRED_FUSED and l0.bias is not None and l2.bias is not None and lin.bias is not None
    if isinstance(normed, _LazyNorm):
        if tail_ok and _predictor_a_gemm_ok(m, normed.x):
            # in_conv's LayerNorm was not materialised: Linear(D,D) + GELU normalises its resident input rows from the row statistics
            # (over every token of x: the GEMM's rows must be dense; the CLS rows' results are simply not read)
            ln = m.in_conv[0]
            g = ops.linear_act(normed.x, l1.weight, l1.bias, ops.ACT_GELU, in_stats=normed.stats, in_ln_weight=ln.weight,
                               in_ln_bias=ln.bias)[:, normed.row0:]
            if ops.predictor_a_tail_ok(g[:, :, :half], l0.weight, l2.weight, lin.weight):
                _, pooled = ops.pool_act(g, prev, ops.ACT_NONE, want_local=False)
                per_image = F.linear(pooled, l0.weight[:, half:], l0.bias)
                return ops.predictor_a_tail(g[:, :, :half], per_image, l0.weight, l2.weight, l2.bias, lin.weight, lin.bias, k, prev=prev)
        normed = normed.value()
    if (tail_ok and _FUSED_PAIR and normed.dtype == torch.bfloat16 and l1.weight.dtype == torch.bfloat16
            and l1.out_features % 192 == 0 and l1.in_features % 64 == 0
            and ops.predictor_a_tail_ok(normed[:, :, :half], l0.weight, l2.weight, lin.weight)):
        # Linear(D,D) + GELU as one tcgen05 GEMM; its local half is read in place by the tail kernel, its global half only pooled
        g = ops.linear_act(normed, l1.weight, l1.bias, ops.ACT_GELU)
        _, pooled = ops.pool_act(g, prev, ops.ACT_NONE, want_local=False)
        per_image = F.linear(pooled, l0.weight[:, half:], l0.bias)
        return ops.predictor_a_tail(g[:, :, :half], per_image, l0.weight, l2.weight, l2.bias, lin.weight, lin.bias, k, prev=prev)
    z = l1(normed)                                               # Linear(D,D) + bias (cuBLAS)
    local, pooled = ops.pool_act(z, prev, ops.ACT_GELU)          # GELU + policy-weighted mean pool, one pass
    # Linear(cat(local, pooled)) = local @ W[:, :half]^T + (pooled @ W[:, half:]^T + b)
    per_image = F.linear(pooled, l0.weight[:, half:], l0.bias)   # (B, D/2)
    if tail_ok and ops.predictor_a_tail_ok(local, l0.weight, l2.weight, lin.weight):
        # split Linear + GELU, Linear + GELU, Linear(., 2), log-softmax and the selection as one tcgen05 kernel
        return ops.predictor_a_tail(local, per_image, l0.weight, l2.weight, l2.bias, lin.weight, lin.bias, k, prev=prev)
    u = F.linear(local, l0.weight[:, :half])
    ops.bias_act_(u, per_image, ops.ACT_GELU)
    z2 = m.out_conv[2](u)                                        # Linear(D/2, D/4) + bias; its GELU is applied by the tail
    lin = m.out_conv[4]
    return ops.score_tail_a(z2, lin.weight, lin.bias, k=k, prev=prev, act_input=ops.ACT_GELU, want_prev_kept=True)


# ---- Variant B predictor (dynamic_vit.py:370-560) --------------------------------------------------
def _predictor_b_tail_parts(m):
    layers = list(m.out_conv)
    # ..., norm, Linear(C,1), Flatten
    return layers[:-3], layers[-3], layers[-2]


def predictor_b_hidden(m, x, normed=None):
    h = _seq_forward(m.in_conv, x) if normed is None else m.in_conv[2](m.in_conv[1](normed))
    B, N, C = h.shape
    half = C // 2
    if ops.pool_concat_train_ok(h) and torch.is_grad_enabled() and h.requires_grad:
        h = ops.pool_concat_train(h)
    else:
        pooled = torch.mean(h[:, :, half:], dim=1, keepdim=True)
        h = torch.cat([h[:, :, :half], pooled.expand(B, N, half)], dim=-1)
    body, norm, lin = _predictor_b_tail_parts(m)
    return _seq_forward(body, h), norm, lin


def _act_code(a):
    if isinstance(a, torch.nn.ReLU):
        return ops.ACT_RELU
    if isinstance(a, torch.nn.GELU) and getattr(a, "approximate", "none") == "none":
        return ops.ACT_GELU
    return None


def _ln_ok(n, dtype):
    return _is_plain_ln(n) and n.normalized_shape[0] % 8 == 0 and n.normalized_shape[0] <= (1536 if dtype == torch.bfloat16 else 768)


def _predictor_b_fusable(m, dtype):
    ic, oc = list(m.in_conv), list(m.out_conv)
    if len(ic) != 3 or len(oc) < 3 or len(oc) % 3 != 0 or not m.topk_selection:
        return False
    if not (_is_plain_ln(ic[0]) and isinstance(ic[1], torch.nn.Linear) and _act_code(ic[2]) is not None):
        return False
    for i in range(0, len(oc) - 3, 3):
        if not (_ln_ok(oc[i], dtype) and isinstance(oc[i + 1], torch.nn.Linear) and _act_code(oc[i + 2]) is not None):
            return False
    return (_is_plain_ln(oc[-3]) and isinstance(oc[-2], torch.nn.Linear) and oc[-2].out_features == 1
            and oc[-2].in_features % 8 == 0 and 8 <= oc[-2].in_features <= 1024 and ic[1].out_features % 16 == 0)


def _linear_act(x, lin, act):
    """act(lin(x)): the tcgen05 GEMM with the activation in its epilogue when the shape allows, else cuBLAS + in-place act."""
    if (_FUSED_PAIR and x.dtype == torch.bfloat16 and lin.weight.dtype == torch.bfloat16
            and (lin.out_features % 256 == 0 or lin.out_features % 192 == 0) and 192 <= lin.out_features <= 4096
            and lin.in_features % 64 == 0):
        return ops.linear_act(x, lin.weight, lin.bias, act)
    u = lin(x)
    return ops.bias_act_(u, None, act)


def predictor_b_select_fused(m, normed, k):
    """Inference form of Variant B's PredictorLG.forward + selection (dynamic_vit.py:536-560, :858-862) for the LayerNorm
    architectures: Linear+activation as one GEMM (or cuBLAS + in-place activation), the mean-pool / expand / concat as
    one in-place kernel, every inner LayerNorm as the d2s kernel, LayerNorm+Linear(.,1)+softmax+top-k in the tail."""
    z = _linear_act(normed, m.in_conv[1], _act_code(m.in_conv[2]))
    h = ops.pool_concat_(z)
    oc = list(m.out_conv)
    for i in range(0, len(oc) - 3, 3):
        _, hn = ops.add_layernorm(h, None, oc[i].weight, oc[i].bias, oc[i].eps, want_sum=False)
        h = _linear_act(hn, oc[i + 1], _act_code(oc[i + 2]))
    norm, lin = oc[-3], oc[-2]
    prob_mode = ops.PROB_SOFTMAX if m.loss_type in ["kl_div", "mse"] else ops.PROB_SIGMOID
    scores, probs, kept, dropped = ops.score_tail_b(h, norm.weight, norm.bias, lin.weight, lin.bias, k, norm.eps, prob_mode)
    return scores.to(normed.dtype), probs.to(normed.dtype), kept, dropped


def predictor_b_forward(m, x, policy=None, current_sigma=0.0005, cls_attn=None, k_select=None, normed=None):
    """Returns (scores, keep_probs) like the reference; with k_select also (kept, dropped) from the fused
    tail kernel.  Like the reference, only the topk_selection=True configuration is defined (:537)."""
    if not m.topk_selection:
        return None
    h, norm, lin = predictor_b_hidden(m, x, normed)
    prob_mode = ops.PROB_SOFTMAX if m.loss_type in ["kl_div", "mse"] else ops.PROB_SIGMOID
    if _needs_grad(h, lin.weight) or not _tail_ok(h):
        scores = lin(norm_forward(norm, h)).flatten(-2, -1)
        probs = F.softmax(scores, dim=-1) if prob_mode == ops.PROB_SOFTMAX else torch.sigmoid(scores)
        if k_select is None:
            return scores, probs
        kept, dropped = ops.select_topk(probs, k_select, ops.ORDER_INDEX_ASC)
        return scores, probs, kept, dropped
    if isinstance(norm, torch.nn.LayerNorm):
        ln_w, ln_b, ln_eps = norm.weight, norm.bias, norm.eps
    else:  # BatchNormLayer: normalise upstream, the kernel then skips its LayerNorm
        h, ln_w, ln_b, ln_eps = norm(h), None, None, 0.0
    scores, probs, kept, dropped = ops.score_tail_b(h, ln_w, ln_b, lin.weight, lin.bias, k_select or 0, ln_eps,
                                                    prob_mode, select=k_select is not None)
    out_dtype = x.dtype if x is not None else normed.dtype
    scores, probs = scores.to(out_dtype), probs.to(out_dtype)
    if k_select is None:
        return scores, probs
    return scores, probs, kept, dropped


def predictor_b_varlen(m, x, n):
    """Variant B's PredictorLG.forward at inference (dynamic_vit.py:536-554) over a padded batch: x (B,Nmax,D) spatial tokens of
    which image b has n[b] (int32, device).  The mean pool and the softmax run over each image's valid rows only (the varlen pool
    and tail kernels); every other layer works row by row.  Returns (scores, keep probabilities) (B,Nmax); pad entries are -inf / 0."""
    if not m.topk_selection:
        raise RuntimeError("PredictorLG is only defined for topk_selection=True (dynamic_vit.py:537)")
    h = ops.pool_concat_varlen_(_seq_forward(m.in_conv, x).contiguous(), n)
    body, norm, lin = _predictor_b_tail_parts(m)
    h = _seq_forward(body, h)
    if not _tail_ok(h):
        raise RuntimeError(f"predictor width {h.shape[-1]} is outside the d2s tail kernel (multiples of 8 in [8, 1024])")
    prob_mode = ops.PROB_SOFTMAX if m.loss_type in ["kl_div", "mse"] else ops.PROB_SIGMOID
    if isinstance(norm, torch.nn.LayerNorm):
        ln_w, ln_b, ln_eps = norm.weight, norm.bias, norm.eps
    else:  # BatchNormLayer (eval: a per-channel affine map, row by row): normalise upstream, the kernel then skips its LayerNorm
        h, ln_w, ln_b, ln_eps = norm(h), None, None, 0.0
    scores, probs = ops.score_tail_b_varlen(h, n, ln_w, ln_b, lin.weight, lin.bias, ln_eps, prob_mode)
    return scores.to(x.dtype), probs.to(x.dtype)


# ---- model forwards ------------------------------------------------------------------------------------
def _embed_stream(model, img):
    """The residual stream after patch embedding; on the inference path the token assembly is left pending (fused with the first
    block's norm1)."""
    patches = patch_embed_forward(model.patch_embed, img)
    if (patches.is_cuda and not _needs_grad(patches, model.cls_token, model.pos_embed) and isinstance(model.pos_drop, torch.nn.Dropout)
            and (model.pos_drop.p == 0 or not model.training) and model.pos_embed.shape[1] == patches.shape[1] + 1
            and patches.dtype in (torch.float32, torch.bfloat16) and patches.shape[-1] % 8 == 0
            and patches.shape[-1] <= (1536 if patches.dtype == torch.bfloat16 else 768)):
        return _Stream(None, asm=(patches, model.cls_token, model.pos_embed))
    B = patches.shape[0]
    x = torch.cat((model.cls_token.to(patches.dtype).expand(B, -1, -1), patches), dim=1)
    return _Stream(model.pos_drop(x + model.pos_embed.to(patches.dtype)))


def _head(model, x):
    # training heads: the final norm keeps torch autocast's fp32 output (the token features go straight into the losses)
    if _is_plain_ln(model.norm) and x.is_cuda and x.shape[-1] % 8 == 0 and x.shape[-1] <= 768 and _d2s_float(x):
        x = ops.layer_norm(x, model.norm.weight, model.norm.bias, model.norm.eps,
                           out_dtype=torch.float32 if torch.is_autocast_enabled("cuda") else None)
    else:
        x = model.norm(x)
    features = x[:, 1:]
    return model.head(model.pre_logits(x[:, 0])), features


def draw_gumbel(like):
    """Same draw as torch F.gumbel_softmax: -log(Exponential(1))."""
    return -torch.empty_like(like, memory_format=torch.legacy_contiguous_format).exponential_().log()


def _pred_ln(pred):
    ln = pred.in_conv[0]
    return ln if _is_plain_ln(ln) else None


def variant_a_forward(model, img):
    """DefaultVisionTransformerDiffPruning.forward (default_dynamic_vit.py:435-487).
    Injected Gumbel noise for parity runs: set model._d2s_gumbels = [tensor (B,196,2) per stage]."""
    st = _embed_stream(model, img)
    B = st.shape[0]
    dt, dev = st._probe().dtype, st._probe().device
    p_count = 0
    out_pred_prob = []
    prev_decision = torch.ones(B, INIT_N, 1, dtype=dt, device=dev)
    policy = torch.ones(B, INIT_N + 1, 1, dtype=dt, device=dev)
    injected = getattr(model, "_d2s_gumbels", None)
    model.kept_token_indices = []
    prev_f32 = None                                  # eval fast path: (B,N) fp32 decisions, None = all ones
    for i, blk in enumerate(model.blocks):
        if i in model.pruning_loc:
            pred = model.score_predictor[p_count]
            if model.training:
                x = st.value()
                pred_score = predictor_a_forward(pred, x, prev_decision, row0=1).reshape(B, -1, 2)
                g = injected[p_count] if injected is not None else draw_gumbel(pred_score)
                hard = ops.gumbel_keep_decision(pred_score, g, prev_decision)
                out_pred_prob.append(hard.reshape(B, INIT_N))
                policy = torch.cat([torch.ones(B, 1, 1, dtype=hard.dtype, device=hard.device), hard], dim=1)
                st.block(blk, policy=policy)
                prev_decision = hard
            else:
                k = int(INIT_N * model.token_ratio[p_count])
                ln = _pred_ln(pred)
                if (ln is not None and _predictor_a_fusable(pred) and st._probe().is_cuda and _d2s_float(st._probe())
                        and not _needs_grad(st.x, st.y, ln.weight)):
                    # residual add folded into the predictor's LayerNorm over x[:, 1:]; fused predictor body
                    x, hn = st.normed(ln, row0=1, lazy=_LAZY_NORM1 and _predictor_a_gemm_ok(pred, st._probe()))
                    _, keep_policy, prev_f32 = predictor_a_select(pred, hn, prev_f32, k)
                    prev_decision = None                 # materialised on demand below
                else:
                    x = st.value()
                    if prev_decision is None:
                        prev_decision = prev_f32.unsqueeze(-1).to(dt)
                    h = predictor_a_hidden(pred, x[:, 1:], prev_decision)
                    lin = pred.out_conv[4]
                    if _tail_ok(h):
                        _, keep_policy = ops.score_tail_a(h, lin.weight, lin.bias, k=k)
                    else:                                # widths outside the tail kernel: torch tail, d2s selection
                        logp = pred.out_conv[5](lin(h))
                        keep_policy, _ = ops.select_topk(logp[:, :, 0], k, ops.ORDER_SCORE_DESC, want_dropped=False)
                    prev_decision = ops.batch_index_select(prev_decision, keep_policy)
                    prev_f32 = prev_decision.reshape(B, -1).float()
                model.kept_token_indices.append(keep_policy)
                st.gather(x, keep_policy)
                st.block(blk)
            p_count += 1
        else:
            st.block(blk, policy if model.training else None)
    if model.training:
        x, features = _head(model, st.value())
        if model.distill:
            return x, features, prev_decision.detach(), out_pred_prob
        return x, out_pred_prob
    return model.head(model.pre_logits(st.cls_normed(model.norm)))


def variant_b_forward(model, img, stacked_cls_attn_weights=None):
    """VisionTransformerDiffPruning.forward (dynamic_vit.py:814-1015)."""
    if (model.patch_score_threshold is not None and not model.training
            and (_THRESHOLD_INFERENCE or getattr(model, "d2s_threshold_inference", False))):
        # OPT-IN.  The reference's inference branch of this mode cannot run (dynamic_vit.py:936 reads `score`, which is only
        # assigned in a comment at :933, and :947 indexes with a float mask).  What it evidently intends -- the same cumulative-score
        # threshold on pred_score, then a variable-length removal of the dropped tokens, batch size 1 by design
        # (mask_predictor.py:249-254) -- is the equal-count case of the padded-batch forward (forward_varlen)
        return _variant_b_threshold_eval(model, img, ragged=False)
    st = _embed_stream(model, img)
    B, T0, D = st.shape
    dt, dev = st._probe().dtype, st._probe().device
    N = T0 - 1
    p_count = 0
    model.num_kept_tokens = []
    model.cls_attns = []
    model.pred_logits = []
    model.kept_token_indices = []
    model.dropped_token_indices = []
    keep_mask = torch.ones((B, N + 1), dtype=dt, device=dev)
    pred_logits = None
    thr = model.patch_score_threshold
    for i, blk in enumerate(model.blocks):
        if i in model.pruning_loc:
            num_keep_node = int(INIT_N * model.token_ratio[p_count])
            pred = model.score_predictor[p_count]
            if thr is None:
                ln = _pred_ln(pred)
                if (ln is not None and pred.topk_selection and st._probe().is_cuda and _d2s_float(st._probe())
                        and not _needs_grad(st.x, st.y, ln.weight)):
                    x, hn = st.normed(ln, row0=1)
                    if _predictor_b_fusable(pred, hn.dtype):
                        pred_logits, pred_score, kept, dropped = predictor_b_select_fused(pred, hn, num_keep_node)
                    else:
                        pred_logits, pred_score, kept, dropped = predictor_b_forward(pred, None, k_select=num_keep_node, normed=hn)
                else:
                    x = st.value()
                    pred_logits, pred_score, kept, dropped = predictor_b_forward(pred, x[:, 1:], k_select=num_keep_node)
                model.kept_token_indices.append(kept)
                model.dropped_token_indices.append(dropped)
                model.pred_logits.append(pred_logits)
                st.gather(x, kept)
                cls_attn = st.block(blk, return_cls_attn=True)
                model.cls_attns.append(cls_attn[:, :, 1:])
            elif model.training:
                # dynamic keep ratio: cumulative-score threshold -> 0/1 policy (dynamic_vit.py:880-894); sort + cumsum +
                # compare + scatter are one d2s kernel (ops.threshold_select)
                x = st.value()
                pred_logits, pred_score = predictor_b_forward(pred, x[:, 1:])
                if pred_score.is_cuda:
                    spatial_mask, kept_count = ops.threshold_select(pred_score.detach(), thr)
                    model.keep_ratios = kept_count.to(torch.float32) / N
                else:
                    val, idx = torch.sort(pred_score.detach().clone(), stable=True)
                    th = torch.cumsum(val, dim=-1) > thr
                    model.keep_ratios = torch.sum(th, dim=1).detach().clone() / N
                    spatial_mask = torch.zeros((B, N), device=dev, dtype=torch.bool).scatter(1, idx, th)
                model.min_keep_ratio = torch.min(model.keep_ratios).item()
                model.avg_keep_ratio = torch.mean(model.keep_ratios).item()
                model.max_keep_ratio = torch.max(model.keep_ratios).item()
                model.kept_token_indices.append(spatial_mask.unsqueeze(-1).repeat(1, 1, D).flatten())
                model.dropped_token_indices.append(~spatial_mask.unsqueeze(-1).repeat(1, 1, D).flatten())
                keep_mask = torch.cat((torch.ones(B, 1, dtype=dt, device=dev), spatial_mask), dim=1).float()
                st.block(blk, policy=keep_mask.unsqueeze(-1))
            else:
                # the reference's inference branch of this mode reads an undefined name (dynamic_vit.py:936)
                raise NotImplementedError("patch_score_threshold inference is undefined in the reference "
                                          "(vit_models/dynamic_vit.py:936 uses `score` before assignment); "
                                          "set model.d2s_threshold_inference = True (or D2S_THRESHOLD_INFERENCE=1) for the intended behaviour")
            p_count += 1
        else:
            if model.training and thr is not None:
                st.block(blk, policy=keep_mask.unsqueeze(-1))
            else:
                cls_attn = st.block(blk, return_cls_attn=True)
                model.cls_attns.append(cls_attn[:, :, 1:])
    if model.training:
        x, features = _head(model, st.value())
        if thr is not None:
            return x, features, pred_logits, keep_mask[:, 1:]
        return x, features, model.pred_logits, model.kept_token_indices
    logits = model.head(model.pre_logits(st.cls_normed(model.norm)))
    return logits, model.cls_attns, model.pred_logits, model.kept_token_indices


def _variant_b_threshold_eval(model, img, ragged):
    """Inference of the dynamic keep-ratio mode (what dynamic_vit.py:935-960 intends) over a padded batch: at each pruning stage
    the predictor scores the valid tokens, the prefix-sum select kernel picks each image's kept set (ascending, -1 padded), ONE host
    read of the per-image counts sizes the next stage (Tmax = 1 + max count), and the gather of CLS + kept tokens runs fused with
    the block's norm1; the stream then carries per-image lengths that the attention kernel honours.  The pruning block and the
    later ones run without a policy.  ragged=False: forward()'s dense outputs, which need equal counts (batch size 1).
    Returns (logits, cls_attns, pred_logits, kept): cls_attns of the blocks that are not pruning stages (B,H,Tmax_i-1), zero past
    an image's tokens; pred_logits (B,Nmax_s), -inf past them; kept (B,Kmax_s) int64 stage-relative ascending, -1 padded."""
    thr = model.patch_score_threshold
    st = _embed_stream(model, img)
    B, T0, _ = st.shape
    N = T0 - 1
    model.num_kept_tokens = []
    model.cls_attns = []
    model.pred_logits = []
    model.kept_token_indices = []
    model.dropped_token_indices = []
    n = None                                       # valid spatial tokens per image (B) int32 on the device
    p_count = 0
    for i, blk in enumerate(model.blocks):
        if i in model.pruning_loc:
            x = st.value()
            if n is None:
                n = torch.full((B,), x.shape[1] - 1, dtype=torch.int32, device=x.device)
            pred_logits, pred_score = predictor_b_varlen(model.score_predictor[p_count], x[:, 1:], n)
            _, count, kept = ops.threshold_select(pred_score.detach(), thr, want_indices=True, lengths=n)
            counts = count.tolist()                # the stage's one host read: the output shape depends on it
            if not ragged and len(set(counts)) != 1:
                raise RuntimeError(f"patch_score_threshold inference: images keep different token counts {counts}; like the "
                                   "reference's x.flatten()[mask].reshape(B, -1, D) forward() is for batch size 1 here -- "
                                   "model.forward_varlen(x) runs such a batch (padded outputs)")
            model.keep_ratios = count.to(torch.float32) / N
            model.min_keep_ratio, model.max_keep_ratio = min(counts) / N, max(counts) / N
            model.avg_keep_ratio = sum(counts) / len(counts) / N
            kept = kept[:, :max(counts)].contiguous()
            model.kept_token_indices.append(kept)
            model.pred_logits.append(pred_logits)
            st.gather(x, kept, count)
            n = count
            st.block(blk)
            p_count += 1
        else:
            cls_attn = st.block(blk, return_cls_attn=True)
            model.cls_attns.append(cls_attn[:, :, 1:])
    logits = model.head(model.pre_logits(st.cls_normed(model.norm)))
    return logits, model.cls_attns, model.pred_logits, model.kept_token_indices


def variant_b_forward_varlen(model, img):
    """VisionTransformerDiffPruning.forward_varlen: the dynamic keep-ratio inference of a whole batch in which images keep
    different token counts (padded outputs, see _variant_b_threshold_eval)."""
    if model.training:
        raise ValueError("forward_varlen is an inference path: call model.eval() first (training uses the keep-mask policy)")
    if model.patch_score_threshold is None:
        raise ValueError("forward_varlen runs the dynamic keep-ratio mode: the model has no patch_score_threshold")
    return _variant_b_threshold_eval(model, img, ragged=True)


def variant_b_forward_cls_attn(model, img):
    """VisionTransformerDiffPruning.forward_cls_attn (dynamic_vit.py:1018-1033)."""
    st = _embed_stream(model, img)
    final = None
    last = len(model.blocks) - 1
    for i, blk in enumerate(model.blocks):
        final = st.block(blk, return_cls_attn=(i == last))
    return final


_SHADOWS = weakref.WeakKeyDictionary()      # frozen fp32 model -> (weights fingerprint, bf16 copy)


def _frozen_bf16_shadow(model, img):
    """A frozen eval model called under bf16 autocast (the distillation teacher of ddp_training.py:77-81 / train.py:40-42)
    computes in bf16 anyway -- through a cast of every fp32 weight and bias on every call and, here, through the unfused
    fallbacks, because the fused inference kernels take bf16 weights.  Its weights cannot change between steps, so a bf16 copy
    is kept and the call runs on the fused inference path.  The copy is rebuilt when any parameter's storage or version counter
    changes (load_state_dict, .to(), in-place edits through the tensor itself); invalidate_frozen_copies() drops it explicitly.
    Numerics: torch autocast keeps the fp32 residual stream and fp32 LayerNorm / softmax of an fp32 module; the copy computes
    like `model.to(bfloat16)` (bf16 residual stream).  Teacher logits / tokens / CLS rows agree with the per-call-cast path to
    bf16 accuracy (3e-2 of the tensor's max, pinned by tests/test_gpu_models.py::test_frozen_teacher_under_autocast_...).
    Returns None when this does not apply."""
    if not (_FROZEN_BF16 and img.is_cuda and not model.training and torch.is_autocast_enabled("cuda")
            and torch.get_autocast_dtype("cuda") == torch.bfloat16):
        return None
    params = list(model.parameters())
    if not params or any(p.requires_grad or p.dtype != torch.float32 or not p.is_cuda for p in params):
        return None
    # storage + version counter of every parameter and buffer.  Edits that bypass the version counter (`p.data.copy_()`, an EMA
    # teacher updated through .data) are NOT seen: call invalidate_frozen_copies(model) after those.
    fp = hash(tuple((p.data_ptr(), p._version) for p in params + list(model.buffers())))
    hit = _SHADOWS.get(model)
    if hit is None or hit[0] != fp:
        hit = (fp, copy.deepcopy(model).to(torch.bfloat16).eval())
        _SHADOWS[model] = hit
    return hit[1]


def invalidate_frozen_copies(model=None):
    """Drop the cached bf16 copy of `model` (all cached copies when None): the next call under bf16 autocast rebuilds it."""
    if model is None:
        _SHADOWS.clear()
    else:
        _SHADOWS.pop(model, None)


def teacher_forward(model, img, with_cls_attn=True):
    """VisionTransformerTeacher.forward (dynamic_vit.py:1150-1176) / DefaultVisionTransformerTeacher.forward
    (default_dynamic_vit.py:581-598, with_cls_attn=False)."""
    shadow = _frozen_bf16_shadow(model, img)
    if shadow is not None:
        with torch.no_grad():
            return teacher_forward(shadow, img.to(torch.bfloat16), with_cls_attn)
    st = _embed_stream(model, img)
    rows = []
    for blk in model.blocks:
        ca = st.block(blk, return_cls_attn=with_cls_attn)
        if with_cls_attn:
            rows.append(ca.detach())
    _, feature = st.normed(model.norm)
    cls = model.head(model.pre_logits(feature[:, 0]))
    tokens = feature[:, 1:]
    if with_cls_attn:
        return cls, tokens, torch.stack(rows, dim=1)
    return cls, tokens


def teacher_forward_cls_attention(model, img):
    """VisionTransformerTeacher.forward_cls_attention (dynamic_vit.py:1134-1148)."""
    st = _embed_stream(model, img)
    rows = []
    for blk in model.blocks:
        rows.append(st.block(blk, return_cls_attn=True).detach())
    return torch.stack(rows, dim=1)
