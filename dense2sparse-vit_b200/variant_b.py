"""Variant B -- the reference author's Dense2Sparse model (vit_models/dynamic_vit.py): one score per token,
hard top-k with kept tokens in spatial order in both training and inference, CLS-attention rows collected
from every block.  Same class names, constructor arguments, side attributes and state-dict keys."""
import torch
import torch.nn as nn

from . import engine, ops
from .layers import _VitBackbone
from .perturbed_topk import PerturbedTopK

batch_index_select = ops.batch_index_select  # dynamic_vit.py:39-60 (unused there, kept for API parity)


class BatchNormLayer(nn.Module):
    """BatchNorm1d over the channel dim of (B,N,C) tokens (dynamic_vit.py:350-367)."""

    def __init__(self, input_dim=384):
        super().__init__()
        self.bn = nn.BatchNorm1d(input_dim)

    def forward(self, x):
        return self.bn(x.transpose(1, 2)).transpose(1, 2)


def _stage(norm, d_in, d_out, act):
    return [norm(d_in), nn.Linear(d_in, d_out), act]


class PredictorLG(nn.Module):
    """dynamic_vit.py:370-560.  Four architectures (small|large x LayerNorm|BatchNorm) with the reference's
    Sequential indices; forward -> (scores (B,N), keep_probs (B,N)), only defined for topk_selection=True."""

    def __init__(self, embed_dim=384, topk_selection=False, k=None, small_predictor=False,
                 loss_type="kl_div", use_bn=False):
        super().__init__()
        self.small_predictor = small_predictor
        self.k = k
        self.topk_selection = topk_selection
        self.loss_type = loss_type
        self.act = nn.ReLU()
        self.flatten = nn.Flatten(start_dim=-2, end_dim=-1)
        self.softmax = nn.Softmax(dim=-1)
        D = embed_dim
        norm = BatchNormLayer if use_bn else nn.LayerNorm
        if small_predictor:
            act = (lambda: self.act) if use_bn else nn.GELU
            widths = [D, D // 2, D // 4]
            self.in_conv = nn.Sequential(*_stage(norm, D, D, act()))
        else:
            act = lambda: self.act  # noqa: E731  (the reference shares one ReLU instance)
            widths = [4 * D, 2 * D, D, D // 2, D // 4]
            self.in_conv = nn.Sequential(*_stage(norm, D, 4 * D, act()))
        layers = []
        for a, b in zip(widths[:-1], widths[1:]):
            layers += _stage(norm, a, b, act())
        layers += [norm(widths[-1]), nn.Linear(widths[-1], 1), nn.Flatten(start_dim=-2, end_dim=-1)]
        self.out_conv = nn.Sequential(*layers)
        self.topk = PerturbedTopK(k)

    def forward(self, x, policy=None, current_sigma=0.0005, cls_attn=None):
        return engine.predictor_b_forward(self, x, policy, current_sigma, cls_attn)


class VisionTransformerDiffPruning(_VitBackbone):
    """dynamic_vit.py:640-1033.  Populates kept_token_indices / dropped_token_indices / pred_logits /
    cls_attns on every forward, as the reference's callers expect (train.py:66-70, evaluate.py:53-57)."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12,
                 num_heads=12, mlp_ratio=4., qkv_bias=True, qk_scale=None, representation_size=None,
                 drop_rate=0., attn_drop_rate=0., drop_path_rate=0., hybrid_backbone=None, norm_layer=None,
                 pruning_loc=None, token_ratio=None, distill=False, attn_selection=False, attn_selection_threshold=0.0,
                 topk_selection=False, early_exit=False, mean_heads=False, random_drop=False, small_predictor=False,
                 predictor_loss_type=False, predictor_bn=False, patch_score_threshold=None):
        super().__init__(img_size, patch_size, in_chans, num_classes, embed_dim, depth, num_heads, mlp_ratio, qkv_bias,
                         qk_scale, representation_size, drop_rate, attn_drop_rate, drop_path_rate, hybrid_backbone,
                         norm_layer)
        self.score_predictor = nn.ModuleList([
            PredictorLG(embed_dim, topk_selection=topk_selection, k=int(token_ratio[i] * (img_size / patch_size) ** 2),
                        small_predictor=small_predictor, loss_type=predictor_loss_type, use_bn=predictor_bn)
            for i in range(len(pruning_loc))])
        self.num_kept_tokens = []
        self.attn_selection = attn_selection
        self.attn_selection_threshold = attn_selection_threshold
        self.topk_selection = topk_selection
        if self.topk_selection:
            self.current_sigma = 0.05
        self.mean_heads = mean_heads
        self.random_drop = random_drop
        self.current_score = None
        self.early_exit = early_exit
        if early_exit:
            self.early_exit_head = nn.Sequential(
                (norm_layer or (lambda d: nn.LayerNorm(d, eps=1e-6)))(embed_dim),
                nn.Linear(self.num_features, num_classes) if num_classes > 0 else nn.Identity())
        self.cls_attns = []
        self.pred_logits = []
        self.kept_token_indices = None
        self.dropped_token_indices = None
        self.patch_score_threshold = patch_score_threshold
        self.keep_ratios = None
        self.min_keep_ratio = None
        self.avg_keep_ratio = None
        self.max_keep_ratio = None
        self.unpruned = False
        self.distill = distill
        self.pruning_loc = pruning_loc
        self.token_ratio = token_ratio
        self._finish_init()

    def forward(self, x, stacked_cls_attn_weights=None):
        return engine.variant_b_forward(self, x, stacked_cls_attn_weights)

    def forward_cls_attn(self, x):
        return engine.variant_b_forward_cls_attn(self, x)

    def forward_varlen(self, x):
        """Dynamic keep-ratio inference (patch_score_threshold set, eval mode) of a batch whose images keep different token counts:
        (logits (B, classes), cls_attns, pred_logits, kept) in forward()'s eval order, ragged entries padded -- kept[s] (B,Kmax_s)
        int64 stage-relative ascending with -1, pred_logits[s] (B,Nmax_s) with -inf, cls_attns[i] (B,H,Tmax_i-1) with zeros.
        Sets keep_ratios (per image) and min / avg / max_keep_ratio of the last stage."""
        return engine.variant_b_forward_varlen(self, x)


class VisionTransformerTeacher(_VitBackbone):
    """dynamic_vit.py:1036-1176: unpruned ViT returning (logits, tokens, cls_attn (B,depth,H,T))."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._finish_init()

    def forward_cls_attention(self, x):
        return engine.teacher_forward_cls_attention(self, x)

    def forward(self, x):
        return engine.teacher_forward(self, x, with_cls_attn=True)


_ARCH = {  # dynamic_vit.py:1216-1364
    "tiny": dict(patch_size=16, embed_dim=192, depth=12, num_heads=3, mlp_ratio=4, qkv_bias=True),
    "small": dict(patch_size=16, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, qkv_bias=True),
    "base": dict(patch_size=16, embed_dim=768, depth=12, num_heads=12, mlp_ratio=4, qkv_bias=True),
}


def _student(arch, pruning_locs, keep_ratios, state_dict=None, **kwargs):
    model = VisionTransformerDiffPruning(pruning_loc=pruning_locs, token_ratio=keep_ratios, distill=True,
                                         **_ARCH[arch], **kwargs)
    if state_dict is not None:  # the reference downloads DeiT weights here; offline callers pass them in
        model.load_state_dict(state_dict.get("model", state_dict), strict=False)
    return model


def dynamic_vit_tiny_patch16_224_student(pruning_locs, keep_ratios, **kwargs):
    return _student("tiny", pruning_locs, keep_ratios, **kwargs)


def dynamic_vit_small_patch16_224_student(pruning_locs, keep_ratios, **kwargs):
    return _student("small", pruning_locs, keep_ratios, **kwargs)


def dynamic_vit_base_patch16_224_student(pruning_locs, keep_ratios, **kwargs):
    return _student("base", pruning_locs, keep_ratios, **kwargs)


def dynamic_vit_teacher(arch="small", state_dict=None, **kwargs):
    model = VisionTransformerTeacher(**_ARCH[arch], **kwargs)
    if state_dict is not None:
        model.load_state_dict(state_dict.get("model", state_dict), strict=False)
    return model
