"""Generate tests/golden/*.npz by executing the UNMODIFIED reference (imported from /root/reference
through refload.py) on seeded synthetic inputs.  Run in the build container only:

    python tests/golden/make_goldens.py

The reference has no tests or golden vectors of its own (SURVEY.md section 4); these files are what
pins the oracle.  Inputs and weights are regenerated from seeds by fixtures.py; the .npz files hold the
reference's outputs plus checksums of the regenerated inputs (to detect RNG drift).
"""
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fixtures as fx  # noqa: E402
import refload  # noqa: E402

torch.set_num_threads(4)
ref = refload.load_reference()


def shapes_of(module):
    return {k: tuple(v.shape) for k, v in module.state_dict().items()}


def load_seeded(module, seed):
    sd = fx.seeded_state_dict(shapes_of(module), seed)
    module.load_state_dict(sd, strict=True)
    return sd


# ------------------------------------------------------------------------------------------
def ops_goldens():
    A, meta = {}, {"cases": {}}

    # batch_index_select (default_dynamic_vit.py:37-53), 3-D and 2-D
    x = fx.randn(1, 3, 10, 8)
    idx = torch.stack([torch.randperm(10, generator=fx.gen(2 + i))[:4] for i in range(3)])
    A["bis3_idx"] = idx
    A["bis3_out"] = ref.ddvit.batch_index_select(x, idx)
    x2 = fx.randn(3, 3, 10)
    A["bis2_out"] = ref.ddvit.batch_index_select(x2, idx)
    meta["cases"]["bis"] = dict(x_seed=1, x_shape=[3, 10, 8], x2_seed=3, x2_shape=[3, 10])

    # softmax_with_policy (dynamic_vit.py:195-214): hard 0/1 policy, fractional policy, all-ones
    attn_mod = ref.dvit.Attention(dim=128, num_heads=2, qkv_bias=True)
    s = fx.randn(10, 2, 3, 17, 17, scale=3.0)
    pol = (torch.rand(2, 17, 1, generator=fx.gen(11)) > 0.4).float()
    pol[:, 0] = 1.0
    A["swp_policy"] = pol
    A["swp_out"] = attn_mod.softmax_with_policy(s, pol)
    polf = torch.rand(2, 17, 1, generator=fx.gen(12))
    A["swp_policy_frac"] = polf
    A["swp_out_frac"] = attn_mod.softmax_with_policy(s, polf)
    A["swp_out_ones"] = attn_mod.softmax_with_policy(s, torch.ones(2, 17, 1))
    # the third textual copy in default_dynamic_vit.py must agree
    attn_mod_a = ref.ddvit.Attention(dim=128, num_heads=2, qkv_bias=True)
    assert torch.equal(attn_mod_a.softmax_with_policy(s, pol), A["swp_out"])
    meta["cases"]["swp"] = dict(s_seed=10, s_shape=[2, 3, 17, 17], s_scale=3.0)

    # gradient of softmax_with_policy w.r.t. scores and policy
    s_g = s.clone().requires_grad_(True)
    p_g = polf.clone().requires_grad_(True)
    up = fx.randn(13, 2, 3, 17, 17)
    (attn_mod.softmax_with_policy(s_g, p_g) * up).sum().backward()
    A["swp_grad_s"], A["swp_grad_p"] = s_g.grad, p_g.grad
    meta["cases"]["swp"]["up_seed"] = 13

    # Attention.forward, Variant B signature (dynamic_vit.py:216-236), with and without policy
    sd = load_seeded(attn_mod, 20)
    xa = fx.randn(21, 2, 21, 128)
    pol_a = (torch.rand(2, 21, 1, generator=fx.gen(22)) > 0.3).float()
    pol_a[:, 0] = 1.0
    with torch.no_grad():
        o, ca = attn_mod(xa, None, return_cls_attn=True)
        A["attn_out"], A["attn_cls"] = o, ca
        o, ca = attn_mod(xa, pol_a, return_cls_attn=True)
        A["attn_out_pol"], A["attn_cls_pol"] = o, ca
    A["attn_policy"] = pol_a
    meta["cases"]["attn"] = dict(w_seed=20, x_seed=21, x_shape=[2, 21, 128], dim=128, heads=2,
                                 sd_sum=fx.sd_checksum(sd), shapes={k: list(v) for k, v in shapes_of(attn_mod).items()})

    # gumbel keep decision (default_dynamic_vit.py:454) incl. gradient of the straight-through path
    logits = F.log_softmax(fx.randn(30, 2, 50, 2, scale=2.0), dim=-1).requires_grad_(True)
    prev = (torch.rand(2, 50, 1, generator=fx.gen(31)) > 0.2).float()
    torch.manual_seed(32)
    with refload.record_gumbels() as rec:
        hard = F.gumbel_softmax(logits, hard=True)[:, :, 0:1] * prev
    upg = fx.randn(33, 2, 50, 1)
    (hard * upg).sum().backward()
    A["gum_noise"], A["gum_prev"], A["gum_hard"], A["gum_grad"] = rec.gumbels[0], prev, hard.detach(), logits.grad
    meta["cases"]["gumbel"] = dict(logit_seed=30, shape=[2, 50, 2], scale=2.0, up_seed=33)

    # selection call sites transcribed as torch calls (dynamic_vit.py:858-862; default_dynamic_vit.py:463)
    sc = torch.softmax(fx.randn(40, 4, 196), dim=-1)
    srt = torch.argsort(sc, dim=1, descending=True)
    assert all(len(torch.unique(sc[b])) == 196 for b in range(4)), "tie in golden scores"
    A["sel_keptB"] = torch.sort(srt[:, :137], dim=1)[0]
    A["sel_dropB"] = torch.sort(srt[:, 137:], dim=1)[0]
    A["sel_keptA"] = srt[:, :137]
    meta["cases"]["select"] = dict(seed=40, shape=[4, 196], k=137)

    # PerturbedTopK forward/backward with injected noise (peturbed_topk.py:16-80)
    for tag, (b, d, k, ns, sigma) in {"ptk_small": (3, 32, 10, 20, 0.05), "ptk_vit": (2, 196, 98, 50, 0.05)}.items():
        xs = torch.softmax(fx.randn(50, b, d), dim=-1).requires_grad_(True)
        noise = fx.randn(51, b, ns, d)
        gout = fx.randn(52, b, k, d)
        with refload.inject_normal(noise):
            ind = ref.ptopk.PerturbedTopK(k, num_samples=ns, sigma=sigma)(xs, current_sigma=sigma)
        (ind * gout).sum().backward()
        A[tag + "_ind"], A[tag + "_gx"] = ind.detach(), xs.grad
        meta["cases"][tag] = dict(b=b, d=d, k=k, ns=ns, sigma=sigma, x_seed=50, noise_seed=51, gout_seed=52)

    # PredictorLG Variant A (default_dynamic_vit.py:304-330)
    pa = ref.ddvit.PredictorLG(128)
    sd = load_seeded(pa, 60)
    xp = fx.randn(61, 2, 30, 128)
    polp = (torch.rand(2, 30, 1, generator=fx.gen(62)) > 0.3).float()
    with torch.no_grad():
        A["predA_out"] = pa(xp, polp)
    A["predA_policy"] = polp
    meta["cases"]["predA"] = dict(w_seed=60, x_seed=61, x_shape=[2, 30, 128], sd_sum=fx.sd_checksum(sd),
                                  shapes={k: list(v) for k, v in shapes_of(pa).items()})

    # PredictorLG Variant B, all four architectures (dynamic_vit.py:370-560), eval mode
    for small in (False, True):
        for bn in (False, True):
            tag = f"predB_{'small' if small else 'large'}_{'bn' if bn else 'ln'}"
            pb = ref.dvit.PredictorLG(128, topk_selection=True, k=137, small_predictor=small,
                                      loss_type="kl_div", use_bn=bn).eval()
            sd = load_seeded(pb, 70)
            with torch.no_grad():
                sc_, pr_ = pb(xp)
            A[tag + "_scores"], A[tag + "_probs"] = sc_, pr_
            meta["cases"][tag] = dict(w_seed=70, x_seed=61, x_shape=[2, 30, 128], small=small, bn=bn,
                                      sd_sum=fx.sd_checksum(sd), shapes={k: list(v) for k, v in shapes_of(pb).items()})
    fx.save_npz("golden_ops.npz", A, meta)
    print("golden_ops.npz:", len(A), "arrays")


# ------------------------------------------------------------------------------------------
def margin_ok(score, k, rel=1e-3):
    """Reject weight seeds that put the K-th/K+1-th scores closer than `rel` (near-tie at the cut)."""
    v = torch.sort(score, dim=1, descending=True).values
    gap = (v[:, k - 1] - v[:, k]).abs()
    return bool((gap > rel * v[:, k - 1].abs()).all())


def model_goldens():
    A, meta = {}, {}
    c = fx.SMALL_CFG
    common = dict(patch_size=c["patch_size"], embed_dim=c["embed_dim"], depth=c["depth"], num_heads=c["num_heads"],
                  num_classes=c["num_classes"], mlp_ratio=4, qkv_bias=True)
    img = fx.randn(100, 2, 3, 224, 224)
    meta["img"] = dict(seed=100, shape=[2, 3, 224, 224], sum=fx.checksum(img))
    locs, ratios = [1, 2], [0.7, 0.49]

    # ---- Variant A (DynamicViT): eval + train with recorded gumbels
    ma = ref.ddvit.DefaultVisionTransformerDiffPruning(pruning_loc=locs, token_ratio=ratios, distill=True, **common)
    sd = load_seeded(ma, 101)
    meta["A"] = dict(w_seed=101, locs=locs, ratios=ratios, sd_sum=fx.sd_checksum(sd),
                     shapes={k: list(v) for k, v in shapes_of(ma).items()})
    ma.eval()
    with torch.no_grad():
        A["A_eval_logits"] = ma(img)
    ma.train()
    torch.manual_seed(102)
    with refload.record_gumbels() as rec:
        logits, feats, final_dec, decs = ma(img)
    A["A_train_logits"], A["A_train_feats"], A["A_train_final"] = logits.detach(), feats.detach(), final_dec
    for i, (g, d) in enumerate(zip(rec.gumbels, decs)):
        A[f"A_train_gumbel{i}"], A[f"A_train_dec{i}"] = g, d.detach()
    # gradient parity targets: d(sum(logits*u) + sum(dec_i * v_i)) / d(selected params)
    u = fx.randn(103, *logits.shape)
    loss = (logits * u).sum() + sum((d * fx.randn(104 + i, *d.shape)).sum() for i, d in enumerate(decs))
    ma.zero_grad()
    loss.backward()
    for name in ["score_predictor.0.out_conv.4.weight", "score_predictor.0.in_conv.1.weight",
                 "score_predictor.1.out_conv.0.weight", "blocks.1.attn.qkv.weight", "blocks.3.mlp.fc2.bias",
                 "blocks.0.attn.qkv.weight", "cls_token"]:
        A["A_grad::" + name] = dict(ma.named_parameters())[name].grad.clone()
    meta["A"]["u_seed"], meta["A"]["v_seed0"] = 103, 104

    # ---- Variant B (Dense2Sparse): eval + train, large LN predictor, top-k mode
    mb = ref.dvit.VisionTransformerDiffPruning(pruning_loc=locs, token_ratio=ratios, distill=True,
                                               topk_selection=True, predictor_loss_type="kl_div", **common)
    sd = load_seeded(mb, 111)
    meta["B"] = dict(w_seed=111, locs=locs, ratios=ratios, sd_sum=fx.sd_checksum(sd),
                     shapes={k: list(v) for k, v in shapes_of(mb).items()})
    mb.eval()
    with torch.no_grad():
        logits, cls_attns, pred_logits, kept = mb(img)
    A["B_eval_logits"] = logits
    for i, t in enumerate(cls_attns):
        A[f"B_eval_cls{i}"] = t
    for i, (pl, kp, dr) in enumerate(zip(pred_logits, kept, mb.dropped_token_indices)):
        A[f"B_eval_pl{i}"], A[f"B_eval_kept{i}"], A[f"B_eval_drop{i}"] = pl, kp, dr
        assert margin_ok(torch.softmax(pl, -1), kp.shape[1]), "near-tie at the cut; pick another seed"
    mb.train()
    logits, feats, pred_logits, kept = mb(img)
    A["B_train_logits"], A["B_train_feats"] = logits.detach(), feats.detach()
    for i, kp in enumerate(kept):
        A[f"B_train_kept{i}"] = kp
    u = fx.randn(113, *logits.shape)
    loss = (logits * u).sum() + sum((pl * fx.randn(114 + i, *pl.shape)).sum() for i, pl in enumerate(pred_logits))
    mb.zero_grad()
    loss.backward()
    for name in ["score_predictor.0.out_conv.13.weight", "score_predictor.1.in_conv.1.weight",
                 "blocks.0.attn.qkv.weight", "blocks.2.attn.proj.weight", "pos_embed"]:
        A["B_grad::" + name] = dict(mb.named_parameters())[name].grad.clone()
    meta["B"]["u_seed"], meta["B"]["v_seed0"] = 113, 114
    # The reference's own fp32 CPU backward of the stage-0 predictor is off by up to 1e-2 (relative) from
    # its fp64 backward (torch CPU reduction order over the expanded global-pool branch); the parity target
    # for gradients is therefore the reference run in float64, stored as float32.
    mb64 = ref.dvit.VisionTransformerDiffPruning(pruning_loc=locs, token_ratio=ratios, distill=True,
                                                 topk_selection=True, predictor_loss_type="kl_div", **common)
    mb64.load_state_dict(sd)
    mb64 = mb64.double().train()
    logits64, _, pred_logits64, kept64 = mb64(img.double())
    assert all(torch.equal(a, b) for a, b in zip(kept64, kept))
    loss64 = (logits64 * u.double()).sum() + sum((pl * fx.randn(114 + i, *pl.shape).double()).sum()
                                                 for i, pl in enumerate(pred_logits64))
    mb64.zero_grad()
    loss64.backward()
    for name in ["score_predictor.0.out_conv.13.weight", "score_predictor.0.out_conv.1.weight",
                 "score_predictor.0.in_conv.1.weight", "score_predictor.1.in_conv.1.weight",
                 "blocks.0.attn.qkv.weight", "blocks.2.attn.proj.weight", "pos_embed"]:
        A["B_grad64::" + name] = dict(mb64.named_parameters())[name].grad.float().clone()

    # ---- Variant B threshold (dynamic keep ratio) training branch (dynamic_vit.py:880-894)
    mt = ref.dvit.VisionTransformerDiffPruning(pruning_loc=[1], token_ratio=[0.7], distill=True, topk_selection=True,
                                               predictor_loss_type="kl_div", patch_score_threshold=0.3,
                                               small_predictor=True, **common)
    sd = load_seeded(mt, 121)
    meta["Bthr"] = dict(w_seed=121, locs=[1], ratios=[0.7], threshold=0.3, small=True, sd_sum=fx.sd_checksum(sd),
                        shapes={k: list(v) for k, v in shapes_of(mt).items()})
    mt.train()
    logits, feats, pl, keep_mask = mt(img)
    A["Bthr_logits"], A["Bthr_pl"], A["Bthr_mask"] = logits.detach(), pl.detach(), keep_mask.detach()

    # ---- Teachers
    tb = ref.dvit.VisionTransformerTeacher(**common).eval()
    sd = load_seeded(tb, 131)
    meta["T"] = dict(w_seed=131, sd_sum=fx.sd_checksum(sd), shapes={k: list(v) for k, v in shapes_of(tb).items()})
    with torch.no_grad():
        lg, tok, ca = tb(img)
    A["T_logits"], A["T_tokens"], A["T_cls_attn"] = lg, tok, ca
    ta = ref.ddvit.DefaultVisionTransformerTeacher(**common).eval()
    ta.load_state_dict(sd, strict=True)
    with torch.no_grad():
        lg2, tok2 = ta(img)
    assert torch.allclose(lg, lg2, atol=1e-6) and torch.allclose(tok, tok2, atol=1e-6)

    # Variant A per-stage kept indices are not returned by the reference's eval forward; expose them by
    # re-running its own lines on a hook-free copy: record argsort outputs via a wrapper around batch_index_select
    rec_idx = []
    orig = ref.ddvit.batch_index_select

    def spy(x, idx):
        rec_idx.append(idx.clone())
        return orig(x, idx)

    ref.ddvit.batch_index_select = spy
    try:
        ma.eval()
        with torch.no_grad():
            again = ma(img)
    finally:
        ref.ddvit.batch_index_select = orig
    assert torch.equal(again, A["A_eval_logits"])
    # calls alternate: (x, now_policy), (prev_decision, keep_policy)
    for s in range(len(locs)):
        A[f"A_eval_kept{s}"] = rec_idx[2 * s + 1]
    fx.save_npz("golden_models.npz", A, meta, sample=True)
    print("golden_models.npz:", len(A), "arrays")


if __name__ == "__main__":
    ops_goldens()
    model_goldens()
