"""Pin the CPU oracle (oracle/) against outputs of the unmodified reference (tests/golden/*.npz,
produced by tests/golden/make_goldens.py).  CPU only."""
import pytest
import torch

import fixtures as fx
from oracle import model as om
from oracle import ops as oo

OPS, OPS_META = fx.load_npz("golden_ops.npz")
MOD, MOD_META = fx.load_npz("golden_models.npz")
C = OPS_META["cases"]

FP32_TOL = dict(rtol=1e-4, atol=1e-6)   # north_star: 1e-4 relative in fp32


def sd_for(meta_case):
    sd = fx.seeded_state_dict(meta_case["shapes"], meta_case["w_seed"])
    got = fx.sd_checksum(sd)
    assert got == pytest.approx(meta_case["sd_sum"], rel=1e-9), "torch CPU RNG drifted: regenerate goldens"
    return sd


def test_batch_index_select_bit_exact():
    c = C["bis"]
    x = fx.randn(c["x_seed"], *c["x_shape"])
    assert torch.equal(oo.batch_index_select(x, OPS["bis3_idx"]), OPS["bis3_out"])
    x2 = fx.randn(c["x2_seed"], *c["x2_shape"])
    assert torch.equal(oo.batch_index_select(x2, OPS["bis3_idx"]), OPS["bis2_out"])
    with pytest.raises(NotImplementedError):
        oo.batch_index_select(torch.zeros(2, 2, 2, 2), OPS["bis3_idx"])


def test_select_matches_reference_call_sites():
    c = C["select"]
    sc = torch.softmax(fx.randn(c["seed"], *c["shape"]), dim=-1)
    kept, dropped = oo.select_topk(sc, c["k"], oo.ORDER_INDEX_ASC)
    assert torch.equal(kept, OPS["sel_keptB"]) and torch.equal(dropped, OPS["sel_dropB"])
    kept_a, _ = oo.select_topk(sc, c["k"], oo.ORDER_SCORE_DESC)
    assert torch.equal(kept_a, OPS["sel_keptA"])


def test_select_tie_rule_lower_index_first():
    sc = torch.tensor([[0.5, 0.7, 0.5, 0.7, 0.1, float("nan"), -0.0, 0.0]])
    kept, dropped = oo.select_topk(sc, 4, oo.ORDER_SCORE_DESC)
    assert kept.tolist() == [[5, 1, 3, 0]]          # NaN largest, then ties by index
    kept, dropped = oo.select_topk(sc, 4, oo.ORDER_INDEX_ASC)
    assert kept.tolist() == [[0, 1, 3, 5]] and dropped.tolist() == [[2, 4, 6, 7]]


def test_gather_scatter_roundtrip():
    x = fx.randn(5, 2, 9, 4)
    kept = torch.tensor([[0, 3, 7], [1, 2, 5]])
    g = oo.gather_tokens_with_cls(x, kept)
    assert torch.equal(g[:, 0], x[:, 0]) and torch.equal(g[0, 2], x[0, 4])
    gx = oo.scatter_tokens_bwd(g, kept, 9)
    assert torch.equal(gx[0, 4], x[0, 4]) and float(gx[0, 2].abs().sum()) == 0.0


def test_softmax_with_policy():
    c = C["swp"]
    s = fx.randn(c["s_seed"], *c["s_shape"], scale=c["s_scale"])
    assert torch.equal(oo.softmax_with_policy(s, OPS["swp_policy"]), OPS["swp_out"])
    torch.testing.assert_close(oo.softmax_with_policy(s, OPS["swp_policy_frac"]), OPS["swp_out_frac"], **FP32_TOL)
    torch.testing.assert_close(oo.softmax_with_policy(s, torch.ones(2, 17, 1)), OPS["swp_out_ones"], **FP32_TOL)


def test_softmax_with_policy_grads():
    c = C["swp"]
    s = fx.randn(c["s_seed"], *c["s_shape"], scale=c["s_scale"]).requires_grad_(True)
    p = OPS["swp_policy_frac"].clone().requires_grad_(True)
    up = fx.randn(c["up_seed"], *c["s_shape"])
    (oo.softmax_with_policy(s, p) * up).sum().backward()
    torch.testing.assert_close(s.grad, OPS["swp_grad_s"], rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(p.grad, OPS["swp_grad_p"], rtol=1e-4, atol=1e-6)


def test_attention_forward():
    c = C["attn"]
    sd = sd_for(c)
    x = fx.randn(c["x_seed"], *c["x_shape"])
    o, ca = oo.attention(x, sd["qkv.weight"], sd["qkv.bias"], sd["proj.weight"], sd["proj.bias"], c["heads"],
                         policy=None, return_cls_attn=True)
    torch.testing.assert_close(o, OPS["attn_out"], **FP32_TOL)
    torch.testing.assert_close(ca, OPS["attn_cls"], **FP32_TOL)
    o, ca = oo.attention(x, sd["qkv.weight"], sd["qkv.bias"], sd["proj.weight"], sd["proj.bias"], c["heads"],
                         policy=OPS["attn_policy"], return_cls_attn=True)
    torch.testing.assert_close(o, OPS["attn_out_pol"], **FP32_TOL)
    torch.testing.assert_close(ca, OPS["attn_cls_pol"], **FP32_TOL)
    # attention_core (what the kernel replaces) is consistent with attention()
    qkv = torch.nn.functional.linear(x, sd["qkv.weight"], sd["qkv.bias"]).view(2, 21, 3, c["heads"], -1)
    core, cls = oo.attention_core(qkv, c["heads"], policy=OPS["attn_policy"][..., 0])
    o2 = torch.nn.functional.linear(core, sd["proj.weight"], sd["proj.bias"])
    torch.testing.assert_close(o2, OPS["attn_out_pol"], **FP32_TOL)
    torch.testing.assert_close(cls, OPS["attn_cls_pol"], **FP32_TOL)


def test_gumbel_keep_decision_and_grad():
    c = C["gumbel"]
    logp = torch.log_softmax(fx.randn(c["logit_seed"], *c["shape"], scale=c["scale"]), dim=-1)
    hard, y0 = oo.gumbel_keep_decision(logp, OPS["gum_noise"], OPS["gum_prev"])
    assert torch.equal(hard, OPS["gum_hard"])
    assert set(hard.unique().tolist()) <= {0.0, 1.0}
    g = oo.gumbel_keep_decision_bwd(fx.randn(c["up_seed"], 2, 50, 1), y0, OPS["gum_prev"])
    torch.testing.assert_close(g, OPS["gum_grad"], rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("tag", ["ptk_small", "ptk_vit"])
def test_perturbed_topk(tag):
    c = C[tag]
    x = torch.softmax(fx.randn(c["x_seed"], c["b"], c["d"]), dim=-1)
    noise = fx.randn(c["noise_seed"], c["b"], c["ns"], c["d"])
    ind, eg = oo.perturbed_topk_fwd(x, noise, c["k"], c["sigma"])
    assert torch.equal(ind, OPS[tag + "_ind"])                  # counts are integers: bit-exact
    torch.testing.assert_close(ind.sum(-1), torch.ones(c["b"], c["k"]))
    gx = oo.perturbed_topk_bwd(fx.randn(c["gout_seed"], c["b"], c["k"], c["d"]), eg)
    torch.testing.assert_close(gx, OPS[tag + "_gx"], rtol=1e-4, atol=1e-5)


def test_predictor_a():
    c = C["predA"]
    sd = {"p." + k: v for k, v in sd_for(c).items()}
    x = fx.randn(c["x_seed"], *c["x_shape"])
    out = oo.predictor_a(sd, "p", x, OPS["predA_policy"])
    torch.testing.assert_close(out, OPS["predA_out"], **FP32_TOL)
    hid = oo.predictor_a_hidden(sd, "p", x, OPS["predA_policy"])
    torch.testing.assert_close(oo.score_tail_a(hid, sd["p.out_conv.4.weight"], sd["p.out_conv.4.bias"]),
                               OPS["predA_out"], **FP32_TOL)


@pytest.mark.parametrize("small", [False, True])
@pytest.mark.parametrize("bn", [False, True])
def test_predictor_b(small, bn):
    tag = f"predB_{'small' if small else 'large'}_{'bn' if bn else 'ln'}"
    c = C[tag]
    sd = {"p." + k: v for k, v in sd_for(c).items()}
    x = fx.randn(c["x_seed"], *c["x_shape"])
    scores, probs = oo.predictor_b(sd, "p", x, small=small, use_bn=bn)
    torch.testing.assert_close(scores, OPS[tag + "_scores"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(probs, OPS[tag + "_probs"], rtol=1e-4, atol=1e-7)


# ---------------------------------------------------------------------------------------- models
def _img():
    m = MOD_META["img"]
    img = fx.randn(m["seed"], *m["shape"])
    assert fx.checksum(img) == pytest.approx(m["sum"], rel=1e-9)
    return img


def _cfg(meta, **kw):
    c = fx.SMALL_CFG
    return om.VitCfg(embed_dim=c["embed_dim"], depth=c["depth"], num_heads=c["num_heads"], patch_size=c["patch_size"],
                     num_classes=c["num_classes"], pruning_loc=meta.get("locs", []), token_ratio=meta.get("ratios", []), **kw)


def test_variant_a_eval():
    m = MOD_META["A"]
    out = om.variant_a_eval(sd_for(m), _cfg(m), _img())
    for s in range(len(m["locs"])):
        assert torch.equal(out["kept"][s], MOD[f"A_eval_kept{s}"])
    torch.testing.assert_close(out["logits"], MOD["A_eval_logits"], **FP32_TOL)


def test_variant_a_train():
    m = MOD_META["A"]
    gum = [MOD[f"A_train_gumbel{i}"] for i in range(len(m["locs"]))]
    out = om.variant_a_train(sd_for(m), _cfg(m), _img(), gum)
    for i in range(len(m["locs"])):
        assert torch.equal(out["decisions"][i], MOD[f"A_train_dec{i}"])
    assert torch.equal(out["final_decision"], MOD["A_train_final"])
    torch.testing.assert_close(out["logits"], MOD["A_train_logits"], **FP32_TOL)
    torch.testing.assert_close(*fx.golden_view(MOD, MOD_META, "A_train_feats", out["features"])[:2], rtol=1e-4, atol=1e-5)


def test_variant_b_eval_and_train():
    m = MOD_META["B"]
    sd, img = sd_for(m), _img()
    out = om.variant_b_forward(sd, _cfg(m), img, training=False)
    for s in range(len(m["locs"])):
        assert torch.equal(out["kept"][s], MOD[f"B_eval_kept{s}"])
        assert torch.equal(out["dropped"][s], MOD[f"B_eval_drop{s}"])
        torch.testing.assert_close(out["pred_logits"][s], MOD[f"B_eval_pl{s}"], rtol=1e-4, atol=1e-5)
    for i in range(fx.SMALL_CFG["depth"]):
        torch.testing.assert_close(out["cls_attns"][i], MOD[f"B_eval_cls{i}"], rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(out["logits"], MOD["B_eval_logits"], **FP32_TOL)
    out = om.variant_b_forward(sd, _cfg(m), img, training=True)
    for s in range(len(m["locs"])):
        assert torch.equal(out["kept"][s], MOD[f"B_train_kept{s}"])
    torch.testing.assert_close(out["logits"], MOD["B_train_logits"], **FP32_TOL)
    torch.testing.assert_close(*fx.golden_view(MOD, MOD_META, "B_train_feats", out["features"])[:2], rtol=1e-4, atol=1e-5)


def test_variant_b_gradients_vs_fp64_reference():
    """Autograd through the oracle reproduces the reference's float64 gradients (the reference's own fp32 CPU
    backward is only accurate to ~1e-2 on the stage-0 predictor; see make_goldens.py)."""
    m = MOD_META["B"]
    sd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in sd_for(m).items()}
    out = om.variant_b_forward(sd, _cfg(m), _img(), training=True)
    u = fx.randn(m["u_seed"], *out["logits"].shape)
    loss = (out["logits"] * u).sum() + sum((pl * fx.randn(m["v_seed0"] + i, *pl.shape)).sum()
                                           for i, pl in enumerate(out["pred_logits"]))
    loss.backward()
    keys = [k for k in MOD if k.startswith("B_grad64::")]
    assert len(keys) == 7
    for key in keys:
        g, ref, amax = fx.golden_view(MOD, MOD_META, key, sd[key.split("::")[1]].grad)
        assert float((g - ref).abs().max()) / amax < 1e-4, key


def test_variant_b_threshold_train():
    m = MOD_META["Bthr"]
    cfg = _cfg(m, small_predictor=True, patch_score_threshold=m["threshold"])
    out = om.variant_b_threshold_train(sd_for(m), cfg, _img())
    assert torch.equal(out["keep_mask"], MOD["Bthr_mask"])
    torch.testing.assert_close(out["pred_logits"], MOD["Bthr_pl"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(out["logits"], MOD["Bthr_logits"], **FP32_TOL)


def test_teacher():
    m = MOD_META["T"]
    logits, tokens, cls_attn = om.teacher_forward(sd_for(m), _cfg(m), _img())
    torch.testing.assert_close(logits, MOD["T_logits"], **FP32_TOL)
    torch.testing.assert_close(*fx.golden_view(MOD, MOD_META, "T_tokens", tokens)[:2], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(cls_attn, MOD["T_cls_attn"], rtol=1e-4, atol=1e-7)


# ------------------------------------------------------------------------------------------ loss-side consumers
def _loss_goldens():
    return fx.load_npz("golden_losses.npz")


@pytest.mark.parametrize("case", ["one_stage", "two_stage", "three_stage"])
@pytest.mark.parametrize("loss_type", ["kl_div", "mse"])
def test_oracle_mask_loss_matches_reference(case, loss_type):
    from oracle import losses as ol
    G, meta = _loss_goldens()
    c = meta["cases"][case]
    inp = fx.loss_inputs(c["seed"], ratios=tuple(c["ratios"]))
    assert torch.allclose(torch.tensor([fx.checksum(inp["cls_attn"]), fx.checksum(inp["token_t"])]).double(),
                          G[f"{case}::in_checksum"].double(), rtol=1e-9), "fixture RNG drifted"
    pl = [p.clone().requires_grad_(True) for p in inp["pred_logits"]]
    loss, accs = ol.mask_loss(pl, inp["cls_attn"], inp["kept"], c["ratios"], loss_type)
    loss.backward()
    torch.testing.assert_close(loss.detach(), G[f"{case}::{loss_type}::loss"], rtol=1e-5, atol=1e-6)
    for i, p in enumerate(pl):
        torch.testing.assert_close(p.grad, G[f"{case}::{loss_type}::grad{i}"], rtol=1e-4, atol=1e-7)
    for i in range(len(c["ratios"])):
        assert float(accs[i]) == pytest.approx(float(G[f"{case}::{loss_type}::acc{i}"]), abs=1e-7)


@pytest.mark.parametrize("case", ["one_stage", "two_stage", "three_stage"])
@pytest.mark.parametrize("mix", [False, True])
def test_oracle_backbone_loss_matches_reference(case, mix):
    from oracle import losses as ol
    G, meta = _loss_goldens()
    c = meta["cases"][case]
    inp = fx.loss_inputs(c["seed"], ratios=tuple(c["ratios"]))
    ls, ts = inp["logits_s"].clone().requires_grad_(True), inp["token_s"].clone().requires_grad_(True)
    loss, parts = ol.backbone_loss(ls, ts, inp["logits_t"], inp["token_t"], inp["kept"], inp["soft"] if mix else inp["labels"],
                                   soft_labels=mix)
    loss.backward()
    tag = f"{case}::backbone{'_mix' if mix else ''}"
    torch.testing.assert_close(loss.detach(), G[f"{tag}::loss"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(ls.grad, G[f"{tag}::grad_logits"], rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(ts.grad, G[f"{tag}::grad_tokens"], rtol=1e-4, atol=1e-8)
    # the reference's metric names swap the two KL terms (losses.py:236-237)
    assert float(parts["cls_kl"].detach()) == pytest.approx(float(G[f"{tag}::train_token_kl_loss"]), rel=1e-5)
    assert float(parts["token_kl"].detach()) == pytest.approx(float(G[f"{tag}::train_cls_kl_loss"]), rel=1e-5)


def test_oracle_loss_masks_and_reference_defects():
    from oracle import losses as ol
    G, meta = _loss_goldens()
    sc = torch.softmax(fx.randn(510, 5, 196), dim=-1)
    assert torch.equal(ol.topk_mask(sc, 0.7), G["mask_pred"]) and torch.equal(ol.topk_mask(sc, 0.49 / 0.7), G["mask_cls"])
    assert meta["bce_error"] == "NameError" and meta["threshold_error"] == "UnboundLocalError"
    with pytest.raises(NameError):
        ol.mask_loss([torch.randn(4, 196)], torch.rand(4, 4, 3, 197), [torch.zeros(4, 137, dtype=torch.long)], [0.7], "bce")
    with pytest.raises(UnboundLocalError):
        ol.backbone_loss(torch.randn(4, 16), torch.randn(4, 10, 32), torch.randn(4, 16), torch.randn(4, 196, 32),
                         [torch.zeros(40, dtype=torch.long)], torch.zeros(4, dtype=torch.long), patch_score_threshold=0.9)
