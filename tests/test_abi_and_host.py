"""CPU-side checks: the C-ABI library loads and exports every symbol include/d2s.h declares (no compute calls),
argument errors are reported before any launch, host-side sharding logic, and the 2-rank (gloo) data-parallel
path of the batch-sharded hot path."""
import ctypes
import json
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "d2s.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(d2s_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol(d2s):
    lib = d2s._lib.load()
    names = _header_symbols()
    assert len(names) >= 16
    for n in names:
        assert hasattr(lib, n), f"libd2s_b200.so does not export {n}"
    assert sorted(d2s._lib.ALL_SYMBOLS) == names, "ctypes SIGNATURES out of sync with include/d2s.h"
    assert lib.d2s_version() == 100
    assert isinstance(d2s._lib.launch_count(), int)


def test_no_torch_or_cxx_types_in_abi():
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(ROOT, "dense2sparse-vit_b200", "libd2s_b200.so")],
                         capture_output=True, text=True, check=True).stdout
    exported = [ln.split()[-1] for ln in out.splitlines() if " T " in ln]
    assert set(_header_symbols()) <= set(exported)
    assert not [s for s in exported if "at::" in s or "torch" in s.lower()]


def test_argument_errors_precede_any_launch(d2s):
    """Shape / null checks run on the host before cudaLaunch: safe to exercise without a GPU."""
    lib = d2s._lib.load()
    before = d2s._lib.launch_count()
    assert lib.d2s_select_topk_f32(None, 1, 196, 10, 0, None, None, None) == 1
    assert b"null" in lib.d2s_last_error()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    assert lib.d2s_select_topk_f32(p, 1, 5000, 10, 0, p, p, None) == 1 and b"N=5000" in lib.d2s_last_error()
    assert lib.d2s_select_topk_f32(p, 1, 196, 500, 0, p, p, None) == 1 and b"K=500" in lib.d2s_last_error()
    assert lib.d2s_gather_tokens(p, 7, 1, 4, 8, p, 2, 1, p, None) == 1 and b"dtype" in lib.d2s_last_error()
    assert lib.d2s_gather_tokens(p + 4, 0, 1, 4, 8, p, 2, 1, p, None) == 2            # misaligned -> D2S_ERR_ALIGN
    assert lib.d2s_ptopk_fwd(p, p, 1, 500, 10, 8, 0.05, p, p, None) == 1 and b"N=500" in lib.d2s_last_error()
    assert lib.d2s_ptopk_fwd(p, p, 1, 196, 98, 8, 0.0, p, p, None) == 1 and b"sigma" in lib.d2s_last_error()
    assert lib.d2s_attn_policy_fwd(p, None, 1, 1, 8, 2, 48, 0.1, 1e-6, p, None, None, None) == 1
    assert b"head dim" in lib.d2s_last_error()
    assert lib.d2s_softmax_policy_fwd(p, None, 0, 1, 1, 5000, 1e-6, p, None, None) == 1
    # the tcgen05 GEMM family and the training-attention helpers: shape / alignment contracts
    assert lib.d2s_linear_residual_ln_bf16(p, p, p, p, p, p, 1e-6, 256, 576, 384, p, p, None) == 1 and b"N in {192, 384, 768}" in lib.d2s_last_error()
    assert lib.d2s_linear_residual_ln_bf16(p, p, p, p, None, None, 1e-6, 256, 384, 384, p, p, None) == 1 and b"gamma" in lib.d2s_last_error()
    assert lib.d2s_linear_residual_ln_bf16(p, p, p, p, p, p, 1e-6, 256, 384, 100, p, p, None) == 1 and b"K %" in lib.d2s_last_error()
    assert lib.d2s_linear_act_pair_bf16(p, p, p, 256, 300, 384, 1, p, None, None) == 1 and b"N % 256" in lib.d2s_last_error()
    assert lib.d2s_linear_act_pair_bf16(p + 8, p, p, 256, 256, 384, 1, p, None, None) == 2
    assert lib.d2s_mlp_residual_ln_bf16(p, p, p, p, p, p, p, p, 1e-6, 256, 768, 3072, 1, 0, p, p, None) == 1 and b"D == 384" in lib.d2s_last_error()
    assert lib.d2s_mlp_residual_ln_bf16(p, p, p, p, p, p, p, p, 1e-6, 256, 384, 1000, 1, 0, p, p, None) == 1 and b"HID" in lib.d2s_last_error()
    assert lib.d2s_mlp_residual_ln_bf16(None, p, p, p, p, p, p, p, 1e-6, 256, 384, 1536, 1, 0, p, p, None) == 1 and b"null" in lib.d2s_last_error()
    assert lib.d2s_mlp_residual_ln_bf16(p, p, p, p, p, p, p, p, 1e-6, 256, 384, 1536, 197, 1, p, p, None) == 1 and b"norm_row0" in lib.d2s_last_error()
    assert lib.d2s_softmax_policy_fwd_ld(p, None, 1, 1, 197, 200, 197, 1e-6, p, None, None) == 1 and b"ld" in lib.d2s_last_error()
    assert lib.d2s_softmax_policy_bwd_ld(p, None, p, p, 1, 1, 300, 304, 304, 1e-6, p, None, None) == 1 and b"T=300" in lib.d2s_last_error()
    assert lib.d2s_split_heads_bf16(p, 1, 197, 100, 3, 6, 64, p, None) == 1 and b"Tp=100" in lib.d2s_last_error()
    assert lib.d2s_merge_heads_bf16(p, 1, 197, 200, 3, 6, 60, p, None) == 1 and b"hd=60" in lib.d2s_last_error()
    assert d2s._lib.launch_count() == before
    # empty batches are a no-op, not an error
    assert lib.d2s_mlp_residual_ln_bf16(p, p, p, p, p, p, p, p, 1e-6, 0, 384, 1536, 1, 0, p, p, None) == 0
    assert lib.d2s_split_heads_bf16(p, 0, 197, 200, 3, 6, 64, p, None) == 0
    assert lib.d2s_assemble_layernorm(p, p, p, p, p, 1, 2, 196, 380, 1e-6, p, p, None) == 1 and b"D=380" in lib.d2s_last_error()
    assert lib.d2s_assemble_layernorm(p, None, p, p, p, 1, 2, 196, 384, 1e-6, p, p, None) == 1
    assert lib.d2s_colsum_bf16(p, 16, 12, p, None) == 1 and b"N=12" in lib.d2s_last_error()
    assert lib.d2s_gelu_bwd_colsum_bf16(p, p, 16, 12, p, p, None) == 1 and b"N=12" in lib.d2s_last_error()
    assert lib.d2s_gelu_bwd_colsum_bf16(p, None, 16, 16, p, p, None) == 1
    assert lib.d2s_colsum_bf16(None, 16, 16, p, None) == 1
    assert lib.d2s_select_topk_f32(p, 0, 196, 10, 0, p, p, None) == 0
    assert lib.d2s_gather_tokens(p, 0, 0, 4, 8, p, 2, 1, p, None) == 0


def test_ops_refuse_cpu_tensors(d2s):
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        d2s.ops.select_topk(torch.rand(2, 196), 10)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        d2s.ops.gather_tokens(torch.rand(2, 5, 8), torch.zeros(2, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        d2s.ops.perturbed_topk(torch.rand(2, 196), 98, 10, 0.05, noise=torch.zeros(2, 10, 196))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "dense2sparse-vit_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{fn} imports the oracle"


def test_package_reads_only_its_documented_environment_variables():
    """The D2S_* variables the package reads: a semantic opt-in, input validation, and the profiling-build hooks.  Every other
    configuration is fixed in the code, so what runs does not depend on the environment."""
    pkg = os.path.join(ROOT, "dense2sparse-vit_b200")
    names = set()
    for sub in (pkg, os.path.join(pkg, "csrc")):
        for fn in os.listdir(sub):
            if fn.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(sub, fn)).read()
                names |= set(re.findall(r"(?:os\.environ(?:\.get)?\s*[\(\[]|getenv\s*\()\s*[\"'](\w+)[\"']", src))
    assert {n for n in names if n.startswith("D2S_")} == {"D2S_THRESHOLD_INFERENCE", "D2S_CHECK_INDICES", "D2S_NVCC_EXTRA",
                                                           "D2S_GEMM_TRACE"}


def test_shard_range_partitions(d2s):
    sr = d2s.runner.shard_range
    for gb, w in [(1024, 1), (1024, 8), (1000, 8), (7, 8), (0, 4)]:
        spans = [sr(gb, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == gb
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [hi - lo for lo, hi in spans]
        assert max(sizes) - min(sizes) <= 1


def test_state_dict_names_follow_reference(d2s):
    a = d2s.variant_a.DefaultVisionTransformerDiffPruning(patch_size=16, embed_dim=64, depth=2, num_heads=2,
                                                          pruning_loc=[1], token_ratio=[0.7], distill=True)
    keys = set(a.state_dict())
    for k in ["patch_embed.proj.weight", "cls_token", "pos_embed", "blocks.0.norm1.weight", "blocks.1.attn.qkv.bias",
              "blocks.0.attn.proj.weight", "blocks.0.mlp.fc1.weight", "blocks.0.mlp.fc2.bias", "norm.weight", "head.bias",
              "score_predictor.0.in_conv.0.weight", "score_predictor.0.in_conv.1.weight", "score_predictor.0.out_conv.0.weight",
              "score_predictor.0.out_conv.2.weight", "score_predictor.0.out_conv.4.bias"]:
        assert k in keys, k
    b = d2s.variant_b.VisionTransformerDiffPruning(patch_size=16, embed_dim=64, depth=2, num_heads=2, pruning_loc=[1],
                                                   token_ratio=[0.7], topk_selection=True, predictor_loss_type="kl_div")
    kb = set(b.state_dict())
    assert {"score_predictor.0.in_conv.1.weight", "score_predictor.0.out_conv.13.weight",
            "score_predictor.0.out_conv.12.weight"} <= kb
    s = d2s.variant_b.VisionTransformerDiffPruning(patch_size=16, embed_dim=64, depth=2, num_heads=2, pruning_loc=[1],
                                                   token_ratio=[0.7], topk_selection=True, small_predictor=True,
                                                   predictor_bn=True, predictor_loss_type="mse")
    assert "score_predictor.0.out_conv.6.bn.running_mean" in set(s.state_dict())


# The hot-path attribute surface of the reference's modules (SURVEY.md 8b): what patch.install() must replace, and nothing else.
_REFERENCE_SURFACE = {
    "peturbed_topk": ["PerturbedTopK.__call__"],
    "default_dynamic_vit": ["batch_index_select", "Attention.softmax_with_policy", "Attention.forward", "Block.forward",
                            "PatchEmbed.forward", "PredictorLG.forward", "DefaultVisionTransformerDiffPruning.forward",
                            "DefaultVisionTransformerTeacher.forward"],
    "dynamic_vit": ["batch_index_select", "PerturbedTopK", "Attention.softmax_with_policy", "Attention.forward", "Block.forward",
                    "PatchEmbed.forward", "PredictorLG.forward", "VisionTransformerDiffPruning.forward",
                    "VisionTransformerDiffPruning.forward_cls_attn", "VisionTransformerTeacher.forward",
                    "VisionTransformerTeacher.forward_cls_attention"],
}


def _reference_stand_ins(d2s):
    """Module objects named like the reference's vit_models modules, carrying the surface above plus attributes install() must
    leave alone (Mlp, helpers).  Every original is a distinct function that fails if it runs; dynamic_vit.PerturbedTopK is the
    class of peturbed_topk, as the reference imports it.  The Variant A model class builds like the reference's (same
    constructor, same submodules), so a patched forward runs on real tensors."""
    import types

    def original():
        def f(*a, **k):
            raise AssertionError("the reference's own code ran: install() did not replace it")
        return f

    mods = {}
    for name, surface in _REFERENCE_SURFACE.items():
        mod = types.ModuleType("vit_models." + name)
        mod.untouched_helper = original()
        mod.Mlp = type("Mlp", (), {"__module__": mod.__name__, "forward": original()})
        for entry in surface:
            owner, _, attr = entry.rpartition(".")
            if not owner:
                setattr(mod, attr, mods["peturbed_topk"].PerturbedTopK if attr == "PerturbedTopK" else original())
                continue
            if not hasattr(mod, owner):
                base = (d2s.variant_a.DefaultVisionTransformerDiffPruning,) if owner == "DefaultVisionTransformerDiffPruning" else ()
                setattr(mod, owner, type(owner, base, {"__module__": mod.__name__, "untouched": original()}))
            setattr(getattr(mod, owner), attr, original())
        mods[name] = mod
    return mods


def _attribute_snapshot(mods):
    """(module, attribute) and (module, Class.attribute) -> object, for the classes each module defines."""
    snap = {}
    for name, mod in mods.items():
        for attr, val in vars(mod).items():
            snap[(name, attr)] = val
            if isinstance(val, type) and val.__module__ == mod.__name__:
                for cattr, cval in vars(val).items():
                    snap[(name, f"{attr}.{cattr}")] = cval
    return snap


def test_patch_install_swaps_reference_surface(d2s):
    """install() must replace exactly the hot-path attribute surface of SURVEY.md 8b and uninstall() must restore it."""
    mods = _reference_stand_ins(d2s)
    before = _attribute_snapshot(mods)
    d2s.patch.install(ddvit=mods["default_dynamic_vit"], dvit=mods["dynamic_vit"], ptopk=mods["peturbed_topk"])
    try:
        after = _attribute_snapshot(mods)
        assert set(after) == set(before)
        changed = {k for k in before if after[k] is not before[k]}
        assert changed == {(name, entry) for name, surface in _REFERENCE_SURFACE.items() for entry in surface}
        ddvit, dvit = mods["default_dynamic_vit"], mods["dynamic_vit"]
        assert ddvit.batch_index_select is d2s.ops.batch_index_select and dvit.batch_index_select is d2s.ops.batch_index_select
        assert dvit.PerturbedTopK is d2s.perturbed_topk.PerturbedTopK
        m = ddvit.DefaultVisionTransformerDiffPruning(patch_size=16, embed_dim=64, depth=2, num_heads=2,
                                                      pruning_loc=[1], token_ratio=[0.7], distill=True).eval()
        with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):   # patched forward reaches the kernels
            with torch.no_grad():
                m(torch.randn(1, 3, 224, 224))
    finally:
        d2s.patch.uninstall()
    restored = _attribute_snapshot(mods)
    assert set(restored) == set(before) and all(restored[k] is before[k] for k in before)


# ---- multi-rank path on CPU (gloo, world_size 2) ----------------------------------------------------
_WORKER = r'''
import os, sys, json, torch, torch.distributed as dist
sys.path.insert(0, os.environ["D2S_ROOT"]); sys.path.insert(0, os.path.join(os.environ["D2S_ROOT"], "tests", "golden"))
import d2s, fixtures as fx
from oracle import ops as oo
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
GB, N, K = 10, 196, 137
score = torch.softmax(fx.randn(5, GB, N), -1)                 # the same global batch on every rank
lo, hi = d2s.runner.shard_range(GB, rank, world)
kept, _ = oo.select_topk(score[lo:hi], K, oo.ORDER_INDEX_ASC)   # rank-local work: no data-path collective
sizes = [d2s.runner.shard_range(GB, r, world) for r in range(world)]
parts = [torch.empty(h - l, K, dtype=torch.int64) for l, h in sizes]
dist.all_gather(parts, kept) if len({p.shape for p in parts}) == 1 else dist.all_gather_object(parts, kept)
full, _ = oo.select_topk(score, K, oo.ORDER_INDEX_ASC)
ok = torch.equal(torch.cat([torch.as_tensor(p) for p in parts]), full)
ms = torch.tensor([10.0 + rank])                              # max-over-ranks timing reduction used by bench.py
dist.all_reduce(ms, op=dist.ReduceOp.MAX)
# training's one collective: runner.FlatGrads -- every gradient a view of one flat buffer, one all-reduce, mean over the ranks
torch.manual_seed(7)
net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Tanh(), torch.nn.Linear(5, 3))
xs, ys = fx.randn(11, GB, 6), fx.randn(12, GB, 3)
ref_net = __import__("copy").deepcopy(net)
((ref_net(xs) - ys) ** 2).mean(dim=1).mean().backward()          # the global-batch gradient, computed in one process
fg = d2s.runner.FlatGrads(net.parameters())
views = [p.grad for p in net.parameters()]
fg.zero()
((net(xs[lo:hi]) - ys[lo:hi]) ** 2).mean(dim=1).mean().backward()  # equal shard sizes: mean of shard means = global mean
fg.all_reduce()
grads_ok = all(p.grad is v for p, v in zip(net.parameters(), views)) and all(
    torch.allclose(p.grad, q.grad, rtol=1e-5, atol=1e-7) for p, q in zip(net.parameters(), ref_net.parameters()))
offs, total = d2s.runner.flat_layout(list(net.parameters()))
layout_ok = all(o % 8 == 0 for o in offs) and total == fg.flat.numel() and offs == fg.offsets
fs = d2s.runner.FlatGrads(__import__("copy").deepcopy(net).parameters(), average=False)   # sum: the optimizer folds 1/world in
fs.flat.fill_(float(rank + 1))
fs.all_reduce()
sum_ok = bool((fs.flat == 3.0).all())
if rank == 0:
    print(json.dumps({"ok": bool(ok), "max_ms": float(ms), "world": world, "env": d2s.runner.dist_env(),
                      "grads_ok": bool(grads_ok), "layout_ok": bool(layout_ok), "sum_ok": sum_ok}))
dist.destroy_process_group()
'''


def _torchrun(args, env_extra=None, timeout=240):
    env = dict(os.environ, D2S_ROOT=ROOT, OMP_NUM_THREADS="2")
    env.update(env_extra or {})
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533"] + args
    return subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout, cwd=ROOT)


def test_two_rank_gloo_sharding(tmp_path):
    w = tmp_path / "worker.py"
    w.write_text(_WORKER)
    r = _torchrun([str(w)])
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    out = json.loads(line)
    assert out["ok"] and out["max_ms"] == 11.0 and out["world"] == 2 and out["env"] == [0, 0, 2]
    # the gradient all-reduce of the training path (runner.FlatGrads): mean over the ranks == the global-batch gradient
    assert out["grads_ok"] and out["layout_ok"] and out["sum_ok"]


def test_bench_reference_arm_contract_two_ranks():
    """`bench.py --impl reference` under torchrun: rank 0 alone prints one JSON line, others exit 0."""
    r = _torchrun([os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                   "--cpu-batch", "1"], timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    out = json.loads(lines[0])
    for k in ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]:
        assert k in out, k
    assert out["impl"] == "reference" and out["n_gpus"] == 2 and out["value"] > 0
    assert out["cpu_baseline"]["kind"] == "port" and out["e2e"]["h2d_bytes_per_step"] == 0


def test_distill_loss_masked_token_term_equals_indexing_the_kept_rows(d2s):
    """DistillDiffPruningLoss computes the kept-token KL as a masked mean (static shapes, CUDA-graph friendly); it must equal
    the boolean-indexing form, including the all-dropped case."""
    import torch
    import torch.nn.functional as F
    torch.manual_seed(5)
    B, N, C, K = 3, 12, 16, 10

    class Teacher(torch.nn.Module):
        def forward(self, x):
            g = torch.Generator().manual_seed(9)
            return torch.randn(B, K, generator=g), torch.randn(B, N, C, generator=g)

    crit = d2s.losses.DistillDiffPruningLoss(Teacher(), keep_ratio=[0.7, 0.49, 0.343])
    pred, tok = torch.randn(B, K), torch.randn(B, N, C)
    scores = [torch.rand(B, N) for _ in range(3)]
    labels = torch.randint(0, K, (B,))
    for mask in ((torch.rand(B, N, 1) > 0.5).float(), torch.zeros(B, N, 1)):
        loss, parts = crit(torch.zeros(B, 3, 8, 8), (pred, tok, mask, scores), labels)
        keep = mask.reshape(B * N) > 0.5
        _, tt = Teacher()(None)
        tp_k, tt_k = tok.reshape(B * N, C)[keep], tt.reshape(B * N, C)[keep]
        ref = tok.new_zeros(()) if tp_k.shape[0] == 0 else F.kl_div(F.log_softmax(tp_k, -1), F.log_softmax(tt_k, -1),
                                                                     reduction="batchmean", log_target=True)
        torch.testing.assert_close(parts["token_kl"], ref, rtol=1e-5, atol=1e-6)
        assert torch.isfinite(loss)


def test_training_path_helpers_fall_back_to_the_modules_off_the_gpu(d2s):
    """ops.linear_train / linear_gelu_train are the plain modules whenever the fused bf16 CUDA path does not apply (here: CPU
    tensors) -- same values, ordinary autograd; they never touch the library in that case."""
    import torch
    torch.manual_seed(3)
    lin, act = torch.nn.Linear(16, 24), torch.nn.GELU()
    x = torch.randn(5, 16, requires_grad=True)
    before = d2s._lib.launch_count()
    y = d2s.ops.linear_train(lin, x)
    z = d2s.ops.linear_gelu_train(lin, act, x)
    assert torch.equal(y, lin(x)) and torch.equal(z, act(lin(x)))
    z.sum().backward()
    assert x.grad is not None and lin.weight.grad is not None
    assert d2s._lib.launch_count() == before
    m = d2s.layers.Mlp(16, 32)
    assert torch.equal(m(x), m.drop(m.fc2(m.drop(m.act(m.fc1(x))))))


def test_traffic_json_is_reproducible_from_the_committed_ncu_capture(tmp_path):
    """profiles/traffic.json (bench.py's `roofline.traffic`) is exactly what scripts/make_traffic_json.py derives from the committed
    ncu capture it names as its source."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    committed = json.load(open(os.path.join(root, "profiles", "traffic.json")))
    src = committed["mlp_pair_kernel"]["source"].split()[0]
    out = tmp_path / "traffic.json"
    subprocess.run([sys.executable, os.path.join(root, "scripts", "make_traffic_json.py"), os.path.join(root, src), str(out)],
                   check=True, capture_output=True)
    assert json.load(open(out)) == committed
    k = committed["mlp_pair_kernel"]
    # algorithmic bytes per launch, averaged over the step's 11 launches: (B,T,D) bf16 in and out (+ the predictor norm in 3 of
    # them) = 2.27 / 4 of the 409.3 MB the kernel moved while it still read a normalised copy and wrote the next one
    assert k["launches_per_step"] == 11 and 0.35 < k["dram_bytes_per_step"] / (11 * 409.3e6) < 0.7
