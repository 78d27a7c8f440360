#!/usr/bin/env python
"""Throughput of the token-sparsification hot path inside DynamicViT DeiT-S/16, keep rate 0.7, 224 px.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl d2s|reference] [--batch B] [--legs a,b,...] [--dump-outputs DIR]

A "step" is one inference pass of the pruned model over one batch of synthetic images (BASELINE.json configs[1]: batch 1024
per GPU, bf16).  N > 1 = one process per GPU (torchrun); the batch dimension is sharded with no data-path collective (weak
scaling: every rank owns its own 1024 images).  Rank 0 prints ONE JSON line.

  value          images/s, inputs resident in HBM, CUDA-graph replay of the whole forward, CUDA-event timed, max over ranks
  e2e            images/s through the public API (runner.InferenceRunner, uint8_input=True) with pinned HOST uint8 images in and
                 HOST logits out every step; e2e_float_input = the same with host-normalised bf16 images (twice the copy)
  parity_checked the gate run before any timing: 8 images through the fp32 GPU path and the bf16 path against the CPU oracle
  roofline       the step's dominant d2s kernel (the one-kernel MLP, tensor-bound), aggregated over its launches per step
  kernels        every d2s kernel of the step timed alone inside a CUDA graph (no host launch time), rotating buffers > L2
  train          BASELINE configs[2]: Variant A training step (student fwd+bwd, frozen teacher on a second stream, distillation
                 losses, AdamW as one flat kernel), bf16 autocast, batch 256 per GPU, whole step one CUDA graph; N > 1: one NCCL
                 all-reduce of the flat gradient buffer per step; train.e2e: pinned host batch copied in under the previous step
  ptopk          BASELINE configs[3]: PerturbedTopK forward + backward (N=196, k=98, 500 samples), B in {1, 8, 64, 256}
  sweep          BASELINE configs[4]: select / gather / scatter, D in {384, 768}, bf16 and fp32, keep 0.3-0.9, B 1-4096
  arch_base      the same inference path at DeiT-B widths (D = 768, 12 heads, hidden 3072), batch 512
  variant_b      Dense2Sparse (Variant B): inference at batch 1024 and the reference's train.py loop (MaskLoss + BackboneLoss) at 256
  h2d_only       the host->device copy of the e2e leg alone (its ceiling), at N ranks
  gpu_eager_baseline  the oracle's restatement of the reference forward executed by torch eager on the same GPU in bf16
  cpu_baseline   the CPU restatement of the reference forward (oracle/), timed on this box's host cores
  --impl reference   times that CPU forward alone (the reference is pure PyTorch; see DESIGN.md section 7)

--steps K is the number of timed steps of every leg that times the project's own path (value, e2e, train, arch_base, variant_b).
--dump-outputs DIR writes what the timed path computed in its last step (rank 0): the logits and the kept-token indices of every
stage, as DIR/<name>.npy in float32.  Weights and inputs are seeded, so two builds run with the same arguments can be compared
output for output.  bench.py writes nothing into the repository tree (it may be read-only).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.dont_write_bytecode = True   # no __pycache__ in the repository tree for the modules only bench.py imports
ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests", "golden")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "images/sec DynamicViT DeiT-S kr=0.7 @224"
UNIT = "images/s"
LOCS, RATIOS = [3, 6, 9], [0.7, 0.7 ** 2, 0.7 ** 3]   # upstream DynamicViT convention (SURVEY.md 8d cfg 1/2)
DEIT_S = dict(patch_size=16, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, qkv_bias=True)
DEIT_B = dict(patch_size=16, embed_dim=768, depth=12, num_heads=12, mlp_ratio=4, qkv_bias=True)     # BASELINE configs[3] / [4] widths
GFLOP_PER_IMG = 5.96                                    # SURVEY.md 8d, Variant A 3 stages
TRAIN_GFLOP_PER_IMG = 36.8                              # SURVEY.md 8d: 3 x 9.2 (student fwd+bwd at T=197) + 9.2 (teacher fwd)
ALL_LEGS = ("parity", "infer", "e2e", "h2d", "train", "kernels", "ptopk", "sweep", "base", "variant_b", "eager", "cpu")
W_SEED = 61                                             # seeded weights (tests/golden/fixtures.py): well-spread predictor scores
L2_BYTES = 126e6
DUMP_BYTES = 64 << 20                                   # --dump-outputs: at most this much in all


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="d2s", choices=["d2s", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="images per GPU per step")
    ap.add_argument("--train-batch", type=int, default=256, help="images per GPU per training step (BASELINE configs[2])")
    ap.add_argument("--train-steps", type=int, default=None, help="timed training steps (default: --steps)")
    ap.add_argument("--cpu-batch", type=int, default=8, help="images per CPU step (BASELINE configs[0])")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--teacher-stream", type=int, default=1, help="training leg: run the frozen teacher on a second stream (1) or inline (0)")
    ap.add_argument("--torch-adamw", action="store_true", help="training leg: torch.optim.AdamW(capturable) instead of runner.FlatAdamW")
    ap.add_argument("--skip-cpu", action="store_true", help="omit the cpu_baseline leg (debugging only)")
    ap.add_argument("--legs", default=",".join(ALL_LEGS), help="comma-separated subset of: " + ", ".join(ALL_LEGS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed path's outputs of its last step (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "d2s":
        ap.error("--dump-outputs writes the outputs of the d2s arm")
    if args.train_steps is None:
        args.train_steps = args.steps
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return dict(hbm=float(p["hbm_gbs"]), tf_burst=float(p["bf16_tflops"]),
                    tf_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


def seeded_weights(model):
    """Random weights with non-degenerate predictor scores, a pure function of the architecture (fixtures.seeded_state_dict)."""
    import fixtures as fx
    sd = fx.seeded_state_dict({k: tuple(v.shape) for k, v in model.state_dict().items()}, W_SEED)
    model.load_state_dict(sd)
    return sd


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle's restatement of DefaultVisionTransformerDiffPruning.forward (eval), all host threads
# ---------------------------------------------------------------------------------------------------
def cpu_forward_setup(batch):
    import torch
    from oracle import model as om           # bench.py's cpu legs are allowed to execute oracle/
    import d2s
    m = d2s.pkg.variant_a.DefaultVisionTransformerDiffPruning(pruning_loc=LOCS, token_ratio=RATIOS, distill=True, **DEIT_S)
    sd = {k: v.detach().float() for k, v in seeded_weights(m).items()}
    cfg = om.VitCfg(embed_dim=384, depth=12, num_heads=6, pruning_loc=LOCS, token_ratio=RATIOS)
    img = torch.randn(batch, 3, 224, 224, generator=torch.Generator().manual_seed(42))
    return om, sd, cfg, img


def time_cpu(batch, steps, warmup, budget_s=None):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    om, sd, cfg, img = cpu_forward_setup(batch)
    with torch.no_grad():
        for _ in range(warmup):
            om.variant_a_eval(sd, cfg, img)
        times = []
        t_begin = time.perf_counter()
        for _ in range(steps):
            t0 = time.perf_counter()
            om.variant_a_eval(sd, cfg, img)
            times.append(time.perf_counter() - t0)
            if budget_s is not None and time.perf_counter() - t_begin > budget_s and len(times) >= 3:
                break
    total = sum(times)
    return dict(img_s=batch * len(times) / total, ms_per_step=1e3 * total / len(times), steps=len(times),
                cores=torch.get_num_threads())


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    r = time_cpu(args.cpu_batch, args.steps, args.warmup)
    sample = (f"{r['steps']} steps x batch {args.cpu_batch} fp32 images, oracle.model.variant_a_eval "
              f"(CPU restatement of default_dynamic_vit.py:435-487), torch {r['cores']} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["img_s"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "DynamicViT DeiT-S/16 keep_rate=0.7 (3 stages @3,6,9) inference, 224px, synthetic images",
                   "cpu_batch": args.cpu_batch, "pruning_loc": LOCS, "token_ratio": RATIOS},
        "cpu_baseline": {"value": r["img_s"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["img_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


# ---------------------------------------------------------------------------------------------------
# GPU arm: helpers
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


def time_graphed(calls, torch, launches=24, replays=5):
    """Average GPU duration (ms) of one kernel launch.  `calls` is a list of closures doing the SAME launch on different
    argument sets (rotating buffers: their combined footprint should exceed the L2); `launches` of them are captured
    round-robin into one CUDA graph, so no host launch time sits between kernels; the graph is replayed `replays` times between
    two CUDA events on the replaying stream."""
    reps = max(1, launches // len(calls))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for c in calls:
            c()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(reps):
            for c in calls:
                c()
    graph.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(replays):
        graph.replay()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / (replays * reps * len(calls))
    del graph
    return ms


def nsets_for(bytes_per_call):
    """How many rotating argument sets make the working set larger than twice the L2 (at most 8, at least 1)."""
    return int(max(1, min(8, -(-2 * L2_BYTES // max(1.0, float(bytes_per_call))))))


def dump_outputs(out_dir, arrays):
    """Write each batch-major array as out_dir/<name>.npy in float32 (the indices are small integers: exact).  Above DUMP_BYTES
    in all, the same fixed, seeded sample of rows (images) is taken from every array."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    rows = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    if rows * row_bytes > DUMP_BYTES:
        keep = np.sort(np.random.RandomState(0).choice(rows, DUMP_BYTES // row_bytes, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def row(kernel, shape, ms, algo_bytes, launches_per_step=None, flops=None):
    r = dict(kernel=kernel, shape=shape, us=ms * 1e3, algo_bytes=algo_bytes, gbs=algo_bytes / ms / 1e6)
    if launches_per_step is not None:
        r["launches_per_step"] = launches_per_step
    if flops is not None:
        r["tflops"] = flops / ms / 1e9
    return r


# ---------------------------------------------------------------------------------------------------
# parity gate
# ---------------------------------------------------------------------------------------------------
def parity_gate(pkg, model16, sd, dev, torch):
    """8 images, before anything is timed: (1) the fp32 GPU path against the CPU oracle on the same weights -- kept-token sets
    bit-exact at all three stages, logits 1e-4; (2) the bf16 model that is about to be timed against the fp32 oracle on the
    bf16-ROUNDED weights and images -- tokens may only change sides where the fp32 score is within bf16 noise of the cut."""
    import copy
    from oracle import model as om
    cfg = om.VitCfg(embed_dim=384, depth=12, num_heads=6, pruning_loc=LOCS, token_ratio=RATIOS)
    img = torch.randn(8, 3, 224, 224, generator=torch.Generator().manual_seed(7)).bfloat16().float()
    sd32 = {k: v.detach().float() for k, v in sd.items()}
    ref = om.variant_a_eval(sd32, cfg, img)
    m32 = pkg.variant_a.DefaultVisionTransformerDiffPruning(pruning_loc=LOCS, token_ratio=RATIOS, distill=True, **DEIT_S)
    m32.load_state_dict(sd32)
    m32 = m32.to(dev).eval()
    with torch.no_grad():
        l32 = m32(img.to(dev)).cpu()
    # Variant A keeps the tokens in descending-score order and indexes every stage relative to the previous stage's order.  Two
    # kept tokens whose fp32 scores differ by less than the CPU/GPU rounding difference (~1e-6) may swap places (attention is
    # permutation equivariant: nothing downstream changes), which shifts the stage-relative indices of the next stage.  What
    # must be bit-identical is the set of ORIGINAL token ids kept at every stage.
    def original_ids(kept_list):
        ids, out = None, []
        for k in kept_list:
            ids = k if ids is None else torch.gather(ids, 1, k)
            out.append(torch.sort(ids, 1).values)
        return out
    mine, theirs = original_ids([k.cpu() for k in m32.kept_token_indices]), original_ids(ref["kept"])
    kept_exact = all(torch.equal(a, b) for a, b in zip(mine, theirs))
    order_same = all(torch.equal(m32.kept_token_indices[s].cpu(), ref["kept"][s]) for s in range(3))
    rel32 = float((l32 - ref["logits"]).abs().max() / ref["logits"].abs().max())
    del m32
    sdr = {k: (v.bfloat16().float() if v.is_floating_point() else v) for k, v in sd32.items()}
    refr = om.variant_a_eval(sdr, cfg, img)
    with torch.no_grad():
        l16 = model16(img.to(dev, torch.bfloat16)).float().cpu()
    k16 = model16.kept_token_indices[0].cpu()
    s32 = refr["scores"][0][:, :, 0]
    K = k16.shape[1]
    srt = torch.sort(s32, dim=-1, descending=True).values
    near = ((s32 - srt[:, K - 1:K]).abs() < 0.05).sum(1)
    a, b = torch.zeros(8, 196, dtype=torch.bool), torch.zeros(8, 196, dtype=torch.bool)
    a.scatter_(1, k16, True)
    b.scatter_(1, refr["kept"][0], True)
    flips = (a ^ b).sum(1)
    margin_ok = bool((flips <= 2 * near).all()) and bool((flips[(srt[:, K - 1] - srt[:, K]) > 0.05] == 0).all())
    out = {"images": 8, "oracle": "oracle.model.variant_a_eval (CPU fp32; equals the unmodified reference to 2e-6 at this config)",
           "fp32_kept_token_sets_bit_exact": kept_exact, "fp32_kept_order_identical": order_same, "fp32_logits_max_rel": rel32,
           "bf16_stage1_flipped_tokens": int(flips.sum()), "bf16_flips_within_fp32_score_margin": margin_ok,
           "bf16_logits_rel_l2_incl_flips": float((l16 - refr["logits"]).norm() / refr["logits"].norm()),
           "ok": bool(kept_exact and rel32 <= 1e-4 and margin_ok and bool(torch.isfinite(l16).all()))}
    if not out["ok"]:
        raise SystemExit("bench.py: parity gate failed, nothing is timed: " + json.dumps(out))
    return out


# ---------------------------------------------------------------------------------------------------
# per-kernel breakdown (graph-timed)
# ---------------------------------------------------------------------------------------------------
def kernel_breakdown(ops, B, dev, torch, pk):
    """Time every d2s kernel of one forward alone, at the shapes the step launches them with.
    Returns (rows, roofline dict for the dominant kernel)."""
    D, H, hd, N0 = 384, 6, 64, 196
    e = 2  # bf16
    rows = []
    bf = torch.bfloat16
    Ks = [int(N0 * r) for r in RATIOS]
    Ts = [N0 + 1] + [k + 1 for k in Ks]                   # tokens per block group: 197, 138, 97, 68
    agg = {k: dict(ms=0.0, by=0.0, fl=0.0, n=0) for k in ("attn", "pair", "mlp")}

    def acc(key, ms, by, fl, n):
        a = agg[key]
        a["ms"] += n * ms; a["by"] += n * by; a["fl"] += n * fl; a["n"] += n

    gw, gb = torch.ones(D, device=dev, dtype=bf), torch.zeros(D, device=dev, dtype=bf)
    wp = torch.randn(D, D, device=dev, dtype=bf) * 0.05
    w1 = torch.randn(4 * D, D, device=dev, dtype=bf) * 0.05
    w2 = torch.randn(D, 4 * D, device=dev, dtype=bf) * 0.02
    b1 = torch.zeros(4 * D, device=dev, dtype=bf)
    for gi, T in enumerate(Ts):
        by_attn = B * (e * 4 * T * D)                      # q,k,v in + out, bf16 (SURVEY.md 8d row 4)
        ns = nsets_for(by_attn)
        qkvs = [torch.randn(B, T, 3 * D, device=dev, dtype=bf) for _ in range(ns)]
        ms = time_graphed([lambda q=q: ops.attention_core(q, H) for q in qkvs], torch, launches=12)
        fl = B * 4.0 * H * T * T * hd
        rows.append(row("attn_policy_fwd(tcgen05)", f"B={B},T={T},H={H},hd={hd}", ms, by_attn, 3, fl))
        acc("attn", ms, by_attn, fl, 3)
        del qkvs
        xs = [(torch.randn(B, T, D, device=dev, dtype=bf), torch.randn(B, T, D, device=dev, dtype=bf)) for _ in range(2)]
        # qkv projection on the CTA-pair GEMM (192-column tiles, input rows resident): write-bound, 3 of its 4 (B,T,D) units are stores
        wq, bq = torch.randn(3 * D, D, device=dev, dtype=bf) * 0.05, torch.zeros(3 * D, device=dev, dtype=bf)
        by, fl = B * T * e * 4 * D, 2.0 * B * T * D * 3 * D
        sts_q = [torch.stack([x.float().mean(-1), torch.rsqrt(x.float().var(-1, unbiased=False) + 1e-6)], -1).reshape(-1, 2).contiguous()
                 for x, _ in xs]
        ms = time_graphed([lambda x=x, st=st: ops.linear_act(x, wq, bq, ops.ACT_NONE, in_stats=st, in_ln_weight=gw, in_ln_bias=gb)
                           for (x, _), st in zip(xs, sts_q)], torch, launches=12)
        rows.append(row("linear_act(norm1 + qkv projection, tcgen05 pair, 192-column tiles)", f"M={B * T},N={3 * D},K={D}", ms, by, 3, fl))
        del sts_q
        # attn.proj + residual; norm2 is NOT materialised: the kernel writes x' and per-row (mean, rstd), the MLP kernel applies the norm
        by, fl = B * T * (e * 3 * D + 8), 2.0 * B * T * D * D
        ms = time_graphed([lambda x=x, y=y: ops.linear_residual_ln(y, wp, gb, x, eps=1e-6, want_norm=False, want_stats=True) for x, y in xs],
                          torch, launches=12)
        rows.append(row("linear_residual_ln(proj+add+row statistics, tcgen05 pair)", f"M={B * T},N={D},K={D}", ms, by, 3, fl))
        acc("pair", ms, by, fl, 3)
        # the MLP branch in one kernel (norm2 on its input tile + fc1 + GELU + fc2 + residual + next LayerNorm): the step's dominant
        # kernel, tensor-bound (4.7 MFLOP per token against 2.3 KB of HBM traffic: x' in (also the residual), x'' and hn out)
        sts = [torch.stack([x.float().mean(-1), torch.rsqrt(x.float().var(-1, unbiased=False) + 1e-6)], -1).reshape(-1, 2).contiguous()
               for x, _ in xs]
        # (x' and its statistics in, x'' and ITS statistics out: the next norm1 is applied by the qkv GEMM)
        by, fl = B * T * (e * 2 * D + 16), 4.0 * B * T * D * 4 * D
        ms = time_graphed([lambda x=x, st=st: ops.mlp_residual_ln(None, w1, b1, w2, gb, x, None, None, 1e-6, want_norm=False, in_stats=st,
                                                                  in_ln_weight=gw, in_ln_bias=gb, want_stats=True)
                           for (x, _), st in zip(xs, sts)], torch, launches=8)
        rows.append(row("mlp_residual_ln(norm2+fc1+GELU+fc2+add+row statistics, tcgen05 pair)", f"M={B * T},D={D},HID={4 * D}", ms, by, 2, fl))
        acc("mlp", ms, by, fl, 2)
        if gi < 3:   # the block in front of a pruning stage: the LayerNorm is the predictor's, over x[:, 1:]
            ms = time_graphed([lambda x=x, st=st: ops.mlp_residual_ln(None, w1, b1, w2, gb, x, gw, gb, 1e-6, norm_row0=1, in_stats=st,
                                                                      in_ln_weight=gw, in_ln_bias=gb) for (x, _), st in zip(xs, sts)],
                              torch, launches=8)
            by = B * (e * D * (2 * T + T - 1) + 8 * T)
            rows.append(row("mlp_residual_ln(... LN over x[:,1:])", f"M={B * T},D={D},HID={4 * D}", ms, by, 1, fl))
            acc("mlp", ms, by, fl, 1)
        del sts
        if gi == 0:  # the first block's norm1: token assembly fused with the LayerNorm
            pos, cls = torch.randn(1, T, D, device=dev, dtype=bf), torch.randn(1, 1, D, device=dev, dtype=bf)
            ps = [torch.randn(B, T - 1, D, device=dev, dtype=bf) for _ in range(2)]
            ms = time_graphed([lambda p=p: ops.assemble_layernorm(p, cls, pos, gw, gb, 1e-6) for p in ps], torch, launches=12)
            rows.append(row("assemble_layernorm(token assembly + norm1)", f"B={B},T={T},D={D}", ms, B * T * D * e * 3, 1))
            imgs = [torch.randn(B, 3, 224, 224, device=dev, dtype=bf) for _ in range(2)]
            ms = time_graphed([lambda i=i: ops.patchify(i, 16, 16) for i in imgs], torch, launches=12)
            rows.append(row("patchify(im2col)", f"B={B},3x224x224", ms, B * 3 * 224 * 224 * e * 2, 1))
            del imgs, ps
        del xs
    n_in = N0
    for s, K in enumerate(Ks):
        T_in = n_in + 1
        by = B * (3 * e * D * (K + 1) + 8 * (K + 1))
        ns = nsets_for(by)
        sets = []
        for _ in range(ns):
            x = torch.randn(B, T_in, D, device=dev, dtype=bf)
            kept, _ = ops.select_topk(torch.rand(B, n_in, device=dev), K, ops.ORDER_SCORE_DESC, want_dropped=False)
            sets.append((x, kept))
        ms = time_graphed([lambda x=x, k=k: ops.gather_layernorm(x, k, gw, gb, 1e-6) for x, k in sets], torch)
        rows.append(row("gather_layernorm(kept-token gather + norm1)", f"B={B},T={T_in},D={D},K={K}", ms, by, 1))
        del sets
        # second half of the predictor + selection as one tcgen05 kernel (what engine.predictor_a_select launches after the first
        # Linear and pool_act): reads local (B,N,D/2) and the per-image bias rows, writes log-probs, kept indices, gathered decisions
        prev = (torch.rand(B, n_in, device=dev) > 0.1).float() if s else None
        H2 = D // 2
        by = B * (e * n_in * H2 + e * H2 + 8 * n_in + 8 * K + 4 * K + (4 * n_in if s else 0))
        w2, w3, b3 = (torch.randn(H2, D, device=dev) * 0.05).to(bf), (torch.randn(H2 // 2, H2, device=dev) * 0.07).to(bf), torch.zeros(H2 // 2, device=dev, dtype=bf)
        W, bias = torch.randn(2, D // 4, device=dev) * 0.1, torch.zeros(2, device=dev)
        pim = torch.randn(B, H2, device=dev, dtype=bf) * 0.3
        locs = [torch.randn(B, n_in, H2, device=dev, dtype=bf) * 0.5 for _ in range(nsets_for(by))]
        if ops.predictor_a_tail_ok(locs[0], w2, w3, W):
            ms = time_graphed([lambda h=h: ops.predictor_a_tail(h, pim, w2, w3, b3, W, bias, K, prev=prev) for h in locs], torch)
            rows.append(row("predictor_a_tail(Linear+GELU x2 + Linear + log-softmax + top-K + prev gather, tcgen05)",
                            f"B={B},N={n_in},C={H2},K={K}", ms, by, 1))
        zs = [torch.randn(B, n_in, D, device=dev, dtype=bf) for _ in range(nsets_for(B * n_in * D * e * 1.5))]
        ms = time_graphed([lambda z=z: ops.pool_act(z, prev, ops.ACT_GELU) for z in zs], torch)
        rows.append(row("pool_act(GELU + policy-weighted mean pool)", f"B={B},N={n_in},C={D}", ms, B * n_in * D * e * 1.5, 1))
        n_in = K
        del locs, zs
    # dominant kernel of the step (profiles/: ~38 % of the serialised step): the one-kernel MLP.  Tensor-bound: 4 * D * 4D flops
    # per token against 4 * D * 2 bytes of HBM traffic (the hidden activations stay on chip).  Aggregated over its launches at
    # the four token counts; peak = the measured burst bf16 GEMM rate (the kernel is timed alone).
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            tj = json.load(fh)["mlp_pair_kernel"]
            traffic = tj["dram_bytes_per_step"] / tj["launches_per_step"]
    except (OSError, KeyError, ValueError):
        pass
    m, p, a = agg["mlp"], agg["pair"], agg["attn"]
    roof = {"kernel": f"mlp_pair_kernel (norm2 + fc1 + GELU + fc2 + residual + LayerNorm, {m['n']} launches/step, T=197/138/97/68)",
            "bound": "tensor", "achieved": m["fl"] / m["ms"] / 1e9, "peak": pk["tf_burst"], "unit": "TFLOP/s",
            "frac": m["fl"] / m["ms"] / 1e9 / pk["tf_burst"], "traffic": traffic, "peak_source": pk["source"],
            "flops_per_launch": m["fl"] / m["n"], "algo_bytes_per_launch": m["by"] / m["n"], "ms_per_launch": m["ms"] / m["n"],
            "ms_per_step_in_kernel": m["ms"],
            "frac_of_sustained_peak": m["fl"] / m["ms"] / 1e9 / pk["tf_sustained"],
            "hbm": {"achieved": m["by"] / m["ms"] / 1e6, "peak": pk["hbm"], "unit": "GB/s", "frac": m["by"] / m["ms"] / 1e6 / pk["hbm"]},
            "proj_ln": {"kernel": f"gemm_pair_kernel<LN> (proj + residual + row statistics, {p['n']} launches/step)", "bound": "hbm",
                        "achieved": p["by"] / p["ms"] / 1e6, "frac": p["by"] / p["ms"] / 1e6 / pk["hbm"],
                        "ms_per_step_in_kernel": p["ms"]},
            "attention": {"kernel": f"attn_tc_fwd_kernel ({a['n']} launches/step)", "bound": "hbm",
                          "achieved": a["by"] / a["ms"] / 1e6, "frac": a["by"] / a["ms"] / 1e6 / pk["hbm"],
                          "ms_per_step_in_kernel": a["ms"],
                          "tensor": {"achieved": a["fl"] / a["ms"] / 1e9, "frac": a["fl"] / a["ms"] / 1e9 / pk["tf_burst"]}},
            "timing": "each kernel alone, launches captured in a CUDA graph (no host launch time), rotating argument sets > 2x L2"}
    return rows, roof


# ---------------------------------------------------------------------------------------------------
# BASELINE configs[3]: PerturbedTopK, configs[4]: select / gather sweep
# ---------------------------------------------------------------------------------------------------
def ptopk_leg(ops, dev, torch, pk):
    N, K, S = 196, 98, 500
    out = []
    for B in (1, 8, 64, 256):
        nsets = nsets_for(B * 4 * S * N)
        xs = [torch.softmax(torch.randn(B, N, device=dev), -1) for _ in range(nsets)]
        noises = [torch.randn(B, S, N, device=dev) for _ in range(nsets)]
        ind = torch.empty(B, K, N, device=dev)
        eg = torch.empty(B, K, N, device=dev)
        gx = torch.empty(B, N, device=dev)
        go = torch.randn(B, K, N, device=dev)
        call = ops._lib.call
        st = lambda: torch.cuda.current_stream().cuda_stream   # noqa: E731
        f_ms = time_graphed([lambda x=x, nz=nz: call("d2s_ptopk_fwd", x.data_ptr(), nz.data_ptr(), B, N, K, S, 0.05, ind.data_ptr(),
                                                     eg.data_ptr(), st()) for x, nz in zip(xs, noises)], torch)
        r_ms = time_graphed([lambda x=x: call("d2s_ptopk_fwd_rng", x.data_ptr(), 7, B, N, K, S, 0.05, ind.data_ptr(), eg.data_ptr(), st())
                             for x in xs], torch)
        b_ms = time_graphed([lambda: call("d2s_ptopk_bwd", go.data_ptr(), eg.data_ptr(), B, N, K, gx.data_ptr(), st())], torch)
        f_by, b_by = B * (4 * N + 4 * S * N + 8 * K * N), B * (8 * K * N + 4 * N)
        out.append({"B": B, "fwd_us": f_ms * 1e3, "fwd_gbs": f_by / f_ms / 1e6, "fwd_frac_hbm": f_by / f_ms / 1e6 / pk["hbm"],
                    "fwd_rng_us": r_ms * 1e3, "bwd_us": b_ms * 1e3, "bwd_gbs": b_by / b_ms / 1e6,
                    "fwd_bwd_us": (f_ms + b_ms) * 1e3, "selections_per_s": B * S / f_ms * 1e3,
                    "reference_materialises_bytes": B * S * K * N * (4 + 8)})
        del xs, noises
    return {"config": "PerturbedTopK N=196 (DeiT-B/16 spatial tokens), k=98, num_samples=500, sigma=0.05, injected noise; fwd also "
                      "writes the backward's expected-gradient tensor; algorithmic bytes per SURVEY.md 8d row (2)", "rows": out}


def sweep_leg(ops, dev, torch, pk):
    N = 196
    rows = []
    for B in (1, 8, 64, 1024, 4096):
        for ratio in (0.3, 0.7, 0.9):
            if B < 64 and ratio != 0.7:
                continue                              # the launch-bound batches at the headline keep rate only
            K = int(N * ratio)
            scs = [torch.rand(B, N, device=dev) for _ in range(nsets_for(B * 12 * N))]
            ms = time_graphed([lambda s=s: ops.select_topk(s, K, ops.ORDER_INDEX_ASC) for s in scs], torch)
            rows.append(row("select_topk(index asc, +dropped)", f"B={B},N={N},K={K}", ms, B * (4 * N + 8 * N)))
            kept, _ = ops.select_topk(scs[0], K, ops.ORDER_INDEX_ASC)
            for D in (384, 768):
                for dt, e, name in ((torch.bfloat16, 2, "bf16"), (torch.float32, 4, "f32")):
                    if B == 4096 and ratio != 0.7:
                        continue                      # the largest batch at the headline keep rate only
                    by_f = B * (2 * e * D * (K + 1) + 8 * (K + 1))
                    xs = [torch.randn(B, N + 1, D, device=dev, dtype=dt) for _ in range(nsets_for(by_f))]
                    ms = time_graphed([lambda x=x: ops.gather_tokens(x, kept) for x in xs], torch, launches=16)
                    rows.append(row("gather_tokens fwd", f"B={B},T={N + 1},D={D},K={K},{name}", ms, by_f))
                    del xs
                    by_b = B * (e * D * ((K + 1) + (N + 1)) + 8 * (K + 1))
                    gs = [torch.randn(B, K + 1, D, device=dev, dtype=dt) for _ in range(nsets_for(by_b))]
                    ms = time_graphed([lambda g=g: ops.scatter_tokens_bwd(g, kept, N + 1) for g in gs], torch, launches=16)
                    rows.append(row("scatter_tokens bwd", f"B={B},T={N + 1},D={D},K={K},{name}", ms, by_b))
                    del gs
    for r in rows:
        r["frac_hbm"] = r["gbs"] / pk["hbm"]
    return {"config": "N=196; D in {384,768}; keep 0.3/0.7/0.9; B in {1,8,64,1024,4096} (B < 64 and B = 4096 at keep 0.7 only); bf16 and fp32; HBM fraction of the measured peak",
            "rows": rows}


# ---------------------------------------------------------------------------------------------------
# BASELINE configs[2]: training step
# ---------------------------------------------------------------------------------------------------
def train_leg(pkg, args, dev, rank, world, torch, dist, pk):
    B = args.train_batch
    torch.manual_seed(0)
    student = pkg.variant_a.DefaultVisionTransformerDiffPruning(pruning_loc=LOCS, token_ratio=RATIOS, distill=True, **DEIT_S)
    seeded_weights(student)
    student = student.to(dev).train()
    teacher = pkg.variant_a.DefaultVisionTransformerTeacher(**DEIT_S).to(dev).eval()
    for p in teacher.parameters():
        p.requires_grad_(False)
    crit = pkg.losses.DistillDiffPruningLoss(teacher, keep_ratio=RATIOS)
    if args.torch_adamw:
        opt = torch.optim.AdamW(student.parameters(), lr=5e-4, weight_decay=0.05, capturable=True)
        grads = pkg.runner.FlatGrads(student.parameters())
        wcache = pkg.ops.BF16WeightCache(student.parameters())
    else:            # AdamW as one d2s kernel over flat (parameter, gradient, moment) buffers; it also writes the bf16 weight copies
        opt = pkg.runner.FlatAdamW(student.parameters(), lr=5e-4, weight_decay=0.05)
        grads, wcache = opt.grads, opt.weight_cache
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    x = torch.randn(B, 3, 224, 224, device=dev, generator=g)
    y = torch.randint(0, 1000, (B,), device=dev, generator=g)

    tstream = torch.cuda.Stream(device=dev) if args.teacher_stream else None

    def fwd_loss(xx, yy):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if tstream is not None:          # the frozen teacher's forward on a second stream, concurrent with the student's
                crit.start_teacher(xx, tstream)
            return crit(xx, student(xx), yy)[0]

    n0 = pkg._lib.launch_count()
    run = pkg.runner.TrainStepRunner(fwd_loss, opt, x, y, warmup=2, use_graph=not args.no_graph, grads=grads, weight_cache=wcache)
    per_step = (pkg._lib.launch_count() - n0) // (3 if not args.no_graph else 2)
    W, K = 3, args.train_steps
    for _ in range(W):
        run()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        loss = run()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    # host -> device fed variant of the same step: pinned fp32 images + labels copied in every step (the e2e form)
    hx, hy = x.cpu().pin_memory(), y.cpu().pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run.prefetch(hx, hy)                    # the copy of step k + 1 runs on a copy stream under step k
    for k in range(K):
        loss = run.step_prefetched()
        if k + 1 < K:
            run.prefetch(hx, hy)
    lv = float(loss.detach())               # device -> host read of the step's result
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.barrier()
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    t = float(ms.item()) / K
    val = world * B / (t / 1e3)
    grad_bytes = grads.flat.numel() * 4
    out = {"metric": "training images/sec DynamicViT (Variant A, 3 stages @3,6,9) DeiT-S kr=0.7 @224", "value": val, "unit": UNIT,
           "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": t, "batch_per_gpu": B, "dtype": "bf16 autocast, fp32 master weights",
           "workload": "student fwd+bwd (Gumbel keep decisions, policy attention at T=197) + frozen DeiT-S teacher fwd + "
                       "DistillDiffPruningLoss (cls + ratio + cls-KL + token-KL) + AdamW",
           "cuda_graph": not args.no_graph, "d2s_launches_per_step": int(per_step), "final_loss": lv,
           "e2e": {"value": world * B * K / float(e2e_s.item()), "unit": UNIT, "h2d_bytes_per_step": hx.numel() * 4 + hy.numel() * 8,
                   "d2h_bytes_per_step": 4},
           "collective": (f"one NCCL all-reduce of the flat fp32 gradient buffer ({grad_bytes / 1e6:.1f} MB) per step, captured in the "
                          f"step's CUDA graph between backward and AdamW" if world > 1 else "none (single GPU)"),
           "allreduce_floor_ms": (2 * (world - 1) / world * grad_bytes / 725e9 * 1e3) if world > 1 else 0.0,
           "teacher": "second stream, concurrent with the student forward (forks from and rejoins the captured stream)" if args.teacher_stream else "inline",
           "optimizer": "torch.optim.AdamW(capturable)" if args.torch_adamw else "runner.FlatAdamW (d2s_adamw_flat_f32: one launch, also writes the bf16 weight copies)",
           "limiter": "tensor + HBM bound single-GPU step; the all-reduce is not overlapped with backward (it is ~1-2 % of the step)",
           "tensor_frac_of_sustained_peak": val / world * TRAIN_GFLOP_PER_IMG / 1e3 / pk["tf_sustained"]}
    wcache.close()
    grads.close()
    del run, student, teacher, opt, grads, wcache
    torch.cuda.empty_cache()
    return out


def base_leg(pkg, dev, torch, pk, K, no_graph=False):
    """DeiT-B widths (D = 768, 12 heads, hidden 3072; dynamic_vit.py:1301-1303) through the same inference path: attention on
    the tcgen05 kernel, proj / fc2 + residual + LayerNorm as the CTA-pair GEMM with the row kept in two 384-column halves,
    fc1 + GELU as the CTA-pair GEMM; qkv stays the library GEMM and the hidden activations make an HBM round trip (the
    128 x 768 fp32 fc2 accumulator does not fit next to the hidden chunks in TMEM)."""
    B = 512
    model = pkg.variant_a.DefaultVisionTransformerDiffPruning(pruning_loc=LOCS, token_ratio=RATIOS, distill=True, **DEIT_B)
    seeded_weights(model)
    runner = pkg.runner.InferenceRunner(model, B, dev, dtype=torch.bfloat16, use_graph=not no_graph, warmup=2)
    n0 = pkg._lib.launch_count()
    with torch.no_grad():
        runner.model(runner.static_in)
    torch.cuda.synchronize()
    launches = pkg._lib.launch_count() - n0
    g = torch.Generator(device=dev).manual_seed(7)
    runner.static_in.copy_(torch.randn(runner.static_in.shape, device=dev, generator=g).to(runner.static_in.dtype))
    for _ in range(3):
        runner.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        runner.replay()
    e1.record()
    torch.cuda.synchronize()
    out = runner.logits
    ms = e0.elapsed_time(e1) / K
    gflop = 4.0 * GFLOP_PER_IMG * 0.985      # widths x2 -> GEMM FLOPs x4; the attention part (score / PV) grows x2 only
    val = B / (ms / 1e3)
    res = {"metric": "images/sec DynamicViT DeiT-B kr=0.7 @224", "value": val, "unit": UNIT, "ms_per_step": ms, "batch": B,
           "dtype": "bf16", "cuda_graph": not no_graph, "d2s_launches_per_step": int(launches), "outputs_finite": bool(torch.isfinite(out.float()).all()),
           "model_tensor_frac": {"gflop_per_img": gflop, "achieved_tflops": val * gflop / 1e3, "peak": pk["tf_sustained"],
                                 "frac": val * gflop / 1e3 / pk["tf_sustained"]},
           "path": "attn_tc_fwd + gemm_pair<LN> (N = 768: two halves) + gemm_pair<ACT> (fc1 + GELU); qkv on the library GEMM"}
    del runner, model
    torch.cuda.empty_cache()
    return res


def variant_b_leg(pkg, dev, torch, K, no_graph=False):
    """Dense2Sparse (Variant B, dynamic_vit.py:814-1015): one pruning stage at block 3, keep ratio 0.7, top-k selection, the
    large LayerNorm predictor, CLS-attention rows collected in every block.  Inference at batch 1024 (CUDA graph) and the
    reference's training loop (train.py:40-66: student + teacher with CLS attention, MaskLoss + BackboneLoss, AdamW) at batch
    256, eager -- the losses keep host-side running metrics."""
    import types
    kw = dict(pruning_loc=[3], token_ratio=[0.7], distill=True, topk_selection=True, predictor_loss_type="kl_div", **DEIT_S)
    model = pkg.variant_b.VisionTransformerDiffPruning(**kw)
    seeded_weights(model)
    B = 1024
    runner = pkg.runner.InferenceRunner(model, B, dev, dtype=torch.bfloat16, use_graph=not no_graph, warmup=2)
    g = torch.Generator(device=dev).manual_seed(11)
    runner.static_in.copy_(torch.randn(runner.static_in.shape, device=dev, generator=g).to(runner.static_in.dtype))
    for _ in range(3):
        runner.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        runner.replay()
    e1.record()
    torch.cuda.synchronize()
    ms_inf = e0.elapsed_time(e1) / K
    finite = bool(torch.isfinite(runner.logits.float()).all())
    del runner, model
    torch.cuda.empty_cache()
    # ---- training loop of train.py
    Bt = 256
    torch.manual_seed(0)
    student = pkg.variant_b.VisionTransformerDiffPruning(**kw)
    seeded_weights(student)
    student = student.to(dev).train()
    teacher = pkg.variant_b.VisionTransformerTeacher(**DEIT_S).to(dev).eval()
    for p in teacher.parameters():
        p.requires_grad_(False)
    mask_loss = pkg.losses.MaskLoss(types.SimpleNamespace(keep_ratios=[0.7], mask_loss_type="kl_div", batch_size=Bt, device=dev), "train")
    backbone_loss = pkg.losses.BackboneLoss(types.SimpleNamespace(mixup=0.0, patch_score_threshold=None))
    opt = pkg.runner.FlatAdamW(student.parameters(), lr=5e-4, weight_decay=0.05)
    x = torch.randn(Bt, 3, 224, 224, device=dev, generator=g)
    y = torch.randint(0, 1000, (Bt,), device=dev, generator=g)
    metrics = {}

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            with torch.no_grad():
                logits_t, token_t, cls_attn = teacher(x)
            logits_s, token_s, pred_logits, kept = student(x)
            loss = mask_loss(pred_logits, cls_attn, kept, metrics) + backbone_loss(logits_s, token_s, logits_t, token_t, kept, y, metrics)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss
    for _ in range(3):
        loss = step()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(K):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms_tr = e0.elapsed_time(e1) / K
    out = {"inference": {"metric": "images/sec Dense2Sparse (Variant B) DeiT-S 1 stage@3 kr=0.7 @224", "value": B / (ms_inf / 1e3), "unit": UNIT,
                         "ms_per_step": ms_inf, "batch": B, "dtype": "bf16", "cuda_graph": not no_graph, "outputs_finite": finite,
                         "outputs": "logits + 12 CLS-attention rows + predictor logits + kept indices"},
           "train": {"metric": "training images/sec Dense2Sparse (Variant B) DeiT-S 1 stage@3 kr=0.7 @224", "value": Bt / (ms_tr / 1e3), "unit": UNIT,
                     "ms_per_step": ms_tr, "batch": Bt, "dtype": "bf16 autocast, fp32 master weights", "cuda_graph": False,
                     "final_loss": float(loss.detach()),
                     "workload": "train.py:40-66: student fwd+bwd + frozen teacher fwd (CLS attention rows) + MaskLoss(kl_div) + BackboneLoss + "
                                 "runner.FlatAdamW, eager (the losses keep host-side running metrics)"}}
    opt.close()
    del student, teacher, opt
    torch.cuda.empty_cache()
    return out


def gpu_eager_leg(sd, dev, B, torch):
    """The oracle's restatement of the reference forward (plain torch ops: F.linear / matmul / softmax / sort / gather -- what
    `reference_model.to(bfloat16).cuda()` executes) run by torch eager on this GPU at the benchmarked batch and dtype."""
    from oracle import model as om
    cfg = om.VitCfg(embed_dim=384, depth=12, num_heads=6, pruning_loc=LOCS, token_ratio=RATIOS)
    sd16 = {k: (v.to(dev, torch.bfloat16) if v.is_floating_point() else v.to(dev)) for k, v in sd.items()}
    x = torch.randn(B, 3, 224, 224, device=dev).bfloat16()
    with torch.no_grad():
        for _ in range(2):
            om.variant_a_eval(sd16, cfg, x)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = 5
        for _ in range(n):
            om.variant_a_eval(sd16, cfg, x)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    return {"value": B / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "kind": "port",
            "what": f"oracle.model.variant_a_eval on cuda tensors, torch eager (cuBLAS / ATen kernels), bf16, batch {B}, inputs resident"}


def h2d_leg(dev, B, world, torch, dist):
    host = [torch.zeros(B, 3, 224, 224, dtype=torch.bfloat16).pin_memory() for _ in range(2)]
    dst = [torch.empty(B, 3, 224, 224, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    for i in range(2):
        dst[i].copy_(host[i], non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 8
    e0.record()
    for i in range(n):
        dst[i & 1].copy_(host[i & 1], non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    nbytes = host[0].numel() * 2
    return {"bytes_per_step": nbytes, "ms_max_over_ranks": float(ms), "gbs_per_gpu": nbytes / float(ms) / 1e6,
            "img_s_ceiling": world * B / (float(ms) / 1e3),
            "what": "pinned bf16 image batch -> device, nothing else running, every rank at once (the e2e leg's copy ceiling)"}


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    import d2s
    pkg = d2s.pkg
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    legs = set(args.legs.split(","))
    if args.skip_cpu:
        legs.discard("cpu")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (d2s arm) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    B, K, W = args.batch, args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    model = pkg.variant_a.DefaultVisionTransformerDiffPruning(pruning_loc=LOCS, token_ratio=RATIOS, distill=True, **DEIT_S)
    sd = seeded_weights(model)
    runner = pkg.runner.InferenceRunner(model, B, dev, dtype=torch.bfloat16, use_graph=not args.no_graph, warmup=2)
    # the captured forward's kept-index tensors, which every replay rewrites (an eager forward rebinds model.kept_token_indices)
    graph_kept = list(runner.model.kept_token_indices)
    line = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic"}

    # ---- parity gate: nothing is timed unless the path about to be timed reproduces the oracle ----------------------
    if "parity" in legs and rank == 0:
        line["parity_checked"] = parity_gate(pkg, runner.model, sd, dev, torch)
    barrier()

    # kernels per forward: count one eager forward through the C ABI (the graph replays exactly these)
    n0 = pkg._lib.launch_count()
    with torch.no_grad():
        runner.model(runner.static_in)
    torch.cuda.synchronize()
    launches_per_step = pkg._lib.launch_count() - n0
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    runner.static_in.copy_(torch.randn(runner.static_in.shape, device=dev, generator=g).to(torch.bfloat16))

    # ---- value: inputs resident in HBM ------------------------------------------------------------
    for _ in range(W):
        runner.replay()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(K):
        runner.replay()
    ev1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    barrier()
    clocks = sampler.stop() if sampler else None
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    value = world * B * K / (total_ms / 1e3)
    logits_ok = bool(torch.isfinite(runner.logits.float()).all())
    if args.dump_outputs and rank == 0:
        kept = graph_kept if runner.graph is not None else runner.model.kept_token_indices
        dump_outputs(args.dump_outputs, {"logits": runner.logits, **{f"kept_token_indices_{s}": k for s, k in enumerate(kept)}})

    # ---- e2e: pinned host images -> device -> forward -> host logits, every step -----------------------
    e2e = None
    if "e2e" in legs:
        host = [torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(100 + i)).to(torch.bfloat16).pin_memory()
                for i in range(2)]
        h2d = host[0].numel() * host[0].element_size()
        d2h = runner.logits.numel() * runner.logits.element_size()
        for i in range(2):
            runner.step_prefetched(runner.prefetch(host[i & 1]))
        barrier()
        t0 = time.perf_counter()
        slot = runner.prefetch(host[0])
        out_host = None
        for i in range(K):
            # start the next step's copy before this step's compute is enqueued: the copy overlaps the compute
            nxt = runner.prefetch(host[(i + 1) & 1]) if i + 1 < K else None
            out_host = runner.step_prefetched(slot)
            slot = nxt
        torch.cuda.synchronize()
        e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        barrier()
        if world > 1:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        logits_ok = logits_ok and bool(torch.isfinite(out_host.float()).all())
        e2e = {"value": world * B * K / float(e2e_s.item()), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "note": "pinned bf16 host images, double-buffered H2D on a copy stream overlapping the previous step, "
                       "host logits read back every step; wall clock between device synchronisations"}
        del host
    h2d_only = h2d_leg(dev, B, world, torch, dist) if "h2d" in legs else None
    del runner
    torch.cuda.empty_cache()
    # the same end-to-end step fed with RAW uint8 pixels (normalisation inside the im2col kernel): half the bytes over PCIe
    e2e_u8 = None
    if "e2e" in legs:
        model_u8 = pkg.variant_a.DefaultVisionTransformerDiffPruning(pruning_loc=LOCS, token_ratio=RATIOS, distill=True, **DEIT_S)
        model_u8.load_state_dict(sd)
        ru = pkg.runner.InferenceRunner(model_u8, B, dev, dtype=torch.bfloat16, use_graph=not args.no_graph, warmup=2, uint8_input=True)
        host8 = [torch.randint(0, 256, (B, 3, 224, 224), generator=torch.Generator().manual_seed(200 + i), dtype=torch.uint8).pin_memory()
                 for i in range(2)]
        for i in range(2):
            ru.step_prefetched(ru.prefetch(host8[i & 1]))
        barrier()
        t0 = time.perf_counter()
        slot = ru.prefetch(host8[0])
        for i in range(K):
            nxt = ru.prefetch(host8[(i + 1) & 1]) if i + 1 < K else None
            out_host = ru.step_prefetched(slot)
            slot = nxt
        torch.cuda.synchronize()
        u8_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        barrier()
        if world > 1:
            dist.all_reduce(u8_s, op=dist.ReduceOp.MAX)
        e2e_u8 = {"value": world * B * K / float(u8_s.item()), "unit": UNIT, "h2d_bytes_per_step": host8[0].numel(),
                  "d2h_bytes_per_step": ru.logits.numel() * ru.logits.element_size(), "outputs_finite": bool(torch.isfinite(out_host.float()).all()),
                  "note": "pinned uint8 host images (raw pixels); ToTensor + Normalize run inside the patch-embedding im2col kernel, "
                          "bit-identical to host-side normalisation (tests/test_gpu_models.py::test_runner_uint8_input_...)"}
        del ru, model_u8, host8
    torch.cuda.empty_cache()

    # ---- training step (all ranks: the gradient all-reduce is the path's one collective) -----------------------------
    train = train_leg(pkg, args, dev, rank, world, torch, dist, pk) if "train" in legs else None

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- rank 0: per-kernel breakdown, roofline, kernel-family legs, baselines ----------------------------------------
    line.update({
        "value": value, "ms_per_step": total_ms / K,
        "config": {"workload": "DynamicViT DeiT-S/16 keep_rate=0.7 (3 stages @3,6,9; ratios 0.7/0.49/0.343) inference, "
                               "224px, batch 1024 per GPU, bf16, random (seeded) weights",
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world} (batch-sharded, no collective)",
                   "cuda_graph": not args.no_graph,
                   "l2": "inputs larger than L2: 308 MB of images and >1 GB of activations per step vs 126 MB L2",
                   "outputs_finite": logits_ok},
        "gpu_launches": int(launches_per_step * K), "d2s_launches_per_step": int(launches_per_step), "clocks": clocks,
        "model_tensor_frac": {"gflop_per_img": GFLOP_PER_IMG, "achieved_tflops": value / world * GFLOP_PER_IMG / 1e3,
                              "peak": pk["tf_sustained"], "frac": value / world * GFLOP_PER_IMG / 1e3 / pk["tf_sustained"],
                              "peak_source": pk["source"] + " (sustained)"}})
    # headline end-to-end number: the uint8-input form of the public API (same logits bit for bit; normalisation runs on the GPU);
    # the form fed with already-normalised bf16 tensors -- what round 1 reported, bound by the 2x larger copy -- stays beside it
    if e2e_u8 is not None:
        line["e2e"] = e2e_u8
        if e2e is not None:
            line["e2e_float_input"] = e2e
    elif e2e is not None:
        line["e2e"] = e2e
    if h2d_only is not None:
        line["h2d_only"] = h2d_only
    if train is not None:
        line["train"] = train
    time.sleep(2.0)   # kernels are timed alone against the BURST peaks: let the clocks recover from the sustained loops
    if "kernels" in legs:
        rows, roof = kernel_breakdown(pkg.ops, B, dev, torch, pk)
        own_ms = sum(r["us"] * 1e-3 * r["launches_per_step"] for r in rows)
        line.update({"roofline": roof, "d2s_kernel_ms_per_step": own_ms, "d2s_kernel_share_of_step": own_ms / (total_ms / K),
                     "kernels": rows})
        torch.cuda.empty_cache()
    if "ptopk" in legs:
        line["ptopk"] = ptopk_leg(pkg.ops, dev, torch, pk)
    if "sweep" in legs:
        line["sweep"] = sweep_leg(pkg.ops, dev, torch, pk)
    if "base" in legs and rank == 0:
        line["arch_base"] = base_leg(pkg, dev, torch, pk, K, args.no_graph)
    if "variant_b" in legs and rank == 0:
        line["variant_b"] = variant_b_leg(pkg, dev, torch, K, args.no_graph)
        torch.cuda.empty_cache()
    if "eager" in legs:
        line["gpu_eager_baseline"] = gpu_eager_leg(sd, dev, B, torch)
        torch.cuda.empty_cache()
    if "cpu" in legs:
        c = time_cpu(args.cpu_batch, steps=40, warmup=1, budget_s=15.0)
        line["cpu_baseline"] = {
            "value": c["img_s"], "unit": UNIT, "cores": c["cores"], "kind": "port",
            "sample": f"{c['steps']} forwards of batch {args.cpu_batch} fp32 (BASELINE configs[0]) through "
                      f"oracle.model.variant_a_eval, same architecture and pruning schedule"}
    _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_JSON_FD = None


def _emit(line):
    """The ONE JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def _stdout_for_json_only():
    """Libraries print to stdout too (NCCL's version banner under NCCL_DEBUG=VERSION lands in front of the JSON line):
    everything written to fd 1 from here on goes to stderr, the JSON line goes to a saved copy of the real stdout."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def main():
    args = parse()
    if not (args.impl != "reference" and args.gpus > 1 and "WORLD_SIZE" not in os.environ):   # (not in the torchrun launcher)
        _stdout_for_json_only()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_gpu(args)


if __name__ == "__main__":
    main()
