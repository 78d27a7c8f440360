"""Training attention beyond 256 tokens on one GPU: forward + backward of ops.attention_train on the key-blocked kernels
(d2s_attn_long_fwd_stats + d2s_attn_long_bwd) against the path they replace (engine.attention_pre_proj with _LONG_ATTN = False:
torch matmuls around ops.softmax_with_policy, (B,H,T,T) scores and probabilities saved for the backward); then a DeiT-S-width
training step at 384 px with the kernels switched on and off.

    python scripts/bench_attn_long_train.py [--out FILE.json] [--iters 10] [--skip-model]

Attention alone: B in {64, 256}, H in {6, 12}, T = 577 with and without a fractional keep policy (new path and baseline), T = 785
and 1025 (new path only; the baseline's softmax kernel stops at T = 1024, and 785 is timed for the scaling).  One timed call is
forward + backward (a loss sum(out * gout) with a fixed gout) on one of several argument sets whose total size exceeds twice the
126 MB L2, cycled, so every call reads its qkv from HBM; warm-up first, CUDA events around --iters calls per set, the two paths
alternated per case.  Peak memory: torch.cuda.max_memory_allocated over one call, above what was allocated before it.
Floors computed from the shapes: exponentials B H T^2 (recomputed once in the backward) at 16 per clock per SM (MUFU ex2) at the
card's maximum SM clock, and the five B H T^2 64 MMAs of the backward (2 FLOP each) at 2250 TFLOP/s dense bf16 (data sheet).
The card's name, power limit and maximum SM clock are read in the same run.
Model: DeiT-S/16 width, depth 12, 384 px, B = 64, bf16 autocast, forward + cross-entropy + backward (no optimizer step),
kernels on / off alternated in one process: img/s and peak memory.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import d2s  # noqa: E402

pkg = d2s.pkg
HD = 64
L2_BYTES = 126 * 2 ** 20
TENSOR_FLOPS = 2.25e15


def card():
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None, "sm_max_mhz": None, "sm_mhz_now": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"], info["sm_mhz_now"] = float(q[0]), float(q[1]), float(q[2])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def baseline(qkv, H, policy):
    """engine.attention_pre_proj's torch branch (what bf16 training above 256 tokens ran before the key-blocked kernels)."""
    B, T, C3 = qkv.shape
    C = C3 // 3
    q, k, v = qkv.reshape(B, T, 3, H, HD).permute(2, 0, 3, 1, 4).unbind(0)
    attn = pkg.ops.softmax_with_policy((q @ k.transpose(-2, -1)) * HD ** -0.5, policy)
    return (attn @ v).transpose(1, 2).reshape(B, T, C)


def kernel(qkv, H, policy):
    return pkg.ops.attention_train(qkv, H, policy=policy)[0]


def fwd_bwd(fn, qkv, H, pol, go):
    q = qkv.detach().requires_grad_(True)
    p = pol.detach().requires_grad_(True) if pol is not None else None
    o = fn(q, H, p)
    o.backward(go)
    return q.grad


def time_case(fn, sets, H, iters):
    for s in sets:                         # warm-up every argument set
        fwd_bwd(fn, *s[:1], H, *s[1:])
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fwd_bwd(fn, sets[0][0], H, *sets[0][1:])
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters * len(sets)):
        s = sets[i % len(sets)]
        fwd_bwd(fn, s[0], H, *s[1:])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / (iters * len(sets)), peak


def floors(B, H, T, clk_hz):
    ex2 = B * H * T * T * 2                # forward and backward each exponentiate every score once
    mma_bwd = 5 * 2 * B * H * T * T * HD
    return {"ex2_bwd_us": (ex2 / 2) / (16 * 148 * clk_hz) * 1e6 if clk_hz else None,
            "ex2_fwd_bwd_us": ex2 / (16 * 148 * clk_hz) * 1e6 if clk_hz else None,
            "tensor_bwd_us": mma_bwd / TENSOR_FLOPS * 1e6,
            "tensor_fwd_bwd_us": (mma_bwd + 2 * 2 * B * H * T * T * HD) / TENSOR_FLOPS * 1e6}


def kernel_cases(res, iters, clk_hz):
    rows = []
    for B in (64, 256):
        for H in (6, 12):
            for T, pol_on in ((577, False), (577, True), (785, True), (1025, True)):
                g = torch.Generator(device="cuda").manual_seed(T + H + B)
                per_set = B * T * 3 * H * HD * 2 * 2
                nsets = max(2, -(-2 * L2_BYTES // per_set))
                sets = []
                for _ in range(nsets):
                    qkv = (torch.randn(B, T, 3 * H * HD, device="cuda", generator=g) * 0.7).bfloat16()
                    pol = torch.rand(B, T, device="cuda", generator=g) if pol_on else None
                    if pol is not None:
                        pol[:, 0] = 1
                    go = (torch.randn(B, T, H * HD, device="cuda", generator=g) * 0.5).bfloat16()
                    sets.append((qkv, pol, go))
                row = {"B": B, "H": H, "T": T, "policy": pol_on, **floors(B, H, T, clk_hz)}
                paths = [("kernel", kernel)] + ([("baseline", baseline)] if T == 577 else [])
                t = {n: [] for n, _ in paths}
                for _ in range(2):                               # alternate the paths
                    for n, fn in paths:
                        try:
                            ti, pk = time_case(fn, sets, H, iters)
                        except torch.cuda.OutOfMemoryError:
                            ti, pk = None, None
                            torch.cuda.empty_cache()
                        t[n].append(ti)
                        row[f"{n}_peak_mem_gb"] = pk / 1e9 if pk is not None else None
                for n in t:
                    ok = [x for x in t[n] if x is not None]
                    row[f"{n}_us"] = min(ok) * 1e6 if ok else None
                if row.get("baseline_us") and row.get("kernel_us"):
                    row["speedup"] = row["baseline_us"] / row["kernel_us"]
                if row.get("kernel_us") and row["ex2_fwd_bwd_us"]:
                    row["kernel_share_of_ex2_floor"] = row["ex2_fwd_bwd_us"] / row["kernel_us"]
                    row["kernel_share_of_tensor_floor"] = row["tensor_fwd_bwd_us"] / row["kernel_us"]
                rows.append(row)
                print(json.dumps(row), flush=True)
                del sets
                torch.cuda.empty_cache()
    res["attention"] = rows


def model_case(res, iters):
    B = 64
    m = pkg.variant_a.DefaultVisionTransformerTeacher(img_size=384, patch_size=16, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4,
                                                      qkv_bias=True, num_classes=1000).cuda().train()
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, 3, 384, 384, device="cuda", generator=gen)
    y = torch.randint(0, 1000, (B,), device="cuda", generator=gen)

    def step():
        m.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = m(x)
            logits = out[0] if isinstance(out, tuple) else out
            loss = torch.nn.functional.cross_entropy(logits.float(), y)
        loss.backward()

    times, peaks = {True: [], False: []}, {}
    for on in (True, False):                                     # warm-up both paths
        pkg.engine._LONG_ATTN = on
        step()
    for _ in range(3):
        for on in (True, False):
            pkg.engine._LONG_ATTN = on
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                step()
            e1.record()
            torch.cuda.synchronize()
            times[on].append(e0.elapsed_time(e1) * 1e-3 / iters)
            peaks[on] = torch.cuda.max_memory_allocated() / 1e9
    pkg.engine._LONG_ATTN = True
    row = {"model": "DeiT-S/16 width, depth 12, fine-tuning step (fwd + CE + bwd)", "img": 384, "B": B,
           "ms_kernel_on": [t * 1e3 for t in times[True]], "ms_kernel_off": [t * 1e3 for t in times[False]],
           "img_s_kernel_on": B / min(times[True]), "img_s_kernel_off": B / min(times[False]),
           "peak_mem_gb_kernel_on": peaks[True], "peak_mem_gb_kernel_off": peaks[False]}
    print(json.dumps(row), flush=True)
    res["model"] = row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--skip-model", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attn_long_train: no CUDA device (this measurement runs on the GPU only)")
    res = {"card": card()}
    clk = res["card"]["sm_max_mhz"]
    kernel_cases(res, args.iters, clk * 1e6 if clk else None)
    if not args.skip_model:
        model_case(res, args.iters)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
