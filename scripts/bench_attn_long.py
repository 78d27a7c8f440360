"""Attention beyond 256 tokens on one GPU: the key-blocked tcgen05 kernel (d2s_attn_long_fwd) against the torch fallback it
replaces (two library matmuls around the d2s policy-softmax kernel, a (B,H,T,T) score tensor in HBM), and at T = 197 against the
one-block kernel (d2s_attn_policy_fwd); then whole models at 384 / 512 px with the kernel switched on and off.

    python scripts/bench_attn_long.py [--out FILE.json] [--reps 20] [--iters 10] [--skip-models]

Kernel times: DeiT-S heads (H = 6, hd = 64), B = 256, T in {197, 577, 785, 1025}, with and without the CLS-row output.  Each
case is a CUDA graph of --reps launches cycling over argument sets (qkv, out[, cls_row]) whose total size exceeds twice the
126 MB L2, so every launch reads its qkv from HBM; the graph is replayed --iters times between CUDA events.  Bounds computed from
the shapes: HBM bytes (qkv read once, out / cls_row written once) at 7.7 TB/s, tensor FLOPs 4 B H T^2 64 at 2250 TFLOP/s dense
bf16, and exponentials B H T^2 at 16 per clock per SM (MUFU ex2) at the card's maximum SM clock, read with the power limit in the
same run.  The torch fallback is timed only where it runs (T <= 1024: its softmax kernel's limit).
Model level: DeiT-S/16 at 384 px through runner.InferenceRunner (CUDA graph, bf16, B = 256) -- the teacher, Variant A eval and
Variant B eval (fixed ratios 0.7 / 0.49 / 0.343, stages 3 / 6 / 9) -- with engine._LONG_ATTN on and off, timed in alternation
in the same process; forward_varlen (Variant B, threshold 0.3) at 384 px and the teacher at 512 px run with the kernel only
(the fallback path raises / cannot run there).  Inputs are seeded random normal images resident on the GPU.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import d2s  # noqa: E402

pkg = d2s.pkg
H, HD = 6, 64
L2_BYTES = 126 * 2 ** 20
HBM_BPS, TENSOR_FLOPS = 7.7e12, 2.25e15
DEIT_S = dict(patch_size=16, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, qkv_bias=True, num_classes=1000)
LOCS, RATIOS = [3, 6, 9], [0.7, 0.49, 0.343]


def card():
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None, "sm_max_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def fallback(qkv, want_cls):
    """engine.attention_pre_proj's torch path (what bf16 above 256 tokens ran before the key-blocked kernel)."""
    B, T, C3 = qkv.shape
    C = C3 // 3
    q, k, v = qkv.reshape(B, T, 3, H, HD).permute(2, 0, 3, 1, 4).unbind(0)
    attn = pkg.ops.softmax_with_policy((q @ k.transpose(-2, -1)) * HD ** -0.5, None)
    o = (attn @ v).transpose(1, 2).reshape(B, T, C)
    return o, (attn[:, :, 0, :] if want_cls else None)


def graph_time(fn, sets, reps, iters):
    """Mean time of one fn(*set) launch: `reps` launches cycling over `sets` captured in one CUDA graph, replayed `iters` times."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for a in sets:          # warm-up: module load, allocator, function attributes
            fn(*a)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for r in range(reps):
            fn(*sets[r % len(sets)])
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    del g
    return e0.elapsed_time(e1) * 1e-3 / (iters * reps)


def kernel_cases(res, reps, iters, clk_hz):
    B = 256
    out = []
    for T in (197, 577, 785, 1025):
        qkv_bytes, out_bytes = B * T * 3 * H * HD * 2, B * T * H * HD * 2
        nsets = max(2, math.ceil(2 * L2_BYTES / (qkv_bytes + out_bytes)) + 1)
        gen = torch.Generator(device="cuda").manual_seed(T)
        sets = [torch.randn(B, T, 3 * H * HD, device="cuda", generator=gen).bfloat16() for _ in range(nsets)]
        for want_cls in (False, True):
            row = {"B": B, "H": H, "T": T, "cls_row": want_cls, "arg_sets": nsets}
            nbytes = qkv_bytes + out_bytes + (B * H * T * 4 if want_cls else 0)
            flops, exps = 4.0 * B * H * T * T * HD, float(B * H * T * T)
            floors = {"hbm": nbytes / HBM_BPS, "tensor": flops / TENSOR_FLOPS}
            if clk_hz:
                floors["mufu_ex2"] = exps / (16 * 148 * clk_hz)
            row.update(bytes=nbytes, flops=flops, exponentials=exps, floors_us={k: v * 1e6 for k, v in floors.items()})
            outs = [(torch.empty(B, T, H * HD, dtype=torch.bfloat16, device="cuda"),
                     torch.empty(B, H, T, dtype=torch.float32, device="cuda") if want_cls else None) for _ in range(nsets)]
            lib = pkg._lib.load()
            stream = torch.cuda.current_stream

            def long_fn(q, o, c):
                rc = lib.d2s_attn_long_fwd(q.data_ptr(), None, None, B, T, H, HD, HD ** -0.5, 1e-6, o.data_ptr(),
                                           c.data_ptr() if c is not None else None, stream().cuda_stream)
                assert rc == 0, lib.d2s_last_error()
            args = [(sets[i], outs[i][0], outs[i][1]) for i in range(nsets)]
            t = graph_time(long_fn, args, reps, iters)
            bound = max(floors, key=floors.get)
            row["long_us"] = t * 1e6
            row["long_bound"] = bound
            row["long_share_of_bound"] = floors[bound] / t
            if T <= 256:
                def short_fn(q, o, c):
                    rc = lib.d2s_attn_policy_fwd(q.data_ptr(), None, 1, B, T, H, HD, HD ** -0.5, 1e-6, o.data_ptr(),
                                                 c.data_ptr() if c is not None else None, None, stream().cuda_stream)
                    assert rc == 0, lib.d2s_last_error()
                row["one_block_kernel_us"] = graph_time(short_fn, args, reps, iters) * 1e6
            if T <= 1024:
                row["torch_fallback_us"] = graph_time(lambda q, o, c: fallback(q, c is not None), args, max(2, reps // 4), iters) * 1e6
                row["speedup_vs_fallback"] = row["torch_fallback_us"] / row["long_us"]
                o_fb, c_fb = fallback(sets[0], True)
                o_k, c_k = pkg.ops.attention_long(sets[0], H, want_cls_row=True)
                row["max_abs_diff_vs_fallback"] = float((o_fb.float() - o_k.float()).abs().max())
            out.append(row)
            print(json.dumps(row), flush=True)
            del outs, args
        del sets
        torch.cuda.empty_cache()
    res["kernel"] = out


def make_model(kind, img, thr=None):
    torch.manual_seed(0)
    if kind == "teacher":
        m = pkg.variant_a.DefaultVisionTransformerTeacher(img_size=img, **DEIT_S)
    elif kind == "variant_a":
        m = pkg.variant_a.DefaultVisionTransformerDiffPruning(img_size=img, pruning_loc=LOCS, token_ratio=RATIOS, distill=True, **DEIT_S)
    else:
        m = pkg.variant_b.VisionTransformerDiffPruning(img_size=img, pruning_loc=LOCS, token_ratio=RATIOS, distill=True, topk_selection=True,
                                                       predictor_loss_type="kl_div", patch_score_threshold=thr, **DEIT_S)
    return m


def replay_time(runner, iters):
    runner.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        runner.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / iters


def model_cases(res, iters):
    B = 256
    gen = torch.Generator(device="cuda").manual_seed(1)
    x384 = torch.randn(B, 3, 384, 384, device="cuda", generator=gen).bfloat16()
    rows = []
    for kind in ("teacher", "variant_a", "variant_b"):
        runners = {}
        for on in (True, False):
            pkg.engine._LONG_ATTN = on
            r = pkg.runner.InferenceRunner(make_model(kind, 384), B, torch.device("cuda"), dtype=torch.bfloat16, img_shape=(3, 384, 384),
                                           use_graph=True, warmup=1)
            r.static_in.copy_(x384)
            runners[on] = r
        pkg.engine._LONG_ATTN = True
        times = {True: [], False: []}
        for _ in range(3):                       # alternate: on, off, on, off, ...
            for on in (True, False):
                times[on].append(replay_time(runners[on], iters))
        row = {"model": kind, "img": 384, "B": B, "ms_kernel_on": [t * 1e3 for t in times[True]],
               "ms_kernel_off": [t * 1e3 for t in times[False]]}
        row["img_s_kernel_on"] = B / min(times[True])
        row["img_s_kernel_off"] = B / min(times[False])
        rows.append(row)
        print(json.dumps(row), flush=True)
        del runners
        torch.cuda.empty_cache()
    with torch.no_grad():
        m = make_model("variant_b", 384, thr=0.3).cuda().eval().to(torch.bfloat16)
        m.forward_varlen(x384)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            m.forward_varlen(x384)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3 / iters
        row = {"model": "variant_b forward_varlen (threshold 0.3)", "img": 384, "B": B, "ms_kernel_on": t * 1e3, "img_s_kernel_on": B / t}
        rows.append(row)
        print(json.dumps(row), flush=True)
        del m
    torch.cuda.empty_cache()
    x512 = torch.randn(B, 3, 512, 512, device="cuda", generator=gen).bfloat16()
    r = pkg.runner.InferenceRunner(make_model("teacher", 512), B, torch.device("cuda"), dtype=torch.bfloat16, img_shape=(3, 512, 512),
                                   use_graph=True, warmup=1)
    r.static_in.copy_(x512)
    t = replay_time(r, iters)
    row = {"model": "teacher", "img": 512, "B": B, "ms_kernel_on": t * 1e3, "img_s_kernel_on": B / t}
    rows.append(row)
    print(json.dumps(row), flush=True)
    res["models"] = rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--skip-models", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attn_long: no CUDA device (this measurement runs on the GPU only)")
    res = {"card": card()}
    clk = res["card"]["sm_max_mhz"]
    kernel_cases(res, args.reps, args.iters, clk * 1e6 if clk else None)
    if not args.skip_models:
        model_cases(res, args.iters)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
