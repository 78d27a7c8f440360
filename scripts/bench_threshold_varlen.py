"""Throughput of the dynamic keep-ratio (patch_score_threshold) inference on one GPU: the padded-batch forward (forward_varlen)
against the batch-1 form it replaces and against the fixed-ratio forward at the same mean keep ratios.

    python scripts/bench_threshold_varlen.py [--out FILE.json] [--iters 10]

Model: DeiT-S/16 Variant B, pruning stages at blocks 3 / 6 / 9, bf16, seeded random weights (torch.manual_seed(0) before the
module's own initialisation).  The threshold is calibrated first (bisection on a 256-image batch) so that the first stage keeps
on average ~70 % of its tokens; the fixed-ratio model then runs with token_ratio set to the measured mean kept fractions of the
three stages (relative to the 196 patch tokens, as token_ratio is defined), the same weights and eager execution (no CUDA graph:
the varlen forward cannot be captured, one host read per stage sizes the next one).
Reported: img/s of forward_varlen at B = 256 and 1024, of the batch-1 opt-in over 256 images, of the fixed-ratio forward at
B = 256 and 1024, and per stage the pad fraction 1 - sum(len) / (B * Tmax) of the padded layout; card name and power limit are
read in the same run.  Inputs are random normal images resident on the GPU (no host copies in the timed window).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import d2s  # noqa: E402

ARCH = dict(patch_size=16, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, qkv_bias=True, num_classes=1000)
LOCS = [3, 6, 9]
TARGET = 0.7


def card():
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def model(ratios, thr):
    torch.manual_seed(0)
    m = d2s.variant_b.VisionTransformerDiffPruning(pruning_loc=LOCS, token_ratio=ratios, distill=True, topk_selection=True,
                                                   predictor_loss_type="kl_div", patch_score_threshold=thr, **ARCH)
    return m.cuda().eval().to(torch.bfloat16)


def kept_counts(kept):
    return [(k >= 0).sum(dim=1) for k in kept]


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_threshold_varlen: no CUDA device (this measurement runs on the GPU only)")
    gen = torch.Generator(device="cuda").manual_seed(1)
    imgs = torch.randn(1024, 3, 224, 224, device="cuda", generator=gen).to(torch.bfloat16)
    m = model([0.7, 0.49, 0.343], 0.3)
    res = {"model": "DeiT-S/16 Variant B, stages [3, 6, 9], bf16, seeded random weights", "card": card()}
    with torch.no_grad():
        # threshold calibration: first-stage mean keep ratio ~ TARGET (it falls as the threshold rises)
        lo, hi = 0.0, 1.0
        for _ in range(14):
            m.patch_score_threshold = (lo + hi) / 2
            _, _, _, kept = m.forward_varlen(imgs[:256])
            r = float(kept_counts(kept)[0].float().mean()) / 196
            lo, hi = (m.patch_score_threshold, hi) if r > TARGET else (lo, m.patch_score_threshold)
        thr = m.patch_score_threshold
        _, _, _, kept = m.forward_varlen(imgs)
        counts = kept_counts(kept)
        ratios = [float(c.float().mean()) / 196 for c in counts]
        res["threshold"] = thr
        res["mean_keep_ratio_per_stage"] = ratios
        pads = []
        for c in counts:
            lens = c + 1
            pads.append(1.0 - float(lens.sum()) / (lens.numel() * int(lens.max())))
        res["pad_fraction_per_stage_B1024"] = pads
        for B in (256, 1024):
            x = imgs[:B]
            res[f"varlen_img_s_B{B}"] = B / timed(lambda: m.forward_varlen(x), args.iters)
        m.d2s_threshold_inference = True
        one = imgs[:256]
        res["batch1_opt_in_img_s_256_images"] = 256 / timed(lambda: [m(one[b:b + 1]) for b in range(256)], 1, warmup=1)
        f = model([r for r in ratios], None)
        f.load_state_dict(m.state_dict())
        for B in (256, 1024):
            x = imgs[:B]
            res[f"fixed_ratio_img_s_B{B}"] = B / timed(lambda: f(x), args.iters)
        res["fixed_ratio_token_ratio"] = ratios
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
