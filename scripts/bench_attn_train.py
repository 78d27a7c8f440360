"""Training attention (ops.attention_train) forward + backward at BASELINE configs[2] shapes and at 208 < T <= 256 (the flash pair
at T <= 208, the key-blocked pair above), CUDA-event timed, with the gradient errors against torch fp32 autograd of the reference
formulas.  The card's name, power limit and maximum SM clock are read in the same run.  profiles/r06_attn_train_blocked_vs_gemm.json
holds these shapes against the head-major GEMM path the key-blocked pair replaced at 208 < T <= 256.

    python scripts/bench_attn_train.py [--B 256] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import d2s  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None, "sm_max_mhz": None, "sm_mhz_now": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"], info["sm_mhz_now"] = float(q[0]), float(q[1]), float(q[2])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def ref_attention(qkv, H, policy, eps=1e-6):
    B, T, _ = qkv.shape
    hd = qkv.shape[-1] // 3 // H
    v = qkv.view(B, T, 3, H, hd)
    q, k, vv = v[:, :, 0].transpose(1, 2), v[:, :, 1].transpose(1, 2), v[:, :, 2].transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * hd ** -0.5
    if policy is None:
        p = torch.softmax(s, -1)
    else:
        pp = policy.reshape(B, 1, 1, T)
        m = pp + (1 - pp) * torch.eye(T, device=qkv.device).view(1, 1, T, T)
        e = torch.exp(s - s.amax(-1, keepdim=True)) * m
        p = (e + eps / T) / (e.sum(-1, keepdim=True) + eps)
    return (p @ vv).transpose(1, 2).reshape(B, T, H * hd)


def timed(step, iters):
    for _ in range(3):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / iters


def case(B, T, H, with_pol, g, iters):
    hd = 64
    qkv = (torch.randn(B, T, 3 * H * hd, device="cuda", generator=g) * 0.7).bfloat16()
    pol = None
    if with_pol:
        pol = (torch.rand(B, T, 1, device="cuda", generator=g) > 0.3).float()
        pol[:, 0] = 1
    go = (torch.randn(B, T, H * hd, device="cuda", generator=g) * 0.5).bfloat16()
    q2 = qkv.float().requires_grad_(True)
    p2 = None if pol is None else pol.clone().requires_grad_(True)
    nb = 32                                             # fp32 reference on a slice (memory)
    o2 = ref_attention(q2[:nb], H, None if p2 is None else p2[:nb])
    (o2 * go[:nb].float()).sum().backward()
    row = {"B": B, "T": T, "H": H, "hd": hd, "policy": with_pol}
    q1 = qkv.clone().requires_grad_(True)
    p1 = None if pol is None else pol.clone().requires_grad_(True)

    def fwd():
        return d2s.pkg.ops.attention_train(q1, H, policy=p1)[0]

    def fwd_bwd():
        q1.grad = None
        fwd().backward(go)

    (fwd().float() * go.float()).sum().backward()
    dq = q1.grad[:nb].float()
    row["dqkv_relmax"] = float((dq - q2.grad[:nb]).abs().max() / q2.grad[:nb].abs().max())
    row["dqkv_rell2"] = float((dq - q2.grad[:nb]).norm() / q2.grad[:nb].norm())
    if pol is not None:
        row["dpol_relmax"] = float((p1.grad[:nb] - p2.grad[:nb]).abs().max() / p2.grad[:nb].abs().max())
        row["dpol_rell2"] = float((p1.grad[:nb] - p2.grad[:nb]).norm() / p2.grad[:nb].norm())
    row["fwd_us"] = timed(fwd, iters)
    row["fwd+bwd_us"] = timed(fwd_bwd, iters)
    hbm = B * T * H * hd * 2 * (4 + 8)                  # fwd: q,k,v in + o out; bwd: q,k,v,o,do in + dq,dk,dv out
    row["fwd+bwd_gbs"] = hbm / row["fwd+bwd_us"] / 1e3
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=256)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attn_train: no CUDA device (this measurement runs on the GPU only)")
    B = args.B
    res = {"card": card(), "rows": []}
    print(json.dumps(res["card"]), flush=True)
    g = torch.Generator(device="cuda").manual_seed(1)
    # T = 197 / 138 / 97: DeiT at 224 px before and after pruning (flash pair); 209 / 226 / 256: the key-blocked pair.  At B = 256,
    # H = 6, T = 226 one qkv tensor is 133 MB, above the 126 MB L2.
    shapes = [(197, 6, True), (197, 6, False), (138, 6, False), (97, 6, False)]
    shapes += [(T, 6, p) for T in (209, 226, 256) for p in (True, False)] + [(226, 12, True)]
    for T, H, with_pol in shapes:
        row = case(B, T, H, with_pol, g, args.iters)
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
