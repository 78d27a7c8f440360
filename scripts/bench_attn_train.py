"""Training attention (ops.attention_train) forward + backward at BASELINE configs[2] shapes: the tcgen05 flash kernels against
the head-major GEMM path they replace (D2S flag flipped in-process), CUDA-event timed, with the gradient errors of both
against torch fp32 autograd of the reference formulas.

    python scripts/bench_attn_train.py [B]
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import d2s  # noqa: E402


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


def main():
    ops = d2s.pkg.ops
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    H, hd = 6, 64
    g = torch.Generator(device="cuda").manual_seed(1)
    rows = []
    for T, with_pol in ((197, True), (197, False), (138, False), (97, False)):
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
        row = {"B": B, "T": T, "policy": with_pol}
        for name, fn in (("flash", ops._AttentionFlash.apply), ("gemm", ops._AttentionTrain.apply)):
            q1 = qkv.clone().requires_grad_(True)
            p1 = None if pol is None else pol.clone().requires_grad_(True)

            def fwd():
                return fn(q1, p1, H, float(hd ** -0.5), 1e-6, False)[0]

            o1 = fwd()
            (o1.float() * go.float()).sum().backward()
            dq = q1.grad[:nb].float()
            row[name + "_dqkv_relmax"] = float((dq - q2.grad[:nb]).abs().max() / q2.grad[:nb].abs().max())
            row[name + "_dqkv_rell2"] = float((dq - q2.grad[:nb]).norm() / q2.grad[:nb].norm())
            if pol is not None:
                row[name + "_dpol_relmax"] = float((p1.grad[:nb] - p2.grad[:nb]).abs().max() / p2.grad[:nb].abs().max())
                row[name + "_dpol_rell2"] = float((p1.grad[:nb] - p2.grad[:nb]).norm() / p2.grad[:nb].norm())
            for what in ("fwd", "fwd+bwd"):
                def step():
                    o = fwd()
                    if what != "fwd":
                        q1.grad = None
                        o.backward(go)
                for _ in range(3):
                    step()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(10):
                    step()
                e1.record()
                torch.cuda.synchronize()
                row[f"{name}_{what}_us"] = 100.0 * e0.elapsed_time(e1)
        hbm = B * T * H * hd * 2 * (4 + 8)                  # fwd: q,k,v in + o out; bwd: q,k,v,o,do in + dq,dk,dv out
        row["flash_fwd+bwd_gbs"] = hbm / row["flash_fwd+bwd_us"] / 1e3
        rows.append(row)
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
