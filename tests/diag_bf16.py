"""Where does the bf16 deviation come from?  (developer diagnostic, run on the GPU box; not collected by pytest)

    python tests/diag_bf16.py [small|deit_s] ...

Truth = the fp32 oracle on the bf16-ROUNDED weights and images (identical inputs), so what is measured is compute precision
only.  Rows: the d2s bf16 path with its fusions on / off, plain torch eager in bf16 (the oracle's restatement executed on the
GPU in bf16 -- what `reference_model.to(torch.bfloat16)` computes), and the d2s fp32 path."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import d2s  # noqa: E402
import fixtures as fx  # noqa: E402
from oracle import model as om  # noqa: E402

CFGS = {"small": dict(embed_dim=128, depth=4, num_heads=2, locs=[1, 2]),
        "deit_s": dict(embed_dim=384, depth=12, num_heads=6, locs=[3, 6, 9])}


def err(a, ref):
    a, ref = a.float().cpu(), ref.float().cpu()
    return float((a - ref).abs().max() / ref.abs().max()), float((a - ref).norm() / ref.norm())


def main(names):
    pkg = d2s.pkg
    dev = torch.device("cuda:0")
    for name in names:
        c = CFGS[name]
        ratios = [1.0] * len(c["locs"])
        kw = dict(patch_size=16, embed_dim=c["embed_dim"], depth=c["depth"], num_heads=c["num_heads"], num_classes=16,
                  pruning_loc=c["locs"], token_ratio=ratios, distill=True)
        m = pkg.variant_a.DefaultVisionTransformerDiffPruning(**kw)
        sd = fx.seeded_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, 11)
        sdr = {k: (v.bfloat16().float() if v.is_floating_point() else v) for k, v in sd.items()}
        img = fx.randn(7, 8, 3, 224, 224).bfloat16().float()
        cfg = om.VitCfg(embed_dim=c["embed_dim"], depth=c["depth"], num_heads=c["num_heads"], num_classes=16,
                        pruning_loc=c["locs"], token_ratio=ratios)
        truth = om.variant_a_eval(sdr, cfg, img)["logits"]
        truth_unrounded = om.variant_a_eval(sd, cfg, img)["logits"]
        print(f"== {name}: max|logit| {float(truth.abs().max()):.3f}; weight rounding alone moves the fp32 logits by "
              f"{err(truth, truth_unrounded)}")
        m.load_state_dict(sdr)
        m = m.to(dev).eval()
        with torch.no_grad():
            l32 = m(img.to(dev))
        print(f"d2s fp32 GPU                      {err(l32, truth)}")
        m16 = m.to(torch.bfloat16)
        x16 = img.to(dev, torch.bfloat16)
        sd16 = {k: v.to(dev, torch.bfloat16) if v.is_floating_point() else v.to(dev) for k, v in sdr.items()}
        with torch.no_grad():
            lt = om.variant_a_eval(sd16, cfg, x16)["logits"]
        print(f"torch eager bf16 (oracle on GPU)  {err(lt, truth)}")
        with torch.no_grad():
            print(f"d2s bf16 fused                    {err(m16(x16), truth)}")
            for flags in (("_FUSED_MLP",), ("_FUSED_MLP", "_FUSED_PAIR")):
                for f in flags:
                    setattr(pkg.engine, f, False)
                print(f"d2s bf16 without {'+'.join(flags):<30} {err(m16(x16), truth)}")
                for f in flags:
                    setattr(pkg.engine, f, True)


if __name__ == "__main__":
    main(sys.argv[1:] or ["small", "deit_s"])
