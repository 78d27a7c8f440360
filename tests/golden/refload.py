"""Load the UNMODIFIED reference hot-path modules from a checkout of marc345/Dense2Sparse-ViT (REF_ROOT).

Golden-generation infrastructure: used by make_goldens.py and make_loss_goldens.py only.  The tests, smoke()
and bench.py read the stored goldens and never import this module: the reference is not part of this repository.

The reference needs six timm names (vit_models/dynamic_vit.py:30-32,
vit_models/default_dynamic_vit.py:30-32); timm is not installed, so a stub
package is injected.  The files are loaded by path under a fake `vit_models`
package so the star-importing vit_models/__init__.py:1-13 (which pulls the whole
model zoo) is bypassed and `from .peturbed_topk import ...` still resolves.
"""
import importlib.util
import os
import sys
import types

import torch

REF_ROOT = os.environ.get("D2S_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "vit_models", "dynamic_vit.py"))


def _install_timm_stub():
    if "timm" in sys.modules and not getattr(sys.modules["timm"], "_d2s_stub", False):
        return  # a real timm exists; use it
    timm = types.ModuleType("timm")
    timm._d2s_stub = True
    data = types.ModuleType("timm.data")
    data.IMAGENET_DEFAULT_MEAN = (0.485, 0.456, 0.406)
    data.IMAGENET_DEFAULT_STD = (0.229, 0.224, 0.225)
    models = types.ModuleType("timm.models")
    layers = types.ModuleType("timm.models.layers")

    class DropPath(torch.nn.Module):  # never instantiated: every factory uses drop_path_rate=0
        def __init__(self, p=0.0):
            super().__init__()
            self.p = p

        def forward(self, x):
            if self.p == 0.0 or not self.training:
                return x
            raise NotImplementedError("stub DropPath only supports p=0")

    def to_2tuple(x):
        return tuple(x) if isinstance(x, (tuple, list)) else (x, x)

    layers.DropPath = DropPath
    layers.to_2tuple = to_2tuple
    layers.trunc_normal_ = torch.nn.init.trunc_normal_
    registry = types.ModuleType("timm.models.registry")
    registry.register_model = lambda fn: fn
    loss = types.ModuleType("timm.loss")

    class SoftTargetCrossEntropy(torch.nn.Module):
        def forward(self, x, target):
            return torch.sum(-target * torch.nn.functional.log_softmax(x, dim=-1), dim=-1).mean()

    loss.SoftTargetCrossEntropy = SoftTargetCrossEntropy
    timm.data, timm.models, timm.loss = data, models, loss
    models.layers, models.registry = layers, registry
    for name, mod in [("timm", timm), ("timm.data", data), ("timm.models", models),
                      ("timm.models.layers", layers), ("timm.models.registry", registry),
                      ("timm.loss", loss)]:
        sys.modules[name] = mod


_cache = {}


def load_reference():
    """Returns a namespace with .ptopk, .dvit (Variant B), .ddvit (Variant A) reference modules."""
    if "ns" in _cache:
        return _cache["ns"]
    if not reference_available():
        raise RuntimeError(f"reference not found under {REF_ROOT}")
    _install_timm_stub()
    pkg_name = "_d2s_ref_vit_models"
    pkg = types.ModuleType(pkg_name)
    pkg.__path__ = [os.path.join(REF_ROOT, "vit_models")]
    sys.modules[pkg_name] = pkg

    def _load(stem):
        full = f"{pkg_name}.{stem}"
        spec = importlib.util.spec_from_file_location(full, os.path.join(REF_ROOT, "vit_models", stem + ".py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[full] = mod
        spec.loader.exec_module(mod)
        return mod

    ns = types.SimpleNamespace()
    ns.ptopk = _load("peturbed_topk")
    ns.dvit = _load("dynamic_vit")
    ns.ddvit = _load("default_dynamic_vit")
    _cache["ns"] = ns
    return ns


class record_gumbels:
    """Context manager: run reference code that calls F.gumbel_softmax unmodified and recover the
    exact Gumbel noise each call drew (torch/nn/functional.py gumbel_softmax:
    `-empty_like(logits).exponential_().log()`), by replaying the RNG state around the call."""

    def __init__(self):
        self.gumbels = []

    def __enter__(self):
        import torch.nn.functional as F
        self._F = F
        self._orig = F.gumbel_softmax
        rec = self

        def wrapped(logits, tau=1, hard=False, eps=1e-10, dim=-1):
            st = torch.get_rng_state()
            out = rec._orig(logits, tau=tau, hard=hard, eps=eps, dim=dim)
            st2 = torch.get_rng_state()
            torch.set_rng_state(st)
            g = -torch.empty_like(logits, memory_format=torch.legacy_contiguous_format).exponential_().log()
            torch.set_rng_state(st2)
            rec.gumbels.append(g.detach().clone())
            return out

        F.gumbel_softmax = wrapped
        return self

    def __exit__(self, *a):
        self._F.gumbel_softmax = self._orig
        return False


class inject_normal:
    """Context manager: make the reference's `torch.normal(mean, std, size=...)` call
    (vit_models/peturbed_topk.py:29) return a supplied noise tensor."""

    def __init__(self, noise):
        self.noise = noise

    def __enter__(self):
        self._orig = torch.normal
        noise = self.noise

        def fake(*args, **kw):
            size = kw.get("size")
            assert size is not None and tuple(size) == tuple(noise.shape), (size, noise.shape)
            return noise.clone()

        torch.normal = fake
        return self

    def __exit__(self, *a):
        torch.normal = self._orig
        return False
