"""Execution helpers around the models: CUDA-graph inference, host->device pipelining, data-parallel sharding.

Everything per-image on the hot path is independent (SURVEY.md section 8e): inference is sharded by batch
across ranks with no collective; training uses torch DistributedDataParallel (NCCL gradient all-reduce), which
is the reference's own design (ddp_training.py:93).
"""
import os

import torch

from . import ops


def shard_range(global_batch: int, rank: int, world: int):
    """Contiguous slice [lo, hi) of a global batch owned by `rank`; sizes differ by at most one image."""
    base, rem = divmod(global_batch, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def dist_env():
    """(rank, local_rank, world) from the torchrun environment; (0, 0, 1) when launched plainly."""
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def wrap_ddp(model, device=None, **kw):
    """DistributedDataParallel exactly as the reference intends (ddp_training.py:93): one process per GPU,
    bucketed gradient all-reduce overlapped with backward."""
    from torch.nn.parallel import DistributedDataParallel as DDP
    if device is not None and device.type == "cuda":
        return DDP(model, device_ids=[device.index], output_device=device.index, find_unused_parameters=False, **kw)
    return DDP(model, find_unused_parameters=False, **kw)


class InferenceRunner:
    """Captures one eval forward of `model` at a fixed batch shape into a CUDA graph and replays it.

    The per-stage launches around the big GEMMs (predictor tail+select, gather, attention) are small; a graph
    removes their launch latency from the step (SURVEY.md section 7, hard part 7).  Outputs are static tensors
    owned by the graph's memory pool: read them (or copy them out) before the next replay.
    """

    IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)   # timm IMAGENET_DEFAULT_MEAN / _STD

    def __init__(self, model, batch, device, dtype=torch.bfloat16, img_shape=(3, 224, 224), use_graph=True, warmup=3,
                 uint8_input=False, mean=IMAGENET_MEAN, std=IMAGENET_STD):
        """uint8_input: the runner takes RAW uint8 images (B,3,H,W); ToTensor + Normalize(mean, std) -- what the reference's
        data loaders do on the host (build_data_sets.py) -- run inside the patch-embedding im2col kernel, bit-identically.  The
        host -> device copy of the end-to-end path shrinks to a quarter of fp32 / half of bf16."""
        self.model = model.eval().to(device=device, dtype=dtype)
        self.device, self.dtype, self.batch = device, dtype, batch
        if uint8_input:
            self.model.patch_embed.d2s_input_norm = (torch.tensor(mean, dtype=torch.float32, device=device),
                                                     torch.tensor(std, dtype=torch.float32, device=device))
        self.static_in = torch.zeros(batch, *img_shape, dtype=torch.uint8 if uint8_input else dtype, device=device)
        self.graph = None
        self.static_out = None
        self._stage = None
        self._copy_stream = None
        self._host_out = None
        with torch.no_grad():
            side = torch.cuda.Stream(device=device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                for _ in range(max(1, warmup)):
                    out = self.model(self.static_in)
            torch.cuda.current_stream(device).wait_stream(side)
            torch.cuda.synchronize(device)
            if use_graph:
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    out = self.model(self.static_in)
            self.static_out = out

    @property
    def logits(self):
        out = self.static_out
        return out[0] if isinstance(out, (tuple, list)) else out

    def replay(self):
        """One forward over whatever currently sits in static_in."""
        if self.graph is not None:
            self.graph.replay()
        else:
            with torch.no_grad():
                self.static_out = self.model(self.static_in)
        return self.static_out

    def __call__(self, x):
        self.static_in.copy_(x, non_blocking=True)
        return self.replay()

    # ---- end-to-end path: pinned host images in, host logits out ------------------------------------
    def _ensure_pipeline(self):
        if self._stage is None:
            self._stage = [torch.empty_like(self.static_in) for _ in range(2)]
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._ready = [torch.cuda.Event() for _ in range(2)]
            self._free = [torch.cuda.Event() for _ in range(2)]
            self._host_out = torch.empty(self.logits.shape, dtype=self.logits.dtype).pin_memory()
            self._slot = 0
            self._used = [False, False]
            # One captured forward PER staging buffer: the step reads the images where the copy stream put them, instead of
            # moving them into static_in first (a 2 x (B,3,H,W) device-to-device pass per step, ~1 % of the step).
            self._slot_graphs = None
            if self.graph is not None:
                self._slot_graphs = []
                with torch.no_grad():
                    for k in range(2):
                        self._stage[k].copy_(self.static_in)
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g):
                            out = self.model(self._stage[k])
                        self._slot_graphs.append((g, out[0] if isinstance(out, (tuple, list)) else out))
                torch.cuda.synchronize(self.device)

    def prefetch(self, x_host):
        """Start the host->device copy of a later step's images on the copy stream; returns the staging slot."""
        self._ensure_pipeline()
        k = self._slot
        with torch.cuda.stream(self._copy_stream):
            if self._used[k]:  # the compute stream must have consumed this staging buffer
                self._copy_stream.wait_event(self._free[k])
            self._stage[k].copy_(x_host, non_blocking=True)
            self._ready[k].record(self._copy_stream)
        self._slot ^= 1
        return k

    def step_prefetched(self, k):
        """Run one forward on the images whose copy was started by `k = prefetch(...)`; returns pinned host
        logits (valid after the caller synchronises the current stream)."""
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(self._ready[k])
        if self._slot_graphs is not None:
            g, logits = self._slot_graphs[k]
            g.replay()                              # reads self._stage[k] in place
            self._free[k].record(cur)               # (the slot is refilled one step later: its copy waits for this step to end)
            self._used[k] = True
            self._host_out.copy_(logits, non_blocking=True)
            return self._host_out
        self.static_in.copy_(self._stage[k], non_blocking=True)
        self._free[k].record(cur)
        self._used[k] = True
        self.replay()
        self._host_out.copy_(self.logits, non_blocking=True)
        return self._host_out

    def step_from_host(self, x_host):
        """Unpipelined end-to-end step: H2D copy, forward, D2H of the logits, all on the current stream."""
        self._ensure_pipeline()
        self.static_in.copy_(x_host, non_blocking=True)
        self.replay()
        self._host_out.copy_(self.logits, non_blocking=True)
        return self._host_out


def flat_layout(params, align=8):
    """Offsets of `params` in a flat buffer, each start rounded up to `align` elements (16 B for bf16, 32 B for fp32: what the
    vectorised kernels, TMA descriptors and library GEMMs reading views of the buffer need).  Returns (offsets, total)."""
    offs, off = [], 0
    for p in params:
        offs.append(off)
        off += (p.numel() + align - 1) // align * align
    return offs, off


class FlatGrads:
    """All trainable parameters' gradients as views into ONE fp32 buffer, so that data-parallel training needs a single NCCL
    all-reduce per step (<= 91 MB for DeiT-S, 0.2 ms at NVLink 5 bus bandwidth against a >= 20 ms step) and the collective can
    sit INSIDE the captured CUDA graph of the step, between backward and the optimizer.  autograd accumulates in place into an
    existing .grad, so the views survive backward; zero() replaces optimizer.zero_grad().  The views are also registered as
    gradient SLOTS with ops: the d2s training nodes (Linear, Linear+GELU, LayerNorm) write their parameter gradients there
    directly instead of handing them to autograd's per-parameter accumulate pass."""

    def __init__(self, params, group=None, average=True):
        import torch.distributed as dist
        self.params = [p for p in params if p.requires_grad]
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.group = group
        self.average = average                       # False: the optimizer folds the 1/world in (FlatAdamW's grad_scale)
        dev = self.params[0].device
        self.offsets, total = flat_layout(self.params)
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        for p, off in zip(self.params, self.offsets):
            if p.dtype != torch.float32:
                raise TypeError("FlatGrads expects fp32 master parameters (bf16 autocast training)")
            p.grad = self.flat[off:off + p.numel()].view_as(p)
        ops.register_grad_slots(self.params)

    def zero(self):
        self.flat.zero_()
        ops.reset_grad_slots(self.params)

    def all_reduce(self):
        """Sum (average=True: mean) of the gradients over the ranks (the one collective of the path: ddp_training.py:93 uses
        DDP's buckets)."""
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(self.flat, group=self.group)
            if self.average:
                self.flat.mul_(1.0 / self.world)

    def close(self):
        ops.unregister_grad_slots(self.params)


class FlatAdamW(torch.optim.Optimizer):
    """torch.optim.AdamW's update (decoupled weight decay, bias correction; no amsgrad / maximize) as ONE d2s kernel launch per
    parameter group over flat buffers: the parameters are re-pointed into one fp32 buffer (same layout as .grads, a FlatGrads
    this optimizer owns), the moments are flat, and the kernel also writes the bf16 copy of the updated weights that the next
    forward's GEMMs read (.weight_cache, an ops.BF16WeightCache whose refresh() is a no-op).  lr and the step count live in
    device memory, so a step captured in a CUDA graph follows an lr schedule: schedulers keep writing group["lr"] and
    sync_hyper() (called by TrainStepRunner before every step) copies a changed value to the device.

    torch's capturable multi-tensor AdamW costs ~380 launches and ~1.4 ms for DeiT-S (22 M parameters) inside the graph; this
    is ~0.1 ms: 30 bytes per parameter at HBM speed."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, group=None, bf16_shadow=True):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        flat_params, self._ranges = [], []
        for g in self.param_groups:
            g["params"] = [p for p in g["params"] if p.requires_grad]
            flat_params += g["params"]
        if not flat_params:
            raise ValueError("FlatAdamW: no trainable parameters")
        dev = flat_params[0].device
        if dev.type != "cuda" or any(p.dtype != torch.float32 or p.device != dev for p in flat_params):
            raise TypeError("FlatAdamW expects fp32 parameters on one CUDA device")
        self.grads = FlatGrads(flat_params, group=group, average=False)
        offs, total = self.grads.offsets, self.grads.flat.numel()
        self.flat_p = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros_like(self.flat_p)
        self.exp_avg_sq = torch.zeros_like(self.flat_p)
        self.shadow = torch.zeros(total, dtype=torch.bfloat16, device=dev) if bf16_shadow else None
        with torch.no_grad():
            for p, off in zip(flat_params, offs):
                view = self.flat_p[off:off + p.numel()].view_as(p)
                view.copy_(p)
                p.data = view
            if self.shadow is not None:
                self.shadow.copy_(self.flat_p)
        self.weight_cache = None
        if self.shadow is not None:
            self.weight_cache = ops.BF16WeightCache(flat_params, copies=[self.shadow[off:off + p.numel()].view_as(p)
                                                                         for p, off in zip(flat_params, offs)])
        i = 0
        for g in self.param_groups:                  # one contiguous range of the flat layout per group
            n = len(g["params"])
            begin = offs[i] if n else 0
            end = (offs[i + n] if i + n < len(offs) else total) if n else 0
            self._ranges.append((begin, end))
            g["_lr_dev"] = torch.full((1,), float(g["lr"]), dtype=torch.float32, device=dev)
            g["_lr_host"] = float(g["lr"])
            i += n
        self.step_t = torch.zeros(1, dtype=torch.float32, device=dev)

    def sync_hyper(self):
        """Host-side lr changes (schedulers write group["lr"]) -> the device copies the kernel reads."""
        for g in self.param_groups:
            if float(g["lr"]) != g["_lr_host"]:
                g["_lr_host"] = float(g["lr"])
                g["_lr_dev"].fill_(g["_lr_host"])

    def zero_grad(self, set_to_none=False):
        self.grads.zero()                            # the gradient views must survive: never set to None

    @torch.no_grad()
    def step(self, closure=None):
        if closure is not None:
            raise NotImplementedError("FlatAdamW.step: closures are not supported")
        if not torch.cuda.is_current_stream_capturing():
            self.sync_hyper()
        self.step_t.add_(1.0)
        scale = 1.0 / self.grads.world
        for g, (begin, end) in zip(self.param_groups, self._ranges):
            b1, b2 = g["betas"]
            ops.adamw_flat(self.flat_p, self.grads.flat, self.exp_avg, self.exp_avg_sq, self.shadow, begin, end, g["_lr_dev"],
                           self.step_t, b1, b2, g["eps"], g["weight_decay"], scale)

    # ---- checkpoint / resume (the moments live in flat buffers, not in torch's per-parameter `state`) ----
    def state_dict(self):
        groups = [{k: v for k, v in g.items() if k != "params" and not k.startswith("_")} for g in self.param_groups]
        return {"step": float(self.step_t.item()), "exp_avg": self.exp_avg.detach().clone(), "exp_avg_sq": self.exp_avg_sq.detach().clone(),
                "param_groups": groups, "numel": [p.numel() for g in self.param_groups for p in g["params"]]}

    def load_state_dict(self, sd):
        numel = [p.numel() for g in self.param_groups for p in g["params"]]
        if list(sd["numel"]) != numel or sd["exp_avg"].numel() != self.exp_avg.numel():
            raise ValueError("FlatAdamW.load_state_dict: the checkpoint was written for a different parameter list")
        with torch.no_grad():
            self.exp_avg.copy_(sd["exp_avg"])
            self.exp_avg_sq.copy_(sd["exp_avg_sq"])
            self.step_t.fill_(float(sd["step"]))
        for g, saved in zip(self.param_groups, sd["param_groups"]):
            g.update(saved)
        self.sync_hyper()

    def close(self):
        self.grads.close()
        if self.weight_cache is not None:
            self.weight_cache.close()


class TrainStepRunner:
    """One whole training step -- forward, loss, backward, [gradient all-reduce,] optimizer -- captured in a CUDA graph and
    replayed.

    A DeiT-S training step is ~1100 kernel launches, most of them short (autograd's elementwise tail, weight casts, the
    optimizer): eager, the step is within ~2 ms of being bound by host-side launch latency.  All shapes of the training path are
    static (training prunes by masks, not by gathers; the losses use masked reductions), so the step captures as is.
    `step_fn(x, y)` must run forward + loss and return the loss tensor; the optimizer must be constructed with
    capturable=True.  `grads` (a FlatGrads over the optimizer's parameters) makes the step data-parallel: one NCCL all-reduce of
    the flat gradient buffer is captured between backward and the optimizer step (one process per GPU, torchrun)."""

    def __init__(self, step_fn, optimizer, x, y, warmup=3, use_graph=True, grads=None, weight_cache=None):
        """weight_cache: an ops.BF16WeightCache over the trained parameters -- refreshed right after every optimizer step
        (inside the captured graph), so the forward's Linear layers read per-step bf16 copies instead of casting every weight."""
        self.step_fn, self.opt, self.grads, self.weight_cache = step_fn, optimizer, grads, weight_cache
        self.static_x, self.static_y = x.clone(), y.clone()
        self.graph, self.loss = None, None
        dev = x.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):          # allocations, cuBLAS workspaces, NCCL channels, lazily built state: outside the capture
                self._eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        if use_graph:
            self.graph = torch.cuda.CUDAGraph()
            if self.grads is None:
                self.opt.zero_grad(set_to_none=True)
            with torch.cuda.graph(self.graph):
                self._body()

    def _body(self):
        if self.grads is not None:
            self.grads.zero()
        self.loss = self.step_fn(self.static_x, self.static_y)
        self.loss.backward()
        if self.grads is not None:
            self.grads.all_reduce()
        self.opt.step()
        if self.weight_cache is not None:
            self.weight_cache.refresh()

    def _eager(self):
        if self.grads is None:
            self.opt.zero_grad(set_to_none=True)
        self._body()
        return self.loss

    # ---- pipelined input: the next batch's host -> device copy runs on a copy stream while the current step computes --------
    def prefetch(self, x_host, y_host):
        """Start copying a LATER step's batch (pinned host tensors) into a device staging buffer on the copy stream."""
        dev = self.static_x.device
        if getattr(self, "_stage", None) is None:
            self._stage = (torch.empty_like(self.static_x), torch.empty_like(self.static_y))
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._ready, self._taken = torch.cuda.Event(), torch.cuda.Event()
            self._taken.record(torch.cuda.current_stream(dev))
        self._copy_stream.wait_event(self._taken)             # the previous staged batch has been moved into the step's inputs
        with torch.cuda.stream(self._copy_stream):
            self._stage[0].copy_(x_host, non_blocking=True)
            self._stage[1].copy_(y_host, non_blocking=True)
            self._ready.record(self._copy_stream)

    def step_prefetched(self):
        """One optimisation step on the batch staged by prefetch(): a device-to-device move into the graph's inputs, then the step."""
        cur = torch.cuda.current_stream(self.static_x.device)
        cur.wait_event(self._ready)
        self.static_x.copy_(self._stage[0], non_blocking=True)
        self.static_y.copy_(self._stage[1], non_blocking=True)
        self._taken.record(cur)
        return self()

    def __call__(self, x=None, y=None):
        """One optimisation step on (x, y) (default: the tensors already in place); returns the (static) loss tensor."""
        if x is not None:
            self.static_x.copy_(x, non_blocking=True)
        if y is not None:
            self.static_y.copy_(y, non_blocking=True)
        if hasattr(self.opt, "sync_hyper"):
            self.opt.sync_hyper()                    # lr schedule -> device memory (outside the graph)
        if self.graph is None:
            return self._eager()
        self.graph.replay()
        return self.loss
