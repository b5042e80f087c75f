"""The training step as two replayed CUDA graphs around ONE gradient all-reduce (BASELINE.json configs[3]; reference
models/trainer.py:247-262, 299-310: forward, loss, backward, optimizer step).

The eager step of this network is ~1300 small launches, so one GPU spends more time being fed from Python than computing
(21 ms eager against 10.4 ms of device time at batch 8), and stock DistributedDataParallel adds its bucket bookkeeping and — because
the module, like the reference's, owns 48 parameters no forward ever reads — a per-step unused-parameter search on top.
``GraphedTrainStep`` removes both without touching the arithmetic:

* graph 1 = forward, loss, backward (gradients written straight into the flat buffer);  graph 2 = the optimizer step (a
  ``capturable`` torch optimizer);
* every parameter that receives a gradient gets a view into ONE flat fp32 buffer as its ``.grad`` (with the parameter's own
  strides, channels_last included), so the data-parallel exchange is a single ``all_reduce(mean)`` of that buffer between the
  two graphs (NCCL over NVLink on GPUs; any ``torch.distributed`` backend works) — no DDP wrapper, no buckets, no hooks;
* parameters that received no gradient during the warm-up are frozen (``requires_grad_(False)``): the optimizer would skip them
  anyway (their ``.grad`` is None in the eager loop too).

``use_graph=False`` runs the same step eagerly (same flat buffer, same all-reduce) — what the CPU / gloo tests exercise.
The module is generic: any ``nn.Module``, any loss callable, any batch tuple whose last element is the target.

Mixed precision (``amp=torch.float16`` or ``torch.bfloat16``): graph 1 runs the forward and the loss under autocast.  For fp16 the
step is ``torch.amp.GradScaler`` with its defaults, kept on the device so that nothing waits for the host: graph 1 runs the
backward from ``loss * scale``; after the all-reduce (so every rank sees the same overflow) graph 2 unscales the flat buffer and
sets ``found_inf`` (``torch._amp_foreach_non_finite_check_and_unscale_``), the optimizer skips its update on the device when
``found_inf`` is set (``_step_supports_amp_scaling``: fused Adam, AdamW or SGD), and ``torch._amp_update_scale_`` moves the
scale.  bf16 has fp32's exponent range and needs no scaler.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

# torch.amp.GradScaler's defaults
INIT_SCALE, GROWTH_FACTOR, BACKOFF_FACTOR, GROWTH_INTERVAL = 2.0 ** 16, 2.0, 0.5, 2000


def _grad_view(flat, offset, p):
    """a view of flat[offset : offset + p.numel()] with p's shape AND strides (dense parameters only)"""
    g = flat[offset:offset + p.numel()]
    if p.is_contiguous():
        return g.view_as(p)
    if p.dim() == 4 and p.is_contiguous(memory_format=torch.channels_last):
        return g.view(p.shape[0], p.shape[2], p.shape[3], p.shape[1]).permute(0, 3, 1, 2)
    raise RuntimeError(f"GraphedTrainStep: parameter of shape {tuple(p.shape)} / strides {p.stride()} is not dense")


class GraphedTrainStep:
    """step(*batch) -> loss (a static tensor: clone it if you keep it across steps).

    net            the module (left in train() mode)
    loss_fn        loss_fn(output, target) -> scalar
    example_batch  tuple of tensors (inputs..., target) fixing shapes / dtypes / device; step() copies each batch into static
                   buffers of these shapes
    make_optimizer callable(list_of_live_parameters) -> torch optimizer (pass capturable=True for Adam-family optimizers when
                   use_graph); optimizers whose all-zero state equals their fresh state (Adam family, SGD with momentum) are
                   supported — the state is created by one throw-away step before capture and zeroed again
    group          torch.distributed process group (default: the world group if initialised, else single process);
                   distributed=False keeps the step local even inside an initialised process group
    amp            None (fp32), torch.float16 (autocast + device-side loss scaling: the optimizer must support
                   ``_step_supports_amp_scaling``, i.e. fused=True Adam / AdamW / SGD) or torch.bfloat16 (autocast)
    """

    def __init__(self, net, loss_fn, example_batch, make_optimizer, group=None, use_graph=True, warmup=3, distributed=True,
                 amp=None):
        if amp not in (None, torch.float16, torch.bfloat16):
            raise ValueError(f"GraphedTrainStep: amp must be None, torch.float16 or torch.bfloat16, not {amp}")
        self.amp, self.scaled = amp, amp == torch.float16
        self.net, self.loss_fn, self.group = net.train(), loss_fn, group
        self.world = dist.get_world_size(group) if (distributed and dist.is_available() and dist.is_initialized()) else 1
        self.static = [t.clone() for t in example_batch]
        dev = self.static[0].device
        self.use_graph = bool(use_graph) and dev.type == "cuda"
        if self.scaled:                                                          # GradScaler's state, on the device
            self.scale = torch.full((1,), INIT_SCALE, dtype=torch.float32, device=dev)
            self.growth_tracker = torch.zeros(1, dtype=torch.int32, device=dev)
            self.found_inf = torch.zeros((), dtype=torch.float32, device=dev)
        buffers = [(b, b.clone()) for b in net.buffers()]                       # BatchNorm running stats must not see the warm-up
        for p in net.parameters():
            p.grad = None
        side = torch.cuda.Stream(dev) if dev.type == "cuda" else None
        if side is not None:
            side.wait_stream(torch.cuda.current_stream(dev))
        with (torch.cuda.stream(side) if side is not None else _null()):
            for _ in range(max(1, warmup)):                                      # lazy initialisation (layouts, autotuning) + liveness
                self._forward_backward(zero=False)
            self.live = [p for p in net.parameters() if p.grad is not None]
            self.flat = torch.zeros(sum(p.numel() for p in self.live), dtype=self.live[0].dtype, device=dev)
            off = 0
            for p in self.live:
                p.grad = _grad_view(self.flat, off, p)
                off += p.numel()
            self.frozen = [p for p in net.parameters() if p.grad is None and p.requires_grad]
            for p in self.frozen:
                p.requires_grad_(False)
            self.opt = make_optimizer(self.live)
            if self.scaled and not getattr(self.opt, "_step_supports_amp_scaling", False):
                for p in net.parameters():
                    p.grad = None
                for p in self.frozen:
                    p.requires_grad_(True)
                with torch.no_grad():
                    for b, s in buffers:
                        b.copy_(s)
                raise ValueError(f"GraphedTrainStep(amp=torch.float16): {type(self.opt).__name__} cannot skip a step on the device "
                                 "when a gradient overflowed, so every step would wait for the host; use an optimizer with "
                                 "_step_supports_amp_scaling (fused=True Adam, AdamW or SGD)")
            if self.scaled:
                self.opt.found_inf = self.found_inf                              # read by the fused step: skip when set
            saved = [p.detach().clone() for p in self.live]
            self._optimizer_step()                                               # creates the optimizer state outside any capture
            with torch.no_grad():
                for p, s in zip(self.live, saved):
                    p.copy_(s)
                for st in self.opt.state.values():
                    for v in st.values():
                        if torch.is_tensor(v):
                            v.zero_()
                for b, s in buffers:
                    b.copy_(s)
                if self.scaled:
                    self.scale.fill_(INIT_SCALE)
                    self.growth_tracker.zero_()
            if self.use_graph:
                self._forward_backward(zero=True)                                # once more with the flat views in place
                with torch.no_grad():
                    for b, s in buffers:
                        b.copy_(s)
        if side is not None:
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
        self.loss = None
        if self.use_graph:
            self.g_fb, self.g_opt = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g_fb):
                self.loss = self._forward_backward(zero=True)
            with torch.cuda.graph(self.g_opt):
                self._optimizer_step()

    def _forward_backward(self, zero):
        # graphs need the autocast weight cache off; it changes no value
        with torch.autocast(self.static[0].device.type, dtype=self.amp, cache_enabled=False) if self.amp else _null():
            loss = self.loss_fn(self.net(*self.static[:-1]), self.static[-1])
        if not zero:                                                             # warm-up: marks the live parameters
            loss.backward()
            return loss.detach()
        # the gradients are WRITTEN into the flat buffer (no zeroing pass, no per-parameter accumulation kernels): autograd
        # returns them, one multi-tensor copy moves them into the views the optimizer reads as .grad
        grads = torch.autograd.grad(loss * self.scale if self.scaled else loss, self.live)
        torch._foreach_copy_([p.grad for p in self.live], list(grads))
        return loss.detach()

    def _optimizer_step(self):
        if self.scaled:                                                          # GradScaler.unscale_ / step / update
            self.found_inf.zero_()
            torch._amp_foreach_non_finite_check_and_unscale_([self.flat], self.found_inf, self.scale.double().reciprocal().float())
        self.opt.step()
        if self.scaled:
            torch._amp_update_scale_(self.scale, self.growth_tracker, self.found_inf, GROWTH_FACTOR, BACKOFF_FACTOR, GROWTH_INTERVAL)

    def scaler_state_dict(self):
        """the loss scaler's state in torch.amp.GradScaler.state_dict() form ({} without one, like a disabled GradScaler), so a
        checkpoint moves between this step and an eager GradScaler loop"""
        if not self.scaled:
            return {}
        return {"scale": float(self.scale), "growth_factor": GROWTH_FACTOR, "backoff_factor": BACKOFF_FACTOR,
                "growth_interval": GROWTH_INTERVAL, "_growth_tracker": int(self.growth_tracker)}

    def load_scaler_state_dict(self, state):
        """restore a torch.amp.GradScaler.state_dict() (or scaler_state_dict()); the growth / backoff settings are baked into the
        captured step and must be GradScaler's defaults"""
        if not self.scaled:
            if state:
                raise ValueError("GraphedTrainStep.load_scaler_state_dict: this step has no loss scaler (amp is not torch.float16)")
            return
        if not state:
            raise ValueError("GraphedTrainStep.load_scaler_state_dict: the state is empty (saved from a disabled GradScaler?)")
        fixed = {"growth_factor": GROWTH_FACTOR, "backoff_factor": BACKOFF_FACTOR, "growth_interval": GROWTH_INTERVAL}
        for k, v in fixed.items():
            if state[k] != v:
                raise ValueError(f"GraphedTrainStep.load_scaler_state_dict: {k} = {state[k]}, the step runs with {v}")
        self.scale.fill_(state["scale"])
        self.growth_tracker.fill_(state["_growth_tracker"])

    def all_reduce(self):
        if self.world > 1:
            if self.flat.is_cuda:
                dist.all_reduce(self.flat, op=dist.ReduceOp.AVG, group=self.group)
            else:                                                                # gloo has no AVG
                dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=self.group)
                self.flat.div_(self.world)

    def step(self, *batch, sync_gradients=True):
        if len(batch) != len(self.static):
            raise ValueError(f"GraphedTrainStep.step: expected {len(self.static)} tensors, got {len(batch)}")
        for s, b in zip(self.static, batch):
            if b is not s:
                if b.shape != s.shape:                                           # copy_ would broadcast (a last, smaller batch x N)
                    raise ValueError(f"GraphedTrainStep.step: batch tensor of shape {tuple(b.shape)}, the step was built for "
                                     f"{tuple(s.shape)}; run other shapes through the eager loop")
                s.copy_(b, non_blocking=True)
        if self.use_graph:
            self.g_fb.replay()
        else:
            self.loss = self._forward_backward(zero=True)
        if sync_gradients:
            self.all_reduce()
        if self.use_graph:
            self.g_opt.replay()
        else:
            self._optimizer_step()
        return self.loss


class _null:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False
