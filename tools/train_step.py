"""configs[3]: LEVIR-CD training step of the drop-in module (batch 8 per GPU, 256x256, synthetic labels, CE loss, AdamW).
Training runs on the stock-autograd route (DESIGN.md "Training step"); under torchrun the module is wrapped in
DistributedDataParallel (NCCL gradient all-reduce, as BASELINE.json's config 4 describes).  After the last step the
module is switched to eval() and the NATIVE forward is checked against the autograd route on the updated weights.
   python tools/train_step.py [--steps 10]                                   (1 GPU)
   python tools/train_step.py --graph --amp fp16                             (mixed precision: autocast, device-side loss scaling)
   python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/train_step.py    (DDP)
Prints one JSON line from rank 0."""
import argparse, contextlib, json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
import torch.nn.functional as F
from dahitra_b200.networks import define_G


class Args:
    net_G = "newUNetTrans"


ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--batch", type=int, default=8)
ap.add_argument("--as-written", action="store_true", help="pixel decoders as the reference writes them (q / k / v / out projections) instead of the collapsed algebra")
ap.add_argument("--stock", action="store_true", help="pixel decoders on stock torch ops instead of the native training kernels (csrc/train_decoder.cu)")
ap.add_argument("--nchw", action="store_true", help="keep activations / parameters NCHW-contiguous instead of the module's default torch.channels_last training layout")
ap.add_argument("--two-pass-trunk", action="store_true", help="run the trunk once per image set (the reference's two forward_single calls) instead of one batch with per-set BatchNorm")
ap.add_argument("--freeze-unused", action="store_true", help="net.freeze_unused_parameters(): DDP without find_unused_parameters")
ap.add_argument("--graphed-route", action="store_true", help="eager loop (loss, backward(), optimizer as written) with the network's forward / backward replayed from CUDA graphs (net.graphed_training, training.GraphedRoute)")
ap.add_argument("--foreach-adamw", action="store_true", help="with --graph: torch's foreach AdamW inside the optimizer graph instead of the fused one")
ap.add_argument("--graph", action="store_true", help="capture forward + backward + AdamW step in ONE CUDA graph and replay it (1 GPU)")
ap.add_argument("--amp", choices=("fp16", "bf16"), help="mixed precision: forward and loss under autocast; fp16 with loss scaling "
                "(torch.amp.GradScaler in the eager loop, GraphedTrainStep(amp=torch.float16) with --graph)")
a = ap.parse_args()
amp = {None: None, "fp16": torch.float16, "bf16": torch.bfloat16}[a.amp]
scaler = torch.amp.GradScaler("cuda", enabled=amp == torch.float16)
world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl")
torch.manual_seed(0)
net = define_G(Args(), gpu_ids=[local]).train()
net.collapsed_training = not a.as_written
net.native_training = not (a.stock or a.as_written)
model = net
if a.freeze_unused:
    net.freeze_unused_parameters()
if world > 1 and not a.graph:
    # like the reference, the module owns parameters its forward never uses (scale-2 transformer, conv_pred, layer4)
    model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[local], find_unused_parameters=not a.freeze_unused)
opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.01, capturable=a.graph)           # models/trainer.py:39-40
g = torch.Generator(device="cuda").manual_seed(100 + rank)
x1 = torch.rand(a.batch, 3, 256, 256, device="cuda", generator=g) * 2 - 1
x2 = torch.rand(a.batch, 3, 256, 256, device="cuda", generator=g) * 2 - 1
y = (torch.rand(a.batch, 256, 256, device="cuda", generator=g) < 0.1).long()
net.channels_last_training = not a.nchw
net.graphed_training = a.graphed_route
net.paired_trunk_training = not a.two_pass_trunk
losses = []
w2 = torch.ones(2, device="cuda")


ts, flat_grad = None, None


def one_step(sync=True):
    if ts is not None:
        return ts.step(x1, x2, y, sync_gradients=sync)
    opt.zero_grad(set_to_none=True)
    ctx = model.no_sync() if (world > 1 and not sync) else contextlib.nullcontext()
    with ctx:
        with torch.autocast("cuda", dtype=amp, enabled=amp is not None):
            loss = F.cross_entropy(model(x1, x2), y, weight=w2, ignore_index=255)   # models/losses.py:9-26
        scaler.scale(loss).backward()
    scaler.step(opt)
    scaler.update()
    return loss


def timed(n, sync=True):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        losses.append(one_step(sync).detach().clone())
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / n], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms)


for _ in range(3):                               # warm-up (cuDNN autotune, allocator, DDP bucket rebuild)
    if not a.graph:                              # (GraphedTrainStep does its own warm-up)
        losses.append(one_step().detach())
if a.graph:
    # forward + backward and the AdamW step replayed from two CUDA graphs around ONE flat NCCL all-reduce (no DDP wrapper):
    # dahitra_b200/train_graph.py
    from dahitra_b200.train_graph import GraphedTrainStep
    ts = GraphedTrainStep(net, lambda out, tgt: F.cross_entropy(out, tgt, weight=w2, ignore_index=255), (x1, x2, y),
                          lambda ps: torch.optim.AdamW(ps, lr=1e-3, weight_decay=0.01, capturable=True, fused=not a.foreach_adamw),
                          amp=amp)
    flat_grad = ts.flat
step_ms = timed(a.steps)
dt = step_ms * a.steps / 1e3
if world > 1:                                   # replicas must hold identical weights after the all-reduced steps
    w = torch.cat([p.detach().flatten()[:64] for p in net.parameters()])
    ref = w.clone()
    dist.broadcast(ref, 0)
    same = bool(torch.equal(w, ref))
    flag = torch.tensor([int(same)], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    replicas_equal = bool(flag.item())
else:
    replicas_equal = None
# (measured AFTER the replica check: steps without the all-reduce let the replicas drift apart on purpose)
# the gradient all-reduce: (a) exposed share = step with - step without the all-reduce (DDP no_sync), (b) the collective
# alone on a flat fp32 buffer of the gradients' size
nosync_ms, ar_ms, grad_bytes = None, None, 4 * sum(p.numel() for p in net.parameters() if p.requires_grad)
if world > 1:
    nosync_ms = timed(max(3, a.steps // 2), sync=False)
    flat = torch.zeros(grad_bytes // 4, device="cuda")
    for _ in range(2):
        dist.all_reduce(flat)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); dist.barrier()
    e0.record()
    for _ in range(5):
        dist.all_reduce(flat)
    e1.record()
    torch.cuda.synchronize()
    ar_ms = e0.elapsed_time(e1) / 5
losses = [float(l) for l in losses]
no_grad = [n for n, p in net.named_parameters() if p.grad is None]
gnorm = float(torch.sqrt(sum((p.grad.float() ** 2).sum() for p in net.parameters() if p.grad is not None)))
net.eval()
with torch.no_grad():
    y_native = net(x1, x2)                      # native sm_100a forward on the UPDATED weights
y_auto = net._forward_autograd(x1, x2).detach()
native_vs_autograd = float((y_native - y_auto).abs().max())
if rank == 0:
    print(json.dumps(dict(decoder="as written (stock ops)" if a.as_written else "collapsed algebra, stock ops (modules.PixelDecoder.forward_collapsed)" if a.stock
                          else "native sm_100a forward + backward kernels (csrc/train_decoder.cu)",
                      workload=f"LEVIR-CD training step, batch {a.batch} x {world} GPU(s), CE loss, AdamW ({'one CUDA graph per iteration, ' if a.graph else ''}autograd route"
                                   + ((", one flat NCCL all-reduce of the live gradients)" if a.graph else ", DDP/NCCL all-reduce)") if world > 1 else ")"),
                          ddp=(None if (world == 1 or a.graph) else ("unused parameters frozen, find_unused_parameters=False" if a.freeze_unused else "find_unused_parameters=True")),
                          loop=("GraphedTrainStep" if a.graph else "eager loop, network forward / backward replayed from CUDA graphs (graphed_training)" if a.graphed_route else "eager"),
                          precision=("fp32 (TF32 convolutions: torch's default allow_tf32)" if amp is None else f"autocast {a.amp}"
                                     + (", loss scaling (GradScaler defaults)" if amp == torch.float16 else "")),
                          trunk="one pass per image set" if a.two_pass_trunk else "both image sets per convolution launch, BatchNorm per set", memory_format="contiguous (NCHW)" if a.nchw else "channels_last (set by the module)", steps=a.steps, step_ms=step_ms, steps_per_s=a.steps / dt, pairs_per_s=a.steps * a.batch * world / dt,
                          pairs_per_s_per_gpu=a.steps * a.batch / dt,
                          step_ms_without_allreduce=nosync_ms, exposed_allreduce_share=(None if nosync_ms is None else max(0.0, 1 - nosync_ms / step_ms)),
                          allreduce_alone_ms=ar_ms, gradient_bytes=grad_bytes,
                          allreduce_alone_share_of_step=(None if ar_ms is None else ar_ms / step_ms),
                          optimizer="AdamW(lr=1e-3, weight_decay=0.01)" + (", fused, capturable" if (a.graph and not a.foreach_adamw) else ""), timing="CUDA events over the timed steps after 3 warm-up steps, max over ranks",
                          loss_first=losses[0], loss_last=losses[-1], grad_norm_last=gnorm, params_without_grad=len(no_grad),
                          replicas_equal=replicas_equal, native_vs_autograd_after_training_max_abs=native_vs_autograd)))
if world > 1:
    dist.destroy_process_group()
