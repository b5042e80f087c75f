"""configs[4] of BASELINE.json: 1024x1024 pre/post pairs cut into 16 tiles of 256x256 on the device, pushed through the
LEVIR-variant module built with output_nc=5, in a reduced-precision mode ("bf16" by default; "h16" stores every activation as
one FP16 plane as well), compared on the 16 tiles of the first pair against the repository's fp32 mode and against the fp64
oracle (oracle.dahitra_oracle.forward_levir; separately stated tolerance: |d| <= 2e-3 + 2e-2 |ref|, argmax agreement >= 99.5 %).
Inputs are decoded uint8 HWC images already on the device; the timed region = normalise + tile + forward + fused argmax.
   python tools/bench_tiled1024.py [--batches 1,4,16,64] [--mode bf16|h16|...]          (one GPU)
   python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/bench_tiled1024.py   (N GPUs, by pair)
Prints one JSON line per batch size from rank 0."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from oracle import dahitra_oracle as O
from dahitra_b200.networks import BASE_Transformer_UNet, init_weights
from dahitra_b200.inputs import normalize_u8

ap = argparse.ArgumentParser()
ap.add_argument("--batches", default="1,4,16,64")
ap.add_argument("--mode", default="bf16")
ap.add_argument("--steps", type=int, default=10)
a = ap.parse_args()
world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl")
torch.manual_seed(0)
net = BASE_Transformer_UNet(3, 5, 'learned', resnet_stages_num=4, with_decoder_pos='learned', enc_depth=1, dec_depth=8)
init_weights(net, 'normal', 0.02)
net = net.cuda().eval()
CHUNK = 128                                                     # tiles per forward call (7 GB of workspace)


def parity_of(y, m, y_ref):
    d = (y.double() - y_ref.double()).abs()
    return dict(max_abs=float(d.max()), mean_abs=float(d.mean()), outside_tol=int((d > 2e-3 + 2e-2 * y_ref.double().abs()).sum()),
                elements=d.numel(), argmax_agree=float((m == y_ref.argmax(1)).float().mean()), tol="2e-3 + 2e-2*|ref|, argmax >= 99.5 %")


def run(pre, post, mode, want_logits=False):
    net.set_mode(mode)
    t1, t2 = normalize_u8(pre, "levir", tile=256), normalize_u8(post, "levir", tile=256)
    maps, logits = [], []
    for c in range(0, t1.shape[0], CHUNK):
        y = net._engine.forward_pair(net, t1[c:c + CHUNK], t2[c:c + CHUNK], want_argmax=True)
        maps.append(net._engine.last_argmax.clone())
        if want_logits:
            logits.append(y.clone())
    return torch.cat(maps), (torch.cat(logits) if want_logits else None)


for B in [int(b) for b in a.batches.split(",")]:
    Bl = max(1, B // world)                                     # pairs per GPU (sharded by pair, no collective)
    g = torch.Generator(device="cuda").manual_seed(7 + rank)
    pre = torch.randint(0, 256, (Bl, 1024, 1024, 3), device="cuda", generator=g, dtype=torch.uint8)
    post = torch.randint(0, 256, (Bl, 1024, 1024, 3), device="cuda", generator=g, dtype=torch.uint8)
    with torch.no_grad():
        m_ref, y_ref = run(pre[:1], post[:1], "fp32", want_logits=True)
        m_low, y_low = run(pre[:1], post[:1], a.mode, want_logits=True)
        parity = parity_of(y_low, m_low, y_ref)
        if B == int(a.batches.split(",")[0]):                     # the fp64 oracle on the same 16 tiles (CPU, once)
            sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
            t1, t2 = (normalize_u8(t, "levir", tile=256).cpu() for t in (pre[:1], post[:1]))
            ref64 = O.forward_levir(sd, t1, t2, dtype=torch.float64)
            parity_oracle = parity_of(y_low.cpu(), m_low.cpu(), ref64)
        for _ in range(3):
            run(pre, post, a.mode)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            run(pre, post, a.mode)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / a.steps], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(json.dumps(dict(workload="1024x1024 pairs tiled to 16 x 256x256 on the device, LEVIR-variant module with output_nc=5",
                              mode=a.mode, n_gpus=world, pairs_per_step=Bl * world, tiles_per_step=16 * Bl * world, ms_per_step=float(ms),
                              value=Bl * world / float(ms) * 1e3, unit="1024x1024 pairs/s", parity_vs_fp32_mode=parity,
                              parity_vs_fp64_oracle=parity_oracle)), flush=True)
if world > 1:
    dist.destroy_process_group()
