#!/usr/bin/env python
"""bench.py — image-pairs/sec of the newUNetTrans bitemporal forward (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload levir256|xbd1024] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

A "step" is one forward over one batch of synthetic image pairs (weights: torch.manual_seed(0) + define_G
random init, exactly what the reference builds).  Workload = BASELINE.json configs[1]: LEVIR 256x256, 64 pairs
per GPU per step, sharded by pair with no collective (weak scaling: every rank runs 64 pairs).
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (which may be read-only)

import torch  # noqa: E402

WORKLOADS = {
    "levir256": dict(H=256, W=256, pairs=64, nc=2, variant="levir",
                     desc="newUNetTrans LEVIR-CD 256x256 batched inference, 64 pairs per GPU per step"),
    "xbd1024": dict(H=1024, W=1024, pairs=8, nc=5, variant="xbd",
                    desc="xBD 1024x1024 pre/post pair 5-class forward, 8 pairs per GPU per step"),
}
DEFAULT_MODE = "tf32x3"     # == dahitra_b200.engine.DEFAULT_MODE: what a user of the module gets without configuration
FALLBACK_PEAKS = dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0)


class Args:
    net_G = "newUNetTrans"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                        bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"]))), "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.proc, self.path = None, f"/tmp/dahitra_clocks_{os.getpid()}.csv"
        try:
            uuid = str(torch.cuda.get_device_properties(device).uuid)
            sel = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            self.cmd = ["nvidia-smi", "-i", sel, f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"]
        except Exception:
            self.cmd = None

    def start(self):
        if self.cmd is None:
            return
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(self.cmd, stdout=self.f, stderr=subprocess.DEVNULL)
            time.sleep(0.25)
        except Exception:
            self.proc = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ----------------------------------------------------------------------------------------------- CPU legs
REF_COPY = os.path.join(ROOT, "baseline", "_ref", "ref")     # unmodified reference sources (baseline/install_reference.py)


def _reference_module(wl):
    """The UNMODIFIED reference network built by the reference's own code from baseline/_ref/ref (import shims only: timm /
    matplotlib stubs, no ImageNet download).  -> (callable(x1, x2) -> logits, kind) or raises."""
    from dahitra_b200 import launch
    nets = launch.install(REF_COPY, stub_missing=True, offline_trunk=True, rebind=False)
    torch.manual_seed(0)
    if wl["variant"] == "levir":
        net = nets.define_G(Args(), gpu_ids=[]).eval()                        # reference models/networks.py:130-168
        assert type(net).__module__ == "models.networks"
        return (lambda a, b: net(a, b)), "reference"
    cwd = os.getcwd()
    xroot = os.path.join(REF_COPY, "xBD_code")
    os.chdir(xroot)                                                           # relative SourceFileLoader in the module
    sys.path.insert(0, xroot)
    try:
        import zoo.model_transformer_encoding as X                            # reference xBD variant
    finally:
        os.chdir(cwd)
    X.bitmodule._resnet = lambda arch, block, layers, pretrained, progress, **kw: X.bitmodule.ResNet(block, layers, **kw)
    net = X.BASE_Transformer_UNet(input_nc=3, output_nc=wl["nc"], token_len=4, resnet_stages_num=4, with_pos="learned",
                                  with_decoder_pos="learned", enc_depth=1, dec_depth=8).eval()
    return (lambda a, b: net(torch.cat([a, b], 1))), "reference"


def _port_module(wl):
    """Fallback when the reference copy is absent: the oracle port of the reference forward (checker / baseline only)."""
    from oracle import dahitra_oracle as O
    from dahitra_b200.networks import define_G
    from dahitra_b200.xbd import BASE_Transformer_UNet as XNet
    torch.manual_seed(0)
    if wl["variant"] == "levir":
        sd = define_G(Args(), gpu_ids=[]).state_dict()
    else:
        sd = XNet(input_nc=3, output_nc=wl["nc"], token_len=4, resnet_stages_num=4, with_pos="learned",
                  with_decoder_pos="learned", enc_depth=1, dec_depth=8).state_dict()
    sd = {k: v.detach() for k, v in sd.items()}
    if wl["variant"] == "levir":
        return (lambda a, b: O.forward_levir(sd, a, b)), "port"
    return (lambda a, b: O.forward_xbd(sd, torch.cat([a, b], 1))), "port"


def cpu_pairs_per_sec(wl, pairs, steps, warmup):
    """The reference's CPU forward on the host cores (all threads): the unmodified reference module when
    baseline/_ref/ref is present, else the oracle port.  -> (pairs/s, s/step, kind, note)"""
    from dahitra_b200 import synth
    import contextlib
    note = None
    try:
        with contextlib.redirect_stdout(sys.stderr):          # the reference prints while it builds; stdout carries ONE JSON line
            fn, kind = _reference_module(wl)
    except Exception as e:                                    # noqa: BLE001 — reported in the JSON line
        note = "reference copy not importable (%s: %s); timed the oracle port instead" % (type(e).__name__, str(e)[:120])
        fn, kind = _port_module(wl)
    x1, x2 = synth.synth_pair(pairs, wl["H"], wl["W"], seed=1, kind="uniform")
    with torch.no_grad():
        for _ in range(warmup):
            fn(x1, x2)
        ts = []
        for _ in range(steps):
            t = time.perf_counter(); fn(x1, x2); ts.append(time.perf_counter() - t)
    sec = sum(ts) / len(ts)
    return pairs / sec, sec, kind, note


def run_reference(a, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    # LEVIR: the workload's own 64-pair batch per step (about 6 s per step on 16 cores); xBD 1024^2: one pair per step
    # (a full 8-pair step takes > 20 s and > 60 GB of host memory in the reference's decoder)
    pairs = a.ref_pairs or (wl["pairs"] if wl["variant"] == "levir" else 1)
    v, sec, kind, note = cpu_pairs_per_sec(wl, pairs, a.steps, min(a.warmup, 1))
    sample = (f"{pairs} pairs per step ({'the whole' if pairs == wl['pairs'] else 'a sample of the'} {wl['pairs']}-pair workload), "
              f"{a.steps} steps after {min(a.warmup, 1)} warm-up, eager PyTorch CPU fp32, {torch.get_num_threads()} threads")
    line = dict(impl="reference", metric="image-pairs/sec", value=v, unit="pairs/s", n_gpus=a.gpus, steps=a.steps,
                warmup=a.warmup, ms_per_step=sec * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic",
                config=dict(workload=wl["desc"], H=wl["H"], W=wl["W"], pairs_per_gpu=wl["pairs"], sample_pairs=pairs,
                            weights="torch.manual_seed(0); define_G random init" if wl["variant"] == "levir" else "torch.manual_seed(0); module default init"),
                cpu_baseline=dict(value=v, unit="pairs/s", cores=torch.get_num_threads(), kind=kind, sample=sample),
                e2e=dict(value=v, unit="pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    if note:
        line["note"] = note
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------- native arm
def _bind_to_gpu_numa_node(local):
    """Run this rank (and first-touch its pinned staging buffers) on the CPUs NVML reports as local to its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def _time_steps(fn, steps, barrier):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


DUMP_BYTES = 64 * 10**6     # --dump-outputs: all files together


def dump_outputs(out_dir, arrays):
    """Write each (B, C, H, W) tensor as out_dir/<name>.npy in float32.  When the whole set would exceed DUMP_BYTES, each array
    is reduced to its C values at a seeded sample of its (b, y, x) positions: <name>.npy is then (n, C) and <name>_index.npy
    (n, 3) holds those positions (float32, exact).  The sample is the same for every run with the same arguments, so two runs or
    two builds write files that compare element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    headers = 2 * 4096 * len(arrays)
    if sum(t.numel() for t in arrays.values()) * 4 + headers <= DUMP_BYTES:
        for name, t in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
        return
    full = sum(t.numel() // t.shape[1] * (t.shape[1] + 3) * 4 for t in arrays.values())     # every position, values + index
    for name, t in arrays.items():
        B, C, H, W = t.shape
        n = B * H * W * (DUMP_BYTES - headers) // full
        pos = torch.randperm(B * H * W, generator=torch.Generator().manual_seed(0))[:n].sort().values
        x = t.detach().float().permute(0, 2, 3, 1).reshape(-1, C).cpu()[pos]
        idx = torch.stack([pos // (H * W), pos // W % H, pos % W], 1).float()
        np.save(os.path.join(out_dir, name + ".npy"), x.numpy())
        np.save(os.path.join(out_dir, name + "_index.npy"), idx.numpy())


def _training_leg(dev, batch=8, steps=10):
    import contextlib
    import torch.nn.functional as F
    from dahitra_b200.networks import define_G
    from dahitra_b200.train_graph import GraphedTrainStep
    torch.manual_seed(0)
    with contextlib.redirect_stdout(sys.stderr):
        net = define_G(Args(), gpu_ids=[dev.index]).train()
    g = torch.Generator(device=dev).manual_seed(100)
    x1 = torch.rand(batch, 3, 256, 256, device=dev, generator=g) * 2 - 1
    x2 = torch.rand(batch, 3, 256, 256, device=dev, generator=g) * 2 - 1
    y = (torch.rand(batch, 256, 256, device=dev, generator=g) < 0.1).long()
    with torch.enable_grad():
        ts = GraphedTrainStep(net, F.cross_entropy, (x1, x2, y),
                              lambda ps: torch.optim.AdamW(ps, lr=1e-3, weight_decay=0.01, capturable=True, fused=True), distributed=False)
        for _ in range(3):
            ts.step(x1, x2, y)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        first = float(ts.loss)
        e0.record()
        for _ in range(steps):
            ts.step(x1, x2, y)
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return dict(workload=f"LEVIR-CD training step, batch {batch}, CE loss, AdamW(1e-3, wd 0.01), one GPU (models/trainer.py:247-262)",
                route="native pixel-decoder / tokenizer forward + backward kernels, channels_last, GraphedTrainStep (two CUDA graphs, fused AdamW)",
                ms_per_step=ms, pairs_per_s_per_gpu=batch / (ms / 1e3), steps=steps, loss_before=first, loss_after=float(ts.loss),
                note="reported next to the headline; multi-GPU form with the NCCL gradient all-reduce: tools/train_step.py --graph")


def run_native(a, wl):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the native arm has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = _bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from dahitra_b200.networks import define_G
    from dahitra_b200.xbd import BASE_Transformer_UNet as XNet
    from dahitra_b200 import synth
    from dahitra_b200.pipeline import PairPipeline

    H, W, Bp = wl["H"], wl["W"], (a.pairs or wl["pairs"])
    levir = wl["variant"] == "levir"
    import contextlib
    torch.manual_seed(0)
    with contextlib.redirect_stdout(sys.stderr):              # init_weights prints like the reference's; stdout carries ONE JSON line
        if levir:
            net = define_G(Args(), gpu_ids=[local]).eval()
        else:
            net = XNet(input_nc=3, output_nc=wl["nc"], token_len=4, resnet_stages_num=4, with_pos="learned",
                       with_decoder_pos="learned", enc_depth=1, dec_depth=8).to(dev).eval()
    sd_cpu = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    from dahitra_b200.engine import MODES
    net.set_mode(a.flags if a.flags is not None else a.mode)
    mode_name = next((k for k, v in MODES.items() if v == net._engine.flags), f"flags{net._engine.flags}")
    # rotating input sets so consecutive steps never re-read the same inputs from L2 (3 x 100 MB > 126 MB L2;
    # the multi-GB per-step intermediates stream through HBM regardless)
    nsets = 3
    sets = []
    for i in range(nsets):
        x1, x2 = synth.synth_pair(Bp, H, W, seed=100 + 10 * rank + i, kind="uniform")
        sets.append((x1.to(dev), x2.to(dev)))

    def fwd(x1, x2):
        return net(x1, x2) if levir else net._engine.forward_pair(net, x1, x2)

    def step(i):
        return fwd(*sets[i % nsets])

    last = {}

    def timed_step(i):
        y = step(i)
        if i == a.steps - 1:
            last["logits"] = y

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for i in range(max(a.warmup, 3)):
            step(i)
        barrier()
        sampler = ClockSampler(dev) if rank == 0 else None
        if sampler:
            sampler.start()
        ms = _time_steps(timed_step, a.steps, barrier)
        # ---- strong scaling (configs[1] as written: ONE global batch of 64 pairs split 64/N per rank, no collective)
        gB = wl["pairs"]
        sB = max(1, gB // world)
        ssets = [(s[0][:sB].contiguous(), s[1][:sB].contiguous()) for s in sets]
        for i in range(3):
            fwd(*ssets[i % nsets])
        ms_strong = _time_steps(lambda i: fwd(*ssets[i % nsets]), a.steps, barrier)
        # the same as replayed CUDA graphs (one per input set): at 64/N pairs per rank the step is ~40 dependent launches of
        # 8-15 us each, and N processes issuing them from Python share the host's cores
        sgraphs = []
        for sset in ssets:
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_):
                y_ = fwd(*sset)
            sgraphs.append((g_, y_))
        for i in range(3):
            sgraphs[i % nsets][0].replay()
        ms_strong_graph = _time_steps(lambda i: sgraphs[i % nsets][0].replay(), a.steps, barrier)
        del sgraphs
        # ---- e2e through the public pipeline API, host buffers in / class maps out, copies inside the timed region.
        #      Primary: uint8 HWC images as an image reader delivers them (normalised on the device, bit-identical to the
        #      reference loaders); sub-key f32: already-normalised fp32 NCHW host tensors (4x the PCIe bytes).
        kind = "levir" if levir else "xbd"
        g = torch.Generator().manual_seed(500 + rank)
        hu8 = [(torch.randint(0, 256, (Bp, H, W, 3), generator=g, dtype=torch.uint8).pin_memory(),
                torch.randint(0, 256, (Bp, H, W, 3), generator=g, dtype=torch.uint8).pin_memory()) for _ in range(nsets)]
        hx = [(s[0].cpu().pin_memory(), s[1].cpu().pin_memory()) for s in sets]

        def run_pipe(pipe, host):
            for _ in pipe.run(host[i % nsets] for i in range(3)):
                pass
            barrier()
            # steady state of one pipe.run over K + 3 batches: the clock starts when result #3 is handed out and stops at
            # result #K+3, so K uploads, K forwards and K downloads lie inside it
            t_fill = time.perf_counter()
            nres, t0 = 0, None
            for _pred in pipe.run(host[i % nsets] for i in range(a.steps + 3)):
                nres += 1
                if nres == 3:
                    t0 = time.perf_counter()
            sec = time.perf_counter() - t0
            barrier()
            fill = (time.perf_counter() - t_fill) * a.steps / (a.steps + 3)
            assert nres == a.steps + 3
            return sec, fill

        def h2d_alone(host, like):
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d1, d2 = torch.empty_like(like[0], device=dev), torch.empty_like(like[1], device=dev)
            torch.cuda.synchronize()
            h0.record()
            for i in range(3):
                d1.copy_(host[i % nsets][0], non_blocking=True)
                d2.copy_(host[i % nsets][1], non_blocking=True)
            h1.record()
            torch.cuda.synchronize()
            return h0.elapsed_time(h1) / 3

        e2e_sec, e2e_fill_sec = run_pipe(PairPipeline(net, out="argmax_u8", inputs="u8_hwc", kind=kind), hu8)
        f32_sec, f32_fill_sec = run_pipe(PairPipeline(net, out="argmax_u8"), hx)
        h2d_u8_ms, h2d_f32_ms = h2d_alone(hu8, hu8[0]), h2d_alone(hx, hx[0])
        # what models/evaluator.py:89-103 does, un-pipelined: .to(device), forward, argmax, int64 map to the host, sync
        pred_h = torch.empty((Bp, H, W), dtype=torch.int64).pin_memory()

        def e2e_step(i):
            h1, h2 = hx[i % nsets]
            y = fwd(h1.to(dev, non_blocking=True), h2.to(dev, non_blocking=True))
            pred_h.copy_(torch.argmax(y, dim=1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for i in range(2):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(a.steps):
            e2e_step(i)
        barrier()
        e2e_sync_sec = time.perf_counter() - t0
        clocks = sampler.stop() if sampler else None
        # ---- per-launch profile (after the timed regions): roofline of the dominant kernel
        prof = None
        if rank == 0:
            runs = [net._engine.profile_pair(net, *sets[i % nsets]) for i in range(3)]
            prof = [dict(name=r["name"], flops=r["flops"], bytes=r["bytes"],
                         ms=statistics.mean(x[j]["ms"] for x in runs)) for j, r in enumerate(runs[0])]
        # ---- in-run parity of the timed mode, outside the timed region: (1) against the ORACLE (CPU restatement of the
        #      reference, fp64) on a few pairs of the timed inputs, (2) against the strict fp32 mode on 8 pairs
        parity, strict = None, None
        if rank == 0 and not a.no_parity:
            from oracle import dahitra_oracle as O             # checker only
            npar = 2 if levir else 1
            xa, xb = sets[0][0][:npar].contiguous(), sets[0][1][:npar].contiguous()
            y_mode = fwd(xa, xb).double().cpu()
            torch.set_num_threads(os.cpu_count())
            t0 = time.perf_counter()
            if levir:
                y_orc = O.forward_levir(sd_cpu, xa.cpu(), xb.cpu(), dtype=torch.float64)
            else:
                y_orc = O.forward_xbd(sd_cpu, torch.cat([xa.cpu(), xb.cpu()], 1), dtype=torch.float64)
            d = (y_mode - y_orc).abs()
            parity = dict(against="oracle (CPU restatement of the reference forward, fp64), same weights, %d pair(s) of the timed inputs" % npar,
                          max_abs=float(d.max()), mean_abs=float(d.mean()), ref_abs_max=float(y_orc.abs().max()),
                          outside_tol=int((d > 1e-4 + 1e-3 * y_orc.abs()).sum()), tol="1e-4 + 1e-3*|ref|", elements=d.numel(),
                          argmax_agree=float((y_mode.argmax(1) == y_orc.argmax(1)).float().mean()),
                          oracle_seconds=time.perf_counter() - t0)
        if rank == 0 and levir and not a.no_parity:
            nb = min(8, Bp)
            xa, xb = sets[0][0][:nb].contiguous(), sets[0][1][:nb].contiguous()
            y_mode = net(xa, xb).double()
            saved = net._engine.flags
            net._engine.flags = 0
            y_ref = net(xa, xb).double()
            d = (y_mode - y_ref).abs()
            parity["vs_strict_fp32_mode"] = dict(pairs=nb, max_abs=float(d.max()), outside_tol=int((d > 1e-4 + 1e-3 * y_ref.abs()).sum()),
                                                 argmax_agree=float((y_mode.argmax(1) == y_ref.argmax(1)).float().mean()))
            # the other shipped modes on the same workload (5 steps each): throughput + their own parity against fp32
            strict = {}
            for other in ("fp32", "tf32", "f16"):
                if MODES[other] == saved:
                    continue
                net._engine.flags = MODES[other]
                y_o = net(xa, xb).double()
                for i in range(2):
                    step(i)
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                s0.record()
                for i in range(5):
                    step(i)
                s1.record()
                torch.cuda.synchronize()
                do = (y_o - y_ref).abs()
                strict[other] = dict(value=Bp / (s0.elapsed_time(s1) / 5 / 1e3), unit="pairs/s per GPU",
                                     max_abs_vs_fp32=float(do.max()), outside_tol=int((do > 1e-4 + 1e-3 * y_ref.abs()).sum()),
                                     argmax_agree=float((y_o.argmax(1) == y_ref.argmax(1)).float().mean()))
            net._engine.flags = saved
    tmax = torch.tensor([ms, e2e_sec * 1e3, e2e_sync_sec * 1e3, ms_strong, f32_sec * 1e3, h2d_u8_ms, h2d_f32_ms, ms_strong_graph],
                        device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms, e2e_ms, e2e_sync_ms, ms_strong, f32_ms, h2d_u8_ms, h2d_f32_ms, ms_strong_graph = (float(v) for v in tmax)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- configs[3] next to the headline (rank 0 only, no collective: the other ranks are gone): the LEVIR training step,
    #      batch 8, CE loss, AdamW, on the native training kernels as two replayed CUDA graphs (dahitra_b200/train_graph.py).
    #      Reported, not part of `value`; tools/train_step.py is the multi-GPU form with the gradient all-reduce.
    training = None
    if levir and not a.no_train:
        try:
            training = _training_leg(dev)
        except Exception as e:                                  # never lose the headline line to the side measurement
            training = dict(error=repr(e)[:300])
    peaks, peak_src = load_peaks()
    ms_step = ms / a.steps
    value = world * Bp / (ms_step / 1e3)
    e2e_value = world * Bp * a.steps / (e2e_ms / 1e3)
    top = max(prof, key=lambda r: r["ms"])
    ridge = peaks["bf16_tflops_sustained"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
    ai = top["flops"] / max(top["bytes"], 1.0)
    if ai > ridge:
        achieved = top["flops"] / (top["ms"] * 1e-3) / 1e12
        roof = dict(kernel=top["name"], bound="tensor", achieved=achieved, peak=peaks["bf16_tflops_sustained"],
                    unit="TFLOP/s", frac=achieved / peaks["bf16_tflops_sustained"])
        # what the tensor pipe actually executes per algorithmic product, in units of one 16-bit (kind::f16) MMA pass:
        # single-pass 16-bit = 1, single-pass TF32 = 2 (half rate), folded x3 = 3 (one N-doubled + one narrow 16-bit pass),
        # three TF32 passes = 6
        fl = net._engine.flags
        mult = 1.0 if (fl & 1024) else ((3.0 if (fl & 2048) else 4.0 if (fl & 512) else 6.0) if (fl & 2) else (1.0 if (fl & 2048) else 2.0))
        roof["tensor_pipe"] = dict(mma_tflops_16bit_equiv=achieved * mult, passes_16bit_equiv_per_product=mult,
                                   peak_tflops=peaks["bf16_tflops_sustained"],
                                   frac=achieved * mult / peaks["bf16_tflops_sustained"],
                                   note="executed kind::f16-equivalent MMA throughput (a kind::tf32 pass counts 2) against the measured bf16 rate")
    else:
        achieved = top["bytes"] / (top["ms"] * 1e-3) / 1e9
        roof = dict(kernel=top["name"], bound="hbm", achieved=achieved, peak=peaks["hbm_gbs"], unit="GB/s",
                    frac=achieved / peaks["hbm_gbs"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")      # per-launch DRAM bytes from the committed ncu capture
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(mode_name, {}).get(top["name"])
    prof_ms = sum(r["ms"] for r in prof)
    roof.update(traffic=traffic, peak_source=f"MEASURED_PEAKS.json ({peak_src}; sustained bf16 for a kernel inside a step)",
                ai_flop_per_byte=ai, launch_ms=top["ms"], share_of_step=top["ms"] / prof_ms,
                algorithmic_flops=top["flops"], algorithmic_bytes=top["bytes"],
                whole_step=dict(algorithmic_gflop=sum(r["flops"] for r in prof) / 1e9,
                                algorithmic_mb=sum(r["bytes"] for r in prof) / 1e6, profiled_ms=prof_ms,
                                hbm_frac=sum(r["bytes"] for r in prof) / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                tensor_frac=sum(r["flops"] for r in prof) / (ms_step * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"]))
    kernels = sorted(prof, key=lambda r: -r["ms"])[:6]
    if a.dump_kernels:
        os.makedirs(os.path.dirname(os.path.abspath(a.dump_kernels)), exist_ok=True)
        json.dump(dict(flags=net._engine.flags, pairs=Bp, H=H, W=W, peaks=peaks, launches=prof), open(a.dump_kernels, "w"), indent=1)
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count())
        try:
            os.sched_setaffinity(0, range(os.cpu_count()))          # the CPU leg uses every host core
        except Exception:
            pass
        cp = 16 if levir else 1
        v, sec, ckind, note = cpu_pairs_per_sec(wl, cp, 2, 1)
        cpu = dict(value=v, unit="pairs/s", cores=torch.get_num_threads(), kind=ckind,
                   sample=f"{'unmodified reference module' if ckind == 'reference' else 'oracle port'} (eager PyTorch CPU fp32), {cp} pairs per call of the "
                          f"{wl['pairs']}-pair workload, mean of 2 calls after 1 warm-up ({sec:.2f} s/call)")
        if note:
            cpu["note"] = note
    in_u8, in_f32 = 2 * Bp * 3 * H * W, 2 * Bp * 3 * H * W * 4
    line = dict(metric="image-pairs/sec", value=value, unit="pairs/s", n_gpus=world, steps=a.steps, warmup=max(a.warmup, 3),
                ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype={"fp32": "f32", "tf32": "tf32", "tf32_fast": "tf32", "tf32x3": "x3 error-compensated f16 products (f16 main + scaled-remainder corrections; decoder: 3xTF32), fp32 accumulate",
                       "tf32x3_unfolded": "x3 error-compensated (convs: f16 main + bf16 corrections; stem/decoder: 3xTF32), fp32 accumulate and storage",
                       "tf32x3_tf32main": "x3 error-compensated (tf32 main + bf16 corrections), fp32 accumulate and storage",
                       "tf32x3_pure": "3xTF32 (error-compensated), fp32 accumulate and storage", "bf16": "bf16 operands, fp32 accumulate and storage",
                       "f16": "f16 operands, fp32 accumulate and storage"}.get(mode_name, "f32/tf32"),
                data="synthetic",
                config=dict(workload=wl["desc"], H=H, W=W, pairs_per_gpu=Bp, global_pairs_per_step=world * Bp,
                            sharding="by image pair, one process per GPU, no collective",
                            weights="torch.manual_seed(0); define_G random init" if levir else "torch.manual_seed(0); module default init",
                            mode=mode_name, flags=net._engine.flags,
                            l2="3 rotating input sets (3x%.0f MB) + multi-GB per-step intermediates >> 126 MB L2" % (in_f32 / 1e6)),
                clocks=clocks,
                training_step=training,
                strong_scaling=dict(global_pairs_per_step=sB * world, pairs_per_gpu=sB, value=sB * world / (ms_strong / a.steps / 1e3),
                                    unit="pairs/s", ms_per_step=ms_strong / a.steps,
                                    cuda_graph=dict(value=sB * world / (ms_strong_graph / a.steps / 1e3), ms_per_step=ms_strong_graph / a.steps,
                                                    note="the same forward captured once per input set and replayed"),
                                    note="configs[1] as written: one global batch split evenly over the ranks, no collective; "
                                         "efficiency at N = this value / (N=1 value)"),
                e2e=dict(value=e2e_value, unit="pairs/s", h2d_bytes_per_step=in_u8, d2h_bytes_per_step=Bp * H * W,
                         ms_per_step=e2e_ms / a.steps, over_value=e2e_value / value,
                         timing="steady state of one PairPipeline.run: K results between the 3rd and the (K+3)th hand-out (wall clock)",
                         ms_per_step_including_fill=e2e_fill_sec * 1e3 / a.steps, h2d_alone_ms_per_step=h2d_u8_ms,
                         host_numa_cpus=numa_cpus,
                         api="dahitra_b200.pipeline.PairPipeline(net, inputs='u8_hwc').run(pinned uint8 HWC host batches): H2D of batch i+1 "
                             "overlaps the forward of batch i; normalisation on the device; uint8 class map D2H every step",
                         f32_inputs=dict(value=world * Bp * a.steps / (f32_ms / 1e3), h2d_bytes_per_step=in_f32, d2h_bytes_per_step=Bp * H * W,
                                         ms_per_step=f32_ms / a.steps, h2d_alone_ms_per_step=h2d_f32_ms,
                                         api="PairPipeline(net).run(pinned fp32 NCHW host batches)"),
                         unpipelined=dict(value=world * Bp * a.steps / (e2e_sync_ms / 1e3), h2d_bytes_per_step=in_f32, d2h_bytes_per_step=Bp * H * W * 8,
                                          api="net(x1.to(dev), x2.to(dev)); torch.argmax(.,1) -> pinned host int64 map; per-step sync")),
                parity=parity, other_modes=strict,
                gpu_launches=len(prof) * a.steps, launches_per_step=len(prof),
                roofline=roof, top_kernels=[dict(name=k["name"], ms=round(k["ms"], 4)) for k in kernels])
    if cpu:
        line["cpu_baseline"] = cpu
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, last)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="levir256", choices=list(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=None, help="pairs per GPU per step (default: the workload's)")
    ap.add_argument("--mode", default=DEFAULT_MODE, help="precision mode of the native engine: fp32 | tf32 | tf32_fast | tf32x3")
    ap.add_argument("--flags", type=int, default=None, help="raw DH_FLAG_* bitmask (overrides --mode)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step leg (configs[3], rank 0, ~5 s)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity block (oracle on CPU + other modes)")
    ap.add_argument("--ref-pairs", type=int, default=None, help="--impl reference: pairs per step (default: the workload batch for LEVIR, 1 for xBD)")
    ap.add_argument("--dump-kernels", default=None, help="write the per-launch table (name, ms, flops, bytes) to this JSON file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned (rank 0) to DIR/<name>.npy in float32, at most 64 MB in all "
                         "(beyond that, the values at a fixed seeded sample of (b, y, x) positions, listed in DIR/<name>_index.npy); "
                         "the inputs depend only on the arguments")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the native arm's outputs; the reference arm times other inputs (one CPU sample)")
    wl = WORKLOADS[a.workload]
    if a.impl == "reference":
        return run_reference(a, wl)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.gpus != world and world == 1 and a.gpus > 1:
        # convenience: re-launch under torchrun when asked for N>1 without it
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_native(a, wl)


if __name__ == "__main__":
    sys.exit(main())
