"""LEVIR-CD training step in fp32 (TF32 convolutions, torch's default) against mixed precision (autocast fp16 with loss scaling,
autocast bf16), for the graphed step (GraphedTrainStep) and the eager loop: tools/train_step.py runs once per configuration, the
configurations alternating over several rounds in one session so that drift of the shared machine lands on all of them alike.
Records the card's name and power limit with the numbers.
   python tools/train_step_amp_ab.py --out profiles/r03_train_step_amp.json [--rounds 2] [--steps 100] [--batch 8]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ap = argparse.ArgumentParser()
ap.add_argument("--out", required=True)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("--steps", type=int, default=100)
ap.add_argument("--batch", type=int, default=8)
a = ap.parse_args()

CONFIGS = [(loop, amp) for loop in ("graph", "eager") for amp in (None, "fp16", "bf16")]
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()
runs = {f"{loop} {amp or 'fp32'}": [] for loop, amp in CONFIGS}
for r in range(a.rounds):
    for loop, amp in CONFIGS:
        cmd = [sys.executable, os.path.join(HERE, "train_step.py"), "--steps", str(a.steps), "--batch", str(a.batch)]
        cmd += ["--graph"] if loop == "graph" else []
        cmd += ["--amp", amp] if amp else []
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            sys.exit(f"{' '.join(cmd)} failed:\n{p.stdout}\n{p.stderr}")
        res = json.loads(p.stdout.strip().splitlines()[-1])
        runs[f"{loop} {amp or 'fp32'}"].append(res)
        print(f"round {r} {loop:5s} {amp or 'fp32'}: {res['step_ms']:.3f} ms/step, loss {res['loss_first']:.4f} -> {res['loss_last']:.4f}",
              flush=True)
summary = {k: dict(step_ms_median=statistics.median(x["step_ms"] for x in v), step_ms_all=[x["step_ms"] for x in v],
                   pairs_per_s_median=statistics.median(x["pairs_per_s"] for x in v), loss_last=[x["loss_last"] for x in v],
                   native_vs_autograd_after_training_max_abs=[x["native_vs_autograd_after_training_max_abs"] for x in v])
           for k, v in runs.items()}
for loop in ("graph", "eager"):
    base = summary[f"{loop} fp32"]["step_ms_median"]
    for amp in ("fp16", "bf16"):
        summary[f"{loop} {amp}"]["speedup_vs_fp32"] = base / summary[f"{loop} {amp}"]["step_ms_median"]
out = dict(workload=f"LEVIR-CD training step, batch {a.batch}, 256x256, 1 GPU, CE loss, AdamW (tools/train_step.py)",
           card=card, timing=f"CUDA events over {a.steps} steps after warm-up, one process per run; configurations alternated over "
                             f"{a.rounds} rounds in one session; median over the rounds",
           summary=summary, runs=runs)
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps({k: (v["step_ms_median"], v.get("speedup_vs_fp32")) for k, v in summary.items()}))
