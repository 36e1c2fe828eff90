"""Cost of per-env randomised dynamics on the bench workload: per-step time of the same workload with
randomisation off and on, for the latency build at 4096 envs, the throughput build at 65 536 envs and the body
build at 4096 envs (configs/bench12_walk.yaml, configs/bench12_walk_body.yaml; the "on" arm adds the ranges of
configs/bench12_walk_rand.yaml).  Timed like bench.py: random actions, the L2 flushed by a 256 MiB write before
every step, CUDA events around each step, summed.  The two arms of a build alternate in rounds so that drift of a
shared machine falls on both.  Prints one JSON line per build and writes them all, with the card name and power
limit read in the same run, to --out.

    python tools/gpu_rand_cost.py --out profiles/rand_cost.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from solorl_b200.envs import SoloVecEnv  # noqa: E402

RAND_KEYS = ("randomize_friction", "randomize_base_mass", "randomize_motor_strength")
CASES = (("latency", "bench12_walk.yaml", 4096), ("throughput", "bench12_walk.yaml", 65536),
         ("body", "bench12_walk_body.yaml", 4096))


def load(name):
    with open(os.path.join(ROOT, "configs", name)) as f:
        return yaml.safe_load(f)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def timed_steps(env, acts, flush, steps):
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.fill_(float(i))
        evs[i][0].record()
        env.sim.step(acts[i % len(acts)])
        evs[i][1].record()
    torch.cuda.synchronize()
    return float(sum(a.elapsed_time(b) for a, b in evs)) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_rand_cost.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    rand = load("bench12_walk_rand.yaml")
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    lines = []
    for build, cfg_name, n in CASES:
        cfg_off = load(cfg_name)
        cfg_on = dict(cfg_off, **{k: rand[k] for k in RAND_KEYS})
        envs = {"off": SoloVecEnv(cfg_off, n, device=dev, seed=0), "on": SoloVecEnv(cfg_on, n, device=dev, seed=0)}
        g = torch.Generator(device=dev).manual_seed(1000)
        acts = [torch.rand(n, envs["off"].sim.act_dim, device=dev, generator=g) * 2 - 1 for _ in range(16)]
        for e in envs.values():
            e.reset()
            for i in range(args.warmup):
                e.sim.step(acts[i % len(acts)])
        torch.cuda.synchronize()
        ms = {"off": [], "on": []}
        for _ in range(args.rounds):
            for arm in ("off", "on"):
                ms[arm].append(timed_steps(envs[arm], acts, flush, args.steps))
        line = {"build": build, "config": cfg_name, "envs": n,
                "variant_off": envs["off"].sim.step_variant, "variant_on": envs["on"].sim.step_variant,
                "ms_per_step_off": float(np.median(ms["off"])), "ms_per_step_on": float(np.median(ms["on"])),
                "rounds_off": ms["off"], "rounds_on": ms["on"], "steps_per_round": args.steps,
                "l2": "flushed (256 MiB write) before every timed step, per-step CUDA events summed"}
        line["cost_pct"] = 100.0 * (line["ms_per_step_on"] / line["ms_per_step_off"] - 1.0)
        print(json.dumps(line), flush=True)
        lines.append(line)
        for e in envs.values():
            e.close()
    rec = {"card": card(), "torch": torch.__version__, "results": lines}
    print(json.dumps({"card": rec["card"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
