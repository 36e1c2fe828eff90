"""Cost of random pushes on the bench workload: per-step time of the same workload as it is (plain), with
randomised dynamics (+rand) and with randomised dynamics and pushes (+rand+push), for the latency build at 4096
envs, the throughput build at 65 536 envs and the body build at 4096 envs (the configs of tools/gpu_rand_cost.py;
+rand adds the ranges of configs/bench12_walk_rand.yaml, +push the push keys of configs/bench12_walk_push.yaml).
Timed as tools/gpu_rand_cost.py times: random actions, the L2 flushed before every step, CUDA events around each
step, summed; the three arms of a build alternate in rounds.  Prints one JSON line per build and writes them all,
with the card name and power limit read in the same run, to --out.

    python tools/gpu_push_cost.py --out profiles/push_cost.json
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from solorl_b200.envs import SoloVecEnv  # noqa: E402
from tools.gpu_rand_cost import CASES, RAND_KEYS, card, load, timed_steps  # noqa: E402

PUSH_KEYS = ("push_force", "push_interval", "push_duration")
ARMS = ("plain", "rand", "rand_push")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_push_cost.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    rand, push = load("bench12_walk_rand.yaml"), load("bench12_walk_push.yaml")
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    lines = []
    for build, cfg_name, n in CASES:
        plain = load(cfg_name)
        with_rand = dict(plain, **{k: rand[k] for k in RAND_KEYS})
        cfgs = {"plain": plain, "rand": with_rand, "rand_push": dict(with_rand, **{k: push[k] for k in PUSH_KEYS})}
        envs = {arm: SoloVecEnv(cfgs[arm], n, device=dev, seed=0) for arm in ARMS}
        g = torch.Generator(device=dev).manual_seed(1000)
        acts = [torch.rand(n, envs["plain"].sim.act_dim, device=dev, generator=g) * 2 - 1 for _ in range(16)]
        for e in envs.values():
            e.reset()
            for i in range(args.warmup):
                e.sim.step(acts[i % len(acts)])
        torch.cuda.synchronize()
        ms = {arm: [] for arm in ARMS}
        for _ in range(args.rounds):
            for arm in ARMS:
                ms[arm].append(timed_steps(envs[arm], acts, flush, args.steps))
        line = {"build": build, "config": cfg_name, "envs": n, "steps_per_round": args.steps,
                "l2": "flushed (256 MiB write) before every timed step, per-step CUDA events summed"}
        for arm in ARMS:
            line[f"variant_{arm}"] = envs[arm].sim.step_variant
            line[f"ms_per_step_{arm}"] = float(np.median(ms[arm]))
            line[f"rounds_{arm}"] = ms[arm]
        line["push_cost_pct_vs_rand"] = 100.0 * (line["ms_per_step_rand_push"] / line["ms_per_step_rand"] - 1.0)
        line["push_cost_pct_vs_plain"] = 100.0 * (line["ms_per_step_rand_push"] / line["ms_per_step_plain"] - 1.0)
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
