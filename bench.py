#!/usr/bin/env python
"""bench.py — env-steps/sec of the batched Solo12 env step (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (this repo's CUDA path)
  python bench.py --impl reference --gpus N --steps K ...   (CPU arm: the reference's path)
  ... --dump-outputs DIR    also write obs / reward / done of the last timed step as DIR/<name>.npy (rank 0)

Workload (BASELINE.json configs[1]): Solo12, task walk, torque control, num_history_stack 1,
frame_skip 4 at 1/240 s, 4096 envs per GPU, random actions U(-1,1)^12, auto-reset on.
A "step" is one vectorised env step of all envs of a rank (= 4 physics substeps + observation +
reward + termination + auto-reset per env).  `value` times the step with actions already in
HBM; `e2e` times the same step through the host-buffer C-ABI call (solo_step_host: H2D actions,
kernel, D2H obs/reward/done, sync).  N > 1: one process per GPU (torchrun), independent env
shards, no data-path collective ("weak" scaling); time = max over ranks.

The reference's own arithmetic for this path is PyBullet, which is not installable in this
image, so the CPU arm (`--impl reference`, and the `cpu_baseline` object) times this repo's
double-precision CPU restatement (oracle/, kind "port") on all host threads.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
CONFIG = {"model_urdf": "solo12", "mode": "headless", "episode_length": 400, "frame_skip": 4,
          "control": "torque", "task": "walk", "num_history_stack": 1, "flat_ground": True}
WORKLOAD = "configs/basic12.yaml-shaped: Solo12 walk, torque control, H=1, frame_skip 4, random actions"


def workload_config(n, world):
    """`config` of the JSON line: the workload, IDENTICAL in both arms (`--impl ours` / `--impl reference`); what
    differs between the arms (kernel build, host cores, how resets are produced) is reported under `run`."""
    return {"workload": WORKLOAD, "envs_per_gpu": n, "robot": "solo12", "task": "walk", "control": "torque",
            "num_history_stack": 1, "episode_length": 400, "frame_skip": 4, "solver_iters": 50,
            "solver_residual_threshold": 1e-7, "joint_limits": 1, "body_contacts": 0,
            "resets": "every auto-reset settles 5..11 zero-torque control steps (baseEnv.py:79-80): simulated by the CPU "
                      "arm, looked up in the bit-identical reset cache by the GPU arm",
            "l2": "GPU arm: flushed (256 MiB write) between timed steps, per-step CUDA events summed; CPU arm: not applicable",
            "parallelism": f"env-shard x{world}"}


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(path, arrays):
    """Write what the timed path returned in its last step as `path/<name>.npy`, float32, so that two builds can be
    compared output for output.  Above 64 MiB in all, the same fixed, seeded sample of rows (envs) is kept in every
    array."""
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes for a in arrays.values()) // n
    keep = (DUMP_LIMIT_BYTES - 1024 * len(arrays)) // row_bytes     # 1 KiB per file covers the .npy header
    if keep < n:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def algorithmic_flops_per_env_step(nj, nc_sum, sweep_feet, frame_skip=4):
    """SURVEY.md §8(d): F_step = S (F_ABA + F_int) + sum_substeps (F_setup + F_PGS) + 400 with m = 3 nc
    rows per substep.  nc_sum = sum over the S substeps of feet in contact; sweep_feet = sum over
    substeps of feet in contact x PGS sweeps actually run (K = 50 only when the residual test never
    fires), both measured by the kernel (solo_get_work_counters)."""
    nb, ndof = nj + 1, nj + 6
    f_aba = 429 * nb - 502
    f_setup = 3.0 * nc_sum * (250 * nb + 2 * ndof)
    f_pgs = 3.0 * sweep_feet * (4 * ndof + 10)
    f_int = 80 * nb
    return frame_skip * (f_aba + f_int) + f_setup + f_pgs + 400


def algorithmic_bytes_per_env_step(nj, D):
    """SURVEY.md §8(d): read state(13+2nj)+action(nj)+contact(4)+scalars(8+3); write state+obs(D)+
    reward+done+contact+scalars, fp32."""
    rd = (16 + 2 * nj) + nj + 4 + 12
    wr = (16 + 2 * nj) + D + 2 + 4 + 12
    return 4 * (rd + wr)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled from a thread (a query takes
    ~0.1 ms, the timed region of a default run a few ms), `nvidia-smi -lms` as the fallback when the NVML binding
    is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None
        self.nvml, self.h, self.sm, self.bits, self.run = None, None, [], 0, False
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = gpu_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[gpu_index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while self.run:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.bits |= int(reasons(self.h))
            except Exception:
                break
            time.sleep(0.0002)

    def start(self):
        if self.nvml is not None:
            self.run = True
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.run = False
            self.t.join(timeout=1.0)
            if not self.sm:            # the region was shorter than one query: sample right after it
                try:
                    self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM)))
                except Exception:
                    pass
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(v for b, v in self.BITS.items() if self.bits & b), "samples": len(self.sm),
                    "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for k, nme in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
            dist.init_process_group("nccl")
        else:
            dist.init_process_group("gloo")
    return rank, world, local


def host_threads():
    """All host threads this process may run on.  Not omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1 to
    every rank, which would time the CPU arm on a single thread at N > 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


CPU_RESET_NOTE = ("resets simulated: every auto-reset runs its 5..11 zero-torque settle steps, as the reference does "
                  "(baseEnv.py:79-80); the GPU arm looks the same trajectories up in its reset cache (bit-identical, "
                  "reset_mode 'cached') and reports the simulate-mode figure under 'reset_mode_simulate'")


def pin_rank_to_cores(local, world):
    """One core set per rank.  The ranks of a torchrun job inherit the SAME affinity mask (all eight ranks of the
    round-1 scaling run shared CPUs 0-31), and each spins in a stream synchronise once per host-buffer step, so
    they fought over cores: e2e efficiency 0.92 at N = 8 with the device figure at 0.99."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if world <= 1 or len(cpus) < world:
            return len(cpus)
        per = len(cpus) // world
        mine = cpus[local * per:(local + 1) * per]
        os.sched_setaffinity(0, mine)
        return len(mine)
    except Exception:
        return None


def make_cpu_env(n, nthreads):
    from oracle.oracle import OracleVecEnv
    from solorl_b200.abi import params_from_config
    from solorl_b200.model import SoloModel
    m = SoloModel.resolve(CONFIG["model_urdf"])
    p = params_from_config(CONFIG, m)
    v = OracleVecEnv(m, p, n, seed=1, nthreads=nthreads)
    v.reset()
    rng = np.random.default_rng(1)
    acts = [rng.uniform(-1, 1, size=(n, v.act_dim)).astype(np.float32) for _ in range(8)]
    return v, acts


def cpu_baseline(seconds=12.0, nthreads=None, n=ENVS_PER_GPU):
    """The oracle port on all host threads, stepping the SAME batch as the GPU arm (all `n` envs per step) for a
    bounded time."""
    nthreads = nthreads or host_threads()
    v, acts = make_cpu_env(n, nthreads)
    for i in range(2):
        v.step(acts[i])
    t0, steps = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds or steps < 3:
        v.step(acts[steps % 8])
        steps += 1
    dt = time.perf_counter() - t0
    return {"value": n * steps / dt, "unit": "env-steps/s", "cores": nthreads, "kind": "port",
            "sample": f"{n} envs x {steps} steps ({dt:.1f} s) of the same workload; fp64 CPU restatement "
                      f"(oracle/), not PyBullet (not installable in this image); " + CPU_RESET_NOTE}


def pybullet_direct_baseline(seconds=30.0):
    """BASELINE.md B0: the reference's own vec-env on PyBullet DIRECT, one worker process per host core, random
    actions as in agents/td3/train.py:98.  Needs pybullet / gym / pybullet_envs and a checkout of the reference
    (SOLORL_REFERENCE, baseline/_ref/soloRL or /root/reference); returns (result, reason)."""
    try:
        import pybullet  # noqa: F401
        import gym  # noqa: F401
    except Exception as e:
        return None, f"pybullet not installed ({type(e).__name__})"
    ref = None
    for cand in (os.environ.get("SOLORL_REFERENCE"), os.path.join(ROOT, "baseline", "_ref", "soloRL"), "/root/reference"):
        if cand and os.path.exists(os.path.join(cand, "baseEnv.py")):
            ref = os.path.abspath(cand)
            break
    if ref is None:
        return None, "no checkout of the reference found (set SOLORL_REFERENCE)"
    try:
        import tempfile
        import torch
        parent, name = os.path.split(ref.rstrip("/"))
        if name != "soloRL":
            parent = tempfile.mkdtemp(prefix="solorl_ref_")
            os.symlink(ref, os.path.join(parent, "soloRL"))
        sys.path.insert(0, parent)
        from soloRL.agents.ppo.envs import make_vec_envs as ref_make_vec_envs
        from soloRL.baseEnv import SoloBaseEnv as RefEnv
        cfg = dict(CONFIG, model_urdf=os.path.join(ref, "solo_description", "robots", "solo12.urdf"), mode="direct")
        n = host_threads()
        envs = ref_make_vec_envs(cfg, n, RefEnv, 0.99, torch.device("cpu"))
        envs.reset()
        A = envs.action_space.shape[0]
        for _ in range(100):
            envs.step(torch.randn(n, A))
        t0, steps = time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds:
            envs.step(torch.randn(n, A))
            steps += 1
        dt = time.perf_counter() - t0
        envs.close()
        return {"value": n * steps / dt, "unit": "env-steps/s", "cores": n, "kind": "reference",
                "sample": f"{n} PyBullet DIRECT worker processes x {steps} steps ({dt:.1f} s), reference code unmodified"}, None
    except Exception as e:
        return None, f"reference vec-env failed: {e!r}"[:300]


def run_reference(args):
    """CPU arm.  Rank 0 alone runs; a step = one vec step of ALL `--envs` envs (the GPU arm's batch), on every
    host thread this process may use (own pthread pool: independent of the OMP_NUM_THREADS=1 torchrun exports)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nthreads = host_threads()
    n = args.envs
    pyb, reason = pybullet_direct_baseline(20.0)
    v, acts = make_cpu_env(n, nthreads)
    for i in range(args.warmup):
        v.step(acts[i % 8])
    t0 = time.perf_counter()
    for i in range(args.steps):
        obs, rew, done = v.step(acts[i % 8])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"obs": obs, "reward": rew, "done": done})
    val = n * args.steps / dt
    sample = (f"{n} envs per step (the GPU arm's batch) on {nthreads} host threads; fp64 CPU restatement (oracle/), "
              f"PyBullet itself is not installable in this image; " + CPU_RESET_NOTE)
    line = {"impl": "reference", "metric": "env-steps/sec", "value": val, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(n, int(os.environ.get("WORLD_SIZE", "1"))),
            "run": {"envs_per_step": n, "reset_mode": "simulate", "host_threads": nthreads},
            "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": nthreads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "pybullet_direct": pyb, "reason": reason}
    if pyb is not None:       # the reference itself ran: it is the arm
        line.update(value=pyb["value"], cpu_baseline=pyb, e2e=dict(line["e2e"], value=pyb["value"]))
    print(json.dumps(line), flush=True)


def time_policy_rollout(cfg, n, dev, rank, world, barrier, T=32, reps=10):
    """env-steps/s of policy rollouts: Policy (agents/ppo/policy.py layout, init_layer orthogonal gain sqrt 2,
    log-std 0), torch.manual_seed(1), stochastic sampling, rollout buffer appends included."""
    import torch
    from solorl_b200.agents.policy import Policy
    from solorl_b200.agents.storage import OPBuffer
    from solorl_b200.agents.train import EpisodeTracker, Rollout
    from solorl_b200.envs import make_vec_envs
    torch.manual_seed(1)
    envs = make_vec_envs(cfg, n, device=dev, seed=2, env_id_offset=rank * n)
    ac = Policy(envs.observation_space.shape, envs.action_space, None, {"hidden_size": 64}).to(dev)
    buf = OPBuffer(T, n, envs.observation_space.shape, envs.action_space.shape[0], dev)
    buf.obs[0].copy_(envs.reset())
    ro = Rollout(envs, ac, buf, EpisodeTracker(dev), T, use_graph=True)
    for _ in range(3):
        ro(); buf.reset()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ro(); buf.reset()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    envs.close()
    return {"value": world * n * T * reps / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms / (T * reps),
            "rollout_steps": T, "cuda_graph": ro.graph is not None,
            "what": "policy act + env step + rollout-buffer append per step, device resident"}


def time_ppo_train(cfg, n, dev, rank, world, barrier, T=32, updates=6):
    """BASELINE.json configs[4]: PPO training throughput, env-steps/s over whole updates = T-step policy rollout
    (one CUDA graph) + GAE kernel + the clipped-surrogate update (ppo_epoch x mini-batches, each one CUDA graph
    with the gradient all-reduce inside) + the 3-scalar advantage all-reduce.  Timed with CUDA events, max over
    ranks.  The share of the collective is measured by repeating the same updates with the gradient all-reduce
    switched off (graphs re-captured): (t_with - t_without) / t_with."""
    import torch
    from solorl_b200.agents.policy import Policy
    from solorl_b200.agents.ppo import PPO, broadcast_parameters
    from solorl_b200.agents.storage import OPBuffer
    from solorl_b200.agents.train import EpisodeTracker, Rollout
    from solorl_b200.envs import make_vec_envs
    torch.manual_seed(1 + rank)
    envs = make_vec_envs(cfg, n, device=dev, seed=2, env_id_offset=rank * n)
    ac = Policy(envs.observation_space.shape, envs.action_space, None, {"hidden_size": 64}).to(dev)
    broadcast_parameters(ac)
    hp = dict(clip_param=0.1, ppo_epoch=5, mini_batch_size=16384, value_loss_coef=0.5, entropy_coef=0.0)
    agent = PPO(ac, hp["clip_param"], hp["ppo_epoch"], hp["mini_batch_size"], hp["value_loss_coef"], hp["entropy_coef"],
                lr=3e-4, max_grad_norm=0.5)
    buf = OPBuffer(T, n, envs.observation_space.shape, envs.action_space.shape[0], dev)
    buf.obs[0].copy_(envs.reset_inplace())
    ro = Rollout(envs, ac, buf, EpisodeTracker(dev), T, use_graph=True)

    def one_update():
        ro()
        with torch.no_grad():
            nv = ac.get_value(buf.obs[-1]).detach()
        buf.compute_returns(nv, True, 0.99, 0.95)
        agent.update(buf)
        buf.reset()

    def timed(k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            one_update()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        return ms / k

    for _ in range(3):                       # eager warm-up steps + graph captures
        one_update()
    ms_with = timed(updates)
    nccl_share = None
    if world > 1:
        agent.sync_enabled = False
        agent._graph, agent._graph_key, agent._warm = None, None, 0
        for _ in range(2):
            one_update()
        ms_without = timed(updates)
        agent.sync_enabled = True
        nccl_share = max(0.0, (ms_with - ms_without) / ms_with)
    envs.close()
    mb_steps = hp["ppo_epoch"] * (n * T // hp["mini_batch_size"])
    return {"value": world * n * T / (ms_with * 1e-3), "unit": "env-steps/s", "ms_per_update": ms_with,
            "rollout_steps": T, "mini_batch_steps_per_update": mb_steps, "hyper": hp,
            "grad_allreduce": {"numel": agent.flat.numel, "bytes": agent.flat.numel * 4, "calls_per_update": mb_steps,
                               "pack_unpack_kernels": 0, "share_of_update_time": nccl_share,
                               "how": "same updates with the collective switched off, (t_with - t_without) / t_with"},
            "what": "rollout (policy act + env step + buffer append, one CUDA graph) + GAE + PPO update incl. NCCL "
                    "gradient and advantage all-reduce; whole updates, CUDA events, max over ranks"}


def time_ppo_stand(cfg, n, dev, max_seconds=30.0, target_return=175.0):
    """north_star: 'PPO Stand reaching the reference's return in under 5 minutes wall-clock'.  One GPU, the trainer of
    training/train_ppo.py (solorl_b200.agents.train.train: rollouts on the CUDA vec-env, GAE kernel, PPO updates) on the
    Stand task from random initialisation, stopped at `target_return` (mean return of the training episodes finished
    since the last log; a standing robot collects ~0.47 per step x 400 steps = 188) or after `max_seconds`.  The
    reference publishes no return figure (BASELINE.md), so the target is stated, not compared."""
    import contextlib
    from solorl_b200.agents.train import default_args, train
    from solorl_b200.envs import SoloBaseEnv
    args = default_args(num_agents=n, num_steps=32, mini_batch_size=4 * n, ppo_epoch=5, lr=3e-4, use_gae=True,
                        entropy_coef=0.0, num_env_steps=int(1e10), log_interval=10, save_interval=10 ** 9,
                        max_seconds=max_seconds, target_return=target_return, seed=2301)
    with contextlib.redirect_stdout(sys.stderr):
        out = train(args, dict(cfg, task="stand"), SoloBaseEnv)
    last = out["last"]
    hit = [h for h in out["history"] if h["episodes"] > 0 and h["episode_return"] >= target_return]
    return {"task": "stand", "envs": n, "target_return": target_return,
            "seconds_to_target": hit[0]["seconds"] if hit else None, "max_seconds": max_seconds,
            "final_return": last.get("episode_return"), "final_episode_length": last.get("episode_length"),
            "env_steps": last.get("steps"), "env_steps_per_s": last.get("fps"), "updates": out["updates"],
            "hyper": {"num_steps": 32, "mini_batch_size": 4 * n, "ppo_epoch": 5, "lr": 3e-4, "use_gae": True,
                      "entropy_coef": 0.0, "seed": 2301},
            "what": "wall-clock from the first rollout (CUDA-graph capture included) to the first log line whose mean "
                    "training-episode return reaches the target"}


def time_saturated(cfg, dev, n, steps=60):
    """Device-resident env-steps/s of the same workload at a batch that fills the GPU (several resident waves
    of the 16-warps-per-SM throughput build), with the work counters of that run."""
    import torch
    from solorl_b200.envs import SoloVecEnv
    env = SoloVecEnv(cfg, n, device=dev, seed=3)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(7)
    acts = [torch.rand(n, env.sim.act_dim, device=dev, generator=g) * 2 - 1 for _ in range(4)]
    ncs, sws = [], []
    for i in range(12):
        env.sim.step(acts[i % 4])
        w = env.sim.get_work_counters().float().mean(0)
        ncs.append(w[0].item()); sws.append(w[1].item())
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        env.sim.step(acts[i % 4])          # state (n x 0.8 KB = 52 MB at 65536 envs) + obs exceed what L2 keeps hot
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    nj = env.sim.nj
    env.close()
    return {"envs": n, "value": n / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms, "step_kernel_build": "throughput",
            "flops_per_env_step": algorithmic_flops_per_env_step(nj, float(np.mean(ncs)), float(np.mean(sws)))}


def time_reset_simulate(cfg, n, dev, steps=40):
    """The headline workload with reset_mode 'simulate' (settle steps run in the step path, what the CPU arms and
    the reference do) instead of the bit-identical reset cache."""
    import torch
    from solorl_b200.envs import SoloVecEnv
    env = SoloVecEnv(dict(cfg, reset_mode="simulate"), n, device=dev, seed=1)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(11)
    acts = [torch.rand(n, env.sim.act_dim, device=dev, generator=g) * 2 - 1 for _ in range(8)]
    for i in range(20):
        env.sim.step(acts[i % 8])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = env.sim.launch_count
    e0.record()
    for i in range(steps):
        env.sim.step(acts[i % 8])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    out = {"value": n / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms,
           "launches_per_step": (env.sim.launch_count - l0) / steps,
           "what": "device-resident, back-to-back steps, settle steps simulated after every auto-reset"}
    env.close()
    return out


def time_body_contacts(cfg, n, dev, steps=60):
    """The headline workload with body_contacts on (knees and base-box corners collide with the ground, SURVEY
    section 8f n4): a collapsed robot rests on its body instead of sinking to the z < 0.05 termination, so fewer
    envs reset per step and the envs that lie on the ground solve 5-11 contact points on the general path."""
    import torch
    from solorl_b200.envs import SoloVecEnv
    env = SoloVecEnv(dict(cfg, body_contacts=1), n, device=dev, seed=1)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(11)
    acts = [torch.rand(n, env.sim.act_dim, device=dev, generator=g) * 2 - 1 for _ in range(8)]
    for i in range(100):                 # past the first collapses: the work mix is the steady one
        env.sim.step(acts[i % 8])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dones, pts = 0.0, []
    e0.record()
    for i in range(steps):
        env.sim.step(acts[i % 8])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    for i in range(8):
        env.sim.step(acts[i % 8])
        dones += float(env.sim.done.sum())
        pts.append(float(env.sim.get_work_counters()[:, 0].float().mean()) / 4.0)
    out = {"value": n / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms,
           "resets_per_env_step": dones / (8 * n), "mean_contact_points_per_substep": float(np.mean(pts)),
           "what": "device-resident, back-to-back steps, body_contacts = 1 (step_kernel<..., BODY>)"}
    env.close()
    return out


def time_gae(dev, peaks, T=400, N=ENVS_PER_GPU, reps=20):
    """HBM view of the rollout-buffer kernel (solo_gae): 20 B per (t, env)."""
    import torch
    from solorl_b200.sim import gae
    g = torch.Generator(device=dev).manual_seed(3)
    r = torch.randn(T, N, device=dev, generator=g)
    v = torch.randn(T + 1, N, device=dev, generator=g)
    m = (torch.rand(T + 1, N, device=dev, generator=g) > 0.02).float()
    ret = torch.zeros(T + 1, N, device=dev)
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    for _ in range(3):
        gae(r, v, m, ret, 0.99, 0.95, True)

    def timed(flush_by_write):
        tot = 0.0
        for i in range(reps):
            # the 33 MB of the rollout would otherwise sit in the 126 MB L2.  A WRITE flush leaves the L2 full of dirty
            # lines whose write-back then competes with the kernel's own traffic; a READ flush leaves clean lines.
            if flush_by_write:
                flush.fill_(float(i))
            else:
                flush.sum()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gae(r, v, m, ret, 0.99, 0.95, True)
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / reps

    ms_w, ms = timed(True), timed(False)
    gbs = 20.0 * T * N / (ms * 1e-3) / 1e9
    peak = peaks.get("hbm_gbs", 6650.0)
    return {"kernel": "gae_chunked_kernel", "T": T, "N": N, "ms": ms, "bound": "hbm", "achieved": gbs, "peak": peak,
            "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes": 20 * T * N,
            "l2": "flushed between launches by READING a 192 MiB buffer (clean lines)",
            "ms_after_write_flush": ms_w}


def measured_traffic(n, variant):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE step_kernel launch from the committed `ncu --set full`
    capture of this workload (profiles/step_kernel_traffic.json names the commit and the command); None when no
    capture matches the batch size and kernel build of this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")) as f:
            recs = json.load(f)["captures"]
        for r in recs:
            if r["envs"] == n and r["build"] == variant:
                return r["dram_bytes_read"] + r["dram_bytes_write"], r["source"]
    except Exception:
        pass
    return None, None


def run_ours(args):
    import torch
    from solorl_b200 import _lib, build
    from solorl_b200.envs import SoloVecEnv
    rank, world, local = dist_setup(args.gpus)
    cores = pin_rank_to_cores(local, world)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    _lib.lib()   # fail loudly if the extension is missing
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n = args.envs
    cfg = dict(CONFIG)
    env = SoloVecEnv(cfg, n, device=dev, seed=args.seed, env_id_offset=rank * n)
    sim = env.sim
    nj, A, D = sim.nj, sim.act_dim, sim.d
    env.reset()
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    nact = 16
    acts = [torch.rand(n, A, device=dev, generator=g) * 2 - 1 for _ in range(nact)]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    ncs, sweeps, resets = [], [], []

    def sample_work(d):
        w = sim.get_work_counters().float().mean(0)
        ncs.append(w[0].item())
        sweeps.append(w[1].item())
        resets.append(d.mean().item())

    for i in range(max(args.warmup, 3)):
        _, _, d, _ = env.step(acts[i % nact])
        sample_work(d)

    # ---- device-resident timing: exactly K steps, L2 flushed between timed steps -------------
    sampler = ClockSampler(local)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.start()
    launches0 = sim.launch_count
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(float(i))
        evs[i][0].record()
        out = sim.step(acts[i % nact])
        evs[i][1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = sim.launch_count - launches0
    clocks = sampler.stop()
    step_ms = np.array([a.elapsed_time(b) for a, b in evs])
    total_ms = float(step_ms.sum())
    if args.dump_outputs and rank == 0:       # the step's buffers are overwritten by the steps below
        dump_outputs(args.dump_outputs, {k: t.cpu().numpy() for k, t in zip(("obs", "reward", "done"), out)})
    for i in range(16):
        _, _, d, _ = env.step(acts[i % nact])
        sample_work(d)
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        total_ms = float(t.item())
    value = world * n * args.steps / (total_ms * 1e-3)

    # ---- back-to-back (no flush) timing of the same K steps, for reference ---------------------
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        sim.step(acts[i % nact])
    e1.record()
    barrier()
    b2b_ms = e0.elapsed_time(e1) / args.steps

    # ---- end to end through the host-buffer C-ABI call -----------------------------------------
    h_act = [torch.empty(n, A, dtype=torch.float32).pin_memory() for _ in range(4)]
    for i, t in enumerate(h_act):
        t.copy_(acts[i].cpu())
    h_obs = torch.empty(n, D, dtype=torch.float32).pin_memory()
    h_rew = torch.empty(n, dtype=torch.float32).pin_memory()
    h_done = torch.empty(n, dtype=torch.float32).pin_memory()
    p_act = [t.data_ptr() for t in h_act]                 # pinned host addresses, reused every step
    p_obs, p_rew, p_done = h_obs.data_ptr(), h_rew.data_ptr(), h_done.data_ptr()
    for i in range(3):
        sim.step_host_ptr(p_act[i % 4], p_obs, p_rew, p_done)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        sim.step_host_ptr(p_act[i % 4], p_obs, p_rew, p_done)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * n * args.steps / e2e_s

    # ---- policy rollout (reference-shaped MLP 64-64 tanh policy, stochastic actions), one CUDA graph of
    #      T x (act -> env step -> buffer append); reported next to the random-action figure -------------
    policy_rollout = None
    if not args.no_policy_rollout:
        try:
            policy_rollout = time_policy_rollout(cfg, n, dev, rank, world, barrier)
        except Exception as e:      # the headline metric does not depend on it
            policy_rollout = {"error": repr(e)[:200]}

    # ---- PPO training with the gradient all-reduce (BASELINE.json configs[4]); the one collective of the system ---
    ppo_train = None
    if not args.no_ppo_train:
        try:
            ppo_train = time_ppo_train(cfg, n, dev, rank, world, barrier)
        except Exception as e:
            ppo_train = {"error": repr(e)[:300]}

    # ---- the same kernel when the batch fills the machine (throughput build, 65536 envs): how far the code is
    #      from the FP32 peak once it is no longer limited by the 4096-env batch of the headline workload ------
    saturated = None
    if not args.no_saturated and world == 1:
        try:
            saturated = time_saturated(cfg, dev, args.saturated_envs)
        except Exception as e:
            saturated = {"error": repr(e)[:200]}

    if rank != 0:
        env.close()
        return

    # ---- roofline of the dominant kernel (step_kernel: one launch per step) ----------------------
    nc_sum, sweep_feet = float(np.mean(ncs)), float(np.mean(sweeps))
    flops = algorithmic_flops_per_env_step(nj, nc_sum, sweep_feet) * n
    kernel_ms = total_ms / args.steps if world == 1 else float(step_ms.mean())
    fma_tflops = C.c_double()
    fma_ms = C.c_double()
    bl = C.CDLL(build.BENCH_LIB)
    bl.solo_bench_fma_peak.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    rc = bl.solo_bench_fma_peak(local, C.byref(fma_tflops), C.byref(fma_ms))
    peak = fma_tflops.value if rc == 0 else 74.5
    achieved = flops / (kernel_ms * 1e-3) / 1e12
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    abytes = algorithmic_bytes_per_env_step(nj, D) * n
    variant = sim.step_variant
    traffic, traffic_src = measured_traffic(n, variant)
    roofline = {
        "bound": "fp32", "kernel": "step kernel, build '%s'" % variant, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
        "frac": achieved / peak,
        "traffic": traffic, "traffic_source": traffic_src,
        "traffic_unit": "bytes per launch (algorithmic: %d)" % (algorithmic_bytes_per_env_step(nj, D) * n),
        "peak_source": "FP32 FMA microbenchmark measured live in this run (solo_bench_fma_peak)" if rc == 0
        else "fallback 148 SM x 128 lanes x 2 x 1.965 GHz",
        "algorithmic_flops_per_env_step": algorithmic_flops_per_env_step(nj, nc_sum, sweep_feet),
        "mean_contacts_per_substep": nc_sum / 4.0,
        "mean_pgs_sweeps_per_contact_substep": (sweep_feet / nc_sum) if nc_sum > 0 else 0.0,
        "resets_per_env_step": float(np.mean(resets)), "kernel_ms": kernel_ms,
        "hbm": {"bound": "hbm", "achieved": abytes / (kernel_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": abytes / (kernel_ms * 1e-3) / 1e9 / hbm_peak,
                "algorithmic_bytes_per_env_step": algorithmic_bytes_per_env_step(nj, D),
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s"},
    }
    line = {
        "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(n, world),
        "run": {"reset_mode": "cached", "step_kernel_build": variant, "host_cores_of_this_rank": cores},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": n * A * 4,
                "d2h_bytes_per_step": n * (D + 2) * 4, "ms_per_step": e2e_s / args.steps * 1e3,
                "api": "solo_step_host (pinned host buffers read and written by the step kernel through their mapped alias, one sync per step)"},
        "roofline": roofline,
        "back_to_back_ms_per_step": b2b_ms, "wall_ms_per_step_incl_flush": t_wall / args.steps * 1e3,
        "policy_rollout": policy_rollout,
        "ppo_train": ppo_train,
        "saturated": saturated,
    }
    if saturated and "flops_per_env_step" in saturated:
        ach = saturated["flops_per_env_step"] * saturated["value"] / 1e12
        saturated.update({"achieved_tflops": ach, "peak_tflops": peak, "frac": ach / peak})
    if world == 1:
        try:
            line["reset_mode_simulate"] = time_reset_simulate(cfg, n, dev)
        except Exception as e:
            line["reset_mode_simulate"] = {"error": repr(e)[:200]}
        if not args.no_ppo_train:
            try:
                line["ppo_stand"] = time_ppo_stand(cfg, n, dev)
            except Exception as e:
                line["ppo_stand"] = {"error": repr(e)[:300]}
        try:
            line["body_contacts"] = time_body_contacts(cfg, n, dev)
        except Exception as e:
            line["body_contacts"] = {"error": repr(e)[:200]}
        try:
            line["gae"] = time_gae(dev, peaks)
        except Exception as e:
            line["gae"] = {"error": repr(e)[:200]}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args.cpu_seconds, n=n)
        line["pybullet_direct"], line["reason"] = pybullet_direct_baseline(20.0)   # SURVEY §8(d)(i) / BASELINE.md B0
    print(json.dumps(line), flush=True)
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU (BASELINE: 4096)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-policy-rollout", action="store_true")
    ap.add_argument("--no-ppo-train", action="store_true")
    ap.add_argument("--no-saturated", action="store_true")
    ap.add_argument("--saturated-envs", type=int, default=65536)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write obs/reward/done of the last timed step as DIR/<name>.npy (float32, at most 64 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    # (the CPU arm never imports torch: ranks > 0 of a torchrun launch exit at once and leave the host cores to rank 0)
    if args.impl != "reference" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        try:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


if __name__ == "__main__":
    main()
