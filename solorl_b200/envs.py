"""GPU-resident vec-env with the reference's ``--num-agents`` interface.

Drop-in for ``agents/ppo/envs.py`` (and the td3/sac copies): ``make_vec_envs`` returns
an object with the methods the trainers use — ``reset()``, ``step(actions)``,
``observation_space``, ``action_space``, ``close()``, ``get_observation()``,
``increment_curriculum()`` and the attribute chain ``envs.envs.ob_rms`` /
``envs.envs.venv`` (reference ``agents/ppo/train.py:32-45,88,126``,
``testing/test_ppo.py:88-109``) — but N environments are ONE CUDA handle instead of N
OS processes exchanging pickles over pipes (``agents/ppo/envs.py:66-95``), and every
tensor stays on the device: no ``.cpu().numpy()`` / ``torch.from_numpy().to(device)``
hop per step (``agents/ppo/envs.py:189-196``).
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from .abi import CONTROL_VPD, params_from_config
from .model import SoloModel
from .sim import SoloSim

_DR_KEYS = (("dr/stand_rew", "dr_stand"), ("dr/joint_pose_rew", "dr_joint_pose"),
            ("dr/torque_rew", "dr_torque"), ("dr/roll_pitch_balance_rew", "dr_balance"),
            ("dr/progress_rew", "dr_progress"))


class Box:
    """Minimal stand-in for ``gym.spaces.Box`` (gym is not a dependency): the trainers only
    read ``.shape`` and ``.__class__.__name__`` (agents/ppo/train.py:34-45)."""

    def __init__(self, low, high):
        self.low = np.asarray(low, dtype=np.float32)
        self.high = np.asarray(high, dtype=np.float32)
        self.shape = self.low.shape
        self.dtype = np.float32

    def sample(self):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return np.random.uniform(lo, hi).astype(np.float32)

    def __repr__(self):
        return f"Box{self.shape}"


class LazyInfos:
    """The ``infos`` tuple of ``VecEnvWrapper.step`` (agents/ppo/envs.py:94-95) without building
    N dicts per step: the episode records live on the device and are copied to the host only
    when somebody looks.  ``infos[i]`` is the info dict of baseEnv.py:63-66 for envs whose
    episode ended at this step and ``{}`` otherwise (nobody reads non-terminal infos:
    agents/ppo/train.py:90-100, agents/td3/train.py:108-115)."""

    def __init__(self, sim: SoloSim, done: torch.Tensor, snapshot: bool = True):
        """snapshot=True (the public step()): the done flags and the episode records are copied on the
        device NOW (two small device-to-device copies, no host sync), so that an infos object inspected
        after later steps still describes ITS step; snapshot=False reads the live buffers lazily (the
        in-repo rollout, which never looks at infos)."""
        self._sim = sim
        self._rec = None
        self._done_np = None
        if snapshot:
            self._done = done.detach().clone()
            self._stats = sim.episode_stats_snapshot()
        else:
            self._done, self._stats = done, None

    def _fetch(self):
        if self._done_np is None:
            self._done_np = self._done.detach().cpu().numpy() > 0.5
            if self._done_np.any():
                self._rec = (self._sim.episode_stats() if self._stats is None
                             else self._stats.cpu().numpy().view(self._sim.stats_dtype))
        return self._rec

    @staticmethod
    def _to_dict(r):
        d = {"timeout": bool(r["timeout"]), "success": bool(r["success"])}
        for k, f in _DR_KEYS:
            d[k] = float(r[f])
        d["episode_length"] = int(r["episode_length"])
        d["episode_reward"] = float(r["episode_reward"])    # last-step reward (SURVEY F8)
        d["episode_return"] = float(r["episode_return"])    # sum of rewards (extension)
        d["goals_reached"] = int(r["goals_reached"])
        d["nan"] = bool(r["nan"])                           # ended by the non-finite-state guard
        # keys the PPO loop reads but only BaseControlEnv provides (SURVEY F9c)
        d["max_velocity"] = 0.0
        d["min_force"] = 0.0
        d["max_force"] = 0.0
        return d

    def done_indices(self):
        self._fetch()
        return np.nonzero(self._done_np)[0]

    def done_records(self):
        """Structured array of the finished episodes' records (may be empty)."""
        rec = self._fetch()
        idx = np.nonzero(self._done_np)[0]
        return rec[idx] if rec is not None else np.zeros(0, dtype=self._sim.episode_stats().dtype)

    def __len__(self):
        return self._sim.n

    def __getitem__(self, i):
        rec = self._fetch()
        if rec is None or not self._done_np[i]:
            return {}
        return self._to_dict(rec[i])

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]


class SoloVecEnv:
    """N SoloBaseEnv instances (baseEnv.py:6-187) stepped by one kernel launch; auto-reset on
    done exactly as the reference's worker does (agents/ppo/envs.py:38-40)."""

    def __init__(self, config: dict, num_envs: int, device=None, seed: int = 0, env_id_offset: int = 0):
        self.config = dict(config)
        self.model = SoloModel.resolve(config["model_urdf"])        # baseEnv.py:8 (required key)
        _ = config["mode"]                                          # baseEnv.py:16 (required key; GUI unsupported)
        self.params = params_from_config(config, self.model)
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else "cuda:0"
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("SoloVecEnv runs on a CUDA device only (no CPU fallback)")
        self.device = device
        self.sim = SoloSim(self.model, self.params, num_envs, device=device.index or 0, seed=seed,
                           env_id_offset=env_id_offset)
        self.nenvs = num_envs
        nj = self.model.nj
        adim = nj + (2 if self.params.control == CONTROL_VPD else 0)      # baseEnv.py:20-24
        self.action_space = Box(-np.ones(adim), np.ones(adim))
        self.observation_space = Box(-np.inf * np.ones(self.sim.d), np.inf * np.ones(self.sim.d))  # :26-27
        self.goal_radius = float(self.params.goal_radius)
        self.closed = False

    def reset(self):
        """The handle's persistent observation buffer (overwritten by the next reset/step): the zero-copy call
        of the in-repo trainers.  ``PyTorchEnvWrapper`` hands out copies."""
        return self.sim.reset()

    def step(self, actions, snapshot: bool = False):
        """Returns the handle's persistent obs / reward / done buffers (overwritten by the next step) and a
        lazy infos object; ``snapshot=True`` freezes the infos of this step (see LazyInfos)."""
        obs, rew, done = self.sim.step(actions)
        return obs, rew, done, LazyInfos(self.sim, done, snapshot=snapshot)

    def get_observation(self):
        return self.sim.get_observation()

    def get_env_params(self):
        """[N,3] (friction, base_mass_scale, motor_strength) of each env's current episode: privileged inputs
        for an asymmetric critic, or logging (see the ``randomize_*`` config keys)."""
        return self.sim.env_params()

    def get_push_force(self):
        """[N,3] push (fx, fy, 0) in N, base axes, that the next step applies to each env: privileged inputs for
        an asymmetric critic, or logging (see the ``push_*`` config keys)."""
        return self.sim.push_force()

    def get_torques(self):
        raise NotImplementedError("get_torques is a gait-env call (env.robot.tau_ff)")  # envs.py:45-46

    def increment_curriculum(self, value: float = 1.0):
        """Pointgoal curriculum: increment_goal_radius (solo.py:332-334)."""
        self.goal_radius += value
        self.sim.set_goal_radius(self.goal_radius)

    def close(self):
        if not self.closed:
            self.sim.close()
            self.closed = True

    def __len__(self):
        return self.nenvs


class VecNormalize:
    """``agents/running_mean_std.py:73-127`` as instantiated by ``make_vec_envs``
    (``ob=False, ret=False``): a pass-through that only tracks the discounted return, kept on
    the device.  Preserves the attribute surface the callers touch: ``ob_rms``, ``ret_rms``,
    ``eval()``, ``venv`` and attribute forwarding to the wrapped env."""

    def __init__(self, venv, ob=False, ret=False, clipob=10., cliprew=10., gamma=0.99, epsilon=1e-8):
        if ob or ret:
            raise NotImplementedError("the reference only instantiates VecNormalize(ob=False, ret=False)")
        self.venv = venv
        self.nenvs = venv.nenvs
        self.ob_rms = None
        self.ret_rms = None
        self.clipob, self.cliprew, self.gamma, self.epsilon = clipob, cliprew, gamma, epsilon
        self.ret = torch.zeros(self.nenvs, dtype=torch.float32, device=venv.device)
        self.training = True

    def step(self, actions, **kw):
        obs, rews, news, infos = self.venv.step(actions, **kw)
        # in place, so that a CUDA graph captured around step() keeps updating the same tensor
        self.ret.mul_(self.gamma).add_(rews)               # running_mean_std.py:98
        self.ret.mul_((news <= 0.5).to(self.ret.dtype))    # :105
        return obs, rews, news, infos

    def reset(self):
        self.ret.zero_()
        return self.venv.reset()

    def eval(self):
        self.training = False

    def close(self):
        return self.venv.close()

    def __len__(self):
        return self.nenvs

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(f"attempted to get missing private attribute '{name}'")
        return getattr(self.venv, name)


class PyTorchEnvWrapper:
    """``agents/ppo/envs.py:183-222``: same return shapes (obs [N,D] f32, reward [N,1] f32,
    done [N] f32, infos sequence), tensors already on the device.

    ``step`` / ``reset`` return FRESH tensors, like the reference's ``torch.from_numpy(...).to(device)``
    (envs.py:192-196): a caller may keep ``obs`` next to ``next_obs`` (the TD3/SAC pattern
    ``buffer.append(obs, a, r, next_obs, 1 - done); obs = next_obs``) and inspect ``infos`` later.  The
    copies are three small device-to-device launches; ``step_inplace`` / ``reset_inplace`` are the
    zero-copy calls the in-repo trainers use (they copy into their own buffers right away) and return
    the handle's persistent buffers, which the next call overwrites."""

    def __init__(self, envs, device):
        self.envs = envs
        self.nenvs = len(envs)
        self.device = device

    def step(self, actions):
        ob, rw, done, info = self.envs.step(actions, snapshot=True)
        return ob.clone(), rw.unsqueeze(-1).clone(), done.clone(), info

    def step_inplace(self, actions):
        ob, rw, done, info = self.envs.step(actions)
        return ob, rw.unsqueeze(-1), done, info

    def reset(self):
        return self.envs.reset().clone()

    def reset_inplace(self):
        return self.envs.reset()

    def close(self):
        self.envs.close()

    def get_observation(self):
        return self.envs.get_observation()

    def get_env_params(self):
        return self.envs.get_env_params()

    def get_push_force(self):
        return self.envs.get_push_force()

    def get_torques(self):
        return self.envs.get_torques()

    def increment_curriculum(self):
        self.envs.increment_curriculum()

    @property
    def observation_space(self):
        return self.envs.observation_space

    @property
    def action_space(self):
        return self.envs.action_space

    def __len__(self):
        return self.nenvs


class SoloBaseEnv:
    """Single-env façade with the gym-0.x contract of ``baseEnv.py`` (``reset() -> obs``,
    ``step(a) -> (obs-or-None, reward, done, info)``); also the class object passed as
    ``env_constructor`` for ``--env-name base`` (training/train_ppo.py:76-78)."""

    def __init__(self, config, device=None, seed: int = 0):
        self._vec = SoloVecEnv(config, 1, device=device, seed=seed)
        self.config = config
        self.action_space = self._vec.action_space
        self.observation_space = self._vec.observation_space
        self._pending = None

    def reset(self):
        # after a finished episode the batched step has already reset the env (masked auto-reset in the kernel,
        # the worker's behaviour of agents/ppo/envs.py:38-40): hand that observation out instead of resetting twice
        if self._pending is not None:
            obs, self._pending = self._pending, None
            return obs
        return self._vec.reset()[0].cpu().numpy().astype(np.float64)

    def step(self, action):
        a = torch.as_tensor(np.asarray(action, dtype=np.float32)[None], device=self._vec.device)
        obs, rew, done, infos = self._vec.step(a)
        d = bool(done[0].item() > 0.5)
        info = infos[0]
        o = obs[0].cpu().numpy().astype(np.float64)
        if d:                     # baseEnv.py:54: the terminal step returns obs = None; reset() gives the next one
            self._pending = o
            return None, float(rew[0].item()), d, info
        self._pending = None
        return o, float(rew[0].item()), d, info

    def get_observation(self):
        return self._vec.get_observation()[0].cpu().numpy().astype(np.float64)

    def close(self):
        self._vec.close()


def make_vec_envs(config, num_envs, env_constructor=SoloBaseEnv, gamma=0.99,
                  device: Optional[torch.device] = None, training=True, seed: int = 0,
                  env_id_offset: int = 0):
    """``agents/ppo/envs.py:14-30`` with the same signature.  ``env_constructor`` is
    :class:`SoloBaseEnv` or :class:`solorl_b200.gait.SoloGaitEnvContact` (the env shell with a pluggable
    controller; the other reference env classes cannot be constructed from any shipped config)."""
    name = getattr(env_constructor, "__name__", "")
    if name not in ("SoloBaseEnv", "SoloGaitEnvContact"):
        raise NotImplementedError(f"env_constructor {env_constructor!r}: SoloBaseEnv and SoloGaitEnvContact are built")
    if device is None or torch.device(device).type != "cuda":
        device = torch.device("cuda", torch.cuda.current_device())
    if name == "SoloGaitEnvContact":
        from .gait import SoloGaitVecEnv
        envs = SoloGaitVecEnv(config, num_envs, device=device, seed=seed, env_id_offset=env_id_offset)
    else:
        envs = SoloVecEnv(config, num_envs, device=device, seed=seed, env_id_offset=env_id_offset)
    envs = VecNormalize(envs, ob=False, ret=False, clipob=100, cliprew=100, gamma=gamma)
    if not training:
        envs.eval()
    return PyTorchEnvWrapper(envs, torch.device(device))
