"""``SoloSim``: torch-tensor view of one ``SoloHandle`` (one per GPU per process).

PyTorch is plumbing here (device memory + the current CUDA stream); every call goes
through the C-ABI of ``include/solo_b200.h`` with raw device pointers.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .abi import (EPISODE_STATS_DTYPE, SoloSimParams, dims, model_table)
from .model import SoloModel


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class SoloSim:
    def __init__(self, model: SoloModel, params: SoloSimParams, num_envs: int, device=0,
                 seed: int = 0, env_id_offset: int = 0):
        self.L = _lib.lib()   # raises if the CUDA extension was not built
        if not torch.cuda.is_available():
            raise RuntimeError("solorl_b200 needs a CUDA device (there is no CPU fallback)")
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.model, self.params, self.n = model, params, int(num_envs)
        self.nj, self.act_dim, self.d0, self.d = dims(model, params)
        self._table = model_table(model)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.L.solo_create(C.byref(self._table), C.byref(params), self.n, self.device.index,
                                          int(seed) & (2 ** 64 - 1), int(env_id_offset), C.byref(h)))
        self.h = h
        f32 = dict(dtype=torch.float32, device=self.device)
        self.obs = torch.zeros(self.n, self.d, **f32)
        self.reward = torch.zeros(self.n, **f32)
        self.done = torch.zeros(self.n, **f32)
        self._stats = torch.zeros(self.n * EPISODE_STATS_DTYPE.itemsize, dtype=torch.uint8, device=self.device)

    def close(self):
        if getattr(self, "h", None):
            self.L.solo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _f32(self, t, shape):
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device).contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    # ---- env step path ------------------------------------------------------------
    def reset(self, mask=None):
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        _lib.check(self.L.solo_reset(self.h, _ptr(m), _ptr(self.obs), self._stream()), self.h)
        return self.obs

    def step(self, actions):
        a = self._f32(actions, (self.n, self.act_dim))
        _lib.check(self.L.solo_step(self.h, _ptr(a), _ptr(self.obs), _ptr(self.reward), _ptr(self.done),
                                    self._stream()), self.h)
        return self.obs, self.reward, self.done

    def step_host(self, actions_np, obs_np, reward_np, done_np):
        """Host-buffer call (numpy / pinned-tensor memory): H2D, step, D2H, sync."""
        _lib.check(self.L.solo_step_host(self.h, C.c_void_p(actions_np.ctypes.data), C.c_void_p(obs_np.ctypes.data),
                                         C.c_void_p(reward_np.ctypes.data), C.c_void_p(done_np.ctypes.data),
                                         self._stream()), self.h)

    def step_host_ptr(self, actions_ptr, obs_ptr, reward_ptr, done_ptr):
        """The same call with raw host addresses (ints), for callers that reuse their buffers: building four
        ctypes pointers from numpy arrays costs more than the C call itself."""
        _lib.check(self.L.solo_step_host(self.h, actions_ptr, obs_ptr, reward_ptr, done_ptr, self._stream()), self.h)

    def get_observation(self):
        out = torch.empty(self.n, self.d, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_get_observation(self.h, _ptr(out), self._stream()), self.h)
        return out

    def episode_stats(self):
        """numpy structured array (one record per env; valid where done == 1). Syncs."""
        _lib.check(self.L.solo_episode_stats(self.h, _ptr(self._stats), self._stream()), self.h)
        return self._stats.cpu().numpy().view(EPISODE_STATS_DTYPE)

    stats_dtype = EPISODE_STATS_DTYPE

    def episode_stats_snapshot(self):
        """A private device copy of the current episode records (uint8 bytes of SoloEpisodeStats[N]); no sync."""
        out = torch.empty_like(self._stats)
        _lib.check(self.L.solo_episode_stats(self.h, _ptr(out), self._stream()), self.h)
        return out

    def episode_stats_device(self):
        """The same records without leaving the device: (float32 view [N,12], int32 view [N,12]) of
        ``SoloEpisodeStats[N]``; columns 0,1,6..10 are floats (episode_reward, episode_return, dr/*),
        columns 2..5 and 11 ints (episode_length, success, timeout, goals_reached, nan).  No sync."""
        _lib.check(self.L.solo_episode_stats(self.h, _ptr(self._stats), self._stream()), self.h)
        w = EPISODE_STATS_DTYPE.itemsize // 4
        return self._stats.view(torch.float32).view(self.n, w), self._stats.view(torch.int32).view(self.n, w)

    def accumulate_episode_stats(self, done, acc):
        """Fold the records of envs with done == 1 into ``acc`` (float64 [13] on the device, see
        solo_accumulate_episode_stats); one small launch, no sync."""
        if not (acc.is_cuda and acc.dtype == torch.float64 and acc.numel() == 13 and acc.is_contiguous()):
            raise ValueError("acc must be a contiguous float64 CUDA tensor of 13 elements")
        d = self._f32(done, (self.n,))
        _lib.check(self.L.solo_accumulate_episode_stats(self.h, _ptr(d), _ptr(acc), self._stream()), self.h)

    def env_params(self):
        """float32 [N,3] on the device: the (friction, base_mass_scale, motor_strength) each env runs its episode
        with (drawn at its last reset on a randomised handle, nominal otherwise).  No sync."""
        out = torch.empty(self.n, 3, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_get_env_params(self.h, _ptr(out), self._stream()), self.h)
        return out

    def push_force(self):
        """float32 [N,3] on the device: the push (fx, fy, 0) in N, base axes, that the next step applies to each
        env (zero outside a push window and without pushes).  No sync."""
        out = torch.empty(self.n, 3, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_get_push_force(self.h, _ptr(out), self._stream()), self.h)
        return out

    def set_goal_radius(self, r):
        _lib.check(self.L.solo_set_goal_radius(self.h, float(r)), self.h)

    # ---- parity hooks ---------------------------------------------------------------
    def get_state(self):
        out = torch.empty(self.n, 13 + 2 * self.nj, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_get_state(self.h, _ptr(out), self._stream()), self.h)
        return out

    def set_state(self, state):
        s = self._f32(state, (self.n, 13 + 2 * self.nj))
        _lib.check(self.L.solo_set_state(self.h, _ptr(s), self._stream()), self.h)

    def set_goals(self, goals):
        g = self._f32(goals, (self.n, 2))
        _lib.check(self.L.solo_set_goals(self.h, _ptr(g), self._stream()), self.h)

    def set_contacts(self, force):
        """Inject the per-foot contact record (normal force [N,4], negative = no contact point)."""
        f = self._f32(force, (self.n, 4))
        _lib.check(self.L.solo_set_contacts(self.h, _ptr(f), self._stream()), self.h)

    def get_contacts(self):
        out = torch.empty(self.n, 4, 3, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_get_contacts(self.h, _ptr(out), self._stream()), self.h)
        return out

    def get_work_counters(self):
        """int32 [N,2]: (feet-in-contact, feet-in-contact x PGS sweeps) summed over the substeps of the last step."""
        out = torch.empty(self.n, 2, dtype=torch.int32, device=self.device)
        _lib.check(self.L.solo_get_work_counters(self.h, _ptr(out), self._stream()), self.h)
        return out

    def forward_dynamics(self, state, tau):
        s = self._f32(state, (self.n, 13 + 2 * self.nj))
        t = self._f32(tau, (self.n, self.nj))
        out = torch.empty(self.n, 6 + self.nj, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_forward_dynamics(self.h, _ptr(s), _ptr(t), _ptr(out), self._stream()), self.h)
        return out

    def substep(self, tau):
        t = self._f32(tau, (self.n, self.nj))
        _lib.check(self.L.solo_substep(self.h, _ptr(t), self._stream()), self.h)

    def action_to_torque(self, actions):
        a = self._f32(actions, (self.n, self.act_dim))
        out = torch.empty(self.n, self.nj, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_action_to_torque(self.h, _ptr(a), _ptr(out), self._stream()), self.h)
        return out

    # ---- gait-env actuator interface (SURVEY §8f n2) ------------------------------------
    def actuator_step(self, cmd, n_ticks=1):
        """cmd [N,5,nj] = q_des, v_des, P, D, tau_ff; n_ticks simulator ticks at params.dt."""
        c = self._f32(cmd, (self.n, 5, self.nj))
        _lib.check(self.L.solo_actuator_step(self.h, _ptr(c), int(n_ticks), self._stream()), self.h)

    def set_external_force(self, force):
        """Base-frame force [N,3] at the base origin for the following actuator_step calls (gait-env pushes)."""
        f = self._f32(force, (self.n, 3))
        _lib.check(self.L.solo_set_external_force(self.h, _ptr(f), self._stream()), self.h)

    def get_feet(self):
        out = torch.empty(self.n, 4, 3, dtype=torch.float32, device=self.device)
        _lib.check(self.L.solo_get_feet(self.h, _ptr(out), self._stream()), self.h)
        return out

    @property
    def step_variant(self):
        return self.L.solo_step_variant(self.h).decode()

    @property
    def launch_count(self):
        return int(self.L.solo_launch_count(self.h))


def gae(rewards, values, masks, returns, gamma, lam, use_gae=True):
    """Device-resident reverse-scan GAE (replaces OPBuffer.compute_returns,
    agents/ppo/storage.py:35-55).  rewards [T,N(,1)], values/masks/returns [T+1,N(,1)];
    writes returns[:T] in place."""
    L = _lib.lib()
    T = rewards.shape[0]
    N = rewards[0].numel()
    for t in (rewards, values, masks, returns):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise ValueError("solo_gae needs contiguous float32 CUDA tensors")
    if values.shape[0] != T + 1 or masks.shape[0] != T + 1 or returns.shape[0] != T + 1:
        raise ValueError("values/masks/returns must have T+1 rows")
    stream = C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream)
    _lib.check(L.solo_gae(_ptr(rewards), _ptr(values), _ptr(masks), _ptr(returns), T, N,
                          float(gamma), float(lam), int(bool(use_gae)), stream))
    return returns
