"""Random pushes on the GPU (SoloSimParams.push_*): the device's schedule against the host build of the sampler,
its independence of sharding and of the reset mode, the pushed physics against the fp64 oracle given the same
force, agreement of a zero force with the build without pushes, the effect on a trained policy, and the calls a
push does not reach."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle.oracle import OracleEnv
from solorl_b200 import abi
from solorl_b200.model import SoloModel
from tests.emu import push_sampler
from tests.helpers import flag_slots, make_config, obs_diff, random_states

pytestmark = pytest.mark.gpu

ROBOTS = ("solo8", "solo12")
RANGES = {"randomize_friction": [0.5, 1.25], "randomize_base_mass": [0.8, 1.2],
          "randomize_motor_strength": [0.8, 1.2]}
PUSH = {"push_force": 15.0, "push_interval": 6, "push_duration": 2}
EVERY_STEP = {"push_interval": 1, "push_duration": 1}


def cuda(x):
    return torch.as_tensor(np.asarray(x, dtype=np.float32)).cuda()


def make_sim(robot, n, seed=0, env_id_offset=0, **kw):
    from solorl_b200.sim import SoloSim
    cfg = make_config(robot, **kw)
    m = SoloModel.resolve(robot)
    p = abi.params_from_config(cfg, m)
    return SoloSim(m, p, n, device=0, seed=seed, env_id_offset=env_id_offset), m, p


def host_push(p, seed, episode, t, gid0=0):
    """[n,3] the host sampler's push for envs gid0.. at their (episode, t)."""
    return np.stack([push_sampler.push_sample(p, seed, gid0 + i, 1, int(episode[i]), int(t[i]), 1)[0, 0]
                     for i in range(len(episode))])


# ---- the schedule ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("reset_mode", ["cached", "simulate"])
def test_device_pushes_equal_the_host_sampler(reset_mode):
    """Before every step of a rollout with auto-resets and one masked reset, the getter returns the host sampler's
    push for each env's (episode, steps completed in it)."""
    n, seed = 128, 9
    sim, m, p = make_sim("solo12", n, seed=seed, task="walk", episode_length=15, reset_mode=reset_mode, **PUSH)
    assert sim.step_variant == "latency+push"
    sim.reset()
    episode, t = np.ones(n, np.int64), np.zeros(n, np.int64)
    g = torch.Generator(device="cuda").manual_seed(3)
    pushed, ndone = 0, 0
    for k in range(40):
        if k == 11:
            mask = np.zeros(n, dtype=bool)
            mask[::5] = True
            sim.reset(mask=torch.as_tensor(mask, device="cuda"))
            episode[mask] += 1
            t[mask] = 0
        got = sim.push_force().cpu().numpy()
        np.testing.assert_array_equal(got, host_push(p, seed, episode, t), err_msg=f"step {k}")
        pushed += int(np.any(got != 0, axis=1).sum())
        _, _, d = sim.step(torch.rand(n, sim.act_dim, device="cuda", generator=g) * 2 - 1)
        done = d.cpu().numpy() > 0.5
        t += 1
        episode[done] += 1
        t[done] = 0
        ndone += int(done.sum())
    assert ndone >= n and pushed > 0.2 * 40 * n
    sim.close()


def test_one_handle_equals_two_shards():
    """Pushes and randomised dynamics together depend on the global env id, not on the sharding."""
    n = 64
    kw = dict(task="walk", episode_length=20, **RANGES, **PUSH)
    whole, _, _ = make_sim("solo12", 2 * n, seed=3, **kw)
    parts = [make_sim("solo12", n, seed=3, env_id_offset=k * n, **kw)[0] for k in range(2)]
    assert whole.step_variant == "latency+rand+push"
    whole.reset()
    for s in parts:
        s.reset()
    g = torch.Generator(device="cuda").manual_seed(2)
    for t in range(30):
        assert torch.equal(whole.push_force(), torch.cat([s.push_force() for s in parts]))
        a = torch.rand(2 * n, whole.act_dim, device="cuda", generator=g) * 2 - 1
        o, r, d = whole.step(a)
        for k, s in enumerate(parts):
            ok, rk, dk = s.step(a[k * n:(k + 1) * n])
            assert torch.equal(o[k * n:(k + 1) * n], ok) and torch.equal(r[k * n:(k + 1) * n], rk)
            assert torch.equal(d[k * n:(k + 1) * n], dk)
    assert torch.equal(whole.get_state(), torch.cat([s.get_state() for s in parts]))
    assert torch.equal(whole.env_params(), torch.cat([s.env_params() for s in parts]))
    for s in [whole] + parts:
        s.close()


def test_cached_reset_equals_simulated_reset_bitwise_under_pushes():
    from solorl_b200.envs import SoloVecEnv
    for robot, task in (("solo12", "pointgoal"), ("solo8", "walk")):
        cfg = make_config(robot, task=task, H=1, episode_length=15, **RANGES, **PUSH)
        e1 = SoloVecEnv(cfg, 96, device="cuda:0", seed=5)
        e2 = SoloVecEnv(dict(cfg, reset_mode="simulate"), 96, device="cuda:0", seed=5)
        assert torch.equal(e1.reset(), e2.reset())
        g = torch.Generator(device="cuda").manual_seed(1)
        ndone = 0
        for t in range(40):
            assert torch.equal(e1.get_push_force(), e2.get_push_force())
            a = torch.rand(96, e1.sim.act_dim, device="cuda", generator=g) * 2 - 1
            o1, r1, d1, _ = e1.step(a)
            o2, r2, d2, _ = e2.step(a)
            assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2)
            ndone += int(d1.sum().item())
        assert ndone >= 96 * 2
        assert torch.equal(e1.sim.get_state(), e2.sim.get_state())
        assert torch.equal(e1.get_env_params(), e2.get_env_params())
        e1.close()
        e2.close()


# ---- the pushed physics against the fp64 oracle ---------------------------------------------------------------
@pytest.mark.parametrize("build", ("latency", "throughput"))
@pytest.mark.parametrize("robot", ROBOTS)
def test_contact_free_step_with_push_matches_oracle_1e4(robot, build, monkeypatch):
    """One control step (frame_skip substeps) of airborne envs pushed in every step by up to 50 N per axis: the
    GPU state against the oracle given the same state and the getter's force, 1e-4 relative; and the push moves
    every env by more than 100x that bound against the same step without pushes."""
    monkeypatch.setenv("SOLO_STEP_VARIANT", build)
    rng = np.random.default_rng(171)
    n, tol = 64, 1e-4
    sim, m, p = make_sim(robot, n, task="walk", episode_length=1000, push_force=50.0, **EVERY_STEP)
    ref_sim, _, _ = make_sim(robot, n, task="walk", episode_length=1000)
    assert sim.step_variant == build + "+push"
    nj = sim.nj
    s0 = random_states(rng, n, nj)
    s0[:, 2] += 1.0
    s0[:, 13:13 + nj] = np.clip(s0[:, 13:13 + nj], -9.0, 9.0)
    a = rng.uniform(-1, 1, size=(n, sim.act_dim)).astype(np.float32)
    states, forces = [], []
    for s in (sim, ref_sim):
        s.reset()
        s.set_state(cuda(s0))
        forces.append(s.push_force().cpu().numpy())
        s.step(torch.from_numpy(a).cuda())
        states.append(s.get_state().cpu().numpy().astype(np.float64))
    f = forces[0]
    assert np.all(np.any(f[:, :2] != 0, axis=1)) and np.all(f[:, 2] == 0) and np.all(forces[1] == 0)
    got, unpushed = states
    worst, moved = 0.0, np.inf
    for i in range(n):
        o = OracleEnv(m, p)
        o.reset()
        o.set_state(s0[i])
        o.set_external_force(f[i].astype(np.float64))
        o.step(a[i].astype(np.float64))
        ref = o.get_state()
        scale = np.maximum(1.0, np.abs(ref))
        worst = max(worst, float((np.abs(ref - got[i]) / scale).max()))
        moved = min(moved, float((np.abs(unpushed[i] - got[i]) / scale).max()))
    assert worst < tol, worst
    assert moved > 100 * tol, moved
    sim.close()
    ref_sim.close()


def test_stance_steps_with_push_match_oracle_5e3():
    """Reset and two control steps with contact, every step pushed by up to 20 N per axis: the shape and bound of
    test_gpu_parity._one_step_vs_oracle, the oracle given the getter's force before each step."""
    from solorl_b200.envs import SoloVecEnv
    n, seed, nref = 32, 31, 8
    cfg = make_config("solo12", task="walk", control="torque", H=1, episode_length=50, push_force=20.0, **EVERY_STEP)
    env = SoloVecEnv(cfg, n, device="cuda:0", seed=seed)
    ors = [OracleEnv(env.model, env.params, seed=seed, env_id=i) for i in range(nref)]
    obs = env.reset().cpu().numpy()
    fl = flag_slots(ors[0].d0, env.sim.nj, 2)
    worst = 0.0
    for i, o in enumerate(ors):
        df = obs_diff(o.reset(), obs[i], o.d0); df[fl] = 0
        worst = max(worst, df.max())
    rng = np.random.default_rng(seed)
    for t in range(2):
        f = env.get_push_force().cpu().numpy()
        assert np.all(np.any(f[:nref, :2] != 0, axis=1))
        a = rng.uniform(-1, 1, size=(n, env.sim.act_dim)).astype(np.float32)
        ob, rw, dn, _ = env.step(torch.from_numpy(a).cuda())
        ob, rw, dn = ob.cpu().numpy(), rw.cpu().numpy(), dn.cpu().numpy()
        for i, o in enumerate(ors):
            o.set_external_force(f[i].astype(np.float64))
            oo, r, d, _ = o.step(a[i].astype(np.float64), auto_reset=True)
            assert d == (dn[i] > 0.5)
            df = obs_diff(oo, ob[i], o.d0); df[fl] = 0
            worst = max(worst, (df / np.maximum(1.0, np.abs(oo))).max(), abs(r - rw[i]) / max(1.0, abs(r)))
    env.close()
    assert worst < 5e-3, worst


def test_zero_force_agrees_with_the_build_without_pushes():
    """push_force 0: the push build (another binary) follows the build without pushes within the bounds of
    test_degenerate_ranges_agree_with_the_plain_build_on_a_rollout, over 50 steps."""
    from solorl_b200.envs import SoloVecEnv
    cfg = make_config("solo12", task="walk", H=1)
    envs = [SoloVecEnv(c, 256, device="cuda:0", seed=4)
            for c in (cfg, dict(cfg, push_force=0.0, push_interval=10, push_duration=4))]
    assert [e.sim.step_variant for e in envs] == ["latency", "latency+push"]
    for e in envs:
        e.reset()
    g = torch.Generator(device="cuda").manual_seed(3)
    for t in range(50):
        assert torch.count_nonzero(envs[1].get_push_force()) == 0
        a = torch.rand(256, 12, device="cuda", generator=g) * 2 - 1
        (o0, r0, d0, _), (o1, r1, d1, _) = (e.step(a) for e in envs)
        assert torch.equal(d0, d1), t
        assert (r0 - r1).abs().max() < 1e-4, t
        df = obs_diff(o0.cpu().numpy(), o1.cpu().numpy(), 38)
        df[:, flag_slots(38, 12, 2)] = 0
        assert df.max() < 1e-3, t
    for e in envs:
        e.close()


def test_pushes_make_the_trained_stand_policy_fall():
    """The golden Stand policy through make_vec_envs (evaluate), 256 episodes each, seeds fixed: without pushes it
    holds the pose, with pushes of up to 40 N per axis for 10 of every 50 control steps it falls.  Measured on a
    B200 (1000 W): 0 of 256 episodes end in a fall without pushes, 256 of 256 with them."""
    from solorl_b200.agents.evaluate import evaluate, load_policy
    from solorl_b200.envs import Box
    from tests.helpers import GOLDEN
    space = Box(-np.ones(12), np.ones(12))
    pol, _ = load_policy(os.path.join(GOLDEN, "ppo_stand_solo12.pt"), (76,), space)
    cfg = make_config("solo12", "stand", "torque", 1)
    falls = {}
    for name, extra in (("none", {}), ("pushed", {"push_force": 40.0, "push_interval": 50, "push_duration": 10})):
        res = evaluate(pol, dict(cfg, **extra), num_runs=256, num_envs=256, seed=21)
        assert len(res["success"]) == 256
        falls[name] = int((res["success"] == 0).sum())
    print("falls", falls)
    assert falls["pushed"] > falls["none"] + 50, falls


# ---- what pushes do not reach, plumbing and rejections --------------------------------------------------------
def test_substep_and_actuator_step_ignore_the_pushes():
    """solo_substep (the step build with pushes, run in substep mode) and solo_actuator_step (the gait envs'
    kernel) give what a handle without pushes gives: a 50 N push over one airborne substep would change the base
    velocity by ~0.1 m/s."""
    rng = np.random.default_rng(181)
    n = 64
    sims = [make_sim("solo12", n, task="walk", **kw)[0] for kw in ({}, dict(push_force=50.0, **EVERY_STEP))]
    nj = sims[0].nj
    s0 = random_states(rng, n, nj)
    s0[:, 2] += 1.0
    tau = rng.uniform(-3, 3, size=(n, nj))
    cmd = np.zeros((n, 5, nj), np.float32)
    cmd[:, 0] = s0[:, 13:13 + nj]
    cmd[:, 2], cmd[:, 3] = 3.0, 0.2
    sub, act = [], []
    for s in sims:
        s.reset()
        assert np.any(s.push_force().cpu().numpy() != 0) == (s is sims[1])
        s.set_state(cuda(s0))
        s.substep(cuda(tau))
        sub.append(s.get_state().cpu().numpy().astype(np.float64))
        s.set_state(cuda(s0))
        s.actuator_step(cuda(cmd), 3)
        act.append(s.get_state().cpu().numpy())
    assert (np.abs(sub[0] - sub[1]) / np.maximum(1.0, np.abs(sub[0]))).max() < 1e-5
    np.testing.assert_array_equal(act[0], act[1])
    for s in sims:
        s.close()


def test_variant_strings(monkeypatch):
    cases = [({}, {}, "latency"), (RANGES, {}, "latency+rand"), ({}, PUSH, "latency+push"),
             (RANGES, PUSH, "latency+rand+push"), ({"body_contacts": 1}, PUSH, "body+push"),
             (dict(RANGES, body_contacts=1), PUSH, "body+rand+push")]
    for a, b, want in cases:
        sim, _, _ = make_sim("solo8", 16, task="walk", **a, **b)
        assert sim.step_variant == want
        sim.close()
    monkeypatch.setenv("SOLO_STEP_VARIANT", "throughput")
    for a, want in (({}, "throughput+push"), (RANGES, "throughput+rand+push")):
        sim, _, _ = make_sim("solo8", 16, task="walk", **a, **PUSH)
        assert sim.step_variant == want
        sim.close()


def test_public_wrappers_reach_the_push_force():
    from solorl_b200.envs import make_vec_envs
    envs = make_vec_envs(make_config("solo8", task="walk", push_force=30.0, **EVERY_STEP), 32)
    envs.reset()
    f = envs.get_push_force()
    assert f.shape == (32, 3) and f.is_cuda and torch.count_nonzero(f[:, :2]) > 0
    envs.close()
    envs = make_vec_envs(make_config("solo8", task="walk"), 32)
    envs.reset()
    assert torch.count_nonzero(envs.get_push_force()) == 0
    envs.close()


def test_create_rejects_bad_pushes(monkeypatch):
    from solorl_b200 import _lib
    L = _lib.lib()
    m = SoloModel.builtin("solo12")
    t = abi.model_table(m)
    good = abi.params_from_config(make_config("solo12", task="walk", **PUSH), m)
    h = C.c_void_p()
    for field, value in (("push_force", -1.0), ("push_force", float("nan")), ("push_force", float("inf")),
                         ("push_interval", -1), ("push_duration", 0), ("push_duration", 7)):
        p = abi.SoloSimParams.from_buffer_copy(good)
        setattr(p, field, value)
        assert L.solo_create(C.byref(t), C.byref(p), 16, 0, 0, 0, C.byref(h)) == -1, field     # SOLO_E_ARG
        assert b"push" in L.solo_last_error(None), field
    p = abi.SoloSimParams.from_buffer_copy(good)
    p.episode_length, p.push_interval, p.push_duration = 2 ** 31 - 1, 1, 1
    assert L.solo_create(C.byref(t), C.byref(p), 16, 0, 0, 0, C.byref(h)) == -1
    assert b"push" in L.solo_last_error(None)
    monkeypatch.setenv("SOLO_STEP_VARIANT", "wide")
    assert L.solo_create(C.byref(t), C.byref(good), 64, 0, 0, 0, C.byref(h)) == -1
    assert b"push" in L.solo_last_error(None) and b"wide" in L.solo_last_error(None)
