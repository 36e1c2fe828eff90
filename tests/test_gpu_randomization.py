"""Per-env randomised dynamics on the GPU (SoloSimParams.randomize): the device draws against the host build of
the sampler, the draws' independence of sharding and their renewal at exactly the envs that reset, and the
physics of each env against an fp64 oracle built with that env's friction, base mass and motor strength."""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from oracle.oracle import OracleEnv
from solorl_b200 import abi
from solorl_b200.model import SoloModel
from tests.emu import dyn_sampler
from tests.helpers import flag_slots, limit_states, make_config, obs_diff, random_states, stance_states

pytestmark = pytest.mark.gpu

ROBOTS = ("solo8", "solo12")
TOL_QDD = 1e-5
TOL_ENV = 1e-6
TOL_CONTACT = 1e-3
RANGES = {"randomize_friction": [0.5, 1.25], "randomize_base_mass": [0.8, 1.2],
          "randomize_motor_strength": [0.8, 1.2]}


def cuda(x):
    return torch.as_tensor(np.asarray(x, dtype=np.float32)).cuda()


def make_sim(robot, n, seed=0, env_id_offset=0, **kw):
    from solorl_b200.sim import SoloSim
    cfg = make_config(robot, **kw)
    m = SoloModel.resolve(robot)
    p = abi.params_from_config(cfg, m)
    return SoloSim(m, p, n, device=0, seed=seed, env_id_offset=env_id_offset), m, p


def oracle_for(m, p, row):
    """The fp64 oracle of one env of a randomised handle: its friction, its base mass and inertia."""
    mu, sm, _ = (float(x) for x in row)
    q = abi.SoloSimParams.from_buffer_copy(p)
    q.friction = mu
    mm = dataclasses.replace(m, base_mass=sm * m.base_mass, base_inertia=sm * np.asarray(m.base_inertia))
    return OracleEnv(mm, q)


# ---- the draws ------------------------------------------------------------------------------------------------
def test_device_draws_equal_the_host_sampler():
    n = 300
    sim, m, p = make_sim("solo12", n, seed=9, task="walk", **RANGES)
    assert sim.step_variant == "latency+rand"
    for episode in (1, 2):
        sim.reset()
        got = sim.env_params().cpu().numpy()
        np.testing.assert_array_equal(got, dyn_sampler.sample(p, 9, 0, n, episode))
    sim.close()


def test_before_the_first_reset_and_without_randomisation_the_rows_are_nominal():
    sim, _, p = make_sim("solo8", 40, task="walk", friction=0.8)
    assert p.randomize == 0 and sim.step_variant == "latency"
    sim.reset()
    sim.step(torch.rand(40, sim.act_dim, device="cuda") * 2 - 1)
    want = np.tile(np.float32([0.8, 1.0, 1.0]), (40, 1))
    np.testing.assert_array_equal(sim.env_params().cpu().numpy(), want)
    sim.close()
    sim, _, _ = make_sim("solo8", 40, task="walk", friction=0.8, **RANGES)
    np.testing.assert_array_equal(sim.env_params().cpu().numpy(), want)
    sim.close()


def test_one_handle_equals_two_shards():
    """The draws and the physics they drive depend on the global env id, not on the sharding."""
    n = 64
    whole, _, _ = make_sim("solo12", 2 * n, seed=3, task="walk", episode_length=20, **RANGES)
    parts = [make_sim("solo12", n, seed=3, env_id_offset=k * n, task="walk", episode_length=20, **RANGES)[0]
             for k in range(2)]
    whole.reset()
    for s in parts:
        s.reset()
    g = torch.Generator(device="cuda").manual_seed(2)
    for t in range(30):
        a = torch.rand(2 * n, whole.act_dim, device="cuda", generator=g) * 2 - 1
        o, r, d = whole.step(a)
        for k, s in enumerate(parts):
            ok, rk, dk = s.step(a[k * n:(k + 1) * n])
            assert torch.equal(o[k * n:(k + 1) * n], ok) and torch.equal(r[k * n:(k + 1) * n], rk)
            assert torch.equal(d[k * n:(k + 1) * n], dk)
    assert torch.equal(whole.env_params(), torch.cat([s.env_params() for s in parts]))
    for s in [whole] + parts:
        s.close()


def test_masked_and_auto_resets_redraw_exactly_the_resetting_envs():
    n = 256
    sim, _, p = make_sim("solo12", n, seed=4, task="walk", episode_length=7, **RANGES)
    sim.reset()
    episode = np.ones(n, dtype=np.int64)
    before = sim.env_params().cpu().numpy()
    mask = np.zeros(n, dtype=bool)
    mask[::3] = True
    sim.reset(mask=torch.as_tensor(mask, device="cuda"))
    episode[mask] += 1
    after = sim.env_params().cpu().numpy()
    assert (np.any(after != before, axis=1) == mask).all()
    g = torch.Generator(device="cuda").manual_seed(5)
    ndone = 0
    for t in range(20):
        before = after
        _, _, d = sim.step(torch.rand(n, sim.act_dim, device="cuda", generator=g) * 2 - 1)
        done = d.cpu().numpy() > 0.5
        episode[done] += 1
        ndone += int(done.sum())
        after = sim.env_params().cpu().numpy()
        assert (np.any(after != before, axis=1) == done).all()
    assert ndone >= n
    for ep in np.unique(episode):      # every row is the host sampler's draw for the env's current episode
        idx = np.nonzero(episode == ep)[0]
        want = dyn_sampler.sample(p, 4, 0, n, int(ep))
        np.testing.assert_array_equal(after[idx], want[idx])
    sim.close()


def test_goal_draws_are_those_of_a_plain_handle():
    """The dynamics draw has a draw index of its own: the pointgoal goals (and settle counts) stay as they are."""
    sims = [make_sim("solo12", 64, seed=8, task="pointgoal", H=0, **kw)[0] for kw in ({}, RANGES)]
    pg = 14 + 8 * 3
    obs = [s.reset()[:, pg + 2:pg + 4].clone() for s in sims]
    assert torch.equal(obs[0], obs[1])
    for s in sims:
        s.close()


# ---- per-env physics against the fp64 oracle ------------------------------------------------------------------
@pytest.mark.parametrize("robot", ROBOTS)
def test_forward_dynamics_per_env_1e5(robot):
    rng = np.random.default_rng(120)
    n = 256
    sim, m, p = make_sim(robot, n, randomize_base_mass=[0.5, 1.5])
    sim.reset()
    prm = sim.env_params().cpu().numpy()
    assert prm[:, 1].min() < 0.6 and prm[:, 1].max() > 1.4
    s = random_states(rng, n, sim.nj)
    tau = rng.uniform(-3, 3, size=(n, sim.nj)).astype(np.float32).astype(np.float64)
    got = sim.forward_dynamics(cuda(s), cuda(tau)).cpu().numpy().astype(np.float64)
    worst = 0.0
    for i in range(n):
        o = oracle_for(m, p, prm[i])
        o.set_state(s[i])
        ref = o.forward_dynamics(tau[i])
        worst = max(worst, np.linalg.norm(ref[6:] - got[i, 6:]) / np.linalg.norm(ref[6:]),
                    np.linalg.norm(ref - got[i]) / np.linalg.norm(ref))
    assert worst < TOL_QDD, worst
    sim.close()


@pytest.mark.parametrize("control", ["torque", "pd", "vpd"])
def test_action_to_torque_per_env_1e6(control):
    rng = np.random.default_rng(121)
    n = 128
    sim, m, p = make_sim("solo12", n, control=control, randomize_motor_strength=[0.5, 1.5])
    sim.reset()
    st = sim.env_params().cpu().numpy()[:, 2].astype(np.float64)
    s = random_states(rng, n, sim.nj, vel_scale=0.2)
    a = rng.uniform(-1.5, 1.5, size=(n, sim.act_dim))
    if control == "vpd":
        a[:, -2] = rng.uniform(0, 6, size=n)
        a[:, -1] = rng.uniform(0, 0.3, size=n)
    a = a.astype(np.float32).astype(np.float64)
    sim.set_state(cuda(s))
    got = sim.action_to_torque(cuda(a)).cpu().numpy()
    o = OracleEnv(m, p)
    nj = sim.nj
    for i in range(n):
        o.set_state(s[i])
        if control == "torque":
            scale = np.ones(nj)
        else:      # 1e-6 relative to the operands of the PD law, as test_action_to_torque_1e6
            kp, kd = (a[i, -2], a[i, -1]) if control == "vpd" else (p.kp, p.kd)
            q_ref = np.clip(a[i, :nj], -1, 1) * 10.0
            scale = np.maximum(1.0, abs(kp) * (np.abs(q_ref) + np.abs(s[i, 13:13 + nj])) + abs(kd) * np.abs(s[i, 13 + nj:]))
        assert (np.abs(st[i] * o.action_to_torque(a[i]) - got[i]) < TOL_ENV * scale * st[i]).all()
    sim.close()


def _hold_torque(s, nj, target, kp=3.0, kd=0.05):
    return np.clip(kp * (target - s[:, 13:13 + nj]) - kd * s[:, 13 + nj:], -3, 3)


@pytest.mark.parametrize("build", ("latency", "throughput"))
@pytest.mark.parametrize("robot", ROBOTS)
def test_contact_substep_per_env_1e3(robot, build, monkeypatch):
    """test_contact_substep_1e3 with every env on its own friction (0.4 .. 1.25) and base mass."""
    monkeypatch.setenv("SOLO_STEP_VARIANT", build)
    rng = np.random.default_rng(124)
    n = 64
    sim, m, p = make_sim(robot, n, randomize_friction=[0.4, 1.25], randomize_base_mass=[0.8, 1.2])
    assert sim.step_variant == build + "+rand"
    sim.reset()
    prm = sim.env_params().cpu().numpy()
    nj = sim.nj
    cur = stance_states(rng, n, nj)
    target = cur[:, 13:13 + nj].copy()
    oracles = {i: oracle_for(m, p, prm[i]) for i in range(0, n, 2)}
    errs, ncs = [], []
    for t in range(40):
        tau = (_hold_torque(cur, nj, target) + rng.normal(size=(n, nj)) * 0.3).astype(np.float32).astype(np.float64)
        sim.set_state(cuda(cur))
        sim.substep(cuda(tau))
        nxt = sim.get_state().cpu().numpy().astype(np.float64)
        con = sim.get_contacts().cpu().numpy()
        for i, o in oracles.items():
            o.set_state(cur[i])
            o.substep(tau[i])
            ref = o.get_state()
            errs.append((np.abs(ref - nxt[i]) / np.maximum(1.0, np.abs(ref))).max())
            co = o.get_contacts()
            assert (co[:, 1] == con[i, :, 1]).all()
            assert np.abs(co[:, 2] - con[i, :, 2]).max() < 2e-2 * max(1.0, co[:, 2].max())
            ncs.append(co[:, 1].sum())
        cur = nxt
    assert np.mean(ncs) > 2.5
    assert max(errs) < TOL_CONTACT, (max(errs), np.median(errs))
    sim.close()


@pytest.mark.parametrize("robot", ROBOTS)
def test_joint_limit_substep_per_env_1e3(robot):
    rng = np.random.default_rng(143)
    n = 96
    sim, m, p = make_sim(robot, n, joint_limits=1, **RANGES)
    sim.reset()
    prm = sim.env_params().cpu().numpy()
    nj = sim.nj
    s0 = limit_states(rng, n, nj)
    s0[1::2, 13:13 + nj] = np.clip(s0[1::2, 13:13 + nj], -9.5, 9.5)
    tau = rng.uniform(-3, 3, size=(n, nj)).astype(np.float32).astype(np.float64)
    sim.set_state(cuda(s0))
    sim.substep(cuda(tau))
    got = sim.get_state().cpu().numpy().astype(np.float64)
    con = sim.get_contacts().cpu().numpy()
    errs, rows = [], 0
    for i in range(n):
        o = oracle_for(m, p, prm[i])
        o.set_state(s0[i]); o.substep(tau[i])
        ref = o.get_state()
        errs.append((np.abs(ref - got[i]) / np.maximum(1.0, np.abs(ref))).max())
        rows += o.last_limit_rows
        assert (o.get_contacts()[:, 1] == con[i, :, 1]).all()
    assert rows > n / 2
    assert max(errs) < TOL_CONTACT, (max(errs), np.median(errs))
    sim.close()


@pytest.mark.parametrize("robot", ROBOTS)
def test_body_contact_substep_per_env_1e3(robot):
    """test_body_contact_substep_1e3 with per-env friction and base mass: the same bounds on the samples whose
    fp64 oracle is stable under a one-ulp perturbation of its input, the same exceedance budget."""
    from tests.helpers import collapsed_states
    rng = np.random.default_rng(161)
    n = 96
    sim, m, p = make_sim(robot, n, body_contacts=1, randomize_friction=[0.4, 1.25], randomize_base_mass=[0.8, 1.2])
    assert sim.step_variant == "body+rand"
    sim.reset()
    prm = sim.env_params().cpu().numpy()
    nj = sim.nj
    pairs = [(oracle_for(m, p, prm[i]), oracle_for(m, p, prm[i])) for i in range(n)]
    cur = np.concatenate([collapsed_states(rng, 64, robot, params=p), stance_states(rng, 32, nj)])
    cur = cur[rng.permutation(n)]
    errs, sens, body, total = [], [], 0, 0
    for t in range(20):
        tau = (rng.normal(size=(n, nj)) * 0.5).astype(np.float32).astype(np.float64)
        sim.set_state(cuda(cur))
        sim.substep(cuda(tau))
        nxt = sim.get_state().cpu().numpy().astype(np.float64)
        con = sim.get_contacts().cpu().numpy()
        pert = cur * (1 + rng.choice([-1, 1], size=cur.shape) * 6e-8)
        for i, (o, o2) in enumerate(pairs):
            o.set_state(cur[i]); o.substep(tau[i])
            o2.set_state(pert[i]); o2.substep(tau[i])
            ref = o.get_state()
            assert (o.get_contacts()[:, 1] == con[i, :, 1]).all()
            scale = np.maximum(1.0, np.abs(ref))
            errs.append((np.abs(ref - nxt[i]) / scale).max())
            sens.append((np.abs(ref - o2.get_state()) / scale).max())
        body += int((cur[:, 2] < 0.12).sum()); total += n
        cur = nxt
    errs, sens = np.array(errs), np.array(sens)
    stable = sens < 1e-4
    assert body > 0.5 * total and stable.mean() > 0.9
    assert np.isfinite(nxt).all()
    assert np.median(errs) < 1e-4 and np.quantile(errs, 0.99) < TOL_CONTACT
    rate = float((errs[stable] > TOL_CONTACT).mean())
    assert rate <= 2e-3 and errs[stable].max() < 1e-2, (rate, errs[stable].max())
    sim.close()


# ---- reset modes and the plain build --------------------------------------------------------------------------
def test_cached_reset_equals_simulated_reset_bitwise_under_randomisation():
    from solorl_b200.envs import SoloVecEnv
    for robot, task in (("solo12", "pointgoal"), ("solo8", "walk")):
        cfg = make_config(robot, task=task, H=1, episode_length=15, **RANGES)
        e1 = SoloVecEnv(cfg, 96, device="cuda:0", seed=5)
        e2 = SoloVecEnv(dict(cfg, reset_mode="simulate"), 96, device="cuda:0", seed=5)
        assert torch.equal(e1.reset(), e2.reset())
        assert torch.equal(e1.get_env_params(), e2.get_env_params())
        g = torch.Generator(device="cuda").manual_seed(1)
        ndone = 0
        for t in range(40):
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


def test_degenerate_ranges_agree_with_the_plain_build_on_a_rollout():
    """Ranges of width zero at the nominal values: the randomised build (another binary) follows the plain one
    within the bounds test_builds_agree_on_a_rollout holds two builds to, over 50 steps."""
    from solorl_b200.envs import SoloVecEnv
    cfg = make_config("solo12", task="walk", H=1)
    degenerate = dict(cfg, randomize_friction=[1.0, 1.0], randomize_base_mass=[1.0, 1.0],
                      randomize_motor_strength=[1.0, 1.0])
    envs = [SoloVecEnv(c, 256, device="cuda:0", seed=4) for c in (cfg, degenerate)]
    assert [e.sim.step_variant for e in envs] == ["latency", "latency+rand"]
    for e in envs:
        e.reset()
    g = torch.Generator(device="cuda").manual_seed(3)
    for t in range(50):
        a = torch.rand(256, 12, device="cuda", generator=g) * 2 - 1
        (o0, r0, d0, _), (o1, r1, d1, _) = (e.step(a) for e in envs)
        assert torch.equal(d0, d1), t
        assert (r0 - r1).abs().max() < 1e-4, t
        df = obs_diff(o0.cpu().numpy(), o1.cpu().numpy(), 38)
        df[:, flag_slots(38, 12, 2)] = 0
        assert df.max() < 1e-3, t
    for e in envs:
        e.close()


def test_public_wrappers_reach_the_env_params():
    from solorl_b200.envs import make_vec_envs
    envs = make_vec_envs(make_config("solo8", task="walk", **RANGES), 32)
    envs.reset()
    prm = envs.get_env_params()
    assert prm.shape == (32, 3) and prm.is_cuda
    envs.close()


# ---- rejections -----------------------------------------------------------------------------------------------
def test_create_rejects_bad_randomisation(monkeypatch):
    from solorl_b200 import _lib
    L = _lib.lib()
    m = SoloModel.builtin("solo12")
    t = abi.model_table(m)
    good = abi.params_from_config(make_config("solo12", task="walk", **RANGES), m)
    h = C.c_void_p()
    for field, value in (("friction_lo", -0.1), ("friction_hi", 0.4), ("base_mass_scale_lo", 0.0),
                         ("base_mass_scale_hi", 0.5), ("motor_strength_lo", 0.0), ("motor_strength_hi", 0.5)):
        p = abi.SoloSimParams.from_buffer_copy(good)
        setattr(p, field, value)
        assert L.solo_create(C.byref(t), C.byref(p), 16, 0, 0, 0, C.byref(h)) == -1, field     # SOLO_E_ARG
        assert b"randomize" in L.solo_last_error(None)
    monkeypatch.setenv("SOLO_STEP_VARIANT", "wide")
    assert L.solo_create(C.byref(t), C.byref(good), 64, 0, 0, 0, C.byref(h)) == -1
    assert b"wide" in L.solo_last_error(None)
    plain = abi.params_from_config(make_config("solo12", task="walk"), m)
    assert L.solo_create(C.byref(t), C.byref(plain), 64, 0, 0, 0, C.byref(h)) == 0       # wide without randomisation
    L.solo_destroy(h)
