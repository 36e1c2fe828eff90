"""Random pushes, the parts that run without a GPU: the config keys and their mapping onto SoloSimParams, and the
push schedule the step kernel computes (solo_env.cuh sample_push), built for the host."""
import numpy as np
import pytest
from scipy import stats

from solorl_b200 import abi
from solorl_b200.model import SoloModel
from tests.emu import dyn_sampler, push_sampler
from tests.helpers import make_config

PUSH = {"push_force": 15.0, "push_interval": 50, "push_duration": 5}
FIELDS = ("push_force", "push_interval", "push_duration")


def params(**kw):
    m = SoloModel.builtin("solo12")
    return abi.params_from_config(make_config("solo12", task="walk", **kw), m)


def fields(p):
    return {f: getattr(p, f) for f, _ in p._fields_}


def pushes(F, I, D, seed=0, gid0=0, n=64, episode=1, t0=0, T=None):
    p = params(push_force=F, push_interval=I, push_duration=D)
    return push_sampler.push_sample(p, seed, gid0, n, episode, t0, 3 * I if T is None else T)


# ---- config mapping ---------------------------------------------------------------------------------
def test_keys_map_onto_the_fields():
    p = params(**PUSH)
    assert (p.push_force, p.push_interval, p.push_duration) == (15.0, 50, 5)


def test_without_the_keys_the_params_are_those_of_today():
    p, q = params(), abi.default_params()
    assert p.push_interval == 0
    for f in FIELDS:
        assert getattr(p, f) == 0 == getattr(q, f)
    with_keys, without = fields(params(**PUSH)), fields(p)
    assert {f for f in without if without[f] != with_keys[f]} == set(FIELDS)


@pytest.mark.parametrize("keys", [("push_force",), ("push_force", "push_interval"), ("push_force", "push_duration"),
                                  ("push_interval", "push_duration")])
def test_a_missing_key_raises(keys):
    with pytest.raises(ValueError):
        params(**{k: PUSH[k] for k in keys})


@pytest.mark.parametrize("key,bad", [
    ("push_force", -1.0),
    ("push_force", float("nan")),
    ("push_force", float("inf")),
    ("push_force", "strong"),
    ("push_interval", 0),              # interval 0 with a force set
    ("push_interval", -5),
    ("push_interval", 2.5),
    ("push_interval", "often"),
    ("push_duration", 0),
    ("push_duration", 51),             # longer than the interval
    ("push_duration", None),
])
def test_malformed_values_raise(key, bad):
    with pytest.raises(ValueError):
        params(**{**PUSH, key: bad})


def test_duration_equal_to_interval_and_zero_force_are_valid():
    p = params(push_force=0.0, push_interval=3, push_duration=3)
    assert (p.push_force, p.push_interval, p.push_duration) == (0.0, 3, 3)


def test_bench_config_declares_the_pushes():
    import yaml
    from tests.helpers import ROOT
    with open(f"{ROOT}/configs/bench12_walk_push.yaml") as f:
        cfg = yaml.safe_load(f)
    with open(f"{ROOT}/configs/bench12_walk.yaml") as f:
        base = yaml.safe_load(f)
    assert {k: cfg[k] for k in FIELDS} == PUSH
    assert {k: v for k, v in cfg.items() if k not in FIELDS} == base


# ---- the schedule ---------------------------------------------------------------------------------
CASES = [(15.0, 50, 5), (40.0, 7, 3), (2.0, 10, 1), (8.0, 4, 4)]


@pytest.mark.parametrize("F,I,D", CASES)
def test_every_interval_holds_one_window_of_constant_force(F, I, D):
    for seed, episode in ((0, 1), (9, 2), (2 ** 40 + 3, 7)):
        x = pushes(F, I, D, seed=seed, gid0=1000 * episode, n=128, episode=episode, T=4 * I)
        assert np.all(x[..., 2] == 0.0)
        f32 = np.float32(F)
        assert np.all(np.abs(x[..., :2]) <= f32)
        on = np.any(x[..., :2] != 0.0, axis=-1)           # a drawn force is 0 with probability ~2^-24 per axis
        for j in range(4):
            win = on[:, j * I:(j + 1) * I]
            assert np.all(win.sum(axis=1) == D)
            first = np.argmax(win, axis=1)
            for i in range(x.shape[0]):
                assert np.all(win[i, first[i]:first[i] + D])      # contiguous, inside the interval
                f = x[i, j * I + first[i]:j * I + first[i] + D, :2]
                assert np.all(f == f[0])                          # a rectangular pulse


def test_zero_force_gives_zero_pushes():
    x = pushes(0.0, 6, 2, n=256)
    assert np.all(x == 0.0)


def test_duration_equal_to_interval_pushes_every_step():
    x = pushes(20.0, 5, 5, n=256, T=50)
    assert np.all(np.any(x[..., :2] != 0.0, axis=-1))


def test_the_schedule_is_deterministic_and_does_not_depend_on_sharding():
    a = pushes(15.0, 10, 3, seed=11, gid0=100, n=64, episode=3, T=40)
    np.testing.assert_array_equal(a, pushes(15.0, 10, 3, seed=11, gid0=100, n=64, episode=3, T=40))
    np.testing.assert_array_equal(a[32:], pushes(15.0, 10, 3, seed=11, gid0=132, n=32, episode=3, T=40))
    np.testing.assert_array_equal(a[:, 25:], pushes(15.0, 10, 3, seed=11, gid0=100, n=64, episode=3, t0=25, T=15))
    assert not np.array_equal(a, pushes(15.0, 10, 3, seed=12, gid0=100, n=64, episode=3, T=40))
    assert not np.array_equal(a, pushes(15.0, 10, 3, seed=11, gid0=100, n=64, episode=4, T=40))


def test_window_starts_are_uniform():
    I, D = 12, 4
    x = pushes(10.0, I, D, n=4096, T=4 * I)
    on = np.any(x[..., :2] != 0.0, axis=-1).reshape(4096, 4, I)
    starts = np.argmax(on, axis=2).ravel()
    counts = np.bincount(starts, minlength=I - D + 1)
    assert counts.size == I - D + 1
    res = stats.chisquare(counts)
    assert res.pvalue > 1e-3, (counts, res)


def test_forces_are_uniform():
    F, I = 15.0, 3
    x = pushes(F, I, I, n=65536 // 4, T=4 * I).astype(np.float64)   # I = D: one window per interval
    f = x[:, ::I, :2].reshape(-1, 2)
    assert f.shape[0] == 65536
    for c in range(2):
        res = stats.kstest(f[:, c], "uniform", args=(-F, 2 * F))
        assert res.pvalue > 1e-3, (c, res)
    assert abs(np.corrcoef(f[:, 0], f[:, 1])[0, 1]) < 0.02


def test_dynamics_draws_do_not_depend_on_the_push_fields():
    ranges = {"randomize_friction": [0.5, 1.25], "randomize_base_mass": [0.8, 1.2],
              "randomize_motor_strength": [0.8, 1.2]}
    a = dyn_sampler.sample(params(**ranges), seed=3, gid0=0, n=512, episode=2)
    b = dyn_sampler.sample(params(**ranges, **PUSH), seed=3, gid0=0, n=512, episode=2)
    np.testing.assert_array_equal(a, b)


def test_the_sampler_rejects_what_solo_create_rejects():
    for f, v in (("push_force", -1.0), ("push_force", float("nan")), ("push_interval", -1), ("push_duration", 0),
                 ("push_duration", 51)):
        p = params(**PUSH)
        setattr(p, f, v)
        with pytest.raises(ValueError):
            push_sampler.push_sample(p, 0, 0, 1, 1, 0, 1)
    p = params(**PUSH, episode_length=2 ** 31 - 1)
    p.push_interval, p.push_duration = 1, 1
    with pytest.raises(ValueError):
        push_sampler.push_sample(p, 0, 0, 1, 1, 0, 1)
    p = params()                                   # pushes off: all zero
    assert np.all(push_sampler.push_sample(p, 0, 0, 4, 1, 0, 10) == 0.0)
