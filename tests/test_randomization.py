"""Per-env randomised dynamics, the parts that run without a GPU: the config keys and their mapping onto
SoloSimParams, and the sampler that begin_reset calls (solo_env.cuh sample_env_dyn), built for the host."""
import numpy as np
import pytest
from scipy import stats

from solorl_b200 import abi
from solorl_b200.model import SoloModel
from tests.emu import dyn_sampler
from tests.helpers import make_config

RANGES = {"randomize_friction": [0.5, 1.25], "randomize_base_mass": [0.8, 1.2],
          "randomize_motor_strength": [0.8, 1.2]}
FIELDS = {"randomize_friction": ("friction_lo", "friction_hi"),
          "randomize_base_mass": ("base_mass_scale_lo", "base_mass_scale_hi"),
          "randomize_motor_strength": ("motor_strength_lo", "motor_strength_hi")}


def params(**kw):
    m = SoloModel.builtin("solo12")
    return abi.params_from_config(make_config("solo12", task="walk", **kw), m)


def fields(p):
    return {f: getattr(p, f) for f, _ in p._fields_}


# ---- config mapping ---------------------------------------------------------------------------------
def test_keys_map_onto_the_fields():
    p = params(**RANGES)
    assert p.randomize == 1
    for key, (lo, hi) in FIELDS.items():
        assert (getattr(p, lo), getattr(p, hi)) == tuple(RANGES[key])


@pytest.mark.parametrize("key", sorted(RANGES))
def test_a_missing_key_gives_the_nominal_degenerate_range(key):
    p = params(friction=0.8, **{key: RANGES[key]})
    assert p.randomize == 1
    nominal = {"randomize_friction": 0.8, "randomize_base_mass": 1.0, "randomize_motor_strength": 1.0}
    for other, (lo, hi) in FIELDS.items():
        want = tuple(RANGES[other]) if other == key else (nominal[other], nominal[other])
        assert (getattr(p, lo), getattr(p, hi)) == want, other


def test_without_the_keys_the_params_are_those_of_today():
    p, q = params(), abi.default_params()
    assert p.randomize == 0
    for f in ("friction_lo", "friction_hi", "base_mass_scale_lo", "base_mass_scale_hi", "motor_strength_lo",
              "motor_strength_hi"):
        assert getattr(p, f) == 0.0 == getattr(q, f)
    with_keys = fields(params(**RANGES))
    without = fields(p)
    changed = {f for f in without if without[f] != with_keys[f]}
    assert changed == {"randomize"} | {f for lo_hi in FIELDS.values() for f in lo_hi}


@pytest.mark.parametrize("key,bad", [
    ("randomize_friction", [1.0, 0.5]),          # reversed
    ("randomize_friction", [-0.1, 1.0]),         # negative friction
    ("randomize_base_mass", [1.2, 0.8]),
    ("randomize_base_mass", [0.0, 1.0]),         # a zero scale
    ("randomize_base_mass", [-1.0, 1.0]),
    ("randomize_motor_strength", [0.0, 0.0]),
    ("randomize_motor_strength", [1.1, 0.9]),
    ("randomize_motor_strength", [0.9]),          # not a pair
    ("randomize_motor_strength", 1.0),
    ("randomize_friction", [0.5, float("nan")]),
])
def test_malformed_ranges_raise(key, bad):
    with pytest.raises(ValueError):
        params(**{key: bad})


def test_zero_friction_is_a_valid_range():
    p = params(randomize_friction=[0.0, 0.0])
    assert (p.friction_lo, p.friction_hi) == (0.0, 0.0)


def test_bench_config_declares_the_ranges():
    import yaml
    from tests.helpers import ROOT
    with open(f"{ROOT}/configs/bench12_walk_rand.yaml") as f:
        cfg = yaml.safe_load(f)
    with open(f"{ROOT}/configs/bench12_walk.yaml") as f:
        base = yaml.safe_load(f)
    assert {k: cfg[k] for k in RANGES} == RANGES
    assert {k: v for k, v in cfg.items() if k not in RANGES} == base


# ---- the sampler ----------------------------------------------------------------------------------
def test_draws_lie_inside_their_ranges():
    p = params(**RANGES)
    x = dyn_sampler.sample(p, seed=3, gid0=0, n=20000, episode=1).astype(np.float64)
    for c, key in enumerate(("randomize_friction", "randomize_base_mass", "randomize_motor_strength")):
        lo, hi = (float(np.float32(v)) for v in RANGES[key])
        assert x[:, c].min() >= lo and x[:, c].max() <= hi, key


def test_degenerate_ranges_give_exactly_the_nominal_values():
    p = params(friction=0.7, randomize_base_mass=[1.0, 1.0])
    x = dyn_sampler.sample(p, seed=1, gid0=0, n=1000, episode=4)
    assert np.all(x[:, 0] == np.float32(0.7)) and np.all(x[:, 1:] == 1.0)


def test_draws_are_deterministic_in_seed_id_and_episode():
    p = params(**RANGES)
    a = dyn_sampler.sample(p, seed=11, gid0=100, n=64, episode=3)
    b = dyn_sampler.sample(p, seed=11, gid0=100, n=64, episode=3)
    np.testing.assert_array_equal(a, b)
    # each id's draw depends on its global id only, not on where a batch starts (sharding invariance)
    c = dyn_sampler.sample(p, seed=11, gid0=132, n=32, episode=3)
    np.testing.assert_array_equal(a[32:], c)
    assert not np.array_equal(a, dyn_sampler.sample(p, seed=12, gid0=100, n=64, episode=3))


def test_another_episode_gives_other_values():
    p = params(**RANGES)
    a = dyn_sampler.sample(p, seed=5, gid0=0, n=256, episode=1)
    b = dyn_sampler.sample(p, seed=5, gid0=0, n=256, episode=2)
    assert np.all(np.any(a != b, axis=1))


def test_draws_are_uniform():
    p = params(**RANGES)
    x = dyn_sampler.sample(p, seed=0, gid0=0, n=65536, episode=1).astype(np.float64)
    for c, key in enumerate(("randomize_friction", "randomize_base_mass", "randomize_motor_strength")):
        lo, hi = RANGES[key]
        res = stats.kstest(x[:, c], "uniform", args=(lo, hi - lo))
        assert res.pvalue > 1e-3, (key, res)
    # the three values of an env come from different words of the draw
    assert abs(np.corrcoef(x[:, 1], x[:, 2])[0, 1]) < 0.02


def test_the_sampler_rejects_what_solo_create_rejects():
    p = params(**RANGES)
    p.base_mass_scale_lo = 0.0
    with pytest.raises(ValueError):
        dyn_sampler.sample(p, seed=0, gid0=0, n=1, episode=1)
    p = params(**RANGES)
    p.friction_lo, p.friction_hi = 1.0, 0.5
    with pytest.raises(ValueError):
        dyn_sampler.sample(p, seed=0, gid0=0, n=1, episode=1)


# (seed, global env id, episode) -> settle count and pointgoal goal drawn by the reset, as the per-env RNG gave them
# before randomised dynamics existed: the dynamics draw uses a draw index of its own and must not move these
RESET_DRAWS = [
    (0, 0, 1, 10, -1.9396580457687378, -1.0589866638183594),
    (0, 0, 2, 11, -1.7129273414611816, -1.1489453315734863),
    (0, 5, 1, 9, -1.3158607482910156, 1.1578704118728638),
    (0, 5, 2, 6, -1.2884635925292969, 1.8264122009277344),
    (7, 123456789012, 1, 11, -1.1433446407318115, 1.5089809894561768),
    (7, 123456789012, 2, 7, 1.5139118432998657, 1.893282175064087),
    (2 ** 40 + 3, 17, 1, 7, -1.0428180694580078, -1.8668508529663086),
    (2 ** 40 + 3, 17, 2, 7, -1.3615608215332031, 1.4409078359603882),
]


def test_goal_and_settle_draws_are_unchanged():
    from tests.emu.emu import EmuEnv
    m = SoloModel.builtin("solo12")
    p = abi.params_from_config(make_config("solo12", task="pointgoal", H=0), m)
    pg = 14 + 8 * 3
    envs = {}
    for seed, gid, ep, k, gx, gy in RESET_DRAWS:
        e = envs.setdefault((seed, gid), EmuEnv(m, p, seed=seed, env_id=gid))
        o = e.reset()
        assert e.settle_count_last == k, (seed, gid, ep)
        assert (o[pg + 2] * 2, o[pg + 3] * 2) == (np.float32(gx), np.float32(gy)), (seed, gid, ep)
