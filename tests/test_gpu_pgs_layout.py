"""The four-row PGS sweep (joint-limit rows on) pinned bit for bit: single substeps of fixed states, hashed and
compared with hashes recorded by the build before the sweep placed its rows on lanes by sweep position
(tests/golden/pgs_layout_hashes.json).  Any change of a bit in the state or the contact records fails.

Cases: both robots, the latency and throughput builds, cone and pyramid friction, and five state sets:
  stance     a bent-leg stance, 3-4 feet in contact, no joint at a limit;
  limits     the stance with joints at or past the +-10 rad URDF limits in 1-4 legs of every env (limit_states):
             contact rows and several limit rows in one env, relaxed as one group;
  air        the same joints at their limits in free flight: limit rows only;
  sweeps50   the stance with the residual exit off: every contact substep runs all 50 sweeps;
  limits50   the limit states with the residual exit off.

Regenerate (only when the arithmetic is meant to change): python tests/test_gpu_pgs_layout.py --write"""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.helpers import GOLDEN, limit_states, make_config, stance_states  # noqa: E402

pytestmark = pytest.mark.gpu

GOLDEN_FILE = os.path.join(GOLDEN, "pgs_layout_hashes.json")
N = 256
CASES = [f"{robot}-{build}-{'cone' if cone else 'pyramid'}-{kind}"
         for robot in ("solo12", "solo8") for build in ("latency", "throughput") for cone in (1, 0)
         for kind in ("stance", "limits", "air", "sweeps50", "limits50")]
LIMIT_KINDS = ("limits", "air", "limits50")
JOINT_LIMIT = 10.0   # the URDF limits of every Solo joint (joint_state_limit)


def _states(kind, nj, seed):
    rng = np.random.default_rng(seed)
    if kind in LIMIT_KINDS:
        return limit_states(rng, N, nj, airborne=(kind == "air"))
    return stance_states(rng, N, nj)


def limit_legs(state, nj):
    """Per env, the number of legs with a joint at or past its limit: the limit rows of the substep."""
    q = np.abs(state[:, 13:13 + nj]).reshape(len(state), 4, nj // 4)
    return (q >= JOINT_LIMIT).any(axis=2).sum(axis=1)


def run_case(case, joint_limits=1):
    """One substep from fixed states: the sha256 of the float32 state and contact records after it, the number of
    contact points, and the number of limit rows per env of the input."""
    import torch
    from solorl_b200.abi import params_from_config
    from solorl_b200.model import SoloModel
    from solorl_b200.sim import SoloSim
    robot, build, cone, kind = case.split("-")
    os.environ["SOLO_STEP_VARIANT"] = build
    extra = {"cone_friction": 1 if cone == "cone" else 0, "joint_limits": joint_limits}
    if kind.endswith("50"):
        extra["solver_residual_threshold"] = 0.0
    cfg = make_config(robot, **extra)
    m = SoloModel.resolve(robot)
    sim = SoloSim(m, params_from_config(cfg, m), N, device=0, seed=0)
    try:
        nj = sim.nj
        seed = sum(map(ord, case))
        cur = _states(kind, nj, seed)
        rng = np.random.default_rng(seed + 1)
        tau = np.clip(rng.normal(size=(N, nj)) * 1.5, -3, 3).astype(np.float32)
        sim.set_state(torch.as_tensor(cur.astype(np.float32)).cuda())
        sim.substep(torch.as_tensor(tau).cuda())
        state = sim.get_state().cpu().numpy().astype(np.float32)
        con = sim.get_contacts().cpu().numpy().astype(np.float32)
        torch.cuda.synchronize()
    finally:
        sim.close()
        os.environ.pop("SOLO_STEP_VARIANT", None)
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(state).tobytes())
    h.update(np.ascontiguousarray(con).tobytes())
    return h.hexdigest(), int((con[:, :, 1] > 0).sum()), limit_legs(cur, nj)


@pytest.mark.parametrize("case", CASES)
def test_pgs_substep_bits_are_pinned(case):
    with open(GOLDEN_FILE) as f:
        golden = json.load(f)
    digest, contacts, nlim = run_case(case)
    kind = case.split("-")[3]
    if kind in LIMIT_KINDS:
        # several limit rows in one env for a good share of the envs, and the rows act on the result
        assert (nlim >= 2).sum() >= N // 4 and (nlim >= 4).sum() > 0, np.bincount(nlim)
        assert run_case(case, joint_limits=0)[0] != digest, "the limit rows do not change the substep"
    else:
        assert (nlim == 0).all()
    if kind != "air":
        assert contacts > 0, "no contact rows: the case does not reach the sweep"
    assert digest == golden[case], f"{case}: state bits changed"


if __name__ == "__main__":
    if "--write" in sys.argv:
        out = {c: run_case(c)[0] for c in CASES}
        with open(GOLDEN_FILE, "w") as f:
            json.dump(out, f, indent=1, sort_keys=True)
            f.write("\n")
        print("wrote", GOLDEN_FILE)
    else:
        for c in CASES:
            digest, contacts, nlim = run_case(c)
            print(c, digest, contacts, np.bincount(nlim, minlength=5).tolist())
