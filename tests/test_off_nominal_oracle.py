"""The reference solve at states off the nominal band (robot_gym.util.synthetic.make_off_nominal_states).

The GPU tests of these families (tests/test_gpu_off_nominal.py) take the C oracle as the reference and the numpy oracle
as the arbiter.  This pins, without a GPU, that the two agree there -- tilted and steep attitudes, fast bodies,
landing and lift-off, feet far out, coincident, colinear and at body height, all 16 contact patterns -- over the whole
horizon at h = 5, 10 and 20, and that the numpy solve verifies every env with its active-set polish.  Active sets here
reach 120 of 200 rows (every stance block at a corner of its friction pyramid)."""
import numpy as np
import pytest

from oracle import c_oracle, convex_mpc as cm
from robot_gym.model.robots.descriptions import GHOST
from robot_gym.util import synthetic

HEIGHT = GHOST.GetCtrlConstants().MPC_BODY_HEIGHT
ENVS = {5: 40, 10: 32, 20: 15}    # the numpy oracle takes ~0.3 s per env at h = 20


def test_families_are_seeded_float32_and_start_from_make_states():
    base = synthetic.make_states(64, GHOST, seed=5)
    far = synthetic.make_off_nominal_states(64, "feet_far", GHOST, seed=5)
    for name in ("com_velocity_body", "base_rpy", "base_rpy_rate", "command", "planned_contacts", "motor_angles"):
        assert getattr(far, name).tobytes() == getattr(base, name).tobytes(), name      # fields a family does not override
    assert far.foot_positions_base.tobytes() != base.foot_positions_base.tobytes()
    for family in synthetic.OFF_NOMINAL_FAMILIES:
        a = synthetic.make_off_nominal_states(64, family, GHOST, seed=5)
        b = synthetic.make_off_nominal_states(64, family, GHOST, seed=5)
        for name in ("com_velocity_body", "base_rpy", "base_rpy_rate", "foot_positions_base", "command",
                     "base_velocity_world", "base_orientation_xyzw", "planned_contacts"):
            x = getattr(a, name)
            assert x.dtype == getattr(base, name).dtype and x.shape == getattr(base, name).shape, (family, name)
            assert x.tobytes() == getattr(b, name).tobytes(), (family, name)
            assert np.all(np.isfinite(x.astype(np.float64))), (family, name)
        assert a.foot_positions_base.flags.c_contiguous
    with pytest.raises(ValueError):
        synthetic.make_off_nominal_states(4, "upside_down")
    pitch = synthetic.make_off_nominal_states(256, "steep_pitch", seed=1).base_rpy[:, 1]
    assert np.all((np.abs(pitch) >= 1.3) & (np.abs(pitch) <= 1.5)) and (pitch > 0).any() and (pitch < 0).any()
    pat = synthetic.make_off_nominal_states(32, "patterns", seed=1).planned_contacts
    assert len({tuple(r) for r in pat}) == 16
    co = synthetic.make_off_nominal_states(8, "feet_coincident", seed=1).foot_positions_base.reshape(8, 4, 3)
    assert np.array_equal(co[:, 3], co[:, 0]) and np.array_equal(co[:, 1], co[:, 2])


@pytest.mark.parametrize("horizon", [5, 10, 20])
@pytest.mark.parametrize("family", synthetic.OFF_NOMINAL_FAMILIES)
def test_c_oracle_matches_the_polished_numpy_oracle(family, horizon):
    n = ENVS[horizon]
    st = synthetic.make_off_nominal_states(n, family, GHOST, seed=300 + horizon)
    mp = cm.MpcParams(horizon=horizon)
    _, ref, _ = c_oracle.solve_batch(mp, st, HEIGHT, want_horizon=True)
    worst = 0.0
    for i in range(n):
        exact, info = cm.compute_contact_forces(
            mp, st.com_velocity_body[i].astype(np.float64), st.base_rpy[i].astype(np.float64),
            st.base_rpy_rate[i].astype(np.float64), st.planned_contacts[i], st.foot_positions_base[i].astype(np.float64),
            [0, 0, HEIGHT], [float(st.command[i, 0]), float(st.command[i, 1]), 0.0], [0, 0, 0],
            [0, 0, float(st.command[i, 2])], return_info=True)
        if not st.planned_contacts[i].any():
            assert np.all(exact == 0) and np.all(ref[i] == 0), (family, horizon, i)
            continue
        assert info.get("polished"), (family, horizon, i)
        rel = np.abs(ref[i].reshape(-1) - exact).max() / max(1.0, np.abs(exact).max())
        assert rel < 1e-6, (family, horizon, i, rel)
        worst = max(worst, rel)
    print(f"[{family} h={horizon}] C vs numpy oracle, worst relative {worst:.1e} over {n} envs")
