"""Parity against the REAL reference (gurobipy + dmpcpwa + the reference sources), wherever those exist.
SURVEY.md 8c: the MIQP half of the path is "parity unpinned" in this container (no Gurobi, no dmpcpwa, no
network); this test closes the pin automatically on a box that has them:
    HVP_REFERENCE_DIR=/path/to/hybrid-vehicle-platoon python -m pytest tests/test_live_gurobi.py -m gpu
It is skipped everywhere else: without gurobipy, without dmpcpwa, or without HVP_REFERENCE_DIR naming a checkout of
the reference.  Tolerances are BASELINE.json's: objective 1e-6 relative, inputs 1e-5."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REF = os.environ.get("HVP_REFERENCE_DIR")


@pytest.fixture(scope="module")
def ref():
    pytest.importorskip("gurobipy")
    pytest.importorskip("dmpcpwa")
    if not REF or not os.path.isdir(REF):
        pytest.skip("HVP_REFERENCE_DIR does not name a checkout of the reference sources")
    sys.path.insert(0, REF)
    import fleet_decent_mld as ref_decent        # the reference's own module
    import models as ref_models
    from misc.spacing_policy import ConstantSpacingPolicy
    return ref_decent, ref_models, ConstantSpacingPolicy


@pytest.mark.parametrize("role", ["leader_front", "interior", "trailer"])
def test_local_miqp_vs_gurobi(ref, role):
    ref_decent, ref_models, RefSpacing = ref
    import hybrid_vehicle_platoon_b200 as hvp
    N, ts = 6, 1.0
    system = ref_models.Platoon(1, "pwa_gear", [800.0]).get_vehicle_system_dicts(ts)[0]
    kw = dict(is_front=role == "leader_front", is_leader=role == "leader_front", is_trailer=role == "trailer")
    gmpc = ref_decent.LocalMpcMld(N, system, RefSpacing(50), True, kw["is_front"], kw["is_leader"], kw["is_trailer"],
                                  1, 0.0, False)
    ours = hvp.LocalMpcMld(N, hvp.Platoon(1, "pwa_gear", [800.0]).get_vehicle_system_dicts(ts)[0],
                           hvp.ConstantSpacingPolicy(50), True, kw["is_front"], kw["is_leader"], kw["is_trailer"])
    rng = np.random.default_rng(42)
    k = np.arange(N + 1)
    for _ in range(25):
        v = rng.uniform(6, 33); p = rng.uniform(500, 2500)
        state = np.array([[p], [v]])
        mk = lambda dp, dv: np.stack([p + dp + (v + dv) * k, np.full(N + 1, v + dv)])
        xf, xb, xl = mk(rng.uniform(40, 120), rng.uniform(-3, 3)), mk(-rng.uniform(40, 120), rng.uniform(-3, 3)), \
            mk(rng.uniform(-20, 20), rng.uniform(-3, 3))
        for m in (gmpc, ours):
            m.set_x_front(xf); m.set_x_back(xb); m.set_leader_x(xl)
        ug, ig = gmpc.solve_mpc(state, raises=False)
        uo, io = ours.solve_mpc(state, raises=False)
        assert np.isinf(ig["cost"]) == np.isinf(io["cost"])
        if np.isinf(ig["cost"]):
            continue
        assert abs(io["cost"] - ig["cost"]) <= 1e-6 * max(1.0, abs(ig["cost"]))
        assert np.abs(io["u"] - ig["u"]).max() < 1e-5
        assert np.abs(io["x"] - ig["x"]).max() < 1e-4


def test_cent_miqp_vs_gurobi(ref):
    _, ref_models, RefSpacing = ref
    from mpcs.cent_mld import MpcMldCent as RefCent
    import hybrid_vehicle_platoon_b200 as hvp
    n, N, ts = 3, 5, 1.0
    gmpc = RefCent(n, N, ref_models.Platoon(n, "pwa_gear", [800.0] * n).get_vehicle_system_dicts(ts), RefSpacing(50), 0, True, 1)
    ours = hvp.MpcMldCent(n, N, hvp.Platoon(n, "pwa_gear", [800.0] * n).get_vehicle_system_dicts(ts),
                          hvp.ConstantSpacingPolicy(50), 0, True)
    rng = np.random.default_rng(43)
    k = np.arange(N + 1)
    for _ in range(10):
        v = rng.uniform(8, 30, n); p = 3000.0 - np.cumsum(rng.uniform(40, 140, n))
        state = np.stack([p, v], 1).reshape(2 * n, 1)
        lead = np.stack([p[0] + rng.uniform(-20, 20) + 20.0 * k, np.full(N + 1, 20.0)])
        gmpc.set_leader_traj(lead); ours.set_leader_traj(lead)
        ug, ig = gmpc.solve_mpc(state, raises=False)
        uo, io = ours.solve_mpc(state, raises=False)
        assert np.isinf(ig["cost"]) == np.isinf(io["cost"])
        if np.isfinite(ig["cost"]):
            assert abs(io["cost"] - ig["cost"]) <= 1e-6 * max(1.0, abs(ig["cost"]))
            assert np.abs(io["u"] - ig["u"]).max() < 1e-5
