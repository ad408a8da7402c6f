"""CPU: the host build of the flat kernel's core (csrc/flat_core.cuh, the code every flat_miqp_kernel instantiation and
the CPU port compile) against the oracle's exhaustive leaf enumeration, at every horizon the flat kernel serves and
beyond, on the distributions and edges where the search goes wrong: stressed and heterogeneous platoons, headway
spacing, tightened acceleration rows, the leader anywhere in the platoon, start velocities on and next to the region
edges and outside the velocity range, and all eight role combinations -- the cooperative and scalar cores included."""
import numpy as np
import pytest

import harness
from gen_cases import EDGES, platoon_local_problems

LIMITS = (3.94, 45.84)                      # velocity range of the vehicle model (vmin, vmax)


def _compare(r, ro, min_opt=0.0):
    """status exactly, objective to 1e-9 relative; inputs, states and region sequences where the optimum is unique
    (second-best leaf more than 1e-6 relative away)."""
    np.testing.assert_array_equal(r["status"], ro["status"])
    ok = ro["status"] == 2
    assert ok.mean() >= min_opt, ok.mean()
    np.testing.assert_allclose(r["obj"][ok], ro["obj"][ok], rtol=1e-9, atol=1e-12)
    assert np.isinf(r["obj"][~ok]).all()
    with np.errstate(invalid="ignore"):
        uniq = ok & ((ro["second"] - ro["obj"]) > 1e-6 * np.abs(ro["obj"]))
    if uniq.any():
        assert np.abs(r["u"][uniq] - ro["u"][uniq]).max() < 1e-7
        assert np.abs(r["x"][uniq] - ro["x"][uniq]).max() < 1e-6
        np.testing.assert_array_equal(r["modes"][uniq], ro["modes"][uniq])
    return ok


# (N, scenarios of 10 vehicles, leader index, stress, heterogeneous masses, d0, t0, tightening).  Tightening shrinks
# with N: at N = 9 a tightening of 0.3 leaves no stressed problem feasible.
CASES = [
    (2, 40, 0, True, True, 10.0, 3.0, 0.3),
    (3, 40, 5, True, True, 10.0, 3.0, 0.2),
    (4, 30, 9, True, True, 10.0, 3.0, 0.0),
    (5, 30, 0, True, False, 50.0, 0.0, 0.2),
    (6, 30, 5, True, True, 10.0, 3.0, 0.1),
    (6, 20, 9, False, False, 50.0, 0.0, 0.0),
    (7, 20, 9, True, True, 10.0, 3.0, 0.05),
    (8, 10, 0, True, True, 10.0, 3.0, 0.02),
    (9, 6, 5, True, True, 10.0, 3.0, 0.0),
    (9, 4, 9, False, True, 50.0, 0.0, 0.01),
]


@pytest.mark.parametrize("N,S,li,stress,hetero,d0,t0,tight", CASES)
def test_flat_core_matches_oracle(oracle, N, S, li, stress, hetero, d0, t0, tight):
    rng = np.random.default_rng(700 + 10 * N + li)
    c = platoon_local_problems(rng, S, 10, N, li, stress, hetero)
    args = (N, c["flags"], c["mass"], c["x0"], c["xf"], c["xb"], c["xl"])
    ro = oracle.local_miqp(*args, d0=d0, t0=t0, tight=tight)
    r = harness.local_miqp(*args, d0=d0, t0=t0, tight=tight, flat=True)
    _compare(r, ro, min_opt=0.5)


def _edge_velocities(rng, B):
    vals = np.concatenate([EDGES, LIMITS, [0.0, 1.0, 50.0]])
    jitter = np.array([0.0, 1e-12, -1e-12, 1e-9])
    return rng.choice(vals, B) + rng.choice(jitter, B)


@pytest.mark.parametrize("N,S", [(2, 12), (3, 12), (4, 12), (5, 12), (6, 12), (7, 8), (8, 4), (9, 3)])
@pytest.mark.parametrize("kind", ["flat", "coop"])
def test_region_edge_start_velocities(oracle, N, S, kind):
    """v0 exactly on a region edge or a velocity limit (where two regions, or none, contain it), 1e-12 on either side
    and 1e-9 above, and out of range (0, 1, 50): a third of these problems are infeasible, the rest branch at
    the root."""
    rng = np.random.default_rng(40 + N)
    c = platoon_local_problems(rng, S, 10, N, int(rng.integers(0, 10)), True, True)
    x0 = c["x0"].copy()
    x0[:, 1] = _edge_velocities(rng, len(x0))
    for tight in (0.0, 0.1):
        args = (N, c["flags"], c["mass"], x0, c["xf"], c["xb"], c["xl"])
        ro = oracle.local_miqp(*args, d0=10.0, t0=3.0, tight=tight)
        r = harness.local_miqp(*args, d0=10.0, t0=3.0, tight=tight, flat=kind == "flat", coop=kind == "coop")
        ok = _compare(r, ro, min_opt=0.3)
        assert (~ok).mean() > 0.1                      # the infeasible side is exercised


@pytest.mark.parametrize("N", [4, 6])
@pytest.mark.parametrize("flags", range(8))
@pytest.mark.parametrize("kind", ["flat", "coop", "scalar"])
def test_every_role_combination(oracle, N, flags, kind):
    """All eight FRONT|LEADER|TRAILER combinations on one batch of stressed problems.  flags = 5 (front and trailer,
    not the leader: a one-vehicle platoon whose leader reference is off) has no tracking term and no neighbour rows;
    its objective is the input cost alone, 0 wherever u = 0 is feasible."""
    rng = np.random.default_rng(90 + N)
    c = platoon_local_problems(rng, 12, 10, N, 0, True, True)
    f = np.full(len(c["x0"]), flags, np.int32)
    args = (N, f, c["mass"], c["x0"], c["xf"], c["xb"], c["xl"])
    ro = oracle.local_miqp(*args, d0=10.0, t0=3.0)
    r = harness.local_miqp(*args, d0=10.0, t0=3.0, flat=kind == "flat", coop=kind == "coop")
    _compare(r, ro, min_opt=0.9)


@pytest.mark.parametrize("N", [4, 6, 9])
@pytest.mark.parametrize("kind", ["flat", "coop", "scalar"])
def test_unread_references_may_be_null(oracle, N, kind):
    """NULL for the references a role never reads: all three for flags = 5, xf and xb for flags = 7 (front, leader
    and trailer).  Same answers as the oracle, whose zeros stand in for the missing arrays."""
    rng = np.random.default_rng(60 + N)
    c = platoon_local_problems(rng, 6 if N < 9 else 2, 10, N, 0, True, True)
    B = len(c["x0"])
    for flags, refs in ((5, (None, None, None)), (7, (None, None, c["xl"]))):
        f = np.full(B, flags, np.int32)
        ro = oracle.local_miqp(N, f, c["mass"], c["x0"], *refs, d0=10.0, t0=3.0)
        r = harness.local_miqp(N, f, c["mass"], c["x0"], *refs, d0=10.0, t0=3.0, flat=kind == "flat", coop=kind == "coop")
        _compare(r, ro, min_opt=0.9)
        if flags == 5:
            assert (ro["obj"][ro["status"] == 2] >= 0).all()
