"""GPU: every launch route of the per-vehicle MIQP (csrc/local_miqp.cu launch_local_miqp) at every horizon it serves,
against the oracle (exhaustive leaf enumeration + exact QP) and, for batches too large for the oracle, against the host
build of the flat core (tests/host_harness, flat=True; itself checked against the oracle in test_host_flat_parity.py).

    route (automatic choice)                      taken when
    coop_split_kernel<8>                          N <= 8, batch <= 64, the stream has a launch slot, max_nodes == 0
    coop_miqp_kernel<8>, one problem per warp     N <= 8, batch <= 1184
    coop_miqp_kernel<8>, packed                   N <= 8, 1184 < batch < 8192
    coop_miqp_kernel<16>                          N >= 9 (N = 9 below 8192 only)
    flat_miqp_kernel<N,1,0> (adoption)            N = 4..9, batch >= 8192
    flat_miqp_kernel<N,0,0>                       no launch slot (capture on a stream the context has not seen)
    flat_miqp_kernel<N,1,1>                       modes_hint given

Routes that only an environment knob selects (HVP_LOCAL_KERNEL, HVP_FLAT_STEAL) are read once per process, so they run
in a subprocess (scripts/stress_local.py).  Adoption makes flat results depend on timing at round-off level: objectives
are compared to 1e-9 relative, inputs and region sequences only where the optimum is unique."""
import os
import subprocess
import sys

import numpy as np
import pytest

import harness
import hybrid_vehicle_platoon_b200 as hvp
from gen_cases import EDGES, platoon_local_problems

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIMITS = (3.94, 45.84)
ORACLE_SAMPLE = {2: 2000, 3: 2000, 4: 2000, 5: 2000, 6: 2000, 7: 1000, 8: 500, 9: 300, 10: 60, 11: 16, 12: 8}
TIGHT = {2: 0.3, 3: 0.2, 4: 0.1, 5: 0.1, 6: 0.05, 7: 0.05, 8: 0.02, 9: 0.02, 10: 0.01, 11: 0.0, 12: 0.0}


def _problems(seed, N, B, edge_share=0.1, role_share=0.05):
    """B stressed, heterogeneous problems (headway spacing is the caller's d0 / t0), the leader at the front, in the
    middle or at the back; a share of start velocities on or next to region edges and velocity limits or out of range
    (infeasible ones among them), and a share of problems with arbitrary role flags (flags = 5 included)."""
    rng = np.random.default_rng(seed)
    S = -(-B // 10)
    c = platoon_local_problems(rng, S, 10, N, int(rng.choice([0, 5, 9])), True, True)
    c = {k: np.ascontiguousarray(v[:B]) for k, v in c.items()}
    e = rng.random(B) < edge_share
    vals = np.concatenate([EDGES, LIMITS, [0.0, 1.0, 50.0]])
    c["x0"][e, 1] = rng.choice(vals, e.sum()) + rng.choice([0.0, 1e-12, -1e-12, 1e-9], e.sum())
    f = rng.random(B) < role_share
    c["flags"][f] = rng.integers(0, 8, f.sum())
    return c


def _args(N, c, idx=slice(None)):
    return (N, c["flags"][idx], c["mass"][idx], c["x0"][idx], c["xf"][idx], c["xb"][idx], c["xl"][idx])


def _vs_oracle(r, ro, min_opt=0.5):
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


def _vs_host(r, rh):
    """the whole batch against the host build of the same core: status exactly, objective to round-off (the device
    contracts FMAs, the host build does not)"""
    np.testing.assert_array_equal(r["status"], rh["status"])
    ok = rh["status"] == 2
    np.testing.assert_allclose(r["obj"][ok], rh["obj"][ok], rtol=1e-9, atol=1e-12)


def _sample(oracle, r, c, N, d0, t0, tight, seed, n=None):
    B = len(c["x0"])
    n = min(B, n or ORACLE_SAMPLE[N])
    idx = np.sort(np.random.default_rng(seed).choice(B, n, replace=False))
    ro = oracle.local_miqp(*_args(N, c, idx), d0=d0, t0=t0, tight=tight)
    return _vs_oracle({k: v[idx] for k, v in r.items() if isinstance(v, np.ndarray)}, ro)


# ---- flat_miqp_kernel<N,1,0>: batches of 8192 and more, every horizon -------------------------------------------
@pytest.mark.parametrize("N", [4, 5, 6, 7, 8, 9])
def test_flat_route_every_horizon(hvp_ctx, oracle, N):
    B = 8192 + 37
    c = _problems(1000 + N, N, B, edge_share=0.15)
    d0, t0, tight = 10.0, 3.0, TIGHT[N]
    r = hvp.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight, ctx=hvp_ctx)
    rh = harness.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight, flat=True)
    _vs_host(r, rh)
    assert (r["status"] == 3).mean() > 0.01                 # infeasible lanes beside long trees and adopters
    _sample(oracle, r, c, N, d0, t0, tight, seed=N)


# ---- coop_miqp_kernel<8>: one problem per warp and packed; coop_split_kernel<8> ------------------------------------
@pytest.mark.parametrize("N", [2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("B", [1, 10, 64, 300, 2000])      # split, split, split, one per warp, packed
def test_coop_routes(hvp_ctx, oracle, N, B):
    if N >= 8 and B == 2000:
        B = 1300                                             # still packed (> 1184); the oracle's share stays small
    c = _problems(2000 + 10 * N + B, N, B)
    d0, t0, tight = 10.0, 3.0, TIGHT[N]
    r = hvp.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight, ctx=hvp_ctx)
    if B > ORACLE_SAMPLE[N]:
        rh = harness.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight, coop=True)
        _vs_host(r, rh)
        _sample(oracle, r, c, N, d0, t0, tight, seed=N)
    else:
        ro = oracle.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight)
        _vs_oracle(r, ro, min_opt=0.3 if B >= 10 else 0.0)


def test_coop_packed_short_horizons_at_flat_sizes(hvp_ctx, oracle):
    """N = 2, 3 have no flat instantiation: 8192 problems and more stay on the packed cooperative kernel"""
    for N in (2, 3):
        c = _problems(2100 + N, N, 9000)
        r = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, tight=TIGHT[N], ctx=hvp_ctx)
        _vs_host(r, harness.local_miqp(*_args(N, c), d0=10.0, t0=3.0, tight=TIGHT[N], coop=True))
        _sample(oracle, r, c, N, 10.0, 3.0, TIGHT[N], seed=N, n=1000)


# ---- coop_miqp_kernel<16>: N = 9..12 -------------------------------------------------------------------------------
@pytest.mark.parametrize("N,B", [(9, 300), (10, 60), (11, 16), (12, 4)])
def test_coop16_long_horizons(hvp_ctx, oracle, N, B):
    c = _problems(3000 + N, N, B, edge_share=0.05)
    d0, t0, tight = 10.0, 3.0, TIGHT[N]
    r = hvp.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight, ctx=hvp_ctx)
    ro = oracle.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight)
    _vs_oracle(r, ro)


def test_coop16_at_flat_sizes(hvp_ctx, oracle):
    """N = 10 at 8192 problems: no flat instantiation, so the packed coop<16> kernel.  (The host coop core needs ~50 ms
    a problem at N = 10: the first 600 are compared with the one-problem-per-warp route instead, a sample with the
    oracle.)"""
    N, B = 10, 8192
    c = _problems(3100, N, B, edge_share=0.05)
    r = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, tight=TIGHT[N], ctx=hvp_ctx)
    head = slice(0, 600)
    _vs_host({k: v[head] for k, v in r.items() if isinstance(v, np.ndarray)},
             hvp.local_miqp(*_args(N, c, head), d0=10.0, t0=3.0, tight=TIGHT[N], ctx=hvp_ctx))
    _sample(oracle, r, c, N, 10.0, 3.0, TIGHT[N], seed=N, n=40)


# ---- flat_miqp_kernel<N,0,0>: no launch slot (capture on a stream the context has never seen) ----------------------
def _device(c, dev):
    import torch
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in c.items()}


def _outputs(B, N, dev):
    import torch
    f64, i32 = torch.float64, torch.int32
    return dict(u=torch.empty((B, N), dtype=f64, device=dev), x=torch.empty((B, 2, N + 1), dtype=f64, device=dev),
                modes=torch.empty((B, N), dtype=i32, device=dev), obj=torch.empty(B, dtype=f64, device=dev),
                status=torch.empty(B, dtype=i32, device=dev), nodes=torch.empty(B, dtype=i32, device=dev))


def _host(o):
    return {k: v.cpu().numpy() for k, v in o.items()}


@pytest.mark.parametrize("N,B", [(6, 8192 + 5), (9, 8192), (5, 48)])
def test_captured_solve_without_launch_slot(oracle, N, B):
    """A new context has no launch slots; a solve captured on a fresh stream gets none (nothing is allocated during
    capture), so it runs without adoption scratch: flat<N,0,0> for 8192 problems and more, the one-problem-per-warp
    cooperative kernel instead of the split for 64 or fewer.  Two replays agree with the eager solve and the oracle."""
    import torch
    from hybrid_vehicle_platoon_b200 import api
    dev = torch.device("cuda", 0)
    ctx = hvp.Context(0)
    try:
        c = _problems(4000 + N, N, B)
        d0, t0, tight = 10.0, 3.0, TIGHT[N]
        eager = hvp.local_miqp(*_args(N, c), d0=d0, t0=t0, tight=tight, ctx=ctx)      # the context's own stream
        d = _device(c, dev)
        out = _outputs(B, N, dev)
        desc = api.local_desc(N, d0, t0, tight)
        s = torch.cuda.Stream(device=dev)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            api.local_miqp_device(desc, B, d["flags"], d["mass"], d["x0"], d["xf"], d["xb"], d["xl"], out["u"], out["x"],
                                  out["modes"], out["obj"], out["status"], out["nodes"], None, ctx=ctx,
                                  stream=torch.cuda.current_stream().cuda_stream)
        for _ in range(2):
            for v in out.values():
                v.fill_(-7)
            g.replay()
            torch.cuda.synchronize()
            r = _host(out)
            _vs_host(r, eager)
            _sample(oracle, r, c, N, d0, t0, tight, seed=N, n=min(B, 300))
        del g
    finally:
        torch.cuda.synchronize()
        ctx.close()


# ---- flat_miqp_kernel<N,1,1>: MIP start ---------------------------------------------------------------------------
@pytest.mark.parametrize("N", [4, 5, 6, 7, 8, 9])
def test_hint_every_flat_horizon(hvp_ctx, oracle, N):
    """optimal, shifted, random and garbage hints: the proven optimum of the un-hinted solve, status for status"""
    import torch
    from hybrid_vehicle_platoon_b200 import api
    dev = torch.device("cuda", 0)
    B = 8192
    c = _problems(5000 + N, N, B)
    d0, t0, tight = 10.0, 3.0, TIGHT[N]
    d = _device(c, dev)
    desc = api.local_desc(N, d0, t0, tight)
    rng = np.random.default_rng(N)

    def solve(hint):
        o = _outputs(B, N, dev)
        api.local_miqp_device(desc, B, d["flags"], d["mass"], d["x0"], d["xf"], d["xb"], d["xl"], o["u"], o["x"],
                              o["modes"], o["obj"], o["status"], o["nodes"], None, ctx=hvp_ctx,
                              stream=torch.cuda.current_stream().cuda_stream,
                              modes_hint=None if hint is None else torch.from_numpy(hint.astype(np.int32)).to(dev))
        torch.cuda.synchronize()
        return _host(o)

    base = solve(None)
    shifted = np.concatenate([base["modes"][:, 1:], base["modes"][:, -1:]], axis=1)
    n = min(B, ORACLE_SAMPLE[N])
    idx = np.sort(rng.choice(B, n, replace=False))
    ro = oracle.local_miqp(*_args(N, c, idx), d0=d0, t0=t0, tight=tight)
    for name, h in (("optimal", base["modes"]), ("shifted", shifted), ("random", rng.integers(0, 7, (B, N))),
                    ("garbage", rng.integers(-5, 12, (B, N)))):
        r = solve(h)
        _vs_host(r, base)
        _vs_oracle({k: v[idx] for k, v in r.items()}, ro)


# ---- solver options per route ----------------------------------------------------------------------------------
def _gap_ok(loose, exact, gap):
    ok = exact["status"] == 2
    np.testing.assert_array_equal(loose["status"], exact["status"])
    tol = 1e-9 * np.abs(exact["obj"][ok])
    assert (loose["obj"][ok] >= exact["obj"][ok] - tol).all()
    assert (loose["obj"][ok] - gap * np.abs(loose["obj"][ok]) <= exact["obj"][ok] + tol).all()


@pytest.mark.parametrize("B", [40, 9000])                    # coop_split / flat
def test_mip_gap_per_route(hvp_ctx, B):
    N = 7
    c = _problems(6000 + B, N, B)
    exact = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, ctx=hvp_ctx)
    loose = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, mip_gap=0.05, ctx=hvp_ctx)
    _gap_ok(loose, exact, 0.05)
    assert loose["nodes"].sum() < exact["nodes"].sum()


@pytest.mark.parametrize("B", [40, 9000])                    # one-problem-per-warp coop (no split) / flat without adoption
def test_node_limit_per_route(hvp_ctx, B):
    """max_nodes > 0 turns the split and the adoption off: the budgeted search ends with status 5 (node limit) and its
    incumbent (HVP_NODE_LIMIT = 8), or proves the optimum (2) / infeasibility (3) within the budget"""
    N = 7
    c = _problems(6100 + B, N, B)
    exact = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, ctx=hvp_ctx)
    lim = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, max_nodes=3, ctx=hvp_ctx)
    assert set(np.unique(lim["status"])) <= {2, 3, 8} and (lim["status"] == 8).any()
    ok = exact["status"] == 2
    done = lim["status"] == 2
    np.testing.assert_allclose(lim["obj"][done], exact["obj"][done], rtol=1e-9)
    assert (exact["status"][lim["status"] == 3] == 3).all()
    has = np.isfinite(lim["obj"]) & ok
    assert (lim["obj"][has] >= exact["obj"][has] - 1e-9 * np.abs(exact["obj"][has])).all()
    full = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, max_nodes=1 << 30, ctx=hvp_ctx)
    np.testing.assert_array_equal(full["status"], exact["status"])
    np.testing.assert_allclose(full["obj"][ok], exact["obj"][ok], rtol=1e-9)


# ---- time limit: one problem, one budget, and an honest status -------------------------------------------------------
def time_limit_invariant(ctx, N, B, limits=(0.01, 0.03, 0.1, 0.3, 1.0), seed=7000):
    """For every problem and every limit: status 2 => the proven optimum (1e-9 relative); 3 => really infeasible;
    9 => obj >= optimum or inf; nothing else.  Returns the status counts per limit."""
    c = _problems(seed + N + B, N, B, edge_share=0.02)
    exact = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, ctx=ctx)
    ok = exact["status"] == 2
    assert set(np.unique(exact["status"])) <= {2, 3}
    counts = {}
    for ms in limits:
        r = hvp.local_miqp(*_args(N, c), d0=10.0, t0=3.0, time_limit_ms=ms, ctx=ctx)
        st = r["status"]
        assert set(np.unique(st)) <= {2, 3, 9}, (ms, np.unique(st))
        two = st == 2
        assert ok[two].all(), ms
        bad = np.abs(r["obj"][two] - exact["obj"][two]) > 1e-9 * np.maximum(1.0, np.abs(exact["obj"][two]))
        assert not bad.any(), (ms, int(bad.sum()), int(np.nonzero(two)[0][bad][0]))
        assert (~ok[st == 3]).all(), ms
        nine = (st == 9) & np.isfinite(r["obj"])
        assert (r["obj"][nine] >= exact["obj"][nine] - 1e-9 * np.abs(exact["obj"][nine])).all(), ms
        assert ok[nine].all(), ms
        counts[ms] = {int(s): int((st == s).sum()) for s in (2, 3, 9)}
    return counts


@pytest.mark.parametrize("N,B", [(9, 16384), (6, 48), (6, 600)])       # flat with adoption / coop_split / coop
def test_time_limit_invariant(hvp_ctx, N, B):
    counts = time_limit_invariant(hvp_ctx, N, B)
    print(N, B, counts)
    assert any(v.get(9, 0) for v in counts.values())         # the ladder reaches problems that run out of time


# ---- forced routes (environment knobs are read once per process) ----------------------------------------------------
@pytest.mark.parametrize("steal", ["1", "0"])
def test_forced_route_campaign(steal):
    """HVP_LOCAL_KERNEL=flat puts small batches on the flat kernel, where nearly every tree is searched with adopters;
    with HVP_FLAT_STEAL=0 as well they run on flat<N,0,0>.  N = 4..9 against the oracle."""
    env = dict(os.environ, HVP_LOCAL_KERNEL="flat", HVP_FLAT_STEAL=steal)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "stress_local.py"), "11", "--scale", "0.25"],
                       env=env, capture_output=True, text=True, timeout=300)
    print(p.stdout[-3000:], p.stderr[-2000:])
    assert p.returncode == 0 and "failures: 0" in p.stdout
