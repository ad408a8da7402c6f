"""GPU: local-MIQP kernel through the C ABI vs the oracle (exhaustive leaf enumeration + exact QP).
Tolerances are BASELINE.json's: objective 1e-6 relative, inputs 1e-5, modes identical where the
optimum is unique (tests assert much tighter: 1e-9 / 1e-7)."""
import numpy as np
import pytest

import hybrid_vehicle_platoon_b200 as hvp
from gen_cases import platoon_local_problems

pytestmark = pytest.mark.gpu


def _check(r, ro):
    np.testing.assert_array_equal(r["status"], ro["status"])
    ok = ro["status"] == 2
    np.testing.assert_allclose(r["obj"][ok], ro["obj"][ok], rtol=1e-9)
    # inputs / states / region sequences are compared wherever the optimum is unique (second-best leaf
    # more than 1e-6 relative away -- BASELINE.json's own qualifier); two leaves whose objectives agree to
    # 1e-9 are both "the optimum" at the solvers' tolerances
    with np.errstate(invalid="ignore"):
        uniq = ok & ((ro["second"] - ro["obj"]) > 1e-6 * np.abs(ro["obj"]))
    assert uniq.sum() >= 0.9 * ok.sum()
    assert np.abs(r["u"][uniq] - ro["u"][uniq]).max() < 1e-7
    assert np.abs(r["x"][uniq] - ro["x"][uniq]).max() < 1e-6
    np.testing.assert_array_equal(r["modes"][uniq], ro["modes"][uniq])
    assert np.isinf(r["obj"][~ok]).all()


@pytest.mark.parametrize("N,n,stress,hetero,d0,t0,li,n_scen", [
    (6, 10, False, False, 50.0, 0.0, 0, 200),     # BASELINE config 2 shape
    (6, 10, True, True, 10.0, 3.0, 0, 200),
    (6, 10, True, True, 10.0, 3.0, 9, 100),       # leader at the back
    (4, 5, True, False, 50.0, 0.0, 2, 100),
    (5, 3, True, True, 10.0, 3.0, 1, 100),
    (8, 15, True, True, 10.0, 3.0, 0, 8),         # config-3 shape (n=15, N=8)
    (7, 10, False, True, 50.0, 0.0, 0, 20),
])
def test_matches_oracle(hvp_ctx, oracle, N, n, stress, hetero, d0, t0, li, n_scen):
    rng = np.random.default_rng(N * 100 + n + li)
    c = platoon_local_problems(rng, n_scen, n, N, li, stress, hetero)
    args = (N, c["flags"], c["mass"], c["x0"], c["xf"], c["xb"], c["xl"])
    r = hvp.local_miqp(*args, d0=d0, t0=t0, ctx=hvp_ctx)
    ro = oracle.local_miqp(*args, d0=d0, t0=t0)
    _check(r, ro)
    assert r["nodes"].mean() < ro["leaves"].mean()


def test_horizon_10(hvp_ctx, oracle):
    rng = np.random.default_rng(1)
    c = platoon_local_problems(rng, 4, 5, 10)
    args = (10, c["flags"], c["mass"], c["x0"], c["xf"], c["xb"], c["xl"])
    _check(hvp.local_miqp(*args, ctx=hvp_ctx), oracle.local_miqp(*args))


def test_infeasible_edge_and_tightening(hvp_ctx, oracle):
    N = 6
    k = np.arange(N + 1)
    xl = np.stack([3000 + 20.0 * k, np.full(N + 1, 20.0)])[None]
    edge = oracle.pwa_gear_system(800.0)[4][2]
    x0 = np.array([[3000.0, 1.0], [3000.0, edge], [3000.0, 45.84], [3000.0, 3.94], [9990.0, 30.0]])
    xls = np.repeat(xl, len(x0), 0)
    z = np.zeros_like(xls)
    for tight in (0.0, 0.2):
        r = hvp.local_miqp(N, 7, 800.0, x0, z, z, xls, tight=tight, ctx=hvp_ctx)
        ro = oracle.local_miqp(N, np.full(len(x0), 7), 800.0, x0, z, z, xls, tight=tight)
        _check(r, ro)
    assert r["status"][0] == 3


def test_empty_batch_and_bad_args(hvp_ctx):
    r = hvp.local_miqp(6, np.zeros(0, np.int32), np.zeros(0), np.zeros((0, 2)), ctx=hvp_ctx)
    assert r["u"].shape == (0, 6)
    with pytest.raises(RuntimeError, match="out of range"):
        hvp.local_miqp(40, 7, 800.0, np.zeros((1, 2)), ctx=hvp_ctx)


def test_bench_size_properties(hvp_ctx, oracle):
    """BASELINE size (4096 scenarios x 10 vehicles, N=6): every problem optimal; cost invariant under
    a common translation of all positions; subset agrees with the oracle."""
    rng = np.random.default_rng(1234 + 1)
    N, n, S = 6, 10, 4096
    c = platoon_local_problems(rng, S, n, N)
    args = (N, c["flags"], c["mass"], c["x0"])
    r = hvp.local_miqp(*args, c["xf"], c["xb"], c["xl"], ctx=hvp_ctx)
    assert (r["status"] == 2).all()
    sh = 64.0
    x0 = c["x0"].copy(); x0[:, 0] += sh
    xf, xb, xl = c["xf"].copy(), c["xb"].copy(), c["xl"].copy()
    for a in (xf, xb, xl):
        a[:, 0, :] += sh
    r2 = hvp.local_miqp(N, c["flags"], c["mass"], x0, xf, xb, xl, ctx=hvp_ctx)
    np.testing.assert_allclose(r2["obj"], r["obj"], rtol=1e-9)
    assert np.abs(r2["u"] - r["u"]).max() < 1e-7
    idx = rng.choice(S * n, 2000, replace=False)
    ro = oracle.local_miqp(N, c["flags"][idx], c["mass"][idx], c["x0"][idx], c["xf"][idx], c["xb"][idx],
                           c["xl"][idx])
    sub = {k: v[idx] for k, v in r.items() if isinstance(v, np.ndarray)}
    _check(sub, ro)


def test_chunked_host_path_equals_device_path():
    """Large host batches go through in chunks on side streams (hvp_local_miqp_host): same results as one device
    launch on the same inputs, remainder chunk included."""
    import torch
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import api
    from gen_cases import platoon_local_problems
    N, n, S = 6, 10, 40000 + 7                       # 400 070 problems: three chunks of 98 304 and a merged remainder
    cs = platoon_local_problems(np.random.default_rng(5), S, n, N)
    r = hvp.local_miqp(N, cs["flags"], cs["mass"], cs["x0"], cs["xf"], cs["xb"], cs["xl"])
    dev = torch.device("cuda", 0)
    B = S * n
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in cs.items()}
    u = torch.empty((B, N), dtype=torch.float64, device=dev); x = torch.empty((B, 2, N + 1), dtype=torch.float64, device=dev)
    mo = torch.empty((B, N), dtype=torch.int32, device=dev); ob = torch.empty(B, dtype=torch.float64, device=dev)
    st = torch.empty(B, dtype=torch.int32, device=dev); no = torch.empty(B, dtype=torch.int32, device=dev)
    api.local_miqp_device(api.local_desc(N), B, d["flags"], d["mass"], d["x0"], d["xf"], d["xb"], d["xl"], u, x, mo, ob, st, no,
                          None, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert (r["status"] == 2).all() and bool((st == 2).all())
    # Not bit-equal by design: in the tail of a launch idle lanes adopt open branches of busy ones, so WHICH lane solves
    # a leaf (and from which sequence of rank-1 updates of H^-1) depends on the launch shape -- round-off level
    # differences, and a different one of two leaves that tie within the 1e-9 acceptance threshold.
    assert np.allclose(r["obj"], ob.cpu().numpy(), rtol=1e-9, atol=0)
    du = np.abs(r["u"] - u.cpu().numpy()).max(axis=1)
    assert (du < 1e-6).mean() > 0.999, (du < 1e-6).mean()
    assert (np.abs(r["x"] - x.cpu().numpy()).max(axis=(1, 2)) < 1e-6).mean() > 0.999


# ---- solver options at the boundary (SURVEY.md 8b: mip_gap, time_limit, status 9) -----------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kernel_batch", [96, 12000])       # cooperative kernel / flat kernel
def test_mip_gap_and_time_limit_options(hvp_ctx, kernel_batch):
    """mip_gap > 0 prunes nodes whose bound is within the gap of the incumbent: fewer nodes, objective within the gap of
    the proven optimum; a time limit far below one tree's duration returns status 9 (or 2 / 3 for the problems that
    finished in time) and whatever it returns as a solution is feasible for the optimum's bound (obj >= optimum)."""
    rng = np.random.default_rng(5)
    S = kernel_batch // 10
    c = platoon_local_problems(rng, S, 10, 6, stress=True)
    args = (6, c["flags"], c["mass"], c["x0"], c["xf"], c["xb"], c["xl"])
    exact = hvp.local_miqp(*args, ctx=hvp_ctx)
    loose = hvp.local_miqp(*args, mip_gap=0.05, ctx=hvp_ctx)
    ok = exact["status"] == 2
    assert (loose["status"] == exact["status"]).all()
    assert (loose["obj"][ok] >= exact["obj"][ok] - 1e-9 * np.abs(exact["obj"][ok])).all()
    # Gurobi's definition: (incumbent - best bound) <= gap * |incumbent|, and the best bound is at most the optimum
    assert (loose["obj"][ok] - 0.05 * np.abs(loose["obj"][ok]) <= exact["obj"][ok] + 1e-9 * np.abs(exact["obj"][ok])).all()
    assert loose["nodes"].sum() < exact["nodes"].sum()
    timed = hvp.local_miqp(*args, time_limit_ms=1e-3, ctx=hvp_ctx)        # 1 microsecond per problem
    assert set(np.unique(timed["status"])) <= {2, 3, 9} and (timed["status"] == 9).any()
    has = np.isfinite(timed["obj"]) & ok
    assert (timed["obj"][has] >= exact["obj"][has] - 1e-9 * np.abs(exact["obj"][has])).all()
    with pytest.raises(RuntimeError):
        hvp.local_miqp(*args, mip_gap=-0.1, ctx=hvp_ctx)


@pytest.mark.gpu
def test_modes_hint_never_changes_the_optimum(hvp_ctx):
    """hvp_local_desc.modes_hint (MIP start): the optimal sequence itself, the shifted sequence, random sequences and
    garbage as hints all return the proven optimum of the un-hinted solve; a good hint cuts the node count."""
    import torch
    from hybrid_vehicle_platoon_b200 import api
    rng = np.random.default_rng(21)
    N, n, S = 6, 10, 1024                                   # 10 240 problems: the flat kernel
    c = platoon_local_problems(rng, S, n, N, stress=True)
    B = S * n
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d = {k: t(v) for k, v in c.items()}
    f64, i32 = torch.float64, torch.int32

    def solve(hint):
        u = torch.empty((B, N), dtype=f64, device=dev); x = torch.empty((B, 2, N + 1), dtype=f64, device=dev)
        mo = torch.empty((B, N), dtype=i32, device=dev); ob = torch.empty(B, dtype=f64, device=dev)
        st = torch.empty(B, dtype=i32, device=dev); no = torch.empty(B, dtype=i32, device=dev)
        api.local_miqp_device(api.local_desc(N), B, d["flags"], d["mass"], d["x0"], d["xf"], d["xb"], d["xl"], u, x, mo, ob, st,
                              no, None, ctx=hvp_ctx, stream=torch.cuda.current_stream().cuda_stream, modes_hint=hint)
        torch.cuda.synchronize()
        return dict(u=u.cpu().numpy(), modes=mo.cpu().numpy(), obj=ob.cpu().numpy(), status=st.cpu().numpy(), nodes=no.cpu().numpy())

    base = solve(None)
    ok = base["status"] == 2
    shifted = np.concatenate([base["modes"][:, 1:], base["modes"][:, -1:]], axis=1)
    hints = {"optimal": base["modes"], "shifted": shifted, "random": rng.integers(0, 7, (B, N)).astype(np.int32),
             "garbage": rng.integers(-5, 12, (B, N)).astype(np.int32)}
    for name, h in hints.items():
        r = solve(t(h.astype(np.int32)))
        assert (r["status"] == base["status"]).all(), name
        rel = np.abs(r["obj"][ok] - base["obj"][ok]) / np.maximum(1.0, np.abs(base["obj"][ok]))
        assert rel.max() < 1e-9, (name, rel.max(), int(rel.argmax()))
        if name == "optimal":
            assert r["nodes"][ok].mean() < base["nodes"][ok].mean(), (r["nodes"][ok].mean(), base["nodes"][ok].mean())


@pytest.mark.gpu
def test_more_streams_than_launch_slots(hvp_ctx):
    """The library keeps the launch state of the per-vehicle kernel (work counter, adoption scratch) per STREAM, for 64
    streams; a caller that keeps creating streams takes over the least recently used slot whose last launch has finished.
    90 distinct streams one after the other, then 8 of them in flight at once: every launch returns the first one's
    answers (objective to round-off -- adoption makes the order of incumbents timing-dependent -- statuses exactly).
    torch.cuda.Stream() hands out a pool of 32 streams round robin, so the streams are created with cudaStreamCreate."""
    import ctypes
    import torch
    from hybrid_vehicle_platoon_b200 import api
    torch.cuda.init()
    cudart = ctypes.CDLL("libcudart.so.12")
    rng = np.random.default_rng(33)
    N, n, S = 6, 10, 1024                                   # 10 240 problems: the flat kernel
    c = platoon_local_problems(rng, S, n, N, stress=True)
    B = S * n
    dev = torch.device("cuda", 0)
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in c.items()}
    f64, i32 = torch.float64, torch.int32

    def launch(stream):
        out = dict(u=torch.empty((B, N), dtype=f64, device=dev), x=torch.empty((B, 2, N + 1), dtype=f64, device=dev),
                   mo=torch.empty((B, N), dtype=i32, device=dev), ob=torch.empty(B, dtype=f64, device=dev),
                   st=torch.empty(B, dtype=i32, device=dev), no=torch.empty(B, dtype=i32, device=dev))
        with torch.cuda.stream(stream):
            api.local_miqp_device(api.local_desc(N), B, d["flags"], d["mass"], d["x0"], d["xf"], d["xb"], d["xl"], out["u"],
                                  out["x"], out["mo"], out["ob"], out["st"], out["no"], None, ctx=hvp_ctx, stream=stream.cuda_stream)
        return out

    torch.cuda.synchronize()
    base = launch(torch.cuda.current_stream())
    torch.cuda.synchronize()
    ok = base["st"] == 2

    def same(o):
        assert torch.equal(o["st"], base["st"])
        assert torch.allclose(o["ob"][ok], base["ob"][ok], rtol=1e-9, atol=0)

    handles, keep = [], []
    try:
        for _ in range(90):
            h = ctypes.c_void_p()
            assert cudart.cudaStreamCreate(ctypes.byref(h)) == 0
            handles.append(h)
            s = torch.cuda.ExternalStream(h.value, device=dev)
            keep.append(s)
            o = launch(s)
            s.synchronize()
            same(o)
        assert len({s.cuda_stream for s in keep}) > 64          # more streams than launch slots: the takeover runs
        outs = [launch(s) for s in keep[-8:]]                   # eight launches in flight, each on a stream of its own
        torch.cuda.synchronize()
        for o in outs:
            same(o)
    finally:
        torch.cuda.synchronize()
        for h in handles:
            cudart.cudaStreamDestroy(h)
