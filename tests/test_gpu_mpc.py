"""GPU parity of the compiled-MPC kernel (csrc/pm_kernel.cu through include/hvp.h hvp_mpc_*) against the
CPU oracle (oracle/hvp_oracle_mpc.c) on the same seeded inputs.  Tolerances: objective 1e-8 relative
(BASELINE.json asks 1e-6), inputs 1e-6 (asks 1e-5), mode sequences identical where the optimum is unique."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import oracle as O
import gen_mpc_cases as G


def _compare(r, ro, what, check_modes=True):
    assert (r["status"] == ro["status"]).all(), (what, r["status"], ro["status"])
    ok = ro["status"] == 2
    assert np.allclose(r["obj"][ok], ro["obj"][ok], rtol=1e-8, atol=1e-7), (what, np.abs(r["obj"][ok] - ro["obj"][ok]).max())
    assert np.abs(r["u"][ok] - ro["u"][ok]).max() < 1e-6, (what, np.abs(r["u"][ok] - ro["u"][ok]).max())
    assert np.abs(r["x"][ok] - ro["x"][ok]).max() < 1e-6, what
    if r["extra"].size:
        assert np.abs(r["extra"][ok] - ro["extra"][ok]).max() < 1e-5, what
    if check_modes:
        uniq = ok & (ro["second"] - ro["obj"] > 1e-6 * np.maximum(1.0, np.abs(ro["obj"])))
        assert (r["modes"][uniq] == ro["modes"][uniq]).all(), what


@pytest.fixture(scope="module")
def hvp():
    import hybrid_vehicle_platoon_b200 as h
    return h


@pytest.mark.parametrize("n,N,stress,t0", [(2, 3, False, 0.0), (3, 3, True, 0.0), (2, 4, True, 3.0), (3, 5, False, 0.0)])
def test_cent_vs_oracle(hvp, n, N, stress, t0):
    rng = np.random.default_rng(100 + n * 10 + N)
    B = 24
    x0, params = G.cent_cases(rng, B, n, N, stress)
    d0 = 10.0 if t0 else 50.0
    mpc = hvp.api.CompiledMpc(G.CENT, N, n_local=n, d0=d0, t0=t0)
    r = mpc.solve(x0, 800.0, params)
    exhaustive = n * N <= 9
    ro = O.mpc_solve(O.CENT, n, N, x0, 800.0, params, d0=d0, t0=t0, method=0 if exhaustive else 1)
    _compare(r, ro, f"cent n={n} N={N}")
    assert (r["nodes"] > 0).all()


@pytest.mark.parametrize("nf,nb,rl,N,t0", [(0, 1, 0, 4, 0.0), (1, 1, 1, 3, 0.0), (2, 2, O.NO_LEADER, 3, 3.0),
                                           (2, 0, -1 + 1, 4, 0.0), (1, 2, -1, 3, 0.0)])
def test_event_vs_oracle(hvp, nf, nb, rl, N, t0):
    rng = np.random.default_rng(200 + nf * 7 + nb * 3 + N)
    B = 24
    nl = (nf > 0) + 1 + (nb > 0)
    x0, params = G.event_cases(rng, B, nf, nb, N, stress=True)
    d0 = 10.0 if t0 else 50.0
    mpc = hvp.api.CompiledMpc(G.EVENT, N, n_local=nl, leader_index=rl, n_front=nf, n_behind=nb, d0=d0, t0=t0)
    r = mpc.solve(x0, 800.0, params)
    ro = O.mpc_solve(O.EVENT, nl, N, x0, 800.0, params, leader_index=rl, n_front=nf, n_behind=nb, d0=d0, t0=t0,
                     method=0 if nl * N <= 9 else 1)
    _compare(r, ro, f"event nf={nf} nb={nb}")


@pytest.mark.parametrize("flags,N", [(0, 4), (G.FRONT | G.LEADER, 4), (G.TRAILER, 5), (G.LEADER, 3), (0, 8)])
def test_admm_vs_oracle(hvp, flags, N):
    rng = np.random.default_rng(300 + flags * 5 + N)
    B = 16
    x0, params = G.admm_cases(rng, B, N, stress=True)
    mass = rng.uniform(700, 1000, (B, 1))
    mpc = hvp.api.CompiledMpc(G.ADMM, N, flags=flags, rho=0.5)
    r = mpc.solve(x0, mass, params)
    ro = O.mpc_solve(O.ADMM, 1, N, x0, mass, params, flags=flags, rho=0.5, method=0 if N <= 5 else 1)
    _compare(r, ro, f"admm flags={flags} N={N}")


@pytest.mark.parametrize("nf,nb,leader,N", [(0, 1, True, 6), (1, 1, False, 8), (1, 0, False, 5)])
def test_gadmm_fixed_mode_qp_vs_oracle(hvp, nf, nb, leader, N):
    rng = np.random.default_rng(400 + nf + 2 * nb + N)
    B = 32
    x0, params, modes = G.gadmm_cases(rng, B, nf, nb, N)
    flags = G.LEADER if leader else 0
    mpc = hvp.api.CompiledMpc(G.GADMM, N, flags=flags, n_front=nf, n_behind=nb, rho=0.5)
    r = mpc.solve(x0, 800.0, params, fixed_modes=modes)
    ro = O.mpc_solve(O.GADMM, 1, N, x0, 800.0, params, flags=flags, n_front=nf, n_behind=nb, rho=0.5,
                     fixed_modes=modes)
    _compare(r, ro, f"gadmm nf={nf} nb={nb}", check_modes=False)
    assert (r["nodes"][r["status"] == 2] == 1).all()
    assert (ro["status"] == 2).sum() >= B // 2


@pytest.mark.parametrize("kind,nl,N", [(G.LOCAL, 1, 5), (G.CENT, 2, 3), (G.ADMM, 1, 4)])
def test_friction_gear_model_vs_oracle(hvp, kind, nl, N):
    """MpcGear variants: pwa_friction model with six discrete gears (mpcs/mpc_gear.py:30-135)."""
    rng = np.random.default_rng(500 + kind * 3 + N)
    B = 24
    if kind == G.CENT:
        x0, params = G.cent_cases(rng, B, nl, N, stress=True)
        flags = 0
    elif kind == G.ADMM:
        x0, params = G.admm_cases(rng, B, N, stress=True)
        flags = 0
    else:
        full = G.platoon_states(rng, B, 3, stress=True)
        x0 = full[:, 1:2]
        lead = x0[:, 0] + [30.0, 2.0]
        params = np.concatenate([G.const_vel(a, N).reshape(B, -1) for a in (full[:, 0], full[:, 2], lead)], axis=1)
        flags = 0
    mpc = hvp.api.CompiledMpc(kind, N, n_local=nl, model=1, flags=flags)
    assert mpc.n_modes == 12
    r = mpc.solve(x0, 800.0, params)
    ro = O.mpc_solve(kind, nl, N, x0, 800.0, params, model=1, flags=flags, method=0 if nl * N <= 6 else 1)
    _compare(r, ro, f"gear kind={kind}")
    ok = ro["status"] == 2
    gears = mpc.gears(r["modes"])
    assert ((gears[ok] >= 1) & (gears[ok] <= 6)).all()
    # the chosen gear's window contains the predicted velocity (mpc_gear.py:101-110)
    vl = np.array([3.94, 5.43, 7.56, 9.96, 13.70, 19.10]); vh = np.array([9.46, 13.04, 18.15, 23.90, 32.93, 45.84])
    v = r["x"][:, :, 1, :N]
    assert (v[ok] >= vl[gears[ok] - 1] - 1e-6).all() and (v[ok] <= vh[gears[ok] - 1] + 1e-6).all()


def test_local_kind_matches_local_kernel(hvp):
    """The compiled LOCAL formulation and the specialised per-vehicle kernel solve the same problem, for every role
    combination.  flags = 5 (front and trailer, not the leader) has no tracking term at all: the per-vehicle kernel
    solves it (test_host_flat_parity.py, test_gpu_local_routes.py); the compiled formulation, built on a positive
    definite tracking Hessian, refuses it when it is created instead of returning wrong answers."""
    from gen_cases import platoon_local_problems
    rng = np.random.default_rng(77)
    N, n = 6, 10
    cs = platoon_local_problems(rng, 4, n, N, stress=True, hetero=True)
    B = len(cs["x0"])
    params = np.concatenate([cs[k].reshape(B, -1) for k in ("xf", "xb", "xl")], axis=1)
    with pytest.raises(RuntimeError, match="not positive definite"):
        hvp.api.CompiledMpc(G.LOCAL, N, flags=5)
    for fl in (0, 1, 2, 3, 4, 6, 7):
        r = hvp.local_miqp(N, np.full(B, fl, np.int32), cs["mass"], cs["x0"], cs["xf"], cs["xb"], cs["xl"])
        mpc = hvp.api.CompiledMpc(G.LOCAL, N, flags=fl)
        g = mpc.solve(cs["x0"][:, None, :], cs["mass"][:, None], params)
        assert (g["status"] == r["status"]).all(), fl
        ok = g["status"] == 2
        assert ok.mean() > 0.9, fl
        assert np.allclose(g["obj"][ok], r["obj"][ok], rtol=1e-9), fl
        assert np.abs(g["u"][ok][:, 0] - r["u"][ok]).max() < 1e-7, fl


def test_mpc_edge_cases(hvp):
    mpc = hvp.api.CompiledMpc(G.CENT, 3, n_local=2)
    # empty batch
    r = mpc.solve(np.zeros((0, 2, 2)), np.zeros((0, 2)), np.zeros((0, mpc.n_param)))
    assert r["obj"].shape == (0,)
    # infeasible: initial velocity outside every region-reachable box
    x0 = np.array([[[3000.0, 60.0], [2900.0, 20.0]]])
    r = mpc.solve(x0, 800.0, np.zeros((1, mpc.n_param)))
    assert r["status"][0] == 3 and np.isinf(r["obj"][0])
    # bad descriptors
    with pytest.raises(RuntimeError):
        hvp.api.CompiledMpc(G.CENT, 3, n_local=2, leader_index=5)
    with pytest.raises(RuntimeError):
        hvp.api.CompiledMpc(G.EVENT, 3, n_local=3, n_front=1, n_behind=0)
    with pytest.raises(RuntimeError):
        hvp.api.CompiledMpc(99, 3)


def _oracle_eval(kind, nl, N, mass, params, xg, ug, tol=1e-6, **kw):
    """Independent restatement of eval_cost (fleet_event_based.py:308-327) on the oracle's dense
    input-space QP: modes from consistency of the pinned data, objective + L1 penalties at u."""
    a, b, c, lo, hi, _ = O.mode_table(kw.get("model", 0), mass)
    R = len(a)
    cands = []
    for i in range(nl):
        row = []
        for k in range(N):
            v = xg[i, 1, k]
            ok = [r for r in range(R) if lo[r] - tol <= v <= hi[r] + tol and
                  (k == N - 1 or abs(xg[i, 1, k + 1] - (a[r] * v + b[r] * ug[i, k] + c[r])) <= tol)]
            if k < N - 1 and abs(xg[i, 0, k + 1] - xg[i, 0, k] - v) > tol:
                return np.inf
            if not ok:
                return np.inf
            row.append(ok if k == N - 1 else ok[:1])
        cands.append(row)
    import itertools
    best = np.inf
    for last in itertools.product(*[cands[i][N - 1] for i in range(nl)]):
        modes = np.array([[cands[i][k][0] for k in range(N - 1)] + [last[i]] for i in range(nl)], np.int32)
        q = O.mpc_build_qp(kind, nl, N, xg[:, :, 0], mass, params, modes, **kw)
        if q is None:
            continue
        H, g, c0, A, bb, w = q
        z = ug.reshape(-1)
        s = A @ z - bb
        hard = ~np.isfinite(w)
        if (s[hard] > tol).any():
            continue
        f = 0.5 * z @ H @ z + g @ z + c0 + (w[~hard] * np.maximum(s[~hard], 0)).sum()
        best = min(best, f)
    return best


def test_event_eval_cost_vs_oracle(hvp):
    rng = np.random.default_rng(600)
    N, nf, nb, nl = 5, 2, 1, 3
    B = 24
    x0, params = G.event_cases(rng, B, nf, nb, N, stress=True)
    mpc = hvp.api.CompiledMpc(G.EVENT, N, n_local=nl, leader_index=0, n_front=nf, n_behind=nb)
    r = mpc.solve(x0, 800.0, params)
    ok = r["status"] == 2
    # (1) the optimal solution itself: eval_cost reproduces the optimal objective
    c = mpc.eval_cost(800.0, params, r["x"], r["u"])
    assert np.allclose(c[ok], r["obj"][ok], rtol=1e-9)
    # (2) shifted guesses (drop column 0, repeat the last: fleet_event_based.py:591-603)
    xs = np.concatenate([r["x"][..., 1:], r["x"][..., -1:]], axis=-1)
    us = np.concatenate([r["u"][..., 1:], r["u"][..., -1:]], axis=-1)
    c = mpc.eval_cost(800.0, params, xs, us)
    co = np.array([_oracle_eval(O.EVENT, nl, N, 800.0, params[i], xs[i], us[i], leader_index=0, n_front=nf,
                                n_behind=nb) if ok[i] else np.inf for i in range(B)])
    fin = np.isfinite(co)
    assert (np.isfinite(c[ok]) == fin[ok]).all()
    assert np.allclose(c[ok & fin], co[ok & fin], rtol=1e-9)
    assert fin.sum() >= 3
    # (3) an inconsistent guess is infeasible
    xbad = r["x"].copy(); xbad[:, 0, 1, 2] += 0.5
    assert np.isinf(mpc.eval_cost(800.0, params, xbad, r["u"])).all()


@pytest.mark.parametrize("budget", ["3", "12"])
def test_tree_split_matches_oracle(hvp, monkeypatch, budget):
    """Heavy trees are split over 32 warps that share the incumbent (pm_kernel.cu pass 1-3).  With a tiny node
    budget almost every problem takes that path; the result must not change."""
    monkeypatch.setenv("HVP_MPC_BUDGET", budget)
    rng = np.random.default_rng(700)
    B, n, N = 48, 3, 4
    x0, params = G.cent_cases(rng, B, n, N, stress=True)
    mpc = hvp.api.CompiledMpc(G.CENT, N, n_local=n)
    r = mpc.solve(x0, 800.0, params)
    ro = O.mpc_solve(O.CENT, n, N, x0, 800.0, params, method=1)
    _compare(r, ro, "cent split")
    monkeypatch.setenv("HVP_MPC_SPLIT", "0")
    r0 = hvp.api.CompiledMpc(G.CENT, N, n_local=n).solve(x0, 800.0, params)
    assert np.allclose(r0["obj"], r["obj"], rtol=1e-9, equal_nan=True)
    assert (r["nodes"] >= 1).all()
    # ADMM formulation with extras, N = 6
    x0, params = G.admm_cases(rng, 32, 6, stress=True)
    monkeypatch.setenv("HVP_MPC_SPLIT", "1")
    mpc = hvp.api.CompiledMpc(G.ADMM, 6, rho=0.5)
    r = mpc.solve(x0, 800.0, params)
    ro = O.mpc_solve(O.ADMM, 1, 6, x0, 800.0, params, rho=0.5, method=1)
    _compare(r, ro, "admm split")


@pytest.mark.parametrize("kind", ["local", "cent"])
def test_real_vehicle_as_reference_vs_oracle(hvp, kind):
    """real_vehicle_as_reference (cent_mld.py:85-105,162-169; fleet_seq_mld.py:137,211-219): the leader keeps the
    spacing policy's distance to the reference vehicle and a (soft) safe distance behind it."""
    rng = np.random.default_rng(333)
    B, N = 24, 4
    if kind == "local":
        from gen_cases import platoon_local_problems
        cs = platoon_local_problems(rng, B, 1, N, stress=True)          # single vehicles: front + leader + trailer
        fl = int(G.FRONT | G.LEADER | G.TRAILER | O.REAL_REF)
        x0 = cs["x0"][:, None, :]
        lead = G.const_vel(np.stack([cs["x0"][:, 0] + rng.uniform(20, 90, B), rng.uniform(10, 30, B)], 1), N)
        params = np.concatenate([np.zeros((B, 2 * 2 * (N + 1))), lead.reshape(B, -1)], axis=1)
        mpc = hvp.api.CompiledMpc(G.LOCAL, N, flags=fl)
        r = mpc.solve(x0, 800.0, params)
        ro = O.mpc_solve(O.LOCAL, 1, N, x0, 800.0, params, flags=fl, method=0)
    else:
        n = 2
        x0, params = G.cent_cases(rng, B, n, N, stress=True)
        params = G.const_vel(np.stack([x0[:, 0, 0] + rng.uniform(20, 90, B), rng.uniform(10, 30, B)], 1), N).reshape(B, -1)
        mpc = hvp.api.CompiledMpc(G.CENT, N, n_local=n, flags=int(O.REAL_REF))
        r = mpc.solve(x0, 800.0, params)
        ro = O.mpc_solve(O.CENT, n, N, x0, 800.0, params, flags=int(O.REAL_REF), method=0)
    _compare(r, ro, f"real_ref {kind}")
    assert (ro["status"] == 2).sum() >= B // 2


def test_local_mpc_mld_real_vehicle_reference_routes_to_compiled(hvp):
    sys_ = hvp.Platoon(1, "pwa_gear", [800.0]).get_vehicle_system_dicts(1.0)[0]
    m = hvp.LocalMpcMld(4, sys_, hvp.ConstantSpacingPolicy(50), True, True, True, True, None, 0.0, True)
    assert isinstance(m, hvp.mpc.LocalMpcGear)
    lead = np.stack([2000.0 + 70.0 + 20.0 * np.arange(5), np.full(5, 20.0)])
    m.set_leader_x(lead)
    u0, info = m.solve_mpc(np.array([[2000.0], [18.0]]))
    assert np.isfinite(info["cost"]) and u0.shape == (1, 1)
    plain = hvp.LocalMpcMld(4, sys_, hvp.ConstantSpacingPolicy(50), True, True, True, True)
    assert type(plain) is hvp.LocalMpcMld


@pytest.mark.gpu
def test_compiled_mip_gap_and_time_limit(hvp):
    """Solver options of hvp_mpc_desc (SURVEY.md 8b): a 5 % gap gives objectives within 5 % of the proven optimum with
    fewer nodes; a 1-microsecond time limit ends trees with status 9 and never reports an objective below the optimum."""
    rng = np.random.default_rng(3)
    n, N = 3, 5
    x0, params = G.cent_cases(rng, 64, n, N, stress=True)
    exact = hvp.api.CompiledMpc(G.CENT, N, n_local=n).solve(x0, 800.0, params)
    loose = hvp.api.CompiledMpc(G.CENT, N, n_local=n, mip_gap=0.05).solve(x0, 800.0, params)
    ok = exact["status"] == 2
    assert (loose["status"] == exact["status"]).all()
    a = np.abs(exact["obj"][ok])
    assert (loose["obj"][ok] >= exact["obj"][ok] - 1e-8 * a).all()
    assert (loose["obj"][ok] - 0.05 * np.abs(loose["obj"][ok]) <= exact["obj"][ok] + 1e-8 * a).all()   # Gurobi's MIPGap definition
    assert loose["nodes"].sum() < exact["nodes"].sum()
    timed = hvp.api.CompiledMpc(G.CENT, N, n_local=n, time_limit_ms=1e-3).solve(x0, 800.0, params)
    assert set(np.unique(timed["status"])) <= {2, 3, 9} and (timed["status"] == 9).any()
    has = np.isfinite(timed["obj"]) & ok
    assert (timed["obj"][has] >= exact["obj"][has] - 1e-8 * np.abs(exact["obj"][has])).all()
    with pytest.raises(RuntimeError):
        hvp.api.CompiledMpc(G.CENT, N, n_local=n, mip_gap=1.5)
