"""On-device closed loops of the naive-ADMM controller: sweep.BatchedAdmmSweep (fused glue kernel hvp_admm_step_dev,
both vehicle models) and fleet_naive_admm.simulate_many.

* The reference's own fleet_naive_admm.py closed loops (tests/golden/fleet_golden.npz) through simulate_many, and the
  discrete-gear one through the sweep, at the bar test_fleet_golden holds simulate() to for this controller.
* The fused loop against the torch glue it replaces, an infeasible scenario beside ordinary ones, a large batch,
  real_vehicle_as_reference.
* Each phase of the glue kernel against a numpy restatement, bit for bit, the older hvp_admm_round_dev against it, and
  its rejected arguments."""
import ctypes as C

import numpy as np
import pytest

from test_fleet_golden import G, META, _tol, agree, make_sim

pytestmark = pytest.mark.gpu


def _reset_states(sim, seeds):
    """Initial states of simulate(sim, seed=s) for each seed: PlatoonEnv.reset with MldAgent.evaluate's seed."""
    from hybrid_vehicle_platoon_b200._sim import make_env_and_systems
    env, _, _, _ = make_env_and_systems(sim)
    return np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                                dtype=np.float64).reshape(-1) for s in seeds])


def _check_schema(out, n, T, w):
    assert out["X"].shape == (T + 1, 2 * n) and out["U"].shape == (T, w) and out["R"].shape == (T, 1, 1)
    assert out["node_counts"].shape == (T, 1) and out["violations"].shape == (T,)
    assert out["solve_times"].shape == (T, 1) and np.isnan(out["solve_times"]).all()
    assert (out["node_counts"] >= 1).all()


def test_simulate_many_matches_reference_goldens(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    names = ["admm_default_s1", "admm_default_s2", "admm_default_s3"]
    sim = make_sim(META[names[0]]["spec"])
    T, n = 30, sim.n
    outs = hvp.fleet_naive_admm.simulate_many(sim, [1, 2, 3], admm_iters=10, ep_len=T, ctx=hvp_ctx)
    for nm, out in zip(names, outs):
        np.testing.assert_array_equal(out["X"][0], G[f"{nm}/X"][0])          # reset and seed path
        agree(nm, out, *_tol("admm"))
        _check_schema(out, n, T, n)
        assert out["leader_x"].shape == (2, 200)


@pytest.mark.parametrize("name", ["admm_task2_C3_n15_N8", "admm_task2_lead1_s0"])
def test_simulate_many_matches_reference_golden_shapes(hvp_ctx, name):
    import hybrid_vehicle_platoon_b200 as hvp
    m = META[name]
    sp = m["spec"]
    out, = hvp.fleet_naive_admm.simulate_many(make_sim(sp), [m["seed"]], admm_iters=m["kw"]["admm_iters"],
                                              leader_index=sp.get("leader_index") or 0, ep_len=sp["ep_len"], ctx=hvp_ctx)
    np.testing.assert_array_equal(out["X"][0], G[f"{name}/X"][0])
    agree(name, out, *_tol("admm"))
    _check_schema(out, sp["n"], sp["ep_len"], sp["n"])


def test_friction_golden_through_sweep_and_simulate_many(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import sweep as S
    nm = "admm_friction_gear"
    sp, kw = META[nm]["spec"], META[nm]["kw"]
    sim = make_sim(sp)
    n, T = sp["n"], sp["ep_len"]
    gX, gU = G[f"{nm}/X"], G[f"{nm}/U"]
    tx, tu = _tol("admm")
    sw = S.BatchedAdmmSweep(n, sp["N"], admm_iters=kw["admm_iters"], spacing_policy=sim.spacing_policy,
                            model="pwa_friction", ctx=hvp_ctx)
    try:
        r = sw.run(gX[0][None], G[f"{nm}/leader_x"], T)
    finally:
        sw.close()
    assert (r["status"] == 2).all() and (r["errors"] == 0).all() and (r["failed_at"] == [-1, -1, 0]).all()
    assert r["U"].shape == (T, 1, 2 * n)
    dX, dU = np.abs(r["X"][:, 0] - gX).max(), np.abs(r["U"][:, 0] - gU).max()
    assert dX < tx and dU < tu, (dX, dU)
    np.testing.assert_array_equal(r["U"][:, 0, n:], gU[:, n:])                 # the gears exactly
    np.testing.assert_allclose(r["R"][:, 0], G[f"{nm}/R"].reshape(-1), rtol=1e-7, atol=tx)
    out, = hvp.fleet_naive_admm.simulate_many(sim, [2], admm_iters=4, ep_len=T, ctx=hvp_ctx)
    agree(nm, out, tx, tu)
    np.testing.assert_array_equal(out["U"][:, n:], gU[:, n:])
    _check_schema(out, n, T, 2 * n)


def _agree_or_both_fail(simulate_one, many_out, failed_at, errors, tx, ty):
    """simulate() of one seed against its episode of a batched run: equal at the controller's tolerance, or simulate()
    raises and the batched run reports a solve that was not optimal or a rollout error.  Returns True if compared."""
    try:
        one = simulate_one()
    except (RuntimeError, RuntimeWarning):
        assert failed_at[0] >= 0 or (errors != 0).any()
        return False
    assert failed_at[0] < 0
    dX, dU = np.abs(many_out["X"] - one["X"]).max(), np.abs(many_out["U"] - one["U"]).max()
    assert dX < tx and dU < ty, (dX, dU)
    np.testing.assert_allclose(np.asarray(many_out["R"]).reshape(-1), np.asarray(one["R"]).reshape(-1), rtol=1e-7, atol=tx)
    return True


def _failed_of(sim, seeds, T, iters, hvp_ctx, **kw):
    """The sweep's failed_at / errors for the seeds' episodes (simulate_many does not return them)."""
    from hybrid_vehicle_platoon_b200 import sweep as S
    from hybrid_vehicle_platoon_b200._sim import make_env_and_systems
    env, _, _, _ = make_env_and_systems(sim, kw.get("leader_index", 0))
    sw = S.BatchedAdmmSweep(sim.n, sim.N, admm_iters=iters, masses=env.unwrapped.masses, spacing_policy=sim.spacing_policy,
                            model=sim.vehicle_model_type, real_vehicle_as_reference=sim.real_vehicle_as_reference,
                            ctx=hvp_ctx, **kw)
    try:
        r = sw.run(_reset_states(sim, seeds), sim.leader_trajectory.get_leader_trajectory(), T)
    finally:
        sw.close()
    return r


def test_friction_seeds_match_simulate(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    sim = make_sim(META["admm_friction_gear"]["spec"])
    n, T, iters, seeds = sim.n, 6, 4, [3, 4, 5, 6]
    outs = hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=iters, ep_len=T, strict=False, ctx=hvp_ctx)
    r = _failed_of(sim, seeds, T, iters, hvp_ctx)
    tx, tu = _tol("admm")
    done = sum(_agree_or_both_fail(lambda: hvp.fleet_naive_admm.simulate(sim, admm_iters=iters, seed=s, ep_len=T), out,
                                   r["failed_at"][j], r["errors"][:, j], tx, tu)
               for j, (s, out) in enumerate(zip(seeds, outs)))
    assert done >= 2


@pytest.mark.parametrize("n,li", [(4, 0), (5, 2)])
def test_fused_matches_torch_glue(hvp_ctx, n, li):
    from hybrid_vehicle_platoon_b200 import sweep as S
    from test_host_fleets import SmallSim
    N, T, iters = 4, 5, 3
    sim = SmallSim(n, N, T, headway=True)
    x0 = _reset_states(sim, [5, 6, 9, 11])
    lx = sim.leader_trajectory.get_leader_trajectory()
    out = {}
    for fused in (True, False):
        sw = S.BatchedAdmmSweep(n, N, admm_iters=iters, leader_index=li, spacing_policy=sim.spacing_policy, fused=fused,
                                ctx=hvp_ctx)
        try:
            out[fused] = sw.run(x0, lx, T)
        finally:
            sw.close()
    a, b = out[True], out[False]
    assert (a["nodes"] >= 1).all()
    for k in ("X", "U", "R", "violations", "errors", "status", "nodes", "failed_at"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


def test_torch_glue_rejects_friction(hvp_ctx):
    from hybrid_vehicle_platoon_b200 import sweep as S
    with pytest.raises(ValueError, match="pwa_gear"):
        S.BatchedAdmmSweep(3, 3, model="pwa_friction", fused=False, ctx=hvp_ctx)
    with pytest.raises(ValueError, match="model"):
        S.BatchedAdmmSweep(3, 3, model="pwa", ctx=hvp_ctx)


def _bad_state(sim, seed):
    """The reset state of `seed` with vehicle 1 at 60 m/s: even full braking leaves it above v_max = 45.84 m/s at
    stage 1, so vehicle 1's local MIQP is infeasible."""
    x = _reset_states(sim, [seed])[0]
    x[3] = 60.0
    return x


def test_infeasible_scenario_is_reported_and_isolated(hvp_ctx, monkeypatch):
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import sweep as S
    from hybrid_vehicle_platoon_b200.env import PlatoonEnv
    n, N, T = 3, 5, 1           # one step: the rollout of a vehicle at 60 m/s reports an error and leaves NaN behind
    sim = hvp.Sim()
    sim.n, sim.N = n, N
    lx = sim.leader_trajectory.get_leader_trajectory()
    good = _reset_states(sim, [0, 1, 2])
    bad_seed = 7
    bad = _bad_state(sim, bad_seed)
    mixed = np.concatenate([good[:1], bad[None], good[1:]])
    # the single-scenario simulate() from that state raises
    target = int(np.random.SeedSequence(bad_seed).generate_state(1)[0])
    orig = PlatoonEnv.reset

    def reset(self, *, seed=None, options=None):
        x, info = orig(self, seed=seed, options=options)
        if seed == target:
            self.x = bad.reshape(-1, 1).copy()
            x = self.x
        return x, info

    monkeypatch.setattr(PlatoonEnv, "reset", reset)
    with pytest.raises(RuntimeError, match="Infeasible problem encountered"):
        hvp.fleet_naive_admm.simulate(sim, admm_iters=3, seed=bad_seed, ep_len=T)
    res = {}
    for fused in (True, False):
        sw = S.BatchedAdmmSweep(n, N, admm_iters=3, fused=fused, ctx=hvp_ctx)
        try:
            res[fused] = (sw.run(mixed, lx, T), sw.run(good, lx, T))
        finally:
            sw.close()
    r, ref = res[True]
    np.testing.assert_array_equal(r["failed_at"][1], [0, 0, 3])
    assert (r["failed_at"][[0, 2, 3]] == [-1, -1, 0]).all()
    assert r["status"][0, 1, 1] != 2 and r["U"][0, 1, 1] == 0.0
    keep = [0, 2, 3]
    for k in ("X", "U", "R", "violations", "errors", "status", "failed_at"):
        np.testing.assert_array_equal(r[k][:, keep] if k != "failed_at" else r[k][keep], ref[k], err_msg=k)
    for k in ("X", "U", "R", "violations", "errors", "status", "nodes", "failed_at"):
        np.testing.assert_array_equal(r[k], res[False][0][k], err_msg=k)        # the torch glue zeros the same way
    # simulate_many: strict raises naming the seed and the timestep, strict=False returns every episode
    seeds = [0, bad_seed, 1]
    with pytest.raises(RuntimeError, match=f"status 3.*seed {bad_seed}, timestep 0"):
        hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=3, ep_len=T, ctx=hvp_ctx)
    outs = hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=3, ep_len=T, strict=False, ctx=hvp_ctx)
    assert len(outs) == 3
    np.testing.assert_array_equal(outs[1]["X"][0], bad)
    np.testing.assert_array_equal(outs[0]["X"], ref["X"][:, 0])


def test_large_batch_matches_simulate(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    n, N, T, B, iters = 5, 5, 3, 1024, 4
    sim = hvp.Sim()
    sim.n, sim.N = n, N
    seeds = list(range(B))
    outs = hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=iters, ep_len=T, strict=False, ctx=hvp_ctx)
    assert len(outs) == B
    r = _failed_of(sim, seeds, T, iters, hvp_ctx)
    assert (r["failed_at"][:, 0] < 0).mean() > 0.9
    tx, tu = _tol("admm")
    done = sum(_agree_or_both_fail(lambda: hvp.fleet_naive_admm.simulate(sim, admm_iters=iters, seed=s, ep_len=T), outs[s],
                                   r["failed_at"][s], r["errors"][:, s], tx, tu)
               for s in (0, 333, 777, 1023))
    assert done >= 3


@pytest.mark.parametrize("platoon", [False, True])
def test_real_vehicle_as_reference_matches_simulate(hvp_ctx, platoon):
    import hybrid_vehicle_platoon_b200 as hvp
    from test_host_fleets import SmallSim
    n, N, T, iters, seeds = 3, 4, 6, 4, [1, 2]
    sim = SmallSim(n, N, T)
    sim.real_vehicle_as_reference, sim.start_from_platoon = True, platoon
    outs = hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=iters, ep_len=T, strict=False, ctx=hvp_ctx)
    r = _failed_of(sim, seeds, T, iters, hvp_ctx)
    tx, tu = _tol("admm")
    done = sum(_agree_or_both_fail(lambda: hvp.fleet_naive_admm.simulate(sim, admm_iters=iters, seed=s, ep_len=T), out,
                                   r["failed_at"][j], r["errors"][:, j], tx, tu)
               for j, (s, out) in enumerate(zip(seeds, outs)))
    assert done >= 1
    with pytest.raises(NotImplementedError):
        hvp.fleet_naive_admm.simulate(sim, admm_iters=iters, seed=1, ep_len=T, leader_index=1)
    with pytest.raises(NotImplementedError):
        hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=iters, ep_len=T, leader_index=1, ctx=hvp_ctx)


def test_simulate_many_rejects_one_vehicle(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    from test_host_fleets import SmallSim
    with pytest.raises(ValueError, match="two vehicles"):
        hvp.fleet_naive_admm.simulate_many(SmallSim(1, 3, 3), [0], ctx=hvp_ctx)


# ---- the glue kernel (hvp_admm_step_dev) against numpy --------------------------------------------------------------
class _Rig:
    """An hvp_admm_step over torch buffers: n = 5 vehicles in four roles whose indices are not in vehicle order -- the
    front, the trailer, vehicles 1 and 3 together, vehicle 2 alone -- so that roles and rows are all exercised."""
    ROLE_OF = [2, 0, 3, 0, 1]

    def __init__(self, torch, S, N=3, T=3, gears=False, seed=0, L=20):
        from hybrid_vehicle_platoon_b200 import _lib
        self.torch, self.n, self.N, self.S, self.T = torch, 5, N, S, T
        n, np1, blk = self.n, N + 1, 2 * (N + 1)
        self.blk = blk
        self.rng = rng = np.random.default_rng(seed)
        cu = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
        self.cu = cu
        g = self.g = _lib.AdmmStep()
        g.n, g.N, g.S, g.nroles, g.T, g.rho = n, N, S, 4, T, 0.5
        self.table = np.array([1, 2, 3, 4, 5, 6, 6, 2, 4], np.int32)
        g.n_modes = len(self.table)
        for k, v in enumerate(self.table):
            g.mode_gear[k] = int(v)
        for i, r in enumerate(self.ROLE_OF):
            g.role_of[i] = r
        self.t_idx = torch.zeros(1, dtype=torch.int64, device="cuda")
        self.r_idx = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.x = cu(rng.normal(size=(S, n, 2)))
        self.cons = {k: cu(rng.normal(size=(S, n, 2, np1))) for k in ("y_front", "y_back", "zf", "zb", "xs")}
        self.ND = cu(rng.integers(0, 50, (T, S)).astype(np.int32))
        self.FA = cu(np.full((S, 3), 99, np.int32))
        self.U_log = cu(np.full((T, S, 2 * n if gears else n), np.nan))
        self.ST = cu(np.full((T, S, n), -5, np.int32))
        self.u0 = cu(np.full((S, n), np.nan))
        self.gear0 = cu(np.full((S, n), -1, np.int32)) if gears else None
        self.members = [[i for i in range(n) if self.ROLE_OF[i] == r] for r in range(4)]
        self.buf = []
        for r, mem in enumerate(self.members):
            B = S * len(mem)
            hf, hb = int(mem[0] > 0), int(mem[0] < n - 1)
            b = dict(params=cu(np.full((B, 5 * blk), -7.0)), x0=cu(np.full((B, 1, 2), np.nan)),
                     u=cu(rng.normal(size=(B, 1, N))), x=cu(rng.normal(size=(B, 1, 2, np1))),
                     extra=cu(rng.normal(size=(B, max((hf + hb) * blk, 1)))),
                     modes=cu(rng.integers(-2, len(self.table) + 3, (B, 1, N)).astype(np.int32)),
                     status=cu(np.full(B, 2, np.int32)), nodes=cu(rng.integers(1, 900, B).astype(np.int32)))
            self.buf.append(b)
            Gr = g.role[r]
            for k, v in b.items():
                setattr(Gr, k, v.data_ptr())
            Gr.has_front, Gr.has_back = hf, hb
        ptr = lambda t_: None if t_ is None else t_.data_ptr()
        g.t, g.r, g.x = self.t_idx.data_ptr(), self.r_idx.data_ptr(), self.x.data_ptr()
        for k, v in self.cons.items():
            setattr(g, k, v.data_ptr())
        g.ND, g.failed_at, g.U_log, g.ST, g.u0, g.gear0 = self.ND.data_ptr(), self.FA.data_ptr(), self.U_log.data_ptr(), \
            self.ST.data_ptr(), self.u0.data_ptr(), ptr(self.gear0)
        self.set_leader(cu(rng.normal(size=(2, L))))

    def row(self, s, i):
        """(role, row) of vehicle i of scenario s: rows [scenario][vehicle of the role], vehicles in index order."""
        r = self.ROLE_OF[i]
        return r, s * len(self.members[r]) + self.members[r].index(i)

    def set_leader(self, lx):
        self.lx = lx
        self.g.leader_x, self.g.leader_len, self.g.leader_per_scenario = lx.data_ptr(), lx.shape[-1], int(lx.ndim == 3)

    def window(self, t):
        lx, L, N = self.np(self.lx), self.lx.shape[-1], self.N
        cols = np.minimum(np.arange(t, t + N + 1), L - 1)
        return np.broadcast_to(lx, (self.S, 2, L))[:, :, cols].reshape(self.S, self.blk)

    def per_vehicle(self, key):
        """A role buffer as [S][n][...] in vehicle order; rows of `extra` padded with NaN to two blocks."""
        rows = [[self.np(self.buf[self.row(s, i)[0]][key])[self.row(s, i)[1]] for i in range(self.n)] for s in range(self.S)]
        if key == "extra":
            out = np.full((self.S, self.n, 2 * self.blk), np.nan)
            for s in range(self.S):
                for i in range(self.n):
                    out[s, i, :rows[s][i].size] = rows[s][i]
            return out
        return np.array(rows)

    def call(self, phase, ctx, t=0, r=0):
        from hybrid_vehicle_platoon_b200 import api
        self.t_idx.fill_(t)
        self.r_idx.fill_(r)
        api.admm_step_device(self.g, phase=phase, ctx=ctx)
        ctx.synchronize()

    def np(self, a):
        return None if a is None else a.cpu().numpy().copy()


def _params_ref(rig, win, c):
    """[S][n][5 blk]: [leader window | y_front | zf | y_back | zb]."""
    S, n, blk = rig.S, rig.n, rig.blk
    f = lambda k: c[k].reshape(S, n, blk)
    return np.concatenate([np.broadcast_to(win[:, None], (S, n, blk)), f("y_front"), f("zf"), f("y_back"), f("zb")], -1)


def _check_params(rig, P):
    for s in range(rig.S):
        for i in range(rig.n):
            r, b = rig.row(s, i)
            np.testing.assert_array_equal(rig.np(rig.buf[r]["params"])[b], P[s, i], err_msg=f"params s={s} i={i}")


def test_pack_phase_matches_numpy(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    S, N, L = 3, 3, 20
    rig = _Rig(torch, S, N, L=L)
    n = rig.n
    x = rig.np(rig.x)
    for shared in (True, False):
        lx_np = rig.rng.normal(size=(2, L) if shared else (S, 2, L))
        rig.set_leader(torch.as_tensor(lx_np, device="cuda"))
        for t in (0, 5, L - N - 1, L - 2):                  # past the end of the trajectory: its last column
            c = {k: rig.np(v) for k, v in rig.cons.items()}
            rig.call(_lib.ADMM_PACK, hvp_ctx, t=t)
            if t > 0:           # shifted previous predictions: drop column 0, repeat the last one
                sh = np.concatenate((c["xs"][..., 1:], c["xs"][..., -1:]), axis=-1)
                c["zf"][:, 1:] = sh[:, :-1]
                c["zb"][:, :-1] = sh[:, 1:]
            for k, v in rig.cons.items():
                np.testing.assert_array_equal(rig.np(v), c[k], err_msg=f"{k} t={t}")
            np.testing.assert_array_equal(rig.per_vehicle("x0").reshape(S, n, 2), x)
            _check_params(rig, _params_ref(rig, rig.window(t), c))


def _round_ref(rig, c, xo, ext, st, nodes, ND, FA, t, r):
    """fleet_naive_admm.py:421-468 with solve_mpc(raises=False)'s zeros, then the logs; on numpy copies."""
    S, n, blk, rho = rig.S, rig.n, rig.blk, rig.g.rho
    ok = (st == 2)[..., None]
    own = np.where(ok, xo.reshape(S, n, blk), 0.0)
    cf = np.zeros((S, n, blk)); cb = np.zeros((S, n, blk))
    for i in range(n):
        o = 0
        if i > 0:
            cf[:, i] = np.where(ok[:, i], ext[:, i, :blk], 0.0); o = blk
        if i < n - 1:
            cb[:, i] = np.where(ok[:, i], ext[:, i, o:o + blk], 0.0)
    z = np.empty((S, n, blk))
    z[:, 0] = (own[:, 0] + cf[:, 1]) / 2.0
    z[:, n - 1] = (own[:, n - 1] + cb[:, n - 2]) / 2.0
    z[:, 1:n - 1] = (own[:, 1:n - 1] + cf[:, 2:] + cb[:, :n - 2]) / 3.0
    sh = lambda a: a.reshape(a.shape[0], a.shape[1], 2, -1)
    c["xs"] = sh(own)
    c["y_front"][:, 1:] += rho * sh(cf[:, 1:] - z[:, :-1])
    c["y_back"][:, :-1] += rho * sh(cb[:, :-1] - z[:, 1:])
    c["zf"][:, 1:] = sh(z[:, :-1])
    c["zb"][:, :-1] = sh(z[:, 1:])
    if 0 <= t < rig.T:
        ND[t] = np.maximum(ND[t], nodes.max(1))
        for s in range(S):
            if t == 0 and r == 0:
                FA[s] = (-1, -1, 0)
            bad = np.nonzero(st[s] != 2)[0]
            if FA[s, 0] < 0 and bad.size:
                FA[s] = (t, r, st[s, bad[0]])


def test_round_phase_matches_numpy(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    S, N, T = 8, 3, 3
    rig = _Rig(torch, S, N, T=T, seed=1)
    n, np1, rng = rig.n, N + 1, rig.rng
    ND, FA = rig.np(rig.ND), rig.np(rig.FA)
    # (t, r): the reset at (0, 0), a later first failure, failures after the first, a round past the logs
    for t, r in ((0, 0), (0, 1), (1, 0), (2, 3), (T, 0)):
        c = {k: rig.np(v) for k, v in rig.cons.items()}
        st = rng.choice(np.array([2, 2, 2, 3, 9, 12], np.int32), (S, n))
        st[0] = 2                                           # scenario 0: never fails
        st[1] = [2, 3, 9, 2, 2] if (t, r) == (0, 1) else 2  # scenario 1: first fails at (0, 1), vehicle 1 (status 3)
        nodes = rng.integers(1, 900, (S, n)).astype(np.int32)
        for s in range(S):
            for i in range(n):
                ro, b = rig.row(s, i)
                rig.buf[ro]["status"][b] = int(st[s, i]); rig.buf[ro]["nodes"][b] = int(nodes[s, i])
        xo, ext = rig.per_vehicle("x"), rig.per_vehicle("extra")
        rig.call(_lib.ADMM_ROUND, hvp_ctx, t=t, r=r)
        _round_ref(rig, c, xo, ext, st, nodes, ND, FA, t, r)
        for k, v in rig.cons.items():
            np.testing.assert_array_equal(rig.np(v), c[k], err_msg=f"{k} t={t} r={r}")
        _check_params(rig, _params_ref(rig, rig.window(t), c))
        np.testing.assert_array_equal(rig.np(rig.ND), ND, err_msg=f"ND t={t} r={r}")
        np.testing.assert_array_equal(rig.np(rig.FA), FA, err_msg=f"failed_at t={t} r={r}")
    fa = rig.np(rig.FA)
    np.testing.assert_array_equal(fa[0], [-1, -1, 0])
    np.testing.assert_array_equal(fa[1], [0, 1, 3])


@pytest.mark.parametrize("gears", [False, True])
def test_adopt_phase_matches_numpy(hvp_ctx, gears):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    S, N, T = 6, 4, 3
    rig = _Rig(torch, S, N, T=T, gears=gears, seed=2)
    n = rig.n
    st = rig.rng.choice(np.array([2, 2, 3, 9], np.int32), (S, n))
    for s in range(S):
        for i in range(n):
            ro, b = rig.row(s, i)
            rig.buf[ro]["status"][b] = int(st[s, i])
    u, modes = rig.per_vehicle("u")[:, :, 0, 0], rig.per_vehicle("modes")[:, :, 0, 0]
    ok = st == 2
    u0 = np.where(ok, u, 0.0)
    gear0 = np.where(ok, rig.table[np.clip(modes, 0, len(rig.table) - 1)], 6)
    assert (modes < 0).any() and (modes >= len(rig.table)).any()
    U_log, ST = rig.np(rig.U_log), rig.np(rig.ST)
    for t in (0, 2, T):                             # t == T: past the logs, only u0 / gear0
        rig.call(_lib.ADMM_ADOPT, hvp_ctx, t=t)
        np.testing.assert_array_equal(rig.np(rig.u0), u0)
        if gears:
            np.testing.assert_array_equal(rig.np(rig.gear0), gear0)
        if t < T:
            U_log[t] = np.concatenate([u0, gear0.astype(np.float64)], 1) if gears else u0
            ST[t] = st
        np.testing.assert_array_equal(rig.np(rig.U_log), U_log)
        np.testing.assert_array_equal(rig.np(rig.ST), ST)


def test_admm_round_dev_equals_step(hvp_ctx):
    """The older entry hvp_admm_round_dev runs the same device code: with every status 2 its pack and round equal the
    step's PACK at t = 0 and ROUND bit for bit."""
    import torch
    from hybrid_vehicle_platoon_b200 import _lib, api
    S, N = 5, 3
    a, b = _Rig(torch, S, N, seed=3), _Rig(torch, S, N, seed=3)
    n = a.n
    ar = _lib.AdmmRound()
    ar.n, ar.N, ar.S, ar.nroles, ar.rho = n, N, S, 4, 0.5
    for i, r in enumerate(_Rig.ROLE_OF):
        ar.role_of[i] = r
    for r in range(4):
        R, B = ar.role[r], b.buf[r]
        R.params, R.x, R.extra = B["params"].data_ptr(), B["x"].data_ptr(), B["extra"].data_ptr()
        R.has_front, R.has_back = b.g.role[r].has_front, b.g.role[r].has_back
    lwin = torch.as_tensor(np.ascontiguousarray(b.window(0)), device="cuda")
    ar.lwin = lwin.data_ptr()
    ar.y_front, ar.y_back, ar.zf, ar.zb, ar.xs = (b.cons[k].data_ptr() for k in ("y_front", "y_back", "zf", "zb", "xs"))
    a.call(_lib.ADMM_PACK, hvp_ctx, t=0)
    api.admm_round_device(ar, pack_only=True, ctx=hvp_ctx)
    hvp_ctx.synchronize()
    for _ in range(2):
        for r in range(4):
            np.testing.assert_array_equal(a.np(a.buf[r]["params"]), b.np(b.buf[r]["params"]))
        for k in a.cons:
            np.testing.assert_array_equal(a.np(a.cons[k]), b.np(b.cons[k]), err_msg=k)
        a.call(_lib.ADMM_ROUND, hvp_ctx, t=0)
        api.admm_round_device(ar, ctx=hvp_ctx)
        hvp_ctx.synchronize()


def test_admm_step_rejects_bad_arguments(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    L = _lib.lib()

    def case(phase, gears=True, **kw):
        rig = _Rig(torch, 3, gears=gears)
        rig.g.phase = phase
        for k, v in kw.items():
            if k == "role_of":                              # (vehicle, value)
                rig.g.role_of[v[0]] = v[1]
            elif k.startswith("role_"):                     # role_<r>_<field>
                _, r, f = k.split("_", 2)
                setattr(rig.g.role[int(r)], f, v)
            else:
                setattr(rig.g, k, v)
        return rig

    P, R, A = _lib.ADMM_PACK, _lib.ADMM_ROUND, _lib.ADMM_ADOPT
    cases = [case(P, n=1), case(P, n=65), case(P, N=0), case(P, S=-1), case(3), case(-1), case(P, nroles=0),
             case(P, nroles=5), case(R, T=-1), case(P, leader_len=0), case(R, leader_len=0), case(A, n_modes=0),
             case(A, n_modes=17), case(P, role_of=(0, 4)), case(P, role_of=(1, -1)),
             case(P, role_of=(0, 0)), case(P, role_of=(4, 0)), case(P, role_1_has_back=1), case(P, role_2_has_front=1),
             case(P, t=None), case(P, x=None), case(P, leader_x=None), case(P, xs=None), case(P, y_front=None),
             case(P, zb=None), case(P, role_0_params=None), case(P, role_3_x0=None),
             case(R, r=None), case(R, leader_x=None), case(R, ND=None), case(R, failed_at=None), case(R, role_1_x=None),
             case(R, role_0_extra=None), case(R, role_2_status=None), case(R, role_3_nodes=None),
             case(R, role_2_params=None),
             case(A, u0=None), case(A, U_log=None), case(A, ST=None), case(A, role_0_u=None), case(A, role_1_status=None),
             case(A, role_2_modes=None)]
    before = hvp_ctx.launch_count
    for rig in cases:
        assert L.hvp_admm_step_dev(hvp_ctx.handle, C.byref(rig.g), None) < 0, rig.g.phase
        assert "admm_step" in _lib.last_error()
    assert L.hvp_admm_step_dev(hvp_ctx.handle, None, None) < 0
    assert "admm_step" in _lib.last_error()
    # S == 0 is a no-op, not an error
    assert L.hvp_admm_step_dev(hvp_ctx.handle, C.byref(case(R, S=0).g), None) == 0
    assert hvp_ctx.launch_count == before
    # the valid versions of the same calls do launch; without gears neither modes nor n_modes are needed
    valid = [case(P), case(R), case(A), case(A, gears=False, n_modes=0, role_2_modes=None)]
    for rig in valid:
        assert L.hvp_admm_step_dev(hvp_ctx.handle, C.byref(rig.g), None) == 0, _lib.last_error()
    hvp_ctx.synchronize()
    assert hvp_ctx.launch_count == before + len(valid)
