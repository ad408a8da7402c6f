"""On-device closed loops of the centralized controller: sweep.BatchedCentSweep and fleet_cent_mld.simulate_many.

* The reference's own fleet_cent_mld.py closed loops (tests/golden/fleet_golden.npz) through simulate_many and through the
  sweep directly, at the bar test_fleet_golden.agree holds simulate() to.
* The 1-norm cost (quadratic_cost=False: MILPs) is certified step by step against HiGHS on the explicit big-M model
  (tests/mld_bigm.py), not compared trajectory to trajectory: an LP optimum is often a face, and which vertex the
  multi-warp search returns depends on timing.
* Non-optimal scenarios, a large batch, and the fused glue kernel (hvp_cent_step_dev) against numpy."""
import ctypes as C

import numpy as np
import pytest

import mld_bigm as MB
from test_fleet_golden import G, META, agree, make_sim

pytestmark = pytest.mark.gpu

GOLDEN_SETS = [["cent_task2_C1_s0", "cent_task2_C1_s1", "cent_task2_C1_s2"], ["cent_task2_lead1"], ["cent_friction_gear"]]


def _reset_states(sim, seeds):
    """Initial states of simulate(sim, seed=s) for each seed: PlatoonEnv.reset with MldAgent.evaluate's seed."""
    from hybrid_vehicle_platoon_b200._sim import make_env_and_systems
    env, _, _, _ = make_env_and_systems(sim, forward_quadratic=True)
    return np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                                dtype=np.float64).reshape(-1) for s in seeds])


def _golden_sweep(names, ctx):
    """One BatchedCentSweep over golden runs that share (n, N, leader, model, ep_len); per-scenario masses and leaders."""
    from hybrid_vehicle_platoon_b200 import sweep as S
    sims = [make_sim(META[nm]["spec"]) for nm in names]
    sp = META[names[0]]["spec"]
    masses = np.array([[800.0] * s.n if s.masses is None else s.masses for s in sims])
    x0 = np.stack([G[f"{nm}/X"][0] for nm in names])
    lx = np.stack([G[f"{nm}/leader_x"] for nm in names])
    sw = S.BatchedCentSweep(sp["n"], sp["N"], masses=masses, spacing_policy=sims[0].spacing_policy,
                            leader_index=sp.get("leader_index") or 0, model=sp.get("model", "pwa_gear"), ctx=ctx)
    try:
        return sw.run(x0, lx, sp["ep_len"], strict=True)
    finally:
        sw.close()


def test_simulate_many_matches_reference_goldens(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    names = ["cent_default_C1_s0", "cent_default_C1_s1", "cent_default_C1_s2"]
    sim = make_sim(META[names[0]]["spec"])
    outs = hvp.fleet_cent_mld.simulate_many(sim, [META[nm]["seed"] for nm in names], ctx=hvp_ctx)
    T = META[names[0]]["spec"]["ep_len"]
    for nm, out in zip(names, outs):
        np.testing.assert_array_equal(out["X"][0], G[f"{nm}/X"][0])          # reset and seed path
        agree(nm, out, 1e-6)
        assert out["R"].shape == (T, 1, 1) and out["node_counts"].shape == (T, 1) and out["violations"].shape == (T,)
        assert out["solve_times"].shape == (T, 1) and np.isnan(out["solve_times"]).all()
        assert (out["node_counts"] >= 1).all()


@pytest.mark.parametrize("names", GOLDEN_SETS, ids=lambda v: v[0])
def test_sweep_matches_reference_goldens(hvp_ctx, names):
    r = _golden_sweep(names, hvp_ctx)
    assert (r["status"] == 2).all() and (r["aborted_at"] == -1).all() and (r["errors"] == 0).all()
    for j, nm in enumerate(names):
        gX, gU = G[f"{nm}/X"], G[f"{nm}/U"]
        assert r["U"][:, j].shape == gU.shape
        dX, dU = np.abs(r["X"][:, j] - gX).max(), np.abs(r["U"][:, j] - gU).max()
        assert dX < 1e-6 and dU < 1e-6, (nm, dX, dU)
        np.testing.assert_allclose(r["R"][:, j], G[f"{nm}/R"].reshape(-1), rtol=1e-7, atol=1e-6)
        np.testing.assert_array_equal(np.where(r["violations"][:, j] != 0, 100.0, 0.0), G[f"{nm}/violations"])
        if META[nm]["spec"].get("model") == "pwa_friction":     # [u_g ; gears]: the gears exactly
            n = gU.shape[1] // 2
            np.testing.assert_array_equal(r["U"][:, j, n:], gU[:, n:])


def _one_norm_stage_cost(x, u, lx_t, n):
    """env.py:126-180 with the 1-norm: leader tracking, constant spacing 50 m, input effort."""
    p, v = x[0::2], x[1::2]
    e = abs(p[0] - lx_t[0]) + 0.1 * abs(v[0] - lx_t[1])
    for i in range(1, n):
        e += abs(p[i] - p[i - 1] + 50.0) + 0.1 * abs(v[i] - v[i - 1])
    return e + np.abs(u).sum()


def test_one_norm_closed_loop_certified_by_highs(hvp_ctx):
    """sim.quadratic_cost = False through simulate_many and through the sweep.  At every logged (t, s): HiGHS on the
    explicit big-M MILP at the logged state and leader window has the optimum the sweep logged (1e-6 relative); HiGHS
    with the stage-0 inputs fixed to the ones the loop applied reaches that optimum (so the applied input is optimal,
    whichever optimal vertex was picked); R[t] is the 1-norm stage cost."""
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import sweep as S
    from hybrid_vehicle_platoon_b200.models import Platoon
    n, N, T, seeds = 3, 4, 6, [0, 1, 2, 3]
    sim = hvp.Sim()
    sim.n, sim.N, sim.ep_len, sim.quadratic_cost = n, N, T, False
    systems = Platoon(n, "pwa_gear", masses=[800.0] * n).get_vehicle_system_dicts(1.0)
    lx = sim.leader_trajectory.get_leader_trajectory()
    opt = {}

    def optimum(x, t):
        key = (x.tobytes(), t)
        if key not in opt:
            M, _, _, _ = MB.build_cent(systems, N, x.reshape(n, 2), lx[:, t:t + N + 1], quadratic=False)
            ok, _, obj = MB.solve_milp(M)
            assert ok, (t, x)
            opt[key] = obj
        return opt[key]

    def certify(x, u, r, t):
        obj = optimum(x, t)
        M, _, us, _ = MB.build_cent(systems, N, x.reshape(n, 2), lx[:, t:t + N + 1], quadratic=False)
        for v in range(n):
            M.lb[int(us[v][0, 0])] = u[v] - 1e-7
            M.ub[int(us[v][0, 0])] = u[v] + 1e-7
        ok, _, obj_u = MB.solve_milp(M)
        assert ok and abs(obj_u - obj) <= 1e-5 * max(1.0, abs(obj)), (t, obj_u, obj)
        e = _one_norm_stage_cost(x, u, lx[:, t], n)
        assert abs(r - e) <= 1e-9 * max(1.0, e), (t, r, e)
        return obj

    for j, out in enumerate(hvp.fleet_cent_mld.simulate_many(sim, seeds, ctx=hvp_ctx)):
        for t in range(T):
            certify(out["X"][t], out["U"][t], float(out["R"][t].reshape(-1)[0]), t)
    sw = S.BatchedCentSweep(n, N, quadratic_cost=False, ctx=hvp_ctx)
    try:
        r = sw.run(_reset_states(sim, seeds), lx, T, strict=True)
    finally:
        sw.close()
    for s in range(len(seeds)):
        for t in range(T):
            obj = certify(r["X"][t, s], r["U"][t, s], r["R"][t, s], t)
            assert abs(r["obj"][t, s] - obj) <= 1e-6 * max(1.0, abs(obj)), (s, t, r["obj"][t, s], obj)


def test_friction_one_norm_consistent_with_single_problem_mpc(hvp_ctx):
    """Friction model x 1-norm: a CONSISTENCY check, not an independent one (tests/mld_bigm.py models pwa_gear only).
    At every step the logged objective equals MpcGearCent.solve_mpc (the single-problem path of the same compiled
    formulation) at the logged state, and the logged gears are a valid gear index."""
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import sweep as S
    from hybrid_vehicle_platoon_b200.models import Platoon
    n, N, T = 2, 3, 4
    sim = hvp.Sim()
    sim.n, sim.N, sim.vehicle_model_type, sim.quadratic_cost = n, N, "pwa_friction", False
    lx = sim.leader_trajectory.get_leader_trajectory()
    x0 = _reset_states(sim, [0, 1, 2])
    sw = S.BatchedCentSweep(n, N, quadratic_cost=False, model="pwa_friction", ctx=hvp_ctx)
    try:
        r = sw.run(x0, lx, T, strict=True)
    finally:
        sw.close()
    assert r["U"].shape == (T, 3, 2 * n)
    g = r["U"][:, :, n:]
    assert ((g >= 1) & (g <= 6) & (g == np.round(g))).all()
    systems = Platoon(n, "pwa_friction", masses=[800.0] * n).get_vehicle_system_dicts(1.0)
    mpc = hvp.fleet_cent_mld.MpcGearCent(n, N, systems, quadratic_cost=False, ctx=hvp_ctx)
    for s in range(x0.shape[0]):
        for t in range(T):
            mpc.set_leader_traj(lx[:, t:t + N + 1])
            _, info = mpc.solve_mpc(r["X"][t, s].reshape(2 * n, 1))
            assert abs(info["cost"] - r["obj"][t, s]) <= 1e-6 * max(1.0, abs(info["cost"])), (s, t, info["cost"], r["obj"][t, s])


def test_infeasible_scenario_is_reported_and_isolated(hvp_ctx):
    """A platoon whose second vehicle starts at 48 m/s: the MPC's velocity box (<= 45.84 m/s from stage 1 on) and its
    deceleration row (at most 2 m/s per step) leave no feasible point -- confirmed by HiGHS on the big-M model."""
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import sweep as S
    from hybrid_vehicle_platoon_b200.models import Platoon
    n, N, T = 3, 5, 8
    sim = hvp.Sim()
    sim.n, sim.N = n, N
    lx = sim.leader_trajectory.get_leader_trajectory()
    good = _reset_states(sim, [0, 1, 2])
    bad = good[0].copy()
    bad[3] = 48.0
    systems = Platoon(n, "pwa_gear", masses=[800.0] * n).get_vehicle_system_dicts(1.0)
    M, _, _, _ = MB.build_cent(systems, N, bad.reshape(n, 2), lx[:, :N + 1], quadratic=False)
    assert not MB.solve_milp(M)[0]
    x0 = np.concatenate([good[:1], bad[None], good[1:]])
    sw = S.BatchedCentSweep(n, N, ctx=hvp_ctx)
    try:
        r = sw.run(x0, lx, T)
        ref = sw.run(good, lx, T)
        with pytest.raises(RuntimeError, match="scenario 1 at timestep 0"):
            sw.run(x0, lx, T, strict=True)
    finally:
        sw.close()
    assert r["status"][0, 1] != 2 and r["aborted_at"][1] == 0
    assert (r["aborted_at"][[0, 2, 3]] == -1).all()
    np.testing.assert_array_equal(r["U"][0, 1], np.zeros(n))
    keep = [0, 2, 3]
    for k in ("X", "U", "R", "obj", "status", "violations", "errors"):
        np.testing.assert_array_equal(r[k][:, keep], ref[k], err_msg=k)
    # friction: zero throttle and gear 6 for the failed scenario (one step: the rollout of gear 6 at 48 m/s is outside
    # that gear's velocity window, which the rollout reports as its own error)
    sw = S.BatchedCentSweep(n, N, model="pwa_friction", ctx=hvp_ctx)
    try:
        rf = sw.run(x0, lx, 1)
    finally:
        sw.close()
    assert rf["status"][0, 1] != 2 and rf["aborted_at"][1] == 0
    np.testing.assert_array_equal(rf["U"][0, 1], np.r_[np.zeros(n), np.full(n, 6.0)])
    assert (rf["status"][0, keep] == 2).all()


def test_large_batch_matches_simulate(hvp_ctx):
    """2048 C1 platoons from the reference's reset distribution x 10 steps: heavy trees go through the split and
    adoption passes of the compiled-MPC kernel; every solve is optimal, and sampled scenarios follow simulate()."""
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import sweep as S
    n, N, T, B = 3, 5, 10, 2048
    sim = hvp.Sim()
    sim.n, sim.N = n, N
    lx = sim.leader_trajectory.get_leader_trajectory()
    x0 = _reset_states(sim, range(B))
    sw = S.BatchedCentSweep(n, N, ctx=hvp_ctx)
    try:
        r = sw.run(x0, lx, T, strict=True)
    finally:
        sw.close()
    assert (r["status"] == 2).all() and (r["errors"] == 0).all()
    for s in (0, 517, 1234, 2047):
        out = hvp.fleet_cent_mld.simulate(sim, seed=s, ep_len=T)
        dX, dU = np.abs(r["X"][:, s] - out["X"]).max(), np.abs(r["U"][:, s] - out["U"]).max()
        assert dX < 1e-6 and dU < 1e-6, (s, dX, dU)
        np.testing.assert_allclose(r["R"][:, s], out["R"].reshape(-1), rtol=1e-7, atol=1e-6)


# ---- the glue kernel (hvp_cent_step_dev) against numpy ------------------------------------------------------------
def _step_struct(torch, n, N, S, *, lx=None, params=None, T=0, tensors=None, gear_table=None):
    from hybrid_vehicle_platoon_b200 import _lib
    g = _lib.CentStep()
    g.n, g.N, g.S = n, N, S
    t_idx = torch.zeros(1, dtype=torch.int64, device="cuda")
    g.t = t_idx.data_ptr()
    if lx is not None:
        g.leader_per_scenario, g.leader_len = int(lx.ndim == 3), lx.shape[-1]
        g.leader_x, g.params, g.n_param = lx.data_ptr(), params.data_ptr(), params.shape[1]
    if tensors is not None:
        g.T = T
        for k, v in tensors.items():
            setattr(g, k, None if v is None else v.data_ptr())
    if gear_table is not None:
        g.n_modes = len(gear_table)
        for k, v in enumerate(gear_table):
            g.mode_gear[k] = int(v)
    return g, t_idx


def test_pack_phase_matches_numpy(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib, api
    rng = np.random.default_rng(5)
    n, N, S, L = 3, 5, 7, 40
    for shared in (True, False):
        lx_np = rng.normal(size=(2, L) if shared else (S, 2, L))
        lx = torch.as_tensor(lx_np, device="cuda")
        npar = 2 * (N + 1) + 3                           # extra columns must be left alone
        params = torch.full((S, npar), -7.0, dtype=torch.float64, device="cuda")
        g, t_idx = _step_struct(torch, n, N, S, lx=lx, params=params)
        for t in (0, 3, L - N - 1, L - 2, L + 5):
            t_idx.fill_(t)
            api.cent_step_device(g, phase=_lib.CENT_PACK, ctx=hvp_ctx)
            hvp_ctx.synchronize()
            cols = np.minimum(np.arange(t, t + N + 1), L - 1)          # past the end: the last column
            ref = np.broadcast_to(lx_np, (S, 2, L))[:, :, cols].reshape(S, -1)
            got = params.cpu().numpy()
            np.testing.assert_array_equal(got[:, :2 * (N + 1)], ref, err_msg=f"shared={shared} t={t}")
            assert (got[:, 2 * (N + 1):] == -7.0).all()


def test_adopt_phase_matches_numpy(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib, api
    rng = np.random.default_rng(6)
    n, N, S, T = 3, 4, 9, 3
    cu = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    for model in (_lib.MODEL_PWA_GEAR, _lib.MODEL_FRICTION_GEAR):
        cm = api.CompiledMpc(_lib.MPC_CENT, N, n_local=n, model=model, ctx=hvp_ctx)
        table = cm.mode_gear
        cm.close()
        for with_gear in (True, False):
            w = 2 * n if with_gear else n
            bufs = dict(u0=cu(np.full((S, n), np.nan)), gear0=cu(np.full((S, n), -1, np.int32)) if with_gear else None,
                        U_log=cu(np.full((T, S, w), np.nan)), obj_log=cu(np.full((T, S), np.nan)),
                        status_log=cu(np.full((T, S), -1, np.int32)), nodes_log=cu(np.full((T, S), -1, np.int32)),
                        aborted_at=cu(np.full(S, 77, np.int32)))
            ab_ref = np.full(S, 77, np.int32)
            for t in range(T + 1):                    # the last t is past the logs: only u0 / gear0 are written
                u = rng.normal(size=(S, n, N)); modes = rng.integers(-1, len(table) + 2, (S, n, N)).astype(np.int32)
                status = rng.choice(np.array([2, 2, 2, 3, 8, 9, 12], np.int32), S)
                obj = rng.normal(size=S); nodes = rng.integers(1, 500, S).astype(np.int32)
                ins = dict(u=cu(u), modes=cu(modes), obj=cu(obj), status=cu(status), nodes=cu(nodes))
                g, t_idx = _step_struct(torch, n, N, S, T=T, tensors={**ins, **bufs}, gear_table=table if with_gear else None)
                t_idx.fill_(t)
                api.cent_step_device(g, phase=_lib.CENT_ADOPT, ctx=hvp_ctx)
                hvp_ctx.synchronize()
                ok = (status == 2)[:, None]
                u0 = np.where(ok, u[:, :, 0], 0.0)
                gear = np.where(ok, table[np.clip(modes[:, :, 0], 0, len(table) - 1)], 6)
                np.testing.assert_array_equal(bufs["u0"].cpu().numpy(), u0)
                if with_gear:
                    np.testing.assert_array_equal(bufs["gear0"].cpu().numpy(), gear)
                if t < T:
                    row = np.concatenate([u0, gear.astype(np.float64)], 1) if with_gear else u0
                    np.testing.assert_array_equal(bufs["U_log"].cpu().numpy()[t], row)
                    np.testing.assert_array_equal(bufs["obj_log"].cpu().numpy()[t], obj)
                    np.testing.assert_array_equal(bufs["status_log"].cpu().numpy()[t], status)
                    np.testing.assert_array_equal(bufs["nodes_log"].cpu().numpy()[t], nodes)
                    if t == 0:
                        ab_ref = np.where(status == 2, -1, 0).astype(np.int32)
                    else:
                        ab_ref = np.where((status != 2) & (ab_ref < 0), t, ab_ref).astype(np.int32)
                np.testing.assert_array_equal(bufs["aborted_at"].cpu().numpy(), ab_ref)


def test_cent_step_rejects_bad_arguments(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    L = _lib.lib()
    n, N, S, T = 3, 4, 5, 2
    lx = torch.zeros((2, 30), dtype=torch.float64, device="cuda")
    params = torch.zeros((S, 2 * (N + 1)), dtype=torch.float64, device="cuda")
    e = lambda *s, dt=torch.float64: torch.zeros(s, dtype=dt, device="cuda")
    i32 = torch.int32
    full = dict(u=e(S, n, N), modes=e(S, n, N, dt=i32), obj=e(S), status=e(S, dt=i32), nodes=e(S, dt=i32), u0=e(S, n),
                gear0=e(S, n, dt=i32), U_log=e(T, S, 2 * n), obj_log=e(T, S), status_log=e(T, S, dt=i32),
                nodes_log=e(T, S, dt=i32), aborted_at=e(S, dt=i32))

    def pack(**kw):
        g, t = _step_struct(torch, n, N, S, lx=lx, params=params)
        g.phase = _lib.CENT_PACK
        for k, v in kw.items():
            setattr(g, k, v)
        return g, t

    def adopt(**kw):
        g, t = _step_struct(torch, n, N, S, T=T, tensors=full, gear_table=[1, 2, 3, 4, 5, 6, 6])
        g.phase = _lib.CENT_ADOPT
        for k, v in kw.items():
            setattr(g, k, v)
        return g, t

    cases = [pack(n=0), pack(N=0), pack(S=-1), pack(phase=2), pack(n_param=2 * N + 1), pack(leader_len=0),
             pack(leader_x=None), pack(params=None), pack(t=None), adopt(T=-1), adopt(n_modes=0), adopt(n_modes=17),
             adopt(modes=None)] + [adopt(**{k: None}) for k in full if k not in ("gear0", "modes")]
    before = hvp_ctx.launch_count
    for g, keep in cases:
        assert L.hvp_cent_step_dev(hvp_ctx.handle, C.byref(g), None) < 0
        assert "cent_step" in _lib.last_error()
    assert L.hvp_cent_step_dev(hvp_ctx.handle, None, None) < 0
    assert hvp_ctx.launch_count == before
    # the valid versions of the same calls do launch
    for g, keep in (pack(), adopt(), adopt(gear0=None, modes=None, n_modes=0)):
        assert L.hvp_cent_step_dev(hvp_ctx.handle, C.byref(g), None) == 0
    hvp_ctx.synchronize()
    assert hvp_ctx.launch_count == before + 3
