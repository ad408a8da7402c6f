"""On-device closed loops of the event-based controller: sweep.BatchedEventSweep (fused glue kernel hvp_event_iter_dev,
both vehicle models) and fleet_event_based.simulate_many.

* The reference's own fleet_event_based.py closed loops (tests/golden/fleet_golden.npz) through simulate_many, and the
  discrete-gear one through the sweep, at the bar test_fleet_golden holds simulate() to for this controller.
* The fused loop against the torch glue it replaces, an infeasible scenario beside ordinary ones, a large batch.
* Each phase of the glue kernel against a numpy restatement, bit for bit, and its rejected arguments."""
import ctypes as C

import numpy as np
import pytest

from test_fleet_golden import G, META, _tol, agree, make_sim

pytestmark = pytest.mark.gpu


def _reset_states(sim, seeds):
    """Initial states of simulate(sim, seed=s) for each seed: PlatoonEnv.reset with MldAgent.evaluate's seed."""
    from hybrid_vehicle_platoon_b200._sim import make_env_and_systems
    env, _, _, _ = make_env_and_systems(sim, forward_real_ref=False)
    return np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                                dtype=np.float64).reshape(-1) for s in seeds])


def test_simulate_many_matches_reference_goldens(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    names = ["event_default_s1", "event_default_s2", "event_default_s3"]
    sim = make_sim(META[names[0]]["spec"])
    T = META[names[0]]["spec"]["ep_len"]
    outs = hvp.fleet_event_based.simulate_many(sim, [1, 2, 3], event_iters=4, ep_len=T, ctx=hvp_ctx)
    n = sim.n
    for nm, out in zip(names, outs):
        np.testing.assert_array_equal(out["X"][0], G[f"{nm}/X"][0])          # reset and seed path
        agree(nm, out, *_tol("event"))
        assert out["X"].shape == (T + 1, 2 * n) and out["U"].shape == (T, n) and out["R"].shape == (T, 1, 1)
        assert out["node_counts"].shape == (T, 1) and out["violations"].shape == (T,) and out["leader_x"].shape == (2, 200)
        assert out["solve_times"].shape == (T, 1) and np.isnan(out["solve_times"]).all()
        assert (out["node_counts"] >= 1).all()


def test_friction_golden_through_sweep(hvp_ctx):
    from hybrid_vehicle_platoon_b200 import sweep as S
    nm = "event_friction_gear"
    sp, kw = META[nm]["spec"], META[nm]["kw"]
    sim = make_sim(sp)
    n = sp["n"]
    sw = S.BatchedEventSweep(n, sp["N"], event_iters=kw["event_iters"], spacing_policy=sim.spacing_policy,
                             model="pwa_friction", ctx=hvp_ctx)
    try:
        r = sw.run(G[f"{nm}/X"][0][None], G[f"{nm}/leader_x"], sp["ep_len"])
    finally:
        sw.close()
    assert r["feasible"].all() and (r["errors"] == 0).all()
    gX, gU = G[f"{nm}/X"], G[f"{nm}/U"]
    assert r["U"].shape == (sp["ep_len"], 1, 2 * n)
    tx, tu = _tol("event")
    dX, dU = np.abs(r["X"][:, 0] - gX).max(), np.abs(r["U"][:, 0] - gU).max()
    assert dX < tx and dU < tu, (dX, dU)
    np.testing.assert_array_equal(r["U"][:, 0, n:], gU[:, n:])                 # the gears exactly
    np.testing.assert_allclose(r["R"][:, 0], G[f"{nm}/R"].reshape(-1), rtol=1e-7, atol=tx)


@pytest.mark.parametrize("n,li", [(4, 0), (5, 2)])
def test_fused_matches_torch_glue(hvp_ctx, n, li):
    from hybrid_vehicle_platoon_b200 import sweep as S
    from test_host_fleets import SmallSim
    N, T, iters = 4, 6, 3
    sim = SmallSim(n, N, T)
    x0 = _reset_states(sim, [5, 6, 9, 11])
    lx = sim.leader_trajectory.get_leader_trajectory()
    out = {}
    for fused in (True, False):
        sw = S.BatchedEventSweep(n, N, event_iters=iters, leader_index=li, fused=fused, ctx=hvp_ctx)
        try:
            out[fused] = sw.run(x0, lx, T)
        finally:
            sw.close()
    a, b = out[True], out[False]
    assert (a["winners"] >= 0).any() and a["feasible"].all()
    np.testing.assert_array_equal(a["winners"], b["winners"])
    np.testing.assert_array_equal(a["feasible"], b["feasible"])
    assert np.abs(a["X"] - b["X"]).max() <= 1e-9 and np.abs(a["U"] - b["U"]).max() <= 1e-9
    np.testing.assert_array_equal(a["errors"], b["errors"])


def _bad_state(sim, seed):
    """The reset state of `seed` with vehicle 1 at 60 m/s: even full braking leaves it above v_max = 45.84 m/s at
    stage 1, so every local MIQP containing vehicle 1 -- all of them when n = 3 -- is infeasible."""
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
    with pytest.raises(RuntimeWarning, match="No feasible solution found for any event based agent"):
        hvp.fleet_event_based.simulate(sim, seed=bad_seed, ep_len=T)
    sw = S.BatchedEventSweep(n, N, ctx=hvp_ctx)
    try:
        r = sw.run(np.concatenate([good[:1], bad[None], good[1:]]), lx, T)
        ref = sw.run(good, lx, T)
    finally:
        sw.close()
    assert not r["feasible"][0, 1] and (r["winners"][0, 1] == -1).all()
    keep = [0, 2, 3]
    for k in ("X", "U", "R", "violations", "errors", "winners", "feasible"):
        np.testing.assert_array_equal(r[k][:, keep], ref[k], err_msg=k)
    # simulate_many: strict raises naming the seed and the timestep, strict=False returns every episode
    seeds = [0, bad_seed, 1]
    with pytest.raises(RuntimeWarning, match=f"seed {bad_seed}, timestep 0"):
        hvp.fleet_event_based.simulate_many(sim, seeds, ep_len=T, ctx=hvp_ctx)
    outs = hvp.fleet_event_based.simulate_many(sim, seeds, ep_len=T, strict=False, ctx=hvp_ctx)
    assert len(outs) == 3
    np.testing.assert_array_equal(outs[1]["X"][0], bad)
    assert np.abs(outs[0]["X"] - ref["X"][:, 0]).max() <= 1e-9


def test_large_batch_matches_simulate(hvp_ctx):
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import sweep as S
    n, N, T, B = 5, 5, 6, 1024
    sim = hvp.Sim()
    sim.n, sim.N = n, N
    lx = sim.leader_trajectory.get_leader_trajectory()
    x0 = _reset_states(sim, range(B))
    sw = S.BatchedEventSweep(n, N, ctx=hvp_ctx)
    try:
        r = sw.run(x0, lx, T)
    finally:
        sw.close()
    assert r["feasible"].all() and (r["errors"] == 0).all()
    tx, tu = _tol("event")
    for s in (0, 333, 777, 1023):
        out = hvp.fleet_event_based.simulate(sim, seed=s, ep_len=T)
        dX, dU = np.abs(r["X"][:, s] - out["X"]).max(), np.abs(r["U"][:, s] - out["U"]).max()
        assert dX < tx and dU < tu, (s, dX, dU)
        np.testing.assert_allclose(r["R"][:, s], out["R"].reshape(-1), rtol=1e-7, atol=tx)


# ---- the glue kernel (hvp_event_iter_dev) against numpy --------------------------------------------------------------
def _members(n, i):
    f = 0 if (n == 2 or i == 0) else (n - 2 if i == n - 1 else i - 1)
    return list(range(f, f + (2 if (n == 2 or i == 0 or i == n - 1) else 3)))


class _Rig:
    """An hvp_event_iter over torch buffers: n = 5 agents in three groups -- the two ends, and the interior agents with
    their slots permuted -- so that rows, slots and member lists are all exercised."""

    def __init__(self, torch, S, N=3, T=3, iters=2, gears=False, n_param_extra=2, seed=0):
        from hybrid_vehicle_platoon_b200 import _lib
        self.torch, self.n, self.N, self.S, self.T, self.iters = torch, 5, N, S, T, iters
        n, np1 = self.n, N + 1
        self.rng = rng = np.random.default_rng(seed)
        self.groups = [([0], 2, True), ([4], 2, False), ([3, 1, 2], 3, True)]     # agents in slot order, n_local, leader
        self.npar = 6 * np1 + n_param_extra
        cu = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
        self.cu = cu
        g = self.g = _lib.EventIter()
        g.n, g.N, g.S, g.iters, g.ngroups, g.T, g.threshold = n, N, S, iters, 3, T, 10.0
        self.table = np.array([1, 2, 3, 4, 5, 6, 6, 2, 4], np.int32)
        g.n_modes = len(self.table)
        for k, v in enumerate(self.table):
            g.mode_gear[k] = int(v)
        self.t_idx = torch.zeros(1, dtype=torch.int64, device="cuda")
        self.x = cu(rng.normal(size=(S, n, 2)))
        self.SG = cu(rng.normal(size=(S, n, 2, np1)))
        self.UG = cu(rng.normal(size=(S, n, N)))
        self.GG = cu(rng.integers(1, 7, (S, n, N)).astype(np.int32)) if gears else None
        self.active = cu(np.ones(S, np.uint8))
        self.WIN = cu(np.full((T, S, iters), -1, np.int32))
        self.FEAS = cu(np.ones((T, S), np.uint8))
        self.ND = cu(np.zeros((T, S), np.int32))
        self.U_log = cu(np.full((T, S, 2 * n if gears else n), np.nan))
        self.u0 = cu(np.full((S, n), np.nan))
        self.gear0 = cu(np.full((S, n), -1, np.int32)) if gears else None
        self.buf = []
        for r, (agents, nl, lead) in enumerate(self.groups):
            B = S * len(agents)
            b = dict(x0=cu(np.full((B, nl, 2), np.nan)), xg=cu(np.full((B, nl, 2, np1), np.nan)),
                     ug=cu(np.full((B, nl, N), np.nan)), params=cu(np.full((B, self.npar), -7.0)),
                     cost=cu(np.zeros(B)), u=cu(np.zeros((B, nl, N))), x=cu(np.zeros((B, nl, 2, np1))),
                     modes=cu(np.zeros((B, nl, N), np.int32)), obj=cu(np.zeros(B)), status=cu(np.zeros(B, np.int32)),
                     nodes=cu(np.zeros(B, np.int32)))
            self.buf.append(b)
            Gr = g.group[r]
            for k, v in b.items():
                setattr(Gr, k, v.data_ptr())
            Gr.n_local, Gr.n_param, Gr.has_leader = nl, self.npar, int(lead)
            for slot, i in enumerate(agents):
                g.group_of[i], g.slot_of[i] = r, slot
        ptr = lambda t_: None if t_ is None else t_.data_ptr()
        g.t, g.x, g.SG, g.UG, g.GG, g.active = self.t_idx.data_ptr(), self.x.data_ptr(), self.SG.data_ptr(), \
            self.UG.data_ptr(), ptr(self.GG), self.active.data_ptr()
        g.WIN, g.FEAS, g.ND, g.U_log, g.u0, g.gear0 = self.WIN.data_ptr(), self.FEAS.data_ptr(), self.ND.data_ptr(), \
            self.U_log.data_ptr(), self.u0.data_ptr(), ptr(self.gear0)

    def row(self, s, i):
        """(group, row) of agent i of scenario s."""
        for r, (agents, _, _) in enumerate(self.groups):
            if i in agents:
                return r, s * len(agents) + agents.index(i)

    def set_leader(self, lx):
        self.lx = lx
        self.g.leader_x, self.g.leader_len, self.g.leader_per_scenario = lx.data_ptr(), lx.shape[-1], int(lx.ndim == 3)

    def call(self, phase, ctx, t=0, it=0):
        from hybrid_vehicle_platoon_b200 import api
        self.t_idx.fill_(t)
        self.g.it = it
        api.event_iter_device(self.g, phase=phase, ctx=ctx)
        ctx.synchronize()

    def np(self, a):
        return None if a is None else a.cpu().numpy().copy()


def test_pack_phase_matches_numpy(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    S, N, L = 4, 3, 30
    rig = _Rig(torch, S, N)
    n, blk = rig.n, 2 * (N + 1)
    x, SG, UG = rig.np(rig.x), rig.np(rig.SG), rig.np(rig.UG)
    for shared in (True, False):
        lx_np = rig.rng.normal(size=(2, L) if shared else (S, 2, L))
        rig.set_leader(torch.as_tensor(lx_np, device="cuda"))
        for t in (0, 7, L - N - 1, L - 2):                  # past the end of the trajectory: its last column
            rig.call(_lib.EVENT_PACK, hvp_ctx, t=t)
            cols = np.minimum(np.arange(t, t + N + 1), L - 1)
            win = np.broadcast_to(lx_np, (S, 2, L))[:, :, cols].reshape(S, blk)
            for s in range(S):
                for i in range(n):
                    r, b = rig.row(s, i)
                    got = {k: rig.np(v)[b] for k, v in rig.buf[r].items() if k in ("x0", "xg", "ug", "params")}
                    mem = _members(n, i)
                    np.testing.assert_array_equal(got["x0"], x[s, mem])
                    np.testing.assert_array_equal(got["xg"], SG[s, mem])
                    np.testing.assert_array_equal(got["ug"], UG[s, mem])
                    P = got["params"]
                    np.testing.assert_array_equal(P[:blk], win[s] if rig.groups[r][2] else np.zeros(blk))
                    np.testing.assert_array_equal(P[blk:2 * blk], SG[s, i - 2].reshape(-1) if i > 1 else np.zeros(blk))
                    np.testing.assert_array_equal(P[2 * blk:3 * blk], SG[s, i + 2].reshape(-1) if i < n - 2 else np.zeros(blk))
                    assert (P[3 * blk:] == -7.0).all()


def _select_ref(rig, c0, obj, status, nodes, u, xo, modes, t, it, state):
    """fleet_event_based.py:60-82 for every active scenario, on numpy copies of the rig's state."""
    SG, UG, GG, active, WIN, FEAS, ND = state
    n = rig.n
    for s in range(rig.S):
        if not active[s]:
            continue
        best, bi, feas = -np.inf, -1, False
        for i in range(n):
            c1 = obj[s, i] if status[s, i] == 2 else np.inf
            with np.errstate(invalid="ignore"):
                dec = c0[s, i] - c1
            feas |= bool(np.isfinite(c1))
            if dec > rig.g.threshold and (bi < 0 or dec > best):
                best, bi = dec, i
        FEAS[t, s] &= feas
        ND[t, s] = max(ND[t, s], nodes[s].max())
        WIN[t, s, it] = bi
        if bi < 0:
            active[s] = 0
            continue
        for l, j in enumerate(_members(n, bi)):
            SG[s, j] = xo[s, bi, l]
            UG[s, j] = u[s, bi, l]
            if GG is not None:
                GG[s, j] = rig.table[np.clip(modes[s, bi, l], 0, len(rig.table) - 1)]


@pytest.mark.parametrize("gears", [False, True])
def test_select_phase_matches_numpy(hvp_ctx, gears):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    S, N, T, iters = 10, 3, 3, 2
    rig = _Rig(torch, S, N, T=T, iters=iters, gears=gears, seed=1)
    n, np1, rng = rig.n, N + 1, rig.rng
    state = [rig.np(a) for a in (rig.SG, rig.UG, rig.GG, rig.active, rig.WIN, rig.FEAS, rig.ND)]
    inf = np.inf
    for t, it in ((1, 0), (1, 1), (2, 0)):
        c0 = rng.uniform(0, 100, (S, n)); obj = rng.uniform(0, 100, (S, n))
        status = rng.choice(np.array([2, 2, 2, 3, 9], np.int32), (S, n))
        nodes = rng.integers(1, 900, (S, n)).astype(np.int32)
        c0[0] = [50, 90, 40, 90, 10]; obj[0] = [1, 2, 3, 2, 0]; status[0] = 2             # equal maxima: agent 1 wins
        c0[1] = [30, 20, 40, 25, 12]; obj[1] = [20, 15, 30, 20, 10]; status[1] = 2         # dec == threshold at agent 0
        c0[2] = [inf, 5, inf, 7, 1]; obj[2] = [3, 1, 9, 2, 0]; status[2] = 2               # inf decreases: agent 0
        c0[3] = [inf, inf, 5, 5, 5]; status[3] = [3, 3, 9, 12, 8]                        # inf - inf, nothing solved
        c0[4] = [100, 50, 60, 70, 20]; obj[4] = [-900, 10, 20, 30, 5]; status[4] = [9, 2, 2, 2, 2]   # non-optimal
        c0[5] = [1, 2, 3, 4, 5]; obj[5] = [2, 3, 4, 5, 6]; status[5] = 2                   # every decrease negative
        c0[6] = [inf, 1, 2, 3, 4]; obj[6] = [1, 1, 1, 1, 1]; status[6] = [2, 3, 3, 3, 3]   # only agent 0: +inf decrease
        if (t, it) == (1, 1):                       # scenario 7 stopped iterating in this timestep: left untouched
            rig.active[7] = 0
            state[3][7] = 0
        u = rng.normal(size=(S, n, 3, N)); xo = rng.normal(size=(S, n, 3, 2, np1))
        modes = rng.integers(-2, len(rig.table) + 3, (S, n, 3, N)).astype(np.int32)
        for s in range(S):
            for i in range(n):
                r, b = rig.row(s, i)
                nl = rig.groups[r][1]
                B = rig.buf[r]
                B["cost"][b] = float(c0[s, i]); B["obj"][b] = float(obj[s, i])
                B["status"][b] = int(status[s, i]); B["nodes"][b] = int(nodes[s, i])
                B["u"][b] = rig.cu(u[s, i, :nl]); B["x"][b] = rig.cu(xo[s, i, :nl]); B["modes"][b] = rig.cu(modes[s, i, :nl])
        rig.call(_lib.EVENT_SELECT, hvp_ctx, t=t, it=it)
        _select_ref(rig, c0, obj, status, nodes, u, xo, modes, t, it, state)
        for name, got, ref in zip(("SG", "UG", "GG", "active", "WIN", "FEAS", "ND"),
                                  (rig.SG, rig.UG, rig.GG, rig.active, rig.WIN, rig.FEAS, rig.ND), state):
            if got is not None:
                np.testing.assert_array_equal(rig.np(got), ref, err_msg=f"{name} t={t} it={it}")
    win = rig.np(rig.WIN)
    assert win[1, 0, 0] == 1 and win[1, 1, 0] == -1 and win[1, 2, 0] == 0 and win[1, 3, 0] == -1
    assert win[1, 4, 0] != 0 and win[1, 5, 0] == -1 and win[1, 6, 0] == 0 and win[1, 7, 1] == -1
    assert not rig.np(rig.FEAS)[1, 3]


@pytest.mark.parametrize("gears", [False, True])
def test_adopt_phase_matches_numpy(hvp_ctx, gears):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    S, N, T = 6, 4, 3
    rig = _Rig(torch, S, N, T=T, gears=gears, seed=2)
    rig.active[::2] = 0
    for t in (0, 2, T):                             # t == T: past the logs, only u0 / gear0 and the shift
        SG, UG, GG, U_log = rig.np(rig.SG), rig.np(rig.UG), rig.np(rig.GG), rig.np(rig.U_log)
        rig.call(_lib.EVENT_ADOPT, hvp_ctx, t=t)
        np.testing.assert_array_equal(rig.np(rig.u0), UG[:, :, 0])
        if gears:
            np.testing.assert_array_equal(rig.np(rig.gear0), GG[:, :, 0])
        if t < T:
            U_log[t] = np.concatenate([UG[:, :, 0], GG[:, :, 0].astype(np.float64)], 1) if gears else UG[:, :, 0]
        np.testing.assert_array_equal(rig.np(rig.U_log), U_log)
        sh = lambda a: np.concatenate((a[..., 1:], a[..., -1:]), axis=-1)
        np.testing.assert_array_equal(rig.np(rig.SG), sh(SG))
        np.testing.assert_array_equal(rig.np(rig.UG), sh(UG))
        if gears:
            np.testing.assert_array_equal(rig.np(rig.GG), sh(GG))
        assert (rig.np(rig.active) == 1).all()


def test_event_iter_rejects_bad_arguments(hvp_ctx):
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    L = _lib.lib()
    lx = torch.zeros((2, 30), dtype=torch.float64, device="cuda")

    def case(phase, gears=True, **kw):
        rig = _Rig(torch, 3, gears=gears)
        rig.set_leader(lx)
        rig.g.phase = phase
        for k, v in kw.items():
            if k in ("group_of", "slot_of"):                # (agent, value)
                getattr(rig.g, k)[v[0]] = v[1]
            elif k.startswith("group_"):                    # group_<r>_<field>
                _, r, f = k.split("_", 2)
                setattr(rig.g.group[int(r)], f, v)
            else:
                setattr(rig.g, k, v)
        return rig

    P, SEL, A = _lib.EVENT_PACK, _lib.EVENT_SELECT, _lib.EVENT_ADOPT
    cases = [case(P, n=1), case(P, n=65), case(P, N=0), case(P, S=-1), case(3), case(P, ngroups=0), case(P, ngroups=9),
             case(P, group_of=(2, 3)), case(P, group_of=(0, -1)), case(P, slot_of=(2, 3)), case(P, slot_of=(1, 2)),
             case(P, slot_of=(4, 1)), case(P, group_0_n_local=3), case(P, group_of=(4, 0)), case(SEL, it=-1),
             case(SEL, it=2), case(P, iters=0, it=0), case(SEL, n_modes=0), case(SEL, n_modes=17), case(A, T=-1),
             case(P, group_2_n_param=23), case(P, leader_len=0),
             case(P, x=None), case(P, leader_x=None), case(P, SG=None), case(P, UG=None), case(P, t=None),
             case(P, group_1_params=None), case(P, group_2_xg=None), case(P, group_0_x0=None), case(P, group_0_ug=None),
             case(SEL, active=None), case(SEL, WIN=None), case(SEL, FEAS=None), case(SEL, ND=None),
             case(SEL, group_2_cost=None), case(SEL, group_0_u=None), case(SEL, group_1_x=None), case(SEL, group_2_obj=None),
             case(SEL, group_2_status=None), case(SEL, group_0_nodes=None), case(SEL, group_1_modes=None),
             case(A, active=None), case(A, U_log=None), case(A, u0=None), case(A, gear0=None)]
    before = hvp_ctx.launch_count
    for rig in cases:
        assert L.hvp_event_iter_dev(hvp_ctx.handle, C.byref(rig.g), None) < 0, rig.g.phase
        assert "event_iter" in _lib.last_error()
    assert L.hvp_event_iter_dev(hvp_ctx.handle, None, None) < 0
    # S == 0 is a no-op, not an error
    assert L.hvp_event_iter_dev(hvp_ctx.handle, C.byref(case(SEL, S=0).g), None) == 0
    assert hvp_ctx.launch_count == before
    # the valid versions of the same calls do launch; without gears neither modes nor gear0 nor n_modes are needed
    valid = [case(P), case(SEL, it=1), case(A), case(SEL, gears=False, n_modes=0, group_1_modes=None),
             case(A, gears=False, gear0=None)]
    for rig in valid:
        assert L.hvp_event_iter_dev(hvp_ctx.handle, C.byref(rig.g), None) == 0, _lib.last_error()
    hvp_ctx.synchronize()
    assert hvp_ctx.launch_count == before + len(valid)
