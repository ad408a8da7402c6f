"""Whole-episode closed loops for MANY scenarios at once, state resident on the device (SURVEY.md 8f rank 1;
the batched replacement of the serial loops in n_sweep*.py for the decentralized controller).

One timestep of `BatchedDecentSweep.run` is, for all S scenarios together:
  observe  -- constant-velocity extrapolation of every vehicle's neighbours (fleet_decent_mld.py:348-428)
              and the leader-trajectory window leader_x[:, t:t+N+1] (:329-331), as a handful of torch ops;
  solve    -- the S*n per-vehicle MIQPs in ONE launch of the local-MIQP kernel (hvp_local_miqp_dev);
  step     -- PlatoonEnv.step for all scenarios in ONE launch of the rollout kernel (hvp_rollout_step_dev);
nothing crosses PCIe until the episode's result tensors are read back.  Scenarios are independent, so
multi-GPU runs shard them by rank with no collective (DESIGN.md 6)."""
from __future__ import annotations

import numpy as np

from . import api
from ._lib import FRONT, LEADER, TRAILER, default_context
from .misc import ConstantSpacingPolicy, Params, spacing_params


def _graphs_enabled():
    import os
    return os.environ.get("HVP_SWEEP_GRAPH", "1") != "0"


class _StepGraph:
    """One timestep (or one consensus phase) of a sweep as a CUDA graph.

    `body` is a closure that enqueues a FIXED sequence of launches -- the library's kernels through the C ABI and the
    torch glue between them -- on torch's current stream, reading and writing only tensors that live as long as the
    sweep; everything that changes from step to step (the timestep index, the leader window, where the logs go) is
    addressed through DEVICE-side indices that the body itself advances.  The first `warm` calls run eagerly (they size
    the library's scratch buffers and torch's allocator, neither of which may happen during capture); the next call
    captures the body once and every later call is a single graph launch, so the per-kernel launch and Python costs
    that bounded the closed loops (VERDICT r01: 4.3x between kernel-only and closed-loop g-ADMM) are paid once.
    HVP_SWEEP_GRAPH=0 keeps every call eager (A/B and debugging)."""

    _side = {}          # one capture stream per device, shared by every sweep (the library keeps per-stream launch state)

    def __init__(self, torch, body, warm: int = 1, enabled: bool = True):
        self.torch, self.body, self.warm = torch, body, warm
        self.calls, self.graph = 0, None
        self.enabled = enabled and _graphs_enabled()
        if self.enabled:
            d = torch.cuda.current_device()
            if d not in _StepGraph._side:
                _StepGraph._side[d] = torch.cuda.Stream(device=d)
            self.stream = _StepGraph._side[d]

    def __call__(self):
        torch = self.torch
        if not self.enabled:
            self.body()
            return
        cur = torch.cuda.current_stream()
        if self.calls < self.warm:
            # eager, but already on the stream the capture will use: the library allocates its per-stream launch state
            # (work counter, adoption scratch) on first use, which must not happen during capture
            self.calls += 1
            self.stream.wait_stream(cur)
            with torch.cuda.stream(self.stream):
                self.body()
            cur.wait_stream(self.stream)
            return
        if self.graph is None:
            # No cyclic collection while capturing: a collected handle of an earlier sweep frees device memory in its
            # finaliser, and any cudaFree invalidates a capture in torch's (global) capture mode.  torch.cuda.graph
            # collects once on entry; this keeps it from happening again inside the body.
            import gc
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            was_on = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.graph(g, stream=self.stream):
                    self.body()
            finally:
                if was_on:
                    gc.enable()
            self.graph = g
        self.calls += 1
        self.graph.replay()

    def close(self):
        """Drops the captured graph and the closure NOW.  body <-> graph <-> the run's tensors form reference cycles, so
        without this a finished run's graph (and the private memory pool of its capture) lives until the cycle collector
        gets to it, and the next run's capture allocates beside it: measured 0.92-1.19 s instead of 0.245 s for the
        g-ADMM leg run back to back (scripts/diag_gadmm_repeat.py)."""
        self.graph = None
        self.body = None


class _Fork:
    """Runs independent pieces of a timestep on side streams (fork from / join to torch's current stream; both are
    captured when the surrounding body is being recorded into a CUDA graph).  The launches of the different ROLES of
    a round (front / interior / trailer) are independent -- different compiled formulations, disjoint output slices --
    and the small ones (1 vehicle per scenario) are pure latency next to the interior one."""
    _pool = {}

    def __init__(self, torch, k, enabled: bool = True, private: bool = False, priority: int = 0):
        import os
        self.enabled = enabled and os.environ.get("HVP_SWEEP_FORK", "1") != "0"
        d = torch.cuda.current_device()
        # private: streams of its own (sweeps that run side by side on different streams must not meet on shared ones)
        pool = [] if private else _Fork._pool.setdefault(d, [])
        while self.enabled and len(pool) < k:
            pool.append(torch.cuda.Stream(device=d, priority=priority))
        self.torch, self.streams = torch, pool[:k]

    def run(self, pieces):
        torch = self.torch
        if not self.enabled:
            for piece in pieces:
                piece()
            return
        cur = torch.cuda.current_stream()
        for st, piece in zip(self.streams, pieces):
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                piece()
        for st in self.streams[:len(pieces)]:
            cur.wait_stream(st)


class BatchedDecentSweep:
    """S independent platoons of n vehicles under the decentralized MLD-MPC (TrackingDecentMldCoordinator
    with the constant-velocity estimator), pwa_gear model, horizon N."""

    def __init__(self, n: int, N: int, masses=None, spacing_policy=ConstantSpacingPolicy(50), leader_index: int = 0,
                 d_safe: float = Params.d_safe, device: int = 0, ctx=None, solver: str = "auto", use_hint: bool = False, graph: bool = False, fused=None,
                 batch_hint=None):
        import os
        import torch
        self.torch = torch
        self.use_hint = use_hint
        self.graph = graph
        # fused: the observe step as one CUDA kernel (csrc/coord.cu hvp_decent_observe_dev) instead of ~N + 6 torch launches
        self.fused = (os.environ.get("HVP_SWEEP_FUSED", "1") != "0") if fused is None else bool(fused)
        self.n, self.N, self.leader_index = n, N, leader_index
        self.dev = torch.device("cuda", device)
        self.ctx = ctx or default_context(device)
        self.d0, self.t0 = spacing_params(spacing_policy)
        self.d_safe = d_safe
        self.masses = None if masses is None else np.asarray(masses, dtype=np.float64)   # (n,) or (S,n)
        self.ldesc = api.local_desc(N, self.d0, self.t0)
        # Which kernel solves the local MIQPs.  "local": the specialised per-vehicle kernel (csrc/local_miqp.cu) --
        # fastest on the short-horizon, constant-spacing problems of the headline benchmark.  "compiled": the LOCAL
        # formulation of the compiled-MPC kernel (csrc/pm_kernel.cu), whose interval-hull tightening and splitting of
        # heavy trees over many warps tame the long tail of hard instances -- long horizons and the time-headway policy
        # (N = 10, headway: worst tree 13 000 -> 6 000 nodes, searched by 64 static workers plus every waiting worker that
        # adopts a piece of it; 464 -> 13 ms per timestep of ~3 000 MIQPs).
        if solver not in ("auto", "local", "compiled"):
            raise ValueError("solver must be 'auto', 'local' or 'compiled'")
        # "auto" follows the measured crossover (scripts/diag_mixed.py, n = 10, 5 timesteps, 300 / 4096 scenarios, end of
        # round 2 -- with waiting workers adopting sub-trees the compiled route's tail is short, its throughput is still the
        # lower one, so the crossover depends on the batch):
        #   constant spacing, ms local | compiled:  N = 8: 10 | 23 and 29 | 78;  N = 9: 38 | 33 and 54 | 101;  N = 10: 66 | 46 and 369 | 137
        #   time headway:  N = 6: 18 | 18 and 23 | 62;  N = 7: 48 | 26 and 57 | 97;  N = 8: 123 | 35 and 151 | 158;  N = 9: 605 | 48 and 411 | 270
        # batch_hint = problems per launch the caller expects (None: large).
        if solver == "auto" and os.environ.get("HVP_SWEEP_SOLVER") in ("local", "compiled"):      # A/B runs of the crossover
            solver = os.environ["HVP_SWEEP_SOLVER"]
        small = batch_hint is not None and batch_hint <= 8192
        n_const, n_headway = (9, 7) if small else (10, 8)
        self.use_compiled = solver == "compiled" or (solver == "auto" and (N >= n_const or (self.t0 != 0.0 and N >= n_headway)))
        self.role_groups = []
        if self.use_compiled:
            from ._lib import MPC_LOCAL
            roles: dict = {}
            for i in range(n):
                fl = (FRONT if i == 0 else 0) | (TRAILER if i == n - 1 else 0) | (LEADER if i == leader_index else 0)
                roles.setdefault(fl, []).append(i)
            for fl, idx in roles.items():
                cm = api.CompiledMpc(MPC_LOCAL, N, flags=fl, d0=self.d0, t0=self.t0, ctx=self.ctx)
                self.role_groups.append((cm, torch.as_tensor(idx, device=self.dev), len(idx)))

    def run(self, x0, leader_x, ep_len: int):
        """x0 (S,2n) initial states (e.g. PlatoonEnv.reset of each scenario), leader_x (2,>=ep_len+N+1) shared
        or (S,2,>=ep_len+N+1) per scenario.  Returns dict of numpy arrays: X (T+1,S,2n), U (T,S,n), R (T,S),
        violations (T,S) uint8, errors (T,S) int32, nodes (T,S,n) int32, status (T,S,n) int32."""
        torch, dev, n, N = self.torch, self.dev, self.n, self.N
        f64 = torch.float64
        x = torch.as_tensor(np.ascontiguousarray(x0, dtype=np.float64), device=dev)
        S = x.shape[0]
        B = S * n
        lx = torch.as_tensor(np.ascontiguousarray(leader_x, dtype=np.float64), device=dev)
        if lx.ndim == 2:
            lx = lx.unsqueeze(0).expand(S, -1, -1)
        if lx.shape[2] < ep_len + N + 1:
            raise ValueError("leader trajectory shorter than ep_len + N + 1")
        flags = np.zeros((S, n), np.int32)
        flags[:, 0] |= FRONT; flags[:, -1] |= TRAILER; flags[:, self.leader_index] |= LEADER
        d_flags = torch.as_tensor(flags.reshape(B), device=dev)
        m = np.full((S, n), 800.0) if self.masses is None else np.broadcast_to(self.masses, (S, n))
        d_mass = torch.as_tensor(np.array(m, dtype=np.float64, order="C"), device=dev)
        edesc = api.env_desc(n, self.leader_index, self.d0, self.t0, self.d_safe, True, False, True)
        # per-step work buffers
        xf = torch.zeros((S, n, 2, N + 1), dtype=f64, device=dev)
        xb = torch.zeros((S, n, 2, N + 1), dtype=f64, device=dev)
        xl = torch.zeros((S, n, 2, N + 1), dtype=f64, device=dev)
        pred = torch.empty((S, n, 2, N + 1), dtype=f64, device=dev)
        u = torch.empty((B, N), dtype=f64, device=dev); xs = torch.empty((B, 2, N + 1), dtype=f64, device=dev)
        modes = torch.empty((B, N), dtype=torch.int32, device=dev); obj = torch.empty(B, dtype=f64, device=dev)
        status = torch.empty(B, dtype=torch.int32, device=dev); nodes = torch.empty(B, dtype=torch.int32, device=dev)
        X = torch.empty((ep_len + 1, S, 2 * n), dtype=f64, device=dev)
        U = torch.empty((ep_len, S, n), dtype=f64, device=dev)
        R = torch.empty((ep_len, S), dtype=f64, device=dev)
        V = torch.empty((ep_len, S), dtype=torch.uint8, device=dev)
        E = torch.empty((ep_len, S), dtype=torch.int32, device=dev)
        ND = torch.empty((ep_len, S, n), dtype=torch.int32, device=dev)
        ST = torch.empty((ep_len, S, n), dtype=torch.int32, device=dev)
        X[0] = x
        ts = float(Params.ts)
        # everything a timestep touches is static; the timestep itself is a DEVICE index the body advances
        x_cur = x.clone()
        x_next = torch.empty_like(x_cur)
        u0 = torch.empty((S, n), dtype=f64, device=dev)
        r_t = torch.empty(S, dtype=f64, device=dev); v_t = torch.empty(S, dtype=torch.uint8, device=dev)
        e_t = torch.empty(S, dtype=torch.int32, device=dev)
        nd_t = torch.empty((S, n), dtype=torch.int32, device=dev); st_t = torch.empty((S, n), dtype=torch.int32, device=dev)
        t_idx = torch.zeros(1, dtype=torch.int64, device=dev)
        win = torch.arange(N + 1, dtype=torch.int64, device=dev)
        lxc = lx.contiguous()
        # MIP start of the next timestep: this timestep's optimal region sequences shifted by one stage (-1 = no hint).
        # OFF by default -- measured (r02, 4096 platoons x 20 steps, n = 10, N = 6): 11.9 -> 19.2 nodes per MIQP and 57.8 ->
        # 81.9 ms with the shifted sequence as the first leaf.  The first dive from the root relaxation already lands on a
        # better leaf than last step's shifted sequence does, and a worse first incumbent prunes less; the OPTIMAL
        # sequence as a hint does cut the nodes (tests/test_gpu_local_miqp.py), so the entry stays for callers that have
        # a good start (a Gurobi MIP start is the same kind of advice).
        hint = torch.full((B, N), -1, dtype=torch.int32, device=dev) if self.use_hint else None

        obs = None
        if self.fused:
            from . import _lib
            obs = _lib.DecentObserve()
            obs.n, obs.N, obs.S, obs.leader_index, obs.ts = n, N, S, self.leader_index, ts
            obs.leader_len, obs.leader_per_scenario = lxc.shape[2], 1
            obs.x, obs.leader_x, obs.t = x_cur.data_ptr(), lxc.data_ptr(), t_idx.data_ptr()
            obs.xf, obs.xb, obs.xl = xf.data_ptr(), xb.data_ptr(), xl.data_ptr()

        def body():
            stream = torch.cuda.current_stream().cuda_stream
            xv = x_cur.view(S, n, 2)
            if obs is not None:
                api.decent_observe_device(obs, ctx=self.ctx, stream=stream)
            else:
                # ---- observe: p_{k+1} = p_k + ts v_k (sequential sums, as the reference), v constant ----
                pred[:, :, 0, 0] = xv[:, :, 0]
                pred[:, :, 1, :] = xv[:, :, 1:2]
                for k in range(N):
                    pred[:, :, 0, k + 1] = pred[:, :, 0, k] + ts * pred[:, :, 1, k]
                xf[:, 1:] = pred[:, :-1]
                xb[:, :-1] = pred[:, 1:]
                xl[:, self.leader_index] = lxc.index_select(2, t_idx + win)           # leader_x[:, t:t+N+1] (:329-331)
            # ---- solve all S*n local MIQPs ----
            if self.use_compiled:      # one launch per role (front / interior / trailer, leader where applicable)
                for cm, ii, k in self.role_groups:
                    Bk = S * k
                    params = torch.cat((xf[:, ii].reshape(S, k, -1), xb[:, ii].reshape(S, k, -1),
                                        xl[:, ii].reshape(S, k, -1)), dim=2).reshape(Bk, -1).contiguous()
                    uo = torch.empty((Bk, 1, N), dtype=f64, device=dev); xo = torch.empty((Bk, 1, 2, N + 1), dtype=f64, device=dev)
                    mo = torch.empty((Bk, 1, N), dtype=torch.int32, device=dev); ob = torch.empty(Bk, dtype=f64, device=dev)
                    st = torch.empty(Bk, dtype=torch.int32, device=dev); no = torch.empty(Bk, dtype=torch.int32, device=dev)
                    cm.solve_device(Bk, xv[:, ii].reshape(Bk, 1, 2).contiguous(), d_mass[:, ii].reshape(Bk, 1).contiguous(),
                                    params, None, uo, xo, None, mo, ob, st, no, None, stream=stream)
                    u0[:, ii] = uo.view(S, k, N)[:, :, 0]
                    nd_t[:, ii] = no.view(S, k)
                    st_t[:, ii] = st.view(S, k)
            else:
                api.local_miqp_device(self.ldesc, B, d_flags, d_mass.view(B), x_cur.view(B, 2), xf.view(B, 2, N + 1),
                                      xb.view(B, 2, N + 1), xl.view(B, 2, N + 1), u, xs, modes, obj, status, nodes,
                                      None, ctx=self.ctx, stream=stream, modes_hint=hint)
                if hint is not None:
                    hint[:, :N - 1] = modes[:, 1:]
                    hint[:, N - 1] = modes[:, N - 1]
                u0.copy_(u[:, 0].view(S, n))
                nd_t.copy_(nodes.view(S, n))
                st_t.copy_(status.view(S, n))
            # ---- step every platoon ----
            lead_now = lxc.index_select(2, t_idx).squeeze(2).contiguous()
            api.rollout_step_device(edesc, S, x_cur, u0, None, d_mass, lead_now, x_next, r_t, v_t, e_t, ctx=self.ctx,
                                    stream=stream)
            # ---- logs at the device-side timestep, then advance ----
            X.index_copy_(0, t_idx + 1, x_next.unsqueeze(0))
            U.index_copy_(0, t_idx, u0.unsqueeze(0)); R.index_copy_(0, t_idx, r_t.unsqueeze(0))
            V.index_copy_(0, t_idx, v_t.unsqueeze(0)); E.index_copy_(0, t_idx, e_t.unsqueeze(0))
            ND.index_copy_(0, t_idx, nd_t.unsqueeze(0)); ST.index_copy_(0, t_idx, st_t.unsqueeze(0))
            x_cur.copy_(x_next)
            t_idx.add_(1)

        # measured (r02): this loop is kernel-bound (one MIQP launch of S*n problems per timestep), eager 54 ms vs graph 59 ms
        # for 4096 platoons x 20 steps -- the graph is off by default here and on where the glue dominates (g-ADMM)
        step = _StepGraph(torch, body, enabled=self.graph)
        for t in range(ep_len):
            step()
        torch.cuda.synchronize()
        step.close()
        return dict(X=X.cpu().numpy(), U=U.cpu().numpy(), R=R.cpu().numpy(), violations=V.cpu().numpy(),
                    errors=E.cpu().numpy(), nodes=ND.cpu().numpy(), status=ST.cpu().numpy())


class MixedSizeDecentSweep:
    """Platoons of DIFFERENT sizes n under the decentralized controller with a common horizon N and spacing policy.
    A per-vehicle MIQP does not depend on n, so every timestep solves the vehicles of ALL platoons in one launch
    (one per role on the compiled route); only observe and the rollout run per platoon size.  This is what keeps the
    GPU filled in the Monte-Carlo sweep of BASELINE.json configs[3], where a (n, N, policy) cell holds ~25 scenarios."""

    def __init__(self, N: int, spacing_policy=ConstantSpacingPolicy(50), leader_index: int = 0,
                 d_safe: float = Params.d_safe, device: int = 0, ctx=None, solver: str = "auto", batch_hint=None):
        import torch
        self.torch, self.N, self.leader_index, self.d_safe = torch, N, leader_index, d_safe
        self.dev = torch.device("cuda", device)
        self.ctx = ctx or default_context(device)
        self.d0, self.t0 = spacing_params(spacing_policy)
        self.ldesc = api.local_desc(N, self.d0, self.t0)
        probe = BatchedDecentSweep(2, N, spacing_policy=spacing_policy, device=device, ctx=self.ctx, solver=solver,
                                   batch_hint=batch_hint)
        self.use_compiled = probe.use_compiled                      # same measured crossover
        self.cms = {}
        self._fork = None

    def _cm(self, fl):
        from ._lib import MPC_LOCAL
        if fl not in self.cms:
            self.cms[fl] = api.CompiledMpc(MPC_LOCAL, self.N, flags=int(fl), d0=self.d0, t0=self.t0, ctx=self.ctx)
        return self.cms[fl]

    def run(self, parts, ep_len: int):
        """parts: list of (n, x0 (S,2n), leader_x (S,2,>=ep_len+N+1), masses (S,n)).  Returns one result dict per
        part with the layout of BatchedDecentSweep.run."""
        self.prepare(parts, ep_len)
        for t in range(ep_len):
            self.step(t)
        return self.finish()

    def prepare(self, parts, ep_len: int):
        """All per-vehicle data lives in FLAT arrays over the vehicles of every platoon (platoon-major, front to back), so
        observe is a handful of torch ops for the whole group; each part's state / result tensors are views into them.
        prepare / step(t) / finish are separate so that several sweeps can be stepped in turn on different CUDA
        streams (run_mixed_sweep): every call only ENQUEUES work on the current torch stream."""
        torch, dev, N, li = self.torch, self.dev, self.N, self.leader_index
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        ts = float(Params.ts)
        T = ep_len
        B = sum(np.asarray(x0).shape[0] * n for n, x0, _, _ in parts)
        Stot = sum(np.asarray(x0).shape[0] for _, x0, _, _ in parts)
        XF = torch.empty((T + 1, B, 2), dtype=f64, device=dev)          # states of every vehicle, every timestep
        UF = torch.empty((T, B), dtype=f64, device=dev)
        NDF = torch.empty((T, B), dtype=i32, device=dev); STF = torch.empty((T, B), dtype=i32, device=dev)
        flags_np = np.zeros(B, np.int32); first_np = np.zeros(B, bool); last_np = np.zeros(B, bool)
        mass_np = np.empty(B); lead_np = []; lxs = []
        st_parts, off, soff = [], 0, 0
        for n, x0, lx, masses in parts:
            x0 = np.ascontiguousarray(x0, dtype=np.float64)
            S = x0.shape[0]
            lx = np.asarray(lx, dtype=np.float64)
            if lx.shape[2] < T + np1:
                raise ValueError("leader trajectory shorter than ep_len + N + 1")
            sl = slice(off, off + S * n)
            fl = np.zeros((S, n), np.int32)
            fl[:, 0] |= FRONT; fl[:, -1] |= TRAILER; fl[:, li] |= LEADER
            flags_np[sl] = fl.reshape(-1)
            fi = np.zeros((S, n), bool); fi[:, 0] = True; first_np[sl] = fi.reshape(-1)
            la = np.zeros((S, n), bool); la[:, -1] = True; last_np[sl] = la.reshape(-1)
            mass_np[sl] = np.ascontiguousarray(masses, dtype=np.float64).reshape(-1)
            lead_np.append(off + np.arange(S) * n + li)
            lxs.append(lx[:, :, :T + np1])
            XF[0, sl] = torch.as_tensor(x0.reshape(S * n, 2), device=dev)
            st_parts.append(dict(n=n, S=S, sl=sl, ssl=slice(soff, soff + S),
                                 edesc=api.env_desc(n, li, self.d0, self.t0, self.d_safe, True, False, True),
                                 R=torch.empty((T, S), dtype=f64, device=dev), V=torch.empty((T, S), dtype=torch.uint8, device=dev),
                                 E=torch.empty((T, S), dtype=i32, device=dev)))
            off += S * n; soff += S
        d_flags = torch.as_tensor(flags_np, device=dev)
        d_mass = torch.as_tensor(mass_np, device=dev)
        not_first = torch.as_tensor(~first_np, device=dev).view(B, 1, 1)
        not_last = torch.as_tensor(~last_np, device=dev).view(B, 1, 1)
        lead_idx = torch.as_tensor(np.concatenate(lead_np) if lead_np else np.zeros(0, np.int64), device=dev)
        # leader trajectories of every scenario, time-major so that a window / a column is one contiguous slice
        LX = torch.as_tensor(np.ascontiguousarray(np.concatenate(lxs, 0).transpose(2, 0, 1)) if lxs else np.zeros((T + np1, 0, 2)),
                             device=dev)                                                     # (T+N+1, Stot, 2)
        xf = torch.zeros((B, 2, np1), dtype=f64, device=dev); xb = torch.zeros((B, 2, np1), dtype=f64, device=dev)
        xl = torch.zeros((B, 2, np1), dtype=f64, device=dev); pred = torch.empty((B, 2, np1), dtype=f64, device=dev)
        u = torch.empty((B, N), dtype=f64, device=dev); xs = torch.empty((B, 2, np1), dtype=f64, device=dev)
        modes = torch.empty((B, N), dtype=i32, device=dev); obj = torch.empty(B, dtype=f64, device=dev)
        status = torch.empty(B, dtype=i32, device=dev); nodes = torch.empty(B, dtype=i32, device=dev)
        roles = [(int(fl), torch.as_tensor(np.nonzero(flags_np == fl)[0], device=dev)) for fl in np.unique(flags_np)] \
            if self.use_compiled else []
        zero = torch.zeros((), dtype=f64, device=dev)
        self._w = dict(T=T, B=B, XF=XF, UF=UF, NDF=NDF, STF=STF, st_parts=st_parts, d_flags=d_flags, d_mass=d_mass,
                       not_first=not_first, not_last=not_last, lead_idx=lead_idx, LX=LX, xf=xf, xb=xb, xl=xl, pred=pred, u=u,
                       xs=xs, modes=modes, obj=obj, status=status, nodes=nodes, roles=roles, zero=zero)

    def step(self, t: int):
        """Enqueue timestep t (observe, solve, rollout) on the current torch stream."""
        torch, dev, N = self.torch, self.dev, self.N
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        ts = float(Params.ts)
        w = self._w
        B, XF, UF, d_mass, pred, xf, xb, xl, u = w["B"], w["XF"], w["UF"], w["d_mass"], w["pred"], w["xf"], w["xb"], w["xl"], w["u"]
        status, nodes, LX = w["status"], w["nodes"], w["LX"]
        stream = torch.cuda.current_stream().cuda_stream
        x = XF[t]
        # ---- observe, for the vehicles of every platoon at once (fleet_decent_mld.py:348-428) ----
        pred[:, 0, 0] = x[:, 0]
        pred[:, 1, :] = x[:, 1:2]
        for k in range(N):
            pred[:, 0, k + 1] = pred[:, 0, k] + ts * pred[:, 1, k]
        if B > 1:
            xf[1:] = torch.where(w["not_first"][1:], pred[:-1], w["zero"])     # the vehicle in front, none for a platoon's first
            xb[:-1] = torch.where(w["not_last"][:-1], pred[1:], w["zero"])     # the vehicle behind, none for a platoon's last
        xl[w["lead_idx"]] = LX[t:t + np1].permute(1, 2, 0)                     # leader window leader_x[:, t:t+N+1]
        # ---- ONE solve for the vehicles of every platoon ----
        if self.use_compiled:
            # one launch sequence per role (front / interior / trailer, leader), each formulation with its own handle and
            # scratch: independent, so they run on forked streams -- the budgeted pass of a small role (a few hundred
            # trees, 2-4 ms of pure latency) hides behind the interior one instead of following it
            def role(fl, ii):
                def piece():
                    Bk = ii.numel()
                    params = torch.cat((xf[ii].reshape(Bk, -1), xb[ii].reshape(Bk, -1), xl[ii].reshape(Bk, -1)), dim=1).contiguous()
                    uo = torch.empty((Bk, 1, N), dtype=f64, device=dev); xo = torch.empty((Bk, 1, 2, np1), dtype=f64, device=dev)
                    mo = torch.empty((Bk, 1, N), dtype=i32, device=dev); ob = torch.empty(Bk, dtype=f64, device=dev)
                    st = torch.empty(Bk, dtype=i32, device=dev); no = torch.empty(Bk, dtype=i32, device=dev)
                    self._cm(fl).solve_device(Bk, x[ii].reshape(Bk, 1, 2).contiguous(), d_mass[ii].reshape(Bk, 1).contiguous(),
                                              params, None, uo, xo, None, mo, ob, st, no, None,
                                              stream=torch.cuda.current_stream().cuda_stream)
                    u[ii] = uo.view(Bk, N); status[ii] = st; nodes[ii] = no
                return piece
            if self._fork is None or len(self._fork.streams) < len(w["roles"]):
                self._fork = _Fork(torch, len(w["roles"]), private=True, priority=-1 if N >= 9 else 0)
            self._fork.run([role(fl, ii) for fl, ii in w["roles"]])
        elif B:
            api.local_miqp_device(self.ldesc, B, w["d_flags"], d_mass, x, xf, xb, xl, u, w["xs"], w["modes"], w["obj"], status,
                                  nodes, None, ctx=self.ctx, stream=stream)
        UF[t] = u[:, 0]; w["NDF"][t] = nodes; w["STF"][t] = status
        # ---- step every platoon: one rollout launch per platoon size, straight into the next state slice ----
        lead_now = LX[t]
        for p in w["st_parts"]:
            S, sl = p["S"], p["sl"]
            api.rollout_step_device(p["edesc"], S, XF[t, sl], UF[t, sl], None, d_mass[sl], lead_now[p["ssl"]],
                                    XF[t + 1, sl], p["R"][t], p["V"][t], p["E"][t], ctx=self.ctx, stream=stream)

    def finish(self):
        """Wait for the device and read the results back (one dict per part)."""
        w = self._w
        T, XF, UF, NDF, STF, st_parts = w["T"], w["XF"], w["UF"], w["NDF"], w["STF"], w["st_parts"]
        self.torch.cuda.synchronize()
        Xh, Uh, Nh, Sh = XF.cpu().numpy(), UF.cpu().numpy(), NDF.cpu().numpy(), STF.cpu().numpy()
        out = []
        for p in st_parts:
            n, S, sl = p["n"], p["S"], p["sl"]
            out.append(dict(X=Xh[:, sl].reshape(T + 1, S, 2 * n), U=Uh[:, sl].reshape(T, S, n), R=p["R"].cpu().numpy(),
                            violations=p["V"].cpu().numpy(), errors=p["E"].cpu().numpy(), nodes=Nh[:, sl].reshape(T, S, n),
                            status=Sh[:, sl].reshape(T, S, n)))
        return out


_MIXED_CACHE: dict = {}          # (ctx, device, N, policy) -> (MixedSizeDecentSweep, its stream, ctx kept alive)


def run_mixed_sweep(scenarios, ep_len: int, rank: int = 0, world: int = 1, device: int = 0, ctx=None):
    """Monte-Carlo sweep over scenarios of MIXED size (BASELINE.json configs[3]): `scenarios` is a list of dicts
    {n, N, x0 (2n,), leader_x (2, >= ep_len+N+1), masses (n,) | None, spacing_policy | None}.  This rank takes
    its load-balanced share (dist.balanced_shards), groups it by (N, spacing policy) -- platoons of every size n
    in one MixedSizeDecentSweep, so a timestep is one solve launch per group, not per (n, N) cell -- and returns
    {scenario index: dict(X (T+1,2n), U (T,n), R (T,), violations, errors, nodes, status)} for its scenarios."""
    from .dist import balanced_shards
    mine = balanced_shards([7 * sc["n"] * sc["N"] for sc in scenarios], world)[rank]
    groups: dict = {}
    for i in mine:
        sc = scenarios[i]
        pol = sc.get("spacing_policy") or ConstantSpacingPolicy(50)
        groups.setdefault((sc["N"], spacing_params(pol)), {}).setdefault(sc["n"], []).append(i)
    import torch
    out, work = {}, []
    for k_, (_, _, cx_) in list(_MIXED_CACHE.items()):          # group objects of a context that has been closed since
        if cx_ is not None and getattr(cx_, "handle", None) is None:
            del _MIXED_CACHE[k_]
    # longest horizons first and on high-priority streams: the N = 10 / time-headway group alone is more than half of the
    # sweep's critical path (scripts/diag_mixed_groups.py), the short-horizon groups fit into its tails
    def weight(item):
        (N_, (d0_, t0_)), _ = item
        return -(N_ + (0.5 if t0_ != 0.0 else 0.0))
    for (N, _), by_n in sorted(groups.items(), key=weight):
        first = next(iter(by_n.values()))[0]
        pol = scenarios[first].get("spacing_policy") or ConstantSpacingPolicy(50)
        parts, index = [], []
        for n, idx in sorted(by_n.items()):
            masses = np.stack([np.full(n, 800.0) if scenarios[i].get("masses") is None
                               else np.asarray(scenarios[i]["masses"], dtype=np.float64) for i in idx])
            parts.append((n, np.stack([scenarios[i]["x0"] for i in idx]), np.stack([scenarios[i]["leader_x"] for i in idx]), masses))
            index.append(idx)
        # The sweep object of a (horizon, policy) group -- its compiled formulations with their device scratch -- and the
        # stream it runs on are kept for the next call: building them is host work and device allocations inside every
        # run, and the library keys its per-stream launch state (work counter, adoption scratch) on the stream handle, of
        # which it keeps 64: fresh streams per run exhausted them after five runs and the later runs lost the adoption
        # scratch of the per-vehicle kernel.
        vehicles = sum(n * len(idx) for n, idx in by_n.items())          # problems per launch of this group
        key = (id(ctx), device, N, spacing_params(pol), vehicles <= 8192)
        if key not in _MIXED_CACHE:
            while len(_MIXED_CACHE) >= 48:                     # bounded: the oldest group object (and its device scratch) goes
                _MIXED_CACHE.pop(next(iter(_MIXED_CACHE)))
            sw = MixedSizeDecentSweep(N, spacing_policy=pol, device=device, ctx=ctx, batch_hint=vehicles)
            _MIXED_CACHE[key] = (sw, torch.cuda.Stream(device=sw.dev, priority=-1 if N >= 9 else 0), ctx)
        sw, stream, _ = _MIXED_CACHE[key]
        with torch.cuda.stream(stream):
            sw.prepare(parts, ep_len)
        work.append((sw, stream, index))
    # The groups are independent and a group's timestep ends in a long tail (its slowest tree): step them in turn, each
    # on its own stream, so that the tails of different groups overlap on the device.
    for t in range(ep_len):
        for sw, stream, _ in work:
            with torch.cuda.stream(stream):
                sw.step(t)
    for sw, stream, index in work:
        with torch.cuda.stream(stream):
            res = sw.finish()
        for r, idx in zip(res, index):
            for j, i in enumerate(idx):
                out[i] = dict(X=r["X"][:, j], U=r["U"][:, j], R=r["R"][:, j], violations=r["violations"][:, j],
                              errors=r["errors"][:, j], nodes=r["nodes"][:, j], status=r["status"][:, j])
    return out


class BatchedAdmmSweep:
    """S independent platoons under the naive (non-convex) ADMM controller (fleet_naive_admm.py:320-587), all
    state on the device.  One timestep = admm_iters rounds; one round = the x-update of all S*n vehicles (one launch
    of the compiled-MPC kernel per distinct role: front / interior / trailer, leader where applicable) followed by
    the z- and y-updates; then one rollout launch.  A vehicle whose solve is not optimal contributes zeros for its
    prediction and its copies and applies zero input (gear 6), as solve_mpc(raises=False) gives it.

    model: "pwa_gear" (gears derived from the velocities) or "pwa_friction" (discrete gears chosen by the MPC; the
    action is [u_g ; gears]).  mip_gap / time_limit_ms: the role solves' options (mpc.OPTIONS in simulate()).
    real_vehicle_as_reference: the rollout's stage cost tracks the real vehicle in front (PlatoonEnv's option).
    fused: the glue of a timestep as the three phases of ONE kernel (hvp_admm_step_dev, csrc/coord.cu) with the
    timestep and round indices on the device; None reads HVP_SWEEP_FUSED (default on).  fused=False keeps the glue as
    torch ops indexed by the host loop, pwa_gear only: the reference the kernel is tested against.
    fork: the roles' solves on forked streams; graph (fused loop): each round replayed as a CUDA graph."""

    def __init__(self, n: int, N: int, admm_iters: int = 20, rho: float = 0.5, masses=None,
                 spacing_policy=ConstantSpacingPolicy(50), leader_index: int = 0, d_safe: float = Params.d_safe,
                 model: str = "pwa_gear", mip_gap: float = 0.0, time_limit_ms: float = 0.0,
                 real_vehicle_as_reference: bool = False, device: int = 0, ctx=None, graph: bool = False,
                 fork: bool = True, fused=None):
        import os
        import torch
        from ._lib import MODEL_FRICTION_GEAR, MODEL_PWA_GEAR, MPC_ADMM
        self.graph, self.fork = graph, fork
        if model not in ("pwa_gear", "pwa_friction"):
            raise ValueError(f"model must be 'pwa_gear' or 'pwa_friction', got {model!r}")
        self.fused = (os.environ.get("HVP_SWEEP_FUSED", "1") != "0") if fused is None else bool(fused)
        self.friction = model == "pwa_friction"
        if self.friction and not self.fused:
            raise ValueError("the torch glue (fused=False) runs the pwa_gear model only")
        if n < 2:
            raise ValueError("the ADMM scheme needs at least two vehicles")
        if self.fused and (n > 64 or admm_iters < 1):
            raise ValueError(f"the fused loop needs n <= 64 and admm_iters >= 1 (n = {n}, admm_iters = {admm_iters})")
        if leader_index != 0 and real_vehicle_as_reference:
            raise NotImplementedError("Not implemented for real vehicle with leader not 0.")   # as PlatoonEnv
        self.torch, self.n, self.N, self.iters, self.rho, self.leader_index = torch, n, N, admm_iters, rho, leader_index
        self.real_ref = bool(real_vehicle_as_reference)
        self.dev = torch.device("cuda", device)
        self.ctx = ctx or default_context(device)
        self.d0, self.t0 = spacing_params(spacing_policy)
        self.d_safe = d_safe
        self.masses = None if masses is None else np.asarray(masses, dtype=np.float64)
        # one compiled formulation per distinct role; vehicles with the same role batch together
        self.role_of = []
        roles: dict = {}
        for i in range(n):
            fl = (FRONT if i == 0 else 0) | (TRAILER if i == n - 1 else 0) | (LEADER if i == leader_index else 0)
            if fl not in roles:
                roles[fl] = api.CompiledMpc(MPC_ADMM, N, model=MODEL_FRICTION_GEAR if self.friction else MODEL_PWA_GEAR,
                                            flags=fl, rho=rho, d0=self.d0, t0=self.t0, mip_gap=mip_gap,
                                            time_limit_ms=time_limit_ms, ctx=self.ctx)
            self.role_of.append(fl)
        self.roles = roles

    def close(self):
        """Releases the compiled formulations (their device scratch)."""
        for cm in self.roles.values():
            cm.close()
        self.roles = {}

    def run(self, x0, leader_x, ep_len: int):
        """x0 (S,2n) initial states, leader_x (2,>=ep_len+N) shared or (S,2,>=ep_len+N) per scenario.  Returns dict of
        numpy arrays: X (T+1,S,2n), U (T,S,n) -- (T,S,2n) = [u_g ; gears] for pwa_friction --, R (T,S), violations (T,S)
        uint8, errors (T,S) int32, status (T,S,n) int32 of the last round, nodes (T,S) int32 (max over the rounds and
        vehicles of a timestep) and failed_at (S,3) int32: (timestep, round, status) of the first solve that was not
        optimal -- the lowest vehicle index within the first such round -- or (-1, -1, 0)."""
        torch, dev, n, N = self.torch, self.dev, self.n, self.N
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        if not self.roles:
            raise RuntimeError("BatchedAdmmSweep is closed")
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        if x0.ndim != 2 or x0.shape[1] != 2 * n:
            raise ValueError(f"x0 must have shape (S, {2 * n}), got {x0.shape}")
        S, T = x0.shape[0], int(ep_len)
        lx_np = np.ascontiguousarray(leader_x, dtype=np.float64)
        if lx_np.ndim not in (2, 3) or lx_np.shape[-2] != 2 or (lx_np.ndim == 3 and lx_np.shape[0] != S):
            raise ValueError(f"leader_x must have shape (2, L) or ({S}, 2, L), got {lx_np.shape}")
        if lx_np.shape[-1] < T + N:
            raise ValueError("leader trajectory shorter than ep_len + N")
        x = torch.as_tensor(x0, device=dev)
        lx = torch.as_tensor(lx_np, device=dev)
        m = np.full((S, n), 800.0) if self.masses is None else np.broadcast_to(self.masses, (S, n))
        d_mass = torch.as_tensor(np.array(m, dtype=np.float64, order="C"), device=dev)
        edesc = api.env_desc(n, self.leader_index, self.d0, self.t0, self.d_safe, True, self.real_ref, True)
        zeros = lambda *s: torch.zeros(s, dtype=f64, device=dev)
        # consensus variables [S][n][2][N+1]: multipliers, the z each vehicle's copies are pulled towards, own predictions
        cons = dict(y_front=zeros(S, n, 2, np1), y_back=zeros(S, n, 2, np1), zf=zeros(S, n, 2, np1),
                    zb=zeros(S, n, 2, np1), xs=zeros(S, n, 2, np1))
        # per-role solve buffers, rows [scenario][vehicle of the role]
        groups = {}
        for fl, cm in self.roles.items():
            idx = [i for i in range(n) if self.role_of[i] == fl]
            k = len(idx); B = S * k
            groups[fl] = dict(cm=cm, idx=torch.as_tensor(idx, device=dev), k=k, B=B,
                              m=d_mass[:, idx].reshape(B, 1).contiguous(),
                              u=torch.empty((B, 1, N), dtype=f64, device=dev), x=torch.empty((B, 1, 2, np1), dtype=f64, device=dev),
                              e=torch.empty((B, max(cm.n_extra, 1)), dtype=f64, device=dev),
                              mo=torch.empty((B, 1, N), dtype=i32, device=dev), ob=torch.empty(B, dtype=f64, device=dev),
                              st=torch.empty(B, dtype=i32, device=dev), no=torch.empty(B, dtype=i32, device=dev))
        X = torch.empty((T + 1, S, 2 * n), dtype=f64, device=dev)
        U = torch.empty((T, S, 2 * n if self.friction else n), dtype=f64, device=dev)
        R = torch.empty((T, S), dtype=f64, device=dev)
        V = torch.empty((T, S), dtype=torch.uint8, device=dev)
        E = torch.empty((T, S), dtype=i32, device=dev)
        ST = torch.empty((T, S, n), dtype=i32, device=dev)
        ND = torch.zeros((T, S), dtype=i32, device=dev)
        FA = torch.tensor([[-1, -1, 0]] * S, dtype=i32, device=dev).reshape(S, 3)
        X[0] = x
        logs = (X, U, R, V, E, ST, ND, FA)
        if self.fused:
            self._run_fused(S, T, x, lx, d_mass, edesc, cons, groups, logs)
        else:
            self._run_torch(S, T, x, lx, d_mass, edesc, cons, groups, logs)
        torch.cuda.synchronize()
        return dict(X=X.cpu().numpy(), U=U.cpu().numpy(), R=R.cpu().numpy(), violations=V.cpu().numpy(),
                    errors=E.cpu().numpy(), status=ST.cpu().numpy(), nodes=ND.cpu().numpy(), failed_at=FA.cpu().numpy())

    def _solve(self, g, x0, params):
        stream = self.torch.cuda.current_stream().cuda_stream
        g["cm"].solve_device(g["B"], x0, g["m"], params, None, g["u"], g["x"], g["e"], g["mo"], g["ob"], g["st"], g["no"],
                             None, stream=stream)

    def _run_fused(self, S, T, x, lx, d_mass, edesc, cons, groups, logs):
        from . import _lib
        torch, dev, n, N = self.torch, self.dev, self.n, self.N
        f64, i32 = torch.float64, torch.int32
        X, U, R, V, E, ST, ND, FA = logs
        g = _lib.AdmmStep()
        g.n, g.N, g.S, g.nroles, g.rho = n, N, S, len(groups), self.rho
        g.leader_per_scenario, g.leader_len, g.T = int(lx.ndim == 3), lx.shape[-1], T
        order = list(groups)
        for i in range(n):
            g.role_of[i] = order.index(self.role_of[i])
        for r, fl in enumerate(order):
            b = groups[fl]
            b["params"] = torch.zeros((b["B"], b["cm"].n_param), dtype=f64, device=dev)
            b["x0"] = torch.zeros((b["B"], 1, 2), dtype=f64, device=dev)
            G = g.role[r]
            for k, key in (("params", "params"), ("x0", "x0"), ("u", "u"), ("x", "x"), ("extra", "e"), ("modes", "mo"),
                           ("status", "st"), ("nodes", "no")):
                setattr(G, k, b[key].data_ptr())
            G.has_front, G.has_back = int(not fl & FRONT), int(not fl & TRAILER)
        table = groups[order[0]]["cm"].mode_gear
        g.n_modes = len(table)
        for k, gear in enumerate(table.tolist()):
            g.mode_gear[k] = gear
        t_idx = torch.zeros(1, dtype=torch.int64, device=dev)
        r_idx = torch.zeros(1, dtype=i32, device=dev)
        u0 = torch.empty((S, n), dtype=f64, device=dev)
        gear0 = torch.empty((S, n), dtype=i32, device=dev) if self.friction else None
        lead_t = torch.empty((S, 2), dtype=f64, device=dev)
        x_cur = x.clone(); x_next = torch.empty_like(x_cur)
        r_t = torch.empty(S, dtype=f64, device=dev); v_t = torch.empty(S, dtype=torch.uint8, device=dev)
        e_t = torch.empty(S, dtype=i32, device=dev)
        g.t, g.r, g.x, g.leader_x = t_idx.data_ptr(), r_idx.data_ptr(), x_cur.data_ptr(), lx.data_ptr()
        for k, t_ in cons.items():
            setattr(g, k, t_.data_ptr())
        g.ND, g.failed_at, g.u0, g.U_log, g.ST = ND.data_ptr(), FA.data_ptr(), u0.data_ptr(), U.data_ptr(), ST.data_ptr()
        g.gear0 = None if gear0 is None else gear0.data_ptr()

        def piece(b):
            return lambda: self._solve(b, b["x0"], b["params"])
        pieces = [piece(b) for b in groups.values()]
        # Measured (r02, 1024 scenarios, n = 15, N = 8, 20 rounds x 3 timesteps): eager 1584 ms, round as a graph 1187 ms,
        # roles on forked streams 976 ms, both 1425 ms -- the MIQP rounds are kernel-bound (2.8 ms per interior launch), what
        # pays is running the two one-vehicle roles beside the interior one; inside a graph the branches did not overlap.
        fork = _Fork(torch, len(pieces), enabled=self.fork)

        def one_round():
            fork.run(pieces)
            api.admm_step_device(g, phase=_lib.ADMM_ROUND, ctx=self.ctx, stream=torch.cuda.current_stream().cuda_stream)
            r_idx.add_(1)

        # one consensus round = one CUDA graph (the role solves + the z / y update): the round, not the timestep, is the
        # unit -- it repeats admm_iters times per timestep with nothing changing but the tensors it updates
        rnd = _StepGraph(torch, one_round, enabled=self.graph)
        stream = torch.cuda.current_stream().cuda_stream
        for _ in range(T):
            r_idx.zero_()
            api.admm_step_device(g, phase=_lib.ADMM_PACK, ctx=self.ctx, stream=stream)
            for _ in range(self.iters):
                rnd()
            api.admm_step_device(g, phase=_lib.ADMM_ADOPT, ctx=self.ctx, stream=stream)
            lead_t.copy_(lx.index_select(-1, t_idx).squeeze(-1))                             # leader_x[:, t]
            api.rollout_step_device(edesc, S, x_cur, u0, gear0, d_mass, lead_t, x_next, r_t, v_t, e_t, ctx=self.ctx,
                                    stream=stream)
            X.index_copy_(0, t_idx + 1, x_next.unsqueeze(0))
            R.index_copy_(0, t_idx, r_t.unsqueeze(0))
            V.index_copy_(0, t_idx, v_t.unsqueeze(0)); E.index_copy_(0, t_idx, e_t.unsqueeze(0))
            x_cur.copy_(x_next)
            t_idx.add_(1)
        torch.cuda.synchronize()
        rnd.close()

    def _run_torch(self, S, T, x, lx, d_mass, edesc, cons, groups, logs):
        torch, dev, n, N, rho = self.torch, self.dev, self.n, self.N, self.rho
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        X, U, R, V, E, ST, ND, FA = logs
        y_front, y_back, zf, zb, xs = (cons[k] for k in ("y_front", "y_back", "zf", "zb", "xs"))
        if lx.ndim == 2:
            lx = lx.unsqueeze(0).expand(S, -1, -1)
        z = torch.zeros((S, n, 2, np1), dtype=f64, device=dev)
        cf, cb = torch.zeros_like(z), torch.zeros_like(z)        # copies x_front / x_back of the last round
        u0 = torch.empty((S, n), dtype=f64, device=dev)
        stat = torch.empty((S, n), dtype=i32, device=dev)
        nd = torch.empty((S, n), dtype=i32, device=dev)
        x_cur = x.clone()                                         # state the rounds of this timestep start from
        lwin = torch.empty((S, 1, 2 * np1), dtype=f64, device=dev)
        three = torch.full((), 3.0, dtype=f64, device=dev)
        zero = torch.zeros((), dtype=f64, device=dev)
        ar = torch.arange(n, device=dev)

        def role_piece(fl, g):
            def piece():
                idx, k, B = g["idx"], g["k"], g["B"]
                params = torch.cat((lwin.expand(S, k, -1), y_front[:, idx].reshape(S, k, -1), zf[:, idx].reshape(S, k, -1),
                                    y_back[:, idx].reshape(S, k, -1), zb[:, idx].reshape(S, k, -1)), dim=2).reshape(B, -1).contiguous()
                x0g = x_cur.view(S, n, 2)[:, idx].reshape(B, 1, 2).contiguous()
                self._solve(g, x0g, params)
                # a solve that is not optimal contributes zeros (solve_mpc(raises=False), LocalMpcADMM._post)
                st = g["st"].view(S, k)
                ok = (st == 2).view(S, k, 1, 1)
                xs[:, idx] = torch.where(ok, g["x"].view(S, k, 2, np1), zero)
                u0[:, idx] = torch.where(ok[:, :, 0, 0], g["u"].view(S, k, N)[:, :, 0], zero)
                stat[:, idx] = st
                nd[:, idx] = g["no"].view(S, k)
                e = g["e"].view(S, k, -1)
                o = 0
                if not fl & FRONT:
                    cf[:, idx] = torch.where(ok, e[:, :, o:o + 2 * np1].reshape(S, k, 2, np1), zero); o += 2 * np1
                if not fl & TRAILER:
                    cb[:, idx] = torch.where(ok, e[:, :, o:o + 2 * np1].reshape(S, k, 2, np1), zero)
            return piece
        pieces = [role_piece(fl, g) for fl, g in groups.items()]
        fork = _Fork(torch, len(pieces), enabled=self.fork)
        stream = torch.cuda.current_stream().cuda_stream
        for t in range(T):
            if t > 0:       # coupling guesses from the previous step's predictions, shifted (fleet_naive_admm.py:392-402)
                sh = torch.cat((xs[..., 1:], xs[..., -1:]), dim=-1)
                zf[:, 1:] = sh[:, :-1]
                zb[:, :-1] = sh[:, 1:]
            lwin.copy_(lx[:, :, t:t + np1].reshape(S, 1, 2 * np1))
            x_cur.copy_(x)
            for r in range(self.iters):
                # ---- x-update: all vehicles of a role in one launch, the roles side by side on forked streams ----
                fork.run(pieces)
                # ---- z-update: average of a vehicle's own prediction and its neighbours' copies of it (:421-447) ----
                z[:, 0] = (xs[:, 0] + cf[:, 1]) / 2.0
                z[:, n - 1] = (xs[:, n - 1] + cb[:, n - 2]) / 2.0
                if n > 2:     # a TRUE division, as numpy's in the reference (torch turns `/ 3.0` into a product with 1/3: one ulp off)
                    z[:, 1:n - 1] = torch.div(xs[:, 1:n - 1] + cf[:, 2:] + cb[:, :n - 2], three)
                # ---- y-update and the z each copy is pulled towards in the next round (:426-468) ----
                y_front[:, 1:] += rho * (cf[:, 1:] - z[:, :-1])
                y_back[:, :-1] += rho * (cb[:, :-1] - z[:, 1:])
                zf[:, 1:] = z[:, :-1]
                zb[:, :-1] = z[:, 1:]
                # ---- logs: largest node count, first solve that was not optimal (lowest vehicle index) ----
                ND[t] = torch.maximum(ND[t], nd.max(dim=1).values)
                bad = stat != 2
                first = torch.where(bad, ar, n).min(dim=1).values
                new = (FA[:, 0] < 0) & (first < n)
                row = torch.stack((torch.full_like(first, t), torch.full_like(first, r),
                                   stat.gather(1, first.clamp(max=n - 1).unsqueeze(1)).squeeze(1)), dim=1).to(i32)
                FA.copy_(torch.where(new.unsqueeze(1), row, FA))
            U[t] = u0
            ST[t] = stat
            api.rollout_step_device(edesc, S, x, U[t], None, d_mass, lx[:, :, t].contiguous(), X[t + 1], R[t], V[t],
                                    E[t], ctx=self.ctx, stream=stream)
            x = X[t + 1]


class BatchedSeqSweep(BatchedDecentSweep):
    """S independent platoons under the SEQUENTIAL MLD-MPC (TrackingSequentialMldCoordinator,
    fleet_seq_mld.py:296-440): per timestep the leader is solved first, then the vehicles in front of it
    (nearest first), then the ones behind -- n waves of S local MIQPs, each wave using the FRESH prediction of
    the neighbour already solved and the shifted previous prediction of the other one."""

    def run(self, x0, leader_x, ep_len: int):
        torch, dev, n, N, li = self.torch, self.dev, self.n, self.N, self.leader_index
        f64, np1 = torch.float64, N + 1
        x = torch.as_tensor(np.ascontiguousarray(x0, dtype=np.float64), device=dev)
        S = x.shape[0]
        lx = torch.as_tensor(np.ascontiguousarray(leader_x, dtype=np.float64), device=dev)
        if lx.ndim == 2:
            lx = lx.unsqueeze(0).expand(S, -1, -1)
        m = np.full((S, n), 800.0) if self.masses is None else np.broadcast_to(self.masses, (S, n))
        d_mass = torch.as_tensor(np.array(m, dtype=np.float64, order="C"), device=dev)
        edesc = api.env_desc(n, li, self.d0, self.t0, self.d_safe, True, False, True)
        ts = float(Params.ts)
        # parameters currently set in each vehicle's controller (persist until overwritten, like the setters)
        xf = torch.zeros((S, n, 2, np1), dtype=f64, device=dev)
        xb = torch.zeros((S, n, 2, np1), dtype=f64, device=dev)
        xl = torch.zeros((S, 2, np1), dtype=f64, device=dev)
        # on_episode_start: constant-velocity extrapolation of the neighbours (fleet_seq_mld.py:411-431)
        xv = x.view(S, n, 2)
        cv = torch.empty((S, n, 2, np1), dtype=f64, device=dev)
        cv[:, :, 0, 0] = xv[:, :, 0]
        cv[:, :, 1, :] = xv[:, :, 1:2]
        for k in range(N):
            cv[:, :, 0, k + 1] = cv[:, :, 0, k] + ts * cv[:, :, 1, k]
        xf[:, 1:] = cv[:, :-1]
        xb[:, :-1] = cv[:, 1:]
        pred = torch.zeros((S, n, 2, np1), dtype=f64, device=dev)      # latest prediction of every vehicle
        have_pred = False
        flags = [(FRONT if i == 0 else 0) | (TRAILER if i == n - 1 else 0) | (LEADER if i == li else 0) for i in range(n)]
        d_flags = [torch.full((S,), f, dtype=torch.int32, device=dev) for f in flags]
        u = torch.empty((S, N), dtype=f64, device=dev); xs = torch.empty((S, 2, np1), dtype=f64, device=dev)
        modes = torch.empty((S, N), dtype=torch.int32, device=dev); obj = torch.empty(S, dtype=f64, device=dev)
        status = torch.empty(S, dtype=torch.int32, device=dev); nodes = torch.empty(S, dtype=torch.int32, device=dev)
        X = torch.empty((ep_len + 1, S, 2 * n), dtype=f64, device=dev)
        U = torch.empty((ep_len, S, n), dtype=f64, device=dev)
        R = torch.empty((ep_len, S), dtype=f64, device=dev)
        V = torch.empty((ep_len, S), dtype=torch.uint8, device=dev)
        E = torch.empty((ep_len, S), dtype=torch.int32, device=dev)
        ND = torch.empty((ep_len, S, n), dtype=torch.int32, device=dev)
        ST = torch.empty((ep_len, S, n), dtype=torch.int32, device=dev)
        X[0] = x
        stream = torch.cuda.current_stream().cuda_stream
        order = [li] + list(range(li - 1, -1, -1)) + list(range(li + 1, n))

        def shifted(p):          # drop column 0, repeat the last, re-extrapolate the last position (:342-344)
            s = torch.cat((p[..., 1:], p[..., -1:]), dim=-1).clone()
            s[:, 0, -1] = s[:, 0, -2] + ts * s[:, 1, -1]
            return s

        for t in range(ep_len):
            xl[:] = lx[:, :, t:t + np1]
            prev = pred.clone()
            for i in order:
                if have_pred:
                    if i != 0:      # front neighbour: fresh if it was solved before me in this step, else shifted
                        xf[:, i] = pred[:, i - 1] if (i > li) else shifted(prev[:, i - 1])
                    if i != n - 1:
                        xb[:, i] = pred[:, i + 1] if (i < li) else shifted(prev[:, i + 1])
                else:               # first step: only the fresh predictions exist (:341, :368, :375)
                    if i > li:
                        xf[:, i] = pred[:, i - 1]
                    if i < li:
                        xb[:, i] = pred[:, i + 1]
                api.local_miqp_device(self.ldesc, S, d_flags[i], d_mass[:, i].contiguous(), x.view(S, n, 2)[:, i].contiguous(),
                                      xf[:, i].contiguous(), xb[:, i].contiguous(), xl, u, xs, modes, obj, status, nodes,
                                      None, ctx=self.ctx, stream=stream)
                pred[:, i] = xs
                U[t, :, i] = u[:, 0]
                ND[t, :, i] = nodes
                ST[t, :, i] = status
            have_pred = True
            api.rollout_step_device(edesc, S, x, U[t], None, d_mass, lx[:, :, t].contiguous(), X[t + 1], R[t], V[t],
                                    E[t], ctx=self.ctx, stream=stream)
            x = X[t + 1]
        torch.cuda.synchronize()
        return dict(X=X.cpu().numpy(), U=U.cpu().numpy(), R=R.cpu().numpy(), violations=V.cpu().numpy(),
                    errors=E.cpu().numpy(), nodes=ND.cpu().numpy(), status=ST.cpu().numpy())


class BatchedGAdmmSweep:
    """S independent platoons under the switching ("g") ADMM controller (fleet_g_admm.py; round logic restated in
    fleet_g_admm.GAdmmCoordinator -- UNVERIFIED-3P).  Every agent holds a fixed PWA region sequence, so a round is
    S*n convex QPs: one launch of the compiled-MPC kernel (fixed_modes path, FP64 tensor-core precompute) per role
    (leader / interior / last); sequences are re-identified from a PWA roll-out of the current inputs as torch ops."""

    def __init__(self, n: int, N: int, admm_iters: int = 100, rho: float = 0.5, masses=None,
                 spacing_policy=ConstantSpacingPolicy(50), d_safe: float = Params.d_safe, device: int = 0, ctx=None,
                 graph: bool = True, fork: bool = False, fused=None):
        import os
        import torch
        from ._lib import MPC_GADMM
        self.graph, self.fork = graph, fork
        # fused: the glue of a round as one CUDA kernel (csrc/coord.cu); False keeps it as torch ops (the reference the
        # fused kernel is tested against)
        self.fused = (os.environ.get("HVP_GADMM_FUSED", "1") != "0") if fused is None else bool(fused)
        from .models import PwaGearVehicle
        if n < 2:
            raise ValueError("the g-ADMM scheme needs at least two vehicles")
        self.torch, self.n, self.N, self.iters, self.rho = torch, n, N, admm_iters, rho
        self.dev = torch.device("cuda", device)
        self.ctx = ctx or default_context(device)
        self.d0, self.t0 = spacing_params(spacing_policy)
        self.d_safe = d_safe
        self.masses = None if masses is None else np.asarray(masses, dtype=np.float64)
        mk = lambda nf, nb, lead: api.CompiledMpc(MPC_GADMM, N, flags=LEADER if lead else 0, n_front=nf, n_behind=nb, rho=rho,
                                                  d0=self.d0, t0=self.t0, ctx=self.ctx)
        self.cm_lead = mk(0, 1, True)
        self.cm_mid = mk(1, 1, False) if n > 2 else None
        self.cm_last = mk(1, 0, False)
        v = PwaGearVehicle(800.0)
        lim = v.v_gear_lim
        f64 = torch.float64
        self.edges = torch.tensor([lim[0], lim[1], lim[2], v.alpha, lim[3], lim[4]], dtype=f64, device=self.dev)
        g = [0, 1, 2, 3, 3, 4, 5]
        self.cf = torch.tensor([v.c1 if r < 4 else v.c2 for r in range(7)], dtype=f64, device=self.dev)
        self.bg = torch.tensor([float(v.b[g[r]]) for r in range(7)], dtype=f64, device=self.dev)
        self.dd = torch.tensor([0.0 if r < 4 else v.d for r in range(7)], dtype=f64, device=self.dev)
        self.mug = v.mu * v.grav

    def _region(self, vel):           # first region whose closed interval (+1e-9) contains v (fleet_g_admm._region_of)
        return self.torch.bucketize(vel, self.edges + 1e-9, right=False)

    def _rollout(self, x, u, mass, tr=None, seq=None):
        """PWA roll-out of all vehicles under inputs u (S,n,N): trajectories (S,n,2,N+1), region sequences (S,n,N)
        (written into `tr` / `seq` when given: the consensus rounds keep them in static tensors)."""
        torch, N = self.torch, self.N
        S, n = u.shape[0], u.shape[1]
        if tr is None:
            tr = torch.empty((S, n, 2, N + 1), dtype=torch.float64, device=self.dev)
            seq = torch.empty((S, n, N), dtype=torch.int64, device=self.dev)
        p, v = x.view(S, n, 2)[:, :, 0].clone(), x.view(S, n, 2)[:, :, 1].clone()
        tr[:, :, 0, 0], tr[:, :, 1, 0] = p, v
        for k in range(N):
            r = self._region(v)
            seq[:, :, k] = r
            a = 1.0 + (-(self.cf[r]) / mass)
            b = self.bg[r] / mass
            c = -self.mug - self.dd[r] / mass
            p, v = p + v, a * v + b * u[:, :, k] + c
            tr[:, :, 0, k + 1], tr[:, :, 1, k + 1] = p, v
        return tr, seq

    def _const_vel_u(self, x, mass):  # PwaGearVehicle.get_u_for_constant_vel (models.py:537-556), vectorised
        S, n = mass.shape
        v = x.view(S, n, 2)[:, :, 1].contiguous()
        r = self.torch.bucketize(v, self.edges + 1e-4, right=False)
        return (1.0 / (self.bg[r] / mass)) * (-(-(self.cf[r]) / mass) * v - (-self.mug - self.dd[r] / mass))

    def _make_admm_fused(self, S, x, mass, lwin):
        """_make_admm with the glue of a round in ONE kernel (csrc/coord.cu, hvp_gadmm_round_dev): a round is the three
        role solves (precompute + QP kernel each) and that kernel -- 7 launches instead of ~290 -- replayed as a graph."""
        from . import _lib
        torch, n, N, dev = self.torch, self.n, self.N, self.dev
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        zer = lambda *s: torch.zeros(s, dtype=f64, device=dev)
        y = zer(S, n, 3, 2, np1); u = zer(S, n, N); tr = zer(S, n, 2, np1); cost = zer(S)
        ok = torch.ones(S, dtype=torch.uint8, device=dev)
        g = _lib.GAdmmRound()
        g.n, g.N, g.S, g.rho, g.mug = n, N, S, self.rho, self.mug
        for k, v in enumerate(self.edges.cpu().tolist()):
            g.edge[k] = v
        for name, t in (("cf", self.cf), ("bg", self.bg), ("dd", self.dd)):
            for k, v in enumerate(t.cpu().tolist()):
                getattr(g, name)[k] = v
        roles = []
        for r, (cm, cnt) in enumerate(((self.cm_lead, 1), (self.cm_last, 1), (self.cm_mid, n - 2))):
            if cnt <= 0:
                continue
            B, na = S * cnt, (3 if r == 2 else 2)
            assert cm.n_param == (1 + 2 * na) * 2 * np1 and cm.n_extra == (na - 1) * 2 * np1
            buf = dict(params=zer(B, cm.n_param), x0=zer(B, 1, 2), mass=zer(B, 1), fm=torch.zeros((B, 1, N), dtype=i32, device=dev),
                       u=zer(B, 1, N), x=zer(B, 1, 2, np1), e=zer(B, cm.n_extra), mo=torch.zeros((B, 1, N), dtype=i32, device=dev),
                       ob=zer(B), st=torch.zeros(B, dtype=i32, device=dev), no=torch.zeros(B, dtype=i32, device=dev))
            R = g.role[r]
            R.params, R.x0, R.mass, R.fixed_modes = (buf[k].data_ptr() for k in ("params", "x0", "mass", "fm"))
            R.u, R.x, R.extra, R.obj, R.status = (buf[k].data_ptr() for k in ("u", "x", "e", "ob", "st"))
            roles.append((cm, B, buf))
        g.x, g.mass, g.lwin = x.data_ptr(), mass.data_ptr(), lwin.data_ptr()
        g.y, g.u, g.tr, g.cost, g.ok = y.data_ptr(), u.data_ptr(), tr.data_ptr(), cost.data_ptr(), ok.data_ptr()
        keep = (y, u, tr, cost, ok, roles, x, mass, lwin)          # the struct holds raw pointers

        def one_round():
            stream = torch.cuda.current_stream().cuda_stream
            for cm, B, b in roles:
                cm.solve_device(B, b["x0"], b["mass"], b["params"], b["fm"], b["u"], b["x"], b["e"], b["mo"], b["ob"],
                                b["st"], b["no"], None, stream=stream)
            api.gadmm_round_device(g, init=False, ctx=self.ctx, stream=stream)

        rnd = _StepGraph(torch, one_round, enabled=self.graph)

        def admm(u_start):
            _ = keep
            u.copy_(u_start)
            api.gadmm_round_device(g, init=True, ctx=self.ctx, stream=torch.cuda.current_stream().cuda_stream)
            for _r in range(self.iters):
                rnd()
            infeas = ((tr[:, :, 1, 1:] > 45.84 + 1e-6) | (tr[:, :, 1, 1:] < 3.94 - 1e-6)).any(dim=2).any(dim=1)
            return u.clone(), cost.clone(), ok.bool() & ~infeas

        admm.close = rnd.close
        return admm

    def _make_admm(self, S, x, mass, lwin):
        """g_admm_control for all S scenarios (fleet_g_admm.py:255-301 + the restated round logic): returns
        admm(u_start) -> (u (S,n,N), cost (S,), ok (S,) bool).  x (S,2n), mass (S,n) and lwin (S,2,N+1) are STATIC
        tensors the caller refreshes per timestep; every consensus variable lives in a static tensor too, so ONE
        ROUND -- the fixed-sequence QPs of all agents (one launch of the compiled-MPC kernel per role, FP64 tensor-core
        precompute), the z / y updates and the re-identification of the PWA sequences -- is one CUDA graph that is
        replayed admm_iters times per warm start."""
        if self.fused:
            return self._make_admm_fused(S, x, mass, lwin)
        torch, n, N, rho, dev = self.torch, self.n, self.N, self.rho, self.dev
        f64, np1 = torch.float64, N + 1
        zer = lambda *s: torch.zeros(s, dtype=f64, device=dev)
        # augmented blocks per vehicle: [front copy (i > 0), own, back copy (i < n-1)], y and z alike
        yF, yO, yB = zer(S, n, 2, np1), zer(S, n, 2, np1), zer(S, n, 2, np1)
        u = zer(S, n, N)
        tr = zer(S, n, 2, np1); seq = torch.zeros((S, n, N), dtype=torch.int64, device=dev)
        zbar = zer(S, n, 2, np1)
        ok = torch.ones(S, dtype=torch.bool, device=dev)
        cost = zer(S)
        own, cF, cB = zer(S, n, 2, np1), zer(S, n, 2, np1), zer(S, n, 2, np1)
        cnt = torch.ones(n, dtype=f64, device=dev); cnt[:-1] += 1; cnt[1:] += 1
        groups = [(self.cm_lead, [0]), (self.cm_last, [n - 1])] + ([(self.cm_mid, list(range(1, n - 1)))] if n > 2 else [])
        groups = [(cm, idx, torch.as_tensor(idx, device=dev)) for cm, idx in groups]

        okp = [torch.ones(S, dtype=torch.bool, device=dev) for _ in groups]
        costp = [zer(S) for _ in groups]

        def role_piece(j, cm, idx, ii):
            def piece():
                stream = torch.cuda.current_stream().cuda_stream
                k = len(idx); B = S * k
                blocks_y, blocks_z = [], []
                if idx[0] > 0:
                    blocks_y.append(yF[:, ii]); blocks_z.append(zbar[:, ii - 1])
                blocks_y.append(yO[:, ii]); blocks_z.append(zbar[:, ii])
                if idx[-1] < n - 1:
                    blocks_y.append(yB[:, ii]); blocks_z.append(zbar[:, ii + 1])
                params = torch.cat([lwin.reshape(S, 1, 2 * np1).expand(S, k, -1)] + [b.reshape(S, k, -1) for b in blocks_y]
                                   + [b.reshape(S, k, -1) for b in blocks_z], dim=2).reshape(B, -1).contiguous()
                x0g = x.view(S, n, 2)[:, ii].reshape(B, 1, 2).contiguous()
                mg = mass[:, ii].reshape(B, 1).contiguous()
                fm = seq[:, ii].reshape(B, 1, N).to(torch.int32).contiguous()
                uo = torch.empty((B, 1, N), dtype=f64, device=dev); xo = torch.empty((B, 1, 2, np1), dtype=f64, device=dev)
                eo = torch.empty((B, max(cm.n_extra, 1)), dtype=f64, device=dev)
                mo = torch.empty((B, 1, N), dtype=torch.int32, device=dev); ob = torch.empty(B, dtype=f64, device=dev)
                st = torch.empty(B, dtype=torch.int32, device=dev); no = torch.empty(B, dtype=torch.int32, device=dev)
                cm.solve_device(B, x0g, mg, params, fm, uo, xo, eo, mo, ob, st, no, None, stream=stream)
                good = (st == 2).view(S, k)
                okp[j].copy_(good.all(dim=1))
                costp[j].copy_(torch.where(good, ob.view(S, k), torch.zeros_like(ob.view(S, k))).sum(dim=1))
                u[:, ii] = torch.where(good.unsqueeze(-1), uo.view(S, k, N), u[:, ii])
                own[:, ii] = xo.view(S, k, 2, np1)
                e = eo.view(S, k, -1)
                o = 0
                if idx[0] > 0:
                    cF[:, ii] = e[:, :, o:o + 2 * np1].reshape(S, k, 2, np1); o += 2 * np1
                if idx[-1] < n - 1:
                    cB[:, ii] = e[:, :, o:o + 2 * np1].reshape(S, k, 2, np1)
            return piece

        pieces = [role_piece(j, cm, idx, ii) for j, (cm, idx, ii) in enumerate(groups)]
        # Measured (r02, 1024 scenarios, n = 15, N = 8, 100 rounds): eager 689 ms, round as a graph 629 ms, forked roles 1086 ms,
        # both 696 ms -- the QP rounds are a few hundred tiny launches, which the graph removes and forking only adds to.
        fork = _Fork(torch, len(pieces), enabled=self.fork)

        def one_round():
            # the roles (leader / last / interior) side by side on forked streams, then the shared sums in group order
            fork.run(pieces)
            cost.zero_()
            for j in range(len(groups)):
                ok.logical_and_(okp[j])
                cost.add_(costp[j])
            # z-update: average of every copy of vehicle j's trajectory (own, the copy held by j+1, the one held by j-1)
            acc = own.clone()
            acc[:, :-1] += cF[:, 1:]
            acc[:, 1:] += cB[:, :-1]
            torch.div(acc, cnt.view(1, n, 1, 1), out=zbar)
            # y-update on every block with the new z
            yO.add_(rho * (own - zbar))
            yF[:, 1:] += rho * (cF[:, 1:] - zbar[:, :-1])
            yB[:, :-1] += rho * (cB[:, :-1] - zbar[:, 1:])
            self._rollout(x, u, mass, tr, seq)

        rnd = _StepGraph(torch, one_round, enabled=self.graph)

        def admm(u_start):
            for t_ in (yF, yO, yB, own, cF, cB):
                t_.zero_()
            u.copy_(u_start)
            self._rollout(x, u, mass, tr, seq)
            zbar.copy_(tr)
            ok.fill_(True)
            for _ in range(self.iters):
                rnd()
            infeas = ((tr[:, :, 1, 1:] > 45.84 + 1e-6) | (tr[:, :, 1, 1:] < 3.94 - 1e-6)).any(dim=2).any(dim=1)
            return u.clone(), cost.clone(), ok & ~infeas

        admm.close = rnd.close

        return admm

    def close(self):
        """Releases the cached consensus round (static buffers + captured graph) of the last batch size."""
        cached = getattr(self, "_round", None)
        if cached is not None:
            cached[4].close()
            self._round = None

    def run(self, x0, leader_x, ep_len: int, strict: bool = False):
        torch, dev, n, N = self.torch, self.dev, self.n, self.N
        f64, np1 = torch.float64, N + 1
        x = torch.as_tensor(np.ascontiguousarray(x0, dtype=np.float64), device=dev)
        S = x.shape[0]
        lx = torch.as_tensor(np.ascontiguousarray(leader_x, dtype=np.float64), device=dev)
        if lx.ndim == 2:
            lx = lx.unsqueeze(0).expand(S, -1, -1)
        m = np.full((S, n), 800.0) if self.masses is None else np.broadcast_to(self.masses, (S, n))
        mass = torch.as_tensor(np.array(m, dtype=np.float64, order="C"), device=dev)
        edesc = api.env_desc(n, 0, self.d0, self.t0, self.d_safe, True, False, True)
        X = torch.empty((ep_len + 1, S, 2 * n), dtype=f64, device=dev)
        U = torch.empty((ep_len, S, n), dtype=f64, device=dev)
        R = torch.empty((ep_len, S), dtype=f64, device=dev)
        V = torch.empty((ep_len, S), dtype=torch.uint8, device=dev)
        E = torch.empty((ep_len, S), dtype=torch.int32, device=dev)
        OK = torch.empty((ep_len, S), dtype=torch.bool, device=dev)
        WS = torch.empty((ep_len, S), dtype=torch.int32, device=dev)
        X[0] = x
        stream = torch.cuda.current_stream().cuda_stream
        prev = None
        # The consensus round (its static buffers and, with graph=True, the captured CUDA graph) is kept for the next run
        # of the same batch size: a capture costs a device synchronisation, a collection and torch.cuda.empty_cache()
        # (torch.cuda.graph does all three on entry), which made one run in six take 0.56-0.65 s instead of 0.245 s.
        cached = getattr(self, "_round", None)
        if cached is not None and cached[0] == S:
            _, x_cur, mass_c, lwin, admm = cached
            x_cur.copy_(x); mass_c.copy_(mass); mass = mass_c
        else:
            self.close()
            x_cur = x.clone()
            lwin = torch.empty((S, 2, np1), dtype=f64, device=dev)
            admm = self._make_admm(S, x_cur, mass, lwin)
            self._round = (S, x_cur, mass, lwin, admm)
        for t in range(ep_len):
            lwin.copy_(lx[:, :, t:t + np1])
            x_cur.copy_(x)
            starts = [self._const_vel_u(x, mass).unsqueeze(-1).expand(S, n, N).clone()]
            if prev is not None:        # shifted previous solution (fleet_g_admm.py:266-272)
                starts.append(torch.cat((prev[..., 1:], prev[..., -1:]), dim=-1))
            best_cost = torch.full((S,), float("inf"), dtype=f64, device=dev)
            best_u = torch.zeros((S, n, N), dtype=f64, device=dev)
            which = torch.zeros(S, dtype=torch.int32, device=dev)
            for w, u in enumerate(starts):
                uu, cost, ok = admm(u)
                cost = torch.where(ok, cost, torch.full_like(cost, float("inf")))
                better = cost < best_cost
                best_cost = torch.where(better, cost, best_cost)
                best_u = torch.where(better.view(S, 1, 1), uu, best_u)
                which = torch.where(better, torch.full_like(which, w + 1), which)
            OK[t] = torch.isfinite(best_cost)
            WS[t] = which
            prev = best_u
            U[t] = best_u[:, :, 0]
            api.rollout_step_device(edesc, S, x, U[t], None, mass, lx[:, :, t].contiguous(), X[t + 1], R[t], V[t], E[t],
                                    ctx=self.ctx, stream=stream)
            x = X[t + 1]
        torch.cuda.synchronize()
        solved = OK.cpu().numpy()
        # The reference RAISES when no warm start of a timestep yields a solution (fleet_g_admm.py:295-297); a batch
        # cannot stop for one scenario, so the outcome is reported instead of hidden: status 2 / 3 per (timestep,
        # scenario) with the Gurobi codes of include/hvp.h, and the first failing timestep of every scenario (-1: none).
        # From that timestep on the scenario's inputs are the zeros the failed step applied -- NOT what the reference
        # would have produced (it has no trajectory there); strict=True turns any failure into the reference's error.
        bad = ~solved
        aborted_at = np.where(bad.any(axis=0), bad.argmax(axis=0), -1).astype(np.int32)
        if strict and bad.any():
            who = np.nonzero(aborted_at >= 0)[0]
            raise RuntimeError(f"No solution found for any of the warm starts: scenarios {who[:8].tolist()}"
                               f"{' ...' if len(who) > 8 else ''} (first at timestep {int(aborted_at[who].min())})")
        return dict(X=X.cpu().numpy(), U=U.cpu().numpy(), R=R.cpu().numpy(), violations=V.cpu().numpy(),
                    errors=E.cpu().numpy(), solved=solved, status=np.where(solved, 2, 3).astype(np.int32),
                    aborted_at=aborted_at, best_warm_start=WS.cpu().numpy())


def friction_gear_from_velocity(v):
    """PwaFrictionVehicle.get_gear_from_velocity over a float64 torch tensor of velocities (any device): gear 1 below
    v_min, 6 above v_max, else the first gear whose OPEN window (vl, vh) contains v.  0 where the scalar method raises
    (v on an end of the velocity range that no open window contains)."""
    import torch
    from .models import Vehicle
    g = torch.zeros(v.shape, dtype=torch.int64, device=v.device)
    for i in reversed(range(len(Vehicle.b))):
        g = torch.where((Vehicle.vl[i] < v) & (v < Vehicle.vh[i]), i + 1, g)
    g = torch.where(v > Vehicle.v_max, 6, g)
    return torch.where(v < Vehicle.v_min, 1, g)


def friction_const_vel_u(v, gear, mass):
    """PwaFrictionVehicle.get_u_for_constant_vel(v, gear) over torch tensors of the same shape (any device), in the
    scalar method's order of operations: (1 / (b_j * (1 / m))) * (-A_r[1, 1] v - c_r[1]) with friction region
    r = 0 for v <= alpha, else 1."""
    import torch
    from .models import PwaFrictionVehicle as V
    f64 = torch.float64
    b = torch.tensor(V.b, dtype=f64, device=v.device)[gear - 1]
    hi = v > V.alpha
    # tensor / tensor only: torch evaluates `scalar / tensor` as a reciprocal times the scalar (two roundings)
    a = -(-torch.tensor([V.c1, V.c2], dtype=f64, device=v.device)[hi.long()] / mass)
    mug = -V.mu * V.grav
    c = torch.where(hi, mug - torch.full_like(mass, V.d) / mass, torch.full_like(mass, mug))
    return (1 / (b * (1 / mass))) * (a * v - c)


class BatchedEventSweep:
    """S independent platoons under the event-based controller (fleet_event_based.py:413-646), state and guesses
    resident on the device.  One iteration = for every distinct local formulation (agents grouped by vehicles in
    front / behind and relative leader position) ONE eval_cost launch and ONE MIQP launch over S x agents problems,
    then the winner selection (largest cost decrease above `threshold`, first agent on ties) and the overwrite of
    the shared guesses.  A scenario whose iteration found no improver is left unchanged by the remaining iterations of
    the timestep, which is the reference's `break`.

    model: "pwa_gear" (gears derived from the velocities) or "pwa_friction" (discrete gears chosen by the MPC; the
    action is [u_g ; gears]).  fused: the glue of an iteration as the three phases of ONE kernel (hvp_event_iter_dev,
    csrc/coord.cu), with no host synchronisation until the results are read back; None reads HVP_SWEEP_FUSED (default
    on).  fused=False keeps the glue as torch ops, pwa_gear only: the reference the kernel is tested against.
    fork / graph (fused loop): the groups' eval and solve launches on forked streams / each iteration replayed as a CUDA
    graph; off by default, the A/B arms of scripts/time_event_sweep.py (DESIGN.md 5b)."""

    def __init__(self, n: int, N: int, event_iters: int = 4, masses=None, spacing_policy=ConstantSpacingPolicy(50),
                 leader_index: int = 0, d_safe: float = Params.d_safe, threshold: float = 10.0, model: str = "pwa_gear",
                 mip_gap: float = 0.0, time_limit_ms: float = 0.0, device: int = 0, ctx=None, fused=None,
                 fork: bool = False, graph: bool = False):
        import os
        import torch
        from ._lib import MODEL_FRICTION_GEAR, MODEL_PWA_GEAR, MPC_EVENT, NO_LEADER
        self.fork, self.graph = fork, graph
        if model not in ("pwa_gear", "pwa_friction"):
            raise ValueError(f"model must be 'pwa_gear' or 'pwa_friction', got {model!r}")
        self.fused = (os.environ.get("HVP_SWEEP_FUSED", "1") != "0") if fused is None else bool(fused)
        self.friction = model == "pwa_friction"
        if self.friction and not self.fused:
            raise ValueError("the torch glue (fused=False) runs the pwa_gear model only")
        if n < 2:
            raise ValueError("the event-based scheme needs at least two vehicles")
        if self.fused and (n > 64 or event_iters < 1):
            raise ValueError(f"the fused loop needs n <= 64 and event_iters >= 1 (n = {n}, event_iters = {event_iters})")
        self.torch, self.n, self.N, self.iters, self.leader_index = torch, n, N, event_iters, leader_index
        self.threshold = float(threshold)
        self.dev = torch.device("cuda", device)
        self.ctx = ctx or default_context(device)
        self.d0, self.t0 = spacing_params(spacing_policy)
        self.d_safe = d_safe
        self.masses = None if masses is None else np.asarray(masses, dtype=np.float64)
        # agents with the same local structure share one compiled formulation (fleet_event_based.py:700-723)
        self.members = [[0, 1] if i == 0 else ([n - 2, n - 1] if i == n - 1 else [i - 1, i, i + 1]) for i in range(n)]
        if n == 2:
            self.members = [[0, 1], [0, 1]]
        groups: dict = {}
        for i in range(n):
            nf = i if i < 2 else 2
            nb = (n - 1) - i if i > n - 3 else 2
            rl = (-1 if i == leader_index - 1 else (0 if i == leader_index else (1 if i == leader_index + 1 else None)))
            groups.setdefault((nf, nb, rl, len(self.members[i])), []).append(i)
        self.groups = []
        for (nf, nb, rl, nl), idx in groups.items():
            cm = api.CompiledMpc(MPC_EVENT, N, n_local=nl, model=MODEL_FRICTION_GEAR if self.friction else MODEL_PWA_GEAR,
                                 leader_index=NO_LEADER if rl is None else rl, n_front=nf, n_behind=nb, d0=self.d0,
                                 t0=self.t0, mip_gap=mip_gap, time_limit_ms=time_limit_ms, ctx=self.ctx)
            self.groups.append((cm, idx, nl, nf, nb, rl))
        from .models import PwaGearVehicle
        v = PwaGearVehicle(800.0)
        lim = v.v_gear_lim
        f64 = torch.float64
        self.edges = torch.tensor([lim[0], lim[1], lim[2], v.alpha, lim[3], lim[4]], dtype=f64, device=self.dev)
        g = [0, 1, 2, 3, 3, 4, 5]
        self.cf = torch.tensor([v.c1 if r < 4 else v.c2 for r in range(7)], dtype=f64, device=self.dev)
        self.bg = torch.tensor([float(v.b[g[r]]) for r in range(7)], dtype=f64, device=self.dev)
        self.dd = torch.tensor([0.0 if r < 4 else v.d for r in range(7)], dtype=f64, device=self.dev)
        self.mug = v.mu * v.grav

    _const_vel_u = BatchedGAdmmSweep._const_vel_u

    def close(self):
        """Releases the compiled formulations (their device scratch)."""
        for cm, *_ in self.groups:
            cm.close()
        self.groups = []

    def run(self, x0, leader_x, ep_len: int):
        """x0 (S,2n) initial states, leader_x (2,>=ep_len+N+1) shared or (S,2,>=ep_len+N+1) per scenario.  Returns dict
        of numpy arrays: X (T+1,S,2n), U (T,S,n) -- (T,S,2n) = [u_g ; gears] for pwa_friction --, R (T,S), violations,
        errors, winners (T,S,event_iters) int32 (-1: nobody improved, or the scenario had stopped iterating), feasible
        (T,S) bool (False: an iteration in which no agent's MIQP was solved, where simulate() raises), nodes (T,S) int32
        (max over iterations and agents)."""
        torch, dev, n, N = self.torch, self.dev, self.n, self.N
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        if not self.groups:
            raise RuntimeError("BatchedEventSweep is closed")
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        if x0.ndim != 2 or x0.shape[1] != 2 * n:
            raise ValueError(f"x0 must have shape (S, {2 * n}), got {x0.shape}")
        S = x0.shape[0]
        lx_np = np.ascontiguousarray(leader_x, dtype=np.float64)
        if lx_np.ndim not in (2, 3) or lx_np.shape[-2] != 2 or (lx_np.ndim == 3 and lx_np.shape[0] != S):
            raise ValueError(f"leader_x must have shape (2, L) or ({S}, 2, L), got {lx_np.shape}")
        if lx_np.shape[-1] < ep_len + np1:
            raise ValueError("leader trajectory shorter than ep_len + N + 1")
        m = np.full((S, n), 800.0) if self.masses is None else np.broadcast_to(self.masses, (S, n))
        m = np.array(m, dtype=np.float64, order="C")
        # first guesses: constant velocity, constant-velocity throttle (fleet_event_based.py:620-634); with discrete
        # gears the gear of the velocity and the throttle in that gear, computed on the host before anything is queued
        gear = None
        if self.friction:
            v_h, m_h = torch.as_tensor(x0[:, 1::2]), torch.as_tensor(m)
            gear = friction_gear_from_velocity(v_h)
            if (gear == 0).any():
                s_, i_ = (int(a) for a in torch.nonzero(gear == 0)[0])
                raise ValueError(f"No gear found for velocity {x0[s_, 2 * i_ + 1]} (scenario {s_}, vehicle {i_})")
            u_first = friction_const_vel_u(v_h, gear, m_h)
        x = torch.as_tensor(x0, device=dev)
        lx = torch.as_tensor(lx_np, device=dev)
        mass = torch.as_tensor(m, device=dev)
        edesc = api.env_desc(n, self.leader_index, self.d0, self.t0, self.d_safe, True, False, True)
        w = 2 * n if self.friction else n
        X = torch.empty((ep_len + 1, S, 2 * n), dtype=f64, device=dev)
        U = torch.empty((ep_len, S, w), dtype=f64, device=dev)
        R = torch.empty((ep_len, S), dtype=f64, device=dev)
        V = torch.empty((ep_len, S), dtype=torch.uint8, device=dev)
        E = torch.empty((ep_len, S), dtype=i32, device=dev)
        WIN = torch.full((ep_len, S, self.iters), -1, dtype=i32, device=dev)
        FEAS = torch.ones((ep_len, S), dtype=torch.bool, device=dev)
        ND = torch.zeros((ep_len, S), dtype=i32, device=dev)
        X[0] = x
        ts = float(Params.ts)
        xv = x.view(S, n, 2)
        SG = torch.empty((S, n, 2, np1), dtype=f64, device=dev)
        SG[:, :, 0, 0] = xv[:, :, 0]
        SG[:, :, 1, :] = xv[:, :, 1:2]
        for k in range(N):
            SG[:, :, 0, k + 1] = SG[:, :, 0, k] + ts * SG[:, :, 1, k]
        if self.friction:
            UG = u_first.to(dev).unsqueeze(-1).expand(S, n, N).contiguous()
            GG = gear.to(device=dev, dtype=i32).unsqueeze(-1).expand(S, n, N).contiguous()
        else:
            UG = self._const_vel_u(x, mass).unsqueeze(-1).expand(S, n, N).contiguous()
            GG = None
        logs = (X, U, R, V, E, WIN, FEAS, ND)
        if self.fused:
            self._run_fused(S, ep_len, x, lx, mass, edesc, SG, UG, GG, logs)
        else:
            self._run_torch(S, ep_len, x, lx, mass, edesc, SG, UG, logs)
        torch.cuda.synchronize()
        return dict(X=X.cpu().numpy(), U=U.cpu().numpy(), R=R.cpu().numpy(), violations=V.cpu().numpy(),
                    errors=E.cpu().numpy(), winners=WIN.cpu().numpy(), feasible=FEAS.cpu().numpy(), nodes=ND.cpu().numpy())

    def _run_fused(self, S, ep_len, x, lx, mass, edesc, SG, UG, GG, logs):
        from . import _lib
        torch, dev, n, N = self.torch, self.dev, self.n, self.N
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        X, U, R, V, E, WIN, FEAS, ND = logs
        g = _lib.EventIter()
        g.n, g.N, g.S, g.iters, g.ngroups = n, N, S, self.iters, len(self.groups)
        g.leader_per_scenario, g.leader_len, g.T, g.threshold = int(lx.ndim == 3), lx.shape[-1], ep_len, self.threshold
        table = self.groups[0][0].mode_gear
        g.n_modes = len(table)
        for k, gear in enumerate(table.tolist()):
            g.mode_gear[k] = gear
        # eval / solve buffers of every group, allocated once per run; rows [scenario][agent of the group]
        bufs = []
        for gi, (cm, idx, nl, nf, nb, rl) in enumerate(self.groups):
            B = S * len(idx)
            mm = torch.as_tensor([self.members[i] for i in idx], device=dev)
            e = lambda *s, dt=f64: torch.empty(s, dtype=dt, device=dev)
            b = dict(cm=cm, B=B, x0=e(B, nl, 2), xg=e(B, nl, 2, np1), ug=e(B, nl, N),
                     params=torch.zeros((B, cm.n_param), dtype=f64, device=dev),
                     m=mass[:, mm].reshape(B, nl).contiguous(), cost=e(B), u=e(B, nl, N), x=e(B, nl, 2, np1),
                     modes=e(B, nl, N, dt=i32), obj=e(B), status=e(B, dt=i32), nodes=e(B, dt=i32))
            bufs.append(b)
            G = g.group[gi]
            for k in ("x0", "xg", "ug", "params", "cost", "u", "x", "modes", "obj", "status", "nodes"):
                setattr(G, k, b[k].data_ptr())
            G.n_local, G.n_param, G.has_leader = nl, cm.n_param, int(rl is not None)
            for slot, i in enumerate(idx):
                g.group_of[i], g.slot_of[i] = gi, slot
        t_idx = torch.zeros(1, dtype=torch.int64, device=dev)
        active = torch.ones(S, dtype=torch.uint8, device=dev)
        u0 = torch.empty((S, n), dtype=f64, device=dev)
        gear0 = torch.empty((S, n), dtype=i32, device=dev) if GG is not None else None
        lead_t = torch.empty((S, 2), dtype=f64, device=dev)
        x_cur = x.clone(); x_next = torch.empty_like(x_cur)
        r_t = torch.empty(S, dtype=f64, device=dev); v_t = torch.empty(S, dtype=torch.uint8, device=dev)
        e_t = torch.empty(S, dtype=i32, device=dev)
        ptr = lambda t_: None if t_ is None else t_.data_ptr()
        g.t, g.x, g.leader_x, g.SG, g.UG, g.GG = t_idx.data_ptr(), x_cur.data_ptr(), lx.data_ptr(), SG.data_ptr(), \
            UG.data_ptr(), ptr(GG)
        g.active, g.WIN, g.FEAS, g.ND, g.U_log = active.data_ptr(), WIN.data_ptr(), FEAS.data_ptr(), ND.data_ptr(), U.data_ptr()
        g.u0, g.gear0 = u0.data_ptr(), ptr(gear0)

        def piece(b):
            def run_group():
                stream = torch.cuda.current_stream().cuda_stream
                b["cm"].eval_device(b["B"], b["m"], b["params"], b["xg"], b["ug"], b["cost"], stream=stream)
                b["cm"].solve_device(b["B"], b["x0"], b["m"], b["params"], None, b["u"], b["x"], None, b["modes"], b["obj"],
                                     b["status"], b["nodes"], None, stream=stream)
            return run_group
        fork = _Fork(torch, len(bufs), enabled=self.fork)
        pieces = [piece(b) for b in bufs]

        def iteration(it):
            def body():
                stream = torch.cuda.current_stream().cuda_stream
                g.it = it
                api.event_iter_device(g, phase=_lib.EVENT_PACK, ctx=self.ctx, stream=stream)
                fork.run(pieces)
                api.event_iter_device(g, phase=_lib.EVENT_SELECT, ctx=self.ctx, stream=stream)
            return _StepGraph(torch, body, enabled=self.graph)
        iterations = [iteration(it) for it in range(self.iters)]

        stream = torch.cuda.current_stream().cuda_stream
        for _ in range(ep_len):
            for step in iterations:
                step()
            api.event_iter_device(g, phase=_lib.EVENT_ADOPT, ctx=self.ctx, stream=stream)
            lead_t.copy_(lx.index_select(-1, t_idx).squeeze(-1))                             # leader_x[:, t]
            api.rollout_step_device(edesc, S, x_cur, u0, gear0, mass, lead_t, x_next, r_t, v_t, e_t, ctx=self.ctx,
                                    stream=stream)
            X.index_copy_(0, t_idx + 1, x_next.unsqueeze(0))
            R.index_copy_(0, t_idx, r_t.unsqueeze(0))
            V.index_copy_(0, t_idx, v_t.unsqueeze(0)); E.index_copy_(0, t_idx, e_t.unsqueeze(0))
            x_cur.copy_(x_next)
            t_idx.add_(1)
        torch.cuda.synchronize()
        for step in iterations:
            step.close()

    def _run_torch(self, S, ep_len, x, lx, mass, edesc, SG, UG, logs):
        torch, dev, n, N = self.torch, self.dev, self.n, self.N
        f64, i32, np1 = torch.float64, torch.int32, N + 1
        X, U, R, V, E, WIN, FEAS, ND = logs
        if lx.ndim == 2:
            lx = lx.unsqueeze(0).expand(S, -1, -1)
        stream = torch.cuda.current_stream().cuda_stream
        mem = torch.full((n, 3), -1, dtype=torch.int64, device=dev)
        for i, ms in enumerate(self.members):
            mem[i, :len(ms)] = torch.as_tensor(ms, device=dev)
        sidx = torch.arange(S, device=dev)
        zero_blk = torch.zeros((S, 1, 2 * np1), dtype=f64, device=dev)
        for t in range(ep_len):
            lwin = lx[:, :, t:t + np1].reshape(S, 1, 2 * np1)
            xv = x.view(S, n, 2)
            for it in range(self.iters):
                cost0 = torch.empty((S, n), dtype=f64, device=dev)
                cost1 = torch.empty((S, n), dtype=f64, device=dev)
                XS = torch.zeros((S, n, 3, 2, np1), dtype=f64, device=dev)
                US = torch.zeros((S, n, 3, N), dtype=f64, device=dev)
                nd = torch.zeros((S, n), dtype=i32, device=dev)
                for cm, idx, nl, nf, nb, rl in self.groups:
                    k = len(idx); B = S * k
                    mm = torch.as_tensor([self.members[i] for i in idx], device=dev)          # (k, nl)
                    x0g = xv[:, mm].reshape(B, nl, 2).contiguous()
                    mg = mass[:, mm].reshape(B, nl).contiguous()
                    xg = SG[:, mm].reshape(B, nl, 2, np1).contiguous()
                    ug = UG[:, mm].reshape(B, nl, N).contiguous()
                    f2 = torch.stack([SG[:, i - 2].reshape(S, 2 * np1) if i > 1 else zero_blk[:, 0] for i in idx], dim=1)
                    b2 = torch.stack([SG[:, i + 2].reshape(S, 2 * np1) if i < n - 2 else zero_blk[:, 0] for i in idx], dim=1)
                    lead = lwin.expand(S, k, -1) if rl is not None else zero_blk.expand(S, k, -1)
                    params = torch.cat((lead, f2, b2), dim=2).reshape(B, -1).contiguous()
                    c0 = torch.empty(B, dtype=f64, device=dev)
                    cm.eval_device(B, mg, params, xg, ug, c0, stream=stream)
                    uo = torch.empty((B, nl, N), dtype=f64, device=dev); xo = torch.empty((B, nl, 2, np1), dtype=f64, device=dev)
                    mo = torch.empty((B, nl, N), dtype=i32, device=dev); ob = torch.empty(B, dtype=f64, device=dev)
                    st = torch.empty(B, dtype=i32, device=dev); no = torch.empty(B, dtype=i32, device=dev)
                    cm.solve_device(B, x0g, mg, params, None, uo, xo, None, mo, ob, st, no, None, stream=stream)
                    ii = torch.as_tensor(idx, device=dev)
                    cost0[:, ii] = c0.view(S, k)
                    cost1[:, ii] = torch.where(st == 2, ob, torch.full_like(ob, float("inf"))).view(S, k)
                    XS[:, ii, :nl] = xo.view(S, k, nl, 2, np1)
                    US[:, ii, :nl] = uo.view(S, k, nl, N)
                    nd[:, ii] = no.view(S, k)
                dec = cost0 - cost1                                   # inf - inf = nan compares False, as in Python
                valid = dec > self.threshold
                w = torch.argmax(torch.where(valid, dec, torch.full_like(dec, -float("inf"))), dim=1)   # first maximum
                anyv = valid.any(dim=1)
                FEAS[t] &= torch.isfinite(cost1).any(dim=1)
                ND[t] = torch.maximum(ND[t], nd.max(dim=1).values)
                WIN[t, :, it] = torch.where(anyv, w.to(i32), torch.full_like(w, -1, dtype=i32))
                for l in range(3):
                    j = mem[w, l]
                    sel = anyv & (j >= 0)
                    s_ = sidx[sel]
                    SG[s_, j[sel]] = XS[s_, w[sel], l]
                    UG[s_, j[sel]] = US[s_, w[sel], l]
            U[t] = UG[:, :, 0]
            api.rollout_step_device(edesc, S, x, U[t], None, mass, lx[:, :, t].contiguous(), X[t + 1], R[t], V[t], E[t],
                                    ctx=self.ctx, stream=stream)
            x = X[t + 1]
            SG = torch.cat((SG[..., 1:], SG[..., -1:]), dim=-1)        # shifted previous solution (:591-603)
            UG = torch.cat((UG[..., 1:], UG[..., -1:]), dim=-1)


class BatchedCentSweep:
    """S independent platoons under the centralized MLD-MPC (TrackingCentralizedAgent with MpcMldCent / MpcGearCent,
    fleet_cent_mld.py:14-101), all state on the device.  One timestep, for all S scenarios: pack the leader window
    leader_x[:, t:t+N+1] into every parameter row, ONE compiled-MPC launch of S centralized problems, adopt the answers
    (inputs, gears from the mode table, logs) -- pack and adopt are the two phases of hvp_cent_step_dev
    (csrc/coord.cu) -- ONE rollout launch, and the X / R / violation / error logs at the device-side timestep index
    (no host synchronisation and no host copy until the results are read back).
    Either cost norm (quadratic_cost) and either vehicle model: "pwa_gear" (gears derived from the velocities) or
    "pwa_friction" (discrete gears chosen by the MPC; the action is [u_g ; gears])."""

    def __init__(self, n: int, N: int, masses=None, spacing_policy=ConstantSpacingPolicy(50), leader_index: int = 0,
                 quadratic_cost: bool = True, model: str = "pwa_gear", d_safe: float = Params.d_safe,
                 mip_gap: float = 0.0, time_limit_ms: float = 0.0, device: int = 0, ctx=None):
        import torch
        from ._lib import MODEL_FRICTION_GEAR, MODEL_PWA_GEAR, MPC_CENT
        if model not in ("pwa_gear", "pwa_friction"):
            raise ValueError(f"model must be 'pwa_gear' or 'pwa_friction', got {model!r}")
        if n < 1 or N < 1 or n * N > 64:
            raise ValueError(f"the centralized problem needs 1 <= n * N <= 64 (n = {n}, N = {N})")
        if not 0 <= leader_index < n:
            raise ValueError(f"leader_index {leader_index} out of range for n = {n}")
        self.torch, self.n, self.N, self.leader_index = torch, n, N, leader_index
        self.quadratic, self.friction = bool(quadratic_cost), model == "pwa_friction"
        self.dev = torch.device("cuda", device)
        self.ctx = ctx or default_context(device)
        self.d0, self.t0 = spacing_params(spacing_policy)
        self.d_safe = d_safe
        self.masses = None if masses is None else np.asarray(masses, dtype=np.float64)   # (n,) or (S,n)
        self.cm = api.CompiledMpc(MPC_CENT, N, n_local=n, model=MODEL_FRICTION_GEAR if self.friction else MODEL_PWA_GEAR,
                                  leader_index=leader_index, d0=self.d0, t0=self.t0, one_norm=not self.quadratic,
                                  mip_gap=mip_gap, time_limit_ms=time_limit_ms, ctx=self.ctx)

    def close(self):
        """Releases the compiled formulation (its device scratch)."""
        if self.cm is not None:
            self.cm.close()
            self.cm = None

    def run(self, x0, leader_x, ep_len: int, strict: bool = False):
        """x0 (S,2n) initial states, leader_x (2,>=ep_len+N+1) shared or (S,2,>=ep_len+N+1) per scenario.  Returns dict
        of numpy arrays: X (T+1,S,2n), U (T,S,n) -- (T,S,2n) = [u_g ; gears] for pwa_friction --, R (T,S), violations
        (T,S) uint8, errors (T,S) int32, obj (T,S), status (T,S) int32, nodes (T,S) int32 and aborted_at (S,) int32 (the
        first timestep whose solve was not optimal, -1: none).  A non-optimal solve applies zero inputs (gear 6), as
        solve_mpc(raises=False) does; strict=True raises RuntimeError after the run if there was one."""
        from . import _lib
        torch, dev, n, N, cm = self.torch, self.dev, self.n, self.N, self.cm
        f64, i32 = torch.float64, torch.int32
        if cm is None:
            raise RuntimeError("BatchedCentSweep is closed")
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        if x0.ndim != 2 or x0.shape[1] != 2 * n:
            raise ValueError(f"x0 must have shape (S, {2 * n}), got {x0.shape}")
        S, T = x0.shape[0], int(ep_len)
        lx_np = np.ascontiguousarray(leader_x, dtype=np.float64)
        if lx_np.ndim not in (2, 3) or lx_np.shape[-2] != 2 or (lx_np.ndim == 3 and lx_np.shape[0] != S):
            raise ValueError(f"leader_x must have shape (2, L) or ({S}, 2, L), got {lx_np.shape}")
        if lx_np.shape[-1] < T + N + 1:
            raise ValueError("leader trajectory shorter than ep_len + N + 1")
        x = torch.as_tensor(x0, device=dev)
        lx = torch.as_tensor(lx_np, device=dev)
        m = np.full((S, n), 800.0) if self.masses is None else np.broadcast_to(self.masses, (S, n))
        d_mass = torch.as_tensor(np.array(m, dtype=np.float64, order="C"), device=dev)
        edesc = api.env_desc(n, self.leader_index, self.d0, self.t0, self.d_safe, self.quadratic, False, True)
        w = 2 * n if self.friction else n
        # solve buffers and the rollout's inputs, allocated once per run
        params = torch.zeros((S, cm.n_param), dtype=f64, device=dev)
        uo = torch.empty((S, n, N), dtype=f64, device=dev); xo = torch.empty((S, n, 2, N + 1), dtype=f64, device=dev)
        mo = torch.empty((S, n, N), dtype=i32, device=dev); ob = torch.empty(S, dtype=f64, device=dev)
        st = torch.empty(S, dtype=i32, device=dev); no = torch.empty(S, dtype=i32, device=dev)
        u0 = torch.empty((S, n), dtype=f64, device=dev)
        gear0 = torch.empty((S, n), dtype=i32, device=dev) if self.friction else None
        lead_t = torch.empty((S, 2), dtype=f64, device=dev)
        x_cur = x.clone(); x_next = torch.empty_like(x_cur)
        r_t = torch.empty(S, dtype=f64, device=dev); v_t = torch.empty(S, dtype=torch.uint8, device=dev)
        e_t = torch.empty(S, dtype=i32, device=dev)
        t_idx = torch.zeros(1, dtype=torch.int64, device=dev)
        # episode logs
        X = torch.empty((T + 1, S, 2 * n), dtype=f64, device=dev)
        U = torch.empty((T, S, w), dtype=f64, device=dev)
        R = torch.empty((T, S), dtype=f64, device=dev)
        V = torch.empty((T, S), dtype=torch.uint8, device=dev)
        E = torch.empty((T, S), dtype=i32, device=dev)
        OBJ = torch.empty((T, S), dtype=f64, device=dev)
        ST = torch.empty((T, S), dtype=i32, device=dev)
        ND = torch.empty((T, S), dtype=i32, device=dev)
        AB = torch.full((S,), -1, dtype=i32, device=dev)
        X[0] = x

        g = _lib.CentStep()
        g.n, g.N, g.S, g.n_param = n, N, S, cm.n_param
        g.leader_per_scenario, g.leader_len, g.T = int(lx.ndim == 3), lx.shape[-1], T
        g.n_modes = cm.n_modes
        for k, gear in enumerate(cm.mode_gear.tolist()):
            g.mode_gear[k] = gear
        ptr = lambda t_: None if t_ is None else t_.data_ptr()
        g.t, g.leader_x, g.params = t_idx.data_ptr(), lx.data_ptr(), params.data_ptr()
        g.u, g.modes, g.obj, g.status, g.nodes = uo.data_ptr(), mo.data_ptr(), ob.data_ptr(), st.data_ptr(), no.data_ptr()
        g.u0, g.gear0 = u0.data_ptr(), ptr(gear0)
        g.U_log, g.obj_log, g.status_log, g.nodes_log, g.aborted_at = (t_.data_ptr() for t_ in (U, OBJ, ST, ND, AB))

        def body():
            stream = torch.cuda.current_stream().cuda_stream
            api.cent_step_device(g, phase=_lib.CENT_PACK, ctx=self.ctx, stream=stream)        # leader_x[:, t:t+N+1]
            # x_cur (S, 2n) = [p0 v0 p1 v1 ...] is already the solve's x0 layout [S][n][2]
            cm.solve_device(S, x_cur, d_mass, params, None, uo, xo, None, mo, ob, st, no, None, stream=stream)
            api.cent_step_device(g, phase=_lib.CENT_ADOPT, ctx=self.ctx, stream=stream)
            lead_t.copy_(lx.index_select(-1, t_idx).squeeze(-1))                             # leader_x[:, t]
            api.rollout_step_device(edesc, S, x_cur, u0, gear0, d_mass, lead_t, x_next, r_t, v_t, e_t, ctx=self.ctx,
                                    stream=stream)
            X.index_copy_(0, t_idx + 1, x_next.unsqueeze(0))
            R.index_copy_(0, t_idx, r_t.unsqueeze(0))
            V.index_copy_(0, t_idx, v_t.unsqueeze(0)); E.index_copy_(0, t_idx, e_t.unsqueeze(0))
            x_cur.copy_(x_next)
            t_idx.add_(1)

        # Eager launches: replaying a timestep as a CUDA graph was measured no faster at any batch size (0.99-1.02x at
        # S = 10 .. 4096, DESIGN.md 5b) -- the loop is bound by the solve, not by launches
        for _ in range(T):
            body()
        torch.cuda.synchronize()
        out = dict(X=X.cpu().numpy(), U=U.cpu().numpy(), R=R.cpu().numpy(), violations=V.cpu().numpy(),
                   errors=E.cpu().numpy(), obj=OBJ.cpu().numpy(), status=ST.cpu().numpy(), nodes=ND.cpu().numpy(),
                   aborted_at=AB.cpu().numpy())
        if strict and (out["status"] != _lib.OPTIMAL).any():
            # raised after the run: nothing can be raised from inside a captured timestep
            ts_, ss_ = np.nonzero(out["status"] != _lib.OPTIMAL)
            bad = [f"scenario {s} at timestep {t} (status {out['status'][t, s]})" for t, s in zip(ts_[:8], ss_[:8])]
            raise RuntimeError(f"Infeasible problem encountered: {', '.join(bad)}{' ...' if len(ts_) > 8 else ''}")
        return out
