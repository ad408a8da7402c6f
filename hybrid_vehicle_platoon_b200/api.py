"""Batched array-level entry points over the C ABI (numpy = host buffers, torch = device buffers)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import EnvDesc, LocalDesc, MpcDesc, check, default_context, lib


def _hp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _stream_arg(stream):
    """None -> the context's own stream; 0 (torch's default stream handle) -> cudaStreamLegacy;
    anything else is a cudaStream_t."""
    if stream is None:
        return None
    return C.c_void_p(1 if int(stream) == 0 else int(stream))


def _c(a, dt):
    return None if a is None else np.ascontiguousarray(a, dtype=dt)


def env_desc(n, leader_index=0, d0=50.0, t0=0.0, d_safe=25.0, quadratic=True, real_ref=False,
             mass_per_scenario=False) -> EnvDesc:
    flags = (_lib.ENV_QUADRATIC if quadratic else 0) | (_lib.ENV_REAL_VEHICLE_REF if real_ref else 0) \
        | (_lib.ENV_MASS_PER_SCENARIO if mass_per_scenario else 0)
    return EnvDesc(int(n), int(leader_index), int(flags), 0, float(d0), float(t0), float(d_safe))


def rollout_step(x, u, gear=None, mass=None, leader=None, *, d0=50.0, t0=0.0, leader_index=0,
                 d_safe=25.0, quadratic=True, real_ref=False, ctx=None):
    """Batched PlatoonEnv.step (env.py:182-212) on host (numpy) buffers.
    x (B,2n), u (B,n), gear (B,n) int32|None, mass (n,)|(B,n)|None, leader (B,2).
    Returns x_new (B,2n), cost (B,), viol (B,) uint8, err (B,) int32."""
    ctx = ctx or default_context()
    x = _c(x, np.float64); u = _c(u, np.float64)
    B, n2 = x.shape
    n = n2 // 2
    gear = _c(gear, np.int32); mass = _c(mass, np.float64)
    leader = _c(leader, np.float64).reshape(B, 2)
    per = mass is not None and mass.ndim == 2
    d = env_desc(n, leader_index, d0, t0, d_safe, quadratic, real_ref, per)
    x_out = np.empty_like(x); cost = np.empty(B); viol = np.empty(B, np.uint8); err = np.empty(B, np.int32)
    check(lib().hvp_rollout_step_host(ctx.handle, C.byref(d), B, _hp(x), _hp(u), _hp(gear), _hp(mass),
                                      _hp(leader), _hp(x_out), _hp(cost), _hp(viol), _hp(err)))
    return x_out, cost, viol, err


def rollout_step_device(desc: EnvDesc, batch, x, u, gear, mass, leader, x_out, cost, viol, err, *,
                        ctx=None, stream=None):
    """Same on DEVICE buffers (torch CUDA tensors); asynchronous on `stream` (int cudaStream_t)."""
    ctx = ctx or default_context()
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    check(lib().hvp_rollout_step_dev(ctx.handle, C.byref(desc), int(batch), p(x), p(u), p(gear), p(mass),
                                     p(leader), p(x_out), p(cost), p(viol), p(err),
                                     _stream_arg(stream)))


def local_desc(N, d0=50.0, t0=0.0, tight=0.0, max_nodes=0, mip_gap=0.0, time_limit_ms=0.0) -> LocalDesc:
    """mip_gap: relative gap at which nodes are pruned (Gurobi MIPGap; 0 = proven optimal); time_limit_ms: per-problem
    device-clock budget, status 9 with the incumbent when it runs out (0 = none)."""
    return LocalDesc(int(N), int(max_nodes), float(d0), float(t0), float(tight), float(mip_gap), float(time_limit_ms), None)


def local_miqp(N, flags, mass, x0, xf=None, xb=None, xl=None, *, d0=50.0, t0=0.0, tight=0.0,
               max_nodes=0, mip_gap=0.0, time_limit_ms=0.0, ctx=None):
    """Batched LocalMpcMld solves (fleet_decent_mld.py:21-223) on host (numpy) buffers.
    x0 (B,2); xf/xb/xl (B,2,N+1) or None; flags (B,) of FRONT|LEADER|TRAILER; mass (B,)."""
    ctx = ctx or default_context()
    x0 = _c(x0, np.float64)
    B = x0.shape[0]
    flags = _c(np.broadcast_to(flags, (B,)), np.int32)
    mass = _c(np.broadcast_to(mass, (B,)), np.float64)
    xf = _c(xf, np.float64); xb = _c(xb, np.float64); xl = _c(xl, np.float64)
    for a in (xf, xb, xl):
        if a is not None and a.size != B * 2 * (N + 1):
            raise ValueError(f"reference arrays must have shape ({B}, 2, {N + 1})")
    d = local_desc(N, d0, t0, tight, max_nodes, mip_gap, time_limit_ms)
    u = np.empty((B, N)); x = np.empty((B, 2, N + 1)); modes = np.empty((B, N), np.int32)
    obj = np.empty(B); status = np.empty(B, np.int32); nodes = np.empty(B, np.int32)
    iters = np.empty(B, np.int32)
    check(lib().hvp_local_miqp_host(ctx.handle, C.byref(d), B, _hp(flags), _hp(mass), _hp(x0), _hp(xf),
                                    _hp(xb), _hp(xl), _hp(u), _hp(x), _hp(modes), _hp(obj), _hp(status),
                                    _hp(nodes), _hp(iters)))
    return dict(u=u, x=x, modes=modes, obj=obj, status=status, nodes=nodes, qp_iters=iters,
                run_time=max(ctx.last_kernel_ms(), 0.0) * 1e-3)


def local_miqp_device(desc: LocalDesc, batch, flags, mass, x0, xf, xb, xl, u, x, modes, obj, status,
                      nodes, qp_iters=None, *, ctx=None, stream=None, modes_hint=None):
    """Same on DEVICE buffers (torch CUDA tensors); asynchronous on `stream`.  modes_hint: optional (batch, N) int32
    CUDA tensor of region sequences to try first (include/hvp.h)."""
    ctx = ctx or default_context()
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    if modes_hint is not None:
        desc = LocalDesc(desc.N, desc.max_nodes, desc.d0, desc.t0, desc.tight, desc.mip_gap, desc.time_limit_ms,
                         modes_hint.data_ptr())
    check(lib().hvp_local_miqp_dev(ctx.handle, C.byref(desc), int(batch), p(flags), p(mass), p(x0), p(xf),
                                   p(xb), p(xl), p(u), p(x), p(modes), p(obj), p(status), p(nodes),
                                   p(qp_iters), _stream_arg(stream)))


class CompiledMpc:
    """One compiled MPC formulation on the device (hvp_mpc; include/hvp.h).  Built once -- like the
    reference builds one Gurobi model per controller -- and solved for batches of (x0, mass, params)."""

    def __init__(self, kind, N, *, n_local=1, model=_lib.MODEL_PWA_GEAR, flags=0, leader_index=0, n_front=0,
                 n_behind=0, d0=50.0, t0=0.0, tight=0.0, rho=0.5, max_nodes=0, one_norm=False, mip_gap=0.0,
                 time_limit_ms=0.0, ctx=None):
        self.ctx = ctx or default_context()
        self.desc = MpcDesc(int(kind), int(model), int(n_local), int(N), int(flags), int(leader_index),
                            int(n_front), int(n_behind), int(max_nodes), int(bool(one_norm)), float(d0), float(t0),
                            float(tight), float(rho), float(mip_gap), float(time_limit_ms))
        h = C.c_void_p()
        check(lib().hvp_mpc_create(self.ctx.handle, C.byref(self.desc), C.byref(h)))
        self._h = h
        if hasattr(self.ctx, "_register"):
            self.ctx._register(self)
        info = (C.c_int32 * 8)()
        check(lib().hvp_mpc_info(h, info))
        (self.n_var, self.n_extra, self.n_param, self.n_modes, self.n_local, self.N, self.n_rows,
         self.smem_bytes) = list(info)
        self.mode_lo = np.zeros(self.n_modes); self.mode_hi = np.zeros(self.n_modes)
        self.mode_gear = np.zeros(self.n_modes, np.int32)
        check(lib().hvp_mpc_mode_table(h, _hp(self.mode_lo), _hp(self.mode_hi), _hp(self.mode_gear)))

    def solve(self, x0, mass, params, fixed_modes=None):
        """Host (numpy) buffers: x0 (B,nl,2), mass (B,nl), params (B,n_param), fixed_modes (B,nl,N)|None."""
        nl, N = self.n_local, self.N
        x0 = _c(x0, np.float64).reshape(-1, nl, 2)
        B = x0.shape[0]
        mass = _c(np.broadcast_to(np.asarray(mass, dtype=np.float64), (B, nl)), np.float64)
        params = _c(params, np.float64).reshape(B, self.n_param)
        fm = None if fixed_modes is None else _c(fixed_modes, np.int32).reshape(B, nl, N)
        u = np.empty((B, nl, N)); x = np.empty((B, nl, 2, N + 1)); extra = np.empty((B, max(self.n_extra, 1)))
        modes = np.empty((B, nl, N), np.int32); obj = np.empty(B); status = np.empty(B, np.int32)
        nodes = np.empty(B, np.int32); iters = np.empty(B, np.int32)
        check(lib().hvp_mpc_solve_host(self._h, B, _hp(x0), _hp(mass), _hp(params), _hp(fm), _hp(u), _hp(x),
                                       _hp(extra), _hp(modes), _hp(obj), _hp(status), _hp(nodes), _hp(iters)))
        return dict(u=u, x=x, extra=extra[:, :self.n_extra], modes=modes, obj=obj, status=status, nodes=nodes,
                    qp_iters=iters, run_time=max(self.ctx.last_kernel_ms(), 0.0) * 1e-3)

    def solve_device(self, batch, x0, mass, params, fixed_modes, u, x, extra, modes, obj, status, nodes,
                     qp_iters=None, *, stream=None):
        """DEVICE buffers (torch CUDA tensors); asynchronous on `stream`."""
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib().hvp_mpc_solve_dev(self._h, int(batch), p(x0), p(mass), p(params), p(fixed_modes), p(u), p(x),
                                      p(extra), p(modes), p(obj), p(status), p(nodes), p(qp_iters),
                                      _stream_arg(stream)))

    def solve_shard_device(self, batch, x0, mass, params, rank, world, groups, prefix_depth, node_budget, incumbent,
                           u, x, extra, modes, obj, status, nodes, qp_iters=None, *, stream=None):
        """One device's share of split trees (hvp_mpc_solve_shard_dev, include/hvp.h); DEVICE buffers."""
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib().hvp_mpc_solve_shard_dev(self._h, int(batch), p(x0), p(mass), p(params), int(rank), int(world),
                                            int(groups), int(prefix_depth), int(node_budget), p(incumbent), p(u), p(x),
                                            p(extra), p(modes), p(obj), p(status), p(nodes), p(qp_iters),
                                            _stream_arg(stream)))

    def eval_device(self, batch, mass, params, xg, ug, cost, *, stream=None):
        """eval_cost on DEVICE buffers (hvp_mpc_eval_dev); asynchronous on `stream`."""
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib().hvp_mpc_eval_dev(self._h, int(batch), p(mass), p(params), p(xg), p(ug), p(cost), _stream_arg(stream)))

    def eval_cost(self, mass, params, xg, ug):
        """Cost of pinned guesses (fleet_event_based.py:308-327): xg (B,nl,2,N+1), ug (B,nl,N) -> (B,)."""
        nl, N = self.n_local, self.N
        xg = _c(xg, np.float64).reshape(-1, nl, 2, N + 1)
        B = xg.shape[0]
        ug = _c(ug, np.float64).reshape(B, nl, N)
        mass = _c(np.broadcast_to(np.asarray(mass, dtype=np.float64), (B, nl)), np.float64)
        params = _c(params, np.float64).reshape(B, self.n_param)
        cost = np.empty(B)
        check(lib().hvp_mpc_eval_host(self._h, B, _hp(mass), _hp(params), _hp(xg), _hp(ug), _hp(cost)))
        return cost

    def gears(self, modes):
        """Gear (1..6) of each mode index (MpcGear.solve_mpc: argmax sigma + 1, mpc_gear.py:120-125)."""
        return self.mode_gear[np.clip(modes, 0, self.n_modes - 1)]

    def close(self):
        if getattr(self, "_h", None):
            lib().hvp_mpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def microbench_fp64(iters: int = 20000, ctx=None) -> float:
    """Measured FP64 FMA peak of the device in TFLOP/s (roofline denominator of the QP kernel)."""
    ctx = ctx or default_context()
    t = C.c_double(0)
    check(lib().hvp_microbench_fp64(ctx.handle, int(iters), C.byref(t)))
    return t.value


def microbench_smem(iters: int = 20000, ctx=None) -> float:
    """Measured shared-memory read bandwidth of the device in GB/s (smem roofline of the QP kernels)."""
    ctx = ctx or default_context()
    t = C.c_double(0)
    check(lib().hvp_microbench_smem(ctx.handle, int(iters), C.byref(t)))
    return t.value


def gadmm_round_device(g, *, init: bool, ctx=None, stream=None):
    """Fused coordinator glue of one g-ADMM consensus round (hvp_gadmm_round_dev, include/hvp.h); `g` is a
    _lib.GAdmmRound whose pointers refer to torch CUDA tensors the caller keeps alive."""
    ctx = ctx or default_context()
    g.init = 1 if init else 0
    check(lib().hvp_gadmm_round_dev(ctx.handle, C.byref(g), _stream_arg(stream)))


def decent_observe_device(g, *, ctx=None, stream=None):
    """Fused observe step of the decentralized controller (hvp_decent_observe_dev); `g` is a _lib.DecentObserve."""
    ctx = ctx or default_context()
    check(lib().hvp_decent_observe_dev(ctx.handle, C.byref(g), _stream_arg(stream)))


def admm_round_device(g, *, pack_only: bool = False, ctx=None, stream=None):
    """Fused z / y update of a naive-ADMM round (hvp_admm_round_dev); `g` is a _lib.AdmmRound."""
    ctx = ctx or default_context()
    g.pack_only = 1 if pack_only else 0
    check(lib().hvp_admm_round_dev(ctx.handle, C.byref(g), _stream_arg(stream)))


def cent_step_device(g, *, phase: int, ctx=None, stream=None):
    """Fused glue of a centralized timestep (hvp_cent_step_dev): phase _lib.CENT_PACK writes the leader window into the
    parameter rows, _lib.CENT_ADOPT adopts the solve's answer and logs it; `g` is a _lib.CentStep."""
    ctx = ctx or default_context()
    g.phase = int(phase)
    check(lib().hvp_cent_step_dev(ctx.handle, C.byref(g), _stream_arg(stream)))


def event_iter_device(g, *, phase: int, ctx=None, stream=None):
    """Fused glue of an event-based iteration (hvp_event_iter_dev): phase _lib.EVENT_PACK fills the groups' eval / solve
    inputs from the guesses, _lib.EVENT_SELECT picks each scenario's winner and adopts its plan, _lib.EVENT_ADOPT takes
    the first inputs, logs them and shifts the guesses; `g` is a _lib.EventIter."""
    ctx = ctx or default_context()
    g.phase = int(phase)
    check(lib().hvp_event_iter_dev(ctx.handle, C.byref(g), _stream_arg(stream)))


def admm_step_device(g, *, phase: int, ctx=None, stream=None):
    """Fused glue of a naive-ADMM timestep (hvp_admm_step_dev): phase _lib.ADMM_PACK fills the role solves' inputs at the
    start of a timestep, _lib.ADMM_ROUND does a round's z / y update, next parameters and logs, _lib.ADMM_ADOPT takes the
    last round's first inputs and gears and logs them; `g` is a _lib.AdmmStep."""
    ctx = ctx or default_context()
    g.phase = int(phase)
    check(lib().hvp_admm_step_dev(ctx.handle, C.byref(g), _stream_arg(stream)))
