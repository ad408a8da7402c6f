"""ctypes front-end of the CPU oracle (oracle/hvp_oracle.c).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libhvp_oracle.so")

FRONT, LEADER, TRAILER = 1, 2, 4

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lp = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_bp = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("hvp_oracle.c", "hvp_oracle_mpc.c")]
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < max(map(os.path.getmtime, srcs)):
        subprocess.check_call(["make", "-s", "-C", _HERE, "libhvp_oracle.so"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        L.hvo_pwa_gear_system.argtypes = [C.c_double, C.c_double, _dp, _dp, _dp, _dp, _dp]
        L.hvo_gear_from_velocity.argtypes = [C.c_double]
        L.hvo_gear_from_velocity.restype = C.c_int
        L.hvo_traction.argtypes = [C.c_double, C.c_int, C.POINTER(C.c_int)]
        L.hvo_traction.restype = C.c_double
        L.hvo_env_step_batch.argtypes = [C.c_int, C.c_int, _dp, _dp, C.c_void_p, C.c_void_p, C.c_int,
                                         _dp, C.c_double, C.c_double, C.c_int, C.c_double, C.c_int,
                                         _dp, _dp, _bp, _ip]
        L.hvo_env_step_batch.restype = None
        L.hvo_qp_solve.argtypes = [C.c_int, C.c_int, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, _dp,
                                   C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.hvo_qp_solve.restype = C.c_int
        L.hvo_local_miqp_batch.argtypes = [C.c_int, C.c_int, _ip, C.c_double, C.c_double, C.c_double,
                                           _dp, _dp, _dp, _dp, _dp, C.c_int, _dp, _dp, _ip, _dp, _dp,
                                           _ip, _lp]
        L.hvo_local_miqp_batch.restype = None
        L.hvo_local_build_qp_py.argtypes = [C.c_int, C.c_int, C.c_double, C.c_double, C.c_double,
                                            C.c_double, _dp, _dp, _dp, _dp, _ip, _dp, _dp,
                                            C.POINTER(C.c_double), _dp, _dp, _dp]
        L.hvo_local_build_qp_py.restype = C.c_int
        L.hvo_max_threads.restype = C.c_int
        hdr = [C.c_int] * 8 + [C.c_double] * 4
        L.hvo_mpc_solve_batch.argtypes = [C.c_int] + hdr + [C.c_int, C.c_int, _dp, _dp, _dp, C.c_void_p, C.c_int,
                                                          _dp, _dp, _dp, _ip, _dp, _dp, _ip, _lp, _lp]
        L.hvo_mpc_solve_batch.restype = None
        L.hvo_mpc_build_qp_py.argtypes = hdr + [_dp, _dp, _dp, _ip, _dp, _dp, C.POINTER(C.c_double), _dp, _dp, _dp]
        L.hvo_mpc_build_qp_py.restype = C.c_int
        L.hvo_mode_table.argtypes = [C.c_int, C.c_double, _dp, _dp, _dp, _dp, _dp, _ip]
        L.hvo_mode_table.restype = C.c_int
        _lib = L
    return _lib


# ---------------------------------------------------------------------------------------------
def pwa_gear_system(mass: float, ts: float = 1.0):
    a, b, c, lo, hi = (np.zeros(7) for _ in range(5))
    lib().hvo_pwa_gear_system(float(mass), float(ts), a, b, c, lo, hi)
    return a, b, c, lo, hi


def gear_from_velocity(v: float) -> int:
    return lib().hvo_gear_from_velocity(float(v))


def traction(v: float, j: int):
    err = C.c_int(0)
    t = lib().hvo_traction(float(v), int(j), C.byref(err))
    return t, err.value


def env_step(x, u, gear=None, mass=None, leader=None, d0=50.0, t0=0.0, leader_index=0,
             d_safe=25.0, quadratic=True, real_ref=False):
    """Batched restatement of PlatoonEnv.step (env.py:182-212).
    x (B,2n), u (B,n), gear (B,n) int32 or None, mass (n,) / (B,n) / None, leader (B,2)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    B, n2 = x.shape
    n = n2 // 2
    leader = np.ascontiguousarray(leader, dtype=np.float64).reshape(B, 2)
    gp = None
    if gear is not None:
        gear = np.ascontiguousarray(gear, dtype=np.int32)
        gp = gear.ctypes.data_as(C.c_void_p)
    mp, per = None, 0
    if mass is not None:
        mass = np.ascontiguousarray(mass, dtype=np.float64)
        per = int(mass.ndim == 2)
        mp = mass.ctypes.data_as(C.c_void_p)
    x_out = np.empty_like(x)
    cost = np.empty(B)
    viol = np.empty(B, dtype=np.uint8)
    err = np.empty(B, dtype=np.int32)
    flags = int(bool(quadratic)) | (int(bool(real_ref)) << 1)
    lib().hvo_env_step_batch(B, n, x, u, gp, mp, per, leader, float(d0), float(t0), int(leader_index),
                             float(d_safe), flags, x_out, cost, viol, err)
    return x_out, cost, viol, err


def qp_solve(H, g, c0, A, b, wmax):
    H = np.ascontiguousarray(H, dtype=np.float64)
    g = np.ascontiguousarray(g, dtype=np.float64)
    A = np.ascontiguousarray(A, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    wmax = np.ascontiguousarray(wmax, dtype=np.float64)
    n, m = g.shape[0], b.shape[0]
    x = np.zeros(n)
    lam = np.zeros(max(m, 1))
    obj = C.c_double(0)
    it = C.c_int(0)
    st = lib().hvo_qp_solve(n, m, H, g, float(c0), A.reshape(-1) if m else np.zeros(1), b if m else np.zeros(1),
                            wmax if m else np.zeros(1), x, lam, C.byref(obj), C.byref(it))
    return st, x, lam[:m], obj.value, it.value


def local_miqp(N, flags, mass, x0, xf, xb, xl, d0=50.0, t0=0.0, tight=0.0, exhaustive=False):
    """Batched exact solve of per-vehicle local MIQPs (LocalMpcMld, fleet_decent_mld.py:21-223).
    x0 (B,2); xf/xb/xl (B,2,N+1); flags (B,) bitmask FRONT|LEADER|TRAILER; mass (B,)."""
    x0 = np.ascontiguousarray(x0, dtype=np.float64)
    B = x0.shape[0]
    flags = np.ascontiguousarray(np.broadcast_to(flags, (B,)), dtype=np.int32)
    mass = np.ascontiguousarray(np.broadcast_to(mass, (B,)), dtype=np.float64)

    def ref(a):
        if a is None:
            return np.zeros((B, 2, N + 1))
        return np.ascontiguousarray(a, dtype=np.float64).reshape(B, 2, N + 1)

    xf, xb, xl = ref(xf), ref(xb), ref(xl)
    u = np.zeros((B, N))
    xt = np.zeros((B, 2, N + 1))
    modes = np.zeros((B, N), dtype=np.int32)
    obj = np.zeros(B)
    second = np.zeros(B)
    status = np.zeros(B, dtype=np.int32)
    leaves = np.zeros(B, dtype=np.int64)
    lib().hvo_local_miqp_batch(B, int(N), flags, float(d0), float(t0), float(tight), mass, x0, xf, xb,
                               xl, int(exhaustive), u, xt, modes, obj, second, status, leaves)
    return dict(u=u, x=xt, modes=modes, obj=obj, second=second, status=status, leaves=leaves)


def local_build_qp(N, flags, mass, x0, xf, xb, xl, modes, d0=50.0, t0=0.0, tight=0.0):
    """Dense fixed-mode QP (H,g,c0,A,b,wmax) of one local problem, for certification."""
    maxrows = 12 * 16 + 8
    H = np.zeros((N, N)); g = np.zeros(N)
    A = np.zeros(maxrows * N); b = np.zeros(maxrows); w = np.zeros(maxrows)
    c0 = C.c_double(0)
    z = np.zeros((2, N + 1))
    m = lib().hvo_local_build_qp_py(
        int(N), int(flags), float(d0), float(t0), float(tight), float(mass),
        np.ascontiguousarray(x0, dtype=np.float64),
        np.ascontiguousarray(z if xf is None else xf, dtype=np.float64),
        np.ascontiguousarray(z if xb is None else xb, dtype=np.float64),
        np.ascontiguousarray(z if xl is None else xl, dtype=np.float64),
        np.ascontiguousarray(modes, dtype=np.int32), H, g, C.byref(c0), A, b, w)
    return H, g, c0.value, A[: m * N].reshape(m, N), b[:m], w[:m]


CENT, LOCAL, EVENT, ADMM, GADMM = 1, 2, 3, 4, 5
PWA_GEAR, FRICTION_GEAR = 0, 1
REAL_REF, NO_LEADER = 8, -100


def mpc_dims(kind, nl, N, flags=0, n_front=0, n_behind=0):
    """(n_param, n_extra) of a formulation (layout: include/hvp.h)."""
    blk = 2 * (N + 1)
    if kind == CENT:
        return blk, 0
    if kind in (LOCAL, EVENT):
        return 3 * blk, 0
    if kind == ADMM:
        return 5 * blk, (0 if flags & FRONT else blk) + (0 if flags & TRAILER else blk)
    if kind == GADMM:
        na = n_front + n_behind + 1
        return (1 + 2 * na) * blk, (n_front + n_behind) * blk
    raise ValueError(kind)


def mode_table(model, mass=800.0):
    a, b, c, lo, hi = (np.zeros(12) for _ in range(5))
    gear = np.zeros(12, np.int32)
    R = lib().hvo_mode_table(int(model), float(mass), a, b, c, lo, hi, gear)
    return a[:R], b[:R], c[:R], lo[:R], hi[:R], gear[:R]


def mpc_solve(kind, nl, N, x0, mass, params, *, model=PWA_GEAR, flags=0, leader_index=0, n_front=0,
              n_behind=0, d0=50.0, t0=0.0, tight=0.0, rho=0.5, fixed_modes=None, method=1):
    """Batched exact solve of the compiled MPC formulations (hvp_oracle_mpc.c).
    x0 (B,nl,2), mass (B,nl), params (B,npar); method 0 = exhaustive enumeration, 1 = branch and bound."""
    x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(-1, nl, 2)
    B = x0.shape[0]
    npar, ne = mpc_dims(kind, nl, N, flags, n_front, n_behind)
    mass = np.ascontiguousarray(np.broadcast_to(np.asarray(mass, dtype=np.float64), (B, nl)))
    params = np.ascontiguousarray(params, dtype=np.float64).reshape(B, npar)
    fm = None
    if fixed_modes is not None:
        fixed_modes = np.ascontiguousarray(fixed_modes, dtype=np.int32).reshape(B, nl, N)
        fm = fixed_modes.ctypes.data_as(C.c_void_p)
    u = np.zeros((B, nl, N)); xt = np.zeros((B, nl, 2, N + 1)); extra = np.zeros((B, max(ne, 1)))
    modes = np.zeros((B, nl, N), np.int32); obj = np.zeros(B); second = np.zeros(B)
    status = np.zeros(B, np.int32); leaves = np.zeros(B, np.int64); nodes = np.zeros(B, np.int64)
    lib().hvo_mpc_solve_batch(B, int(kind), int(model), int(nl), int(N), int(flags), int(leader_index),
                              int(n_front), int(n_behind), float(d0), float(t0), float(tight), float(rho),
                              int(npar), int(max(ne, 1)), x0, mass, params, fm, int(method), u, xt, extra, modes,
                              obj, second, status, leaves, nodes)
    return dict(u=u, x=xt, extra=extra[:, :ne], modes=modes, obj=obj, second=second, status=status,
                leaves=leaves, nodes=nodes)


def mpc_build_qp(kind, nl, N, x0, mass, params, modes, *, model=PWA_GEAR, flags=0, leader_index=0, n_front=0,
                 n_behind=0, d0=50.0, t0=0.0, tight=0.0, rho=0.5):
    """Dense fixed-mode QP (H,g,c0,A,b,wmax) of one problem in input space, for certification."""
    npar, ne = mpc_dims(kind, nl, N, flags, n_front, n_behind)
    n = nl * N + ne
    maxrows = 2400
    H = np.zeros((n, n)); g = np.zeros(n); A = np.zeros(maxrows * n); b = np.zeros(maxrows); w = np.zeros(maxrows)
    c0 = C.c_double(0)
    m = lib().hvo_mpc_build_qp_py(int(kind), int(model), int(nl), int(N), int(flags), int(leader_index),
                                  int(n_front), int(n_behind), float(d0), float(t0), float(tight), float(rho),
                                  np.ascontiguousarray(x0, dtype=np.float64).reshape(-1),
                                  np.ascontiguousarray(np.broadcast_to(np.asarray(mass, dtype=np.float64), (nl,))),
                                  np.ascontiguousarray(params, dtype=np.float64).reshape(-1),
                                  np.ascontiguousarray(modes, dtype=np.int32).reshape(-1), H, g, C.byref(c0), A, b, w)
    if m < 0:
        return None
    return H, g, c0.value, A[: m * n].reshape(m, n), b[:m], w[:m]


def max_threads() -> int:
    return lib().hvo_max_threads()


def use_all_cores() -> int:
    """Let the batch calls use every host core this process may run on (torchrun exports OMP_NUM_THREADS=1)."""
    import os
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    lib().hvo_set_threads(int(n))
    return max_threads()


# ---------------------------------------------------------------------------------------------
# CPU baseline port (oracle/hvp_cpu_bnb.cpp): the product's branch-and-bound compiled for the host cores.
# Used ONLY by bench.py's cpu_baseline / --impl reference legs and by the test that checks it against the
# enumeration oracle above.
_BNB = {}


def build_cpu_bnb(native: bool = False, force: bool = False) -> str:
    """Generic build: oracle/libhvp_cpu_bnb.so (-O3).  Native build (-O3 -march=native): compiled by the process that
    loads it into a temporary directory removed at exit, so it never travels between hosts and the tree may be
    read-only."""
    src = os.path.join(_HERE, "hvp_cpu_bnb.cpp")
    hdr = os.path.join(_HERE, "..", "hybrid_vehicle_platoon_b200", "csrc", "flat_core.cuh")
    if native:
        import atexit
        import shutil
        import tempfile
        tmp = tempfile.mkdtemp(prefix="hvp_cpu_bnb_")
        atexit.register(shutil.rmtree, tmp, ignore_errors=True)
        out = os.path.join(tmp, "libhvp_cpu_bnb_native.so")
    else:
        out = os.path.join(_HERE, "libhvp_cpu_bnb.so")
    newest = max(os.path.getmtime(src), os.path.getmtime(hdr))
    if force or not os.path.exists(out) or os.path.getmtime(out) < newest:
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        cmd = [cxx, "-O3", "-fopenmp", "-fPIC", "-shared", "-std=c++17"] + (["-march=native"] if native else []) + ["-o", out, src]
        subprocess.check_call(cmd)
    return out


def _bnb_lib(native: bool):
    if native not in _BNB:
        L = C.CDLL(build_cpu_bnb(native))
        L.hvc_local_miqp_bnb.argtypes = [C.c_int, C.c_int, _ip, C.c_double, C.c_double, C.c_double, _dp, _dp, _dp, _dp,
                                         _dp, _dp, _dp, _ip, _dp, _ip, _ip, _ip]
        L.hvc_local_miqp_bnb.restype = C.c_int
        L.hvc_max_threads.restype = C.c_int
        _BNB[native] = L
    return _BNB[native]


def local_miqp_bnb(N, flags, mass, x0, xf, xb, xl, d0=50.0, t0=0.0, tight=0.0, native=False, threads=None):
    """The CPU branch-and-bound port on a batch of local MIQPs (same contract as local_miqp; `nodes` instead of
    `leaves`).  threads=None: every core this process may run on."""
    L = _bnb_lib(native)
    x0 = np.ascontiguousarray(x0, dtype=np.float64)
    B = x0.shape[0]
    c = lambda a, t=np.float64: np.ascontiguousarray(a, dtype=t)
    flags = c(np.broadcast_to(flags, (B,)), np.int32)
    mass = c(np.broadcast_to(mass, (B,)))
    ref = lambda a: np.zeros((B, 2, N + 1)) if a is None else c(a).reshape(B, 2, N + 1)
    if threads is None:
        threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    L.hvc_set_threads(int(threads))
    u = np.zeros((B, N)); x = np.zeros((B, 2, N + 1)); modes = np.zeros((B, N), np.int32)
    obj = np.zeros(B); st = np.zeros(B, np.int32); nodes = np.zeros(B, np.int32); it = np.zeros(B, np.int32)
    rc = L.hvc_local_miqp_bnb(B, int(N), flags, float(d0), float(t0), float(tight), mass, x0, ref(xf), ref(xb), ref(xl),
                              u, x, modes, obj, st, nodes, it)
    if rc != 0:
        raise ValueError(f"hvc_local_miqp_bnb: unsupported horizon N={N}")
    return dict(u=u, x=x, modes=modes, obj=obj, status=st, nodes=nodes, qp_iters=it, threads=L.hvc_max_threads())
