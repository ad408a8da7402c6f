"""ctypes binding of libhvp.so (include/hvp.h).  The CUDA library is the ONLY execution path of
this package: a missing library or a missing GPU raises, nothing falls back to the CPU."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libhvp.so")

OPTIMAL, INFEASIBLE, NODE_LIMIT, TIME_LIMIT, NUMERIC = 2, 3, 8, 9, 12
FRONT, LEADER, TRAILER = 1, 2, 4
ENV_QUADRATIC, ENV_REAL_VEHICLE_REF, ENV_MASS_PER_SCENARIO = 1, 2, 4


class EnvDesc(C.Structure):
    _fields_ = [("n", C.c_int32), ("leader_index", C.c_int32), ("flags", C.c_int32),
                ("reserved", C.c_int32), ("d0", C.c_double), ("t0", C.c_double),
                ("d_safe", C.c_double)]


class LocalDesc(C.Structure):
    _fields_ = [("N", C.c_int32), ("max_nodes", C.c_int32), ("d0", C.c_double), ("t0", C.c_double),
                ("tight", C.c_double), ("mip_gap", C.c_double), ("time_limit_ms", C.c_double),
                ("modes_hint", C.c_void_p)]


class MpcDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("model", C.c_int32), ("n_local", C.c_int32), ("N", C.c_int32),
                ("flags", C.c_int32), ("leader_index", C.c_int32), ("n_front", C.c_int32),
                ("n_behind", C.c_int32), ("max_nodes", C.c_int32), ("one_norm", C.c_int32),
                ("d0", C.c_double), ("t0", C.c_double), ("tight", C.c_double), ("rho", C.c_double),
                ("mip_gap", C.c_double), ("time_limit_ms", C.c_double)]


class GAdmmRole(C.Structure):      # hvp_gadmm_role: the buffers of one role's hvp_mpc_solve_dev call
    _fields_ = [(k, C.c_void_p) for k in ("params", "x0", "mass", "fixed_modes", "u", "x", "extra", "obj", "status")]


class GAdmmRound(C.Structure):     # hvp_gadmm_round
    _fields_ = [("n", C.c_int32), ("N", C.c_int32), ("S", C.c_int32), ("init", C.c_int32), ("rho", C.c_double),
                ("mug", C.c_double), ("edge", C.c_double * 6), ("cf", C.c_double * 7), ("bg", C.c_double * 7),
                ("dd", C.c_double * 7), ("role", GAdmmRole * 3)] + \
               [(k, C.c_void_p) for k in ("x", "mass", "lwin", "y", "u", "tr", "cost", "ok")]


class DecentObserve(C.Structure):  # hvp_decent_observe
    _fields_ = [("n", C.c_int32), ("N", C.c_int32), ("S", C.c_int32), ("leader_index", C.c_int32),
                ("leader_len", C.c_int64), ("leader_per_scenario", C.c_int32), ("reserved", C.c_int32), ("ts", C.c_double)] + \
               [(k, C.c_void_p) for k in ("x", "leader_x", "t", "xf", "xb", "xl")]


class AdmmRole(C.Structure):       # hvp_admm_role
    _fields_ = [("params", C.c_void_p), ("x", C.c_void_p), ("extra", C.c_void_p), ("has_front", C.c_int32),
                ("has_back", C.c_int32)]


class AdmmRound(C.Structure):      # hvp_admm_round
    _fields_ = [("n", C.c_int32), ("N", C.c_int32), ("S", C.c_int32), ("nroles", C.c_int32), ("pack_only", C.c_int32),
                ("reserved", C.c_int32), ("rho", C.c_double), ("role", AdmmRole * 4), ("role_of", C.c_int32 * 64)] + \
               [(k, C.c_void_p) for k in ("lwin", "y_front", "y_back", "zf", "zb", "xs")]


class CentStep(C.Structure):       # hvp_cent_step
    _fields_ = [("n", C.c_int32), ("N", C.c_int32), ("S", C.c_int32), ("phase", C.c_int32), ("n_param", C.c_int32),
                ("leader_per_scenario", C.c_int32), ("leader_len", C.c_int64), ("T", C.c_int64), ("n_modes", C.c_int32),
                ("reserved", C.c_int32), ("mode_gear", C.c_int32 * 16)] + \
               [(k, C.c_void_p) for k in ("t", "leader_x", "params", "u", "modes", "obj", "status", "nodes", "u0", "gear0",
                                          "U_log", "obj_log", "status_log", "nodes_log", "aborted_at")]


class EventGroup(C.Structure):     # hvp_event_group: the buffers of one group's eval and solve launches
    _fields_ = [(k, C.c_void_p) for k in ("x0", "xg", "ug", "params", "cost", "u", "x", "modes", "obj", "status", "nodes")] + \
               [("n_local", C.c_int32), ("n_param", C.c_int32), ("has_leader", C.c_int32), ("reserved", C.c_int32)]


class EventIter(C.Structure):      # hvp_event_iter
    _fields_ = [("n", C.c_int32), ("N", C.c_int32), ("S", C.c_int32), ("phase", C.c_int32), ("iters", C.c_int32),
                ("it", C.c_int32), ("ngroups", C.c_int32), ("leader_per_scenario", C.c_int32), ("leader_len", C.c_int64),
                ("T", C.c_int64), ("threshold", C.c_double), ("n_modes", C.c_int32), ("reserved", C.c_int32),
                ("mode_gear", C.c_int32 * 16), ("group_of", C.c_int32 * 64), ("slot_of", C.c_int32 * 64),
                ("group", EventGroup * 8)] + \
               [(k, C.c_void_p) for k in ("t", "x", "leader_x", "SG", "UG", "GG", "active", "WIN", "FEAS", "ND", "U_log",
                                          "u0", "gear0")]


class AdmmStepRole(C.Structure):   # hvp_admm_step_role: the buffers of one role's solve launch
    _fields_ = [(k, C.c_void_p) for k in ("params", "x0", "u", "x", "extra", "modes", "status", "nodes")] + \
               [("has_front", C.c_int32), ("has_back", C.c_int32)]


class AdmmStep(C.Structure):       # hvp_admm_step
    _fields_ = [("n", C.c_int32), ("N", C.c_int32), ("S", C.c_int32), ("phase", C.c_int32), ("nroles", C.c_int32),
                ("leader_per_scenario", C.c_int32), ("leader_len", C.c_int64), ("T", C.c_int64), ("rho", C.c_double),
                ("n_modes", C.c_int32), ("reserved", C.c_int32), ("mode_gear", C.c_int32 * 16),
                ("role", AdmmStepRole * 4), ("role_of", C.c_int32 * 64)] + \
               [(k, C.c_void_p) for k in ("t", "r", "x", "leader_x", "y_front", "y_back", "zf", "zb", "xs", "ND",
                                          "failed_at", "u0", "gear0", "U_log", "ST")]


CENT_PACK, CENT_ADOPT = 0, 1
EVENT_PACK, EVENT_SELECT, EVENT_ADOPT = 0, 1, 2
ADMM_PACK, ADMM_ROUND, ADMM_ADOPT = 0, 1, 2
MPC_CENT, MPC_LOCAL, MPC_EVENT, MPC_ADMM, MPC_GADMM = 1, 2, 3, 4, 5
MODEL_PWA_GEAR, MODEL_FRICTION_GEAR = 0, 1
REAL_VEHICLE_REF, NO_LEADER = 8, -100


def build(verbose: bool = False) -> str:
    """Compile libhvp.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-j", str(min(8, os.cpu_count() or 1)), "-C", CSRC, "libhvp.so"], capture_output=True, text=True)
    if verbose or out.returncode:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode:
        raise RuntimeError("building libhvp.so failed")
    return LIB_PATH


_lib = None
_vp = C.c_void_p


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(hybrid_vehicle_platoon_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.hvp_version.restype = C.c_int
    L.hvp_last_error.argtypes = [C.c_char_p, C.c_int]
    L.hvp_device_count.restype = C.c_int
    L.hvp_ctx_create.argtypes = [C.c_int, C.POINTER(_vp)]
    L.hvp_ctx_destroy.argtypes = [_vp]
    L.hvp_ctx_stream.argtypes = [_vp]
    L.hvp_ctx_stream.restype = _vp
    L.hvp_ctx_synchronize.argtypes = [_vp]
    L.hvp_ctx_launch_count.argtypes = [_vp]
    L.hvp_ctx_launch_count.restype = C.c_int64
    L.hvp_ctx_last_kernel_ms.argtypes = [_vp]
    L.hvp_ctx_last_kernel_ms.restype = C.c_float
    roll = [_vp, C.POINTER(EnvDesc), C.c_int64] + [_vp] * 9
    L.hvp_rollout_step_dev.argtypes = roll + [_vp]
    L.hvp_rollout_step_host.argtypes = roll
    loc = [_vp, C.POINTER(LocalDesc), C.c_int64] + [_vp] * 13
    L.hvp_local_miqp_dev.argtypes = loc + [_vp]
    L.hvp_local_miqp_host.argtypes = loc
    L.hvp_mpc_create.argtypes = [_vp, C.POINTER(MpcDesc), C.POINTER(_vp)]
    L.hvp_mpc_destroy.argtypes = [_vp]
    L.hvp_mpc_info.argtypes = [_vp, C.POINTER(C.c_int32)]
    L.hvp_mpc_mode_table.argtypes = [_vp, _vp, _vp, _vp]
    mpc = [_vp, C.c_int64] + [_vp] * 12
    L.hvp_mpc_solve_dev.argtypes = mpc + [_vp]
    L.hvp_mpc_solve_host.argtypes = mpc
    L.hvp_mpc_solve_shard_dev.argtypes = [_vp, C.c_int64, _vp, _vp, _vp] + [C.c_int32] * 5 + [_vp] * 10
    L.hvp_mpc_eval_dev.argtypes = [_vp, C.c_int64] + [_vp] * 6
    L.hvp_mpc_eval_host.argtypes = [_vp, C.c_int64] + [_vp] * 5
    L.hvp_gadmm_round_dev.argtypes = [_vp, C.POINTER(GAdmmRound), _vp]
    L.hvp_decent_observe_dev.argtypes = [_vp, C.POINTER(DecentObserve), _vp]
    L.hvp_admm_round_dev.argtypes = [_vp, C.POINTER(AdmmRound), _vp]
    L.hvp_cent_step_dev.argtypes = [_vp, C.POINTER(CentStep), _vp]
    L.hvp_event_iter_dev.argtypes = [_vp, C.POINTER(EventIter), _vp]
    L.hvp_admm_step_dev.argtypes = [_vp, C.POINTER(AdmmStep), _vp]
    L.hvp_microbench_fp64.argtypes = [_vp, C.c_int, C.POINTER(C.c_double)]
    L.hvp_microbench_smem.argtypes = [_vp, C.c_int, C.POINTER(C.c_double)]
    _lib = L
    return L


def last_error() -> str:
    buf = C.create_string_buffer(512)
    lib().hvp_last_error(buf, 512)
    return buf.value.decode()


def check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError(f"libhvp error {rc}: {last_error()}")


class Context:
    """One device + one stream (hvp_ctx)."""

    def __init__(self, device: int = 0):
        L = lib()
        if L.hvp_device_count() <= 0:
            raise RuntimeError("no CUDA device visible: hybrid_vehicle_platoon_b200 has no CPU path")
        h = _vp()
        check(L.hvp_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)
        # compiled formulations built on this context: destroyed WITH it (hvp_mpc_destroy reads its context, so a handle
        # must never outlive it -- and sweeps keep handles in caches that do)
        import weakref
        self._children = weakref.WeakSet()

    def _register(self, child):
        self._children.add(child)

    @property
    def handle(self):
        return self._h

    @property
    def stream(self) -> int:
        return lib().hvp_ctx_stream(self._h) or 0

    def synchronize(self):
        check(lib().hvp_ctx_synchronize(self._h))

    @property
    def launch_count(self) -> int:
        return lib().hvp_ctx_launch_count(self._h)

    def last_kernel_ms(self) -> float:
        return lib().hvp_ctx_last_kernel_ms(self._h)

    def close(self):
        if getattr(self, "_h", None):
            for child in list(getattr(self, "_children", ())):
                child.close()
            lib().hvp_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: dict[int, Context] = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
