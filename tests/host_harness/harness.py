"""ctypes loader of the HOST build of csrc/miqp_core.cuh (test harness only, see harness.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhvp_host_harness.so")
_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


def build(force=False):
    srcs = [os.path.join(_HERE, "harness.cpp"), os.path.join(_HERE, "scalar_solver.h"),
            os.path.join(_HERE, "../../hybrid_vehicle_platoon_b200/csrc/miqp_core.cuh"),
            os.path.join(_HERE, "../../hybrid_vehicle_platoon_b200/csrc/vehicle_model.h"),
            os.path.join(_HERE, "../../hybrid_vehicle_platoon_b200/csrc/coop_core.cuh"),
            os.path.join(_HERE, "../../hybrid_vehicle_platoon_b200/csrc/coop_backend.cuh"),
            os.path.join(_HERE, "../../hybrid_vehicle_platoon_b200/csrc/flat_core.cuh")]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-fPIC", "-shared", "-std=c++17", "-o", _SO, srcs[0]])
    return _SO


def local_miqp(N, flags, mass, x0, xf, xb, xl, d0=50.0, t0=0.0, tight=0.0, max_nodes=0, coop=False, flat=False):
    L = C.CDLL(build())
    fn = L.hvh_flat_miqp_batch if flat else (L.hvh_coop_miqp_batch if coop else L.hvh_local_miqp_batch)
    # references may be None (NULL): legal for the roles that do not read them
    fn.argtypes = [C.c_int, C.c_int, _ip, C.c_double, C.c_double, C.c_double,
                                       C.c_int, _dp, _dp, C.c_void_p, C.c_void_p, C.c_void_p, _dp, _dp, _ip, _dp, _ip,
                                       _ip, _ip]
    B = x0.shape[0]
    c = lambda a, t=np.float64: np.ascontiguousarray(a, dtype=t)
    refs = [None if a is None else c(a) for a in (xf, xb, xl)]
    ptr = lambda a: None if a is None else a.ctypes.data
    u = np.zeros((B, N)); x = np.zeros((B, 2, N + 1)); modes = np.zeros((B, N), np.int32)
    obj = np.zeros(B); st = np.zeros(B, np.int32); nodes = np.zeros(B, np.int32); it = np.zeros(B, np.int32)
    fn(B, N, c(flags, np.int32), d0, t0, tight, max_nodes, c(mass), c(x0), *map(ptr, refs), u, x, modes, obj, st, nodes, it)
    return dict(u=u, x=x, modes=modes, obj=obj, status=st, nodes=nodes, qp_iters=it)


def flat_adopt(N, flags, mass, x0, xf, xb, xl, after_nodes=1, d0=50.0, t0=0.0, tight=0.0):
    """Host emulation of the flat kernel's sub-tree adoption (harness.cpp: hvh_flat_adopt_batch)."""
    L = C.CDLL(build())
    fn = L.hvh_flat_adopt_batch
    fn.argtypes = [C.c_int, C.c_int, _ip, C.c_double, C.c_double, C.c_double, _dp, _dp, _dp, _dp, _dp, C.c_int, _dp, _ip, _ip]
    fn.restype = C.c_int
    B = x0.shape[0]
    c = lambda a, t=np.float64: np.ascontiguousarray(a, dtype=t)
    obj = np.zeros(B); ad = np.zeros(B, np.int32); nodes = np.zeros(B, np.int32)
    rc = fn(B, N, c(flags, np.int32), d0, t0, tight, c(mass), c(x0), c(xf), c(xb), c(xl), int(after_nodes), obj, ad, nodes)
    assert rc == 0
    return dict(obj=obj, adopters=ad, nodes=nodes)


def coop_split(N, M, flags, mass, x0, xf, xb, xl, d0=50.0, t0=0.0, tight=0.0):
    """Host emulation of the M-worker split search of the cooperative solver (harness.cpp: hvh_coop_split_batch)."""
    L = C.CDLL(build())
    fn = L.hvh_coop_split_batch
    fn.argtypes = [C.c_int, C.c_int, C.c_int, _ip, C.c_double, C.c_double, C.c_double, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip]
    B = x0.shape[0]
    c = lambda a, t=np.float64: np.ascontiguousarray(a, dtype=t)
    obj = np.zeros(B); ns = np.zeros(B, np.int32); nm = np.zeros(B, np.int32)
    fn(B, N, int(M), c(flags, np.int32), d0, t0, tight, c(mass), c(x0), c(xf), c(xb), c(xl), obj, ns, nm)
    return dict(obj=obj, nodes_sum=ns, nodes_max=nm)
