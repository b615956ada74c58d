"""TEST INFRASTRUCTURE: host build of the engine's __host__ __device__ functions (see horus_emu.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(os.path.dirname(_HERE))
_OUT = os.path.join(_HERE, "_build", "libhorus_emu.so")
_lib = None


def build(force=False, out=_OUT):
    src = os.path.join(_HERE, "horus_emu.cpp")
    deps = [src, os.path.join(_REPO, "gpuschedule_b200", "csrc", "gs_horus_core.cuh"),
            os.path.join(_REPO, "gpuschedule_b200", "csrc", "gs_horus_host.h"),
            os.path.join(_REPO, "include", "gsched.h"), os.path.join(_REPO, "include", "gsched_horus.h")]
    if not force and os.path.exists(out) and os.path.getmtime(out) >= max(os.path.getmtime(d) for d in deps):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-shared", "-x", "c++",
                    "-I", os.path.join(_REPO, "include"), "-I", os.path.join(_REPO, "gpuschedule_b200", "csrc"),
                    "-o", out, src], check=True)
    return out


def lib(out=_OUT):
    """the host build of the engine's core; `out` is where it is built (bench.py passes a temporary directory,
    because the tree it runs from may be read-only)"""
    global _lib
    if _lib is None:
        _lib = C.CDLL(build(out=out))
        _lib.emu_run_horus.restype = C.c_longlong
    return _lib


def run_horus(cluster, params, table, gauss, rows_cap, max_ticks_per_call=0, words=None, cooperative=False):
    """gauss: standard-normal values (horus / gandiva), or words: raw MT19937 words (any schedule, needed by horus+)"""
    from gpuschedule_b200.capi import HORUS_REC_DTYPE
    from gpuschedule_b200.log_manager import ROW_DTYPE
    n = table.n
    rows = np.zeros(rows_cap, dtype=ROW_DTYPE)
    util = np.zeros(rows_cap, dtype=np.float64)
    util_arr = np.zeros(rows_cap, dtype=np.uint8)
    recs = np.zeros(max(n, 1), dtype=HORUS_REC_DTYPE)
    fin = np.zeros(max(n, 1), dtype=np.int32)
    nfin, events, draws = C.c_longlong(0), C.c_longlong(0), C.c_longlong(0)
    arr = lambda a, dt: np.ascontiguousarray(a, dtype=dt)
    cols = [arr(table.arrive_tick, np.int32), arr(table.gpus, np.int32), arr(table.gpu_per_task, np.int32),
            arr(table.duration, np.float64), arr(table.mem_bytes, np.int64), arr(table.util_avg, np.float64),
            arr(table.util_max, np.float64)]
    ma = table.extra.get("mem_avg_mib")
    ma = None if ma is None else arr(ma, np.float64)
    g = None if gauss is None else arr(gauss, np.float64)
    w = None if words is None else arr(words, np.uint32)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    ticks = lib().emu_run_horus(C.byref(cluster), C.byref(params), C.c_longlong(n), *[p(c) for c in cols], p(ma), p(g),
                                C.c_longlong(0 if g is None else len(g)), p(w), C.c_longlong(0 if w is None else len(w)),
                                p(rows), p(util), p(util_arr), C.c_longlong(rows_cap), p(recs), p(fin),
                                C.byref(nfin), C.byref(events), C.byref(draws), C.c_longlong(max_ticks_per_call), C.c_int(int(cooperative)))
    return ticks, rows[:max(ticks, 0)], util[:max(ticks, 0)], util_arr[:max(ticks, 0)], recs[:n], fin[:nfin.value], events.value, draws.value


_ABI_OUT = os.path.join(_HERE, "_build", "libhorus_abi_emu.so")
_abi_lib = None


def build_abi(force=False):
    """gs_horus.cu itself -- the library's host side, every extern "C" entry point -- compiled with g++ against
    fake_cuda/cuda_runtime.h (device memory = host memory, kernels = the source's own host loop)."""
    src = os.path.join(_REPO, "gpuschedule_b200", "csrc", "gs_horus.cu")
    deps = [src, os.path.join(_HERE, "fake_cuda", "cuda_runtime.h"),
            os.path.join(_REPO, "gpuschedule_b200", "csrc", "gs_horus_core.cuh"),
            os.path.join(_REPO, "gpuschedule_b200", "csrc", "gs_horus_host.h"),
            os.path.join(_REPO, "include", "gsched.h"), os.path.join(_REPO, "include", "gsched_horus.h")]
    if not force and os.path.exists(_ABI_OUT) and os.path.getmtime(_ABI_OUT) >= max(os.path.getmtime(d) for d in deps):
        return _ABI_OUT
    os.makedirs(os.path.dirname(_ABI_OUT), exist_ok=True)
    subprocess.run(["g++", "-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-shared", "-x", "c++",
                    "-I", os.path.join(_HERE, "fake_cuda"), "-I", os.path.join(_REPO, "include"),
                    "-I", os.path.join(_REPO, "gpuschedule_b200", "csrc"), "-o", _ABI_OUT, src], check=True)
    return _ABI_OUT


def abi_lib():
    """the host build of the horus C ABI with the package's own ctypes prototypes on it"""
    global _abi_lib
    if _abi_lib is None:
        from gpuschedule_b200 import capi
        _abi_lib = capi.declare_horus_prototypes(C.CDLL(build_abi()))
    return _abi_lib


def emu_engine_class():
    """TEST INFRASTRUCTURE: capi.HorusEngine bound to the host-emulation build of gs_horus.cu.  The package itself has
    no way to select a library (capi.load_library only accepts the nvcc build); the substitution lives here, in tests/."""
    from gpuschedule_b200 import capi

    class EmuHorusEngine(capi.HorusEngine):
        @staticmethod
        def _library():
            lib = abi_lib()
            assert lib.gs_horus_build_tag() == b"host-emulation"
            return lib

    return EmuHorusEngine
