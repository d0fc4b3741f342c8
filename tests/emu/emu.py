"""TEST INFRASTRUCTURE: drives tests/emu/libmapad_emu.so, a plain-C++ build of the product's per-read
device logic (mapad_b200/csrc/*_core.cuh), so the non-GPU suite can compare it with the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np

from mapad_b200 import abi, api

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
# MAPAD_EMU_DEFS="-DMAPAD_COMPACT_CAND=1 ...": build and load a variant of the device logic (its own .so)
_DEFS = os.environ.get("MAPAD_EMU_DEFS", "").split()
_LIB = os.path.join(_HERE, "libmapad_emu%s.so" % ("_" + "_".join(d.replace("-D", "").replace("=", "") for d in _DEFS) if _DEFS else ""))
_lib = None
SMALL_CHUNKS = any(d.startswith("-DMAPAD_GCHUNK_SHIFT=") for d in _DEFS)  # variant build with tiny pool chunks


def build(force=False):
    csrc = os.path.join(_ROOT, "mapad_b200", "csrc")
    srcs = [os.path.join(_HERE, "emu_harness.cpp"), os.path.join(_HERE, "simt_emu.cpp")] + [os.path.join(csrc, f) for f in ("host_index.cpp", "host_params.cpp", "dev_index_build.cpp")]
    deps = srcs + [os.path.join(_HERE, "simt_emu.hpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc) if os.path.isfile(os.path.join(csrc, f))]
    if force or not os.path.exists(_LIB) or any(os.path.getmtime(d) > os.path.getmtime(_LIB) for d in deps):
        subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-fPIC", "-ffp-contract=off", "-march=x86-64-v3", "-shared", "-o", _LIB] + _DEFS + srcs + ["-ldl"])
    return _LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        L.emu_map_batch.restype = C.c_int
        L.emu_map_batch.argtypes = [C.c_void_p, C.POINTER(abi.Params), C.POINTER(abi.Reads), C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.emu_map_batch_group.restype = C.c_int
        L.emu_map_batch_group.argtypes = [C.c_void_p, C.POINTER(abi.Params), C.POINTER(abi.Reads), C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int,
                                          C.POINTER(C.c_uint32), C.POINTER(C.c_void_p)]
        L.emu_batch_view.argtypes = [C.c_void_p, C.POINTER(abi.Results)]
        L.emu_batch_free.argtypes = [C.c_void_p]
        L.emu_occ4.restype = C.c_int
        L.emu_occ4.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
        L.emu_sa_get.restype = C.c_int
        L.emu_sa_get.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.POINTER(C.c_uint64)]
        L.emu_libm_array.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def map_batch(index, params, seqs=None, quals=None, seeds=None, cap=1 << 16, layout=-1, packed=None, group=None, custom_penalties=None):
    """group=None: the per-thread reference loop (search_core.cuh::search_read); group=dict(G=8, n_groups=3, pool_chunks=64, lpt=1):
    the group kernel of search_group.cuh under the SIMT emulator.  custom_penalties: MAPAD_MODEL_CUSTOM's precomputed table."""
    if packed is None:
        packed = abi.pack_reads(seqs, quals)
    R, keep = api.make_reads(packed[0], packed[1], packed[2], seeds, custom_penalties)
    h = C.c_void_p()
    if group is None:
        rc = lib().emu_map_batch(index.h, C.byref(params), C.byref(R), cap, layout, C.byref(h))
    else:
        ng = int(group.get("n_groups", 3))
        nd = C.c_uint32(0)
        rc = lib().emu_map_batch_group(index.h, C.byref(params), C.byref(R), layout, int(group.get("G", 8)), ng,
                                       int(group.get("pool_chunks", 2 * ng + (4096 if SMALL_CHUNKS else 32))), int(group.get("lpt", 1)), C.byref(nd), C.byref(h))
        map_batch.last_deferred = int(nd.value)
    if rc != 0:
        raise api.MapadError(rc)
    try:
        v = abi.Results()
        lib().emu_batch_view(h, C.byref(v))
        out = abi.BatchResult(v)
        buf = C.create_string_buffer(1 << 16)
        out.xa = []
        for i in range(len(out)):
            k = api.lib().mapad_format_xa(index.h, C.byref(v), i, buf, 1 << 16)
            out.xa.append(buf.raw[:k].decode() if k >= 0 else None)
    finally:
        lib().emu_batch_free(h)
    return out


def occ4(index, row, layout=-1):
    out = (C.c_uint64 * 4)()
    b = C.c_uint32()
    rc = lib().emu_occ4(index.h, layout, row, out, C.byref(b))
    assert rc == 0
    return [int(x) for x in out], int(b.value)


def sa_get(index, row, layout=-1):
    out = C.c_uint64()
    rc = lib().emu_sa_get(index.h, layout, row, C.byref(out))
    assert rc == 0
    return int(out.value)


def libm(fn, values, iarg=0):
    x = np.ascontiguousarray(values, dtype=np.float32)
    y = np.zeros_like(x)
    lib().emu_libm_array(fn, iarg, len(x), x.ctypes.data, y.ctypes.data)
    return y
