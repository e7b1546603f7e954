"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

ctypes view of tests/layered_f32_oracle.c: the binary32 layered min-sum specification (orc_decode_layered_f32) and a batch
frame loop that also runs the fp64 specification orc_decode_layered.  The library is compiled on first use into a temporary
directory, so the tree stays read-only; codes are oracle.oracle.Code objects and layers are lists of check-index arrays
(Context.layers() / Code.auto_layers()).
"""
import atexit
import ctypes as ct
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "layered_f32_oracle.c")

_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="layered_f32_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "liblayered_f32_oracle.so")
        subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-o", so, SRC, "-lm"], check=True)
        L = ct.CDLL(so)
        vp, ip = ct.c_void_p, ct.POINTER(ct.c_int)
        L.orc_decode_layered_batch.argtypes = [vp, ct.c_int, ip, ip, ct.POINTER(ct.c_double), ct.c_int64, ct.c_int, ct.c_int, ct.c_int,
                                               ct.c_double, ct.c_int, ct.c_int, ct.POINTER(ct.c_double), ct.POINTER(ct.c_uint8),
                                               ct.POINTER(ct.c_int32)]
        _lib = L
    return _lib


def decode(code, llr_in, layers, iterations=50, early_term=True, f32=True, minsum=True, ms_scale=1.0, threads=None):
    """[n, nc] fp64 LLRs -> (llr_out [n, nc] fp64, co [n, nc] u8, iters [n] i32) of the layered specification: binary32 min-sum
    (f32=True) or fp64 orc_decode_layered (min-sum or sum-product)."""
    if f32 and not minsum:
        raise ValueError("binary32 sum-product has no exact specification")
    x = np.ascontiguousarray(llr_in, dtype=np.float64).reshape(-1, code.nc)
    n = x.shape[0]
    out = np.empty_like(x)
    co = np.empty(x.shape, dtype=np.uint8)
    its = np.empty(n, dtype=np.int32)
    ptr = np.zeros(len(layers) + 1, dtype=np.int32)
    ptr[1:] = np.cumsum([len(l) for l in layers])
    chk = np.ascontiguousarray(np.concatenate([np.asarray(l, dtype=np.int32) for l in layers]), dtype=np.int32)
    ipp = ct.POINTER(ct.c_int)
    lib().orc_decode_layered_batch(ct.cast(code._p, ct.c_void_p), len(layers), ptr.ctypes.data_as(ipp), chk.ctypes.data_as(ipp),
                                   x.ctypes.data_as(ct.POINTER(ct.c_double)), n, int(iterations), int(early_term), int(minsum),
                                   float(ms_scale), int(f32), int(threads or os.cpu_count() or 1), out.ctypes.data_as(ct.POINTER(ct.c_double)),
                                   co.ctypes.data_as(ct.POINTER(ct.c_uint8)), its.ctypes.data_as(ct.POINTER(ct.c_int32)))
    return out, co, its
