"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

ctypes view of tests/quant_oracle.c, the executable specification of the fixed-point layered min-sum decoder (DESIGN.md §3.7).
The library is compiled on first use into a temporary directory, so the tree stays read-only; codes are oracle.oracle.Code
objects and layers are lists of check-index arrays (Context.layers() / Code.auto_layers()).
"""
import atexit
import ctypes as ct
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "quant_oracle.c")
AWGN, BSC, RAYLEIGH = 1, 2, 4
KIND = {"AWGN": AWGN, "BSC": BSC, "RAYLEIGH": RAYLEIGH}


class Quant(ct.Structure):  # ldpc_b200_quant
    _fields_ = [("ch_bits", ct.c_int), ("msg_bits", ct.c_int), ("post_bits", ct.c_int), ("offset", ct.c_int), ("scale8", ct.c_int),
                ("step", ct.c_double)]


def quant(ch_bits, msg_bits, post_bits, step, offset=0, scale8=8):
    return Quant(int(ch_bits), int(msg_bits), int(post_bits), int(offset), int(scale8), float(step))


_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="quant_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libquant_oracle.so")
        subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-o", so, SRC, "-lm"], check=True)
        L = ct.CDLL(so)
        vp, ip, qp = ct.c_void_p, ct.POINTER(ct.c_int), ct.POINTER(Quant)
        i32p = ct.POINTER(ct.c_int32)
        L.orc_quantize.restype = ct.c_int32
        L.orc_quantize.argtypes = [ct.c_double, qp]
        L.orc_check_q.argtypes = [ct.c_int, i32p, qp, i32p]
        L.orc_decode_layered_q.restype = ct.c_int
        L.orc_decode_layered_q.argtypes = [vp, ct.c_int, ip, ip, ct.POINTER(ct.c_double), ct.c_int, ct.c_int, qp, ct.POINTER(ct.c_double),
                                           ct.POINTER(ct.c_uint8), i32p, ct.POINTER(ct.c_uint64)]
        L.orc_sim_point_layered_q.argtypes = [vp, ct.c_int, ip, ip, ct.c_int, ct.c_double, ct.c_int, ct.c_int, ct.c_int, qp, ct.c_uint64,
                                              ct.c_uint32, ct.c_uint64, ct.c_uint64, ct.c_int, ct.POINTER(ct.c_uint64)]
        _lib = L
    return _lib


def _layers(layers):
    ptr = np.zeros(len(layers) + 1, dtype=np.int32)
    ptr[1:] = np.cumsum([len(l) for l in layers])
    chk = np.ascontiguousarray(np.concatenate([np.asarray(l, dtype=np.int32) for l in layers]), dtype=np.int32)
    return ptr, chk


def _ip(a):
    return a.ctypes.data_as(ct.POINTER(ct.c_int))


def quantize(values, q):
    f = lib().orc_quantize
    return np.array([f(float(v), ct.byref(q)) for v in np.asarray(values, dtype=np.float64).reshape(-1)], dtype=np.int32)


def check(v, q):
    """The check rule on one check's v2c values (list of ints) -> its check-to-variable messages."""
    v = np.ascontiguousarray(v, dtype=np.int32)
    r = np.zeros_like(v)
    lib().orc_check_q(len(v), v.ctypes.data_as(ct.POINTER(ct.c_int32)), ct.byref(q), r.ctypes.data_as(ct.POINTER(ct.c_int32)))
    return r


def decode(code, llr_in, layers, q, iterations=50, early_term=True):
    """[n, nc] fp64 LLRs -> (llr_out [n, nc] = P * step, co [n, nc], iters [n], P [n, nc] int32, clips): clips counts the
    saturations and message clips that changed a value, over all frames."""
    x = np.ascontiguousarray(llr_in, dtype=np.float64).reshape(-1, code.nc)
    out = np.empty_like(x)
    co = np.empty(x.shape, dtype=np.uint8)
    post = np.empty(x.shape, dtype=np.int32)
    its = np.empty(x.shape[0], dtype=np.int32)
    clips = ct.c_uint64(0)
    ptr, chk = _layers(layers)
    for t in range(x.shape[0]):
        its[t] = lib().orc_decode_layered_q(ct.cast(code._p, ct.c_void_p), len(layers), _ip(ptr), _ip(chk),
                                            x[t].ctypes.data_as(ct.POINTER(ct.c_double)), int(iterations), int(early_term), ct.byref(q),
                                            out[t].ctypes.data_as(ct.POINTER(ct.c_double)), co[t].ctypes.data_as(ct.POINTER(ct.c_uint8)),
                                            post[t].ctypes.data_as(ct.POINTER(ct.c_int32)), ct.byref(clips))
    return out, co, its, post, int(clips.value)


def sim_point(code, layers, channel, x, q, coherence=1, seed=0, point=0, frame0=0, nframes=100, iterations=50, early_term=True, threads=1):
    """-> dict(fec, bec, frames, iters) over frames [frame0, frame0 + nframes), all-zero codeword."""
    cnt = (ct.c_uint64 * 4)()
    ptr, chk = _layers(layers)
    lib().orc_sim_point_layered_q(ct.cast(code._p, ct.c_void_p), len(layers), _ip(ptr), _ip(chk), KIND[channel], float(x), int(coherence),
                                  int(iterations), int(early_term), ct.byref(q), int(seed), int(point), int(frame0), int(nframes),
                                  int(threads), cnt)
    return dict(fec=int(cnt[0]), bec=int(cnt[1]), frames=int(cnt[2]), iters=int(cnt[3]))
