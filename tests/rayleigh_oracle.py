"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

ctypes view of tests/rayleigh_oracle.c, the executable specification of the RAYLEIGH channel (DESIGN.md §3.2).  The library
is compiled on first use into a temporary directory, so the tree stays read-only; codes are oracle.oracle.Code objects.
"""
import atexit
import ctypes as ct
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "rayleigh_oracle.c")

_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="rayleigh_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "librayleigh_oracle.so")
        subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-o", so, SRC, "-lm"], check=True)
        L = ct.CDLL(so)
        vp, dp, bp = ct.c_void_p, ct.POINTER(ct.c_double), ct.POINTER(ct.c_uint8)
        L.orc_rayleigh_coeff.restype = ct.c_double
        L.orc_rayleigh_coeff.argtypes = [ct.c_uint64, ct.c_uint32, ct.c_uint64, ct.c_uint32]
        L.orc_channel_frame_rayleigh.argtypes = [vp, vp, ct.c_double, ct.c_int, ct.c_uint64, ct.c_uint32, ct.c_uint64, bp, dp]
        L.orc_sim_point_rayleigh.argtypes = [vp, vp, ct.c_int, ct.c_int, ct.c_int, ct.c_double, ct.c_int, ct.c_uint64, ct.c_uint32,
                                             ct.c_uint64, ct.c_uint64, ct.c_int, ct.POINTER(ct.c_uint64)]
        _lib = L
    return _lib


def _ptr(code):
    return ct.cast(code._p, ct.c_void_p) if code is not None else None


def coeffs(seed, point, frame, c):
    """Fading coefficients h of indices c (iterable) of one frame."""
    f = lib().orc_rayleigh_coeff
    return np.array([f(int(seed), int(point), int(frame), int(j)) for j in c], dtype=np.float64)


def channel_frames(code, x, coherence, seed, point, frame0, nframes, gen=None):
    """-> (cw [n, nc] u8, llr [n, nc] f64) of frames [frame0, frame0 + n)."""
    cw = np.zeros((nframes, code.nc), dtype=np.uint8)
    llr = np.zeros((nframes, code.nc), dtype=np.float64)
    for t in range(nframes):
        lib().orc_channel_frame_rayleigh(_ptr(code), _ptr(gen), float(x), int(coherence), int(seed), int(point), int(frame0 + t),
                                         cw[t].ctypes.data_as(ct.POINTER(ct.c_uint8)), llr[t].ctypes.data_as(ct.POINTER(ct.c_double)))
    return cw, llr


def sim_point(code, x, coherence, seed=0, point=0, frame0=0, nframes=100, decoding="BP", iterations=50, early_term=True, threads=1,
              gen=None):
    """-> dict(fec, bec, frames, iters) over frames [frame0, frame0 + nframes)."""
    cnt = (ct.c_uint64 * 4)()
    lib().orc_sim_point_rayleigh(_ptr(code), _ptr(gen), int(decoding == "BP_MS"), int(iterations), int(early_term), float(x),
                                 int(coherence), int(seed), int(point), int(frame0), int(nframes), int(threads), cnt)
    return dict(fec=int(cnt[0]), bec=int(cnt[1]), frames=int(cnt[2]), iters=int(cnt[3]))
