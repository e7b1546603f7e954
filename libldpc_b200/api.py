"""ctypes binding of the handle-based C ABI (include/ldpc_b200.h, part 2).

Pure plumbing: every call goes straight into libldpc.so; there is no Python or CPU implementation of
the decode path here, and a missing library / missing GPU raises.
"""
import ctypes as ct
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path():
    """libldpc.so beside this file; LDPC_B200_LIB names another build of the same library (debug / phase-timing builds)."""
    return os.environ.get("LDPC_B200_LIB") or os.path.join(_HERE, "libldpc.so")


class decoder_param(ct.Structure):  # reference: src/core/functions.h:107-112, pyLDPC/ldpc.py:16-19
    _fields_ = [("earlyTerm", ct.c_bool), ("iterations", ct.c_uint32), ("type", ct.c_char_p)]


class channel_param(ct.Structure):  # reference: src/core/functions.h:114-119, pyLDPC/ldpc.py:21-24
    _fields_ = [("seed", ct.c_uint64), ("xRange", ct.c_double * 3), ("type", ct.c_char_p)]


class simulation_param(ct.Structure):  # reference: src/core/functions.h:121-127, pyLDPC/ldpc.py:26-30
    _fields_ = [("threads", ct.c_uint32), ("maxFrames", ct.c_uint64), ("fec", ct.c_uint64), ("resultFile", ct.c_char_p)]


class sim_results_t(ct.Structure):  # reference: src/sim/ldpcsim.h:23-31, pyLDPC/ldpc.py:8-14
    _fields_ = [("fer", ct.POINTER(ct.c_double)), ("ber", ct.POINTER(ct.c_double)), ("avg_iter", ct.POINTER(ct.c_double)),
                ("time", ct.POINTER(ct.c_double)), ("fec", ct.POINTER(ct.c_uint64)), ("frames", ct.POINTER(ct.c_uint64))]


class code_info(ct.Structure):
    _fields_ = [(k, ct.c_int) for k in ("nc", "mc", "nnz", "kc", "nct", "mct", "kct", "n_punct", "n_short", "max_degree",
                                         "max_check_degree", "max_var_degree", "has_generator", "g_rows", "g_cols", "g_nnz")]


class tuning(ct.Structure):
    _fields_ = [(k, ct.c_int) for k in ("precision", "residency", "frames_per_cta", "threads_per_cta", "ctas", "bec_deg1_compat", "tmem", "idx16", "zero_codeword", "schedule", "layered_ms_scale64")]


class quant(ct.Structure):  # ldpc_b200_quant
    _fields_ = [("ch_bits", ct.c_int), ("msg_bits", ct.c_int), ("post_bits", ct.c_int), ("offset", ct.c_int), ("scale8", ct.c_int),
                ("step", ct.c_double)]


class error_record(ct.Structure):  # ldpc_b200_error_record
    _fields_ = [("frame", ct.c_uint64), ("bit_errors", ct.c_uint32), ("iterations", ct.c_int32)]


class frame_report(ct.Structure):  # ldpc_b200_frame_report
    _fields_ = [("frame", ct.c_uint64), ("iterations", ct.c_int32), ("bit_errors", ct.c_uint32), ("syndrome_weight", ct.c_uint32),
                ("bits_offset", ct.c_int64), ("checks_offset", ct.c_int64)]


class stats(ct.Structure):
    _fields_ = [("device_ms", ct.c_double), ("launches", ct.c_uint64), ("frames", ct.c_uint64), ("edge_iterations", ct.c_uint64),
                ("frames_per_cta", ct.c_int), ("threads_per_cta", ct.c_int), ("ctas", ct.c_int), ("residency", ct.c_int),
                ("precision", ct.c_int), ("smem_bytes", ct.c_size_t)]


ALLREDUCE_FN = ct.CFUNCTYPE(None, ct.POINTER(ct.c_uint64), ct.c_int, ct.c_void_p)
ROUND_FN = ct.CFUNCTYPE(ct.c_int, ct.c_uint32, ct.c_double, ct.c_uint64, ct.c_uint64, ct.POINTER(ct.c_uint64), ct.c_void_p)
F64, F32 = 0, 1
FIXED = 2  # stats()["precision"] of the fixed-point layered decoder (Context.set_quant)
AUTO, SMEM, GLOBAL = 0, 1, 2
LLR_F64, LLR_F32, LLR_I8 = 0, 1, 2
FLOODING, LAYERED = 0, 1

REFERENCE_SYMBOLS = ("ldpc_setup", "simulate", "calculate_rank", "encode", "decode", "syndrome")
HANDLE_SYMBOLS = ("ldpc_b200_last_error", "ldpc_b200_version", "ldpc_b200_device_count", "ldpc_b200_open", "ldpc_b200_close",
                  "ldpc_b200_info", "ldpc_b200_set_tuning", "ldpc_b200_get_tuning", "ldpc_b200_get_edges", "ldpc_b200_get_bit_pos",
                  "ldpc_b200_get_puncture", "ldpc_b200_get_layout", "ldpc_b200_rank", "ldpc_b200_encode", "ldpc_b200_syndrome",
                  "ldpc_b200_decode_batch", "ldpc_b200_decode_batch_device", "ldpc_b200_decode_bec_batch", "ldpc_b200_channel",
                  "ldpc_b200_sim_point", "ldpc_b200_sim_point_async", "ldpc_b200_simulate", "ldpc_b200_simulate_ex", "ldpc_b200_get_stats",
                  "ldpc_b200_reset_stats", "ldpc_b200_smem_probe", "ldpc_b200_sim_point_log", "ldpc_b200_prepare", "ldpc_b200_decode_batch_ex", "ldpc_b200_decode_batch_device_ex", "ldpc_b200_get_bec_layout", "ldpc_b200_fp64_probe", "ldpc_b200_set_layers", "ldpc_b200_load_layers", "ldpc_b200_get_layers", "ldpc_b200_set_modulation",
                  "ldpc_b200_error_report", "ldpc_b200_set_fading", "ldpc_b200_set_quant", "ldpc_b200_get_quant")

_lib = None


class _Missing:
    """Stands in for a symbol an older build of the library lacks (A/B runs against earlier builds): calling it raises."""
    def __init__(self, name):
        self.name, self.argtypes, self.restype = name, None, None

    def __call__(self, *a):
        raise RuntimeError(f"{self.name} is not exported by this build of libldpc.so")


class _Tolerant:
    def __init__(self, lib):
        object.__setattr__(self, "_lib", lib)
        object.__setattr__(self, "_missing", {})

    def __getattr__(self, name):
        try:
            return getattr(self._lib, name)
        except AttributeError:
            return self._missing.setdefault(name, _Missing(name))


def load_library(path=None):
    """Loads libldpc.so and declares the prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or lib_path()
    if not os.path.exists(p):
        raise RuntimeError(f"{p} is missing: build it with `python -m libldpc_b200.build` (there is no fallback path)")
    L = _Tolerant(ct.CDLL(p))
    vp, i64, u64, u32 = ct.c_void_p, ct.c_int64, ct.c_uint64, ct.c_uint32
    dptr, bptr, iptr = ct.POINTER(ct.c_double), ct.POINTER(ct.c_uint8), ct.POINTER(ct.c_int)
    L.ldpc_b200_last_error.restype = ct.c_char_p
    L.ldpc_b200_version.restype = ct.c_char_p
    L.ldpc_b200_device_count.restype = ct.c_int
    L.ldpc_b200_open.restype = vp
    L.ldpc_b200_open.argtypes = [ct.c_char_p, ct.c_char_p, ct.c_int]
    L.ldpc_b200_close.argtypes = [vp]
    L.ldpc_b200_info.argtypes = [vp, ct.POINTER(code_info)]
    L.ldpc_b200_set_tuning.argtypes = [vp, ct.POINTER(tuning)]
    L.ldpc_b200_get_tuning.argtypes = [vp, ct.POINTER(tuning)]
    L.ldpc_b200_prepare.argtypes = [vp, decoder_param, u64]
    L.ldpc_b200_get_edges.argtypes = [vp, iptr, iptr]
    L.ldpc_b200_get_bit_pos.argtypes = [vp, iptr]
    L.ldpc_b200_get_puncture.argtypes = [vp, iptr, iptr]
    L.ldpc_b200_get_layout.argtypes = [vp, iptr, iptr, iptr, iptr, iptr]
    L.ldpc_b200_get_bec_layout.argtypes = [vp, iptr, iptr]
    L.ldpc_b200_set_modulation.argtypes = [vp, ct.c_int, iptr, iptr]
    L.ldpc_b200_set_fading.argtypes = [vp, ct.c_int]
    L.ldpc_b200_set_quant.argtypes = [vp, ct.POINTER(quant)]
    L.ldpc_b200_get_quant.argtypes = [vp, ct.POINTER(quant)]
    L.ldpc_b200_set_layers.argtypes = [vp, ct.c_int, iptr, iptr]
    L.ldpc_b200_load_layers.argtypes = [vp, ct.c_char_p]
    L.ldpc_b200_get_layers.argtypes = [vp, iptr]
    L.ldpc_b200_rank.argtypes = [vp]
    L.ldpc_b200_encode.argtypes = [vp, bptr, bptr]
    L.ldpc_b200_syndrome.argtypes = [vp, bptr, bptr]
    L.ldpc_b200_decode_batch.argtypes = [vp, decoder_param, dptr, i64, dptr, bptr, ct.POINTER(ct.c_int32)]
    L.ldpc_b200_decode_batch_ex.argtypes = [vp, decoder_param, vp, ct.c_int, ct.c_double, i64, dptr, bptr, ct.POINTER(u32), ct.POINTER(ct.c_int32)]
    L.ldpc_b200_decode_batch_device_ex.argtypes = [vp, decoder_param, vp, ct.c_int, ct.c_double, i64, vp, vp, vp, vp, vp]
    L.ldpc_b200_decode_batch_device.argtypes = [vp, decoder_param, vp, i64, vp, vp, vp, vp]
    L.ldpc_b200_decode_bec_batch.argtypes = [vp, decoder_param, bptr, bptr, i64, bptr, bptr, ct.POINTER(ct.c_int32)]
    L.ldpc_b200_channel.argtypes = [vp, ct.c_char_p, ct.c_double, u64, u32, u64, i64, bptr, dptr, bptr]
    L.ldpc_b200_sim_point.argtypes = [vp, decoder_param, ct.c_char_p, ct.c_double, u64, u32, u64, u64, ct.POINTER(u64), ct.POINTER(ct.c_float)]
    L.ldpc_b200_sim_point_async.argtypes = [vp, decoder_param, ct.c_char_p, ct.c_double, u64, u32, u64, u64, vp, vp]
    L.ldpc_b200_simulate.argtypes = [vp, decoder_param, channel_param, simulation_param, ct.POINTER(sim_results_t), ct.POINTER(ct.c_bool),
                                     ct.c_int, ct.c_int, ALLREDUCE_FN, vp, ct.c_int]
    L.ldpc_b200_simulate_ex.argtypes = [vp, decoder_param, channel_param, simulation_param, ct.POINTER(sim_results_t), ct.POINTER(ct.c_bool),
                                        ct.c_int, ct.c_int, ALLREDUCE_FN, ROUND_FN, vp, ct.c_int]
    L.ldpc_b200_get_stats.argtypes = [vp, ct.POINTER(stats)]
    L.ldpc_b200_reset_stats.argtypes = [vp]
    L.ldpc_b200_smem_probe.argtypes = [vp, ct.POINTER(ct.c_double)]
    L.ldpc_b200_fp64_probe.argtypes = [vp, ct.POINTER(ct.c_double)]
    L.ldpc_b200_sim_point_log.argtypes = [vp, decoder_param, ct.c_char_p, ct.c_double, u64, u32, u64, u64, ct.POINTER(u64), ct.POINTER(error_record),
                                          i64, ct.POINTER(i64)]
    L.ldpc_b200_error_report.argtypes = [vp, decoder_param, ct.c_char_p, ct.c_double, u64, u32, ct.POINTER(u64), i64, ct.POINTER(frame_report),
                                         ct.POINTER(ct.c_int32), i64, ct.POINTER(ct.c_int32), i64, ct.POINTER(i64), ct.POINTER(i64)]
    if path is None:
        _lib = L
    return L


def _p(a, ty):
    return a.ctypes.data_as(ct.POINTER(ty)) if a is not None else None


class Context:
    """One loaded code bound to one CUDA device (device=-1: host-only loader / GF(2) helpers)."""

    def __init__(self, pc_file, gen_file="", device=0, lib=None):
        self.lib = lib or load_library()
        self._h = self.lib.ldpc_b200_open(str(pc_file).encode(), str(gen_file or "").encode(), int(device))
        if not self._h:
            raise RuntimeError("ldpc_b200_open: " + self.lib.ldpc_b200_last_error().decode())
        ci = code_info()
        self._check(self.lib.ldpc_b200_info(self._h, ct.byref(ci)))
        for k, _ in code_info._fields_:
            setattr(self, k, getattr(ci, k))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.ldpc_b200_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(self.lib.ldpc_b200_last_error().decode())

    # ---- host-side views ---------------------------------------------------------------------
    def edges(self):
        r = np.empty(self.nnz, np.int32)
        c = np.empty(self.nnz, np.int32)
        self._check(self.lib.ldpc_b200_get_edges(self._h, _p(r, ct.c_int), _p(c, ct.c_int)))
        return r, c

    def bit_pos(self):
        b = np.empty(max(self.nct, 1), np.int32)
        self._check(self.lib.ldpc_b200_get_bit_pos(self._h, _p(b, ct.c_int)))
        return b[:self.nct]

    def puncture(self):
        p = np.empty(max(self.n_punct, 1), np.int32)
        s = np.empty(max(self.n_short, 1), np.int32)
        self._check(self.lib.ldpc_b200_get_puncture(self._h, _p(p, ct.c_int), _p(s, ct.c_int)))
        return p[:self.n_punct], s[:self.n_short]

    def layout(self):
        es = np.empty(self.nnz, np.int32)
        v = [ct.c_int() for _ in range(4)]
        self._check(self.lib.ldpc_b200_get_layout(self._h, _p(es, ct.c_int), *[ct.byref(x) for x in v]))
        return dict(edge_slot=es, n_slots=v[0].value, frames_per_cta=v[1].value, threads_per_cta=v[2].value, residency=v[3].value)

    def bec_layout(self):
        es = np.empty(self.nnz, np.int32)
        n = ct.c_int()
        self._check(self.lib.ldpc_b200_get_bec_layout(self._h, _p(es, ct.c_int), ct.byref(n)))
        return es, n.value

    def set_modulation(self, M=2, labels=None, bit_mapper=None):
        """M-ASK with bit-metric decoding for the AWGN sweep (M = 2: BPSK).  labels [M] (None: Gray), bit_mapper [log2 M, nct / log2 M]
        variable ids (None: consecutive transmitted positions per symbol)."""
        lab = np.ascontiguousarray(labels, np.int32) if labels is not None else None
        bm = np.ascontiguousarray(bit_mapper, np.int32) if bit_mapper is not None else None
        self._check(self.lib.ldpc_b200_set_modulation(self._h, int(M), _p(lab, ct.c_int), _p(bm, ct.c_int)))

    def set_fading(self, coherence=1):
        """Coherence length of the "RAYLEIGH" channel: transmitted positions per fading coefficient (1: fast fading, 0: one
        coefficient per frame)."""
        self._check(self.lib.ldpc_b200_set_fading(self._h, int(coherence)))

    def set_quant(self, ch_bits, msg_bits=None, post_bits=None, step=None, offset=0, scale8=8):
        """Fixed-point layered min-sum (DESIGN.md §3.7): channel LLRs quantised to ch_bits with LSB `step`, msg_bits check-to-variable
        messages, post_bits posteriors, offset beta in LSBs and normalisation factor scale8 / 8.  set_quant(None) turns it off.
        Needs the layered schedule and BP_MS."""
        if ch_bits is None or ch_bits == 0:
            self._check(self.lib.ldpc_b200_set_quant(self._h, None))
            return
        if msg_bits is None or post_bits is None or step is None:
            raise ValueError("set_quant needs ch_bits, msg_bits, post_bits and step")
        q = quant(int(ch_bits), int(msg_bits), int(post_bits), int(offset), int(scale8), float(step))
        self._check(self.lib.ldpc_b200_set_quant(self._h, ct.byref(q)))

    def quant(self):
        """The fixed-point setting as a dict, or None when it is off."""
        q = quant()
        self._check(self.lib.ldpc_b200_get_quant(self._h, ct.byref(q)))
        return {k: getattr(q, k) for k, _ in quant._fields_} if q.ch_bits else None

    def set_layers(self, layers=None):
        """Layers of the layered schedule: a list of check-index lists, or None for the built-in first-fit layering."""
        if not layers:
            self._check(self.lib.ldpc_b200_set_layers(self._h, 0, None, None))
            return
        ptr = np.zeros(len(layers) + 1, np.int32)
        ptr[1:] = np.cumsum([len(l) for l in layers])
        chk = np.ascontiguousarray(np.concatenate([np.asarray(l, np.int32) for l in layers]), np.int32)
        self._check(self.lib.ldpc_b200_set_layers(self._h, len(layers), _p(ptr, ct.c_int), _p(chk, ct.c_int)))

    def load_layers(self, path):
        self._check(self.lib.ldpc_b200_load_layers(self._h, str(path).encode()))

    def layers(self):
        """The layering in use as a list of check-index arrays."""
        lo = np.zeros(self.mc, np.int32)
        n = self.lib.ldpc_b200_get_layers(self._h, _p(lo, ct.c_int))
        if n < 0:
            raise RuntimeError(self.lib.ldpc_b200_last_error().decode())
        return [np.nonzero(lo == l)[0].astype(np.int32) for l in range(n)]

    def set_tuning(self, **kw):
        t = tuning()
        self._check(self.lib.ldpc_b200_get_tuning(self._h, ct.byref(t)))
        for k, v in kw.items():
            setattr(t, k, int(v))
        self._check(self.lib.ldpc_b200_set_tuning(self._h, ct.byref(t)))

    def rank(self):
        return self.lib.ldpc_b200_rank(self._h)

    def encode(self, info):
        info = np.ascontiguousarray(info, np.uint8)
        cw = np.zeros(self.nc, np.uint8)
        self._check(self.lib.ldpc_b200_encode(self._h, _p(info, ct.c_uint8), _p(cw, ct.c_uint8)))
        return cw

    def syndrome(self, word):
        word = np.ascontiguousarray(word, np.uint8)
        s = np.zeros(self.mc, np.uint8)
        self._check(self.lib.ldpc_b200_syndrome(self._h, _p(word, ct.c_uint8), _p(s, ct.c_uint8)))
        return s

    # ---- GPU path ------------------------------------------------------------------------------
    @staticmethod
    def _dp(decoding, iterations, early_term):
        return decoder_param(bool(early_term), int(iterations), decoding.encode())

    def decode_batch(self, llr, decoding="BP", iterations=50, early_term=True, want_llr=True, want_hard=True, out=None, hard=None, its=None):
        """llr [n, nc] float64 (full length) -> (llr_out [n,nc], hard [n,nc] u8, iters [n] i32).
        out / hard / its may be caller-provided C-contiguous arrays (e.g. views of pinned host memory)."""
        llr = np.ascontiguousarray(llr, np.float64).reshape(-1, self.nc)
        n = llr.shape[0]
        if out is None and want_llr:
            out = np.empty_like(llr)
        if hard is None and want_hard:
            hard = np.empty((n, self.nc), np.uint8)
        if its is None:
            its = np.empty(n, np.int32)
        assert out is None or (out.dtype == np.float64 and out.size == n * self.nc and out.flags.c_contiguous)
        assert hard is None or (hard.dtype == np.uint8 and hard.size == n * self.nc and hard.flags.c_contiguous)
        assert its.dtype == np.int32 and its.size == n and its.flags.c_contiguous
        self._check(self.lib.ldpc_b200_decode_batch(self._h, self._dp(decoding, iterations, early_term), _p(llr, ct.c_double), n,
                                                    _p(out, ct.c_double), _p(hard, ct.c_uint8), _p(its, ct.c_int32)))
        return out, hard, its

    def decode_batch_ex(self, llr, decoding="BP", iterations=50, early_term=True, scale=1.0, want_llr=False, want_hard=False, want_bits=True,
                        out=None, hard=None, bits=None, its=None):
        """Narrow encodings of decode_batch: llr [n, nc] float64 / float32 / int8 (LLR = int8 * scale); decisions bit-packed
        (bits [n, ceil(nc/32)] uint32, variable i = bit i%32 of word i/32).  -> (llr_out | None, hard | None, bits | None, iters)."""
        llr = np.ascontiguousarray(llr).reshape(-1, self.nc)
        ty = {np.dtype(np.float64): LLR_F64, np.dtype(np.float32): LLR_F32, np.dtype(np.int8): LLR_I8}[llr.dtype]
        n = llr.shape[0]
        hw = (self.nc + 31) // 32
        if out is None and want_llr:
            out = np.empty((n, self.nc), np.float64)
        if hard is None and want_hard:
            hard = np.empty((n, self.nc), np.uint8)
        if bits is None and want_bits:
            bits = np.empty((n, hw), np.uint32)
        if its is None:
            its = np.empty(n, np.int32)
        assert bits is None or (bits.dtype == np.uint32 and bits.size == n * hw and bits.flags.c_contiguous)
        self._check(self.lib.ldpc_b200_decode_batch_ex(self._h, self._dp(decoding, iterations, early_term), llr.ctypes.data_as(ct.c_void_p), ty,
                                                       float(scale), n, _p(out, ct.c_double), _p(hard, ct.c_uint8), _p(bits, ct.c_uint32),
                                                       _p(its, ct.c_int32)))
        return out, hard, bits, its

    def unpack_bits(self, bits):
        """bit-packed decisions [n, ceil(nc/32)] uint32 -> [n, nc] uint8"""
        b = np.unpackbits(np.ascontiguousarray(bits).view(np.uint8), axis=1, bitorder="little")
        return b[:, :self.nc]

    def decode_bec_batch(self, inp, cw, iterations=50, early_term=True):
        inp = np.ascontiguousarray(inp, np.uint8).reshape(-1, self.nc)
        cw = np.ascontiguousarray(cw, np.uint8).reshape(-1, self.nc)
        n = inp.shape[0]
        out = np.empty_like(inp)
        hard = np.empty_like(inp)
        its = np.empty(n, np.int32)
        self._check(self.lib.ldpc_b200_decode_bec_batch(self._h, self._dp("BP", iterations, early_term), _p(inp, ct.c_uint8),
                                                        _p(cw, ct.c_uint8), n, _p(out, ct.c_uint8), _p(hard, ct.c_uint8), _p(its, ct.c_int32)))
        return out, hard, its

    def channel(self, channel, x, seed, point, frame0, n):
        """Decoder inputs the simulator generates for frames [frame0, frame0+n): (cw, llr)."""
        cw = np.empty((n, self.nc), np.uint8)
        llr = np.zeros((n, self.nc), np.float64) if channel != "BEC" else None
        u8 = np.zeros((n, self.nc), np.uint8) if channel == "BEC" else None
        self._check(self.lib.ldpc_b200_channel(self._h, channel.encode(), float(x), int(seed), int(point), int(frame0), int(n),
                                               _p(cw, ct.c_uint8), _p(llr, ct.c_double), _p(u8, ct.c_uint8)))
        return cw, (u8 if channel == "BEC" else llr)

    def sim_point(self, channel, x, seed=0, point=0, frame0=0, nframes=1000, decoding="BP", iterations=50, early_term=True):
        cnt = (ct.c_uint64 * 4)()
        ms = ct.c_float()
        self._check(self.lib.ldpc_b200_sim_point(self._h, self._dp(decoding, iterations, early_term), channel.encode(), float(x), int(seed),
                                                 int(point), int(frame0), int(nframes), cnt, ct.byref(ms)))
        return dict(fec=int(cnt[0]), bec=int(cnt[1]), frames=int(cnt[2]), iters=int(cnt[3]), device_ms=float(ms.value))

    def sim_point_log(self, channel, x, seed=0, point=0, frame0=0, nframes=1000, decoding="BP", iterations=50, early_term=True, capacity=4096):
        """sim_point + the per-error diagnostics log: (counters dict, list of (global frame, bit errors, iterations), frames in error)."""
        cnt = (ct.c_uint64 * 4)()
        rec = (error_record * max(int(capacity), 1))()
        n = ct.c_int64()
        self._check(self.lib.ldpc_b200_sim_point_log(self._h, self._dp(decoding, iterations, early_term), channel.encode(), float(x), int(seed),
                                                     int(point), int(frame0), int(nframes), cnt, rec, int(capacity), ct.byref(n)))
        m = min(int(n.value), int(capacity))
        log = sorted((int(rec[i].frame), int(rec[i].bit_errors), int(rec[i].iterations)) for i in range(m))
        return dict(fec=int(cnt[0]), bec=int(cnt[1]), frames=int(cnt[2]), iters=int(cnt[3])), log, int(n.value)

    def error_report(self, channel, x, seed, point, frame, decoding="BP", iterations=50, early_term=True):
        """Replays ONE logged frame (the channel is counter-based, so its input is regenerated exactly) and returns what the
        reference's log_error prints: failed bit indices (transmitted positions), failed check indices, syndrome weight."""
        cw, llr = self.channel(channel, x, seed, point, frame, 1)
        if channel == "BEC":
            out, hard, its = self.decode_bec_batch(llr, cw, iterations, early_term)
        else:
            out, hard, its = self.decode_batch(llr, decoding, iterations, early_term)
        r, c = self.edges()
        synd = np.zeros(self.mc, np.uint8)
        np.bitwise_xor.at(synd, r, hard[0][c])
        tx = self.bit_pos()
        bad = tx[hard[0][tx] != cw[0][tx]]
        return dict(frame=int(frame), iterations=int(its[0]), failed_bits=[int(b) for b in bad], hamming_distance=int(len(bad)),
                    failed_checks=[int(i) for i in np.nonzero(synd)[0]], syndrome_weight=int(synd.sum()))

    def error_reports(self, channel, x, seed, point, frames, decoding="BP", iterations=50, early_term=True):
        """error_report for many frames at once, on the GPU (ldpc_b200_error_report): one dict per entry of `frames` (global frame
        indices of sweep point `point`; any order, repeats allowed), with the keys and values of error_report, under the current
        tuning.  With M-ASK the decisions are compared with the all-zero word the decoder sees."""
        fr = np.ascontiguousarray(frames, np.uint64).reshape(-1)
        n = fr.size
        rep = (frame_report * max(n, 1))()
        cap = [max(4096, 64 * n)] * 2
        for attempt in range(2):
            bits, checks = np.empty(cap[0], np.int32), np.empty(cap[1], np.int32)
            nb, nk = ct.c_int64(-1), ct.c_int64(-1)
            rc = self.lib.ldpc_b200_error_report(self._h, self._dp(decoding, iterations, early_term), channel.encode(), float(x), int(seed), int(point),
                                                 _p(fr, ct.c_uint64), n, rep, _p(bits, ct.c_int32), cap[0], _p(checks, ct.c_int32), cap[1],
                                                 ct.byref(nb), ct.byref(nk))
            if rc == 0:
                break
            if attempt or nb.value < 0 or (nb.value <= cap[0] and nk.value <= cap[1]):
                self._check(rc)
            cap = [nb.value, nk.value]      # the lists did not fit: once more with their exact sizes
        out = []
        for i in range(n):
            r = rep[i]
            fb = bits[r.bits_offset:r.bits_offset + r.bit_errors].tolist()
            fc = checks[r.checks_offset:r.checks_offset + r.syndrome_weight].tolist()
            out.append(dict(frame=int(r.frame), iterations=int(r.iterations), failed_bits=fb, hamming_distance=int(r.bit_errors),
                            failed_checks=fc, syndrome_weight=int(r.syndrome_weight)))
        return out

    def prepare(self, decoding="BP", iterations=50, early_term=True, nframes=1 << 20):
        """Runs the one-off kernel-shape trial for this (decoder, precision) now, so that asynchronous launches use its outcome."""
        self._check(self.lib.ldpc_b200_prepare(self._h, self._dp(decoding, iterations, early_term), int(nframes)))

    def sim_point_async(self, d_counters_ptr, stream_ptr, channel, x, seed=0, point=0, frame0=0, nframes=1000, decoding="BP",
                        iterations=50, early_term=True):
        self._check(self.lib.ldpc_b200_sim_point_async(self._h, self._dp(decoding, iterations, early_term), channel.encode(), float(x),
                                                       int(seed), int(point), int(frame0), int(nframes), ct.c_void_p(d_counters_ptr),
                                                       ct.c_void_p(stream_ptr)))

    def decode_batch_device(self, d_llr, n, d_llr_out, d_hard, d_iters, stream_ptr, decoding="BP", iterations=50, early_term=True):
        self._check(self.lib.ldpc_b200_decode_batch_device(self._h, self._dp(decoding, iterations, early_term), ct.c_void_p(d_llr), int(n),
                                                           ct.c_void_p(d_llr_out), ct.c_void_p(d_hard), ct.c_void_p(d_iters),
                                                           ct.c_void_p(stream_ptr)))

    def simulate(self, snr, channel="AWGN", decoding="BP", iterations=50, early_term=True, seed=0, max_frames=int(10e9), fec=50,
                 result_file="", rank=0, world=1, allreduce=None, quiet=True, max_points=512, round_fn=None):
        """Blocking sweep with the reference's semantics; returns the per-point result arrays.
        allreduce(values_ptr, n, user) sums a uint64 array over ranks; round_fn (tests / custom hosts)
        replaces the GPU launch, see ldpc_b200_simulate_ex."""
        res = sim_results_t(*[(ct.c_double * max_points)() for _ in range(4)], (ct.c_uint64 * max_points)(), (ct.c_uint64 * max_points)())
        stop = ct.c_bool(False)
        cb = ALLREDUCE_FN(allreduce) if allreduce is not None else ct.cast(None, ALLREDUCE_FN)
        cp = channel_param(int(seed), (ct.c_double * 3)(*snr), channel.encode())
        sp = simulation_param(1, int(max_frames), int(fec), str(result_file).encode())
        rf = ROUND_FN(round_fn) if round_fn is not None else ct.cast(None, ROUND_FN)
        self._check(self.lib.ldpc_b200_simulate_ex(self._h, self._dp(decoding, iterations, early_term), cp, sp, ct.byref(res), ct.byref(stop),
                                                   int(rank), int(world), cb, rf, None, int(bool(quiet))))
        n = int(np.sum(np.array(res.frames[0:max_points]) > 0))
        return {k: np.array(getattr(res, k)[0:n]) for k, _ in sim_results_t._fields_}

    def smem_probe(self):
        """Sustained shared-memory read bandwidth of this device, GB/s."""
        v = ct.c_double()
        self._check(self.lib.ldpc_b200_smem_probe(self._h, ct.byref(v)))
        return float(v.value)

    def fp64_probe(self):
        """Sustained FP64 instruction rate of this device, G thread-instructions/s."""
        v = ct.c_double()
        self._check(self.lib.ldpc_b200_fp64_probe(self._h, ct.byref(v)))
        return float(v.value)

    def stats(self, reset=False):
        s = stats()
        self._check(self.lib.ldpc_b200_get_stats(self._h, ct.byref(s)))
        d = {k: getattr(s, k) for k, _ in stats._fields_}
        if reset:
            self._check(self.lib.ldpc_b200_reset_stats(self._h))
        return d
