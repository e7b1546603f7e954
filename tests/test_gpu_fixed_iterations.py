"""Fixed-iteration min-sum decoding by the lock-step batch loop of the TMEM-mirror kernels (tile4.cuh, compiled without early
termination) against the same decode by the general half-iteration loop: the shared-memory kernel without the mirror, which
is compiled with early termination and runs with it switched off.  Posteriors, decisions, iteration counts and the five
counters (frames in error, bit errors, frames, reference iterations, executed iterations) must be bit-identical, for ragged
last batches, several batches per CTA, both automatic shapes, every frame source and iteration limits down to one.  The C
oracle is a second control where it is cheap."""
import ctypes as ct

import numpy as np
import pytest

from conftest import H_IRREGULAR

pytestmark = pytest.mark.gpu

SMEM = 1
AUTO = dict(frames_per_cta=0, threads_per_cta=0, ctas=0)
# h.txt in fp64: two CTAs per SM x 256 threads with 16-bit index tables, or one CTA per SM x 512 threads with 32-bit ones
SHAPES = {"pair16": dict(residency=SMEM, tmem=0, idx16=2, frames_per_cta=2, threads_per_cta=256, ctas=296),
          "one32": dict(residency=SMEM, tmem=0, idx16=1, **AUTO)}
CONTROL = dict(residency=SMEM, tmem=1, idx16=0, **AUTO)
ITERS = [1, 2, 3, 50]
# one frame, a ragged single batch, two batches of which the last is ragged (2 * 296 CTAs + 1), several batches per CTA
FRAMES = [1, 3, 2 * 296 + 1, 7 * 4 * 148 + 5]


def _tuning(ctx):
    from libldpc_b200 import api
    t = api.tuning()
    ctx._check(ctx.lib.ldpc_b200_get_tuning(ctx._h, ct.byref(t)))
    return {k: getattr(t, k) for k, _ in api.tuning._fields_}


@pytest.fixture
def ctx(gpu_ctx):
    saved = _tuning(gpu_ctx)
    yield gpu_ctx
    gpu_ctx.set_modulation(2)
    gpu_ctx.set_tuning(**saved)


@pytest.fixture(scope="module")
def irregular(built_lib):
    from libldpc_b200 import api
    from oracle import oracle as O
    c = api.Context(H_IRREGULAR, "", device=0)
    yield c, O.Code(H_IRREGULAR)
    c.close()


def _run(ctx, tuning, fn):
    """fn() under `tuning`, with the executed iterations of the launches it made (the fifth counter)"""
    ctx.set_tuning(**tuning)
    ctx.stats(reset=True)
    r = fn()
    return r, ctx.stats()["edge_iterations"]


def _llrs(rng, oc, n):
    llr = rng.normal(1.0, 1.6, size=(n, oc.nc))
    llr[:, oc.puncture] = 0.0
    llr[:, oc.shorten] = 99999.9
    llr[0, ::7] = -0.0
    return llr


def _same_decode(a, b):
    (out_a, hard_a, its_a), ei_a = a
    (out_b, hard_b, its_b), ei_b = b
    assert np.array_equal(its_a, its_b)
    assert np.array_equal(hard_a, hard_b)
    assert np.array_equal(out_a.view(np.uint64), out_b.view(np.uint64))  # bit patterns, -0.0 included
    assert ei_a == ei_b


def _counters(r):
    return {k: r[k] for k in ("fec", "bec", "frames", "iters")}


def _same_counters(a, b):
    assert a == b and a[0]["frames"] > 0


@pytest.mark.parametrize("n", FRAMES)
@pytest.mark.parametrize("iters", ITERS)
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_decode_batch_h(ctx, oracle_code, shape, iters, n):
    llr = _llrs(np.random.default_rng(1000 * iters + n), oracle_code, n)
    dec = lambda: ctx.decode_batch(llr, "BP_MS", iters, False)
    got = _run(ctx, dict(precision=0, **SHAPES[shape]), dec)
    _same_decode(got, _run(ctx, dict(precision=0, **CONTROL), dec))
    assert got[1] == n * iters * len(ctx.edges()[0]) and np.all(got[0][2] == iters)
    if n <= 3:
        ro, rc, ri = oracle_code.decode(llr, iters, False, True)
        assert np.array_equal(got[0][0].view(np.uint64), ro.view(np.uint64)) and np.array_equal(got[0][1], rc) and np.array_equal(got[0][2], ri)


@pytest.mark.parametrize("n", [1, 3, 301, 5003])
@pytest.mark.parametrize("iters", ITERS)
@pytest.mark.parametrize("idx16", [2, 1])
def test_decode_batch_irregular(irregular, idx16, iters, n):
    """degree-0/1 variables, checks of degree 2..15 (the generic body above 8), punctured and shortened positions"""
    c, oc = irregular
    llr = _llrs(np.random.default_rng(7 * iters + n), oc, n)
    dec = lambda: c.decode_batch(llr, "BP_MS", iters, False)
    got = _run(c, dict(precision=0, residency=SMEM, tmem=0, idx16=idx16, **AUTO), dec)
    _same_decode(got, _run(c, dict(precision=0, **CONTROL), dec))
    if n <= 3:
        ro, rc, ri = oc.decode(llr, iters, False, True)
        assert np.array_equal(got[0][0].view(np.uint64), ro.view(np.uint64)) and np.array_equal(got[0][1], rc) and np.array_equal(got[0][2], ri)


@pytest.mark.parametrize("iters", ITERS)
def test_sweep_irregular(irregular, iters):
    c, oc = irregular
    sweep = lambda: _counters(c.sim_point("BSC", 0.04, seed=3, point=1, frame0=77, nframes=1001, decoding="BP_MS", iterations=iters, early_term=False))
    got = _run(c, dict(precision=0, residency=SMEM, tmem=0, idx16=2, **AUTO), sweep)
    _same_counters(got, _run(c, dict(precision=0, **CONTROL), sweep))
    o = oc.sim_point("BSC", 0.04, seed=3, point=1, frame0=77, nframes=1001, decoding="BP_MS", iterations=iters, early_term=False, threads=8)
    assert got[0] == o


SWEEPS = [("AWGN", -4.5, 0), ("BSC", 0.075, 0), ("RAYLEIGH", -1.5, 0), ("AWGN", -4.5, 1)]  # (channel, x, 1: codewords through G)


@pytest.mark.parametrize("n", [3, 2 * 296 + 1, 7 * 4 * 148 + 5])
@pytest.mark.parametrize("iters", [1, 2, 50])
@pytest.mark.parametrize("channel,x,gen", SWEEPS)
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_sweep_h(ctx, shape, channel, x, gen, iters, n):
    """the fused count + refill pass (all-zero codeword) and the staged route (-G)"""
    sweep = lambda: _counters(ctx.sim_point(channel, x, seed=9, point=2, frame0=1 << 33, nframes=n, decoding="BP_MS", iterations=iters,
                                            early_term=False))
    zc = dict(precision=0, zero_codeword=1 - gen)
    got = _run(ctx, dict(zc, **SHAPES[shape]), sweep)
    _same_counters(got, _run(ctx, dict(zc, **CONTROL), sweep))
    assert got[0]["iters"] == n * iters


@pytest.mark.parametrize("iters", [1, 50])
def test_sweep_f32_and_4ask(ctx, iters):
    n = 7 * 8 * 148 + 3
    sweep = lambda: _counters(ctx.sim_point("AWGN", -3.0, seed=4, point=0, frame0=0, nframes=n, decoding="BP_MS", iterations=iters,
                                            early_term=False))
    for prec in (1, 0):
        ctx.set_modulation(2)
        t = dict(precision=prec, zero_codeword=1)
        _same_counters(_run(ctx, dict(t, residency=SMEM, tmem=0, idx16=0, **AUTO), sweep), _run(ctx, dict(t, **CONTROL), sweep))
    ctx.set_modulation(4)
    for shape in sorted(SHAPES):
        t = dict(precision=0, zero_codeword=1)
        _same_counters(_run(ctx, dict(t, **SHAPES[shape]), sweep), _run(ctx, dict(t, **CONTROL), sweep))


@pytest.mark.parametrize("iters", [1, 3, 50])
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_decode_batch_ex_narrow_inputs(ctx, oracle_code, shape, iters):
    n = 2 * 296 + 1
    rng = np.random.default_rng(iters)
    llr = _llrs(rng, oracle_code, n)
    for inp, scale in ((llr.astype(np.float32), 1.0), (np.clip(np.rint(llr * 8), -127, 127).astype(np.int8), 0.125)):
        dec = lambda: ctx.decode_batch_ex(inp, "BP_MS", iters, False, scale=scale, want_llr=True, want_hard=True, want_bits=True)
        (out, hard, bits, its), ei = _run(ctx, dict(precision=0, **SHAPES[shape]), dec)
        (out_c, hard_c, bits_c, its_c), ei_c = _run(ctx, dict(precision=0, **CONTROL), dec)
        assert np.array_equal(out.view(np.uint64), out_c.view(np.uint64)) and np.array_equal(hard, hard_c)
        assert np.array_equal(bits, bits_c) and np.array_equal(its, its_c) and ei == ei_c


@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_error_log_and_replay(ctx, shape):
    kw = dict(seed=12, point=3, frame0=5000, nframes=7 * 4 * 148 + 5, decoding="BP_MS", iterations=20, early_term=False)
    log = lambda: ctx.sim_point_log("AWGN", -4.6, capacity=1 << 14, **kw)
    t = dict(precision=0, zero_codeword=1)
    got = _run(ctx, dict(t, **SHAPES[shape]), log)
    ctl = _run(ctx, dict(t, **CONTROL), log)
    (cnt, rec, n_err), _ = got
    assert got == ctl and n_err == cnt["fec"] > 0 and len(rec) == n_err
    frames = [r[0] for r in rec[:64]]
    rep = lambda: ctx.error_reports("AWGN", -4.6, 12, 3, frames, "BP_MS", 20, False)
    reps = _run(ctx, dict(t, **SHAPES[shape]), rep)
    assert reps == _run(ctx, dict(t, **CONTROL), rep)
    assert [r["hamming_distance"] for r in reps[0]] == [r[1] for r in rec[:64]]
