"""Fixed-iteration min-sum decoding when the lock-step kernel cannot take a shape.  The lock-step kernel (tile4.cuh, TMEM
mirror, compiled without early termination) keeps every gather address of a thread in TMEM and reads its segment
descriptors from the kernel parameters.  When the addresses do not fit the mirror's TMEM allocation, or the descriptors do
not fit K4Params::ls_seg, the engine runs the early-termination mirror kernel with early termination off instead.  Each
case is compared bit for bit with the shared-memory kernel without the mirror, and the launch must name the kernel that
ran (LDPC_B200_DEBUG) and report the shape the caller pinned."""
import ctypes as ct

import numpy as np
import pytest

from conftest import H_FILE

pytestmark = pytest.mark.gpu

SMEM = 1
AUTO = dict(frames_per_cta=0, threads_per_cta=0, ctas=0)
CONTROL = dict(precision=0, residency=SMEM, tmem=1, idx16=0, **AUTO)


def _tuning(ctx):
    from libldpc_b200 import api
    t = api.tuning()
    ctx._check(ctx.lib.ldpc_b200_get_tuning(ctx._h, ct.byref(t)))
    return {k: getattr(t, k) for k, _ in api.tuning._fields_}


def _many_degrees_code(path, seed=5):
    """checks of degree 2, 3, 4, 5, 6 and variables of degree 0 to 7, most in whole warp tasks for every warp and a few single
    tasks: at one frame lane per node and 512 threads the 16 warps need 16 x (4 + 5) = 144 descriptors with the
    terminators, while the mirror and the gather addresses fit 412 of the 512 TMEM columns.  At 256 threads 96 descriptors
    and 378 columns.  The shared-memory tables fit with 32-bit entries (229 120 bytes)."""
    cdeg = sum(([d] * n for d, n in ((2, 512), (3, 512), (4, 768), (5, 32), (6, 32))), [])
    vdeg = sum(([d] * n for d, n in ((0, 32), (1, 512), (2, 512), (3, 512), (4, 584), (5, 32), (6, 32), (7, 32))), [])
    assert sum(vdeg) == sum(cdeg)
    rng = np.random.default_rng(seed)
    cs = np.repeat(np.arange(len(cdeg)), cdeg)
    vs = np.repeat(np.arange(len(vdeg)), vdeg)
    rng.shuffle(vs)
    while True:  # no check may list a variable twice
        _, first = np.unique(cs.astype(np.int64) * len(vdeg) + vs, return_index=True)
        dup = np.setdiff1d(np.arange(len(cs)), first)
        if len(dup) == 0:
            break
        for i in dup:
            j = rng.integers(len(vs))
            vs[i], vs[j] = vs[j], vs[i]
    with open(path, "w") as f:
        f.writelines("%d %d\n" % (c, v) for c, v in zip(cs, vs))


@pytest.fixture(scope="module")
def h_ctx(built_lib):
    from libldpc_b200 import api
    from oracle import oracle as O
    c = api.Context(H_FILE, "", device=0)
    yield c, O.Code(H_FILE)
    c.close()


@pytest.fixture(scope="module")
def many_ctx(built_lib, tmp_path_factory):
    from libldpc_b200 import api
    from oracle import oracle as O
    path = str(tmp_path_factory.mktemp("codes") / "many_degrees_h.txt")
    _many_degrees_code(path)
    c = api.Context(path, "", device=0)
    yield c, O.Code(path)
    c.close()


def _llrs(rng, oc, n):
    llr = rng.normal(1.0, 1.6, size=(n, oc.nc))
    llr[:, oc.puncture] = 0.0
    llr[:, oc.shorten] = 99999.9
    llr[0, ::7] = -0.0
    return llr


def _run(ctx, tuning, fn, capfd, monkeypatch):
    """fn() under `tuning`: its result, the stats of the launch and the tile kernels the launches name"""
    saved = _tuning(ctx)
    monkeypatch.setenv("LDPC_B200_DEBUG", "1")
    try:
        ctx.set_tuning(**tuning)
        ctx.stats(reset=True)
        capfd.readouterr()
        r = fn()
        err = capfd.readouterr().err
        st = ctx.stats()
    finally:
        monkeypatch.delenv("LDPC_B200_DEBUG")
        ctx.set_tuning(**saved)
    kernels = {ln.split("tile kernel: ", 1)[1].strip() for ln in err.splitlines() if ln.startswith("[launch] tile kernel: ")}
    return r, st, kernels


def _same(a, b):
    (out_a, hard_a, its_a), (out_b, hard_b, its_b) = a, b
    assert np.array_equal(its_a, its_b) and np.array_equal(hard_a, hard_b)
    assert np.array_equal(out_a.view(np.uint64), out_b.view(np.uint64))  # bit patterns, -0.0 included


# (context fixture, threads per CTA, kernel): h.txt at one frame lane per node and 192 threads needs 316 TMEM columns for
# the mirror and the gather addresses but allocates 256 for the mirror; 256 threads fit them (228).  The many-degree code
# exceeds the descriptor cap at 512 threads and fits at 256.
CASES = [("h_ctx", 192, "half-iteration, TMEM mirror"), ("h_ctx", 256, "lock-step"),
         ("many_ctx", 512, "half-iteration, TMEM mirror"), ("many_ctx", 256, "lock-step")]


@pytest.mark.parametrize("iters", [1, 3, 50])
@pytest.mark.parametrize("idx16", [1, 2])
@pytest.mark.parametrize("code,threads,kernel", CASES)
def test_fallback_decode_equals_mirrorless_kernel(request, capfd, monkeypatch, code, threads, kernel, idx16, iters):
    ctx, oc = request.getfixturevalue(code)
    n = 2 * 148 * 2 + 3  # two CTAs per SM's worth of frames and a ragged last batch
    llr = _llrs(np.random.default_rng(31 * iters + threads), oc, n)
    dec = lambda: ctx.decode_batch(llr, "BP_MS", iters, False)
    shape = dict(precision=0, residency=SMEM, tmem=0, idx16=idx16, frames_per_cta=2, threads_per_cta=threads, ctas=0)
    got, st, kernels = _run(ctx, shape, dec, capfd, monkeypatch)
    ctl, st_c, kernels_c = _run(ctx, CONTROL, dec, capfd, monkeypatch)
    assert kernels == {kernel} and kernels_c == {"half-iteration"}
    _same(got, ctl)
    assert np.all(got[2] == iters)
    assert st["frames_per_cta"] == 2 and st["threads_per_cta"] == threads and st["residency"] == SMEM
    assert st["frames"] == n and st["edge_iterations"] == n * iters * len(ctx.edges()[0]) == st_c["edge_iterations"]
    if iters <= 3:
        ro, rc, ri = oc.decode(llr[:3], iters, False, True)
        assert np.array_equal(got[0][:3].view(np.uint64), ro.view(np.uint64)) and np.array_equal(got[1][:3], rc) and np.array_equal(got[2][:3], ri)


@pytest.mark.parametrize("code,threads,kernel", CASES)
def test_fallback_sweep_equals_mirrorless_kernel(request, capfd, monkeypatch, code, threads, kernel):
    ctx, _ = request.getfixturevalue(code)
    sweep = lambda: {k: v for k, v in ctx.sim_point("AWGN", -1.0, seed=8, point=1, frame0=3, nframes=7 * 296 + 5, decoding="BP_MS",
                                                     iterations=20, early_term=False).items() if k in ("fec", "bec", "frames", "iters")}
    shape = dict(precision=0, residency=SMEM, tmem=0, idx16=1, frames_per_cta=2, threads_per_cta=threads, ctas=0, zero_codeword=1)
    got, _, kernels = _run(ctx, shape, sweep, capfd, monkeypatch)
    ctl, _, _ = _run(ctx, dict(CONTROL, zero_codeword=1), sweep, capfd, monkeypatch)
    assert kernels == {kernel} and got == ctl and got["frames"] == 7 * 296 + 5 and got["iters"] == 20 * got["frames"]
