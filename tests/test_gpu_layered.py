"""The floating-point layered decoders (lay_kernel<double | float, ALG_MS | ALG_BP, *>) on the GPU against their specifications:
orc_decode_layered (fp64) and orc_decode_layered_f32 (binary32 min-sum, tests/layered_f32_oracle.c).  Min-sum is compared bit for
bit (posteriors as uint64, decisions, iteration counts), fp64 sum-product within BP_RTOL with identical iteration counts.

Results must not depend on where a frame is decoded: on which CTA, after which batch, beside which neighbours, on the grid, the
shard split or the pipeline chunking.  Several tests therefore run every batch on one CTA (ctas = 1), so that each batch starts
from the state the previous one left behind.  Layered jobs also run no kernel-shape trial: nothing may be written to the tune
cache under the flooding kernel's key."""
import ctypes as ct
import os
import subprocess

import numpy as np
import pytest

import layered_f32_oracle as LF
from conftest import G_FILE, H_FILE, H_IRREGULAR, ROOT
from test_gpu_parity import BP_RTOL, _rel_err

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "libldpc_b200", "ldpcsim")
FPC = {"f64": (4, 8), "f32": (8, 16)}        # frames per CTA: 2 or 4 lanes x the 16-byte vector (2 doubles, 4 floats)
X = {"BP_MS": -4.4, "BP": -5.2}               # AWGN points with frames that converge and frames that fail (h.txt, 25 iterations)
TUNING = ("schedule", "precision", "frames_per_cta", "threads_per_cta", "ctas", "zero_codeword", "layered_ms_scale64")


def _prec(p):
    from libldpc_b200 import api
    return {"f64": api.F64, "f32": api.F32}[p]


def _tuning(c):
    from libldpc_b200 import api
    t = api.tuning()
    c._check(c.lib.ldpc_b200_get_tuning(c._h, ct.byref(t)))
    return {k: getattr(t, k) for k in TUNING}


@pytest.fixture
def lay(gpu_ctx):
    """The session context (h.txt) on the layered schedule with the all-zero codeword; its tuning and fading are put back."""
    from libldpc_b200 import api
    saved = _tuning(gpu_ctx)
    gpu_ctx.set_tuning(schedule=api.LAYERED, zero_codeword=1)
    try:
        yield gpu_ctx
    finally:
        gpu_ctx.set_fading(1)
        gpu_ctx.set_tuning(**saved)


@pytest.fixture(scope="module")
def irregular(built_lib):
    from libldpc_b200 import api
    from oracle import oracle as O
    c = api.Context(H_IRREGULAR, "", device=0)
    c.set_tuning(schedule=api.LAYERED)
    yield c, O.Code(H_IRREGULAR)
    c.close()


@pytest.fixture(scope="module")
def bg1(built_lib):
    from conftest import large_code_files
    from libldpc_b200 import api
    from oracle import oracle as O
    path = large_code_files()["bg1"]
    c = api.Context(path, "", device=0)
    c.set_tuning(schedule=api.LAYERED)
    yield c, O.Code(path)
    c.close()


def _spec(code, llr, layers, iters, et, prec, alg, ms_scale=1.0):
    return LF.decode(code, llr, layers, iters, et, f32=prec == "f32", minsum=alg == "BP_MS", ms_scale=ms_scale)


def _same(got, want, alg, what):
    out, hard, its = got
    ro, rc, ri = want
    assert np.array_equal(its, ri), (what, np.nonzero(its != ri)[0][:8], its[its != ri][:8], ri[its != ri][:8])
    if alg == "BP_MS":
        assert np.array_equal(hard, rc) and np.array_equal(out.view(np.uint64), ro.view(np.uint64)), what
    else:
        assert (hard == rc).mean() >= 0.9999 and _rel_err(out, ro).max() < BP_RTOL, what


def _identical(a, b, what):
    assert all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(a, b)), what


def _clean_frames(c, oc, layers, n):
    """n channel frames at 8 dB that every specification (fp64 min-sum and sum-product, binary32 min-sum) stops after the first
    iteration.  Most frames at this point need two: h.txt's 128 punctured positions start at 0."""
    _, llr = c.channel("AWGN", 8.0, seed=41, point=0, frame0=0, n=16 * n)
    keep = np.ones(len(llr), bool)
    for prec, alg in (("f64", "BP_MS"), ("f64", "BP"), ("f32", "BP_MS")):
        keep &= _spec(oc, llr, layers, 3, True, prec, alg)[2] == 0
    assert keep.sum() >= n
    return llr[keep][:n]


# ---- a. a batch that ends at an odd limit with lanes still decoding must not leak its syndrome flags into the next batch ----
@pytest.mark.parametrize("iters", [1, 2, 3, 4, 5, 25])
@pytest.mark.parametrize("prec, fpc", [("f64", 4), ("f64", 8), ("f32", 8), ("f32", 16)])
@pytest.mark.parametrize("alg", ["BP_MS", "BP"])
def test_syndrome_flags_do_not_leak_into_the_next_batch(lay, oracle_code, prec, fpc, alg, iters):
    """One CTA decodes every batch in turn: F frames that fail, then F frames that stop after their first iteration, four
    times.  At an odd limit the failing batch ends with its flags in slot 0, the slot the next batch tests at iteration 0; the
    even limits are controls (their last flags are in slot 1, which iteration 0 clears before iteration 1 uses it)."""
    layers = lay.layers()
    _, hard = lay.channel("AWGN", -9.0, seed=40, point=0, frame0=0, n=4 * fpc)
    clean = _clean_frames(lay, oracle_code, layers, 4 * fpc)
    llr = np.concatenate([np.concatenate([hard[k * fpc:(k + 1) * fpc], clean[k * fpc:(k + 1) * fpc]]) for k in range(4)])
    is_clean = np.tile(np.repeat([False, True], fpc), 4)
    lay.set_tuning(precision=_prec(prec), frames_per_cta=fpc, ctas=1)
    got = lay.decode_batch(llr, alg, iters, True)
    assert lay.stats()["ctas"] == 1 and lay.stats()["frames_per_cta"] == fpc
    want_its = np.where(is_clean, 0, iters)
    if prec == "f32" and alg == "BP":                 # no exact specification: the iteration counts are the whole claim
        assert np.array_equal(got[2], want_its), got[2]
        return
    want = _spec(oracle_code, llr, layers, iters, True, prec, alg)
    assert np.array_equal(want[2], want_its)          # every hard frame reaches the limit, every clean one stops at iteration 0
    _same(got, want, alg, iters)


# ---- b. batch decode against the specification across grid shapes ----
@pytest.mark.parametrize("prec, alg", [("f64", "BP_MS"), ("f64", "BP"), ("f32", "BP_MS")])
def test_batch_decode_equals_specification_across_shapes(lay, oracle_code, prec, alg):
    layers = lay.layers()
    n = 5 * max(FPC[prec]) + 3
    _, llr = lay.channel("AWGN", X[alg], seed=31, point=0, frame0=0, n=n)
    llr[3::7] = _clean_frames(lay, oracle_code, layers, len(llr[3::7]))   # frames that stop at iteration 0 among failing ones
    llr[2, ::9] = -0.0
    llr[5, oracle_code.bit_pos[::4]] = -0.0
    lay.set_tuning(precision=_prec(prec))
    for iters in (1, 5, 25):
        for et in (True, False):
            want = _spec(oracle_code, llr, layers, iters, et, prec, alg)
            if iters == 25 and et:
                assert (want[2] == 0).any() and (want[2] == 25).any() and ((want[2] > 0) & (want[2] < 25)).any()
            for fpc in FPC[prec]:
                for ctas in (1, 7, 0):
                    lay.set_tuning(frames_per_cta=fpc, ctas=ctas)
                    for threads in (64, 256, 512):
                        lay.set_tuning(threads_per_cta=threads)
                        m = 5 * fpc + 3
                        _same(lay.decode_batch(llr[:m], alg, iters, et), tuple(w[:m] for w in want), alg, (iters, et, fpc, ctas, threads))
                    lay.set_tuning(threads_per_cta=0)
                    for m in (1, fpc - 1, fpc + 1):                         # ragged batches
                        _same(lay.decode_batch(llr[:m], alg, iters, et), tuple(w[:m] for w in want), alg, (iters, et, fpc, ctas, m))


@pytest.mark.parametrize("prec, alg", [("f64", "BP_MS"), ("f64", "BP"), ("f32", "BP_MS")])
def test_irregular_code_equals_specification(irregular, prec, alg):
    """Check degrees 2-15, layers of 1-25 checks, punctured and shortened positions."""
    c, oc = irregular
    layers = c.layers()
    assert oc.layers_valid(layers)
    _, llr = c.channel("AWGN", 0.5, seed=8, point=0, frame0=0, n=5 * max(FPC[prec]) + 3)
    llr[1, ::5] = -0.0
    try:
        c.set_tuning(precision=_prec(prec))
        for iters, et in ((5, True), (25, True), (5, False)):
            want = _spec(oc, llr, layers, iters, et, prec, alg)
            if iters == 25:
                assert (want[2] < 25).any() and (want[2] == 25).any()
            for fpc in FPC[prec]:
                for ctas, threads in ((1, 64), (1, 512), (0, 256)):
                    c.set_tuning(frames_per_cta=fpc, ctas=ctas, threads_per_cta=threads)
                    _same(c.decode_batch(llr, alg, iters, et), want, alg, (iters, et, fpc, ctas, threads))
    finally:
        c.set_tuning(precision=_prec("f64"), frames_per_cta=0, ctas=0, threads_per_cta=0)


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_bg1_shaped_code_on_one_cta(bg1, prec):
    c, oc = bg1
    layers = c.layers()
    _, llr = oc.channel_frames("AWGN", -0.6, 9, 0, 0, 40)
    try:
        c.set_tuning(precision=_prec(prec), ctas=1)
        for q in (0, 48):
            c.set_tuning(layered_ms_scale64=q)
            for iters, et in ((25, True), (5, False)):
                want = _spec(oc, llr, layers, iters, et, prec, "BP_MS", ms_scale=(q or 64) / 64.0)
                _same(c.decode_batch(llr, "BP_MS", iters, et), want, "BP_MS", (q, iters, et))
    finally:
        c.set_tuning(precision=_prec("f64"), ctas=0, layered_ms_scale64=0)


# ---- c. a frame's result does not depend on its neighbours or its CTA, in all four floating-point instantiations ----
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("alg", ["BP_MS", "BP"])
def test_result_does_not_depend_on_position(lay, oracle_code, prec, alg):
    layers = lay.layers()
    _, llr = lay.channel("AWGN", X[alg], seed=17, point=0, frame0=0, n=64)
    llr[::5] = _clean_frames(lay, oracle_code, layers, len(llr[::5]))
    lay.set_tuning(precision=_prec(prec))
    iters = 25
    alone = [lay.decode_batch(llr[i:i + 1], alg, iters, True) for i in range(len(llr))]
    alone = tuple(np.concatenate([a[k] for a in alone]) for k in range(3))
    perm = np.random.default_rng(5).permutation(len(llr))
    lay.set_tuning(ctas=1)
    shuffled = lay.decode_batch(llr[perm], alg, iters, True)
    inv = np.argsort(perm)
    shuffled = tuple(a[inv] for a in shuffled)
    lay.set_tuning(ctas=0)
    grid = lay.decode_batch(llr, alg, iters, True)
    _identical(alone, shuffled, "alone / shuffled on one CTA")
    _identical(alone, grid, "alone / default grid")
    assert (alone[2] == 0).any() and (alone[2] == iters).any()
    if not (prec == "f32" and alg == "BP"):
        _same(grid, _spec(oracle_code, llr, layers, iters, True, prec, alg), alg, "specification")


def test_f32_sum_product_is_statistically_consistent(lay):
    """Binary32 sum-product has no exact specification: on the same 20000 frames its FER is fp64's within binomial tolerance."""
    n = 20000
    kw = dict(seed=11, point=0, frame0=0, nframes=n, decoding="BP", iterations=25, early_term=True)
    a = lay.sim_point("AWGN", X["BP"], **kw)
    lay.set_tuning(precision=_prec("f32"))
    b = lay.sim_point("AWGN", X["BP"], **kw)
    p = a["fec"] / n
    assert 0.01 < p < 0.9, a
    assert abs(a["fec"] - b["fec"]) <= 4 * np.sqrt(2 * p * (1 - p) * n) + 5, (a, b)
    assert abs(a["iters"] - b["iters"]) <= 0.02 * a["iters"], (a, b)


# ---- d. sweeps: the layered kernel's own frame generator and accounting against the specification's frame loop ----
# (channel, x, coherence, iterations).  On h.txt no AWGN, BSC or fast-fading point has frames that stop at iteration 0 beside
# frames that reach the limit (at 1 dB still no frame stops at 0, the 128 punctured positions start at 0); those cases pin the
# generators and the counters.  Quasi-static fading (one coefficient per frame) mixes both at one point.
SWEEPS = [("AWGN", -4.4, 1, 25), ("AWGN", -2.0, 1, 5), ("BSC", 0.16, 1, 5), ("RAYLEIGH", -3.5, 1, 25), ("RAYLEIGH", 7.0, 0, 5),
          ("RAYLEIGH", 7.0, 0, 25)]


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("channel, x, L, iters", SWEEPS)
def test_sweep_equals_specification_frame_loop(lay, oracle_code, prec, channel, x, L, iters):
    n, seed, point, frame0 = 3000, 21, 2, 7
    lay.set_fading(L)
    lay.set_tuning(precision=_prec(prec))
    cw, llr = lay.channel(channel, x, seed=seed, point=point, frame0=frame0, n=n)
    assert not cw.any()
    _, co, ri = _spec(oracle_code, llr, lay.layers(), iters, True, prec, "BP_MS")
    errs = co[:, oracle_code.bit_pos].sum(1).astype(np.int64)
    want = dict(fec=int((errs > 0).sum()), bec=int(errs.sum()), frames=n, iters=int(ri.sum()))
    assert (ri == iters).mean() >= 0.05, (ri == iters).mean()
    if L == 0:
        assert (ri == 0).mean() >= 0.2, (ri == 0).mean()
    kw = dict(seed=seed, point=point, decoding="BP_MS", iterations=iters, early_term=True)
    key = ("fec", "bec", "frames", "iters")
    for ctas in (1, 7, 0):
        for threads in (128, 512):
            lay.set_tuning(ctas=ctas, threads_per_cta=threads)
            got = lay.sim_point(channel, x, frame0=frame0, nframes=n, **kw)
            assert {k: got[k] for k in key} == want, (ctas, threads, got)
    lay.set_tuning(ctas=0, threads_per_cta=0)
    for cut in (1, 1000, 2999):
        a = lay.sim_point(channel, x, frame0=frame0, nframes=cut, **kw)
        b = lay.sim_point(channel, x, frame0=frame0 + cut, nframes=n - cut, **kw)
        assert {k: a[k] + b[k] for k in key} == want, cut
    cnt, log, n_err = lay.sim_point_log(channel, x, frame0=frame0, nframes=n, capacity=n, **kw)
    bad = np.nonzero(errs)[0]
    assert cnt == want and n_err == len(bad)
    assert log == [(frame0 + int(t), int(errs[t]), int(ri[t])) for t in bad]


# ---- e. the CLI: one shard or three on the same device give the same results file ----
def _rows(out):
    lines = out.read_text().split("\n")
    assert lines[0] == "snr fer ber frames avg_iter frame_time"
    return [l.split()[:5] for l in lines[1:] if l]


def _cli(out, *args, env=None):
    r = subprocess.run([CLI, H_FILE, str(out), *args], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    return _rows(out)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("dec, iters", [("BP_MS", 5), ("BP", 3)])
def test_cli_shards_give_identical_results(built_lib, tmp_path, prec, dec, iters):
    args = ["-5.0", "-3.5", "0.5", "--schedule", "layered", "--precision", prec, "--decoding", dec, "-i", str(iters), "-s", "4",
            "--frame-error-count", "300", "--max-frames", "200000"]
    one = _cli(tmp_path / "one.txt", *args, "--devices", "0")
    three = _cli(tmp_path / "three.txt", *args, "--devices", "0,0,0")
    assert len(one) >= 3 and one == three, (one, three)


# ---- f. layered jobs run no kernel-shape trial and write nothing to the tune cache ----
def test_layered_jobs_leave_the_tune_cache_alone(built_lib, tmp_path):
    from libldpc_b200 import api
    d = tmp_path / "tune"
    d.mkdir()
    saved = {k: os.environ.get(k) for k in ("LDPC_B200_TUNE_CACHE", "LDPC_B200_PAIR")}
    os.environ["LDPC_B200_TUNE_CACHE"] = str(d)
    os.environ.pop("LDPC_B200_PAIR", None)          # it presets the trial's outcome, and the control below needs the trial
    c = api.Context(H_FILE, G_FILE, device=0)
    try:
        c.set_tuning(schedule=api.LAYERED, zero_codeword=1)
        n = 25000
        _, llr = c.channel("AWGN", -4.0, seed=1, point=0, frame0=0, n=n)
        c.decode_batch(llr, "BP_MS", 10, True, want_llr=False)
        c.sim_point("AWGN", -4.0, seed=1, nframes=n, decoding="BP_MS", iterations=10)
        assert list(d.iterdir()) == []
        _cli(tmp_path / "res.txt", "-4.5", "-4.0", "0.5", "--schedule", "layered", "--decoding", "BP_MS", "-i", "10",
             "--frame-error-count", "50", "--max-frames", "60000", env=dict(os.environ))
        assert list(d.iterdir()) == []
        c.set_tuning(schedule=api.FLOODING, zero_codeword=0)               # control: the same job on flooding runs the trial
        c.decode_batch(llr, "BP_MS", 10, True, want_llr=False)
        assert len(list(d.iterdir())) == 1
    finally:
        c.close()
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
