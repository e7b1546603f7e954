"""The fixed-point layered min-sum decoder on the GPU against its specification (tests/quant_oracle.c, DESIGN.md §3.7): batch
decode bit for bit, the fused sweep's counters against the oracle frame loop on AWGN / BSC / RAYLEIGH, the replay of logged
frames, switching it off, the rejected combinations, the FER against fp64 and the CLI."""
import os
import subprocess

import numpy as np
import pytest

import quant_oracle as Q
from conftest import H_FILE, ROOT

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "libldpc_b200", "ldpcsim")
THREADS = os.cpu_count() or 1
PARAMS = [(6, 6, 8, 0.5, 0, 8), (5, 5, 7, 0.25, 1, 8), (4, 4, 6, 0.5, 0, 6), (8, 8, 16, 0.25, 0, 8)]


@pytest.fixture(scope="module", autouse=True)
def tune_cache(tmp_path_factory):
    """Shape-trial outcomes go to a directory of this module's own; quantised runs must leave it empty."""
    d = tmp_path_factory.mktemp("tune_cache")
    old = os.environ.get("LDPC_B200_TUNE_CACHE")
    os.environ["LDPC_B200_TUNE_CACHE"] = str(d)
    yield d
    if old is None:
        del os.environ["LDPC_B200_TUNE_CACHE"]
    else:
        os.environ["LDPC_B200_TUNE_CACHE"] = old


@pytest.fixture
def ctx(gpu_ctx):
    """h.txt on the layered schedule with the all-zero codeword; restores the defaults afterwards."""
    from libldpc_b200 import api
    gpu_ctx.set_tuning(schedule=api.LAYERED, zero_codeword=1)
    yield gpu_ctx
    gpu_ctx.set_quant(None)
    gpu_ctx.set_fading(1)
    gpu_ctx.set_modulation(2)
    gpu_ctx.set_tuning(precision=api.F64, residency=api.AUTO, schedule=api.FLOODING, zero_codeword=0, frames_per_cta=0, ctas=0)


@pytest.fixture(scope="module")
def bg1_ctx(built_lib):
    from conftest import large_code_files
    from libldpc_b200 import api
    from oracle import oracle as O
    path = large_code_files()["bg1"]
    c = api.Context(path, "", device=0)
    c.set_tuning(schedule=api.LAYERED)
    yield c, O.Code(path)
    c.close()


def _set(c, p):
    ch, msg, post, step, beta, a = p
    c.set_quant(ch, msg, post, step, offset=beta, scale8=a)
    return Q.quant(ch, msg, post, step, beta, a)


@pytest.mark.parametrize("p", PARAMS)
@pytest.mark.parametrize("et", [True, False])
def test_batch_decode_equals_specification_h(ctx, oracle_code, p, et):
    from libldpc_b200 import api
    q = _set(ctx, p)
    assert ctx.quant() == dict(ch_bits=p[0], msg_bits=p[1], post_bits=p[2], offset=p[4], scale8=p[5], step=p[3])
    cw, llr = ctx.channel("AWGN", -4.4, seed=31, point=0, frame0=0, n=101)
    llr[3, ::9] = -0.0
    layers = ctx.layers()
    for iters in (1, 5, 20):
        ro, rc, ri, _, _ = Q.decode(oracle_code, llr, layers, q, iters, et)
        if iters == 20 and et and p != PARAMS[2]:             # (4, 4, 6) with a = 6 fails every frame at this point
            assert (ri < iters).any() and (ri == iters).any()        # frames that converge and frames that fail
        for fpc in (16, 32):
            ctx.set_tuning(frames_per_cta=fpc, ctas=2)                 # several batches per CTA
            out, hard, its = ctx.decode_batch(llr, "BP_MS", iters, et)
            assert np.array_equal(its, ri) and np.array_equal(hard, rc), (iters, fpc)
            assert np.array_equal(out.view(np.uint64), ro.view(np.uint64)), (iters, fpc)
            st = ctx.stats()
            assert st["precision"] == api.FIXED and st["frames_per_cta"] == fpc and st["ctas"] == 2


@pytest.mark.parametrize("p", PARAMS)
def test_batch_decode_equals_specification_bg1(bg1_ctx, p):
    c, oc = bg1_ctx
    q = _set(c, p)
    layers = c.layers()
    _, llr = oc.channel_frames("AWGN", -0.6, 9, 0, 0, 40)
    try:
        for et in (True, False):
            for iters in (1, 5, 20):
                ro, rc, ri, _, _ = Q.decode(oc, llr, layers, q, iters, et)
                for fpc in (16, 32):
                    c.set_tuning(frames_per_cta=fpc, ctas=1)
                    out, hard, its = c.decode_batch(llr, "BP_MS", iters, et)
                    assert np.array_equal(its, ri) and np.array_equal(hard, rc), (et, iters, fpc)
                    assert np.array_equal(out.view(np.uint64), ro.view(np.uint64)), (et, iters, fpc)
    finally:
        c.set_quant(None)
        c.set_tuning(frames_per_cta=0, ctas=0)


# (channel, x, coherence, early termination, iterations): points where 0.05 < FER < 0.9 for (6, 6, 8, step 0.5)
SWEEP_CASES = [("AWGN", -4.4, 1, True, 20), ("AWGN", -4.4, 1, False, 10), ("BSC", 0.25, 1, True, 20),
               ("RAYLEIGH", -3.5, 1, True, 20), ("RAYLEIGH", 1.0, 0, True, 20)]


@pytest.mark.parametrize("channel, x, L, et, iters", SWEEP_CASES)
def test_sweep_counters_equal_oracle_frame_loop(ctx, oracle_code, channel, x, L, et, iters):
    q = _set(ctx, PARAMS[0])
    ctx.set_fading(L)
    n, seed, point, frame0 = 1500, 21, 2, 7
    got = ctx.sim_point(channel, x, seed=seed, point=point, frame0=frame0, nframes=n, decoding="BP_MS", iterations=iters, early_term=et)
    want = Q.sim_point(oracle_code, ctx.layers(), channel, x, q, coherence=L, seed=seed, point=point, frame0=frame0, nframes=n,
                       iterations=iters, early_term=et, threads=THREADS)
    assert 0.05 < want["fec"] / n < 0.9, want
    assert {k: got[k] for k in want} == want


def test_replay_of_logged_frames(ctx):
    _set(ctx, PARAMS[1])
    cnt, log, n_err = ctx.sim_point_log("AWGN", -4.4, seed=3, point=4, frame0=0, nframes=2000, decoding="BP_MS", iterations=15,
                                        early_term=True, capacity=4096)
    assert n_err == cnt["fec"] == len(log) > 0
    reps = ctx.error_reports("AWGN", -4.4, 3, 4, [f for f, _, _ in log], decoding="BP_MS", iterations=15, early_term=True)
    assert [(r["frame"], r["hamming_distance"], r["iterations"]) for r in reps] == log


def test_large_job_runs_no_shape_trial(ctx, tune_cache):
    _set(ctx, PARAMS[0])
    ctx.sim_point("AWGN", -3.0, seed=1, nframes=40000, decoding="BP_MS", iterations=10)
    _, llr = ctx.channel("AWGN", -3.0, 1, 0, 0, 25000)
    ctx.decode_batch(llr, "BP_MS", 10, True, want_llr=False)
    assert list(tune_cache.iterdir()) == []


def test_switching_off_restores_the_float_decoder(ctx, built_lib):
    from conftest import G_FILE
    from libldpc_b200 import api
    _, llr = ctx.channel("AWGN", -4.4, seed=5, point=0, frame0=0, n=200)
    _set(ctx, PARAMS[0])
    ctx.decode_batch(llr, "BP_MS", 20, True)
    ctx.sim_point("AWGN", -4.4, nframes=500, decoding="BP_MS", iterations=20)
    ctx.set_quant(None)
    assert ctx.quant() is None
    fresh = api.Context(H_FILE, G_FILE, device=0)
    fresh.set_tuning(schedule=api.LAYERED, zero_codeword=1)
    try:
        for c in (ctx, fresh):
            c.set_tuning(frames_per_cta=0)
        a = ctx.decode_batch(llr, "BP_MS", 20, True)
        b = fresh.decode_batch(llr, "BP_MS", 20, True)
        assert all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(a, b))
        assert ctx.stats()["precision"] == api.F64
        kw = dict(seed=2, point=1, frame0=0, nframes=3000, decoding="BP_MS", iterations=20)
        assert ctx.sim_point("AWGN", -4.4, **kw)["fec"] == fresh.sim_point("AWGN", -4.4, **kw)["fec"]
    finally:
        fresh.close()


def test_rejections(ctx):
    from libldpc_b200 import api
    _, llr = ctx.channel("AWGN", -4.0, 0, 0, 0, 8)
    with pytest.raises(RuntimeError, match="bit widths"):
        ctx.set_quant(6, 8, 7, 0.5)
    with pytest.raises(RuntimeError, match="offset"):
        ctx.set_quant(6, 3, 8, 0.5, offset=3)
    with pytest.raises(RuntimeError, match="scale8"):
        ctx.set_quant(6, 6, 8, 0.5, scale8=9)
    with pytest.raises(RuntimeError, match="step"):
        ctx.set_quant(6, 6, 8, 0.0)
    assert ctx.quant() is None                                             # a failed call keeps the previous setting
    _set(ctx, PARAMS[0])
    with pytest.raises(RuntimeError, match="bit widths"):
        ctx.set_quant(17, 16, 16, 0.5)
    assert ctx.quant()["ch_bits"] == 6
    with pytest.raises(RuntimeError, match="min-sum only"):
        ctx.decode_batch(llr, "BP", 5, True)
    with pytest.raises(RuntimeError, match="min-sum only"):
        ctx.sim_point("AWGN", -4.0, nframes=10, decoding="BP")
    with pytest.raises(RuntimeError, match="does not apply to the BEC"):
        ctx.sim_point("BEC", 0.3, nframes=10, decoding="BP_MS")
    cw, u8 = ctx.channel("BEC", 0.3, 0, 0, 0, 4)
    with pytest.raises(RuntimeError, match="does not apply to the BEC"):
        ctx.decode_bec_batch(u8, cw, 5, True)
    with pytest.raises(RuntimeError, match="narrow encodings"):
        ctx.decode_batch_ex(llr.astype(np.float32), "BP_MS", 5, True)
    with pytest.raises(RuntimeError, match="narrow encodings"):
        ctx.decode_batch_ex(llr, "BP_MS", 5, True, want_bits=True)
    for fpc in (4, 8, 64):
        ctx.set_tuning(frames_per_cta=fpc)
        with pytest.raises(RuntimeError, match="frames_per_cta must be 0, 16 or 32"):
            ctx.decode_batch(llr, "BP_MS", 5, True)
        with pytest.raises(RuntimeError, match="frames_per_cta must be 0, 16 or 32"):
            ctx.sim_point("AWGN", -4.0, nframes=10, decoding="BP_MS")
    ctx.set_tuning(frames_per_cta=0)
    ctx.set_modulation(4)
    with pytest.raises(RuntimeError, match="BPSK only"):
        ctx.sim_point("AWGN", 2.0, nframes=10, decoding="BP_MS")
    ctx.set_modulation(2)
    ctx.set_tuning(schedule=api.FLOODING)
    with pytest.raises(RuntimeError, match="layered schedule only"):
        ctx.decode_batch(llr, "BP_MS", 5, True)
    with pytest.raises(RuntimeError, match="layered schedule only"):
        ctx.sim_point("AWGN", -4.0, nframes=10, decoding="BP_MS")
    ctx.set_tuning(schedule=api.LAYERED)
    ctx.decode_batch(llr, "BP_MS", 5, True)                               # the valid combination still works


def test_fer_orders_by_message_width(ctx):
    n = 20000
    kw = dict(seed=9, point=0, frame0=0, nframes=n, decoding="BP_MS", iterations=20, early_term=True)
    x = -4.0
    fp64 = ctx.sim_point("AWGN", x, **kw)["fec"] / n
    ctx.set_quant(8, 8, 10, 0.125)
    q8 = ctx.sim_point("AWGN", x, **kw)["fec"] / n
    ctx.set_quant(3, 3, 6, 1.0)
    q3 = ctx.sim_point("AWGN", x, **kw)["fec"] / n
    sd = np.sqrt(2 * fp64 * (1 - fp64) / n)
    assert 0.02 < fp64 < 0.5 and abs(q8 - fp64) < 4 * sd, (fp64, q8, q3)
    assert q3 > q8, (q3, q8)


def _results(out):
    lines = out.read_text().split("\n")
    assert lines[0] == "snr fer ber frames avg_iter frame_time"
    return [l.split()[:5] for l in lines[1:] if l]


def _cli(out, *extra):
    r = subprocess.run([CLI, H_FILE, str(out), "-5", "-3.9", "0.5", "--schedule", "layered", "--decoding", "BP_MS", "-i", "20",
                        "--quantize", "6,6,8", "--llr-step", "0.5", "--ms-offset", "1", "--frame-error-count", "40", "--max-frames", "200000",
                        *extra], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Fixed point" in r.stdout
    return _results(out)


def test_cli_shards_and_error_log(built_lib, tmp_path):
    one = _cli(tmp_path / "one.txt")
    assert len(one) == 3 and float(one[0][1]) > 0
    assert _cli(tmp_path / "three.txt", "--devices", "0,0,0") == one
    log = tmp_path / "err.log"
    assert _cli(tmp_path / "logged.txt", "--error-log", str(log)) == one
    lines = log.read_text().split("\n")
    assert len(lines) > 2 and lines[0].startswith("snr frame iterations")
