"""The RAYLEIGH channel on the GPU: the channel kernel bit for bit against the specification (tests/rayleigh_oracle.c), the fused
sweep's counters against the oracle frame loop, the f32 / global-residency / layered paths against host accounting of the batch
decode, the batched replay of logged frames, the CLI, and the FER against AWGN and quasi-static fading."""
import os
import subprocess

import numpy as np
import pytest

import rayleigh_oracle as R
from conftest import H_FILE, ROOT

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "libldpc_b200", "ldpcsim")
THREADS = os.cpu_count() or 1


@pytest.fixture
def ctx(gpu_ctx):
    """h.txt with its generator matrix; restores the defaults afterwards."""
    from libldpc_b200 import api
    yield gpu_ctx
    gpu_ctx.set_fading(1)
    gpu_ctx.set_modulation(2)
    gpu_ctx.set_tuning(precision=api.F64, residency=api.AUTO, schedule=api.FLOODING, zero_codeword=0)


@pytest.mark.parametrize("L", [1, 7, 0])
@pytest.mark.parametrize("with_gen", [False, True])
def test_channel_equals_oracle(ctx, oracle_code, oracle_gen, L, with_gen):
    ctx.set_fading(L)
    ctx.set_tuning(zero_codeword=0 if with_gen else 1)
    x, seed, point, frame0, n = -1.5, 0xDEADBEEF12, 5, (1 << 32) + 3, 24
    cw, llr = ctx.channel("RAYLEIGH", x, seed, point, frame0, n)
    ocw, ollr = R.channel_frames(oracle_code, x, L, seed, point, frame0, n, gen=oracle_gen if with_gen else None)
    assert np.array_equal(cw, ocw)
    assert cw.any() == with_gen
    assert np.array_equal(llr.view(np.uint64), ollr.view(np.uint64))


# (L, x, early termination, iterations): points where 0.05 < FER < 0.9
COUNTER_CASES = [(1, -4.0, True, 30), (1, -4.0, False, 20), (0, 0.0, True, 30), (0, 0.0, False, 20)]


@pytest.mark.parametrize("L, x, et, iters", COUNTER_CASES)
@pytest.mark.parametrize("with_gen", [False, True])
def test_sweep_counters_equal_oracle_frame_loop(ctx, oracle_code, oracle_gen, L, x, et, iters, with_gen):
    ctx.set_fading(L)
    ctx.set_tuning(zero_codeword=0 if with_gen else 1)
    n, seed, point, frame0 = 1500, 21, 2, 7
    got = ctx.sim_point("RAYLEIGH", x, seed=seed, point=point, frame0=frame0, nframes=n, decoding="BP_MS", iterations=iters, early_term=et)
    want = R.sim_point(oracle_code, x, L, seed=seed, point=point, frame0=frame0, nframes=n, decoding="BP_MS", iterations=iters,
                       early_term=et, threads=THREADS, gen=oracle_gen if with_gen else None)
    assert 0.05 < want["fec"] / n < 0.9, want
    assert {k: got[k] for k in want} == want


@pytest.mark.parametrize("shape", ["f32", "global", "layered"])
@pytest.mark.parametrize("L", [1, 0])
def test_other_shapes_equal_host_accounting(ctx, shape, L):
    from libldpc_b200 import api
    tun = {"f32": dict(precision=api.F32), "global": dict(residency=api.GLOBAL), "layered": dict(schedule=api.LAYERED)}[shape]
    ctx.set_fading(L)
    ctx.set_tuning(zero_codeword=1, **tun)
    x = -4.0 if L == 1 else 0.0
    n, seed, point, frame0 = 3000, 5, 1, 11
    got = ctx.sim_point("RAYLEIGH", x, seed=seed, point=point, frame0=frame0, nframes=n, decoding="BP_MS", iterations=25, early_term=True)
    cw, llr = ctx.channel("RAYLEIGH", x, seed, point, frame0, n)
    _, hard, its = ctx.decode_batch(llr, "BP_MS", 25, True, want_llr=False)
    tx = ctx.bit_pos()
    errs = (hard[:, tx] != cw[:, tx]).sum(1)
    assert errs.any()
    assert got["frames"] == n and got["iters"] == int(its.sum())
    assert got["fec"] == int((errs > 0).sum()) and got["bec"] == int(errs.sum())


@pytest.mark.parametrize("L", [1, 0])
def test_replay_of_logged_frames(ctx, L):
    ctx.set_fading(L)
    x = -4.0 if L == 1 else 0.0
    cnt, log, n_err = ctx.sim_point_log("RAYLEIGH", x, seed=3, point=4, frame0=0, nframes=2000, decoding="BP_MS", iterations=30,
                                        early_term=True, capacity=4096)
    assert n_err == cnt["fec"] == len(log) > 0
    reps = ctx.error_reports("RAYLEIGH", x, 3, 4, [f for f, _, _ in log], decoding="BP_MS", iterations=30, early_term=True)
    assert [(r["frame"], r["hamming_distance"], r["iterations"]) for r in reps] == log


def _results(out):
    """rows of a results file without the frame-time column"""
    lines = out.read_text().split("\n")
    assert lines[0] == "snr fer ber frames avg_iter frame_time"
    return [l.split()[:5] for l in lines[1:] if l]


def _cli(out, *extra):
    r = subprocess.run([CLI, H_FILE, str(out), "-5", "-2.9", "1", "--channel", "RAYLEIGH", "--decoding", "BP_MS", "-i", "30",
                        "--frame-error-count", "40", "--max-frames", "200000", *extra], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    return _results(out)


@pytest.mark.parametrize("L", ["1", "0"])
def test_cli_shards_and_error_log(built_lib, tmp_path, L):
    one = _cli(tmp_path / "one.txt", "--coherence", L)
    assert len(one) == 3
    fer = [float(r[1]) for r in one]
    assert fer[0] > 0 and (L == "0" or fer == sorted(fer, reverse=True))
    assert _cli(tmp_path / "three.txt", "--coherence", L, "--devices", "0,0,0") == one
    log = tmp_path / "err.log"
    assert _cli(tmp_path / "logged.txt", "--coherence", L, "--error-log", str(log)) == one
    lines = log.read_text().split("\n")
    assert len(lines) > 2 and lines[0].startswith("snr frame iterations")


def test_fer_exceeds_awgn_and_fast_fading(ctx):
    n = 20000
    kw = dict(seed=9, point=0, frame0=0, nframes=n, decoding="BP_MS", iterations=30, early_term=True)
    ctx.set_tuning(zero_codeword=1)
    awgn = ctx.sim_point("AWGN", -4.0, **kw)["fec"] / n
    fast = ctx.sim_point("RAYLEIGH", -4.0, **kw)["fec"] / n
    assert fast > awgn
    fast = ctx.sim_point("RAYLEIGH", -3.0, **kw)["fec"] / n
    ctx.set_fading(0)
    slow = ctx.sim_point("RAYLEIGH", -3.0, **kw)["fec"] / n
    assert 0 < fast < 0.1 and slow > fast


def test_fading_arguments(ctx):
    with pytest.raises(RuntimeError, match="coherence"):
        ctx.set_fading(-1)
    ctx.set_modulation(4)
    with pytest.raises(RuntimeError, match="BPSK only"):
        ctx.channel("RAYLEIGH", 0.0, 0, 0, 0, 1)
    with pytest.raises(RuntimeError, match="BPSK only"):
        ctx.sim_point("RAYLEIGH", 0.0, nframes=10)


def test_reference_simulate_accepts_rayleigh(built_lib):
    """The six-symbol simulate() (through the pyLDPC-style wrapper) with channel_param.type = "RAYLEIGH", coherence length 1."""
    from libldpc_b200.ldpc import LDPC
    code = LDPC(H_FILE)
    code.simulate(snr=[-4.0, -3.0, 0.5], channel="RAYLEIGH", decoding="BP_MS", iterations=30, maxFrames=30000, fec=30, seed=4)
    code.wait()
    res = code.get_results()
    assert len(res["fer"]) == 2 and all(f > 0 for f in res["frames"]) and res["fer"][0] > res["fer"][1] > 0
