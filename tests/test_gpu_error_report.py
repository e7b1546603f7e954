"""Batched replay of frames in error (ldpc_b200_error_report, Context.error_reports) and `ldpcsim --error-log`: the batched
reports against the one-frame-per-call reference Context.error_report and a vectorised host reference, the capacity contract,
and the CLI's log against the sweep."""
import ctypes as ct
import os
import subprocess

import numpy as np
import pytest

from conftest import H_FILE, ROOT

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "libldpc_b200", "ldpcsim")
FIELDS = ("frame", "iterations", "failed_bits", "hamming_distance", "failed_checks", "syndrome_weight")


@pytest.fixture(scope="module")
def h_ctx(built_lib):
    """h.txt without a generator matrix: the context the CLI opens without -G."""
    from libldpc_b200 import api
    ctx = api.Context(H_FILE, "", device=0)
    yield ctx
    ctx.close()


def _restore(ctx):
    from libldpc_b200 import api
    ctx.set_modulation(2)
    ctx.set_tuning(precision=api.F64, schedule=api.FLOODING, zero_codeword=0, bec_deg1_compat=1)


# (name, channel, x, decoding, iterations, tuning, modulation M, frames swept)
CASES = [
    ("awgn_ms", "AWGN", -5.0, "BP_MS", 30, dict(zero_codeword=1), 2, 600),
    ("awgn_bp_gen", "AWGN", -4.8, "BP", 20, dict(zero_codeword=0), 2, 600),
    ("bsc", "BSC", 0.16, "BP_MS", 30, dict(zero_codeword=1), 2, 8 << 20),     # error-floor region: errors are rare
    ("bec_compat1", "BEC", 0.9, "BP", 50, dict(zero_codeword=1, bec_deg1_compat=1), 2, 2000),
    ("bec_compat0", "BEC", 0.9, "BP", 50, dict(zero_codeword=1, bec_deg1_compat=0), 2, 2000),
    ("bec_gen_compat1", "BEC", 0.9, "BP", 50, dict(zero_codeword=0, bec_deg1_compat=1), 2, 2000),
    ("bec_gen_compat0", "BEC", 0.9, "BP", 50, dict(zero_codeword=0, bec_deg1_compat=0), 2, 2000),
    ("ask4", "AWGN", -3.0, "BP_MS", 30, dict(zero_codeword=0), 4, 600),
    ("layered_ms", "AWGN", -5.0, "BP_MS", 20, dict(schedule=1, zero_codeword=1), 2, 600),
    ("f32_ms_gen", "AWGN", -5.0, "BP_MS", 30, dict(precision=1, zero_codeword=0), 2, 600),
]


@pytest.mark.parametrize("name,channel,x,decoding,iters,tuning,M,n", CASES, ids=[c[0] for c in CASES])
def test_batched_reports_equal_per_frame_reports(gpu_ctx, name, channel, x, decoding, iters, tuning, M, n):
    """Frames logged by sim_point_log, shuffled and with a repeat, replayed in one call: the same six fields as error_report
    frame by frame, and each replay's (iterations, bit errors) equal to the sweep's record of that frame."""
    seed, point, f0 = 23, 3, 1 << 33
    kw = dict(decoding=decoding, iterations=iters, early_term=True)
    try:
        gpu_ctx.set_tuning(**tuning)
        if M != 2:
            gpu_ctx.set_modulation(M)
        cnt, log, n_err = gpu_ctx.sim_point_log(channel, x, seed=seed, point=point, frame0=f0, nframes=n, capacity=min(n, 1 << 16), **kw)
        assert n_err == len(log) == cnt["fec"] > 3, (name, cnt)
        rng = np.random.default_rng(5)
        pick = [log[i] for i in rng.permutation(len(log))[:40]]
        pick.append(pick[len(pick) // 2])
        reps = gpu_ctx.error_reports(channel, x, seed, point, [p[0] for p in pick], **kw)
        assert len(reps) == len(pick)
        for (frame, bit_errors, its), rep in zip(pick, reps):
            assert list(rep) == list(FIELDS)
            assert (rep["frame"], rep["iterations"], rep["hamming_distance"]) == (frame, its, bit_errors), name
            assert len(rep["failed_bits"]) == bit_errors and len(rep["failed_checks"]) == rep["syndrome_weight"]
            ref = gpu_ctx.error_report(channel, x, seed, point, frame, **kw)
            if M == 2:
                assert rep == ref, (name, frame)
            else:
                # error_report compares the decisions with the channel's scrambling bits; the decoder sees the all-zero word
                # (ldpc_b200_set_modulation), which is what the sweep counts and the batched report compares with
                assert {k: rep[k] for k in ("frame", "iterations", "failed_checks", "syndrome_weight")} == \
                    {k: ref[k] for k in ("frame", "iterations", "failed_checks", "syndrome_weight")}, (name, frame)
                cw, llr = gpu_ctx.channel(channel, x, seed, point, frame, 1)
                _, hard, _ = gpu_ctx.decode_batch(llr, decoding, iters, True, want_llr=False)
                tx = gpu_ctx.bit_pos()
                assert rep["failed_bits"] == [int(b) for b in tx[hard[0][tx] != 0]], (name, frame)
    finally:
        _restore(gpu_ctx)


def _host_reports(ctx, channel, x, seed, point, frame0, n, decoding, iters, block=4000):
    """Vectorised reference for the contiguous frames [frame0, frame0 + n): channel(), decode_batch (or the erasure decode),
    failed bits over the transmitted positions and a syndrome over the edges."""
    from scipy import sparse
    r, c = ctx.edges()
    Hs = sparse.csr_matrix((np.ones(len(r), np.int32), (r, c)), shape=(ctx.mc, ctx.nc))
    tx = ctx.bit_pos()
    out = []
    for o in range(0, n, block):
        m = min(block, n - o)
        cw, llr = ctx.channel(channel, x, seed, point, frame0 + o, m)
        if channel == "BEC":
            _, hard, its = ctx.decode_bec_batch(llr, cw, iters, True)
        else:
            _, hard, its = ctx.decode_batch(llr, decoding, iters, True, want_llr=False)
        synd = np.asarray(Hs @ hard.T.astype(np.int32)) & 1      # [mc][m]
        bad = hard[:, tx] != cw[:, tx]
        for i in range(m):
            fb = tx[bad[i]]
            fc = np.nonzero(synd[:, i])[0]
            out.append(dict(frame=frame0 + o + i, iterations=int(its[i]), failed_bits=[int(b) for b in fb], hamming_distance=len(fb),
                            failed_checks=[int(k) for k in fc], syndrome_weight=len(fc)))
    return out


def test_many_frames_span_several_chunks(h_ctx):
    """40,000 contiguous frames of h.txt (about 370 MB of decoder input: several 32 MB chunks), failures and successes mixed."""
    n, f0, x = 40000, 12345, -4.2
    reps = h_ctx.error_reports("AWGN", x, 7, 1, np.arange(f0, f0 + n), decoding="BP_MS", iterations=20)
    ref = _host_reports(h_ctx, "AWGN", x, 7, 1, f0, n, "BP_MS", 20)
    failed = sum(r["hamming_distance"] > 0 for r in ref)
    assert 50 < failed < n - 50
    assert reps == ref


def test_many_frames_bec(h_ctx):
    n, f0 = 5000, 99
    reps = h_ctx.error_reports("BEC", 0.89, 2, 0, np.arange(f0, f0 + n), iterations=50)
    ref = _host_reports(h_ctx, "BEC", 0.89, 2, 0, f0, n, "BP", 50)
    assert sum(r["hamming_distance"] > 0 for r in ref) > 10
    assert reps == ref


def test_dvbs2_shaped_code(built_lib):
    """The DVB-S2-shaped code (nc = 64800): a few frames per chunk, long lists."""
    from conftest import large_code_files
    from libldpc_b200 import api
    ctx = api.Context(large_code_files()["dvbs2"], "", device=0)
    try:
        n, x = 240, -2.5
        reps = ctx.error_reports("AWGN", x, 4, 0, np.arange(n), decoding="BP_MS", iterations=30)
        ref = _host_reports(ctx, "AWGN", x, 4, 0, 0, n, "BP_MS", 30, block=60)
        assert reps == ref
        assert sum(r["hamming_distance"] > 0 for r in ref) > 0
    finally:
        ctx.close()


def test_capacity_contract_and_bad_arguments(h_ctx):
    """Too-small list capacities fail, write nothing and return the exact sizes; bad arguments fail with a message."""
    from libldpc_b200 import api
    L = h_ctx.lib
    dp = api.decoder_param(True, 30, b"BP_MS")
    frames = np.arange(100, 400, dtype=np.uint64)
    good = h_ctx.error_reports("AWGN", -5.0, 3, 0, frames, decoding="BP_MS", iterations=30)
    nb_want = sum(r["hamming_distance"] for r in good)
    nk_want = sum(r["syndrome_weight"] for r in good)
    assert nb_want > 0 and nk_want > 0

    def call(fr, n, bcap, kcap, channel=b"AWGN", ctx=h_ctx._h, rep=True):
        reps = (api.frame_report * max(n, 1))()
        for r in reps:
            r.frame, r.bits_offset = 777, -5
        bits = np.full(max(bcap, 1), -7, np.int32)
        checks = np.full(max(kcap, 1), -7, np.int32)
        nb, nk = ct.c_int64(-1), ct.c_int64(-1)
        fp = fr.ctypes.data_as(ct.POINTER(ct.c_uint64)) if fr is not None else None
        rc = L.ldpc_b200_error_report(ctx, dp, channel, -5.0, 3, 0, fp, n, reps if rep else None, bits.ctypes.data_as(ct.POINTER(ct.c_int32)), bcap,
                                      checks.ctypes.data_as(ct.POINTER(ct.c_int32)), kcap, ct.byref(nb), ct.byref(nk))
        return rc, reps, bits, checks, nb.value, nk.value

    for bcap, kcap in ((0, 0), (nb_want - 1, nk_want), (nb_want, nk_want - 1)):
        rc, reps, bits, checks, nb, nk = call(frames, len(frames), bcap, kcap)
        assert rc != 0 and "capacities" in L.ldpc_b200_last_error().decode()
        assert (nb, nk) == (nb_want, nk_want)
        assert (bits == -7).all() and (checks == -7).all() and all(r.frame == 777 and r.bits_offset == -5 for r in reps)
    rc, reps, bits, checks, nb, nk = call(frames, len(frames), nb_want, nk_want)
    assert rc == 0 and (nb, nk) == (nb_want, nk_want)
    for r, g in zip(reps, good):
        assert list(bits[r.bits_offset:r.bits_offset + r.bit_errors]) == g["failed_bits"]
        assert list(checks[r.checks_offset:r.checks_offset + r.syndrome_weight]) == g["failed_checks"]
    rc, *_, nb, nk = call(frames, 0, 0, 0)
    assert rc == 0 and (nb, nk) == (0, 0)
    assert call(frames, -1, 10, 10)[0] != 0
    assert call(frames, len(frames), -1, 10)[0] != 0
    assert call(None, 5, 10, 10)[0] != 0 and "null" in L.ldpc_b200_last_error().decode()
    assert call(frames, len(frames), 10, 10, rep=False)[0] != 0
    assert call(frames, 5, 10, 10, channel=b"XYZ")[0] != 0 and "No channel selected" in L.ldpc_b200_last_error().decode()
    assert call(frames, 5, 10, 10, channel=None)[0] != 0
    assert call(frames, 5, 10, 10, ctx=None)[0] != 0
    with pytest.raises(RuntimeError, match="No channel selected"):
        h_ctx.error_reports("XYZ", 1.0, 0, 0, [1])
    assert h_ctx.error_reports("AWGN", 1.0, 0, 0, []) == []


def _sweep_points(lo, hi, step, eps_axis):
    xs, v = [], lo
    while v < hi:
        xs.append(v)
        v += step
    return xs[::-1] if eps_axis else xs


def _run_cli(out, args, log=None, devices="0"):
    cmd = [CLI, H_FILE, str(out)] + args + ["--devices", devices] + (["--error-log", str(log)] if log else [])
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    return [l.split() for l in out.read_text().split("\n")[1:-1]]    # one row per point; empty while a point has no frame error


SWEEPS = [
    ("AWGN", ["-5.5", "-4.4", "0.5", "--decoding", "BP_MS", "--frame-error-count", "25", "--max-frames", "60000", "-i", "30", "-s", "4"],
     (-5.5, -4.4, 0.5), "BP_MS", 30),
    ("BEC", ["0.80", "0.9", "0.05", "--channel", "BEC", "--frame-error-count", "25", "--max-frames", "200000", "-s", "4"],
     (0.80, 0.9, 0.05), "BP", 50),
]


@pytest.mark.parametrize("channel,args,rng,decoding,iters", SWEEPS, ids=[s[0] for s in SWEEPS])
def test_cli_error_log(h_ctx, tmp_path, channel, args, rng, decoding, iters):
    """ldpcsim --error-log: the results file equals the one without the flag (all columns but the frame time); per point at
    most --frame-error-count lines, which are the first frames in error in frame order, each equal to error_report; the log is
    byte-identical for one, two and three shards."""
    fec = 25
    plain = _run_cli(tmp_path / "plain.txt", args)
    logs = []
    for devs in ("0", "0,0", "0,0,0"):
        log = tmp_path / ("err_%d.log" % len(logs))
        rows = _run_cli(tmp_path / ("res_%d.txt" % len(logs)), args, log=log, devices=devs)
        assert [r[:5] for r in rows] == [r[:5] for r in plain]
        logs.append(log.read_bytes())
    assert logs[0] == logs[1] == logs[2]
    lines = logs[0].decode().split("\n")
    assert lines[0] == "snr frame iterations bit_errors syndrome_weight failed_bits failed_checks" and lines[-1] == ""
    xs = _sweep_points(*rng, eps_axis=channel != "AWGN")
    name_of = {"%f" % x: i for i, x in enumerate(xs)}
    by_point = {}
    for l in lines[1:-1]:
        snr, frame, its, be, sw, fb, fc = l.split(" ")
        by_point.setdefault(name_of[snr], []).append((int(frame), int(its), int(be), int(sw), fb, fc))
    assert list(by_point) == sorted(by_point) and set(by_point) == {i for i, r in enumerate(plain) if r}   # points in execution order
    kw = dict(decoding=decoding, iterations=iters, early_term=True)
    for i, entries in by_point.items():
        frames_i = int(plain[i][3])
        assert plain[i][0] == "%f" % xs[i]
        _, log, n_err = h_ctx.sim_point_log(channel, xs[i], seed=4, point=i, frame0=0, nframes=frames_i, capacity=frames_i, **kw)
        assert [e[0] for e in entries] == [f for f, _, _ in log[:fec]]
        for (frame, its, be, sw, fb, fc), (lf, lbe, lits) in zip(entries, log):
            ref = h_ctx.error_report(channel, xs[i], 4, i, frame, **kw)
            assert (its, be, sw) == (ref["iterations"], ref["hamming_distance"], ref["syndrome_weight"]) == (lits, lbe, sw)
            assert fb == (",".join(map(str, ref["failed_bits"])) or "-") and fc == (",".join(map(str, ref["failed_checks"])) or "-")
