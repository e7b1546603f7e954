"""Cost of the error-floor diagnostics: reports/s of the batched replay (Context.error_reports, one call) against the
one-frame-per-call reference (a loop of Context.error_report) on frames that a sweep logged, and the wall time of ldpcsim
with and without --error-log.  Prints one JSON object (and writes it to --out) with the card's name and power limit, read
in the same run.

    python profiles/error_report_rate.py [--out FILE]
"""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "codes"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0]


def replay_rates(api, ctx, name, channel, x, decoding, iters, n_logged, sweep, loop_frames):
    """Logs n_logged frames in error at one point, then times both replay paths on them."""
    frames, f0 = [], 0
    while len(frames) < n_logged and f0 < 50 * sweep:
        _, log, _ = ctx.sim_point_log(channel, x, seed=1, point=0, frame0=f0, nframes=sweep, decoding=decoding, iterations=iters,
                                      capacity=sweep)
        frames += [f for f, _, _ in log]
        f0 += sweep
    frames = frames[:n_logged]
    kw = dict(decoding=decoding, iterations=iters, early_term=True)
    ctx.error_reports(channel, x, 1, 0, frames[:64], **kw)           # warm-up: tables, kernel attributes, shape trial
    ctx.error_report(channel, x, 1, 0, frames[0], **kw)
    t = time.perf_counter()
    reps = ctx.error_reports(channel, x, 1, 0, frames, **kw)
    batched = time.perf_counter() - t
    # the C ABI call alone, with list capacities that fit at once (error_reports may have to replay twice to learn them)
    nb, nk = sum(r["hamming_distance"] for r in reps), sum(r["syndrome_weight"] for r in reps)
    fr = np.ascontiguousarray(frames, np.uint64)
    rep = (api.frame_report * len(frames))()
    bits, checks = np.empty(max(nb, 1), np.int32), np.empty(max(nk, 1), np.int32)
    t = time.perf_counter()
    rc = ctx.lib.ldpc_b200_error_report(ctx._h, ctx._dp(decoding, iters, True), channel.encode(), float(x), 1, 0,
                                        fr.ctypes.data_as(ct.POINTER(ct.c_uint64)), len(frames), rep, bits.ctypes.data_as(ct.POINTER(ct.c_int32)),
                                        bits.size, checks.ctypes.data_as(ct.POINTER(ct.c_int32)), checks.size, None, None)
    abi = time.perf_counter() - t
    assert rc == 0
    t = time.perf_counter()
    for f in frames[:loop_frames]:
        ctx.error_report(channel, x, 1, 0, f, **kw)
    loop = time.perf_counter() - t
    return dict(code=name, channel=channel, x=x, decoding=decoding, iterations=iters, frames=len(frames),
                mean_failed_bits=float(np.mean([r["hamming_distance"] for r in reps])),
                failed_bits=nb, failed_checks=nk, batched_s=batched, batched_reports_per_s=len(frames) / batched,
                abi_call_s=abi, abi_reports_per_s=len(frames) / abi,
                loop_frames=loop_frames, loop_s=loop, loop_reports_per_s=loop_frames / loop)


def cli_times(h_file, tmp):
    cli = os.path.join(ROOT, "libldpc_b200", "ldpcsim")
    out = {}
    # BASELINE config 5's BSC point (eps = 0.08, no frame errors in reach) with a frame budget, and a point with errors
    for tag, rng, extra in (("C5_bsc_0.08", ["0.08", "0.0801", "0.01"], ["--max-frames", str(1 << 27)]),
                            ("bsc_0.18", ["0.18", "0.1801", "0.01"], ["--max-frames", str(1 << 27), "--frame-error-count", "200"])):
        for logged in (False, True):
            res_file = os.path.join(tmp, "res.txt")
            if os.path.exists(res_file):
                os.remove(res_file)
            cmd = [cli, h_file, res_file] + rng + ["--channel", "BSC", "--decoding", "BP_MS", "-i", "50"] + extra
            if logged:
                cmd += ["--error-log", os.path.join(tmp, "err.log")]
            t = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True)
            wall = time.perf_counter() - t
            assert r.returncode == 0, r.stdout + r.stderr
            row = open(res_file).read().split("\n")[1].split() if os.path.exists(res_file) else None   # written at frame errors only
            out["%s_%s" % (tag, "error_log" if logged else "plain")] = dict(wall_s=wall, results_row=row)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    args = ap.parse_args()
    from libldpc_b200 import api
    import gen_codes
    h_file = os.path.join(ROOT, "codes", "ref_h_n1152_m1024.txt")
    res = dict(card=card())
    ctx = api.Context(h_file, "", device=0)
    res["h_txt"] = replay_rates(api, ctx, "h.txt", "AWGN", -5.0, "BP_MS", 50, 10000, 20000, 500)
    ctx.close()
    with tempfile.TemporaryDirectory() as tmp:
        big = gen_codes.ensure(("dvbs2",), directory=tmp)
        ctx = api.Context(big["dvbs2"], "", device=0)
        res["dvbs2"] = replay_rates(api, ctx, "dvbs2", "AWGN", -2.5, "BP_MS", 30, 10000, 10000, 50)
        ctx.close()
        res["ldpcsim"] = cli_times(h_file, tmp)
    res["card_after"] = card()
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
