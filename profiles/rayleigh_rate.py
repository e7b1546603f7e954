"""Cost of the RAYLEIGH channel in the fused sweep: device-timed frames/s of RAYLEIGH (coherence L = 1 and L = 0) against AWGN
at the same x, on h.txt with min-sum at 50 fixed iterations, on h.txt with early termination at a high-SNR point (where the
channel is a large share of a frame), and on the BG1-shaped code.  The three channels are timed in alternation, several times;
the median and the spread are reported.  Prints one JSON object (and writes it to --out) with the card's name and power limit,
read in the same run.

    python profiles/rayleigh_rate.py [--out FILE] [--reps N]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "codes"))

CHANNELS = (("AWGN", 1), ("RAYLEIGH", 1), ("RAYLEIGH", 0))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0]


def rates(ctx, x, frames, et, reps, decoding="BP_MS", iters=50):
    """frames/s (CUDA-event time of the sweep kernel inside sim_point) of every channel of CHANNELS, timed in alternation"""
    kw = dict(decoding=decoding, iterations=iters, early_term=et)
    for ch, L in CHANNELS:   # warm-up and the one-off shape trial
        ctx.set_fading(L)
        ctx.sim_point(ch, x, seed=1, point=0, frame0=0, nframes=min(frames, 1 << 16), **kw)
    runs = {"%s_L%d" % (ch, L) if ch == "RAYLEIGH" else ch: [] for ch, L in CHANNELS}
    its = dict.fromkeys(runs, 0)
    for r in range(reps):
        for (ch, L), name in zip(CHANNELS, runs):
            ctx.set_fading(L)
            res = ctx.sim_point(ch, x, seed=2 + r, point=0, frame0=0, nframes=frames, **kw)
            runs[name].append(frames / (res["device_ms"] * 1e-3))
            its[name] += res["iters"]
    out = {}
    for name, v in runs.items():
        v = np.array(v)
        out[name] = dict(frames_per_s_median=float(np.median(v)), spread=float((v.max() - v.min()) / np.median(v)),
                         runs=[float(a) for a in v], avg_ref_iterations=its[name] / (frames * reps))
    base = out["AWGN"]["frames_per_s_median"]
    for name in out:
        out[name]["vs_awgn"] = out[name]["frames_per_s_median"] / base
    return dict(x=x, frames=frames, early_term=et, decoding=decoding, iterations=iters, channels=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    from libldpc_b200 import api
    import gen_codes
    res = dict(card=card())
    h_file = os.path.join(ROOT, "codes", "ref_h_n1152_m1024.txt")
    ctx = api.Context(h_file, "", device=0)
    res["h_ms50_fixed"] = rates(ctx, -5.0, 1 << 21, False, args.reps)
    res["h_ms50_et_high_snr"] = rates(ctx, 0.0, 1 << 22, True, args.reps)
    ctx.close()
    with tempfile.TemporaryDirectory() as tmp:
        big = gen_codes.ensure(("bg1",), directory=tmp)
        ctx = api.Context(big["bg1"], "", device=0)
        res["bg1_ms50_fixed"] = rates(ctx, -0.5, 1 << 14, False, args.reps)
        ctx.close()
    res["card_after"] = card()
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
