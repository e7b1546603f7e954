"""Cost of the fixed-point layered decoder: device-timed frames/s of layered fp64 min-sum against quantised (6, 6, 8) layered
min-sum (step 0.5, the same normalisation: 0.75 on the BG1-shaped code, 1 on h.txt) in the fused sweep, on the BG1-shaped code and
on h.txt, at 50 fixed iterations and on an early-termination sweep point.  The two decoders are timed in alternation, several
times, on the same card; the median and the spread are reported with the FER of both.  Prints one JSON object (and writes it
to --out) with the card's name and power limit, read in the same run.

    python profiles/quant_rate.py [--out FILE] [--reps N]
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

QUANT = (6, 6, 8, 0.5)  # ch_bits, msg_bits, post_bits, step


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0]


def rates(ctx, x, frames, et, reps, scale8=8, iters=50):
    """frames/s (CUDA-event time of the sweep kernel inside sim_point) of fp64 and quantised layered min-sum, in alternation"""
    kw = dict(decoding="BP_MS", iterations=iters, early_term=et)

    def use(name):
        if name == "fp64":
            ctx.set_quant(None)
        else:
            ctx.set_quant(QUANT[0], QUANT[1], QUANT[2], QUANT[3], scale8=scale8)

    names = ("fp64", "q668")
    for name in names:   # warm-up
        use(name)
        ctx.sim_point("AWGN", x, seed=1, nframes=min(frames, 1 << 14), **kw)
    runs = {n: [] for n in names}
    fec = dict.fromkeys(names, 0)
    for r in range(reps):
        for name in names:
            use(name)
            res = ctx.sim_point("AWGN", x, seed=2 + r, nframes=frames, **kw)
            runs[name].append(frames / (res["device_ms"] * 1e-3))
            fec[name] += res["fec"]
    out = {}
    for name, v in runs.items():
        v = np.array(v)
        out[name] = dict(frames_per_s_median=float(np.median(v)), spread=float((v.max() - v.min()) / np.median(v)),
                         runs=[float(a) for a in v], fer=fec[name] / (frames * reps))
    out["q668"]["vs_fp64"] = out["q668"]["frames_per_s_median"] / out["fp64"]["frames_per_s_median"]
    ctx.set_quant(None)
    return dict(x=x, frames=frames, early_term=et, iterations=iters, scale8=scale8, decoders=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    from libldpc_b200 import api
    import gen_codes
    os.environ.setdefault("LDPC_B200_TUNE_CACHE", "off")
    res = dict(card=card(), quant=dict(ch_bits=QUANT[0], msg_bits=QUANT[1], post_bits=QUANT[2], step=QUANT[3]))
    with tempfile.TemporaryDirectory() as tmp:
        big = gen_codes.ensure(("bg1",), directory=tmp)
        ctx = api.Context(big["bg1"], "", device=0)
        ctx.set_tuning(schedule=api.LAYERED, layered_ms_scale64=48)
        res["bg1_fixed50"] = rates(ctx, 0.5, 1 << 14, False, args.reps, scale8=6)
        res["bg1_et"] = rates(ctx, 1.0, 1 << 15, True, args.reps, scale8=6)
        ctx.close()
    h_file = os.path.join(ROOT, "codes", "ref_h_n1152_m1024.txt")
    ctx = api.Context(h_file, "", device=0)
    ctx.set_tuning(schedule=api.LAYERED)
    res["h_fixed50"] = rates(ctx, -4.0, 1 << 20, False, args.reps)
    res["h_et"] = rates(ctx, -3.0, 1 << 21, True, args.reps)
    ctx.close()
    res["card_after"] = card()
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
