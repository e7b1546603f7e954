#!/usr/bin/env python
"""bench.py — decoded coded Gb/s of the LDPC decode hot path on B200 (contract: see DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, NCCL)

Headline workload (BASELINE.json configs[1]): codes/ref_h_n1152_m1024.txt (n=1024, k=128 transmitted), AWGN,
BP_MS, -i 50, every frame running the full 50 iterations (the "@50 iters" of the metric, i.e. --no-early-term).  One
step = one pass of channel -> decode -> accounting over FRAMES_PER_STEP frames per GPU (weak scaling: frames shard
over GPUs, counters are all-reduced once per step).  --dump-outputs DIR writes what the last timed step returned to its
caller, the counters {frame errors, bit errors, frames, sum of reference iteration counts, sum of executed iterations}
over all GPUs, as DIR/counters.npy (float64); the frames of every step are fixed by the seed and the step index.

Besides the headline the line carries (N=1): `configs` — all five BASELINE.json configurations, each device-timed with
its own roofline (shared memory / HBM / FP64 pipe); `e2e` — the batch decode call with HOST buffers; `cpu_baseline` — the
unmodified reference CLI on this box's host cores.
"""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H_FILE = os.path.join(ROOT, "codes", "ref_h_n1152_m1024.txt")
SNR_DB = -4.5
ITERS = 50
DECODING = "BP_MS"
FRAMES_PER_STEP = 148 * 4 * 512          # per GPU and step (303,104 frames ~ 65 ms of B200 time)
NCT, NC, NNZ, MC = 1024, 1152, 3456, 1024
METRIC = "decoded coded Gb/s @50 iters"
UNIT = "Gb/s"
WORKLOAD = ("h.txt n=1024 k=128 (1152x1024, nnz 3456), AWGN Es/sigma^2=-4.5 dB, BP_MS min-sum, -i 50, "
            "fixed 50 iterations/frame (--no-early-term)")
FP64_PER_BOXPLUS = 50                    # FP64 instructions of one pairwise box-plus (fallback; the per-code figures come from ncu, profiles/roofline_traffic.json)
I8_SCALE = 0.25                          # LLR = int8 * 0.25 on the narrow e2e path (exact in double)


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def read_traffic():
    """DRAM bytes per launch of each configuration's kernel from one `ncu` pass (profiles/traffic.py -> roofline_traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the UNMODIFIED reference CLI (oracle/_ref/ldpcsim_ref) on host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(frames, threads, snr=SNR_DB):
    """Runs the reference's own ldpcsim on `frames` frames of the bench workload at `snr`; returns (seconds, frames, kind)."""
    ref = os.path.join(ROOT, "oracle", "_ref", "ldpcsim_ref")
    if os.path.exists(ref):
        out = f"/tmp/bench_ref_{os.getpid()}.txt"
        cmd = [ref, H_FILE, out, str(snr), str(snr + 0.25), "0.5", "--decoding", DECODING, "-i", str(ITERS), "--no-early-term",
               "--max-frames", str(frames), "--frame-error-count", "1000000000", "-t", str(threads), "-s", "0"]
        t0 = time.perf_counter()
        subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL)
        dt = time.perf_counter() - t0
        done = frames
        try:  # the reference overshoots max-frames by up to `threads` frames; use what it reports (it only reports when frames erred)
            last = [l for l in open(out).read().splitlines()[1:] if l.strip()]
            if last:
                done = int(last[-1].split()[3])
            os.remove(out)
        except Exception:
            pass
        return dt, done, "reference"
    # the reference could not be compiled for this box: time the C restatement instead
    from oracle import oracle as O
    c = O.Code(H_FILE)
    t0 = time.perf_counter()
    c.sim_point("AWGN", snr, seed=0, point=0, frame0=0, nframes=frames, decoding=DECODING, iterations=ITERS, early_term=False, threads=threads)
    return time.perf_counter() - t0, frames, "port"


def cpu_baseline(budget_s=10.0):
    threads = os.cpu_count() or 1
    dt, done, kind = cpu_reference_run(threads * 8, threads)          # calibration
    rate = done / dt
    frames = max(int(rate * budget_s), threads * 8)
    dt, done, kind = cpu_reference_run(frames, threads)
    gbps = done * NCT / dt / 1e9
    # the same fixed work at a point without frame errors (+2 dB): there the reference never enters its critical section
    # (no results-file rewrite per error, BASELINE.md 4.3); -4.5 dB has FER 0.19
    dt0, done0, _ = cpu_reference_run(frames, threads, snr=2.0)
    return {"value": gbps, "unit": UNIT, "cores": threads, "kind": kind, "frames_per_s": done / dt,
            "sample": f"{done} frames of the bench workload via {'oracle/_ref/ldpcsim_ref' if kind == 'reference' else 'oracle port'} "
                      f"-t {threads} --no-early-term in {dt:.1f} s",
            "zero_error_point": {"value": done0 * NCT / dt0 / 1e9, "unit": UNIT, "snr_db": 2.0,
                                 "sample": f"{done0} frames at +2 dB (no frame errors, same fixed 50 iterations) in {dt0:.1f} s"}}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    dt, done, kind = cpu_reference_run(threads * 8, threads)
    rate = done / dt
    per_step = max(int(rate * min(8.0, 150.0 / max(args.steps + args.warmup, 1))), threads * 4)
    for _ in range(args.warmup):
        cpu_reference_run(per_step, threads)
    tot_t, tot_f = 0.0, 0
    for _ in range(args.steps):
        dt, done, kind = cpu_reference_run(per_step, threads)
        tot_t += dt
        tot_f += done
    gbps = tot_f * NCT / tot_t / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": gbps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": tot_t / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": WORKLOAD, "frames_per_step": per_step},
            "cpu_baseline": {"value": gbps, "unit": UNIT, "cores": threads, "kind": kind,
                             "sample": f"{tot_f} frames in {tot_t:.1f} s, {args.steps} steps of {per_step} frames, -t {threads}"},
            "e2e": {"value": gbps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# the five BASELINE configurations (N = 1): device-timed kernels, each with the roofline that bounds it
# ------------------------------------------------------------------------------------------------
def boxplus_per_iteration(nnz, mc):
    return 3 * nnz - 4 * mc      # pairwise updates of the forward/backward recursion per frame-iteration (SURVEY.md 8 a5)


def run_configs(api, smem_peak, fp64_peak, hbm_peak, traffic):
    sys.path.insert(0, os.path.join(ROOT, "codes"))
    import gen_codes
    codes_dir = tempfile.TemporaryDirectory()      # generated outside the tree, which may be read-only
    big = gen_codes.ensure(directory=codes_dir.name)
    out = {}

    def measure(ctx, channel, xs, decoding, et, frames, reps=2):
        """device-timed (CUDA events around the kernel, inside sim_point) pass over `frames` frames at every x; best of reps"""
        tot_ms, tot_frames, tot_edge, launches = 0.0, 0, 0, 0
        for i, x in enumerate(xs):
            ctx.sim_point(channel, x, seed=1, point=i, frame0=0, nframes=min(frames, 1 << 16), decoding=decoding, iterations=ITERS, early_term=et)  # warm-up / shape trial
            best = None
            for r in range(reps):
                ctx.stats(reset=True)
                res = ctx.sim_point(channel, x, seed=2 + r, point=i, frame0=0, nframes=frames, decoding=decoding, iterations=ITERS, early_term=et)
                st = ctx.stats()
                if best is None or res["device_ms"] < best[0]:
                    best = (res["device_ms"], st["edge_iterations"], res)
            tot_ms += best[0]; tot_frames += frames; tot_edge += best[1]; launches += reps + 1
        return tot_ms, tot_frames, tot_edge, st, launches

    def entry(name, ctx, ms, frames, edge_it, st, bound, what, extra=None, msg_bytes=32):
        t = ms * 1e-3
        e = {"workload": what, "value": frames * ctx.nct / t / 1e9, "unit": UNIT, "frames_per_s": frames / t, "edge_updates_per_s": edge_it / t,
             "device_ms": ms, "frames": frames,
             "kernel_shape": {"frames_per_cta": st["frames_per_cta"], "threads_per_cta": st["threads_per_cta"], "ctas": st["ctas"],
                              "residency": {1: "smem", 2: "global"}.get(st["residency"], "?")}}
        achieved = edge_it * msg_bytes / t / 1e9
        tr = traffic.get(name)
        if bound == "smem":
            e["roofline"] = {"bound": "smem", "achieved": achieved, "peak": smem_peak, "unit": "GB/s", "frac": achieved / smem_peak,
                             "traffic": tr, "peak_source": "ldpc_b200_smem_probe in this run"}
        elif bound == "hbm":
            e["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                             "traffic": tr, "peak_source": "MEASURED_PEAKS.json hbm_gbs"}
        if extra:
            e.update(extra)
        out[name] = e

    def fp64_block(ctx, edge_it, ms, key):
        # FP64 instructions the kernel executes per edge-iteration on this code: counted by ncu (smsp__inst_executed_pipe_fp64.sum of
        # one launch, profiles/traffic.py); the formula is the fallback when that file is missing
        per_edge_it = traffic.get("_fp64_thread_instructions_per_edge_iteration", {}).get(
            key, FP64_PER_BOXPLUS * boxplus_per_iteration(ctx.nnz, ctx.mc) / ctx.nnz + 2.0)
        ach = edge_it * per_edge_it / (ms * 1e-3) / 1e9
        return {"fp64_pipe": {"bound": "fp64_pipe", "achieved": ach, "peak": fp64_peak, "unit": "G thread-instructions/s", "frac": ach / fp64_peak,
                              "fp64_instructions_per_edge_iteration": per_edge_it,
                              "note": "pipe utilisation: FP64 instructions the kernel executes (ncu count per edge-iteration x edge-iterations of this run) over the measured DFMA issue rate",
                              "peak_source": "ldpc_b200_fp64_probe in this run (independent DFMA chains on every SM)"}}

    launches = 0
    # ---- h.txt --------------------------------------------------------------------------------
    ctx = api.Context(H_FILE, "", device=0)
    ctx.set_tuning(precision=api.F64)
    ms, fr, ed, st, l = measure(ctx, "AWGN", [SNR_DB], "BP", False, 148 * 4 * 64)
    launches += l
    entry("C1_bp_fixed50", ctx, ms, fr, ed, st, "smem", "configs[0] h.txt, AWGN -4.5 dB, BP (sum-product, fp64), 50 fixed iterations", fp64_block(ctx, ed, ms, "C1_bp_fixed50"))
    ms, fr, ed, st, l = measure(ctx, "AWGN", [0.0, 0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 3.5], "BP", True, 148 * 4 * 256)
    launches += l
    entry("C1_et_sweep", ctx, ms, fr, ed, st, "smem", "configs[0] h.txt, AWGN 0 ... 3.5 dB step 0.5 (8 points), BP, -i 50, early termination", fp64_block(ctx, ed, ms, "C1_bp_fixed50"))
    ms, fr, ed, st, l = measure(ctx, "AWGN", [-6.0, -5.5, -5.0, -4.5, -4.0, -3.5], "BP_MS", True, 148 * 4 * 256)
    launches += l
    entry("C2_et", ctx, ms, fr, ed, st, "smem", "configs[1] h.txt, AWGN -6 ... -3.5 dB step 0.5 (6 points), BP_MS, -i 50, early termination")
    ms, fr, ed, st, l = measure(ctx, "BSC", [0.08], "BP_MS", True, 1 << 22)
    launches += l
    entry("C5_bsc", ctx, ms, fr, ed, st, "smem", "configs[4] h.txt, BSC eps = 0.08 (error-floor region), BP_MS, -i 50, early termination")
    ms, fr, ed, st, l = measure(ctx, "BEC", [0.70], "BP", True, 1 << 24)
    launches += l
    # bit-sliced erasure kernel: one known-bit per edge and frame; per edge-iteration and 32-frame word it reads 2 x 2 and writes 2 words
    entry("C5_bec", ctx, ms, fr, ed, st, "smem", "configs[4] h.txt, BEC eps = 0.70 (error-floor region), erasure decoder, -i 50, early termination",
          {"note": "roofline in bytes the bit-sliced kernel moves through shared memory (24 B per edge-iteration and 32-frame word); the kernel is "
                   "bound by instruction issue (Philox channel + boolean folds), not by this pipe"}, msg_bytes=24.0 / 32.0)
    ctx.close()
    # ---- BG1-shaped, Z = 384 ----------------------------------------------------------------------
    # (the one-off shape trial a long sweep would run first: ldpc_b200_prepare; frame counts are whole waves of every kernel shape)
    ctx = api.Context(big["bg1"], "", device=0)
    ctx.prepare("BP_MS", ITERS, False)
    ms, fr, ed, st, l = measure(ctx, "AWGN", [-0.5], "BP_MS", False, 148 * 32)
    launches += l
    entry("C3_bg1_ms", ctx, ms, fr, ed, st, "hbm", "configs[2] NR-BG1-shaped QC code Z=384 (26112 x 17664, nnz 121344), AWGN -0.5 dB, BP_MS fp64, 50 fixed iterations")
    ctx.close()
    # ---- DVB-S2-shaped, n = 64800 -----------------------------------------------------------------
    ctx = api.Context(big["dvbs2"], "", device=0)
    ctx.prepare("BP", ITERS, False)
    ms, fr, ed, st, l = measure(ctx, "AWGN", [1.0], "BP", False, 148 * 16)
    launches += l
    entry("C4_dvbs2_bp_noet", ctx, ms, fr, ed, st, "hbm", "configs[3] DVB-S2-shaped IRA code n=64800 r=1/2 (nnz 226799), AWGN +1 dB, BP fp64, --no-early-term",
          fp64_block(ctx, ed, ms, "C4_dvbs2_bp_noet"))
    ctx.close()
    codes_dir.cleanup()
    return out, launches


def decode_latency():
    """Single-frame decode() of the six-symbol reference ABI (what a pyLDPC user loops over): wall time per call."""
    from libldpc_b200 import api
    import numpy as np
    L = ct.CDLL(api.lib_path())
    n, m, nct, mct = ct.c_int(), ct.c_int(), ct.c_int(), ct.c_int()
    L.ldpc_setup(H_FILE.encode(), b"", ct.byref(n), ct.byref(m), ct.byref(nct), ct.byref(mct))
    L.decode.restype = ct.c_int
    L.decode.argtypes = [api.decoder_param, ct.POINTER(ct.c_double), ct.POINTER(ct.c_double)]
    rng = np.random.default_rng(0)
    llr = (2.0 * (1.0 + rng.normal(0, 1.68, nct.value)) / 2.82).astype(np.float64)
    out = np.empty(nct.value, np.float64)
    dp = api.decoder_param(True, 50, b"BP_MS")
    for _ in range(20):
        L.decode(dp, llr.ctypes.data_as(ct.POINTER(ct.c_double)), out.ctypes.data_as(ct.POINTER(ct.c_double)))
    t0 = time.perf_counter()
    reps = 300
    for _ in range(reps):
        it = L.decode(dp, llr.ctypes.data_as(ct.POINTER(ct.c_double)), out.ctypes.data_as(ct.POINTER(ct.c_double)))
    us = (time.perf_counter() - t0) / reps * 1e6
    return {"us_per_call": us, "frames_per_s": 1e6 / us, "iterations_returned": int(it),
            "call": "decode() of the reference's C ABI (src/shared.cpp:47-65): one frame of nct doubles in, posteriors out, BP_MS -i 50 with early termination"}


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from libldpc_b200 import api, build as B

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the decode path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL writes its version banner to fd 1 at communicator creation: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.all_reduce(torch.zeros(1, device="cuda"))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    if not os.path.exists(api.lib_path()):
        if rank == 0:
            B.build()
        if world > 1:
            dist.barrier()
    ctx = api.Context(H_FILE, "", device=local)
    ctx.set_tuning(precision=api.F64)
    # the one-off kernel-shape trials (blocking) happen here; the timed steps below are asynchronous launches
    for et in (False, True):
        ctx.prepare(DECODING, ITERS, et, nframes=FRAMES_PER_STEP)
    stream = torch.cuda.Stream()
    counters = torch.zeros(8, dtype=torch.int64, device="cuda")
    n_step = FRAMES_PER_STEP

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_cnt = torch.zeros(8, dtype=torch.int64, device="cuda")
    last_cnt = torch.zeros(8, dtype=torch.int64, device="cuda")   # the last timed step's counters (--dump-outputs)

    def step(i, early_term=False, last=False):
        """one pass of channel -> decode -> accounting over this rank's n_step frames (+ the counter all-reduce when sharded);
        last: the step's counters go to last_cnt as well (world > 1) or instead of counters (world == 1)"""
        frame0 = (i * world + rank) * n_step
        if world == 1:
            ctx.sim_point_async((last_cnt if last else counters).data_ptr(), stream.cuda_stream, "AWGN", SNR_DB, seed=0, point=0,
                                frame0=frame0, nframes=n_step, decoding=DECODING, iterations=ITERS, early_term=early_term)
            return
        with torch.cuda.stream(stream):
            step_cnt.zero_()
            ctx.sim_point_async(step_cnt.data_ptr(), stream.cuda_stream, "AWGN", SNR_DB, seed=0, point=0, frame0=frame0, nframes=n_step,
                                decoding=DECODING, iterations=ITERS, early_term=early_term)
            dist.all_reduce(step_cnt)        # 64 B over NVLink: the only collective of the path
            counters.add_(step_cnt)
            if last:
                last_cnt.copy_(step_cnt)

    def timed(nsteps, first, early_term=False, keep_last=False):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(nsteps):
            step(first + i, early_term, last=keep_last and i == nsteps - 1)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for i in range(args.warmup):
        step(10_000 + i)
    barrier()
    counters.zero_()
    ctx.stats(reset=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(args.steps, 0, keep_last=True)
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.stats()["launches"]
    total_frames = n_step * world * args.steps
    value = total_frames * NCT / (ms * 1e-3) / 1e9
    if world == 1:
        counters.add_(last_cnt)
    cnt = counters.cpu().tolist()
    assert cnt[2] == total_frames, (cnt, total_frames)   # every frame of every rank was decoded and counted
    last = last_cnt.cpu().numpy()[:5]
    assert last[2] == n_step * world, last
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "counters.npy"), last.astype(np.float64))

    # per-launch duration of the dominant kernel (single launch per step) with events on the launch stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scratch = torch.zeros(8, dtype=torch.int64, device="cuda")
    kms = []
    for i in range(3):
        torch.cuda.synchronize()
        e0.record(stream)
        ctx.sim_point_async(scratch.data_ptr(), stream.cuda_stream, "AWGN", SNR_DB, seed=0, point=0, frame0=(20_000 + i) * n_step, nframes=n_step,
                            decoding=DECODING, iterations=ITERS, early_term=False)
        e1.record(stream)
        torch.cuda.synchronize()
        kms.append(e0.elapsed_time(e1))
    kernel_ms = sum(kms) / len(kms)
    hbm_peak, hbm_src = read_peaks()
    traffic = read_traffic()
    alg_bytes = n_step * ITERS * NNZ * 4 * 8          # 4 message touches x 8 B (f64) per edge-iteration (SURVEY.md §8d)
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    st = ctx.stats()
    smem_peak = ctx.smem_probe()                      # measured here: LDS.128 streaming from every SM, GB/s
    fp64_peak = ctx.fp64_probe()
    # shared-memory bytes the kernel really moves per edge-iteration (DESIGN.md §3.3): out gather + c2v store (check phase),
    # c2v gather (variable phase) = 3 x 8 B, + posterior store 8 B per variable; c2v re-read and channel LLR come from TMEM
    smem_bytes = n_step * ITERS * (NNZ * 3 * 8 + NC * 8)
    # early-termination throughput of the same point (reported, not the headline)
    ms_et = timed(max(args.steps // 2, 1), 30_000, early_term=True)
    et_frames = n_step * world * max(args.steps // 2, 1)

    # f32 message mode (reported, not the headline)
    ctx.set_tuning(precision=api.F32)
    ctx.prepare(DECODING, ITERS, False, nframes=FRAMES_PER_STEP)
    step(40_000)
    ms_f32 = timed(max(args.steps // 2, 1), 40_001)
    ctx.set_tuning(precision=api.F64)

    # ---- end to end, HOST buffers, through the C ABI (copies inside the timed region) ----------------------------------
    #   e2e      : ldpc_b200_decode_batch_ex — this rank's frames as int8 LLRs (LLR = value * 0.25, what a quantising front
    #              end delivers) in PINNED host memory -> H2D -> 50-iteration min-sum decode -> D2H of bit-packed decisions +
    #              iteration counts; the frames are the bench workload's (AWGN -4.5 dB, produced beforehand by the channel
    #              kernel, then quantised); every frame runs the full 50 iterations.  1152 + 148 B per frame cross PCIe.
    #   e2e_f64  : ldpc_b200_decode_batch — the same frames as fp64 LLRs in, one byte per decision out (the types of the
    #              reference's own decode(), 9216 + 1156 B per frame)
    #   e2e_simulate: the reference's own sweep entry point (what `ldpcsim` / pyLDPC.simulate call): parameter structs in,
    #              result arrays out; the frames are generated on the device, so no bulk input crosses PCIe by construction
    # the int8 call decodes one bench step (FRAMES_PER_STEP frames per call and rank, like the device-timed step); the fp64 call keeps a
    # smaller batch (9216 B per frame of pinned host memory: 56832 frames = 0.5 GB per rank)
    nb8 = n_step
    nb = 148 * 4 * 96
    # NUMA placement of the caller's buffers (what a deployment does): run this rank on the cores next to its GPU while the
    # pinned buffers are allocated and first touched, so that 8 ranks do not pull their LLRs through one socket
    old_affinity = _bind_near_gpu(torch.cuda.get_device_properties(local))
    pin_in = torch.empty((nb, NC), dtype=torch.float64, pin_memory=True)
    pin_i8 = torch.empty((nb8, NC), dtype=torch.int8, pin_memory=True)
    for f0 in range(0, nb8, nb):                  # frames of the bench workload from the channel kernel, quantised piece by piece
        m = min(nb, nb8 - f0)
        _, gen = ctx.channel("AWGN", SNR_DB, 5 + rank, 0, f0, m)
        if f0 == 0:
            pin_in.numpy()[:] = gen
        pin_i8.numpy()[f0:f0 + m] = np.clip(np.rint(gen / I8_SCALE), -127, 127).astype(np.int8)
        del gen
    hw = (NC + 31) // 32
    pin_hard = torch.empty((nb, NC), dtype=torch.uint8, pin_memory=True)
    pin_bits = torch.empty((nb8, hw), dtype=torch.int32, pin_memory=True)
    pin_its = torch.empty(nb8, dtype=torch.int32, pin_memory=True)
    bits_np = pin_bits.numpy().view(np.uint32)
    reps = 3

    def run_e2e(fn):
        fn()                                          # untimed warm-up
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        t = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([t], device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = float(tt.item())
        return t

    t_f64 = run_e2e(lambda: ctx.decode_batch(pin_in.numpy(), DECODING, ITERS, False, want_llr=False, hard=pin_hard.numpy(), its=pin_its.numpy()[:nb]))
    assert int(pin_its.numpy()[:nb].min()) == ITERS and int(pin_its.numpy()[:nb].max()) == ITERS
    t_i8 = run_e2e(lambda: ctx.decode_batch_ex(pin_i8.numpy(), DECODING, ITERS, False, scale=I8_SCALE, bits=bits_np, its=pin_its.numpy()))
    assert int(pin_its.numpy().min()) == ITERS and int(pin_its.numpy().max()) == ITERS
    # parity of the narrow path inside the bench: the same quantised values fed as doubles give the same decisions
    chk = 592
    ctx.decode_batch(pin_i8.numpy()[:chk].astype(np.float64) * I8_SCALE, DECODING, ITERS, False, want_llr=False, hard=pin_hard.numpy()[:chk], its=pin_its.numpy()[:chk])
    assert np.array_equal(ctx.unpack_bits(bits_np[:chk]), pin_hard.numpy()[:chk]), "int8 path and fp64 path disagree"
    e2e_i8 = reps * nb8 * world * NCT / t_i8 / 1e9
    e2e_f64 = reps * nb * world * NCT / t_f64 / 1e9
    if old_affinity:
        os.sched_setaffinity(0, old_affinity)   # the CPU baseline below uses every host core

    sim_frames = n_step * max(args.steps // 2, 1) * world
    barrier()
    t0 = time.perf_counter()
    if world > 1:
        from libldpc_b200 import dist as D
        res = D.simulate_distributed(ctx, [SNR_DB, SNR_DB + 0.25, 0.5], decoding=DECODING, iterations=ITERS, early_term=False, seed=1,
                                     max_frames=sim_frames, fec=10 ** 12)
    else:
        res = ctx.simulate([SNR_DB, SNR_DB + 0.25, 0.5], decoding=DECODING, iterations=ITERS, early_term=False, seed=1,
                           max_frames=sim_frames, fec=10 ** 12)
    t_sim = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([t_sim], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_sim = float(t.item())
    sim_done = int(res["frames"][0])
    e2e_sim = sim_done * NCT / t_sim / 1e9

    if rank == 0:
        shape = "tile4_kernel<double,MS,SMEM,lanes=%d,TMEM>, %d CTAs/SM x %d threads" % (st["frames_per_cta"] // 2, max(1, st["ctas"] // 148), st["threads_per_cta"])
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": n_step, "sharding": f"frames x{world}",
                       "l2_policy": "no HBM-resident inputs: LLRs are generated in-kernel (Philox) and messages live in shared memory; nothing to flush",
                       "frames_per_cta": st["frames_per_cta"], "threads_per_cta": st["threads_per_cta"], "ctas": st["ctas"],
                       "residency": {1: "smem", 2: "global"}.get(st["residency"], "?"), "smem_bytes": st["smem_bytes"]},
            "frames_per_s": total_frames / (ms * 1e-3),
            "edge_updates_per_s": total_frames * ITERS * NNZ / (ms * 1e-3),
            # The messages of this code are SHARED-MEMORY resident: the bound that applies is the shared-memory pipe (SURVEY.md 8d),
            # measured in this run by an LDS.128 streaming probe.  achieved = algorithmic message bytes (4 x 8 B per edge-iteration).
            "roofline": {"bound": "smem", "achieved": achieved, "peak": smem_peak, "unit": "GB/s", "frac": achieved / smem_peak,
                         "traffic": traffic.get("headline"),
                         "peak_source": "measured in this run: ldpc_b200_smem_probe (LDS.128 streaming from all SMs)",
                         "kernel": shape, "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": alg_bytes,
                         "achieved_moved": smem_bytes / (kernel_ms * 1e-3) / 1e9, "frac_moved": smem_bytes / (kernel_ms * 1e-3) / 1e9 / smem_peak,
                         "note": "algorithmic = 32 B per edge-iteration (read v2c, write c2v, read c2v, write v2c in fp64); moved = bytes the kernel "
                                 "actually passes through shared memory (24 B per edge-iteration + 8 B per variable-iteration: v2c is never stored, "
                                 "the thread-private c2v re-read and channel LLR are served from Tensor Memory); `traffic` = DRAM bytes per launch "
                                 "(ncu), ~0 because nothing of the decode loop touches HBM",
                         "hbm_quotient": {"peak": hbm_peak, "peak_source": hbm_src, "frac": achieved / hbm_peak,
                                          "note": "the same algorithmic bytes over the measured HBM copy peak: > 1 because the messages never leave "
                                                  "the SM — not a roofline fraction, kept for comparison with HBM-resident decoders"}},
            "e2e": {"value": e2e_i8, "unit": UNIT, "h2d_bytes_per_step": int(nb8 * NC), "d2h_bytes_per_step": int(nb8 * (hw * 4 + 4)),
                    "call": "ldpc_b200_decode_batch_ex (C ABI): pinned host int8 LLR frames (LLR = value x 0.25) in -> H2D -> 50-iteration min-sum "
                            "decode on exactly those doubles -> D2H bit-packed decisions + iteration counts to pinned host memory; 3-stream "
                            "double-buffered pipeline inside the call; decisions checked against the fp64 call on the same values",
                    "frames": reps * nb8 * world, "seconds": t_i8, "h2d_gb_per_s_per_rank": reps * nb8 * NC / t_i8 / 1e9},
            "e2e_f64": {"value": e2e_f64, "unit": UNIT, "h2d_bytes_per_step": int(nb * NC * 8), "d2h_bytes_per_step": int(nb * (NC + 4)),
                        "call": "ldpc_b200_decode_batch (C ABI): the same frames as fp64 LLRs in, one byte per decision out — the types of the "
                                "reference's own decode()",
                        "frames": reps * nb * world, "seconds": t_f64, "h2d_gb_per_s_per_rank": reps * nb * NC * 8 / t_f64 / 1e9},
            "e2e_simulate": {"value": e2e_sim, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 40,
                             "call": "ldpc_b200_simulate_ex (the reference's sweep entry point behind simulate()/ldpcsim): parameter structs in, "
                                     "per-point result arrays out; frames are generated on the device; pipelined rounds",
                             "frames": sim_done, "seconds": t_sim},
            "et_on": {"value": et_frames * NCT / (ms_et * 1e-3) / 1e9, "unit": UNIT, "frames_per_s": et_frames / (ms_et * 1e-3)},
            "f32_messages": {"value": n_step * world * max(args.steps // 2, 1) * NCT / (ms_f32 * 1e-3) / 1e9, "unit": UNIT},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "counters_sample": {"fec": int(res["fec"][0]), "frames": sim_done, "fer": float(res["fer"][0]), "avg_iter": float(res["avg_iter"][0])},
        }
        if world == 1:
            try:
                line["configs"], cfg_launches = run_configs(api, smem_peak, fp64_peak, hbm_peak, traffic)
                line["gpu_launches_configs"] = cfg_launches
            except Exception as e:
                line["configs"] = {"error": str(e)}
            try:
                line["decode_single_frame"] = decode_latency()
            except Exception as e:
                line["decode_single_frame"] = {"error": str(e)}
            try:
                line["cpu_baseline"] = cpu_baseline()
            except Exception as e:  # keep the GPU line even if the host run fails
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _bind_near_gpu(prop):
    """Pins this process to the CPUs local to the GPU's PCIe root (sysfs local_cpulist); returns the previous affinity
    (None when nothing was changed)."""
    try:
        bdf = "%04x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        old = os.sched_getaffinity(0)
        cpus &= old
        if not cpus or cpus == old:
            return None
        os.sched_setaffinity(0, cpus)
        return old
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
