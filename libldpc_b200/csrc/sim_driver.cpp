// Monte-Carlo sweep driver with the reference's observable behaviour
// (src/sim/ldpcsim.cpp:97-263): half-open x list, reversed order for BSC/BEC, per-point counters,
// stop rule fec >= minFec || frames >= maxFrames || *stopFlag, results-file layout, console table,
// sim_results_t fill.  Frames are processed in (pipelined) rounds on the GPU instead of one at a time; every
// frame of every launched round is counted.  The frame -> Philox substream mapping depends only on
// (seed, point, global frame index), and each round's frame range is split contiguously over
// `world` ranks, so the totals do not depend on the number of GPUs.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "engine.hpp"

namespace b200
{
    int run_sweep(Engine &eng, const decoder_param &dp, const channel_param &cp, const simulation_param &sp,
                  sim_results_t *results, bool *stop_flag, int rank, int world, ldpc_b200_allreduce_fn allreduce,
                  void *user, bool quiet, bool write_file, ldpc_b200_round_fn round_fn)
    {
        const std::string ch = cp.type ? cp.type : "";
        if (ch != "AWGN" && ch != "BSC" && ch != "BEC" && ch != "RAYLEIGH") throw std::runtime_error("No channel selected.");
        if (world < 1 || rank < 0 || rank >= world) throw std::runtime_error("bad rank/world");
        if (world > 1 && !allreduce) throw std::runtime_error("world > 1 needs an allreduce callback");

        std::vector<double> xs; // ldpcsim.cpp:104-110 (floating-point accumulation kept as is)
        if (!(cp.xRange[2] > 0)) throw std::runtime_error("snr step must be > 0");
        for (double v = cp.xRange[0]; v < cp.xRange[1]; v += cp.xRange[2]) xs.push_back(v);
        const bool eps_axis = (ch == "BSC" || ch == "BEC");
        if (eps_axis) std::reverse(xs.begin(), xs.end()); // ldpcsim.cpp:116-122

        const uint64_t min_fec = sp.fec, max_frames = sp.maxFrames;
        std::vector<std::string> lines(xs.size() + 1);
        lines[0] = "snr fer ber frames avg_iter frame_time"; // ldpcsim.cpp:130
        const bool lead = (rank == 0);
        if (lead && !quiet)
        {
            std::cout << "========================================================================================" << std::endl;
            std::cout << "  FEC   |      FRAME     |   " << (eps_axis ? "EPS" : "SNR") << "   |    BER     |    FER     | AVGITERS  |  TIME/FRAME   \n";
            std::cout << "========+================+=========+============+============+===========+==============" << std::endl;
        }

        // Rounds.  A round is a contiguous range of global frame indices, split contiguously over the ranks.  Its size is a
        // multiple of 9472 = 148 x 64 frames — whole waves of every persistent-grid shape of the kernels (148 or 296 CTAs x 2 ... 16
        // frames) for 1, 2, 4 or 8 ranks — doubling while no error has been seen and then steered towards the remaining error
        // budget.  The rounds are PIPELINED: round k+1 is issued before the counters of round k are read (two slots on the
        // engine's stream), so the device never waits for the host, the all-reduce or the results file; the stop rule therefore
        // acts one round late and every frame of every issued round is counted (bounded overshoot, unbiased).  The schedule
        // depends only on reduced counters — not on the number of ranks or shards, the kernel shape or who processes the
        // frames (GPU launch or injected callback) — so 1 GPU and N GPUs produce the same counters.
        const bool pipelined = round_fn == nullptr;
        if (pipelined && ch != "BEC") eng.prepare(dp, max_frames); // the one-off shape trial (large jobs only)
        const uint64_t wave = 9472;
        auto whole_waves = [&](uint64_t n) { return std::max<uint64_t>((n + wave / 2) / wave, 1) * wave; };
        const uint64_t round0 = wave, round_cap = whole_waves(1ull << 22);
        for (size_t i = 0; i < xs.size(); ++i)
        {
            uint64_t fec = 0, bec = 0, frames = 0, iters = 0, cursor = 0; // cursor: frames launched so far
            uint64_t round = round0;
            const auto t0 = std::chrono::high_resolution_clock::now();
            bool stop = false, stopped = false;
            struct Pending { bool live = false; uint64_t n_this = 0, lo = 0, hi = 0; } pend[2];
            int k = 0;
            auto launch_round = [&](int slot) -> bool
            { // launches the next round into `slot` unless the frame budget is used up
                const uint64_t n_this = std::min<uint64_t>(round, max_frames > cursor ? max_frames - cursor : 0);
                if (n_this == 0) return false;
                Pending &pd = pend[slot];
                pd.live = true;
                pd.n_this = n_this;
                pd.lo = cursor + n_this * (uint64_t)rank / (uint64_t)world;
                pd.hi = cursor + n_this * (uint64_t)(rank + 1) / (uint64_t)world;
                cursor += n_this;
                if (pipelined && pd.hi > pd.lo) eng.round_launch(slot, dp, ch, xs[i], cp.seed, (uint32_t)i, pd.lo, pd.hi - pd.lo);
                return true;
            };
            launch_round(0);
            while (pend[k & 1].live)
            {
                Pending &pd = pend[k & 1];
                // keep the device busy: the following round goes out before this one is read (not known to be needed yet)
                if (!stop) launch_round((k + 1) & 1);
                uint64_t c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                if (pd.hi > pd.lo)
                {
                    if (round_fn)
                    {
                        if (round_fn((uint32_t)i, xs[i], pd.lo, pd.hi - pd.lo, c, user) != 0) throw std::runtime_error("round callback failed");
                    }
                    else eng.round_collect(k & 1, c);
                }
                pd.live = false;
                c[5] = (stop_flag && *stop_flag) ? 1 : 0;
                if (world > 1) allreduce(c, 8, user);
                stopped = stopped || c[5] != 0; // the REDUCED flag: every rank leaves the sweep at the same place
                fec += c[0]; bec += c[1]; frames += c[2]; iters += c[3];
                const bool new_errors = c[0] > 0;
                if (new_errors)
                { // what the reference does inside its critical section at every frame error, ldpcsim.cpp:190-249
                    const auto now = std::chrono::high_resolution_clock::now();
                    const uint64_t us = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(now - t0).count();
                    const uint64_t t_frame = us / frames;
                    const double fer = (double)fec / frames;
                    const double ber = (double)bec / ((double)frames * eng.H.nc); // denominator nc, ldpcsim.cpp:204
                    const double avg_it = (double)iters / frames;
                    if (lead && !quiet)
                    {
                        printf("\r %2lu/%2lu  |  %12lu  |  %.3f  |  %.2e  |  %.2e  |  %.1e  |  %.3fms", (unsigned long)fec, (unsigned long)min_fec,
                               (unsigned long)frames, xs[i], ber, fer, avg_it, (double)t_frame * 1e-3);
                        fflush(stdout);
                    }
                    char buf[160];
                    snprintf(buf, sizeof(buf), "%lf %.3e %.3e %lu %.3e %.6f", xs[i], fer, ber, (unsigned long)frames, avg_it, (double)t_frame * 1e-6);
                    lines[i + 1] = buf;
                    if (lead && write_file && sp.resultFile && sp.resultFile[0])
                    {
                        std::ofstream fp(sp.resultFile);
                        if (fp.good()) for (const auto &l : lines) fp << l << "\n";
                        else printf("Warning: can not open logfile for writing\n");
                    }
                    if (results)
                    {
                        results->fer[i] = fer;
                        results->ber[i] = ber;
                        results->avg_iter[i] = avg_it;
                        results->time[i] = (double)t_frame * 1e-6;
                        results->fec[i] = fec;
                        results->frames[i] = frames;
                    }
                }
                stop = stop || (fec >= min_fec) || (frames >= max_frames) || stopped; // ldpcsim.cpp:255
                if (fec == 0) round = std::min(whole_waves(round * 2), round_cap);
                else
                {
                    const double need = (double)(min_fec > fec ? min_fec - fec : 0) * ((double)frames / (double)fec) * 1.2;
                    round = whole_waves((uint64_t)std::min<double>(std::max<double>(need, (double)round0), (double)round_cap));
                }
                ++k;
            }
            if (lead && !quiet) printf("\n");
            if (stopped) break;
        }
        return 0;
    }
} // namespace b200
