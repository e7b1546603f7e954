// Error report of replayed frames (ldpc_b200_error_report): for every frame, the transmitted positions whose decision differs
// from the transmitted word (in transmitted order) and the checks the decisions leave unsatisfied (ascending).  One warp per
// frame, 32 positions / checks per step, order-preserving compaction by ballot.  Two launches: COUNT writes the per-frame
// counts, the host scans them into offsets, WRITE fills the lists at those offsets (CSR output, no per-frame worst-case
// buffers).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b200
{
    struct ReportParams
    {
        const uint8_t *hard;    // [n][nc] replayed decisions
        const uint8_t *cw;      // [n][nc] transmitted word; null = the all-zero word (M-ASK: the decoder sees the descrambled frame)
        const int32_t *bit_pos; // [nct] transmitted positions
        const int32_t *chk_ptr; // [mc + 1] check-major CSR of H ...
        const int32_t *chk_var; // [nnz] ... variable of every edge
        int nc, nct, mc;
        int64_t n;
        uint32_t *counts;        // COUNT: [n][2] bit errors, syndrome weight
        const int64_t *offsets;  // WRITE: [n][2] where the frame's failed bits / failed checks start
        int32_t *failed_bits, *failed_checks;
    };

    template <bool WRITE>
    __global__ void __launch_bounds__(256) report_kernel(ReportParams p)
    {
        const int lane = threadIdx.x & 31;
        const uint32_t below = (1u << lane) - 1u;
        const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
        for (int64_t f = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); f < p.n; f += warps)
        {
            const uint8_t *h = p.hard + f * p.nc;
            const uint8_t *c = p.cw ? p.cw + f * p.nc : nullptr;
            int32_t *bits = WRITE ? p.failed_bits + p.offsets[2 * f] : nullptr;
            int32_t *checks = WRITE ? p.failed_checks + p.offsets[2 * f + 1] : nullptr;
            uint32_t nb = 0, nk = 0;
            for (int t0 = 0; t0 < p.nct; t0 += 32)
            {
                const int t = t0 + lane;
                int v = 0;
                bool bad = false;
                if (t < p.nct)
                {
                    v = p.bit_pos[t];
                    bad = h[v] != (c ? c[v] : (uint8_t)0);
                }
                const uint32_t m = __ballot_sync(0xffffffffu, bad);
                if (WRITE && bad) bits[nb + __popc(m & below)] = v;
                nb += __popc(m);
            }
            for (int k0 = 0; k0 < p.mc; k0 += 32)
            {
                const int k = k0 + lane;
                uint32_t s = 0;
                if (k < p.mc)
                    for (int e = p.chk_ptr[k]; e < p.chk_ptr[k + 1]; ++e) s ^= h[p.chk_var[e]];
                const bool bad = s != 0;
                const uint32_t m = __ballot_sync(0xffffffffu, bad);
                if (WRITE && bad) checks[nk + __popc(m & below)] = k;
                nk += __popc(m);
            }
            if (!WRITE && lane == 0)
            {
                p.counts[2 * f] = nb;
                p.counts[2 * f + 1] = nk;
            }
        }
    }
} // namespace b200
