// Layered-schedule decode kernel (opt-in; SURVEY.md 8f row 4).  The schedule is the legacy tree's layer loop
// (gpu/device/kernel.cpp:52-75: check update of one layer, a-posteriori update, next layer) with the check-node rules of the live
// decoder (forward/backward recursion with box-plus or min-sum, src/decoding/decoder.cpp:30-44); oracle/ldpc_oracle.c
// orc_decode_layered is its specification and the parity tests compare against it bit for bit (min-sum).  Results differ from
// the flooding reference BY DESIGN (about half the iterations at equal error rate), so it is never the default.
//
// State per frame lane: c2v per edge slot and the posterior `out` per variable; neither v2c nor the channel LLR is kept:
//   v2c = out - c2v_old;  c2v_new = check rule(v2c of the other edges);  out = v2c + c2v_new        (all inside the check's thread)
// A layer never contains two checks that share a variable (validated on the host), so the in-place posterior update is race
// free and ONE barrier per layer is all the synchronisation there is; there is no variable phase.  Early termination is tested
// once per iteration by a gather-only syndrome pass over all checks.
//
// Mapping: as in tile4.cuh — 16-byte vectors of VEC frame lanes, LANES warp lanes per node, NPW = 32/LANES checks of equal degree
// per warp task, per-(layer, warp) task lists stored as run-length segments.  Frames run in lock step per CTA (a batch of
// LANES*VEC frames starts and retires together; converged lanes are frozen by masked stores).  Global residency only (the mode
// is for quasi-cyclic codes of the 5G NR kind, whose state does not fit shared memory).
#pragma once
#include "tile4.cuh"

namespace b200
{
    struct LayParams
    {
        const uint32_t *seg;   // [(layer * warps + warp) * max_segs + s][4]: {degree | nodes << 8 | tasks << 16, first slot, 0, 0}; first word 0 ends a list
        const uint32_t *idx;   // [n_slots] byte offset of the out record gathered by the slot's edge (variable id * 16 * LANES)
        int n_layers, max_segs, n_slots, nc, nct, n_punct, n_short;
        const int32_t *tx_var, *punct, *shorten; // variable ids
        int max_iter, early_term, kind;
        const double *llr_in;
        double sigma, llr_scale, delta;
        double ms_scale; // normalisation factor of the min-sum check output (1 = the reference's plain min-sum)
        uint32_t thr;
        uint64_t seed;
        uint32_t point;
        uint64_t frame0, n_frames;
        double *llr_out;
        uint8_t *hard_out;
        int32_t *iters_out;
        unsigned long long *counters; // [5]
        unsigned long long *err_log, *err_count;
        unsigned long long err_cap;
        unsigned char *state;
        size_t state_stride;
    };

    // One check of degree `deg`: thread (node j, vector sub).  slot0 = first slot of the node (slot of edge k = slot0 + k * NPW).
    // fz: lanes whose old c2v counts as +0 (first visit); live: lanes that may be written (the others are frozen: converged).
    template <typename T, int ALG, int LANES>
    __device__ __forceinline__ void cn_lay(unsigned char *out_sub, unsigned char *c2v_sub, const uint32_t *__restrict__ idx, uint32_t slot0, int deg,
                                           uint32_t fz, uint32_t live, T ms_scale)
    {
        typedef Vec<T> V;
        constexpr int VEC = V::N, NPW = 32 / LANES, RS = 16 * LANES, TS = (int)sizeof(T);
        constexpr uint32_t VMASK = (1u << VEC) - 1u;
        auto load_v = [&](int k, uint32_t &eo) -> V
        {
            const uint32_t s = slot0 + (uint32_t)k * NPW;
            eo = __ldg(idx + s);
            const V o = *reinterpret_cast<const V *>(out_sub + eo);
            V c = *reinterpret_cast<const V *>(c2v_sub + (size_t)s * RS);
            V v;
#pragma unroll
            for (int e = 0; e < VEC; ++e) v.e[e] = o.e[e] - (((fz >> e) & 1u) ? T(0) : c.e[e]);
            return v;
        };
        auto store = [&](int k, uint32_t eo, const V &v, const V &r)
        { // c2v = r, out = v2c + c2v (the posterior update of gpu/device/kernel.cpp:272-296, in place)
            const uint32_t s = slot0 + (uint32_t)k * NPW;
            V o;
#pragma unroll
            for (int e = 0; e < VEC; ++e) o.e[e] = v.e[e] + r.e[e];
            if (live == VMASK)
            {
                *reinterpret_cast<V *>(c2v_sub + (size_t)s * RS) = r;
                *reinterpret_cast<V *>(out_sub + eo) = o;
            }
            else
            {
#pragma unroll
                for (int e = 0; e < VEC; ++e)
                    if ((live >> e) & 1u)
                    {
                        *reinterpret_cast<T *>(c2v_sub + (size_t)s * RS + e * TS) = r.e[e];
                        *reinterpret_cast<T *>(out_sub + eo + e * TS) = o.e[e];
                    }
            }
        };
        if (ALG == ALG_MS)
        { // exact minimum over the other edges, XOR of sign bits (= the F/B recursion with f = sign*sign*min for every input)
            T m1[VEC], m2[VEC];
            int arg[VEC];
            unsigned long long smask[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) { m1[e] = Num<T>::inf(); m2[e] = Num<T>::inf(); arg[e] = 0; smask[e] = 0; }
            for (int k = 0; k < deg; ++k)
            {
                uint32_t eo;
                const V v = load_v(k, eo);
#pragma unroll
                for (int e = 0; e < VEC; ++e)
                {
                    smask[e] |= (unsigned long long)(Num<T>::hi(v.e[e]) >> 31) << k;
                    const bool lt1 = Num<T>::abs(v.e[e]) < Num<T>::abs(m1[e]), lt2 = Num<T>::abs(v.e[e]) < Num<T>::abs(m2[e]);
                    m2[e] = lt1 ? m1[e] : (lt2 ? v.e[e] : m2[e]);
                    arg[e] = lt1 ? k : arg[e];
                    m1[e] = lt1 ? v.e[e] : m1[e];
                }
            }
            uint32_t tot[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) tot[e] = (uint32_t)__popcll(smask[e]) & 1u;
            for (int k = 0; k < deg; ++k)
            {
                uint32_t eo;
                const V v = load_v(k, eo); // the same operands as in the first pass: the same value
                V r;
#pragma unroll
                for (int e = 0; e < VEC; ++e)
                {
                    const uint32_t sg = tot[e] ^ (uint32_t)((smask[e] >> k) & 1ull);
                    r.e[e] = mag_sign(((k == arg[e]) ? m2[e] : m1[e]) * ms_scale, sg << 31); // x 1 is exact: plain min-sum unchanged
                }
                store(k, eo, v, r);
            }
        }
        else
        { // forward/backward box-plus recursion, file order (decoder.cpp:30-44)
            V v[64], F[64];
            uint32_t eo[64];
            for (int k = 0; k < deg; ++k) v[k] = load_v(k, eo[k]);
            if constexpr (sizeof(T) == 8 && B200_BP_EDOMAIN)
            {
                // fp64: the same function of the inputs on E = e^-|x| (kernels.cuh bp_check; arbitrary degree as in tile4.cuh
                // cn4_any): d exponentials, forward / backward values as plain numbers, d logarithms of the joined fractions.
                // All outputs are formed before the first in-place store, so the rare exact path below can still take over.
                if (deg >= 3)
                {
                    unsigned long long smask[VEC];
                    double shift[VEC];
                    V Ek[64], R[64];
#pragma unroll
                    for (int e = 0; e < VEC; ++e)
                    {
                        uint32_t mh = 0x7fffffffu;
                        smask[e] = 0;
                        for (int k = 0; k < deg; ++k)
                        {
                            const uint32_t h = Num<T>::hi(v[k].e[e]);
                            smask[e] |= (unsigned long long)(h >> 31) << k;
                            mh = min(mh, h & 0x7fffffffu);
                        }
                        shift[e] = (mh >= 0x40440000u && mh < 0x7ff00000u) ? __hiloint2double((int)mh, 0) - 40.0 : 0.0;
                    }
                    for (int k = 0; k < deg; ++k)
                    {
#pragma unroll
                        for (int e = 0; e < VEC; ++e) Ek[k].e[e] = bp_exp_neg(fabs(v[k].e[e]) - shift[e]);
                        if (k == 0) F[0] = Ek[0];
                        else if (k < deg - 1)
                        {
#pragma unroll
                            for (int e = 0; e < VEC; ++e) F[k].e[e] = bp_join(F[k - 1].e[e], Ek[k].e[e]);
                        }
                    }
                    bool anyfar = false, far;
                    V B = Ek[deg - 1];
                    for (int k = deg - 1; k >= 0; --k)
                    {
#pragma unroll
                        for (int e = 0; e < VEC; ++e)
                        {
                            double N, Dn;
                            if (k == deg - 1) { N = F[deg - 2].e[e]; Dn = 1.0; }
                            else if (k == 0) { N = B.e[e]; Dn = 1.0; }
                            else { N = F[k - 1].e[e] + B.e[e]; Dn = __fma_rn(F[k - 1].e[e], B.e[e], 1.0); }
                            const double l = bp_log_frac(N, Dn, shift[e], far);
                            anyfar |= far;
                            const uint32_t sg = (((uint32_t)__popcll(smask[e]) ^ (uint32_t)(smask[e] >> k)) & 1u) << 31;
                            R[k].e[e] = __hiloint2double((int)(((uint32_t)__double2hiint(l) & 0x7fffffffu) | sg), __double2loint(l));
                            if (k > 0 && k < deg - 1) B.e[e] = bp_join(B.e[e], Ek[k].e[e]);
                        }
                    }
                    if (!anyfar)
                    {
                        for (int k = deg - 1; k >= 0; --k) store(k, eo[k], v[k], R[k]);
                        return;
                    }
                }
            }
            F[0] = v[0];
            for (int k = 1; k < deg; ++k)
            {
#pragma unroll
                for (int e = 0; e < VEC; ++e) F[k].e[e] = boxplus(F[k - 1].e[e], v[k].e[e]);
            }
            V B = v[deg - 1];
            store(deg - 1, eo[deg - 1], v[deg - 1], F[deg - 2]);
            for (int k = deg - 2; k >= 1; --k)
            {
                V r;
#pragma unroll
                for (int e = 0; e < VEC; ++e) r.e[e] = boxplus(F[k - 1].e[e], B.e[e]);
                store(k, eo[k], v[k], r);
#pragma unroll
                for (int e = 0; e < VEC; ++e) B.e[e] = boxplus(B.e[e], v[k].e[e]);
            }
            store(0, eo[0], v[0], B);
        }
    }

    // parity of the hard decisions of one check's variables, per frame lane of the vector (decoder.h:47-64)
    template <typename T, int LANES>
    __device__ __forceinline__ uint32_t synd_lay(const unsigned char *out_sub, const uint32_t *__restrict__ idx, uint32_t slot0, int deg)
    {
        typedef Vec<T> V;
        constexpr int VEC = V::N, NPW = 32 / LANES;
        uint32_t par = 0;
        for (int k = 0; k < deg; ++k)
        {
            const V o = *reinterpret_cast<const V *>(out_sub + __ldg(idx + slot0 + (uint32_t)k * NPW));
#pragma unroll
            for (int e = 0; e < VEC; ++e) par ^= (o.e[e] <= T(0)) ? (1u << e) : 0u;
        }
        return par;
    }

    template <typename T, int ALG, int LANES>
    __global__ void __launch_bounds__(512, 1) lay_kernel(const LayParams p)
    {
        typedef Vec<T> V;
        constexpr int VEC = V::N, FPC = LANES * VEC, NPW = 32 / LANES, RS = 16 * LANES, TS = (int)sizeof(T);
        constexpr uint32_t VMASK = (1u << VEC) - 1u;
        __shared__ uint32_t s_synd[2], s_err[FPC];
        __shared__ unsigned long long s_cnt[5];
        const int tid = threadIdx.x, nthreads = blockDim.x, lane = tid & 31, warp = tid >> 5, warps = nthreads >> 5;
        const int sub = lane & (LANES - 1), j = lane / LANES;
        unsigned char *c2v = p.state + p.state_stride * blockIdx.x;
        unsigned char *out = c2v + (size_t)RS * p.n_slots;
        unsigned char *out_sub = out + sub * 16, *c2v_sub = c2v + sub * 16;
        if (tid < 5) s_cnt[tid] = 0;
        if (tid < 2) s_synd[tid] = 0;
        if (tid < FPC) s_err[tid] = 0;
        __syncthreads();

        // every segment of this warp in layer l: f(degree, nodes in the task, first slot of the thread's node)
        auto for_tasks = [&](int l, auto &&f)
        {
            const uint32_t *sp = p.seg + 4 * ((size_t)(l * warps + warp) * p.max_segs);
            for (;; sp += 4)
            {
                const uint4 sg = __ldg(reinterpret_cast<const uint4 *>(sp));
                if (sg.x == 0) break;
                const int deg = (int)(sg.x & 0xFFu), cnt = (int)((sg.x >> 8) & 0xFFu);
                uint32_t slot0 = sg.y + (uint32_t)j;
                for (int nt = (int)(sg.x >> 16); nt > 0; --nt, slot0 += (uint32_t)deg * NPW)
                    if (j < cnt) f(deg, slot0);
            }
        };

        const int nblk = (p.nct + 3) >> 2;
        for (unsigned long long batch = blockIdx.x; batch * FPC < p.n_frames; batch += gridDim.x)
        {
            const unsigned long long f0 = batch * FPC;
            const uint32_t valid = (p.n_frames - f0 >= FPC) ? ((FPC == 32) ? 0xFFFFFFFFu : ((1u << FPC) - 1u)) : ((1u << (uint32_t)(p.n_frames - f0)) - 1u);
            // ---- decoder input = the initial posterior (channel specification as in tile4.cuh frame_pass; all-zero codeword) ----
            for (int g = 0; g < FPC; ++g)
            {
                unsigned char *dst = out + (g / VEC) * 16 + (g % VEC) * TS;
                auto put = [&](int var, T v) { *reinterpret_cast<T *>(dst + (size_t)var * RS) = v; };
                if (!((valid >> g) & 1u))
                {
                    for (int i = tid; i < p.nc; i += nthreads) put(i, T(1));
                    continue;
                }
                if (p.kind == SRC_LLR)
                {
                    const double *src = p.llr_in + (size_t)(f0 + g) * p.nc;
                    for (int i = tid; i < p.nc; i += nthreads) put(i, (T)src[i]);
                    continue;
                }
                const unsigned long long frame = p.frame0 + f0 + g;
                for (int q = tid; q < nblk; q += nthreads)
                {
                    const u32x4 r = channel_block(p.seed, p.point, 0, frame, (uint32_t)q);
                    if (p.kind == SRC_AWGN)
                    {
                        float z[4];
                        normal_pair(r.x, r.y, z[0], z[1]);
                        normal_pair(r.z, r.w, z[2], z[3]);
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (q + k * nblk < p.nct) put(p.tx_var[q + k * nblk], (T)__dmul_rn(__dadd_rn(__dmul_rn((double)z[k], p.sigma), 1.0), p.llr_scale));
                    }
                    else
                    {
                        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (q + k * nblk < p.nct) put(p.tx_var[q + k * nblk], (T)((w[k] < p.thr) ? -p.delta : p.delta));
                    }
                }
                for (int i = tid; i < p.n_punct; i += nthreads) put(p.punct[i], T(0));
                for (int i = tid; i < p.n_short; i += nthreads) put(p.shorten[i], (T)(p.kind == SRC_AWGN ? 99999.9 : p.delta));
            }
            __syncthreads();

            uint32_t live = valid;       // CTA-uniform: lanes still decoding
            int ret[FPC];                // CTA-uniform: reference iteration count per lane
#pragma unroll
            for (int g = 0; g < FPC; ++g) ret[g] = p.max_iter;
            unsigned long long executed = 0;
            for (int it = 0; it < p.max_iter && live; ++it)
            {
                const uint32_t mylive = (live >> (sub * VEC)) & VMASK, fz = (it == 0) ? VMASK : 0u;
                for (int l = 0; l < p.n_layers; ++l)
                {
                    for_tasks(l, [&](int deg, uint32_t slot0) { cn_lay<T, ALG, LANES>(out_sub, c2v_sub, p.idx, slot0, deg, fz, mylive, (T)p.ms_scale); });
                    __syncthreads(); // the next layer reads the posteriors this one wrote
                }
                executed += (unsigned long long)__popc(live);
                if (p.early_term)
                {
                    uint32_t bad = 0;
                    for (int l = 0; l < p.n_layers; ++l)
                        for_tasks(l, [&](int deg, uint32_t slot0) { bad |= synd_lay<T, LANES>(out_sub, p.idx, slot0, deg); });
                    const uint32_t m = __reduce_or_sync(0xffffffffu, bad << (sub * VEC));
                    if (lane == 0 && m) atomicOr(&s_synd[it & 1], m);
                    __syncthreads();
                    const uint32_t conv = live & ~s_synd[it & 1]; // decoder.cpp:66-72: stop BEFORE ++I
                    if (tid == 0) s_synd[(it + 1) & 1] = 0;       // read two barriers ago
#pragma unroll
                    for (int g = 0; g < FPC; ++g)
                        if ((conv >> g) & 1u) ret[g] = it;
                    live &= ~conv;
                }
            }
            // ---- retire the batch: bit errors over the transmitted positions (ldpcsim.cpp:184-190), outputs, counters ----
            for (int g = 0; g < FPC; ++g)
                if ((valid >> g) & 1u)
                {
                    const unsigned char *src = out + (g / VEC) * 16 + (g % VEC) * TS;
                    uint32_t n = 0;
                    for (int i = tid; i < p.nct; i += nthreads) n += (*reinterpret_cast<const T *>(src + (size_t)p.tx_var[i] * RS) <= T(0)) ? 1u : 0u;
                    n = __reduce_add_sync(0xffffffffu, n);
                    if (lane == 0 && n) atomicAdd(&s_err[g], n);
                    if (p.llr_out || p.hard_out)
                    {
                        const size_t o = (size_t)(f0 + g) * p.nc;
                        for (int i = tid; i < p.nc; i += nthreads)
                        {
                            const T v = *reinterpret_cast<const T *>(src + (size_t)i * RS);
                            if (p.llr_out) p.llr_out[o + i] = (double)v;
                            if (p.hard_out) p.hard_out[o + i] = (v <= T(0)) ? 1 : 0;
                        }
                    }
                    if (tid == 0 && p.iters_out) p.iters_out[f0 + g] = ret[g];
                }
            __syncthreads();
            if (tid == 0)
            {
                unsigned long long fec = 0, bec = 0, rs = 0;
                for (int g = 0; g < FPC; ++g)
                    if ((valid >> g) & 1u)
                    {
                        const uint32_t e = s_err[g];
                        fec += e ? 1 : 0; bec += e; rs += (unsigned long long)ret[g];
                        if (e && p.err_log)
                        {
                            const unsigned long long slot = atomicAdd(p.err_count, 1ull);
                            if (slot < p.err_cap)
                            {
                                p.err_log[2 * slot] = p.frame0 + f0 + g;
                                p.err_log[2 * slot + 1] = (unsigned long long)e | ((unsigned long long)(uint32_t)ret[g] << 32);
                            }
                        }
                        s_err[g] = 0;
                    }
                s_cnt[0] += fec; s_cnt[1] += bec; s_cnt[2] += (unsigned long long)__popc(valid); s_cnt[3] += rs; s_cnt[4] += executed;
            }
            __syncthreads();
        }
        if (tid < 5 && s_cnt[tid]) atomicAdd(&p.counters[tid], s_cnt[tid]);
    }

    // the layered kernel for (precision, algorithm, lanes per node: 2 or 4); layered.cu instantiates them
    const void *layered_kernel(bool f32, int alg, int lanes);
} // namespace b200
