// sm_100a decode kernel, vector-tile mapping over run-length SEGMENTS: Philox channel -> flooding
// min-sum / box-plus decode -> hard decision + error accounting, fused into ONE persistent kernel.
//
// Mapping.  A CTA keeps FPC = LANES * VEC frames in flight (VEC = 16/sizeof(T): 2 doubles or 4
// floats).  Every per-frame array is stored as 16-byte vectors of VEC adjacent frame lanes,
// [index][LANES] vectors per index ("records" of RS = 16*LANES bytes).  One thread owns ONE vector of
// one node: warp lane l serves node l / LANES of the warp's current task and vector l % LANES, so a warp
// walking the NPW = 32/LANES nodes of a task moves 512 contiguous bytes per access (conflict free in
// shared memory, whole sectors in HBM/L2) with one LDS.128/STS.128 (LDG/STG.128) per VEC messages, and
// every index load / address computation is shared by VEC frames.
//
// Work list (SegLayout, code.cpp).  Nodes of equal degree are packed NPW at a time into warp tasks and
// the tasks of a warp are stored run-length encoded as segments; message slots, variable positions and
// index entries are numbered in that order.  A warp therefore decodes one 16-byte descriptor per
// SEGMENT, dispatches once on the (warp-uniform) degree to a fully unrolled body and then only advances
// two pointers by compile-time strides per task.  A node's index entries are contiguous, pre-scaled to
// byte offsets, and fetched with one vector load.
//
// State per frame lane: c2v per edge slot, posterior `out` and channel LLR per variable position.
// v2c is never stored — it is recomputed as out - c2v, which is exactly the value the reference
// stores (src/decoding/decoder.cpp:60-63), so results stay bit-identical while one of the
// reference's two message arrays disappears.  A fresh frame starts with c2v = +0 and out = LLRin,
// which makes its first check pass read LLRin exactly (x - (+0) == x for every x, -0 included),
// i.e. decoder.cpp:16-19 without a special case.
//
// A frame lane that finishes (syndrome clear after an iteration, or iteration limit) is retired —
// its bit errors are counted once, from the final posterior (src/sim/ldpcsim.cpp:184-190) — and
// refilled at once with the next frame (LLRs regenerated from the counter-based Philox stream), so
// early termination never leaves lanes idle waiting for the slowest frame of a batch.
#pragma once
#include <cstdio>
#include <utility>

#include "kernels.cuh"

namespace b200
{
    // ------------------------------------------------------------------------------------------
    // 16-byte vectors of frame lanes
    // ------------------------------------------------------------------------------------------
    template <typename T> struct Vec;
    template <> struct __align__(16) Vec<double> { static constexpr int N = 2; double e[2]; };
    template <> struct __align__(16) Vec<float> { static constexpr int N = 4; float e[4]; };

    template <bool SMEM, typename T, int OFF> struct VAcc;
    template <int OFF> struct VAcc<true, double, OFF>
    {
        static __device__ __forceinline__ Vec<double> ld(uint32_t a)
        {
            Vec<double> v;
            asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+%3];" : "=d"(v.e[0]), "=d"(v.e[1]) : "r"(a), "n"(OFF));
            return v;
        }
        static __device__ __forceinline__ void st(uint32_t a, const Vec<double> &v)
        {
            asm volatile("st.shared.v2.f64 [%0+%1], {%2, %3};" ::"r"(a), "n"(OFF), "d"(v.e[0]), "d"(v.e[1]) : "memory");
        }
    };
    template <int OFF> struct VAcc<true, float, OFF>
    {
        static __device__ __forceinline__ Vec<float> ld(uint32_t a)
        {
            Vec<float> v;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];" : "=f"(v.e[0]), "=f"(v.e[1]), "=f"(v.e[2]), "=f"(v.e[3]) : "r"(a), "n"(OFF));
            return v;
        }
        static __device__ __forceinline__ void st(uint32_t a, const Vec<float> &v)
        {
            asm volatile("st.shared.v4.f32 [%0+%1], {%2, %3, %4, %5};" ::"r"(a), "n"(OFF), "f"(v.e[0]), "f"(v.e[1]), "f"(v.e[2]), "f"(v.e[3]) : "memory");
        }
    };
    template <typename T, int OFF> struct VAcc<false, T, OFF>
    {
        static __device__ __forceinline__ Vec<T> ld(const unsigned char *a) { return *reinterpret_cast<const Vec<T> *>(a + OFF); }
        static __device__ __forceinline__ void st(unsigned char *a, const Vec<T> &v) { *reinterpret_cast<Vec<T> *>(a + OFF) = v; }
    };

    // read-only words (tables): 4 / 8 / 16 bytes
    template <bool SMEM, int OFF> struct WAcc;
    template <int OFF> struct WAcc<true, OFF>
    {
        static __device__ __forceinline__ uint32_t ld1(uint32_t a) { return lds_u32<OFF>(a); }
        static __device__ __forceinline__ uint2 ld2(uint32_t a)
        {
            uint2 v;
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+%3];" : "=r"(v.x), "=r"(v.y) : "r"(a), "n"(OFF));
            return v;
        }
        static __device__ __forceinline__ uint4 ld4(uint32_t a)
        {
            uint4 v;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4+%5];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a), "n"(OFF));
            return v;
        }
    };
    template <int OFF> struct WAcc<false, OFF>
    {
        static __device__ __forceinline__ uint32_t ld1(const unsigned char *a) { return __ldg(reinterpret_cast<const uint32_t *>(a + OFF)); }
        static __device__ __forceinline__ uint2 ld2(const unsigned char *a) { return __ldg(reinterpret_cast<const uint2 *>(a + OFF)); }
        static __device__ __forceinline__ uint4 ld4(const unsigned char *a) { return __ldg(reinterpret_cast<const uint4 *>(a + OFF)); }
    };

    // ------------------------------------------------------------------------------------------
    // Tensor Memory as thread-private scratch.  tcgen05.ld/st with shape 32x32b.x4: thread i of a warp
    // moves four 32-bit columns of TMEM lane (warp % 4) * 32 + i, i.e. one 16-byte vector per thread and
    // instruction, on a data path separate from shared memory (LDTM / STTM).  Used as a write-through
    // mirror of the two arrays only their owning thread ever reads back (a check task's own c2v slots, a
    // variable task's channel LLR), which takes those reads off the shared-memory pipe that bounds the kernel.
    // ------------------------------------------------------------------------------------------
    template <typename T> struct TmAcc;
    template <> struct TmAcc<double>
    {
        static __device__ __forceinline__ Vec<double> ld(uint32_t taddr)
        {
            uint32_t a, b, c, d;
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(taddr) : "memory");
            Vec<double> v;
            v.e[0] = __hiloint2double((int)b, (int)a);
            v.e[1] = __hiloint2double((int)d, (int)c);
            return v;
        }
        static __device__ __forceinline__ void st(uint32_t taddr, const Vec<double> &v)
        {
            asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(__double2loint(v.e[0])), "r"(__double2hiint(v.e[0])),
                         "r"(__double2loint(v.e[1])), "r"(__double2hiint(v.e[1]))
                         : "memory");
        }
    };
    template <> struct TmAcc<float>
    {
        static __device__ __forceinline__ Vec<float> ld(uint32_t taddr)
        {
            Vec<float> v;
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=f"(v.e[0]), "=f"(v.e[1]), "=f"(v.e[2]), "=f"(v.e[3]) : "r"(taddr) : "memory");
            return v;
        }
        static __device__ __forceinline__ void st(uint32_t taddr, const Vec<float> &v)
        {
            asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "f"(v.e[0]), "f"(v.e[1]), "f"(v.e[2]), "f"(v.e[3]) : "memory");
        }
    };
    // a segment descriptor is the same in every lane (one address per warp): say so with a broadcast, so that the degree
    // dispatch, the task loop and the TMEM addresses derived from it are uniform-datapath work
    __device__ __forceinline__ uint4 uniform4(uint4 v)
    {
        v.x = __shfl_sync(0xFFFFFFFFu, v.x, 0); v.y = __shfl_sync(0xFFFFFFFFu, v.y, 0);
        v.z = __shfl_sync(0xFFFFFFFFu, v.z, 0); v.w = __shfl_sync(0xFFFFFFFFu, v.w, 0);
        return v;
    }
    __device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
    __device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

    // Lock-step kernel (TM, ET = false): every thread keeps the shared-memory address of each gather of its tasks in its TMEM
    // lane.  A task of degree D owns W = D rounded up to a power of two columns (one tcgen05.ld.32x32b.xW); the generic-degree
    // bodies (checks above 8, variables above 16 or of degree 0) own none and keep reading the index tables.
    __host__ __device__ constexpr int ls_idx_cols(bool check, int deg)
    {
        if (check ? (deg < 2 || deg > 8) : (deg < 1 || deg > 16)) return 0;
        int w = 1;
        while (w < deg) w <<= 1;
        return w;
    }
    // segment descriptors the lock-step kernel takes from its parameters (K4Params::ls_seg): check lists, then variable lists
    constexpr int K4_LS_SEGS = 128;
    template <int D> __device__ __forceinline__ void tm_ld_idx(uint32_t taddr, uint32_t (&e)[D])
    {
        constexpr int W = ls_idx_cols(false, D);
        uint32_t w[W];
        if constexpr (W == 1) asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(w[0]) : "r"(taddr) : "memory");
        else if constexpr (W == 2) asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(w[0]), "=r"(w[1]) : "r"(taddr) : "memory");
        else if constexpr (W == 4)
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(taddr) : "memory");
        else if constexpr (W == 8)
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                         : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "r"(taddr) : "memory");
        else
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                         : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]),
                           "=r"(w[8]), "=r"(w[9]), "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15])
                         : "r"(taddr) : "memory");
#pragma unroll
        for (int k = 0; k < D; ++k) e[k] = w[k];
    }
    __device__ __forceinline__ void tm_st1(uint32_t taddr, uint32_t v) { asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(v) : "memory"); }

    // compile-time loop: f(std::integral_constant<int, 0>) ... f(std::integral_constant<int, N-1>)
    template <typename F, int... K>
    __device__ __forceinline__ void static_for_impl(F &&f, std::integer_sequence<int, K...>) { (f(std::integral_constant<int, K>{}), ...); }
    template <int N, typename F>
    __device__ __forceinline__ void static_for(F &&f) { static_for_impl(f, std::make_integer_sequence<int, N>{}); }

    // bytes between the index blocks of consecutive nodes (SegLayout::idx_stride)
    __host__ __device__ constexpr int idx_stride_of(int deg, int isz)
    {
        const int b = deg * isz;
        return b <= 2 ? 2 : b <= 4 ? 4 : b <= 8 ? 8 : (b + 15) & ~15;
    }

    // All D index entries of one node -> byte offsets.  Entries are uint32 byte offsets or uint16 offsets in
    // 16-byte units (shared-memory residency of codes whose tables would not fit otherwise).  Blocks of up
    // to 8 bytes are node-major; longer ones are 16-byte chunks, chunk-major (SegLayout, code.hpp): chunk q of
    // node j at + q*NPW*16 + j*16.
    template <bool SMEM, typename IdxT, int LANES, int D> struct IdxLoad
    {
        typedef typename PtrOf<SMEM>::type P;
        static constexpr int ISZ = (int)sizeof(IdxT), STRIDE = idx_stride_of(D, ISZ), NW = (STRIDE + 3) / 4;
        static constexpr int CH = STRIDE < 16 ? STRIDE : 16, CSTEP = (32 / LANES) * 16;
        static __device__ __forceinline__ void load(P p, uint32_t (&e)[D])
        {
            uint32_t w[NW];
            if constexpr (STRIDE == 2) w[0] = Acc<SMEM, uint16_t, 0>::ld(p);
            else if constexpr (STRIDE == 4) w[0] = WAcc<SMEM, 0>::ld1(p);
            else if constexpr (STRIDE == 8) { const uint2 t = WAcc<SMEM, 0>::ld2(p); w[0] = t.x; w[1] = t.y; }
            else
                static_for<STRIDE / 16>([&](auto q) {
                    const uint4 t = WAcc<SMEM, q.value * CSTEP>::ld4(p);
                    w[4 * q.value] = t.x; w[4 * q.value + 1] = t.y; w[4 * q.value + 2] = t.z; w[4 * q.value + 3] = t.w;
                });
#pragma unroll
            for (int k = 0; k < D; ++k)
            {
                if constexpr (ISZ == 4) e[k] = w[k];
                else e[k] = ((k & 1) ? (w[k >> 1] >> 16) : (w[k >> 1] & 0xFFFFu)) << 4;
            }
        }
    };
    // one 16-byte chunk (EPC = 16/sizeof(IdxT) entries) of a long index block -> byte offsets (generic-degree paths)
    template <bool SMEM, typename IdxT> struct IdxChunk
    {
        typedef typename PtrOf<SMEM>::type P;
        static constexpr int EPC = 16 / (int)sizeof(IdxT);
        static __device__ __forceinline__ void load(P p, uint32_t (&e)[EPC])
        {
            const uint4 t = WAcc<SMEM, 0>::ld4(p);
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int k = 0; k < EPC; ++k)
            {
                if constexpr (sizeof(IdxT) == 4) e[k] = w[k];
                else e[k] = ((k & 1) ? (w[k >> 1] >> 16) : (w[k >> 1] & 0xFFFFu)) << 4;
            }
        }
    };

    struct K4Params
    {
        // code tables (device global memory), SegLayout of code.hpp
        const uint32_t *cn_seg, *vn_seg; // [warps][max_segs][4]
        const unsigned char *cn_idx, *vn_idx;
        uint32_t cn_idx_bytes, vn_idx_bytes; // multiples of 16
        int cn_max_segs, vn_max_segs;
        const uint32_t *var_pos;                       // [nc] variable id -> position
        const int32_t *tx_pos, *punct_pos, *short_pos; // positions of transmitted (ascending id) / punctured / shortened variables
        int n_slots, n_pos;
        int nc, nct, n_punct, n_short;
        // decoder
        int max_iter, early_term;
        // frame source
        int kind;
        int coherence; // SRC_RAYLEIGH: transmitted positions per fading coefficient (0: one per frame)
        const double *llr_in; // SRC_LLR: [n_frames][nc]; or one of the narrow encodings below (exactly one of the three is set)
        const float *llr_in_f32;  // widened exactly to the decoder's type
        const int8_t *llr_in_i8;  // quantised LLRs: value = i8 * i8_scale, evaluated in double (exact for a power-of-two scale)
        double i8_scale;
        double sigma, sigma2, delta, llr_scale; // llr_scale = 2 / sigma2
        uint32_t thr;
        uint64_t seed;
        uint32_t point;
        uint64_t frame0, n_frames;
        // sinks (indexed by frame - frame0); any may be null
        double *llr_out;
        uint8_t *hard_out;
        uint32_t *hard_bits; // bit-packed hard decisions [n_frames][hard_words] (bit i%32 of word i/32)
        int hard_words;
        int32_t *iters_out;
        unsigned long long *counters; // [5] fec, bec, frames, sum(ret iters), sum(executed iterations)
        // per-error diagnostics log (may be null): records {global frame, bit errors, iterations}, err_count = frames in error
        unsigned long long *err_log;     // [err_cap][2]: frame, bit_errors | (uint32)iterations << 32
        unsigned long long *err_count;
        unsigned long long err_cap;
        // global-memory residency: per-CTA state block
        unsigned char *state;
        size_t state_stride;
        // transmitted codewords (-G, src/sim/channel.cpp:44-60): generator matrix by column (variable id) and
        // the variable id of every transmitted position; g_rows = 0 -> all-zero codeword
        const int32_t *g_col_ptr, *g_row;
        const int32_t *tx_var;
        int g_rows, g_cols, u_words; // u_words = ceil(g_rows / 32)
        AskParams ask; // kind == SRC_ASK
        // TMEM mirror (TM kernels): columns allocated per CTA (power of two >= 32), columns per warp window,
        // column offset of the variable-side (channel LLR) part inside a warp window
        uint32_t tm_alloc_cols, tm_cols_per_warp, tm_vn_off;
        // lock-step kernel (TM, ET = false): column offset of the gather addresses inside a warp window (ls_idx_cols), and the
        // segment descriptors of SegLayout in the parameter bank -- check lists at [warp * cn_max_segs], then variable lists at
        // [warps * cn_max_segs + warp * vn_max_segs] -- so that a warp reads them as uniform values, not through shared memory.
        // The last word of a warp's first variable descriptor (0 in SegLayout) holds the number of its check-side address columns.
        uint32_t tm_idx_off;
        uint32_t ls_seg[4 * K4_LS_SEGS];
    };

    // raw value of smaller magnitude (min-sum keeps raw values; magnitude and sign are fixed at the store)
#ifndef B200_BP_CALL_FROM
#define B200_BP_CALL_FROM 5 // shared-memory fp64 sum-product: check bodies of this degree and above are calls (0: all inlined)
#endif
#ifndef B200_BP_LANES_TOGETHER
#define B200_BP_LANES_TOGETHER 1 // fp64 sum-product: both frame lanes of a vector in one basic block (1: shared-memory kernels, 2: all, 0: none)
#endif
#ifndef B200_BP_EDOMAIN
#define B200_BP_EDOMAIN 1 // fp64 sum-product checks on E = e^-|x| (kernels.cuh bp_check; cn4_any and layered.cuh for arbitrary degree); 0: the pairwise recursion (A/B builds)
#endif
    template <typename T> __device__ __forceinline__ T min_mag(T a, T b) { return (Num<T>::abs(b) < Num<T>::abs(a)) ? b : a; }
    // |mag| with the sign bit of word s (bit 31)
    __device__ __forceinline__ double mag_sign(double m, uint32_t s)
    {
        return __hiloint2double((int)(((uint32_t)__double2hiint(m) & 0x7FFFFFFFu) | (s & 0x80000000u)), __double2loint(m));
    }
    __device__ __forceinline__ float mag_sign(float m, uint32_t s) { return __uint_as_float((__float_as_uint(m) & 0x7FFFFFFFu) | (s & 0x80000000u)); }

    // ------------------------------------------------------------------------------------------
    // check-node update of one node, degree D (compile time).
    //   out_sub : &out[0][sub]            gathered record at + index entry
    //   c2v0    : &c2v[first slot][lane]  slot k at + k*512 (slots of a node are NPW records apart)
    //   ip      : the node's index block
    // Returns, per frame lane of the vector (bit e), the parity of the hard decisions of the check's
    // variables (= the syndrome bit of the previous iteration's output, decoder.h:47-64), which comes for
    // free with the gather.
    // ------------------------------------------------------------------------------------------
    template <typename T, typename IdxT, bool SMEM, int LANES, int ALG, int D>
    struct Cn4
    {
        typedef typename PtrOf<SMEM>::type P;
        typedef Vec<T> V;
        static constexpr int VEC = V::N, CS = 512;

        // CSRC: the old c2v values come from shared/global memory (0, 2) or from the thread's TMEM mirror at
        // columns tc + 4k (1, 3); 2 and 3 force the fresh frame lanes `fz` to +0; 4: every lane's old c2v is +0 (first check
        // phase of a lock-step batch), so v2c = out and no c2v is read; TMW: new values are also written to the mirror.
        // nx: in = this node's index entries (byte offsets), out = those of the node at ip_next when `more`
        // (software prefetch: the load is in flight while this node is computed).
        // PAR: also return the syndrome bits (only early termination consumes them, decoder.cpp:66-72).
        // fz (CSRC >= 2 only): frame lanes of this vector that hold a fresh frame — their old c2v is +0 by definition
        // (decoder.cpp:16-19) whatever the slots still contain, so a refill never has to clear the message array.
        template <int CSRC, bool TMW, bool PAR>
        static __device__ __forceinline__ uint32_t run(P out_sub, P c2v0, uint32_t (&nx)[D], P ip_next, bool more, uint32_t tc, uint32_t fz)
        {
            uint32_t eo[D];
#pragma unroll
            for (int k = 0; k < D; ++k) eo[k] = nx[k];
            if (more) IdxLoad<SMEM, IdxT, LANES, D>::load(ip_next, nx);
            bool par[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) par[e] = false;

            if constexpr (ALG == ALG_MS && D > 4)
            {
                // one pass: running smallest / second smallest raw values, position of the smallest, sign bits
                T m1[VEC], m2[VEC];
                uint32_t arg[VEC], sm[VEC];
#pragma unroll
                for (int e = 0; e < VEC; ++e) { m1[e] = Num<T>::inf(); m2[e] = Num<T>::inf(); arg[e] = 0; sm[e] = 0; }
                static_for<D>([&](auto k) {
                    const V o = VAcc<SMEM, T, 0>::ld(out_sub + eo[k.value]);
                    V c;
                    if constexpr (CSRC == 1 || CSRC == 3) { c = TmAcc<T>::ld(tc + 4 * k.value); tm_wait_ld(); }
                    else if constexpr (CSRC != 4) c = VAcc<SMEM, T, k.value * CS>::ld(c2v0);
                    if constexpr (CSRC == 2 || CSRC == 3)
                    {
#pragma unroll
                        for (int e = 0; e < VEC; ++e) c.e[e] = ((fz >> e) & 1u) ? T(0) : c.e[e];
                    }
#pragma unroll
                    for (int e = 0; e < VEC; ++e)
                    {
                        T v = o.e[e]; // out - (+0) == out for every out, -0 included
                        if constexpr (CSRC != 4) v = o.e[e] - c.e[e]; // == the reference's stored v2c (decoder.cpp:62); LLRin on a fresh frame (:18)
                        if constexpr (PAR) par[e] ^= (o.e[e] <= T(0));
                        sm[e] |= (Num<T>::hi(v) >> 31) << k.value;
                        const bool lt1 = Num<T>::abs(v) < Num<T>::abs(m1[e]), lt2 = Num<T>::abs(v) < Num<T>::abs(m2[e]);
                        m2[e] = lt1 ? m1[e] : (lt2 ? v : m2[e]);
                        arg[e] = lt1 ? (uint32_t)k.value : arg[e];
                        m1[e] = lt1 ? v : m1[e];
                    }
                });
                // sign of message k = total sign ^ own sign: bit k of sm
#pragma unroll
                for (int e = 0; e < VEC; ++e) sm[e] ^= (__popc(sm[e]) & 1u) ? ((D >= 32) ? 0xFFFFFFFFu : ((1u << D) - 1u)) : 0u;
                static_for<D>([&](auto k) {
                    V r;
#pragma unroll
                    for (int e = 0; e < VEC; ++e) r.e[e] = mag_sign((arg[e] == (uint32_t)k.value) ? m2[e] : m1[e], sm[e] << (31 - k.value));
                    VAcc<SMEM, T, k.value * CS>::st(c2v0, r);
                    if constexpr (TMW) TmAcc<T>::st(tc + 4 * k.value, r);
                });
            }
            else
            {
                V v[D], r[D], c[D];
                static_for<D>([&](auto k) {
                    if constexpr (CSRC == 1 || CSRC == 3) c[k.value] = TmAcc<T>::ld(tc + 4 * k.value);
                    else if constexpr (CSRC != 4) c[k.value] = VAcc<SMEM, T, k.value * CS>::ld(c2v0);
                });
                if constexpr (CSRC == 1 || CSRC == 3) tm_wait_ld();
                if constexpr (CSRC == 2 || CSRC == 3)
                {
#pragma unroll
                    for (int k = 0; k < D; ++k)
                    {
#pragma unroll
                        for (int e = 0; e < VEC; ++e) c[k].e[e] = ((fz >> e) & 1u) ? T(0) : c[k].e[e];
                    }
                }
                static_for<D>([&](auto k) {
                    const V o = VAcc<SMEM, T, 0>::ld(out_sub + eo[k.value]);
#pragma unroll
                    for (int e = 0; e < VEC; ++e)
                    {
                        if constexpr (CSRC == 4) v[k.value].e[e] = o.e[e];
                        else v[k.value].e[e] = o.e[e] - c[k.value].e[e];
                        if constexpr (PAR) par[e] ^= (o.e[e] <= T(0));
                    }
                });
#pragma unroll
                for (int e = 0; e < VEC; ++e)
                {
                    if constexpr (ALG == ALG_MS)
                    {
                        // min-sum: f = sign*sign*min (decoder.h:17-20) through the forward/backward recursion of
                        // decoder.cpp:30-44.  Magnitude: exact minimum over the other edges; sign: XOR of sign BITS
                        // (std::signbit semantics, -0.0 is negative).
                        if constexpr (D == 2) { r[0].e[e] = v[1].e[e]; r[1].e[e] = v[0].e[e]; }
                        else
                        {
                            uint32_t sx = 0;
#pragma unroll
                            for (int k = 0; k < D; ++k) sx ^= Num<T>::hi(v[k].e[e]);
                            T m[D];
                            if constexpr (D == 3)
                            {
                                m[0] = min_mag(v[1].e[e], v[2].e[e]); m[1] = min_mag(v[0].e[e], v[2].e[e]); m[2] = min_mag(v[0].e[e], v[1].e[e]);
                            }
                            else
                            {
                                const T m01 = min_mag(v[0].e[e], v[1].e[e]), m23 = min_mag(v[2].e[e], v[3].e[e]);
                                m[0] = min_mag(v[1].e[e], m23); m[1] = min_mag(v[0].e[e], m23);
                                m[2] = min_mag(m01, v[3].e[e]); m[3] = min_mag(m01, v[2].e[e]);
                            }
#pragma unroll
                            for (int k = 0; k < D; ++k) r[k].e[e] = mag_sign(m[k], sx ^ Num<T>::hi(v[k].e[e]));
                        }
                    }
                    else if constexpr (sizeof(T) == 8 && D >= 3 && B200_BP_EDOMAIN)
                    {
                        // sum-product in fp64: the same function of the inputs evaluated on E = e^-|x|, both frame lanes of the
                        // vector together (kernels.cuh bp_check)
                        constexpr bool TOGETHER = B200_BP_LANES_TOGETHER == 2 || (B200_BP_LANES_TOGETHER == 1 && SMEM);
                        if constexpr (TOGETHER)
                        {
                            if (e == 0)
                            {
                                double x[VEC][D], y[VEC][D];
#pragma unroll
                                for (int w = 0; w < VEC; ++w)
#pragma unroll
                                    for (int k = 0; k < D; ++k) x[w][k] = v[k].e[w];
                                bp_check<D, VEC>(x, y);
#pragma unroll
                                for (int w = 0; w < VEC; ++w)
#pragma unroll
                                    for (int k = 0; k < D; ++k) r[k].e[w] = y[w][k];
                            }
                        }
                        else
                        {
                            double x[1][D], y[1][D];
#pragma unroll
                            for (int k = 0; k < D; ++k) x[0][k] = v[k].e[e];
                            bp_check<D, 1>(x, y);
#pragma unroll
                            for (int k = 0; k < D; ++k) r[k].e[e] = y[0][k];
                        }
                    }
                    else
                    {
                        // sum-product: the reference's forward/backward box-plus recursion, file order
                        T F[D];
                        F[0] = v[0].e[e];
#pragma unroll
                        for (int k = 1; k < D; ++k) F[k] = boxplus(F[k - 1], v[k].e[e]);
                        T B = v[D - 1].e[e];
                        r[D - 1].e[e] = F[D - 2];
#pragma unroll
                        for (int k = D - 2; k >= 1; --k) { r[k].e[e] = boxplus(F[k - 1], B); B = boxplus(B, v[k].e[e]); }
                        r[0].e[e] = B;
                    }
                }
                static_for<D>([&](auto k) {
                    VAcc<SMEM, T, k.value * CS>::st(c2v0, r[k.value]);
                    if constexpr (TMW) TmAcc<T>::st(tc + 4 * k.value, r[k.value]);
                });
            }
            uint32_t bits = 0;
#pragma unroll
            for (int e = 0; e < VEC; ++e) bits |= par[e] ? (1u << e) : 0u;
            return bits;
        }
        // lock-step kernel: nx holds this node's gather addresses (shared-memory byte addresses: run() with out_sub = 0 and no
        // index load); those of the next task (TMEM columns ti_next) are loaded while this one runs.  The wait of the c2v mirror
        // load covers them; the first check phase of a batch reads no mirror and waits at the end of the task.
        template <int CSRC>
        static __device__ __forceinline__ void run_ls(uint32_t (&nx)[D], uint32_t ti_next, bool more, P c2v0, uint32_t tc)
        {
            uint32_t ga[D];
#pragma unroll
            for (int k = 0; k < D; ++k) ga[k] = nx[k];
            if (more) tm_ld_idx<D>(ti_next, nx);
            run<CSRC, true, false>(P(0), c2v0, ga, P(0), false, tc, 0u);
            if constexpr (CSRC == 4) tm_wait_ld();
        }
    };

    // Out-of-line copy of a fixed-degree body.  The fp64 sum-product bodies of degree >= B200_BP_CALL_FROM need more registers than
    // the 128 a 512-thread CTA leaves; inlined, they make the allocator spill the decode loop's state around the whole degree
    // switch, and with the L1 carved out for shared memory every reload is an L2 round trip -- also on codes that never execute
    // those bodies (h.txt: check degrees 3 and 4).  Behind a call only the call site pays.
    template <typename T, typename IdxT, bool SMEM, int LANES, int ALG, int D, int CSRC, bool TMW, bool PAR>
    __device__ __noinline__ uint32_t cn4_call(typename PtrOf<SMEM>::type out_sub, typename PtrOf<SMEM>::type c2v0, typename PtrOf<SMEM>::type ip, uint32_t tc, uint32_t fz)
    {
        uint32_t nx[D];
        IdxLoad<SMEM, IdxT, LANES, D>::load(ip, nx);
        return Cn4<T, IdxT, SMEM, LANES, ALG, D>::template run<CSRC, TMW, PAR>(out_sub, c2v0, nx, ip, false, tc, fz);
    }

    // arbitrary degree (9..64): running min1/min2 + sign mask for min-sum, parked forward values for box-plus.
    // The index block is walked in 16-byte chunks (chunk q at ip + q*NPW*16).
    template <typename T, typename IdxT, bool SMEM, int LANES, int ALG>
    __device__ __noinline__ uint32_t cn4_any(typename PtrOf<SMEM>::type out_sub, typename PtrOf<SMEM>::type c2v0, typename PtrOf<SMEM>::type ip, int deg,
                                             uint32_t fz)
    {
        typedef Vec<T> V;
        typedef IdxChunk<SMEM, IdxT> IC;
        constexpr int VEC = V::N, CS = 512, EPC = IC::EPC, CSTEP = (32 / LANES) * 16;
        uint32_t par = 0;
        if (ALG == ALG_MS)
        {
            T m1[VEC], m2[VEC];
            int arg[VEC];
            unsigned long long smask[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) { m1[e] = Num<T>::inf(); m2[e] = Num<T>::inf(); arg[e] = 0; smask[e] = 0; }
            for (int k0 = 0; k0 < deg; k0 += EPC, ip += CSTEP)
            {
                uint32_t eo[EPC];
                IC::load(ip, eo);
#pragma unroll
                for (int q = 0; q < EPC; ++q)
                {
                    const int k = k0 + q;
                    if (k < deg)
                    {
                        const V o = VAcc<SMEM, T, 0>::ld(out_sub + eo[q]);
                        V c = VAcc<SMEM, T, 0>::ld(c2v0 + k * CS);
#pragma unroll
                        for (int e = 0; e < VEC; ++e) c.e[e] = ((fz >> e) & 1u) ? T(0) : c.e[e];
#pragma unroll
                        for (int e = 0; e < VEC; ++e)
                        {
                            const T v = o.e[e] - c.e[e];
                            par ^= (o.e[e] <= T(0)) ? (1u << e) : 0u;
                            smask[e] |= (unsigned long long)(Num<T>::hi(v) >> 31) << k;
                            const bool lt1 = Num<T>::abs(v) < Num<T>::abs(m1[e]), lt2 = Num<T>::abs(v) < Num<T>::abs(m2[e]);
                            m2[e] = lt1 ? m1[e] : (lt2 ? v : m2[e]);
                            arg[e] = lt1 ? k : arg[e];
                            m1[e] = lt1 ? v : m1[e];
                        }
                    }
                }
            }
            uint32_t tot[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) tot[e] = (uint32_t)__popcll(smask[e]) & 1u;
            for (int k = 0; k < deg; ++k)
            {
                V r;
#pragma unroll
                for (int e = 0; e < VEC; ++e)
                {
                    const uint32_t s = tot[e] ^ (uint32_t)((smask[e] >> k) & 1ull);
                    r.e[e] = mag_sign((k == arg[e]) ? m2[e] : m1[e], s << 31);
                }
                VAcc<SMEM, T, 0>::st(c2v0 + k * CS, r);
            }
        }
        else
        {
            // box-plus forward/backward with the forward values parked in the output slots: slot k first
            // receives F[k-1]; the backward sweep turns it into f(F[k-1], B[k+1]) (decoder.cpp:33-44).
            // v[k] is needed again by the backward sweep (out and the old c2v are gone by then).
            V v[64];
            [[maybe_unused]] unsigned long long smask[VEC];
            [[maybe_unused]] uint32_t mh[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) { smask[e] = 0; mh[e] = 0x7fffffffu; }
            for (int k0 = 0; k0 < deg; k0 += EPC, ip += CSTEP)
            {
                uint32_t eo[EPC];
                IC::load(ip, eo);
#pragma unroll
                for (int q = 0; q < EPC; ++q)
                {
                    const int k = k0 + q;
                    if (k < deg)
                    {
                        const V o = VAcc<SMEM, T, 0>::ld(out_sub + eo[q]);
                        V c = VAcc<SMEM, T, 0>::ld(c2v0 + k * CS);
#pragma unroll
                        for (int e = 0; e < VEC; ++e) c.e[e] = ((fz >> e) & 1u) ? T(0) : c.e[e];
                        V vk;
#pragma unroll
                        for (int e = 0; e < VEC; ++e)
                        {
                            vk.e[e] = o.e[e] - c.e[e];
                            par ^= (o.e[e] <= T(0)) ? (1u << e) : 0u;
                            if constexpr (sizeof(T) == 8)
                            {
                                const uint32_t h = Num<T>::hi(vk.e[e]);
                                smask[e] |= (unsigned long long)(h >> 31) << k;
                                mh[e] = min(mh[e], h & 0x7fffffffu);
                            }
                        }
                        v[k] = vk;
                    }
                }
            }
            bool exact = true;
            if constexpr (sizeof(T) == 8 && B200_BP_EDOMAIN)
            {
                // fp64: the check on E = e^-|x| (kernels.cuh bp_check): forward and backward values as plain numbers
                // (one division per step), the outputs as logarithms of the joined fractions; the exponentials are
                // recomputed in the backward sweep rather than kept in a second local array.
                double shift[VEC];
                V Fp, B;
#pragma unroll
                for (int e = 0; e < VEC; ++e)
                    shift[e] = (mh[e] >= 0x40440000u && mh[e] < 0x7ff00000u) ? __hiloint2double((int)mh[e], 0) - 40.0 : 0.0;
                for (int k = 0; k < deg; ++k)
                {
                    const V vk = v[k];
                    V Ek;
#pragma unroll
                    for (int e = 0; e < VEC; ++e) Ek.e[e] = bp_exp_neg(fabs(vk.e[e]) - shift[e]);
                    if (k == 0) Fp = Ek;
                    else
                    {
                        VAcc<SMEM, T, 0>::st(c2v0 + k * CS, Fp); // E of F[k-1]
#pragma unroll
                        for (int e = 0; e < VEC; ++e) Fp.e[e] = bp_join(Fp.e[e], Ek.e[e]);
                    }
                }
                bool anyfar = false, far;
#pragma unroll
                for (int e = 0; e < VEC; ++e) B.e[e] = bp_exp_neg(fabs(v[deg - 1].e[e]) - shift[e]);
                for (int k = deg - 1; k >= 0; --k)
                {
                    V f = B;
                    if (k > 0) f = VAcc<SMEM, T, 0>::ld(c2v0 + k * CS);
                    const V vk = v[k];
                    V r;
#pragma unroll
                    for (int e = 0; e < VEC; ++e)
                    {
                        double N, Dn;
                        if (k == deg - 1) { N = f.e[e]; Dn = 1.0; }
                        else if (k == 0) { N = B.e[e]; Dn = 1.0; }
                        else { N = f.e[e] + B.e[e]; Dn = __fma_rn(f.e[e], B.e[e], 1.0); }
                        const double l = bp_log_frac(N, Dn, shift[e], far);
                        anyfar |= far;
                        const uint32_t sg = (((uint32_t)__popcll(smask[e]) ^ (uint32_t)(smask[e] >> k)) & 1u) << 31;
                        r.e[e] = __hiloint2double((int)(((uint32_t)__double2hiint(l) & 0x7fffffffu) | sg), __double2loint(l));
                        if (k > 0 && k < deg - 1) B.e[e] = bp_join(B.e[e], bp_exp_neg(fabs(vk.e[e]) - shift[e]));
                    }
                    VAcc<SMEM, T, 0>::st(c2v0 + k * CS, r);
                }
                exact = anyfar; // rare: inputs beyond the clamp of the exponential decide an output
            }
            if (exact)
            {
                V Fp, B;
                for (int k = 0; k < deg; ++k)
                {
                    const V vk = v[k];
                    if (k == 0) Fp = vk;
                    else
                    {
                        VAcc<SMEM, T, 0>::st(c2v0 + k * CS, Fp); // F[k-1] (slot deg-1 thereby gets its final value)
#pragma unroll
                        for (int e = 0; e < VEC; ++e) Fp.e[e] = boxplus(Fp.e[e], vk.e[e]);
                    }
                }
                B = v[deg - 1];
                for (int k = deg - 2; k >= 1; --k)
                {
                    const V f = VAcc<SMEM, T, 0>::ld(c2v0 + k * CS);
                    V r;
#pragma unroll
                    for (int e = 0; e < VEC; ++e) { r.e[e] = boxplus(f.e[e], B.e[e]); B.e[e] = boxplus(B.e[e], v[k].e[e]); }
                    VAcc<SMEM, T, 0>::st(c2v0 + k * CS, r);
                }
                VAcc<SMEM, T, 0>::st(c2v0, B);
            }
        }
        return par;
    }

    // variable node: posterior = LLRin + sum of incoming c2v, strictly in file order (decoder.cpp:50-56)
    template <typename T, typename IdxT, bool SMEM, int LANES, int D>
    struct Vn4
    {
        typedef typename PtrOf<SMEM>::type P;
        typedef Vec<T> V;
        static __device__ __forceinline__ V run(P c2v_sub, uint32_t (&nx)[D], P ip_next, bool more, V acc)
        {
            uint32_t eo[D];
#pragma unroll
            for (int k = 0; k < D; ++k) eo[k] = nx[k];
            if (more) IdxLoad<SMEM, IdxT, LANES, D>::load(ip_next, nx);
            V m[D];
#pragma unroll
            for (int k = 0; k < D; ++k) m[k] = VAcc<SMEM, T, 0>::ld(c2v_sub + eo[k]);
#pragma unroll
            for (int k = 0; k < D; ++k)
            {
#pragma unroll
                for (int e = 0; e < V::N; ++e) acc.e[e] += m[k].e[e];
            }
            return acc;
        }
        // lock-step kernel: gather addresses in nx, the next task's loaded from TMEM columns ti_next meanwhile (the caller waits)
        static __device__ __forceinline__ V run_ls(uint32_t (&nx)[D], uint32_t ti_next, bool more, V acc)
        {
            uint32_t ga[D];
#pragma unroll
            for (int k = 0; k < D; ++k) ga[k] = nx[k];
            if (more) tm_ld_idx<D>(ti_next, nx);
            return run(P(0), ga, P(0), false, acc);
        }
    };
    // arbitrary degree (> 8): 16-byte index chunks (chunk q at ip + q*NPW*16)
    template <typename T, typename IdxT, bool SMEM, int LANES>
    __device__ __forceinline__ Vec<T> vn4_any(typename PtrOf<SMEM>::type c2v_sub, typename PtrOf<SMEM>::type ip, int deg, Vec<T> acc)
    {
        typedef Vec<T> V;
        typedef IdxChunk<SMEM, IdxT> IC;
        constexpr int EPC = IC::EPC, CSTEP = (32 / LANES) * 16;
        for (int k0 = 0; k0 < deg; k0 += EPC, ip += CSTEP)
        {
            uint32_t eo[EPC];
            IC::load(ip, eo);
            if (k0 + EPC <= deg)
            {
                V m[EPC];
#pragma unroll
                for (int q = 0; q < EPC; ++q) m[q] = VAcc<SMEM, T, 0>::ld(c2v_sub + eo[q]);
#pragma unroll
                for (int q = 0; q < EPC; ++q)
                {
#pragma unroll
                    for (int e = 0; e < V::N; ++e) acc.e[e] += m[q].e[e];
                }
            }
            else
            {
#pragma unroll
                for (int q = 0; q < EPC; ++q)
                    if (k0 + q < deg)
                    {
                        const V m = VAcc<SMEM, T, 0>::ld(c2v_sub + eo[q]);
#pragma unroll
                        for (int e = 0; e < V::N; ++e) acc.e[e] += m.e[e];
                    }
            }
        }
        return acc;
    }

    // ------------------------------------------------------------------------------------------
    // the persistent kernel
    // ------------------------------------------------------------------------------------------
#ifndef B200_TILE_MAX_THREADS
#define B200_TILE_MAX_THREADS 512 // compile-time cap of threads per CTA (register budget = 65536 / cap)
#endif
    // TM: keep the write-through TMEM mirror (K4Params::tm_*; shared-memory residency only).
    // ET: compiled with early termination support (syndrome in the check phase); ET = false serves --no-early-term runs.
    // MINB: resident CTAs per SM the kernel is compiled for (register budget 65536 / (MINB * B200_TILE_MAX_THREADS)): 1 everywhere
    // except the narrow global-residency min-sum variant (2: more warps, 64 registers), which quasi-cyclic codes prefer.
    // The shared-memory fp64 sum-product kernel is compiled for fewer threads: its check bodies want ~170 registers, and at 128
    // the allocator parks the decode loop's CTA-uniform state in local memory -- with the L1 carved out for shared memory every
    // reload after a barrier is an L2 round trip with all warps waiting (ncu: 16 % of the warp time in long-scoreboard stalls).
    // 12 warps x 168 registers beat 16 x 128 by 11 % on h.txt.
#ifndef B200_BP64_SMEM_THREADS
#define B200_BP64_SMEM_THREADS 384
#endif
    constexpr int tile_thread_cap(bool f64, int alg, bool smem)
    {
        return (f64 && alg == ALG_BP && smem && B200_BP64_SMEM_THREADS < B200_TILE_MAX_THREADS) ? B200_BP64_SMEM_THREADS : B200_TILE_MAX_THREADS;
    }
    template <typename T, typename IdxT, int ALG, bool SMEM, int LANES, bool TM, bool ET, int MINB>
    __global__ void __launch_bounds__(tile_thread_cap(sizeof(T) == 8, ALG, SMEM), MINB) tile4_kernel(const K4Params p)
    {
        static_assert(SMEM || !TM, "the TMEM mirror belongs to shared-memory residency");
        typedef typename PtrOf<SMEM>::type P;
        typedef Vec<T> V;
        constexpr int VEC = V::N, FPC = LANES * VEC, NPW = 32 / LANES;
        constexpr int TS = (int)sizeof(T), RS = 16 * LANES, ISZ = (int)sizeof(IdxT);
        constexpr uint32_t ALL = (FPC == 32) ? 0xFFFFFFFFu : ((1u << FPC) - 1u), VMASK = (1u << VEC) - 1u;
        extern __shared__ __align__(16) unsigned char dyn_smem[];
        struct LaneCnt { unsigned long long bec, ret, its; uint32_t fec, frames; }; // per frame lane, owned by lane g of warp 0 (no atomics)
        __shared__ unsigned long long s_old[FPC];
        __shared__ LaneCnt s_cnt[FPC];
        __shared__ uint32_t s_err[FPC];
        __shared__ int s_ret[FPC];
        __shared__ uint32_t s_synd[2];
        __shared__ uint2 s_ctrl[2]; // {frames at the iteration limit, frames with >= 1 completed iteration}
        __shared__ uint32_t s_tmem;

        const int tid = threadIdx.x, nthreads = blockDim.x;
        // the warp index through a broadcast: the compiler then keeps everything derived from it in uniform registers
        // (shared-memory residency only: the global-residency kernels lost 25-30 % with it, their loads want to stay in flight)
        const int lane = tid & 31, warp = SMEM ? __shfl_sync(0xFFFFFFFFu, tid >> 5, 0) : (tid >> 5), warps = nthreads >> 5;
        const int sub = lane & (LANES - 1), j = lane / LANES;

        // ---- carve state and tables --------------------------------------------------------
        P c2v, out, llr, cn_seg, vn_seg, cn_idx, vn_idx;
        uint32_t a_u = (uint32_t)__cvta_generic_to_shared(dyn_smem); // information words of the frames in flight: [FPC][u_words]
        uint32_t a_tx = 0, a_pu = 0, a_sh = 0;                       // shared-memory residency: position tables (uint16)
        if constexpr (SMEM)
        {
            uint32_t q = (uint32_t)__cvta_generic_to_shared(dyn_smem);
            const uint32_t a_c2v = q; q += RS * p.n_slots;
            const uint32_t a_out = q; q += RS * p.n_pos;
            const uint32_t a_llr = q; q += RS * p.n_pos;
            const uint32_t a_cs = q; q += 16 * p.cn_max_segs * warps;
            const uint32_t a_vs = q; q += 16 * p.vn_max_segs * warps;
            const uint32_t a_ci = q; q += p.cn_idx_bytes;
            const uint32_t a_vi = q; q += p.vn_idx_bytes;
            // positions of the transmitted / punctured / shortened variables as 16-bit entries: a refill reads them on its
            // critical path (two L2 round trips per event when they sat in global memory)
            a_tx = q; q += 2 * ((p.nct + 3) & ~3);
            a_pu = q; q += 2 * p.n_punct;
            a_sh = q; q += 2 * p.n_short;
            q = (q + 15u) & ~15u;
            a_u = q;
            for (int i = tid; i < p.nct; i += nthreads) sts_u16<0>(a_tx + 2 * i, (uint32_t)p.tx_pos[i]);
            for (int i = tid; i < p.n_punct; i += nthreads) sts_u16<0>(a_pu + 2 * i, (uint32_t)p.punct_pos[i]);
            for (int i = tid; i < p.n_short; i += nthreads) sts_u16<0>(a_sh + 2 * i, (uint32_t)p.short_pos[i]);
            if constexpr (ET || !TM) // the lock-step kernel takes its descriptors from the parameters
            {
                for (int i = tid; i < 4 * p.cn_max_segs * warps; i += nthreads) sts_u32<0>(a_cs + 4 * i, p.cn_seg[i]);
                for (int i = tid; i < 4 * p.vn_max_segs * warps; i += nthreads) sts_u32<0>(a_vs + 4 * i, p.vn_seg[i]);
            }
            for (int i = tid; i < (int)(p.cn_idx_bytes >> 2); i += nthreads) sts_u32<0>(a_ci + 4 * i, reinterpret_cast<const uint32_t *>(p.cn_idx)[i]);
            for (int i = tid; i < (int)(p.vn_idx_bytes >> 2); i += nthreads) sts_u32<0>(a_vi + 4 * i, reinterpret_cast<const uint32_t *>(p.vn_idx)[i]);
            c2v = a_c2v; out = a_out; llr = a_llr; cn_seg = a_cs; vn_seg = a_vs; cn_idx = a_ci; vn_idx = a_vi;
        }
        else
        {
            unsigned char *q = p.state + p.state_stride * blockIdx.x;
            unsigned char *g_c2v = q; q += (size_t)RS * p.n_slots;
            unsigned char *g_out = q; q += (size_t)RS * p.n_pos;
            unsigned char *g_llr = q;
            c2v = g_c2v; out = g_out; llr = g_llr;
            cn_seg = (unsigned char *)p.cn_seg; vn_seg = (unsigned char *)p.vn_seg;
            cn_idx = (unsigned char *)p.cn_idx; vn_idx = (unsigned char *)p.vn_idx;
        }
        uint32_t tm_w = 0; // this warp's TMEM window: lane partition (warp % 4), columns (warp / 4) * tm_cols_per_warp ...
        if constexpr (TM)
        {
            if (warp == 0)
            {
                asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(&s_tmem)), "r"(p.tm_alloc_cols) : "memory");
                asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tm_w = s_tmem + (((uint32_t)(warp & 3) * 32u) << 16) + (uint32_t)(warp >> 2) * p.tm_cols_per_warp;
        }
        if constexpr (TM && !ET)
        {
            // The work of a thread is the same in every phase of the launch: write the shared-memory address of each of its
            // gathers (check side: `out` record + sub, variable side: c2v record + sub) into its TMEM lane once, task after
            // task in list order (ls_idx_cols columns each).  The index tables were staged above.
            constexpr int EPC = 16 / ISZ;
            uint32_t ti = tm_w + p.tm_idx_off;
            for (int side = 0; side < 2; ++side)
            {
                const int ms = side ? p.vn_max_segs : p.cn_max_segs, s0 = (side ? warps * p.cn_max_segs : 0) + warp * ms;
                const P base = (side ? c2v : out) + sub * 16, tab = side ? vn_idx : cn_idx;
                for (int s = s0; s < s0 + ms; ++s)
                {
                    const uint4 sg = make_uint4(p.ls_seg[4 * s], p.ls_seg[4 * s + 1], p.ls_seg[4 * s + 2], 0u);
                    if (sg.x == 0) break;
                    const int deg = (int)(sg.x & 0xFFu), nt = (int)(sg.x >> 16);
                    const int w = ls_idx_cols(side == 0, deg), st = idx_stride_of(deg, ISZ);
                    for (int t = 0; t < nt && w > 0; ++t)
                        for (int k = 0; k < w; ++k, ++ti)
                        {
                            uint32_t a = 0;
                            if (k < deg)
                            {
                                const uint32_t o = sg.z + (uint32_t)(st < 16 ? (t * NPW + j) * st + k * ISZ : t * NPW * st + (k / EPC) * NPW * 16 + j * 16 + (k % EPC) * ISZ);
                                a = base + (ISZ == 4 ? lds_u32<0>(tab + o) : lds_u16<0>(tab + o) << 4);
                            }
                            tm_st1(ti, a);
                        }
                }
            }
            tm_wait_st();
        }
        if (tid < FPC)
        {
            s_err[tid] = 0; s_old[tid] = 0; s_ret[tid] = 0;
            s_cnt[tid].bec = 0; s_cnt[tid].ret = 0; s_cnt[tid].its = 0; s_cnt[tid].fec = 0; s_cnt[tid].frames = 0;
        }
        if (tid == 0)
        {
            s_synd[0] = 0; s_synd[1] = 0;
            s_ctrl[0] = make_uint2(0, 0); s_ctrl[1] = make_uint2(0, 0);
        }
        __syncthreads();

        // per-frame iteration counter and global frame index: lane g of warp 0 owns frame lane g
        int it = 0;
        unsigned long long my_gf = 0;
        // CTA-uniform scheduling state, kept in registers by every thread (no shared round trip): frame lanes in flight, lanes
        // that sit out the next variable phase, and the CTA's frame cursor (its k-th frame is blockIdx.x + gridDim.x * k)
        uint32_t active = 0, skip = 0;
        unsigned long long next_k = 0;
        const unsigned long long k_end = (blockIdx.x < p.n_frames) ? (p.n_frames - blockIdx.x + gridDim.x - 1) / gridDim.x : 0ull;
#ifdef B200_PHASE_TIMING
        long long pt_refill = 0, pt_nrefill = 0, pt_rf[4] = {0, 0, 0, 0}; // stages: bit errors (+ arrival skew), bookkeeping, outputs, generate
#endif
        // A refill rewrites c2v / llr in shared memory behind the TMEM mirror's back: the next check phase and the
        // next variable phase read shared memory (and refresh the mirror).  CTA-uniform.
        bool cn_stale = true, vn_stale = true;
        uint32_t fresh = 0; // frame lanes refilled since the last check phase (CTA-uniform)


        // bit of the codeword of frame lane g at transmitted index t: parity of the information bits selected by
        // column tx_var[t] of the generator matrix (src/core/sparse.h:162-187); 0 without a generator matrix
        auto cw_bit = [&](int g, int t) -> uint32_t
        {
            if (p.g_rows <= 0) return 0u;
            const int v = p.tx_var[t];
            if (v >= p.g_cols) return 0u;
            uint32_t b = 0;
            for (int q = p.g_col_ptr[v]; q < p.g_col_ptr[v + 1]; ++q)
            {
                const int r = p.g_row[q];
                b ^= lds_u32<0>(a_u + 4 * (g * p.u_words + (r >> 5))) >> (r & 31);
            }
            return b & 1u;
        };

        // One pass over the transmitted positions of frame lane g (all threads of the CTA cooperate; thread <-> Philox block q
        // <-> transmitted indices 4q .. 4q+3), doing either or both of
        //   count  : bit errors of the lane's final decisions against the transmitted word (ldpcsim.cpp:184-190) -> s_err[g]
        //   refill : the decoder input of global frame gf, with the fresh-frame state out = LLRin (c2v = +0 is implied by the
        //            `fresh` mask: the message array is never cleared).
        // Doing both in ONE pass needs no barrier in between: a thread reads the old posterior of exactly the positions it then
        // overwrites.  (Caller-supplied LLRs are indexed by variable, not by transmitted index: they take separate passes.)
        auto frame_pass = [&](int g, bool count, bool refill, unsigned long long gf)
        {
            const int eo = (g / VEC) * 16 + (g % VEC) * TS; // byte offset of lane g inside a record
            const P dl = llr + eo, dout = out + eo;
            auto put = [&](int pos, T v)
            {
                Acc<SMEM, T, 0>::st(dl + pos * RS, v);
                Acc<SMEM, T, 0>::st(dout + pos * RS, v);
            };
            const bool has_g = p.g_rows > 0;
            const unsigned long long frame = p.frame0 + gf;
            const bool gen = refill && p.kind != SRC_LLR && p.kind != SRC_ASK;
            uint32_t nerr = 0;
#ifdef B200_PHASE_TIMING
            const long long fp0 = clock64();
#endif
            const int nblk = (p.nct + 3) >> 2;
            for (int q = tid; q < nblk; q += nthreads)
            {
                // value k of Philox block q belongs to the transmitted index q + k*nblk: for every k the threads of a warp then
                // touch neighbouring transmitted indices, i.e. (mostly) neighbouring records — with 4q + k they strode four
                // records apart and every one of the pass's scattered loads / stores was a 16-way bank conflict
                int pos[4];
                bool ok[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                {
                    const int t = q + k * nblk;
                    ok[k] = t < p.nct;
                    if constexpr (SMEM) pos[k] = ok[k] ? (int)lds_u16<0>(a_tx + 2 * t) : 0;
                    else pos[k] = ok[k] ? __ldg(p.tx_pos + t) : 0;
                }
                if (count)
                {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (ok[k]) nerr += ((Acc<SMEM, T, 0>::ld(dout + pos[k] * RS) <= T(0)) ? 1u : 0u) ^ ((has_g && !refill) ? cw_bit(g, q + k * nblk) : 0u);
                }
                if (gen)
                {
                    const u32x4 r = channel_block(p.seed, p.point, 0, frame, (uint32_t)q);
                    if (p.kind == SRC_AWGN)
                    { // y = sigma*z + x, x = 1 - 2*cw (BPSK), LLR = 2y/sigma^2 (src/sim/channel.cpp:56-68,88-92), evaluated as
                      // y * (2/sigma^2) with the factor rounded once on the host (channel specification, oracle orc_channel_frame)
                        float z[4];
                        normal_pair(r.x, r.y, z[0], z[1]);
                        normal_pair(r.z, r.w, z[2], z[3]);
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (ok[k])
                            {
                                const double x = (has_g && cw_bit(g, q + k * nblk)) ? -1.0 : 1.0;
                                const double y = __dadd_rn(__dmul_rn((double)z[k], p.sigma), x);
                                put(pos[k], (T)__dmul_rn(y, p.llr_scale));
                            }
                    }
                    else if (p.kind == SRC_RAYLEIGH)
                    { // the AWGN noise with the faded amplitude h: y = sigma*z + h*x, LLR = y*h*(2/sigma^2) (DESIGN.md §3.2)
                        float z[4];
                        normal_pair(r.x, r.y, z[0], z[1]);
                        normal_pair(r.z, r.w, z[2], z[3]);
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (ok[k])
                            {
                                const int t = q + k * nblk;
                                const double h = rayleigh_coeff(p.seed, p.point, frame, p.coherence ? (uint32_t)(t / p.coherence) : 0u);
                                const double y = __dadd_rn(__dmul_rn((double)z[k], p.sigma), (has_g && cw_bit(g, t)) ? -h : h);
                                put(pos[k], (T)__dmul_rn(__dmul_rn(y, h), p.llr_scale));
                            }
                    }
                    else
                    { // BSC: y = x ^ Bernoulli(eps), LLR = delta*(1-2y) (src/sim/channel.cpp:123-162)
                        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (ok[k]) put(pos[k], (T)((((w[k] < p.thr) ? 1u : 0u) ^ (has_g ? cw_bit(g, q + k * nblk) : 0u)) ? -p.delta : p.delta));
                    }
                }
            }
#ifdef B200_PHASE_TIMING
            const long long fp1 = clock64();
            pt_rf[1] += fp1 - fp0;
#endif
            if (gen)
            {
                const T sv = (T)(p.kind == SRC_BSC ? p.delta : 99999.9);
                if constexpr (SMEM)
                {
                    for (int i = tid; i < p.n_punct; i += nthreads) put((int)lds_u16<0>(a_pu + 2 * i), T(0));
                    for (int i = tid; i < p.n_short; i += nthreads) put((int)lds_u16<0>(a_sh + 2 * i), sv);
                }
                else
                {
                    for (int i = tid; i < p.n_punct; i += nthreads) put(p.punct_pos[i], T(0));
                    for (int i = tid; i < p.n_short; i += nthreads) put(p.short_pos[i], sv);
                }
            }
            else if (refill && p.kind == SRC_ASK)
            { // M-ASK / bit-metric: thread <-> Philox block q <-> symbols q + k*nsblk; LLRs land at the positions of the mapped variables
                const int nsblk = (p.ask.n_sym + 3) >> 2;
                for (int q = tid; q < nsblk; q += nthreads)
                {
                    const u32x4 r = channel_block(p.seed, p.point, 0, frame, (uint32_t)q);
                    float z[4];
                    normal_pair(r.x, r.y, z[0], z[1]);
                    normal_pair(r.z, r.w, z[2], z[3]);
                    for (int k = 0; k < 4; ++k)
                        if (q + k * nsblk < p.ask.n_sym)
                            ask_symbol(p.ask, p.seed, p.point, frame, q + k * nsblk, z[k], p.sigma, p.sigma2, [&](int v, double l, uint32_t) { put((int)p.var_pos[v], (T)l); });
                }
                for (int i = tid; i < p.n_punct; i += nthreads) put(p.punct_pos[i], T(0));
                for (int i = tid; i < p.n_short; i += nthreads) put(p.short_pos[i], (T)99999.9);
            }
            else if (refill)
            {
                if (p.llr_in_f32)
                {
                    const float *src = p.llr_in_f32 + (size_t)gf * p.nc;
                    for (int i = tid; i < p.nc; i += nthreads) put((int)p.var_pos[i], (T)src[i]);
                }
                else if (p.llr_in_i8)
                {
                    const int8_t *src = p.llr_in_i8 + (size_t)gf * p.nc;
                    for (int i = tid; i < p.nc; i += nthreads) put((int)p.var_pos[i], (T)__dmul_rn((double)src[i], p.i8_scale));
                }
                else
                {
                    const double *src = p.llr_in + (size_t)gf * p.nc;
                    for (int i = tid; i < p.nc; i += nthreads) put((int)p.var_pos[i], (T)src[i]);
                }
            }
#ifdef B200_PHASE_TIMING
            const long long fp2 = clock64();
            pt_rf[2] += fp2 - fp1;
#endif
            if (count)
            {
                nerr = __reduce_add_sync(0xffffffffu, nerr);
                if (lane == 0 && nerr) atomicAdd(&s_err[g], nerr);
            }
#ifdef B200_PHASE_TIMING
            pt_rf[3] += clock64() - fp2;
#endif
        };
        // fresh information word of frame gf from Philox stream 1 (bit k = bit k%32 of word k/32) into lane g's slot; cw = u*G
        auto draw_info_word = [&](int g, unsigned long long gf)
        {
            for (int w = tid; w < p.u_words; w += nthreads)
            {
                const u32x4 r = channel_block(p.seed, p.point, 1, p.frame0 + gf, (uint32_t)w >> 2);
                const uint32_t q4[4] = {r.x, r.y, r.z, r.w};
                uint32_t v = q4[w & 3];
                if (32 * w + 32 > p.g_rows) v &= (1u << (p.g_rows - 32 * w)) - 1u;
                sts_u32<0>(a_u + 4 * (g * p.u_words + w), v);
            }
        };

        // Retires the frame lanes in `mask` and hands each a new frame if any is left.
        //   synd / started : syndrome flags and ">= 1 iteration done" flags valid for this decision
        //   as_skip        : the new frames must sit out the variable phase that follows
        // Which lanes get a frame is plain arithmetic on CTA-uniform registers; the counters live in per-lane shared rows that
        // only lane g of warp 0 touches.  Sweeps (frames made on the device, no per-frame outputs, all-zero codeword) take ONE
        // fused count + refill pass and ONE barrier per event; decode-API launches and -G sweeps take the staged route.
        auto retire_and_refill = [&](uint32_t mask, uint32_t synd, uint32_t started, bool as_skip, bool first_fill)
        {
#ifdef B200_PHASE_TIMING
            const long long rf0 = clock64();
#endif
            const unsigned long long left = k_end - next_k;
            const uint32_t n_new = (uint32_t)min((unsigned long long)__popc(mask), left);
            uint32_t gm = 0; // the lanes that receive a frame: the lowest n_new set bits of `mask`
#pragma unroll
            for (int g = 0; g < FPC; ++g)
                if (((mask >> g) & 1u) && (uint32_t)__popc(mask & ((1u << g) - 1u)) < n_new) gm |= 1u << g;
            auto new_frame = [&](int g) { return (unsigned long long)blockIdx.x + (unsigned long long)gridDim.x * (next_k + (unsigned long long)__popc(mask & ((1u << g) - 1u))); };
            const bool outputs = !first_fill && (p.llr_out || p.hard_out || p.hard_bits || p.iters_out);
            const bool fused = p.kind != SRC_LLR && p.kind != SRC_ASK && p.g_rows <= 0 && !outputs;
            auto bookkeeping = [&]()
            {
                if (warp != 0) return;
                const bool mine = lane < FPC && ((mask >> lane) & 1u);
                if (mine && !first_fill)
                {
                    const bool conv = ET && p.early_term && ((started >> lane) & 1u) && !((synd >> lane) & 1u);
                    const int ret = conv ? it - 1 : p.max_iter; // the reference breaks before ++I (decoder.cpp:66-77)
                    const uint32_t e = s_err[lane];
                    s_err[lane] = 0;
                    LaneCnt c = s_cnt[lane];
                    c.fec += e ? 1u : 0u; c.bec += e; c.frames += 1u; c.ret += (unsigned long long)ret; c.its += (unsigned long long)it;
                    s_cnt[lane] = c;
                    s_ret[lane] = ret;
                    s_old[lane] = my_gf;
                    if (e && p.err_log)
                    { // the frame can be regenerated from its global index (counter-based channel): that is the whole record
                        const unsigned long long slot = atomicAdd(p.err_count, 1ull);
                        if (slot < p.err_cap)
                        {
                            p.err_log[2 * slot] = p.frame0 + my_gf;
                            p.err_log[2 * slot + 1] = (unsigned long long)e | ((unsigned long long)(uint32_t)ret << 32);
                        }
                    }
                }
                if (mine)
                {
                    it = 0;
                    if ((gm >> lane) & 1u) my_gf = new_frame(lane);
                }
            };
            // Up to two rounds of ONE frame_pass call site (a second inlined copy would double the cold code):
            //   fused : round 0 = count + refill, then the barrier and the bookkeeping
            //   staged: round 0 = count (skipped on the first fill); bookkeeping, outputs, information words; round 1 = refill
#pragma unroll 1
            for (int round = 0; round < (fused ? 1 : 2); ++round)
            {
                const bool count = round == 0 && !first_fill, refill = fused || round == 1;
                if (count || refill)
                {
#pragma unroll 1
                    for (int g = 0; g < FPC; ++g)
                        if ((mask >> g) & 1u)
                        {
                            const bool rf = refill && ((gm >> g) & 1u);
                            if (count || rf) frame_pass(g, count, rf, new_frame(g));
                        }
                    __syncthreads();
                }
#ifdef B200_PHASE_TIMING
                if (round == 0) pt_rf[0] += clock64() - rf0;
#endif
                if (round == 0) bookkeeping();
                if (!fused && round == 0)
                {
                    if (outputs)
                    {
                        __syncthreads();
                        for (int g = 0; g < FPC; ++g)
                            if ((mask >> g) & 1u)
                            {
                                const int eo = (g / VEC) * 16 + (g % VEC) * TS;
                                const unsigned long long fr = s_old[g];
                                const size_t o = (size_t)fr * p.nc;
                                if (p.llr_out || p.hard_out)
                                    for (int i = tid; i < p.nc; i += nthreads)
                                    {
                                        const T v = Acc<SMEM, T, 0>::ld(out + eo + p.var_pos[i] * RS);
                                        if (p.llr_out) p.llr_out[o + i] = (double)v;
                                        if (p.hard_out) p.hard_out[o + i] = (v <= T(0)) ? 1 : 0; // decoder.cpp:58
                                    }
                                if (p.hard_bits)
                                { // bit-packed decisions: bit i%32 of word i/32, rows of hard_words 32-bit words per frame
                                    uint32_t *dst = p.hard_bits + (size_t)fr * p.hard_words;
                                    for (int i0 = 32 * warp; i0 < p.nc; i0 += 32 * (nthreads >> 5))
                                    {
                                        const int i = i0 + lane;
                                        const bool one = i < p.nc && Acc<SMEM, T, 0>::ld(out + eo + p.var_pos[i] * RS) <= T(0);
                                        const uint32_t wbits = __ballot_sync(0xffffffffu, one);
                                        if (lane == 0) dst[i0 >> 5] = wbits;
                                    }
                                }
                                if (tid == 0 && p.iters_out) p.iters_out[fr] = s_ret[g];
                            }
                    }
                    __syncthreads(); // the old posteriors and information words have been consumed
                    if (p.g_rows > 0 && gm)
                    {
                        for (int g = 0; g < FPC; ++g)
                            if ((gm >> g) & 1u) draw_info_word(g, new_frame(g));
                        __syncthreads();
                    }
                }
            }
            next_k += n_new;
            active = (active & ~mask) | gm;
            skip = as_skip ? gm : 0u;
            fresh |= gm;
            cn_stale = true;
            vn_stale = true;
#ifdef B200_PHASE_TIMING
            pt_refill += clock64() - rf0;
            pt_nrefill += 1;
#endif
        };

        const P c2v_lane = c2v + lane * 16, c2v_sub = c2v + sub * 16, out_sub = out + sub * 16;
        const P out_lane = out + lane * 16, llr_lane = llr + lane * 16;
        const P cn_seg_w = cn_seg + 16 * p.cn_max_segs * warp, vn_seg_w = vn_seg + 16 * p.vn_max_segs * warp;

#ifdef B200_PHASE_TIMING
        long long pt_cn = 0, pt_wb = 0, pt_vn = 0, pt_wa = 0, pt_n = 0, pt_hdr = 0, pt_nseg = 0, pt_ntask = 0, pt_rel = 0;
        __shared__ long long s_pt[2][32]; // work-end time stamps of the warps (a barrier releases at their maximum)
        long long pt_vcyc[3] = {0, 0, 0}, pt_vtask[3] = {0, 0, 0};
#endif
        // state of the half-iteration loop (ET kernels, below)
        uint32_t pend_mask = ALL, pend_synd = 0, pend_started = 0; // the initial fill is the first event
        bool pend_skip = false, pend_first = true, pend_clear = false;
        int par_i = 1; // parity of the iteration in progress (double-buffered control words); the first check half makes it 0
#ifdef B200_PHASE_TIMING
        long long pt1 = 0, pt2 = 0;
#endif
        // ---- check-node phase (+ syndrome of the previous iteration's decisions, ORed into `bad`: ET kernels) -----
        uint32_t bad = 0;
        auto cn_phase = [&](auto csrc)
        {
            constexpr int CSRC = decltype(csrc)::value;
            const uint32_t fz = (fresh >> (sub * VEC)) & VMASK;
            uint32_t tc = tm_w;
            uint4 sg_next = WAcc<SMEM, 0>::ld4(cn_seg_w);
            for (P sp = cn_seg_w;;)
            {
#ifdef B200_PHASE_TIMING
                const long long ph0 = clock64();
#endif
                const uint4 sg = SMEM ? uniform4(sg_next) : sg_next;
                if (sg.x == 0) break;
                sp += 16;
                sg_next = WAcc<SMEM, 0>::ld4(sp); // the next descriptor (or the terminator) is in flight while this segment runs
                // threads of nodes missing from a ragged task run along on padded slots / zero index entries
                const int deg = (int)(sg.x & 0xFFu);
                const uint32_t keep = (j < (int)((sg.x >> 8) & 0xFFu)) ? 0xFFFFFFFFu : 0u;
                int nt = (int)(sg.x >> 16);
                P c2v0 = c2v_lane + sg.y;
                const P ib = cn_idx + sg.z;
#ifdef B200_PHASE_TIMING
#define B200_PT_HDR pt_hdr += clock64() - ph0; pt_nseg += 1; pt_ntask += nt;
#else
#define B200_PT_HDR
#endif
#define B200_CN_CASE(D)                                                                                      \
    case D:                                                                                                  \
    {                                                                                                        \
        constexpr int ST = idx_stride_of(D, ISZ);                                                            \
        P ip = ib + j * (ST < 16 ? ST : 16);                                                                 \
        uint32_t nx[D];                                                                                      \
        IdxLoad<SMEM, IdxT, LANES, D>::load(ip, nx);                                                         \
        B200_PT_HDR                                                                                          \
        _Pragma("unroll 1") for (; nt > 0; --nt)                                                             \
        {                                                                                                    \
            if constexpr (B200_BP_CALL_FROM > 0 && SMEM && ALG == ALG_BP && sizeof(T) == 8 && D >= B200_BP_CALL_FROM) \
                bad |= cn4_call<T, IdxT, SMEM, LANES, ALG, D, CSRC, TM, ET>(out_sub, c2v0, ip, tc, fz) & keep; \
            ip += NPW * ST;                                                                                  \
            if constexpr (!(B200_BP_CALL_FROM > 0 && SMEM && ALG == ALG_BP && sizeof(T) == 8 && D >= B200_BP_CALL_FROM)) \
                bad |= Cn4<T, IdxT, SMEM, LANES, ALG, D>::template run<CSRC, TM, ET>(out_sub, c2v0, nx, ip, nt > 1, tc, fz) & keep; \
            c2v0 += D * 512;                                                                                 \
            if constexpr (TM) tc += 4 * D;                                                                   \
        }                                                                                                    \
        break;                                                                                               \
    }
                switch (deg) // warp-uniform
                {
                    B200_CN_CASE(2)
                    B200_CN_CASE(3)
                    B200_CN_CASE(4)
                    B200_CN_CASE(5)
                    B200_CN_CASE(6)
                    B200_CN_CASE(7)
                    B200_CN_CASE(8)
                default: // not mirrored: always served from shared / global memory
                {
                    const int st = idx_stride_of(deg, ISZ);
                    P ip = ib + j * 16;
                    for (; nt > 0; --nt)
                    {
                        bad |= cn4_any<T, IdxT, SMEM, LANES, ALG>(out_sub, c2v0, ip, deg, CSRC == 4 ? VMASK : CSRC >= 2 ? fz : 0u) & keep;
                        c2v0 += deg * 512;
                        ip += NPW * st;
                    }
                    break;
                }
                }
#undef B200_CN_CASE
            }
            if constexpr (TM) tm_wait_st();
        };
        // ---- variable-node phase: posterior (hard decision = its sign, taken where it is consumed); frame lanes outside
        //      `mylive` (bits of this thread's vector) keep their posterior.  The lock-step loop never clears a bit. ----
        uint32_t mylive = VMASK;
        auto vn_phase = [&](auto lsrc)
        {
            constexpr int LSRC = decltype(lsrc)::value;
            uint32_t tl = tm_w + p.tm_vn_off;
            uint4 sg_next = WAcc<SMEM, 0>::ld4(vn_seg_w);
            for (P sp = vn_seg_w;;)
            {
                const uint4 sg = SMEM ? uniform4(sg_next) : sg_next;
                if (sg.x == 0) break;
                sp += 16;
                sg_next = WAcc<SMEM, 0>::ld4(sp);
                const int deg = (int)(sg.x & 0xFFu);
                int nt = (int)(sg.x >> 16);
#ifdef B200_PHASE_TIMING
                const long long vs0 = clock64();
                const int vcls = deg == 1 ? 0 : deg == 2 ? 1 : 2;
                pt_vtask[vcls] += nt;
#endif
                P lp = llr_lane + sg.y, op = out_lane + sg.y;
                const P ib = vn_idx + sg.z;
                auto channel_llr = [&]() -> V // decoder.cpp:50
                {
                    V a;
                    if constexpr (LSRC == 1) { a = TmAcc<T>::ld(tl); tm_wait_ld(); }
                    else
                    {
                        a = VAcc<SMEM, T, 0>::ld(lp);
                        if constexpr (TM) TmAcc<T>::st(tl, a);
                    }
                    return a;
                };
                auto finish = [&](const V &acc)
                {
                    if (mylive == VMASK) VAcc<SMEM, T, 0>::st(op, acc);
                    else
                    {
#pragma unroll
                        for (int e = 0; e < VEC; ++e)
                            if ((mylive >> e) & 1u) Acc<SMEM, T, 0>::st(op + e * TS, acc.e[e]);
                    }
                    lp += 512;
                    op += 512;
                    if constexpr (TM) tl += 4;
                };
#define B200_VN_CASE(D)                                                                                      \
    case D:                                                                                                  \
    {                                                                                                        \
        constexpr int ST = idx_stride_of(D, ISZ);                                                            \
        P ip = ib + j * (ST < 16 ? ST : 16);                                                                 \
        uint32_t nx[D];                                                                                      \
        IdxLoad<SMEM, IdxT, LANES, D>::load(ip, nx);                                                         \
        _Pragma("unroll 1") for (; nt > 0; --nt)                                                             \
        {                                                                                                    \
            ip += NPW * ST;                                                                                  \
            finish(Vn4<T, IdxT, SMEM, LANES, D>::run(c2v_sub, nx, ip, nt > 1, channel_llr()));               \
        }                                                                                                    \
        break;                                                                                               \
    }
                switch (deg)
                {
                case 0:
                    for (; nt > 0; --nt) finish(channel_llr());
                    break;
                    B200_VN_CASE(1)
                    B200_VN_CASE(2)
                    B200_VN_CASE(3)
                    B200_VN_CASE(4)
                    B200_VN_CASE(5)
                    B200_VN_CASE(6)
                    B200_VN_CASE(7)
                    B200_VN_CASE(8)
                default:
                {
                    auto generic = [&]()
                    {
                        const int st = idx_stride_of(deg, ISZ);
                        P ip = ib + j * 16;
                        for (; nt > 0; --nt)
                        {
                            finish(vn4_any<T, IdxT, SMEM, LANES>(c2v_sub, ip, deg, channel_llr()));
                            ip += NPW * st;
                        }
                    };
                    if constexpr (SMEM)
                    { // the 128-register kernels also unroll degrees 9..16: every gather of the node is in flight before the
                      // (strictly ordered) additions start
                        switch (deg)
                        {
                            B200_VN_CASE(9)
                            B200_VN_CASE(10)
                            B200_VN_CASE(11)
                            B200_VN_CASE(12)
                            B200_VN_CASE(13)
                            B200_VN_CASE(14)
                            B200_VN_CASE(15)
                            B200_VN_CASE(16)
                        default: generic(); break;
                        }
                    }
                    else generic();
                    break;
                }
                }
#undef B200_VN_CASE
#ifdef B200_PHASE_TIMING
                pt_vcyc[vcls] += clock64() - vs0;
#endif
            }
            if constexpr (TM && LSRC == 0) tm_wait_st();
        };


        // The retire / refill event has exactly ONE call site per kernel.  (The event is ~1 k instructions of cold code; inlined at
        // three sites it no longer shared the 32 KB instruction cache with the decode loop and every event paid for instruction
        // fetches from L2.)
        if constexpr (!ET)
        {
            // ---- the phases of the lock-step kernel: the same bodies, the descriptors read from the parameter bank (uniform) and
            //      the gather addresses from TMEM (written by the prologue), one task ahead.  CSRC 4 / LSRC 0: first iteration of a
            //      batch (no old c2v; the channel LLRs are read from shared memory and mirrored) -----------------------------
            auto cn_phase_ls = [&](auto csrc)
            {
                constexpr int CSRC = decltype(csrc)::value;
                uint32_t tc = tm_w, ti = tm_w + p.tm_idx_off;
                for (int s = warp * p.cn_max_segs;; ++s)
                {
                    const uint4 sg = make_uint4(p.ls_seg[4 * s], p.ls_seg[4 * s + 1], p.ls_seg[4 * s + 2], 0u);
                    if (sg.x == 0) break;
                    const int deg = (int)(sg.x & 0xFFu);
                    int nt = (int)(sg.x >> 16);
                    P c2v0 = c2v_lane + sg.y;
#define B200_CN_LS_CASE(D)                                                                                   \
    case D:                                                                                                  \
    {                                                                                                        \
        uint32_t nx[D];                                                                                      \
        tm_ld_idx<D>(ti, nx);                                                                                \
        tm_wait_ld();                                                                                        \
        _Pragma("unroll 1") for (; nt > 0; --nt)                                                             \
        {                                                                                                    \
            ti += ls_idx_cols(true, D);                                                                      \
            Cn4<T, IdxT, SMEM, LANES, ALG, D>::template run_ls<CSRC>(nx, ti, nt > 1, c2v0, tc);              \
            c2v0 += D * 512;                                                                                 \
            tc += 4 * D;                                                                                     \
        }                                                                                                    \
        break;                                                                                               \
        }
                    switch (deg) // warp-uniform
                    {
                        B200_CN_LS_CASE(2)
                        B200_CN_LS_CASE(3)
                        B200_CN_LS_CASE(4)
                        B200_CN_LS_CASE(5)
                        B200_CN_LS_CASE(6)
                        B200_CN_LS_CASE(7)
                        B200_CN_LS_CASE(8)
                    default: // neither mirrored nor in TMEM: index tables and c2v in shared memory
                    {
                        const int st = idx_stride_of(deg, ISZ);
                        P ip = cn_idx + sg.z + j * 16;
                        for (; nt > 0; --nt)
                        {
                            cn4_any<T, IdxT, SMEM, LANES, ALG>(out_sub, c2v0, ip, deg, CSRC == 4 ? VMASK : 0u);
                            c2v0 += deg * 512;
                            ip += NPW * st;
                        }
                        break;
                    }
                    }
#undef B200_CN_LS_CASE
                }
                tm_wait_st();
            };
            auto vn_phase_ls = [&](auto lsrc)
            {
                constexpr int LSRC = decltype(lsrc)::value;
                // the variable-side addresses follow the warp's check-side ones: the first variable descriptor's last word holds
                // the check-side column count (Engine::launch)
                const int s0 = warps * p.cn_max_segs + warp * p.vn_max_segs;
                uint32_t tl = tm_w + p.tm_vn_off, ti = tm_w + p.tm_idx_off + p.ls_seg[4 * s0 + 3];
                for (int s = s0;; ++s)
                {
                    const uint4 sg = make_uint4(p.ls_seg[4 * s], p.ls_seg[4 * s + 1], p.ls_seg[4 * s + 2], 0u);
                    if (sg.x == 0) break;
                    const int deg = (int)(sg.x & 0xFFu);
                    int nt = (int)(sg.x >> 16);
                    P lp = llr_lane + sg.y, op = out_lane + sg.y;
                    // channel LLR (decoder.cpp:50); from the mirror its wait also covers the gather addresses loaded by the last task
                    auto channel_llr = [&]() -> V
                    {
                        V a;
                        if constexpr (LSRC == 1) a = TmAcc<T>::ld(tl);
                        else
                        {
                            a = VAcc<SMEM, T, 0>::ld(lp);
                            TmAcc<T>::st(tl, a);
                        }
                        tm_wait_ld();
                        return a;
                    };
                    auto finish = [&](const V &acc)
                    {
                        VAcc<SMEM, T, 0>::st(op, acc);
                        lp += 512;
                        op += 512;
                        tl += 4;
                    };
#define B200_VN_LS_CASE(D)                                                                                   \
    case D:                                                                                                  \
    {                                                                                                        \
        uint32_t nx[D];                                                                                      \
        tm_ld_idx<D>(ti, nx);                                                                                \
        _Pragma("unroll 1") for (; nt > 0; --nt)                                                             \
        {                                                                                                    \
            ti += ls_idx_cols(false, D);                                                                     \
            const V a = channel_llr();                                                                       \
            finish(Vn4<T, IdxT, SMEM, LANES, D>::run_ls(nx, ti, nt > 1, a));                                 \
        }                                                                                                    \
        break;                                                                                               \
        }
                    switch (deg)
                    {
                    case 0:
                        for (; nt > 0; --nt) finish(channel_llr());
                        break;
                        B200_VN_LS_CASE(1)
                        B200_VN_LS_CASE(2)
                        B200_VN_LS_CASE(3)
                        B200_VN_LS_CASE(4)
                        B200_VN_LS_CASE(5)
                        B200_VN_LS_CASE(6)
                        B200_VN_LS_CASE(7)
                        B200_VN_LS_CASE(8)
                        B200_VN_LS_CASE(9)
                        B200_VN_LS_CASE(10)
                        B200_VN_LS_CASE(11)
                        B200_VN_LS_CASE(12)
                        B200_VN_LS_CASE(13)
                        B200_VN_LS_CASE(14)
                        B200_VN_LS_CASE(15)
                        B200_VN_LS_CASE(16)
                    default:
                    {
                        const int st = idx_stride_of(deg, ISZ);
                        P ip = vn_idx + sg.z + j * 16;
                        for (; nt > 0; --nt)
                        {
                            finish(vn4_any<T, IdxT, SMEM, LANES>(c2v_sub, ip, deg, channel_llr()));
                            ip += NPW * st;
                        }
                        break;
                    }
                    }
#undef B200_VN_LS_CASE
                }
                if constexpr (LSRC == 0) tm_wait_st();
            };

            // Without early termination every frame lane of the CTA is filled by the same event and reaches max_iter in the same
            // iteration, so the CTA decodes in lock-step batches: fill, max_iter x (check phase, barrier, variable phase,
            // barrier), retire -- the event's call site is the top of a batch and nothing is decided per half iteration.  In a
            // ragged last batch the lanes without a frame compute on whatever their slots hold (arithmetic on shared memory and
            // TMEM only, nothing can fault); nothing reads those lanes.
            for (bool first = true;; first = false)
            {
                retire_and_refill(first ? ALL : active, 0u, 0u, false, first);
                if (!active) break; // CTA-uniform
                for (int i = 0; i < p.max_iter; ++i)
                {
                    // first iteration of a batch: every old c2v is +0 and the channel LLRs sit in shared memory only (the variable
                    // phase refreshes their mirror); the later ones read the mirror
                    if (i == 0) cn_phase_ls(std::integral_constant<int, 4>{});
                    else cn_phase_ls(std::integral_constant<int, 1>{});
#ifdef B200_PHASE_TIMING
                    pt1 = clock64();
                    if (lane == 0) s_pt[0][warp] = pt1;
#endif
                    __syncthreads(); // B
#ifdef B200_PHASE_TIMING
                    pt2 = 0;
                    for (int w = 0; w < warps; ++w) pt2 = max(pt2, s_pt[0][w]);
#endif
                    if (i == 0) vn_phase_ls(std::integral_constant<int, 0>{});
                    else vn_phase_ls(std::integral_constant<int, 1>{});
#ifdef B200_PHASE_TIMING
                    const long long pt3 = clock64();
                    if (lane == 0) s_pt[1][warp] = pt3;
#endif
                    __syncthreads(); // A
#ifdef B200_PHASE_TIMING
                    long long pt4 = 0;
                    for (int w = 0; w < warps; ++w) pt4 = max(pt4, s_pt[1][w]);
                    if (pt_rel) { pt_cn += pt1 - pt_rel; pt_wb += pt2 - pt1; pt_vn += pt3 - pt2; pt_wa += pt4 - pt3; ++pt_n; }
                    pt_rel = pt4;
#endif
                }
                it = p.max_iter;
            }
        }
        else
        {
        // The loop advances by HALF iterations (even h: check phase, odd h: variable phase) so that the event can be called at
        // the top of a half: a frame lane found finished is recorded as pending and handled when the next half begins.
        for (uint32_t h = 0;; ++h)
        {
            if (pend_mask)
            {
                retire_and_refill(pend_mask, pend_synd, pend_started, pend_skip, pend_first);
                if (pend_clear && warp == 0 && lane == 0) s_ctrl[par_i ^ 1].x &= ~pend_mask; // consumed (everyone read it before the event's barriers)
                pend_mask = 0; pend_first = false; pend_clear = false;
            }
            if (!(h & 1u))
            {
            if (!active) break; // CTA-uniform
            par_i ^= 1;

            // ---- check-node phase (+ syndrome of the previous iteration's decisions) ----------
            bad = 0;
            // right after a refill the fresh lanes' old c2v is forced to +0 (the mirror itself never goes stale: the check
            // phase is the only writer of c2v and writes through)
            if (!cn_stale) cn_phase(std::integral_constant<int, TM ? 1 : 0>{});
            else cn_phase(std::integral_constant<int, TM ? 3 : 2>{});
            cn_stale = false;
            fresh = 0;
            // syndrome flags per frame lane: frame = sub*VEC + e
            if constexpr (ET)
            {
                const uint32_t m = __reduce_or_sync(0xffffffffu, bad << (sub * VEC));
                if (lane == 0 && m) atomicOr(&s_synd[par_i], m);
            }
#ifdef B200_PHASE_TIMING
            pt1 = clock64();
            if (lane == 0) s_pt[0][warp] = pt1;
#endif
            __syncthreads(); // B
#ifdef B200_PHASE_TIMING
            pt2 = 0; // release time of barrier B = arrival of the last warp
            for (int w = 0; w < warps; ++w) pt2 = max(pt2, s_pt[0][w]);
#endif

            // ---- decision: converged (decoder.cpp:66-72) or out of iterations: retired when the variable half begins; the
            //      new frames sit out that variable phase ---------------------
            {
                const uint32_t synd = s_synd[par_i];
                const uint2 ctrl = s_ctrl[par_i];
                const uint32_t done = active & (((ET && p.early_term) ? (~synd & ctrl.y) : 0u) | ctrl.x);
                if (done) { pend_mask = done; pend_synd = synd; pend_started = ctrl.y; pend_skip = true; }
            }
            }
            else
            {
            // bookkeeping for the variable phase that follows and the next decision
            const uint32_t live = active & ~skip;
            if (warp == 0)
            {
                if (lane < FPC && ((live >> lane) & 1u)) ++it;
                const bool act = lane < FPC && ((active >> lane) & 1u);
                const uint32_t started = __ballot_sync(0xffffffffu, act && it >= 1);
                const uint32_t limit = __ballot_sync(0xffffffffu, act && it >= p.max_iter);
                if (lane == 0) { s_ctrl[par_i ^ 1] = make_uint2(limit, started); s_synd[par_i ^ 1] = 0; }
            }

            // ---- variable-node phase: posterior (hard decision = its sign, taken where it is consumed) ----
            mylive = (live >> (sub * VEC)) & VMASK;
            if (live)
            {
                if (TM && !vn_stale) vn_phase(std::integral_constant<int, TM ? 1 : 0>{});
                else vn_phase(std::integral_constant<int, 0>{});
                vn_stale = false;
            }
            skip = 0;
#ifdef B200_PHASE_TIMING
            const long long pt3 = clock64();
            if (lane == 0) s_pt[1][warp] = pt3;
#endif
            __syncthreads(); // A: variable-phase writes visible to the next check phase
#ifdef B200_PHASE_TIMING
            long long pt4 = 0; // release time of barrier A
            for (int w = 0; w < warps; ++w) pt4 = max(pt4, s_pt[1][w]);
            if (pt_rel) { pt_cn += pt1 - pt_rel; pt_wb += pt2 - pt1; pt_vn += pt3 - pt2; pt_wa += pt4 - pt3; ++pt_n; }
            pt_rel = pt4;
#endif
            // ---- without early termination a frame at the iteration limit retires before a check phase is spent on it
            //      (its result is fixed: decoder.cpp:22,74-77); its successor joins the next check phase
            if (!ET || !p.early_term)
            {
                const uint32_t lim = s_ctrl[par_i ^ 1].x & active;
                if (lim) { pend_mask = lim; pend_synd = 0; pend_started = 0; pend_skip = false; pend_clear = true; }
            }
            }
        }
        }
#ifdef B200_PHASE_TIMING
        if (blockIdx.x == 0 && lane == 0)
            printf("warp %2d: iterations %lld  check work %lld  wait-B %lld  decision+variable work %lld  wait-A %lld  (cycles per iteration, from barrier release); check segments/it %lld tasks/it %lld header cycles/seg %lld\n", warp, pt_n,
                   pt_cn / pt_n, pt_wb / pt_n, pt_vn / pt_n, pt_wa / pt_n, pt_nseg / pt_n, pt_ntask / pt_n, pt_hdr / (pt_nseg ? pt_nseg : 1));
        if (blockIdx.x == 0 && tid == 0)
            printf("refills: %lld events, %lld cycles each (pass + barrier %lld: block loop %lld, punctured/shortened %lld, count reduce %lld); iterations %lld\n", pt_nrefill,
                   pt_refill / (pt_nrefill ? pt_nrefill : 1), pt_rf[0] / (pt_nrefill ? pt_nrefill : 1), pt_rf[1] / (pt_nrefill ? pt_nrefill : 1),
                   pt_rf[2] / (pt_nrefill ? pt_nrefill : 1), pt_rf[3] / (pt_nrefill ? pt_nrefill : 1), pt_n);
        if (blockIdx.x == 0 && lane == 0)
            printf("warp %2d: variable segments: deg1 %lld tasks/it %lld cycles/task | deg2 %lld tasks/it %lld cycles/task | other %lld tasks/it %lld cycles/task\n", warp,
                   pt_vtask[0] / (pt_n + 1), pt_vcyc[0] / (pt_vtask[0] ? pt_vtask[0] : 1), pt_vtask[1] / (pt_n + 1), pt_vcyc[1] / (pt_vtask[1] ? pt_vtask[1] : 1),
                   pt_vtask[2] / (pt_n + 1), pt_vcyc[2] / (pt_vtask[2] ? pt_vtask[2] : 1));
#endif

        __syncthreads();
        if (tid < FPC)
        {
            const LaneCnt c = s_cnt[tid];
            if (c.fec) atomicAdd(&p.counters[0], (unsigned long long)c.fec);
            if (c.bec) atomicAdd(&p.counters[1], c.bec);
            if (c.frames) atomicAdd(&p.counters[2], (unsigned long long)c.frames);
            if (c.ret) atomicAdd(&p.counters[3], c.ret);
            if (c.its) atomicAdd(&p.counters[4], c.its);
        }
        if constexpr (TM)
        {
            if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s_tmem), "r"(p.tm_alloc_cols) : "memory");
        }
    }
} // namespace b200
