// Device-side building blocks shared by the sm_100a kernels of the decode hot path (tile4.cuh: BP / min-sum,
// bec_kernel.cuh: erasure decoder, engine.cu: stand-alone channel kernel): the counter-based Philox4x32-10
// channel stream, memory-space access policies (shared window with explicit ld/st.shared, or global memory),
// numeric helpers and the pairwise box-plus of the reference (src/decoding/decoder.h:12-15).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b200
{
    // ------------------------------------------------------------------------------------------
    // Philox4x32-10 (Salmon et al., SC'11) — counter-based, stateless
    // ------------------------------------------------------------------------------------------
    struct u32x4 { uint32_t x, y, z, w; };

    __host__ __device__ __forceinline__ u32x4 philox4x32_10(u32x4 c, uint32_t k0, uint32_t k1)
    {
        for (int r = 0; r < 10; ++r)
        {
            const uint64_t p0 = (uint64_t)0xD2511F53u * c.x;
            const uint64_t p1 = (uint64_t)0xCD9E8D57u * c.z;
            u32x4 n;
            n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k0;
            n.y = (uint32_t)p1;
            n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k1;
            n.w = (uint32_t)p0;
            c = n;
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        return c;
    }

    // counter = (block index j, frame lo, frame hi, point | stream << 24), key = seed
    __host__ __device__ __forceinline__ u32x4 channel_block(uint64_t seed, uint32_t point, uint32_t stream, uint64_t frame, uint32_t j)
    {
        u32x4 c = {j, (uint32_t)frame, (uint32_t)(frame >> 32), (point & 0xFFFFFFu) | (stream << 24)};
        return philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    }

    // Standard-normal pair of the channel specification (oracle/ldpc_oracle.c normal_pair_v2 is the same arithmetic, bit for
    // bit): Box-Muller in binary32 with correctly rounded operations only (+, *, fma, 1/x, sqrt; explicit intrinsics so that
    // nothing is contracted or reordered).  wr: 32 radius bits; wa: bits 7..0 extend the radius uniform to 40 bits (tails to
    // 7.4 sigma), bits 31..8 are the angle (octant + 21-bit fraction).  ~60 instructions per pair, no library call, no fp64.
    __device__ __forceinline__ void normal_pair(uint32_t wr, uint32_t wa, float &z0, float &z1)
    {
        const unsigned long long T = ((((unsigned long long)wr << 8) | (unsigned long long)(wa & 0xFFu)) << 1) | 1ull; // 2U+1 < 2^41
        const uint32_t tb = __float_as_uint(__ull2float_rz(T)); // truncation: exponent 40 - lz, top 24 bits
        float f = __uint_as_float((tb & 0x7FFFFFu) | 0x3F800000u);
        int e = 168 - (int)(tb >> 23); // 41 - (exponent - 127): u1 ~ f 2^-e
        const bool big = f > 1.41421354f;
        f = big ? __fmul_rn(f, 0.5f) : f;
        e = big ? e - 1 : e;
        const float g = __fadd_rn(f, -1.0f);
        const float s = __fmul_rn(g, __frcp_rn(__fadd_rn(2.0f, g)));
        const float s2 = __fmul_rn(s, s);
        float q = 0x1.c71c72p-4f;
        q = __fmaf_rn(q, s2, 0x1.24924ap-3f);
        q = __fmaf_rn(q, s2, 0x1.99999ap-3f);
        q = __fmaf_rn(q, s2, 0x1.555556p-2f);
        q = __fmaf_rn(q, s2, 1.0f);
        const float lnf = __fmul_rn(__fmul_rn(2.0f, s), q);
        const float n = __fmaf_rn((float)e, 0x1.62e430p-1f, -lnf);
        const float r = __fsqrt_rn(__fmul_rn(2.0f, n));
        const uint32_t a = wa >> 8, oct = a >> 21;
        const float phi = __fmul_rn(__fadd_rn((float)(a & 0x1FFFFFu), 0.5f), 0x1.921fb6p-22f);
        const float x2 = __fmul_rn(phi, phi);
        float sp = 0x1.71de3ap-19f;
        sp = __fmaf_rn(sp, x2, -0x1.a01a02p-13f);
        sp = __fmaf_rn(sp, x2, 0x1.111112p-7f);
        sp = __fmaf_rn(sp, x2, -0x1.555556p-3f);
        const float sn0 = __fmaf_rn(__fmul_rn(phi, x2), sp, phi);
        float cp = -0x1.27e4fcp-22f;
        cp = __fmaf_rn(cp, x2, 0x1.a01a02p-16f);
        cp = __fmaf_rn(cp, x2, -0x1.6c16c2p-10f);
        cp = __fmaf_rn(cp, x2, 0x1.555556p-5f);
        cp = __fmaf_rn(cp, x2, -0.5f);
        const float cs0 = __fmaf_rn(cp, x2, 1.0f);
        float c = (oct & 1u) ? sn0 : cs0, sn = (oct & 1u) ? cs0 : sn0;
        if (oct & 2u) { const float t = c; c = -sn; sn = t; }
        if (oct & 4u) { c = -c; sn = -sn; }
        z0 = __fmul_rn(r, c);
        z1 = __fmul_rn(r, sn);
    }

    // Rayleigh fading coefficient c of a frame (DESIGN.md §3.2): the first normal pair (a, b) of Philox block c of stream 3,
    // h = sqrt((a^2 + b^2) / 2) in fp64, so E[h^2] = 1.  The squares of binary32 values are exact in fp64, the sum is rounded
    // once, the halving is exact and the square root is correctly rounded: the oracle's sqrt gives the same bits.
    __device__ __forceinline__ double rayleigh_coeff(uint64_t seed, uint32_t point, uint64_t frame, uint32_t c)
    {
        const u32x4 r = channel_block(seed, point, 3, frame, c);
        float a, b;
        normal_pair(r.x, r.y, a, b);
        const double s = __dadd_rn(__dmul_rn((double)a, (double)a), __dmul_rn((double)b, (double)b));
        return __dsqrt_rn(__dmul_rn(0.5, s));
    }

    // SRC_ASK: AWGN with M-ASK + bit-metric decoding; SRC_RAYLEIGH: BPSK over flat Rayleigh fading, perfect CSI
    enum { SRC_LLR = 0, SRC_AWGN = 1, SRC_BSC = 2, SRC_BEC = 3, SRC_ASK = 4, SRC_RAYLEIGH = 5 };

    // M-ASK with bit-metric decoding (legacy tree gpu/device/kernel.cpp:141-219, gpu/sim/ldpcsim.cpp:240-323; specification:
    // oracle/ldpc_oracle.c orc_channel_frame_ask).  Tables in global memory.
    struct AskParams
    {
        int M, bits, n_sym;
        const double *X;  // [M] constellation points, unit average energy
        const int32_t *label, *rev; // [M] label of point j / point of label l
        const int32_t *bm; // [bits][n_sym] variable id carrying bit level k of symbol i
    };
    // One symbol: scrambling bits of its variables -> point -> y -> bit-metric LLRs (already multiplied by 1 - 2c).  z: the
    // symbol's standard normal.  put(variable id, LLR, scrambling bit) is called once per bit level.
    template <typename F>
    __device__ __forceinline__ void ask_symbol(const AskParams &a, uint64_t seed, uint32_t point, uint64_t frame, int i, float z, double sigma,
                                               double sigma2, F &&put)
    {
        int tmp = 0;
        uint32_t cbit[8];
        for (int k = 0; k < a.bits; ++k)
        {
            const int v = a.bm[k * a.n_sym + i];
            const u32x4 w = channel_block(seed, point, 2, frame, (uint32_t)v >> 7);
            const uint32_t q4[4] = {w.x, w.y, w.z, w.w};
            cbit[k] = (q4[(v >> 5) & 3] >> (v & 31)) & 1u;
            tmp += (int)cbit[k] << (a.bits - 1 - k);
        }
        const double y = __dadd_rn(__dmul_rn((double)z, sigma), a.X[a.rev[tmp]]);
        for (int k = 0; k < a.bits; ++k)
        {
            double t0 = 0, t1 = 0;
            for (int j = 0; j < a.M; ++j)
            {
                const double d = y - a.X[j];
                const double e = exp(-d * d / (2 * sigma2)) * (1.0 / a.M);
                if (a.label[j] & (1 << (a.bits - 1 - k))) t1 += e; else t0 += e;
            }
            double val = log(t0 / t1);
            if (isinf(val)) val = val > 0 ? 9999.9 : -9999.9;
            put(a.bm[k * a.n_sym + i], cbit[k] ? -val : val, cbit[k]);
        }
    }
    enum { ALG_MS = 0, ALG_BP = 1 };
    constexpr uint32_t IDLE = 0xFFFFFFFFu;

    // ------------------------------------------------------------------------------------------
    // memory-space policies: shared window (32-bit byte addresses, explicit ld/st.shared so that no
    // generic-address arithmetic is rematerialised in the inner loops) or global memory
    // ------------------------------------------------------------------------------------------
    // (explicit overload set instead of partial specialisation: OFF must be an immediate)
#define B200_SMEM_LD(NAME, TYPE, PTXT, CONS)                                                        \
    template <int OFF> __device__ __forceinline__ TYPE NAME(uint32_t a)                             \
    {                                                                                               \
        TYPE v;                                                                                     \
        asm volatile("ld.shared." PTXT " %0, [%1+%2];" : "=" CONS(v) : "r"(a), "n"(OFF));           \
        return v;                                                                                   \
    }
#define B200_SMEM_ST(NAME, TYPE, PTXT, CONS)                                                        \
    template <int OFF> __device__ __forceinline__ void NAME(uint32_t a, TYPE v)                     \
    {                                                                                               \
        asm volatile("st.shared." PTXT " [%0+%1], %2;" ::"r"(a), "n"(OFF), CONS(v) : "memory");     \
    }
    B200_SMEM_LD(lds_f64, double, "f64", "d")
    B200_SMEM_LD(lds_f32, float, "f32", "f")
    B200_SMEM_LD(lds_u32, uint32_t, "u32", "r")
    B200_SMEM_ST(sts_f64, double, "f64", "d")
    B200_SMEM_ST(sts_f32, float, "f32", "f")
    B200_SMEM_ST(sts_u32, uint32_t, "u32", "r")
    template <int OFF> __device__ __forceinline__ uint32_t lds_u16(uint32_t a)
    {
        uint16_t v;
        asm volatile("ld.shared.u16 %0, [%1+%2];" : "=h"(v) : "r"(a), "n"(OFF));
        return v;
    }
    template <int OFF> __device__ __forceinline__ void sts_u16(uint32_t a, uint32_t v)
    {
        asm volatile("st.shared.u16 [%0+%1], %2;" ::"r"(a), "n"(OFF), "h"((uint16_t)v) : "memory");
    }

    // typed front ends ----------------------------------------------------------------------------
    template <bool SMEM, typename V, int OFF> struct Acc;
    template <int OFF> struct Acc<true, double, OFF>
    {
        static __device__ __forceinline__ double ld(uint32_t a) { return lds_f64<OFF>(a); }
        static __device__ __forceinline__ void st(uint32_t a, double v) { sts_f64<OFF>(a, v); }
    };
    template <int OFF> struct Acc<true, float, OFF>
    {
        static __device__ __forceinline__ float ld(uint32_t a) { return lds_f32<OFF>(a); }
        static __device__ __forceinline__ void st(uint32_t a, float v) { sts_f32<OFF>(a, v); }
    };
    template <int OFF> struct Acc<true, uint32_t, OFF>
    {
        static __device__ __forceinline__ uint32_t ld(uint32_t a) { return lds_u32<OFF>(a); }
        static __device__ __forceinline__ void st(uint32_t a, uint32_t v) { sts_u32<OFF>(a, v); }
    };
    template <int OFF> struct Acc<true, uint16_t, OFF>
    {
        static __device__ __forceinline__ uint32_t ld(uint32_t a) { return lds_u16<OFF>(a); }
        static __device__ __forceinline__ void st(uint32_t a, uint32_t v) { sts_u16<OFF>(a, v); }
    };
    template <typename V, int OFF> struct Acc<false, V, OFF>
    {
        static __device__ __forceinline__ V ld(const unsigned char *a) { return *reinterpret_cast<const V *>(a + OFF); }
        static __device__ __forceinline__ void st(unsigned char *a, V v) { *reinterpret_cast<V *>(a + OFF) = v; }
    };
    template <bool SMEM> struct PtrOf { typedef uint32_t type; };
    template <> struct PtrOf<false> { typedef unsigned char *type; };

    template <typename T> struct Num;
    template <> struct Num<double>
    {
        static __device__ __forceinline__ uint32_t hi(double v) { return (uint32_t)__double2hiint(v); }
        static __device__ __forceinline__ double abs(double v) { return fabs(v); }
        // mag >= 0; sign bit taken from bit 31 of s
        static __device__ __forceinline__ double with_sign(double mag, uint32_t s) { return __hiloint2double(__double2hiint(mag) | (int)(s & 0x80000000u), __double2loint(mag)); }
        static __device__ __forceinline__ double inf() { return __longlong_as_double(0x7ff0000000000000ll); }
        static __device__ __forceinline__ double min_(double a, double b) { return fmin(a, b); }
        static __device__ __forceinline__ double exp_(double v) { return exp(v); }
        static __device__ __forceinline__ double log_(double v) { return log(v); }
    };
    template <> struct Num<float>
    {
        static __device__ __forceinline__ uint32_t hi(float v) { return __float_as_uint(v); }
        static __device__ __forceinline__ float abs(float v) { return fabsf(v); }
        static __device__ __forceinline__ float with_sign(float mag, uint32_t s) { return __uint_as_float(__float_as_uint(mag) | (s & 0x80000000u)); }
        static __device__ __forceinline__ float inf() { return __uint_as_float(0x7f800000u); }
        static __device__ __forceinline__ float min_(float a, float b) { return fminf(a, b); }
        static __device__ __forceinline__ float exp_(float v) { return __expf(v); }
        static __device__ __forceinline__ float log_(float v) { return __logf(v); }
    };

#ifdef __CUDACC__
    // ---- fp64 exponential and the Jacobian correction log((1 + e^-a) / (1 + e^-b)), a, b >= 0, without the math library -----
    // The library exp / log spend a third of a sum-product kernel's issue slots on materialising 64-bit polynomial
    // coefficients (two moves per constant, every call).  Here the coefficients sit in the constant bank and arrive as
    // uniform loads; the logarithm of the ratio is 2 atanh((u - v) / (2 + u + v)), |argument| <= 1/3, so no range
    // reduction, no table.  Accuracy of the pairwise correction against the exact value: 3.1e-16 absolute at most over 2e7
    // random pairs -- the same as the reference's own double expression (3.4e-16); the parity bar needs ~1e-14
    // (profiles/r1/bp_accuracy.md).  The pairwise box-plus serves the layered kernel, checks of degree > 8 and the rare exact
    // path of bp_check below.
    // e^r on |r| <= ln 2 / 2: minimax polynomial of degree 11 (Remez at 60 digits, profiles/gen_bp_tables.py; 1.2e-17 with the
    // coefficients rounded to binary64; the Taylor polynomial needs degree 13 for the same error)
    static __constant__ double BP_EXP_C[12] = {0x1.0000000000000p+0, 0x1.0000000000000p+0, 0x1.0000000000011p-1, 0x1.555555555556ap-3, 0x1.555555554f0b8p-5,
                                               0x1.111111110c4b2p-7, 0x1.6c16c188007dap-10, 0x1.a01a01bec709ap-13, 0x1.a01991a047428p-16, 0x1.71ddd953a34f1p-19,
                                               0x1.28b410c11893dp-22, 0x1.af8db1c459b51p-26};
    static __constant__ double BP_ATH_C[17] = {1.0, 1.0 / 3, 1.0 / 5, 1.0 / 7, 1.0 / 9, 1.0 / 11, 1.0 / 13, 1.0 / 15, 1.0 / 17, 1.0 / 19, 1.0 / 21,
                                               1.0 / 23, 1.0 / 25, 1.0 / 27, 1.0 / 29, 1.0 / 31, 1.0 / 33}; // 1/(2k+1)
    // -log2(e), 1.5 * 2^52 (rounds to an integer in the low mantissa bits), ln 2 high and low part, (argument clamp 708: e^-708 ~ 3e-308)
    static __constant__ double BP_K[5] = {-1.4426950408889634, 6755399441055744.0, 0.6931471803691238, 1.9082149292705877e-10, 708.0};

    __device__ __forceinline__ double bp_exp_neg(double z) // e^-z, z >= 0 (clamped at ~708: e^-708 is still a normal number)
    {
        const double zc = __hiloint2double(min(__double2hiint(z), 0x40862000), __double2loint(z)); // z >= 0: the high words order like integers
        const double t = __fma_rn(zc, BP_K[0], BP_K[1]);
        const double k = t - BP_K[1];               // round(-z log2 e)
        double r = __fma_rn(k, -BP_K[2], -zc);      // -z - k ln 2, |r| <= ln 2 / 2
        r = __fma_rn(k, -BP_K[3], r);
        double p = BP_EXP_C[11];
#pragma unroll
        for (int i = 10; i >= 0; --i) p = __fma_rn(p, r, BP_EXP_C[i]);
        return __hiloint2double(__double2hiint(p) + (int)((uint32_t)__double2loint(t) << 20), __double2loint(p)); // * 2^k (k >= -1022)
    }
    __device__ __forceinline__ double bp_log_ratio(double u, double v) // log((1 + u) / (1 + v)), u, v in [0, 1]
    {
        const double w = (u - v) / ((2.0 + u) + v);
        const double s = w * w;
        double p = BP_ATH_C[16];
#pragma unroll
        for (int i = 15; i >= 0; --i) p = __fma_rn(p, s, BP_ATH_C[i]);
        return 2.0 * w * p;
    }
#endif

    template <typename T> __device__ __forceinline__ T boxplus(T x, T y);

#ifdef __CUDACC__
    // ---- fp64 sum-product check node on E = e^-|x| -----------------------------------------------------------------------
    // The reference evaluates a degree-d check as 3(d-2) pairwise box-plus operations (decoder.cpp:30-44 with decoder.h:12-15:
    // two exp, a division and a log each, ~70 FP64 instructions here).  In terms of E = e^-|x| the magnitude of x [+] y is
    //     E(x [+] y) = (Ex + Ey) / (1 + Ex Ey)                       (tanh(x/2) = (1 - Ex) / (1 + Ex) in the tanh rule)
    // so the same function of the d inputs costs d exponentials, fraction-valued forward / backward products (E = N / D carried
    // as the pair: folding in a raw input is two FMAs, joining a forward with a backward value four operations, no division) and
    // d logarithms log(D / N) -- ~45 FP64 instructions per edge for any degree (d = 7: 3.2 x fewer than the pairwise chain), all
    // of them independent chains instead of one d-deep dependent recursion.  Unlike tanh / atanh this form has no cancellation:
    // E keeps full relative precision down to e^-708, and log(D / N) = e0 ln 2 + 2 atanh((D - N') / (D + N')) with N' = N 2^e0
    // brought within a factor 2^0.59 of D is accurate to ~2e-16 absolute + 1e-16 relative -- the same as the reference's own
    // double expression (tests/study_bp_edomain.py: posteriors after 50 iterations within 1.3e-7 of the oracle's, bar 1e-4).
    // Large inputs: with m = min |x| over the check (taken from the high words), all inputs are shifted by max(0, m - 40) before
    // the exponential and the shift is added back after the logarithm (exact: once every E <= e^-40 the denominators are 1 to
    // 1e-34); an output whose magnitude would exceed ~665 above the shift (inputs beyond the e^-708 clamp decide it: shortened
    // positions at 99999.9) makes the thread redo the check with the reference's pairwise recursion.
    // Per edge: exponential 16 FP64 instructions, logarithm 18 (5 of them the division), ~4 for the products.
    // 2 atanh(w) / w as a function of s = w^2 on [0, 0.0405]: minimax polynomial of degree 7 (6e-17; profiles/gen_bp_tables.py)
    static __constant__ double BP_LOG_C[8] = {0x1.0000000000000p+1, 0x1.55555555558bap-1, 0x1.99999998be9bbp-2, 0x1.249249cc9eae0p-2,
                                              0x1.c71bf34d80545p-3, 0x1.7476dda759777p-3, 0x1.382eecef5e3a5p-3, 0x1.3bc09a1b49468p-3};
    static __constant__ double BP_LOG_K[3] = {0.6931471805599453, 4503601774854144.0 /* 2^52 + 2^31 */, 40.0};

    // log(D / N) + shift for 0 < N <~ D, both normal; far: beyond the range the clamp of bp_exp_neg keeps exact
    __device__ __forceinline__ double bp_log_frac(double N, double D, double shift, bool &far)
    {
        // e0 = round of the difference of the high words (a piecewise-linear log2, off by < 0.086 each): D / (N 2^e0) lies within
        // 2^+-0.59, |w| <= 0.2003
        const int hn = __double2hiint(N), hd = __double2hiint(D);
        const int e0 = (hd - hn + 0x80000) >> 20;
        const double Ns = __hiloint2double(hn + (int)((uint32_t)e0 << 20), __double2loint(N));
        const double num = D - Ns, den = D + Ns;
        // num / den, den in [1, 2^9): reciprocal seed (2^-23), one Newton step, quotient, one residual correction (error e^4)
        double rc;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(rc) : "d"(den));
        rc = __fma_rn(rc, __fma_rn(-den, rc, 1.0), rc);
        double w = num * rc;
        w = __fma_rn(__fma_rn(-den, w, num), rc, w);
        const double s = w * w;
        double p = BP_LOG_C[7];
#pragma unroll
        for (int i = 6; i >= 0; --i) p = __fma_rn(p, s, BP_LOG_C[i]);
        far = e0 > 960;
        const double e0d = __hiloint2double(0x43300000, (int)((uint32_t)e0 ^ 0x80000000u)) - BP_LOG_K[1];
        return __fma_rn(w, p, __fma_rn(e0d, BP_LOG_K[0], shift));
    }

    // E(x [+] y) from E(x), E(y) as a plain number: (a + b) / (1 + a b), a, b in (0, 1] (the arbitrary-degree path)
    __device__ __forceinline__ double bp_join(double a, double b)
    {
        const double num = a + b, den = __fma_rn(a, b, 1.0);
        double rc;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(rc) : "d"(den));
        rc = __fma_rn(rc, __fma_rn(-den, rc, 1.0), rc);
        const double q = num * rc;
        return __fma_rn(__fma_rn(-den, q, num), rc, q);
    }

    // W frame lanes of one check at a time: the fast paths of all lanes form ONE basic block (the rare exact path is tested once,
    // after all of them), so the scheduler interleaves W * D independent chains and every coefficient load serves W lanes.
    template <int D, int W>
    __device__ __forceinline__ void bp_check(const double (&x)[W][D], double (&r)[W][D])
    {
        static_assert(D >= 3, "degree-2 checks swap their inputs");
        uint32_t sx[W];
        double shift[W], E[W][D], FN[W][D - 1], FD[W][D - 1];
#pragma unroll
        for (int w = 0; w < W; ++w)
        {
            uint32_t mh = 0x7fffffffu;
            sx[w] = 0;
#pragma unroll
            for (int k = 0; k < D; ++k)
            {
                const uint32_t h = (uint32_t)__double2hiint(x[w][k]);
                sx[w] ^= h;
                mh = min(mh, h & 0x7fffffffu);
            }
            shift[w] = (mh >= 0x40440000u && mh < 0x7ff00000u) ? __hiloint2double((int)mh, 0) - BP_LOG_K[2] : 0.0;
        }
#pragma unroll
        for (int k = 0; k < D; ++k)
#pragma unroll
            for (int w = 0; w < W; ++w) E[w][k] = bp_exp_neg(fabs(x[w][k]) - shift[w]);
        bool anyfar = false, far;
#pragma unroll
        for (int w = 0; w < W; ++w)
        {
            FN[w][0] = E[w][0];
            FD[w][0] = 1.0;
#pragma unroll
            for (int k = 1; k < D - 1; ++k)
            {
                FN[w][k] = __fma_rn(E[w][k], FD[w][k - 1], FN[w][k - 1]);
                FD[w][k] = __fma_rn(E[w][k], FN[w][k - 1], FD[w][k - 1]);
            }
        }
        double BN[W], BD[W], QN[W][D], QD[W][D]; // the fractions whose logarithms are the outputs
#pragma unroll
        for (int w = 0; w < W; ++w)
        {
            BN[w] = E[w][D - 1];
            BD[w] = 1.0;
            QN[w][D - 1] = FN[w][D - 2];
            QD[w][D - 1] = FD[w][D - 2];
#pragma unroll
            for (int k = D - 2; k >= 1; --k)
            {
                QN[w][k] = __fma_rn(FN[w][k - 1], BD[w], BN[w] * FD[w][k - 1]);
                QD[w][k] = __fma_rn(FN[w][k - 1], BN[w], FD[w][k - 1] * BD[w]);
                const double bn = __fma_rn(E[w][k], BD[w], BN[w]), bd = __fma_rn(E[w][k], BN[w], BD[w]);
                BN[w] = bn;
                BD[w] = bd;
            }
            QN[w][0] = BN[w];
            QD[w][0] = BD[w];
        }
#pragma unroll
        for (int k = 0; k < D; ++k)
#pragma unroll
            for (int w = 0; w < W; ++w)
            {
                const double l = bp_log_frac(QN[w][k], QD[w][k], shift[w], far);
                anyfar |= far;
                const uint32_t sg = (sx[w] ^ (uint32_t)__double2hiint(x[w][k])) & 0x80000000u;
                r[w][k] = __hiloint2double((int)(((uint32_t)__double2hiint(l) & 0x7fffffffu) | sg), __double2loint(l));
            }
        if (anyfar) // rare: the reference's pairwise recursion for all W lanes, rolled loops over a local copy
        {
            double lx[W][D], lf[W][D];
#pragma unroll
            for (int w = 0; w < W; ++w)
#pragma unroll
                for (int k = 0; k < D; ++k) lx[w][k] = x[w][k];
#pragma unroll 1
            for (int w = 0; w < W; ++w)
            {
                lf[w][0] = lx[w][0];
#pragma unroll 1
                for (int k = 1; k < D; ++k) lf[w][k] = boxplus(lf[w][k - 1], lx[w][k]);
                double B = lx[w][D - 1];
                lf[w][D - 1] = lf[w][D - 2];
#pragma unroll 1
                for (int k = D - 2; k >= 1; --k)
                {
                    const double f = lf[w][k - 1];
                    lf[w][k] = boxplus(f, B);
                    B = boxplus(B, lx[w][k]);
                }
                lf[w][0] = B;
            }
#pragma unroll
            for (int w = 0; w < W; ++w)
#pragma unroll
                for (int k = 0; k < D; ++k) r[w][k] = lf[w][k];
        }
    }
#endif

    // pairwise box-plus with the Jacobian correction, decoder.h:12-15 (same expression, same order)
    template <typename T>
    __device__ __forceinline__ T boxplus(T x, T y)
    {
        const T ax = Num<T>::abs(x), ay = Num<T>::abs(y);
        const T m = (ay < ax) ? ay : ax;
        const T sm = Num<T>::with_sign(m, Num<T>::hi(x) ^ Num<T>::hi(y));
        if constexpr (sizeof(T) == 8) return sm + bp_log_ratio(bp_exp_neg(Num<T>::abs(x + y)), bp_exp_neg(Num<T>::abs(x - y)));
        else
        {
            const T num = T(1) + Num<T>::exp_(-Num<T>::abs(x + y));
            const T den = T(1) + Num<T>::exp_(-Num<T>::abs(x - y));
            return sm + Num<T>::log_(num / den);
        }
    }

} // namespace b200
