/* TEST INFRASTRUCTURE — NOT PRODUCT CODE.
 *
 * Executable specification of the "RAYLEIGH" channel (DESIGN.md §3.2): BPSK over flat Rayleigh fading with perfect channel
 * state information at the receiver.  It builds on the counter-based channel of oracle/ldpc_oracle.c (Philox blocks, the
 * binary32 Box-Muller normal pair, the AWGN noise and codewords), which is compiled into this library unchanged.
 *
 * Build: gcc -O2 -std=c11 -fPIC -shared -fopenmp -ffp-contract=off -o librayleigh_oracle.so rayleigh_oracle.c -lm
 * (tests/rayleigh_oracle.py does this in a temporary directory).  -ffp-contract=off keeps every product and sum rounded on its
 * own, as the CUDA kernels evaluate them.
 */
#include "../oracle/ldpc_oracle.c"

/* Fading coefficient c of a frame: the first normal pair (a, b) of Philox block c of stream 3, h = sqrt((a^2 + b^2) / 2).  The
 * squares of binary32 values are exact in fp64, the sum is rounded once, the halving is exact and sqrt is correctly rounded. */
double orc_rayleigh_coeff(uint64_t seed, uint32_t point, uint64_t frame, uint32_t c)
{
    uint32_t w[4];
    float ab[2];
    philox_block(seed, point, 3, frame, c, w);
    normal_pair_v2(w[0], w[1], ab);
    const double a = ab[0], b = ab[1];
    return sqrt(0.5 * (a * a + b * b));
}

/* One faded frame at average SNR x dB, coherence length L (transmitted index t uses coefficient t / L; L = 0: coefficient 0 for
 * the whole frame).  The codeword, the noise z_t and the punctured / shortened values are the AWGN channel's; on the transmitted
 * positions y = z sigma + h (1 - 2 cw) and LLR = (y h) (2 / sigma^2). */
void orc_channel_frame_rayleigh(const orc_code *c, const orc_code *g, double x, int L, uint64_t seed, uint32_t point, uint64_t frame,
                                uint8_t *cw, double *llr)
{
    orc_channel_frame(c, g, ORC_AWGN, x, seed, point, frame, cw, llr, NULL);
    const double sigma2 = pow(10, -x / 10), sigma = sqrt(sigma2), scale = 2.0 / sigma2;
    const int nb = (c->nct + 3) / 4;
    for (int q = 0; q < nb; ++q)
    {
        double z[4];
        orc_normal_block(seed, point, frame, (uint32_t)q, z);
        for (int k = 0; k < 4; ++k)
        {
            const int t = q + k * nb;
            if (t >= c->nct) continue;
            const double h = orc_rayleigh_coeff(seed, point, frame, L ? (uint32_t)(t / L) : 0u);
            const int v = c->bit_pos[t];
            const double y = z[k] * sigma + (cw[v] ? -h : h);
            llr[v] = (y * h) * scale;
        }
    }
}

/* Monte-Carlo point over frames [frame0, frame0 + nframes) of the RAYLEIGH channel, as orc_sim_point: counters = {fec, bec,
 * frames, iters}. */
void orc_sim_point_rayleigh(const orc_code *c, const orc_code *g, int minsum, int iterations, int early_term, double x, int L,
                            uint64_t seed, uint32_t point, uint64_t frame0, uint64_t nframes, int threads, uint64_t counters[4])
{
    uint64_t fec = 0, bec = 0, iters = 0;
    if (threads < 1) threads = 1;
#pragma omp parallel num_threads(threads) reduction(+ : fec, bec, iters)
    {
        uint8_t *cw = (uint8_t *)malloc(c->nc), *co = (uint8_t *)malloc(c->nc);
        double *lf = (double *)malloc(sizeof(double) * c->nc), *lo = (double *)malloc(sizeof(double) * c->nc);
#pragma omp for schedule(dynamic, 4)
        for (uint64_t t = 0; t < nframes; ++t)
        {
            orc_channel_frame_rayleigh(c, g, x, L, seed, point, frame0 + t, cw, lf);
            iters += (uint64_t)orc_decode(c, lf, iterations, early_term, minsum, lo, co);
            const int be = orc_count_bit_errors(c, co, cw);
            if (be > 0) { bec += (uint64_t)be; ++fec; }
        }
        free(cw); free(co); free(lf); free(lo);
    }
    counters[0] = fec; counters[1] = bec; counters[2] = nframes; counters[3] = iters;
}
