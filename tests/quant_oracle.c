/* TEST INFRASTRUCTURE — NOT PRODUCT CODE.
 *
 * Executable specification of the fixed-point layered min-sum decoder (DESIGN.md §3.7): quantised channel LLRs, integer
 * check-to-variable messages and posteriors with saturating arithmetic, an offset and a normalisation factor a/8.  The layer
 * loop, the `cw < 2` skip, the first-visit rule and the stop rule are those of orc_decode_layered (oracle/ldpc_oracle.c); the
 * channels are the counter-based AWGN / BSC channel of the oracle and the RAYLEIGH channel of tests/rayleigh_oracle.c, which
 * are compiled into this library unchanged.
 *
 * Build: gcc -O2 -std=c11 -fPIC -shared -fopenmp -ffp-contract=off -o libquant_oracle.so quant_oracle.c -lm
 * (tests/quant_oracle.py does this in a temporary directory).  -ffp-contract=off keeps L / step and P * step rounded on their own,
 * as the CUDA kernel evaluates them (__ddiv_rn, __dmul_rn).
 */
#include "rayleigh_oracle.c"

enum { ORC_RAYLEIGH = 4 };

/* the parameters of ldpc_b200_quant (include/ldpc_b200.h), same layout */
typedef struct
{
    int ch_bits, msg_bits, post_bits, offset, scale8;
    double step;
} orc_quant;

static inline int32_t qmax(int bits) { return (int32_t)((1u << (bits - 1)) - 1u); } /* M(q) = 2^(q-1) - 1 */
static inline int32_t sat(int32_t x, int32_t m) { return x > m ? m : x < -m ? -m : x; }

/* clamp(round(L / step), -M(Qc), M(Qc)); round half away from zero, the division correctly rounded */
int32_t orc_quantize(double L, const orc_quant *q)
{
    const double m = (double)qmax(q->ch_bits);
    double r = round(L / q->step);
    if (r > m) r = m;
    if (r < -m) r = -m;
    return (int32_t)r;
}

/* The check rule on the v2c values v[0 .. deg) (already saturated to the posterior range): r[j] = s_j max(floor(m_j a / 8) - beta, 0)
 * with m_j = min over k != j of min(|v_k|, M(Qm)) and s_j the product of the signs of the other v_k (0 counts as positive). */
void orc_check_q(int deg, const int32_t *v, const orc_quant *q, int32_t *r)
{
    const int32_t mm = qmax(q->msg_bits);
    for (int j = 0; j < deg; ++j)
    {
        int32_t m = mm;
        int neg = 0;
        for (int k = 0; k < deg; ++k)
        {
            if (k == j) continue;
            const int32_t a = v[k] < 0 ? -v[k] : v[k];
            if (a < m) m = a;
            neg ^= v[k] < 0;
        }
        int32_t mag = (m * q->scale8) / 8 - q->offset; /* m * a >= 0: the division is the floor */
        if (mag < 0) mag = 0;
        r[j] = neg ? -mag : mag;
    }
}

/* Fixed-point layered min-sum of one frame.  llr_in[nc] fp64 channel LLRs; llr_out[nc] = P * step, co[nc] = (P <= 0); post[nc]
 * (may be NULL) the integer posteriors; *clips (may be NULL) += the number of times a saturation or the message clip changed a
 * value.  Returns the iteration count of orc_decode_layered. */
int orc_decode_layered_q(const orc_code *c, int nl, const int *layer_ptr, const int *layer_check, const double *llr_in, int iterations,
                         int early_term, const orc_quant *q, double *llr_out, uint8_t *co, int32_t *post, uint64_t *clips)
{
    const int32_t pm = qmax(q->post_bits), mm = qmax(q->msg_bits);
    int32_t *P = (int32_t *)malloc(sizeof(int32_t) * (c->nc + 1));
    int32_t *R = (int32_t *)calloc(c->nnz + 1, sizeof(int32_t)); /* 0: the first visit of a check reads the posterior itself */
    int32_t *v = (int32_t *)malloc(sizeof(int32_t) * (c->max_degree + 2));
    int32_t *r = (int32_t *)malloc(sizeof(int32_t) * (c->max_degree + 2));
    uint64_t nclip = 0;
    for (int i = 0; i < c->nc; ++i) { P[i] = orc_quantize(llr_in[i], q); co[i] = 0; }
    int I = 0;
    while (I < iterations)
    {
        for (int l = 0; l < nl; ++l)
            for (int t = layer_ptr[l]; t < layer_ptr[l + 1]; ++t)
            {
                const int *cn = c->row_edge + c->row_ptr[layer_check[t]];
                const int cw = c->row_ptr[layer_check[t] + 1] - c->row_ptr[layer_check[t]];
                if (cw < 2) continue;
                for (int j = 0; j < cw; ++j)
                {
                    const int32_t raw = P[c->e_col[cn[j]]] - R[cn[j]];
                    v[j] = sat(raw, pm);
                    nclip += (v[j] != raw) + (v[j] > mm || v[j] < -mm);
                }
                orc_check_q(cw, v, q, r);
                for (int j = 0; j < cw; ++j)
                {
                    const int32_t raw = v[j] + r[j];
                    R[cn[j]] = r[j];
                    P[c->e_col[cn[j]]] = sat(raw, pm);
                    nclip += P[c->e_col[cn[j]]] != raw;
                }
            }
        for (int i = 0; i < c->nc; ++i) co[i] = (P[i] <= 0);
        if (early_term && orc_is_codeword(c, co)) break; /* before ++I, like the live decoder */
        ++I;
    }
    for (int i = 0; i < c->nc; ++i)
    {
        co[i] = (P[i] <= 0);
        llr_out[i] = (double)P[i] * q->step;
        if (post) post[i] = P[i];
    }
    if (clips) *clips += nclip;
    free(P); free(R); free(v); free(r);
    return I;
}

/* Monte-Carlo point of the fixed-point layered decoder over frames [frame0, frame0 + nframes) of kind ORC_AWGN, ORC_BSC or
 * ORC_RAYLEIGH (coherence length L), all-zero codeword: counters = {fec, bec, frames, iters} as orc_sim_point. */
void orc_sim_point_layered_q(const orc_code *c, int nl, const int *layer_ptr, const int *layer_check, int kind, double x, int L,
                             int iterations, int early_term, const orc_quant *q, uint64_t seed, uint32_t point, uint64_t frame0,
                             uint64_t nframes, int threads, uint64_t counters[4])
{
    uint64_t fec = 0, bec = 0, iters = 0;
    if (threads < 1) threads = 1;
#pragma omp parallel num_threads(threads) reduction(+ : fec, bec, iters)
    {
        uint8_t *cw = (uint8_t *)malloc(c->nc), *co = (uint8_t *)malloc(c->nc), *lu = (uint8_t *)malloc(c->nc);
        double *lf = (double *)malloc(sizeof(double) * c->nc), *lo = (double *)malloc(sizeof(double) * c->nc);
#pragma omp for schedule(dynamic, 4)
        for (uint64_t t = 0; t < nframes; ++t)
        {
            if (kind == ORC_RAYLEIGH) orc_channel_frame_rayleigh(c, NULL, x, L, seed, point, frame0 + t, cw, lf);
            else orc_channel_frame(c, NULL, kind, x, seed, point, frame0 + t, cw, lf, lu);
            iters += (uint64_t)orc_decode_layered_q(c, nl, layer_ptr, layer_check, lf, iterations, early_term, q, lo, co, NULL, NULL);
            const int be = orc_count_bit_errors(c, co, cw);
            if (be > 0) { bec += (uint64_t)be; ++fec; }
        }
        free(cw); free(co); free(lu); free(lf); free(lo);
    }
    counters[0] = fec; counters[1] = bec; counters[2] = nframes; counters[3] = iters;
}
