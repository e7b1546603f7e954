/* TEST INFRASTRUCTURE — NOT PRODUCT CODE.
 *
 * Executable specification of the binary32 layered min-sum decoder (lay_kernel<float, ALG_MS, *>, DESIGN.md §3.7).  The layer
 * loop, the `cw < 2` skip, the first-visit rule (+0 as the old check-to-variable message) and the stop rule are those of
 * orc_decode_layered (oracle/ldpc_oracle.c, compiled into this library unchanged); the state is binary32 throughout:
 *   - decoder input = (float) of the fp64 LLR (99999.9 on shortened positions becomes 99999.8984375);
 *   - check output = sign-bit XOR of the others x their exact minimum magnitude, then x (float)ms_scale, rounded once;
 *   - llr_out = (double) of the posterior.
 * Min-sum needs nothing but +, -, compares, sign bits and that one product, so the kernel has nothing to contract into an FMA and
 * must equal this function bit for bit.  Sum-product in binary32 (__expf / __logf on the device) has no exact specification.
 *
 * Build: gcc -O2 -std=c11 -fPIC -shared -fopenmp -ffp-contract=off -o liblayered_f32_oracle.so layered_f32_oracle.c -lm
 * (tests/layered_f32_oracle.py does this in a temporary directory).
 */
#include "../oracle/ldpc_oracle.c"

static inline int sgnf(float x) { return 1 - 2 * (signbit(x) ? 1 : 0); } /* -0.0f is negative, as sgn() */
static inline float fminf_first(float a, float b) { return (b < a) ? b : a; }

static float f_minsum_f32(float x, float y) { return (float)(sgnf(x) * sgnf(y)) * fminf_first(fabsf(x), fabsf(y)); }

int orc_decode_layered_f32(const orc_code *c, int nl, const int *layer_ptr, const int *layer_check, const double *llr_in, int iterations,
                           int early_term, double ms_scale, double *llr_out, uint8_t *co)
{
    const float scale = (float)ms_scale;
    float *P = (float *)malloc(sizeof(float) * (c->nc + 1));
    float *c2v = (float *)calloc(c->nnz + 1, sizeof(float)); /* +0: the first visit of a check reads the posterior itself */
    float *F = (float *)calloc(c->max_degree + 2, sizeof(float));
    float *B = (float *)calloc(c->max_degree + 2, sizeof(float));
    float *v = (float *)calloc(c->max_degree + 2, sizeof(float));
    for (int i = 0; i < c->nc; ++i) { P[i] = (float)llr_in[i]; co[i] = 0; }
    int I = 0;
    while (I < iterations)
    {
        for (int l = 0; l < nl; ++l)
            for (int q = layer_ptr[l]; q < layer_ptr[l + 1]; ++q)
            {
                const int *cn = c->row_edge + c->row_ptr[layer_check[q]];
                const int cw = c->row_ptr[layer_check[q] + 1] - c->row_ptr[layer_check[q]];
                if (cw < 2) continue;
                for (int j = 0; j < cw; ++j) v[j] = P[c->e_col[cn[j]]] - c2v[cn[j]];
                F[0] = v[0];
                B[cw - 1] = v[cw - 1];
                for (int j = 1; j < cw; ++j)
                {
                    F[j] = f_minsum_f32(F[j - 1], v[j]);
                    B[cw - 1 - j] = f_minsum_f32(B[cw - j], v[cw - j - 1]);
                }
                for (int j = 0; j < cw; ++j)
                {
                    const float r = ((j == 0) ? B[1] : (j == cw - 1) ? F[cw - 2] : f_minsum_f32(F[j - 1], B[j + 1])) * scale;
                    c2v[cn[j]] = r;
                    P[c->e_col[cn[j]]] = v[j] + r;
                }
            }
        for (int i = 0; i < c->nc; ++i) co[i] = (P[i] <= 0);
        if (early_term && orc_is_codeword(c, co)) break; /* before ++I, like the live decoder */
        ++I;
    }
    for (int i = 0; i < c->nc; ++i)
    {
        co[i] = (P[i] <= 0);
        llr_out[i] = (double)P[i];
    }
    free(P); free(c2v); free(F); free(B); free(v);
    return I;
}

/* n frames of llr_in[n][nc] through the layered specification: f32 != 0 -> orc_decode_layered_f32 (min-sum), otherwise
 * orc_decode_layered (fp64, min-sum or sum-product).  Frames are independent; `threads` OpenMP threads share them. */
void orc_decode_layered_batch(const orc_code *c, int nl, const int *layer_ptr, const int *layer_check, const double *llr_in, int64_t n,
                              int iterations, int early_term, int minsum, double ms_scale, int f32, int threads, double *llr_out,
                              uint8_t *co, int32_t *iters)
{
    if (threads < 1) threads = 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1)
    for (int64_t t = 0; t < n; ++t)
    {
        const size_t o = (size_t)t * (size_t)c->nc;
        iters[t] = f32 ? orc_decode_layered_f32(c, nl, layer_ptr, layer_check, llr_in + o, iterations, early_term, ms_scale, llr_out + o, co + o)
                       : orc_decode_layered(c, nl, layer_ptr, layer_check, llr_in + o, iterations, early_term, minsum, ms_scale, llr_out + o,
                                            co + o);
    }
}
