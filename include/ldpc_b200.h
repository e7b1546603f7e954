/* libldpc_b200 — C ABI of the B200-native LDPC decode path.
 *
 * Part 1 is the drop-in boundary: the six symbols and four POD structs that the reference's
 * libldpc.so exports (reference: src/shared.cpp:9-78, src/core/functions.h:107-127,
 * src/sim/ldpcsim.h:23-31) and that pyLDPC/ldpc.py binds through ctypes (pyLDPC/ldpc.py:8-50,
 * 102,130,160-166,200,216).  Same names, same argument meaning, same struct layouts (LP64),
 * structs passed BY VALUE exactly as the reference does.
 *
 * Part 2 is the handle-based API the tests, bench.py, the ldpcsim CLI and the multi-GPU host use.
 * Plain pointers and sizes only; no C++/torch types.  Every int-returning function returns 0 on
 * success and a negative value on failure with the text available from ldpc_b200_last_error().
 * There is no CPU fallback: anything that decodes or simulates needs a CUDA device and fails
 * loudly without one.  Loader / GF(2) helpers are host-side (they are one-off O(nnz) utilities in
 * the reference as well) and work without a GPU.
 */
#ifndef LDPC_B200_H
#define LDPC_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

/* The library is built with -fvisibility=hidden: only the functions declared here are exported. */
#if defined(__GNUC__)
#define LDPC_B200_API __attribute__((visibility("default")))
#else
#define LDPC_B200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------ */
/* Part 1 — reference-compatible boundary                                                     */
/* ------------------------------------------------------------------------------------------ */

/* reference: src/core/functions.h:107-112 (16 bytes: bool @0, u32 @4, char* @8) */
typedef struct
{
    bool earlyTerm;
    uint32_t iterations;
    const char *type; /* "BP_MS" = min-sum; anything else = BP (src/decoding/decoder.h:76) */
} decoder_param;

/* reference: src/core/functions.h:114-119 (40 bytes) */
typedef struct
{
    uint64_t seed;
    double xRange[3]; /* MIN MAX STEP, half-open sweep (src/sim/ldpcsim.cpp:104-110) */
    const char *type; /* "AWGN" | "BSC" | "BEC" | "RAYLEIGH" (B200 extension: x = average SNR in dB; coherence length of the
                         context, ldpc_b200_set_fading, default 1) */
} channel_param;

/* reference: src/core/functions.h:121-127 (32 bytes) */
typedef struct
{
    uint32_t threads; /* accepted for compatibility; the GPU path ignores it */
    uint64_t maxFrames;
    uint64_t fec;
    const char *resultFile;
} simulation_param;

/* reference: src/sim/ldpcsim.h:23-31 (48 bytes); caller-allocated arrays indexed by point in
 * execution order (reversed for BSC/BEC, src/sim/ldpcsim.cpp:114-122) */
typedef struct
{
    double *fer;
    double *ber;
    double *avg_iter;
    double *time;
    uint64_t *fec;
    uint64_t *frames;
} sim_results_t;

/* replaces src/shared.cpp:11-24 — loads the code (and optional generator) into the process-global
 * context; prints "Error: ..." and exit(EXIT_FAILURE)s on file errors like src/core/ldpc.cpp:16-20 */
LDPC_B200_API void ldpc_setup(const char *pcFile, const char *genFile, int *n, int *m, int *nct, int *mct);
/* replaces src/shared.cpp:26-30 — blocking Monte-Carlo sweep; fills results[] per point; polls *stopFlag */
LDPC_B200_API void simulate(decoder_param decoderParams, channel_param channelParam, simulation_param simParam,
              sim_results_t *results, bool *stopFlag);
/* replaces src/shared.cpp:32-35 */
LDPC_B200_API int calculate_rank(void);
/* replaces src/shared.cpp:37-45 — infoWord[kct] -> codeWord[nct] (transmitted positions of u*G) */
LDPC_B200_API void encode(uint8_t *infoWord, uint8_t *codeWord);
/* replaces src/shared.cpp:47-65 — llr[nct] in, llrOut[nct] out, returns the 0-based iteration count
 * (src/decoding/decoder.cpp:66-77).  Punctured and shortened inputs are 0.0 (shared.cpp:50).
 * Unlike the reference there is no sticky min-sum state between calls (reference quirk: decoder.h:73-80). */
LDPC_B200_API int decode(decoder_param decoderParams, double *llr, double *llrOut);
/* replaces src/shared.cpp:67-77 — word[nc] -> syndrome[mc] */
LDPC_B200_API void syndrome(uint8_t *word, uint8_t *syndrome);

/* ------------------------------------------------------------------------------------------ */
/* Part 2 — handle-based B200 API                                                             */
/* ------------------------------------------------------------------------------------------ */

/* A context owns one loaded code, its device tables on ONE CUDA device, a stream and workspaces.  It is not
 * thread-safe: use one context per host thread (and per GPU); different contexts may be used concurrently, also on
 * different devices of one process.  Every function returns 0 on success and non-zero on failure (message:
 * ldpc_b200_last_error(), thread-local); compute entry points fail when no CUDA device is present — there is no CPU
 * fallback. */
typedef struct ldpc_b200_ctx ldpc_b200_ctx;

enum { LDPC_B200_F64 = 0, LDPC_B200_F32 = 1 };          /* arithmetic / message type of the decoder */
enum { LDPC_B200_FIXED = 2 }; /* ldpc_b200_stats.precision of the fixed-point layered decoder (ldpc_b200_set_quant); not a tuning value */
enum { LDPC_B200_AUTO = 0, LDPC_B200_SMEM = 1, LDPC_B200_GLOBAL = 2 }; /* message residency */

typedef struct
{
    int nc, mc, nnz, kc;     /* src/core/ldpc.h:47-53 */
    int nct, mct, kct;       /* src/core/ldpc.h:55-59 */
    int n_punct, n_short;
    int max_degree;          /* src/core/ldpc.cpp:83-87 */
    int max_check_degree, max_var_degree;
    int has_generator, g_rows, g_cols, g_nnz;
} ldpc_b200_code_info;

typedef struct
{
    int precision;        /* LDPC_B200_F64 (bit-exact parity mode, default) | LDPC_B200_F32 */
    int residency;        /* LDPC_B200_AUTO | _SMEM | _GLOBAL */
    int frames_per_cta;   /* 0 = auto (power of two, 1..32) */
    int threads_per_cta;  /* 0 = auto; capped at the kernel's build (512; 384 for the shared-memory fp64 sum-product kernel) */
    int ctas;             /* 0 = auto (148 x resident CTAs) */
    int bec_deg1_compat;  /* 1 (default) = erased degree-1 variable nodes send 0 like the reference's UB outcome */
    int tmem;             /* 0 = auto (Tensor-Memory mirror of thread-private state when it fits), 1 = off */
    int idx16;            /* index entries of the shared-memory tables: 0 = auto (16-bit entries and two CTAs per SM where a one-off
                             timed trial finds that shape faster, else 32-bit), 1 = always 32-bit, 2 = 16-bit whenever the code is
                             small enough for them */
    int zero_codeword;    /* 0 (default) = with a generator matrix loaded the sweep transmits random codewords like the
                             reference's -G; 1 = always the all-zero codeword */
    int schedule;         /* LDPC_B200_FLOODING (default: the reference's schedule, src/decoding/decoder.cpp:11-78) | LDPC_B200_LAYERED
                             (opt-in: the legacy tree's layer loop, gpu/device/kernel.cpp:52-75; results differ from the flooding
                             reference by design; AWGN / BSC sweeps with the all-zero codeword and the batch decode call) */
    int layered_ms_scale64; /* layered schedule, BP_MS only: check outputs are multiplied by this / 64 (normalised min-sum; 0 or 64 = the
                               reference's plain min-sum, 48 = 0.75).  Plain min-sum is unstable under the layered schedule on
                               codes with many punctured / high-degree columns (profiles/r2/layered.md) */
} ldpc_b200_tuning;
enum { LDPC_B200_FLOODING = 0, LDPC_B200_LAYERED = 1 };

LDPC_B200_API const char *ldpc_b200_last_error(void);
LDPC_B200_API const char *ldpc_b200_version(void);
/* number of CUDA devices visible (0 when there is no GPU / driver) */
LDPC_B200_API int ldpc_b200_device_count(void);

/* Loads pcFile (+ genFile, may be NULL/"") on the host.  device >= 0 binds the context to that CUDA
 * device (tables are uploaded lazily on first use); device = -1 keeps it host-only.  NULL on failure. */
LDPC_B200_API ldpc_b200_ctx *ldpc_b200_open(const char *pcFile, const char *genFile, int device);
LDPC_B200_API void ldpc_b200_close(ldpc_b200_ctx *ctx);
LDPC_B200_API int ldpc_b200_info(const ldpc_b200_ctx *ctx, ldpc_b200_code_info *info);
LDPC_B200_API int ldpc_b200_set_tuning(ldpc_b200_ctx *ctx, const ldpc_b200_tuning *t);
LDPC_B200_API int ldpc_b200_get_tuning(const ldpc_b200_ctx *ctx, ldpc_b200_tuning *t);

/* One launch in flight per context at a time is the supported use.  Launches of one context that do overlap (different
 * caller streams) are still safe: the per-CTA message workspace in HBM (large codes, byte-wise erasure decoder) is shared
 * by the launches of a context and every launch waits, on its own stream, for the previous user of that workspace.
 *
 * The kernel shape of a (decoder type, precision) pair is picked by a one-off timed trial before the first large job.  The
 * blocking entry points run it themselves; the asynchronous ones (ldpc_b200_decode_batch_device, ldpc_b200_sim_point_async)
 * never block and use the cached outcome or the default shape.  Call ldpc_b200_prepare once (blocking) to have the trial
 * done before a stream of asynchronous launches; n_frames = the size of the job (jobs below ~20000 frames skip the trial). */
LDPC_B200_API int ldpc_b200_prepare(ldpc_b200_ctx *ctx, decoder_param dp, uint64_t n_frames);

/* Layers of the layered schedule: n_layers lists of check indices (layer l = layer_check[layer_ptr[l] .. layer_ptr[l+1])), every
 * check in exactly one layer, no two checks of a layer sharing a variable.  n_layers = 0 selects the built-in first-fit layering
 * (one layer per block row on quasi-cyclic codes).  ldpc_b200_load_layers reads the legacy tree's layer file (gpu/ldpc/ldpc.cpp:
 * 111-138: "nl: N", then per layer "cn[i]: W" and W check indices).  ldpc_b200_get_layers returns the layering in use
 * (layer_of[mc]; the return value is the number of layers, negative on failure). */
LDPC_B200_API int ldpc_b200_set_layers(ldpc_b200_ctx *ctx, int n_layers, const int *layer_ptr, const int *layer_check);
LDPC_B200_API int ldpc_b200_load_layers(ldpc_b200_ctx *ctx, const char *layer_file);
LDPC_B200_API int ldpc_b200_get_layers(ldpc_b200_ctx *ctx, int *layer_of /*[mc]*/);

/* Higher-order modulation of the AWGN sweep (opt-in; the legacy tree's M-ASK with bit-metric decoding: constellation
 * gpu/sim/ldpcsim.cpp:6-20, labels / bit mapper :64-140, encode_all0 + map_c_to_x :240-271, calc_llrs :273-323 =
 * gpu/device/kernel.cpp:141-219).  M = 4, 8, ... 256 points X_j = (-M + 1 + 2j) / sqrt(mean energy), uniform; labels[M] = the
 * log2(M)-bit label of point j (NULL: binary reflected Gray code); bit_mapper[log2 M][nct / log2 M] = the variable carrying bit
 * level k (most significant first) of symbol i (NULL: symbol i carries transmitted positions i*bits ... i*bits + bits - 1); nct must
 * be a multiple of log2 M.  Frames carry random scrambling bits and the LLRs are multiplied by (1 - 2c), so the decoder sees the
 * all-zero codeword, as in the legacy tree.  M = 2 returns to BPSK (the reference's channel_awgn).  Applies to "AWGN" in
 * ldpc_b200_channel / _sim_point* / _simulate*; flooding schedule. */
LDPC_B200_API int ldpc_b200_set_modulation(ldpc_b200_ctx *ctx, int M, const int *labels, const int *bit_mapper);

/* Coherence length of the "RAYLEIGH" channel (not in the reference): BPSK over flat Rayleigh fading with perfect channel state
 * information at the receiver.  Transmitted index t uses fading coefficient floor(t / coherence) of its frame; coherence = 1 (the
 * default) is fast fading, 0 is one coefficient per frame (quasi-static).  Coefficient c is h = sqrt((a^2 + b^2) / 2) of the first
 * normal pair of Philox block c of stream 3, E[h^2] = 1; y = sigma z + h (1 - 2 cw) with the AWGN channel's noise z at average
 * SNR x dB, LLR = y h 2 / sigma^2 (DESIGN.md 3.2).  Per context; negative values fail.  RAYLEIGH with M-ASK (M > 2) fails. */
LDPC_B200_API int ldpc_b200_set_fading(ldpc_b200_ctx *ctx, int coherence);

/* Fixed-point layered min-sum (not in the reference; DESIGN.md 3.7), the decoder of a hardware implementation: the fp64 channel
 * LLR L (the channel's own, or the caller's for the batch decode) enters as clamp(round(L / step), -M(ch_bits), M(ch_bits)) with
 * M(q) = 2^(q-1) - 1, round half away from zero; the check-to-variable messages have msg_bits and the posteriors post_bits, with
 * saturating int32 arithmetic; a check sends sign * max(floor(m * scale8 / 8) - offset, 0), m = the smallest magnitude of the other
 * edges clipped to M(msg_bits).  Valid: 2 <= msg_bits <= post_bits <= 16, 2 <= ch_bits <= post_bits, 0 <= offset < M(msg_bits),
 * 1 <= scale8 <= 8, step > 0.  Decisions are P <= 0; llr_out receives P * step.
 * Per context.  q = NULL or ch_bits = 0 turns it off; invalid parameters fail and keep the previous setting.  While it is on, the
 * layered schedule (tuning.schedule = LDPC_B200_LAYERED, tuning.precision ignored) runs the int16 kernel: 16 or 32 frames per CTA
 * (tuning.frames_per_cta 0 = 32), ldpc_b200_get_stats reports precision = LDPC_B200_FIXED, and no kernel-shape trial runs.  Every
 * decoding entry point fails while it is on with the flooding schedule, decoder type BP, the BEC, M-ASK (M > 2), the narrow
 * encodings of the batch decode or another frames_per_cta. */
typedef struct
{
    int ch_bits, msg_bits, post_bits; /* bits of the channel LLR, of the check-to-variable messages and of the posterior */
    int offset;                       /* beta, in LSBs */
    int scale8;                       /* normalisation factor scale8 / 8 */
    double step;                      /* LLR value of one LSB */
} ldpc_b200_quant;
LDPC_B200_API int ldpc_b200_set_quant(ldpc_b200_ctx *ctx, const ldpc_b200_quant *q);
LDPC_B200_API int ldpc_b200_get_quant(const ldpc_b200_ctx *ctx, ldpc_b200_quant *q); /* ch_bits = 0: off */

/* host-side views of the loaded code (file order; sizes from ldpc_b200_info) */
LDPC_B200_API int ldpc_b200_get_edges(const ldpc_b200_ctx *ctx, int *rows /*[nnz]*/, int *cols /*[nnz]*/);
LDPC_B200_API int ldpc_b200_get_bit_pos(const ldpc_b200_ctx *ctx, int *bit_pos /*[nct]*/);
LDPC_B200_API int ldpc_b200_get_puncture(const ldpc_b200_ctx *ctx, int *punct /*[n_punct]*/, int *shorten /*[n_short]*/);
/* device schedule for the current tuning (for tests): for every edge e (file order) the check-major
 * message slot it lives in; n_slots = padded slot count */
LDPC_B200_API int ldpc_b200_get_layout(ldpc_b200_ctx *ctx, int *edge_slot /*[nnz]*/, int *n_slots, int *frames_per_cta,
                         int *threads_per_cta, int *residency);

/* message slots of the bit-sliced erasure kernel (for tests): slot % 32 is the shared-memory bank; edge k of 32 consecutive
 * checks, and edge k of 32 consecutive variables, never share a bank (a 32-colouring of the edges) */
LDPC_B200_API int ldpc_b200_get_bec_layout(ldpc_b200_ctx *ctx, int *edge_slot /*[nnz]*/, int *n_slots);

/* GF(2) helpers on the host (reference: src/core/sparse.h:162-218,227-294) */
LDPC_B200_API int ldpc_b200_rank(const ldpc_b200_ctx *ctx);
LDPC_B200_API int ldpc_b200_encode(const ldpc_b200_ctx *ctx, const uint8_t *info /*[g_rows]*/, uint8_t *cw_full /*[nc]*/);
LDPC_B200_API int ldpc_b200_syndrome(const ldpc_b200_ctx *ctx, const uint8_t *word /*[nc]*/, uint8_t *synd /*[mc]*/);

/* Batched flooding decode on the GPU, HOST buffers (copies are part of the call).
 *   llr      [n_frames][nc]  full-length LLRs (punctured/shortened positions included)
 *   llr_out  [n_frames][nc]  posterior LLRs after the last executed iteration (may be NULL)
 *   hard     [n_frames][nc]  decisions (LLR <= 0 -> 1, src/decoding/decoder.cpp:58)   (may be NULL)
 *   iters    [n_frames]      reference iteration count (0-based on success)              (may be NULL)
 * Decoder type/iterations/early termination come from decoder_param (reference semantics). */
LDPC_B200_API int ldpc_b200_decode_batch(ldpc_b200_ctx *ctx, decoder_param dp, const double *llr, int64_t n_frames,
                           double *llr_out, uint8_t *hard, int32_t *iters);
/* The same call with narrower encodings at the host <-> device boundary (the six-symbol decode() and the call above keep
 * double in / byte-per-bit out, src/shared.cpp:47-65).  At 9216 B in + 1152 B out per frame of the n=1152 code the fp64 path
 * is bound by the PCIe / host-memory path once several GPUs share a host; int8 LLRs + bit-packed decisions move 1152 + 144 B.
 *   llr_type  LDPC_B200_LLR_F64: const double*  |  _F32: const float* (widened exactly)  |  _I8: const int8_t*, LLR =
 *             value * llr_scale evaluated in double (exact when llr_scale is a power of two), i.e. the decoder runs on exactly
 *             the doubles {value * llr_scale}: min-sum stays bit-identical to the reference fed those doubles
 *   hard_bits [n_frames][ceil(nc/32)] uint32: decision of variable i = bit i%32 of word i/32 (may be NULL)
 * llr_out / hard / iters as above (any may be NULL). */
enum { LDPC_B200_LLR_F64 = 0, LDPC_B200_LLR_F32 = 1, LDPC_B200_LLR_I8 = 2 };
LDPC_B200_API int ldpc_b200_decode_batch_ex(ldpc_b200_ctx *ctx, decoder_param dp, const void *llr, int llr_type, double llr_scale,
                                            int64_t n_frames, double *llr_out, uint8_t *hard, uint32_t *hard_bits, int32_t *iters);
/* Same with DEVICE buffers (already resident in HBM), asynchronous on `stream` (cudaStream_t). */
LDPC_B200_API int ldpc_b200_decode_batch_device(ldpc_b200_ctx *ctx, decoder_param dp, const double *d_llr, int64_t n_frames,
                                  double *d_llr_out, uint8_t *d_hard, int32_t *d_iters, void *stream);

LDPC_B200_API int ldpc_b200_decode_batch_device_ex(ldpc_b200_ctx *ctx, decoder_param dp, const void *d_llr, int llr_type, double llr_scale,
                                                   int64_t n_frames, double *d_llr_out, uint8_t *d_hard, uint32_t *d_hard_bits,
                                                   int32_t *d_iters, void *stream);

/* BEC decode, HOST buffers: in[n][nc] in {0,1,'E'}, cw[n][nc] true bits (genie check of the
 * reference's vn_update, src/decoding/decoder.h:145-149). */
LDPC_B200_API int ldpc_b200_decode_bec_batch(ldpc_b200_ctx *ctx, decoder_param dp, const uint8_t *in, const uint8_t *cw,
                               int64_t n_frames, uint8_t *out, uint8_t *hard, int32_t *iters);

/* Philox channel only: writes the decoder inputs the simulator would generate for global frames
 * [frame0, frame0+n) of sweep point `point`: cw[n][nc] (may be NULL), and llr[n][nc] doubles
 * (AWGN/BSC/RAYLEIGH) or llr_u8[n][nc] (BEC).  HOST buffers. */
LDPC_B200_API int ldpc_b200_channel(ldpc_b200_ctx *ctx, const char *channel, double x, uint64_t seed, uint32_t point,
                      uint64_t frame0, int64_t n_frames, uint8_t *cw, double *llr, uint8_t *llr_u8);

/* One Monte-Carlo round of one sweep point, fully on the GPU (channel -> decode -> accounting):
 * global frames [frame0, frame0+n_frames) of channel "AWGN", "BSC", "BEC" or "RAYLEIGH".  counters[4] += {frame errors, bit errors, frames,
 * sum of reference iteration counts} (src/sim/ldpcsim.cpp:175-190).  Blocking; counters on the host.
 * device_ms (may be NULL) receives the CUDA-event time of the kernel(s). */
LDPC_B200_API int ldpc_b200_sim_point(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed,
                        uint32_t point, uint64_t frame0, uint64_t n_frames, uint64_t counters[4], float *device_ms);
/* Same round with the per-error diagnostics log (the reference's log_error, src/sim/ldpcsim.cpp:282-405, live in
 * gpu/sim/ldpcsim.cpp:351-464): every frame that ends with >= 1 bit error over the transmitted positions is recorded
 * (up to `capacity` records, unordered; *n_errors receives the number of frames in error, which may exceed capacity).
 * A record names the GLOBAL frame index: because the channel is counter-based, ldpc_b200_channel(frame0 = record.frame,
 * n = 1) regenerates that frame's decoder input exactly and ldpc_b200_decode_batch replays the decoding, which yields
 * the failed bit / check indices and the syndrome weight (libldpc_b200/api.py: Context.error_report).  All four channels. */
typedef struct
{
    uint64_t frame;      /* global frame index of the sweep point */
    uint32_t bit_errors; /* Hamming distance to the transmitted word over the transmitted positions */
    int32_t iterations;  /* reference iteration count of the frame (0-based on success, decoder.cpp:66-77) */
} ldpc_b200_error_record;
LDPC_B200_API int ldpc_b200_sim_point_log(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed,
                            uint32_t point, uint64_t frame0, uint64_t n_frames, uint64_t counters[4],
                            ldpc_b200_error_record *records, int64_t capacity, int64_t *n_errors);
/* Batched replay of frames in error, on the GPU: for every global frame index frames[i] of sweep point `point` the channel
 * regenerates the decoder input, the decoder runs under the context's current tuning (precision, residency, schedule,
 * modulation; the erasure decode mode on "BEC") and the decisions are compared with the transmitted word.  reports[i] describes
 * frames[i] (same order; repeated and unsorted indices are allowed); its failed bits are failed_bits[bits_offset ..
 * bits_offset + bit_errors): the variable ids of the transmitted positions whose decision differs, in transmitted order; its
 * failed checks are failed_checks[checks_offset .. checks_offset + syndrome_weight): the unsatisfied checks of the decisions,
 * ascending.  syndrome_weight = 0 with bit_errors > 0 is an undetected error (the decoder stopped on another codeword).  With
 * M-ASK the decoder sees the all-zero word (ldpc_b200_set_modulation), and the decisions are compared with it.
 * *bits_needed / *checks_needed (may be NULL) receive the total list lengths.  When a capacity is too small the call fails and
 * writes nothing but those two: call again with capacities of at least that size.  Blocking; HOST buffers. */
typedef struct
{
    uint64_t frame;                      /* global frame index of the sweep point */
    int32_t iterations;                  /* reference iteration count of the replayed decode */
    uint32_t bit_errors;                 /* = number of failed_bits of this frame */
    uint32_t syndrome_weight;            /* = number of failed_checks of this frame */
    int64_t bits_offset, checks_offset;  /* into failed_bits / failed_checks */
} ldpc_b200_frame_report;
LDPC_B200_API int ldpc_b200_error_report(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed,
                                         uint32_t point, const uint64_t *frames, int64_t n_frames, ldpc_b200_frame_report *reports,
                                         int32_t *failed_bits, int64_t bits_capacity, int32_t *failed_checks, int64_t checks_capacity,
                                         int64_t *bits_needed, int64_t *checks_needed);
/* Asynchronous variant: d_counters is a DEVICE array of 5 uint64 that the kernel accumulates into
 * ({frame errors, bit errors, frames, sum of reference iteration counts, sum of executed iterations}). */
LDPC_B200_API int ldpc_b200_sim_point_async(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed,
                              uint32_t point, uint64_t frame0, uint64_t n_frames, uint64_t *d_counters, void *stream);

/* Whole sweep with the reference's semantics (x list, reversed order for BSC/BEC, stop rule, results
 * file layout — src/sim/ldpcsim.cpp:97-263).  Channels "AWGN", "BSC", "BEC" and "RAYLEIGH" (ascending SNR like AWGN).  rank/world shard the frames of every round across
 * processes; `allreduce` (may be NULL when world == 1) is called once per round with a small host
 * array of uint64 counters to be summed over ranks (the caller wires it to NCCL/gloo).  quiet != 0 suppresses the console table. */
typedef void (*ldpc_b200_allreduce_fn)(uint64_t *values, int n, void *user); /* in-place sum over ranks */
LDPC_B200_API int ldpc_b200_simulate(ldpc_b200_ctx *ctx, decoder_param dp, channel_param cp, simulation_param sp,
                       sim_results_t *results, bool *stopFlag, int rank, int world,
                       ldpc_b200_allreduce_fn allreduce, void *user, int quiet);
/* Same sweep with the frame processor injected: round_fn (if non-NULL) is called instead of the GPU
 * launch to process global frames [frame0, frame0+n_frames) of sweep point `point` at channel value x
 * and must add {frame errors, bit errors, frames, iterations} to counters4.  Lets a multi-GPU host
 * drive its own asynchronous launches, and lets the host-side logic (sharding, stop rule, results
 * writer) be exercised on machines without a GPU.  Returns non-zero from round_fn to abort. */
typedef int (*ldpc_b200_round_fn)(uint32_t point, double x, uint64_t frame0, uint64_t n_frames,
                                  uint64_t *counters4, void *user);
LDPC_B200_API int ldpc_b200_simulate_ex(ldpc_b200_ctx *ctx, decoder_param dp, channel_param cp, simulation_param sp,
                          sim_results_t *results, bool *stopFlag, int rank, int world,
                          ldpc_b200_allreduce_fn allreduce, ldpc_b200_round_fn round_fn, void *user, int quiet);

/* execution statistics of the last simulate/sim_point/decode_batch call on this context */
typedef struct
{
    double device_ms;        /* CUDA-event time summed over kernel launches */
    uint64_t launches;       /* kernel launches */
    uint64_t frames;         /* frames decoded */
    uint64_t edge_iterations;/* sum over frames of executed iterations x nnz */
    int frames_per_cta, threads_per_cta, ctas, residency, precision;
    size_t smem_bytes;
} ldpc_b200_stats;
LDPC_B200_API int ldpc_b200_get_stats(const ldpc_b200_ctx *ctx, ldpc_b200_stats *s);
/* Measurement aid: sustained shared-memory read bandwidth of the context's device in GB/s (a conflict-free
 * LDS.128 streaming kernel on every SM) — the roofline that bounds the shared-memory-resident decode kernel. */
LDPC_B200_API int ldpc_b200_smem_probe(ldpc_b200_ctx *ctx, double *gb_per_s);
/* Measurement aid: sustained FP64 instruction rate in G thread-instructions/s (independent DFMA chains on every SM) — the
 * roofline of the fp64 sum-product kernel, which is bound by the FP64 pipe. */
LDPC_B200_API int ldpc_b200_fp64_probe(ldpc_b200_ctx *ctx, double *ginst_per_s);
LDPC_B200_API int ldpc_b200_reset_stats(ldpc_b200_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* LDPC_B200_H */
