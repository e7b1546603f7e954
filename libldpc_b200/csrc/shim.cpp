// C-ABI shim: the six reference symbols (src/shared.cpp:9-78) over a process-global context, plus
// the handle-based ldpc_b200_* API (include/ldpc_b200.h).  No exceptions cross this boundary.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "engine.hpp"

static_assert(sizeof(decoder_param) == 16, "decoder_param layout (src/core/functions.h:107-112)");
static_assert(offsetof(decoder_param, iterations) == 4 && offsetof(decoder_param, type) == 8, "decoder_param layout");
static_assert(sizeof(channel_param) == 40 && offsetof(channel_param, xRange) == 8 && offsetof(channel_param, type) == 32, "channel_param layout");
static_assert(sizeof(simulation_param) == 32 && offsetof(simulation_param, maxFrames) == 8 && offsetof(simulation_param, fec) == 16 &&
                  offsetof(simulation_param, resultFile) == 24, "simulation_param layout");
static_assert(sizeof(sim_results_t) == 48, "sim_results_t layout (src/sim/ldpcsim.h:23-31)");
static_assert(sizeof(ldpc_b200_frame_report) == 40 && offsetof(ldpc_b200_frame_report, bits_offset) == 24, "ldpc_b200_frame_report layout");

struct ldpc_b200_ctx
{
    std::unique_ptr<b200::Engine> eng;
};

namespace
{
    thread_local std::string g_error;
    std::unique_ptr<ldpc_b200_ctx> g_ctx; // the reference keeps one code per process (src/shared.cpp:4-5)

    template <typename F>
    int guarded(F &&f)
    {
        try
        {
            f();
            g_error.clear();
            return 0;
        }
        catch (const std::exception &e)
        {
            g_error = e.what();
            return -1;
        }
        catch (...)
        {
            g_error = "unknown error";
            return -1;
        }
    }

    b200::Engine &global_engine()
    {
        if (!g_ctx) throw std::runtime_error("ldpc_setup() has not been called");
        return *g_ctx->eng;
    }

    [[noreturn]] void die(const char *where, const std::string &what)
    {
        // the reference prints to stdout and exits (src/core/ldpc.cpp:16-20, src/sim/ldpcsim.cpp:77-81)
        std::cout << "Error: " << where << " " << what << std::endl;
        std::cerr << "libldpc_b200: " << where << " " << what << std::endl;
        std::exit(EXIT_FAILURE);
    }
} // namespace

extern "C"
{
    // ---- part 1: reference boundary ---------------------------------------------------------------

    void ldpc_setup(const char *pcFile, const char *genFile, int *n, int *m, int *nct, int *mct)
    {
        auto ctx = std::make_unique<ldpc_b200_ctx>();
        try
        {
            int dev = 0;
            if (const char *e = std::getenv("LDPC_B200_DEVICE")) dev = std::atoi(e);
            ctx->eng = std::make_unique<b200::Engine>(pcFile ? pcFile : "", genFile ? genFile : "", dev);
            if (const char *e = std::getenv("LDPC_B200_PRECISION"))
                ctx->eng->tuning.precision = (std::string(e) == "f32") ? LDPC_B200_F32 : LDPC_B200_F64;
        }
        catch (const std::exception &e)
        {
            die("ldpc_code():", e.what());
        }
        g_ctx = std::move(ctx);
        const auto &H = g_ctx->eng->H;
        *n = H.nc; *m = H.mc; *nct = H.nct(); *mct = H.mct();
    }

    void simulate(decoder_param decoderParams, channel_param channelParam, simulation_param simParam, sim_results_t *results, bool *stopFlag)
    {
        try
        {
            // LIB_SHARED build of the reference: table header only, no results file (src/sim/ldpcsim.cpp:128-139,201-238)
            b200::run_sweep(global_engine(), decoderParams, channelParam, simParam, results, stopFlag, 0, 1, nullptr, nullptr, true, false);
        }
        catch (const std::exception &e)
        {
            die("ldpc_sim::ldpc_sim()", e.what());
        }
    }

    int calculate_rank(void)
    {
        try { return global_engine().H.rank(); }
        catch (const std::exception &e) { die("calculate_rank():", e.what()); }
    }

    void encode(uint8_t *infoWord, uint8_t *codeWord)
    {
        try
        {
            auto &eng = global_engine();
            if (!eng.has_gen) throw std::runtime_error("no generator matrix loaded");
            // u has kct entries (src/shared.cpp:39); rows beyond it do not contribute
            std::vector<uint8_t> u(eng.G.mc, 0), cw(std::max(eng.G.nc, eng.H.nc), 0);
            const int k = std::min(eng.H.kct(), eng.G.mc);
            for (int i = 0; i < k; ++i) u[i] = infoWord[i] ? 1 : 0;
            eng.G.multiply_left(u.data(), cw.data());
            for (int i = 0; i < eng.H.nct(); ++i) codeWord[i] = cw[eng.H.bit_pos[i]];
        }
        catch (const std::exception &e) { die("encode():", e.what()); }
    }

    int decode(decoder_param decoderParams, double *llr, double *llrOut)
    {
        try
        {
            auto &eng = global_engine();
            const int nc = eng.H.nc, nct = eng.H.nct();
            std::vector<double> in(nc, 0.0), out(nc, 0.0); // src/shared.cpp:50: untransmitted positions enter as 0.0
            for (int i = 0; i < nct; ++i) in[eng.H.bit_pos[i]] = llr[i];
            int32_t iters = 0;
            if (decoderParams.iterations == 0)
            { // the reference's loop does not run: zero-initialised output, returns 0 (src/decoding/decoder.cpp:21-22)
                for (int i = 0; i < nct; ++i) llrOut[i] = 0.0;
                return 0;
            }
            eng.decode_batch_host(decoderParams, in.data(), LDPC_B200_LLR_F64, 1.0, 1, out.data(), nullptr, nullptr, &iters);
            for (int i = 0; i < nct; ++i) llrOut[i] = out[eng.H.bit_pos[i]];
            return iters;
        }
        catch (const std::exception &e) { die("decode():", e.what()); }
    }

    void syndrome(uint8_t *word, uint8_t *synd)
    {
        try
        {
            auto &eng = global_engine();
            std::vector<uint8_t> s(eng.H.mc, 0);
            eng.H.multiply_right(word, s.data());
            std::memcpy(synd, s.data(), s.size());
        }
        catch (const std::exception &e) { die("syndrome():", e.what()); }
    }

    // ---- part 2: handle API ----------------------------------------------------------------------------

    const char *ldpc_b200_last_error(void) { return g_error.c_str(); }
    const char *ldpc_b200_version(void) { return "libldpc_b200 0.1 (sm_100a)"; }

    ldpc_b200_ctx *ldpc_b200_open(const char *pcFile, const char *genFile, int device)
    {
        ldpc_b200_ctx *ctx = nullptr;
        guarded([&] {
            auto c = std::make_unique<ldpc_b200_ctx>();
            c->eng = std::make_unique<b200::Engine>(pcFile ? pcFile : "", genFile ? genFile : "", device);
            ctx = c.release();
        });
        return ctx;
    }

    void ldpc_b200_close(ldpc_b200_ctx *ctx) { delete ctx; }

    int ldpc_b200_info(const ldpc_b200_ctx *ctx, ldpc_b200_code_info *info)
    {
        return guarded([&] {
            if (!ctx || !info) throw std::runtime_error("null argument");
            const auto &H = ctx->eng->H;
            const auto &G = ctx->eng->G;
            info->nc = H.nc; info->mc = H.mc; info->nnz = H.nnz; info->kc = H.kc();
            info->nct = H.nct(); info->mct = H.mct(); info->kct = H.kct();
            info->n_punct = (int)H.puncture.size(); info->n_short = (int)H.shorten.size();
            info->max_degree = H.max_degree; info->max_check_degree = H.max_cn_degree; info->max_var_degree = H.max_vn_degree;
            info->has_generator = ctx->eng->has_gen ? 1 : 0;
            info->g_rows = ctx->eng->has_gen ? G.mc : 0; info->g_cols = ctx->eng->has_gen ? G.nc : 0; info->g_nnz = G.nnz;
        });
    }

    int ldpc_b200_set_tuning(ldpc_b200_ctx *ctx, const ldpc_b200_tuning *t)
    {
        return guarded([&] {
            if (!ctx || !t) throw std::runtime_error("null argument");
            if (t->precision != LDPC_B200_F64 && t->precision != LDPC_B200_F32) throw std::runtime_error("bad precision");
            if (t->residency < 0 || t->residency > 2) throw std::runtime_error("bad residency");
            if (t->schedule != LDPC_B200_FLOODING && t->schedule != LDPC_B200_LAYERED) throw std::runtime_error("bad schedule");
            if (t->layered_ms_scale64 < 0 || t->layered_ms_scale64 > 64) throw std::runtime_error("layered_ms_scale64 must be 0 .. 64");
            ctx->eng->tuning = *t;
        });
    }

    int ldpc_b200_get_tuning(const ldpc_b200_ctx *ctx, ldpc_b200_tuning *t)
    {
        return guarded([&] {
            if (!ctx || !t) throw std::runtime_error("null argument");
            *t = ctx->eng->tuning;
        });
    }

    int ldpc_b200_prepare(ldpc_b200_ctx *ctx, decoder_param dp, uint64_t n_frames)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            ctx->eng->prepare(dp, n_frames);
        });
    }

    int ldpc_b200_set_modulation(ldpc_b200_ctx *ctx, int M, const int *labels, const int *bit_mapper)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            ctx->eng->set_modulation(M, labels, bit_mapper);
        });
    }

    int ldpc_b200_set_fading(ldpc_b200_ctx *ctx, int coherence)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            ctx->eng->set_fading(coherence);
        });
    }

    int ldpc_b200_set_quant(ldpc_b200_ctx *ctx, const ldpc_b200_quant *q)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            ctx->eng->set_quant(q);
        });
    }

    int ldpc_b200_get_quant(const ldpc_b200_ctx *ctx, ldpc_b200_quant *q)
    {
        return guarded([&] {
            if (!ctx || !q) throw std::runtime_error("null argument");
            *q = ctx->eng->quant;
        });
    }

    int ldpc_b200_set_layers(ldpc_b200_ctx *ctx, int n_layers, const int *layer_ptr, const int *layer_check)
    {
        return guarded([&] {
            if (!ctx || n_layers < 0 || (n_layers > 0 && (!layer_ptr || !layer_check))) throw std::runtime_error("bad argument");
            std::vector<std::vector<int>> layers((size_t)n_layers);
            for (int l = 0; l < n_layers; ++l) layers[l].assign(layer_check + layer_ptr[l], layer_check + layer_ptr[l + 1]);
            ctx->eng->set_layers(std::move(layers));
        });
    }

    int ldpc_b200_load_layers(ldpc_b200_ctx *ctx, const char *layer_file)
    {
        return guarded([&] {
            if (!ctx || !layer_file) throw std::runtime_error("null argument");
            ctx->eng->set_layers(b200::read_layer_file(layer_file));
        });
    }

    int ldpc_b200_get_layers(ldpc_b200_ctx *ctx, int *layer_of)
    {
        int n = -1;
        guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            const auto &layers = ctx->eng->layers();
            if (layer_of)
                for (size_t l = 0; l < layers.size(); ++l)
                    for (int c : layers[l]) layer_of[c] = (int)l;
            n = (int)layers.size();
        });
        return n;
    }

    int ldpc_b200_get_edges(const ldpc_b200_ctx *ctx, int *rows, int *cols)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            const auto &H = ctx->eng->H;
            for (int e = 0; e < H.nnz; ++e) { rows[e] = H.e_row[e]; cols[e] = H.e_col[e]; }
        });
    }

    int ldpc_b200_get_bit_pos(const ldpc_b200_ctx *ctx, int *bit_pos)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            const auto &H = ctx->eng->H;
            for (int i = 0; i < H.nct(); ++i) bit_pos[i] = H.bit_pos[i];
        });
    }

    int ldpc_b200_get_puncture(const ldpc_b200_ctx *ctx, int *punct, int *shorten)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            const auto &H = ctx->eng->H;
            for (size_t i = 0; i < H.puncture.size(); ++i) punct[i] = H.puncture[i];
            for (size_t i = 0; i < H.shorten.size(); ++i) shorten[i] = H.shorten[i];
        });
    }

    int ldpc_b200_get_layout(ldpc_b200_ctx *ctx, int *edge_slot, int *n_slots, int *frames_per_cta, int *threads_per_cta, int *residency)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            int res = 0;
            size_t smem = 0;
            const auto &l = ctx->eng->layout_for(ctx->eng->tuning.precision, 0, &res, &smem);
            if (edge_slot) for (int e = 0; e < ctx->eng->H.nnz; ++e) edge_slot[e] = l.edge_slot[e];
            if (n_slots) *n_slots = l.n_slots;
            if (frames_per_cta) *frames_per_cta = l.lanes * (ctx->eng->tuning.precision == LDPC_B200_F32 ? 4 : 2);
            if (threads_per_cta) *threads_per_cta = l.threads;
            if (residency) *residency = res;
        });
    }

    int ldpc_b200_get_bec_layout(ldpc_b200_ctx *ctx, int *edge_slot, int *n_slots)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            b200::BecSliceLayout l;
            l.build(ctx->eng->H);
            if (edge_slot) for (int e = 0; e < ctx->eng->H.nnz; ++e) edge_slot[e] = l.edge_slot[e];
            if (n_slots) *n_slots = l.n_slots;
        });
    }

    int ldpc_b200_rank(const ldpc_b200_ctx *ctx)
    {
        int r = -1;
        guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            r = ctx->eng->H.rank();
        });
        return r;
    }

    int ldpc_b200_encode(const ldpc_b200_ctx *ctx, const uint8_t *info, uint8_t *cw_full)
    {
        return guarded([&] {
            if (!ctx || !ctx->eng->has_gen) throw std::runtime_error("no generator matrix loaded");
            std::vector<uint8_t> cw(std::max(ctx->eng->G.nc, ctx->eng->H.nc), 0);
            ctx->eng->G.multiply_left(info, cw.data());
            std::memcpy(cw_full, cw.data(), ctx->eng->H.nc);
        });
    }

    int ldpc_b200_syndrome(const ldpc_b200_ctx *ctx, const uint8_t *word, uint8_t *synd)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            std::memset(synd, 0, ctx->eng->H.mc);
            ctx->eng->H.multiply_right(word, synd);
        });
    }

    int ldpc_b200_decode_batch(ldpc_b200_ctx *ctx, decoder_param dp, const double *llr, int64_t n_frames, double *llr_out, uint8_t *hard, int32_t *iters)
    {
        return guarded([&] {
            if (!ctx || !llr) throw std::runtime_error("null argument");
            ctx->eng->decode_batch_host(dp, llr, LDPC_B200_LLR_F64, 1.0, n_frames, llr_out, hard, nullptr, iters);
        });
    }

    int ldpc_b200_decode_batch_device(ldpc_b200_ctx *ctx, decoder_param dp, const double *d_llr, int64_t n_frames, double *d_llr_out,
                                      uint8_t *d_hard, int32_t *d_iters, void *stream)
    {
        return guarded([&] {
            if (!ctx || !d_llr) throw std::runtime_error("null argument");
            b200::FrameSource src;
            src.kind = 0;
            src.d_llr = d_llr;
            b200::FrameSink sink;
            sink.d_llr_out = d_llr_out; sink.d_hard = d_hard; sink.d_iters = d_iters;
            ctx->eng->launch(dp, src, sink, (uint64_t)n_frames, stream);
        });
    }

    int ldpc_b200_decode_batch_ex(ldpc_b200_ctx *ctx, decoder_param dp, const void *llr, int llr_type, double llr_scale, int64_t n_frames,
                                  double *llr_out, uint8_t *hard, uint32_t *hard_bits, int32_t *iters)
    {
        return guarded([&] {
            if (!ctx || !llr) throw std::runtime_error("null argument");
            ctx->eng->decode_batch_host(dp, llr, llr_type, llr_scale, n_frames, llr_out, hard, hard_bits, iters);
        });
    }

    int ldpc_b200_decode_batch_device_ex(ldpc_b200_ctx *ctx, decoder_param dp, const void *d_llr, int llr_type, double llr_scale, int64_t n_frames,
                                         double *d_llr_out, uint8_t *d_hard, uint32_t *d_hard_bits, int32_t *d_iters, void *stream)
    {
        return guarded([&] {
            if (!ctx || !d_llr) throw std::runtime_error("null argument");
            b200::FrameSource src;
            src.kind = 0;
            if (llr_type == LDPC_B200_LLR_F64) src.d_llr = (const double *)d_llr;
            else if (llr_type == LDPC_B200_LLR_F32) src.d_llr_f32 = (const float *)d_llr;
            else if (llr_type == LDPC_B200_LLR_I8) { src.d_llr_i8 = (const int8_t *)d_llr; src.i8_scale = llr_scale; }
            else throw std::runtime_error("bad llr_type");
            b200::FrameSink sink;
            sink.d_llr_out = d_llr_out; sink.d_hard = d_hard; sink.d_iters = d_iters;
            sink.d_hard_bits = d_hard_bits; sink.hard_words = (ctx->eng->H.nc + 31) / 32;
            ctx->eng->launch(dp, src, sink, (uint64_t)n_frames, stream);
        });
    }

    int ldpc_b200_decode_bec_batch(ldpc_b200_ctx *ctx, decoder_param dp, const uint8_t *in, const uint8_t *cw, int64_t n_frames,
                                   uint8_t *out, uint8_t *hard, int32_t *iters)
    {
        return guarded([&] {
            if (!ctx || !in || !cw) throw std::runtime_error("null argument");
            ctx->eng->decode_bec_host(dp, in, cw, n_frames, out, hard, iters);
        });
    }

    int ldpc_b200_channel(ldpc_b200_ctx *ctx, const char *channel, double x, uint64_t seed, uint32_t point, uint64_t frame0,
                          int64_t n_frames, uint8_t *cw, double *llr, uint8_t *llr_u8)
    {
        return guarded([&] {
            if (!ctx || !channel) throw std::runtime_error("null argument");
            ctx->eng->channel_host(channel, x, seed, point, frame0, n_frames, cw, llr, llr_u8);
        });
    }

    int ldpc_b200_sim_point(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed, uint32_t point,
                            uint64_t frame0, uint64_t n_frames, uint64_t counters[4], float *device_ms)
    {
        return guarded([&] {
            if (!ctx || !channel || !counters) throw std::runtime_error("null argument");
            uint64_t c[5] = {0, 0, 0, 0, 0};
            ctx->eng->sim_point(dp, channel, x, seed, point, frame0, n_frames, c, device_ms);
            for (int i = 0; i < 4; ++i) counters[i] += c[i];
        });
    }

    int ldpc_b200_sim_point_log(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed, uint32_t point,
                                uint64_t frame0, uint64_t n_frames, uint64_t counters[4], ldpc_b200_error_record *records, int64_t capacity,
                                int64_t *n_errors)
    {
        return guarded([&] {
            if (!ctx || !channel || !counters) throw std::runtime_error("null argument");
            uint64_t c[5] = {0, 0, 0, 0, 0};
            ctx->eng->sim_point_log(dp, channel, x, seed, point, frame0, n_frames, c, records, capacity, n_errors);
            for (int i = 0; i < 4; ++i) counters[i] += c[i];
        });
    }

    int ldpc_b200_error_report(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed, uint32_t point,
                               const uint64_t *frames, int64_t n_frames, ldpc_b200_frame_report *reports, int32_t *failed_bits,
                               int64_t bits_capacity, int32_t *failed_checks, int64_t checks_capacity, int64_t *bits_needed,
                               int64_t *checks_needed)
    {
        return guarded([&] {
            if (!ctx || !channel) throw std::runtime_error("null argument");
            if (n_frames < 0 || bits_capacity < 0 || checks_capacity < 0) throw std::runtime_error("error_report: negative size");
            if ((n_frames > 0 && (!frames || !reports)) || (bits_capacity > 0 && !failed_bits) || (checks_capacity > 0 && !failed_checks))
                throw std::runtime_error("null argument");
            std::vector<ldpc_b200_frame_report> rep((size_t)n_frames);
            std::vector<int32_t> bits, checks;
            ctx->eng->error_report(dp, channel, x, seed, point, frames, n_frames, rep.data(), bits, checks);
            const int64_t nb = (int64_t)bits.size(), nk = (int64_t)checks.size();
            if (bits_needed) *bits_needed = nb;
            if (checks_needed) *checks_needed = nk;
            if (nb > bits_capacity || nk > checks_capacity)
                throw std::runtime_error("error_report: the reports need " + std::to_string(nb) + " failed bits and " + std::to_string(nk) +
                                         " failed checks; capacities " + std::to_string(bits_capacity) + " and " + std::to_string(checks_capacity));
            std::copy(rep.begin(), rep.end(), reports);
            std::copy(bits.begin(), bits.end(), failed_bits);
            std::copy(checks.begin(), checks.end(), failed_checks);
        });
    }

    int ldpc_b200_sim_point_async(ldpc_b200_ctx *ctx, decoder_param dp, const char *channel, double x, uint64_t seed, uint32_t point,
                                  uint64_t frame0, uint64_t n_frames, uint64_t *d_counters, void *stream)
    {
        return guarded([&] {
            if (!ctx || !channel || !d_counters) throw std::runtime_error("null argument");
            ctx->eng->sim_point_async(dp, channel, x, seed, point, frame0, n_frames, reinterpret_cast<unsigned long long *>(d_counters), stream);
        });
    }

    int ldpc_b200_simulate(ldpc_b200_ctx *ctx, decoder_param dp, channel_param cp, simulation_param sp, sim_results_t *results,
                           bool *stopFlag, int rank, int world, ldpc_b200_allreduce_fn allreduce, void *user, int quiet)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            b200::run_sweep(*ctx->eng, dp, cp, sp, results, stopFlag, rank, world, allreduce, user, quiet != 0, true);
        });
    }

    int ldpc_b200_simulate_ex(ldpc_b200_ctx *ctx, decoder_param dp, channel_param cp, simulation_param sp, sim_results_t *results,
                              bool *stopFlag, int rank, int world, ldpc_b200_allreduce_fn allreduce, ldpc_b200_round_fn round_fn,
                              void *user, int quiet)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            b200::run_sweep(*ctx->eng, dp, cp, sp, results, stopFlag, rank, world, allreduce, user, quiet != 0, true, round_fn);
        });
    }

    int ldpc_b200_reset_stats(ldpc_b200_ctx *ctx)
    {
        return guarded([&] {
            if (!ctx) throw std::runtime_error("null argument");
            ctx->eng->stats = ldpc_b200_stats{};
        });
    }

    int ldpc_b200_smem_probe(ldpc_b200_ctx *ctx, double *gb_per_s)
    {
        return guarded([&] {
            if (!ctx || !gb_per_s) throw std::runtime_error("null argument");
            *gb_per_s = ctx->eng->smem_probe();
        });
    }

    int ldpc_b200_fp64_probe(ldpc_b200_ctx *ctx, double *ginst_per_s)
    {
        return guarded([&] {
            if (!ctx || !ginst_per_s) throw std::runtime_error("null argument");
            *ginst_per_s = ctx->eng->fp64_probe();
        });
    }

    int ldpc_b200_get_stats(const ldpc_b200_ctx *ctx, ldpc_b200_stats *s)
    {
        return guarded([&] {
            if (!ctx || !s) throw std::runtime_error("null argument");
            *s = ctx->eng->stats;
        });
    }
}
