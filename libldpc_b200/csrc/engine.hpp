// Host engine: owns the loaded code, the device copies of its tile layouts and the workspaces,
// and launches the persistent tile kernel (kernels.cuh).  C++17 host code; the CUDA runtime is only
// touched lazily so that loader / GF(2) helpers work on machines without a GPU.
#pragma once
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <set>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/ldpc_b200.h"
#include "code.hpp"

struct CUevent_st;  // cudaEvent_t = CUevent_st *
struct CUstream_st; // cudaStream_t = CUstream_st *

namespace b200
{
    // Owners of CUDA resources; the deleters are defined in engine.cu, and ignore errors as teardown has nobody to report to.
    struct DeviceFree { void operator()(void *p) const; };
    struct PinnedFree { void operator()(void *p) const; };
    struct EventDestroy { void operator()(CUevent_st *e) const; };
    struct StreamDestroy { void operator()(CUstream_st *s) const; };
    template <typename T>
    using DevPtr = std::unique_ptr<T, DeviceFree>;    // device memory (cudaMalloc)
    template <typename T>
    using PinnedPtr = std::unique_ptr<T, PinnedFree>; // pinned host memory (cudaHostAlloc)
    using Event = std::unique_ptr<CUevent_st, EventDestroy>;
    using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;
    struct DevBuf // device buffer that is grown on demand
    {
        DevPtr<unsigned char> p;
        size_t cap = 0; // bytes
    };

    struct DeviceLayered;    // device-resident LayeredLayout (engine.cu; layered schedule)
    struct DeviceLayout;     // device-resident TileLayout (engine.cu; erasure decoder)
    struct DeviceSegLayout;  // device-resident SegLayout (engine.cu; tile4 kernel)

    struct FrameSource
    {
        int kind = 0;                // SRC_* of kernels.cuh
        const double *d_llr = nullptr; // SRC_LLR: device [n][nc] ...
        const float *d_llr_f32 = nullptr;  // ... or the same frames as binary32
        const int8_t *d_llr_i8 = nullptr;  // ... or as quantised int8 (LLR = value * i8_scale)
        double i8_scale = 1.0;
        const uint8_t *d_bec_in = nullptr, *d_bec_cw = nullptr; // BEC decode mode
        double x = 0;                // channel parameter (snr dB or epsilon)
        uint64_t seed = 0;
        uint32_t point = 0;
        uint64_t frame0 = 0;
    };

    struct FrameSink
    {
        double *d_llr_out = nullptr;
        uint8_t *d_hard = nullptr;
        uint32_t *d_hard_bits = nullptr; // bit-packed decisions, hard_words 32-bit words per frame
        int hard_words = 0;
        uint8_t *d_bec_out = nullptr;
        int32_t *d_iters = nullptr;
        unsigned long long *d_counters = nullptr; // [5]; null -> engine scratch
        unsigned long long *d_err_log = nullptr, *d_err_count = nullptr; // per-error diagnostics log (device), capacity in records
        unsigned long long err_cap = 0;
    };

    class Engine
    {
    public:
        Engine(const std::string &pc_file, const std::string &gen_file, int device);
        ~Engine();

        HostCode H, G;
        bool has_gen = false;
        int device = -1;
        ldpc_b200_tuning tuning{};
        ldpc_b200_stats stats{};

        // Chooses / builds the layout for (precision, algorithm) under the current tuning (host only).
        const SegLayout &layout_for(int precision, int alg, int *residency, size_t *smem_bytes);

        // Launches the tile kernel over n_frames frames on `stream` (0 = engine stream).  Asynchronous unless may_block, which
        // allows the one-off timed shape trials (they run and wait for trial kernels on `stream`).
        void launch(const decoder_param &dp, const FrameSource &src, const FrameSink &sink, uint64_t n_frames, void *stream, bool may_block = false);
        // runs the one-off shape trials for (decoder type, current precision) and a job of n_frames now (blocking)
        void prepare(const decoder_param &dp, uint64_t n_frames);

        // Blocking helpers used by the C ABI
        // llr_type: LDPC_B200_LLR_F64 / _F32 / _I8 (element type of `llr`); hard_bits: bit-packed decisions, ceil(nc/32) words per frame
        void decode_batch_host(const decoder_param &dp, const void *llr, int llr_type, double llr_scale, int64_t n, double *llr_out, uint8_t *hard,
                               uint32_t *hard_bits, int32_t *iters);
        void decode_bec_host(const decoder_param &dp, const uint8_t *in, const uint8_t *cw, int64_t n, uint8_t *out, uint8_t *hard, int32_t *iters);
        void channel_host(const std::string &channel, double x, uint64_t seed, uint32_t point, uint64_t frame0, int64_t n,
                          uint8_t *cw, double *llr, uint8_t *llr_u8);
        void sim_point(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point,
                       uint64_t frame0, uint64_t n_frames, uint64_t counters[5], float *device_ms);
        void sim_point_log(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point, uint64_t frame0,
                           uint64_t n_frames, uint64_t counters[5], ldpc_b200_error_record *records, int64_t capacity, int64_t *n_errors);
        // Replays global frames frames[0 .. n) of a sweep point (any order, repeats allowed) under the current tuning and
        // reports each: reports[i] with offsets into `bits` (failed transmitted positions, in transmitted order) and `checks`
        // (unsatisfied checks, ascending), which are replaced.  Blocking.
        void error_report(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point, const uint64_t *frames,
                          int64_t n, ldpc_b200_frame_report *reports, std::vector<int32_t> &bits, std::vector<int32_t> &checks);
        void sim_point_async(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point,
                             uint64_t frame0, uint64_t n_frames, unsigned long long *d_counters, void *stream, bool may_block = false);

        // Pipelined rounds of the sweep driver: a round is launched into one of two slots (device counters, a pinned host copy,
        // an event) and collected later, so the next round is already running while the host reads the previous one.
        void round_launch(int slot, const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point, uint64_t frame0,
                          uint64_t n_frames);
        void round_collect(int slot, uint64_t counters[5]);
        // frames of one full wave of the persistent grid for this decoder type under the current tuning (rounds are sized in waves)
        uint64_t wave_frames(const decoder_param &dp, const std::string &channel);

        // M-ASK with bit-metric decoding for the AWGN sweep (M = 2: BPSK)
        void set_modulation(int M, const int *labels, const int *bit_mapper);
        int ask_M = 2;
        std::vector<int32_t> ask_labels, ask_rev, ask_bm;
        std::vector<double> ask_X;

        // Rayleigh fading: transmitted positions per fading coefficient (0 = one coefficient per frame, quasi-static)
        void set_fading(int coherence)
        {
            if (coherence < 0) throw std::runtime_error("fading: the coherence length must be >= 0");
            fading_L = coherence;
        }
        int fading_L = 1;

        // fixed-point layered min-sum (DESIGN.md §3.7): ch_bits = 0 is off; set_quant validates and keeps the old setting on failure
        void set_quant(const ldpc_b200_quant *q);
        ldpc_b200_quant quant{};
        bool quantised() const { return quant.ch_bits > 0; }

        // layered schedule: the layering in use (empty = built-in first-fit layering, made on first use)
        void set_layers(std::vector<std::vector<int>> layers);
        const std::vector<std::vector<int>> &layers();

        // sustained shared-memory read bandwidth of the device in GB/s (LDS.128 streaming from every SM)
        double smem_probe();
        // sustained FP64 instruction rate of the device in G thread-instructions/s (DFMA streaming from every SM)
        double fp64_probe();

        void ensure_cuda();
        void *engine_stream() const { return stream_.get(); }

    private:
        struct Config
        {
            int precision, alg, residency, lanes, fpc, threads, ctas;
            size_t smem_bytes;
            bool tm;                                  // TMEM mirror in use
            bool wide;                                // global residency: the 1-CTA-per-SM / 128-register kernel build
            bool idx16;                               // 16-bit index entries (shared-memory residency with the TMEM mirror)
            uint32_t tm_alloc_cols, tm_cols_per_warp, tm_vn_off;
            bool lockstep;                            // fixed iterations run the lock-step kernel (its gather addresses and descriptors fit)
            uint32_t tm_idx_off;                      // lock-step kernel: column of the gather addresses inside a warp window
        };
        Config choose(int precision, int alg, uint64_t n_frames);
        const SegLayout &get_seg_layout(int lanes, int threads, int isz = 4);
        DeviceSegLayout &device_seg_layout(int lanes, int threads, int isz = 4);
        const TileLayout &get_layout(int fpc, int threads);
        struct TrialGuard; // puts back what a shape trial changes (engine.cu)
        void autotune_global(int alg, const decoder_param &dp, CUstream_st *s);
        void autotune_pair(int alg, const decoder_param &dp, CUstream_st *s);
        // one shape trial: frames per ms of the current shape on synthetic AWGN frames; 0 when it is not a candidate
        double trial_rate(const decoder_param &dp, double snr, unsigned long long *d_cnt, uint64_t frames, CUstream_st *s,
                          const std::function<bool()> &eligible = nullptr);
        float time_ms(CUstream_st *s, const std::function<void()> &work); // device time of `work` on s (ev0_ .. ev1_; blocking)
        void maybe_autotune(int alg, const decoder_param &dp, uint64_t n_frames, CUstream_st *s);
        // frames of one full wave of the persistent grid for a batch job of this decoder type (runs the shape trial first where it applies)
        int64_t batch_wave(const decoder_param &dp, uint64_t n_frames, CUstream_st *s);
        // the fixed-point layered kernel's shape under the current tuning: lanes per node, threads, the kernel, CTAs per SM
        void quant_shape(int *lanes, int *threads, const void **fn, int *per_sm);
        // outcomes of the shape trials are remembered across processes: $LDPC_B200_TUNE_CACHE (a directory; "off" disables) or
        // ~/.cache/libldpc_b200, one small text file per (code, device)
        std::string tune_cache_file();
        void tune_cache_load();
        void tune_cache_store();
        bool tune_cache_loaded_ = false;
        std::string device_name_;
        void launch_layered(const decoder_param &dp, const FrameSource &src, const FrameSink &sink, uint64_t n_frames, CUstream_st *s);
        std::vector<std::vector<int>> layers_;
        std::map<std::pair<int, int>, std::unique_ptr<LayeredLayout>> lay_layouts_;
        void launch_bec(const decoder_param &dp, const FrameSource &src, const FrameSink &sink, uint64_t n_frames, CUstream_st *s);
        DeviceLayout &device_layout(int fpc, int threads, bool idx16);
        void ensure_state(size_t bytes, CUstream_st *s);
        void release_state(CUstream_st *s);
        bool try_seg_layout(int lanes, int threads, int isz);
        int channel_kind(const std::string &name) const; // SRC_* of a channel name; RAYLEIGH needs BPSK
        void launch_channel(int kind, double x, uint64_t seed, uint32_t point, uint64_t frame0, const uint64_t *frames, int64_t n,
                            uint8_t *d_cw, double *d_llr, uint8_t *d_u8, CUstream_st *s);
        const void *tile_fn(const Config &c, bool et); // the tile kernel of c (early termination: et), its attributes set
        // dynamic shared-memory opt-in (max_shared: and the all-shared carveout) of a kernel, set on this engine's first use of it
        void set_smem_attributes(const void *fn, int smem_optin, bool max_shared);
        std::set<const void *> attrs_set_; // kernels whose attributes this engine has set (it is bound to one device)
        // stats of the last launch, and of a finished job (from its counters)
        void note_launch(int fpc, int threads, int ctas, int residency, int precision, size_t smem_bytes);
        void account(double ms, uint64_t frames, uint64_t executed_iterations);

        bool cuda_ready_ = false;
        int sm_count_ = 148;
        size_t smem_optin_ = 227 * 1024, smem_per_sm_ = 228 * 1024;
        std::map<std::pair<int, int>, int> pair_tuned_; // (precision, alg) -> 1 when the two-CTAs-per-SM shape won its trial (shared-memory residency)
        int force_pair_ = -1;                           // trial: -1 = use pair_tuned_, 0/1 = force
        std::map<std::pair<int, int>, std::unique_ptr<TileLayout>> layouts_;
        std::map<std::tuple<int, int, int>, std::unique_ptr<SegLayout>> seg_layouts_;
        std::map<std::tuple<int, int, int, int, int, size_t>, int> occupancy_;
        std::map<std::pair<int, int>, std::tuple<int, int, int>> tuned_; // (precision, alg) -> autotuned (lanes, threads, wide), global residency
        bool in_autotune_ = false;
        int force_wide_ = -1; // autotune trials: -1 = use tuned_/default, 0/1 = force
        std::unique_ptr<BecSliceLayout> bs_layout_;
        void ask_fill(void *ask_params); // uploads the tables on first use and fills an AskParams
        bool state_used_ = false;

        // CUDA resources.  Members are destroyed in reverse order: device layouts first, then buffers and events, then the
        // copy streams, and the engine stream last.
        Stream stream_;
        Event ev0_, ev1_;
        // host-buffer batch decode pipeline (decode_batch_host): copy streams, per-buffer events, cached device buffers
        Stream copy_in_, copy_out_;
        Event ev_in_[2], ev_k_[2], ev_out_[2];
        DevBuf db_in_[2], db_out_[2], db_hard_[2], db_it_[2], db_bits_[2];
        DevPtr<unsigned long long> d_round_[2]; // sweep rounds in flight
        PinnedPtr<unsigned long long> h_round_[2];
        Event ev_round_[2], ev_round0_[2], ev_rdone_[2];
        DevBuf state_;  // per-CTA state block (ensure_state)
        Event ev_state_; // recorded after every launch that uses the state block
        DevPtr<int32_t> d_bit_pos_, d_punct_, d_short_;
        DevPtr<int32_t> d_g_col_ptr_, d_g_row_; // generator matrix by column (device)
        DevPtr<int32_t> d_chk_ptr_, d_chk_var_; // check-major CSR of H: variable ids (error_report)
        DevPtr<int32_t> d_bs_row_ptr_, d_bs_col_ptr_; // bit-sliced BEC kernel
        DevPtr<uint16_t> d_bs_row_slot_, d_bs_col_slot_;
        DevPtr<uint8_t> d_bs_tx_flag_;
        DevPtr<unsigned long long> d_counters_;
        DevPtr<double> d_ask_X_;
        DevPtr<int32_t> d_ask_label_, d_ask_rev_, d_ask_bm_;
        std::map<std::tuple<int, int, bool>, std::unique_ptr<DeviceLayout>> dev_layouts_;
        std::map<std::tuple<int, int, int>, std::unique_ptr<DeviceSegLayout>> dev_seg_layouts_;
        std::map<std::pair<int, int>, std::unique_ptr<DeviceLayered>> dev_lay_;
    };

    // reference-semantics sweep driver (sim_driver.cpp)
    int run_sweep(Engine &eng, const decoder_param &dp, const channel_param &cp, const simulation_param &sp,
                  sim_results_t *results, bool *stop_flag, int rank, int world, ldpc_b200_allreduce_fn allreduce,
                  void *user, bool quiet, bool write_file, ldpc_b200_round_fn round_fn = nullptr);
} // namespace b200
