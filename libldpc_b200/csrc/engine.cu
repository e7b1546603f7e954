#include "engine.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <tuple>
#include <sys/stat.h>
#include <unistd.h>

#include "tile_launch.cuh"
#include "bec_kernel.cuh"
#include "bec_slice.cuh"
#include "layered.cuh"
#include "report.cuh"

namespace b200
{
#define CUDA_OK(call)                                                                                              \
    do                                                                                                             \
    {                                                                                                              \
        cudaError_t e_ = (call);                                                                                   \
        if (e_ != cudaSuccess)                                                                                     \
            throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #call);        \
    } while (0)

    void DeviceFree::operator()(void *p) const { cudaFree(p); }
    void PinnedFree::operator()(void *p) const { cudaFreeHost(p); }
    void EventDestroy::operator()(CUevent_st *e) const { cudaEventDestroy(e); }
    void StreamDestroy::operator()(CUstream_st *s) const { cudaStreamDestroy(s); }

    struct DeviceLayout
    {
        DevPtr<uint32_t> cn_desc, vn_desc;
        DevPtr<void> cn_col, vn_slot, vn_id;
        const TileLayout *host = nullptr;
    };

    struct DeviceLayered
    {
        DevPtr<uint32_t> seg, idx;
        const LayeredLayout *host = nullptr;
    };

    struct DeviceSegLayout
    {
        DevPtr<uint32_t> cn_seg, vn_seg, var_pos;
        DevPtr<uint8_t> cn_idx, vn_idx;
        DevPtr<int32_t> tx_pos, punct_pos, short_pos;
        const SegLayout *host = nullptr;
    };

    namespace
    {
        template <typename T>
        DevPtr<T> device_alloc(size_t count)
        {
            T *d = nullptr;
            CUDA_OK(cudaMalloc(&d, count * sizeof(T)));
            return DevPtr<T>(d);
        }

        Event make_event(unsigned flags)
        {
            cudaEvent_t e = nullptr;
            CUDA_OK(cudaEventCreateWithFlags(&e, flags));
            return Event(e);
        }

        Stream make_stream()
        {
            cudaStream_t s = nullptr;
            CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
            return Stream(s);
        }

        // waits for the device, then replaces the buffer by one of `bytes` when it is smaller (kernels or copies in flight may use it)
        void grow(DevBuf &b, size_t bytes)
        {
            if (bytes <= b.cap) return;
            CUDA_OK(cudaDeviceSynchronize());
            b.p.reset();
            b.cap = 0;
            b.p = device_alloc<unsigned char>(bytes);
            b.cap = bytes;
        }

        template <typename V>
        DevPtr<V> upload(const std::vector<V> &v)
        {
            DevPtr<V> d = device_alloc<V>(std::max<size_t>(v.size(), 1));
            if (!v.empty()) CUDA_OK(cudaMemcpy(d.get(), v.data(), v.size() * sizeof(V), cudaMemcpyHostToDevice));
            return d;
        }

        template <typename IdxT>
        DevPtr<void> upload_idx(const std::vector<uint32_t> &v)
        {
            std::vector<IdxT> tmp(v.size() ? v.size() : 1);
            for (size_t i = 0; i < v.size(); ++i) tmp[i] = static_cast<IdxT>(v[i]);
            return upload(tmp);
        }

        size_t tile_smem_bytes(const TileLayout &l, size_t sizeof_t, int nc, bool idx16)
        {
            const size_t idx = idx16 ? 2 : 4;
            size_t b = sizeof_t * ((size_t)l.n_slots + 2 * (size_t)nc) * l.fpc;
            b += 4 * ((size_t)l.cn_rounds + l.vn_rounds) * l.nt;
            b += idx * ((size_t)l.n_slots + l.n_vslots + (size_t)l.vn_rounds * l.nt);
            return b + 16;
        }

        // pos_entries: transmitted (padded to a multiple of 4) + punctured + shortened positions, kept as uint16 beside the tables
        size_t seg_smem_bytes(const SegLayout &l, size_t pos_entries)
        {
            const size_t rs = 16 * (size_t)l.lanes;
            size_t b = rs * ((size_t)l.n_slots + 2 * (size_t)l.n_pos);
            b += 16 * ((size_t)l.cn_max_segs + l.vn_max_segs) * l.warps;
            b += l.cn_idx.size() + l.vn_idx.size(); // both multiples of 16
            b += (2 * pos_entries + 15) & ~(size_t)15;
            return b + 16;
        }

        int alg_of(const decoder_param &dp) { return dp.type && std::string(dp.type) == "BP_MS" ? ALG_MS : ALG_BP; } // src/decoding/decoder.h:76

        // a persistent grid of `ctas` CTAs, but no more CTAs than work items (`need`) and at least one
        int clamp_grid(int ctas, uint64_t need) { return (uint64_t)ctas > need ? (int)std::max<uint64_t>(need, 1) : ctas; }

        // Channel constants of a point: AWGN (M-ASK, Rayleigh fading) at x dB -> noise variance, deviation and LLR scale
        // (src/sim/channel.cpp:39-40); BSC / BEC with probability x -> the BSC's LLR magnitude (src/sim/channel.cpp:139) and the
        // 32-bit threshold of a uniform word.  The other channel's fields stay 0.
        struct ChannelConsts
        {
            double sigma2 = 0, sigma = 0, llr_scale = 0, delta = 0;
            uint32_t thr = 0;
        };
        ChannelConsts channel_consts(int kind, double x)
        {
            ChannelConsts c;
            if (kind == SRC_AWGN || kind == SRC_ASK || kind == SRC_RAYLEIGH)
            {
                c.sigma2 = std::pow(10.0, -x / 10.0);
                c.sigma = std::sqrt(c.sigma2);
                c.llr_scale = 2.0 / c.sigma2;
            }
            else if (kind == SRC_BSC || kind == SRC_BEC)
            {
                c.delta = std::log((1 - x) / x);
                const double t = std::floor(x * 4294967296.0);
                c.thr = t <= 0 ? 0u : (t >= 4294967295.0 ? 4294967295u : (uint32_t)t);
            }
            return c;
        }

        // Launches a kernel that takes one parameter struct.  As after <<<...>>>, the error is read (and cleared) with
        // cudaGetLastError.
        template <typename P>
        void launch_kernel(const void *fn, int ctas, int threads, size_t smem_bytes, cudaStream_t s, P params, const char *what)
        {
            void *args[] = {&params};
            (void)cudaLaunchKernel(fn, dim3(ctas), dim3(threads), args, smem_bytes, s);
            const cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " (" + what + " launch)");
        }
    } // namespace

    // ------------------------------------------------------------------------------------------

    Engine::Engine(const std::string &pc_file, const std::string &gen_file, int dev) : device(dev)
    {
        H.load(pc_file, true);
        if (!gen_file.empty())
        {
            G.load(gen_file, false);
            has_gen = true;
        }
        tuning.precision = LDPC_B200_F64;
        tuning.residency = LDPC_B200_AUTO;
        tuning.bec_deg1_compat = 1;
    }

    Engine::~Engine()
    {
        if (cuda_ready_) cudaSetDevice(device); // the members free themselves on this device
    }

    void Engine::ensure_cuda()
    {
        if (cuda_ready_)
        {
            CUDA_OK(cudaSetDevice(device));
            return;
        }
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n == 0)
            throw std::runtime_error("no CUDA device available: libldpc_b200 has no CPU fallback for decoding/simulation");
        if (device < 0) device = 0;
        if (device >= n) throw std::runtime_error("CUDA device index out of range");
        CUDA_OK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_OK(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10) throw std::runtime_error(std::string("libldpc_b200 is built for sm_100a only; found ") + prop.name);
        sm_count_ = prop.multiProcessorCount;
        device_name_ = prop.name;
        smem_optin_ = prop.sharedMemPerBlockOptin;
        smem_per_sm_ = prop.sharedMemPerMultiprocessor;
        stream_ = make_stream();
        ev0_ = make_event(cudaEventDefault);
        ev1_ = make_event(cudaEventDefault);
        std::vector<int32_t> bp(H.bit_pos.begin(), H.bit_pos.end()), pu(H.puncture.begin(), H.puncture.end()), sh(H.shorten.begin(), H.shorten.end());
        d_bit_pos_ = upload(bp);
        d_punct_ = upload(pu);
        d_short_ = upload(sh);
        if (has_gen)
        { // generator matrix by column (= variable id), rows in file order
            std::vector<int32_t> cp(G.col_ptr.begin(), G.col_ptr.end()), rows(G.nnz);
            for (int q = 0; q < G.nnz; ++q) rows[q] = (int32_t)G.e_row[G.col_edge[q]];
            d_g_col_ptr_ = upload(cp);
            d_g_row_ = upload(rows);
        }
        d_counters_ = device_alloc<unsigned long long>(8);
        CUDA_OK(cudaMemset(d_counters_.get(), 0, 8 * sizeof(unsigned long long)));
        cuda_ready_ = true;
    }

    const SegLayout &Engine::get_seg_layout(int lanes, int threads, int isz)
    {
        auto key = std::make_tuple(lanes, threads, isz);
        auto it = seg_layouts_.find(key);
        if (it == seg_layouts_.end())
        {
            auto l = std::make_unique<SegLayout>();
            l->build(H, lanes, threads, isz);
            it = seg_layouts_.emplace(key, std::move(l)).first;
        }
        return *it->second;
    }

    // false when the layout cannot be built (e.g. the padded slots of a code with many distinct degrees do not fit 16-bit entries)
    bool Engine::try_seg_layout(int lanes, int threads, int isz)
    {
        try
        {
            get_seg_layout(lanes, threads, isz);
            return true;
        }
        catch (const std::exception &)
        {
            return false;
        }
    }

    // Configuration policy.  A CTA holds lanes * VEC frames (VEC = 2 doubles / 4 floats per 16-byte
    // vector).  Shared-memory residency is used whenever the code fits: the widest tile that fits
    // with the default thread count wins (it shares every index load / address computation between
    // the most frames); otherwise messages live in global memory (L2 / HBM).
    const SegLayout &Engine::layout_for(int precision, int alg, int *residency, size_t *smem_bytes)
    {
        const int vec = precision == LDPC_B200_F32 ? 4 : 2;
        // compile-time caps of the kernels (tile4.cuh): shared-memory residency (the fp64 sum-product kernel has a lower one), global residency
        const int max_threads = tile_thread_cap(precision != LDPC_B200_F32, alg, true), g_max_threads = B200_TILE_MAX_THREADS;
        const int threads = tuning.threads_per_cta > 0 ? std::min(tuning.threads_per_cta, max_threads) : max_threads;
        int want_lanes = 0;
        if (tuning.frames_per_cta > 0)
        {
            if (tuning.frames_per_cta % vec) throw std::runtime_error("frames_per_cta must be a multiple of the vector width (2 for f64, 4 for f32)");
            want_lanes = tuning.frames_per_cta / vec;
            if (want_lanes != 1 && want_lanes != 2 && want_lanes != 4)
                throw std::runtime_error("frames_per_cta / vector width must be 1, 2 or 4");
        }
        const size_t limit = std::min<size_t>(smem_optin_ > 2048 ? smem_optin_ - 2048 : 0, (size_t)TILE_SMEM_OPTIN);
        // information words of the frames in flight (random codewords through the generator matrix), 16-byte rounded
        auto u_bytes = [&](int lanes) -> size_t { return has_gen ? (((size_t)4 * lanes * vec * ((G.mc + 31) / 32)) + 15) & ~(size_t)15 : 0; };
        size_t pos_entries = ((size_t)H.nct() + 3) & ~(size_t)3;
        for (int v : H.puncture) if (v >= 0 && v < H.nc) ++pos_entries;
        for (int v : H.shorten) if (v >= 0 && v < H.nc) ++pos_entries;
        if (tuning.residency != LDPC_B200_GLOBAL)
        {
            // 16-bit entries (record offset / 16) need every record offset of the layout below 2^16
            auto fits16 = [&](int lanes) { return (size_t)lanes * (size_t)(H.nnz + 32 * 64) < 65536 && (size_t)lanes * (size_t)(H.nc + 32 * 64) < 65536; };
            for (int lanes = 4; lanes >= 1; lanes >>= 1)
            {
                if (want_lanes && lanes != want_lanes) continue;
                bool i16 = tuning.idx16 == 2 && tuning.tmem == 0 && fits16(lanes);
                if (i16 && !try_seg_layout(lanes, threads, 2)) i16 = false; // many distinct degrees: the padded layout can still exceed 16 bits
                const SegLayout &l = get_seg_layout(lanes, threads, i16 ? 2 : 4);
                const size_t need = seg_smem_bytes(l, pos_entries) + u_bytes(lanes);
                if (need <= limit)
                {
                    // Nothing pinned by the caller and the widest tile that fits is two lanes: the same frames as TWO
                    // CTAs per SM of one lane and half the threads each hide each other's barriers and latencies
                    // (h.txt f64: 4.36 -> 4.47 Gb/s fixed-iteration, 6.48 -> 7.19 Gb/s with early termination).  The
                    // tables only fit twice with 16-bit entries.  Taken when the one-off trial (autotune_pair) found it
                    // faster on this device; choose() falls back when the pair cannot be resident.
                    bool want_pair = force_pair_ == 1;
                    if (force_pair_ < 0)
                    {
                        auto it = pair_tuned_.find(std::make_pair(precision, alg));
                        want_pair = it != pair_tuned_.end() && it->second == 1;
                    }
                    if (want_pair && lanes == 2 && !want_lanes && tuning.threads_per_cta <= 0 && tuning.idx16 == 0 && tuning.tmem == 0 &&
                        tuning.ctas <= 0 && fits16(1) && try_seg_layout(1, max_threads / 2, 2))
                    {
                        const SegLayout &l1 = get_seg_layout(1, max_threads / 2, 2);
                        const size_t need1 = seg_smem_bytes(l1, pos_entries) + u_bytes(1);
                        if (2 * (need1 + 2048) <= smem_per_sm_)
                        {
                            *residency = LDPC_B200_SMEM;
                            *smem_bytes = need1;
                            return l1;
                        }
                    }
                    *residency = LDPC_B200_SMEM;
                    *smem_bytes = need;
                    return l;
                }
            }
            if (tuning.residency == LDPC_B200_SMEM) throw std::runtime_error("code does not fit shared-memory residency with this tuning");
        }
        *residency = LDPC_B200_GLOBAL;
        int g_lanes = want_lanes ? want_lanes : 1, g_threads = tuning.threads_per_cta > 0 ? std::min(tuning.threads_per_cta, g_max_threads) : g_max_threads;
        if (!want_lanes && tuning.threads_per_cta <= 0)
        { // global residency, nothing pinned by the caller: the autotuned (lanes, threads) of this (precision, algorithm)
            auto it = tuned_.find(std::make_pair(precision, alg));
            if (it != tuned_.end()) { g_lanes = std::get<0>(it->second); g_threads = std::get<1>(it->second); }
        }
        *smem_bytes = u_bytes(g_lanes);
        return get_seg_layout(g_lanes, g_threads);
    }

    Engine::Config Engine::choose(int precision, int alg, uint64_t n_frames)
    {
        Config c{};
        c.precision = precision;
        c.alg = alg;
        const SegLayout &l = layout_for(precision, alg, &c.residency, &c.smem_bytes);
        c.lanes = l.lanes;
        c.fpc = l.lanes * (precision == LDPC_B200_F32 ? 4 : 2);
        c.threads = l.threads;
        // Tensor-Memory mirror (shared-memory residency): every warp gets a window of 4 columns per mirrored 16-byte
        // vector (its check tasks' c2v slots, then its variable tasks' channel LLRs); the windows of the warps that
        // share a TMEM lane partition (warp % 4) lie side by side in the 512 columns.
        c.tm = false;
        c.tm_alloc_cols = c.tm_cols_per_warp = c.tm_vn_off = 0;
        c.lockstep = false;
        c.tm_idx_off = 0;
        c.wide = false;
        if (c.residency == LDPC_B200_GLOBAL)
        {
            if (force_wide_ >= 0) c.wide = force_wide_ != 0;
            else
            {
                auto it = tuned_.find(std::make_pair(precision, alg));
                if (it != tuned_.end() && tuning.frames_per_cta <= 0 && tuning.threads_per_cta <= 0) c.wide = std::get<2>(it->second) != 0;
            }
        }
        if (c.residency == LDPC_B200_SMEM && tuning.tmem == 0)
        {
            // the lock-step kernel also keeps every gather address of a warp's tasks in its window (ls_idx_cols per task)
            uint32_t cn_max = 0, vn_max = 0, idx_max = 0;
            for (int w = 0; w < l.warps; ++w)
            {
                uint32_t cn = 0, vn = 0, idx = 0;
                for (int sgi = 0; sgi < l.cn_max_segs; ++sgi)
                {
                    const uint32_t d = l.cn_seg[4 * ((size_t)w * l.cn_max_segs + sgi)];
                    if (!d) break;
                    cn += (d & 0xFFu) * (d >> 16);
                    idx += (uint32_t)ls_idx_cols(true, (int)(d & 0xFFu)) * (d >> 16);
                }
                for (int sgi = 0; sgi < l.vn_max_segs; ++sgi)
                {
                    const uint32_t d = l.vn_seg[4 * ((size_t)w * l.vn_max_segs + sgi)];
                    if (!d) break;
                    vn += d >> 16;
                    idx += (uint32_t)ls_idx_cols(false, (int)(d & 0xFFu)) * (d >> 16);
                }
                cn_max = std::max(cn_max, cn);
                vn_max = std::max(vn_max, vn);
                idx_max = std::max(idx_max, idx);
            }
            const uint32_t windows = (uint32_t)((l.warps + 3) / 4), per_warp = 4 * (cn_max + vn_max), total = per_warp * windows;
            if (total <= 512)
            {
                uint32_t cols = 32;
                while (cols < total) cols <<= 1;
                c.tm = true;
                c.tm_alloc_cols = cols; c.tm_cols_per_warp = per_warp; c.tm_vn_off = 4 * cn_max;
                // Fixed iterations run the lock-step kernel when the gather addresses fit the mirror's allocation (the shape, the
                // occupancy and the TMEM a CTA holds stay as they are) and the descriptors fit K4Params::ls_seg; otherwise the
                // early-termination kernel runs them with early termination off.
                if ((per_warp + idx_max) * windows <= cols && (size_t)l.warps * (size_t)(l.cn_max_segs + l.vn_max_segs) <= (size_t)K4_LS_SEGS)
                {
                    c.lockstep = true;
                    c.tm_idx_off = per_warp;
                    c.tm_cols_per_warp = per_warp + idx_max;
                }
            }
        }
        c.idx16 = l.isz == 2;
        const bool pair = c.idx16 && tuning.idx16 == 0; // the automatic two-CTAs-per-SM shape of layout_for
        // the 16-bit tables only exist for the TMEM-mirror kernels; the pair needs both CTAs' TMEM windows at once
        if (c.idx16 && (!c.tm || (pair && c.tm_alloc_cols > 256)))
        {
            if (pair)
            {
                if (force_pair_ == 1) throw std::runtime_error("the two-CTAs-per-SM shape does not fit");
                pair_tuned_[std::make_pair(precision, alg)] = 0;
                return choose(precision, alg, n_frames);
            }
            const int saved = tuning.idx16; // asked for by the caller: redo the choice with 32-bit entries
            tuning.idx16 = 1;
            try
            {
                const Config c32 = choose(precision, alg, n_frames);
                tuning.idx16 = saved;
                return c32;
            }
            catch (...)
            {
                tuning.idx16 = saved;
                throw;
            }
        }
        int ctas = tuning.ctas;
        if (ctas <= 0)
        { // persistent grid: every SM gets as many CTAs as the runtime keeps resident
            auto key = std::make_tuple(precision, alg, c.residency * 8 + (c.tm ? 1 : 0) + (c.wide ? 2 : 0) + (c.idx16 ? 4 : 0), c.lanes, c.threads, c.smem_bytes);
            auto it = occupancy_.find(key);
            if (it == occupancy_.end())
            {
                int n = 0;
                CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, tile_fn(c, true), c.threads, c.smem_bytes));
                it = occupancy_.emplace(key, n).first;
            }
            if (it->second < 1) throw std::runtime_error("tile kernel does not fit on this device with the current tuning");
            int per_sm = it->second;
            // every resident CTA of a TM kernel holds tm_alloc_cols of the SM's 512 TMEM columns: do not launch more
            // CTAs per SM than can hold their allocation at the same time (the others would wait inside tcgen05.alloc)
            if (std::getenv("LDPC_B200_DEBUG"))
                fprintf(stderr, "[choose] lanes %d threads %d smem %zu tm %d cols %u idx16 %d occupancy %d\n", c.lanes, c.threads, c.smem_bytes, (int)c.tm,
                        c.tm_alloc_cols, (int)c.idx16, per_sm);
            if (c.tm) per_sm = std::max(1, std::min(per_sm, (int)(512u / c.tm_alloc_cols)));
            // the occupancy calculator answers 1 for the pair although two CTAs are resident (measured: 296 CTAs run at
            // 1.47 x the rate of 148); the shape is only ever chosen after it won the timed trial on this device
            if (pair) per_sm = 2;
            ctas = sm_count_ * per_sm;
        }
        c.ctas = clamp_grid(ctas, (n_frames + c.fpc - 1) / c.fpc);
        return c;
    }

    const void *Engine::tile_fn(const Config &c, bool et)
    {
        const bool smem = c.residency == LDPC_B200_SMEM;
        const void *fn = tile_kernel(c.precision == LDPC_B200_F32, c.alg, c.lanes, smem, c.tm, et || !c.lockstep, c.wide, c.idx16);
        set_smem_attributes(fn, TILE_SMEM_OPTIN, smem);
        return fn;
    }

    void Engine::set_smem_attributes(const void *fn, int smem_optin, bool max_shared)
    {
        if (attrs_set_.count(fn)) return;
        CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin));
        // all of the L1/shared array as shared memory: the shared-memory kernels keep their working set there (two CTAs per
        // SM need it); the global-residency kernels keep the default split, they live off the L1 cache
        if (max_shared) cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        attrs_set_.insert(fn);
    }

    void Engine::note_launch(int fpc, int threads, int ctas, int residency, int precision, size_t smem_bytes)
    {
        stats.launches += 1;
        stats.frames_per_cta = fpc; stats.threads_per_cta = threads; stats.ctas = ctas;
        stats.residency = residency; stats.precision = precision; stats.smem_bytes = smem_bytes;
    }

    void Engine::account(double ms, uint64_t frames, uint64_t executed_iterations)
    {
        stats.device_ms += ms;
        stats.frames += frames;
        stats.edge_iterations += executed_iterations * (uint64_t)H.nnz;
    }

    DeviceSegLayout &Engine::device_seg_layout(int lanes, int threads, int isz)
    {
        auto key = std::make_tuple(lanes, threads, isz);
        auto it = dev_seg_layouts_.find(key);
        if (it != dev_seg_layouts_.end()) return *it->second;
        const SegLayout &l = get_seg_layout(lanes, threads, isz);
        auto d = std::make_unique<DeviceSegLayout>();
        d->host = &l;
        d->cn_seg = upload(l.cn_seg);
        d->vn_seg = upload(l.vn_seg);
        d->var_pos = upload(l.var_pos);
        d->cn_idx = upload(l.cn_idx);
        d->vn_idx = upload(l.vn_idx);
        std::vector<int32_t> tx, pu, sh;
        for (int v : H.bit_pos) tx.push_back((int32_t)l.var_pos[v]);
        for (int v : H.puncture) if (v >= 0 && v < H.nc) pu.push_back((int32_t)l.var_pos[v]);
        for (int v : H.shorten) if (v >= 0 && v < H.nc) sh.push_back((int32_t)l.var_pos[v]);
        d->tx_pos = upload(tx);
        d->punct_pos = upload(pu);
        d->short_pos = upload(sh);
        return *dev_seg_layouts_.emplace(key, std::move(d)).first->second;
    }

    const TileLayout &Engine::get_layout(int fpc, int threads)
    {
        auto key = std::make_pair(fpc, threads);
        auto it = layouts_.find(key);
        if (it == layouts_.end())
        {
            auto l = std::make_unique<TileLayout>();
            l->build(H, fpc, threads);
            it = layouts_.emplace(key, std::move(l)).first;
        }
        return *it->second;
    }

    DeviceLayout &Engine::device_layout(int fpc, int threads, bool idx16)
    {
        auto key = std::make_tuple(fpc, threads, idx16);
        auto it = dev_layouts_.find(key);
        if (it != dev_layouts_.end()) return *it->second;
        const TileLayout &l = *layouts_.at(std::make_pair(fpc, threads));
        auto d = std::make_unique<DeviceLayout>();
        d->host = &l;
        d->cn_desc = upload(l.cn_desc);
        d->vn_desc = upload(l.vn_desc);
        if (idx16)
        {
            d->cn_col = upload_idx<uint16_t>(l.cn_col);
            d->vn_slot = upload_idx<uint16_t>(l.vn_slot);
            d->vn_id = upload_idx<uint16_t>(l.vn_id);
        }
        else
        {
            d->cn_col = upload_idx<uint32_t>(l.cn_col);
            d->vn_slot = upload_idx<uint32_t>(l.vn_slot);
            d->vn_id = upload_idx<uint32_t>(l.vn_id);
        }
        return *dev_layouts_.emplace(key, std::move(d)).first->second;
    }

    // The per-CTA state block (global residency, byte-wise erasure kernel) is ONE allocation per context: every launch that
    // uses it first waits for the previous user (an event recorded after that launch), whatever streams the two run on, so
    // overlapping launches of one context serialise instead of overwriting each other's messages.
    void Engine::ensure_state(size_t bytes, cudaStream_t s)
    {
        grow(state_, bytes);
        if (!ev_state_) ev_state_ = make_event(cudaEventDisableTiming);
        else if (state_used_) CUDA_OK(cudaStreamWaitEvent(s, ev_state_.get(), 0));
    }

    void Engine::release_state(cudaStream_t s)
    {
        CUDA_OK(cudaEventRecord(ev_state_.get(), s));
        state_used_ = true;
    }

    // Shared-memory streaming probe: every CTA (1024 threads, one per SM) reads a 128 KB window with
    // conflict-free LDS.128 (each warp 512 contiguous bytes per instruction), 8 loads in flight per thread.
    // Gives the sustained shared-memory read bandwidth of this device under load — the roofline that applies
    // to the shared-memory-resident decode kernel.
    __global__ void __launch_bounds__(1024, 1) smem_probe_kernel(int iters, uint32_t stride, const uint32_t *__restrict__ offs, uint32_t *sink)
    {
        extern __shared__ __align__(16) unsigned char probe_smem[];
        const uint32_t base = (uint32_t)__cvta_generic_to_shared(probe_smem) + threadIdx.x * 16u;
        for (int i = threadIdx.x; i < 8 * 16384 / 4; i += blockDim.x) reinterpret_cast<uint32_t *>(probe_smem)[i] = i;
        uint32_t o[8]; // run-time block offsets (u * 16 KB): keeps the address stream opaque to the compiler
#pragma unroll
        for (int u = 0; u < 8; ++u) o[u] = offs[u];
        __syncthreads();
        uint32_t acc = 0, off = 0;
        for (int i = 0; i < iters; ++i)
        {
            uint32_t v[8][4];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[u][0]), "=r"(v[u][1]), "=r"(v[u][2]), "=r"(v[u][3]) : "r"(base + ((off + o[u]) & 0x1FFFFu)) : "memory");
#pragma unroll
            for (int u = 0; u < 8; ++u) acc += v[u][0] ^ v[u][1] ^ v[u][2] ^ v[u][3];
            off += stride;
        }
        sink[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    }

    double Engine::smem_probe()
    {
        ensure_cuda();
        const int iters = 4096, threads = 1024, smem = 8 * 16384;
        CUDA_OK(cudaFuncSetAttribute(smem_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        const DevPtr<uint32_t> sink = device_alloc<uint32_t>((size_t)sm_count_ * threads);
        std::vector<uint32_t> h(8);
        for (int u = 0; u < 8; ++u) h[u] = (uint32_t)u * 16384u;
        const DevPtr<uint32_t> offs = upload(h);
        cudaStream_t s = stream_.get();
        double best = 0;
        for (int rep = 0; rep < 4; ++rep)
        {
            const float ms = time_ms(s, [&] { smem_probe_kernel<<<sm_count_, threads, smem, s>>>(iters, 16384u, offs.get(), sink.get()); });
            const double gbs = (double)sm_count_ * threads * 16.0 * 8.0 * iters / (ms * 1e-3) / 1e9;
            if (rep > 0) best = std::max(best, gbs);
        }
        return best;
    }

    // FP64 pipe probe: every SM runs 1024 threads of independent DFMA chains (8 per thread).  Gives the sustained FP64
    // instruction rate of this device — the roofline of the fp64 sum-product kernel, which is bound by that pipe.
    __global__ void __launch_bounds__(1024, 1) fp64_probe_kernel(int iters, double a, double b, double *sink)
    {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (double)(threadIdx.x + u) * 1e-3;
        for (int i = 0; i < iters; ++i)
        {
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = __fma_rn(v[u], a, b);
        }
        double acc = 0;
#pragma unroll
        for (int u = 0; u < 8; ++u) acc += v[u];
        sink[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    }

    double Engine::fp64_probe()
    {
        ensure_cuda();
        const int iters = 8192, threads = 1024;
        const DevPtr<double> sink = device_alloc<double>((size_t)sm_count_ * threads);
        cudaStream_t s = stream_.get();
        double best = 0;
        for (int rep = 0; rep < 4; ++rep)
        {
            const float ms = time_ms(s, [&] { fp64_probe_kernel<<<sm_count_, threads, 0, s>>>(iters, 0.999999, 1e-9, sink.get()); });
            const double ginst = (double)sm_count_ * threads * 8.0 * iters / (ms * 1e-3) / 1e9; // thread-level DFMA per second / 1e9
            if (rep > 0) best = std::max(best, ginst);
        }
        return best;
    }

    int Engine::channel_kind(const std::string &name) const
    {
        if (name == "AWGN") return SRC_AWGN;
        if (name == "BSC") return SRC_BSC;
        if (name == "BEC") return SRC_BEC;
        if (name == "RAYLEIGH")
        {
            if (ask_M > 2) throw std::runtime_error("the RAYLEIGH channel is BPSK only: set the modulation back to M = 2");
            return SRC_RAYLEIGH;
        }
        throw std::runtime_error("No channel selected."); // message of src/sim/ldpcsim.cpp:72
    }

    void Engine::launch(const decoder_param &dp, const FrameSource &src, const FrameSink &sink, uint64_t n_frames, void *stream, bool may_block)
    {
        if (n_frames == 0) return;
        ensure_cuda();
        cudaStream_t s = stream ? (cudaStream_t)stream : stream_.get();
        if (dp.iterations == 0) throw std::runtime_error("iterations must be >= 1");
        if (quantised())
        { // the fixed-point decoder is layered min-sum on BPSK frames with fp64 LLRs: anything else is an error, not a fallback
            if (tuning.schedule != LDPC_B200_LAYERED) throw std::runtime_error("quantised decoding runs on the layered schedule only (tuning.schedule = LDPC_B200_LAYERED)");
            if (src.kind == SRC_BEC || src.d_bec_in) throw std::runtime_error("quantised decoding does not apply to the BEC");
            if (alg_of(dp) != ALG_MS) throw std::runtime_error("quantised decoding is min-sum only (decoder type BP_MS)");
            if (src.kind == SRC_AWGN && ask_M > 2) throw std::runtime_error("quantised decoding is BPSK only: set the modulation back to M = 2");
            if (src.d_llr_f32 || src.d_llr_i8 || sink.d_hard_bits)
                throw std::runtime_error("quantised decoding takes fp64 LLRs and byte decisions: the narrow encodings are not supported");
        }

        if (src.kind == SRC_BEC || src.d_bec_in)
        {
            launch_bec(dp, src, sink, n_frames, s);
            return;
        }

        if (tuning.schedule == LDPC_B200_LAYERED)
        {
            launch_layered(dp, src, sink, n_frames, s);
            return;
        }
        const int alg = alg_of(dp);
        // the one-off shape trials time kernels and wait for them: only on the blocking entry points.  The asynchronous ones
        // (caller stream, possibly under graph capture) use the cached outcome or the default shape.
        if (may_block) maybe_autotune(alg, dp, n_frames, s);
        const Config c = choose(tuning.precision, alg, n_frames);
        DeviceSegLayout &dl = device_seg_layout(c.lanes, c.threads, c.idx16 ? 2 : 4);
        const SegLayout &l = *dl.host;

        K4Params kp{};
        kp.cn_seg = dl.cn_seg.get(); kp.vn_seg = dl.vn_seg.get();
        kp.cn_idx = dl.cn_idx.get(); kp.vn_idx = dl.vn_idx.get(); kp.var_pos = dl.var_pos.get();
        kp.cn_idx_bytes = (uint32_t)l.cn_idx.size(); kp.vn_idx_bytes = (uint32_t)l.vn_idx.size();
        kp.cn_max_segs = l.cn_max_segs; kp.vn_max_segs = l.vn_max_segs;
        kp.tx_pos = dl.tx_pos.get(); kp.punct_pos = dl.punct_pos.get(); kp.short_pos = dl.short_pos.get();
        kp.n_slots = l.n_slots; kp.n_pos = l.n_pos;
        kp.nc = H.nc; kp.nct = H.nct();
        kp.n_punct = 0; kp.n_short = 0;
        for (int v : H.puncture) if (v >= 0 && v < H.nc) ++kp.n_punct;
        for (int v : H.shorten) if (v >= 0 && v < H.nc) ++kp.n_short;
        kp.max_iter = (int)dp.iterations;
        kp.early_term = dp.earlyTerm ? 1 : 0;
        kp.kind = (src.kind == SRC_AWGN && ask_M > 2) ? SRC_ASK : src.kind;
        if (kp.kind == SRC_ASK) ask_fill(&kp.ask);
        kp.coherence = fading_L;
        kp.llr_in = src.d_llr; kp.llr_in_f32 = src.d_llr_f32; kp.llr_in_i8 = src.d_llr_i8; kp.i8_scale = src.i8_scale;
        const ChannelConsts cc = channel_consts(src.kind, src.x);
        kp.sigma2 = cc.sigma2; kp.sigma = cc.sigma; kp.llr_scale = cc.llr_scale; kp.delta = cc.delta; kp.thr = cc.thr;
        kp.seed = src.seed; kp.point = src.point; kp.frame0 = src.frame0; kp.n_frames = n_frames;
        kp.llr_out = sink.d_llr_out; kp.hard_out = sink.d_hard; kp.iters_out = sink.d_iters;
        kp.hard_bits = sink.d_hard_bits; kp.hard_words = sink.hard_words;
        kp.counters = sink.d_counters ? sink.d_counters : d_counters_.get();
        kp.err_log = sink.d_err_log; kp.err_count = sink.d_err_count; kp.err_cap = sink.err_cap;
        if (c.residency == LDPC_B200_GLOBAL)
        {
            kp.state_stride = ((16 * (size_t)c.lanes * ((size_t)l.n_slots + 2 * (size_t)l.n_pos)) + 255) & ~(size_t)255;
            ensure_state(kp.state_stride * c.ctas, s);
            kp.state = state_.p.get();
        }
        kp.tm_alloc_cols = c.tm_alloc_cols; kp.tm_cols_per_warp = c.tm_cols_per_warp; kp.tm_vn_off = c.tm_vn_off;
        if (c.lockstep)
        { // the segment descriptors travel in the parameters: check lists, then variable lists (tile4.cuh K4Params::ls_seg)
            kp.tm_idx_off = c.tm_idx_off;
            std::copy(l.cn_seg.begin(), l.cn_seg.end(), kp.ls_seg);
            std::copy(l.vn_seg.begin(), l.vn_seg.end(), kp.ls_seg + l.cn_seg.size());
            for (int w = 0; w < l.warps; ++w)
            { // where the warp's variable-side addresses start: after its check-side ones
                uint32_t cols = 0;
                for (int sgi = 0; sgi < l.cn_max_segs; ++sgi)
                {
                    const uint32_t d = l.cn_seg[4 * ((size_t)w * l.cn_max_segs + sgi)];
                    if (!d) break;
                    cols += (uint32_t)ls_idx_cols(true, (int)(d & 0xFFu)) * (d >> 16);
                }
                kp.ls_seg[l.cn_seg.size() + 4 * (size_t)w * l.vn_max_segs + 3] = cols;
            }
        }
        // transmitted codewords: random information words through G when a generator matrix is loaded (the reference's -G,
        // src/sim/ldpcsim.cpp:162-165); decoding caller-supplied LLRs has no transmitted word
        kp.tx_var = d_bit_pos_.get();
        if (has_gen && !tuning.zero_codeword && src.kind != SRC_LLR && kp.kind != SRC_ASK)
        {
            kp.g_col_ptr = d_g_col_ptr_.get(); kp.g_row = d_g_row_.get();
            kp.g_rows = G.mc; kp.g_cols = G.nc; kp.u_words = (G.mc + 31) / 32;
        }
        if (std::getenv("LDPC_B200_DEBUG"))
            fprintf(stderr, "[launch] tile kernel: %s\n", kp.early_term ? "early termination" : c.lockstep ? "lock-step" : c.tm ? "half-iteration, TMEM mirror" : "half-iteration");
        launch_kernel(tile_fn(c, kp.early_term != 0), c.ctas, c.threads, c.smem_bytes, s, kp, "tile kernel");
        if (c.residency == LDPC_B200_GLOBAL) release_state(s);
        note_launch(c.fpc, c.threads, c.ctas, c.residency, c.precision, c.smem_bytes);
    }

    // Global residency has no single best tile shape: quasi-cyclic codes whose neighbouring checks gather neighbouring
    // variables like narrow records and many CTAs, codes with scattered gathers like wide records (whole 64-byte
    // sectors per gather).  One-off trial of a few (lanes, threads) shapes on synthetic AWGN frames, fixed iterations;
    // the winner is cached per (precision, algorithm) and used whenever the caller pins nothing.
    // One-off tile-shape trials, run before the first large job of a (precision, algorithm) when the caller pinned nothing:
    // global residency -> autotune_global, shared-memory residency -> autotune_pair.  `n_frames` is the size of the whole
    // job (a batch decode passes its total, not the size of one pipeline piece).
    std::string Engine::tune_cache_file()
    {
        std::string dir;
        if (const char *e = std::getenv("LDPC_B200_TUNE_CACHE"))
        {
            dir = e;
            if (dir.empty() || dir == "off" || dir == "0") return "";
        }
        else if (const char *h = std::getenv("HOME")) dir = std::string(h) + "/.cache/libldpc_b200";
        else return "";
        // FNV-1a over the edge list, the header lists and the device name: the trials depend on nothing else
        uint64_t hsh = 1469598103934665603ull;
        auto mix = [&](uint64_t v) { for (int b = 0; b < 8; ++b) { hsh ^= (v >> (8 * b)) & 0xFF; hsh *= 1099511628211ull; } };
        mix((uint64_t)H.nc); mix((uint64_t)H.mc); mix((uint64_t)H.nnz);
        for (int e = 0; e < H.nnz; ++e) mix(((uint64_t)H.e_row[e] << 32) | (uint32_t)H.e_col[e]);
        for (int v : H.puncture) mix((uint64_t)v + 1);
        for (int v : H.shorten) mix((uint64_t)v + (1ull << 40));
        for (char ch : device_name_) mix((uint64_t)(unsigned char)ch);
        mix((uint64_t)B200_TILE_MAX_THREADS);
        char name[64];
        snprintf(name, sizeof(name), "/tune_%016llx_v2.txt", (unsigned long long)hsh);
        return dir + name;
    }

    void Engine::tune_cache_load()
    {
        if (tune_cache_loaded_) return;
        tune_cache_loaded_ = true;
        const std::string f = tune_cache_file();
        if (f.empty()) return;
        FILE *fp = fopen(f.c_str(), "r");
        if (!fp) return;
        char kind;
        int prec, alg, a, b, c;
        while (fscanf(fp, " %c %d %d %d %d %d", &kind, &prec, &alg, &a, &b, &c) == 6)
        {
            if (kind == 'g') tuned_[std::make_pair(prec, alg)] = std::make_tuple(a, b, c);
            else if (kind == 'p') pair_tuned_[std::make_pair(prec, alg)] = a;
        }
        fclose(fp);
    }

    void Engine::tune_cache_store()
    {
        const std::string f = tune_cache_file();
        if (f.empty()) return;
        const std::string dir = f.substr(0, f.rfind('/'));
        std::string cmd_dir;
        for (size_t i = 1; i <= dir.size(); ++i) // mkdir -p
            if (i == dir.size() || dir[i] == '/') mkdir(dir.substr(0, i).c_str(), 0755);
        const std::string tmp = f + ".tmp" + std::to_string((long)getpid());
        FILE *fp = fopen(tmp.c_str(), "w");
        if (!fp) return;
        for (const auto &kv : tuned_) fprintf(fp, "g %d %d %d %d %d\n", kv.first.first, kv.first.second, std::get<0>(kv.second), std::get<1>(kv.second), std::get<2>(kv.second));
        for (const auto &kv : pair_tuned_) fprintf(fp, "p %d %d %d 0 0\n", kv.first.first, kv.first.second, kv.second);
        fclose(fp);
        rename(tmp.c_str(), f.c_str());
    }

    void Engine::maybe_autotune(int alg, const decoder_param &dp, uint64_t n_frames, cudaStream_t s)
    {
        // The trials time launch(), which serves the layered schedule (and the fixed-point decoder) with the layered kernel: its
        // outcome would be stored, and cached on disk, as the flooding kernel's shape.  The layered kernel has no shape trial.
        if (quantised() || tuning.schedule != LDPC_B200_FLOODING) return;
        tune_cache_load();
        const auto key = std::make_pair(tuning.precision, alg);
        if (in_autotune_ || n_frames < 20000 || tuning.frames_per_cta > 0 || tuning.threads_per_cta > 0 || tuned_.count(key) || pair_tuned_.count(key)) return;
        int res = 0;
        size_t sb = 0;
        layout_for(tuning.precision, alg, &res, &sb);
        if (res == LDPC_B200_GLOBAL) { autotune_global(alg, dp, s); tune_cache_store(); }
        else if (tuning.idx16 == 0 && tuning.tmem == 0 && tuning.ctas <= 0)
        { // LDPC_B200_PAIR=0/1 presets the outcome (runs under a profiler, whose serialised replays distort the trial)
            const char *preset = std::getenv("LDPC_B200_PAIR");
            if (preset && (preset[0] == '0' || preset[0] == '1')) pair_tuned_[key] = preset[0] == '1';
            else { autotune_pair(alg, dp, s); tune_cache_store(); }
        }
    }

    // A shape trial pins the tuning and the trial switches, and its launches count in the stats: all of it is put back however
    // the trial ends.
    struct Engine::TrialGuard
    {
        Engine &e;
        const ldpc_b200_tuning saved_tuning;
        const ldpc_b200_stats saved_stats;
        explicit TrialGuard(Engine &eng) : e(eng), saved_tuning(eng.tuning), saved_stats(eng.stats) { e.in_autotune_ = true; }
        ~TrialGuard()
        {
            e.tuning = saved_tuning;
            e.stats = saved_stats;
            e.in_autotune_ = false;
            e.force_wide_ = e.force_pair_ = -1;
        }
    };

    float Engine::time_ms(cudaStream_t s, const std::function<void()> &work)
    {
        CUDA_OK(cudaEventRecord(ev0_.get(), s));
        work();
        CUDA_OK(cudaEventRecord(ev1_.get(), s));
        CUDA_OK(cudaEventSynchronize(ev1_.get()));
        float ms = 0;
        CUDA_OK(cudaEventElapsedTime(&ms, ev0_.get(), ev1_.get()));
        return ms;
    }

    // A warm-up launch of frames / 4 (tables, attributes, state block), then `frames` timed.  `eligible`, asked after the
    // warm-up, can still turn the shape down.
    double Engine::trial_rate(const decoder_param &dp, double snr, unsigned long long *d_cnt, uint64_t frames, cudaStream_t s,
                              const std::function<bool()> &eligible)
    {
        FrameSource src;
        src.kind = SRC_AWGN;
        src.x = snr;
        src.seed = 0x5eed;
        FrameSink sink;
        sink.d_counters = d_cnt;
        try
        {
            launch(dp, src, sink, frames / 4, s, true);
            if (eligible && !eligible()) return 0;
            return (double)frames / time_ms(s, [&] { launch(dp, src, sink, frames, s, true); });
        }
        catch (const std::exception &)
        { // a shape that does not fit is simply not a candidate
            cudaGetLastError();
            return 0;
        }
    }

    void Engine::autotune_global(int alg, const decoder_param &dp, cudaStream_t s)
    {
        const auto key = std::make_pair(tuning.precision, alg);
        const TrialGuard guard(*this);
        const DevPtr<unsigned long long> d_cnt = device_alloc<unsigned long long>(8);
        CUDA_OK(cudaMemsetAsync(d_cnt.get(), 0, 8 * sizeof(unsigned long long), s));
        const int vec = tuning.precision == LDPC_B200_F32 ? 4 : 2;
        decoder_param tdp = dp;
        tdp.earlyTerm = false;
        tdp.iterations = std::min<uint32_t>(dp.iterations, 20); // enough iterations that decoding, not frame generation, dominates
        const uint64_t frames = (uint64_t)sm_count_ * 2 * 16;   // whole waves for every shape (the widest holds 16 frames per CTA)
        double best = 0;
        std::tuple<int, int, int> best_cfg(1, std::min(512, B200_TILE_MAX_THREADS), 0);
        const int cand[9][3] = {{1, 512, 0}, {2, 512, 0}, {4, 512, 0}, {1, 512, 1}, {2, 512, 1}, {4, 512, 1}, {1, 256, 0}, {2, 256, 0}, {4, 256, 0}};
        for (const auto &cd : cand)
        {
            if (cd[2] && alg != ALG_MS) continue; // the wide build only differs for min-sum
            force_wide_ = cd[2];
            tuning.residency = LDPC_B200_GLOBAL;
            tuning.frames_per_cta = cd[0] * vec;
            tuning.threads_per_cta = cd[1];
            tuning.zero_codeword = 1;
            const double rate = trial_rate(tdp, 3.0, d_cnt.get(), frames, s);
            if (rate > best) { best = rate; best_cfg = std::make_tuple(cd[0], cd[1], cd[2]); }
        }
        tuned_[key] = best_cfg;
    }

    // Shared-memory residency, nothing pinned by the caller: one CTA per SM (two lanes, 32-bit index tables) against two
    // CTAs per SM (one lane, half the threads, 16-bit tables) on the same frames, timed once per (precision, algorithm).
    void Engine::autotune_pair(int alg, const decoder_param &dp, cudaStream_t s)
    {
        const auto key = std::make_pair(tuning.precision, alg);
        const TrialGuard guard(*this);
        const DevPtr<unsigned long long> d_cnt = device_alloc<unsigned long long>(8);
        CUDA_OK(cudaMemsetAsync(d_cnt.get(), 0, 8 * sizeof(unsigned long long), s));
        decoder_param tdp = dp;
        tdp.iterations = std::min<uint32_t>(dp.iterations, 20);
        tuning.zero_codeword = 1;
        const uint64_t frames = (uint64_t)sm_count_ * 2 * 64; // whole waves for both shapes
        const int pair_threads = tile_thread_cap(tuning.precision != LDPC_B200_F32, alg, true) / 2;
        double rate[2] = {0, 0};
        for (int cand = 0; cand < 2; ++cand)
        {
            force_pair_ = cand;
            // not eligible: the one-CTA shape ran
            rate[cand] = trial_rate(tdp, -4.0, d_cnt.get(), frames, s, [&] { return cand == 0 || stats.threads_per_cta == pair_threads; });
        }
        if (std::getenv("LDPC_B200_DEBUG")) fprintf(stderr, "[autotune_pair] one CTA/SM %.1f frames/ms, two CTAs/SM %.1f frames/ms\n", rate[0], rate[1]);
        pair_tuned_[key] = rate[1] > 1.01 * rate[0] ? 1 : 0;
    }

    void Engine::set_modulation(int M, const int *labels, const int *bit_mapper)
    {
        if (M == 2) { ask_M = 2; return; }
        int bits = 0;
        while ((1 << bits) < M) ++bits;
        if (M < 4 || M > 256 || (1 << bits) != M) throw std::runtime_error("modulation: M must be 2 (BPSK) or a power of two 4 ... 256");
        if (H.nct() % bits) throw std::runtime_error("modulation: the number of transmitted bits is not a multiple of log2(M)"); // gpu/sim/ldpcsim.cpp:115-118
        const int n_sym = H.nct() / bits;
        std::vector<int32_t> lab(M), rev(M, -1), bm((size_t)bits * n_sym);
        for (int j = 0; j < M; ++j) lab[j] = labels ? labels[j] : (j ^ (j >> 1));
        for (int j = 0; j < M; ++j)
        {
            if (lab[j] < 0 || lab[j] >= M || rev[lab[j]] >= 0) throw std::runtime_error("modulation: labels must be a permutation of 0 ... M-1");
            rev[lab[j]] = j;
        }
        std::vector<char> used(H.nc, 0);
        for (int k = 0; k < bits; ++k)
            for (int i = 0; i < n_sym; ++i)
            {
                const int v = bit_mapper ? bit_mapper[(size_t)k * n_sym + i] : H.bit_pos[(size_t)i * bits + k];
                if (v < 0 || v >= H.nc || used[v]++) throw std::runtime_error("modulation: the bit mapper must name every transmitted variable once");
                bm[(size_t)k * n_sym + i] = v;
            }
        for (int v : H.bit_pos) if (!used[v]) throw std::runtime_error("modulation: the bit mapper must name every transmitted variable once");
        std::vector<double> X(M);
        double m = 0;
        for (int j = 0; j < M; ++j) { X[j] = (double)-M + 1 + 2 * j; m += X[j] * X[j] * (1.0 / M); } // gpu/sim/ldpcsim.cpp:10-14
        for (int j = 0; j < M; ++j) X[j] = X[j] / std::sqrt(m);
        ask_M = M; ask_labels = lab; ask_rev = rev; ask_bm = bm; ask_X = X;
        if (cuda_ready_)
        {
            cudaSetDevice(device);
            cudaDeviceSynchronize();
            d_ask_X_.reset(); d_ask_label_.reset(); d_ask_rev_.reset(); d_ask_bm_.reset();
        }
    }

    void Engine::ask_fill(void *out)
    {
        if (!d_ask_bm_) // uploaded last: present means all four are
        {
            d_ask_X_ = upload(ask_X); d_ask_label_ = upload(ask_labels); d_ask_rev_ = upload(ask_rev); d_ask_bm_ = upload(ask_bm);
        }
        AskParams &a = *static_cast<AskParams *>(out);
        a.M = ask_M;
        a.bits = 0;
        while ((1 << a.bits) < ask_M) ++a.bits;
        a.n_sym = H.nct() / a.bits;
        a.X = d_ask_X_.get(); a.label = d_ask_label_.get(); a.rev = d_ask_rev_.get(); a.bm = d_ask_bm_.get();
    }

    void Engine::set_layers(std::vector<std::vector<int>> layers)
    {
        if (!layers.empty()) validate_layers(H, layers);
        layers_ = std::move(layers);
        dev_lay_.clear();
        lay_layouts_.clear();
    }

    const std::vector<std::vector<int>> &Engine::layers()
    {
        if (layers_.empty()) layers_ = auto_layers(H);
        return layers_;
    }

    // Layered schedule (opt-in, tuning.schedule): layered.cuh.  Global residency, frames in lock step per CTA.
    void Engine::launch_layered(const decoder_param &dp, const FrameSource &src, const FrameSink &sink, uint64_t n_frames, cudaStream_t s)
    {
        if (src.d_llr_f32 || src.d_llr_i8 || sink.d_hard_bits) throw std::runtime_error("layered schedule: the narrow encodings are served by the flooding path only");
        if (src.kind == SRC_AWGN && ask_M > 2) throw std::runtime_error("layered schedule: higher-order modulation is served by the flooding path only");
        if (has_gen && !tuning.zero_codeword && src.kind != SRC_LLR)
            throw std::runtime_error("layered schedule: sweeps transmit the all-zero codeword (set tuning.zero_codeword = 1 with a generator matrix loaded)");
        const bool q = quantised();
        const int vec = q ? 8 : tuning.precision == LDPC_B200_F32 ? 4 : 2;
        int lanes = 4, threads = 0, per_sm = 0;
        const void *fn = nullptr;
        if (q) quant_shape(&lanes, &threads, &fn, &per_sm);
        else
        {
            if (tuning.frames_per_cta > 0)
            {
                if (tuning.frames_per_cta != 2 * vec && tuning.frames_per_cta != 4 * vec) throw std::runtime_error("layered schedule: frames_per_cta / vector width must be 2 or 4");
                lanes = tuning.frames_per_cta / vec;
            }
            threads = tuning.threads_per_cta > 0 ? std::min(tuning.threads_per_cta, 512) : 256;
        }
        auto key = std::make_pair(lanes, threads);
        auto it = dev_lay_.find(key);
        if (it == dev_lay_.end())
        {
            auto l = std::make_unique<LayeredLayout>();
            l->build(H, layers(), lanes, threads);
            auto d = std::make_unique<DeviceLayered>();
            d->host = l.get();
            d->seg = upload(l->seg);
            d->idx = upload(l->idx);
            lay_layouts_[key] = std::move(l);
            it = dev_lay_.emplace(key, std::move(d)).first;
        }
        const LayeredLayout &l = *it->second->host;
        LayParams lp{};
        lp.seg = it->second->seg.get(); lp.idx = it->second->idx.get();
        lp.n_layers = l.n_layers; lp.max_segs = l.max_segs; lp.n_slots = l.n_slots;
        lp.nc = H.nc; lp.nct = H.nct(); lp.n_punct = (int)H.puncture.size(); lp.n_short = (int)H.shorten.size();
        lp.tx_var = d_bit_pos_.get(); lp.punct = d_punct_.get(); lp.shorten = d_short_.get();
        lp.max_iter = (int)dp.iterations; lp.early_term = dp.earlyTerm ? 1 : 0; lp.kind = src.kind;
        lp.coherence = fading_L;
        lp.llr_in = src.d_llr;
        const ChannelConsts cc = channel_consts(src.kind, src.x);
        lp.sigma = cc.sigma; lp.llr_scale = cc.llr_scale; lp.delta = cc.delta; lp.thr = cc.thr;
        lp.ms_scale = (tuning.layered_ms_scale64 > 0 ? tuning.layered_ms_scale64 : 64) / 64.0;
        lp.seed = src.seed; lp.point = src.point; lp.frame0 = src.frame0; lp.n_frames = n_frames;
        lp.llr_out = sink.d_llr_out; lp.hard_out = sink.d_hard; lp.iters_out = sink.d_iters;
        lp.counters = sink.d_counters ? sink.d_counters : d_counters_.get();
        lp.err_log = sink.d_err_log; lp.err_count = sink.d_err_count; lp.err_cap = sink.err_cap;
        if (q)
        {
            lp.q_step = quant.step;
            lp.q_ch_max = (1 << (quant.ch_bits - 1)) - 1; lp.q_msg_max = (1 << (quant.msg_bits - 1)) - 1; lp.q_post_max = (1 << (quant.post_bits - 1)) - 1;
            lp.q_offset = quant.offset; lp.q_scale8 = quant.scale8;
        }
        const int fpc = lanes * vec;
        if (!q)
        {
            fn = layered_kernel(tuning.precision == LDPC_B200_F32, alg_of(dp), lanes);
            CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, 0));
        }
        if (per_sm < 1) throw std::runtime_error("layered kernel does not fit on this device");
        const int ctas = clamp_grid(tuning.ctas > 0 ? tuning.ctas : sm_count_ * per_sm, (n_frames + fpc - 1) / fpc);
        lp.state_stride = ((16 * (size_t)lanes * ((size_t)l.n_slots + (size_t)H.nc)) + 255) & ~(size_t)255;
        ensure_state(lp.state_stride * ctas, s);
        lp.state = state_.p.get();
        launch_kernel(fn, ctas, threads, 0, s, lp, "layered kernel");
        release_state(s);
        note_launch(fpc, threads, ctas, LDPC_B200_GLOBAL, q ? LDPC_B200_FIXED : tuning.precision, 0);
    }

    void Engine::quant_shape(int *lanes, int *threads, const void **fn, int *per_sm)
    {
        if (tuning.frames_per_cta != 0 && tuning.frames_per_cta != 16 && tuning.frames_per_cta != 32)
            throw std::runtime_error("quantised decoding: frames_per_cta must be 0, 16 or 32");
        *lanes = tuning.frames_per_cta == 16 ? 2 : 4;
        *threads = tuning.threads_per_cta > 0 ? std::min(tuning.threads_per_cta, 512) : 256;
        *fn = layered_kernel_q(*lanes);
        CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, *fn, *threads, 0));
    }

    int64_t Engine::batch_wave(const decoder_param &dp, uint64_t n_frames, cudaStream_t s)
    {
        if (quantised())
        {
            int lanes, threads, per_sm;
            const void *fn;
            quant_shape(&lanes, &threads, &fn, &per_sm);
            return (int64_t)sm_count_ * std::max(per_sm, 1) * lanes * 8;
        }
        maybe_autotune(alg_of(dp), dp, n_frames, s);
        const Config c = choose(tuning.precision, alg_of(dp), ~0ull >> 1);
        return (int64_t)c.ctas * c.fpc;
    }

    void Engine::set_quant(const ldpc_b200_quant *q)
    {
        if (!q || q->ch_bits == 0) { quant = ldpc_b200_quant{}; return; }
        if (!(q->msg_bits >= 2 && q->msg_bits <= q->post_bits && q->post_bits <= 16 && q->ch_bits >= 2 && q->ch_bits <= q->post_bits))
            throw std::runtime_error("quantisation: bit widths must satisfy 2 <= msg_bits <= post_bits <= 16 and 2 <= ch_bits <= post_bits");
        if (q->offset < 0 || q->offset >= (1 << (q->msg_bits - 1)) - 1) throw std::runtime_error("quantisation: offset must satisfy 0 <= offset < 2^(msg_bits-1) - 1");
        if (q->scale8 < 1 || q->scale8 > 8) throw std::runtime_error("quantisation: scale8 must be 1 .. 8");
        if (!(q->step > 0) || !std::isfinite(q->step)) throw std::runtime_error("quantisation: step must be a finite value > 0");
        quant = *q;
    }

    void Engine::launch_bec(const decoder_param &dp, const FrameSource &src, const FrameSink &sink, uint64_t n_frames, cudaStream_t s)
    {
        // Sweep mode (frames generated on the device, only the counters and the error log leave it): the bit-sliced kernel, 32
        // frames per word, when one word's state (bit-planes per edge and per variable) fits shared memory; the byte-wise
        // kernel below serves caller-supplied frames (decode API: per-frame outputs) and larger codes.
        const bool use_gen = has_gen && !tuning.zero_codeword && !src.d_bec_in; // random codewords u*G (src/sim/channel.cpp:177-191)
        const bool logging = sink.d_err_log != nullptr;
        const bool slice_mode = !src.d_bec_in && !sink.d_bec_out && !sink.d_hard && !sink.d_iters && H.min_cn_degree >= 2 && H.max_cn_degree <= 32 &&
                                H.max_vn_degree <= 32 * 64 && tuning.residency != LDPC_B200_GLOBAL;
        const size_t slice_limit = smem_optin_ > 2048 ? smem_optin_ - 2048 : 0;
        if (slice_mode)
        {
            if (!bs_layout_)
            {
                bs_layout_ = std::make_unique<BecSliceLayout>();
                try { bs_layout_->build(H); }
                catch (const std::exception &) { bs_layout_->n_slots = 0; } // too large / too dense: the byte-wise kernel serves it
            }
        }
        const bool gen_variant = use_gen || logging;
        const uint32_t thr = channel_consts(SRC_BEC, src.x).thr;
        const size_t n_slots = bs_layout_ ? (size_t)bs_layout_->n_slots : 0;
        const size_t group_words = gen_variant ? 2 * n_slots + 3 * (size_t)H.nc + 40 : n_slots + (size_t)H.nc + 8;
        const size_t slice_group_bytes = 4 * group_words;
        // the information words of a 32-frame group are transposed in the (not yet used) message area
        const bool scratch_ok = !use_gen || (size_t)(32 * 4 * ((G.mc + 127) / 128) + G.mc) <= n_slots;
        if (slice_mode && n_slots > 0 && slice_group_bytes <= slice_limit && scratch_ok)
        {
            if (!d_bs_row_ptr_)
            {
                std::vector<int32_t> rp(H.row_ptr.begin(), H.row_ptr.end()), cp(H.col_ptr.begin(), H.col_ptr.end());
                std::vector<uint8_t> tf(H.nc, 0);
                for (int v : H.bit_pos) tf[v] = 1;
                d_bs_row_ptr_ = upload(rp); d_bs_col_ptr_ = upload(cp);
                d_bs_row_slot_ = upload(bs_layout_->row_slot); d_bs_col_slot_ = upload(bs_layout_->col_slot);
                d_bs_tx_flag_ = upload(tf);
            }
            BecSliceParams bp{};
            bp.row_ptr = d_bs_row_ptr_.get(); bp.row_slot = d_bs_row_slot_.get(); bp.col_ptr = d_bs_col_ptr_.get(); bp.col_slot = d_bs_col_slot_.get();
            bp.tx_var = d_bit_pos_.get(); bp.punct = d_punct_.get(); bp.shorten = d_short_.get(); bp.tx_flag = d_bs_tx_flag_.get();
            bp.nc = H.nc; bp.mc = H.mc; bp.nnz = H.nnz; bp.nct = H.nct(); bp.n_slots = (int)n_slots;
            bp.n_punct = (int)H.puncture.size(); bp.n_short = (int)H.shorten.size();
            bp.max_iter = (int)dp.iterations; bp.early_term = dp.earlyTerm ? 1 : 0; bp.deg1_compat = tuning.bec_deg1_compat;
            bp.thr = thr;
            bp.seed = src.seed; bp.point = src.point; bp.frame0 = src.frame0; bp.n_frames = n_frames;
            bp.counters = sink.d_counters ? sink.d_counters : d_counters_.get();
            if (use_gen) { bp.g_col_ptr = d_g_col_ptr_.get(); bp.g_row = d_g_row_.get(); bp.g_rows = G.mc; bp.g_cols = G.nc; }
            bp.err_log = sink.d_err_log; bp.err_count = sink.d_err_count; bp.err_cap = sink.err_cap;
            const uint64_t n_words = (n_frames + 31) / 32;
            int groups = (int)std::min<size_t>(8, slice_limit / slice_group_bytes);
            groups = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)groups, n_words));
            bp.groups_per_cta = groups;
            bp.group_words = (int)group_words;
            const int ctas = clamp_grid(tuning.ctas > 0 ? tuning.ctas : sm_count_, (n_words + groups - 1) / groups);
            const void *fn = gen_variant ? (const void *)bec_slice_kernel<true> : (const void *)bec_slice_kernel<false>;
            set_smem_attributes(fn, (int)slice_limit, false);
            launch_kernel(fn, ctas, groups * BEC_TPG, groups * slice_group_bytes, s, bp, "bit-sliced erasure kernel");
            note_launch(32 * groups, groups * BEC_TPG, ctas, LDPC_B200_SMEM, -1, groups * slice_group_bytes);
            return;
        }
        const int threads = 1024;
        const TileLayout &l = get_layout(32, threads);
        const bool idx16 = std::max({l.n_slots, l.n_vslots, H.nc}) <= 65535;
        DeviceLayout &dl = device_layout(32, threads, idx16);
        BecParams bp{};
        bp.cn_desc = dl.cn_desc.get(); bp.vn_desc = dl.vn_desc.get(); bp.cn_col = dl.cn_col.get(); bp.vn_slot = dl.vn_slot.get(); bp.vn_id = dl.vn_id.get();
        bp.bit_pos = d_bit_pos_.get(); bp.punct = d_punct_.get(); bp.shorten = d_short_.get();
        bp.cn_rounds = l.cn_rounds; bp.vn_rounds = l.vn_rounds; bp.n_slots = l.n_slots;
        bp.nc = H.nc; bp.nct = H.nct(); bp.n_punct = (int)H.puncture.size(); bp.n_short = (int)H.shorten.size();
        bp.max_iter = (int)dp.iterations; bp.early_term = dp.earlyTerm ? 1 : 0; bp.deg1_compat = tuning.bec_deg1_compat;
        bp.kind = src.d_bec_in ? SRC_LLR : SRC_BEC;
        bp.in = src.d_bec_in; bp.cw = src.d_bec_cw;
        bp.thr = thr;
        bp.seed = src.seed; bp.point = src.point; bp.frame0 = src.frame0; bp.n_frames = n_frames;
        bp.out = sink.d_bec_out; bp.hard = sink.d_hard; bp.iters_out = sink.d_iters;
        bp.counters = sink.d_counters ? sink.d_counters : d_counters_.get();
        if (use_gen) { bp.g_col_ptr = d_g_col_ptr_.get(); bp.g_row = d_g_row_.get(); bp.g_rows = G.mc; bp.g_cols = G.nc; }
        bp.err_log = sink.d_err_log; bp.err_count = sink.d_err_count; bp.err_cap = sink.err_cap;
        const int ctas = clamp_grid(tuning.ctas > 0 ? tuning.ctas : sm_count_, (n_frames + 31) / 32);
        bp.state_stride = (((2 * (size_t)l.n_slots + 3 * (size_t)H.nc) * 32) + 255) & ~(size_t)255;
        ensure_state(bp.state_stride * ctas, s);
        bp.state = state_.p.get();
        launch_kernel(idx16 ? (const void *)bec_kernel<uint16_t> : (const void *)bec_kernel<uint32_t>, ctas, threads, 0, s, bp, "erasure kernel");
        release_state(s);
        note_launch(32, threads, ctas, LDPC_B200_GLOBAL, -1, 0);
    }

    // ------------------------------------------------------------------------------------------
    // blocking helpers
    // ------------------------------------------------------------------------------------------

    void Engine::sim_point_async(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point,
                                 uint64_t frame0, uint64_t n_frames, unsigned long long *d_counters, void *stream, bool may_block)
    {
        FrameSource src;
        src.kind = channel_kind(channel);
        src.x = x; src.seed = seed; src.point = point; src.frame0 = frame0;
        FrameSink sink;
        sink.d_counters = d_counters;
        launch(dp, src, sink, n_frames, stream, may_block);
    }

    // One-off shape trials of (decoder type, current precision) for a job of n_frames, on the engine stream.  Blocking.
    void Engine::prepare(const decoder_param &dp, uint64_t n_frames)
    {
        ensure_cuda();
        maybe_autotune(alg_of(dp), dp, n_frames, stream_.get());
    }

    void Engine::sim_point(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point,
                           uint64_t frame0, uint64_t n_frames, uint64_t counters[5], float *device_ms)
    {
        (void)channel_kind(channel); // argument errors first, as the reference's constructor does (ldpcsim.cpp:32-72)
        ensure_cuda();
        cudaStream_t s = stream_.get();
        CUDA_OK(cudaMemsetAsync(d_counters_.get(), 0, 8 * sizeof(unsigned long long), s));
        CUDA_OK(cudaEventRecord(ev0_.get(), s));
        sim_point_async(dp, channel, x, seed, point, frame0, n_frames, d_counters_.get(), s, true);
        CUDA_OK(cudaEventRecord(ev1_.get(), s));
        unsigned long long h[5];
        CUDA_OK(cudaMemcpyAsync(h, d_counters_.get(), sizeof(h), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaStreamSynchronize(s));
        float ms = 0;
        CUDA_OK(cudaEventElapsedTime(&ms, ev0_.get(), ev1_.get()));
        if (device_ms) *device_ms = ms;
        for (int i = 0; i < 5; ++i) counters[i] = h[i];
        account(ms, h[2], h[4]);
    }

    void Engine::round_launch(int slot, const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point, uint64_t frame0,
                              uint64_t n_frames)
    {
        (void)channel_kind(channel);
        ensure_cuda();
        cudaStream_t s = stream_.get();
        if (!ev_rdone_[slot]) // created last: present means the slot is complete
        {
            d_round_[slot] = device_alloc<unsigned long long>(8);
            unsigned long long *h = nullptr;
            CUDA_OK(cudaHostAlloc((void **)&h, 8 * sizeof(unsigned long long), cudaHostAllocDefault));
            h_round_[slot].reset(h);
            ev_round_[slot] = make_event(cudaEventDefault);
            ev_round0_[slot] = make_event(cudaEventDefault);
            ev_rdone_[slot] = make_event(cudaEventDisableTiming);
        }
        CUDA_OK(cudaMemsetAsync(d_round_[slot].get(), 0, 8 * sizeof(unsigned long long), s));
        CUDA_OK(cudaEventRecord(ev_round0_[slot].get(), s));
        sim_point_async(dp, channel, x, seed, point, frame0, n_frames, d_round_[slot].get(), s, true);
        CUDA_OK(cudaEventRecord(ev_round_[slot].get(), s));
        CUDA_OK(cudaMemcpyAsync(h_round_[slot].get(), d_round_[slot].get(), 5 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaEventRecord(ev_rdone_[slot].get(), s));
    }

    void Engine::round_collect(int slot, uint64_t counters[5])
    {
        CUDA_OK(cudaSetDevice(device));
        CUDA_OK(cudaEventSynchronize(ev_rdone_[slot].get())); // only this round: the next one may already be running behind it
        float ms = 0;
        CUDA_OK(cudaEventElapsedTime(&ms, ev_round0_[slot].get(), ev_round_[slot].get()));
        for (int i = 0; i < 5; ++i) counters[i] = h_round_[slot].get()[i];
        account(ms, counters[2], counters[4]);
    }

    uint64_t Engine::wave_frames(const decoder_param &dp, const std::string &channel)
    {
        ensure_cuda();
        if (channel_kind(channel) == SRC_BEC) return (uint64_t)sm_count_ * 8 * 32; // bit-sliced kernel: up to 8 words of 32 frames per CTA
        if (quantised()) return (uint64_t)batch_wave(dp, 0, stream_.get());
        const Config c = choose(tuning.precision, alg_of(dp), ~0ull >> 1);
        return (uint64_t)c.ctas * c.fpc;
    }

    void Engine::sim_point_log(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point, uint64_t frame0,
                               uint64_t n_frames, uint64_t counters[5], ldpc_b200_error_record *records, int64_t capacity, int64_t *n_errors)
    {
        const int kind = channel_kind(channel);
        if (capacity < 0 || (capacity > 0 && !records)) throw std::runtime_error("bad error-log buffer");
        ensure_cuda();
        cudaStream_t s = stream_.get();
        const DevPtr<unsigned long long> d_log = device_alloc<unsigned long long>(std::max<size_t>((size_t)capacity, 1) * 2);
        const DevPtr<unsigned long long> d_cnt = device_alloc<unsigned long long>(1);
        CUDA_OK(cudaMemsetAsync(d_cnt.get(), 0, sizeof(unsigned long long), s));
        CUDA_OK(cudaMemsetAsync(d_counters_.get(), 0, 8 * sizeof(unsigned long long), s));
        FrameSource src;
        src.kind = kind;
        src.x = x; src.seed = seed; src.point = point; src.frame0 = frame0;
        FrameSink sink;
        sink.d_counters = d_counters_.get();
        sink.d_err_log = d_log.get(); sink.d_err_count = d_cnt.get(); sink.err_cap = (unsigned long long)capacity;
        launch(dp, src, sink, n_frames, s, true);
        unsigned long long h[5], n = 0;
        CUDA_OK(cudaMemcpyAsync(h, d_counters_.get(), sizeof(h), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaMemcpyAsync(&n, d_cnt.get(), sizeof(n), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaStreamSynchronize(s));
        const size_t m = (size_t)std::min<unsigned long long>(n, (unsigned long long)capacity);
        std::vector<unsigned long long> raw(2 * std::max<size_t>(m, 1));
        if (m) CUDA_OK(cudaMemcpy(raw.data(), d_log.get(), m * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < m; ++i)
        {
            records[i].frame = raw[2 * i];
            records[i].bit_errors = (uint32_t)(raw[2 * i + 1] & 0xFFFFFFFFull);
            records[i].iterations = (int32_t)(uint32_t)(raw[2 * i + 1] >> 32);
        }
        if (n_errors) *n_errors = (int64_t)n;
        for (int i = 0; i < 5; ++i) counters[i] = h[i];
        account(0, h[2], h[4]); // no device time: the launch is not timed
    }

    // Host-buffer batch decode: a double-buffered pipeline over three streams — H2D of chunk k+1, the decode
    // kernel of chunk k and D2H of chunk k-1 overlap (kernels stay on ONE stream, so the per-CTA state block of
    // global residency is never shared by two launches).  Device buffers are cached in the engine.  With pinned
    // caller buffers the copies run at full PCIe rate; pageable buffers work too (the driver stages them).
    void Engine::decode_batch_host(const decoder_param &dp, const void *llr, int llr_type, double llr_scale, int64_t n, double *llr_out, uint8_t *hard,
                                   uint32_t *hard_bits, int32_t *iters)
    {
        if (n <= 0) return;
        if (llr_type != LDPC_B200_LLR_F64 && llr_type != LDPC_B200_LLR_F32 && llr_type != LDPC_B200_LLR_I8) throw std::runtime_error("bad llr_type");
        ensure_cuda();
        cudaStream_t sk = stream_.get();
        const size_t nc = H.nc;
        const size_t esz = llr_type == LDPC_B200_LLR_F64 ? 8 : llr_type == LDPC_B200_LLR_F32 ? 4 : 1; // bytes per input LLR
        const size_t hw = (nc + 31) / 32;                                                              // words per frame of packed decisions
        // chunk = whole waves of the persistent grid (CTAs x frames per CTA), about 32 MB of input: no partly filled last wave
        // per launch, and a short pipeline fill
        int64_t chunk = std::max<int64_t>((int64_t)((32ull << 20) / (nc * esz)), 1), wave = 1;
        {
            wave = batch_wave(dp, (uint64_t)n, sk);
            chunk = std::max<int64_t>(wave, chunk / wave * wave);
        }
        chunk = std::min<int64_t>(n, chunk);
        // Piece sizes: the pipeline fills with the H2D copy of the first piece and drains with the kernel and D2H copy of the
        // last one, so both ends ramp (1, 2, 4 ... waves up to the steady chunk, and down again); the ragged remainder of
        // the batch rides in the last piece.
        std::vector<int64_t> pieces;
        {
            std::vector<int64_t> ramp;
            int64_t ramp_sum = 0;
            for (int64_t w = wave; w < chunk; w *= 2) { ramp.push_back(w); ramp_sum += w; }
            const int64_t ragged = n % wave, body = n - ragged;
            if (body >= 2 * ramp_sum + 2 * chunk)
            {
                pieces = ramp;
                for (int64_t left = body - 2 * ramp_sum; left > 0;)
                {
                    const int64_t m = std::min(chunk, left);
                    pieces.push_back(m);
                    left -= m;
                }
                for (auto it = ramp.rbegin(); it != ramp.rend(); ++it) pieces.push_back(*it);
                pieces.back() += ragged;
            }
            else
                for (int64_t left = n; left > 0;)
                {
                    int64_t m = std::min(chunk, left);
                    if (left - m > 0 && left - m < wave) m = left; // no sliver launch of its own
                    pieces.push_back(m);
                    left -= m;
                }
        }
        int64_t max_piece = 0;
        for (int64_t m : pieces) max_piece = std::max(max_piece, m);
        chunk = max_piece;
        if (!ev_out_[1]) // created last: present means all are
        {
            copy_in_ = make_stream();
            copy_out_ = make_stream();
            for (int b = 0; b < 2; ++b)
            {
                ev_in_[b] = make_event(cudaEventDisableTiming);
                ev_k_[b] = make_event(cudaEventDisableTiming);
                ev_out_[b] = make_event(cudaEventDisableTiming);
            }
        }
        // a batch that is a single piece (decode() of the six-symbol ABI: one frame per call) has nothing to overlap: copies and kernel
        // run in order on ONE stream, without the cross-stream event hand-offs (each costs microseconds of latency)
        const bool single = pieces.size() == 1;
        cudaStream_t si = single ? sk : copy_in_.get(), so = single ? sk : copy_out_.get();
        for (int b = 0; b < 2; ++b)
        {
            grow(db_in_[b], (size_t)chunk * nc * esz);
            if (llr_out) grow(db_out_[b], (size_t)chunk * nc * sizeof(double));
            if (hard) grow(db_hard_[b], (size_t)chunk * nc);
            if (hard_bits) grow(db_bits_[b], (size_t)chunk * hw * sizeof(uint32_t));
            if (iters) grow(db_it_[b], (size_t)chunk * sizeof(int32_t));
        }
        unsigned long long h[5] = {0, 0, 0, 0, 0};
        try
        {
        CUDA_OK(cudaMemsetAsync(d_counters_.get(), 0, 8 * sizeof(unsigned long long), sk));
        CUDA_OK(cudaEventRecord(ev0_.get(), sk));
        int64_t k = 0, o = 0;
        for (size_t pi = 0; pi < pieces.size(); o += pieces[pi], ++pi, ++k)
        {
            const int b = (int)(k & 1);
            const int64_t m = pieces[pi];
            if (k >= 2) CUDA_OK(cudaStreamWaitEvent(si, ev_k_[b].get(), 0)); // the kernel that read this input buffer is done
            CUDA_OK(cudaMemcpyAsync(db_in_[b].p.get(), (const unsigned char *)llr + (size_t)o * nc * esz, (size_t)m * nc * esz, cudaMemcpyHostToDevice, si));
            if (!single)
            {
                CUDA_OK(cudaEventRecord(ev_in_[b].get(), si));
                CUDA_OK(cudaStreamWaitEvent(sk, ev_in_[b].get(), 0));
            }
            if (k >= 2) CUDA_OK(cudaStreamWaitEvent(sk, ev_out_[b].get(), 0)); // the copy-out of this output buffer is done
            FrameSource src;
            src.kind = SRC_LLR;
            if (llr_type == LDPC_B200_LLR_F64) src.d_llr = (const double *)db_in_[b].p.get();
            else if (llr_type == LDPC_B200_LLR_F32) src.d_llr_f32 = (const float *)db_in_[b].p.get();
            else { src.d_llr_i8 = (const int8_t *)db_in_[b].p.get(); src.i8_scale = llr_scale; }
            FrameSink sink;
            sink.d_llr_out = llr_out ? (double *)db_out_[b].p.get() : nullptr;
            sink.d_hard = hard ? db_hard_[b].p.get() : nullptr;
            sink.d_hard_bits = hard_bits ? (uint32_t *)db_bits_[b].p.get() : nullptr;
            sink.hard_words = (int)hw;
            sink.d_iters = iters ? (int32_t *)db_it_[b].p.get() : nullptr;
            launch(dp, src, sink, (uint64_t)m, sk);
            if (!single)
            {
                CUDA_OK(cudaEventRecord(ev_k_[b].get(), sk));
                CUDA_OK(cudaStreamWaitEvent(so, ev_k_[b].get(), 0));
            }
            if (llr_out) CUDA_OK(cudaMemcpyAsync(llr_out + o * nc, db_out_[b].p.get(), m * nc * sizeof(double), cudaMemcpyDeviceToHost, so));
            if (hard) CUDA_OK(cudaMemcpyAsync(hard + o * nc, db_hard_[b].p.get(), m * nc, cudaMemcpyDeviceToHost, so));
            if (hard_bits) CUDA_OK(cudaMemcpyAsync(hard_bits + o * hw, db_bits_[b].p.get(), m * hw * sizeof(uint32_t), cudaMemcpyDeviceToHost, so));
            if (iters) CUDA_OK(cudaMemcpyAsync(iters + o, db_it_[b].p.get(), m * sizeof(int32_t), cudaMemcpyDeviceToHost, so));
            if (!single) CUDA_OK(cudaEventRecord(ev_out_[b].get(), so));
        }
        CUDA_OK(cudaEventRecord(ev1_.get(), sk));
        CUDA_OK(cudaMemcpyAsync(h, d_counters_.get(), sizeof(h), cudaMemcpyDeviceToHost, sk));
        CUDA_OK(cudaStreamSynchronize(sk));
        if (!single) CUDA_OK(cudaStreamSynchronize(so));
        }
        catch (...)
        { // copies in flight still reference the caller's buffers and the cached device buffers: drain all three streams first
            cudaStreamSynchronize(si); cudaStreamSynchronize(sk); cudaStreamSynchronize(so);
            throw;
        }
        float ms = 0;
        CUDA_OK(cudaEventElapsedTime(&ms, ev0_.get(), ev1_.get()));
        account(ms, h[2], h[4]);
    }

    void Engine::decode_bec_host(const decoder_param &dp, const uint8_t *in, const uint8_t *cw, int64_t n, uint8_t *out, uint8_t *hard, int32_t *iters)
    {
        if (n <= 0) return;
        ensure_cuda();
        cudaStream_t s = stream_.get();
        const size_t nc = H.nc;
        const DevPtr<uint8_t> d_in = device_alloc<uint8_t>(n * nc), d_cw = device_alloc<uint8_t>(n * nc);
        const DevPtr<uint8_t> d_out = device_alloc<uint8_t>(n * nc), d_hard = device_alloc<uint8_t>(n * nc);
        const DevPtr<int32_t> d_it = device_alloc<int32_t>(n);
        CUDA_OK(cudaMemcpyAsync(d_in.get(), in, n * nc, cudaMemcpyHostToDevice, s));
        CUDA_OK(cudaMemcpyAsync(d_cw.get(), cw, n * nc, cudaMemcpyHostToDevice, s));
        CUDA_OK(cudaMemsetAsync(d_counters_.get(), 0, 8 * sizeof(unsigned long long), s));
        FrameSource src;
        src.kind = SRC_LLR;
        src.d_bec_in = d_in.get(); src.d_bec_cw = d_cw.get();
        FrameSink sink;
        sink.d_bec_out = d_out.get(); sink.d_hard = d_hard.get(); sink.d_iters = d_it.get();
        launch(dp, src, sink, (uint64_t)n, s, true);
        if (out) CUDA_OK(cudaMemcpyAsync(out, d_out.get(), n * nc, cudaMemcpyDeviceToHost, s));
        if (hard) CUDA_OK(cudaMemcpyAsync(hard, d_hard.get(), n * nc, cudaMemcpyDeviceToHost, s));
        if (iters) CUDA_OK(cudaMemcpyAsync(iters, d_it.get(), n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaStreamSynchronize(s));
    }

    // Stand-alone channel kernel: the same generator code as the fused path, one thread per Philox block.  Output row fr holds
    // global frame frame0 + fr, or with GATHER frames[fr] (the replay of a list of logged frames).
    template <bool GATHER>
    __global__ void channel_kernel(int kind, int nc, int nct, const int32_t *__restrict__ bit_pos, const int32_t *__restrict__ punct, int n_punct,
                                   const int32_t *__restrict__ shorten, int n_short, double sigma, double llr_scale, double delta, uint32_t thr,
                                   uint64_t seed, uint32_t point, uint64_t frame0, int64_t n_frames, uint8_t *cw, double *llr, uint8_t *llr_u8,
                                   const int32_t *__restrict__ g_col_ptr, const int32_t *__restrict__ g_row, int g_rows, int g_cols, AskParams ask,
                                   double sigma2, const uint64_t *__restrict__ frames, int coherence)
    {
        auto frame_of = [&](int64_t fr) -> uint64_t { return GATHER ? frames[fr] : frame0 + fr; };
        if (kind == SRC_ASK)
        { // M-ASK with bit-metric decoding: one thread per Philox block of four symbols (same arithmetic as tile4.cuh frame_pass)
            const int nsblk = (ask.n_sym + 3) / 4;
            const int64_t total = n_frames * (int64_t)nsblk;
            for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x)
            {
                const int64_t fr = g / nsblk;
                const int q = (int)(g % nsblk);
                const size_t base = (size_t)fr * nc;
                const u32x4 r = channel_block(seed, point, 0, frame_of(fr), (uint32_t)q);
                float z[4];
                normal_pair(r.x, r.y, z[0], z[1]);
                normal_pair(r.z, r.w, z[2], z[3]);
                for (int k = 0; k < 4; ++k)
                    if (q + k * nsblk < ask.n_sym)
                        ask_symbol(ask, seed, point, frame_of(fr), q + k * nsblk, z[k], sigma, sigma2, [&](int v, double l, uint32_t c) {
                            llr[base + v] = l;
                            if (cw) cw[base + v] = (uint8_t)c;
                        });
                if (q == 0)
                {
                    for (int i = 0; i < n_punct; ++i) { llr[base + punct[i]] = 0.0; if (cw) cw[base + punct[i]] = 0; }
                    for (int i = 0; i < n_short; ++i) { llr[base + shorten[i]] = 99999.9; if (cw) cw[base + shorten[i]] = 0; }
                }
            }
            return;
        }
        // codeword bit of variable v in frame fr: parity of the Philox stream-1 information bits selected by column v of G
        // (same rule as the fused kernels); 0 without a generator matrix.
        auto cw_bit = [&](int64_t fr, int v) -> uint32_t
        {
            if (g_rows <= 0 || v >= g_cols) return 0u;
            uint32_t b = 0;
            for (int q = g_col_ptr[v]; q < g_col_ptr[v + 1]; ++q)
            {
                const int r = g_row[q];
                const u32x4 w = channel_block(seed, point, 1, frame_of(fr), (uint32_t)r >> 7);
                const uint32_t q4[4] = {w.x, w.y, w.z, w.w};
                b ^= q4[(r >> 5) & 3] >> (r & 31);
            }
            return b & 1u;
        };
        const int nblk = (nct + 3) / 4; // value q of Philox block j serves the transmitted index j + q*nblk, on every channel
        const int64_t total = n_frames * (int64_t)nblk;
        for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x)
        {
            const int64_t fr = g / nblk;
            const int j = (int)(g % nblk);
            const u32x4 r = channel_block(seed, point, 0, frame_of(fr), (uint32_t)j);
            const size_t base = (size_t)fr * nc;
            if (kind == SRC_AWGN)
            { // the same arithmetic as the fused path (tile4.cuh frame_pass)
                float z[4];
                normal_pair(r.x, r.y, z[0], z[1]);
                normal_pair(r.z, r.w, z[2], z[3]);
                for (int q = 0; q < 4; ++q)
                {
                    const int t = j + q * nblk;
                    if (t >= nct) break;
                    const uint32_t b = cw_bit(fr, bit_pos[t]);
                    const double y = __dadd_rn(__dmul_rn((double)z[q], sigma), b ? -1.0 : 1.0);
                    llr[base + bit_pos[t]] = __dmul_rn(y, llr_scale);
                    if (cw) cw[base + bit_pos[t]] = (uint8_t)b;
                }
            }
            else if (kind == SRC_RAYLEIGH)
            { // the same arithmetic as the fused path (tile4.cuh frame_pass)
                float z[4];
                normal_pair(r.x, r.y, z[0], z[1]);
                normal_pair(r.z, r.w, z[2], z[3]);
                for (int q = 0; q < 4; ++q)
                {
                    const int t = j + q * nblk;
                    if (t >= nct) break;
                    const uint32_t b = cw_bit(fr, bit_pos[t]);
                    const double h = rayleigh_coeff(seed, point, frame_of(fr), coherence ? (uint32_t)(t / coherence) : 0u);
                    const double y = __dadd_rn(__dmul_rn((double)z[q], sigma), b ? -h : h);
                    llr[base + bit_pos[t]] = __dmul_rn(__dmul_rn(y, h), llr_scale);
                    if (cw) cw[base + bit_pos[t]] = (uint8_t)b;
                }
            }
            else
            {
                const uint32_t w[4] = {r.x, r.y, r.z, r.w};
                for (int q = 0; q < 4; ++q)
                {
                    const int t = j + q * nblk;
                    if (t >= nct) break;
                    const bool hit = w[q] < thr;
                    if (kind == SRC_BSC)
                    {
                        const uint32_t b = cw_bit(fr, bit_pos[t]);
                        llr[base + bit_pos[t]] = ((hit ? 1u : 0u) ^ b) ? -delta : delta;
                        if (cw) cw[base + bit_pos[t]] = (uint8_t)b;
                    }
                    else
                    { // y = 'E' w.p. eps else x (src/sim/channel.cpp:193-205)
                        const uint32_t b = cw_bit(fr, bit_pos[t]);
                        llr_u8[base + bit_pos[t]] = hit ? (uint8_t)'E' : (uint8_t)b;
                        if (cw) cw[base + bit_pos[t]] = (uint8_t)b;
                    }
                }
            }
            if (j == 0)
            {
                for (int i = 0; i < n_punct; ++i)
                {
                    if (kind == SRC_BEC) llr_u8[base + punct[i]] = (uint8_t)'E';
                    else llr[base + punct[i]] = 0.0;
                }
                for (int i = 0; i < n_short; ++i)
                {
                    if (kind == SRC_BEC) llr_u8[base + shorten[i]] = (uint8_t)cw_bit(fr, shorten[i]); // the true bit (channel.cpp:219-222)
                    else llr[base + shorten[i]] = (kind == SRC_BSC) ? delta : 99999.9;
                }
                if (cw)
                { // non-transmitted positions carry their codeword bit too
                    for (int i = 0; i < n_punct; ++i) cw[base + punct[i]] = (uint8_t)cw_bit(fr, punct[i]);
                    for (int i = 0; i < n_short; ++i) cw[base + shorten[i]] = (uint8_t)cw_bit(fr, shorten[i]);
                }
            }
        }
    }

    // Enqueues the channel kernel on s: rows of global frames frame0 + fr, or frames[fr] when `frames` (device) is given.
    // kind = SRC_AWGN is M-ASK under the current modulation; SRC_RAYLEIGH uses the context's coherence length.
    void Engine::launch_channel(int kind, double x, uint64_t seed, uint32_t point, uint64_t frame0, const uint64_t *frames, int64_t n,
                                uint8_t *d_cw, double *d_llr, uint8_t *d_u8, cudaStream_t s)
    {
        AskParams ask{};
        if (kind == SRC_AWGN && ask_M > 2) { kind = SRC_ASK; ask_fill(&ask); }
        const ChannelConsts cc = channel_consts(kind, x);
        const int g_rows = (has_gen && !tuning.zero_codeword) ? G.mc : 0, g_cols = has_gen ? G.nc : 0;
        auto fn = frames ? channel_kernel<true> : channel_kernel<false>;
        fn<<<sm_count_ * 4, 256, 0, s>>>(kind, H.nc, H.nct(), d_bit_pos_.get(), d_punct_.get(), (int)H.puncture.size(), d_short_.get(),
                                         (int)H.shorten.size(), cc.sigma, cc.llr_scale, cc.delta, cc.thr, seed, point, frame0, n, d_cw, d_llr, d_u8,
                                         d_g_col_ptr_.get(), d_g_row_.get(), g_rows, g_cols, ask, cc.sigma2, frames, fading_L);
        CUDA_OK(cudaGetLastError());
    }

    void Engine::channel_host(const std::string &channel, double x, uint64_t seed, uint32_t point, uint64_t frame0, int64_t n,
                              uint8_t *cw, double *llr, uint8_t *llr_u8)
    {
        if (n <= 0) return;
        ensure_cuda();
        const int kind = channel_kind(channel);
        cudaStream_t s = stream_.get();
        const size_t nc = H.nc;
        DevPtr<double> d_llr;
        DevPtr<uint8_t> d_u8, d_cw;
        if (kind == SRC_BEC) { if (!llr_u8) throw std::runtime_error("llr_u8 buffer required for BEC"); d_u8 = device_alloc<uint8_t>(n * nc); }
        else { if (!llr) throw std::runtime_error("llr buffer required"); d_llr = device_alloc<double>(n * nc); }
        if (cw) d_cw = device_alloc<uint8_t>(n * nc);
        launch_channel(kind, x, seed, point, frame0, nullptr, n, d_cw.get(), d_llr.get(), d_u8.get(), s);
        if (d_llr) CUDA_OK(cudaMemcpyAsync(llr, d_llr.get(), n * nc * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (d_u8) CUDA_OK(cudaMemcpyAsync(llr_u8, d_u8.get(), n * nc, cudaMemcpyDeviceToHost, s));
        if (d_cw) CUDA_OK(cudaMemcpyAsync(cw, d_cw.get(), n * nc, cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaStreamSynchronize(s));
    }

    // Replay of logged frames: the gather channel regenerates their decoder inputs, the decode runs under the current tuning
    // (the erasure decode mode on the BEC, as decode_bec_host), and report_kernel compares the decisions with the transmitted
    // word.  Chunks of about 32 MB of decoder input, whole waves of the persistent grid.
    void Engine::error_report(const decoder_param &dp, const std::string &channel, double x, uint64_t seed, uint32_t point, const uint64_t *frames,
                              int64_t n, ldpc_b200_frame_report *reports, std::vector<int32_t> &bits, std::vector<int32_t> &checks)
    {
        const int kind = channel_kind(channel);
        if (n < 0 || (n > 0 && (!frames || !reports))) throw std::runtime_error("error_report: bad frame list");
        bits.clear();
        checks.clear();
        if (n == 0) return;
        ensure_cuda();
        cudaStream_t s = stream_.get();
        const bool bec = kind == SRC_BEC, ask = kind == SRC_AWGN && ask_M > 2;
        const size_t nc = H.nc;
        if (!d_chk_var_)
        {
            std::vector<int32_t> ptr(H.row_ptr.begin(), H.row_ptr.end()), var(H.nnz);
            for (int q = 0; q < H.nnz; ++q) var[q] = (int32_t)H.e_col[H.row_edge[q]];
            d_chk_ptr_ = upload(ptr);
            d_chk_var_ = upload(var);
        }
        int64_t chunk = std::max<int64_t>((int64_t)((32ull << 20) / (nc * (bec ? 1 : sizeof(double)))), 1);
        if (!bec)
        {
            const int64_t wave = batch_wave(dp, (uint64_t)n, s);
            chunk = std::max<int64_t>(wave, chunk / wave * wave);
        }
        chunk = std::min<int64_t>(chunk, n);
        const DevPtr<uint64_t> d_frames = device_alloc<uint64_t>(chunk);
        const DevPtr<uint8_t> d_cw = device_alloc<uint8_t>(chunk * nc), d_hard = device_alloc<uint8_t>(chunk * nc);
        DevPtr<uint8_t> d_u8;
        DevPtr<double> d_llr;
        if (bec) d_u8 = device_alloc<uint8_t>(chunk * nc);
        else d_llr = device_alloc<double>(chunk * nc);
        const DevPtr<int32_t> d_iters = device_alloc<int32_t>(chunk);
        const DevPtr<uint32_t> d_counts = device_alloc<uint32_t>(2 * chunk);
        const DevPtr<int64_t> d_offsets = device_alloc<int64_t>(2 * chunk);
        DevBuf d_bits, d_checks;
        std::vector<int32_t> iters(chunk);
        std::vector<uint32_t> counts(2 * chunk);
        std::vector<int64_t> offsets(2 * chunk);
        ReportParams rp{};
        rp.hard = d_hard.get(); rp.cw = ask ? nullptr : d_cw.get(); // M-ASK: the decoder sees the all-zero word (set_modulation)
        rp.bit_pos = d_bit_pos_.get(); rp.chk_ptr = d_chk_ptr_.get(); rp.chk_var = d_chk_var_.get();
        rp.nc = H.nc; rp.nct = H.nct(); rp.mc = H.mc;
        rp.counts = d_counts.get(); rp.offsets = d_offsets.get();
        for (int64_t o = 0; o < n; o += chunk)
        {
            const int64_t m = std::min(chunk, n - o);
            CUDA_OK(cudaMemcpyAsync(d_frames.get(), frames + o, m * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
            launch_channel(kind, x, seed, point, 0, d_frames.get(), m, ask ? nullptr : d_cw.get(), d_llr.get(), d_u8.get(), s);
            FrameSource src;
            src.kind = SRC_LLR;
            if (bec) { src.d_bec_in = d_u8.get(); src.d_bec_cw = d_cw.get(); }
            else src.d_llr = d_llr.get();
            FrameSink sink;
            sink.d_hard = d_hard.get(); sink.d_iters = d_iters.get();
            launch(dp, src, sink, (uint64_t)m, s);
            rp.n = m;
            const int blocks = clamp_grid(sm_count_ * 8, (uint64_t)(m + 7) / 8); // 8 warps (frames) per block
            report_kernel<false><<<blocks, 256, 0, s>>>(rp);
            CUDA_OK(cudaGetLastError());
            CUDA_OK(cudaMemcpyAsync(counts.data(), d_counts.get(), 2 * m * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
            CUDA_OK(cudaMemcpyAsync(iters.data(), d_iters.get(), m * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
            CUDA_OK(cudaStreamSynchronize(s));
            int64_t nb = 0, nk = 0;
            for (int64_t i = 0; i < m; ++i)
            {
                offsets[2 * i] = nb; offsets[2 * i + 1] = nk;
                ldpc_b200_frame_report &r = reports[o + i];
                r.frame = frames[o + i]; r.iterations = iters[i];
                r.bit_errors = counts[2 * i]; r.syndrome_weight = counts[2 * i + 1];
                r.bits_offset = (int64_t)bits.size() + nb; r.checks_offset = (int64_t)checks.size() + nk;
                nb += counts[2 * i];
                nk += counts[2 * i + 1];
            }
            if (nb + nk == 0) continue;
            grow(d_bits, std::max<int64_t>(nb, 1) * sizeof(int32_t));
            grow(d_checks, std::max<int64_t>(nk, 1) * sizeof(int32_t));
            rp.failed_bits = (int32_t *)d_bits.p.get(); rp.failed_checks = (int32_t *)d_checks.p.get();
            CUDA_OK(cudaMemcpyAsync(d_offsets.get(), offsets.data(), 2 * m * sizeof(int64_t), cudaMemcpyHostToDevice, s));
            report_kernel<true><<<blocks, 256, 0, s>>>(rp);
            CUDA_OK(cudaGetLastError());
            const size_t b0 = bits.size(), k0 = checks.size();
            bits.resize(b0 + nb);
            checks.resize(k0 + nk);
            if (nb) CUDA_OK(cudaMemcpyAsync(bits.data() + b0, d_bits.p.get(), nb * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
            if (nk) CUDA_OK(cudaMemcpyAsync(checks.data() + k0, d_checks.p.get(), nk * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
            CUDA_OK(cudaStreamSynchronize(s));
        }
    }
} // namespace b200

extern "C" int ldpc_b200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}
