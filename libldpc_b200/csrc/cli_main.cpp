// ldpcsim — command-line front end with the reference's interface (src/sim_cpu.cpp:7-22):
//   ldpcsim [options] codefile output-file MIN MAX STEP
//   -G/--gen-matrix FILE  -i/--num-iterations N (50)  -s/--seed N (0)  -t/--num-threads N (1, ignored)
//   --channel AWGN|BSC|BEC (AWGN; B200 extra: RAYLEIGH)  --decoding BP|BP_MS (BP)  --max-frames N (10e9)
//   --frame-error-count N (50)  --no-early-term  -h/--help  -v/--version
// Negative MIN/MAX are positionals, as with the reference's argument parser.
// B200 extras (do not exist in the reference): --precision f64|f32, --device N, --gpus N / --devices LIST (frames of every
// round sharded over N GPUs of this process, one host thread per shard; the counters are summed on the host, results do not
// depend on the number of shards), --error-log FILE (per sweep point, the first --frame-error-count frames in error, replayed on the
// GPU: failed bits and checks; see the usage text), --channel RAYLEIGH with --coherence L (flat Rayleigh fading, DESIGN.md §3.2),
// --quantize CH,MSG,POST --llr-step D [--ms-offset B] (fixed-point layered min-sum, DESIGN.md §3.7).
// The CLI is a client of the C ABI only (include/ldpc_b200.h): the library exports nothing else.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <array>
#include <cstring>
#include <iostream>
#include <map>
#include <stdexcept>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/ldpc_b200.h"

namespace
{
    const char *USAGE =
        "Usage: ldpc [options] codefile output-file snr-range \n\n"
        "Positional arguments:\n"
        "codefile            \tLDPC parity-check matrix file containing all non-zero entries.\n"
        "output-file         \tResults output file.\n"
        "snr-range           \t{MIN} {MAX} {STEP}\n\n"
        "Optional arguments:\n"
        "-h --help           \tshows help message and exits\n"
        "-v --version        \tprints version information and exits\n"
        "-G --gen-matrix     \tGenerator matrix file.\n"
        "-i --num-iterations \tNumber of iterations for decoding. (Default: 50)\n"
        "-s --seed           \tRNG seed. (Default: 0)\n"
        "-t --num-threads    \tNumber of frames to be decoded in parallel. (Default: 1; ignored, the GPU batches frames)\n"
        "--channel           \tSpecifies channel: \"AWGN\", \"BSC\", \"BEC\" (Default: AWGN); B200 only: \"RAYLEIGH\" (BPSK over flat Rayleigh\n"
        "                    \tfading with perfect CSI at the receiver, x = average SNR in dB)\n"
        "--decoding          \tSpecifies decoding algorithm: \"BP\", \"BP_MS\" (Default: BP)\n"
        "--max-frames        \tLimit number of decoded frames.\n"
        "--frame-error-count \tMaximum frame errors for given simulation point.\n"
        "--no-early-term     \tDisable early termination for decoding.\n"
        "--precision         \tB200 only: message arithmetic \"f64\" (bit-exact with the reference, default) or \"f32\"\n"
        "--device            \tB200 only: CUDA device index (Default: 0)\n"
        "--gpus              \tB200 only: number of GPUs to shard every round of frames over, starting at --device (Default: 1, 0 = all)\n"
        "--schedule          \tB200 only: \"flooding\" (the reference's schedule, default) or \"layered\" (opt-in; results differ by design)\n"
        "--ms-scale          \tB200 only: with --schedule layered and BP_MS: normalisation factor of the check outputs in 1/64 steps (Default: 1 = plain min-sum)\n"
        "--modulation        \tB200 only: M-ASK with bit-metric decoding on the AWGN channel, M = 4, 8, ... (Gray labels, consecutive bit mapper; Default: 2 = BPSK)\n"
        "--layers            \tB200 only: layer file for --schedule layered (legacy format: nl: N / cn[i]: W / W check indices); default: built-in layering\n"
        "--devices           \tB200 only: explicit device list for the shards, e.g. 0,1,2,3 (an index may repeat: several shards on one GPU)\n"
        "--coherence         \tB200 only: with --channel RAYLEIGH: transmitted bits per fading coefficient, >= 0 (Default: 1 = fast fading;\n"
        "                    \t0 = one coefficient per frame)\n"
        "--error-log         \tB200 only: file of the frames in error: per point the first --frame-error-count of them in frame order, one line\n"
        "                    \teach: snr frame iterations bit_errors syndrome_weight failed_bits failed_checks (comma-separated lists, - = empty;\n"
        "                    \tsyndrome_weight 0 with bit_errors > 0 is an undetected error); written after every round\n"
        "--quantize          \tB200 only: fixed-point layered min-sum with CH,MSG,POST bits of the channel LLR, the check-to-variable messages\n"
        "                    \tand the posterior (2 <= MSG <= POST <= 16, 2 <= CH <= POST); needs --schedule layered, --decoding BP_MS and\n"
        "                    \t--llr-step; not on the BEC or with --modulation > 2.  --ms-scale is then a multiple of 1/8\n"
        "--llr-step          \tB200 only: with --quantize: LLR value of one LSB (> 0); channel LLRs enter as clamp(round(L / step))\n"
        "--ms-offset         \tB200 only: with --quantize: min-sum offset in LSBs, 0 <= B < 2^(MSG-1) - 1 (Default: 0)\n";

    bool looks_numeric(const std::string &s)
    {
        if (s.empty()) return false;
        char *end = nullptr;
        std::strtod(s.c_str(), &end);
        return end && *end == 0;
    }

    // Multi-GPU rounds: the sweep driver hands one round [frame0, frame0 + n) of a sweep point to this callback, which
    // splits it contiguously over the contexts (one per GPU, one host thread each) and sums the counters.  The frame ->
    // Philox substream mapping depends only on the global frame index, so the totals do not depend on the split.
    struct MultiGpu
    {
        std::vector<ldpc_b200_ctx *> ctxs;
        decoder_param dp;
        std::string channel;
        uint64_t seed = 0;
        // --error-log
        FILE *log = nullptr;
        uint64_t log_budget = 0;              // frames logged per point (--frame-error-count)
        std::map<uint32_t, uint64_t> logged;  // point -> frames logged so far
        uint64_t mismatches = 0;              // logged frames whose replay differs from the sweep's record
        ~MultiGpu()
        {
            for (auto *c : ctxs) ldpc_b200_close(c);
            if (log) fclose(log);
        }
    };
    int multi_gpu_round(uint32_t point, double x, uint64_t frame0, uint64_t n, uint64_t *counters, void *user)
    {
        MultiGpu &m = *static_cast<MultiGpu *>(user);
        const size_t g = m.ctxs.size();
        std::vector<std::array<uint64_t, 4>> part(g);
        std::vector<std::string> err(g);
        std::vector<std::thread> th;
        for (size_t i = 0; i < g; ++i)
            th.emplace_back([&, i] {
                const uint64_t lo = frame0 + n * i / g, hi = frame0 + n * (i + 1) / g;
                part[i] = {0, 0, 0, 0};
                if (hi == lo) return;
                if (ldpc_b200_sim_point(m.ctxs[i], m.dp, m.channel.c_str(), x, m.seed, point, lo, hi - lo, part[i].data(), nullptr) != 0)
                    err[i] = ldpc_b200_last_error(); // thread-local message of the failing call
            });
        for (auto &t : th) t.join();
        for (size_t i = 0; i < g; ++i)
        {
            if (!err[i].empty()) { std::cout << "Error: GPU " << i << ": " << err[i] << std::endl; return 1; }
            for (int k = 0; k < 4; ++k) counters[k] += part[i][k];
        }
        return 0;
    }

    void write_list(FILE *f, const int32_t *v, uint32_t n)
    {
        if (n == 0) fputs("-", f);
        for (uint32_t i = 0; i < n; ++i) fprintf(f, i ? ",%d" : "%d", (int)v[i]);
    }

    // A round with the error log.  Every shard records its frames in error (a slice whose errors overflow the record buffer is
    // run again with room for all of them: the counters are deterministic); the records are merged in global frame order and
    // the first ones, up to what is left of the point's budget, are replayed on the first context and appended to the log.  The
    // logged set therefore depends only on (seed, point, frames decoded), not on the shards or the round split.
    int logged_round(uint32_t point, double x, uint64_t frame0, uint64_t n, uint64_t *counters, void *user)
    {
        MultiGpu &m = *static_cast<MultiGpu *>(user);
        const size_t g = m.ctxs.size();
        std::vector<std::array<uint64_t, 4>> part(g, std::array<uint64_t, 4>{0, 0, 0, 0});
        std::vector<std::vector<ldpc_b200_error_record>> recs(g);
        std::vector<std::string> err(g);
        std::vector<std::thread> th;
        for (size_t i = 0; i < g; ++i)
            th.emplace_back([&, i] {
                const uint64_t lo = frame0 + n * i / g, hi = frame0 + n * (i + 1) / g;
                if (hi == lo) return;
                int64_t cap = 256, n_err = 0;
                for (;;)
                {
                    part[i] = {0, 0, 0, 0};
                    recs[i].resize((size_t)cap);
                    if (ldpc_b200_sim_point_log(m.ctxs[i], m.dp, m.channel.c_str(), x, m.seed, point, lo, hi - lo, part[i].data(), recs[i].data(), cap,
                                                &n_err) != 0)
                    {
                        err[i] = ldpc_b200_last_error();
                        return;
                    }
                    if (n_err <= cap) break;
                    cap = n_err;
                }
                recs[i].resize((size_t)n_err);
            });
        for (auto &t : th) t.join();
        std::vector<ldpc_b200_error_record> all;
        for (size_t i = 0; i < g; ++i)
        {
            if (!err[i].empty()) { std::cout << "Error: GPU " << i << ": " << err[i] << std::endl; return 1; }
            for (int k = 0; k < 4; ++k) counters[k] += part[i][k];
            all.insert(all.end(), recs[i].begin(), recs[i].end());
        }
        std::sort(all.begin(), all.end(), [](const ldpc_b200_error_record &a, const ldpc_b200_error_record &b) { return a.frame < b.frame; });
        uint64_t &logged = m.logged[point];
        all.resize((size_t)std::min<uint64_t>(all.size(), m.log_budget > logged ? m.log_budget - logged : 0));
        if (all.empty()) return 0;
        std::vector<uint64_t> frames(all.size());
        for (size_t j = 0; j < all.size(); ++j) frames[j] = all[j].frame;
        std::vector<ldpc_b200_frame_report> rep(all.size());
        std::vector<int32_t> bits(4096), checks(4096);
        for (int attempt = 0;; ++attempt)
        {
            int64_t nb = 0, nk = 0;
            if (ldpc_b200_error_report(m.ctxs[0], m.dp, m.channel.c_str(), x, m.seed, point, frames.data(), (int64_t)frames.size(), rep.data(),
                                       bits.data(), (int64_t)bits.size(), checks.data(), (int64_t)checks.size(), &nb, &nk) == 0)
                break;
            if (attempt > 0 || (nb <= (int64_t)bits.size() && nk <= (int64_t)checks.size()))
            {
                std::cout << "Error: error log: " << ldpc_b200_last_error() << std::endl;
                return 1;
            }
            bits.resize((size_t)std::max<int64_t>(nb, 1));
            checks.resize((size_t)std::max<int64_t>(nk, 1));
        }
        for (size_t j = 0; j < rep.size(); ++j)
        {
            const ldpc_b200_frame_report &r = rep[j];
            if (r.iterations != all[j].iterations || r.bit_errors != all[j].bit_errors) ++m.mismatches;
            fprintf(m.log, "%lf %llu %d %u %u ", x, (unsigned long long)r.frame, (int)r.iterations, (unsigned)r.bit_errors, (unsigned)r.syndrome_weight);
            write_list(m.log, bits.data() + r.bits_offset, r.bit_errors);
            fputs(" ", m.log);
            write_list(m.log, checks.data() + r.checks_offset, r.syndrome_weight);
            fputs("\n", m.log);
        }
        logged += rep.size();
        if (fflush(m.log) != 0 || ferror(m.log))
        {
            std::cout << "Error: error log: write failed" << std::endl;
            return 1;
        }
        return 0;
    }

    std::vector<int> parse_devices(const std::string &list)
    {
        std::vector<int> v;
        size_t pos = 0;
        while (pos <= list.size())
        {
            const size_t c = list.find(',', pos);
            const std::string tok = list.substr(pos, c == std::string::npos ? std::string::npos : c - pos);
            if (tok.empty()) throw std::runtime_error("--devices expects a comma-separated list of CUDA device indices");
            v.push_back(std::stoi(tok));
            if (c == std::string::npos) break;
            pos = c + 1;
        }
        return v;
    }

    template <typename V>
    void print_list(std::ostream &os, const std::vector<V> &v)
    { // vector printer of src/core/functions.h:62-77
        os << "[";
        for (size_t i = 0; i < v.size(); ++i) os << v[i] << (i + 1 < v.size() ? ", " : "");
        os << "]";
    }
} // namespace

int main(int argc, char **argv)
{
    std::string gen, channel = "AWGN", decoding = "BP", precision = "f64";
    unsigned iterations = 50, threads = 1;
    unsigned long seed = 0, max_frames = (unsigned long)10e9, fec = 50;
    bool early_term = true;
    int device = 0, gpus = 1;
    std::string device_list, schedule = "flooding", layer_file, error_log;
    double ms_scale = 1.0;
    int modulation = 2;
    int coherence = 1;
    bool coherence_set = false;
    std::string quantize;
    double llr_step = 0;
    int ms_offset = 0;
    bool llr_step_set = false, ms_offset_set = false, ms_scale_set = false;
    std::vector<std::string> pos;
    try
    {
        for (int i = 1; i < argc; ++i)
        {
            const std::string a = argv[i];
            auto value = [&]() -> std::string
            {
                if (i + 1 >= argc) throw std::runtime_error("Too few arguments for '" + a + "'.");
                return argv[++i];
            };
            if (a == "-h" || a == "--help") { std::cout << USAGE; return 0; }
            else if (a == "-v" || a == "--version") { std::cout << ldpc_b200_version() << std::endl; return 0; }
            else if (a == "-G" || a == "--gen-matrix") gen = value();
            else if (a == "-i" || a == "--num-iterations") iterations = (unsigned)std::stoul(value());
            else if (a == "-s" || a == "--seed") seed = std::stoul(value());
            else if (a == "-t" || a == "--num-threads") threads = (unsigned)std::stoul(value());
            else if (a == "--channel") channel = value();
            else if (a == "--decoding") decoding = value();
            else if (a == "--max-frames") max_frames = std::stoul(value());
            else if (a == "--frame-error-count") fec = std::stoul(value());
            else if (a == "--no-early-term") early_term = false;
            else if (a == "--precision") precision = value();
            else if (a == "--device") device = std::stoi(value());
            else if (a == "--gpus") gpus = std::stoi(value());
            else if (a == "--devices") device_list = value();
            else if (a == "--schedule") schedule = value();
            else if (a == "--layers") layer_file = value();
            else if (a == "--ms-scale") { ms_scale = std::stod(value()); ms_scale_set = true; }
            else if (a == "--modulation") modulation = std::stoi(value());
            else if (a == "--error-log") error_log = value();
            else if (a == "--coherence") { coherence = std::stoi(value()); coherence_set = true; }
            else if (a == "--quantize") quantize = value();
            else if (a == "--llr-step") { llr_step = std::stod(value()); llr_step_set = true; }
            else if (a == "--ms-offset") { ms_offset = std::stoi(value()); ms_offset_set = true; }
            else if (a.size() > 1 && a[0] == '-' && !looks_numeric(a)) throw std::runtime_error("Unknown argument: " + a);
            else pos.push_back(a);
        }
        if (pos.size() < 5) throw std::runtime_error("Too few arguments");
        if (pos.size() > 5) throw std::runtime_error("Maximum number of positional arguments exceeded");
        const double snr[3] = {std::stod(pos[2]), std::stod(pos[3]), std::stod(pos[4])};
        if (snr[0] > snr[1]) throw std::runtime_error("snr min > snr max");
        if (precision != "f64" && precision != "f32") throw std::runtime_error("--precision must be f64 or f32");
        if (schedule != "flooding" && schedule != "layered") throw std::runtime_error("--schedule must be flooding or layered");
        if (coherence_set && channel != "RAYLEIGH") throw std::runtime_error("--coherence applies to --channel RAYLEIGH only");
        if (coherence < 0) throw std::runtime_error("--coherence must be >= 0");
        if (channel == "RAYLEIGH" && modulation != 2) throw std::runtime_error("--channel RAYLEIGH is BPSK only: --modulation must be 2");
        ldpc_b200_quant qt{};
        if (quantize.empty())
        {
            if (llr_step_set) throw std::runtime_error("--llr-step applies to --quantize only");
            if (ms_offset_set) throw std::runtime_error("--ms-offset applies to --quantize only");
        }
        else
        {
            if (schedule != "layered") throw std::runtime_error("--quantize needs --schedule layered");
            if (decoding != "BP_MS") throw std::runtime_error("--quantize needs --decoding BP_MS");
            if (channel == "BEC") throw std::runtime_error("--quantize does not apply to --channel BEC");
            if (modulation != 2) throw std::runtime_error("--quantize needs --modulation 2");
            if (!llr_step_set) throw std::runtime_error("--quantize needs --llr-step");
            if (!(llr_step > 0)) throw std::runtime_error("--llr-step must be > 0");
            if (std::sscanf(quantize.c_str(), "%d,%d,%d", &qt.ch_bits, &qt.msg_bits, &qt.post_bits) != 3 ||
                std::count(quantize.begin(), quantize.end(), ',') != 2)
                throw std::runtime_error("--quantize expects CH,MSG,POST (three bit widths)");
            if (!(qt.msg_bits >= 2 && qt.msg_bits <= qt.post_bits && qt.post_bits <= 16 && qt.ch_bits >= 2 && qt.ch_bits <= qt.post_bits))
                throw std::runtime_error("--quantize: bit widths must satisfy 2 <= MSG <= POST <= 16 and 2 <= CH <= POST");
            if (ms_offset < 0 || ms_offset >= (1 << (qt.msg_bits - 1)) - 1) throw std::runtime_error("--ms-offset must be >= 0 and < 2^(MSG-1) - 1");
            const double a8 = ms_scale * 8.0;
            if (ms_scale_set && !(a8 >= 1 && a8 <= 8 && a8 == std::floor(a8))) throw std::runtime_error("--ms-scale must be a multiple of 1/8 in [1/8, 1] with --quantize");
            qt.offset = ms_offset;
            qt.scale8 = ms_scale_set ? (int)a8 : 8;
            qt.step = llr_step;
        }

        std::vector<int> devices;
        if (!device_list.empty()) devices = parse_devices(device_list);
        else
        {
            if (gpus == 0) gpus = std::max(ldpc_b200_device_count(), 1);
            if (gpus < 1) throw std::runtime_error("--gpus must be >= 0");
            for (int g = 0; g < gpus; ++g) devices.push_back(device + g);
        }
        MultiGpu m;
        if (!error_log.empty())
        { // truncated now: a file that cannot be written fails before any work
            m.log = fopen(error_log.c_str(), "w");
            if (!m.log)
            {
                std::cout << "Error: --error-log: cannot open " << error_log << " for writing" << std::endl;
                return EXIT_FAILURE;
            }
            fputs("snr frame iterations bit_errors syndrome_weight failed_bits failed_checks\n", m.log);
            fflush(m.log);
            m.log_budget = fec;
        }
        ldpc_b200_ctx *ctx = ldpc_b200_open(pos[0].c_str(), gen.c_str(), devices[0]);
        if (!ctx)
        {
            std::cout << "Error: ldpc_code(): " << ldpc_b200_last_error() << std::endl; // src/core/ldpc.cpp:16-20
            return EXIT_FAILURE;
        }
        m.ctxs.push_back(ctx);
        ldpc_b200_tuning tn;
        ldpc_b200_get_tuning(ctx, &tn);
        tn.precision = precision == "f32" ? LDPC_B200_F32 : LDPC_B200_F64;
        tn.schedule = schedule == "layered" ? LDPC_B200_LAYERED : LDPC_B200_FLOODING;
        if (tn.schedule == LDPC_B200_LAYERED) tn.zero_codeword = 1; // the layered sweep transmits the all-zero word
        tn.layered_ms_scale64 = (int)(ms_scale * 64.0 + 0.5);
        ldpc_b200_set_tuning(ctx, &tn);
        if (modulation != 2 && ldpc_b200_set_modulation(ctx, modulation, nullptr, nullptr) != 0)
        {
            std::cout << "Error: modulation: " << ldpc_b200_last_error() << std::endl;
            return EXIT_FAILURE;
        }
        if (channel == "RAYLEIGH" && ldpc_b200_set_fading(ctx, coherence) != 0)
        {
            std::cout << "Error: fading: " << ldpc_b200_last_error() << std::endl;
            return EXIT_FAILURE;
        }
        if (!layer_file.empty() && ldpc_b200_load_layers(ctx, layer_file.c_str()) != 0)
        {
            std::cout << "Error: layers: " << ldpc_b200_last_error() << std::endl;
            return EXIT_FAILURE;
        }
        if (qt.ch_bits && ldpc_b200_set_quant(ctx, &qt) != 0)
        {
            std::cout << "Error: quantize: " << ldpc_b200_last_error() << std::endl;
            return EXIT_FAILURE;
        }
        ldpc_b200_code_info H;
        ldpc_b200_info(ctx, &H);
        std::vector<int> puncture(std::max(H.n_punct, 1)), shorten(std::max(H.n_short, 1));
        ldpc_b200_get_puncture(ctx, puncture.data(), shorten.data());
        puncture.resize(H.n_punct);
        shorten.resize(H.n_short);
        const char *bar = "========================================================================================";
        std::cout << bar << std::endl;
        std::cout << "Parity-Check Matrix: " << pos[0] << std::endl;
        std::cout << "Generator Matrix: " << gen << std::endl;
        // code summary, src/core/ldpc.cpp:112-130
        std::cout << "N : " << H.nc << "\nM : " << H.mc << "\nK : " << H.kc << "\nNNZ : " << H.nnz << "\n";
        std::cout << "puncture[" << puncture.size() << "] : ";
        print_list(std::cout, puncture);
        std::cout << "\nshorten[" << shorten.size() << "] : ";
        print_list(std::cout, shorten);
        std::cout << "\nRate : " << 1. - (double)H.mct / (double)H.nct << "\n";
        std::cout << "N (transmitted) : " << H.nct << "\nM (transmitted) : " << H.mct << "\nK (transmitted) : " << H.kct << "\n" << std::endl;
        std::cout << bar << std::endl;

        decoder_param dp{early_term, iterations, decoding.c_str()};
        channel_param cp{seed, {snr[0], snr[1], snr[2]}, channel.c_str()};
        simulation_param sp{threads, max_frames, fec, pos[1].c_str()};
        // parameter dump, src/core/functions.cpp:19-42 and src/sim/ldpcsim.cpp:84-95
        std::cout << "== Decoder Parameters\n Type: " << dp.type << "\n Iterations: " << dp.iterations << "\n Early Termination: " << dp.earlyTerm << "\n";
        std::cout << "== Channel Parameters\n Type: " << cp.type << "\n Seed: " << cp.seed << "\n Range: Min: " << cp.xRange[0] << ", Max: " << cp.xRange[1]
                  << ", Step: " << cp.xRange[2] << "\n";
        if (tn.schedule == LDPC_B200_LAYERED)
            std::cout << "== Schedule\n layered (" << ldpc_b200_get_layers(ctx, nullptr) << " layers" << (layer_file.empty() ? ", built-in layering" : (", " + layer_file)) << ")\n";
        if (qt.ch_bits)
            std::cout << "== Fixed point\n bits (channel, message, posterior): " << qt.ch_bits << ", " << qt.msg_bits << ", " << qt.post_bits << "\n LLR step: " << qt.step
                      << "\n Offset: " << qt.offset << "\n Scale: " << qt.scale8 << "/8\n";
        std::cout << "== Simulation Parameters\n Threads: " << sp.threads << "\n FEC: " << sp.fec << "\n Max Frames: " << sp.maxFrames
                  << "\n Output File: " << sp.resultFile << "\n" << std::endl;
        std::cout << bar << std::endl;
        bool stop = false;
        int rc;
        if (devices.size() == 1 && !m.log) rc = ldpc_b200_simulate(ctx, dp, cp, sp, nullptr, &stop, 0, 1, nullptr, nullptr, 0);
        else
        { // the logged sweep takes the round callback on any number of devices
            m.dp = dp; m.channel = channel; m.seed = seed;
            for (size_t g = 1; g < devices.size(); ++g)
            {
                ldpc_b200_ctx *c = ldpc_b200_open(pos[0].c_str(), gen.c_str(), devices[g]);
                if (!c) { std::cout << "Error: ldpc_code(): " << ldpc_b200_last_error() << std::endl; return EXIT_FAILURE; }
                ldpc_b200_set_tuning(c, &tn);
                if (!layer_file.empty()) ldpc_b200_load_layers(c, layer_file.c_str());
                m.ctxs.push_back(c); // closed with the others from here on
                if (modulation != 2) ldpc_b200_set_modulation(c, modulation, nullptr, nullptr);
                if (channel == "RAYLEIGH" && ldpc_b200_set_fading(c, coherence) != 0)
                {
                    std::cout << "Error: fading: GPU " << devices[g] << ": " << ldpc_b200_last_error() << std::endl;
                    return EXIT_FAILURE;
                }
                if (qt.ch_bits && ldpc_b200_set_quant(c, &qt) != 0)
                {
                    std::cout << "Error: quantize: GPU " << devices[g] << ": " << ldpc_b200_last_error() << std::endl;
                    return EXIT_FAILURE;
                }
            }
            if (devices.size() > 1)
            {
                std::cout << "GPUs: " << devices.size() << " shards on devices ";
                print_list(std::cout, devices);
                std::cout << std::endl;
            }
            rc = ldpc_b200_simulate_ex(ctx, dp, cp, sp, nullptr, &stop, 0, 1, nullptr, m.log ? logged_round : multi_gpu_round, &m, 0);
        }
        if (rc != 0)
        {
            std::cout << "Error: ldpc_sim::ldpc_sim() " << ldpc_b200_last_error() << std::endl; // src/sim/ldpcsim.cpp:77-81
            return EXIT_FAILURE;
        }
        if (m.mismatches)
        {
            std::cout << "Warning: " << m.mismatches << " frame(s) of the error log replayed with other iteration or bit-error counts than the "
                      << "sweep recorded: their lines do not describe the failure" << std::endl;
            return EXIT_FAILURE;
        }
    }
    catch (const std::exception &e)
    {
        std::cout << e.what() << std::endl; // src/sim_cpu.cpp:77-82
        std::cout << USAGE;
        return EXIT_FAILURE;
    }
    return 0;
}
