// Variant choice of the tile kernel family.  Each (T, ALG, lanes) is instantiated in its own translation unit
// (tile_<alg>_<prec>_l<lanes>.cu) so that the build can compile them in parallel.
#pragma once
#include <stdexcept>

#include "tile4.cuh"

namespace b200
{
    constexpr int TILE_SMEM_OPTIN = 232448 - 2048; // 227 KB minus the kernel's static shared memory (scheduling state, a copy of the arguments)

    // Variants per (T, ALG, lanes): shared-memory residency with the TMEM mirror (with / without the
    // early-termination syndrome: --no-early-term min-sum runs skip it), shared-memory residency without the mirror,
    // global residency (min-sum: a narrow 2-CTA/64-register and a wide 1-CTA/128-register build).  Index entries are
    // 32-bit byte offsets, or 16-bit with the TMEM mirror (idx16).
    // lanes = warp lanes per node (frames per CTA = lanes * 16/sizeof(T)).
    // wide (global residency, min-sum): the 1-CTA-per-SM / 128-register build instead of the 2-CTA / 64-register one
    template <typename T, int ALG, int L>
    const void *tile_variant(bool smem, bool tm, bool et, bool wide, bool idx16)
    {
        constexpr int NB = (ALG == ALG_MS) ? (1024 / B200_TILE_MAX_THREADS) : 1;
        typedef uint32_t U32;
        typedef uint16_t U16;
        if (smem && tm && idx16 && (et || ALG != ALG_MS)) return (const void *)tile4_kernel<T, U16, ALG, true, L, true, true, 1>;
        if (smem && tm && idx16) return (const void *)tile4_kernel<T, U16, ALG, true, L, true, ALG != ALG_MS, 1>;
        if (smem && tm && (et || ALG != ALG_MS)) return (const void *)tile4_kernel<T, U32, ALG, true, L, true, true, 1>;
        if (smem && tm) return (const void *)tile4_kernel<T, U32, ALG, true, L, true, ALG != ALG_MS, 1>;
        if (smem) return (const void *)tile4_kernel<T, U32, ALG, true, L, false, true, 1>;
        if (wide) return (const void *)tile4_kernel<T, U32, ALG, false, L, false, true, 1>;
        return (const void *)tile4_kernel<T, U32, ALG, false, L, false, true, NB>;
    }

    extern template const void *tile_variant<double, ALG_BP, 1>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<double, ALG_BP, 2>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<double, ALG_BP, 4>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<double, ALG_MS, 1>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<double, ALG_MS, 2>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<double, ALG_MS, 4>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<float, ALG_BP, 1>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<float, ALG_BP, 2>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<float, ALG_BP, 4>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<float, ALG_MS, 1>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<float, ALG_MS, 2>(bool, bool, bool, bool, bool);
    extern template const void *tile_variant<float, ALG_MS, 4>(bool, bool, bool, bool, bool);

    // the tile kernel for (precision, algorithm, lanes per node: 1, 2 or 4) and the variant switches
    inline const void *tile_kernel(bool f32, int alg, int lanes, bool smem, bool tm, bool et, bool wide, bool idx16)
    {
        typedef const void *(*Variant)(bool, bool, bool, bool, bool);
        static const Variant variants[2][2][3] = {
            {{tile_variant<double, ALG_MS, 1>, tile_variant<double, ALG_MS, 2>, tile_variant<double, ALG_MS, 4>},
             {tile_variant<double, ALG_BP, 1>, tile_variant<double, ALG_BP, 2>, tile_variant<double, ALG_BP, 4>}},
            {{tile_variant<float, ALG_MS, 1>, tile_variant<float, ALG_MS, 2>, tile_variant<float, ALG_MS, 4>},
             {tile_variant<float, ALG_BP, 1>, tile_variant<float, ALG_BP, 2>, tile_variant<float, ALG_BP, 4>}}};
        if (lanes != 1 && lanes != 2 && lanes != 4) throw std::runtime_error("lanes per node must be 1, 2 or 4");
        return variants[f32][alg == ALG_BP][lanes / 2](smem, tm, et, wide, idx16);
    }
} // namespace b200
