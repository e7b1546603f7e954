// layered-schedule kernel instantiations (layered.cuh)
#include <stdexcept>

#include "layered.cuh"

namespace b200
{
    const void *layered_kernel(bool f32, int alg, int lanes)
    {
        static const void *const kernels[2][2][2] = {
            {{(const void *)lay_kernel<double, ALG_MS, 2>, (const void *)lay_kernel<double, ALG_MS, 4>},
             {(const void *)lay_kernel<double, ALG_BP, 2>, (const void *)lay_kernel<double, ALG_BP, 4>}},
            {{(const void *)lay_kernel<float, ALG_MS, 2>, (const void *)lay_kernel<float, ALG_MS, 4>},
             {(const void *)lay_kernel<float, ALG_BP, 2>, (const void *)lay_kernel<float, ALG_BP, 4>}}};
        if (lanes != 2 && lanes != 4) throw std::runtime_error("layered schedule: lanes per node must be 2 or 4");
        return kernels[f32][alg == ALG_BP][lanes == 4];
    }
} // namespace b200
