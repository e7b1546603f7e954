// tile kernel instantiation: T = double, algorithm = ALG_MS, lanes per node = 1
#include "tile_launch.cuh"
namespace b200
{
    template const void *tile_variant<double, ALG_MS, 1>(bool, bool, bool, bool, bool);
}
