// tile kernel instantiation: T = float, algorithm = ALG_BP, lanes per node = 1
#include "tile_launch.cuh"
namespace b200
{
    template const void *tile_variant<float, ALG_BP, 1>(bool, bool, bool, bool, bool);
}
