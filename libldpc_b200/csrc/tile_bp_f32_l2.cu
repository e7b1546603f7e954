// tile kernel instantiation: T = float, algorithm = ALG_BP, lanes per node = 2
#include "tile_launch.cuh"
namespace b200
{
    template const void *tile_variant<float, ALG_BP, 2>(bool, bool, bool, bool, bool);
}
