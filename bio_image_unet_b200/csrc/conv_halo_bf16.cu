// bf16 instantiations of the halo-tile convolution kernel (conv_halo.cuh)
#include <cstring>
#include "conv_halo.cuh"
namespace biu {
BIU_HALO_INSTANCES(, FMT_BF16)
}  // namespace biu
