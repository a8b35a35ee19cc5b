// tf32 (fp32 storage) instantiations of the halo-tile convolution kernel (conv_halo.cuh)
#include <cstring>
#include "conv_halo.cuh"
namespace biu {
BIU_HALO_INSTANCES(, FMT_TF32)
}  // namespace biu
