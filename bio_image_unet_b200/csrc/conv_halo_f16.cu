// fp16 instantiations of the halo-tile convolution kernel (conv_halo.cuh)
#include <cstring>
#include "conv_halo.cuh"
namespace biu {
BIU_DEFINE_HALO_DISPATCH(halo_dispatch_f16, FMT_F16)
BIU_DEFINE_HALO_PAIRS(halo_max_pairs_f16, FMT_F16)
}  // namespace biu
