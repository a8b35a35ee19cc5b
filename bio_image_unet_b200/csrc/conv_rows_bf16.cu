// bf16 instantiations of the row-streaming folded-tap convolution kernel (conv_rows.cuh)
#include "conv_rows.cuh"
namespace biu {
BIU_ROWS_INSTANCES(, FMT_BF16)
}  // namespace biu
