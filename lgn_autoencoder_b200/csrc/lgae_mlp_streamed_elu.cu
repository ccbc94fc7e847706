// Streamed-weight CGMLP kernels (lgae_mlp_streamed.cuh) with the elu activation.
#include "lgae_mlp_streamed.cuh"

namespace lgae {

LGAE_MLP_STREAMED_INSTANCES(, LGAE_ACT_ELU)

}  // namespace lgae
