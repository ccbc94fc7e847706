// Streamed-weight CGMLP kernels (lgae_mlp_streamed.cuh) with the leakyrelu activation.
#include "lgae_mlp_streamed.cuh"

namespace lgae {

LGAE_MLP_STREAMED_INSTANCES(, LGAE_ACT_LEAKYRELU)

}  // namespace lgae
