// CGMLP kernels (lgae_mlp.cuh) with the tanh and atan activations.
#include "lgae_mlp.cuh"

namespace lgae {

LGAE_MLP_INSTANCES(, LGAE_ACT_TANH)
LGAE_MLP_INSTANCES(, LGAE_ACT_ATAN)

}  // namespace lgae
