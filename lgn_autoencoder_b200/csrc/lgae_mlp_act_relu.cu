// CGMLP kernels (lgae_mlp.cuh) with the ReLU and ELU activations.
#include "lgae_mlp.cuh"

namespace lgae {

LGAE_MLP_INSTANCES(, LGAE_ACT_RELU)
LGAE_MLP_INSTANCES(, LGAE_ACT_ELU)

}  // namespace lgae
