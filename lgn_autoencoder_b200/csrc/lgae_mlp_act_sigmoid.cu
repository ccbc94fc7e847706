// CGMLP kernels (lgae_mlp.cuh) with the sigmoid and log-sigmoid activations.
#include "lgae_mlp.cuh"

namespace lgae {

LGAE_MLP_INSTANCES(, LGAE_ACT_SIGMOID)
LGAE_MLP_INSTANCES(, LGAE_ACT_LOGSIGMOID)

}  // namespace lgae
