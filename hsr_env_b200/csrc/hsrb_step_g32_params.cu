// Action kernel with per-environment parameters, 32 lanes per environment (see hsrb_kernels.cuh).
#include "hsrb_kernels.cuh"
HSRB_DEFINE_G_PARAMS(32)
