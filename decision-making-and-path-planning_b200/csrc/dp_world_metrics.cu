// csrc/dp_world_metrics.cu -- the world step with episode metrics armed (include/dmpp_b200.h section 11): the METRICS = true
// instances of dp_world_kernel (dp_world_step.cuh), in a translation unit of their own so that the disarmed instances of
// dp_world.cu stay what they were.
#include "dp_world_step.cuh"

template struct WorldStep<true, false, false>;
