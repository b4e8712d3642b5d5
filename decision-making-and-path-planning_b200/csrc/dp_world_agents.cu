// csrc/dp_world_agents.cu -- the world step with reactive agents armed (include/dmpp_b200.h section 12): the REACT = true
// instances of dp_world_kernel (dp_world_step.cuh), with and without junctions and episode metrics, in a translation unit of
// their own so that the disarmed instances of dp_world.cu and dp_world_metrics.cu stay what they were.
#include "dp_world_step.cuh"

template struct WorldStep<false, true, false>;
template struct WorldStep<true, true, false>;
