// csrc/dp_world_lanechange.cu -- the world step with lane-changing agents armed (include/dmpp_b200.h section 13, on top of the
// reactive agents of section 12): the LANECHG = true instances of dp_world_kernel (dp_world_step.cuh), with and without
// junctions and episode metrics, in a translation unit of their own so that the disarmed and react-only instances stay what
// they were.
#include "dp_world_step.cuh"

template struct WorldStep<false, true, true>;
template struct WorldStep<true, true, true>;
