// csrc/dp_world_traffic.cu -- the world step whose agents obey the V2X events (include/dmpp_b200.h section 15, on top of the
// reactive agents of section 12 and the V2X events of section 14): the TRAFFIC = true instances of dp_world_kernel
// (dp_world_step.cuh), with and without junctions, episode metrics and lane changes, in a translation unit of their own so that
// the other instances stay what they were.
#include "dp_world_step.cuh"

template struct WorldStep<false, true, false, true>;
template struct WorldStep<true, true, false, true>;
template struct WorldStep<false, true, true, true>;
template struct WorldStep<true, true, true, true>;
