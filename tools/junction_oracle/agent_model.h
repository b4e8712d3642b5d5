// tools/junction_oracle/agent_model.h -- TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
//
// Frozen arithmetic of the reactive agents (include/dmpp_b200.h section 12), the specification the REACT instances of the world
// step are tested against.  Same discipline as the world step: IEEE binary64, operations in the order written, no contraction,
// min updates `if (x < m) m = x`.
//   react  rewrite ag[k].v, k < n, of one scene from the state at the start of its step (h0 = the header before the world step,
//          every agent reading the old state of the others), on a header that names a lane; then junction::world_step runs
//          unchanged.  v0[k]: the desired speeds of the scene.  acc_out (nullable): acc_out[k] = agent k's clamped IDM
//          acceleration, for the agents that react (v0[k] > 0; the lane changes of lane_change.h start from it).
#pragma once
#include "world_junction.h"

namespace agents {

// the ego as a candidate (section 12): its lane (-1: none) and, in *se, its station
int ego_lane(const junction::JMap& jm, const dp_world_params& wp, const dp_scene_hdr& h0, double* se);
// len(gl): the last entry of the lane's cump
double lane_len(const junction::JMap& jm, int gl);

void react(const junction::JMap& jm, const dp_world_params& wp, const dp_agent_model_params& mp, const dp_scene_hdr& h0, dp_agent* ag,
           int n, const double* v0, double* acc_out = nullptr);

}  // namespace agents
