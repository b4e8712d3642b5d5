// tools/junction_oracle/lane_change.h -- TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
//
// Frozen arithmetic of the lane-changing agents (include/dmpp_b200.h section 13), the specification the LANECHG instances of the
// world step are tested against.  Same discipline as agent_model.h: IEEE binary64, operations in the order written, no
// contraction, min updates `if (x < m) m = x`.
//   init  the placement step (rec == NULL): st[k] = {agents[k].lat, 0, 0, 0} for k < n, whatever the header names.
//   step  the react phase of agent_model.h and then the lane changes of one scene, in place (ag[k], st[k], k < n), from the state
//         at the start of its step (h0 = the header before the world step); a header that names no lane leaves everything
//         alone.  junction::world_step then runs unchanged.  tw (nullable): the V2X events of v2x_traffic.h join section 12's
//         leader and the leader of at_c and of the safety test on the target lane (when tw->tp.obey); kind_out as agent_model.h.
#pragma once
#include "v2x_traffic.h"
#include "world_junction.h"

namespace lanechg {

void init(const dp_agent* ag, int n, dp_lane_change_state* st);

void step(const junction::JMap& jm, const dp_world_params& wp, const dp_agent_model_params& am, const dp_lane_change_params& lp,
          const dp_scene_hdr& h0, dp_agent* ag, int n, const double* v0, dp_lane_change_state* st, const traffic::World* tw = nullptr,
          int* kind_out = nullptr);

}  // namespace lanechg
