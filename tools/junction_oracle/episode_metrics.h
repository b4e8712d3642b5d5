// tools/junction_oracle/episode_metrics.h -- TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
//
// Frozen arithmetic of the closed-loop episode metrics (include/dmpp_b200.h section 11), the specification the armed world-step
// kernels are tested against.  Same discipline as the world step: IEEE binary64, operations in the order written, no contraction,
// min / max updates `if (x < m) m = x` / `if (x > m) m = x`, the ego frame through spec::spec_sincos_deg.
//   init    the row of a placement step (rec == NULL), whatever the header names
//   update  one step: h0 = the header before the world step, h = after it, agents / ox / oy after it, r = the record it applied
#pragma once
#include "world_junction.h"

namespace metrics {

void init(dp_episode_metrics& m);
void update(const junction::JMap& jm, const dp_world_params& wp, const dp_metrics_params& mp, dp_episode_metrics& m, const dp_scene_hdr& h0,
            const dp_scene_hdr& h, const dp_agent* ag, const double* ox, const double* oy, int n_agents, const dp_plan_record& r);
// the kernel's test: a header that names a lane of the map (others leave world and row alone)
bool header_valid(const oracle::MapView& m, const dp_scene_hdr& h);

}  // namespace metrics
