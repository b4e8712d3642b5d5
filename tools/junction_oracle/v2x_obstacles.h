// tools/junction_oracle/v2x_obstacles.h -- TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
//
// Frozen rules of the V2X road users the planner sees (include/dmpp_b200.h section 16), the specification dp_world_obstacles_kernel
// is tested against: the view a cycle runs on and the world's row.  Same discipline as the world step: IEEE binary64, operations
// in the order written, no contraction, the ego frame through spec::spec_sincos_deg, the pedestrian through v2x::pedestrian.
//   init    the row of the first launch of an episode
//   launch  one obstacles launch at cycle k on the world h / ox / oy (max_obs slots): the view into hv / vx / vy (not on the
//           tally; slots at and beyond the view's n_obs are left as they are) and the row; prev = the record of cycle k - 1
//           (nullptr at k == 0); wp_x / wp_y the whole warning list in map coordinates
#pragma once
#include "world_junction.h"

namespace v2xobs {

void init(dp_v2x_obstacle_stats& r);
void launch(const junction::JMap& jm, const dp_v2x_obstacle_params& op, int max_obs, const dp_v2x_event_spec& s, const double* wp_x,
            const double* wp_y, const dp_scene_hdr& h, const double* ox, const double* oy, const dp_plan_record* prev, int k, bool tally,
            dp_scene_hdr* hv, double* vx, double* vy, dp_v2x_obstacle_stats& r);

}  // namespace v2xobs
