// tools/junction_oracle/world_junction.h -- TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
//
// Frozen arithmetic of the world step of the closed-loop episode runner WITH junction transitions (include/dmpp_b200.h
// section 9, dp_world_params.pre_junction_pts = J > 0), the specification dp_world_kernel<true> is tested against.  With J <= 0
// world_step is oracle::world_step (oracle/world_spec.cpp), the segment-only step, called as it is.  Same arithmetic discipline as
// oracle/: IEEE binary64, operations in the order written, no contraction, headings through spec::calc_global_dir.
//
// Compares as frozen here (J > 0):
//   every nearest-point search is the localisation's (squared distance, strict '<', lowest index wins, window clipped to the lane);
//   0 -> 1  ego connector c >= 0 and the NEW id[lane_num-1] >= lane_size - 1 - J (after this step's localisation, also when
//           rec == nullptr);
//   1 -> 2  d2(connector, [0, loc_fwd]) <  d2(approach road, windows around id[]) -- a tie stays in pos 1;
//   2 -> 0  d2(departure road, [0, loc_fwd] on every lane) <  d2(connector, id[last_lanenum-1] window) -- a tie stays in pos 2;
//   at most one transition per step; the ego's speed and walk do not depend on pos except through the end_margin stop;
//   agents: u < L of a lane's last segment stays on it, u >= L moves to the successor with u - L (at most 8 successors per step).
#pragma once
#include <vector>
#include "../../include/dmpp_b200.h"
#include "../../oracle/planner_oracle.h"

namespace junction {

// the map view of oracle/ plus lane_next of dp_map_upload: the successor of every lane, -1 none; and its cump: per point i of a
// lane, the segment lengths sqrt(dx*dx + dy*dy) of points 0 .. i-1 added in index order (dp_map_prep_kernel)
struct JMap {
    oracle::MapView m;
    std::vector<int> next;
    std::vector<double> cump;
    void set(const dp_map_desc& d);
};

// the ego's connector (include/dmpp_b200.h section 9): lowest c leaving (road, lane) towards h.next_roadnum, -1 none
int ego_connector(const oracle::MapView& m, const dp_scene_hdr& h, int road, int lane);

// one world step of one scene; rec == nullptr: place the agents and localise only (and the 0 -> 1 / 1 -> 2 / 2 -> 0 rules).
// last_x / last_y: the carried local path (road_points of the cycle that produced rec).
void world_step(const JMap& m, const dp_params& p, const dp_world_params& wp, dp_scene_hdr& h, dp_agent* agents, double* ox,
                double* oy, const dp_plan_record* rec, const double* last_x, const double* last_y);

}  // namespace junction
