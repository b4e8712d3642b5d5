// tools/junction_oracle/v2x_world.h -- TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
//
// Frozen rules of the V2X events in closed-loop episodes (include/dmpp_b200.h section 14), the specification dp_world_v2x_kernel is
// tested against: the data builder, the row and the apply rule, around the handlers of oracle/v2x_oracle.cpp (pinned to the
// unmodified reference by tests/test_v2x.py), called unchanged.  Same discipline as the world step: IEEE binary64, operations in
// the order written, no contraction, GlobalToWGS84 through spec::global_to_wgs84.
//   build  the cycle's dp_v2x_data of one world at cycle k, with the signal state the red-crossing rule carries
//   init   the row of the first launch of an episode
//   cycle  one V2X launch: k < cycles with rec (the handlers on pos 0 headers, the apply rule, the row), or the tally (rec ==
//          nullptr); wp_lat / wp_lng: the whole warning list through GlobalToWGS84
#pragma once
#include "world_junction.h"

namespace v2x {

struct World {
    dp_v2x_data v;
    double d;                          // metres from the ego's point to the stop index on its lane (0 off the approach)
    int state;                         // spat_state: 6 / 7 / 3, 0 without a signal
    bool on, ped_on;                   // on the governed approach (pos 0 / 1); the pedestrian is active
};
World build(const junction::JMap& jm, const dp_params& p, const dp_v2x_event_spec& s, const dp_scene_hdr& h, int k);
void init(dp_v2x_episode_stats& r);
// flags (nullable) receives the flags of a launch with rec (the tally leaves them); a header that names no lane gets zero flags and leaves the row alone
void cycle(const junction::JMap& jm, const dp_params& p, const dp_v2x_world_params& vp, const dp_v2x_event_spec& s, const double* wp_lat,
           const double* wp_lng, const dp_scene_hdr& h, int k, dp_plan_record* rec, dp_v2x_episode_stats& r, dp_v2x_flags* flags);

}  // namespace v2x
