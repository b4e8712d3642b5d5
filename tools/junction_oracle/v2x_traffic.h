// tools/junction_oracle/v2x_traffic.h -- TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
//
// Frozen arithmetic of the agents that obey the V2X events (include/dmpp_b200.h section 15), the specification the TRAFFIC
// instances of the world step are tested against.  Same discipline as agent_model.h: IEEE binary64, operations in the order
// written, no contraction, min updates `if (x < m) m = x`.
//   world    the events of one world at the world step of cycle k (h0 = the header before the step): section 14's signal state
//            and pedestrian (v2x_world.h), the governed lanes, the parameters
//   leader   section 12's extra candidates of one agent, after its vehicle scan: the line, then the pedestrian, each replacing
//            (lead, best) with `if (!lead || g < best)`; returns the kind that leads in the end (0 a vehicle or none, 1 the line,
//            2 the pedestrian).  agents::react applies it when obey, and counts it either way
//   side     the same two candidates on section 13's target lane m at (i_m, s_m, u); lanechg::step's side() uses the result for
//            at_c and the safety test when obey
//   update   the row after the motion of section 9: a1 = the agents as the motion started (after the lane changes), a2 / ox / oy
//            = after it, line_n / ped_n = the step's counts of the leader kinds
#pragma once
#include "world_junction.h"

namespace traffic {

struct World {
    double px = 0, py = 0;             // the pedestrian (ped_on)
    int gb = 0, ge = 0;                // the governed lanes [gb, ge)
    int sig_stop = -1;
    bool line = false, red = false, ped_on = false;   // line: state 7 or 3; red: state 3
    dp_v2x_traffic_params tp{};
};

World world(const junction::JMap& jm, const dp_v2x_traffic_params& tp, const dp_v2x_event_spec& s, const dp_scene_hdr& h0, int k);
int leader(const junction::JMap& jm, const World& w, const dp_agent_model_params& am, int l0, int l1, int l2, double D1, double D2, double sk,
           double v, int i, double u, bool* lead, double* best);
bool side(const junction::JMap& jm, const World& w, const dp_agent_model_params& am, int m, int im, double sm, double u, double v, bool* lead,
          double* g);
void init(dp_v2x_traffic_stats& r);
void update(const junction::JMap& jm, const World& w, const dp_agent_model_params& am, double vehicle_width, dp_v2x_traffic_stats& r,
            const dp_agent* a1, const dp_agent* a2, const double* ox, const double* oy, int n, int line_n, int ped_n);

}  // namespace traffic
