// tools/junction_oracle/v2x_traffic.cpp -- TEST INFRASTRUCTURE (CPU oracle), see v2x_traffic.h.
#include "v2x_traffic.h"

#include <cmath>
#include <cstring>
#include <limits>

#include "v2x_world.h"

namespace traffic {

namespace {
bool governed(const World& w, int l) { return l >= w.gb && l < w.ge; }

// S(l)
double stop_station(const junction::JMap& jm, const World& w, int l) {
    const int off = jm.m.d.lane_pt_off[l], cnt = jm.m.lane_size(l);
    const int stop = w.sig_stop < 0 || w.sig_stop > cnt - 1 ? cnt - 1 : w.sig_stop;
    return jm.cump[off + stop];
}

// the line ds ahead: within look and stoppable within b_commit
bool line_gap(const World& w, const dp_agent_model_params& am, double ds, double v, double* g) {
    if (!(ds <= am.look)) return false;
    const double gg = ds - am.length;
    if (!(gg > 0 && v * v <= 2.0 * w.tp.b_commit * gg)) return false;
    *g = gg;
    return true;
}

// the pedestrian in the frame of segment (i, i + 1) of lane l at offset u
bool frame(const junction::JMap& jm, const World& w, int l, int i, double u, double* lon, double* lat) {
    const spec::P2 Q = jm.m.pt(l, i), R = jm.m.pt(l, i + 1);
    const double dx = R.x - Q.x, dy = R.y - Q.y, L = std::sqrt(dx * dx + dy * dy);
    if (!(L > 0)) return false;
    const double q = u / L, Px = Q.x + q * dx, Py = Q.y + q * dy, tx = dx / L, ty = dy / L;
    const double ex = w.px - Px, ey = w.py - Py;
    *lon = ex * tx + ey * ty; *lat = ey * tx - ex * ty;
    return true;
}

bool ped_gap(const junction::JMap& jm, const World& w, const dp_agent_model_params& am, int l, int i, double u, double* g) {
    double lon, lat;
    if (!w.ped_on || !frame(jm, w, l, i, u, &lon, &lat)) return false;
    if (!(0 < lon && lon <= am.look && std::fabs(lat) <= w.tp.ped_half_width)) return false;
    *g = lon - am.length;
    return true;
}
}  // namespace

World world(const junction::JMap& jm, const dp_v2x_traffic_params& tp, const dp_v2x_event_spec& s, const dp_scene_hdr& h0, int k) {
    World w;
    const double t = (double)k * h0.period_ms / 1000.0;
    const int state = v2x::signal_state(s, t);
    w.line = state == 7 || state == 3; w.red = state == 3;
    if (s.sig_road > 0) { w.gb = jm.m.d.road_lane_base[s.sig_road - 1]; w.ge = jm.m.d.road_lane_base[s.sig_road]; w.sig_stop = s.sig_stop; }
    w.ped_on = v2x::pedestrian(s, t, &w.px, &w.py);
    w.tp = tp;
    return w;
}

int leader(const junction::JMap& jm, const World& w, const dp_agent_model_params& am, int l0, int l1, int l2, double D1, double D2, double sk,
           double v, int i, double u, bool* lead, double* best) {
    int kind = 0;
    double g;
    if (w.line) {                                           // the first governed lane of the chain decides
        double ds = 0;
        bool have = false;
        if (governed(w, l0)) {
            const double S = stop_station(jm, w, l0);
            if (S > sk) { ds = S - sk; have = true; }
        } else if (l1 >= 0 && governed(w, l1)) { ds = D1 + stop_station(jm, w, l1); have = true; }
        else if (l2 >= 0 && governed(w, l2)) { ds = D2 + stop_station(jm, w, l2); have = true; }
        if (have && line_gap(w, am, ds, v, &g) && (!*lead || g < *best)) { *best = g; *lead = true; kind = 1; }
    }
    if (ped_gap(jm, w, am, l0, i, u, &g) && (!*lead || g < *best)) { *best = g; *lead = true; kind = 2; }
    return kind;
}

bool side(const junction::JMap& jm, const World& w, const dp_agent_model_params& am, int m, int im, double sm, double u, double v, bool* lead,
          double* g) {
    bool won = false;
    double c;
    if (w.line && governed(w, m)) {
        const double S = stop_station(jm, w, m);
        if (S > sm && line_gap(w, am, S - sm, v, &c) && (!*lead || c < *g)) { *g = c; *lead = won = true; }
    }
    if (ped_gap(jm, w, am, m, im, u, &c) && (!*lead || c < *g)) { *g = c; *lead = won = true; }
    return won;
}

void init(dp_v2x_traffic_stats& r) {
    std::memset(&r, 0, sizeof(r));
    r.min_ped_dist = std::numeric_limits<double>::infinity();
}

void update(const junction::JMap& jm, const World& w, const dp_agent_model_params& am, double vehicle_width, dp_v2x_traffic_stats& r,
            const dp_agent* a1, const dp_agent* a2, const double* ox, const double* oy, int n, int line_n, int ped_n) {
    const int* po = jm.m.d.lane_pt_off;
    for (int k = 0; k < n; ++k) {
        const int l = a1[k].lane;
        if (w.red && governed(w, l)) {
            const double S = stop_station(jm, w, l), s1 = jm.cump[po[l] + a1[k].i] + a1[k].u;
            if (s1 < S && (a2[k].lane != l || jm.cump[po[l] + a2[k].i] + a2[k].u >= S)) r.red_runs += 1;
        }
        if (w.ped_on) {
            double lon, lat;
            if (frame(jm, w, a2[k].lane, a2[k].i, a2[k].u, &lon, &lat) && 0 <= lon && lon <= am.length && std::fabs(lat) <= vehicle_width / 2.0)
                r.ped_hits += 1;
            const double dx = ox[k] - w.px, dy = oy[k] - w.py, d = std::sqrt(dx * dx + dy * dy);
            if (d < r.min_ped_dist) r.min_ped_dist = d;
        }
    }
    r.line_steps += line_n; r.ped_steps += ped_n;
}

}  // namespace traffic
