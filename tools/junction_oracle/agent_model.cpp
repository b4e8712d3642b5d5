// tools/junction_oracle/agent_model.cpp -- TEST INFRASTRUCTURE (CPU oracle), see agent_model.h.
#include "agent_model.h"

#include <cmath>
#include <limits>
#include <vector>

#include "episode_metrics.h"

namespace agents {

double lane_len(const junction::JMap& jm, int gl) { return jm.cump[jm.m.d.lane_pt_off[gl + 1] - 1]; }

int ego_lane(const junction::JMap& jm, const dp_world_params& wp, const dp_scene_hdr& h0, double* se) {
    const oracle::MapView& m = jm.m;
    const int pos = (wp.pre_junction_pts > 0 && (h0.pos == 1 || h0.pos == 2)) ? h0.pos : 0;
    int le = -1, idx = 0;
    if (pos != 2) { le = m.lane_index(h0.road_num, h0.lane_num); idx = h0.id[h0.lane_num - 1]; }
    else if (h0.conn >= 0 && h0.conn < m.d.n_conn && h0.last_lanenum >= 1 && h0.last_lanenum <= DP_LANESUM) {
        le = m.d.conn[h0.conn].lane; idx = h0.id[h0.last_lanenum - 1];
    }
    *se = 0;
    if (le >= 0) {
        const int cnt = m.lane_size(le);
        if (idx > cnt - 1) idx = cnt - 1;
        if (idx < 0) idx = 0;
        *se = jm.cump[m.d.lane_pt_off[le] + idx];
    }
    return le;
}

void react(const junction::JMap& jm, const dp_world_params& wp, const dp_agent_model_params& mp, const dp_scene_hdr& h0, dp_agent* ag,
           int n, const double* v0, double* acc_out) {
    const oracle::MapView& m = jm.m;
    if (!metrics::header_valid(m, h0)) return;
    const double inf = std::numeric_limits<double>::infinity();
    const double dt = h0.period_ms / 1000.0;
    // the start-of-step state of every agent
    std::vector<double> S(n), V(n);
    std::vector<int> L(n);
    for (int k = 0; k < n; ++k) {
        S[k] = jm.cump[m.d.lane_pt_off[ag[k].lane] + ag[k].i] + ag[k].u;
        V[k] = ag[k].v; L[k] = ag[k].lane;
    }
    // the ego: lane, station, speed
    double se = 0;
    const int le = ego_lane(jm, wp, h0, &se);
    const double ve = h0.velocity / 3.6;
    for (int k = 0; k < n; ++k) {
        const double vd = v0[k];
        if (!(vd > 0)) continue;
        const double sk = S[k], v = V[k];
        const int l0 = L[k], l1 = jm.next[l0], l2 = l1 >= 0 ? jm.next[l1] : -1;
        const double D1 = lane_len(jm, l0) - sk;
        const double D2 = l1 >= 0 ? D1 + lane_len(jm, l1) : 0.0;
        // the leader: smallest gap, the ego first on a tie, then the lowest agent index
        double best = inf, vl = 0;
        bool lead = false;
        if (le >= 0) {
            double ds = inf;
            if (le == l0 && se >= sk) ds = se - sk;
            if (le == l1) { const double c = D1 + se; if (c < ds) ds = c; }
            if (l2 >= 0 && le == l2) { const double c = D2 + se; if (c < ds) ds = c; }
            if (ds <= mp.look) { best = ds - mp.ego_rear; vl = ve; lead = true; }
        }
        for (int j = 0; j < n; ++j) {
            double ds = inf;
            if (L[j] == l0 && (S[j] > sk || (S[j] == sk && j > k))) ds = S[j] - sk;
            if (L[j] == l1) { const double c = D1 + S[j]; if (c < ds) ds = c; }
            if (l2 >= 0 && L[j] == l2) { const double c = D2 + S[j]; if (c < ds) ds = c; }
            if (ds <= mp.look) {
                const double g = ds - mp.length;
                if (!lead || g < best) { best = g; vl = V[j]; lead = true; }
            }
        }
        // IDM, delta = 4
        const double r = v / vd;
        double fr = r * r;
        fr = fr * fr;
        double acc;
        if (lead) {
            const double dv = v - vl;
            double z = v * mp.T + v * dv / (2.0 * std::sqrt(mp.a_max * mp.b));
            if (z < 0) z = 0;
            const double ss = mp.s0 + z;
            if (best > 0) { const double q = ss / best; acc = mp.a_max * (1.0 - fr - q * q); }
            else acc = -mp.b_max;
        } else acc = mp.a_max * (1.0 - fr);
        if (acc < -mp.b_max) acc = -mp.b_max;
        if (acc_out) acc_out[k] = acc;
        double vn = v + acc * dt;
        if (vn < 0) vn = 0;
        ag[k].v = vn;
    }
}

}  // namespace agents
