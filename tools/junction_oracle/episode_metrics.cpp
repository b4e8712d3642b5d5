// tools/junction_oracle/episode_metrics.cpp -- TEST INFRASTRUCTURE (CPU oracle), see episode_metrics.h.
#include "episode_metrics.h"

#include <cmath>
#include <cstring>
#include <limits>

#include "../../oracle/cshare_spec.h"

namespace metrics {

void init(dp_episode_metrics& m) {
    const double inf = std::numeric_limits<double>::infinity();
    std::memset(&m, 0, sizeof(m));
    m.min_clearance = inf; m.min_lead_gap = inf; m.min_ttc = inf;
    m.max_accel = -inf; m.min_accel = inf;
    m.first_collision_step = -1; m.first_collision_agent = -1;
    m.last_behavior = -1;
}

bool header_valid(const oracle::MapView& m, const dp_scene_hdr& h) {
    return !(h.road_num < 1 || h.road_num > m.d.n_roads || h.lane_num < 1 || h.lane_num > m.lanes_of(h.road_num) ||
             h.lane_num > DP_LANESUM);
}

void update(const junction::JMap& jm, const dp_world_params& wp, const dp_metrics_params& mp, dp_episode_metrics& m, const dp_scene_hdr& h0,
            const dp_scene_hdr& h, const dp_agent* ag, const double* ox, const double* oy, int n_agents, const dp_plan_record& r) {
    const oracle::MapView& mv = jm.m;
    const double inf = std::numeric_limits<double>::infinity();
    // the step's own quantities, as the world step computed them from the header before it
    const double v = h0.velocity, vn = h.velocity, dt = h0.period_ms / 1000.0;
    const int pos = (wp.pre_junction_pts > 0 && (h0.pos == 1 || h0.pos == 2)) ? h0.pos : 0;
    const bool stop_zone = wp.pre_junction_pts <= 0 || (pos == 0 && junction::ego_connector(mv, h0, h0.road_num, h0.lane_num) < 0);
    const bool at_end = stop_zone && h0.id[h0.lane_num - 1] >= mv.lane_size(mv.lane_index(h0.road_num, h0.lane_num)) - wp.end_margin;
    const double ds = at_end ? 0.0 : (v + vn) * 0.5 / 3.6 * dt;
    double c, s;
    spec::spec_sincos_deg(h.dir, &c, &s);
    // ---- the agents in the ego frame ----
    double dmin = inf, gmin = inf, tmin = inf;
    int first = -1;
    bool front = false, rear = false;
    for (int k = 0; k < n_agents; ++k) {
        const double dx = ox[k] - h.x, dy = oy[k] - h.y;
        const double lon = dx * c + dy * s, lat = dy * c - dx * s, alat = std::fabs(lat);
        if (-mp.rear <= lon && lon <= mp.front && -mp.half_width <= lat && lat <= mp.half_width) {
            if (first < 0) first = k;
            if (lon >= 0) front = true;
            else rear = true;
        }
        const double ex = lon > mp.front ? lon - mp.front : (lon < -mp.rear ? -mp.rear - lon : 0.0);
        const double ey = alat > mp.half_width ? alat - mp.half_width : 0.0;
        const double d = std::sqrt(ex * ex + ey * ey);
        if (d < dmin) dmin = d;
        if (lon > mp.front && alat <= mp.corridor_half) {
            const double gap = lon - mp.front;
            const spec::P2 a = mv.pt(ag[k].lane, ag[k].i), b = mv.pt(ag[k].lane, ag[k].i + 1);
            const double ddx = b.x - a.x, ddy = b.y - a.y;
            const double L = std::sqrt(ddx * ddx + ddy * ddy);
            const double va = L == 0 ? 0.0 : ag[k].v * (ddx / L * c + ddy / L * s);
            const double closing = vn / 3.6 - va;
            const double ttc = closing > 0 ? gap / closing : inf;
            if (gap < gmin) gmin = gap;
            if (ttc < tmin) tmin = ttc;
        }
    }
    // ---- the row ----
    const int step_no = m.steps + 1;
    m.distance = m.distance + ds;
    if (dmin < m.min_clearance) m.min_clearance = dmin;
    if (gmin < m.min_lead_gap) m.min_lead_gap = gmin;
    if (tmin < m.min_ttc) m.min_ttc = tmin;
    if (dt > 0) {
        const double a = (vn - v) / 3.6 / dt;
        if (a > m.max_accel) m.max_accel = a;
        if (a < m.min_accel) m.min_accel = a;
        if (m.accel_steps > 0) {
            const double j = std::fabs(a - m.last_accel) / dt;
            if (j > m.max_abs_jerk) m.max_abs_jerk = j;
        }
        m.last_accel = a; m.accel_steps += 1;
    }
    const double le = std::fabs(r.path_lat_dis), de = std::fabs(r.path_dir_err);
    if (le > m.max_abs_lat_err) m.max_abs_lat_err = le;
    if (de > m.max_abs_dir_err) m.max_abs_dir_err = de;
    if (first >= 0) {
        m.collision_steps += 1;
        if (m.first_collision_step < 0) { m.first_collision_step = step_no; m.first_collision_agent = first; }
    }
    if (front) m.collision_steps_front += 1;
    if (rear) m.collision_steps_rear += 1;
    if (tmin < mp.ttc_warn) m.ttc_warn_steps += 1;
    if (vn == 0) m.stopped_steps += 1;
    if (at_end) m.end_stop_steps += 1;
    m.replans += r.afresh_planning; m.aeb_steps += r.acc_flag;
    const int b = r.behavior;
    if (b < 8) m.behavior_steps[b] += 1;
    if (m.steps > 0 && b != m.last_behavior) m.behavior_switches += 1;
    m.last_behavior = b;
    m.steps = step_no;
}

}  // namespace metrics
