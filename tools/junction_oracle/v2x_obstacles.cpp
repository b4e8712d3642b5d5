// tools/junction_oracle/v2x_obstacles.cpp -- TEST INFRASTRUCTURE (CPU oracle), see v2x_obstacles.h.
#include "v2x_obstacles.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>

#include "episode_metrics.h"
#include "v2x_world.h"
#include "../../oracle/cshare_spec.h"

namespace v2xobs {

namespace {
// section 11's box at the header's pose: inside?  *d = the clearance
bool box_point(const dp_v2x_obstacle_params& op, const dp_scene_hdr& h, double c, double s, double ox, double oy, double* d) {
    const double dx = ox - h.x, dy = oy - h.y;
    const double lon = dx * c + dy * s, lat = dy * c - dx * s, alat = std::fabs(lat);
    const double ex = lon > op.front ? lon - op.front : (lon < -op.rear ? -op.rear - lon : 0.0);
    const double ey = alat > op.half_width ? alat - op.half_width : 0.0;
    *d = std::sqrt(ex * ex + ey * ey);
    return -op.rear <= lon && lon <= op.front && -op.half_width <= lat && lat <= op.half_width;
}
bool in_range(double range, const dp_scene_hdr& h, double px, double py) {
    const double dx = px - h.x, dy = py - h.y;
    return std::sqrt(dx * dx + dy * dy) <= range;
}
}  // namespace

void init(dp_v2x_obstacle_stats& r) {
    std::memset(&r, 0, sizeof(r));
    r.min_ped_clearance = std::numeric_limits<double>::infinity();
    r.min_works_clearance = std::numeric_limits<double>::infinity();
    r.first_ped_hit = -1; r.first_works_hit = -1;
    r.last_ped_slot = -1;
}

void launch(const junction::JMap& jm, const dp_v2x_obstacle_params& op, int max_obs, const dp_v2x_event_spec& s, const double* wp_x,
            const double* wp_y, const dp_scene_hdr& h, const double* ox, const double* oy, const dp_plan_record* prev, int k, bool tally,
            dp_scene_hdr* hv, double* vx, double* vy, dp_v2x_obstacle_stats& r) {
    if (k == 0) init(r);
    const int na = std::min((int)h.n_obs, max_obs);
    if (!tally) {                                       // the plain copy; a header that names a lane then gets its points appended
        *hv = h;
        std::copy(ox, ox + na, vx); std::copy(oy, oy + na, vy);
    }
    if (!metrics::header_valid(jm.m, h)) return;
    const double t = (double)k * h.period_ms / 1000.0;
    double c, sn;
    spec::spec_sincos_deg(h.dir, &c, &sn);
    if (prev && prev->ob_flag) {
        const int oi = prev->ob_index;
        if (r.last_ped_slot >= 0 && oi == r.last_ped_slot) r.ped_bound_cycles += 1;
        if (oi >= r.last_works_first && oi < r.last_works_end) r.works_bound_cycles += 1;
    }
    double px = 0, py = 0, d;
    const bool ped_on = v2x::pedestrian(s, t, &px, &py);
    if (ped_on) {
        if (box_point(op, h, c, sn, px, py, &d)) { r.ped_hits += 1; if (r.first_ped_hit < 0) r.first_ped_hit = k; }
        if (d < r.min_ped_clearance) r.min_ped_clearance = d;
    }
    if (s.has_works) {
        bool hit = box_point(op, h, c, sn, s.rw_x, s.rw_y, &d);
        if (d < r.min_works_clearance) r.min_works_clearance = d;
        for (int i = 0; i < s.wp_count; ++i) {
            hit = box_point(op, h, c, sn, wp_x[s.wp_first + i], wp_y[s.wp_first + i], &d) || hit;
            if (d < r.min_works_clearance) r.min_works_clearance = d;
        }
        if (hit) { r.works_hits += 1; if (r.first_works_hit < 0) r.first_works_hit = k; }
    }
    if (tally) return;
    int cnt = na, ped_slot = -1, dropped = 0;
    auto put = [&](double x, double y) {
        if (cnt < max_obs) { vx[cnt] = x; vy[cnt] = y; ++cnt; return true; }
        ++dropped;
        return false;
    };
    if ((op.what & 1) && ped_on && in_range(op.range, h, px, py) && put(px, py)) ped_slot = cnt - 1;
    const int wf = cnt;
    if (s.has_works) {
        if ((op.what & 2) && in_range(op.range, h, s.rw_x, s.rw_y)) put(s.rw_x, s.rw_y);
        if (op.what & 4)
            for (int i = 0; i < s.wp_count; ++i)
                if (in_range(op.range, h, wp_x[s.wp_first + i], wp_y[s.wp_first + i])) put(wp_x[s.wp_first + i], wp_y[s.wp_first + i]);
    }
    r.views += 1; r.ped_cycles += ped_slot >= 0; r.works_cycles += cnt > wf; r.dropped += dropped;
    r.last_ped_slot = ped_slot; r.last_works_first = wf; r.last_works_end = cnt;
    if (cnt > na) hv->n_obs = (uint16_t)cnt;
}

}  // namespace v2xobs
