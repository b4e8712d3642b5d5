// tools/junction_oracle/v2x_world.cpp -- TEST INFRASTRUCTURE (CPU oracle), see v2x_world.h.
#include "v2x_world.h"

#include <cmath>
#include <cstring>
#include <limits>

#include "episode_metrics.h"
#include "../../oracle/cshare_spec.h"
#include "../../oracle/v2x_oracle.h"

namespace v2x {

namespace {
void gps(const dp_params& p, double x, double y, double* lat, double* lng) {
    spec::global_to_wgs84(spec::Datum{p.lat0, p.lng0, p.k_lat, p.k_lng}, x, y, lat, lng);
}
}  // namespace

int signal_state(const dp_v2x_event_spec& s, double t) {
    int state = 0;
    if (s.sig_road > 0) {
        double ph = std::fmod(t + s.sig_offset, s.sig_cycle);
        if (ph < 0) ph += s.sig_cycle;
        state = ph < s.sig_green ? 6 : (ph < s.sig_green + s.sig_yellow ? 7 : 3);
    }
    return state;
}

bool pedestrian(const dp_v2x_event_spec& s, double t, double* px, double* py) {
    const bool on = s.has_ped && s.ped_t_on <= t && t <= s.ped_t_off;
    if (on) {
        const double tp = t - s.ped_t_on;
        *px = s.ped_x + s.ped_vx * tp; *py = s.ped_y + s.ped_vy * tp;
    }
    return on;
}

World build(const junction::JMap& jm, const dp_params& p, const dp_v2x_event_spec& s, const dp_scene_hdr& h, int k) {
    const oracle::MapView& m = jm.m;
    const double t = (double)k * h.period_ms / 1000.0;
    World w;
    std::memset(&w, 0, sizeof(w));
    dp_v2x_data& v = w.v;
    w.state = signal_state(s, t);
    w.on = s.sig_road > 0 && h.road_num == s.sig_road && h.pos != 2;
    if (w.on) {
        const int gl = m.lane_index(h.road_num, h.lane_num), off = m.d.lane_pt_off[gl], cnt = m.lane_size(gl);
        const int stop = s.sig_stop < 0 || s.sig_stop > cnt - 1 ? cnt - 1 : s.sig_stop;
        int i = h.id[h.lane_num - 1];
        if (i > cnt - 1) i = cnt - 1;
        if (i < 0) i = 0;
        w.d = jm.cump[off + stop] - jm.cump[off + i];
    }
    v.spat_state = w.state;
    v.spat_lane_occupied = (w.on && w.d >= 0 && w.d <= s.sig_range) ? 1 : 0;
    double px = 0, py = 0;
    w.ped_on = pedestrian(s, t, &px, &py);
    if (w.ped_on) {
        const double dx = px - h.x, dy = py - h.y;
        v.ped_distance = std::sqrt(dx * dx + dy * dy);
        gps(p, px, py, &v.ped_lat, &v.ped_lng);
    }
    v.ped_direction = s.ped_direction;
    bool near_works = false;
    if (s.has_works) {
        if (s.rw_rsi) gps(p, s.rw_x, s.rw_y, &v.rsi_lat, &v.rsi_lng);
        v.wp_first = s.wp_first; v.wp_count = s.wp_count;
        const double dx = s.rw_x - h.x, dy = s.rw_y - h.y;
        near_works = std::sqrt(dx * dx + dy * dy) <= s.rw_range;
    }
    gps(p, h.x, h.y, &v.ego_lat, &v.ego_lng);
    v.warn_status = (w.ped_on && v.ped_distance <= s.ped_range) ? 5 : w.on ? 3 : near_works ? 4 : 0;
    return w;
}

void init(dp_v2x_episode_stats& r) {
    std::memset(&r, 0, sizeof(r));
    r.min_ped_distance = std::numeric_limits<double>::infinity();
    r.first_red_crossing = -1;
}

void cycle(const junction::JMap& jm, const dp_params& p, const dp_v2x_world_params& vp, const dp_v2x_event_spec& s, const double* wp_lat,
           const double* wp_lng, const dp_scene_hdr& h, int k, dp_plan_record* rec, dp_v2x_episode_stats& r, dp_v2x_flags* flags) {
    dp_v2x_flags f;
    std::memset(&f, 0, sizeof(f));
    f.lng_distance = 9999; f.lat_distance = 9999;
    if (k == 0) init(r);
    if (!metrics::header_valid(jm.m, h)) {
        if (flags && rec) *flags = f;
        return;
    }
    const World w = build(jm, p, s, h, k);
    const bool run = rec != nullptr && h.pos == 0;
    if (run) oracle::v2x_event(jm.m, p, h, w.v, wp_lat, wp_lng, vp.mode, &f);
    if (r.last_on && r.last_d >= 0 && r.last_phase == 3 && (!w.on || w.d < 0)) {
        r.red_crossings += 1;
        if (r.first_red_crossing < 0) r.first_red_crossing = k - 1;
    }
    if (rec) {
        if (w.ped_on && w.v.ped_distance < r.min_ped_distance) r.min_ped_distance = w.v.ped_distance;
        if (run) {
            const bool stop = f.pedestrian_flag || f.light_flag == 1;
            const bool creep = !stop && f.construction_flag && rec->brakespeed > 3.0;
            r.cycles += 1;
            r.light_cycles[f.light_flag] += 1; r.construction_cycles[f.construction_flag] += 1; r.pedestrian_cycles[f.pedestrian_flag] += 1;
            r.stop_cmds += stop; r.creep_cmds += creep; r.ub_cycles += f.ub;
            if (vp.apply) oracle::v2x_apply(f, *rec);
        }
        r.last_d = w.d; r.last_phase = w.state; r.last_on = w.on;
    }
    if (flags && rec) *flags = f;
}

}  // namespace v2x
