// csrc/dp_world_v2x.cu -- the V2X launch of a closed-loop episode (include/dmpp_b200.h section 14): one warp per world builds
// the cycle's dp_v2x_data from the world's event specification and its header, runs the handlers of dp_v2x.cuh on it, and lane
// 0 applies the flags to the cycle's record and updates the world's row.  Rules frozen in tools/junction_oracle/v2x_world.h
// (IEEE binary64, -fmad=false, operations in that order).  A translation unit of its own: the world-step instances of
// dp_world*.cu compile to what they compiled to before.
#include "dp_world_step.cuh"
#include "dp_v2x.cuh"

static_assert(sizeof(dp_v2x_event_spec) == 160, "dp_v2x_event_spec is 160 bytes");
static_assert(sizeof(dp_v2x_episode_stats) == 80, "dp_v2x_episode_stats is 80 bytes");

namespace {
// the warning list in map coordinates, read through GlobalToWGS84 as the handlers expect it
struct V2xWpGlobal {
    const double* __restrict__ x; const double* __restrict__ y;
    double lat0, lng0, k_lat, k_lng;
    __device__ __forceinline__ double lat(int i) const { return fma(y[i], k_lat, lat0); }
    __device__ __forceinline__ double lng(int i) const { return fma(x[i], k_lng, lng0); }
};

// the cycle's V2X inputs of one world, and the signal state the red-crossing rule carries.  Every lane builds the same values
// (scalar work on broadcast loads), so the handlers need no shuffle of the inputs.
struct V2xWorld { dp_v2x_data v; double d; int state; bool on, ped_on; };
__device__ __forceinline__ V2xWorld v2x_world_data(const DevMap& m, const dp_params& p, const dp_v2x_event_spec& s, const dp_scene_hdr& h, int k) {
    const double t = v2x_time(k, h);
    V2xWorld w;
    dp_v2x_data& v = w.v;
    w.state = v2x_signal_state(s, t);
    w.on = s.sig_road > 0 && h.road_num == s.sig_road && h.pos != 2;
    w.d = 0;
    if (w.on) {
        const int gl = m.road_lane_base[h.road_num - 1] + h.lane_num - 1;
        const int off = m.lane_pt_off[gl], cnt = m.lane_pt_off[gl + 1] - off;
        const int stop = s.sig_stop < 0 || s.sig_stop > cnt - 1 ? cnt - 1 : s.sig_stop;
        int i = h.id[h.lane_num - 1];
        if (i > cnt - 1) i = cnt - 1;
        if (i < 0) i = 0;
        w.d = m.cump[off + stop] - m.cump[off + i];
    }
    v.spat_state = w.state;
    v.spat_lane_occupied = (w.on && w.d >= 0 && w.d <= s.sig_range) ? 1 : 0;
    double px, py;
    w.ped_on = v2x_pedestrian(s, t, &px, &py);
    v.ped_distance = 0; v.ped_lat = 0; v.ped_lng = 0;
    if (w.ped_on) {
        const double dx = px - h.x, dy = py - h.y;
        v.ped_distance = sqrt(dx * dx + dy * dy);
        v.ped_lat = fma(py, p.k_lat, p.lat0); v.ped_lng = fma(px, p.k_lng, p.lng0);
    }
    v.ped_direction = s.ped_direction;
    v.rsi_lat = 0; v.rsi_lng = 0; v.wp_first = 0; v.wp_count = 0;
    bool near_works = false;
    if (s.has_works) {
        if (s.rw_rsi) { v.rsi_lat = fma(s.rw_y, p.k_lat, p.lat0); v.rsi_lng = fma(s.rw_x, p.k_lng, p.lng0); }
        v.wp_first = s.wp_first; v.wp_count = s.wp_count;
        const double dx = s.rw_x - h.x, dy = s.rw_y - h.y;
        near_works = sqrt(dx * dx + dy * dy) <= s.rw_range;
    }
    v.ego_lat = fma(h.y, p.k_lat, p.lat0); v.ego_lng = fma(h.x, p.k_lng, p.lng0);
    v.warn_status = (w.ped_on && v.ped_distance <= s.ped_range) ? 5 : w.on ? 3 : near_works ? 4 : 0;
    return w;
}

__device__ __forceinline__ void v2x_stats_init(dp_v2x_episode_stats& r) {
    r.min_ped_distance = __longlong_as_double(0x7ff0000000000000LL); r.last_d = 0;
    r.cycles = 0;
    for (int i = 0; i < 3; ++i) r.light_cycles[i] = 0;
    for (int i = 0; i < 2; ++i) { r.construction_cycles[i] = 0; r.pedestrian_cycles[i] = 0; }
    r.stop_cmds = 0; r.creep_cmds = 0; r.ub_cycles = 0;
    r.red_crossings = 0; r.first_red_crossing = -1;
    r.last_phase = 0; r.last_on = 0; r.pad = 0;
}

// k: the cycle; rec == nullptr: the tally after the last world step (closes the red-crossing check, runs no handler)
__global__ void __launch_bounds__(WPB * 32) dp_world_v2x_kernel(DevMap m, dp_params p, dp_v2x_world_params vp, int n, int k,
                                                                const dp_scene_hdr* __restrict__ hdr, dp_plan_record* __restrict__ rec,
                                                                const dp_v2x_event_spec* __restrict__ spec, const double* __restrict__ wp_x,
                                                                const double* __restrict__ wp_y, dp_v2x_flags* __restrict__ flags,
                                                                dp_v2x_episode_stats* __restrict__ stats) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int scene = blockIdx.x * WPB + wib;
    if (scene >= n) return;
    const dp_scene_hdr& h = hdr[scene];
    dp_v2x_flags f;
    f.light_flag = 0; f.construction_flag = 0; f.pedestrian_flag = 0; f.ub = 0; f.pad[0] = f.pad[1] = f.pad[2] = 0;
    f.lng_distance = 9999; f.lat_distance = 9999;
    if (k == 0 && lane == 0) v2x_stats_init(stats[scene]);   // the first launch of an episode starts a clean row
    // a header that does not name a lane of the map (device-pointer callers are not validated on the host): zero flags, row alone
    if (h.road_num < 1 || h.road_num > m.n_roads || h.lane_num < 1 ||
        h.lane_num > m.road_lane_base[h.road_num] - m.road_lane_base[h.road_num - 1] || h.lane_num > DP_LANESUM) {
        if (lane == 0 && flags && rec) flags[scene] = f;
        return;
    }
    const dp_v2x_event_spec& s = spec[scene];
    const V2xWorld w = v2x_world_data(m, p, s, h, k);
    const bool run = rec != nullptr && h.pos == 0;          // SegmentDecision is the handlers' only caller (Decision.cpp:283)
    if (run) f = v2x_handlers(m, p, h, w.v, V2xWpGlobal{wp_x, wp_y, p.lat0, p.lng0, p.k_lat, p.k_lng}, vp.mode, lane);
    if (lane != 0) return;
    dp_v2x_episode_stats r = stats[scene];
    if (r.last_on && r.last_d >= 0 && r.last_phase == 3 && (!w.on || w.d < 0)) {   // the step that ended here crossed on red
        r.red_crossings += 1;
        if (r.first_red_crossing < 0) r.first_red_crossing = k - 1;
    }
    if (rec != nullptr) {
        if (w.ped_on && w.v.ped_distance < r.min_ped_distance) r.min_ped_distance = w.v.ped_distance;
        if (run) {
            dp_plan_record& rc = rec[scene];
            const bool stop = f.pedestrian_flag || f.light_flag == 1;
            const bool creep = !stop && f.construction_flag && rc.brakespeed > 3.0;
            r.cycles += 1;
            for (int i = 0; i < 3; ++i) r.light_cycles[i] += f.light_flag == i;        // (unrolled: the row stays in registers)
            for (int i = 0; i < 2; ++i) {
                r.construction_cycles[i] += f.construction_flag == i; r.pedestrian_cycles[i] += f.pedestrian_flag == i;
            }
            r.stop_cmds += stop; r.creep_cmds += creep; r.ub_cycles += f.ub;
            if (vp.apply) v2x_apply_rule(f, rc);
        }
        r.last_d = w.d; r.last_phase = w.state; r.last_on = w.on;
    }
    stats[scene] = r;
    if (flags && rec) flags[scene] = f;              // (the tally leaves the last cycle's flags)
}
}  // namespace

cudaError_t dp_launch_world_v2x(const DevMap& m, const dp_params& p, const DpV2xOpts& o, int n, const dp_scene_hdr* hdr, dp_plan_record* rec,
                                int cycle, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_world_v2x_kernel<<<(n + WPB - 1) / WPB, WPB * 32, 0, st>>>(m, p, o.vp, n, cycle, hdr, rec, o.spec, o.wp_x, o.wp_y, o.flags, o.stats);
    return cudaGetLastError();
}
