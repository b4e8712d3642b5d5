// csrc/dp_v2x.cuh -- the V2X event handlers (Decision.cpp:1824-2434) as one warp-wide device function, and the opt-in apply
// rule of include/dmpp_b200.h section 10.  Two kernels call them: dp_v2x_kernel (dp_world.cu), the batch operator of section 10,
// and dp_world_v2x_kernel (dp_world_v2x.cu), the V2X launch of a closed-loop episode (section 14).  Control flow is warp-uniform,
// the nearest-point and minimum-distance scans over the <= 200 map points ahead are lane-parallel.  Quirks: see
// oracle/v2x_oracle.cpp.
#pragma once
#include "dp_kernels.h"

namespace {
struct V2xPath { const double2* p; const double* len; int n; };   // a slice of a map lane: points, segment lengths (p[i] -> p[i+1])
__device__ __forceinline__ V2xPath v2x_front(const DevMap& m, int gl, int id, int first_off) {
    const int off = m.lane_pt_off[gl], cnt = m.lane_pt_off[gl + 1] - off;
    const int a = min(cnt, id + first_off), b = min(cnt, id + 200 + first_off);
    V2xPath f; f.p = m.xy + off + a; f.len = m.lenp + off + a; f.n = b - a;
    return f;
}
__device__ __forceinline__ int v2x_nearest(const V2xPath& f, double x, double y, int lane) {
    const int i = dp_nearest_plain(f.p, f.n, x, y, lane);
    return i == 0x7fffffff ? 0 : i;                         // CShare::NearestId starts from index 0 / distance 9999
}
// the longitudinal distance idiom (Decision.cpp:1899-1922): segment lengths added in index order; lenp holds the same terms
__device__ __forceinline__ double v2x_lng(const V2xPath& f, int index, double at_zero) {
    if (index >= 2) {
        double d = 0;
        for (int i = 0; i < index; ++i) d += f.len[i];
        return d;
    }
    return index == 1 ? f.len[0] : at_zero;
}
__device__ __forceinline__ double v2x_min_dist(const V2xPath& f, double x, double y, int lane) {
    double best = 9999;
    for (int i = lane; i < f.n; i += 32) { const double2 a = f.p[i]; best = fmin(best, dp_dist_plain(x, y, a.x, a.y)); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmin(best, __shfl_xor_sync(DP_FULL, best, o));
    return best;
}
struct V2xNear { double min_d; float lat, lng; int index; };
// Decision.cpp:2036-2112: the warning list (or the event point alone), the nearest entry by longitudinal distance; false: no
// information.  WP reads entry i of the caller's list as wp.lat(i) / wp.lng(i).
template <class WP>
__device__ __forceinline__ bool v2x_works(const dp_params& p, const dp_v2x_data& v, const WP& wp, const V2xPath& f, int lane, V2xNear* r) {
    const bool single = v.wp_count <= 0;
    if (single && (v.rsi_lat == 0 || v.rsi_lng == 0)) return false;
    const int cnt = single ? 1 : v.wp_count;
    r->min_d = 9999; r->lat = 0.f; r->lng = 0.f; r->index = 0;
    for (int k = 0; k < cnt; ++k) {
        const double la = single ? v.rsi_lat : wp.lat(v.wp_first + k), lo = single ? v.rsi_lng : wp.lng(v.wp_first + k);
        const double gy = (la - p.lat0) / p.k_lat, gx = (lo - p.lng0) / p.k_lng;
        r->index = v2x_nearest(f, gx, gy, lane);
        const double d = v2x_lng(f, r->index, -9999.0);
        if (r->min_d >= d) { r->min_d = d; r->lat = (float)la; r->lng = (float)lo; }
    }
    return true;
}
// the warning list as latitude / longitude arrays (dp_v2x_event_batch)
struct V2xWpLatLng {
    const double* __restrict__ la; const double* __restrict__ lo;
    __device__ __forceinline__ double lat(int i) const { return la[i]; }
    __device__ __forceinline__ double lng(int i) const { return lo[i]; }
};

// V2XEventDecision of one scene (every lane of the warp; the result is the same in every lane).  A header that does not name a
// lane of the map (device-pointer callers are not validated on the host): no flags, `ub` set
template <class WP>
__device__ __forceinline__ dp_v2x_flags v2x_handlers(const DevMap& m, const dp_params& p, const dp_scene_hdr& h, const dp_v2x_data& v,
                                                     const WP& wp, int mode, int lane) {
    unsigned light = 0, cons = 0, ped = 0, ub = 0;
    double lng = 9999, lat = 9999;
    const bool bad_hdr = h.road_num < 1 || h.road_num > m.n_roads || h.lane_num < 1 || h.lane_num > DP_LANESUM ||
                         h.lane_num > m.road_lane_base[h.road_num < 1 || h.road_num > m.n_roads ? 1 : h.road_num] -
                                          m.road_lane_base[h.road_num < 1 || h.road_num > m.n_roads ? 0 : h.road_num - 1];
    const int ln = bad_hdr ? 1 : h.lane_num, gl = bad_hdr ? 0 : m.road_lane_base[h.road_num - 1] + ln - 1, id = bad_hdr ? 0 : h.id[ln - 1];
    if (bad_hdr) ub = 1;
    else if (v.warn_status == 3) {                               // V2XSignalLight
        if (v.spat_lane_occupied == 1) light = (v.spat_state == 3 || v.spat_state == 7) ? 1 : (v.spat_state == 6) ? 2 : 0;
    } else if (v.warn_status == 4 && mode != 1) {           // V2XConstructionEvent
        const V2xPath f = v2x_front(m, gl, id, p.id_more);
        V2xNear r;
        if (v2x_works(p, v, wp, f, lane, &r)) {
            if (r.index + 1 >= f.n) ub = 1;
            else {
                const double gy = ((double)r.lat - p.lat0) / p.k_lat, gx = ((double)r.lng - p.lng0) / p.k_lng;
                const double2 a = f.p[r.index], b = f.p[r.index + 1];
                lat = dp_lat_dis(gx, gy, a.x, a.y, b.x, b.y, p.epsilon);
                lng = r.min_d;
                if (r.min_d >= 0 && r.min_d <= 100) cons = (lat >= 0 && lat < 3.75 / 2) ? 1 : 0;
            }
        }
    } else if (v.warn_status == 4) {                        // V2XConstructionEventTemporal
        const int off = m.lane_pt_off[gl], cnt = m.lane_pt_off[gl + 1] - off;
        if (id >= cnt) ub = 1;
        else {
            const int lane_sum = m.road_lane_base[h.road_num] - m.road_lane_base[h.road_num - 1], chg = m.attr[off + id];
            const V2xPath F = v2x_front(m, gl, id, p.id_more);
            V2xPath LF = F, RF = F; LF.n = 0; RF.n = 0;
            if (chg == 1 && ln > 1) {
                const int idl = h.id[ln - 2], cl = m.lane_pt_off[gl] - m.lane_pt_off[gl - 1];
                if (idl > 0 && idl < cl) LF = v2x_front(m, gl - 1, idl, p.id_more);
            }
            if (chg == 2 && ln < lane_sum) {
                const int idr = h.id[ln], cr = m.lane_pt_off[gl + 2] - m.lane_pt_off[gl + 1];
                if (idr > 0 && idr < cr) RF = v2x_front(m, gl + 1, idr, p.id_more);
            }
            const double ey = (v.ego_lat - p.lat0) / p.k_lat, ex = (v.ego_lng - p.lng0) / p.k_lng;
            const double ry = (v.rsi_lat - p.lat0) / p.k_lat, rx = (v.rsi_lng - p.lng0) / p.k_lng;
            const double rsi_distance = dp_dist_plain(ex, ey, rx, ry);
            if (rsi_distance >= 0 && rsi_distance <= 100) {
                const double f = v2x_min_dist(F, rx, ry, lane), lf = v2x_min_dist(LF, rx, ry, lane), rf = v2x_min_dist(RF, rx, ry, lane);
                const bool left = (lf < rf) && (lf < f) && (lf < 2), right = (rf < lf) && (rf < f) && (rf < 2);
                if (!left && !right && (f < lf) && (f < rf) && (f < 2)) {
                    V2xNear r;
                    if (v2x_works(p, v, wp, F, lane, &r)) { lng = r.min_d; cons = (r.min_d >= 0 && r.min_d <= 100) ? 1 : 0; }
                }
            }
        }
    } else if (v.warn_status == 5) {                        // V2XPedestrianJudge
        const V2xPath f = v2x_front(m, gl, id, 0);
        if (v.ped_distance >= 0 && v.ped_distance <= 100) {
            const double gy = (v.ped_lat - p.lat0) / p.k_lat, gx = (v.ped_lng - p.lng0) / p.k_lng;
            const int index = v2x_nearest(f, gx, gy, lane);
            if (index + 1 >= f.n) ub = 1;
            else {
                const double2 a = f.p[index], b = f.p[index + 1];
                lat = dp_lat_dis(gx, gy, a.x, a.y, b.x, b.y, p.epsilon);
                lng = v2x_lng(f, index, v.ped_distance > 5 ? -9999.0 : 0.0);
                const double width = 3.75 + 3.75 / 2;
                const int lat_time = (lat < 0) ? 1 : 0;     // the reference's counters are locals: never more than one
                if (lng >= 0 && lng <= 100) {
                    if (lat >= width) ped = 0;
                    else if (lat > 1.5 && lat < width) ped = (lat_time < 5) ? 0 : 1;
                    else if (lat <= 1.5 || v.ped_direction == 1) ped = 1;
                }
            }
        }
    }
    if (ub) { light = 0; cons = 0; ped = 0; lng = 9999; lat = 9999; }
    dp_v2x_flags o;
    o.light_flag = (uint16_t)light; o.construction_flag = (uint8_t)cons; o.pedestrian_flag = (uint8_t)ped; o.ub = (uint8_t)ub;
    o.pad[0] = o.pad[1] = o.pad[2] = 0; o.lng_distance = lng; o.lat_distance = lat;
    return o;
}

// the opt-in speed command of include/dmpp_b200.h section 10
__device__ __forceinline__ void v2x_apply_rule(const dp_v2x_flags& f, dp_plan_record& r) {
    if (f.pedestrian_flag || f.light_flag == 1) { r.brakespeed = 0.0; r.acc_flag = 1; r.des_acc = -3.0; }
    else if (f.construction_flag && r.brakespeed > 3.0) r.brakespeed = 3.0;
}
}  // namespace
