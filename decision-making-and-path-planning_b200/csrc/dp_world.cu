// csrc/dp_world.cu -- the two stages either side of the Decision + Planning cycle (SURVEY.md 8f ranks 1 and 3):
//   dp_world_kernel   the world step of the closed-loop episode runner: ego walked along its own plan, agents along their
//                     lanes, windowed re-localisation; one warp per scene, everything in place in HBM
//                     (arithmetic frozen in oracle/world_spec.cpp, junction transitions in tools/junction_oracle/world_junction.cpp;
//                     IEEE binary64, -fmad=false, operations in that order); the kernel and its launcher are in
//                     dp_world_step.cuh, its disarmed instances here, its episode-metrics instances in dp_world_metrics.cu,
//                     its reactive-agent instances in dp_world_agents.cu, its lane-changing instances in dp_world_lanechange.cu;
//                     dp_launch_world picks the instance set from the armed options;
//   dp_v2x_kernel     the V2X event handlers (Decision.cpp:1824-2434) as a batch operator next to the cycle;
//   dp_frames_kernel  the output stage: PlanningOut / PlanningStatus (Planning.cpp:173-214) packed into fixed-layout frames
//                     from the plan record and the carried local path -- byte work bound by HBM: a warp streams one scene
//                     (3.3 KB in, 3.3 KB out), lanes own consecutive 16-byte points so that loads and stores coalesce.
#include "dp_world_step.cuh"

namespace {
__global__ void __launch_bounds__(WPB * 32) dp_frames_kernel(dp_params p, int n, const dp_plan_record* __restrict__ rec,
                                                             const double2* __restrict__ last_path, dp_ctrl_frame* __restrict__ ctrl,
                                                             dp_status_frame* __restrict__ status) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int scene = blockIdx.x * WPB + wib;
    if (scene >= n) return;
    const dp_plan_record* r = rec + scene;
    // heads: lane 0 (64-bit stores into zeroed-by-construction layouts: every byte of the head is written here)
    if (lane == 0) {
        const double lon = r->mindist_lon, bs = r->brakespeed, da = r->des_acc;
        const unsigned light = r->light;
        if (ctrl) {
            dp_ctrl_frame* c = ctrl + scene;
            const unsigned long long w0 = (unsigned long long)r->cnt | ((unsigned long long)r->acc_flag << 16) | (1ull << 40) |
                                          ((unsigned long long)light << 48);          // cnt, apa 0, desacc_vd, desstr_vd 0, road_type 0, sstop 1, light
            *reinterpret_cast<unsigned long long*>(c) = w0;
            c->brakedis = lon; c->brake_speed = 0.0; c->desacc = da; c->desspd = bs; c->desstr = 0.0; c->radius = r->radius;
        }
        if (status) {
            dp_status_frame* s = status + scene;
            const unsigned long long w0 = (unsigned long long)(unsigned)(int)r->afresh_cause | ((unsigned long long)light << 32);
            *reinterpret_cast<unsigned long long*>(s) = w0;
            s->near_ob_dist = lon; s->planspeed = bs; s->planacc = da;
        }
    }
    // every 2nd path point (Planning.cpp:180-183, :203-212); frames are 8-byte aligned only, so points go out as two doubles
    const double2* lp = last_path + (size_t)scene * DP_PATH_POINTS;
    for (int i = lane; i < DP_OUT_POINTS; i += 32) {
        const double2 q = lp[2 * i];
        if (ctrl) {
            double* o = &ctrl[scene].pnts[i][0];
            o[0] = fma(q.y, p.k_lat, p.lat0);               // GlobalToWGS84 (operator specification): lat, then lng
            o[1] = fma(q.x, p.k_lng, p.lng0);
        }
        if (status) {
            double* o = &status[scene].path_points[i][0];
            o[0] = q.x; o[1] = q.y;
        }
    }
}

// ---- V2X event handlers (Decision.cpp:1824-2434), one warp per scene; control flow is warp-uniform, the nearest-point and
// minimum-distance scans over the <= 200 map points ahead are lane-parallel.  Quirks: see oracle/v2x_oracle.cpp. ----
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
// Decision.cpp:2036-2112: the warning list (or the event point alone), the nearest entry by longitudinal distance; false: no information
__device__ __forceinline__ bool v2x_works(const dp_params& p, const dp_v2x_data& v, const double* wp_lat, const double* wp_lng, const V2xPath& f,
                                          int lane, V2xNear* r) {
    const bool single = v.wp_count <= 0;
    if (single && (v.rsi_lat == 0 || v.rsi_lng == 0)) return false;
    const int cnt = single ? 1 : v.wp_count;
    r->min_d = 9999; r->lat = 0.f; r->lng = 0.f; r->index = 0;
    for (int k = 0; k < cnt; ++k) {
        const double la = single ? v.rsi_lat : wp_lat[v.wp_first + k], lo = single ? v.rsi_lng : wp_lng[v.wp_first + k];
        const double gy = (la - p.lat0) / p.k_lat, gx = (lo - p.lng0) / p.k_lng;
        r->index = v2x_nearest(f, gx, gy, lane);
        const double d = v2x_lng(f, r->index, -9999.0);
        if (r->min_d >= d) { r->min_d = d; r->lat = (float)la; r->lng = (float)lo; }
    }
    return true;
}

__global__ void __launch_bounds__(WPB * 32) dp_v2x_kernel(DevMap m, dp_params p, int n, const dp_scene_hdr* __restrict__ hdr,
                                                          const dp_v2x_data* __restrict__ v2x, const double* __restrict__ wp_lat,
                                                          const double* __restrict__ wp_lng, int mode, dp_v2x_flags* __restrict__ out) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int scene = blockIdx.x * WPB + wib;
    if (scene >= n) return;
    const dp_scene_hdr& h = hdr[scene];
    const dp_v2x_data v = v2x[scene];
    unsigned light = 0, cons = 0, ped = 0, ub = 0;
    double lng = 9999, lat = 9999;
    // a header that names no lane of the map (device-pointer callers are not validated on the host): no flags, `ub` set
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
        if (v2x_works(p, v, wp_lat, wp_lng, f, lane, &r)) {
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
                    if (v2x_works(p, v, wp_lat, wp_lng, F, lane, &r)) { lng = r.min_d; cons = (r.min_d >= 0 && r.min_d <= 100) ? 1 : 0; }
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
    if (lane == 0) {
        dp_v2x_flags o;
        o.light_flag = (uint16_t)light; o.construction_flag = (uint8_t)cons; o.pedestrian_flag = (uint8_t)ped; o.ub = (uint8_t)ub;
        o.pad[0] = o.pad[1] = o.pad[2] = 0; o.lng_distance = lng; o.lat_distance = lat;
        out[scene] = o;
    }
}
}  // namespace

namespace {
// the opt-in speed command of include/dmpp_b200.h section 10: one thread per scene, a 128-byte record each
__global__ void dp_v2x_apply_kernel(int n, const dp_v2x_flags* __restrict__ flags, dp_plan_record* __restrict__ rec) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const dp_v2x_flags f = flags[i];
    if (f.pedestrian_flag || f.light_flag == 1) { rec[i].brakespeed = 0.0; rec[i].acc_flag = 1; rec[i].des_acc = -3.0; }
    else if (f.construction_flag && rec[i].brakespeed > 3.0) rec[i].brakespeed = 3.0;
}
}  // namespace
cudaError_t dp_launch_v2x_apply(int n, const dp_v2x_flags* flags, dp_plan_record* rec, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_v2x_apply_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, flags, rec);
    return cudaGetLastError();
}
cudaError_t dp_launch_v2x(const DevMap& m, const dp_params& p, int n, const dp_scene_hdr* hdr, const dp_v2x_data* v2x, const double* wp_lat,
                          const double* wp_lng, int mode, dp_v2x_flags* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_v2x_kernel<<<(n + WPB - 1) / WPB, WPB * 32, 0, st>>>(m, p, n, hdr, v2x, wp_lat, wp_lng, mode, out);
    return cudaGetLastError();
}

template struct WorldStep<false, false, false>;

cudaError_t dp_launch_world(const DevMap& m, const dp_params& p, const DpWorldOpts& o, const DpWorldBufs& b, cudaStream_t st) {
    if (b.n <= 0) return cudaSuccess;
    if (o.v0 && o.lcs) return o.met ? WorldStep<true, true, true>::launch(m, p, o, b, st) : WorldStep<false, true, true>::launch(m, p, o, b, st);
    if (o.v0) return o.met ? WorldStep<true, true, false>::launch(m, p, o, b, st) : WorldStep<false, true, false>::launch(m, p, o, b, st);
    return o.met ? WorldStep<true, false, false>::launch(m, p, o, b, st) : WorldStep<false, false, false>::launch(m, p, o, b, st);
}
cudaError_t dp_world_prepare() {
    for (auto prepare : {WorldStep<false, true, false>::prepare, WorldStep<true, true, false>::prepare, WorldStep<false, true, true>::prepare,
                         WorldStep<true, true, true>::prepare})
        if (const cudaError_t e = prepare(); e != cudaSuccess) return e;
    return cudaSuccess;
}
cudaError_t dp_launch_frames(const dp_params& p, int n, const dp_plan_record* rec, const double2* last_path, dp_ctrl_frame* ctrl,
                             dp_status_frame* status, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_frames_kernel<<<(n + WPB - 1) / WPB, WPB * 32, 0, st>>>(p, n, rec, last_path, ctrl, status);
    return cudaGetLastError();
}
