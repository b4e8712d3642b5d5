// csrc/dp_world_v2x_obstacles.cu -- the obstacles launch of a closed-loop episode (include/dmpp_b200.h section 16): one warp per
// world copies the world's header and obstacle points into the view the next cycle runs on, and lane 0 appends the V2X road users
// within range (the active pedestrian, the road-works point, the zone's warning points) and updates the world's row.  Rules frozen
// in tools/junction_oracle/v2x_obstacles.h (IEEE binary64, -fmad=false, operations in that order).  A translation unit of its own:
// the world-step instances, dp_world_v2x_kernel and the cycle kernels compile to what they compiled to before.
#include <cstddef>
#include "dp_world_step.cuh"

static_assert(sizeof(dp_v2x_obstacle_params) == 40, "dp_v2x_obstacle_params is 40 bytes");
static_assert(sizeof(dp_v2x_obstacle_stats) == 80, "dp_v2x_obstacle_stats is 80 bytes");
static_assert(sizeof(dp_scene_hdr) == 32 * 4, "one 4-byte header word per lane");
static_assert(offsetof(dp_scene_hdr, n_obs) % 4 == 2, "n_obs is the upper half of its header word");

namespace {
// section 11's ego box at the header's pose
struct EgoBox { double x, y, c, s; };
// inside the box?  *d = the clearance
__device__ __forceinline__ bool box_point(const dp_v2x_obstacle_params& op, const EgoBox& b, double ox, double oy, double* d) {
    const double dx = ox - b.x, dy = oy - b.y;
    const double lon = dx * b.c + dy * b.s, lat = dy * b.c - dx * b.s, alat = fabs(lat);
    const double ex = lon > op.front ? lon - op.front : (lon < -op.rear ? -op.rear - lon : 0.0);
    const double ey = alat > op.half_width ? alat - op.half_width : 0.0;
    *d = sqrt(ex * ex + ey * ey);
    return -op.rear <= lon && lon <= op.front && -op.half_width <= lat && lat <= op.half_width;
}
__device__ __forceinline__ bool in_range(double range, const dp_scene_hdr& h, double px, double py) {
    const double dx = px - h.x, dy = py - h.y;
    return sqrt(dx * dx + dy * dy) <= range;
}

__device__ __forceinline__ void obst_stats_init(dp_v2x_obstacle_stats& r) {
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    r.min_ped_clearance = inf; r.min_works_clearance = inf;
    r.views = 0; r.ped_cycles = 0; r.works_cycles = 0; r.dropped = 0;
    r.ped_bound_cycles = 0; r.works_bound_cycles = 0;
    r.ped_hits = 0; r.first_ped_hit = -1; r.works_hits = 0; r.first_works_hit = -1;
    r.last_ped_slot = -1; r.last_works_first = 0; r.last_works_end = 0;
    r.pad[0] = r.pad[1] = r.pad[2] = 0;
}

// k: the cycle the view is built for; tally: the row only, after the last world step (k = the number of cycles)
__global__ void __launch_bounds__(WPB * 32) dp_world_obstacles_kernel(DevMap m, dp_v2x_obstacle_params op, int n, int max_obs, int k, int tally,
                                                                      const dp_scene_hdr* __restrict__ hdr, const double* __restrict__ ox,
                                                                      const double* __restrict__ oy, const dp_plan_record* __restrict__ prev,
                                                                      const dp_v2x_event_spec* __restrict__ spec, const double* __restrict__ wp_x,
                                                                      const double* __restrict__ wp_y, dp_scene_hdr* __restrict__ hv,
                                                                      double* __restrict__ vx, double* __restrict__ vy,
                                                                      dp_v2x_obstacle_stats* __restrict__ stats) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int scene = blockIdx.x * WPB + wib;
    if (scene >= n) return;
    const dp_scene_hdr& h = hdr[scene];
    const uint32_t word = reinterpret_cast<const uint32_t*>(hdr + scene)[lane];   // the header, one word per lane, coalesced
    const int na = min((int)h.n_obs, max_obs);
    const size_t row = (size_t)scene * max_obs;
    // the world's points first: the copy does not wait for lane 0's scalar work (lane 0 appends at slots >= na)
    if (!tally)
        for (int j = lane; j < na; j += 32) { vx[row + j] = ox[row + j]; vy[row + j] = oy[row + j]; }
    if (k == 0 && lane == 0) obst_stats_init(stats[scene]);  // the first launch of an episode starts a clean row
    // a header that does not name a lane of the map: a plain copy, the row alone
    const bool named = !(h.road_num < 1 || h.road_num > m.n_roads || h.lane_num < 1 ||
                         h.lane_num > m.road_lane_base[h.road_num] - m.road_lane_base[h.road_num - 1] || h.lane_num > DP_LANESUM);
    int n_view = h.n_obs;
    if (lane == 0) {
        // loads that do not depend on the header are issued before the lane test, so that they overlap its map lookups
        const dp_v2x_event_spec s = spec[scene];
        dp_v2x_obstacle_stats r = stats[scene];
        const bool bound = prev != nullptr && prev[scene].ob_flag;
        const int oi = prev != nullptr ? prev[scene].ob_index : -1;
        if (named) {
            const double t = v2x_time(k, h);
            EgoBox b;
            b.x = h.x; b.y = h.y;
            dp_sincos_deg(h.dir, &b.c, &b.s);
            if (bound) {                                        // the previous cycle's local path was bounded by one of its event points
                if (r.last_ped_slot >= 0 && oi == r.last_ped_slot) r.ped_bound_cycles += 1;
                if (oi >= r.last_works_first && oi < r.last_works_end) r.works_bound_cycles += 1;
            }
            double px = 0, py = 0, d;
            const bool ped_on = v2x_pedestrian(s, t, &px, &py);
            if (ped_on) {
                if (box_point(op, b, px, py, &d)) { r.ped_hits += 1; if (r.first_ped_hit < 0) r.first_ped_hit = k; }
                if (d < r.min_ped_clearance) r.min_ped_clearance = d;
            }
            if (s.has_works) {
                bool hit = box_point(op, b, s.rw_x, s.rw_y, &d);
                if (d < r.min_works_clearance) r.min_works_clearance = d;
                for (int i = 0; i < s.wp_count; ++i) {
                    hit = box_point(op, b, wp_x[s.wp_first + i], wp_y[s.wp_first + i], &d) || hit;
                    if (d < r.min_works_clearance) r.min_works_clearance = d;
                }
                if (hit) { r.works_hits += 1; if (r.first_works_hit < 0) r.first_works_hit = k; }
            }
            if (!tally) {
                int cnt = na, ped_slot = -1, dropped = 0;
                if ((op.what & 1) && ped_on && in_range(op.range, h, px, py)) {
                    if (cnt < max_obs) { vx[row + cnt] = px; vy[row + cnt] = py; ped_slot = cnt; ++cnt; }
                    else ++dropped;
                }
                const int wf = cnt;
                if (s.has_works) {
                    if ((op.what & 2) && in_range(op.range, h, s.rw_x, s.rw_y)) {
                        if (cnt < max_obs) { vx[row + cnt] = s.rw_x; vy[row + cnt] = s.rw_y; ++cnt; }
                        else ++dropped;
                    }
                    if (op.what & 4)
                        for (int i = 0; i < s.wp_count; ++i) {
                            const double x = wp_x[s.wp_first + i], y = wp_y[s.wp_first + i];
                            if (!in_range(op.range, h, x, y)) continue;
                            if (cnt < max_obs) { vx[row + cnt] = x; vy[row + cnt] = y; ++cnt; }
                            else ++dropped;
                        }
                }
                r.views += 1; r.ped_cycles += ped_slot >= 0; r.works_cycles += cnt > wf; r.dropped += dropped;
                r.last_ped_slot = ped_slot; r.last_works_first = wf; r.last_works_end = cnt;
                if (cnt > na) n_view = cnt;
            }
            stats[scene] = r;
        }
    }
    if (tally) return;
    n_view = __shfl_sync(0xffffffffu, n_view, 0);
    uint32_t w = word;
    if (lane == (int)(offsetof(dp_scene_hdr, n_obs) / 4)) w = (w & 0xffffu) | ((uint32_t)n_view << 16);
    reinterpret_cast<uint32_t*>(hv + scene)[lane] = w;
}
}  // namespace

cudaError_t dp_launch_world_obstacles(const DevMap& m, const DpV2xOpts& v, const DpObstOpts& o, int n, int max_obs, const dp_scene_hdr* hdr,
                                      const double* ox, const double* oy, const dp_plan_record* prev, int cycle, bool tally, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_world_obstacles_kernel<<<(n + WPB - 1) / WPB, WPB * 32, 0, st>>>(m, o.op, n, max_obs, cycle, tally ? 1 : 0, hdr, ox, oy, prev, v.spec,
                                                                       v.wp_x, v.wp_y, o.hv, o.vx, o.vy, o.stats);
    return cudaGetLastError();
}
