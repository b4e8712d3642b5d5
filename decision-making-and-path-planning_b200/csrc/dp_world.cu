// csrc/dp_world.cu -- the two stages either side of the Decision + Planning cycle (SURVEY.md 8f ranks 1 and 3):
//   dp_world_kernel   the world step of the closed-loop episode runner: ego walked along its own plan, agents along their
//                     lanes, windowed re-localisation; one warp per scene, everything in place in HBM
//                     (arithmetic frozen in oracle/world_spec.cpp, junction transitions in tools/junction_oracle/world_junction.cpp;
//                     IEEE binary64, -fmad=false, operations in that order); the kernel and its launcher are in
//                     dp_world_step.cuh, its disarmed instances here, its episode-metrics instances in dp_world_metrics.cu,
//                     its reactive-agent instances in dp_world_agents.cu, its lane-changing instances in dp_world_lanechange.cu;
//                     dp_launch_world picks the instance set from the armed options;
//   dp_v2x_kernel     the V2X event handlers (Decision.cpp:1824-2434, dp_v2x.cuh) as a batch operator next to the cycle (their
//                     closed-loop launch is dp_world_v2x.cu);
//   dp_frames_kernel  the output stage: PlanningOut / PlanningStatus (Planning.cpp:173-214) packed into fixed-layout frames
//                     from the plan record and the carried local path -- byte work bound by HBM: a warp streams one scene
//                     (3.3 KB in, 3.3 KB out), lanes own consecutive 16-byte points so that loads and stores coalesce.
#include "dp_world_step.cuh"
#include "dp_v2x.cuh"

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

// ---- V2X event handlers (Decision.cpp:1824-2434), one warp per scene: the device function of dp_v2x.cuh ----
__global__ void __launch_bounds__(WPB * 32) dp_v2x_kernel(DevMap m, dp_params p, int n, const dp_scene_hdr* __restrict__ hdr,
                                                          const dp_v2x_data* __restrict__ v2x, const double* __restrict__ wp_lat,
                                                          const double* __restrict__ wp_lng, int mode, dp_v2x_flags* __restrict__ out) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int scene = blockIdx.x * WPB + wib;
    if (scene >= n) return;
    const dp_v2x_flags o = v2x_handlers(m, p, hdr[scene], v2x[scene], V2xWpLatLng{wp_lat, wp_lng}, mode, lane);
    if (lane == 0) out[scene] = o;
}
}  // namespace

namespace {
// the opt-in speed command of include/dmpp_b200.h section 10: one thread per scene, a 128-byte record each
__global__ void dp_v2x_apply_kernel(int n, const dp_v2x_flags* __restrict__ flags, dp_plan_record* __restrict__ rec) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    v2x_apply_rule(flags[i], rec[i]);
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
