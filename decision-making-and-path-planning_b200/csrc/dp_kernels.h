// csrc/dp_kernels.h -- launcher prototypes shared by the translation units of libdmpp_b200.so
#pragma once
#include <cuda_runtime.h>
#include "dp_device.cuh"
#include "dp_group.cuh"                        // (DpIo: the plumbing of one cycle launch)

// launch-time state of ONE context (no process-wide statics: two threads may own two contexts): device properties, which
// kernels already carry their shared-memory attributes, and the experiment switch read from the environment by dp_create
struct DpLaunchCfg {
    int sm_count = 0;
    bool attr_warp = false, attr_group[3] = {false, false, false};
    int group_cfg = 0;                         // DP_GROUP_CFG = 0 | 1 | 2: CTA shape of the group kernel (16 x 256, 8 x 128, 8 x 256)
    // L2 persistence for the map arena (dp_map_upload): the warp-kernel launches carry an access-policy window over it, so the
    // ~3 MB of map tables every scene gathers from stay resident in the L2 set-aside whatever streams through in between
    void* l2_base = nullptr; size_t l2_bytes = 0;
};

cudaError_t dp_launch_cycle(const DevMap& m, const dp_params& p, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                            int max_obs, dp_carry* carry, double2* last_path, dp_plan_record* rec, dp_trace_record* trace,
                            double* path_xy, double* path_ll, cudaStream_t st, const DpIo& io, DpLaunchCfg& lc);   // Decision + Planning half, overlapped
// set the shared-memory attributes of the warp kernels (done lazily by dp_launch_cycle; called up front before a stream capture)
void dp_launch_prepare(DpLaunchCfg& lc);
// the closed-loop world step (dp_world_step.cuh): the buffers of one launch, and the option set a context arms.  A model is armed
// by its pointer: met != nullptr episode metrics (include/dmpp_b200.h section 11), v0 != nullptr reactive agents (section 12),
// lcs != nullptr with v0 lane changes (section 13); its parameters are read only while it is armed
struct DpWorldBufs {
    int n, max_obs;
    dp_scene_hdr* hdr; dp_agent* agents; double* ox; double* oy;
    const dp_plan_record* rec;                 // nullptr: the placement step
    const double2* last_path;
};
struct DpWorldOpts {
    dp_world_params wp;
    dp_metrics_params mp; dp_episode_metrics* met = nullptr;
    dp_agent_model_params amp; const double* v0 = nullptr;
    dp_lane_change_params lcp; dp_lane_change_state* lcs = nullptr;
};
cudaError_t dp_launch_world(const DevMap& m, const dp_params& p, const DpWorldOpts& o, const DpWorldBufs& b, cudaStream_t st);
// allow the reactive instances the dynamic shared memory of DP_AGENT_MODEL_MAX_OBS agent slots (current device; set before a capture)
cudaError_t dp_world_prepare();
// the V2X events of a closed-loop episode (include/dmpp_b200.h section 14), armed by spec != nullptr; n: the worlds the specs cover
struct DpV2xOpts {
    dp_v2x_world_params vp = {0, 0};
    const dp_v2x_event_spec* spec = nullptr;
    const double* wp_x = nullptr; const double* wp_y = nullptr;
    dp_v2x_flags* flags = nullptr; dp_v2x_episode_stats* stats = nullptr;
    int n = 0;
};
// one V2X launch of cycle `cycle` (dp_world_v2x.cu); rec == nullptr: the tally after the last world step
cudaError_t dp_launch_world_v2x(const DevMap& m, const dp_params& p, const DpV2xOpts& o, int n, const dp_scene_hdr* hdr, dp_plan_record* rec,
                                int cycle, cudaStream_t st);
cudaError_t dp_launch_v2x(const DevMap& m, const dp_params& p, int n, const dp_scene_hdr* hdr, const dp_v2x_data* v2x, const double* wp_lat,
                          const double* wp_lng, int mode, dp_v2x_flags* out, cudaStream_t st);
cudaError_t dp_launch_v2x_apply(int n, const dp_v2x_flags* flags, dp_plan_record* rec, cudaStream_t st);
cudaError_t dp_launch_frames(const dp_params& p, int n, const dp_plan_record* rec, const double2* last_path, dp_ctrl_frame* ctrl,
                             dp_status_frame* status, cudaStream_t st);
cudaError_t dp_launch_gather_flush(const dp_plan_record* src, int n, const DpIo& io, cudaStream_t st);
cudaError_t dp_launch_gather_wait(const unsigned* flags, int world, unsigned step, cudaStream_t st);
cudaError_t dp_launch_reset(dp_carry* carry, double2* last_path, int first, int count, cudaStream_t st);
cudaError_t dp_launch_map_prep(const double* x, const double* y, const uint16_t* attr, const int32_t* lane_pt_off, int n_lanes, double2* xy,
                               double2* nrm, double* lenp, double* lenf, float* lane_hmax, float* lane_hmin, float* lane_dnmax, double* cump,
                               double* lane_cerr, int32_t* run_end0, int32_t* run_end1, cudaStream_t st);
// the group kernel (dp_group.cuh): ONE launch per cycle, a CTA walks a group of scenes through the cycle phase by phase
cudaError_t dp_launch_group(const DgMap& m, const dp_params& p, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                            int max_obs, dp_carry* carry, double2* last_path, dp_plan_record* rec, dp_trace_record* trace,
                            double* path_xy, double* path_ll, cudaStream_t st, const DpIo& io, DpLaunchCfg& lc);

// operator-level kernels (dp_ops.cu)
// operator kernels take polylines as AoS double2 (the host entry points interleave x/y)
cudaError_t dp_launch_search(int n_paths, const int32_t* path_off, const double2* pxy, const double* ox,
                             const double* oy, int n_obs, const double* lat_min, const double* lat_max, dp_search_slot* out,
                             cudaStream_t st);
cudaError_t dp_launch_create(int n_paths, const int32_t* path_off, const double2* pxy, const double* offset,
                             double2* out_xy, cudaStream_t st);
cudaError_t dp_launch_bezier(int n, const double* poses, double* out_xy, cudaStream_t st);
cudaError_t dp_launch_mean(int n_paths, const int32_t* path_off, const double2* pxy, double* out_xy, cudaStream_t st);
cudaError_t dp_launch_nearest(int n_paths, const int32_t* path_off, const double2* pxy, const double* qx, const double* qy, int32_t* out_id,
                              cudaStream_t st);
// dense candidate sweep (dp_ops.cu): candidates grouped on the host by (offset = row, point count = horizon group)
cudaError_t dp_launch_sweep_prefix(const double* lines, int n_base, int n_rows, const double* row_off, const int4* row_info, double* row_cum,
                                   cudaStream_t st);
cudaError_t dp_launch_sweep(const double* lines, int n_base, int n_lines, int n_rows, const double* row_off, const int4* row_info,
                            const int32_t* group_P, const int32_t* group_row, const int32_t* cand_group, int n_cand, const double* ox,
                            const double* oy, const double* dvx, const double* dvy, int n_obs, double lat_min, double lat_max, double clear_dis,
                            unsigned* group_key, const double* row_cum, double* cand_dis_lng, unsigned long long* best_key, cudaStream_t st);
cudaError_t dp_launch_sweep_fused(const double* lines, int n_base, int n_lines, int n_rows, const double* row_off, const int4* row_info,
                                  const int32_t* group_P, const int32_t* group_first, int first_nogroup, const double* obs4, int obs_stride,
                                  int n_obs, double lat_min, double lat_max, double clear_dis, const double* row_cum,
                                  unsigned long long* row_res, unsigned* done, unsigned long long* host, unsigned long long seq, long long* dbg,
                                  cudaStream_t st);
cudaError_t dp_launch_fma_peak(int which, float* sink, int iters, int blocks, cudaStream_t st);
