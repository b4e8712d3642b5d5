// csrc/dp_world_lanechange.cu -- the world step with lane-changing agents armed (include/dmpp_b200.h section 13, on top of the
// reactive agents of section 12): the LANECHG = true instances of dp_world_kernel (dp_world_step.cuh), with and without
// junctions and episode metrics, in a translation unit of their own so that the disarmed and react-only instances stay what
// they were.
#include "dp_world_step.cuh"

namespace {
template <bool JUNC, bool METRICS>
cudaError_t launch(int g, size_t smem, cudaStream_t st, const DevMap& m, const dp_params& p, const dp_world_params& wp, int n, int max_obs,
                   dp_scene_hdr* hdr, dp_agent* agents, double* obs_x, double* obs_y, const dp_plan_record* rec, const double2* last_path,
                   const dp_metrics_params& mp, dp_episode_metrics* met, const LaneChangeModel& am) {
    dp_world_kernel<JUNC, METRICS, true, true><<<g, WPB * 32, smem, st>>>(m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
    return cudaGetLastError();
}
}  // namespace

cudaError_t dp_world_lanechange_prepare() {
    const int bytes = (int)(WPB * react_stage_bytes(DP_AGENT_MODEL_MAX_OBS));
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(dp_world_kernel<false, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(dp_world_kernel<true, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(dp_world_kernel<false, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(dp_world_kernel<true, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

cudaError_t dp_launch_world_lanechange(const DevMap& m, const dp_params& p, const dp_world_params& wp, int n, int max_obs, dp_scene_hdr* hdr,
                                       dp_agent* agents, double* obs_x, double* obs_y, const dp_plan_record* rec, const double2* last_path,
                                       const dp_metrics_params& mp, dp_episode_metrics* met, const dp_agent_model_params& amp, const double* v0,
                                       const dp_lane_change_params& lcp, dp_lane_change_state* lcs, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int g = (n + WPB - 1) / WPB;
    const size_t smem = WPB * react_stage_bytes(max_obs);
    LaneChangeModel am;
    am.p = amp; am.v0 = v0; am.lc = lcp; am.lcs = lcs;
    const bool junc = wp.pre_junction_pts > 0;
    if (met) return junc ? launch<true, true>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am)
                         : launch<false, true>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
    return junc ? launch<true, false>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am)
                : launch<false, false>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
}
