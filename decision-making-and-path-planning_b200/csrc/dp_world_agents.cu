// csrc/dp_world_agents.cu -- the world step with reactive agents armed (include/dmpp_b200.h section 12): the REACT = true
// instances of dp_world_kernel (dp_world_step.cuh), with and without junctions and episode metrics, in a translation unit of
// their own so that the disarmed instances of dp_world.cu and dp_world_metrics.cu stay what they were.
#include "dp_world_step.cuh"

namespace {
template <bool JUNC, bool METRICS>
cudaError_t launch(int g, size_t smem, cudaStream_t st, const DevMap& m, const dp_params& p, const dp_world_params& wp, int n, int max_obs,
                   dp_scene_hdr* hdr, dp_agent* agents, double* obs_x, double* obs_y, const dp_plan_record* rec, const double2* last_path,
                   const dp_metrics_params& mp, dp_episode_metrics* met, const AgentModel& am) {
    dp_world_kernel<JUNC, METRICS, true><<<g, WPB * 32, smem, st>>>(m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
    return cudaGetLastError();
}
}  // namespace

cudaError_t dp_world_agents_prepare() {
    const int bytes = (int)(WPB * react_stage_bytes(DP_AGENT_MODEL_MAX_OBS));
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(dp_world_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(dp_world_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(dp_world_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(dp_world_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

cudaError_t dp_launch_world_agents(const DevMap& m, const dp_params& p, const dp_world_params& wp, int n, int max_obs, dp_scene_hdr* hdr,
                                   dp_agent* agents, double* obs_x, double* obs_y, const dp_plan_record* rec, const double2* last_path,
                                   const dp_metrics_params& mp, dp_episode_metrics* met, const dp_agent_model_params& amp, const double* v0,
                                   cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int g = (n + WPB - 1) / WPB;
    const size_t smem = WPB * react_stage_bytes(max_obs);
    const AgentModel am = {amp, v0};
    const bool junc = wp.pre_junction_pts > 0;
    if (met) return junc ? launch<true, true>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am)
                         : launch<false, true>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
    return junc ? launch<true, false>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am)
                : launch<false, false>(g, smem, st, m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
}
