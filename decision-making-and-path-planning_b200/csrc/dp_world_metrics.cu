// csrc/dp_world_metrics.cu -- the world step with episode metrics armed (include/dmpp_b200.h section 11): the METRICS = true
// instances of dp_world_kernel (dp_world_step.cuh), in a translation unit of their own so that the disarmed instances of
// dp_world.cu stay what they were.
#include "dp_world_step.cuh"

cudaError_t dp_launch_world_metrics(const DevMap& m, const dp_params& p, const dp_world_params& wp, int n, int max_obs, dp_scene_hdr* hdr,
                                    dp_agent* agents, double* obs_x, double* obs_y, const dp_plan_record* rec, const double2* last_path,
                                    const dp_metrics_params& mp, dp_episode_metrics* met, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int g = (n + WPB - 1) / WPB;
    const AgentModel am = {};
    if (wp.pre_junction_pts > 0) dp_world_kernel<true, true, false><<<g, WPB * 32, 0, st>>>(m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
    else dp_world_kernel<false, true, false><<<g, WPB * 32, 0, st>>>(m, p, wp, n, max_obs, hdr, agents, obs_x, obs_y, rec, last_path, mp, met, am);
    return cudaGetLastError();
}
