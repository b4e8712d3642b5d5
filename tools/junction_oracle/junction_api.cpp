// tools/junction_oracle/junction_api.cpp -- TEST INFRASTRUCTURE. C API of libjunction_oracle.so: the restated cycle of oracle/
// (planner_oracle.cpp, compiled in unchanged) with the junction world step of world_junction.cpp between its cycles; the
// same arrays as oracle_world_step / oracle_run_closed_loop of oracle/oracle_api.cpp.
#include <atomic>
#include <cstring>
#include <thread>
#include <vector>
#include "world_junction.h"

namespace { junction::JMap g_map; bool g_have_map = false; }

extern "C" {

int jo_set_map(const dp_map_desc* m) { g_map.set(*m); g_have_map = true; return 0; }   // caller keeps arrays alive

// lane_next[n_lanes] as the world step sees it
int jo_lane_next(int32_t* out) {
    if (!g_have_map) return -1;
    for (size_t l = 0; l < g_map.next.size(); ++l) out[l] = g_map.next[l];
    return 0;
}

int jo_world_step(const dp_params* p, const dp_world_params* wp, int n, int max_obs, dp_scene_hdr* hdr, dp_agent* agents, double* ox,
                  double* oy, const dp_plan_record* rec, const double* last_path) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s)
        junction::world_step(g_map, *p, *wp, hdr[s], agents + (size_t)s * max_obs, ox + (size_t)s * max_obs, oy + (size_t)s * max_obs,
                             rec ? rec + s : nullptr, last_path ? last_path + (size_t)s * 400 : nullptr,
                             last_path ? last_path + (size_t)s * 400 + 200 : nullptr);
    return 0;
}

long long jo_run_closed_loop(const dp_params* p, const dp_world_params* wp, int n, int cycles, int max_obs, dp_scene_hdr* hdr,
                             dp_agent* agents, double* ox, double* oy, dp_plan_record* rec, dp_scene_hdr* hdr_log, double* obs_log_x,
                             double* obs_log_y, double* path_xy, dp_carry* carry_out, double* last_path_out, int threads,
                             int32_t* ub_scene) {
    if (!g_have_map) return -1;
    if (threads < 1) threads = 1;
    std::atomic<long long> ub(0);
    auto work = [&](int s0, int s1) {
        long long lub = 0;
        for (int s = s0; s < s1; ++s) {
            const long long lub0 = lub;
            oracle::SceneState st;
            oracle::reset_state(st);
            dp_agent* ag = agents + (size_t)s * max_obs;
            double* sx = ox + (size_t)s * max_obs; double* sy = oy + (size_t)s * max_obs;
            junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, nullptr, nullptr, nullptr);
            for (int c = 0; c < cycles; ++c) {
                const size_t e = (size_t)c * n + s;
                if (hdr_log) hdr_log[e] = hdr[s];
                if (obs_log_x) std::memcpy(obs_log_x + e * max_obs, sx, sizeof(double) * max_obs);
                if (obs_log_y) std::memcpy(obs_log_y + e * max_obs, sy, sizeof(double) * max_obs);
                oracle::CycleOut o{};
                o.rec = rec + e;
                o.path_xy = path_xy ? path_xy + e * 400 : nullptr;
                oracle::cycle(g_map.m, *p, hdr[s], sx, sy, st, o, false);
                lub += o.ub_hits;
                junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, rec + e, st.last_x, st.last_y);
            }
            if (ub_scene) ub_scene[s] = (int32_t)(lub - lub0);
            if (carry_out) carry_out[s] = st.c;
            if (last_path_out) {
                std::memcpy(last_path_out + (size_t)s * 400, st.last_x, sizeof(st.last_x));
                std::memcpy(last_path_out + (size_t)s * 400 + 200, st.last_y, sizeof(st.last_y));
            }
        }
        ub += lub;
    };
    if (threads == 1) work(0, n);
    else {
        std::vector<std::thread> th;
        for (int t = 0; t < threads; ++t) th.emplace_back(work, (int)((long long)n * t / threads), (int)((long long)n * (t + 1) / threads));
        for (auto& t : th) t.join();
    }
    return ub.load();
}

}  // extern "C"
