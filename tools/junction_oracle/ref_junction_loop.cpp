// tools/junction_oracle/ref_junction_loop.cpp -- TEST INFRASTRUCTURE. Closed-loop episodes of the UNMODIFIED reference
// (oracle/_ref/libref.so) with the junction world step of world_junction.cpp between its cycles: oracle/ref_closed_loop.cpp
// with two differences.  The reference reads RoadNavi once, before its loop (ref_harness.cpp:220-232), so the entry of the road
// after the junction (path_num + 1: out_lane_no unchanged, stub_attribute 0) is handed to it up front; and the step is
// junction::world_step.
#include <cstring>
#include <vector>
#include "../../oracle/ref_api.h"
#include "world_junction.h"

extern "C" {
const dp_map_desc* ref_map_desc();
void ref_set_cycle_hook(void (*fn)(int, void*), void* user);
void ref_last_path(double* x, double* y);
int ref_run_episode(int cycles, const dp_scene_hdr* hdr, long hdr_stride, const double* obs_x, const double* obs_y, long obs_stride,
                    dp_plan_record* rec, long rec_stride, double* path_xy, long path_xy_stride, double* path_ll, long path_ll_stride,
                    ref_call* calls, int32_t* n_calls, long ncalls_stride, long calls_stride, int calls_cap, dp_carry* carry_out,
                    double* last_path_out);
}

namespace {
struct Loop {
    const junction::JMap* m; const dp_params* p; const dp_world_params* wp; int cycles, max_obs;
    std::vector<dp_scene_hdr> hdr; std::vector<double> ox, oy; std::vector<dp_plan_record> rec; dp_agent* ag;
};
void between(int c, void* user) {
    Loop& L = *(Loop*)user;
    double lx[200], ly[200];
    ref_last_path(lx, ly);
    L.hdr[c + 1] = L.hdr[c];
    std::memcpy(&L.ox[(size_t)(c + 1) * L.max_obs], &L.ox[(size_t)c * L.max_obs], sizeof(double) * L.max_obs);
    std::memcpy(&L.oy[(size_t)(c + 1) * L.max_obs], &L.oy[(size_t)c * L.max_obs], sizeof(double) * L.max_obs);
    junction::world_step(*L.m, *L.p, *L.wp, L.hdr[c + 1], L.ag, &L.ox[(size_t)(c + 1) * L.max_obs], &L.oy[(size_t)(c + 1) * L.max_obs],
                         &L.rec[c], lx, ly);
}
}  // namespace

// same arrays as jo_run_closed_loop; returns the worst ref_run_episode status (0 ok)
extern "C" int ref_run_closed_loop_junction(const dp_params* p, const dp_world_params* wp, int n, int cycles, int max_obs, dp_scene_hdr* hdr,
                                            dp_agent* agents, double* ox, double* oy, dp_plan_record* rec, dp_scene_hdr* hdr_log,
                                            double* obs_log_x, double* obs_log_y, double* path_xy, dp_carry* carry_out, double* last_path_out) {
    junction::JMap m;
    m.set(*ref_map_desc());
    int worst = 0;
    for (int s = 0; s < n; ++s) {
        Loop L;
        L.m = &m; L.p = p; L.wp = wp; L.cycles = cycles; L.max_obs = max_obs;
        L.ag = agents + (size_t)s * max_obs;
        L.hdr.assign(cycles + 1, hdr[s]);
        L.ox.assign((size_t)(cycles + 1) * max_obs, 0.0); L.oy.assign((size_t)(cycles + 1) * max_obs, 0.0);
        L.rec.assign(cycles, dp_plan_record());
        junction::world_step(m, *p, *wp, L.hdr[0], L.ag, L.ox.data(), L.oy.data(), nullptr, nullptr, nullptr);
        for (int c = 1; c <= cycles; ++c) L.hdr[c] = L.hdr[0];     // (RoadNavi is assembled from every cycle's slice before the loop)
        if (wp->pre_junction_pts > 0 && cycles > 1) {             // the RoadNavi entry of the road after the junction; the hook
            L.hdr[1].path_num = (uint16_t)(L.hdr[0].path_num + 1); // overwrites hdr[1] before cycle 1 runs
            L.hdr[1].stub_attribute = 0;
        }
        std::vector<double> pxy(path_xy ? (size_t)cycles * 400 : 0);
        ref_set_cycle_hook(between, &L);
        const int rc = ref_run_episode(cycles, L.hdr.data(), 1, L.ox.data(), L.oy.data(), max_obs, L.rec.data(), 1,
                                       path_xy ? pxy.data() : nullptr, 400, nullptr, 0, nullptr, nullptr, 0, 0, 0,
                                       carry_out ? carry_out + s : nullptr, last_path_out ? last_path_out + (size_t)s * 400 : nullptr);
        ref_set_cycle_hook(nullptr, nullptr);
        if (rc < 0) return rc;
        if (rc > worst) worst = rc;
        for (int c = 0; c < cycles; ++c) {
            const size_t e = (size_t)c * n + s;
            rec[e] = L.rec[c];
            if (hdr_log) hdr_log[e] = L.hdr[c];
            if (obs_log_x) std::memcpy(obs_log_x + e * max_obs, &L.ox[(size_t)c * max_obs], sizeof(double) * max_obs);
            if (obs_log_y) std::memcpy(obs_log_y + e * max_obs, &L.oy[(size_t)c * max_obs], sizeof(double) * max_obs);
            if (path_xy) std::memcpy(path_xy + e * 400, &pxy[(size_t)c * 400], sizeof(double) * 400);
        }
        hdr[s] = L.hdr[cycles];
        std::memcpy(ox + (size_t)s * max_obs, &L.ox[(size_t)cycles * max_obs], sizeof(double) * max_obs);
        std::memcpy(oy + (size_t)s * max_obs, &L.oy[(size_t)cycles * max_obs], sizeof(double) * max_obs);
    }
    return worst;
}
