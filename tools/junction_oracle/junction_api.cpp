// tools/junction_oracle/junction_api.cpp -- TEST INFRASTRUCTURE. C API of libjunction_oracle.so: the restated cycle of oracle/
// (planner_oracle.cpp, compiled in unchanged) with the junction world step of world_junction.cpp between its cycles; the
// same arrays as oracle_world_step / oracle_run_closed_loop of oracle/oracle_api.cpp; in jo_run_closed_loop, the models each
// world step may carry: the episode metrics of episode_metrics.cpp (alone: jo_metrics_step), the reactive agents of
// agent_model.cpp (alone: jo_react_step) and their lane changes of lane_change.cpp (alone: jo_lane_change_step); and the V2X launch
// of v2x_world.cpp between a cycle and its world step (alone: jo_v2x_cycle, its data builder: jo_v2x_data).
#include <algorithm>
#include <atomic>
#include <cstring>
#include <thread>
#include <vector>
#include "agent_model.h"
#include "episode_metrics.h"
#include "lane_change.h"
#include "v2x_world.h"
#include "world_junction.h"
#include "../../oracle/cshare_spec.h"

namespace {
junction::JMap g_map; bool g_have_map = false;
// the warning list through GlobalToWGS84, as the handlers read it
void wp_gps(const dp_params& p, const double* wp_x, const double* wp_y, int n_wp, std::vector<double>& la, std::vector<double>& lo) {
    la.resize((size_t)n_wp); lo.resize((size_t)n_wp);
    for (int i = 0; i < n_wp; ++i) spec::global_to_wgs84(spec::Datum{p.lat0, p.lng0, p.k_lat, p.k_lng}, wp_x[i], wp_y[i], &la[i], &lo[i]);
}
}  // namespace

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

// the closed loop: the junction world step between the cycles of oracle/, the same arrays as oracle_run_closed_loop.  Each model is
// armed by a non-null pair, or off with both NULL: mp / met[n] the episode metrics of include/dmpp_b200.h section 11, accumulated
// after every world step; am / v0[n][max_obs] the reactive agents of section 12, before every world step; lp / lcs[n][max_obs]
// (with am) their lane changes of section 13, states initialised by the placement step and holding the final states; vp / spec[n]
// (wp_x / wp_y[n_wp], flags[n] nullable, stats[n]) the V2X events of section 14 between every cycle and its world step
long long jo_run_closed_loop(const dp_params* p, const dp_world_params* wp, int n, int cycles, int max_obs, dp_scene_hdr* hdr,
                             dp_agent* agents, double* ox, double* oy, dp_plan_record* rec, dp_scene_hdr* hdr_log, double* obs_log_x,
                             double* obs_log_y, double* path_xy, dp_carry* carry_out, double* last_path_out, int threads,
                             int32_t* ub_scene, const dp_metrics_params* mp, dp_episode_metrics* met, const dp_agent_model_params* am,
                             const double* v0, const dp_lane_change_params* lp, dp_lane_change_state* lcs, const dp_v2x_world_params* vp,
                             const dp_v2x_event_spec* spec, const double* wp_x, const double* wp_y, int n_wp, dp_v2x_flags* flags,
                             dp_v2x_episode_stats* stats) {
    if (!g_have_map) return -1;
    if ((!mp) != (!met) || (!am) != (!v0) || (!lp) != (!lcs) || (lcs && !v0) || (!vp) != (!spec) || (spec && !stats)) return -1;
    if (threads < 1) threads = 1;
    std::vector<double> wla, wlo;
    if (spec) wp_gps(*p, wp_x, wp_y, n_wp, wla, wlo);
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
            if (met) metrics::init(met[s]);
            if (lcs) lanechg::init(ag, std::min((int)hdr[s].n_obs, max_obs), lcs + (size_t)s * max_obs);
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
                if (spec) v2x::cycle(g_map, *p, *vp, spec[s], wla.data(), wlo.data(), hdr[s], c, rec + e, stats[s], flags ? flags + s : nullptr);
                const dp_scene_hdr h0 = hdr[s];
                if (lcs) lanechg::step(g_map, *wp, *am, *lp, h0, ag, std::min((int)h0.n_obs, max_obs), v0 + (size_t)s * max_obs,
                                       lcs + (size_t)s * max_obs);
                else if (am) agents::react(g_map, *wp, *am, h0, ag, std::min((int)h0.n_obs, max_obs), v0 + (size_t)s * max_obs);
                junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, rec + e, st.last_x, st.last_y);
                if (met) metrics::update(g_map, *wp, *mp, met[s], h0, hdr[s], ag, sx, sy, std::min((int)h0.n_obs, max_obs), rec[e]);
            }
            if (spec) v2x::cycle(g_map, *p, *vp, spec[s], wla.data(), wlo.data(), hdr[s], cycles, nullptr, stats[s], flags ? flags + s : nullptr);
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

// the react phase alone, for every scene (agents[n][max_obs], v0[n][max_obs], k < min(n_obs, max_obs)), as the armed kernel runs
// it at the start of a step with a record; a header that names no lane leaves its agents alone
int jo_react_step(const dp_world_params* wp, const dp_agent_model_params* am, int n, int max_obs, const dp_scene_hdr* hdr, dp_agent* agents,
                  const double* v0) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s)
        agents::react(g_map, *wp, *am, hdr[s], agents + (size_t)s * max_obs, std::min((int)hdr[s].n_obs, max_obs), v0 + (size_t)s * max_obs);
    return 0;
}

int jo_agent_model_sizeof(void) { return (int)sizeof(dp_agent_model_params); }

// the react and lane-change phases alone, for every scene, in place (agents and lcs [n][max_obs], k < min(n_obs, max_obs)), as the
// armed kernel runs them at the start of a step with a record; a header that names no lane leaves its agents and states alone
int jo_lane_change_step(const dp_world_params* wp, const dp_agent_model_params* am, const dp_lane_change_params* lp, int n, int max_obs,
                        const dp_scene_hdr* hdr, dp_agent* agents, const double* v0, dp_lane_change_state* lcs) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s)
        lanechg::step(g_map, *wp, *am, *lp, hdr[s], agents + (size_t)s * max_obs, std::min((int)hdr[s].n_obs, max_obs),
                      v0 + (size_t)s * max_obs, lcs + (size_t)s * max_obs);
    return 0;
}

int jo_lane_change_sizeof(int which) { return which ? (int)sizeof(dp_lane_change_state) : (int)sizeof(dp_lane_change_params); }

// one world step plus its metric update for every scene, as the armed kernel does it: rec == NULL initialises the rows (also for a
// header that names no lane); a header that names no lane leaves its world and its row alone
int jo_metrics_step(const dp_params* p, const dp_world_params* wp, const dp_metrics_params* mp, int n, int max_obs, dp_scene_hdr* hdr,
                    dp_agent* agents, double* ox, double* oy, const dp_plan_record* rec, const double* last_path, dp_episode_metrics* met) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s) {
        if (!rec) metrics::init(met[s]);
        if (!metrics::header_valid(g_map.m, hdr[s])) continue;
        const dp_scene_hdr h0 = hdr[s];
        dp_agent* ag = agents + (size_t)s * max_obs;
        double* sx = ox + (size_t)s * max_obs; double* sy = oy + (size_t)s * max_obs;
        junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, rec ? rec + s : nullptr, last_path ? last_path + (size_t)s * 400 : nullptr,
                             last_path ? last_path + (size_t)s * 400 + 200 : nullptr);
        if (rec) metrics::update(g_map, *wp, *mp, met[s], h0, hdr[s], ag, sx, sy, std::min((int)h0.n_obs, max_obs), rec[s]);
    }
    return 0;
}

int jo_metrics_sizeof(void) { return (int)sizeof(dp_episode_metrics); }

void jo_sincos_deg(double a, double* c, double* s) { spec::spec_sincos_deg(a, c, s); }

// the V2X data builder alone for every world at cycle k: data[n], and aux[n][3] = (d, spat_state, on + 2 * ped_on); headers must
// name a lane
int jo_v2x_data(const dp_params* p, int n, const dp_v2x_event_spec* spec, const dp_scene_hdr* hdr, int k, dp_v2x_data* data, double* aux) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s) {
        if (!metrics::header_valid(g_map.m, hdr[s])) return -1;
        const v2x::World w = v2x::build(g_map, *p, spec[s], hdr[s], k);
        data[s] = w.v;
        aux[3 * s] = w.d; aux[3 * s + 1] = w.state; aux[3 * s + 2] = (w.on ? 1 : 0) + (w.ped_on ? 2 : 0);
    }
    return 0;
}

// one V2X launch for every world, in place (rec[n] nullable: the tally), as dp_v2x_world_dev runs it
int jo_v2x_cycle(const dp_params* p, const dp_v2x_world_params* vp, int n, const dp_v2x_event_spec* spec, const double* wp_x, const double* wp_y,
                 int n_wp, const dp_scene_hdr* hdr, dp_plan_record* rec, int k, dp_v2x_flags* flags, dp_v2x_episode_stats* stats) {
    if (!g_have_map) return -1;
    std::vector<double> wla, wlo;
    wp_gps(*p, wp_x, wp_y, n_wp, wla, wlo);
    for (int s = 0; s < n; ++s)
        v2x::cycle(g_map, *p, *vp, spec[s], wla.data(), wlo.data(), hdr[s], k, rec ? rec + s : nullptr, stats[s], flags ? flags + s : nullptr);
    return 0;
}

// GlobalToWGS84 of n points
void jo_gps(const dp_params* p, int n, const double* x, const double* y, double* lat, double* lng) {
    for (int i = 0; i < n; ++i) spec::global_to_wgs84(spec::Datum{p->lat0, p->lng0, p->k_lat, p->k_lng}, x[i], y[i], lat + i, lng + i);
}

int jo_v2x_sizeof(int which) { return which ? (int)sizeof(dp_v2x_episode_stats) : (int)sizeof(dp_v2x_event_spec); }

}  // extern "C"
