// tools/junction_oracle/junction_api.cpp -- TEST INFRASTRUCTURE. C API of libjunction_oracle.so: the restated cycle of oracle/
// (planner_oracle.cpp, compiled in unchanged) with the junction world step of world_junction.cpp between its cycles; the
// same arrays as oracle_world_step / oracle_run_closed_loop of oracle/oracle_api.cpp; in jo_run_closed_loop, the models each
// world step may carry (in parts: jo_run_closed_loop_part): the episode metrics of episode_metrics.cpp (alone: jo_metrics_step), the reactive agents of
// agent_model.cpp (alone: jo_react_step) and their lane changes of lane_change.cpp (alone: jo_lane_change_step); and the V2X launch
// of v2x_world.cpp between a cycle and its world step (alone: jo_v2x_cycle, its data builder: jo_v2x_data); and the agents that
// obey the V2X events of v2x_traffic.cpp (alone: jo_traffic_step, its candidates: jo_traffic_leader / jo_traffic_side); and the view of
// the V2X road users every cycle runs on, v2x_obstacles.cpp (alone: jo_v2x_obstacles_view).
#include <algorithm>
#include <atomic>
#include <cstring>
#include <thread>
#include <vector>
#include "agent_model.h"
#include "episode_metrics.h"
#include "lane_change.h"
#include "v2x_obstacles.h"
#include "v2x_traffic.h"
#include "v2x_world.h"
#include "world_junction.h"
#include "world_split.h"
#include "../../oracle/cshare_spec.h"

namespace {
junction::JMap g_map; bool g_have_map = false;
// section 15's row update of one world after its motion, with the step's leader kinds
void traffic_update(const dp_params& p, const dp_agent_model_params& am, const traffic::World& tw, dp_v2x_traffic_stats& r, const dp_agent* a1,
                    const dp_agent* a2, const double* ox, const double* oy, int n, const int* kinds) {
    int line_n = 0, ped_n = 0;
    for (int k = 0; k < n; ++k) { line_n += kinds[k] == 1; ped_n += kinds[k] == 2; }
    traffic::update(g_map, tw, am, p.vehicle_width, r, a1, a2, ox, oy, n, line_n, ped_n);
}
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

// a closed loop in parts (include/dmpp_b200.h section 17): cycles k0 .. k0 + cycles - 1 of the episode, rec / hdr_log / obs_log_* /
// path_xy indexed by the part's cycle j.  k0 == 0: a fresh state (reset_state), the placement step and the row inits; k0 > 0: the
// world hdr / agents / ox / oy, the rows and states, and carry[n] / last_path[n][2][200] (in and out) continue where the previous
// part left them, and prev_rec[n] holds the records of cycle k0 - 1 (required with os).  finish: the V2X and obstacles tallies at
// cycle k0 + cycles.  Each model is armed by a non-null pair, or off with both NULL: mp / met[n] the episode metrics of section 11,
// accumulated after every world step; am / v0[n][max_obs] the reactive agents of section 12, before every world step; lp /
// lcs[n][max_obs] (with am) their lane changes of section 13, states initialised by the placement step; vp / spec[n] (wp_x / wp_y[n_wp],
// flags[n] nullable, stats[n]) the V2X events of section 14 between every cycle and its world step; tp / ts[n] (with am and vp) the
// agents that obey them, section 15; op / os[n] (with vp) the V2X road users the planner sees, section 16: every cycle runs on the view
// its obstacles launch builds, and hdr_log / obs_log_* record the views (slots beyond a view's n_obs hold zeros from the part's start)
long long jo_run_closed_loop_part(const dp_params* p, const dp_world_params* wp, int n, int k0, int cycles, int finish, int max_obs,
                                  dp_scene_hdr* hdr, dp_agent* agents, double* ox, double* oy, const dp_plan_record* prev_rec, dp_plan_record* rec,
                                  dp_scene_hdr* hdr_log, double* obs_log_x, double* obs_log_y, double* path_xy, dp_carry* carry,
                                  double* last_path, int threads, int32_t* ub_scene, const dp_metrics_params* mp, dp_episode_metrics* met,
                                  const dp_agent_model_params* am, const double* v0, const dp_lane_change_params* lp, dp_lane_change_state* lcs,
                                  const dp_v2x_world_params* vp, const dp_v2x_event_spec* spec, const double* wp_x, const double* wp_y,
                                  int n_wp, dp_v2x_flags* flags, dp_v2x_episode_stats* stats, const dp_v2x_traffic_params* tp,
                                  dp_v2x_traffic_stats* ts, const dp_v2x_obstacle_params* op, dp_v2x_obstacle_stats* os) {
    if (!g_have_map) return -1;
    if ((!mp) != (!met) || (!am) != (!v0) || (!lp) != (!lcs) || (lcs && !v0) || (!vp) != (!spec) || (spec && !stats)) return -1;
    if ((!tp) != (!ts) || (ts && (!v0 || !spec))) return -1;
    if ((!op) != (!os) || (os && !spec)) return -1;
    if (k0 < 0 || cycles < 0 || (finish != 0 && finish != 1) || (k0 > 0 && (!carry || !last_path || (os && !prev_rec)))) return -1;
    if (threads < 1) threads = 1;
    std::vector<double> wla, wlo;
    if (spec) wp_gps(*p, wp_x, wp_y, n_wp, wla, wlo);
    std::atomic<long long> ub(0);
    auto work = [&](int s0, int s1) {
        long long lub = 0;
        for (int s = s0; s < s1; ++s) {
            const long long lub0 = lub;
            oracle::SceneState st;
            dp_agent* ag = agents + (size_t)s * max_obs;
            double* sx = ox + (size_t)s * max_obs; double* sy = oy + (size_t)s * max_obs;
            if (k0 == 0) {
                oracle::reset_state(st);
                junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, nullptr, nullptr, nullptr);
                if (met) metrics::init(met[s]);
                if (lcs) lanechg::init(ag, std::min((int)hdr[s].n_obs, max_obs), lcs + (size_t)s * max_obs);
                if (ts) traffic::init(ts[s]);
            } else {
                st.c = carry[s];
                std::memcpy(st.last_x, last_path + (size_t)s * 400, sizeof(st.last_x));
                std::memcpy(st.last_y, last_path + (size_t)s * 400 + 200, sizeof(st.last_y));
            }
            std::vector<int> kinds((size_t)max_obs);
            std::vector<dp_agent> a1((size_t)max_obs);
            // the cycle's inputs: the world, or with os the view of it (slots beyond the view's n_obs keep what they held)
            dp_scene_hdr hv{};
            std::vector<double> vx((size_t)max_obs), vy((size_t)max_obs);
            // the records of the cycle before j (prev_rec at j == 0 of a continued part)
            auto prev_of = [&](int j) -> const dp_plan_record* {
                return j > 0 ? rec + (size_t)(j - 1) * n + s : (k0 > 0 ? prev_rec + s : nullptr);
            };
            for (int j = 0; j < cycles; ++j) {
                const int c = k0 + j;
                const size_t e = (size_t)j * n + s;
                if (os) v2xobs::launch(g_map, *op, max_obs, spec[s], wp_x, wp_y, hdr[s], sx, sy, prev_of(j), c, false, &hv, vx.data(), vy.data(),
                                       os[s]);
                const dp_scene_hdr& ch = os ? hv : hdr[s];
                const double* cx = os ? vx.data() : sx;
                const double* cy = os ? vy.data() : sy;
                if (hdr_log) hdr_log[e] = ch;
                if (obs_log_x) std::memcpy(obs_log_x + e * max_obs, cx, sizeof(double) * max_obs);
                if (obs_log_y) std::memcpy(obs_log_y + e * max_obs, cy, sizeof(double) * max_obs);
                oracle::CycleOut o{};
                o.rec = rec + e;
                o.path_xy = path_xy ? path_xy + e * 400 : nullptr;
                oracle::cycle(g_map.m, *p, ch, cx, cy, st, o, false);
                lub += o.ub_hits;
                if (spec) v2x::cycle(g_map, *p, *vp, spec[s], wla.data(), wlo.data(), hdr[s], c, rec + e, stats[s], flags ? flags + s : nullptr);
                const dp_scene_hdr h0 = hdr[s];
                const int na = std::min((int)h0.n_obs, max_obs);
                traffic::World tw;
                if (ts) tw = traffic::world(g_map, *tp, spec[s], h0, c);
                const traffic::World* twp = ts ? &tw : nullptr;
                if (lcs) lanechg::step(g_map, *wp, *am, *lp, h0, ag, na, v0 + (size_t)s * max_obs, lcs + (size_t)s * max_obs, twp, kinds.data());
                else if (am) agents::react(g_map, *wp, *am, h0, ag, na, v0 + (size_t)s * max_obs, nullptr, twp, kinds.data());
                if (ts) std::copy(ag, ag + na, a1.begin());
                junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, rec + e, st.last_x, st.last_y);
                if (ts && metrics::header_valid(g_map.m, h0)) traffic_update(*p, *am, tw, ts[s], a1.data(), ag, sx, sy, na, kinds.data());
                if (met) metrics::update(g_map, *wp, *mp, met[s], h0, hdr[s], ag, sx, sy, std::min((int)h0.n_obs, max_obs), rec[e]);
            }
            if (finish) {
                if (spec) v2x::cycle(g_map, *p, *vp, spec[s], wla.data(), wlo.data(), hdr[s], k0 + cycles, nullptr, stats[s], flags ? flags + s : nullptr);
                if (os) v2xobs::launch(g_map, *op, max_obs, spec[s], wp_x, wp_y, hdr[s], sx, sy, prev_of(cycles), k0 + cycles, true, nullptr, nullptr,
                                       nullptr, os[s]);
            }
            if (ub_scene) ub_scene[s] = (int32_t)(lub - lub0);
            if (carry) carry[s] = st.c;
            if (last_path) {
                std::memcpy(last_path + (size_t)s * 400, st.last_x, sizeof(st.last_x));
                std::memcpy(last_path + (size_t)s * 400 + 200, st.last_y, sizeof(st.last_y));
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

// the closed loop: the junction world step between the cycles of oracle/, the same arrays as oracle_run_closed_loop, and the models
// of jo_run_closed_loop_part: the whole episode as one part (k0 = 0, finish = 1) from a fresh state
long long jo_run_closed_loop(const dp_params* p, const dp_world_params* wp, int n, int cycles, int max_obs, dp_scene_hdr* hdr,
                             dp_agent* agents, double* ox, double* oy, dp_plan_record* rec, dp_scene_hdr* hdr_log, double* obs_log_x,
                             double* obs_log_y, double* path_xy, dp_carry* carry_out, double* last_path_out, int threads,
                             int32_t* ub_scene, const dp_metrics_params* mp, dp_episode_metrics* met, const dp_agent_model_params* am,
                             const double* v0, const dp_lane_change_params* lp, dp_lane_change_state* lcs, const dp_v2x_world_params* vp,
                             const dp_v2x_event_spec* spec, const double* wp_x, const double* wp_y, int n_wp, dp_v2x_flags* flags,
                             dp_v2x_episode_stats* stats, const dp_v2x_traffic_params* tp, dp_v2x_traffic_stats* ts,
                             const dp_v2x_obstacle_params* op, dp_v2x_obstacle_stats* os) {
    return jo_run_closed_loop_part(p, wp, n, 0, cycles, 1, max_obs, hdr, agents, ox, oy, nullptr, rec, hdr_log, obs_log_x, obs_log_y, path_xy,
                                   carry_out, last_path_out, threads, ub_scene, mp, met, am, v0, lp, lcs, vp, spec, wp_x, wp_y, n_wp, flags,
                                   stats, tp, ts, op, os);
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

// one world step of cycle k with the agents obeying the V2X events, for every scene, in place, as the TRAFFIC kernel runs it: the
// react phase (with lp / lcs non-null: and the lane changes), the world step, the row update; kinds[n][max_obs] (nullable) the leader
// kinds.  rec == NULL initialises the rows and runs the placement step.  The ego walks its last_path[n][400] with rec
int jo_traffic_step(const dp_params* p, const dp_world_params* wp, const dp_agent_model_params* am, const dp_lane_change_params* lp,
                    const dp_v2x_traffic_params* tp, int n, int max_obs, const dp_v2x_event_spec* spec, int k, dp_scene_hdr* hdr, dp_agent* agents,
                    double* ox, double* oy, const double* v0, dp_lane_change_state* lcs, const dp_plan_record* rec, const double* last_path,
                    dp_v2x_traffic_stats* ts, int32_t* kinds) {
    if (!g_have_map || (!lp) != (!lcs)) return -1;
    std::vector<int> kd((size_t)max_obs);
    std::vector<dp_agent> a1((size_t)max_obs);
    for (int s = 0; s < n; ++s) {
        dp_agent* ag = agents + (size_t)s * max_obs;
        double* sx = ox + (size_t)s * max_obs; double* sy = oy + (size_t)s * max_obs;
        const double* lx = last_path ? last_path + (size_t)s * 400 : nullptr;
        if (!rec) {
            traffic::init(ts[s]);
            if (lcs) lanechg::init(ag, std::min((int)hdr[s].n_obs, max_obs), lcs + (size_t)s * max_obs);
            junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, nullptr, nullptr, nullptr);
            continue;
        }
        const dp_scene_hdr h0 = hdr[s];
        const int na = std::min((int)h0.n_obs, max_obs);
        const traffic::World tw = traffic::world(g_map, *tp, spec[s], h0, k);
        std::fill(kd.begin(), kd.end(), 0);
        if (lcs) lanechg::step(g_map, *wp, *am, *lp, h0, ag, na, v0 + (size_t)s * max_obs, lcs + (size_t)s * max_obs, &tw, kd.data());
        else agents::react(g_map, *wp, *am, h0, ag, na, v0 + (size_t)s * max_obs, nullptr, &tw, kd.data());
        std::copy(ag, ag + na, a1.begin());
        junction::world_step(g_map, *p, *wp, hdr[s], ag, sx, sy, rec + s, lx, lx ? lx + 200 : nullptr);
        if (metrics::header_valid(g_map.m, h0)) traffic_update(*p, *am, tw, ts[s], a1.data(), ag, sx, sy, na, kd.data());
        if (kinds)
            for (int j = 0; j < max_obs; ++j) kinds[(size_t)s * max_obs + j] = j < na ? kd[j] : 0;
    }
    return 0;
}

// section 15's candidates alone, for n independent agents of world s (spec[s], hdr[s] at cycle k[s]): the section 12 leader after a
// vehicle scan, lanes[s] = (l0, l1, l2), x[s] = (D1, D2, sk, v, u, best), iv[s] = (i, lead) -> out[s] = (best, lead, kind)
int jo_traffic_leader(const dp_v2x_traffic_params* tp, const dp_agent_model_params* am, int n, const dp_v2x_event_spec* spec,
                      const dp_scene_hdr* hdr, const int32_t* k, const int32_t* lanes, const double* x, const int32_t* iv, double* out) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s) {
        const traffic::World w = traffic::world(g_map, *tp, spec[s], hdr[s], k[s]);
        const double* a = x + 6 * s;
        bool lead = iv[2 * s + 1] != 0;
        double best = a[5];
        const int kind = traffic::leader(g_map, w, *am, lanes[3 * s], lanes[3 * s + 1], lanes[3 * s + 2], a[0], a[1], a[2], a[3], iv[2 * s],
                                         a[4], &lead, &best);
        out[3 * s] = best; out[3 * s + 1] = lead; out[3 * s + 2] = kind;
    }
    return 0;
}

// ... and on a target lane: lanes[s] = (m, i_m), x[s] = (s_m, u, v, g), lead[s] -> out[s] = (g, lead, won)
int jo_traffic_side(const dp_v2x_traffic_params* tp, const dp_agent_model_params* am, int n, const dp_v2x_event_spec* spec, const dp_scene_hdr* hdr,
                    const int32_t* k, const int32_t* lanes, const double* x, const int32_t* lead_in, double* out) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s) {
        const traffic::World w = traffic::world(g_map, *tp, spec[s], hdr[s], k[s]);
        const double* a = x + 4 * s;
        bool lead = lead_in[s] != 0;
        double g = a[3];
        const bool won = traffic::side(g_map, w, *am, lanes[2 * s], lanes[2 * s + 1], a[0], a[1], a[2], &lead, &g);
        out[3 * s] = g; out[3 * s + 1] = lead; out[3 * s + 2] = won;
    }
    return 0;
}

// one obstacles launch of cycle k for every world, as dp_v2x_obstacles_dev runs it: hdr[n] / ox / oy[n][max_obs] the world,
// prev[n] (nullable) the records of cycle k - 1, views hv[n] / vx / vy[n][max_obs] (not written on the tally), stats[n] in place
int jo_v2x_obstacles_view(const dp_v2x_obstacle_params* op, int max_obs, int n, const dp_v2x_event_spec* spec, const double* wp_x,
                          const double* wp_y, const dp_scene_hdr* hdr, const double* ox, const double* oy, const dp_plan_record* prev, int k,
                          int tally, dp_scene_hdr* hv, double* vx, double* vy, dp_v2x_obstacle_stats* stats) {
    if (!g_have_map) return -1;
    for (int s = 0; s < n; ++s) {
        const size_t o = (size_t)s * max_obs;
        v2xobs::launch(g_map, *op, max_obs, spec[s], wp_x, wp_y, hdr[s], ox + o, oy + o, prev ? prev + s : nullptr, k, tally != 0,
                       tally ? nullptr : hv + s, tally ? nullptr : vx + o, tally ? nullptr : vy + o, stats[s]);
    }
    return 0;
}

int jo_v2x_obstacles_sizeof(int which) { return which ? (int)sizeof(dp_v2x_obstacle_stats) : (int)sizeof(dp_v2x_obstacle_params); }

int jo_traffic_sizeof(int which) { return which ? (int)sizeof(dp_v2x_traffic_stats) : (int)sizeof(dp_v2x_traffic_params); }

// the select launch of a split (include/dmpp_b200.h section 18) for the n / M populations of worlds 0 .. n-1: met[n], rows[n] and
// groups[n / M] in place, map[n] the source of every destination (relative to world 0), -1 elsewhere
int jo_world_split_select(const dp_split_params* p, int n, int level, const dp_episode_metrics* met, dp_split_row* rows,
                          dp_split_group* groups, int32_t* map) {
    const int M = p->group;
    if (M < 1 || M > 1024 || n < 0 || n % M != 0 || level < 0) return -1;
    for (int g = 0; g < n / M; ++g) {
        const size_t o = (size_t)g * M;
        split::select(*p, M, g, level, met + o, rows + o, groups[g], map + o);
        for (int j = 0; j < M; ++j)
            if (map[o + j] >= 0) map[o + j] += (int32_t)o;
    }
    return 0;
}

// the perturb launch of a split: every world i < n, agents[n][max_obs] and (nullable) v0[n][max_obs] in place
int jo_world_perturb(const dp_split_params* p, int n, int level, int max_obs, const dp_scene_hdr* hdr, dp_agent* agents, double* v0) {
    for (int i = 0; i < n; ++i)
        split::perturb(*p, level, i, hdr[i].n_obs, max_obs, agents + (size_t)i * max_obs, v0 ? v0 + (size_t)i * max_obs : nullptr);
    return 0;
}

// y[i] = spec_exp(x[i])
int jo_spec_exp(int n, const double* x, double* y) {
    for (int i = 0; i < n; ++i) y[i] = split::spec_exp(x[i]);
    return 0;
}

int jo_split_sizeof(int which) {
    return which == 0 ? (int)sizeof(dp_split_params) : which == 1 ? (int)sizeof(dp_split_row) : (int)sizeof(dp_split_group);
}

}  // extern "C"
