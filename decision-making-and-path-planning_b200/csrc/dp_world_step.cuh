// csrc/dp_world_step.cuh -- the world step of the closed-loop episode runner (dp_world_kernel, see dp_world.cu), with the
// episode metrics of include/dmpp_b200.h section 11, the reactive agents of section 12 and their lane changes (section 13) as
// compile-time options, and its launcher WorldStep<METRICS, REACT, LANECHG>.  dp_world.cu instantiates the disarmed kernels
// (METRICS = REACT = false), dp_world_metrics.cu the metrics instances, dp_world_agents.cu the reactive ones and
// dp_world_lanechange.cu the lane-changing ones: kept in separate translation units, the disarmed instances compile to exactly
// what they compiled to before the options existed.
#pragma once
#include <type_traits>

#include "dp_kernels.h"

namespace {
constexpr int WPB = 4;   // warps (= scenes) per CTA

__device__ __forceinline__ double seg_len(const double2 a, const double2 b, double* ddx, double* ddy) {
    *ddx = b.x - a.x; *ddy = b.y - a.y;
    return sqrt(*ddx * *ddx + *ddy * *ddy);
}

constexpr int WORLD_MAX_HOPS = 8;   // successor lanes an agent may enter in one step (tools/junction_oracle/world_junction.cpp)

// nearest point of map lane gl to (x, y) in [lo, hi] clipped to the lane, lane-parallel: squared distance (returned in every
// lane), index in *bi (lowest on ties, lo when the window is empty) -- the strict '<' scan of the specification
__device__ __forceinline__ double warp_nearest(const DevMap& m, int gl, int lo, int hi, double x, double y, int lane, int* bi_out) {
    const int off = m.lane_pt_off[gl], cnt = m.lane_pt_off[gl + 1] - off;
    if (lo < 0) lo = 0;
    if (hi > cnt - 1) hi = cnt - 1;
    double be = __longlong_as_double(0x7ff0000000000000LL);
    int bi = 0x7fffffff;
    for (int i = lo + lane; i <= hi; i += 32) {
        const double2 q = m.xy[off + i];
        const double dx = x - q.x, dy = y - q.y;
        const double e = dx * dx + dy * dy;
        if (e < be) { be = e; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oe = __shfl_xor_sync(DP_FULL, be, o);
        const int oi = __shfl_xor_sync(DP_FULL, bi, o);
        if (oe < be || (oe == be && oi < bi)) { be = oe; bi = oi; }
    }
    *bi_out = bi == 0x7fffffff ? lo : bi;
    return be;
}

// the ego's connector (include/dmpp_b200.h section 9): lowest c leaving (road, lane_num) towards next_road, -1 none; warp-uniform
__device__ __forceinline__ int ego_connector(const DevMap& m, int road, int lane_num, int next_road, int lane) {
    if (next_road == road) return -1;
    for (int base = 0; base < m.n_conn; base += 32) {
        const int c = base + lane;
        bool hit = false;
        if (c < m.n_conn) { const dp_connector k = m.conn[c]; hit = k.last_road == road && k.next_road == next_road && k.last_lane == lane_num; }
        const unsigned b = __ballot_sync(DP_FULL, hit);
        if (b) return base + __ffs(b) - 1;
    }
    return -1;
}

// ---- episode metrics (include/dmpp_b200.h section 11): the row of a scene travels as MET_WORDS doubles, one per lane ----
constexpr int MET_WORDS = (int)(sizeof(dp_episode_metrics) / sizeof(double));
static_assert(sizeof(dp_episode_metrics) == 192, "dp_episode_metrics is 192 bytes");

__device__ __forceinline__ void metrics_init(dp_episode_metrics& r) {
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    r.distance = 0; r.min_clearance = inf; r.min_lead_gap = inf; r.min_ttc = inf;
    r.max_accel = -inf; r.min_accel = inf; r.max_abs_jerk = 0; r.last_accel = 0;
    r.max_abs_lat_err = 0; r.max_abs_dir_err = 0;
    r.steps = 0; r.first_collision_step = -1; r.first_collision_agent = -1;
    r.collision_steps = 0; r.collision_steps_front = 0; r.collision_steps_rear = 0; r.ttc_warn_steps = 0;
    r.stopped_steps = 0; r.end_stop_steps = 0; r.replans = 0; r.aeb_steps = 0;
    r.accel_steps = 0; r.last_behavior = -1; r.behavior_switches = 0;
    for (int i = 0; i < 8; ++i) r.behavior_steps[i] = 0;
    for (int i = 0; i < 6; ++i) r.pad[i] = 0;
}

// the scalar part of one step's update (lane 0), given the warp's minima over the agents: dmin (clearance), gmin / tmin (lead gap
// / ttc), first (lowest agent inside the box, -1 none), front / rear (an agent inside at lon >= 0 / lon < 0)
__device__ __forceinline__ void metrics_update(dp_episode_metrics& r, const dp_metrics_params& mp, const dp_plan_record& rc, double v,
                                               double vn, double dt, double ds, bool at_end, double dmin, double gmin, double tmin,
                                               int first, bool front, bool rear) {
    const int step_no = r.steps + 1;
    r.distance = r.distance + ds;
    if (dmin < r.min_clearance) r.min_clearance = dmin;
    if (gmin < r.min_lead_gap) r.min_lead_gap = gmin;
    if (tmin < r.min_ttc) r.min_ttc = tmin;
    if (dt > 0) {
        const double a = (vn - v) / 3.6 / dt;
        if (a > r.max_accel) r.max_accel = a;
        if (a < r.min_accel) r.min_accel = a;
        if (r.accel_steps > 0) {
            const double j = fabs(a - r.last_accel) / dt;
            if (j > r.max_abs_jerk) r.max_abs_jerk = j;
        }
        r.last_accel = a; r.accel_steps += 1;
    }
    const double le = fabs(rc.path_lat_dis), de = fabs(rc.path_dir_err);
    if (le > r.max_abs_lat_err) r.max_abs_lat_err = le;
    if (de > r.max_abs_dir_err) r.max_abs_dir_err = de;
    if (first >= 0) {
        r.collision_steps += 1;
        if (r.first_collision_step < 0) { r.first_collision_step = step_no; r.first_collision_agent = first; }
    }
    if (front) r.collision_steps_front += 1;
    if (rear) r.collision_steps_rear += 1;
    if (tmin < mp.ttc_warn) r.ttc_warn_steps += 1;
    if (vn == 0) r.stopped_steps += 1;
    if (at_end) r.end_stop_steps += 1;
    r.replans += rc.afresh_planning; r.aeb_steps += rc.acc_flag;
    const int b = rc.behavior;
    if (b < 8) r.behavior_steps[b] += 1;
    if (r.steps > 0 && b != r.last_behavior) r.behavior_switches += 1;
    r.last_behavior = b;
    r.steps = step_no;
}

// the per-lane state of the armed instances: this lane's word of the row (loaded at entry), the step's distance and end_margin
// stop, the ego frame (c, s) of the new pose, and the minima / flags over the lane's agents
struct MetricLane {
    double word = 0, ds = 0, c = 1, s = 0;
    double d = __builtin_huge_val(), gap = d, ttc = d;
    int first = 0x7fffffff;
    bool at_end = false, front = false, rear = false;
};
struct NoMetrics {};

// the end of an armed step: the warp's minima over the agents (order-free: no NaN and no -0 among d, gap, ttc), the lowest agent
// inside the box (each lane scanned its agents in increasing order, so it is an integer min), lane 0's update of the row staged
// in shared memory, then one coalesced store of the row
__device__ __forceinline__ void metrics_step(MetricLane& ml, double* row, dp_episode_metrics* out, int lane, const dp_metrics_params& mp,
                                             const dp_plan_record& rc, double v, double vn, double dt) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ml.d = fmin(ml.d, __shfl_xor_sync(DP_FULL, ml.d, o));
        ml.gap = fmin(ml.gap, __shfl_xor_sync(DP_FULL, ml.gap, o));
        ml.ttc = fmin(ml.ttc, __shfl_xor_sync(DP_FULL, ml.ttc, o));
    }
    const int first = (int)__reduce_min_sync(DP_FULL, (unsigned)ml.first);
    const bool front = __any_sync(DP_FULL, ml.front), rear = __any_sync(DP_FULL, ml.rear);
    if (lane < MET_WORDS) row[lane] = ml.word;
    __syncwarp();
    if (lane == 0)
        metrics_update(*reinterpret_cast<dp_episode_metrics*>(row), mp, rc, v, vn, dt, ml.ds, ml.at_end, ml.d, ml.gap, ml.ttc,
                       first == 0x7fffffff ? -1 : first, front, rear);
    __syncwarp();
    if (lane < MET_WORDS) reinterpret_cast<double*>(out)[lane] = row[lane];
}

// ---- reactive agents (include/dmpp_b200.h section 12): the intelligent driver model on the lane chain ----
constexpr int REACT_SLOT_BYTES = 24;   // staged per agent slot and world: (station, speed) as a double2 and the lane (int, padded)
// bytes of dynamic shared memory per warp (16-byte aligned: the double2 array comes first)
__host__ __device__ constexpr size_t react_stage_bytes(int max_obs) { return ((size_t)max_obs * REACT_SLOT_BYTES + 15) & ~(size_t)15; }
static_assert(WPB * (react_stage_bytes(DP_AGENT_MODEL_MAX_OBS) + (32 + 2 * MET_WORDS) * 4) <= 227 * 1024,
              "the staging of DP_AGENT_MODEL_MAX_OBS agent slots fits the shared memory of a CTA");
struct AgentModel {
    dp_agent_model_params p;
    const double* v0;                  // [n][max_obs] desired speeds
};
// the model of the LANECHG instances (section 13): the agent model plus the lane-change parameters and states.  A type of its own,
// so that the kernel parameters of the other instances stay what they were
struct LaneChangeModel : AgentModel {
    dp_lane_change_params lc;
    dp_lane_change_state* lcs;         // [n][max_obs]
};

// length of map lane gl: the last entry of its sequential prefix of segment lengths
__device__ __forceinline__ double lane_len(const DevMap& m, int gl) { return m.cump[m.lane_pt_off[gl + 1] - 1]; }

// section 12's IDM acceleration with its clamp (lead false: free road); sab = 2.0 * sqrt(a_max * b)
__device__ __forceinline__ double idm_accel(const dp_agent_model_params& p, double sab, double v, double vd, bool lead, double g, double vl) {
    const double r = v / vd;
    double fr = r * r;
    fr = fr * fr;
    double acc;
    if (lead) {
        const double dv = v - vl;
        double z = v * p.T + v * dv / sab;
        if (z < 0) z = 0;
        const double ss = p.s0 + z;
        if (g > 0) { const double q = ss / g; acc = p.a_max * (1.0 - fr - q * q); }
        else acc = -p.b_max;
    } else acc = p.a_max * (1.0 - fr);
    if (acc < -p.b_max) acc = -p.b_max;
    return acc;
}

// ---- lane-changing agents (include/dmpp_b200.h section 13): MOBIL on the react phase's staging ----
static_assert(sizeof(dp_lane_change_state) == 24, "dp_lane_change_state is 24 bytes");

// the ego as a follower: the interaction term alone (its v0 is unknown), 0 without a leader
__device__ __forceinline__ double lc_ego_idm(const dp_agent_model_params& p, double sab, double v, bool lead, double g, double vl) {
    if (!lead) return 0.0;
    const double dv = v - vl;
    double z = v * p.T + v * dv / sab;
    if (z < 0) z = 0;
    const double ss = p.s0 + z;
    double acc;
    if (g > 0) { const double q = ss / g; acc = -p.a_max * (q * q); }
    else acc = -p.b_max;
    if (acc < -p.b_max) acc = -p.b_max;
    return acc;
}

// an agent that does not change lanes this step: its hold runs down and its lat moves back towards lat_goal
__device__ __forceinline__ void lc_relax(const dp_lane_change_params& c, double dt, double& lat, dp_lane_change_state& s) {
    s.hold = s.hold - dt;
    if (lat != s.lat_goal) {
        const double e = s.lat_goal - lat, w = c.lat_speed * dt;
        lat = fabs(e) <= w ? s.lat_goal : (e > 0 ? lat + w : lat - w);
    }
}

struct LcSide { bool ok; double delta, atc; int im; };

// one side of agent k: target lane ml, abeam station, leader and follower on ml alone, safety and incentive.  (i, u): the agent's
// point and offset; (v, vd, ac): its start-of-step speed, desired speed and react-phase acceleration; (le, se, ve): the ego candidate
__device__ __forceinline__ LcSide lc_side(const DevMap& m, const LaneChangeModel& am, double sab, const double2* SV, const int* L, int n_obs,
                                          const double* v0, int le, double se, double ve, int ml, int i, double u, double v, double vd,
                                          double ac) {
    const dp_agent_model_params& p = am.p;
    const dp_lane_change_params& c = am.lc;
    LcSide r;
    r.ok = false;
    const int off = m.lane_pt_off[ml], cnt = m.lane_pt_off[ml + 1] - off;
    r.im = min(i, cnt - 2);
    const double sm = m.cump[off + r.im] + u;
    if (!(m.cump[off + cnt - 1] - sm >= c.end_guard)) return r;
    bool overlap = false, lead = false, foll = false, lego = false, fego = false;
    double gl = 0, vl = 0, sl = 0, gf = 0, vf = 0, sf = 0;
    int fj = -1;
    if (le == ml) {
        if (se == sm) overlap = true;
        else if (se > sm) { const double ds = se - sm; if (ds <= p.look) { lead = lego = true; gl = ds - p.ego_rear; vl = ve; sl = se; } }
        else { const double ds = sm - se; if (ds <= p.look) { foll = fego = true; gf = ds - c.ego_front; vf = ve; sf = se; } }
    }
    for (int j = 0; j < n_obs; ++j) {                       // warp-uniform j: broadcast reads
        if (L[j] != ml) continue;
        const double2 c2 = SV[j];
        const double sj = c2.x;
        if (sj == sm) overlap = true;
        else if (sj > sm) {
            const double ds = sj - sm;
            if (ds <= p.look) {
                const double g = ds - p.length;
                if (!lead || g < gl) { gl = g; vl = c2.y; sl = sj; lead = true; lego = false; }
            }
        } else {
            const double ds = sm - sj;
            if (ds <= p.look) {
                const double g = ds - p.length;
                if (!foll || g < gf) { gf = g; vf = c2.y; sf = sj; fj = j; foll = true; fego = false; }
            }
        }
    }
    if (overlap || (lead && !(gl > 0)) || (foll && !(gf > 0))) return r;
    r.atc = idm_accel(p, sab, v, vd, lead, gl, vl);
    double af = 0, atf = 0;
    if (fego) {
        af = lc_ego_idm(p, sab, vf, lead, (sl - sf) - c.ego_front, vl);
        atf = lc_ego_idm(p, sab, vf, true, gf, v);
        if (!(atf >= -c.ego_b_safe)) return r;
    } else if (foll) {
        const double vdf = v0[fj];
        if (vdf > 0) {
            af = idm_accel(p, sab, vf, vdf, lead, (sl - sf) - (lego ? p.ego_rear : p.length), vl);
            atf = idm_accel(p, sab, vf, vdf, true, gf, v);
        }
        if (!(atf >= -c.b_safe)) return r;
    }
    r.delta = (r.atc - ac) + c.politeness * (atf - af);
    r.ok = r.delta > c.a_thr;
    return r;
}

// agent k after its react phase (acc = a_c, vn = section 12's new speed): MOBIL, then the change or the relaxation; writes the
// agent and its lane-change state once
__device__ __forceinline__ void lane_change_agent(const DevMap& m, const LaneChangeModel& am, double sab, const double2* SV, const int* L,
                                                  int n_obs, const double* v0, int le, double se, double ve, double dt, int k, double v,
                                                  double vd, double acc, double vn, dp_agent* ag, dp_lane_change_state* lcs) {
    const dp_lane_change_params& c = am.lc;
    dp_agent a = ag[k];
    dp_lane_change_state s = lcs[k];
    const int l0 = a.lane;
    if (l0 < m.road_lane_base[m.n_roads] && a.lat == s.lat_goal && s.hold <= 0 && lane_len(m, l0) - SV[k].x >= c.end_guard) {
        int lo = 1, hi = m.n_roads;                         // the road r: road_lane_base[r-1] <= l0 < road_lane_base[r]
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (m.road_lane_base[mid] <= l0) lo = mid + 1;
            else hi = mid;
        }
        const int b0 = m.road_lane_base[lo - 1], q = l0 - b0, nl = m.road_lane_base[lo] - b0;
        const int attr = m.attr[m.lane_pt_off[l0] + a.i];
        LcSide best;
        best.ok = false;
        int side = 0;
        if (q >= 1 && (attr == 1 || attr == 3)) {
            best = lc_side(m, am, sab, SV, L, n_obs, v0, le, se, ve, l0 - 1, a.i, a.u, v, vd, acc);
            side = -1;
        }
        if (q + 1 < nl && (attr == 2 || attr == 3)) {
            const LcSide rs = lc_side(m, am, sab, SV, L, n_obs, v0, le, se, ve, l0 + 1, a.i, a.u, v, vd, acc);
            if (rs.ok && (!best.ok || rs.delta > best.delta)) { best = rs; side = 1; }
        }
        if (best.ok) {
            const int ml = l0 + side, om = m.lane_pt_off[ml];
            const double2 P = m.xy[m.lane_pt_off[l0] + a.i], Q = m.xy[om + best.im], R = m.xy[om + best.im + 1];
            const double dx = R.x - Q.x, dy = R.y - Q.y, Ls = sqrt(dx * dx + dy * dy);
            const double d = Ls > 0 ? (P.x - Q.x) * (-(dy / Ls)) + (P.y - Q.y) * (dx / Ls) : 0.0;
            a.lat = a.lat + d; a.lane = ml; a.i = best.im;
            double vc = v + best.atc * dt;
            if (vc < 0) vc = 0;
            a.v = vc;
            s.hold = c.cooldown;
            if (side < 0) s.changes_left += 1;
            else s.changes_right += 1;
            ag[k] = a; lcs[k] = s;
            return;
        }
    }
    a.v = vn;
    lc_relax(c, dt, a.lat, s);
    ag[k] = a; lcs[k] = s;
}

// rewrite agents[].v of one scene from the state at the start of the step (Jacobi): stage (lane, s, v) of every agent in the
// warp's slice of dynamic shared memory, then each lane scans the staged candidates for each of its agents (broadcast reads).
// LANECHG: each agent's lane change (section 13) follows its IDM step on the same staging.
template <bool LANECHG, class Model>
__device__ __forceinline__ void react_step(const DevMap& m, const Model& am, const dp_scene_hdr& h, int pos, int n_obs, double dt,
                                           dp_agent* ag, const double* v0, unsigned char* stage, int max_obs, int lane) {
    double2* SV = reinterpret_cast<double2*>(stage);
    int* L = reinterpret_cast<int*>(SV + max_obs);
    for (int k = lane; k < n_obs; k += 32) {
        const dp_agent a = ag[k];
        SV[k] = make_double2(m.cump[m.lane_pt_off[a.lane] + a.i] + a.u, a.v);
        L[k] = a.lane;
    }
    // the ego candidate (warp-uniform): its lane, station and speed from the start-of-step header
    int le = -1, idx = 0;
    if (pos != 2) { le = m.road_lane_base[h.road_num - 1] + h.lane_num - 1; idx = h.id[h.lane_num - 1]; }
    else if (h.conn >= 0 && h.conn < m.n_conn && h.last_lanenum >= 1 && h.last_lanenum <= DP_LANESUM) {
        le = m.conn[h.conn].lane; idx = h.id[h.last_lanenum - 1];
    }
    double se = 0;
    if (le >= 0) {
        const int off = m.lane_pt_off[le], cnt = m.lane_pt_off[le + 1] - off;
        if (idx > cnt - 1) idx = cnt - 1;
        if (idx < 0) idx = 0;
        se = m.cump[off + idx];
    }
    const double ve = h.velocity / 3.6;
    const dp_agent_model_params& p = am.p;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const double sab = 2.0 * sqrt(p.a_max * p.b);
    __syncwarp();
    for (int k = lane; k < n_obs; k += 32) {
        const double vd = v0[k];
        if (!(vd > 0)) {
            if constexpr (LANECHG) {
                dp_lane_change_state* lcs = am.lcs + (v0 - am.v0);   // the scene's states: indexed like v0
                dp_lane_change_state s = lcs[k];
                double lat = ag[k].lat;
                lc_relax(am.lc, dt, lat, s);
                ag[k].lat = lat; lcs[k] = s;
            }
            continue;
        }
        const double2 own = SV[k];
        const double sk = own.x, v = own.y;
        const int l0 = L[k], l1 = m.lane_next[l0], l2 = l1 >= 0 ? m.lane_next[l1] : -1;
        const double D1 = lane_len(m, l0) - sk, D2 = l1 >= 0 ? D1 + lane_len(m, l1) : 0.0;
        double best = inf, vl = 0;
        bool lead = false;
        if (le >= 0) {
            double ds = inf;
            if (le == l0 && se >= sk) ds = se - sk;
            if (le == l1) { const double c = D1 + se; if (c < ds) ds = c; }
            if (l2 >= 0 && le == l2) { const double c = D2 + se; if (c < ds) ds = c; }
            if (ds <= p.look) { best = ds - p.ego_rear; vl = ve; lead = true; }
        }
#pragma unroll 4
        for (int j = 0; j < n_obs; ++j) {                   // warp-uniform j: broadcast reads
            const int lj = L[j];
            const double2 c2 = SV[j];
            const double sj = c2.x;
            double ds = inf;
            if (lj == l0 && (sj > sk || (sj == sk && j > k))) ds = sj - sk;
            if (lj == l1) { const double c = D1 + sj; if (c < ds) ds = c; }
            if (l2 >= 0 && lj == l2) { const double c = D2 + sj; if (c < ds) ds = c; }
            if (ds <= p.look) {
                const double g = ds - p.length;
                if (!lead || g < best) { best = g; vl = c2.y; lead = true; }
            }
        }
        const double acc = idm_accel(p, sab, v, vd, lead, best, vl);
        double vn = v + acc * dt;
        if (vn < 0) vn = 0;
        if constexpr (LANECHG) lane_change_agent(m, am, sab, SV, L, n_obs, v0, le, se, ve, dt, k, v, vd, acc, vn, ag, am.lcs + (v0 - am.v0));
        else ag[k].v = vn;
    }
}

// JUNC = (pre_junction_pts > 0): the segment-only step (false) carries none of the junction code.
// METRICS = episode metrics armed (met != nullptr): the disarmed instances carry none of the metric code; the armed ones read the
// scene's row at entry and write it at the end as one coalesced 192-byte access each, staged behind the header in shared memory.
// REACT = reactive agents armed (am.v0 != nullptr): before the agent loop the armed instances rewrite agents[].v (react_step),
// staging max_obs * REACT_SLOT_BYTES of dynamic shared memory per warp.
// LANECHG = lane changes armed (am.lcs != nullptr, REACT instances only): the react phase is followed per agent by the lane
// change of section 13 on the same staging; the placement step initialises the states.
template <bool JUNC, bool METRICS, bool REACT, bool LANECHG = false>
__global__ void __launch_bounds__(WPB * 32, (METRICS || REACT) ? 8 : 0) dp_world_kernel(DevMap m, dp_params p, dp_world_params wp, int n, int max_obs,
                                                            dp_scene_hdr* __restrict__ hdr, dp_agent* __restrict__ agents,
                                                            double* __restrict__ obs_x, double* __restrict__ obs_y,
                                                            const dp_plan_record* __restrict__ rec, const double2* __restrict__ last_path,
                                                            dp_metrics_params mp, dp_episode_metrics* __restrict__ met,
                                                            std::conditional_t<LANECHG, LaneChangeModel, AgentModel> am) {
    __shared__ __align__(16) uint32_t sh[WPB][METRICS ? 32 + 2 * MET_WORDS : 32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int scene = blockIdx.x * WPB + wib;
    if (scene >= n) return;
    sh[wib][lane] = reinterpret_cast<const uint32_t*>(hdr + scene)[lane];   // one coalesced 128-byte load
    __syncwarp();
    const dp_scene_hdr& h = *reinterpret_cast<const dp_scene_hdr*>(sh[wib]);
    if constexpr (METRICS) {
        if (rec == nullptr) {                               // placement step: a clean row, whatever the header names
            double* row = reinterpret_cast<double*>(&sh[wib][32]);
            if (lane == 0) metrics_init(*reinterpret_cast<dp_episode_metrics*>(row));
            __syncwarp();
            if (lane < MET_WORDS) reinterpret_cast<double*>(met + scene)[lane] = row[lane];
        }
    }
    if constexpr (LANECHG) {
        static_assert(REACT, "lane changes run on the react phase");
        if (rec == nullptr) {                               // placement step: clean states, whatever the header names
            const int no = min((int)h.n_obs, max_obs);
            for (int k = lane; k < no; k += 32) {
                const size_t e = (size_t)scene * max_obs + k;
                dp_lane_change_state s;
                s.lat_goal = agents[e].lat; s.hold = 0; s.changes_left = 0; s.changes_right = 0;
                am.lcs[e] = s;
            }
        }
    }
    // a header that does not name a lane of the map (device-pointer callers are not validated on the host) leaves its world untouched
    if (h.road_num < 1 || h.road_num > m.n_roads || h.lane_num < 1 ||
        h.lane_num > m.road_lane_base[h.road_num] - m.road_lane_base[h.road_num - 1] || h.lane_num > DP_LANESUM) return;
    // metrics state of this lane; an empty object in the disarmed instances, which must compile to what they compiled to before
    std::conditional_t<METRICS, MetricLane, NoMetrics> ml;
    if constexpr (METRICS) {
        if (rec != nullptr && lane < MET_WORDS) ml.word = reinterpret_cast<const double*>(met + scene)[lane];
    }
    const int n_obs = min((int)h.n_obs, max_obs);
    const double dt = h.period_ms / 1000.0;
    const int J = wp.pre_junction_pts;
    const int pos = (JUNC && (h.pos == 1 || h.pos == 2)) ? h.pos : 0;
    double x = h.x, y = h.y, dir = h.dir, vn = h.velocity;
    const bool step = rec != nullptr;
    if (step) {
        // ---- ego: bounded approach to the planned speed, then a walk along the carried local path (every lane computes the same
        // scalars; the path segments come in 32 at a time, one per lane, and are walked in index order through shuffles, so the
        // sequential `rem -= L` of the specification never waits for memory) ----
        const dp_plan_record& r = rec[scene];
        const int gl = m.road_lane_base[h.road_num - 1] + h.lane_num - 1;
        const int cnt = m.lane_pt_off[gl + 1] - m.lane_pt_off[gl];
        const bool stop_zone = !JUNC || (pos == 0 && ego_connector(m, h.road_num, h.lane_num, h.next_roadnum, lane) < 0);
        const bool at_end = stop_zone && h.id[h.lane_num - 1] >= cnt - wp.end_margin;
        const double v = h.velocity, vt = r.brakespeed * 3.6, dvm = wp.a_max * 3.6 * dt;
        double dv = vt - v;
        if (dv > dvm) dv = dvm;
        if (dv < -dvm) dv = -dvm;
        vn = v + dv;
        if (vn < 0) vn = 0;
        if (at_end) vn = 0;
        const double ds = at_end ? 0.0 : (v + vn) * 0.5 / 3.6 * dt;
        if constexpr (METRICS) { ml.ds = ds; ml.at_end = at_end; }
        if (ds > 0) {
            const double2* lp = last_path + (size_t)scene * DP_PATH_POINTS;
            int i = r.afresh_planning ? 0 : r.path_near_id;
            if (i < 0) i = 0;
            if (i > DP_PATH_POINTS - 2) i = DP_PATH_POINTS - 2;
            double rem = ds;
            for (int base = i;; base += 32) {
                const int idx = min(base + lane, DP_PATH_POINTS - 2);
                const double2 a = lp[idx], b = lp[idx + 1];
                double ddx, ddy;
                const double L = seg_len(a, b, &ddx, &ddy);
                int hit = -1;
                for (int k = 0; k < 32; ++k) {
                    const double Lk = __shfl_sync(DP_FULL, L, k);
                    if (rem < Lk || base + k == DP_PATH_POINTS - 2) { hit = k; break; }
                    rem -= Lk;
                }
                if (hit < 0) continue;
                const double ax = __shfl_sync(DP_FULL, a.x, hit), ay = __shfl_sync(DP_FULL, a.y, hit);
                const double bx = __shfl_sync(DP_FULL, b.x, hit), by = __shfl_sync(DP_FULL, b.y, hit);
                const double sdx = __shfl_sync(DP_FULL, ddx, hit), sdy = __shfl_sync(DP_FULL, ddy, hit), Lh = __shfl_sync(DP_FULL, L, hit);
                if (Lh > 0) {
                    double t = rem / Lh;
                    if (t > 1) t = 1;
                    x = ax + t * sdx; y = ay + t * sdy;
                    dir = dp_heading(ax, ay, bx, by, p.epsilon, p.pi);
                } else { x = ax; y = ay; }
                break;
            }
        }
    }
    x = __shfl_sync(DP_FULL, x, 0); y = __shfl_sync(DP_FULL, y, 0);
    if constexpr (METRICS) {
        if (step) {                                     // the ego frame of the new pose
            double c, sn;
            dp_sincos_deg(dir, &c, &sn);
            ml.c = c; ml.s = sn;
        }
    }
    if constexpr (REACT) {
        if (step) {
            extern __shared__ __align__(16) unsigned char react_stage[];
            react_step<LANECHG>(m, am, h, pos, n_obs, dt, agents + (size_t)scene * max_obs, am.v0 + (size_t)scene * max_obs,
                                react_stage + wib * react_stage_bytes(max_obs), max_obs, lane);
        }
    }
    // ---- agents: constant speed along their lanes (junctions on: and on into the lane's successor), then their obstacle points ----
    for (int k = lane; k < n_obs; k += 32) {
        dp_agent a = agents[(size_t)scene * max_obs + k];
        int off = m.lane_pt_off[a.lane], cntk = m.lane_pt_off[a.lane + 1] - off;
        double ddx, ddy;
        if (step) {
            double u = a.u + a.v * dt;
            int i = a.i;
            for (int hop = 0;; ++hop) {
                while (i < cntk - 2) {
                    const double L = seg_len(m.xy[off + i], m.xy[off + i + 1], &ddx, &ddy);
                    if (u < L) break;
                    u -= L; ++i;
                }
                if (i < cntk - 2) break;
                i = cntk - 2;
                const double L = seg_len(m.xy[off + i], m.xy[off + i + 1], &ddx, &ddy);
                const int nx = JUNC && hop < WORLD_MAX_HOPS ? m.lane_next[a.lane] : -1;
                if (u < L || nx < 0) {
                    if (u > L) u = L;
                    break;
                }
                u -= L; a.lane = nx; i = 0;
                off = m.lane_pt_off[nx]; cntk = m.lane_pt_off[nx + 1] - off;
            }
            a.u = u; a.i = i;
            agents[(size_t)scene * max_obs + k] = a;
        }
        const double2 q = m.xy[off + a.i];
        const double L = seg_len(q, m.xy[off + a.i + 1], &ddx, &ddy);
        double ox = q.x, oy = q.y;
        if (L > 0) {
            const double t = a.u / L;
            const double px = q.x + t * ddx, py = q.y + t * ddy;
            ox = px + a.lat * (-(ddy / L));
            oy = py + a.lat * (ddx / L);
        }
        obs_x[(size_t)scene * max_obs + k] = ox;
        obs_y[(size_t)scene * max_obs + k] = oy;
        if constexpr (METRICS) {
            if (step) {                                     // the agent in the ego frame: box, clearance, lead gap and ttc
                const double dx = ox - x, dy = oy - y;
                const double lon = dx * ml.c + dy * ml.s, lat = dy * ml.c - dx * ml.s, alat = fabs(lat);
                if (-mp.rear <= lon && lon <= mp.front && -mp.half_width <= lat && lat <= mp.half_width) {
                    if (k < ml.first) ml.first = k;
                    if (lon >= 0) ml.front = true;
                    else ml.rear = true;
                }
                const double ex = lon > mp.front ? lon - mp.front : (lon < -mp.rear ? -mp.rear - lon : 0.0);
                const double ey = alat > mp.half_width ? alat - mp.half_width : 0.0;
                const double d = sqrt(ex * ex + ey * ey);
                if (d < ml.d) ml.d = d;
                if (lon > mp.front && alat <= mp.corridor_half) {
                    const double gap = lon - mp.front;
                    const double va = L == 0 ? 0.0 : a.v * (ddx / L * ml.c + ddy / L * ml.s);
                    const double closing = vn / 3.6 - va;
                    const double ttc = closing > 0 ? gap / closing : __longlong_as_double(0x7ff0000000000000LL);
                    if (gap < ml.gap) ml.gap = gap;
                    if (ttc < ml.ttc) ml.ttc = ttc;
                }
            }
        }
    }
    if constexpr (METRICS) {
        if (step) metrics_step(ml, reinterpret_cast<double*>(&sh[wib][32]), met + scene, lane, mp, rec[scene], h.velocity, vn, dt);
    }
    // ---- localisation: nearest point per lane inside a window around the previous index (pos 2: the departure road from its
    // start), nearest lane ----
    const int base = m.road_lane_base[h.road_num - 1];
    int nl = m.road_lane_base[h.road_num] - base;
    if (nl > DP_LANESUM) nl = DP_LANESUM;
    double best = __longlong_as_double(0x7ff0000000000000LL);
    int bl = 0, my_id = 0;                                  // lane l keeps the new id of map lane l
    for (int l = 0; l < nl; ++l) {
        int bi;
        const double be = warp_nearest(m, base + l, pos == 2 ? 0 : h.id[l] - wp.loc_back, pos == 2 ? wp.loc_fwd : h.id[l] + wp.loc_fwd,
                                       x, y, lane, &bi);
        if (lane == l) my_id = bi;
        if (be < best) { best = be; bl = l; }
    }
    // ---- junction transitions (warp-uniform; include/dmpp_b200.h section 9) ----
    int o_pos = h.pos, o_conn = h.conn, o_road = h.road_num, o_lane = h.lane_num, o_path = h.path_num, o_stub = h.stub_attribute;
    int o_last_road = h.last_roadnum, o_last_lane = h.last_lanenum, o_next_lane = h.next_lanenum;
    int id_val = my_id, id_n = nl;                          // lanes [0, id_n) of hdr.id get id_val
    if (pos != 2) o_lane = bl + 1;
    if (JUNC) {
        if (pos == 0) {
            const int c = ego_connector(m, h.road_num, o_lane, h.next_roadnum, lane);
            const int my_new = __shfl_sync(DP_FULL, my_id, o_lane - 1);
            const int gl = base + o_lane - 1;
            if (c >= 0 && my_new >= m.lane_pt_off[gl + 1] - m.lane_pt_off[gl] - 1 - J) {
                o_pos = 1; o_conn = c; o_last_road = h.road_num; o_last_lane = o_lane; o_next_lane = m.conn[c].next_lane;
            }
        } else {
            bool conn_ok = true;
            if (pos == 1) {
                const int c = ego_connector(m, h.road_num, o_lane, h.next_roadnum, lane);
                if (c < 0) { o_pos = 0; o_conn = -1; conn_ok = false; }
                else { o_conn = c; o_last_road = h.road_num; o_last_lane = o_lane; o_next_lane = m.conn[c].next_lane; }
            }
            if (conn_ok) {
                const bool have_conn = o_conn >= 0 && o_conn < m.n_conn && o_last_lane >= 1 && o_last_lane <= DP_LANESUM;
                double bc = __longlong_as_double(0x7ff0000000000000LL);
                int ci = 0;
                if (have_conn) {
                    const int idc = h.id[o_last_lane - 1];
                    bc = warp_nearest(m, m.conn[o_conn].lane, pos == 1 ? 0 : idc - wp.loc_back, pos == 1 ? wp.loc_fwd : idc + wp.loc_fwd,
                                      x, y, lane, &ci);
                }
                if (pos == 2 && best < bc) {
                    o_lane = bl + 1; o_pos = 0; o_conn = -1; o_path = h.path_num + 1; o_stub = 0;
                } else if (pos == 2 || bc < best) {
                    if (pos == 1) { o_pos = 2; o_road = h.next_roadnum; o_lane = o_next_lane; }
                    const int lr = m.conn[o_conn].last_road;
                    id_val = ci; id_n = min(m.road_lane_base[lr] - m.road_lane_base[lr - 1], DP_LANESUM);
                }
            }
        }
    }
    // ---- the header of the next cycle, in place ----
    dp_scene_hdr* out = hdr + scene;
    if (lane < id_n) out->id[lane] = id_val;
    if (lane == 0) {
        out->x = x; out->y = y; out->dir = dir; out->velocity = vn;
        out->lane_num = (uint16_t)o_lane;
        if (JUNC) {
            out->road_num = (uint16_t)o_road; out->pos = (uint16_t)o_pos; out->path_num = (uint16_t)o_path;
            out->last_roadnum = (uint16_t)o_last_road; out->last_lanenum = (uint16_t)o_last_lane; out->next_lanenum = (uint16_t)o_next_lane;
            out->stub_attribute = (uint16_t)o_stub; out->conn = o_conn;
        }
    }
}
}  // namespace

// the launches of one instance set, both JUNC instances: each set is instantiated in its own translation unit (the extern
// declarations below name it), and dp_launch_world (dp_world.cu) picks the set from the armed options
template <bool METRICS, bool REACT, bool LANECHG>
struct WorldStep {
    static cudaError_t launch(const DevMap& m, const dp_params& p, const DpWorldOpts& o, const DpWorldBufs& b, cudaStream_t st);
    static cudaError_t prepare();              // REACT: allow the dynamic shared memory of DP_AGENT_MODEL_MAX_OBS agent slots
    static auto kernel(bool junc) { return junc ? dp_world_kernel<true, METRICS, REACT, LANECHG> : dp_world_kernel<false, METRICS, REACT, LANECHG>; }
};
// (defined outside the class: not inline, so the extern declarations below keep the other translation units from instantiating them)
template <bool METRICS, bool REACT, bool LANECHG>
cudaError_t WorldStep<METRICS, REACT, LANECHG>::launch(const DevMap& m, const dp_params& p, const DpWorldOpts& o, const DpWorldBufs& b,
                                                       cudaStream_t st) {
    std::conditional_t<LANECHG, LaneChangeModel, AgentModel> am;
    am.p = o.amp; am.v0 = o.v0;
    if constexpr (LANECHG) { am.lc = o.lcp; am.lcs = o.lcs; }
    const size_t smem = REACT ? WPB * react_stage_bytes(b.max_obs) : 0;
    kernel(o.wp.pre_junction_pts > 0)<<<(b.n + WPB - 1) / WPB, WPB * 32, smem, st>>>(
        m, p, o.wp, b.n, b.max_obs, b.hdr, b.agents, b.ox, b.oy, b.rec, b.last_path, o.mp, o.met, am);
    return cudaGetLastError();
}
template <bool METRICS, bool REACT, bool LANECHG>
cudaError_t WorldStep<METRICS, REACT, LANECHG>::prepare() {
    const int bytes = (int)(WPB * react_stage_bytes(DP_AGENT_MODEL_MAX_OBS));
    for (const bool junc : {false, true}) {
        const cudaError_t e = cudaFuncSetAttribute(kernel(junc), cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}
extern template struct WorldStep<false, false, false>;   // dp_world.cu
extern template struct WorldStep<true, false, false>;    // dp_world_metrics.cu
extern template struct WorldStep<false, true, false>;    // dp_world_agents.cu
extern template struct WorldStep<true, true, false>;
extern template struct WorldStep<false, true, true>;     // dp_world_lanechange.cu
extern template struct WorldStep<true, true, true>;
