// tools/junction_oracle/lane_change.cpp -- TEST INFRASTRUCTURE (CPU oracle), see lane_change.h.
#include "lane_change.h"

#include <cmath>
#include <vector>

#include "agent_model.h"
#include "episode_metrics.h"

namespace lanechg {

namespace {
// section 12's IDM acceleration with its clamp; lead false: free road
double idm(const dp_agent_model_params& p, double v, double vd, bool lead, double g, double vl) {
    const double r = v / vd;
    double fr = r * r;
    fr = fr * fr;
    double acc;
    if (lead) {
        const double dv = v - vl;
        double z = v * p.T + v * dv / (2.0 * std::sqrt(p.a_max * p.b));
        if (z < 0) z = 0;
        const double ss = p.s0 + z;
        if (g > 0) { const double q = ss / g; acc = p.a_max * (1.0 - fr - q * q); }
        else acc = -p.b_max;
    } else acc = p.a_max * (1.0 - fr);
    if (acc < -p.b_max) acc = -p.b_max;
    return acc;
}

// the ego as a follower: the interaction term alone, 0 without a leader
double ego_idm(const dp_agent_model_params& p, double v, bool lead, double g, double vl) {
    if (!lead) return 0.0;
    const double dv = v - vl;
    double z = v * p.T + v * dv / (2.0 * std::sqrt(p.a_max * p.b));
    if (z < 0) z = 0;
    const double ss = p.s0 + z;
    double acc;
    if (g > 0) { const double q = ss / g; acc = -p.a_max * (q * q); }
    else acc = -p.b_max;
    if (acc < -p.b_max) acc = -p.b_max;
    return acc;
}

struct Side { bool ok = false; double delta = 0, atc = 0; int im = 0; };

// the start-of-step state of the scene: stations, speeds and lanes of the agents, the ego candidate
struct Snapshot {
    std::vector<double> S, V;
    std::vector<int> L;
    int le;
    double se, ve;
};

Side side(const junction::JMap& jm, const dp_agent_model_params& p, const dp_lane_change_params& c, const Snapshot& w, const double* v0,
          int ml, int i, double u, double v, double vd, double ac, const traffic::World* tw) {
    const oracle::MapView& m = jm.m;
    Side r;
    const int off = m.d.lane_pt_off[ml], cnt = m.lane_size(ml);
    r.im = i < cnt - 2 ? i : cnt - 2;
    const double sm = jm.cump[off + r.im] + u;
    if (!(agents::lane_len(jm, ml) - sm >= c.end_guard)) return r;
    bool overlap = false, lead = false, foll = false, lego = false, fego = false;
    double gl = 0, vl = 0, sl = 0, gf = 0, vf = 0, sf = 0;
    int fj = -1;
    if (w.le == ml) {                                       // the ego first: agents replace it only with a strictly smaller g
        if (w.se == sm) overlap = true;
        else if (w.se > sm) {
            const double ds = w.se - sm;
            if (ds <= p.look) { lead = lego = true; gl = ds - p.ego_rear; vl = w.ve; sl = w.se; }
        } else {
            const double ds = sm - w.se;
            if (ds <= p.look) { foll = fego = true; gf = ds - c.ego_front; vf = w.ve; sf = w.se; }
        }
    }
    const int n = (int)w.S.size();
    for (int j = 0; j < n; ++j) {
        if (w.L[j] != ml) continue;
        const double sj = w.S[j];
        if (sj == sm) overlap = true;
        else if (sj > sm) {
            const double ds = sj - sm;
            if (ds <= p.look) {
                const double g = ds - p.length;
                if (!lead || g < gl) { gl = g; vl = w.V[j]; sl = sj; lead = true; lego = false; }
            }
        } else {
            const double ds = sm - sj;
            if (ds <= p.look) {
                const double g = ds - p.length;
                if (!foll || g < gf) { gf = g; vf = w.V[j]; sf = sj; fj = j; foll = true; fego = false; }
            }
        }
    }
    bool clead = lead;                                      // the leader of at_c and of the safety test
    double cg = gl, cv = vl;
    if (tw) {                                               // section 15: the line and the pedestrian on ml
        bool tl = lead;
        double tg = gl;
        if (traffic::side(jm, *tw, p, ml, r.im, sm, u, v, &tl, &tg) && tw->tp.obey) { clead = true; cg = tg; cv = 0.0; }
    }
    if (overlap || (clead && !(cg > 0)) || (foll && !(gf > 0))) return r;
    r.atc = idm(p, v, vd, clead, cg, cv);
    double af = 0, atf = 0;
    if (fego) {
        af = ego_idm(p, vf, lead, (sl - sf) - c.ego_front, vl);
        atf = ego_idm(p, vf, true, gf, v);
        if (!(atf >= -c.ego_b_safe)) return r;
    } else if (foll) {
        const double vdf = v0[fj];
        if (vdf > 0) {
            af = idm(p, vf, vdf, lead, (sl - sf) - (lego ? p.ego_rear : p.length), vl);
            atf = idm(p, vf, vdf, true, gf, v);
        }
        if (!(atf >= -c.b_safe)) return r;
    }
    r.delta = (r.atc - ac) + c.politeness * (atf - af);
    r.ok = r.delta > c.a_thr;
    return r;
}

void relax(const dp_lane_change_params& c, double dt, double& lat, dp_lane_change_state& s) {
    s.hold = s.hold - dt;
    if (lat != s.lat_goal) {
        const double e = s.lat_goal - lat, w = c.lat_speed * dt;
        lat = std::fabs(e) <= w ? s.lat_goal : (e > 0 ? lat + w : lat - w);
    }
}
}  // namespace

void init(const dp_agent* ag, int n, dp_lane_change_state* st) {
    for (int k = 0; k < n; ++k) {
        st[k].lat_goal = ag[k].lat; st[k].hold = 0; st[k].changes_left = 0; st[k].changes_right = 0;
    }
}

void step(const junction::JMap& jm, const dp_world_params& wp, const dp_agent_model_params& am, const dp_lane_change_params& lp,
          const dp_scene_hdr& h0, dp_agent* ag, int n, const double* v0, dp_lane_change_state* st, const traffic::World* tw,
          int* kind_out) {
    const oracle::MapView& m = jm.m;
    if (!metrics::header_valid(m, h0)) return;
    const double dt = h0.period_ms / 1000.0;
    Snapshot w;
    w.S.resize(n); w.V.resize(n); w.L.resize(n);
    const std::vector<dp_agent> a0(ag, ag + n);
    for (int k = 0; k < n; ++k) {
        w.S[k] = jm.cump[m.d.lane_pt_off[a0[k].lane] + a0[k].i] + a0[k].u;
        w.V[k] = a0[k].v; w.L[k] = a0[k].lane;
    }
    w.le = agents::ego_lane(jm, wp, h0, &w.se);
    w.ve = h0.velocity / 3.6;
    std::vector<double> acc(n, 0.0);
    agents::react(jm, wp, am, h0, ag, n, v0, acc.data(), tw, kind_out);   // ag[k].v = section 12's speed; acc[k] = a_c
    const int road_lanes = m.d.road_lane_base[m.d.n_roads];
    for (int k = 0; k < n; ++k) {
        dp_agent& a = ag[k];
        dp_lane_change_state& s = st[k];
        const int l0 = a.lane;
        if (v0[k] > 0 && l0 < road_lanes && a.lat == s.lat_goal && s.hold <= 0 && agents::lane_len(jm, l0) - w.S[k] >= lp.end_guard) {
            int r = 1;                                      // the road: road_lane_base[r-1] <= l0 < road_lane_base[r]
            while (m.d.road_lane_base[r] <= l0) ++r;
            const int b0 = m.d.road_lane_base[r - 1], q = l0 - b0, nl = m.d.road_lane_base[r] - b0;
            const int attr = m.attr(l0, a.i);
            Side best;
            int dir = 0;
            if (q >= 1 && (attr == 1 || attr == 3)) {
                best = side(jm, am, lp, w, v0, l0 - 1, a.i, a.u, w.V[k], v0[k], acc[k], tw);
                dir = -1;
            }
            if (q + 1 < nl && (attr == 2 || attr == 3)) {
                const Side rs = side(jm, am, lp, w, v0, l0 + 1, a.i, a.u, w.V[k], v0[k], acc[k], tw);
                if (rs.ok && (!best.ok || rs.delta > best.delta)) { best = rs; dir = 1; }
            }
            if (best.ok) {
                const int ml = l0 + dir;
                const spec::P2 P = m.pt(l0, a.i), Q = m.pt(ml, best.im), R = m.pt(ml, best.im + 1);
                const double dx = R.x - Q.x, dy = R.y - Q.y, Ls = std::sqrt(dx * dx + dy * dy);
                const double d = Ls > 0 ? (P.x - Q.x) * (-(dy / Ls)) + (P.y - Q.y) * (dx / Ls) : 0.0;
                a.lat = a.lat + d; a.lane = ml; a.i = best.im;
                double vc = w.V[k] + best.atc * dt;
                if (vc < 0) vc = 0;
                a.v = vc;
                s.hold = lp.cooldown;
                if (dir < 0) s.changes_left += 1;
                else s.changes_right += 1;
                continue;
            }
        }
        relax(lp, dt, a.lat, s);
    }
}

}  // namespace lanechg
