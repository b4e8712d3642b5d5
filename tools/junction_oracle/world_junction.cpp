// tools/junction_oracle/world_junction.cpp -- TEST INFRASTRUCTURE (CPU oracle), see world_junction.h.
#include "world_junction.h"

#include <cmath>
#include <limits>

#include "../../oracle/world_spec.h"

namespace junction {

namespace {
constexpr int WORLD_MAX_HOPS = 8;   // successor lanes an agent may enter in one step
inline double seg_len(const oracle::MapView& m, int gl, int i, double* ddx, double* ddy) {
    const spec::P2 a = m.pt(gl, i), b = m.pt(gl, i + 1);
    *ddx = b.x - a.x; *ddy = b.y - a.y;
    return std::sqrt(*ddx * *ddx + *ddy * *ddy);
}
// nearest point of lane gl to (x, y) in [lo, hi] clipped to the lane: squared distance (returned), strict '<', lowest index
inline double nearest(const oracle::MapView& m, int gl, int lo, int hi, double x, double y, int* bi) {
    const int cnt = m.lane_size(gl);
    if (lo < 0) lo = 0;
    if (hi > cnt - 1) hi = cnt - 1;
    double be = std::numeric_limits<double>::infinity();
    *bi = lo;
    for (int i = lo; i <= hi; ++i) {
        const spec::P2 q = m.pt(gl, i);
        const double dx = x - q.x, dy = y - q.y;
        const double e = dx * dx + dy * dy;
        if (e < be) { be = e; *bi = i; }
    }
    return be;
}
}  // namespace

int ego_connector(const oracle::MapView& m, const dp_scene_hdr& h, int road, int lane) {
    if (h.next_roadnum == road) return -1;
    for (int c = 0; c < m.d.n_conn; ++c) {
        const dp_connector& k = m.d.conn[c];
        if (k.last_road == road && k.next_road == h.next_roadnum && k.last_lane == lane) return c;
    }
    return -1;
}

void JMap::set(const dp_map_desc& m) {
    this->m.d = m;
    next.assign(m.n_lanes > 0 ? m.n_lanes : 0, -1);
    const int n_road_lanes = m.road_lane_base[m.n_roads];
    for (int r = 1; r <= m.n_roads; ++r)
        for (int gl = m.road_lane_base[r - 1]; gl < m.road_lane_base[r] && gl < m.n_lanes; ++gl)
            for (int c = 0; c < m.n_conn; ++c)
                if (m.conn[c].last_road == r && m.conn[c].last_lane == gl - m.road_lane_base[r - 1] + 1) { next[gl] = m.conn[c].lane; break; }
    for (int c = 0; c < m.n_conn; ++c) {
        const dp_connector& k = m.conn[c];
        if (k.lane < n_road_lanes || k.lane >= m.n_lanes || k.next_road < 1 || k.next_road > m.n_roads) continue;
        if (k.next_lane < 1 || k.next_lane > m.road_lane_base[k.next_road] - m.road_lane_base[k.next_road - 1]) continue;
        next[k.lane] = m.road_lane_base[k.next_road - 1] + k.next_lane - 1;
    }
    cump.assign(m.n_lanes > 0 ? m.lane_pt_off[m.n_lanes] : 0, 0.0);
    for (int gl = 0; gl < m.n_lanes; ++gl) {
        const int off = m.lane_pt_off[gl], cnt = m.lane_pt_off[gl + 1] - off;
        double acc = 0.0;
        for (int i = 0; i < cnt; ++i) {
            double l = 0.0;
            if (i + 1 < cnt) {
                const double dx = m.x[off + i + 1] - m.x[off + i], dy = m.y[off + i + 1] - m.y[off + i];
                l = std::sqrt(dx * dx + dy * dy);
            }
            cump[off + i] = acc; acc += l;
        }
    }
}

void world_step(const JMap& jm, const dp_params& p, const dp_world_params& wp, dp_scene_hdr& h, dp_agent* ag, double* ox, double* oy,
                const dp_plan_record* rec, const double* lx, const double* ly) {
    if (wp.pre_junction_pts <= 0) {                         // junctions off: the frozen segment-only step itself
        oracle::world_step(jm.m, p, wp, h, ag, ox, oy, rec, lx, ly);
        return;
    }
    const oracle::MapView& m = jm.m;
    const int n_obs = h.n_obs;
    const double dt = h.period_ms / 1000.0;
    const int J = wp.pre_junction_pts;
    const int pos = (h.pos == 1 || h.pos == 2) ? h.pos : 0;
    if (rec) {
        // ---- ego: bounded approach to the planned speed, then a walk along the carried local path ----
        const int gl = m.lane_index(h.road_num, h.lane_num), cnt = m.lane_size(gl);
        const bool stop_zone = pos == 0 && ego_connector(m, h, h.road_num, h.lane_num) < 0;
        const bool at_end = stop_zone && h.id[h.lane_num - 1] >= cnt - wp.end_margin;
        const double v = h.velocity, vt = rec->brakespeed * 3.6, dvm = wp.a_max * 3.6 * dt;
        double dv = vt - v;
        if (dv > dvm) dv = dvm;
        if (dv < -dvm) dv = -dvm;
        double vn = v + dv;
        if (vn < 0) vn = 0;
        if (at_end) vn = 0;
        const double ds = at_end ? 0.0 : (v + vn) * 0.5 / 3.6 * dt;
        double x = h.x, y = h.y, dir = h.dir;
        if (ds > 0) {
            int i = rec->afresh_planning ? 0 : rec->path_near_id;   // a fresh path starts at the ego (Planning.cpp:596-611, :845-877)
            if (i < 0) i = 0;
            if (i > DP_PATH_POINTS - 2) i = DP_PATH_POINTS - 2;
            double rem = ds;
            for (;;) {
                const double ax = lx[i], ay = ly[i], bx = lx[i + 1], by = ly[i + 1];
                const double ddx = bx - ax, ddy = by - ay;
                const double L = std::sqrt(ddx * ddx + ddy * ddy);
                if (rem < L || i == DP_PATH_POINTS - 2) {
                    if (L > 0) {
                        double t = rem / L;
                        if (t > 1) t = 1;
                        x = ax + t * ddx; y = ay + t * ddy;
                        dir = spec::calc_global_dir(spec::P2{ax, ay}, spec::P2{bx, by}, p.epsilon, p.pi);
                    } else { x = ax; y = ay; }
                    break;
                }
                rem -= L; ++i;
            }
        }
        h.x = x; h.y = y; h.dir = dir; h.velocity = vn;
        // ---- agents: constant speed along their lanes (junctions on: and on into the lane's successor) ----
        for (int k = 0; k < n_obs; ++k) {
            dp_agent& a = ag[k];
            int lane = a.lane, cntk = m.lane_size(lane);
            double u = a.u + a.v * dt, ddx, ddy;
            int i = a.i;
            for (int hop = 0;; ++hop) {
                while (i < cntk - 2) {
                    const double L = seg_len(m, lane, i, &ddx, &ddy);
                    if (u < L) break;
                    u -= L; ++i;
                }
                if (i < cntk - 2) break;
                i = cntk - 2;
                const double L = seg_len(m, lane, i, &ddx, &ddy);
                const int nx = hop < WORLD_MAX_HOPS ? jm.next[lane] : -1;
                if (u < L || nx < 0) {
                    if (u > L) u = L;
                    break;
                }
                u -= L; lane = nx; i = 0; cntk = m.lane_size(lane);
            }
            a.u = u; a.i = i; a.lane = lane;
        }
    }
    // ---- obstacle points of the agents ----
    for (int k = 0; k < n_obs; ++k) {
        const dp_agent& a = ag[k];
        double ddx, ddy;
        const double L = seg_len(m, a.lane, a.i, &ddx, &ddy);
        const spec::P2 q = m.pt(a.lane, a.i);
        if (L > 0) {
            const double t = a.u / L;
            const double px = q.x + t * ddx, py = q.y + t * ddy;
            ox[k] = px + a.lat * (-(ddy / L));
            oy[k] = py + a.lat * (ddx / L);
        } else { ox[k] = q.x; oy[k] = q.y; }
    }
    // ---- localisation: nearest point per lane inside a window around the previous index, nearest lane ----
    const int nl = m.lanes_of(h.road_num);
    double best = std::numeric_limits<double>::infinity();
    int bl = 0;
    int new_id[DP_LANESUM];
    for (int l = 0; l < nl && l < DP_LANESUM; ++l) {
        const int gl = m.lane_index(h.road_num, l + 1);
        int be_i;
        const double be = nearest(m, gl, pos == 2 ? 0 : h.id[l] - wp.loc_back, pos == 2 ? wp.loc_fwd : h.id[l] + wp.loc_fwd, h.x, h.y, &be_i);
        new_id[l] = be_i;
        if (be < best) { best = be; bl = l; }
    }
    if (pos == 0 || pos == 1) {
        for (int l = 0; l < nl && l < DP_LANESUM; ++l) h.id[l] = new_id[l];
        h.lane_num = (uint16_t)(bl + 1);
    }
    // ---- junction transitions ----
    if (pos == 0) {
        const int c = ego_connector(m, h, h.road_num, h.lane_num);
        if (c >= 0 && h.id[h.lane_num - 1] >= m.lane_size(m.lane_index(h.road_num, h.lane_num)) - 1 - J) {
            h.pos = 1; h.conn = c;
            h.last_roadnum = h.road_num; h.last_lanenum = h.lane_num; h.next_lanenum = m.d.conn[c].next_lane;
        }
        return;
    }
    if (pos == 1) {
        const int c = ego_connector(m, h, h.road_num, h.lane_num);
        if (c < 0) { h.pos = 0; h.conn = -1; return; }
        h.conn = c; h.last_roadnum = h.road_num; h.last_lanenum = h.lane_num; h.next_lanenum = m.d.conn[c].next_lane;
    }
    const bool have_conn = h.conn >= 0 && h.conn < m.d.n_conn && h.last_lanenum >= 1 && h.last_lanenum <= DP_LANESUM;
    double bc = std::numeric_limits<double>::infinity();
    int ci = 0;
    if (have_conn) {
        const int gc = m.d.conn[h.conn].lane, idc = h.id[h.last_lanenum - 1];
        bc = nearest(m, gc, pos == 1 ? 0 : idc - wp.loc_back, pos == 1 ? wp.loc_fwd : idc + wp.loc_fwd, h.x, h.y, &ci);
    }
    if (pos == 1 && !(bc < best)) return;
    if (pos == 2 && best < bc) {
        for (int l = 0; l < nl && l < DP_LANESUM; ++l) h.id[l] = new_id[l];
        h.lane_num = (uint16_t)(bl + 1);
        h.pos = 0; h.conn = -1; h.path_num = (uint16_t)(h.path_num + 1); h.stub_attribute = 0;
        return;
    }
    // pos 2 (entered now or kept): the connector index for every lane of the approach road
    if (pos == 1) { h.pos = 2; h.road_num = h.next_roadnum; h.lane_num = h.next_lanenum; }
    const int nla = m.lanes_of(m.d.conn[h.conn].last_road);
    for (int l = 0; l < nla && l < DP_LANESUM; ++l) h.id[l] = ci;
}

}  // namespace junction
