// tools/emu/dp_emu.cpp -- TEST INFRASTRUCTURE.  Host emulation of the group kernel (csrc/dp_group.cuh compiled with
// -DDP_EMU: every phase of a CTA becomes a loop over its thread ids).  It exists so that the kernel's LOGIC (phase
// structure, pruned scans, rule tree, index math) can be checked against the oracle on a box without a GPU
// (tests/test_emu_vs_oracle.py).  It is never linked into libdmpp_b200.so and nothing in the product loads it.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../../decision-making-and-path-planning_b200/csrc/dp_group.cuh"

namespace {
struct HostMap {
    std::vector<double2> xy, nrm;
    std::vector<double> lenp, lenf;
    std::vector<float> hmax, hmin, dnmax;
    std::vector<double> cump, cerr;
    std::vector<int32_t> re0, re1;
    DgMap m;
    bool ok = false;
} g;
}

extern "C" {

// same precompute as dp_map_prep_kernel (csrc/dp_cycle.cu)
int emu_set_map(const dp_map_desc* d) {
    const size_t np = (size_t)d->n_points;
    g.xy.assign(np, make_double2(0, 0)); g.nrm.assign(np, make_double2(0, 0));
    g.lenp.assign(np, 0.0); g.lenf.assign(np, 0.0);
    g.hmax.assign(d->n_lanes, 0.f); g.dnmax.assign(d->n_lanes, 0.f); g.hmin.assign(d->n_lanes, 1e30f);
    g.cump.assign(np, 0.0); g.cerr.assign(d->n_lanes, 0.0); g.re0.assign(np, 0); g.re1.assign(np, 0);
    for (int gl = 0; gl < d->n_lanes; ++gl) {
        const int off = d->lane_pt_off[gl], n = d->lane_pt_off[gl + 1] - off;
        for (int i = 0; i < n; ++i) {
            const double2 a = make_double2(d->x[off + i], d->y[off + i]);
            g.xy[off + i] = a;
            if (i + 1 < n) {
                const double2 b = make_double2(d->x[off + i + 1], d->y[off + i + 1]);
                const double sx = b.x - a.x, sy = b.y - a.y;
                const double len = sqrt(dg_sq2(sx, sy));
                if (len > 0) g.nrm[off + i] = make_double2(sy / len, -sx / len);
                g.lenp[off + i] = dg_dist_plain(b.x, b.y, a.x, a.y);
                g.lenf[off + i] = len;
                const float h = (float)len * 1.0001f + 1e-6f;
                if (h > g.hmax[gl]) g.hmax[gl] = h;
                const float hl = (float)len * 0.9999f;
                if (hl < g.hmin[gl]) g.hmin[gl] = hl;
            }
        }
        {   // same as dp_map_prep2_kernel: sequential prefix, its rounding bound, run ends
            double acc = 0.0;
            bool dyadic = true;
            for (int i = 0; i < n; ++i) {
                const double t = g.lenp[off + i];
                g.cump[off + i] = acc; acc += t;
                if (t * 1048576.0 != rint(t * 1048576.0)) dyadic = false;
            }
            g.cerr[gl] = (dyadic && acc < 1073741824.0) ? 0.0 : 4.0 * (double)n * 0x1p-53 * acc + 1e-12;
            if (n > 0) { g.re0[off + n - 1] = n - 1; g.re1[off + n - 1] = n - 1; }
            for (int i = n - 2; i >= 0; --i) {
                const int a = d->lanechg_attr[off + i + 1];
                g.re0[off + i] = (a == 1) ? g.re0[off + i + 1] : i;
                g.re1[off + i] = (a & 1) ? g.re1[off + i + 1] : i;
            }
        }
        for (int i = 0; i + 2 < n; ++i) {
            const double2 a = g.nrm[off + i], b = g.nrm[off + i + 1];
            const float dn = (float)sqrt(dg_sq2(b.x - a.x, b.y - a.y)) * 1.0001f + 1e-7f;
            if (dn > g.dnmax[gl]) g.dnmax[gl] = dn;
        }
    }
    DgMap& m = g.m;
    m.xy = g.xy.data(); m.nrm = g.nrm.data(); m.x = d->x; m.y = d->y; m.dir = d->dir;
    m.lenp = g.lenp.data(); m.lenf = g.lenf.data(); m.width = d->lane_width; m.attr = d->lanechg_attr;
    m.road_lane_base = d->road_lane_base; m.lane_pt_off = d->lane_pt_off; m.conn = d->conn;
    m.lane_hmax = g.hmax.data(); m.lane_dnmax = g.dnmax.data(); m.lane_hmin = g.hmin.data();
    m.cump = g.cump.data(); m.lane_cerr = g.cerr.data(); m.run_end0 = g.re0.data(); m.run_end1 = g.re1.data();
    m.n_roads = d->n_roads; m.n_lanes = d->n_lanes; m.n_conn = d->n_conn;
    g.ok = true;
    return 0;
}

// hdr[cycles][n], obs[cycles][n][max_obs], rec[cycles][n], trace / path_xy / path_ll nullable; carry_out[n], last_path_out[n][2][200]
int emu_run_batch_tracks(const dp_params* p, int n, int cycles, int max_obs, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                         const double* vx, const double* vy, const double* dth, int T, dp_plan_record* rec, dp_trace_record* trace,
                         double* path_xy, double* path_ll, dp_carry* carry_out, double* last_path_out, int group);
int emu_run_batch(const dp_params* p, int n, int cycles, int max_obs, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                  dp_plan_record* rec, dp_trace_record* trace, double* path_xy, double* path_ll, dp_carry* carry_out,
                  double* last_path_out, int group) {
    return emu_run_batch_tracks(p, n, cycles, max_obs, hdr, ox, oy, nullptr, nullptr, nullptr, 0, rec, trace, path_xy, path_ll, carry_out,
                                last_path_out, group);
}
// with predicted agent tracks (vx != null): constant-turn-rate parameters [cycles][n][max_obs]
int emu_run_batch_tracks(const dp_params* p, int n, int cycles, int max_obs, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                         const double* vx, const double* vy, const double* dth, int T, dp_plan_record* rec, dp_trace_record* trace,
                         double* path_xy, double* path_ll, dp_carry* carry_out, double* last_path_out, int group) {
    if (!g.ok) return -1;
    constexpr int G = 16, TPB = 256;
    if (group < 1 || group > G) return -2;
    std::vector<dp_carry> carry(n);
    std::vector<double2> last((size_t)n * DP_PATH_POINTS, make_double2(0, 0));
    for (int s = 0; s < n; ++s) {
        std::memset(&carry[s], 0, sizeof(dp_carry));
        carry[s].behavior = 1; carry[s].velocity_expect = 10; carry[s].his_behavior = 1; carry[s].plan_his_behavior = 1;
    }
    DgSmem<G>* sm = new DgSmem<G>();
    DpIo io; std::memset(&io, 0, sizeof(io));
    for (int c = 0; c < cycles; ++c) {
        const size_t e = (size_t)c * n;
        if (vx) { io.trk_vx = vx + e * max_obs; io.trk_vy = vy + e * max_obs; io.trk_dth = dth + e * max_obs; io.trk_T = T; }
        for (int first = 0; first < n; first += group) {
            const int S = (n - first < group) ? n - first : group;
            std::memset(sm, 0xA5, sizeof(*sm));             // uninitialised shared memory
            dg_group_cycle<G, TPB>(g.m, *p, first, S, hdr + e, ox + e * max_obs, oy + e * max_obs, max_obs, carry.data(), last.data(),
                                   rec + e, trace ? trace + e : nullptr, path_xy ? path_xy + e * 400 : nullptr,
                                   path_ll ? path_ll + e * 200 : nullptr, io, *sm);
        }
    }
    delete sm;
    if (carry_out) std::memcpy(carry_out, carry.data(), (size_t)n * sizeof(dp_carry));
    if (last_path_out)
        for (int s = 0; s < n; ++s)
            for (int i = 0; i < DP_PATH_POINTS; ++i) {
                last_path_out[(size_t)s * 400 + i] = last[(size_t)s * DP_PATH_POINTS + i].x;
                last_path_out[(size_t)s * 400 + DP_PATH_POINTS + i] = last[(size_t)s * DP_PATH_POINTS + i].y;
            }
    return 0;
}

}  // extern "C"
