// csrc/dp_group.cuh -- the Decision + Planning cycle as a GROUP kernel (sm_100a): one CTA owns a group of scenes and walks
// them through the cycle phase by phase.
//
// Why this shape (round-2 redesign; the round-1 kernel gave one warp to one scene for the whole cycle and spent 32 lanes on
// every scalar instruction of the rule tree -- 7.6 k warp instructions per scene, 6 % of the FP64 roofline):
//   * scalar phases (Nav_LaneChange, LoadRefPath index math, the BehaviorDecision rule tree, SearchAimPoint,
//     GetVhclLocalState, UpdatePlanJudge, SpeedPlanning ...) run ONE THREAD PER SCENE: a warp advances up to 32 rule trees;
//   * geometry phases are flat work lists over the whole group: one thread per (trajectory, obstacle) pair for the
//     SearchObstacle scans, one per path point for BezierPlanning / MeanPoints, one per (scene, trajectory) for the
//     sequential arclength sums -- every lane has work whatever the obstacle count;
//   * the nearest-point scan is EXACTLY PRUNED: a polyline whose segments are no longer than h satisfies
//     |o - p_j| >= |o - p_i| - |i - j| h, so after sampling one point per cell of 8 only the cells whose sample lies within
//     (best sample + 4 h) can hold the argmin; those are scanned in index order with the reference's strict '<'.  And an
//     obstacle can only pass the corridor test if its nearest path point is closer than Dmax = (Wmax + h/2) / (1 - delta)
//     (Wmax = widest side of the corridor, delta = largest change of direction between consecutive segments; derivation at
//     dg_dmax), so cells farther than Dmax + 4 h are dropped too and most (trajectory, obstacle) pairs end after the 16
//     samples.  The filter runs in FP32 with generous margins, every value that is compared for the result is the FP64 one
//     -- same bits as the full scan;
//   * a scan phase is two compacted passes: pass 1 samples every (trajectory, obstacle) pair and appends the survivors
//     with their cell masks to a list in shared memory, pass 2 gives each survivor to one thread (cells, gates, lateral
//     offset, corridor): lanes stay busy although nine pairs out of ten die in pass 1;
//   * sums the reference evaluates sequentially stay sequential, but never on memory latency: terms are produced by all
//     threads into shared memory first; threshold walks along the map (SearchAimPoint, the lane-change run lengths) are
//     answered from a prefix table with a rounding-error bracket and fall back to the exact loop only inside the bracket;
//   * trajectories are never materialised: a path is a RECIPE (map slice, stride, lateral offset, optional second run, or a
//     window of the local path held in shared memory) evaluated point by point inside the scan;
//   * the carried local path (3200 B per scene, Planning.cpp:6) arrives by one TMA bulk copy per scene
//     (cp.async.bulk + mbarrier) issued at kernel entry and first needed half-way through the cycle.
// Selection = packed (path index << 16 | obstacle index) atomicMin in shared memory: nearest-along-path first, lowest
// obstacle index on ties, independent of the order in which threads arrive (deterministic).
//
// The file is DUAL-TARGET: compiled by nvcc it is the body of dp_group_kernel (dp_cycle.cu); compiled by g++ with -DDP_EMU
// every phase becomes a loop over the CTA's thread ids, which lets tests/ check the kernel's logic against the oracle on a
// box without a GPU (tools/emu, TEST INFRASTRUCTURE -- never linked into libdmpp_b200.so).
// Arithmetic: IEEE binary64, -fmad=false / -ffp-contract=off, fma() exactly where the operator specification says so.
#pragma once
#include <stdint.h>
#include "../../include/dmpp_b200.h"

#if defined(DP_EMU)
#include <cmath>
#include <cstring>
struct double2 { double x, y; };
static inline double2 make_double2(double x, double y) { double2 r; r.x = x; r.y = y; return r; }
struct uint4 { unsigned x, y, z, w; };
#define DG_FN static inline
#define DG_NOINLINE static
#define DG_PHASE(tid) for (int tid = 0; tid < TPB; ++tid)
#define DG_SYNC()
#else
#include <cuda_runtime.h>
#define DG_FN static __device__ __forceinline__
#define DG_NOINLINE static __device__ __noinline__
#define DG_PHASE(tid) for (int tid = (int)threadIdx.x, dg_once_ = 1; dg_once_; dg_once_ = 0)
#define DG_SYNC() __syncthreads()
#endif
#if defined(DP_EMU)
#define DG_MARK(i)
#else
// phase stamps of an instrumented run: thread 0 of every CTA, after the barrier that ends phase i
#define DG_MARK(i) do { if (io.timeline && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); \
                        io.timeline[(size_t)blockIdx.x * 32 + (i)] = (long long)t_; } } while (0)
#endif

#define DG_NREG 4                                  // lane-region trajectories per scene: F, R, NF, NR (junction: slot 0)
#define DG_NSWEEP (2 * (DP_MAX_SWEEP - 1))         // shifted avoid candidates per scene (L1.., R1..)
#define DG_LOCAL (DG_NREG + DG_NSWEEP)             // result slot of the local-path search
#define DG_NRES (DG_LOCAL + 1)
#define DG_SCR DP_PATH_POINTS                      // sequential-sum terms per scene
#define DG_TABCAP 96                               // lane / road offset tables cached in shared memory up to this many entries
#define DG_NQ 8                                    // partial nearest-point searches per scene (25 points each)

struct DgMap {
    const double2* xy;                             // AoS (x, y), built at upload
    const double2* nrm;                            // unit RIGHT normal of segment i -> i+1 (0 at a lane's last point)
    const double* x; const double* y; const double* dir;
    const double* lenp;                            // |p[i+1]-p[i]| = sqrt(dx*dx+dy*dy)        (CalcDistance idiom)
    const double* lenf;                            // |p[i+1]-p[i]| = sqrt(fma(dx,dx,dy*dy))   (SearchObstacle arclength idiom)
    const uint16_t* width; const uint16_t* attr;
    const int32_t* road_lane_base; const int32_t* lane_pt_off;
    const dp_connector* conn;
    const int32_t* lane_next;                      // per lane: successor lane (road lane -> lowest connector leaving it, connector ->
                                                   // its next lane), -1 none; read by the world step with junctions on
    const float* lane_hmax;                        // per lane: upper bound of its segment lengths
    const float* lane_hmin;                        // per lane: lower bound of its segment lengths (0: duplicate points)
    const float* lane_dnmax;                       // per lane: upper bound of |nrm[i+1]-nrm[i]| over the segments of the lane
    const double* cump;                            // per lane: cump[i] = lenp[0] + ... + lenp[i-1], added in index order
    const double* lane_cerr;                       // per lane: bound of |(cump[b]-cump[a]) - (lenp[a] + ... + lenp[b-1] added in order)|;
                                                   // 0 when every term is a multiple of 2^-20 and the total is small: all sums exact
    const int32_t* run_end0; const int32_t* run_end1;   // per point i: first e >= i with e == n-1 or attr[e+1] != 1 (0) / even (1)
    int n_roads, n_lanes, n_conn;
};

// plumbing of one cycle launch, both kernels (dp_cycle.cu: the warp kernel's two halves and the group kernel)
#define DP_MAX_MIRRORS 9
struct DpWait { const unsigned* flag; int n; unsigned value; };
struct DpIo {
    // every finished 128-byte plan record is ALSO stored (one coalesced store each) at mirror[k][scene]: the caller's pinned result
    // buffer (no D2H copy), and/or the gathered-records buffers of the peer GPUs mapped over NVLink (dp_set_record_mirrors, dp_gather_arm)
    dp_plan_record* mirror[DP_MAX_MIRRORS]; int n_mirror;
    // finished Planning warps / scenes of the launch; the last one stores epoch to *host_done (page-locked host memory)
    unsigned* tally; unsigned tally_n; unsigned* host_done; unsigned epoch;
    // fused record gather of a multi-GPU job (dp_gather_*): when the LAST record of the launch is out, flag_value is stored to
    // peer_flag[k] of every rank (one system fence, then relaxed system-scope stores): "rank's slice of this step is complete in your buffer"
    unsigned* peer_flag[DP_MAX_MIRRORS]; int n_peer_flag; unsigned flag_value;
    // ... and the barrier of the PREVIOUS step folded into this launch: after raising its own flags the last warp / CTA waits
    // until wait.flag[0..wait.n) (this rank's flag words of that step, one per rank) all hold wait.value, and only then tells the
    // host -- "this launch is complete" implies "every rank's records of the step before are in my gathered buffer"
    DpWait wait;
    // deferred gather (dp_gather_arm_deferred): the records of the PREVIOUS launch (fwd_src, indexed like rec) are copied to
    // fwd_dst[0..n_fwd) by the warps / CTAs as they START -- the NVLink round trips hide under the cycle -- and the flags above
    // then stand for THAT step: nothing of the gather is left at the end of the launch but one fence, the flags and the wait
    const dp_plan_record* fwd_src; dp_plan_record* fwd_dst[DP_MAX_MIRRORS]; int n_fwd;
    unsigned* tally2; int flag_mode;                        // warp kernel: flags raised at the end of the Decision half (mode 1)
    // warp kernel: per-scene hand-off flags of the overlapped halves (the Decision warp of a scene publishes epoch in done[scene]
    // when its outputs are in memory, the Planning warp of that scene waits for it), and of a submitted cycle's inputs
    // (*in_flag == epoch once they are in the staging set, dp_cycle_submit)
    unsigned* done; const unsigned* in_flag;
    long long* timeline;                           // group kernel, instrumented runs only (tools/group_timeline.py): [block][32] globaltimer stamps
    // group kernel: predicted agent tracks (BASELINE config 5, dp_set_tracks): constant-turn-rate parameters [scene][max_obs] --
    // displacement of step 0 (vx, vy) and heading change per step (deg) -- and the horizon T; null = static obstacles (the reference's semantics)
    const double* trk_vx; const double* trk_vy; const double* trk_dth; int trk_T;
};

#if !defined(DP_EMU)
// one thread: every flag word of a step has arrived (ld.acquire.sys pairs with the st.release.sys of the peers' last warps)
__device__ __forceinline__ void dg_wait_flags(const unsigned* flags, int n, unsigned value) {
    for (int r = 0; r < n; ++r) {
        unsigned v = 0;
        for (long spin = 0; spin < (1L << 26); ++spin) {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + r) : "memory");
            if (v == value) break;
            __nanosleep(100);
        }
        if (v != value) __trap();                           // never spin forever on a rank that is not there
    }
}
// one thread, the last warp / CTA of a launch (or of the warp kernel's Decision half) once every other one has counted itself
// in *tally: re-arm the tally (here: a memset on the copy stream could run as a kernel and find no SM slot), one system fence
// (cumulative: everything the other warps fenced before their increment), this rank's gather flags on every rank (when `raise`),
// the previous step's flags, then the host flag (when `host`)
__device__ __forceinline__ void dg_complete(unsigned* tally, const DpIo& io, bool raise, bool host) {
    *tally = 0;
    __threadfence_system();
#pragma unroll
    for (int k = 0; k < DP_MAX_MIRRORS; ++k)
        if (k < io.n_peer_flag && raise) asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(io.peer_flag[k]), "r"(io.flag_value) : "memory");
    dg_wait_flags(io.wait.flag, io.wait.n, io.wait.value);
    if (host && io.host_done) *reinterpret_cast<volatile unsigned*>(io.host_done) = io.epoch;
}
#endif

// ---- small portable helpers ---------------------------------------------------------------------------------------------
DG_FN int dg_imin(int a, int b) { return a < b ? a : b; }
DG_FN int dg_imax(int a, int b) { return a > b ? a : b; }
DG_FN double dg_inf() {
#if defined(DP_EMU)
    return INFINITY;
#else
    return __longlong_as_double(0x7ff0000000000000LL);
#endif
}
DG_FN float dg_inff() {
#if defined(DP_EMU)
    return INFINITY;
#else
    return __int_as_float(0x7f800000);
#endif
}
DG_FN void dg_atomic_min_u32(unsigned* p, unsigned v) {
#if defined(DP_EMU)
    if (v < *p) *p = v;
#else
    atomicMin(p, v);
#endif
}
DG_FN void dg_atomic_max_i32(int* p, int v) {
#if defined(DP_EMU)
    if (v > *p) *p = v;
#else
    atomicMax(p, v);
#endif
}
DG_FN int dg_atomic_add_i32(int* p, int v) {
#if defined(DP_EMU)
    const int o = *p; *p = o + v; return o;
#else
    return atomicAdd(p, v);
#endif
}
DG_FN unsigned dg_float_bits(float f) {
#if defined(DP_EMU)
    unsigned u; std::memcpy(&u, &f, 4); return u;
#else
    return __float_as_uint(f);
#endif
}
DG_FN float dg_bits_float(unsigned u) {
#if defined(DP_EMU)
    float f; std::memcpy(&f, &u, 4); return f;
#else
    return __uint_as_float(u);
#endif
}
DG_FN double dg_sq2(double dx, double dy) { return fma(dx, dx, dy * dy); }
DG_FN double dg_dist_plain(double ax, double ay, double bx, double by) {
    const double dx = ax - bx, dy = ay - by;
    return sqrt(dx * dx + dy * dy);
}

// spec_sincos_deg / spec_atan: fixed polynomials shared (as text, not as code) with the oracle (oracle/cshare_spec.h)
DG_NOINLINE void dg_sincos_deg(double a, double* c, double* s) {
    const double k = rint(a / 90.0);
    const double r = fma(-90.0, k, a);
    const double x = r * (3.14159265358979323846 / 180.0);
    const double x2 = x * x;
    double ps = -1.0 / 355687428096000.0;
    ps = fma(x2, ps, 1.0 / 1307674368000.0);
    ps = fma(x2, ps, -1.0 / 6227020800.0);
    ps = fma(x2, ps, 1.0 / 39916800.0);
    ps = fma(x2, ps, -1.0 / 362880.0);
    ps = fma(x2, ps, 1.0 / 5040.0);
    ps = fma(x2, ps, -1.0 / 120.0);
    ps = fma(x2, ps, 1.0 / 6.0);
    const double sn = fma(-x * x2, ps, x);
    double pc = 1.0 / 20922789888000.0;
    pc = fma(x2, pc, -1.0 / 87178291200.0);
    pc = fma(x2, pc, 1.0 / 479001600.0);
    pc = fma(x2, pc, -1.0 / 3628800.0);
    pc = fma(x2, pc, 1.0 / 40320.0);
    pc = fma(x2, pc, -1.0 / 720.0);
    pc = fma(x2, pc, 1.0 / 24.0);
    pc = fma(x2, pc, -0.5);
    const double cs = fma(x2, pc, 1.0);
    const long long q = (long long)k;
    const int mq = (int)(((q % 4) + 4) % 4);
    if (mq == 0) { *c = cs; *s = sn; }
    else if (mq == 1) { *c = -sn; *s = cs; }
    else if (mq == 2) { *c = -cs; *s = -sn; }
    else { *c = sn; *s = -cs; }
}
DG_NOINLINE double dg_atan(double z) {
    const double PI_2 = 1.57079632679489661923, PI_4 = 0.78539816339744830962;
    const bool neg = z < 0;
    double a = neg ? -z : z;
    const bool inv = a > 1.0;
    if (inv) a = 1.0 / a;
    const bool shift = a > 0.41421356237309503;
    const double w = shift ? (a - 1.0) / (a + 1.0) : a;
    const double w2 = w * w;
    double p = 1.0 / 47.0;
#pragma unroll
    for (int n = 22; n >= 0; --n) {
        const double c = 1.0 / (double)(2 * n + 1);
        p = fma(-w2, p, c);
    }
    double r = w * p;
    if (shift) r = PI_4 + r;
    if (inv) r = PI_2 - r;
    return neg ? -r : r;
}
// CalcGlobalDir / GetRoadAngle (Planning.cpp:719-750)
DG_NOINLINE double dg_heading(double ax, double ay, double bx, double by, double eps, double pi) {
    double angle;
    if (fabs(bx - ax) < eps && fabs(by - ay) < eps) angle = 0;
    else if (fabs(bx - ax) < eps) angle = (by > ay) ? pi / 2 : 3 * pi / 2;
    else {
        angle = dg_atan((by - ay) / (bx - ax));
        if (bx < ax) angle = angle + pi;
        else if ((bx > ax) && (by < ay)) angle = angle + 2 * pi;
    }
    return angle * 180 / pi;
}
// GetLatDis (Planning.cpp:686-709), LEFT positive
DG_NOINLINE double dg_lat_dis(double cx, double cy, double px, double py, double nx, double ny, double eps) {
    double l;
    if (fabs(px - nx) > eps) {
        const double k = (py - ny) / (px - nx);
        l = fabs((cy - py) - k * (cx - px)) / sqrt(1 + k * k);
    } else l = fabs(px - cx);
    if (l < eps) return 0.0;
    const double c = (nx - px) * (cy - py) - (ny - py) * (cx - px);
    return l * (c > 0 ? 1 : -1);
}
// GetAngleErr (Planning.cpp:760-786)
DG_FN double dg_angle_err(double d1, double d2) {
    double e = d2 - d1;
    if (d1 < 180) e = (d2 - d1 <= 180) ? d2 - d1 : d2 - d1 - 360;
    else if (d1 >= 180) e = (d2 - d1 > -180) ? d2 - d1 : d2 - d1 + 360;
    return e;
}

// ---- trajectories as recipes ---------------------------------------------------------------------------------------------
// Up to two runs of points behind ONE generic base pointer (the AoS map, or the scene's local path in shared memory):
// run 0 = pts[base0 + stride0 * j], j < n0 (stride -1: the rear slices of LoadRefPath); run 1 = pts[base1 + (j - n0)];
// d != 0 (single run only) applies CreateNewPath while the point is read: p + d * n with the precomputed unit normals.
struct DgPath {
    double d, lo, hi;                              // lateral offset (RIGHT positive), corridor window of the search
    int base0, stride0, n0, base1, n1;
    float hb;                                      // upper bound of the trajectory's segment lengths (pruning radius per index step)
    float dmax;                                    // an obstacle farther than this from every point cannot pass the corridor test
    unsigned key;                                  // packed (path index << 16 | obstacle) minimum over the in-corridor obstacles
    int local;                                     // 1: window of the local path in shared memory
};
struct DgView {
    const double2* pts; const double2* nrm;
    int base0, stride0, n0, base1, n1;
    double d;
};
DG_FN double2 dg_pt(const DgView& v, int j) {
    const int idx = (j < v.n0) ? v.base0 + v.stride0 * j : v.base1 + (j - v.n0);
    return v.pts[idx];
}
// CShare::CreateNewPath fused in (segment normal of point j: min(j, P-2); reversed runs use the mirrored normal)
DG_FN double2 dg_pt_off(const DgView& v, int j) {
    double2 q = dg_pt(v, j);
    if (j < v.n0 && v.n0 >= 2) {
        const int jj = dg_imin(j, v.n0 - 2);
        double2 n = (v.stride0 > 0) ? v.nrm[v.base0 + jj] : v.nrm[v.base0 - jj - 1];
        if (v.stride0 < 0) { n.x = -n.x; n.y = -n.y; }
        q.x = fma(v.d, n.x, q.x); q.y = fma(v.d, n.y, q.y);
    }
    return q;
}
DG_FN double2 dg_point_any(const DgView& v, int j) { return (v.d != 0.0) ? dg_pt_off(v, j) : dg_pt(v, j); }
// MODE 0: one plain run (the common case: a lane slice or the local path), MODE 1: anything (second run, lateral offset)
template <int MODE> DG_FN double2 dg_jpt(const DgView& v, int j) {
    if (MODE == 0) return v.pts[v.base0 + v.stride0 * j];
    return dg_point_any(v, j);
}

// Reach of a corridor.  Let D be the distance from an obstacle o to its nearest path point p_j, h an upper bound of the
// segment lengths and delta an upper bound of |dir(k+1) - dir(k)| between consecutive unit segment directions.  The
// specification measures the lateral offset d against segment k = min(j, P-2) and gates the two end points.  Because the
// neighbours of p_j are not closer than p_j, the component t of (o - p_k) along segment k obeys |t| <= h/2 + D delta
// (interior j: t <= |s_k|/2 from p_{j+1}; (o-p_j).dir(k-1) >= -|s_{k-1}|/2 from p_{j-1}, and dir(k) differs from dir(k-1) by
// at most delta; j = 0 and j = P-1: the gate and the one neighbour give 0 <= |t| <= h/2).  With d^2 = D^2 - t^2, an obstacle
// inside the corridor (|d| <= Wmax) has D <= Wmax + h/2 + D delta, i.e. D <= (Wmax + h/2) / (1 - delta).
// Paths with duplicate points (a zero-length segment has d = 0 whatever the distance) or sharp corners get no filter.
DG_FN float dg_dmax(double lo, double hi, float hb, float delta, float hmin) {
    if (!(hmin > 1e-6f) || !(delta < 0.5f)) return dg_inff();
    const float wm = (float)fmax(fabs(lo), fabs(hi));
    return (wm + 0.5f * hb) / (1.0f - delta) * 1.001f + 1e-3f;
}

struct DgArg { double bd; int bj; };

// ---- exactly pruned nearest-point search: argmin_j |o - p_j|^2 with value fma(dx,dx,dy*dy) and strict '<' (lowest index on
// ties), step 1 of the SearchObstacle specification (oracle/cshare_spec.h), restricted to obstacles within dmax of the path.
// Pass 1 (dg_coarse): one sample per cell of 8 points; a cell can hold a point at distance <= X only if its sample is within
// X + 4 hb.  X = min(best sample so far, dmax).  Returns the cells to visit as a bit mask (bit = cell index, P <= 512).
template <class PF>
DG_FN unsigned long long dg_coarse_f(PF pt, const int P, const double ox, const double oy, const float hb, const float dmax) {
    const float FINF = dg_inff();
    float ubf = FINF;                              // upper bound of the minimum DISTANCE over the path, FP32, rounded up
    const float R = 4.0f * hb * 1.0001f + 1e-3f;   // a cell's points are at most 4 index steps from its sample
    unsigned long long mask = 0;
    for (int c0 = 0, ch = 0; c0 < P; c0 += 128, ++ch) {
        float dc[16];
        float mn = FINF;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const int j0 = c0 + 8 * c;
            float f = FINF;
            if (j0 < P) {
                const double2 q = pt(dg_imin(j0 + 4, P - 1));
                const double dx = ox - q.x, dy = oy - q.y;
                f = (float)fma(dx, dx, dy * dy);
            }
            dc[c] = f;
            mn = fminf(mn, f);
        }
        ubf = fminf(ubf, sqrtf(mn) * 1.0001f + 1e-3f);
        const float thr = fminf(ubf, dmax) + R;
        const float thr2 = thr * thr * 1.0001f;
        unsigned m16 = 0;
#pragma unroll
        for (int c = 0; c < 16; ++c) m16 |= (dc[c] <= thr2) ? (1u << c) : 0u;
        mask |= (unsigned long long)m16 << (16 * ch);
    }
    return mask;
}
// Pass 2 (dg_refine): the marked cells in index order, strict '<' keeps the lowest index
template <class PF>
DG_FN DgArg dg_refine_f(PF pt, const int P, const double ox, const double oy, unsigned long long mask) {
    const double INF = dg_inf();
    DgArg r; r.bd = INF; r.bj = 0;
    while (mask) {
#if defined(DP_EMU)
        const int c = __builtin_ctzll(mask);
#else
        const int c = __ffsll((long long)mask) - 1;
#endif
        mask &= mask - 1;
        const int jb = 8 * c;
        double e[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int j = jb + k;
            const double2 q = pt(dg_imin(j, P - 1));
            const double dx = ox - q.x, dy = oy - q.y;
            e[k] = (j < P) ? fma(dx, dx, dy * dy) : INF;
        }
        // tournament that prefers the lower index on ties
        int i01 = 0, i23 = 2, i45 = 4, i67 = 6;
        double e01 = e[0], e23 = e[2], e45 = e[4], e67 = e[6];
        if (e[1] < e01) { e01 = e[1]; i01 = 1; }
        if (e[3] < e23) { e23 = e[3]; i23 = 3; }
        if (e[5] < e45) { e45 = e[5]; i45 = 5; }
        if (e[7] < e67) { e67 = e[7]; i67 = 7; }
        if (e23 < e01) { e01 = e23; i01 = i23; }
        if (e67 < e45) { e45 = e67; i45 = i67; }
        if (e45 < e01) { e01 = e45; i01 = i45; }
        if (e01 < r.bd) { r.bd = e01; r.bj = jb + i01; }
    }
    return r;
}
// Moving agents (BASELINE config 5): fused rollout -> nearest-point search of ONE agent against ONE trajectory.  The agent follows
// the constant-turn-rate model of oracle/cshare_spec.h (rollout_ctr): position j+1 = position j + v_j, v_{j+1} = v_j rotated by
// dtheta, frozen after step T-1; it is at position j when the ego reaches path point j.  The predicted track is never
// materialised: the recurrence advances in registers while the path is walked, strict '<' keeps the lowest index, and the
// agent's position at the argmin is what steps 2-5 of SearchObstacle (gates, lateral offset, corridor) see.
struct DgTrk { double x, y; DgArg a; };
template <class PF>
DG_FN DgTrk dg_track_search(PF pt, const int P, double x, double y, double vx, double vy, const double dth, const int T) {
    double c, s;
    dg_sincos_deg(dth, &c, &s);
    DgTrk r; r.x = x; r.y = y; r.a.bd = dg_inf(); r.a.bj = 0;
    int j = 0;
    for (; j + 4 <= P; j += 4) {                   // four path points in flight per trip: their loads do not wait for the recurrence
        const double2 q0 = pt(j), q1 = pt(j + 1), q2 = pt(j + 2), q3 = pt(j + 3);
#define DG_TRK_STEP(q, jj) { const double dx = x - (q).x, dy = y - (q).y; const double e = fma(dx, dx, dy * dy); \
                             if (e < r.a.bd) { r.a.bd = e; r.a.bj = (jj); r.x = x; r.y = y; } \
                             if ((jj) + 1 < T) { x = x + vx; y = y + vy; const double nvx = fma(c, vx, -(s * vy)), nvy = fma(s, vx, c * vy); vx = nvx; vy = nvy; } }
        DG_TRK_STEP(q0, j) DG_TRK_STEP(q1, j + 1) DG_TRK_STEP(q2, j + 2) DG_TRK_STEP(q3, j + 3)
    }
    for (; j < P; ++j) { const double2 q = pt(j); DG_TRK_STEP(q, j) }
#undef DG_TRK_STEP
    return r;
}
// the agent's position at step j (the same recurrence, for the one selected agent of a trajectory)
DG_FN double2 dg_track_pos(double x, double y, double vx, double vy, const double dth, const int T, const int j) {
    double c, s;
    dg_sincos_deg(dth, &c, &s);
    for (int i = 0; i < j && i + 1 < T; ++i) {
        x = x + vx; y = y + vy;
        const double nvx = fma(c, vx, -(s * vy)), nvy = fma(s, vx, c * vy);
        vx = nvx; vy = nvy;
    }
    return make_double2(x, y);
}

template <int MODE>
DG_FN unsigned long long dg_coarse(const DgView& v, const int P, const double ox, const double oy, const float hb, const float dmax) {
    return dg_coarse_f([&](int j) { return dg_jpt<MODE>(v, j); }, P, ox, oy, hb, dmax);
}
template <int MODE>
DG_FN DgArg dg_refine(const DgView& v, const int P, const double ox, const double oy, unsigned long long mask) {
    return dg_refine_f([&](int j) { return dg_jpt<MODE>(v, j); }, P, ox, oy, mask);
}
// The cells that survive the reach filter hold the true nearest point whenever it lies within dmax; when it does not, the
// best point found may be a different one (and its lateral offset meaningless): such an obstacle cannot be in the corridor
// and is dropped by comparing the FP64 minimum with dmax (dmax already carries its rounding margins).
DG_FN bool dg_within_reach(double bd, float dmax) { return !(bd > (double)dmax * (double)dmax); }
// paths longer than 512 points: both passes chunk by chunk in one thread (bj = -1: nothing within reach)
DG_NOINLINE DgArg dg_scan_long(const DgView v, const int P, const double ox, const double oy, const float hb, const float dmax) {
    const float FINF = dg_inff();
    DgArg r; r.bd = dg_inf(); r.bj = -1;
    float ubf = FINF;
    const float R = 4.0f * hb * 1.0001f + 1e-3f;
    for (int c0 = 0; c0 < P; c0 += 8) {            // plain two-level walk, one cell at a time (rare shape, not tuned)
        const double2 q = dg_point_any(v, dg_imin(c0 + 4, P - 1));
        const double dx = ox - q.x, dy = oy - q.y;
        const float f = (float)fma(dx, dx, dy * dy);
        ubf = fminf(ubf, sqrtf(f) * 1.0001f + 1e-3f);
        const float thr = fminf(ubf, dmax) + R;
        if (f <= thr * thr * 1.0001f) {
            for (int j = c0; j < dg_imin(c0 + 8, P); ++j) {
                const double2 w = dg_point_any(v, j);
                const double ex = ox - w.x, ey = oy - w.y;
                const double e = fma(ex, ex, ey * ey);
                if (e < r.bd) { r.bd = e; r.bj = j; }
            }
            if (r.bj >= 0) ubf = fminf(ubf, sqrtf((float)r.bd) * 1.0001f + 1e-3f);
        }
    }
    return r;
}

// steps 2-5 of the SearchObstacle specification for one obstacle whose nearest path point is bj: end gates, signed lateral
// offset (RIGHT positive) against segment k = min(bj, P-2), corridor test.  Returns the packed selection key, d in *dout.
DG_FN unsigned dg_key(const DgView& v, int P, int bj, int o, double ox, double oy, double lo, double hi, double* dout) {
    const int k = (bj == P - 1) ? P - 2 : bj;
    const double2 pk = dg_point_any(v, k), pk1 = dg_point_any(v, k + 1);
    const double sx = pk1.x - pk.x, sy = pk1.y - pk.y;
    *dout = 0.0;
    if (bj == 0) { if (!(fma(ox - pk.x, sx, (oy - pk.y) * sy) >= 0.0)) return 0xffffffffu; }
    else if (bj == P - 1) { if (!(fma(ox - pk1.x, sx, (oy - pk1.y) * sy) <= 0.0)) return 0xffffffffu; }
    const double cross = fma(ox - pk.x, sy, -((oy - pk.y) * sx));
    const double len2 = dg_sq2(sx, sy);
    {   // FP32 pre-reject of obstacles far outside the corridor (|d| = |cross| / len): saves the FP64 sqrt and division
        const float cf = (float)cross, lf = (float)len2;
        const float wm = (float)fmax(fabs(lo), fabs(hi)) * 1.001f + 0.01f;
        if (cf * cf > wm * wm * lf * 1.001f) return 0xffffffffu;
    }
    const double len = sqrt(len2);
    double d = 0.0;
    if (len > 0) d = cross / len;
    *dout = d;
    if (!(d >= lo && d <= hi)) return 0xffffffffu;
    return ((unsigned)bj << 16) | (unsigned)o;
}

// segment length |p[j+1]-p[j]| of a trajectory in the SearchObstacle idiom sqrt(fma(dx,dx,dy*dy)): table look-up for plain
// map runs (the table holds exactly this expression; a reversed run negates dx and dy, the squares are identical)
DG_FN double dg_seg_fma(const DgView& v, const double* lenf, int j) {
    if (lenf && v.d == 0.0) {
        if (j + 1 < v.n0) return lenf[(v.stride0 > 0) ? v.base0 + j : v.base0 - j - 1];
        if (j >= v.n0) return lenf[v.base1 + (j - v.n0)];
    }
    const double2 a = dg_point_any(v, j), b = dg_point_any(v, j + 1);
    return sqrt(dg_sq2(b.x - a.x, b.y - a.y));
}

struct DgRes { double dis_lat, dis_lng; int ob, pathid, found, pad; };
DG_FN DgRes dg_res_none() {
    DgRes r; r.dis_lat = DP_NOT_FOUND; r.dis_lng = DP_NOT_FOUND; r.ob = -1; r.pathid = 0; r.found = 0; r.pad = 0;
    return r;
}
// sum of n terms in index order: the first min(n, cap) from shared memory (produced in parallel by the phase before), the
// rest through `tail(j)`.  stop_above >= 0: only the decision `sum > stop_above` is consumed (avoid sweep, Decision.cpp:944):
// partial sums of non-negative terms are monotone, the sum may stop at the end of the first block of 8 beyond the threshold.
template <class Tail>
DG_FN double dg_seq_sum(const double* t, int n, int cap, double stop_above, Tail tail) {
    double sum = 0.0;
    const int m = dg_imin(n, cap);
    int j = 0;
    for (; j + 8 <= m; j += 8) {
        const double t0 = t[j], t1 = t[j + 1], t2 = t[j + 2], t3 = t[j + 3], t4 = t[j + 4], t5 = t[j + 5], t6 = t[j + 6], t7 = t[j + 7];
        sum += t0; sum += t1; sum += t2; sum += t3; sum += t4; sum += t5; sum += t6; sum += t7;
        if (stop_above >= 0.0 && sum > stop_above) return sum;
    }
    for (; j < m; ++j) sum += t[j];
    for (; j < n; ++j) {
        sum += tail(j);
        if (stop_above >= 0.0 && sum > stop_above) return sum;
    }
    return sum;
}

// first index j < n whose running sum t[0] + ... + t[j] (index order) satisfies (sum - 4 > far), -1 if none: the walk of
// SearchAimPoint (Planning.cpp:410-432, 505-530).  The first min(n, cap) terms come from shared memory, the rest through
// tail(j); partial sums are evaluated 8 at a time with one exit test per block (terms >= 0: the test is monotone).
template <class Tail>
DG_FN int dg_first_hit(const double* t, int n, int cap, double far, Tail tail) {
    double sum = 0.0;
    const int m = dg_imin(n, cap);
    int j = 0;
    for (; j + 8 <= m; j += 8) {
        const double s0 = sum + t[j], s1 = s0 + t[j + 1], s2 = s1 + t[j + 2], s3 = s2 + t[j + 3];
        const double s4 = s3 + t[j + 4], s5 = s4 + t[j + 5], s6 = s5 + t[j + 6], s7 = s6 + t[j + 7];
        if ((s7 - 4.0) > far) {
            int hit = j + 7;
            if ((s6 - 4.0) > far) hit = j + 6;
            if ((s5 - 4.0) > far) hit = j + 5;
            if ((s4 - 4.0) > far) hit = j + 4;
            if ((s3 - 4.0) > far) hit = j + 3;
            if ((s2 - 4.0) > far) hit = j + 2;
            if ((s1 - 4.0) > far) hit = j + 1;
            if ((s0 - 4.0) > far) hit = j;
            return hit;
        }
        sum = s7;
    }
    for (; j < n; ++j) {
        sum += (j < m) ? t[j] : tail(j);
        if ((sum - 4.0) > far) return j;
    }
    return -1;
}

DG_FN void dg_put_slot(dp_search_slot* slot, const DgRes& r, int evaluated) {
    slot->dis_lat = r.dis_lat; slot->dis_lng = r.dis_lng; slot->ob_index = (int16_t)r.ob;
    slot->pathid = (uint16_t)r.pathid; slot->evaluated = (uint8_t)evaluated; slot->found = r.found ? 1 : 0;
    slot->pad[0] = slot->pad[1] = 0;
}

// avoid-sweep candidate numbering (Decision.cpp:940-974): reference order L0..L(K-1), R0..R(K-1) = g; candidate 0 of either
// side is F itself under the F region's window (result known, never feasible when the sweep runs), so only the 2(K-1)
// shifted candidates u = 0..2(K-1)-1 are scored
DG_FN int dg_sweep_g(int u, int K) { return (u >= K - 1) ? u + 2 : u + 1; }
DG_FN double dg_sweep_offset(int g, int K) { return (g < K) ? -0.3 * g : 0.3 * (g - K); }

// ---- per-scene control block: the scalars that flow from phase to phase ---------------------------------------------------
struct DgCtl {
    double W, v_exp;
    double bx0, by0, bx1, by1, bx2, by2, bx3, by3;  // Bezier control points of the (re)planning request
    double lat, dir_err, remain;
    int N, pos, gl, lane_sum, lane_n, id, side, lanechg, K;
    int navi, navi_t;
    int ub, n_traj, pts;
    int beh, target, light, lanechg_st, obsavoid, dlg;   // Cur_Behavior while the rule tree is split around the sweep
    int sweep_on, sweep_cnt, sweep_pick;
    int rp_base0, rp_n0, rp_base1, rp_n1;          // DecisionOut.refpath as a recipe
    int d_behavior, d_target;
    float faraim;
    int walk_kind, woff, wgl, wfrom, wto, fb_off, fb_idx, fb_n, fb_id;
    int walk_hit, walk_exact;                      // look-ahead walk answered from the prefix table (-1: no hit); 1: the exact loop decides
    int first, near_id, front_id, afresh, cause, plan_dirty, req;   // req: 0 reuse, 1 Bezier, 2 MeanPoints, 3 zero path
    int mean_n, s0;
    unsigned hb2_bits, hmin2_bits, dl2_bits;       // local path: max / min squared segment length, max squared direction change (FP32 bits)
};

// one trajectory of a scan phase, by value
struct DgJob {
    DgView v; double lo, hi; unsigned* key; int P, scene; float hb, dmax;
    const double* tvx; const double* tvy; const double* tdth; int tT;     // the scene's agent tracks (null: static obstacles)
};

template <int G>
struct DgSmem {
    dp_scene_hdr hdr[G];
    dp_carry carry[G];
    dp_plan_record rec[G];
    double2 plan[G][DP_PATH_POINTS];               // term pool of the decision half; last_Bpoints (TMA bulk copy) / road_points afterwards
    double scr[G][DG_SCR + 8];                     // survivor lists of the scan phases; sequential-sum terms of the planning half
    DgPath path[G][DG_NREG + 1];                   // F, R, NF, NR, local
    DgRes res[G][DG_NRES];
    unsigned swkey[G][DG_NSWEEP];
    DgCtl ctl[G];
    double ne[G][DG_NQ]; int ni[G][DG_NQ]; int namb[G][DG_NQ];
    int sweep_list[G];
    int lpo[DG_TABCAP], rlb[DG_TABCAP];
    unsigned long long mbar;
    int nsurv[2];
    int maxN, n_sweep, any_first, any_mean, any_junction, tab_ok;
};
#define DG_POOL (2 * DP_PATH_POINTS)               // doubles in one scene's term pool (its slot of sm.plan)

// ---- TMA bulk copy global -> shared (cp.async.bulk, SASS UBLKCP) with an mbarrier ------------------------------------------
#if !defined(DP_EMU)
DG_FN uint32_t dg_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
DG_FN void dg_mbar_init(unsigned long long* mbar, uint32_t bytes) {
    const uint32_t mb = dg_smem_u32(mbar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
}
DG_FN void dg_bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, unsigned long long* mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dg_smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(dg_smem_u32(mbar)) : "memory");
}
DG_FN void dg_mbar_wait(unsigned long long* mbar) {
    const uint32_t mb = dg_smem_u32(mbar);
    uint32_t done = 0;
    for (int spin = 0; spin < (1 << 24) && !done; ++spin) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(mb) : "memory");
    }
    if (!done) __trap();                           // never spin forever on a broken copy
}
#endif

// forward 120-point / backward 40-point slices of one lane (Decision.cpp:581-596, 611-622, 649-660)
DG_FN void dg_lane_slices(const int* lpo, int gl, int id, int id_more, DgPath& fwd, DgPath& rear, int& ub) {
    const int off = lpo[gl], n = lpo[gl + 1] - off;
    const int a = dg_imin(n, id + id_more), b = dg_imin(n, id + 120 + id_more);
    fwd.base0 = off + a; fwd.stride0 = 1; fwd.n0 = dg_imax(0, b - a);
    const int lo = dg_imax(0, id + id_more - 40);
    int start = a;
    if (start >= n) { start = n - 1; if (a > lo) ++ub; }    // reference reads index == size here (UB); clamp
    rear.base0 = off + start; rear.stride0 = -1; rear.n0 = dg_imax(0, a - lo);
}
// pruning bounds of a (possibly laterally shifted) slice of lane gl: hb >= its segment lengths, dmax = reach of its corridor.
// A shift by d changes a segment vector by d (n[j+1] - n[j]): lengths by at most |d| dn, unit directions by at most
// 2 |d| dn / hmin, so consecutive directions of the shifted line differ by at most dn (1 + 4 |d| / hmin).
DG_FN void dg_bounds(const DgMap& m, int gl, double d, double lo, double hi, float* hb, float* dmax) {
    const float ad = (float)fabs(d) * 1.0001f;
    const float hmax = m.lane_hmax[gl], hmin = m.lane_hmin[gl], dn = m.lane_dnmax[gl];
    *hb = hmax + ad * dn + 1e-4f;
    float delta = dn;
    if (ad > 0.f) delta = (hmin > 1e-6f) ? dn * (1.0f + 4.0f * ad / hmin) * 1.0001f + 1e-6f : 2.0f;
    *dmax = dg_dmax(lo, hi, *hb, delta, hmin - ad * dn);
}
DG_FN DgView dg_view(const DgMap& m, const DgPath& p, const double2* plan) {
    DgView v;
    v.pts = p.local ? plan : m.xy; v.nrm = m.nrm;
    v.base0 = p.base0; v.stride0 = p.stride0; v.n0 = p.n0; v.base1 = p.base1; v.n1 = p.n1; v.d = p.d;
    return v;
}

// does the arclength from `id` along lane gl (points off .. off+n-1), while cond(attr[i+1]) holds, exceed thr?
// (Decision.cpp:1179-1190 and siblings)  mode: 0 = attr == 1, 1 = attr & 1, 2 = never.  The run ends at run_end[id]; its
// length is cump[end] - cump[id] up to the rounding bound lane_cerr: outside that bracket the answer needs no walk, inside
// it the reference's own loop decides (partial sums of non-negative terms are monotone: it stops at the first sum > thr).
DG_NOINLINE bool dg_run_exceeds(const DgMap& m, int gl, int off, int n, int id, int mode, double thr) {
    if (mode == 2 || id >= n - 1) return 0.0 > thr;
    const int e = (mode == 0 ? m.run_end0 : m.run_end1)[off + id];
    const double approx = m.cump[off + e] - m.cump[off + id], err = m.lane_cerr[gl];
    if (approx > thr + err) return true;
    if (approx < thr - err) return false;
    double sum = 0.0;
    for (int i = id; i < n - 1; ++i) {
        const int a = m.attr[off + i + 1];
        const bool ok = (mode == 0) ? (a == 1) : ((a & 1) != 0);
        if (!ok) break;
        sum += m.lenp[off + i];
        if (sum > thr) return true;
    }
    return sum > thr;
}

// nearest-of-200 partial (GetVhclLocalState, Planning.cpp:640-648) over points [i0, i1): squared distances in the reference's
// own operations; `amb` flags a displaced earlier minimum within 2^-49 (its rounded sqrt may tie: resolved by the exact loop)
DG_FN void dg_nearest_part(const double2* pts, int i0, int i1, double x, double y, double* be_out, int* bi_out, int* amb_out) {
    const double TOL = 1.0 + 0x1p-49;
    double be = dg_inf();
    int bi = 0x7fffffff, amb = 0;
    for (int i = i0; i < i1; ++i) {
        const double2 q = pts[i];
        const double dx = x - q.x, dy = y - q.y;
        const double e = dx * dx + dy * dy;
        if (e < be) { if (be <= e * TOL) amb = 1; be = e; bi = i; }
    }
    *be_out = be; *bi_out = bi; *amb_out = amb;
}

#if defined(DP_EMU)
#define DG_BODY static void
#else
#define DG_BODY static __device__ __forceinline__ void
#endif

// ---- one scan phase: every (trajectory jb, obstacle o) pair of the group, jb < njobs, job(jb) describes the trajectory ----
// pass 1 samples the pair and appends the survivors (pair id, cell mask) to a list that lives in sm.scr; pass 2 hands each
// survivor to one thread: marked cells, gates, lateral offset, corridor, packed-key atomicMin into the trajectory's slot.
template <int G, int TPB, class JobFn>
DG_BODY dg_scan_phase(DgSmem<G>& sm, const int njobs, const int first, const double* obs_x, const double* obs_y, const int max_obs, JobFn job) {
    const int maxN = sm.maxN;
    constexpr int TILE = G * 128;                  // pairs per tile: 4 B + 8 B per survivor fit sm.scr (G * 1664 B)
    unsigned* list = reinterpret_cast<unsigned*>(&sm.scr[0][0]);
    unsigned long long* masks = reinterpret_cast<unsigned long long*>(list + TILE);
    const int total = njobs * maxN;
    for (int t0 = 0, tile = 0; t0 < total; t0 += TILE, ++tile) {
        int* cnt = &sm.nsurv[tile & 1];            // (zero on entry: the caller clears both, pass 2 clears the other one)
        DG_PHASE(tid) {
            const int tend = dg_imin(total, t0 + TILE);
            for (int it = t0 + tid; it < tend; it += TPB) {
                const int o = it % maxN, jb = it / maxN;
                const DgJob jq = job(jb);
                if (jq.P < 2 || o >= sm.ctl[jq.scene].N) continue;
                const size_t ob = (size_t)(first + jq.scene) * max_obs + o;
                const double ox = obs_x[ob], oy = obs_y[ob];
                if (jq.tvx) {                      // predicted tracks: fused rollout + search of this agent, no survivor list
                    const DgView& vv = jq.v;
                    const DgTrk t = dg_track_search([&](int j) { return dg_point_any(vv, j); }, jq.P, ox, oy, jq.tvx[o], jq.tvy[o], jq.tdth[o], jq.tT);
                    double d;
                    const unsigned key = dg_key(vv, jq.P, t.a.bj, o, t.x, t.y, jq.lo, jq.hi, &d);
                    if (key != 0xffffffffu) dg_atomic_min_u32(jq.key, key);
                    continue;
                }
                if (jq.P > 512) {                  // longer than the 64-cell mask: the whole search in this thread
                    const DgArg a = dg_scan_long(jq.v, jq.P, ox, oy, jq.hb, jq.dmax);
                    if (a.bj >= 0 && dg_within_reach(a.bd, jq.dmax)) {
                        double d;
                        const unsigned key = dg_key(jq.v, jq.P, a.bj, o, ox, oy, jq.lo, jq.hi, &d);
                        if (key != 0xffffffffu) dg_atomic_min_u32(jq.key, key);
                    }
                    continue;
                }
                const bool plain = (jq.v.n1 == 0 && jq.v.d == 0.0);
                const unsigned long long mk = plain ? dg_coarse<0>(jq.v, jq.P, ox, oy, jq.hb, jq.dmax) : dg_coarse<1>(jq.v, jq.P, ox, oy, jq.hb, jq.dmax);
                if (mk) {
                    const int pos = dg_atomic_add_i32(cnt, 1);
                    list[pos] = (unsigned)(it - t0); masks[pos] = mk;
                }
            }
        }
        DG_SYNC();
        DG_PHASE(tid) {
            if (tid == 0) sm.nsurv[(tile + 1) & 1] = 0;
            const int ns = *cnt;
            for (int e = tid; e < ns; e += TPB) {
                const int it = t0 + (int)list[e];
                const int o = it % maxN, jb = it / maxN;
                const DgJob jq = job(jb);
                const size_t ob = (size_t)(first + jq.scene) * max_obs + o;
                const double ox = obs_x[ob], oy = obs_y[ob];
                const bool plain = (jq.v.n1 == 0 && jq.v.d == 0.0);
                const DgArg a = plain ? dg_refine<0>(jq.v, jq.P, ox, oy, masks[e]) : dg_refine<1>(jq.v, jq.P, ox, oy, masks[e]);
                if (!dg_within_reach(a.bd, jq.dmax)) continue;
                double d;
                const unsigned key = dg_key(jq.v, jq.P, a.bj, o, ox, oy, jq.lo, jq.hi, &d);
                if (key != 0xffffffffu) dg_atomic_min_u32(jq.key, key);
            }
        }
        DG_SYNC();
        DG_PHASE(tid) { if (tid == 0) *cnt = 0; }  // (read again only after the next barrier of the caller or of the next tile)
    }
}

// selected obstacle of one trajectory -> dis_lat (the same operations as pass 2), pathid, obstacle index
DG_FN DgRes dg_selected(const DgView& v, int P, unsigned key, const double* ox, const double* oy, double lo, double hi) {
    DgRes r = dg_res_none();
    if (key == 0xffffffffu || P < 2) return r;
    const int jstar = (int)(key >> 16), ostar = (int)(key & 0xffffu);
    double d;
    dg_key(v, P, jstar, ostar, ox[ostar], oy[ostar], lo, hi, &d);
    r.found = 1; r.pathid = jstar; r.ob = ostar; r.dis_lat = d;
    return r;
}

// =============================================================================================================================
// one CTA = the scenes [first, first + S) of the batch
// =============================================================================================================================
template <int G, int TPB>
DG_BODY dg_group_cycle(const DgMap& m, const dp_params& p, const int first, const int S, const dp_scene_hdr* hdr, const double* obs_x,
                       const double* obs_y, const int max_obs, dp_carry* carry, double2* last_path, dp_plan_record* rec,
                       dp_trace_record* trace, double* path_xy, double* path_ll, const DpIo& io, DgSmem<G>& sm) {
    const double Vw = p.vehicle_width;
    DG_MARK(0);

    // ---- P0: headers and carry in with coalesced 16-byte loads; small map tables to shared memory
    DG_PHASE(tid) {
        const uint4* gh = reinterpret_cast<const uint4*>(hdr + first);
        const uint4* gc = reinterpret_cast<const uint4*>(carry + first);
        uint4* sh = reinterpret_cast<uint4*>(sm.hdr);
        uint4* sc = reinterpret_cast<uint4*>(sm.carry);
        for (int i = tid; i < S * 8; i += TPB) { sh[i] = gh[i]; sc[i] = gc[i]; }
#if !defined(DP_EMU)
        if (io.n_fwd) {                                     // deferred gather: last cycle's records of these scenes go out first
            const uint4* fs = reinterpret_cast<const uint4*>(io.fwd_src + first);
            for (int i = tid; i < S * 8; i += TPB) {
                const uint4 w = __ldcg(fs + i);
#pragma unroll
                for (int q = 0; q < DP_MAX_MIRRORS; ++q)
                    if (q < io.n_fwd) reinterpret_cast<uint4*>(io.fwd_dst[q] + first)[i] = w;
            }
        }
#endif
        if (trace) {
            uint32_t* w = reinterpret_cast<uint32_t*>(trace + first);
            for (int i = tid; i < S * (int)(sizeof(dp_trace_record) / 4); i += TPB) w[i] = 0;
        }
        const bool tab = (m.n_lanes + 1 <= DG_TABCAP) && (m.n_roads + 1 <= DG_TABCAP);
        if (tab) {
            for (int i = tid; i <= m.n_lanes; i += TPB) sm.lpo[i] = m.lane_pt_off[i];
            for (int i = tid; i <= m.n_roads; i += TPB) sm.rlb[i] = m.road_lane_base[i];
        }
        if (tid == 0) {
            sm.maxN = 0; sm.n_sweep = 0; sm.any_first = 0; sm.any_mean = 0; sm.any_junction = 0; sm.tab_ok = tab ? 1 : 0;
            sm.nsurv[0] = sm.nsurv[1] = 0;
        }
    }
    DG_SYNC();
    DG_MARK(1);
    const int* lpo = sm.tab_ok ? sm.lpo : m.lane_pt_off;
    const int* rlb = sm.tab_ok ? sm.rlb : m.road_lane_base;

    // ---- P1 (thread per scene): Nav_LaneChange (Decision.cpp:685-738), LoadRefPath as recipes (:553-673), junction path (:352-367, 438-452)
    DG_PHASE(tid) {
        if (tid >= S) continue;
        const int s = tid;
        const dp_scene_hdr& h = sm.hdr[s];
        DgCtl& c = sm.ctl[s];
        c.N = dg_imin((int)h.n_obs, max_obs); c.pos = h.pos; c.ub = 0; c.n_traj = 0; c.pts = 0;
        c.sweep_on = 0; c.sweep_cnt = 0; c.sweep_pick = -1; c.lane_n = h.lane_num; c.gl = 0; c.lane_sum = 0; c.side = 0; c.K = 0;
        c.rp_base0 = c.rp_n0 = c.rp_base1 = c.rp_n1 = 0; c.navi = 0; c.navi_t = 0; c.W = 0.0; c.lanechg = 0; c.id = 0;
        dg_atomic_max_i32(&sm.maxN, c.N);
        for (int r = 0; r <= DG_NREG; ++r) {
            DgPath& q = sm.path[s][r];
            q.d = 0.0; q.lo = -0.5 * Vw; q.hi = 0.5 * Vw; q.base0 = 0; q.stride0 = 1; q.n0 = 0; q.base1 = 0; q.n1 = 0; q.hb = 0.f;
            q.dmax = dg_inff(); q.key = 0xffffffffu; q.local = 0;
        }
        for (int u = 0; u < DG_NSWEEP; ++u) sm.swkey[s][u] = 0xffffffffu;
        if (c.pos == 0) {
            const int road = h.road_num, lane_n = h.lane_num;
            const int gl = rlb[road - 1] + lane_n - 1;
            const int lane_sum = rlb[road] - rlb[road - 1];
            const int off = lpo[gl], id_sum = lpo[gl + 1] - off;
            const int id = (int)(uint16_t)h.id[lane_n - 1];
            unsigned navi = 4, navi_t = 0;
            for (int i = 0; i < DP_LANESUM && h.out_lane_no[i] != 0; ++i)
                if (lane_n == h.out_lane_no[i]) { navi = 0; break; }
            int out_min = h.out_lane_no[0], out_max = 1;
            for (int i = 0; i < DP_LANESUM; ++i) if (h.out_lane_no[i] > out_max) out_max = h.out_lane_no[i];
            if (navi == 4) {
                int dirn = 0;
                if (lane_n < out_min) { navi = 2; dirn = 2; }
                else if (lane_n > out_max) { navi = 1; dirn = 1; }
                else navi = 0;
                if (dirn) {                                 // CalcNaviLaneChgTimes (Decision.cpp:498-538)
                    int times = 5;
                    for (int i = 0; i < DP_LANESUM && h.out_lane_no[i] != 0; ++i) {
                        const int t = (dirn == 1) ? lane_n - h.out_lane_no[i] : h.out_lane_no[i] - lane_n;
                        if (t < times) times = t;
                    }
                    navi_t = (unsigned)(times & 0xff);
                }
            }
            const int idc = dg_imin(id, id_sum - 1);
            const int lanechg = m.attr[off + idc];
            const double W = m.width[off + idc] / 100.0;
            DgPath& F = sm.path[s][0]; DgPath& R = sm.path[s][1]; DgPath& NF = sm.path[s][2]; DgPath& NR = sm.path[s][3];
            int ub = 0;
            dg_lane_slices(lpo, gl, id, p.id_more, F, R, ub);
            int side = 0, gn = gl;                          // gn: the lane the neighbour pair is read from
            double dn = 0.0;
            // at most ONE neighbour pair exists per cycle: left for attribute 1/3, right only for attribute 2 (the reference
            // never loads the right lane for 3, Decision.cpp:636)
            if (lanechg == 1 || lanechg == 3) {
                side = 1;
                if (lane_n > 1) {
                    const int idl = (int)(uint16_t)h.id[lane_n - 2];
                    const int nl = lpo[gl] - lpo[gl - 1];
                    if (idl > 0 && idl < nl) { dg_lane_slices(lpo, gl - 1, idl, p.id_more, NF, NR, ub); gn = gl - 1; }
                } else {
                    NF.base0 = F.base0; NF.stride0 = F.stride0; NF.n0 = F.n0; NR.base0 = R.base0; NR.stride0 = R.stride0; NR.n0 = R.n0;
                    dn = -1 * W;
                }
            } else if (lanechg == 2) {
                side = 2;
                if (lane_n < lane_sum) {
                    const int idr = (int)(uint16_t)h.id[lane_n];
                    const int nr = lpo[gl + 2] - lpo[gl + 1];
                    if (idr > 0 && idr < nr) { dg_lane_slices(lpo, gl + 1, idr, p.id_more, NF, NR, ub); gn = gl + 1; }
                } else {
                    NF.base0 = F.base0; NF.stride0 = F.stride0; NF.n0 = F.n0; NR.base0 = R.base0; NR.stride0 = R.stride0; NR.n0 = R.n0;
                    dn = W;
                }
            }
            // windows of AroundObstacle (Decision.cpp:811-842): F/R +-Vw/2, left pair [-Vw/2, +W/2], right pair [-W/2, +Vw/2]
            NF.lo = NR.lo = (side == 2) ? -0.5 * W : -0.5 * Vw;
            NF.hi = NR.hi = (side == 2) ? 0.5 * Vw : 0.5 * W;
            NF.d = NR.d = dn;
            dg_bounds(m, gl, 0.0, F.lo, F.hi, &F.hb, &F.dmax);
            R.hb = F.hb; R.dmax = F.dmax;
            dg_bounds(m, gn, dn, NF.lo, NF.hi, &NF.hb, &NF.dmax);
            NR.hb = NF.hb; NR.dmax = NF.dmax;
            c.gl = gl; c.lane_sum = lane_sum; c.id = id; c.side = side; c.lanechg = lanechg; c.W = W;
            c.navi = (int)navi; c.navi_t = (int)navi_t; c.ub = ub;
            int K = 0;
            while (K < DP_MAX_SWEEP && (double)K < (W - Vw) / 0.6) ++K;
            c.K = K;
        } else if (c.pos == 1 || c.pos == 2) {
            // junction reference path as two forward map runs: remaining approach lane + connector (PreStubDecision,
            // Decision.cpp:352-367) or remaining connector + first 60 points of the next lane (StubDecision, :438-452)
            const int gc = (h.conn >= 0 && h.conn < m.n_conn) ? m.conn[h.conn].lane : -1;
            const int coff = gc >= 0 ? lpo[gc] : 0, n_inter = gc >= 0 ? lpo[gc + 1] - coff : 0;
            const int gj = rlb[h.road_num - 1] + h.lane_num - 1;
            const int off = lpo[gj], n = lpo[gj + 1] - off;
            DgPath& F = sm.path[s][0];
            int g0, g1;
            if (c.pos == 1) {
                const int idj = (int)(uint16_t)h.id[h.lane_num - 1];
                F.base0 = off + idj; F.n0 = dg_imax(0, n - idj); F.base1 = coff; F.n1 = n_inter; g0 = gj; g1 = gc;
            } else {
                const int idj = (int)(uint16_t)h.id[h.last_lanenum - 1];
                F.base0 = coff + idj; F.n0 = dg_imax(0, n_inter - idj); F.base1 = off; F.n1 = dg_imin(60, n); g0 = gc; g1 = gj;
            }
            // bounds of the concatenation: both lanes and the joint segment between the two runs (its length, and how much
            // its direction differs from the segments before and after it)
            float hb = 1e-4f, hmin = 1e30f, delta = 0.f;
            if (g0 >= 0 && F.n0 > 1) { hb = fmaxf(hb, m.lane_hmax[g0]); hmin = fminf(hmin, m.lane_hmin[g0]); delta = fmaxf(delta, m.lane_dnmax[g0]); }
            if (g1 >= 0 && F.n1 > 1) { hb = fmaxf(hb, m.lane_hmax[g1]); hmin = fminf(hmin, m.lane_hmin[g1]); delta = fmaxf(delta, m.lane_dnmax[g1]); }
            if (F.n0 > 0 && F.n1 > 0) {
                const double2 a = m.xy[F.base0 + F.n0 - 1], b = m.xy[F.base1];
                const double jx = b.x - a.x, jy = b.y - a.y;
                const double jl = sqrt(dg_sq2(jx, jy));
                hb = fmaxf(hb, (float)jl * 1.0001f + 1e-4f);
                hmin = fminf(hmin, (float)jl * 0.9999f);
                if (jl > 0) {
                    const double nx = jy / jl, ny = -jx / jl;
                    if (F.n0 > 1) { const double2 q = m.nrm[F.base0 + F.n0 - 2]; delta = fmaxf(delta, (float)sqrt(dg_sq2(q.x - nx, q.y - ny)) * 1.0001f + 1e-6f); }
                    if (F.n1 > 1) { const double2 q = m.nrm[F.base1]; delta = fmaxf(delta, (float)sqrt(dg_sq2(q.x - nx, q.y - ny)) * 1.0001f + 1e-6f); }
                }
            }
            F.hb = hb + 1e-4f;
            F.dmax = dg_dmax(F.lo, F.hi, F.hb, delta, hmin);
            sm.any_junction = 1;
            c.rp_base0 = F.base0; c.rp_n0 = F.n0; c.rp_base1 = F.base1; c.rp_n1 = F.n1;
        }
    }
    DG_SYNC();
    DG_MARK(2);
    // ---- P2: AroundObstacle (Decision.cpp:759-881) / the junction search (:370, :455): every (scene, trajectory, obstacle) pair
    dg_scan_phase<G, TPB>(sm, S * DG_NREG, first, obs_x, obs_y, max_obs, [&](int jb) {
        const int s = jb / DG_NREG, r = jb & (DG_NREG - 1);
        DgPath& pa = sm.path[s][r];
        DgJob j;
        j.v = dg_view(m, pa, nullptr); j.lo = pa.lo; j.hi = pa.hi; j.key = &pa.key; j.P = pa.n0 + pa.n1; j.scene = s; j.hb = pa.hb; j.dmax = pa.dmax;
        j.tvx = nullptr; j.tvy = nullptr; j.tdth = nullptr; j.tT = 0;
        if (io.trk_vx && r == 0 && sm.ctl[s].pos != 0) {      // the junction search (Decision.cpp:370, :455) against the moving agents
            const size_t tb = (size_t)(first + s) * max_obs;
            j.tvx = io.trk_vx + tb; j.tvy = io.trk_vy + tb; j.tdth = io.trk_dth + tb; j.tT = io.trk_T;
        }
        return j;
    });
    DG_MARK(3);

    // ---- P3: SearchObstacle outputs of the lane regions.  3a: the arclength terms up to the selected point, all threads, into
    //      the scene's term pool (sm.plan is idle until the carried path is fetched); 3b: one thread per trajectory adds them up
    DG_PHASE(tid) {
        const int lane = tid & 31;
        for (int pr = tid >> 5; pr < S * DG_NREG; pr += TPB / 32) {        // one warp per trajectory: coalesced table reads
            const int s = pr / DG_NREG, r = pr & (DG_NREG - 1);
            const DgPath& pa = sm.path[s][r];
            if (pa.key == 0xffffffffu) continue;
            const bool seg = sm.ctl[s].pos == 0;                            // F: 0..119, R: 120..159, NF: 160..279, NR: 280..319
            const int tb = seg ? (r == 0 ? 0 : r == 1 ? 120 : r == 2 ? 160 : 280) : 0;     // (junction path: the whole pool)
            const int cap = seg ? ((r & 1) ? 40 : 120) : DG_POOL;
            const int nt = dg_imin((int)(pa.key >> 16), cap);
            const DgView v = dg_view(m, pa, nullptr);
            double* pool = reinterpret_cast<double*>(sm.plan[s]) + tb;
            for (int j = lane; j < nt; j += 32) pool[j] = dg_seg_fma(v, m.lenf, j);
        }
    }
    DG_SYNC();
    DG_PHASE(tid) {
        if (tid >= S * DG_NREG) continue;
        const int s = tid / DG_NREG, r = tid & (DG_NREG - 1);
        const DgPath& pa = sm.path[s][r];
        const int P = pa.n0 + pa.n1;
        const size_t ob = (size_t)(first + s) * max_obs;
        const DgView v = dg_view(m, pa, nullptr);
        DgRes res;
        if (io.trk_vx && r == 0 && sm.ctl[s].pos != 0 && pa.key != 0xffffffffu && P >= 2) {
            const int jstar = (int)(pa.key >> 16), ostar = (int)(pa.key & 0xffffu);
            const size_t q = ob + ostar;
            const double2 at = dg_track_pos(obs_x[q], obs_y[q], io.trk_vx[q], io.trk_vy[q], io.trk_dth[q], io.trk_T, jstar);
            double d;
            dg_key(v, P, jstar, ostar, at.x, at.y, pa.lo, pa.hi, &d);
            res = dg_res_none(); res.found = 1; res.pathid = jstar; res.ob = ostar; res.dis_lat = d;
        } else res = dg_selected(v, P, pa.key, obs_x + ob, obs_y + ob, pa.lo, pa.hi);
        if (res.found) {
            const bool seg = sm.ctl[s].pos == 0;
            const int tb = seg ? (r == 0 ? 0 : r == 1 ? 120 : r == 2 ? 160 : 280) : 0;
            const int cap = seg ? ((r & 1) ? 40 : 120) : DG_POOL;
            res.dis_lng = dg_seq_sum(reinterpret_cast<const double*>(sm.plan[s]) + tb, res.pathid, cap, -1.0,
                                     [&](int j) { return dg_seg_fma(v, m.lenf, j); });
        }
        sm.res[s][r] = res;
    }
    DG_SYNC();
    DG_MARK(4);

    // ---- P4 (thread per scene): BehaviorDecision (Decision.cpp:898-1773) up to the avoid sweep; junction speed rule (:373-392)
    DG_PHASE(tid) {
        if (tid >= S) continue;
        const int s = tid;
        const dp_scene_hdr& h = sm.hdr[s];
        DgCtl& k = sm.ctl[s];
        dp_carry& c = sm.carry[s];
        dp_plan_record& out = sm.rec[s];
        dp_trace_record* tr = trace ? trace + first + s : nullptr;
        {   // zero the record (fields are stored as they become final)
            uint32_t* w = reinterpret_cast<uint32_t*>(&out);
            for (int i = 0; i < 32; ++i) w[i] = 0;
        }
        const int pos = k.pos;
        if (pos == 0) {
            const int lane_n = k.lane_n, lane_sum = k.lane_sum, lanechg = k.lanechg, side = k.side, gl = k.gl, id = k.id;
            const double W = k.W;
            const int nslot = (side == 2) ? 4 : 2;
            double gF = 0.0, gNF = 0.0, gNR = 0.0;          // gaps stay 0 (memset state) for paths that are not evaluated
            for (int r = 0; r < DG_NREG; ++r) {
                const int Pr = sm.path[s][r].n0;
                if (Pr != 0) {
                    const DgRes& sr = sm.res[s][r];
                    ++k.n_traj; k.pts += Pr;
                    if (tr) dg_put_slot(&tr->region[r < 2 ? r : nslot + r - 2], sr, 1);
                    if (r == 0) gF = sr.dis_lng; else if (r == 2) gNF = sr.dis_lng; else if (r == 3) gNR = sr.dis_lng;
                }
            }
            const double gLF = (side == 1) ? gNF : 0.0, gLR = (side == 1) ? gNR : 0.0;
            const double gRF = (side == 2) ? gNF : 0.0, gRR = (side == 2) ? gNR : 0.0;
            if (tr) { tr->width_curlane = W; tr->navi_lanechg = (uint32_t)k.navi; tr->navi_lanechg_times = (uint32_t)k.navi_t; }
            const int navi = k.navi;
            int cur_behavior = c.behavior, cur_target = c.target_lanenum, cur_light = c.light_status;
            bool cur_lanechg = c.lanechg_status != 0, cur_obsavoid = c.obsavoid_status != 0;
            int cur_dlg = c.behavior_to_dlg;
            const int his_behavior = c.his_behavior, his_target = c.his_target_lanenum, his_light = c.his_light_status;
            int lane_cur = lane_n;
            int z_light = c.light_status;
            const double period = h.period_ms;
            const int off = lpo[gl], id_sum = lpo[gl + 1] - off;
#define DG_KEEP(reset) do { cur_behavior = 1; cur_target = lane_cur; if (reset) cur_lanechg = false; } while (0)
#define DG_TICK do { c.leftlight_time += period; if (c.leftlight_time > 2000) c.leftlight_time = 2000; } while (0)
            if (lanechg == 0) {                             // :920-1010
                if (gF < 15) {
                    c.no_obsavoid_time = 0;
                    c.obsavoid_time++;
                    if (c.obsavoid_time > 2) {
                        // in-lane avoid sweep (Decision.cpp:940-974): scored by the next two phases, resolved in P6
                        k.sweep_on = 1;
                        k.sweep_cnt = (k.K >= 1) ? 2 * (k.K - 1) : 0;
                        if (k.sweep_cnt > 0) sm.sweep_list[dg_atomic_add_i32(&sm.n_sweep, 1)] = s;
                    } else { cur_behavior = 1; cur_target = lane_cur; cur_light = 0; cur_dlg = 1; }
                } else {
                    if (c.obsavoid_status == 0) { cur_behavior = 1; cur_target = lane_cur; cur_light = 0; cur_dlg = 1; }
                    else {
                        c.no_obsavoid_time++;
                        if (c.no_obsavoid_time > 3) { cur_behavior = 1; cur_target = lane_cur; cur_light = 0; cur_dlg = 1; cur_obsavoid = false; }
                    }
                    cur_dlg = 1;
                }
            } else {                                        // :1012-1772
                c.no_obsavoid_time = 0;
                c.obsavoid_time = 0;
                if (!cur_lanechg) {
                    if (navi != 0) {                        // :1021-1144
                        if (navi == 1) {
                            if (lanechg == 1 || lanechg == 3) {
                                cur_dlg = 2;
                                if (cur_light != 1) { cur_light = 1; c.leftlight_time = 0; }
                                c.leftlight_time += period;
                                if (((gLF > gF + 10) || (gLF > 40)) && gLR > 15 && c.leftlight_time > 2000) {
                                    cur_behavior = 2; cur_target = lane_cur - 1; cur_lanechg = true;
                                } else DG_KEEP(true);
                            } else { DG_KEEP(true); cur_dlg = 4; }
                        } else if (navi == 2) {
                            if (lanechg == 2 || lanechg == 3) {
                                cur_dlg = 3;
                                if (cur_light != 2) { cur_lanechg = true; c.rightlight_time = 0; }   // sic: lanechg_status = 2 (:1094)
                                c.rightlight_time += period;
                                if (((gRF > gF + 10) || (gRF > 40)) && gRR > 15 && c.rightlight_time >= 2000) {
                                    cur_behavior = 3; cur_target = lane_cur + 1; cur_lanechg = true;
                                } else DG_KEEP(true);
                            } else { DG_KEEP(true); cur_dlg = 4; }
                        }
                    } else {                                // :1146-1757
                        if (gF < (2 * 10 + 5)) {
                            c.frontobs_time++;
                            if (c.frontobs_time > 2) {
                                c.frontobs_time = 3;
                                bool has_m1 = false, has_p1 = false;    // exit-lane list contains lane-1 / lane+1
                                for (int i = 0; i < DP_LANESUM && h.out_lane_no[i] != 0; ++i) {
                                    if (h.out_lane_no[i] == lane_cur - 1) has_m1 = true;
                                    if (h.out_lane_no[i] == lane_cur + 1) has_p1 = true;
                                }
                                if (lanechg == 1) {         // :1157-1294
                                    if (lane_cur > 1) {
                                        cur_dlg = 5;
                                        const bool no_back = !has_m1;
                                        bool chg = false;
                                        if (no_back) {
                                            if (dg_run_exceeds(m, gl, off, id_sum, id, 0, 60.0)) {
                                                chg = true;
                                                if (z_light != 1) { z_light = 1; c.leftlight_time = 0; }
                                                c.leftlight_time += period;
                                                if (c.leftlight_time > 2000) c.leftlight_time = 2000;
                                            } else z_light = 0;
                                        } else {
                                            if (dg_run_exceeds(m, gl, off, id_sum, id, 1, 15.0)) {
                                                chg = true;
                                                if (cur_light != 1) { cur_light = 1; c.leftlight_time = 0; }
                                                c.leftlight_time += period;
                                                if (c.leftlight_time > 2000) c.leftlight_time = 2100;
                                            } else cur_light = 0;
                                        }
                                        if (chg && gLF > gF + 10 && gLR > 10 && c.leftlight_time > 1500) {
                                            c.frontobs_time = 0; cur_behavior = 2; cur_target = lane_cur - 1; cur_lanechg = true;
                                        } else DG_KEEP(true);
                                    } else DG_KEEP(true);
                                } else if (lanechg == 2) {  // :1296-1424
                                    if (lane_cur < lane_sum) {
                                        cur_dlg = 6;
                                        const bool no_back = !has_m1;                     // sic (:1307)
                                        bool chg = false;
                                        if (dg_run_exceeds(m, gl, off, id_sum, id, 1, no_back ? 50.0 : 10.0)) {
                                            chg = true;
                                            const int want = no_back ? 2 : 1;
                                            if (cur_light != want) { cur_light = want; c.leftlight_time = 0; }
                                            c.leftlight_time += period;
                                            if (c.leftlight_time > 2000) c.leftlight_time = 2000;
                                        }
                                        if (chg && gRF > gF + 10 && gRR > 10 && c.leftlight_time > 1500) {
                                            c.frontobs_time = 0; cur_behavior = 3; cur_target = lane_cur + 1; cur_lanechg = true;
                                        } else DG_KEEP(true);
                                    } else DG_KEEP(true);
                                } else if (lanechg == 3) {  // :1426-1738
                                    const bool nb_left = !has_m1, nb_right = !has_p1;
                                    bool left_ok = false, right_ok = false;
                                    if (lane_cur > 1) left_ok = dg_run_exceeds(m, gl, off, id_sum, id, nb_left ? 1 : 2, nb_left ? 50.0 : 10.0);
                                    if (lane_cur < lane_sum) right_ok = dg_run_exceeds(m, gl, off, id_sum, id, 1, nb_right ? 50.0 : 10.0);
                                    if (left_ok && !nb_left) {                          // :1545-1594
                                        if (!cur_lanechg) { cur_light = 1; c.leftlight_time = 0; }
                                        DG_TICK;
                                        if (gLF > gF + 10 && gLR > 10 && c.leftlight_time > 2000) {
                                            c.frontobs_time = 0; cur_behavior = 2; cur_target = lane_cur - 1; cur_lanechg = true;
                                        } else DG_KEEP(true);
                                    } else if (right_ok && !nb_right) {                 // :1596-1636
                                        if (cur_light != 2) { cur_light = 2; c.leftlight_time = 0; }
                                        DG_TICK;
                                        if (gRF > gF + 10) {
                                            if (gRR > 10 && c.leftlight_time > 2000) {
                                                c.frontobs_time = 0; cur_behavior = 3; cur_target = lane_cur + 1; cur_lanechg = true;
                                            } else DG_KEEP(false);
                                        }
                                    } else if (left_ok) {                               // :1638-1686
                                        if (cur_light != 1) { cur_lanechg = true; c.leftlight_time = 0; }   // sic (:1642)
                                        DG_TICK;
                                        if (gLF > gF + 10 && gLR > 10 && c.leftlight_time > 2000) {
                                            c.frontobs_time = 0; cur_behavior = 2; cur_target = lane_cur - 1; cur_lanechg = true;
                                        } else DG_KEEP(false);
                                    } else if (right_ok) {                              // :1688-1730
                                        if (cur_light != 2) { cur_light = 2; c.leftlight_time = 0; }
                                        DG_TICK;
                                        if (gRF > gF + 10) {
                                            if (gRR > 10 && c.leftlight_time > 2000) {
                                                c.frontobs_time = 0; cur_behavior = 3; lane_cur = 1; cur_target = 1; cur_lanechg = true;   // sic (:1712)
                                            } else DG_KEEP(false);
                                        }
                                    } else DG_KEEP(true);
                                }
                            } else DG_KEEP(true);           // :1741-1746
                        } else { c.frontobs_time = 0; cur_dlg = 8; DG_KEEP(true); }
                    }
                } else {                                    // lane change in progress, :1760-1771
                    cur_dlg = 9;
                    if (cur_target == lane_cur) { cur_lanechg = false; cur_light = 0; }
                    cur_behavior = his_behavior; cur_target = his_target; cur_light = his_light;
                }
            }
#undef DG_KEEP
#undef DG_TICK
            (void)z_light;
            k.beh = cur_behavior; k.target = cur_target; k.light = cur_light; k.lanechg_st = cur_lanechg ? 1 : 0;
            k.obsavoid = cur_obsavoid ? 1 : 0; k.dlg = cur_dlg;
        } else if (pos == 1 || pos == 2) {
            // =================== PreStubDecision / StubDecision (Decision.cpp:323-486) ===================
            const DgRes& sr = sm.res[s][0];
            ++k.n_traj; k.pts += k.rp_n0 + k.rp_n1;
            if (tr) dg_put_slot(&tr->junction, sr, 1);
            double v_exp; int dlg;
            if (sr.dis_lng < 13) {
                const double v = sr.dis_lng - 3;
                v_exp = v > 0 ? v : 0;
                dlg = 13;
            } else { v_exp = 10; dlg = 1; }
            const int light = (h.stub_attribute == 3) ? 1 : h.stub_attribute;
            k.d_behavior = 1; k.d_target = h.lane_num; k.v_exp = v_exp;
            // members the junction functions write (:394-399) + thread-loop tail (:187-201)
            c.velocity_expect = v_exp; c.behavior_to_dlg = (uint16_t)dlg; c.light_status = (uint16_t)light;
            c.behavior = 1; c.target_roadnum = h.road_num; c.target_lanenum = h.lane_num;
            c.his_behavior = 1; c.his_light_status = (uint16_t)light; c.his_target_lanenum = h.lane_num;
            out.velocity_expect = v_exp; out.behavior = 1; out.target_roadnum = h.road_num; out.target_lanenum = h.lane_num;
            out.light = (uint16_t)light; out.behavior_to_dlg = (uint16_t)dlg; out.sweep_index = -1;
        } else {
            // no decision function runs for other pos values (Decision.cpp:183): members keep their values
            k.d_behavior = c.behavior; k.d_target = c.target_lanenum; k.v_exp = c.velocity_expect;
            c.his_behavior = c.behavior; c.his_light_status = c.light_status; c.his_target_lanenum = c.target_lanenum;
            out.velocity_expect = c.velocity_expect; out.behavior = c.behavior; out.target_roadnum = c.target_roadnum;
            out.target_lanenum = c.target_lanenum; out.light = c.light_status; out.behavior_to_dlg = c.behavior_to_dlg;
            out.sweep_index = -1;
        }
    }
    DG_SYNC();
    DG_MARK(5);

    // ---- P5: the shifted avoid candidates of the armed scenes (Decision.cpp:940-974), all at once
    if (sm.n_sweep > 0) {
        dg_scan_phase<G, TPB>(sm, sm.n_sweep * DG_NSWEEP, first, obs_x, obs_y, max_obs, [&](int jb) {
            const int u = jb % DG_NSWEEP, s = sm.sweep_list[jb / DG_NSWEEP];
            const DgCtl& k = sm.ctl[s];
            DgPath pa = sm.path[s][0];
            DgJob j;
            j.scene = s; j.lo = -0.5 * Vw; j.hi = 0.5 * Vw; j.key = &sm.swkey[s][u];
            j.tvx = nullptr; j.tvy = nullptr; j.tdth = nullptr; j.tT = 0;
            if (u >= k.sweep_cnt) { j.P = 0; j.hb = 0.f; j.dmax = 0.f; j.v = dg_view(m, pa, nullptr); return j; }
            pa.d = dg_sweep_offset(dg_sweep_g(u, k.K), k.K);
            j.v = dg_view(m, pa, nullptr); j.P = pa.n0;
            dg_bounds(m, k.gl, pa.d, j.lo, j.hi, &j.hb, &j.dmax);
            return j;
        });
        DG_MARK(6);
        // 5b: arclength terms of the selected candidates into the scene's term pool (pool / candidates terms each), then one
        // thread per candidate adds them up -- only as far as the `dis_lng > 25` decision needs unless a trace is written
        DG_PHASE(tid) {
            for (int it = tid; it < sm.n_sweep * DG_POOL; it += TPB) {
                const int s = sm.sweep_list[it / DG_POOL], t = it % DG_POOL;
                const DgCtl& k = sm.ctl[s];
                const int cap = DG_POOL / k.sweep_cnt, u = t / cap, j = t - u * cap;
                if (u >= k.sweep_cnt) continue;
                const unsigned key = sm.swkey[s][u];
                if (key == 0xffffffffu || j >= (int)(key >> 16)) continue;
                DgPath pa = sm.path[s][0];
                pa.d = dg_sweep_offset(dg_sweep_g(u, k.K), k.K);
                reinterpret_cast<double*>(sm.plan[s])[t] = dg_seg_fma(dg_view(m, pa, nullptr), nullptr, j);
            }
        }
        DG_SYNC();
        DG_PHASE(tid) {
            if (tid >= sm.n_sweep * DG_NSWEEP) continue;
            const int u = tid % DG_NSWEEP, s = sm.sweep_list[tid / DG_NSWEEP];
            const DgCtl& k = sm.ctl[s];
            if (u >= k.sweep_cnt) continue;
            DgPath pa = sm.path[s][0];
            pa.d = dg_sweep_offset(dg_sweep_g(u, k.K), k.K);
            const size_t ob = (size_t)(first + s) * max_obs;
            const DgView v = dg_view(m, pa, nullptr);
            DgRes res = dg_selected(v, pa.n0, sm.swkey[s][u], obs_x + ob, obs_y + ob, -0.5 * Vw, 0.5 * Vw);
            if (res.found) {
                const int cap = DG_POOL / k.sweep_cnt;
                res.dis_lng = dg_seq_sum(reinterpret_cast<const double*>(sm.plan[s]) + u * cap, res.pathid, cap, trace ? -1.0 : 25.0,
                                         [&](int j) { return dg_seg_fma(v, nullptr, j); });
            }
            sm.res[s][DG_NREG + u] = res;
        }
        DG_SYNC();
        DG_MARK(7);
    }

    // ---- P6 (thread per scene): first feasible candidate, SpeedDecision / RefPath / write-back (Decision.cpp:940-974, 1781-1816,
    //      307-313, 187-201); Calculate_aim_dis (Planning.cpp:242-290) and the recipe of the SearchAimPoint walk (:303-583)
    DG_PHASE(tid) {
        if (tid == 0) {                                     // the term pool is dead: fetch the carried paths (Planning.cpp:6) into sm.plan
#if defined(DP_EMU)
            for (int q = 0; q < S; ++q) std::memcpy(sm.plan[q], last_path + (size_t)(first + q) * DP_PATH_POINTS, DP_PATH_POINTS * sizeof(double2));
#else
            dg_mbar_init(&sm.mbar, (uint32_t)S * DP_PATH_POINTS * (uint32_t)sizeof(double2));
            for (int q = 0; q < S; ++q)
                dg_bulk_load(sm.plan[q], last_path + (size_t)(first + q) * DP_PATH_POINTS, DP_PATH_POINTS * (uint32_t)sizeof(double2), &sm.mbar);
#endif
        }
        if (tid >= S) continue;
        const int s = tid;
        const dp_scene_hdr& h = sm.hdr[s];
        DgCtl& k = sm.ctl[s];
        dp_carry& c = sm.carry[s];
        dp_plan_record& out = sm.rec[s];
        dp_trace_record* tr = trace ? trace + first + s : nullptr;
        const int pos = k.pos;
        if (pos == 0) {
            int cur_behavior = k.beh, cur_target = k.target, cur_light = k.light, cur_dlg = k.dlg;
            bool cur_obsavoid = k.obsavoid != 0;
            int sweep_pick = -1;
            if (k.sweep_on) {
                const int K = k.K, total = 2 * K;
                const int FP = sm.path[s][0].n0;
                int first_u = -1;
                for (int u = 0; u < k.sweep_cnt; ++u) {
                    DgRes r = sm.res[s][DG_NREG + u];
                    if (FP < 2) { r.found = 0; r.dis_lat = DP_NOT_FOUND; r.dis_lng = DP_NOT_FOUND; r.ob = -1; r.pathid = 0; }
                    const int g = dg_sweep_g(u, K);
                    if (tr) dg_put_slot(&tr->sweep[(g / K) * DP_MAX_SWEEP + (g % K)], r, first_u < 0 ? 1 : 2);
                    if (first_u < 0 && r.dis_lng > 25) { first_u = u; sweep_pick = g; }
                    if (first_u >= 0 && !tr) break;
                }
                const int scored = sweep_pick < 0 ? total : sweep_pick + 1;        // what the reference evaluates
                k.n_traj += scored; k.pts += scored * FP;
                if (tr && total > 0) {                                          // L0 and R0: copies of the F region slot
                    dp_search_slot s0 = tr->region[0];
                    s0.evaluated = 1; tr->sweep[0] = s0;
                    s0.evaluated = (uint8_t)(K < scored ? 1 : 2); tr->sweep[DP_MAX_SWEEP] = s0;
                }
                if (sweep_pick >= 0) {
                    const int sd = sweep_pick / K;
                    cur_behavior = sd == 0 ? 4 : 5; cur_target = k.lane_n; cur_light = sd == 0 ? 1 : 2;
                    cur_obsavoid = true; cur_dlg = sd == 0 ? 11 : 12;
                }
            }
            const double v_exp = (cur_behavior == 4 || cur_behavior == 5) ? 5 : 10;
            const int nNF = sm.path[s][2].n0;
            k.rp_n0 = (cur_behavior == 2) ? (k.side == 1 ? nNF : 0) : (cur_behavior == 3) ? (k.side == 2 ? nNF : 0) : sm.path[s][0].n0;
            k.rp_n1 = 0;
            k.d_behavior = cur_behavior; k.d_target = cur_target; k.v_exp = v_exp;
            c.velocity_expect = v_exp;
            c.behavior = (uint16_t)cur_behavior; c.target_roadnum = h.road_num; c.target_lanenum = (uint16_t)cur_target;
            c.light_status = (uint16_t)cur_light; c.behavior_to_dlg = (uint16_t)cur_dlg;
            c.his_behavior = (uint16_t)cur_behavior; c.his_target_lanenum = (uint16_t)cur_target; c.his_light_status = (uint16_t)cur_light;
            c.lanechg_status = (uint8_t)k.lanechg_st; c.obsavoid_status = cur_obsavoid ? 1 : 0;
            out.velocity_expect = v_exp;
            out.behavior = (uint16_t)cur_behavior; out.target_roadnum = h.road_num; out.target_lanenum = (uint16_t)cur_target;
            out.light = (uint16_t)cur_light; out.behavior_to_dlg = (uint16_t)cur_dlg; out.sweep_index = (int16_t)sweep_pick;
        }
        if (tr) tr->refpath_len = (uint16_t)(k.rp_n0 + k.rp_n1);

        // ================================ Planning thread iteration ================================
        float faraim = 0.f;                                 // FLOAT faraim_dis (Planning.cpp:242-290)
        if (pos == 0) {
            faraim = (float)((h.velocity / 3.6) * 5 + 4);
            if (faraim > p.road_faraim_max) faraim = (float)p.road_faraim_max;
            else if (faraim < p.road_faraim_min) faraim = (float)p.road_faraim_min;
        } else if (pos == 1) faraim = (float)p.pre_inter_faraim;
        else if (pos == 2) faraim = (float)p.inter_faraim;
        k.faraim = faraim;
        if (tr) tr->faraim_dis = faraim;
        k.first = (c.plan_count == 0) ? 1 : 0;
        if (k.first) sm.any_first = 1;
        k.walk_kind = 0; k.woff = 0; k.wgl = 0; k.wfrom = 0; k.wto = 0; k.fb_off = 0; k.fb_idx = 0; k.fb_n = 0; k.fb_id = 0;
        if (pos == 0) {
            const int gl = k.gl, lane_n = k.lane_n, lane_sum = k.lane_sum;
            const int d_behavior = k.d_behavior, d_target = k.d_target;
            const int cur_id = h.id[lane_n - 1], cur_sum = lpo[gl + 1] - lpo[gl];
            int left_id = 0, left_sum = 0, right_id = 0, right_sum = 0;
            if (lane_n > 1) { left_id = h.id[lane_n - 2]; left_sum = lpo[gl] - lpo[gl - 1]; }
            if (lane_n < lane_sum) { right_id = h.id[lane_n]; right_sum = lpo[gl + 2] - lpo[gl + 1]; }
            int wl = -1, wfrom = 0, wto = 0, fb_gl = gl, fb_idx = 0, fb_id = 0;   // lane to walk, fallback point
            if (d_target == lane_n) {
                if (d_behavior == 1) { wl = gl; wfrom = cur_id; wto = cur_sum - 1; fb_gl = gl; fb_idx = cur_sum - 1; fb_id = cur_sum - 1; }
            } else {
                if (d_behavior == 2) {
                    if (lane_n > 1) { wl = gl - 1; wfrom = left_id; wto = left_sum - 1; fb_gl = gl; fb_idx = left_sum - 2; fb_id = left_sum - 1; }
                } else if (d_behavior == 3) {
                    if (lane_n < lane_sum) { wl = gl + 1; wfrom = right_id; wto = left_sum - 1; fb_gl = gl + 1; fb_idx = right_sum - 1; fb_id = right_sum - 1; }
                    else if (right_id < left_sum - 1) ++k.ub;
                }
            }
            if (wl >= 0 && wfrom < wto) {
                const int woff = lpo[wl], wn = lpo[wl + 1] - woff;
                bool walk = true;
                if (wfrom < 0) { ++k.ub; walk = false; }
                if (wto > wn - 1) { ++k.ub; wto = wn - 1; if (wfrom >= wto) walk = false; }
                if (walk) {
                    k.walk_kind = 1; k.woff = woff; k.wgl = wl; k.wfrom = wfrom; k.wto = wto;
                    k.fb_off = lpo[fb_gl]; k.fb_n = lpo[fb_gl + 1] - lpo[fb_gl]; k.fb_idx = fb_idx; k.fb_id = fb_id;
                }
            }
        } else if (pos == 1 || pos == 2) {
            if (k.rp_n0 + k.rp_n1 - 1 > 0) k.walk_kind = 2;
        }
        k.walk_hit = -1; k.walk_exact = 0;
        if (k.walk_kind == 1) {
            // "first point whose accumulated arclength - 4 exceeds faraim" (Planning.cpp:410-432) asked of the prefix table:
            // cump[from + j + 1] - cump[from] equals the reference's running sum up to the rounding bound lane_cerr (0 for lanes
            // whose sums are exact).  Terms lie in [hmin, hmax], so the first hit sits in a small index window: binary search
            // there; if the decision at the hit or before it falls inside the rounding bracket, the reference's own loop decides.
            const int cnt = k.wto - k.wfrom;
            int hit = -1;
            const double far = (double)faraim;
            const double* cp = m.cump + k.woff + k.wfrom;
            const double c0 = cp[0], ce = m.lane_cerr[k.wgl], err = ce > 0.0 ? ce + 1e-9 : 0.0;
            const double tgt = far + 4.0;
            const float hmx = m.lane_hmax[k.wgl], hmn = m.lane_hmin[k.wgl];
            int lo = (int)((float)tgt / hmx) - 2, hi = (hmn > 1e-6f) ? (int)((float)tgt / hmn) + 3 : cnt - 1;
            if (lo < 0) lo = 0;
            if (hi > cnt - 1) hi = cnt - 1;
            // invariant: no hit at j < lo (j terms of at most hmax stay below the target); first j in [lo, hi] with a definite hit
            int first_def = hi + 1;
            {
                int a = lo, b = hi;
                while (a <= b) {
                    const int mid = (a + b) >> 1;
                    if ((cp[mid + 1] - c0) - 4.0 > far + err) { first_def = mid; b = mid - 1; } else a = mid + 1;
                }
            }
            bool exact_loop = false;
            if (first_def <= hi) {
                hit = k.wfrom + first_def;
                if (err > 0.0 && first_def > 0 && (cp[first_def] - c0) - 4.0 >= far - err) exact_loop = true;   // the point before it is inside the bracket
            } else if (hi < cnt - 1) exact_loop = true;     // (cannot happen with valid bounds; never guess)
            else if (err > 0.0 && cnt > 0 && (cp[cnt] - c0) - 4.0 >= far - err) exact_loop = true;
            k.walk_hit = hit; k.walk_exact = exact_loop ? 1 : 0;
        }
    }
    DG_SYNC();
    DG_MARK(8);

    // ---- P7: nearest-of-200 partials on the carried path; arclength terms of a junction reference path (it has no prefix table)
#if !defined(DP_EMU)
    dg_mbar_wait(&sm.mbar);
#endif
    DG_PHASE(tid) {
        {
            const int lane = tid & 31;
            for (int s = tid >> 5; s < S; s += TPB / 32) {  // walks the table could not decide: their terms, coalesced
                const DgCtl& k = sm.ctl[s];
                if (k.walk_kind != 1 || !k.walk_exact) continue;
                const int nt = dg_imin(k.wto - k.wfrom, DG_SCR);
                for (int j = lane; j < nt; j += 32) sm.scr[s][j] = m.lenp[k.woff + k.wfrom + j];
            }
        }
        if (sm.any_junction) {
            for (int it = tid; it < S * DG_SCR; it += TPB) {
                const int s = it / DG_SCR, j = it - s * DG_SCR;
                const DgCtl& k = sm.ctl[s];
                if (k.walk_kind == 2 && j < k.rp_n0 + k.rp_n1 - 1) {
                    const DgView v = dg_view(m, sm.path[s][0], nullptr);
                    const double2 a = dg_pt(v, j), b = dg_pt(v, j + 1);
                    sm.scr[s][j] = dg_dist_plain(a.x, a.y, b.x, b.y);
                }
            }
        }
        if (tid < S * DG_NQ) {
            const int s = tid / DG_NQ, q = tid - s * DG_NQ;
            if (!sm.ctl[s].first)
                dg_nearest_part(sm.plan[s], q * (DP_PATH_POINTS / DG_NQ), (q + 1) * (DP_PATH_POINTS / DG_NQ), sm.hdr[s].x, sm.hdr[s].y,
                                &sm.ne[s][q], &sm.ni[s][q], &sm.namb[s][q]);
        }
    }
    DG_SYNC();
    DG_MARK(9);

    // ---- P8 (thread per scene): SearchAimPoint (Planning.cpp:303-583); control points of InitialPlanning on a first cycle (:124-128)
    DG_PHASE(tid) {
        if (tid >= S) continue;
        const int s = tid;
        const dp_scene_hdr& h = sm.hdr[s];
        DgCtl& k = sm.ctl[s];
        dp_carry& c = sm.carry[s];
        double aim_x = c.aim_x, aim_y = c.aim_y, aim_dir = c.aim_dir;
        int aim_id = c.aim_id;
        const double far = (double)k.faraim;
        if (k.walk_kind == 1) {
            int hit = k.walk_hit;
            if (k.walk_exact) {                             // inside the rounding bracket: the reference's loop on the staged terms
                const int j = dg_first_hit(sm.scr[s], k.wto - k.wfrom, DG_SCR, far, [&](int q) { return m.lenp[k.woff + k.wfrom + q]; });
                hit = j >= 0 ? k.wfrom + j : -1;
            }
            if (hit >= 0) {
                aim_x = m.x[k.woff + hit]; aim_y = m.y[k.woff + hit]; aim_dir = m.dir[k.woff + hit]; aim_id = hit;
            } else {
                int fi = k.fb_idx;
                if (fi < 0 || fi >= k.fb_n) { ++k.ub; fi = fi < 0 ? 0 : k.fb_n - 1; }
                aim_x = m.x[k.fb_off + fi]; aim_y = m.y[k.fb_off + fi]; aim_dir = m.dir[k.fb_off + fi]; aim_id = k.fb_id;
            }
        } else if (k.walk_kind == 2) {
            const DgView rv = dg_view(m, sm.path[s][0], nullptr);
            const int n = k.rp_n0 + k.rp_n1;
            const int hit = dg_first_hit(sm.scr[s], n - 1, DG_SCR, far, [&](int q) {
                const double2 a = dg_pt(rv, q), b = dg_pt(rv, q + 1);
                return dg_dist_plain(a.x, a.y, b.x, b.y);
            });
            if (hit >= 0) {
                const double2 a = dg_pt(rv, hit);
                aim_x = a.x; aim_y = a.y;
                if ((size_t)hit < (size_t)n - 4) {
                    const double2 b = dg_pt(rv, hit + 2);
                    aim_dir = dg_heading(a.x, a.y, b.x, b.y, p.epsilon, p.pi);
                } else {
                    int ia = hit - 2; if (ia < 0) { ++k.ub; ia = 0; }
                    const double2 b = dg_pt(rv, ia);
                    aim_dir = dg_heading(b.x, b.y, a.x, a.y, p.epsilon, p.pi);
                }
                aim_id = hit;
            } else {
                int ia = n - 3; if (ia < 0) { ++k.ub; ia = 0; }
                const double2 e = dg_pt(rv, n - 1), b = dg_pt(rv, ia);
                aim_x = e.x; aim_y = e.y;
                aim_dir = dg_heading(b.x, b.y, e.x, e.y, p.epsilon, p.pi);
                aim_id = n - 1;
            }
        }
        k.bx3 = aim_x; k.by3 = aim_y;
        // carried values are read by the planning phases below; the history update is stored in P11
        c.aim_x = aim_x; c.aim_y = aim_y; c.aim_dir = aim_dir; c.aim_id = aim_id;
        k.plan_dirty = 0;
        if (k.first) {                                      // CShare::BezierPlanning control points (oracle/cshare_spec.h)
            const double ex = aim_x - h.x, ey = aim_y - h.y;
            const double L = sqrt(dg_sq2(ex, ey)) / 3.0;
            double c0, s0, c3, s3;
            dg_sincos_deg(h.dir, &c0, &s0);
            dg_sincos_deg(aim_dir, &c3, &s3);
            k.bx0 = h.x; k.by0 = h.y;
            k.bx1 = fma(L, c0, h.x); k.by1 = fma(L, s0, h.y);
            k.bx2 = fma(-L, c3, aim_x); k.by2 = fma(-L, s3, aim_y);
            k.plan_dirty = 1;
        }
    }
    DG_SYNC();
    DG_MARK(10);

    // ---- P8b/c: first cycle of a scene: InitialPlanning runs BEFORE GetVhclLocalState (Planning.cpp:124-131)
    if (sm.any_first) {
        DG_PHASE(tid) {
            for (int it = tid; it < S * DP_PATH_POINTS; it += TPB) {
                const int s = it / DP_PATH_POINTS, i = it - s * DP_PATH_POINTS;
                const DgCtl& k = sm.ctl[s];
                if (!k.first) continue;
                const double t = (double)i / (double)(DP_PATH_POINTS - 1);
                const double u = 1.0 - t;
                const double b0 = u * u * u;
                const double b1 = 3.0 * (u * u) * t;
                const double b2 = 3.0 * u * (t * t);
                const double b3 = t * t * t;
                sm.plan[s][i] = make_double2(fma(b3, k.bx3, fma(b2, k.bx2, fma(b1, k.bx1, b0 * k.bx0))),
                                             fma(b3, k.by3, fma(b2, k.by2, fma(b1, k.by1, b0 * k.by0))));
            }
        }
        DG_SYNC();
    DG_MARK(11);
        DG_PHASE(tid) {
            if (tid < S * DG_NQ) {
                const int s = tid / DG_NQ, q = tid - s * DG_NQ;
                if (sm.ctl[s].first)
                    dg_nearest_part(sm.plan[s], q * (DP_PATH_POINTS / DG_NQ), (q + 1) * (DP_PATH_POINTS / DG_NQ), sm.hdr[s].x, sm.hdr[s].y,
                                    &sm.ne[s][q], &sm.ni[s][q], &sm.namb[s][q]);
            }
        }
        DG_SYNC();
    DG_MARK(12);
    }

    // ---- P9 (thread per scene): GetVhclLocalState part 1 (Planning.cpp:623-660): nearest point, lateral and heading error
    DG_PHASE(tid) {
        if (tid >= S) continue;
        const int s = tid;
        const dp_scene_hdr& h = sm.hdr[s];
        DgCtl& k = sm.ctl[s];
        const dp_carry& c = sm.carry[s];
        const double2* plan = sm.plan[s];
        // combine the partial searches: lowest index among the smallest squared distances; any other value within 2^-49 of
        // the minimum may round to the same sqrt -> the reference's own loop decides
        const double TOL = 1.0 + 0x1p-49;
        double ge = sm.ne[s][0]; int gi = sm.ni[s][0];
        int amb = sm.namb[s][0];
        for (int q = 1; q < DG_NQ; ++q) {
            amb |= sm.namb[s][q];
            if (sm.ne[s][q] < ge) { ge = sm.ne[s][q]; gi = sm.ni[s][q]; }
        }
        for (int q = 0; q < DG_NQ; ++q) if (sm.ne[s][q] != ge && sm.ne[s][q] <= ge * TOL) amb = 1;
        int mi;
        if (!amb) mi = (gi != 0x7fffffff && sqrt(ge) < 9999.0) ? gi : 0x7fffffff;
        else {
            double md = 9999.0; mi = 0x7fffffff;
            for (int i = 0; i < DP_PATH_POINTS; ++i) {
                const double dd = dg_dist_plain(h.x, h.y, plan[i].x, plan[i].y);
                if (dd < md) { md = dd; mi = i; }
            }
        }
        const int near_id = (mi == 0x7fffffff) ? c.path_near_id : mi;
        const int front_id = near_id + 8;
        int idx = (near_id == 199) ? near_id - 1 : near_id;
        if (idx < 0 || idx > 198) { ++k.ub; idx = idx < 0 ? 0 : 198; }
        const double2 pt = plan[idx], pn = plan[idx + 1];
        k.lat = dg_lat_dis(h.x, h.y, pt.x, pt.y, pn.x, pn.y, p.epsilon);
        k.dir_err = dg_angle_err(dg_heading(pt.x, pt.y, pn.x, pn.y, p.epsilon, p.pi), h.dir);
        k.near_id = near_id; k.front_id = front_id;
        if (front_id < 0) ++k.ub;
    }
    DG_SYNC();
    DG_MARK(13);

    // ---- P10: terms of the remaining length (Planning.cpp:662-672), CalcDistance idiom
    DG_PHASE(tid) {
        for (int it = tid; it < S * (DP_PATH_POINTS - 1); it += TPB) {
            const int s = it / (DP_PATH_POINTS - 1), j = it - s * (DP_PATH_POINTS - 1);
            const int f0 = dg_imax(sm.ctl[s].front_id, 0);
            if (j >= f0) {
                const double2 a = sm.plan[s][j], b = sm.plan[s][j + 1];
                sm.scr[s][j - f0] = dg_dist_plain(b.x, b.y, a.x, a.y);
            }
        }
    }
    DG_SYNC();
    DG_MARK(14);

    // ---- P11 (thread per scene): remaining length, UpdatePlanJudge (Planning.cpp:797-832), CalculateRadius on the PREVIOUS
    //      path (:199, 1000-1019), the (re)planning request
    DG_PHASE(tid) {
        if (tid >= S) continue;
        const int s = tid;
        const dp_scene_hdr& h = sm.hdr[s];
        DgCtl& k = sm.ctl[s];
        dp_carry& c = sm.carry[s];
        dp_plan_record& out = sm.rec[s];
        const double2* plan = sm.plan[s];
        const int pos = k.pos, near_id = k.near_id, front_id = k.front_id;
        const double remain = dg_seq_sum(sm.scr[s], dg_imax(0, 199 - dg_imax(front_id, 0)), DG_SCR, -1.0, [](int) { return 0.0; });
        const double lat = k.lat, dir_err = k.dir_err;
        bool afresh = true;
        int cause = 0;
        if (c.plan_his_behavior != k.d_behavior) cause = 1;
        else if (fabs(lat) > 0.2) cause = 2;
        else if (fabs(dir_err) > 45) cause = 3;
        else if (pos == 0 && remain < p.road_remain_distance) cause = 4;
        else if (pos != 0 && remain < p.inter_remain_distance) cause = 4;
        else afresh = false;
        double radius;
        {
            int ia = near_id, ib = (near_id + front_id) / 2, ic = front_id;
            if (ia < 0 || ia > 199) { ++k.ub; ia = ia < 0 ? 0 : 199; }
            if (ib < 0 || ib > 199) { ++k.ub; ib = ib < 0 ? 0 : 199; }
            if (ic < 0 || ic > 199) { ++k.ub; ic = ic < 0 ? 0 : 199; }
            const double2 A = plan[ia], B = plan[ib], Fp = plan[ic];
            const double d1 = dg_dist_plain(A.x, A.y, B.x, B.y), d2 = dg_dist_plain(B.x, B.y, Fp.x, Fp.y), d3 = dg_dist_plain(A.x, A.y, Fp.x, Fp.y);
            const double dd = d1 * d1 + d2 * d2 - d3 * d3;
            const double cosA = dd / (2 * d1 * d2);
            const double sinA = sqrt(1 - cosA * cosA);
            radius = (sinA < 0.001) ? 1000 : 0.5 * d3 / sinA;
        }
        out.path_lat_dis = lat; out.path_dir_err = dir_err; out.remain_dis = remain; out.radius = radius;
        out.aim_x = c.aim_x; out.aim_y = c.aim_y; out.aim_dir = c.aim_dir; out.aim_id = c.aim_id;
        out.afresh_cause = (uint16_t)cause; out.afresh_planning = afresh;
        out.path_near_id = (int16_t)near_id; out.path_front_near_id = (int16_t)front_id;
        c.path_near_id = near_id;
        c.plan_his_behavior = k.d_behavior;                 // history update of Planning.cpp:216
        {
            const int plan_count = c.plan_count;
            uint8_t cnt = (uint8_t)(plan_count + 1);        // BYTE count of CPlanningThread (Planning.cpp:219-223)
            if (cnt % 100 == 1) cnt = 1;
            c.plan_count = cnt;
            out.cnt = (uint8_t)(plan_count % 100);
        }
        // PathPlanning (Planning.cpp:845-877) or reuse (:142-146)
        k.afresh = afresh ? 1 : 0; k.cause = cause; k.req = 0; k.mean_n = 0;
        if (afresh) {
            k.plan_dirty = 1;
            if (pos == 0) {
                // the first-cycle Bezier above used the same two poses: identical points, nothing to redo
                if (!k.first) {
                    const double ax = c.aim_x, ay = c.aim_y;
                    const double ex = ax - h.x, ey = ay - h.y;
                    const double L = sqrt(dg_sq2(ex, ey)) / 3.0;
                    double c0, s0, c3, s3;
                    dg_sincos_deg(h.dir, &c0, &s0);
                    dg_sincos_deg(c.aim_dir, &c3, &s3);
                    k.bx0 = h.x; k.by0 = h.y; k.bx3 = ax; k.by3 = ay;
                    k.bx1 = fma(L, c0, h.x); k.by1 = fma(L, s0, h.y);
                    k.bx2 = fma(-L, c3, ax); k.by2 = fma(-L, s3, ay);
                    k.req = 1;
                }
            } else if (pos == 1 || pos == 2) {
                int n = c.aim_id;
                if (n > DP_PATH_POINTS) { ++k.ub; n = DP_PATH_POINTS; }
                if (n > k.rp_n0 + k.rp_n1) { ++k.ub; n = k.rp_n0 + k.rp_n1; }
                k.mean_n = n; k.req = 2;
                sm.any_mean = 1;
            } else k.req = 3;
        }
    }
    DG_SYNC();
    DG_MARK(15);

    // ---- P11b/c: CShare::MeanPoints (Planning.cpp:872) for junction scenes: segment lengths, then the sequential prefix
    if (sm.any_mean) {
        DG_PHASE(tid) {
            for (int it = tid; it < S * DG_SCR; it += TPB) {
                const int s = it / DG_SCR, j = it - s * DG_SCR;
                const DgCtl& k = sm.ctl[s];
                if (k.req == 2 && j < k.mean_n - 1) {
                    const DgView v = dg_view(m, sm.path[s][0], nullptr);
                    const double2 a = dg_pt(v, j), b = dg_pt(v, j + 1);
                    sm.scr[s][j + 1] = sqrt(dg_sq2(b.x - a.x, b.y - a.y));
                }
            }
        }
        DG_SYNC();
    DG_MARK(16);
        DG_PHASE(tid) {
            if (tid >= S) continue;
            const DgCtl& k = sm.ctl[tid];
            if (k.req == 2 && k.mean_n >= 2) {               // in-place sequential prefix: cum[i+1] = cum[i] + len[i]
                double* cum = sm.scr[tid];
                double acc = 0.0;
                cum[0] = 0.0;
                for (int j = 1; j < k.mean_n; ++j) { acc += cum[j]; cum[j] = acc; }
            }
        }
        DG_SYNC();
    DG_MARK(17);
    }

    // ---- P12: road_points -> sm.plan: CShare::BezierPlanning (Planning.cpp:863) / MeanPoints (:872), one thread per point
    DG_PHASE(tid) {
        for (int it = tid; it < S * DP_PATH_POINTS; it += TPB) {
            const int s = it / DP_PATH_POINTS, i = it - s * DP_PATH_POINTS;
            const DgCtl& k = sm.ctl[s];
            if (k.req == 1) {
                const double t = (double)i / (double)(DP_PATH_POINTS - 1);
                const double u = 1.0 - t;
                const double b0 = u * u * u;
                const double b1 = 3.0 * (u * u) * t;
                const double b2 = 3.0 * u * (t * t);
                const double b3 = t * t * t;
                sm.plan[s][i] = make_double2(fma(b3, k.bx3, fma(b2, k.bx2, fma(b1, k.bx1, b0 * k.bx0))),
                                             fma(b3, k.by3, fma(b2, k.by2, fma(b1, k.by1, b0 * k.by0))));
            } else if (k.req == 2) {
                const int n_in = k.mean_n;
                const DgView v = dg_view(m, sm.path[s][0], nullptr);
                double2 q;
                if (n_in <= 0) q = make_double2(0.0, 0.0);
                else if (n_in == 1) q = dg_pt(v, 0);
                else {
                    const double* cum = sm.scr[s];
                    const double step = cum[n_in - 1] / (double)(DP_PATH_POINTS - 1);
                    const double sv = (double)i * step;
                    int lo_i = 0, hi_i = n_in - 2;          // largest i <= n_in-2 with cum[i] <= sv
                    while (lo_i < hi_i) {
                        const int mid = (lo_i + hi_i + 1) >> 1;
                        if (cum[mid] <= sv) lo_i = mid; else hi_i = mid - 1;
                    }
                    const double seg = cum[lo_i + 1] - cum[lo_i];
                    const double t = seg > 0 ? (sv - cum[lo_i]) / seg : 0.0;
                    const double2 a = dg_pt(v, lo_i), b = dg_pt(v, lo_i + 1);
                    q = make_double2(fma(t, b.x - a.x, a.x), fma(t, b.y - a.y, a.y));
                    if (i == DP_PATH_POINTS - 1) q = dg_pt(v, n_in - 1);
                }
                sm.plan[s][i] = q;
            } else if (k.req == 3) sm.plan[s][i] = make_double2(0.0, 0.0);
        }
        if (tid < S) {                                      // recipe of the local-path search (Planning.cpp:152-168): a window of sm.plan
            DgCtl& k = sm.ctl[tid];
            DgPath& L = sm.path[tid][DG_NREG];
            const int s0 = dg_imax(k.near_id, 0);
            k.s0 = s0;
            L.local = 1; L.base0 = s0; L.stride0 = 1; L.n0 = DP_PATH_POINTS - s0; L.base1 = 0; L.n1 = 0; L.d = 0.0;
            L.lo = (double)(float)(-1.1); L.hi = (double)(float)(1.1); L.key = 0xffffffffu;
            k.hb2_bits = 0; k.hmin2_bits = 0x7f800000u; k.dl2_bits = 0;
        }
    }
    DG_SYNC();
    DG_MARK(18);

    // ---- P13: bounds of the local path for the pruned search (FP32: longest / shortest segment, largest difference of consecutive segments);
    //      path outputs (coalesced)
    DG_PHASE(tid) {
        const int lane = tid & 31;
        for (int s = tid >> 5; s < S; s += TPB / 32) {      // one warp per scene, one atomic per thread and bound
            DgCtl& k = sm.ctl[s];
            float hmx = 0.f, hmn = dg_inff(), dmx = 0.f;    // squared: longest / shortest segment, largest |u - w| of consecutive segments
            for (int j = k.s0 + lane; j < DP_PATH_POINTS - 1; j += 32) {
                const double2 a = sm.plan[s][j], b = sm.plan[s][j + 1];
                const float ux = (float)(b.x - a.x), uy = (float)(b.y - a.y);
                const float l2 = ux * ux + uy * uy;
                hmx = fmaxf(hmx, l2); hmn = fminf(hmn, l2);
                if (j + 2 < DP_PATH_POINTS) {
                    const double2 c = sm.plan[s][j + 2];
                    const float ex = (float)(c.x - b.x) - ux, ey = (float)(c.y - b.y) - uy;
                    dmx = fmaxf(dmx, ex * ex + ey * ey);
                }
            }
#if defined(DP_EMU)
            if (dg_float_bits(hmx) > k.hb2_bits) k.hb2_bits = dg_float_bits(hmx);
            if (dg_float_bits(hmn) < k.hmin2_bits) k.hmin2_bits = dg_float_bits(hmn);
            if (dg_float_bits(dmx) > k.dl2_bits) k.dl2_bits = dg_float_bits(dmx);
#else
            atomicMax(&k.hb2_bits, __float_as_uint(hmx));   // (non-negative floats order like their bit patterns)
            atomicMin(&k.hmin2_bits, __float_as_uint(hmn));
            atomicMax(&k.dl2_bits, __float_as_uint(dmx));
#endif
        }
        for (int it = tid; it < S * DP_PATH_POINTS; it += TPB) {
            const int s = it / DP_PATH_POINTS, i = it - s * DP_PATH_POINTS;
            const double2 q = sm.plan[s][i];
            if (sm.ctl[s].plan_dirty) last_path[(size_t)(first + s) * DP_PATH_POINTS + i] = q;   // the carried path only changes on (re)planning cycles
            if (path_xy) {
                path_xy[(size_t)(first + s) * 400 + i] = q.x; path_xy[(size_t)(first + s) * 400 + DP_PATH_POINTS + i] = q.y;
            }
            if (path_ll && (i & 1) == 0) {                  // every 2nd point -> WGS84 (Planning.cpp:180-183, 203-212)
                path_ll[(size_t)(first + s) * 200 + (i >> 1)] = fma(q.y, p.k_lat, p.lat0);
                path_ll[(size_t)(first + s) * 200 + DP_OUT_POINTS + (i >> 1)] = fma(q.x, p.k_lng, p.lng0);
            }
        }
    }
    DG_SYNC();
    DG_MARK(19);

    // ---- P14: local path collision (Planning.cpp:152-168): every (scene, obstacle) pair against a window of sm.plan
    dg_scan_phase<G, TPB>(sm, S, first, obs_x, obs_y, max_obs, [&](int s) {
        DgPath& pa = sm.path[s][DG_NREG];
        const DgCtl& k = sm.ctl[s];
        DgJob j;
        j.v = dg_view(m, pa, sm.plan[s]); j.lo = pa.lo; j.hi = pa.hi; j.key = &pa.key; j.P = pa.n0; j.scene = s;
        j.tvx = nullptr; j.tvy = nullptr; j.tdth = nullptr; j.tT = 0;
        j.hb = sqrtf(dg_bits_float(k.hb2_bits)) * 1.0001f + 1e-4f;
        const float hmin = sqrtf(dg_bits_float(k.hmin2_bits)) * 0.9999f - 1e-6f;
        // |u/|u| - w/|w|| <= 2 |u - w| / (|u| + |w|) <= |u - w| / hmin for consecutive segment vectors u, w
        const float delta = (hmin > 1e-6f) ? sqrtf(dg_bits_float(k.dl2_bits)) / hmin * 1.001f + 1e-4f : 2.0f;
        j.dmax = dg_dmax(pa.lo, pa.hi, j.hb, delta, hmin);
        return j;
    });
    DG_MARK(20);
    // 14b: arclength terms up to the selected point (SearchObstacle idiom), all threads
    DG_PHASE(tid) {
        for (int it = tid; it < S * (DP_PATH_POINTS - 1); it += TPB) {
            const int s = it / (DP_PATH_POINTS - 1), j = it - s * (DP_PATH_POINTS - 1);
            const DgPath& pa = sm.path[s][DG_NREG];
            if (pa.key == 0xffffffffu || j >= (int)(pa.key >> 16)) continue;
            const double2 a = sm.plan[s][pa.base0 + j], b = sm.plan[s][pa.base0 + j + 1];
            sm.scr[s][j] = sqrt(dg_sq2(b.x - a.x, b.y - a.y));
        }
    }
    DG_SYNC();
    DG_MARK(21);

    // ---- P15 (thread per scene): local search result, SpeedPlanning (Planning.cpp:888-990), the rest of the record
    DG_PHASE(tid) {
        if (tid >= S) continue;
        const int s = tid;
        DgCtl& k = sm.ctl[s];
        dp_plan_record& out = sm.rec[s];
        dp_trace_record* tr = trace ? trace + first + s : nullptr;
        const DgPath& pa = sm.path[s][DG_NREG];
        const int P = pa.n0;
        const size_t ob = (size_t)(first + s) * max_obs;
        DgRes ls = dg_selected(dg_view(m, pa, sm.plan[s]), P, pa.key, obs_x + ob, obs_y + ob, pa.lo, pa.hi);
        if (ls.found) ls.dis_lng = dg_seq_sum(sm.scr[s], ls.pathid, DG_SCR, -1.0, [](int) { return 0.0; });
        ++k.n_traj; k.pts += P;
        if (tr) dg_put_slot(&tr->local, ls, 1);
        double brake = 0.0, des_acc = 0.0;
        bool acc_flag = false;
        if (k.pos <= 2) {
            if (ls.found) {
                if (ls.dis_lng - 4 > 9) brake = 3 + (ls.dis_lng - 9) / (k.faraim - 9) * (k.v_exp - 3);
                else if (ls.dis_lng - 4 > 5) brake = 3;
                else { brake = 0; acc_flag = true; des_acc = -3; }
            } else brake = k.v_exp;
        }
        out.mindist_lat = ls.dis_lat; out.mindist_lon = ls.dis_lng; out.brakespeed = brake; out.des_acc = des_acc;
        out.ob_index = (int16_t)ls.ob; out.ob_pathid = (uint16_t)ls.pathid; out.n_traj = (uint16_t)k.n_traj;
        out.ob_flag = ls.found ? 1 : 0; out.acc_flag = acc_flag;
        if (tr) { tr->ub_hits = (uint16_t)k.ub; tr->pts_scored = (uint32_t)k.pts; }
    }
    DG_SYNC();
    DG_MARK(22);

    // ---- P16: records and carry out with coalesced 16-byte stores; record mirrors (pinned host / peer GPUs); completion flag
    DG_PHASE(tid) {
        const uint4* sr = reinterpret_cast<const uint4*>(sm.rec);
        const uint4* sc = reinterpret_cast<const uint4*>(sm.carry);
        uint4* gr = reinterpret_cast<uint4*>(rec + first);
        uint4* gc = reinterpret_cast<uint4*>(carry + first);
        for (int i = tid; i < S * 8; i += TPB) {
            const uint4 w = sr[i];
            gr[i] = w; gc[i] = sc[i];
#pragma unroll
            for (int q = 0; q < DP_MAX_MIRRORS; ++q)
                if (q < io.n_mirror) reinterpret_cast<uint4*>(io.mirror[q] + first)[i] = w;
        }
    }
    DG_MARK(23);
#if !defined(DP_EMU)
    if (io.tally) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();                                // cumulative: the CTA's stores (ordered before the barrier) before the tally
            if (atomicAdd(io.tally, (unsigned)S) + (unsigned)S == io.tally_n) dg_complete(io.tally, io, true, true);
        }
    }
#endif
}
