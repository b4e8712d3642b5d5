// csrc/dp_cycle.cu -- the Decision + Planning cycle kernel (sm_100a): dp_cycle_kernel<PHASE, WPB>, launched as a Decision
// half and a Planning half that overlap scene by scene (PHASE 1 / 2), see below.
//
// One WARP owns one scene for the whole cycle: LoadRefPath -> AroundObstacle -> BehaviorDecision
// (with the in-lane avoid sweep) -> SpeedDecision/RefPath  (Decision.cpp:216-315, 323-486), then
// Calculate_aim_dis -> SearchAimPoint -> GetVhclLocalState -> UpdatePlanJudge -> PathPlanning ->
// local-path SearchObstacle -> SpeedPlanning -> CalculateRadius -> result packing
// (Planning.cpp:118-217).  Scalar rule-tree state is warp-uniform (every lane holds it, branches
// never diverge); the geometry operators in dp_device.cuh spread their inner loops over the lanes.
// Candidate paths exist only as shared-memory tiles; HBM sees the 128-byte scene header, the
// obstacle SoA rows, the 128-byte carry, the previous local path (the reference's own cross-cycle
// state, Planning.cpp:6) and the 128-byte plan record.
#include <cstdlib>
#include "dp_device.cuh"
#include "dp_fused.cuh"
#include "dp_kernels.h"
#include "dp_group.cuh"

namespace {

struct Beh { int behavior, target, light; bool lanechg, obsavoid; int dlg; };

// a lane slice of the map as a path recipe: map point index base + stride*j, j < P, lateral offset d
struct Slice { int base, stride, P; double d; };

__device__ __forceinline__ void put_slot(dp_search_slot* slot, const SearchRes& r, int evaluated, int lane) {
    if (slot && lane == 0) {
        slot->dis_lat = r.dis_lat; slot->dis_lng = r.dis_lng; slot->ob_index = (int16_t)r.ob;
        slot->pathid = (uint16_t)r.pathid; slot->evaluated = (uint8_t)evaluated; slot->found = r.found ? 1 : 0;
        slot->pad[0] = slot->pad[1] = 0;
    }
}

// forward 120-point / backward 40-point slices of one lane (Decision.cpp:581-596, 611-622, 649-660)
__device__ __forceinline__ void lane_slices(const DevMap& m, int gl, int id, int id_more, Slice& fwd, Slice& rear, int& ub) {
    const int off = m.lane_pt_off[gl], n = m.lane_pt_off[gl + 1] - off;
    const int a = min(n, id + id_more), b = min(n, id + 120 + id_more);
    fwd.base = off + a; fwd.stride = 1; fwd.P = max(0, b - a); fwd.d = 0.0;
    const int lo = max(0, id + id_more - 40);
    int start = a;
    if (start >= n) { start = n - 1; if (a > lo) ++ub; }   // reference reads index == size here (UB); clamp
    rear.base = off + start; rear.stride = -1; rear.P = max(0, a - lo); rear.d = 0.0;
}

// recipe of a slice: map points in place (+ normals when shifted: CreateNewPath fused into the staging)
__device__ __forceinline__ Src slice_src(const DevMap& m, int base, int stride, int P, double d) {
    Src s = dp_src_run(m.xy + base, stride, P);
    s.nrm0 = m.nrm + base; s.d = d;
    return s;
}

// does the arclength from `id` along lane `gl`, while cond(attr[i+1]) holds, exceed thr?
// (Decision.cpp:1179-1190 and siblings; partial sums are monotone, so stopping at the first
// partial sum > thr gives the reference's answer without walking the whole lane)
// mode: 0 = attr == 1, 1 = attr & 1, 2 = never
static __device__ __noinline__ bool run_exceeds(const DevMap& m, WarpSmem& sm, int gl, int id, int mode, double thr, int lane) {
    if (mode == 2) return 0.0 > thr;
    const int off = m.lane_pt_off[gl], n = m.lane_pt_off[gl + 1] - off;
    if (id >= n - 1) return 0.0 > thr;
    {   // the run ends at run_end[id]; its length is cump[end] - cump[id] up to the rounding bound lane_cerr: outside that
        // bracket the answer needs no walk (dp_group.cuh, dg_run_exceeds)
        const int e = (mode == 0 ? m.run_end0 : m.run_end1)[off + id];
        const double approx = m.cump[off + e] - m.cump[off + id], err = m.lane_cerr[gl];
        if (approx > thr + err) return true;
        if (approx < thr - err) return false;
    }
    double sum = 0.0;
    for (int i0 = id; i0 < n - 1; i0 += DP_SCR) {
        const int cnt = min(DP_SCR, n - 1 - i0);
        int first_bad = cnt;                               // first term whose condition fails
        __syncwarp();
        for (int j0 = 0; j0 < cnt; j0 += 32) {
            const int j = j0 + lane;
            bool ok = true;
            if (j < cnt) {
                const int a = m.attr[off + i0 + j + 1];
                ok = (mode == 0) ? (a == 1) : ((a & 1) != 0);
                sm.scr[j] = m.lenp[off + i0 + j];
            }
            const unsigned bad = __ballot_sync(DP_FULL, !ok);
            if (bad) { first_bad = j0 + __ffs(bad) - 1; break; }
        }
        const int cn = min(cnt, first_bad);
        __syncwarp();
        dp_pad_scr(sm, cn, lane);
        __syncwarp();
        const SeqHit hq = dp_seq_first(sm, cn, sum, 0.0, thr);
        if (hq.k >= 0) return true;
        sum = hq.acc;
        if (first_bad < cnt) break;
    }
    return sum > thr;
}

// SearchAimPoint along one map lane (Planning.cpp:410-432 and the lane-change twins): index of the
// first point whose accumulated arclength exceeds faraim + 4, -1 if the walk ends first, -2 if it
// never starts (aim point keeps its previous value)
static __device__ __noinline__ int aim_walk_lane(const DevMap& m, WarpSmem& sm, int gl_walk, int from, int to_excl, float faraim, int lane) {
    if (from >= to_excl) return -2;
    const int off = m.lane_pt_off[gl_walk], n = m.lane_pt_off[gl_walk + 1] - off;
    if (from < 0) return -3;
    if (to_excl > n - 1) { to_excl = n - 1; if (from >= to_excl) return -3; }
    double sum = 0.0;
    for (int i0 = from; i0 < to_excl; i0 += DP_SCR) {
        const int cnt = min(DP_SCR, to_excl - i0);
        __syncwarp();
        for (int j = lane; j < cnt; j += 32) sm.scr[j] = m.lenp[off + i0 + j];
        dp_pad_scr(sm, cnt, lane);
        __syncwarp();
        const SeqHit hq = dp_seq_first(sm, cnt, sum, 4.0, (double)faraim);
        if (hq.k >= 0) return i0 + hq.k;
        sum = hq.acc;
    }
    return -1;
}

// junction reference path: remaining approach lane + connector (pos 1) or remaining connector +
// first 60 points of the next lane (pos 2), read in place (Decision.cpp:352-367, 438-452)
__device__ __forceinline__ Src junction_src(const DevMap& m, int base0, int n0, int base1, int n1) {
    Src s = dp_src_run(m.xy + base0, 1, n0);
    s.p1 = m.xy + base1; s.n1 = n1;
    return s;
}

// junction reference path as two forward map runs: remaining approach lane + connector (PreStubDecision,
// Decision.cpp:352-367) or remaining connector + first 60 points of the next lane (StubDecision, :438-452)
__device__ __forceinline__ void junction_recipe(const DevMap& m, const dp_scene_hdr& h, int& base0, int& n0, int& base1, int& n1) {
    const int gc = (h.conn >= 0 && h.conn < m.n_conn) ? m.conn[h.conn].lane : -1;
    const int coff = gc >= 0 ? m.lane_pt_off[gc] : 0, n_inter = gc >= 0 ? m.lane_pt_off[gc + 1] - coff : 0;
    const int gj = m.road_lane_base[h.road_num - 1] + h.lane_num - 1;
    const int off = m.lane_pt_off[gj], n = m.lane_pt_off[gj + 1] - off;
    if (h.pos == 1) {
        const int idj = (int)(uint16_t)h.id[h.lane_num - 1];
        base0 = off + idj; n0 = max(0, n - idj);
        base1 = coff; n1 = n_inter;
    } else {
        const int idj = (int)(uint16_t)h.id[h.last_lanenum - 1];
        base0 = coff + idj; n0 = max(0, n_inter - idj);
        base1 = off; n1 = min(60, n);
    }
}

// out-of-line copy for the rare trajectories (junction reference path, sweep with more than 16 obstacles)
static __device__ __noinline__ SearchRes dp_search_cold(const Src s, double mx, double my, const double* ox, const double* oy, int N,
                                                        const LaneMap lm, double lo, double hi, WarpSmem& sm, int lane, float hb = 0.f,
                                                        float dmax = 0.f) {
    return dp_search(s, mx, my, ox, oy, N, lm, lo, hi, sm, lane, hb, dmax);
}

// ---- per-scene hand-off between the two overlapped launches ----------------------------------------------------------
// The Planning launch is a programmatic dependent launch: its CTAs become eligible as soon as every Decision CTA has
// STARTED (they trigger at entry), and take the SM slots the Decision launch frees as its short scenes retire, instead of
// waiting for the slowest scene of the batch (the ~16 % that run the avoid sweep).  A scene's Planning warp therefore
// waits for THAT scene's Decision warp only: release/acquire on done[scene] at GPU scope.  No deadlock: when the first
// Planning CTA is scheduled every Decision CTA is already resident, so every awaited flag has a running producer.
__device__ __forceinline__ void dp_publish(unsigned* flag, unsigned epoch, int lane) {
    // the warp barrier orders every lane's stores of this scene before lane 0's store, and a release is cumulative: ONE fence per
    // scene.  (A __threadfence() by all 32 lanes in front of it, as in round 1, is a second full fence on the scene's critical
    // path: 63.5 -> 63.1 us per cycle without it, profiles/README.md.)
    __syncwarp();
    if (lane == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
}
__device__ __forceinline__ void dp_await(const unsigned* flag, unsigned epoch) {
    unsigned v = 0;
#pragma unroll 1
    for (int spin = 0; spin < (1 << 22); ++spin) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (v == epoch) break;
        __nanosleep(spin < 64 ? 100 : 1000);
    }
    if (v != epoch) __trap();                               // never spin forever on a producer that is not there
    __syncwarp();
}
// reads of what the Decision launch of THIS cycle wrote go to L2 (the SM's L1 may hold an older copy of the line)
template <class T> __device__ __forceinline__ T dp_l2(const T* p) { return __ldcg(p); }

}  // namespace

// Which scans of the warp kernel use the exact pruning of dp_group.cuh (measured on the B200, profiles/README.md round 2):
// in the avoid sweep a lane owns a whole 120-point scan of its (candidate, obstacle) pair and pruning pays (78 -> 70 us per
// 4096-scene cycle); in the lane-region and local-path searches the lanes already split a path in chunks of ~40 points, the
// sampling pass costs as much as it saves and the extra code hurts (70 -> 83 us): off.  Large batches run the one-warp CTAs,
// whose instruction footprint matters more than the scan length: no pruning there either.
#ifndef DP_PRUNE_REGION
#define DP_PRUNE_REGION 0
#endif
#ifndef DP_PRUNE_LOCAL
#define DP_PRUNE_LOCAL 0
#endif
#ifndef DP_PRUNE_SWEEP
#define DP_PRUNE_SWEEP (WPB == 4)
#endif
#define DP_CARVEOUT 77
// CTA size of the cycle kernel.  WPB = 4 (7 CTAs = 28 warps per SM) keeps a 4096-scene batch a single wave.  WPB = 1 (25 CTAs
// per SM; the per-CTA shared-memory reservation costs three slots) recycles a warp's slot the moment ITS scene is done
// instead of when the slowest scene of its CTA retires (sweep scenes last twice as long: ncu showed 21.6 of 28 warp slots
// active at 65 536 scenes): 0.942 -> 0.857 ms there, but 1.8 % slower on the one-wave batch.  The launcher picks by batch size.
#ifndef DP_MIN_BLOCKS_W1
#define DP_MIN_BLOCKS_W1 25
#endif
#define DP_MIN_BLOCKS(WPB) ((WPB) == 1 ? DP_MIN_BLOCKS_W1 : 7)

// PHASE 1 / 2: Decision half / Planning half as two launches -- the same work with half the code per kernel: with 28 warps
// per SM in different places of a ~11 k-instruction kernel the instruction cache thrashes (ncu: 25 % `no_instruction` stalls);
// each half alone fits.  The hand-off between the two
// halves is what the reference hands from CDecisionThread to CPlanningThread (DecisionOut, Decision.cpp:187-205),
// already stored in dp_carry / dp_plan_record.
#ifdef DP_DEBUG_CLOCK
// instrumented build only (make debug, tools/scene_timeline.py): per scene and launch {start ns, end ns, SM id, n_traj,
// regions done ns, sweep start ns, sweep end ns, -}
__device__ long long g_dbg_timeline[2 * 65536 * 2 * 8];   // [epoch parity][scene][phase][8]
__device__ __forceinline__ long long dbg_now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return (long long)t; }
#define DBG_MARK(ph, slot) if (lane == 0) g_dbg_timeline[(((size_t)(io.epoch & 1) * 65536 + scene) * 2 + (ph)) * 8 + (slot)] = dbg_now()
#define DBG_END(ph, nt) if (lane == 0) { long long* g = g_dbg_timeline + (((size_t)(io.epoch & 1) * 65536 + scene) * 2 + (ph)) * 8; g[1] = dbg_now(); g[3] = (nt); }
extern "C" int dp_debug_scene_timeline(long long* dst, int n_scenes) {
    (void)n_scenes;
    return (int)cudaMemcpyFromSymbol(dst, g_dbg_timeline, sizeof(g_dbg_timeline));   // dst: [2][65536][2][8]
}
#else
#define DBG_MARK(ph, slot)
#define DBG_END(ph, nt)
#endif

template <int PHASE, int WPB>
__global__ void __launch_bounds__(WPB * 32, DP_MIN_BLOCKS(WPB))
dp_cycle_kernel(DevMap m, dp_params p, int n_scenes, const dp_scene_hdr* __restrict__ hdr, const double* __restrict__ obs_x,
                const double* __restrict__ obs_y, int max_obs, dp_carry* __restrict__ carry, double2* __restrict__ last_path,
                dp_plan_record* __restrict__ rec, dp_trace_record* __restrict__ trace, double* __restrict__ path_xy,
                double* __restrict__ path_ll, DpIo io) {
    __shared__ WarpSmem smem[WPB];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int scene = blockIdx.x * WPB + wib;
    if (scene >= n_scenes) return;
#ifdef DP_DEBUG_CLOCK
    if (lane == 0) {
        unsigned sid;
        asm volatile("mov.u32 %0, %smid;" : "=r"(sid));
        long long* g = g_dbg_timeline + (((size_t)(io.epoch & 1) * 65536 + scene) * 2 + (PHASE == 2 ? 1 : 0)) * 8;
        g[0] = dbg_now(); g[2] = sid; g[4] = g[5] = g[6] = 0;
    }
    const long long dbg_t0 = clock64();
    long long dbg_t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define DBG_T(i) dbg_t[i] = clock64() - dbg_t0
#else
#define DBG_T(i)
#endif
    WarpSmem& sm = smem[wib];
    if (PHASE == 1 && io.done) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // Planning CTAs may start filling in
    if (PHASE == 1 && io.in_flag) dp_await(io.in_flag, io.epoch);                                // chained submit: inputs staged?
    if (PHASE == 2 && io.done) dp_await(io.done + scene, io.epoch);
    // while the header is on its way: ask L2 for the lines the warp needs next and whose addresses do not depend on it -- the two
    // obstacle rows and the carry (otherwise three DRAM round trips in a row at the start of every scene after an L2 flush)
    if (PHASE == 1 && !io.in_flag && lane < 5) {
        const size_t row = (size_t)scene * max_obs, last = (size_t)(max_obs > 0 ? max_obs - 1 : 0);
        const void* a = lane == 0 ? (const void*)(obs_x + row) : lane == 1 ? (const void*)(obs_x + row + last)
                      : lane == 2 ? (const void*)(obs_y + row) : lane == 3 ? (const void*)(obs_y + row + last) : (const void*)(carry + scene);
        asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
    }
    // the 128-byte scene header comes in with one coalesced warp load and is read from shared memory afterwards
    sm.hdr[lane] = (PHASE == 2 || io.in_flag) ? dp_l2(reinterpret_cast<const uint32_t*>(hdr + scene) + lane)   // (staged by a concurrent launch / copy)
                                              : reinterpret_cast<const uint32_t*>(hdr + scene)[lane];
    __syncwarp();
    const dp_scene_hdr& h = *reinterpret_cast<const dp_scene_hdr*>(sm.hdr);
    const double* ox = obs_x + (size_t)scene * max_obs;
    const double* oy = obs_y + (size_t)scene * max_obs;
    const int N = min((int)h.n_obs, max_obs);
    double2* lastp = last_path + (size_t)scene * DP_PATH_POINTS;
    dp_carry* const cg = carry + scene;
    dp_plan_record* const out = rec + scene;                // the record is assembled in place: fields are stored when final
    // deferred gather: last cycle's record of this scene (DpIo) is picked up here, before this cycle overwrites it, and sent
    // when the Decision half of the scene is done: the warps of a launch START together (28 per SM x 148 SMs x world stores at
    // once is a 4 us NVLink burst that every warp then sits behind: +3.9 us per step at 8 GPUs), but they FINISH spread over
    // 15-50 us
    uint32_t fwd_w = 0;
    if (PHASE == 1 && io.n_fwd) fwd_w = __ldcg(reinterpret_cast<const uint32_t*>(io.fwd_src + scene) + lane);
    const LaneMap lm = dp_lane_map(N, lane);
    // this lane's obstacle stays in registers for the whole cycle when N < 32
    const bool lm_act = (lm.nchunk > 1) && (lane < N * lm.nchunk);
    const bool via_l2 = PHASE == 2 || io.in_flag != nullptr;
    const double mx = lm_act ? (via_l2 ? dp_l2(ox + lm.o) : ox[lm.o]) : 0.0, my = lm_act ? (via_l2 ? dp_l2(oy + lm.o) : oy[lm.o]) : 0.0;
    dp_trace_record* tr = trace ? trace + scene : nullptr;
    if (tr && PHASE == 1) {                                 // zero the trace record cooperatively
        uint32_t* w = reinterpret_cast<uint32_t*>(tr);
        for (int i = lane; i < (int)(sizeof(dp_trace_record) / 4); i += 32) w[i] = 0;
        __syncwarp();
    }
    const double Vw = p.vehicle_width;
    const int pos = h.pos;
    int ub = 0, n_traj = 0, pts = 0;
    int rp_base0 = 0, rp_n0 = 0, rp_base1 = 0, rp_n1 = 0;    // DecisionOut.refpath as a recipe (two forward map runs)
    int gl = 0, lane_sum = 0;
    const int lane_n = h.lane_num;
    // decision outputs that the planning half consumes
    int d_behavior = 1, d_target = 0;
    double v_exp = 10.0;

    if (PHASE == 2) {
        // ---- hand-off from the Decision launch ----
        d_behavior = dp_l2(&cg->behavior); d_target = dp_l2(&cg->target_lanenum); v_exp = dp_l2(&cg->velocity_expect);
        n_traj = dp_l2(&out->n_traj);
        if (tr) { ub = dp_l2(&tr->ub_hits); pts = (int)dp_l2(&tr->pts_scored); }
        if (pos == 0) {
            gl = m.road_lane_base[h.road_num - 1] + lane_n - 1;
            lane_sum = m.road_lane_base[h.road_num] - m.road_lane_base[h.road_num - 1];
        } else if (pos == 1 || pos == 2) junction_recipe(m, h, rp_base0, rp_n0, rp_base1, rp_n1);
    } else if (pos == 0) {
        // =========================== SegmentDecision (Decision.cpp:216-315) ===========================
        const int road = h.road_num;
        gl = m.road_lane_base[road - 1] + lane_n - 1;
        lane_sum = m.road_lane_base[road] - m.road_lane_base[road - 1];
        const int off = m.lane_pt_off[gl], id_sum = m.lane_pt_off[gl + 1] - off;
        const int id = (int)(uint16_t)h.id[lane_n - 1];
        // ---- Nav_LaneChange (Decision.cpp:685-738) ----
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
            if (dirn) {                                     // CalcNaviLaneChgTimes (Decision.cpp:498-538)
                int times = 5;
                for (int i = 0; i < DP_LANESUM && h.out_lane_no[i] != 0; ++i) {
                    const int t = (dirn == 1) ? lane_n - h.out_lane_no[i] : h.out_lane_no[i] - lane_n;
                    if (t < times) times = t;
                }
                navi_t = (unsigned)(times & 0xff);
            }
        }
        // ---- LoadRefPath (Decision.cpp:553-673) ----
        const int idc = min(id, id_sum - 1);
        const int lanechg = m.attr[off + idc];
        const double W = m.width[off + idc] / 100.0;
        // F and R always; at most ONE neighbour pair exists per cycle: left for attribute 1/3, right only
        // for attribute 2 (the reference never loads the right lane for 3, Decision.cpp:636)
        Slice F, R, NF, NR;
        NF.base = NR.base = 0; NF.stride = 1; NR.stride = -1; NF.P = NR.P = 0; NF.d = NR.d = 0.0;
        lane_slices(m, gl, id, p.id_more, F, R, ub);
        int side = 0, gn = gl;                              // gn: the lane the neighbour pair is read from
        if (lanechg == 1 || lanechg == 3) {
            side = 1;
            if (lane_n > 1) {
                const int idl = (int)(uint16_t)h.id[lane_n - 2];
                const int nl = m.lane_pt_off[gl] - m.lane_pt_off[gl - 1];
                if (idl > 0 && idl < nl) { lane_slices(m, gl - 1, idl, p.id_more, NF, NR, ub); gn = gl - 1; }
            } else { NF = F; NF.d = -1 * W; NR = R; NR.d = -1 * W; }
        } else if (lanechg == 2) {
            side = 2;
            if (lane_n < lane_sum) {
                const int idr = (int)(uint16_t)h.id[lane_n];
                const int nr = m.lane_pt_off[gl + 2] - m.lane_pt_off[gl + 1];
                if (idr > 0 && idr < nr) { lane_slices(m, gl + 1, idr, p.id_more, NF, NR, ub); gn = gl + 1; }
            } else { NF = F; NF.d = W; NR = R; NR.d = W; }
        }
        // ---- AroundObstacle (Decision.cpp:759-881): the four trajectories in ONE fused pass ----
        const int nslot = (side == 2) ? 4 : 2;
        double gF = 0.0, gNF = 0.0, gNR = 0.0;              // gaps stay 0 (memset state) for paths that are not evaluated
        double bdF = 0.0;                                   // lane o < N: squared distance of obstacle o to its nearest point of F (avoid sweep)
        {
            const int rb[4] = {F.base, R.base, NF.base, NR.base}, rs[4] = {F.stride, R.stride, NF.stride, NR.stride};
            const int rP[4] = {F.P, R.P, NF.P, NR.P};
            const double rd[4] = {0.0, 0.0, NF.d, NR.d};
            dp_region_stage(m, sm, rb, rs, rP, rd, lane);
            const double nlo = (side == 2) ? -0.5 * W : -0.5 * Vw, nhi = (side == 2) ? 0.5 * Vw : 0.5 * W;
            // pruning bounds of the scans (dp_group.cuh): F / R from the ego lane, the neighbour pair from its lane (or the
            // ego lane shifted by +-W when the neighbour is virtual)
            float hbF, dmF, hbN, dmN;
            dg_bounds(m, gl, 0.0, -0.5 * Vw, 0.5 * Vw, &hbF, &dmF);
            dg_bounds(m, gn, NF.d, nlo, nhi, &hbN, &dmN);
            int qoff = 0;
            bdF = __longlong_as_double(0x7ff0000000000000LL);
#pragma unroll 1
            for (int r = 0; r < 4; ++r) {                   // one copy of the search code, four staged trajectories
                const int Pr = (r == 0) ? F.P : (r == 1) ? R.P : (r == 2) ? NF.P : NR.P;
                if (Pr != 0) {
                    Src sp = dp_src_run(m.xy, 1, Pr);
                    sp.q_off = qoff;
                    const SearchRes sr = dp_search(sp, mx, my, ox, oy, N, lm, r < 2 ? -0.5 * Vw : nlo, r < 2 ? 0.5 * Vw : nhi, sm, lane,
                                                   DP_PRUNE_REGION ? (r < 2 ? hbF : hbN) : 0.f, r < 2 ? dmF : dmN, r == 0 ? &bdF : nullptr);
                    ++n_traj; pts += Pr;
                    put_slot(tr ? &tr->region[r < 2 ? r : nslot + r - 2] : nullptr, sr, 1, lane);
                    if (r == 0) gF = sr.dis_lng; else if (r == 2) gNF = sr.dis_lng; else if (r == 3) gNR = sr.dis_lng;
                }
                qoff += Pr;
            }
        }
        const double gLF = (side == 1) ? gNF : 0.0, gLR = (side == 1) ? gNR : 0.0;
        const double gRF = (side == 2) ? gNF : 0.0, gRR = (side == 2) ? gNR : 0.0;
        if (tr && lane == 0) { tr->width_curlane = W; tr->navi_lanechg = navi; tr->navi_lanechg_times = navi_t; }
        DBG_T(5);
        DBG_MARK(0, 4);

        // ---- BehaviorDecision (Decision.cpp:898-1773) ----
        dp_carry c;                                         // (read through L2, 16 bytes at a time)
        {
            const int4* src = reinterpret_cast<const int4*>(cg);
            int4* dst = reinterpret_cast<int4*>(&c);
#pragma unroll
            for (int k = 0; k < (int)(sizeof(dp_carry) / 16); ++k) dst[k] = __ldcg(src + k);
        }
        Beh cur;
        cur.behavior = c.behavior; cur.target = c.target_lanenum; cur.light = c.light_status;
        cur.lanechg = c.lanechg_status != 0; cur.obsavoid = c.obsavoid_status != 0; cur.dlg = c.behavior_to_dlg;
        const int his_behavior = c.his_behavior, his_target = c.his_target_lanenum, his_light = c.his_light_status;
        int lane_cur = lane_n;
        int z_light = c.light_status;
        int sweep_pick = -1;
        const double period = h.period_ms;
        int K = 0;
        while (K < DP_MAX_SWEEP && (double)K < (W - Vw) / 0.6) ++K;
#define DP_KEEP(reset) do { cur.behavior = 1; cur.target = lane_cur; if (reset) cur.lanechg = false; } while (0)
#define DP_TICK do { c.leftlight_time += period; if (c.leftlight_time > 2000) c.leftlight_time = 2000; } while (0)
        if (lanechg == 0) {                                 // :920-1010
            if (gF < 15) {
                c.no_obsavoid_time = 0;
                c.obsavoid_time++;
                if (c.obsavoid_time > 2) {
                    // in-lane avoid sweep: candidates L0..L(K-1), R0..R(K-1), first feasible wins (Decision.cpp:940-974).
                    // With a trace buffer the remaining candidates are scored too (evaluated = 2) but neither counted nor used.
                    // Candidate 0 of either side is F itself under the F region's window: result known (the F slot) and, with
                    // gF < 15, never feasible -- only the 2(K-1) shifted candidates are scored (dp_fused.cuh, dp_sweep_g).
                    const int total = 2 * K, shifted = 2 * (K - 1);
                    DBG_MARK(0, 5);
                    if (shifted > 0 && N > 0 && N <= 16) {
                        dp_sweep_stage(m, sm, F.base, F.P, lane);
                        const float hmaxF = m.lane_hmax[gl], hminF = m.lane_hmin[gl], dnF = m.lane_dnmax[gl];
                        // Which obstacles can matter to ANY candidate?  A point of a candidate is its point of F moved by |d| <= 0.3 (K-1),
                        // so an obstacle is at least (its distance to F) - |d| away from every candidate, and it can only pass a corridor
                        // test from within that candidate's reach (dg_dmax, growing with |d|).  The F region search has just measured the
                        // distance of every obstacle to F: the few that remain are dealt out as (candidate, obstacle) lanes -- normally
                        // all 2(K-1) candidates in ONE pass instead of 32 / N per pass.
                        unsigned relmask = (N >= 32) ? 0xffffffffu : ((1u << N) - 1u);
                        {
                            const float adm = 0.3f * (float)(K - 1) * 1.0001f;
                            const float hbm = hmaxF + adm * dnF + 1e-4f;
                            const float dlt = (hminF > 1e-6f) ? dnF * (1.0f + 4.0f * adm / hminF) * 1.0001f + 1e-6f : 2.0f;
                            const float dmm = dg_dmax(-0.5 * Vw, 0.5 * Vw, hbm, dlt, hminF - adm * dnF);
                            const bool rel = lane < N && !(sqrt(bdF) - (double)adm > (double)dmm * 1.000001 + 1e-6);
                            relmask &= __ballot_sync(DP_FULL, rel);
                            if (relmask == 0u) relmask = 1u;        // nobody within reach: one obstacle stands in (it cannot produce a key either)
                        }
                        const int M = __popc(relmask);
                        const int per = min(8, 32 / M);
                        const int oid = (int)__fns(relmask, 0, lane % M + 1);   // this lane's obstacle: the (lane mod M)-th relevant one
                        const double smx = __shfl_sync(DP_FULL, mx, oid), smy = __shfl_sync(DP_FULL, my, oid);
                        for (int u0 = 0; u0 < shifted && (sweep_pick < 0 || tr); u0 += per) {
                            const int cnt = min(per, shifted - u0);
                            const bool none_yet = sweep_pick < 0;
                            int first_g = -1;
                            const int first = dp_sweep_pass(sm, F.P, u0, cnt, K, smx, smy, M, lm, -0.5 * Vw, 0.5 * Vw, 25.0, tr != nullptr, lane,
                                [&](int g, const SearchRes& r, bool before_first) {
                                    if (before_first && r.dis_lng > 25) first_g = g;
                                    if (tr) put_slot(&tr->sweep[(g / K) * DP_MAX_SWEEP + (g % K)], r, (none_yet && before_first) ? 1 : 2, lane);
                                }, DP_PRUNE_SWEEP ? hmaxF : -1.f, hminF, dnF, oid, relmask);
                            if (sweep_pick < 0 && first >= 0) sweep_pick = first_g;
                        }
                    } else {
                        for (int u = 0; u < shifted && (sweep_pick < 0 || tr); ++u) {   // one candidate at a time (N > 16)
                            const int g = dp_sweep_g(u, K);
                            const double cd = dp_sweep_offset(g, K);
                            float hbC, dmC;
                            dg_bounds(m, gl, cd, -0.5 * Vw, 0.5 * Vw, &hbC, &dmC);
                            const SearchRes s = dp_search_cold(slice_src(m, F.base, 1, F.P, cd), mx, my, ox, oy, N, lm, -0.5 * Vw, 0.5 * Vw, sm, lane, hbC, dmC);
                            const bool before = sweep_pick < 0;
                            put_slot(tr ? &tr->sweep[(g / K) * DP_MAX_SWEEP + (g % K)] : nullptr, s, before ? 1 : 2, lane);
                            if (before && s.dis_lng > 25) sweep_pick = g;
                        }
                    }
                    {
                        const int scored = sweep_pick < 0 ? total : sweep_pick + 1;        // what the reference evaluates
                        n_traj += scored; pts += scored * F.P;
                        if (tr && total > 0) {                                          // L0 and R0: copies of the F region slot
                            __syncwarp();
                            if (lane == 0) {
                                dp_search_slot s0 = tr->region[0];
                                s0.evaluated = 1; tr->sweep[0] = s0;
                                s0.evaluated = (uint8_t)(K < scored ? 1 : 2); tr->sweep[DP_MAX_SWEEP] = s0;
                            }
                        }
                    }
                    DBG_MARK(0, 6);
                    if (sweep_pick >= 0) {
                        const int sd = sweep_pick / K;
                        cur.behavior = sd == 0 ? 4 : 5; cur.target = lane_cur; cur.light = sd == 0 ? 1 : 2;
                        cur.obsavoid = true; cur.dlg = sd == 0 ? 11 : 12;
                    }
                } else { cur.behavior = 1; cur.target = lane_cur; cur.light = 0; cur.dlg = 1; }
            } else {
                if (c.obsavoid_status == 0) { cur.behavior = 1; cur.target = lane_cur; cur.light = 0; cur.dlg = 1; }
                else {
                    c.no_obsavoid_time++;
                    if (c.no_obsavoid_time > 3) { cur.behavior = 1; cur.target = lane_cur; cur.light = 0; cur.dlg = 1; cur.obsavoid = false; }
                }
                cur.dlg = 1;
            }
        } else {                                            // :1012-1772
            c.no_obsavoid_time = 0;
            c.obsavoid_time = 0;
            if (!cur.lanechg) {
                if (navi != 0) {                            // :1021-1144
                    if (navi == 1) {
                        if (lanechg == 1 || lanechg == 3) {
                            cur.dlg = 2;
                            if (cur.light != 1) { cur.light = 1; c.leftlight_time = 0; }
                            c.leftlight_time += period;
                            if (((gLF > gF + 10) || (gLF > 40)) && gLR > 15 && c.leftlight_time > 2000) {
                                cur.behavior = 2; cur.target = lane_cur - 1; cur.lanechg = true;
                            } else DP_KEEP(true);
                        } else { DP_KEEP(true); cur.dlg = 4; }
                    } else if (navi == 2) {
                        if (lanechg == 2 || lanechg == 3) {
                            cur.dlg = 3;
                            if (cur.light != 2) { cur.lanechg = true; c.rightlight_time = 0; }   // sic: lanechg_status = 2 (:1094)
                            c.rightlight_time += period;
                            if (((gRF > gF + 10) || (gRF > 40)) && gRR > 15 && c.rightlight_time >= 2000) {
                                cur.behavior = 3; cur.target = lane_cur + 1; cur.lanechg = true;
                            } else DP_KEEP(true);
                        } else { DP_KEEP(true); cur.dlg = 4; }
                    }
                } else {                                    // :1146-1757
                    if (gF < (2 * 10 + 5)) {
                        c.frontobs_time++;
                        if (c.frontobs_time > 2) {
                            c.frontobs_time = 3;
                            bool has_m1 = false, has_p1 = false;    // exit-lane list contains lane-1 / lane+1
                            for (int i = 0; i < DP_LANESUM && h.out_lane_no[i] != 0; ++i) {
                                if (h.out_lane_no[i] == lane_cur - 1) has_m1 = true;
                                if (h.out_lane_no[i] == lane_cur + 1) has_p1 = true;
                            }
                            if (lanechg == 1) {             // :1157-1294
                                if (lane_cur > 1) {
                                    cur.dlg = 5;
                                    const bool no_back = !has_m1;
                                    bool chg = false;
                                    if (no_back) {
                                        if (run_exceeds(m, sm, gl, id, 0, 60.0, lane)) {
                                            chg = true;
                                            if (z_light != 1) { z_light = 1; c.leftlight_time = 0; }
                                            c.leftlight_time += period;
                                            if (c.leftlight_time > 2000) c.leftlight_time = 2000;
                                        } else z_light = 0;
                                    } else {
                                        if (run_exceeds(m, sm, gl, id, 1, 15.0, lane)) {
                                            chg = true;
                                            if (cur.light != 1) { cur.light = 1; c.leftlight_time = 0; }
                                            c.leftlight_time += period;
                                            if (c.leftlight_time > 2000) c.leftlight_time = 2100;
                                        } else cur.light = 0;
                                    }
                                    if (chg && gLF > gF + 10 && gLR > 10 && c.leftlight_time > 1500) {
                                        c.frontobs_time = 0; cur.behavior = 2; cur.target = lane_cur - 1; cur.lanechg = true;
                                    } else DP_KEEP(true);
                                } else DP_KEEP(true);
                            } else if (lanechg == 2) {      // :1296-1424
                                if (lane_cur < lane_sum) {
                                    cur.dlg = 6;
                                    const bool no_back = !has_m1;                     // sic (:1307)
                                    bool chg = false;
                                    if (run_exceeds(m, sm, gl, id, 1, no_back ? 50.0 : 10.0, lane)) {
                                        chg = true;
                                        const int want = no_back ? 2 : 1;
                                        if (cur.light != want) { cur.light = want; c.leftlight_time = 0; }
                                        c.leftlight_time += period;
                                        if (c.leftlight_time > 2000) c.leftlight_time = 2000;
                                    }
                                    if (chg && gRF > gF + 10 && gRR > 10 && c.leftlight_time > 1500) {
                                        c.frontobs_time = 0; cur.behavior = 3; cur.target = lane_cur + 1; cur.lanechg = true;
                                    } else DP_KEEP(true);
                                } else DP_KEEP(true);
                            } else if (lanechg == 3) {      // :1426-1738
                                const bool nb_left = !has_m1, nb_right = !has_p1;
                                bool left_ok = false, right_ok = false;
                                if (lane_cur > 1) left_ok = run_exceeds(m, sm, gl, id, nb_left ? 1 : 2, nb_left ? 50.0 : 10.0, lane);
                                if (lane_cur < lane_sum) right_ok = run_exceeds(m, sm, gl, id, 1, nb_right ? 50.0 : 10.0, lane);
                                if (left_ok && !nb_left) {                          // :1545-1594
                                    if (!cur.lanechg) { cur.light = 1; c.leftlight_time = 0; }
                                    DP_TICK;
                                    if (gLF > gF + 10 && gLR > 10 && c.leftlight_time > 2000) {
                                        c.frontobs_time = 0; cur.behavior = 2; cur.target = lane_cur - 1; cur.lanechg = true;
                                    } else DP_KEEP(true);
                                } else if (right_ok && !nb_right) {                 // :1596-1636
                                    if (cur.light != 2) { cur.light = 2; c.leftlight_time = 0; }
                                    DP_TICK;
                                    if (gRF > gF + 10) {
                                        if (gRR > 10 && c.leftlight_time > 2000) {
                                            c.frontobs_time = 0; cur.behavior = 3; cur.target = lane_cur + 1; cur.lanechg = true;
                                        } else DP_KEEP(false);
                                    }
                                } else if (left_ok) {                               // :1638-1686
                                    if (cur.light != 1) { cur.lanechg = true; c.leftlight_time = 0; }   // sic (:1642)
                                    DP_TICK;
                                    if (gLF > gF + 10 && gLR > 10 && c.leftlight_time > 2000) {
                                        c.frontobs_time = 0; cur.behavior = 2; cur.target = lane_cur - 1; cur.lanechg = true;
                                    } else DP_KEEP(false);
                                } else if (right_ok) {                              // :1688-1730
                                    if (cur.light != 2) { cur.light = 2; c.leftlight_time = 0; }
                                    DP_TICK;
                                    if (gRF > gF + 10) {
                                        if (gRR > 10 && c.leftlight_time > 2000) {
                                            c.frontobs_time = 0; cur.behavior = 3; lane_cur = 1; cur.target = 1; cur.lanechg = true;   // sic (:1712)
                                        } else DP_KEEP(false);
                                    }
                                } else DP_KEEP(true);
                            }
                        } else DP_KEEP(true);               // :1741-1746
                    } else { c.frontobs_time = 0; cur.dlg = 8; DP_KEEP(true); }
                }
            } else {                                        // lane change in progress, :1760-1771
                cur.dlg = 9;
                if (cur.target == lane_cur) { cur.lanechg = false; cur.light = 0; }
                cur.behavior = his_behavior; cur.target = his_target; cur.light = his_light;
            }
        }
        (void)z_light;
        // ---- SpeedDecision / RefPath / write-back (Decision.cpp:1781-1816, 307-313) + thread-loop tail (:187-201) ----
        v_exp = (cur.behavior == 4 || cur.behavior == 5) ? 5 : 10;
        rp_n0 = (cur.behavior == 2) ? (side == 1 ? NF.P : 0) : (cur.behavior == 3) ? (side == 2 ? NF.P : 0) : F.P;   // only its length is consumed at pos 0
        d_behavior = cur.behavior; d_target = cur.target;
        if (lane == 0) {                                    // decision half of the carry and of the record is final: store it now
            cg->leftlight_time = c.leftlight_time; cg->rightlight_time = c.rightlight_time; cg->velocity_expect = v_exp;
            cg->obsavoid_time = c.obsavoid_time; cg->no_obsavoid_time = c.no_obsavoid_time; cg->frontobs_time = c.frontobs_time;
            cg->behavior = (uint16_t)cur.behavior; cg->target_roadnum = h.road_num; cg->target_lanenum = (uint16_t)cur.target;
            cg->light_status = (uint16_t)cur.light; cg->behavior_to_dlg = (uint16_t)cur.dlg;
            cg->his_behavior = (uint16_t)cur.behavior; cg->his_target_lanenum = (uint16_t)cur.target; cg->his_light_status = (uint16_t)cur.light;
            cg->lanechg_status = cur.lanechg; cg->obsavoid_status = cur.obsavoid;
            out->velocity_expect = v_exp;
            out->behavior = (uint16_t)cur.behavior; out->target_roadnum = h.road_num; out->target_lanenum = (uint16_t)cur.target;
            out->light = (uint16_t)cur.light; out->behavior_to_dlg = (uint16_t)cur.dlg; out->sweep_index = (int16_t)sweep_pick;
        }
    } else if (pos == 1 || pos == 2) {
        // =================== PreStubDecision / StubDecision (Decision.cpp:323-486) ===================
        junction_recipe(m, h, rp_base0, rp_n0, rp_base1, rp_n1);
        const SearchRes s = dp_search_cold(junction_src(m, rp_base0, rp_n0, rp_base1, rp_n1), mx, my, ox, oy, N, lm, -0.5 * Vw, 0.5 * Vw, sm, lane);
        ++n_traj; pts += rp_n0 + rp_n1;
        put_slot(tr ? &tr->junction : nullptr, s, 1, lane);
        int dlg;
        if (s.dis_lng < 13) {
            const double v = s.dis_lng - 3;
            v_exp = v > 0 ? v : 0;
            dlg = 13;
        } else { v_exp = 10; dlg = 1; }
        const int light = (h.stub_attribute == 3) ? 1 : h.stub_attribute;
        d_behavior = 1; d_target = h.lane_num;
        if (lane == 0) {                                    // members the junction functions write (:394-399) + thread-loop tail
            cg->velocity_expect = v_exp; cg->behavior_to_dlg = (uint16_t)dlg; cg->light_status = (uint16_t)light;
            cg->behavior = 1; cg->target_roadnum = h.road_num; cg->target_lanenum = h.lane_num;
            cg->his_behavior = 1; cg->his_light_status = (uint16_t)light; cg->his_target_lanenum = h.lane_num;
            out->velocity_expect = v_exp; out->behavior = 1; out->target_roadnum = h.road_num; out->target_lanenum = h.lane_num;
            out->light = (uint16_t)light; out->behavior_to_dlg = (uint16_t)dlg; out->sweep_index = -1;
        }
    } else {
        // no decision function runs for other pos values (Decision.cpp:183): members keep their values
        d_behavior = cg->behavior; d_target = cg->target_lanenum; v_exp = cg->velocity_expect;
        if (lane == 0) {
            cg->his_behavior = cg->behavior; cg->his_light_status = cg->light_status; cg->his_target_lanenum = cg->target_lanenum;
            out->velocity_expect = v_exp; out->behavior = cg->behavior; out->target_roadnum = cg->target_roadnum;
            out->target_lanenum = cg->target_lanenum; out->light = cg->light_status; out->behavior_to_dlg = cg->behavior_to_dlg;
            out->sweep_index = -1;
        }
    }
    DBG_T(0);
    if (PHASE == 1 && tr && lane == 0) tr->refpath_len = (uint16_t)(rp_n0 + rp_n1);
    if (PHASE == 1) {                                       // hand the counters over and stop: the Planning launch follows
        if (lane == 0) {
            out->n_traj = (uint16_t)n_traj;
            if (tr) { tr->ub_hits = (uint16_t)ub; tr->pts_scored = (uint32_t)pts; }
        }
        DBG_END(0, n_traj);
        if (io.done) dp_publish(io.done + scene, io.epoch, lane);   // (the scene's Planning warp goes on; what follows is off its path)
        if (io.n_fwd) {
#pragma unroll
            for (int k = 0; k < DP_MAX_MIRRORS; ++k)
                if (k < io.n_fwd) reinterpret_cast<uint32_t*>(io.fwd_dst[k] + scene)[lane] = fwd_w;
        }
        if (io.flag_mode == 1 && io.tally2) {               // deferred gather: every forwarded record is out when the last Decision warp retires
            __threadfence(); __syncwarp();                  // (every lane: its forwarded words before the tally)
            // ... and that warp stays until every rank's flag of that step is here: the pair of launches is complete only when the
            // gathered buffer of the step before is (the Planning half needs no tally for it)
            if (lane == 0 && atomicAdd(io.tally2, 1u) == io.tally_n - 1u) dg_complete(io.tally2, io, true, false);
        }
        return;
    }
    // ================================ Planning thread iteration ================================
    // last_Bpoints (Planning.cpp:6) -> sm.plan by one TMA bulk copy; the staging area of the decision half is free now and
    // the copy lands while the aim point is searched
    __syncwarp();
    dp_bulk_prefetch(sm.plan, lastp, DP_PATH_POINTS * (uint32_t)sizeof(double2), &sm.mbar, lane);
    const int plan_his_behavior = dp_l2(&cg->plan_his_behavior), carried_near_id = dp_l2(&cg->path_near_id), plan_count = dp_l2(&cg->plan_count);
    double aim_x = dp_l2(&cg->aim_x), aim_y = dp_l2(&cg->aim_y), aim_dir = dp_l2(&cg->aim_dir);
    int aim_id = dp_l2(&cg->aim_id);
    // ---- Calculate_aim_dis (Planning.cpp:242-290), FLOAT faraim_dis ----
    float faraim = 0.f;
    if (pos == 0) {
        faraim = (float)((h.velocity / 3.6) * 5 + 4);
        if (faraim > p.road_faraim_max) faraim = (float)p.road_faraim_max;
        else if (faraim < p.road_faraim_min) faraim = (float)p.road_faraim_min;
    } else if (pos == 1) faraim = (float)p.pre_inter_faraim;
    else if (pos == 2) faraim = (float)p.inter_faraim;
    if (tr && lane == 0) tr->faraim_dis = faraim;
    // ---- SearchAimPoint (Planning.cpp:303-583) ----
    if (pos == 0) {
        const int cur_id = h.id[lane_n - 1], cur_sum = m.lane_pt_off[gl + 1] - m.lane_pt_off[gl];
        int left_id = 0, left_sum = 0, right_id = 0, right_sum = 0;
        if (lane_n > 1) { left_id = h.id[lane_n - 2]; left_sum = m.lane_pt_off[gl] - m.lane_pt_off[gl - 1]; }
        if (lane_n < lane_sum) { right_id = h.id[lane_n]; right_sum = m.lane_pt_off[gl + 2] - m.lane_pt_off[gl + 1]; }
        int wl = -1, wfrom = 0, wto = 0, fb_gl = gl, fb_idx = 0, fb_id = 0;   // lane to walk, fallback point
        if (d_target == lane_n) {
            if (d_behavior == 1) { wl = gl; wfrom = cur_id; wto = cur_sum - 1; fb_gl = gl; fb_idx = cur_sum - 1; fb_id = cur_sum - 1; }
        } else {
            if (d_behavior == 2) {
                if (lane_n > 1) { wl = gl - 1; wfrom = left_id; wto = left_sum - 1; fb_gl = gl; fb_idx = left_sum - 2; fb_id = left_sum - 1; }
            } else if (d_behavior == 3) {
                if (lane_n < lane_sum) { wl = gl + 1; wfrom = right_id; wto = left_sum - 1; fb_gl = gl + 1; fb_idx = right_sum - 1; fb_id = right_sum - 1; }
                else if (right_id < left_sum - 1) ++ub;
            }
        }
        if (wl >= 0 && wfrom < wto) {
            const int woff = m.lane_pt_off[wl], wn = m.lane_pt_off[wl + 1] - woff;
            int hit = -1;
            bool walk = true;
            if (wfrom < 0) { ++ub; walk = false; }
            if (wto > wn - 1) { ++ub; wto = wn - 1; if (wfrom >= wto) walk = false; }
            // "first point whose accumulated arclength - 4 exceeds faraim" asked of the prefix table (dp_group.cuh, P6): binary
            // search inside the index window the segment-length bounds allow; the exact loop below only runs when the decision at
            // the hit (or at the last point) falls inside the rounding bracket of the table
            bool table_done = false;
            if (walk) {
                const int cnt = wto - wfrom;
                const double far = (double)faraim;
                const double* cp = m.cump + woff + wfrom;
                const double c0 = cp[0], ce = m.lane_cerr[wl], err = ce > 0.0 ? ce + 1e-9 : 0.0;
                const double tgt = far + 4.0;
                const float hmx = m.lane_hmax[wl], hmn = m.lane_hmin[wl];
                int lo = (int)((float)tgt / hmx) - 2, hi = (hmn > 1e-6f) ? (int)((float)tgt / hmn) + 3 : cnt - 1;
                if (lo < 0) lo = 0;
                if (hi > cnt - 1) hi = cnt - 1;
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
                    if (err > 0.0 && first_def > 0 && (cp[first_def] - c0) - 4.0 >= far - err) exact_loop = true;
                } else if (hi < cnt - 1) exact_loop = true;
                else if (err > 0.0 && cnt > 0 && (cp[cnt] - c0) - 4.0 >= far - err) exact_loop = true;
                if (!exact_loop) { table_done = true; hit = (first_def <= hi) ? wfrom + first_def : -1; }
            }
            if (walk) {
                double sum = 0.0;
                for (int i0 = wfrom; i0 < wto && hit < 0 && !table_done; i0 += DP_SCR) {
                    const int cnt = min(DP_SCR, wto - i0);
                    __syncwarp();
                    for (int j = lane; j < cnt; j += 32) sm.scr[j] = m.lenp[woff + i0 + j];
                    dp_pad_scr(sm, cnt, lane);
                    __syncwarp();
                    const SeqHit hq = dp_seq_first(sm, cnt, sum, 4.0, (double)faraim);
                    if (hq.k >= 0) hit = i0 + hq.k;
                    sum = hq.acc;
                }
                if (hit >= 0) {
                    aim_x = m.x[woff + hit]; aim_y = m.y[woff + hit]; aim_dir = m.dir[woff + hit]; aim_id = hit;
                } else {
                    const int offb = m.lane_pt_off[fb_gl], nb = m.lane_pt_off[fb_gl + 1] - offb;
                    int fi = fb_idx;
                    if (fi < 0 || fi >= nb) { ++ub; fi = fi < 0 ? 0 : nb - 1; }
                    aim_x = m.x[offb + fi]; aim_y = m.y[offb + fi]; aim_dir = m.dir[offb + fi]; aim_id = fb_id;
                }
            }
        }
    } else if (pos == 1 || pos == 2) {
        const Src rv = junction_src(m, rp_base0, rp_n0, rp_base1, rp_n1);
        const int n = rp_n0 + rp_n1;
        double sum = 0.0;
        int hit = -1;
        for (int i0 = 0; i0 < n - 1 && hit < 0; i0 += DP_SCR) {
            const int cnt = min(DP_SCR, n - 1 - i0);
            __syncwarp();
            for (int j = lane; j < cnt; j += 32) {
                const double2 a = dp_src_point(rv, i0 + j), b = dp_src_point(rv, i0 + j + 1);
                sm.scr[j] = dp_dist_plain(a.x, a.y, b.x, b.y);
            }
            dp_pad_scr(sm, cnt, lane);
            __syncwarp();
            const SeqHit hq = dp_seq_first(sm, cnt, sum, 4.0, (double)faraim);
            if (hq.k >= 0) hit = i0 + hq.k;
            sum = hq.acc;
        }
        if (hit >= 0) {
            const double2 a = dp_src_point(rv, hit);
            aim_x = a.x; aim_y = a.y;
            if ((size_t)hit < (size_t)n - 4) {
                const double2 b = dp_src_point(rv, hit + 2);
                aim_dir = dp_heading(a.x, a.y, b.x, b.y, p.epsilon, p.pi);
            } else {
                int ia = hit - 2; if (ia < 0) { ++ub; ia = 0; }
                const double2 b = dp_src_point(rv, ia);
                aim_dir = dp_heading(b.x, b.y, a.x, a.y, p.epsilon, p.pi);
            }
            aim_id = hit;
        } else if (n - 1 > 0) {
            int ia = n - 3; if (ia < 0) { ++ub; ia = 0; }
            const double2 e = dp_src_point(rv, n - 1), b = dp_src_point(rv, ia);
            aim_x = e.x; aim_y = e.y;
            aim_dir = dp_heading(b.x, b.y, e.x, e.y, p.epsilon, p.pi);
            aim_id = n - 1;
        }
    }
    DBG_T(1);
    dp_bulk_wait(&sm.mbar);
    DBG_T(2);
    // ---- InitialPlanning on the first cycle (Planning.cpp:124-128) ----
    bool plan_dirty = false;
    const bool first = (plan_count == 0);
    if (first) {
        dp_bezier_to_plan(sm, h.x, h.y, h.dir, aim_x, aim_y, aim_dir, lane);
        plan_dirty = true;
    }
    // ---- GetVhclLocalState (Planning.cpp:623-676) on last_Bpoints ----
    const int mi = dp_nearest_plain(sm.plan, DP_PATH_POINTS, h.x, h.y, lane);   // nearest of the 200 points (Planning.cpp:640-648)
    const int near_id = (mi == 0x7fffffff) ? carried_near_id : mi;
    const int front_id = near_id + 8;
    int idx = (near_id == 199) ? near_id - 1 : near_id;
    if (idx < 0 || idx > 198) { ++ub; idx = idx < 0 ? 0 : 198; }
    const double2 pt = sm.plan[idx], pn = sm.plan[idx + 1];
    const double lat = dp_lat_dis(h.x, h.y, pt.x, pt.y, pn.x, pn.y, p.epsilon);
    double remain;
    {
        const int f0 = max(front_id, 0);
        if (front_id < 0) ++ub;
        const int cnt = max(0, 199 - f0);
        __syncwarp();
        for (int j = lane; j < cnt; j += 32) { const double2 a = sm.plan[f0 + j], b = sm.plan[f0 + j + 1]; sm.scr[j] = dp_dist_plain(b.x, b.y, a.x, a.y); }
        dp_pad_scr(sm, cnt, lane);
        __syncwarp();
        remain = dp_seq_sum(sm, cnt, 0.0);
    }
    const double dir_err = dp_angle_err(dp_heading(pt.x, pt.y, pn.x, pn.y, p.epsilon, p.pi), h.dir);
    DBG_T(3);
    // ---- UpdatePlanJudge (Planning.cpp:797-832) ----
    bool afresh = true;
    int cause = 0;
    if (plan_his_behavior != d_behavior) cause = 1;
    else if (fabs(lat) > 0.2) cause = 2;
    else if (fabs(dir_err) > 45) cause = 3;
    else if (pos == 0 && remain < p.road_remain_distance) cause = 4;
    else if (pos != 0 && remain < p.inter_remain_distance) cause = 4;
    else afresh = false;
    // ---- CalculateRadius reads the PREVIOUS path (Planning.cpp:199, 1000-1019): before overwriting ----
    double radius;
    {
        int ia = near_id, ib = (near_id + front_id) / 2, ic = front_id;
        if (ia < 0 || ia > 199) { ++ub; ia = ia < 0 ? 0 : 199; }
        if (ib < 0 || ib > 199) { ++ub; ib = ib < 0 ? 0 : 199; }
        if (ic < 0 || ic > 199) { ++ub; ic = ic < 0 ? 0 : 199; }
        const double2 A = sm.plan[ia], B = sm.plan[ib], Fp = sm.plan[ic];
        const double d1 = dp_dist_plain(A.x, A.y, B.x, B.y), d2 = dp_dist_plain(B.x, B.y, Fp.x, Fp.y), d3 = dp_dist_plain(A.x, A.y, Fp.x, Fp.y);
        const double dd = d1 * d1 + d2 * d2 - d3 * d3;
        const double cosA = dd / (2 * d1 * d2);
        const double sinA = sqrt(1 - cosA * cosA);
        radius = (sinA < 0.001) ? 1000 : 0.5 * d3 / sinA;
    }
    if (lane == 0) {                                        // local-state half of the record and of the carry is final
        out->path_lat_dis = lat; out->path_dir_err = dir_err; out->remain_dis = remain; out->radius = radius;
        out->aim_x = aim_x; out->aim_y = aim_y; out->aim_dir = aim_dir; out->aim_id = aim_id;
        out->afresh_cause = (uint16_t)cause; out->afresh_planning = afresh;
        out->path_near_id = (int16_t)near_id; out->path_front_near_id = (int16_t)front_id;
        cg->aim_x = aim_x; cg->aim_y = aim_y; cg->aim_dir = aim_dir; cg->aim_id = aim_id; cg->path_near_id = near_id;
        cg->plan_his_behavior = d_behavior;                 // history update of Planning.cpp:216
        uint8_t cnt = (uint8_t)(plan_count + 1);            // BYTE count of CPlanningThread (Planning.cpp:219-223)
        if (cnt % 100 == 1) cnt = 1;
        cg->plan_count = cnt;
        out->cnt = (uint8_t)(plan_count % 100);
    }
    // ---- PathPlanning (Planning.cpp:845-877) or reuse (:142-146): road_points -> sm.plan ----
    if (afresh) {
        plan_dirty = true;
        if (pos == 0) {
            // the first-cycle Bezier above used the same two poses: identical points, nothing to redo
            if (!first) dp_bezier_to_plan(sm, h.x, h.y, h.dir, aim_x, aim_y, aim_dir, lane);
        } else if (pos == 1 || pos == 2) {
            int n = aim_id;
            if (n > DP_PATH_POINTS) { ++ub; n = DP_PATH_POINTS; }
            if (n > rp_n0 + rp_n1) { ++ub; n = rp_n0 + rp_n1; }
            dp_mean_points_to_plan(sm, junction_src(m, rp_base0, rp_n0, rp_base1, rp_n1), n, lane);
        } else {
            __syncwarp();
            for (int i = lane; i < DP_PATH_POINTS; i += 32) sm.plan[i] = make_double2(0.0, 0.0);
            __syncwarp();
        }
    }                                                       // else: road_points = last_Bpoints, already in sm.plan
    DBG_T(4);
    // ---- local path collision (Planning.cpp:152-168): rem_path is a window of sm.plan ----
    const int s0 = max(near_id, 0);
    Src rem = dp_src_run(sm.plan + s0, 1, DP_PATH_POINTS - s0);
    rem.q_off = s0;
    // pruning bounds of the local path (FP32, rounded outwards): longest / shortest segment, largest difference of consecutive
    // segment vectors (|u/|u| - w/|w|| <= |u - w| / hmin bounds the change of direction)
    float hbL = 0.f, dmL = 0.f;
    if (DP_PRUNE_LOCAL) {                                   // (the warp reductions below are never dead code to the compiler: keep them out when unused)
        float hmx = 0.f, hmn = __int_as_float(0x7f800000), dmx = 0.f;
        for (int j = s0 + lane; j < DP_PATH_POINTS - 1; j += 32) {
            const double2 a = sm.plan[j], b = sm.plan[j + 1];
            const float ux = (float)(b.x - a.x), uy = (float)(b.y - a.y);
            const float l2 = ux * ux + uy * uy;
            hmx = fmaxf(hmx, l2); hmn = fminf(hmn, l2);
            if (j + 2 < DP_PATH_POINTS) {
                const double2 c = sm.plan[j + 2];
                const float ex = (float)(c.x - b.x) - ux, ey = (float)(c.y - b.y) - uy;
                dmx = fmaxf(dmx, ex * ex + ey * ey);
            }
        }
        hmx = __uint_as_float(__reduce_max_sync(DP_FULL, __float_as_uint(hmx)));   // (non-negative floats order like their bit patterns)
        hmn = __uint_as_float(__reduce_min_sync(DP_FULL, __float_as_uint(hmn)));
        dmx = __uint_as_float(__reduce_max_sync(DP_FULL, __float_as_uint(dmx)));
        hbL = sqrtf(hmx) * 1.0001f + 1e-4f;
        const float hmin = sqrtf(hmn) * 0.9999f - 1e-6f;
        const float delta = (hmin > 1e-6f) ? sqrtf(dmx) / hmin * 1.001f + 1e-4f : 2.0f;
        dmL = dg_dmax((double)(float)(-1.1), (double)(float)(1.1), hbL, delta, hmin);
    }
    const SearchRes ls = dp_search(rem, mx, my, ox, oy, N, lm, (double)(float)(-1.1), (double)(float)(1.1), sm, lane, DP_PRUNE_LOCAL ? hbL : 0.f, dmL);
    ++n_traj; pts += DP_PATH_POINTS - s0;
    put_slot(tr ? &tr->local : nullptr, ls, 1, lane);
    // ---- SpeedPlanning (Planning.cpp:888-990) ----
    double brake = 0.0, des_acc = 0.0;
    bool acc_flag = false;
    if (pos <= 2) {
        if (ls.found) {
            if (ls.dis_lng - 4 > 9) brake = 3 + (ls.dis_lng - 9) / (faraim - 9) * (v_exp - 3);
            else if (ls.dis_lng - 4 > 5) brake = 3;
            else { brake = 0; acc_flag = true; des_acc = -3; }
        } else brake = v_exp;
    }
    // ---- outputs (Planning.cpp:173-214) and history (:216-223) ----
    if (plan_dirty)                                         // the carried path only changes on (re)planning cycles
        for (int i = lane; i < DP_PATH_POINTS; i += 32) lastp[i] = sm.plan[i];
    if (path_xy)
        for (int i = lane; i < DP_PATH_POINTS; i += 32) {
            const double2 q = sm.plan[i];
            path_xy[(size_t)scene * 400 + i] = q.x; path_xy[(size_t)scene * 400 + DP_PATH_POINTS + i] = q.y;
        }
    if (path_ll) {
        for (int i = lane; i < DP_OUT_POINTS; i += 32) {
            const double2 q = sm.plan[2 * i];
            path_ll[(size_t)scene * 200 + i] = fma(q.y, p.k_lat, p.lat0);
            path_ll[(size_t)scene * 200 + DP_OUT_POINTS + i] = fma(q.x, p.k_lng, p.lng0);
        }
    }
    if (lane == 0) {
        out->mindist_lat = ls.dis_lat; out->mindist_lon = ls.dis_lng; out->brakespeed = brake; out->des_acc = des_acc;
        out->ob_index = (int16_t)ls.ob; out->ob_pathid = (uint16_t)ls.pathid; out->n_traj = (uint16_t)n_traj;
        out->ob_flag = ls.found; out->acc_flag = acc_flag;
#ifdef DP_DEBUG_CLOCK
        out->radius = (double)(clock64() - dbg_t0); out->des_acc = (double)dbg_t0;
        out->path_lat_dis = (double)dbg_t[0]; out->path_dir_err = (double)dbg_t[1]; out->remain_dis = (double)dbg_t[2];
        out->mindist_lat = (double)dbg_t[3]; out->mindist_lon = (double)dbg_t[4]; out->brakespeed = (double)dbg_t[5];
#endif
        if (tr) { tr->ub_hits = (uint16_t)ub; tr->pts_scored = (uint32_t)pts; }
    }
    DBG_END(1, n_traj);
    if (io.n_mirror) {                                      // mirrors: one coalesced 128-byte store each (pinned host / peer GPUs)
        __syncwarp();
        __threadfence_block();
        const uint32_t w = reinterpret_cast<const volatile uint32_t*>(out)[lane];
#pragma unroll
        for (int k = 0; k < DP_MAX_MIRRORS; ++k)             // (static indices: the parameter array stays in the constant bank)
            if (k < io.n_mirror) reinterpret_cast<uint32_t*>(io.mirror[k] + scene)[lane] = w;
    }
    // completion: the last warp of the launch tells the host (page-locked flag) and / or the peers.  Two copies of the same
    // sequence, one per way of launching: a launch call (io.tally set by the caller or for a gather) and a submitted cycle
    // (io.in_flag).  Written as one `if (io.tally)` block it costs the one-wave Planning half 24 B more stack and twice the
    // spill traffic: ptxas allocates registers differently.
    if (io.tally && !io.in_flag) {
        __threadfence();                                    // (every lane: its stores, the mirrors included, before the tally)
        __syncwarp();
        if (lane == 0 && atomicAdd(io.tally, 1u) == io.tally_n - 1u) dg_complete(io.tally, io, io.flag_mode == 0, true);
    }
    if (io.in_flag) {
        __threadfence();                                    // (every lane: its stores, the mirrors included, before the tally)
        __syncwarp();
        if (lane == 0) {
            if (io.tally && atomicAdd(io.tally, 1u) == io.tally_n - 1u) dg_complete(io.tally, io, io.flag_mode == 0, true);
        }
    }
}

// ---- reset carry to constructor state (Decision.cpp:8-29, Planning.cpp:8-11,62) ----
__global__ void dp_reset_kernel(dp_carry* carry, double2* last_path, int first, int count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    dp_carry c;
    memset(&c, 0, sizeof(c));
    c.behavior = 1; c.velocity_expect = 10; c.his_behavior = 1; c.plan_his_behavior = 1;
    carry[first + i] = c;
    double2* lp = last_path + (size_t)(first + i) * DP_PATH_POINTS;
    for (int k = 0; k < DP_PATH_POINTS; ++k) lp[k] = make_double2(0.0, 0.0);
}

// ---- map precompute: AoS points, per-point segment lengths (both idioms), unit right normal, per-lane pruning bounds ----
// lane_hmax[gl] >= every segment length of lane gl, lane_dnmax[gl] >= |nrm[i+1]-nrm[i]| over its segments (FP32, rounded up):
// the radii of the exactly pruned scan (dp_group.cuh).  Positive floats order like their bit patterns: atomicMax on the bits.
__global__ void dp_map_prep_kernel(const double* x, const double* y, const int32_t* lane_pt_off, int n_lanes, double2* xy, double2* nrm,
                                   double* lenp, double* lenf, float* lane_hmax, float* lane_hmin, float* lane_dnmax) {
    const int gl = blockIdx.x;
    if (gl >= n_lanes) return;
    const int off = lane_pt_off[gl], n = lane_pt_off[gl + 1] - off;
    float hm = 0.f, hl = 1e30f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double2 nn = make_double2(0.0, 0.0);
        double l = 0.0, lf = 0.0;
        const double2 a = make_double2(x[off + i], y[off + i]);
        if (i + 1 < n) {
            const double2 b = make_double2(x[off + i + 1], y[off + i + 1]);
            nn = dp_normal(a, b);
            l = dp_dist_plain(b.x, b.y, a.x, a.y);
            lf = sqrt(dp_sq2(b.x - a.x, b.y - a.y));
            hm = fmaxf(hm, (float)lf * 1.0001f + 1e-6f);
            hl = fminf(hl, (float)lf * 0.9999f);
        }
        xy[off + i] = a; nrm[off + i] = nn; lenp[off + i] = l; lenf[off + i] = lf;
    }
    atomicMax(reinterpret_cast<unsigned*>(lane_hmax + gl), __float_as_uint(hm));
    atomicMin(reinterpret_cast<unsigned*>(lane_hmin + gl), __float_as_uint(hl));
    __syncthreads();                                        // this block's normals are in memory (same block reads them back)
    float dm = 0.f;
    for (int i = threadIdx.x; i + 2 < n; i += blockDim.x) {
        const double2 a = nrm[off + i], b = nrm[off + i + 1];
        dm = fmaxf(dm, (float)sqrt(dp_sq2(b.x - a.x, b.y - a.y)) * 1.0001f + 1e-7f);
    }
    atomicMax(reinterpret_cast<unsigned*>(lane_dnmax + gl), __float_as_uint(dm));
}

// per lane, one thread per task: 0 = sequential prefix of lenp (+ the rounding bound of its differences), 1 / 2 = run ends
// of the lane-change attribute tests `attr == 1` / `attr & 1` (Decision.cpp:1179-1190 and siblings; dg_run_exceeds)
__global__ void dp_map_prep2_kernel(const double* lenp, const uint16_t* attr, const int32_t* lane_pt_off, int n_lanes, double* cump,
                                    double* lane_cerr, int32_t* run_end0, int32_t* run_end1) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int gl = t / 3, task = t - gl * 3;
    if (gl >= n_lanes) return;
    const int off = lane_pt_off[gl], n = lane_pt_off[gl + 1] - off;
    if (task == 0) {
        double acc = 0.0;
        bool dyadic = true;                                 // every term a multiple of 2^-20: partial sums in any order are exact
        for (int i = 0; i < n; ++i) {
            const double t = lenp[off + i];
            cump[off + i] = acc; acc += t;
            if (t * 1048576.0 != rint(t * 1048576.0)) dyadic = false;
        }
        lane_cerr[gl] = (dyadic && acc < 1073741824.0) ? 0.0 : 4.0 * (double)n * 0x1p-53 * acc + 1e-12;
    } else {
        int32_t* re = (task == 1) ? run_end0 : run_end1;
        if (n > 0) re[off + n - 1] = n - 1;
        for (int i = n - 2; i >= 0; --i) {
            const int a = attr[off + i + 1];
            const bool ok = (task == 1) ? (a == 1) : ((a & 1) != 0);
            re[off + i] = ok ? re[off + i + 1] : i;
        }
    }
}

// ---- fused gather: wait until every rank's flag of this step has arrived in MY gathered buffer (one thread) ----
__global__ void dp_gather_wait_kernel(const unsigned* flags, int world, unsigned step) { dg_wait_flags(flags, world, step); }

// ---- the group kernel (dp_group.cuh): one CTA = g scenes ----
template <int G, int TPB>
__global__ void __launch_bounds__(TPB, (G <= 8) ? 4 : 2)   // G 16: 2 CTAs x 256 threads x 128 regs; G 8: 4 CTAs/SM (TPB 128: 128 regs, TPB 256: 64 regs)
dp_group_kernel(DgMap m, dp_params p, int n_scenes, int g, const dp_scene_hdr* __restrict__ hdr, const double* __restrict__ obs_x,
                const double* __restrict__ obs_y, int max_obs, dp_carry* __restrict__ carry, double2* __restrict__ last_path,
                dp_plan_record* __restrict__ rec, dp_trace_record* __restrict__ trace, double* __restrict__ path_xy,
                double* __restrict__ path_ll, DpIo io) {
    extern __shared__ __align__(16) unsigned char dg_raw[];
    DgSmem<G>& sm = *reinterpret_cast<DgSmem<G>*>(dg_raw);
    const int first = blockIdx.x * g;
    if (first >= n_scenes) return;
    const int S = min(g, n_scenes - first);
    dg_group_cycle<G, TPB>(m, p, first, S, hdr, obs_x, obs_y, max_obs, carry, last_path, rec, trace, path_xy, path_ll, io, sm);
}

// ---- launchers (called from dp_api.cu) ----
// access-policy window over the map arena: every access inside it is "persisting" (kept in the L2 set-aside)
static void dp_l2_window(cudaLaunchAttribute& a, const DpLaunchCfg& lc) {
    a.id = cudaLaunchAttributeAccessPolicyWindow;
    a.val.accessPolicyWindow.base_ptr = lc.l2_base;
    a.val.accessPolicyWindow.num_bytes = lc.l2_bytes;
    a.val.accessPolicyWindow.hitRatio = 1.0f;
    a.val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    a.val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
}
void dp_launch_prepare(DpLaunchCfg& lc) {
    if (lc.attr_warp) return;                               // 196 of 256 KB as shared memory, the rest stays L1 (per context: no process-wide state)
    cudaFuncSetAttribute(dp_cycle_kernel<1, 4>, cudaFuncAttributePreferredSharedMemoryCarveout, DP_CARVEOUT);
    cudaFuncSetAttribute(dp_cycle_kernel<2, 4>, cudaFuncAttributePreferredSharedMemoryCarveout, DP_CARVEOUT);
    cudaFuncSetAttribute(dp_cycle_kernel<1, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, DP_CARVEOUT);
    cudaFuncSetAttribute(dp_cycle_kernel<2, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, DP_CARVEOUT);
    lc.attr_warp = true;
}
cudaError_t dp_launch_cycle(const DevMap& m, const dp_params& p, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                            int max_obs, dp_carry* carry, double2* last_path, dp_plan_record* rec, dp_trace_record* trace,
                            double* path_xy, double* path_ll, cudaStream_t st, const DpIo& io, DpLaunchCfg& lc) {
    if (n <= 0) return cudaSuccess;
    dp_launch_prepare(lc);
    // batches of at most one wave of 4-warp CTAs stay one wave; larger ones run one warp per CTA (see DP_MIN_BLOCKS)
    const bool wide = n <= lc.sm_count * DP_MIN_BLOCKS(4) * 4;
    const int wpb = wide ? 4 : 1;
    const int blocks = (n + wpb - 1) / wpb, threads = wpb * 32;
    DpIo io1 = io; io1.n_mirror = 0;                        // the records are final in the Planning half
    DpIo io2 = io;
    io1.flag_mode = io2.flag_mode = (io.n_fwd && io.tally2) ? 1 : 0;   // deferred gather: the Decision half forwards and raises the flags
    auto launch = [&](void (*kernel)(DevMap, dp_params, int, const dp_scene_hdr*, const double*, const double*, int, dp_carry*, double2*,
                                     dp_plan_record*, dp_trace_record*, double*, double*, DpIo),
                      const DpIo& hio, bool pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = 0; cfg.stream = st;
        cudaLaunchAttribute at[2];
        int na = 0;
        if (pdl) {
            at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[na].val.programmaticStreamSerializationAllowed = 1;
            ++na;
        }
        if (lc.l2_bytes) dp_l2_window(at[na++], lc);
        cfg.attrs = at; cfg.numAttrs = na;
        return cudaLaunchKernelEx(&cfg, kernel, m, p, n, hdr, ox, oy, max_obs, carry, last_path, rec, trace, path_xy, path_ll, hio);
    };
    cudaError_t e = launch(wide ? dp_cycle_kernel<1, 4> : dp_cycle_kernel<1, 1>, io1, false);
    if (e != cudaSuccess) return e;
    // the Planning half as a programmatic dependent launch WITHOUT a grid-wide dependency wait in the kernel: scenes hand over one
    // by one (dp_publish / dp_await), so Planning CTAs run in the slots the Decision launch frees while its tail finishes
    e = launch(wide ? dp_cycle_kernel<2, 4> : dp_cycle_kernel<2, 1>, io2, io.done != nullptr);
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}
cudaError_t dp_launch_gather_wait(const unsigned* flags, int world, unsigned step, cudaStream_t st) {
    dp_gather_wait_kernel<<<1, 1, 0, st>>>(flags, world, step);
    return cudaGetLastError();
}
// deferred gather, last step of a sequence: nobody launches another cycle to forward its records
__global__ void dp_gather_forward_kernel(const dp_plan_record* __restrict__ src, int n, DpIo io) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;    // one 16-byte piece per thread
    if (i >= n * 8) return;
    const uint4 w = __ldcg(reinterpret_cast<const uint4*>(src) + i);
#pragma unroll
    for (int k = 0; k < DP_MAX_MIRRORS; ++k)
        if (k < io.n_fwd) reinterpret_cast<uint4*>(io.fwd_dst[k])[i] = w;
}
// (the sequence of dg_complete without a tally or host flag, written out: the helper's unrolled flag loop takes 2 registers more here)
__global__ void dp_gather_raise_kernel(DpIo io) {           // (after the forward kernel in stream order: its stores are complete)
    __threadfence_system();
    for (int k = 0; k < io.n_peer_flag; ++k) asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(io.peer_flag[k]), "r"(io.flag_value) : "memory");
    dg_wait_flags(io.wait.flag, io.wait.n, io.wait.value);
}
cudaError_t dp_launch_gather_flush(const dp_plan_record* src, int n, const DpIo& io, cudaStream_t st) {
    dp_gather_forward_kernel<<<(n * 8 + 255) / 256, 256, 0, st>>>(src, n, io);
    dp_gather_raise_kernel<<<1, 1, 0, st>>>(io);
    return cudaGetLastError();
}
cudaError_t dp_launch_reset(dp_carry* carry, double2* last_path, int first, int count, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    dp_reset_kernel<<<(count + 127) / 128, 128, 0, st>>>(carry, last_path, first, count);
    return cudaGetLastError();
}
cudaError_t dp_launch_map_prep(const double* x, const double* y, const uint16_t* attr, const int32_t* lane_pt_off, int n_lanes, double2* xy,
                               double2* nrm, double* lenp, double* lenf, float* lane_hmax, float* lane_hmin, float* lane_dnmax, double* cump,
                               double* lane_cerr, int32_t* run_end0, int32_t* run_end1, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(lane_hmax, 0, (size_t)n_lanes * sizeof(float), st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(lane_dnmax, 0, (size_t)n_lanes * sizeof(float), st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(lane_hmin, 0x7f, (size_t)n_lanes * sizeof(float), st);   // 0x7f7f7f7f = 3.4e38: above every length
    if (e != cudaSuccess) return e;
    dp_map_prep_kernel<<<n_lanes, 256, 0, st>>>(x, y, lane_pt_off, n_lanes, xy, nrm, lenp, lenf, lane_hmax, lane_hmin, lane_dnmax);
    dp_map_prep2_kernel<<<(3 * n_lanes + 63) / 64, 64, 0, st>>>(lenp, attr, lane_pt_off, n_lanes, cump, lane_cerr, run_end0, run_end1);
    return cudaGetLastError();
}

// Group kernel launch.  cfg 0: 16 scenes x 256 threads per CTA, 2 CTAs per SM; cfg 1: 8 scenes x 128 threads, 4 CTAs per SM.
// Scenes per CTA: batches that fit one wave are spread evenly over the resident CTA slots (4096 scenes on 148 SMs: 14 per CTA,
// 293 of 296 slots); larger batches run full groups.
template <int G, int TPB>
static cudaError_t dp_launch_group_t(const DgMap& m, const dp_params& p, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                                     int max_obs, dp_carry* carry, double2* last_path, dp_plan_record* rec, dp_trace_record* trace,
                                     double* path_xy, double* path_ll, cudaStream_t st, const DpIo& io, int sm_count, bool& configured) {
    const size_t smem = sizeof(DgSmem<G>);
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(dp_group_kernel<G, TPB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        cudaFuncSetAttribute(dp_group_kernel<G, TPB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        configured = true;
    }
    const int per_sm = (G <= 8) ? 4 : 2;
    int g = (n + sm_count * per_sm - 1) / (sm_count * per_sm);
    if (g < 1) g = 1;
    if (g > G) g = G;
    const int blocks = (n + g - 1) / g;
    dp_group_kernel<G, TPB><<<blocks, TPB, smem, st>>>(m, p, n, g, hdr, ox, oy, max_obs, carry, last_path, rec, trace, path_xy, path_ll, io);
    return cudaGetLastError();
}
cudaError_t dp_launch_group(const DgMap& m, const dp_params& p, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy,
                            int max_obs, dp_carry* carry, double2* last_path, dp_plan_record* rec, dp_trace_record* trace,
                            double* path_xy, double* path_ll, cudaStream_t st, const DpIo& io, DpLaunchCfg& lc) {
    if (n <= 0) return cudaSuccess;
    const int cfg = lc.group_cfg, sm_count = lc.sm_count;
    if (cfg == 1) return dp_launch_group_t<8, 128>(m, p, n, hdr, ox, oy, max_obs, carry, last_path, rec, trace, path_xy, path_ll, st, io, sm_count, lc.attr_group[1]);
    if (cfg == 2) return dp_launch_group_t<8, 256>(m, p, n, hdr, ox, oy, max_obs, carry, last_path, rec, trace, path_xy, path_ll, st, io, sm_count, lc.attr_group[2]);
    return dp_launch_group_t<16, 256>(m, p, n, hdr, ox, oy, max_obs, carry, last_path, rec, trace, path_xy, path_ll, st, io, sm_count, lc.attr_group[0]);
}
