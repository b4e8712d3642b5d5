// csrc/dp_api.cu -- host side of the C ABI declared in include/dmpp_b200.h.
// Owns the device context: map tables (+ precomputed segment lengths / normals), per-scene
// carry and last-path arrays, pinned staging for the host-pointer entry points, two streams so
// that chunks of a large batch overlap H2D / kernel / D2H.  No CPU compute path exists here:
// every entry point either launches the CUDA kernels or returns an error.
#include <cuda_runtime.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <string>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <vector>
#include "dp_kernels.h"

static_assert(sizeof(dp_scene_hdr) == 128, "dp_scene_hdr layout");
static_assert(sizeof(dp_plan_record) == 128, "dp_plan_record layout");
static_assert(sizeof(dp_carry) == 128, "dp_carry layout");
static_assert(sizeof(dp_search_slot) == 24, "dp_search_slot layout");
static_assert(sizeof(dp_trace_record) == 608, "dp_trace_record layout");

namespace {
thread_local std::string g_err;
int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
    g_err = what;
    if (e != cudaSuccess) { g_err += ": "; g_err += cudaGetErrorString(e); }
    return code;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(DP_ERR_CUDA, #call, e_); } while (0)

const int kChunk = 32768;   // scenes per staged chunk of the host-pointer path
}  // namespace

struct dp_ctx {
    int device = 0;
    dp_params p;
    int max_scenes = 0, max_obs = 0;
    bool have_map = false;
    DgMap gmap;                                             // map tables + pruning bounds + prefix / run-end tables (both kernels)
    DpLaunchCfg lc;                                         // per-context launch state (dp_kernels.h)
    // predicted agent tracks (dp_set_tracks): constant-turn-rate parameters of every obstacle point, indexed by carry slot;
    // tracks_T == 0: static obstacles.  d_trk: the context's own copy for the host-pointer form ([3][max_scenes][max_obs])
    const double* trk_vx = nullptr; const double* trk_vy = nullptr; const double* trk_dth = nullptr;
    double* d_trk = nullptr;
    int tracks_T = 0;
    long long* d_timeline = nullptr;                        // DP_TIMELINE=1: phase stamps of the last group launch (dp_debug_timeline)
    int kernel = 0;                                         // 0: warp-per-scene kernel (dp_cycle.cu), 1: group kernel (dp_group.cuh); see dp_create
    std::vector<void*> map_allocs;
    dp_carry* d_carry = nullptr;
    double2* d_last = nullptr;
    cudaStream_t st[2] = {nullptr, nullptr};
    // staging, two sets
    int chunk = 0;
    dp_scene_hdr* d_hdr[2] = {nullptr, nullptr};  dp_scene_hdr* h_hdr[2] = {nullptr, nullptr};
    double* d_ox[2] = {nullptr, nullptr};         double* h_ox[2] = {nullptr, nullptr};
    double* d_oy[2] = {nullptr, nullptr};         double* h_oy[2] = {nullptr, nullptr};
    dp_plan_record* d_rec[2] = {nullptr, nullptr}; dp_plan_record* h_rec[2] = {nullptr, nullptr};
    dp_trace_record* d_trace[2] = {nullptr, nullptr};
    double* d_pxy[2] = {nullptr, nullptr};
    double* d_pll[2] = {nullptr, nullptr};
    long long launches = 0;
    // closed-loop episodes (dp_run_closed_loop_dev): world-step parameters, the capture stream, the cached episode graph and its key
    DpWorldOpts world;                                      // dp_world_set_params and the armed models (dp_world_set_metrics,
                                                            // dp_world_set_agent_model, dp_world_set_lane_change)
    DpV2xOpts v2x;                                          // dp_world_set_v2x: the V2X launch between cycle and world step
    cudaStream_t ep_stream = nullptr;
    cudaGraphExec_t ep_exec = nullptr;
    const void* ep_key[8] = {}; int ep_dims[3] = {-1, -1, -1};
    long long ep_launches = 0;
    int ep_graph = 1;                                       // DP_EPISODE_GRAPH=0: enqueue the launches directly
    int ep_last_graph = 0;
    // pipelined submit / wait: inputs of cycle k+1 cross PCIe on the copy stream while cycle k computes
    cudaStream_t cp[3] = {nullptr, nullptr, nullptr};       // one copy stream per input array: the three DMAs overlap
    cudaEvent_t in_ready[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
    unsigned long long submitted = 0, waited = 0;
    // overlapped launch of the two halves: per-scene hand-off flags and the epoch of the next cycle
    unsigned* d_done = nullptr;
    unsigned epoch = 0;
    // submitted cycles (dp_cycle_submit): no event or stream wait sits between the launches; inputs and completion are signalled
    // through flags instead
    unsigned* d_inflag = nullptr;                           // [2] "inputs of the cycle in staging set s are on the device"
    unsigned* d_tally = nullptr;                            // [2] finished Planning warps
    unsigned* h_done = nullptr;                             // [2] page-locked: the last Planning warp of a cycle stores its epoch here
                                                            // [2..3] page-locked source words of the in_flag copies
    unsigned wait_epoch[2] = {0, 0};
    // what the next cycle launch carries besides its own plumbing: the record mirrors (dp_set_record_mirrors) and the armed gather
    // (dp_gather_*: mirrors, peer flags, the folded wait, the deferred forward), mirror / fwd_dst indexed by carry slot (make_io)
    DpIo armed = {};
    bool deferred = false;                                  // armed by dp_gather_arm_deferred: one-shot
    dp_plan_record* last_rec = nullptr; int last_first = -1, last_n = 0;   // record array (device) and slot range of the last cycle launch
    unsigned* d_tally_g = nullptr;                          // [2]: launch tally, Decision-half tally of the deferred gather
};

namespace {
// launch plumbing of one cycle call: hand-off flags, then the caller's pinned record buffer (if any), the context's mirrors and
// armed gather offset by the first slot
DpIo make_io(dp_ctx* c, int first, dp_plan_record* host_rec) {
    DpIo io = c->armed;
    if (++c->epoch == 0) ++c->epoch;                        // (0 is what never-written flags hold)
    io.done = c->d_done + first; io.epoch = c->epoch;
    io.n_mirror = 0;
    if (host_rec) io.mirror[io.n_mirror++] = host_rec;
    for (int k = 0; k < c->armed.n_mirror; ++k) io.mirror[io.n_mirror++] = c->armed.mirror[k] + first;
    if (io.n_fwd && c->last_rec) {
        io.fwd_src = c->last_rec;
        for (int k = 0; k < io.n_fwd; ++k) io.fwd_dst[k] += first;
        io.tally2 = c->d_tally_g + 1;
    } else io.n_fwd = 0;
    return io;
}
// record mirrors or a gather armed for the next launch?
bool armed_any(const DpIo& a) { return a.n_mirror || a.n_peer_flag || a.wait.n || a.n_fwd; }
// bookkeeping of every cycle launch: remember its record array (the deferred gather of the NEXT launch forwards it) and drop the
// one-shot deferred state
struct LaunchDone {
    dp_ctx* c; dp_plan_record* rec; int first, n;
    ~LaunchDone() {
        c->last_rec = rec; c->last_first = first; c->last_n = n;
        if (c->deferred) { c->armed = {}; c->deferred = false; }
    }
};
// one cycle of n scenes (carry slots first ..) on stream st: the group kernel (dp_group.cuh), or the warp-per-scene kernel pair
// (dp_cycle.cu)
cudaError_t run_cycle(dp_ctx* c, int first, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy, dp_plan_record* rec,
                      dp_trace_record* trace, double* path_xy, double* path_ll, cudaStream_t st, DpIo io) {
    if (io.n_fwd && (first != c->last_first || n != c->last_n)) return cudaErrorInvalidValue;   // deferred gather: same slot range as the launch before
    LaunchDone done_{c, rec, first, n};
    const bool group = c->kernel == 1 || c->tracks_T > 0;  // (track tiles are only read by the group kernel)
    if (!io.tally) {
        // deferred gather on the warp kernel: the Decision half forwards, flags and waits by itself (tally2), the Planning half ends as
        // it does without a gather; otherwise the launch's last warp / CTA does it and needs the tally
        if (!group && io.n_fwd && io.tally2) io.tally_n = (unsigned)n;
        else if (io.n_peer_flag || io.wait.n) { io.tally = c->d_tally_g; io.tally_n = (unsigned)n; }
    }
    dp_carry* carry = c->d_carry + first;
    double2* last_path = c->d_last + (size_t)first * DP_PATH_POINTS;
    if (!group) {
        c->launches += 2;
        return dp_launch_cycle(c->gmap, c->p, n, hdr, ox, oy, c->max_obs, carry, last_path, rec, trace, path_xy, path_ll, st, io, c->lc);
    }
    if (c->tracks_T > 0) {
        const size_t tb = (size_t)first * c->max_obs;
        io.trk_vx = c->trk_vx + tb; io.trk_vy = c->trk_vy + tb; io.trk_dth = c->trk_dth + tb; io.trk_T = c->tracks_T;
    }
    io.timeline = (n <= 8192) ? c->d_timeline : nullptr;
    if (io.timeline) cudaMemsetAsync(c->d_timeline, 0, (size_t)8192 * 32 * 8, st);
    c->launches += 1;
    return dp_launch_group(c->gmap, c->p, n, hdr, ox, oy, c->max_obs, carry, last_path, rec, trace, path_xy, path_ll, st, io, c->lc);
}
}  // namespace

namespace {
bool is_pinned(const void* p, void** dev = nullptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (dev) *dev = a.devicePointer;                        // device-side alias of the pinned allocation (== p under UVA)
    return a.type == cudaMemoryTypeHost;
}
template <class T> int dev_alloc(T** p, size_t n) {
    cudaError_t e = cudaMalloc((void**)p, n * sizeof(T));
    if (e != cudaSuccess) return fail(DP_ERR_NOMEM, "cudaMalloc", e);
    return DP_OK;
}
int ensure_optional(dp_ctx* c, int which) {   // 0 trace, 1 path_xy, 2 path_ll: allocated on first use
    for (int s = 0; s < 2; ++s) {
        if (which == 0 && !c->d_trace[s]) { int r = dev_alloc(&c->d_trace[s], (size_t)c->chunk); if (r) return r; }
        if (which == 1 && !c->d_pxy[s]) { int r = dev_alloc(&c->d_pxy[s], (size_t)c->chunk * 400); if (r) return r; }
        if (which == 2 && !c->d_pll[s]) { int r = dev_alloc(&c->d_pll[s], (size_t)c->chunk * 200); if (r) return r; }
    }
    return DP_OK;
}
}  // namespace

namespace {
struct Tmp {
    std::vector<void*> v;
    ~Tmp() { for (void* p : v) cudaFree(p); }
    template <class T> T* put(const T* src, size_t n, cudaError_t& e) {
        T* d = nullptr;
        e = cudaMalloc((void**)&d, (n ? n : 1) * sizeof(T));
        if (e != cudaSuccess) return nullptr;
        v.push_back(d);
        if (src && n) e = cudaMemcpy(d, src, n * sizeof(T), cudaMemcpyHostToDevice);
        return d;
    }
};
std::vector<double2> interleave(const double* x, const double* y, size_t n) {
    std::vector<double2> v(n ? n : 1);
    for (size_t i = 0; i < n; ++i) v[i] = make_double2(x[i], y[i]);
    return v;
}
#define PUT(var, T, src, n) T* var = tmp.put<T>(src, n, e); if (e != cudaSuccess) return fail(DP_ERR_CUDA, "operator staging", e)

// Dense sweep: candidates that share an offset share their geometry (dp_ops.cu).  rows = distinct offsets (bit patterns),
// groups = distinct point counts of a row, ascending; cand_group[c] = group of candidate c (-1: fewer than 2 points).
struct SweepGroups {
    std::vector<double> row_off;
    std::vector<int32_t> row_gbeg, group_P, group_row, cand_group, group_first;   // group_first: lowest candidate index of the group
    int32_t first_nogroup = -1;                             // lowest candidate with fewer than 2 points
    std::vector<int32_t> row_info;                          // per row {first group, groups, longest horizon, base line}
};
SweepGroups build_sweep_groups(const int32_t* cand_line, const double* offset, const int32_t* n_pts, int n_cand, int n_base) {
    SweepGroups g;
    struct Key { int32_t line; uint64_t bits; int32_t P; };
    std::vector<Key> keyed((size_t)n_cand);                 // (base line, offset bits, P)
    for (int c = 0; c < n_cand; ++c) {
        uint64_t b; memcpy(&b, &offset[c], 8);
        keyed[c] = {cand_line ? cand_line[c] : 0, b, n_pts[c] < n_base ? n_pts[c] : n_base};
    }
    std::vector<int32_t> order((size_t)n_cand);
    for (int c = 0; c < n_cand; ++c) order[c] = c;
    std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
        const Key &x = keyed[a], &y = keyed[b];
        return x.line != y.line ? x.line < y.line : x.bits != y.bits ? x.bits < y.bits : x.P != y.P ? x.P < y.P : a < b;
    });
    g.cand_group.assign((size_t)n_cand, -1);
    g.row_gbeg.push_back(0);
    std::vector<int32_t> row_line;
    bool have_row = false; uint64_t cur_bits = 0; int32_t cur_P = -1, cur_line = -1;
    for (int32_t c : order) {
        const uint64_t b = keyed[c].bits; const int32_t P = keyed[c].P, line = keyed[c].line;
        if (P < 2) continue;
        if (!have_row || b != cur_bits || line != cur_line) {
            if (have_row) g.row_gbeg.push_back((int32_t)g.group_P.size());
            double off; memcpy(&off, &b, 8);
            g.row_off.push_back(off); row_line.push_back(line); have_row = true; cur_bits = b; cur_line = line; cur_P = -1;
        }
        if (P != cur_P) { g.group_P.push_back(P); g.group_row.push_back((int32_t)g.row_off.size() - 1); g.group_first.push_back(c); cur_P = P; }
        g.cand_group[c] = (int32_t)g.group_P.size() - 1;
        if (c < g.group_first.back()) g.group_first.back() = c;
    }
    for (int c = 0; c < n_cand; ++c) if (g.cand_group[c] < 0) { g.first_nogroup = c; break; }
    if (have_row) g.row_gbeg.push_back((int32_t)g.group_P.size());
    for (size_t r = 0; r + 1 < g.row_gbeg.size(); ++r) {
        const int32_t g0 = g.row_gbeg[r], ng = g.row_gbeg[r + 1] - g0;
        g.row_info.insert(g.row_info.end(), {g0, ng, ng > 0 ? g.group_P[(size_t)g0 + ng - 1] : 0, row_line[r]});   // (horizons ascend within a row)
    }
    return g;
}
}  // namespace

extern "C" {

const char* dp_last_error(void) { return g_err.c_str(); }

void dp_default_params(dp_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->vehicle_width = 1.8; p->epsilon = 1e-6; p->pi = 3.14159265358979323846;
    p->road_faraim_max = 60; p->road_faraim_min = 15; p->pre_inter_faraim = 20; p->inter_faraim = 15;
    p->road_remain_distance = 15; p->inter_remain_distance = 5;
    p->lat0 = 23.0; p->lng0 = 113.0; p->k_lat = 1.0 / 110574.0; p->k_lng = 1.0 / 102470.0;
    p->id_more = 8;
}

int dp_create(dp_ctx** out, int device, const dp_params* params, int max_scenes, int max_obs) {
    if (!out || max_scenes <= 0 || max_obs <= 0 || max_obs > 65535) return fail(DP_ERR_ARG, "dp_create: bad argument");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail(DP_ERR_CUDA, "dp_create: no CUDA device (this library has no CPU path)", e);
    if (device < 0 || device >= ndev) return fail(DP_ERR_ARG, "dp_create: device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(DP_ERR_CUDA, "dp_create: device is not sm_100-class (kernels are built for sm_100a only)");
    dp_ctx* c = new dp_ctx();
    c->device = device;
    if (params) c->p = *params; else dp_default_params(&c->p);
    c->max_scenes = max_scenes; c->max_obs = max_obs;
    if (const char* e = getenv("DP_EPISODE_GRAPH")) c->ep_graph = atoi(e) != 0;
    dp_world_default_params(&c->world.wp);
    dp_metrics_default_params(&c->world.mp);
    dp_agent_model_default_params(&c->world.amp);
    dp_lane_change_default_params(&c->world.lcp);
    // Kernel choice, from the measurements in profiles/README.md (round 2): the warp-per-scene kernel wins while a scene's
    // obstacles fit one warp pass (N < 32: 71 vs 96 us per 4096-scene cycle at N = 10); the group kernel, whose scans are flat
    // (trajectory, obstacle) lists with exact pruning, wins for crowded scenes (N = 200: 135 vs 212 us per 1024 junction scenes).
    c->kernel = (max_obs >= 32) ? 1 : 0;
    if (const char* e = getenv("DP_KERNEL")) c->kernel = (strcmp(e, "warp") == 0) ? 0 : (strcmp(e, "group") == 0) ? 1 : c->kernel;
    CK(cudaDeviceGetAttribute(&c->lc.sm_count, cudaDevAttrMultiProcessorCount, device));
    if (const char* e = getenv("DP_GROUP_CFG")) c->lc.group_cfg = atoi(e);
    if (const char* e = getenv("DP_TIMELINE")) {
        if (atoi(e)) { int rt = dev_alloc(&c->d_timeline, (size_t)8192 * 32); if (rt) { delete c; return rt; } cudaMemset(c->d_timeline, 0, (size_t)8192 * 32 * 8); }
    }
    c->chunk = max_scenes < kChunk ? max_scenes : kChunk;
    int r;
    if ((r = dev_alloc(&c->d_carry, (size_t)max_scenes))) { delete c; return r; }
    if ((r = dev_alloc(&c->d_last, (size_t)max_scenes * DP_PATH_POINTS))) { delete c; return r; }
    if ((r = dev_alloc(&c->d_done, (size_t)max_scenes))) { delete c; return r; }
    if ((r = dev_alloc(&c->d_inflag, 2)) || (r = dev_alloc(&c->d_tally, 2)) || (r = dev_alloc(&c->d_tally_g, 2))) { delete c; return r; }
    CK(cudaMemset(c->d_tally_g, 0, 2 * sizeof(unsigned)));
    CK(cudaMemset(c->d_inflag, 0, 2 * sizeof(unsigned))); CK(cudaMemset(c->d_tally, 0, 2 * sizeof(unsigned)));
    CK(cudaHostAlloc((void**)&c->h_done, 4 * sizeof(unsigned), cudaHostAllocMapped));
    c->h_done[0] = c->h_done[1] = c->h_done[2] = c->h_done[3] = 0;
    CK(cudaMemset(c->d_done, 0, (size_t)max_scenes * sizeof(unsigned)));
    for (int s = 0; s < 2; ++s) {
        CK(cudaStreamCreateWithFlags(&c->st[s], cudaStreamNonBlocking));
        if ((r = dev_alloc(&c->d_hdr[s], (size_t)c->chunk))) return r;
        if ((r = dev_alloc(&c->d_ox[s], (size_t)c->chunk * max_obs))) return r;
        if ((r = dev_alloc(&c->d_oy[s], (size_t)c->chunk * max_obs))) return r;
        if ((r = dev_alloc(&c->d_rec[s], (size_t)c->chunk))) return r;
        CK(cudaMallocHost((void**)&c->h_hdr[s], (size_t)c->chunk * sizeof(dp_scene_hdr)));
        CK(cudaMallocHost((void**)&c->h_ox[s], (size_t)c->chunk * max_obs * sizeof(double)));
        CK(cudaMallocHost((void**)&c->h_oy[s], (size_t)c->chunk * max_obs * sizeof(double)));
        CK(cudaMallocHost((void**)&c->h_rec[s], (size_t)c->chunk * sizeof(dp_plan_record)));
        for (int k = 0; k < 3; ++k) CK(cudaEventCreateWithFlags(&c->in_ready[s][k], cudaEventDisableTiming));
    }
    for (int k = 0; k < 3; ++k) CK(cudaStreamCreateWithFlags(&c->cp[k], cudaStreamNonBlocking));
    *out = c;
    return dp_reset(c, 0, max_scenes);
}

int dp_destroy(dp_ctx* c) {
    if (!c) return DP_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    if (c->lc.l2_bytes) { cudaCtxResetPersistingL2Cache(); cudaGetLastError(); }   // hand the map's lines in the L2 set-aside back
    for (void* p : c->map_allocs) cudaFree(p);
    if (c->ep_exec) cudaGraphExecDestroy(c->ep_exec);
    if (c->ep_stream) cudaStreamDestroy(c->ep_stream);
    cudaFree(c->d_timeline); cudaFree(c->d_trk);
    cudaFree(c->d_carry); cudaFree(c->d_last); cudaFree(c->d_done); cudaFree(c->d_inflag); cudaFree(c->d_tally); cudaFree(c->d_tally_g);
    if (c->h_done) cudaFreeHost(c->h_done);
    for (int s = 0; s < 2; ++s) {
        cudaFree(c->d_hdr[s]); cudaFree(c->d_ox[s]); cudaFree(c->d_oy[s]); cudaFree(c->d_rec[s]);
        cudaFree(c->d_trace[s]); cudaFree(c->d_pxy[s]); cudaFree(c->d_pll[s]);
        cudaFreeHost(c->h_hdr[s]); cudaFreeHost(c->h_ox[s]); cudaFreeHost(c->h_oy[s]); cudaFreeHost(c->h_rec[s]);
        if (c->st[s]) cudaStreamDestroy(c->st[s]);
        for (int k = 0; k < 3; ++k) if (c->in_ready[s][k]) cudaEventDestroy(c->in_ready[s][k]);
    }
    for (int k = 0; k < 3; ++k) if (c->cp[k]) cudaStreamDestroy(c->cp[k]);
    delete c;
    return DP_OK;
}

int dp_map_upload(dp_ctx* c, const dp_map_desc* m) {
    if (!c || !m || m->n_roads <= 0 || m->n_lanes <= 0 || m->n_points <= 0) return fail(DP_ERR_ARG, "dp_map_upload: bad argument");
    CK(cudaSetDevice(c->device));
    for (void* p : c->map_allocs) cudaFree(p);
    c->map_allocs.clear();
    c->have_map = false; c->lc.l2_base = nullptr; c->lc.l2_bytes = 0;   // (until the new tables are complete)
    if (c->ep_exec) { cudaGraphExecDestroy(c->ep_exec); c->ep_exec = nullptr; }   // (a cached episode graph points into the old map)
    // every map table lives in ONE arena (256-byte aligned pieces), so that a single L2 access-policy window covers the map
    const size_t np = (size_t)m->n_points;
    const size_t arena_bytes = 16 * 256 + np * (8 * 3 + 16 * 2 + 8 * 2 + 8 + 4 * 2 + 2 * 2) + (size_t)m->n_lanes * (4 * 3 + 8 + 4) +
                               (size_t)(m->n_roads + m->n_lanes + 2) * 4 + (size_t)m->n_conn * sizeof(dp_connector) + (size_t)m->n_lanes * 4 +
                               33 * 256;
    char* arena = nullptr;
    {
        cudaError_t e = cudaMalloc((void**)&arena, arena_bytes);
        if (e != cudaSuccess) return fail(DP_ERR_NOMEM, "cudaMalloc(map)", e);
        c->map_allocs.push_back(arena);
    }
    size_t arena_used = 0;
    auto up = [&](const void* src, size_t bytes, void** dst) -> int {
        const size_t need = (bytes ? bytes : 8);
        if (arena_used + need > arena_bytes) return fail(DP_ERR_NOMEM, "dp_map_upload: arena");
        *dst = arena + arena_used;
        arena_used = (arena_used + need + 255) & ~(size_t)255;
        if (src && bytes) { cudaError_t e = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice); if (e != cudaSuccess) return fail(DP_ERR_CUDA, "cudaMemcpy(map)", e); }
        return DP_OK;
    };
    // the avoid sweep enumerates i < (W - Vw) / 0.6 candidates per side with no cap (Decision.cpp:940); this library holds
    // DP_MAX_SWEEP of them: a lane wide enough to need more is rejected here instead of diverging silently
    for (size_t i = 0; i < np; ++i)
        if ((m->lane_width[i] / 100.0 - c->p.vehicle_width) / 0.6 > (double)DP_MAX_SWEEP)
            return fail(DP_ERR_ARG, "dp_map_upload: lane too wide for DP_MAX_SWEEP avoid candidates per side");
    for (int i = 0; i < m->n_lanes; ++i)
        if (m->lane_pt_off[i + 1] - m->lane_pt_off[i] > 65535) return fail(DP_ERR_ARG, "dp_map_upload: lane longer than 65535 points");
    // successor of every lane (the world step's agents follow it through junctions): a road lane -> the lane of the lowest
    // connector leaving it, a connector's pseudo-lane -> lane_index(next_road, next_lane); -1 none
    const int n_road_lanes = m->road_lane_base[m->n_roads];
    auto lanes_of = [&](int r) { return m->road_lane_base[r] - m->road_lane_base[r - 1]; };
    for (int k = 0; k < m->n_conn; ++k) {
        const dp_connector& q = m->conn[k];
        if (q.lane < n_road_lanes || q.lane >= m->n_lanes || q.last_road < 1 || q.last_road > m->n_roads || q.next_road < 1 ||
            q.next_road > m->n_roads || q.last_lane < 1 || q.last_lane > lanes_of(q.last_road) || q.next_lane < 1 ||
            q.next_lane > lanes_of(q.next_road))
            return fail(DP_ERR_ARG, "dp_map_upload: connector names no road lane / pseudo-lane of the map");
    }
    std::vector<int32_t> lane_next(m->n_lanes, -1);
    for (int r = 1; r <= m->n_roads; ++r)
        for (int gl = m->road_lane_base[r - 1]; gl < m->road_lane_base[r]; ++gl)
            for (int k = 0; k < m->n_conn; ++k)
                if (m->conn[k].last_road == r && m->conn[k].last_lane == gl - m->road_lane_base[r - 1] + 1) { lane_next[gl] = m->conn[k].lane; break; }
    for (int k = 0; k < m->n_conn; ++k) lane_next[m->conn[k].lane] = m->road_lane_base[m->conn[k].next_road - 1] + m->conn[k].next_lane - 1;
    DgMap d;
    int r;
    double* d_lenf = nullptr; float* d_hmax = nullptr; float* d_dnmax = nullptr; float* d_hmin = nullptr;
    double* d_cump = nullptr; double* d_cerr = nullptr; int32_t* d_re0 = nullptr; int32_t* d_re1 = nullptr;
    if ((r = up(m->x, np * 8, (void**)&d.x))) return r;
    if ((r = up(m->y, np * 8, (void**)&d.y))) return r;
    if ((r = up(m->dir, np * 8, (void**)&d.dir))) return r;
    if ((r = up(nullptr, np * 16, (void**)&d.xy))) return r;
    if ((r = up(nullptr, np * 16, (void**)&d.nrm))) return r;
    if ((r = up(nullptr, np * 8, (void**)&d.lenp))) return r;
    if ((r = up(nullptr, np * 8, (void**)&d_lenf))) return r;
    if ((r = up(nullptr, (size_t)m->n_lanes * 4, (void**)&d_hmax))) return r;
    if ((r = up(nullptr, (size_t)m->n_lanes * 4, (void**)&d_dnmax))) return r;
    if ((r = up(nullptr, (size_t)m->n_lanes * 4, (void**)&d_hmin))) return r;
    if ((r = up(nullptr, np * 8, (void**)&d_cump))) return r;
    if ((r = up(nullptr, (size_t)m->n_lanes * 8, (void**)&d_cerr))) return r;
    if ((r = up(nullptr, np * 4, (void**)&d_re0))) return r;
    if ((r = up(nullptr, np * 4, (void**)&d_re1))) return r;
    if ((r = up(m->lane_width, np * 2, (void**)&d.width))) return r;
    if ((r = up(m->lanechg_attr, np * 2, (void**)&d.attr))) return r;
    if ((r = up(m->road_lane_base, (size_t)(m->n_roads + 1) * 4, (void**)&d.road_lane_base))) return r;
    if ((r = up(m->lane_pt_off, (size_t)(m->n_lanes + 1) * 4, (void**)&d.lane_pt_off))) return r;
    if ((r = up(m->conn, (size_t)m->n_conn * sizeof(dp_connector), (void**)&d.conn))) return r;
    if ((r = up(lane_next.data(), (size_t)m->n_lanes * 4, (void**)&d.lane_next))) return r;
    d.n_roads = m->n_roads; d.n_lanes = m->n_lanes; d.n_conn = m->n_conn;
    CK(dp_launch_map_prep(d.x, d.y, d.attr, d.lane_pt_off, d.n_lanes, (double2*)d.xy, (double2*)d.nrm, (double*)d.lenp, d_lenf, d_hmax, d_hmin,
                          d_dnmax, d_cump, d_cerr, d_re0, d_re1, c->st[0]));
    c->launches += 2;
    CK(cudaStreamSynchronize(c->st[0]));
    d.lenf = d_lenf; d.lane_hmax = d_hmax; d.lane_dnmax = d_dnmax; d.lane_hmin = d_hmin;
    d.cump = d_cump; d.lane_cerr = d_cerr; d.run_end0 = d_re0; d.run_end1 = d_re1;
    c->gmap = d;
    c->have_map = true;
    // L2 persistence (DP_L2_PERSIST=0 switches it off): reserve a set-aside as large as the arena (if the device allows) and let
    // the cycle launches mark their map accesses persisting -- constant tables every scene gathers from should not be evicted
    // by what streams through the cache between two cycles
    c->lc.l2_base = nullptr; c->lc.l2_bytes = 0;
    int want = 1;
    if (const char* e = getenv("DP_L2_PERSIST")) want = atoi(e);
    if (want) {
        int max_persist = 0, max_window = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, c->device);
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, c->device);
        size_t cur = 0;
        cudaDeviceGetLimit(&cur, cudaLimitPersistingL2CacheSize);
        const size_t bytes = arena_used;
        if (max_persist > 0 && bytes <= (size_t)max_persist && bytes <= (size_t)max_window) {
            bool ok = cur >= bytes || cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes + (1u << 20)) == cudaSuccess;
            if (ok) { c->lc.l2_base = arena; c->lc.l2_bytes = bytes; } else cudaGetLastError();
        }
    }
    return DP_OK;
}

int dp_reset(dp_ctx* c, int first, int count) {
    if (!c || first < 0 || count < 0 || first + count > c->max_scenes) return fail(DP_ERR_ARG, "dp_reset: range");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_reset: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    CK(dp_launch_reset(c->d_carry, c->d_last, first, count, c->st[0]));
    ++c->launches;
    CK(cudaStreamSynchronize(c->st[0]));
    return DP_OK;
}

int dp_reset_dev(dp_ctx* c, int first, int count, void* stream) {
    if (!c || first < 0 || count < 0 || first + count > c->max_scenes) return fail(DP_ERR_ARG, "dp_reset_dev: range");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_reset_dev: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    CK(dp_launch_reset(c->d_carry, c->d_last, first, count, (cudaStream_t)stream));
    ++c->launches;
    return DP_OK;
}

int dp_carry_download(dp_ctx* c, int first, int count, dp_carry* hc, double* hl) {
    if (!c || first < 0 || count < 0 || first + count > c->max_scenes) return fail(DP_ERR_ARG, "dp_carry_download: range");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_carry_download: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    if (hc) CK(cudaMemcpy(hc, c->d_carry + first, (size_t)count * sizeof(dp_carry), cudaMemcpyDeviceToHost));
    if (hl) {                                               // device keeps the path as [200] double2; the ABI layout is [2][200]
        std::vector<double2> tmp((size_t)count * DP_PATH_POINTS);
        CK(cudaMemcpy(tmp.data(), c->d_last + (size_t)first * DP_PATH_POINTS, tmp.size() * sizeof(double2), cudaMemcpyDeviceToHost));
        for (int s = 0; s < count; ++s)
            for (int i = 0; i < DP_PATH_POINTS; ++i) {
                hl[(size_t)s * 400 + i] = tmp[(size_t)s * DP_PATH_POINTS + i].x;
                hl[(size_t)s * 400 + DP_PATH_POINTS + i] = tmp[(size_t)s * DP_PATH_POINTS + i].y;
            }
    }
    return DP_OK;
}
int dp_carry_upload(dp_ctx* c, int first, int count, const dp_carry* hc, const double* hl) {
    if (!c || first < 0 || count < 0 || first + count > c->max_scenes) return fail(DP_ERR_ARG, "dp_carry_upload: range");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_carry_upload: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    if (hc) CK(cudaMemcpy(c->d_carry + first, hc, (size_t)count * sizeof(dp_carry), cudaMemcpyHostToDevice));
    if (hl) {
        std::vector<double2> tmp((size_t)count * DP_PATH_POINTS);
        for (int s = 0; s < count; ++s)
            for (int i = 0; i < DP_PATH_POINTS; ++i)
                tmp[(size_t)s * DP_PATH_POINTS + i] = make_double2(hl[(size_t)s * 400 + i], hl[(size_t)s * 400 + DP_PATH_POINTS + i]);
        CK(cudaMemcpy(c->d_last + (size_t)first * DP_PATH_POINTS, tmp.data(), tmp.size() * sizeof(double2), cudaMemcpyHostToDevice));
    }
    return DP_OK;
}

int dp_cycle_batch_dev(dp_ctx* c, int first, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy, dp_plan_record* rec,
                       dp_trace_record* trace, double* path_xy, double* path_ll, void* stream) {
    if (!c || !hdr || !ox || !oy || !rec || n < 0 || first < 0 || first + n > c->max_scenes) return fail(DP_ERR_ARG, "dp_cycle_batch_dev: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_cycle_batch_dev: map not uploaded");
    CK(cudaSetDevice(c->device));
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_cycle_batch_dev: submitted cycles in flight, call dp_cycle_wait first");
    CK(run_cycle(c, first, n, hdr, ox, oy, rec, trace, path_xy, path_ll, (cudaStream_t)stream, make_io(c, first, nullptr)));
    return DP_OK;
}

int dp_run_episode_dev(dp_ctx* c, int first, int n, int cycles, const dp_scene_hdr* hdr, const double* ox, const double* oy, dp_plan_record* rec,
                       void* stream) {
    if (!c || !hdr || !ox || !oy || !rec || n < 0 || cycles < 0 || first < 0 || first + n > c->max_scenes)
        return fail(DP_ERR_ARG, "dp_run_episode_dev: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_run_episode_dev: map not uploaded");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_run_episode_dev: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    const size_t mo = (size_t)c->max_obs;
    // back-to-back launch pairs, no host involvement in between.  (Cycle k+1's Decision launch as a programmatic dependent of
    // cycle k's Planning launch was measured here too: 84 vs 66 us per 4096-scene cycle -- the early Decision CTAs spin in slots
    // the Planning launch needs -- so the episode runner keeps the plain stream order.)
    for (int k = 0; k < cycles; ++k) {
        const DpIo io = make_io(c, first, nullptr);
        CK(run_cycle(c, first, n, hdr + (size_t)k * n, ox + (size_t)k * n * mo, oy + (size_t)k * n * mo, rec + (size_t)k * n, nullptr, nullptr,
                     nullptr, (cudaStream_t)stream, io));
    }
    return DP_OK;
}

int dp_cycle_batch(dp_ctx* c, int first, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy, dp_plan_record* rec,
                   dp_trace_record* trace, double* path_xy, double* path_ll) {
    if (!c || !hdr || !ox || !oy || !rec || n < 0 || first < 0 || first + n > c->max_scenes) return fail(DP_ERR_ARG, "dp_cycle_batch: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_cycle_batch: map not uploaded");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_cycle_batch: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    int r;
    if (trace && (r = ensure_optional(c, 0))) return r;
    if (path_xy && (r = ensure_optional(c, 1))) return r;
    if (path_ll && (r = ensure_optional(c, 2))) return r;
    const size_t mo = (size_t)c->max_obs;
    const bool pin_in = is_pinned(hdr) && is_pinned(ox) && is_pinned(oy);
    const bool pin_rec = is_pinned(rec);
    const bool plain = n <= c->chunk && !trace && !path_xy && !path_ll;
    if (plain && pin_in && pin_rec) {
        // Page-locked buffers: the pipelined machinery with one cycle in flight -- three overlapping input DMAs, the two
        // launches, and the Planning launch storing each finished 128-byte record straight into the caller's buffer.
        int rs = dp_cycle_submit(c, first, n, hdr, ox, oy, rec);
        if (rs != DP_OK) return rs;
        return dp_cycle_wait(c);
    }
    int nchunks = (n + c->chunk - 1) / c->chunk;
    for (int k = 0; k < nchunks; ++k) {
        const int s = k & 1;
        const int i0 = k * c->chunk, cn = (n - i0 < c->chunk) ? n - i0 : c->chunk;
        cudaStream_t st = c->st[s];
        if (k >= 2) {                                       // staging set s is being reused: drain its previous chunk
            CK(cudaStreamSynchronize(st));
            if (!pin_rec) memcpy(rec + (size_t)(k - 2) * c->chunk, c->h_rec[s], (size_t)c->chunk * sizeof(dp_plan_record));
        }
        const dp_scene_hdr* sh = hdr + i0; const double* sx = ox + i0 * mo; const double* sy = oy + i0 * mo;
        if (!pin_in) {
            memcpy(c->h_hdr[s], sh, (size_t)cn * sizeof(dp_scene_hdr));
            memcpy(c->h_ox[s], sx, (size_t)cn * mo * 8);
            memcpy(c->h_oy[s], sy, (size_t)cn * mo * 8);
            sh = c->h_hdr[s]; sx = c->h_ox[s]; sy = c->h_oy[s];
        }
        CK(cudaMemcpyAsync(c->d_hdr[s], sh, (size_t)cn * sizeof(dp_scene_hdr), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(c->d_ox[s], sx, (size_t)cn * mo * 8, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(c->d_oy[s], sy, (size_t)cn * mo * 8, cudaMemcpyHostToDevice, st));
        CK(run_cycle(c, first + i0, cn, c->d_hdr[s], c->d_ox[s], c->d_oy[s], c->d_rec[s], trace ? c->d_trace[s] : nullptr,
                     path_xy ? c->d_pxy[s] : nullptr, path_ll ? c->d_pll[s] : nullptr, st, make_io(c, first + i0, nullptr)));
        CK(cudaMemcpyAsync(pin_rec ? rec + i0 : c->h_rec[s], c->d_rec[s], (size_t)cn * sizeof(dp_plan_record), cudaMemcpyDeviceToHost, st));
        if (trace) CK(cudaMemcpyAsync(trace + i0, c->d_trace[s], (size_t)cn * sizeof(dp_trace_record), cudaMemcpyDeviceToHost, st));
        if (path_xy) CK(cudaMemcpyAsync(path_xy + (size_t)i0 * 400, c->d_pxy[s], (size_t)cn * 400 * 8, cudaMemcpyDeviceToHost, st));
        if (path_ll) CK(cudaMemcpyAsync(path_ll + (size_t)i0 * 200, c->d_pll[s], (size_t)cn * 200 * 8, cudaMemcpyDeviceToHost, st));
    }
    for (int k = (nchunks >= 2 ? nchunks - 2 : 0); k < nchunks; ++k) {
        const int s = k & 1;
        const int i0 = k * c->chunk, cn = (n - i0 < c->chunk) ? n - i0 : c->chunk;
        CK(cudaStreamSynchronize(c->st[s]));
        if (!pin_rec) memcpy(rec + i0, c->h_rec[s], (size_t)cn * sizeof(dp_plan_record));
    }
    return DP_OK;
}

// The records reach the caller's buffer by stores of the kernel (the Planning warps, or the group kernel's CTAs): no copy in the
// tail of a call
int dp_cycle_submit(dp_ctx* c, int first, int n, const dp_scene_hdr* hdr, const double* ox, const double* oy, dp_plan_record* rec) {
    if (!c || !hdr || !ox || !oy || !rec || n < 0 || first < 0 || first + n > c->max_scenes || n > c->chunk)
        return fail(DP_ERR_ARG, "dp_cycle_submit: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_cycle_submit: map not uploaded");
    if (c->submitted - c->waited >= 2) return fail(DP_ERR_STATE, "dp_cycle_submit: two cycles already in flight, call dp_cycle_wait");
    void* dv_rec = nullptr;
    if (!is_pinned(hdr) || !is_pinned(ox) || !is_pinned(oy) || !is_pinned(rec, &dv_rec) || !dv_rec)
        return fail(DP_ERR_ARG, "dp_cycle_submit: buffers must be page-locked (dp_host_alloc)");
    CK(cudaSetDevice(c->device));
    // staging set s was last read by cycle (submitted - 2), which has been waited for: it is free.
    const int s = (int)(c->submitted & 1);
    const size_t mo = (size_t)c->max_obs;
    cudaStream_t st = c->st[0];                             // one compute stream: cycle k+1 reads the carry cycle k wrote
    DpIo io = make_io(c, first, (dp_plan_record*)dv_rec);
    void* dv_done = nullptr;
    CK(cudaHostGetDevicePointer(&dv_done, c->h_done, 0));
    // the last Planning warp / CTA of the cycle stores its epoch to page-locked host memory (dp_cycle_wait polls it: no event round
    // trip) and re-arms the tally word itself, no memset
    io.tally = c->d_tally + s; io.tally_n = (unsigned)n; io.host_done = (unsigned*)dv_done + s;
    c->wait_epoch[s] = n > 0 ? io.epoch : 0u;
    if (c->kernel == 1 || c->tracks_T > 0) {
        // group kernel: the three input DMAs overlap on their own copy streams, the launch waits for their events
        CK(cudaMemcpyAsync(c->d_hdr[s], hdr, (size_t)n * sizeof(dp_scene_hdr), cudaMemcpyHostToDevice, c->cp[0]));
        CK(cudaMemcpyAsync(c->d_ox[s], ox, (size_t)n * mo * 8, cudaMemcpyHostToDevice, c->cp[1]));
        CK(cudaMemcpyAsync(c->d_oy[s], oy, (size_t)n * mo * 8, cudaMemcpyHostToDevice, c->cp[2]));
        for (int k = 0; k < 3; ++k) {
            CK(cudaEventRecord(c->in_ready[s][k], c->cp[k]));
            CK(cudaStreamWaitEvent(st, c->in_ready[s][k], 0));
        }
    } else {
        // warp kernel: nothing but kernels goes into the compute stream.  The copy stream carries the three input DMAs and then a
        // four-byte copy that raises in_flag; the Decision warps wait for that flag
        CK(cudaMemcpyAsync(c->d_hdr[s], hdr, (size_t)n * sizeof(dp_scene_hdr), cudaMemcpyHostToDevice, c->cp[0]));
        CK(cudaMemcpyAsync(c->d_ox[s], ox, (size_t)n * mo * 8, cudaMemcpyHostToDevice, c->cp[0]));
        CK(cudaMemcpyAsync(c->d_oy[s], oy, (size_t)n * mo * 8, cudaMemcpyHostToDevice, c->cp[0]));
        // the flag goes up by a COPY, not a kernel: a one-thread kernel could find every SM slot taken by Decision and Planning
        // CTAs that are waiting for exactly this flag
        c->h_done[2 + s] = io.epoch;
        CK(cudaMemcpyAsync(c->d_inflag + s, c->h_done + 2 + s, sizeof(unsigned), cudaMemcpyHostToDevice, c->cp[0]));
        io.in_flag = c->d_inflag + s;
    }
    CK(run_cycle(c, first, n, c->d_hdr[s], c->d_ox[s], c->d_oy[s], c->d_rec[s], nullptr, nullptr, nullptr, st, io));
    ++c->submitted;
    return DP_OK;
}
int dp_cycle_wait(dp_ctx* c) {
    if (!c) return fail(DP_ERR_ARG, "dp_cycle_wait: null context");
    if (c->submitted == c->waited) return fail(DP_ERR_STATE, "dp_cycle_wait: nothing in flight");
    CK(cudaSetDevice(c->device));
    const int s = (int)(c->waited & 1);
    const unsigned want = c->wait_epoch[s];
    const volatile unsigned* flag = c->h_done + s;
    if (want) {
        const auto t0 = std::chrono::steady_clock::now();
        for (unsigned long long spin = 0; *flag != want; ++spin) {
            if ((spin & 0xfff) == 0xfff) {                  // a kernel that trapped never raises the flag: ask the stream now and then
                const cudaError_t q = cudaStreamQuery(c->st[0]);
                if (q != cudaSuccess && q != cudaErrorNotReady) return fail(DP_ERR_CUDA, "dp_cycle_wait", q);
                if (q == cudaSuccess && *flag != want) return fail(DP_ERR_CUDA, "dp_cycle_wait: the stream drained without the completion flag");
                if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(30)) return fail(DP_ERR_CUDA, "dp_cycle_wait: timed out");
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
    }
    ++c->waited;
    return DP_OK;
}

int dp_set_record_mirrors(dp_ctx* c, int n, void* const* bases) {
    if (!c || n < 0 || n > DP_MAX_MIRRORS - 1 || (n > 0 && !bases)) return fail(DP_ERR_ARG, "dp_set_record_mirrors: bad argument");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_set_record_mirrors: submitted cycles in flight, call dp_cycle_wait first");
    for (int k = 0; k < n; ++k) {
        if (!bases[k]) return fail(DP_ERR_ARG, "dp_set_record_mirrors: null base");
        c->armed.mirror[k] = (dp_plan_record*)bases[k];
    }
    c->armed.n_mirror = n;
    return DP_OK;
}

int dp_set_tracks_dev(dp_ctx* c, int T, const double* vx, const double* vy, const double* dth) {
    if (!c || T < 1 || !vx || !vy || !dth) return fail(DP_ERR_ARG, "dp_set_tracks_dev: bad argument");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_set_tracks_dev: submitted cycles in flight, call dp_cycle_wait first");
    c->trk_vx = vx; c->trk_vy = vy; c->trk_dth = dth; c->tracks_T = T;
    return DP_OK;
}
int dp_set_tracks(dp_ctx* c, int first, int n, int T, const double* vx, const double* vy, const double* dth) {
    if (!c || first < 0 || n < 0 || first + n > c->max_scenes || T < 1 || !vx || !vy || !dth) return fail(DP_ERR_ARG, "dp_set_tracks: bad argument");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_set_tracks: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    const size_t st = (size_t)c->max_scenes * c->max_obs, cnt = (size_t)n * c->max_obs, off = (size_t)first * c->max_obs;
    if (!c->d_trk) { int r = dev_alloc(&c->d_trk, st * 3); if (r) return r; CK(cudaMemset(c->d_trk, 0, st * 3 * 8)); }
    const double* src[3] = {vx, vy, dth};
    for (int k = 0; k < 3; ++k) CK(cudaMemcpyAsync(c->d_trk + (size_t)k * st + off, src[k], cnt * 8, cudaMemcpyHostToDevice, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    c->trk_vx = c->d_trk; c->trk_vy = c->d_trk + st; c->trk_dth = c->d_trk + 2 * st; c->tracks_T = T;
    return DP_OK;
}
int dp_clear_tracks(dp_ctx* c) {
    if (!c) return fail(DP_ERR_ARG, "dp_clear_tracks: null context");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_clear_tracks: submitted cycles in flight, call dp_cycle_wait first");
    c->tracks_T = 0;
    return DP_OK;
}

int dp_debug_timeline(dp_ctx* c, long long* host_out, int n_blocks) {
    if (!c || !host_out || n_blocks < 0 || n_blocks > 8192) return fail(DP_ERR_ARG, "dp_debug_timeline: bad argument");
    if (!c->d_timeline) return fail(DP_ERR_STATE, "dp_debug_timeline: context was created without DP_TIMELINE=1");
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(host_out, c->d_timeline, (size_t)n_blocks * 32 * sizeof(long long), cudaMemcpyDeviceToHost));
    return DP_OK;
}

// ---- fused gather of plan records across the GPUs of one box, through the C ABI (CUDA IPC) ----
struct dp_gather {
    dp_ctx* c = nullptr;
    int world = 0, rank = 0, slots = 0, depth = 0;
    unsigned char* base[DP_MAX_MIRRORS] = {};               // every rank's allocation as seen from here (own: the local pointer)
    bool opened[DP_MAX_MIRRORS] = {};
    size_t rec_bytes = 0;                                   // records come first ([depth][world][slots]), the flags ([depth][world] u32) follow
    unsigned pending = 0;                                   // deferred mode: step whose records have been computed but not forwarded yet
    unsigned forwarded = 0;                                 // ... and the newest step that has been forwarded (flags raised by this rank)
    int lag = 1;                                            // a launch awaits the flags of the step `lag` launches back (dp_gather_set_lag)
};
namespace {
// the buffers / flags of step `step`: this rank's slice and flag word in every rank's buffer, and this rank's flag words of the step
void gather_route(dp_gather* g, unsigned step, dp_plan_record** dst, unsigned** flag, DpWait* wait) {
    const size_t b = step % (unsigned)g->depth;
    for (int r = 0; r < g->world; ++r) {
        dst[r] = reinterpret_cast<dp_plan_record*>(g->base[r]) + (b * g->world + g->rank) * g->slots;
        flag[r] = reinterpret_cast<unsigned*>(g->base[r] + g->rec_bytes) + b * g->world + g->rank;
    }
    if (wait) *wait = {reinterpret_cast<const unsigned*>(g->base[g->rank] + g->rec_bytes) + b * g->world, g->world, step};
}
}  // namespace
static_assert(DP_IPC_BYTES >= sizeof(cudaIpcMemHandle_t), "DP_IPC_BYTES");

int dp_gather_create(dp_ctx* c, int world, int rank, int slots, int depth, dp_gather** out, void* handle_out) {
    if (!c || !out || !handle_out || world < 1 || world > DP_MAX_MIRRORS - 1 || rank < 0 || rank >= world || slots < 1 || slots > c->max_scenes || depth < 1)
        return fail(DP_ERR_ARG, "dp_gather_create: bad argument (world <= 8)");
    CK(cudaSetDevice(c->device));
    dp_gather* g = new dp_gather();
    g->c = c; g->world = world; g->rank = rank; g->slots = slots; g->depth = depth;
    g->rec_bytes = (size_t)depth * world * slots * sizeof(dp_plan_record);
    const size_t bytes = g->rec_bytes + (size_t)depth * world * sizeof(unsigned);
    cudaError_t e = cudaMalloc((void**)&g->base[rank], bytes);
    if (e != cudaSuccess) { delete g; return fail(DP_ERR_NOMEM, "dp_gather_create: cudaMalloc", e); }
    CK(cudaMemset(g->base[rank], 0, bytes));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, g->base[rank]));
    memset(handle_out, 0, DP_IPC_BYTES);
    memcpy(handle_out, &h, sizeof(h));
    *out = g;
    return DP_OK;
}
int dp_gather_attach(dp_gather* g, const void* handles) {
    if (!g || !handles) return fail(DP_ERR_ARG, "dp_gather_attach: bad argument");
    CK(cudaSetDevice(g->c->device));
    for (int r = 0; r < g->world; ++r) {
        if (r == g->rank || g->opened[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const unsigned char*)handles + (size_t)r * DP_IPC_BYTES, sizeof(h));
        CK(cudaIpcOpenMemHandle((void**)&g->base[r], h, cudaIpcMemLazyEnablePeerAccess));
        g->opened[r] = true;
    }
    return DP_OK;
}
int dp_gather_arm(dp_gather* g, unsigned step) {
    if (!g || step == 0) return fail(DP_ERR_ARG, "dp_gather_arm: bad argument (steps count from 1)");
    dp_ctx* c = g->c;                                       // (only read by the NEXT launch call of this thread: fine between pipelined submits)
    for (int r = 0; r < g->world; ++r) if (!g->base[r]) return fail(DP_ERR_STATE, "dp_gather_arm: dp_gather_attach first");
    DpIo a = {};                                            // replaces the mirrors and any armed gather; a wait folded in by dp_gather_chain stays
    a.wait = c->armed.wait;
    gather_route(g, step, a.mirror, a.peer_flag, nullptr);
    a.n_mirror = a.n_peer_flag = g->world;
    a.flag_value = step;
    c->armed = a; c->deferred = false;
    return DP_OK;
}
int dp_gather_arm_deferred(dp_gather* g, unsigned step) {
    if (!g || step == 0) return fail(DP_ERR_ARG, "dp_gather_arm_deferred: bad argument (steps count from 1)");
    dp_ctx* c = g->c;
    for (int r = 0; r < g->world; ++r) if (!g->base[r]) return fail(DP_ERR_STATE, "dp_gather_arm_deferred: dp_gather_attach first");
    DpIo a = {};
    if (g->pending && c->last_rec) {                        // the launch that follows forwards and flags the step before ...
        gather_route(g, g->pending, a.fwd_dst, a.peer_flag, nullptr);
        a.n_fwd = a.n_peer_flag = g->world;
        a.flag_value = g->pending;
        // ... and awaits every rank's flags of that step (lag 1) or of the one before it (lag 2: a full step of slack between the
        // ranks; that step was forwarded by the launch before, so only launches that have one to wait for do)
        const unsigned w = (g->lag == 1) ? g->pending : g->forwarded;
        if (w) {
            dp_plan_record* d_[DP_MAX_MIRRORS]; unsigned* f_[DP_MAX_MIRRORS];
            gather_route(g, w, d_, f_, &a.wait);
        }
        g->forwarded = g->pending;
    }
    c->armed = a; c->deferred = true;
    g->pending = step;
    return DP_OK;
}
int dp_gather_set_lag(dp_gather* g, int lag) {
    if (!g || lag < 1 || lag > 2 || g->depth < lag + 2) return fail(DP_ERR_ARG, "dp_gather_set_lag: lag 1 or 2, depth >= lag + 2");
    g->lag = lag;
    return DP_OK;
}
int dp_gather_flush(dp_gather* g, void* stream) {
    if (!g) return fail(DP_ERR_ARG, "dp_gather_flush: null");
    dp_ctx* c = g->c;
    if (!g->pending || !c->last_rec) return DP_OK;
    CK(cudaSetDevice(c->device));
    DpIo io = {};
    gather_route(g, g->pending, io.fwd_dst, io.peer_flag, &io.wait);
    for (int r = 0; r < g->world; ++r) io.fwd_dst[r] += c->last_first;
    io.n_fwd = io.n_peer_flag = g->world;
    io.flag_value = g->pending;
    if (g->lag == 2 && g->forwarded) {                      // the step before may not have been awaited by any launch yet
        CK(dp_launch_gather_wait(reinterpret_cast<const unsigned*>(g->base[g->rank] + g->rec_bytes) + (size_t)(g->forwarded % (unsigned)g->depth) * g->world,
                                 g->world, g->forwarded, (cudaStream_t)stream));
        ++c->launches;
    }
    CK(dp_launch_gather_flush(c->last_rec, c->last_n, io, (cudaStream_t)stream));
    c->launches += 2;
    g->pending = 0; g->forwarded = 0;
    return DP_OK;
}
int dp_gather_chain(dp_gather* g, unsigned prev_step) {
    if (!g) return fail(DP_ERR_ARG, "dp_gather_chain: null");
    dp_ctx* c = g->c;
    if (prev_step == 0) { c->armed.wait = {}; return DP_OK; }
    if (!g->base[g->rank]) return fail(DP_ERR_STATE, "dp_gather_chain: dp_gather_attach first");
    c->armed.wait = {reinterpret_cast<const unsigned*>(g->base[g->rank] + g->rec_bytes) + (size_t)(prev_step % (unsigned)g->depth) * g->world,
                     g->world, prev_step};
    return DP_OK;
}
int dp_gather_disarm(dp_gather* g) {
    if (!g) return fail(DP_ERR_ARG, "dp_gather_disarm: null");
    g->c->armed = {}; g->c->deferred = false;
    g->pending = 0; g->forwarded = 0;
    return DP_OK;
}
int dp_gather_wait(dp_gather* g, unsigned step, void* stream) {
    if (!g || step == 0) return fail(DP_ERR_ARG, "dp_gather_wait: bad argument");
    CK(cudaSetDevice(g->c->device));
    const size_t b = step % (unsigned)g->depth;
    CK(dp_launch_gather_wait(reinterpret_cast<const unsigned*>(g->base[g->rank] + g->rec_bytes) + b * g->world, g->world, step, (cudaStream_t)stream));
    ++g->c->launches;
    return DP_OK;
}
const void* dp_gather_buffer(dp_gather* g, unsigned step) {
    if (!g) return nullptr;
    return g->base[g->rank] + (size_t)(step % (unsigned)g->depth) * g->world * g->slots * sizeof(dp_plan_record);
}
int dp_gather_destroy(dp_gather* g) {
    if (!g) return DP_OK;
    cudaSetDevice(g->c->device);
    cudaDeviceSynchronize();
    dp_gather_disarm(g);
    for (int r = 0; r < g->world; ++r) {
        if (r == g->rank) cudaFree(g->base[r]);
        else if (g->opened[r]) cudaIpcCloseMemHandle(g->base[r]);
    }
    delete g;
    return DP_OK;
}

int dp_host_alloc(void** p, size_t bytes) {
    if (!p) return fail(DP_ERR_ARG, "dp_host_alloc");
    cudaError_t e = cudaMallocHost(p, bytes ? bytes : 8);
    if (e != cudaSuccess) return fail(DP_ERR_NOMEM, "cudaMallocHost", e);
    return DP_OK;
}
int dp_host_free(void* p) { if (p) cudaFreeHost(p); return DP_OK; }

// ---- operator-level entry points: host buffers in, host buffers out ----

int dp_search_obstacle(dp_ctx* c, int n_paths, const int32_t* path_off, const double* px, const double* py, const double* ox,
                       const double* oy, int n_obs, const double* lat_min, const double* lat_max, dp_search_slot* out) {
    if (!c || n_paths < 0 || !path_off || !lat_min || !lat_max || !out || n_obs < 0 || n_obs > 65535) return fail(DP_ERR_ARG, "dp_search_obstacle: bad argument");
    CK(cudaSetDevice(c->device));
    const size_t np = (size_t)path_off[n_paths];
    for (int i = 0; i < n_paths; ++i) if (path_off[i + 1] - path_off[i] > 65535) return fail(DP_ERR_ARG, "dp_search_obstacle: path longer than 65535 points");
    Tmp tmp; cudaError_t e;
    std::vector<double2> hxy = interleave(px, py, np);
    PUT(d_off, int32_t, path_off, (size_t)n_paths + 1);
    PUT(d_pxy, double2, hxy.data(), np);
    PUT(d_ox, double, ox, (size_t)n_obs); PUT(d_oy, double, oy, (size_t)n_obs);
    PUT(d_lo, double, lat_min, (size_t)n_paths); PUT(d_hi, double, lat_max, (size_t)n_paths);
    PUT(d_out, dp_search_slot, (const dp_search_slot*)nullptr, (size_t)n_paths);
    CK(dp_launch_search(n_paths, d_off, d_pxy, d_ox, d_oy, n_obs, d_lo, d_hi, d_out, c->st[0]));
    ++c->launches;
    CK(cudaMemcpyAsync(out, d_out, (size_t)n_paths * sizeof(dp_search_slot), cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    return DP_OK;
}

int dp_create_new_path(dp_ctx* c, int n_paths, const int32_t* path_off, const double* px, const double* py, const double* offset,
                       double* out_x, double* out_y) {
    if (!c || n_paths < 0 || !path_off || !offset || !out_x || !out_y) return fail(DP_ERR_ARG, "dp_create_new_path: bad argument");
    CK(cudaSetDevice(c->device));
    const size_t np = (size_t)path_off[n_paths];
    Tmp tmp; cudaError_t e;
    std::vector<double2> hxy = interleave(px, py, np);
    PUT(d_off, int32_t, path_off, (size_t)n_paths + 1);
    PUT(d_pxy, double2, hxy.data(), np);
    PUT(d_d, double, offset, (size_t)n_paths);
    PUT(d_o, double2, (const double2*)nullptr, np);
    CK(dp_launch_create(n_paths, d_off, d_pxy, d_d, d_o, c->st[0]));
    ++c->launches;
    CK(cudaMemcpyAsync(hxy.data(), d_o, np * sizeof(double2), cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    for (size_t i = 0; i < np; ++i) { out_x[i] = hxy[i].x; out_y[i] = hxy[i].y; }
    return DP_OK;
}

int dp_bezier_planning(dp_ctx* c, int n, const double* poses, double* out_xy) {
    if (!c || n < 0 || !poses || !out_xy) return fail(DP_ERR_ARG, "dp_bezier_planning: bad argument");
    CK(cudaSetDevice(c->device));
    Tmp tmp; cudaError_t e;
    PUT(d_p, double, poses, (size_t)n * 6);
    PUT(d_o, double, (const double*)nullptr, (size_t)n * 400);
    CK(dp_launch_bezier(n, d_p, d_o, c->st[0]));
    ++c->launches;
    CK(cudaMemcpyAsync(out_xy, d_o, (size_t)n * 400 * 8, cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    return DP_OK;
}

int dp_mean_points(dp_ctx* c, int n_paths, const int32_t* path_off, const double* px, const double* py, double* out_xy) {
    if (!c || n_paths < 0 || !path_off || !out_xy) return fail(DP_ERR_ARG, "dp_mean_points: bad argument");
    for (int i = 0; i < n_paths; ++i) if (path_off[i + 1] - path_off[i] > 2 * DP_TILE) return fail(DP_ERR_ARG, "dp_mean_points: more than 240 input points (reference limit is 200, Planning.cpp:851)");
    CK(cudaSetDevice(c->device));
    const size_t np = (size_t)path_off[n_paths];
    Tmp tmp; cudaError_t e;
    std::vector<double2> hxy = interleave(px, py, np);
    PUT(d_off, int32_t, path_off, (size_t)n_paths + 1);
    PUT(d_pxy, double2, hxy.data(), np);
    PUT(d_o, double, (const double*)nullptr, (size_t)n_paths * 400);
    CK(dp_launch_mean(n_paths, d_off, d_pxy, d_o, c->st[0]));
    ++c->launches;
    CK(cudaMemcpyAsync(out_xy, d_o, (size_t)n_paths * 400 * 8, cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    return DP_OK;
}

int dp_nearest_id(dp_ctx* c, int n_paths, const int32_t* path_off, const double* px, const double* py, const double* qx, const double* qy,
                  int32_t* out_id) {
    if (!c || n_paths < 0 || !path_off || !qx || !qy || !out_id) return fail(DP_ERR_ARG, "dp_nearest_id: bad argument");
    CK(cudaSetDevice(c->device));
    const size_t np = (size_t)path_off[n_paths];
    Tmp tmp; cudaError_t e;
    std::vector<double2> hxy = interleave(px, py, np);
    PUT(d_off, int32_t, path_off, (size_t)n_paths + 1);
    PUT(d_pxy, double2, hxy.data(), np);
    PUT(d_qx, double, qx, (size_t)n_paths);
    PUT(d_qy, double, qy, (size_t)n_paths);
    PUT(d_o, int32_t, (const int32_t*)nullptr, (size_t)n_paths);
    CK(dp_launch_nearest(n_paths, d_off, d_pxy, d_qx, d_qy, d_o, c->st[0]));
    ++c->launches;
    CK(cudaMemcpyAsync(out_id, d_o, (size_t)n_paths * sizeof(int32_t), cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    return DP_OK;
}

int dp_score_candidates(dp_ctx* c, const double* base_x, const double* base_y, int n_base, const double* offset, const int32_t* n_pts,
                        int n_cand, const double* ox, const double* oy, const double* dvx, const double* dvy, int n_obs, double lat_min,
                        double lat_max, double clear_dis, int32_t* best_index, double* best_dis_lng, double* out_dis_lng) {
    if (!c || !base_x || !base_y || n_base < 2 || n_base > 256 || !offset || !n_pts || n_cand <= 0 || n_obs < 0 || n_obs > 192 || !best_index)
        return fail(DP_ERR_ARG, "dp_score_candidates: bad argument (n_base in [2,256], n_obs <= 192)");
    CK(cudaSetDevice(c->device));
    Tmp tmp; cudaError_t e;
    const SweepGroups sg = build_sweep_groups(nullptr, offset, n_pts, n_cand, n_base);
    const int n_rows = (int)sg.row_off.size();
    std::vector<double> line((size_t)2 * n_base);           // lines[1][2][n_base]
    memcpy(line.data(), base_x, (size_t)n_base * 8); memcpy(line.data() + n_base, base_y, (size_t)n_base * 8);
    PUT(d_lines, double, line.data(), line.size());
    PUT(d_roff, double, sg.row_off.data(), sg.row_off.size());
    PUT(d_gP, int32_t, sg.group_P.data(), sg.group_P.size()); PUT(d_cg, int32_t, sg.cand_group.data(), (size_t)n_cand);
    PUT(d_rinfo, int32_t, sg.row_info.data(), sg.row_info.size());
    PUT(d_grow, int32_t, sg.group_row.data(), sg.group_row.size());
    PUT(d_rcum, double, (const double*)nullptr, sg.row_off.size() * 256);
    PUT(d_gkey, unsigned, (const unsigned*)nullptr, sg.group_P.size());
    PUT(d_ox, double, ox, (size_t)n_obs); PUT(d_oy, double, oy, (size_t)n_obs);
    double* d_vx = nullptr; double* d_vy = nullptr;
    if (dvx && dvy) { d_vx = tmp.put<double>(dvx, (size_t)n_obs, e); if (e != cudaSuccess) return fail(DP_ERR_CUDA, "staging", e);
                      d_vy = tmp.put<double>(dvy, (size_t)n_obs, e); if (e != cudaSuccess) return fail(DP_ERR_CUDA, "staging", e); }
    PUT(d_dis, double, (const double*)nullptr, (size_t)n_cand);
    PUT(d_key, unsigned long long, (const unsigned long long*)nullptr, 1);
    CK(cudaMemsetAsync(d_key, 0xff, 8, c->st[0]));
    const int4* d_ri = reinterpret_cast<const int4*>(d_rinfo);
    CK(dp_launch_sweep_prefix(d_lines, n_base, n_rows, d_roff, d_ri, d_rcum, c->st[0]));
    CK(dp_launch_sweep(d_lines, n_base, 1, n_rows, d_roff, d_ri, d_gP, d_grow, d_cg, n_cand, d_ox, d_oy, d_vx, d_vy, n_obs, lat_min, lat_max,
                       clear_dis, d_gkey, d_rcum, d_dis, d_key, c->st[0]));
    c->launches += 3;
    ++c->launches;
    unsigned long long key = ~0ull;
    CK(cudaMemcpyAsync(&key, d_key, 8, cudaMemcpyDeviceToHost, c->st[0]));
    std::vector<double> dis;
    if (out_dis_lng) CK(cudaMemcpyAsync(out_dis_lng, d_dis, (size_t)n_cand * 8, cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    const bool feasible = (key >> 32) == 0;
    *best_index = feasible ? (int32_t)(key & 0xffffffffu) : -1;
    if (best_dis_lng) {
        *best_dis_lng = DP_NOT_FOUND;
        if (feasible) CK(cudaMemcpy(best_dis_lng, d_dis + *best_index, 8, cudaMemcpyDeviceToHost));
    }
    return DP_OK;
}

// ---- latency-mode sweep session: device-resident candidate set + one captured CUDA graph per scoring call ----
struct dp_sweep {
    dp_ctx* c = nullptr;
    int n_base = 0, n_lines = 1, n_cand = 0, max_obs = 0;
    double *d_lines = nullptr, *d_roff = nullptr, *d_rcum = nullptr;   // d_lines: [n_lines][2][n_base] base lines
    double* d_poses = nullptr;                              // Bezier sessions: [n_lines][6] end poses of the lines
    int32_t *d_gP = nullptr, *d_rinfo = nullptr;            // rows / horizon groups of the candidate set (build_sweep_groups)
    int32_t* d_gfirst = nullptr;                            // lowest candidate index per group
    unsigned* d_done = nullptr;                             // row counter of the fused launch (0 between calls)
    int n_rows = 0, n_groups = 0, first_nogroup = -1;
    unsigned long long* d_res = nullptr;                    // {packed key, dis_lng bits} per row of the call in flight
    double* h_obs = nullptr;                                // [4][192] staging of the caller's obstacle arrays
    unsigned long long* h_out = nullptr;                    // page-locked {packed key, dis_lng bits, sequence}: written by the grid's last CTA
    unsigned long long* h_out_dev = nullptr;                // ... as the device addresses it
    unsigned long long seq = 0;
    long long* d_dbg = nullptr;                             // DP_SWEEP_DBG=1: phase stamps of the row owners (tools/sweep_probe.py)
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};

// lines_xy: host [n_lines][2][n_base] or null (Bezier sessions fill the lines on the device, dp_sweep_set_bezier)
static int sweep_create(dp_ctx* c, dp_sweep** out, const double* lines_xy, int n_lines, int n_base, const int32_t* cand_line, const double* offset,
                        const int32_t* n_pts, int n_cand, int max_obs) {
    CK(cudaSetDevice(c->device));
    dp_sweep* s = new dp_sweep();
    s->c = c; s->n_base = n_base; s->n_lines = n_lines; s->n_cand = n_cand; s->max_obs = max_obs;
    const SweepGroups sg = build_sweep_groups(cand_line, offset, n_pts, n_cand, n_base);
    s->n_rows = (int)sg.row_off.size(); s->n_groups = (int)sg.group_P.size();
    const size_t line_bytes = (size_t)n_lines * 2 * n_base * 8;
    CK(cudaMalloc((void**)&s->d_lines, line_bytes)); CK(cudaMemset(s->d_lines, 0, line_bytes));
    CK(cudaMalloc((void**)&s->d_poses, (size_t)n_lines * 6 * 8));
    CK(cudaMalloc((void**)&s->d_roff, (sg.row_off.size() + 1) * 8));
    CK(cudaMalloc((void**)&s->d_gP, (sg.group_P.size() + 1) * 4)); CK(cudaMalloc((void**)&s->d_rinfo, (sg.row_info.size() + 4) * 4));
    CK(cudaMalloc((void**)&s->d_rcum, (sg.row_off.size() + 1) * 256 * 8));
    CK(cudaMalloc((void**)&s->d_gfirst, (sg.group_P.size() + 1) * 4)); CK(cudaMalloc((void**)&s->d_res, (sg.row_off.size() + 1) * 16));
    CK(cudaMalloc((void**)&s->d_done, 4));
    CK(cudaMemset(s->d_done, 0, 4));
    CK(cudaHostAlloc((void**)&s->h_obs, (size_t)4 * 192 * 8, cudaHostAllocMapped));
    CK(cudaHostAlloc((void**)&s->h_out, 3 * 8, cudaHostAllocMapped));
    s->h_out[0] = s->h_out[1] = s->h_out[2] = 0;
    CK(cudaHostGetDevicePointer((void**)&s->h_out_dev, s->h_out, 0));
    s->first_nogroup = sg.first_nogroup;
    if (getenv("DP_SWEEP_DBG")) { CK(cudaMalloc((void**)&s->d_dbg, (size_t)(s->n_rows + 1) * 64)); CK(cudaMemset(s->d_dbg, 0, (size_t)(s->n_rows + 1) * 64)); }
    if (lines_xy) CK(cudaMemcpy(s->d_lines, lines_xy, line_bytes, cudaMemcpyHostToDevice));
    if (s->n_rows) CK(cudaMemcpy(s->d_roff, sg.row_off.data(), sg.row_off.size() * 8, cudaMemcpyHostToDevice));
    if (s->n_groups) CK(cudaMemcpy(s->d_gP, sg.group_P.data(), sg.group_P.size() * 4, cudaMemcpyHostToDevice));
    if (s->n_rows) CK(cudaMemcpy(s->d_rinfo, sg.row_info.data(), sg.row_info.size() * 4, cudaMemcpyHostToDevice));
    if (s->n_groups) CK(cudaMemcpy(s->d_gfirst, sg.group_first.data(), sg.group_first.size() * 4, cudaMemcpyHostToDevice));
    // the arclength prefix of every row does not depend on the obstacles: once, here (Bezier sessions: with every set of poses)
    if (lines_xy) {
        CK(dp_launch_sweep_prefix(s->d_lines, n_base, s->n_rows, s->d_roff, reinterpret_cast<const int4*>(s->d_rinfo), s->d_rcum, c->st[0]));
        ++c->launches;
    }
    CK(cudaStreamSynchronize(c->st[0]));
    CK(cudaEventCreate(&s->e0)); CK(cudaEventCreate(&s->e1));
    *out = s;
    return DP_OK;
}

int dp_sweep_create(dp_ctx* c, dp_sweep** out, const double* base_x, const double* base_y, int n_base, const double* offset,
                    const int32_t* n_pts, int n_cand, int max_obs) {
    if (!c || !out || !base_x || !base_y || n_base < 2 || n_base > 256 || !offset || !n_pts || n_cand <= 0 || max_obs <= 0 || max_obs > 192)
        return fail(DP_ERR_ARG, "dp_sweep_create: bad argument (n_base in [2,256], max_obs <= 192)");
    std::vector<double> line((size_t)2 * n_base);
    memcpy(line.data(), base_x, (size_t)n_base * 8); memcpy(line.data() + n_base, base_y, (size_t)n_base * 8);
    return sweep_create(c, out, line.data(), 1, n_base, nullptr, offset, n_pts, n_cand, max_obs);
}

int dp_sweep_create_lines(dp_ctx* c, dp_sweep** out, const double* lines_xy, int n_lines, int n_base, const int32_t* cand_line,
                          const double* offset, const int32_t* n_pts, int n_cand, int max_obs) {
    if (!c || !out || !lines_xy || n_lines <= 0 || n_base < 2 || n_base > 256 || !cand_line || !offset || !n_pts || n_cand <= 0 || max_obs <= 0 ||
        max_obs > 192)
        return fail(DP_ERR_ARG, "dp_sweep_create_lines: bad argument (n_base in [2,256], max_obs <= 192)");
    for (int i = 0; i < n_cand; ++i) if (cand_line[i] < 0 || cand_line[i] >= n_lines) return fail(DP_ERR_ARG, "dp_sweep_create_lines: cand_line out of range");
    return sweep_create(c, out, lines_xy, n_lines, n_base, cand_line, offset, n_pts, n_cand, max_obs);
}

int dp_sweep_create_bezier(dp_ctx* c, dp_sweep** out, int n_lines, const int32_t* cand_line, const double* offset, const int32_t* n_pts, int n_cand,
                           int max_obs) {
    if (!c || !out || n_lines <= 0 || !cand_line || !offset || !n_pts || n_cand <= 0 || max_obs <= 0 || max_obs > 192)
        return fail(DP_ERR_ARG, "dp_sweep_create_bezier: bad argument (max_obs <= 192)");
    for (int i = 0; i < n_cand; ++i) if (cand_line[i] < 0 || cand_line[i] >= n_lines) return fail(DP_ERR_ARG, "dp_sweep_create_bezier: cand_line out of range");
    return sweep_create(c, out, nullptr, n_lines, DP_PATH_POINTS, cand_line, offset, n_pts, n_cand, max_obs);
}

int dp_sweep_set_bezier(dp_sweep* s, const double* poses, float* device_ms) {
    if (!s || !poses || s->n_base != DP_PATH_POINTS) return fail(DP_ERR_ARG, "dp_sweep_set_bezier: not a Bezier session");
    dp_ctx* c = s->c;
    CK(cudaSetDevice(c->device));
    cudaStream_t st = c->st[0];
    CK(cudaMemcpyAsync(s->d_poses, poses, (size_t)s->n_lines * 6 * 8, cudaMemcpyHostToDevice, st));
    if (device_ms) CK(cudaEventRecord(s->e0, st));
    CK(dp_launch_bezier(s->n_lines, s->d_poses, s->d_lines, st));   // out[n][2][200] IS the lines layout
    CK(dp_launch_sweep_prefix(s->d_lines, s->n_base, s->n_rows, s->d_roff, reinterpret_cast<const int4*>(s->d_rinfo), s->d_rcum, st));
    c->launches += 2;
    if (device_ms) { CK(cudaEventRecord(s->e1, st)); CK(cudaEventSynchronize(s->e1)); CK(cudaEventElapsedTime(device_ms, s->e0, s->e1)); }
    return DP_OK;                                           // (stream order: the next dp_sweep_score sees the new lines)
}

int dp_sweep_lines(dp_sweep* s, double* lines_xy_out) {
    if (!s || !lines_xy_out) return fail(DP_ERR_ARG, "dp_sweep_lines: null");
    CK(cudaSetDevice(s->c->device));
    CK(cudaMemcpyAsync(lines_xy_out, s->d_lines, (size_t)s->n_lines * 2 * s->n_base * 8, cudaMemcpyDeviceToHost, s->c->st[0]));
    CK(cudaStreamSynchronize(s->c->st[0]));
    return DP_OK;
}

int dp_sweep_score(dp_sweep* s, const double* ox, const double* oy, const double* dvx, const double* dvy, int n_obs, double lat_min,
                   double lat_max, double clear_dis, int32_t* best_index, double* best_dis_lng, float* device_ms) {
    if (!s || !best_index || n_obs < 0 || n_obs > s->max_obs || (n_obs > 0 && (!ox || !oy))) return fail(DP_ERR_ARG, "dp_sweep_score: bad argument");
    dp_ctx* c = s->c;
    CK(cudaSetDevice(c->device));
    cudaStream_t st = c->st[0];
    const int mo = 192;                                      // staging stride (SWEEP_MAX_OBS)
    for (int i = 0; i < n_obs; ++i) {
        s->h_obs[i] = ox[i]; s->h_obs[mo + i] = oy[i];
        s->h_obs[2 * mo + i] = dvx ? dvx[i] : 0.0; s->h_obs[3 * mo + i] = dvy ? dvy[i] : 0.0;
    }
    // ONE launch: the obstacle tracks travel in the kernel parameters, the grid's last CTA writes the winner into page-locked
    // memory and re-arms the device state; the host watches the sequence word instead of synchronising the stream
    const unsigned long long seq = ++s->seq;
    if (device_ms) CK(cudaEventRecord(s->e0, st));
    CK(dp_launch_sweep_fused(s->d_lines, s->n_base, s->n_lines, s->n_rows, s->d_roff, reinterpret_cast<const int4*>(s->d_rinfo), s->d_gP, s->d_gfirst,
                             s->first_nogroup, s->h_obs, mo, n_obs, lat_min, lat_max, clear_dis, s->d_rcum, s->d_res, s->d_done, s->h_out_dev, seq,
                             s->d_dbg, st));
    ++c->launches;
    if (device_ms) CK(cudaEventRecord(s->e1, st));
    volatile unsigned long long* ho = s->h_out;
    for (unsigned spin = 1; ho[2] != seq; ++spin) {
        if ((spin & 0xfffff) == 0) {                        // every ~million polls: has the launch died?
            const cudaError_t q = cudaStreamQuery(st);
            if (q != cudaSuccess && q != cudaErrorNotReady) return fail(DP_ERR_CUDA, "dp_sweep_score: launch failed", q);
            if (q == cudaSuccess && ho[2] != seq) return fail(DP_ERR_CUDA, "dp_sweep_score: launch finished without a result");
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    const unsigned long long key = ho[0], dbits = ho[1];
    if (device_ms) { CK(cudaEventSynchronize(s->e1)); CK(cudaEventElapsedTime(device_ms, s->e0, s->e1)); }
    const bool feasible = (key >> 32) == 0;
    *best_index = feasible ? (int32_t)(key & 0xffffffffu) : -1;
    if (best_dis_lng) {
        *best_dis_lng = DP_NOT_FOUND;
        if (feasible) memcpy(best_dis_lng, &dbits, 8);
    }
    return DP_OK;
}
/* diagnostic: globaltimer stamps [n_rows][8] of the last dp_sweep_score (sessions created with DP_SWEEP_DBG=1 only) */
int dp_sweep_debug(dp_sweep* s, long long* out, int n_rows) {
    if (!s || !out || !s->d_dbg || n_rows > s->n_rows + 1) return fail(DP_ERR_STATE, "dp_sweep_debug: session was created without DP_SWEEP_DBG=1");
    CK(cudaSetDevice(s->c->device));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out, s->d_dbg, (size_t)n_rows * 64, cudaMemcpyDeviceToHost));
    return DP_OK;
}

int dp_sweep_destroy(dp_sweep* s) {
    if (!s) return DP_OK;
    cudaSetDevice(s->c->device);
    cudaStreamSynchronize(s->c->st[0]);
    cudaFree(s->d_lines); cudaFree(s->d_poses); cudaFree(s->d_roff); cudaFree(s->d_gP); cudaFree(s->d_rinfo); cudaFree(s->d_rcum);
    cudaFree(s->d_dbg); cudaFree(s->d_gfirst); cudaFree(s->d_res); cudaFree(s->d_done);
    cudaFreeHost(s->h_obs); cudaFreeHost(s->h_out);
    if (s->e0) cudaEventDestroy(s->e0);
    if (s->e1) cudaEventDestroy(s->e1);
    delete s;
    return DP_OK;
}

int dp_measure_fma_peak(dp_ctx* c, double* fp64_tflops, double* fp32_tflops) {
    if (!c) return fail(DP_ERR_ARG, "dp_measure_fma_peak");
    CK(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, c->device));
    float* sink = nullptr;
    CK(cudaMalloc((void**)&sink, 64));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    const int blocks = prop.multiProcessorCount * 8, iters = 4096;
    double out[2] = {0, 0};
    for (int which = 0; which < 2; ++which) {
        double best = 0;
        for (int rep = 0; rep < 4; ++rep) {
            CK(cudaEventRecord(a, c->st[0]));
            CK(dp_launch_fma_peak(which, sink, iters, blocks, c->st[0]));
            ++c->launches;
            CK(cudaEventRecord(b, c->st[0]));
            CK(cudaEventSynchronize(b));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, a, b));
            const double flops = 2.0 * 64.0 * iters * 256.0 * blocks;   // 64 fma per iteration per thread
            const double tf = flops / (ms * 1e-3) / 1e12;
            if (rep > 0 && tf > best) best = tf;
        }
        out[which] = best;
    }
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(sink);
    if (fp64_tflops) *fp64_tflops = out[0];
    if (fp32_tflops) *fp32_tflops = out[1];
    return DP_OK;
}

// ---- (8) output stage ----
int dp_pack_frames_dev(dp_ctx* c, int first, int n, const dp_plan_record* rec, dp_ctrl_frame* ctrl, dp_status_frame* status, void* stream) {
    if (!c || !rec || n < 0 || first < 0 || first + n > c->max_scenes) return fail(DP_ERR_ARG, "dp_pack_frames_dev: bad argument");
    CK(cudaSetDevice(c->device));
    if (!ctrl && !status) return DP_OK;
    c->launches += n > 0 ? 1 : 0;
    CK(dp_launch_frames(c->p, n, rec, c->d_last + (size_t)first * DP_PATH_POINTS, ctrl, status, (cudaStream_t)stream));
    return DP_OK;
}
int dp_pack_frames(dp_ctx* c, int first, int n, const dp_plan_record* rec, dp_ctrl_frame* ctrl, dp_status_frame* status) {
    if (!c || !rec || n < 0 || first < 0 || first + n > c->max_scenes) return fail(DP_ERR_ARG, "dp_pack_frames: bad argument");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_pack_frames: submitted cycles in flight, call dp_cycle_wait first");
    CK(cudaSetDevice(c->device));
    if (n == 0 || (!ctrl && !status)) return DP_OK;
    Tmp t;
    cudaError_t e = cudaSuccess;
    dp_plan_record* d_rec = t.put(rec, (size_t)n, e);
    if (e != cudaSuccess) return fail(DP_ERR_CUDA, "dp_pack_frames: staging", e);
    dp_ctrl_frame* d_c = ctrl ? t.put((const dp_ctrl_frame*)nullptr, (size_t)n, e) : nullptr;
    if (e != cudaSuccess) return fail(DP_ERR_NOMEM, "dp_pack_frames: staging", e);
    dp_status_frame* d_s = status ? t.put((const dp_status_frame*)nullptr, (size_t)n, e) : nullptr;
    if (e != cudaSuccess) return fail(DP_ERR_NOMEM, "dp_pack_frames: staging", e);
    cudaStream_t st = c->st[0];
    c->launches += 1;
    CK(dp_launch_frames(c->p, n, d_rec, c->d_last + (size_t)first * DP_PATH_POINTS, d_c, d_s, st));
    if (ctrl) CK(cudaMemcpyAsync(ctrl, d_c, (size_t)n * sizeof(dp_ctrl_frame), cudaMemcpyDeviceToHost, st));
    if (status) CK(cudaMemcpyAsync(status, d_s, (size_t)n * sizeof(dp_status_frame), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return DP_OK;
}

// ---- (10) V2X event handlers ----
int dp_v2x_event_batch_dev(dp_ctx* c, int n, const dp_scene_hdr* hdr, const dp_v2x_data* v2x, const double* wp_lat, const double* wp_lng, int mode,
                           dp_v2x_flags* out, void* stream) {
    if (!c || !hdr || !v2x || !out || n < 0 || (mode != 0 && mode != 1)) return fail(DP_ERR_ARG, "dp_v2x_event_batch_dev: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_v2x_event_batch_dev: map not uploaded");
    CK(cudaSetDevice(c->device));
    c->launches += n > 0 ? 1 : 0;
    CK(dp_launch_v2x(c->gmap, c->p, n, hdr, v2x, wp_lat, wp_lng, mode, out, (cudaStream_t)stream));
    return DP_OK;
}
int dp_v2x_event_batch(dp_ctx* c, int n, const dp_scene_hdr* hdr, const dp_v2x_data* v2x, const double* wp_lat, const double* wp_lng, int n_wp,
                       int mode, dp_v2x_flags* out) {
    if (!c || !hdr || !v2x || !out || n < 0 || n_wp < 0 || (n_wp > 0 && (!wp_lat || !wp_lng)) || (mode != 0 && mode != 1))
        return fail(DP_ERR_ARG, "dp_v2x_event_batch: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_v2x_event_batch: map not uploaded");
    for (int s = 0; s < n; ++s)                             // the slices must lie inside the list, and the ego inside the map tables
        if (v2x[s].wp_count < 0 || (v2x[s].wp_count > 0 && (v2x[s].wp_first < 0 || v2x[s].wp_first + v2x[s].wp_count > n_wp)) ||
            hdr[s].road_num < 1 || hdr[s].road_num > c->gmap.n_roads || hdr[s].lane_num < 1 || hdr[s].lane_num > DP_LANESUM)
            return fail(DP_ERR_ARG, "dp_v2x_event_batch: scene header or warning-point slice out of range");
    CK(cudaSetDevice(c->device));
    if (n == 0) return DP_OK;
    Tmp t;
    cudaError_t e = cudaSuccess;
    dp_scene_hdr* d_h = t.put(hdr, (size_t)n, e);
    if (e != cudaSuccess) return fail(DP_ERR_CUDA, "dp_v2x_event_batch: staging", e);
    dp_v2x_data* d_v = t.put(v2x, (size_t)n, e);
    if (e != cudaSuccess) return fail(DP_ERR_CUDA, "dp_v2x_event_batch: staging", e);
    double* d_la = t.put(wp_lat, (size_t)n_wp, e);
    if (e != cudaSuccess) return fail(DP_ERR_CUDA, "dp_v2x_event_batch: staging", e);
    double* d_lo = t.put(wp_lng, (size_t)n_wp, e);
    if (e != cudaSuccess) return fail(DP_ERR_CUDA, "dp_v2x_event_batch: staging", e);
    dp_v2x_flags* d_o = t.put((const dp_v2x_flags*)nullptr, (size_t)n, e);
    if (e != cudaSuccess) return fail(DP_ERR_NOMEM, "dp_v2x_event_batch: staging", e);
    c->launches += 1;
    CK(dp_launch_v2x(c->gmap, c->p, n, d_h, d_v, d_la, d_lo, mode, d_o, c->st[0]));
    CK(cudaMemcpyAsync(out, d_o, (size_t)n * sizeof(dp_v2x_flags), cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    return DP_OK;
}

int dp_v2x_apply_dev(dp_ctx* c, int n, const dp_v2x_flags* flags, dp_plan_record* rec, void* stream) {
    if (!c || !flags || !rec || n < 0) return fail(DP_ERR_ARG, "dp_v2x_apply_dev: bad argument");
    CK(cudaSetDevice(c->device));
    c->launches += n > 0 ? 1 : 0;
    CK(dp_launch_v2x_apply(n, flags, rec, (cudaStream_t)stream));
    return DP_OK;
}
int dp_v2x_apply(dp_ctx* c, int n, const dp_v2x_flags* flags, dp_plan_record* rec) {
    if (!c || !flags || !rec || n < 0) return fail(DP_ERR_ARG, "dp_v2x_apply: bad argument");
    CK(cudaSetDevice(c->device));
    if (n == 0) return DP_OK;
    Tmp t;
    cudaError_t e = cudaSuccess;
    dp_v2x_flags* d_f = t.put(flags, (size_t)n, e);
    if (e != cudaSuccess) return fail(DP_ERR_CUDA, "dp_v2x_apply: staging", e);
    dp_plan_record* d_r = t.put((const dp_plan_record*)rec, (size_t)n, e);
    if (e != cudaSuccess) return fail(DP_ERR_CUDA, "dp_v2x_apply: staging", e);
    c->launches += 1;
    CK(dp_launch_v2x_apply(n, d_f, d_r, c->st[0]));
    CK(cudaMemcpyAsync(rec, d_r, (size_t)n * sizeof(dp_plan_record), cudaMemcpyDeviceToHost, c->st[0]));
    CK(cudaStreamSynchronize(c->st[0]));
    return DP_OK;
}

// ---- (9) closed-loop episodes ----
void dp_world_default_params(dp_world_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->a_max = 3.0; p->loc_back = 8; p->loc_fwd = 56; p->end_margin = 160;
}
namespace {
// the world options are baked into the launches of a cached episode graph: a change drops it
int drop_episode_graph(dp_ctx* c) {
    if (c->ep_exec) { cudaGraphExecDestroy(c->ep_exec); c->ep_exec = nullptr; }
    return DP_OK;
}
bool all_finite(std::initializer_list<double> v) {
    for (double x : v) if (!std::isfinite(x)) return false;
    return true;
}
}  // namespace
int dp_world_set_params(dp_ctx* c, const dp_world_params* p) {
    if (!c || !p || !(p->a_max >= 0) || p->loc_back < 0 || p->loc_fwd < 0) return fail(DP_ERR_ARG, "dp_world_set_params: bad argument");
    c->world.wp = *p;
    return drop_episode_graph(c);
}
void dp_metrics_default_params(dp_metrics_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->front = 4.0; p->rear = 1.0; p->half_width = 0.9; p->corridor_half = 1.1; p->ttc_warn = 2.0;
}
int dp_world_set_metrics(dp_ctx* c, const dp_metrics_params* p, dp_episode_metrics* m) {
    if (!c || (m && !p)) return fail(DP_ERR_ARG, "dp_world_set_metrics: bad argument");
    if (p) {
        if (!all_finite({p->front, p->rear, p->half_width, p->corridor_half, p->ttc_warn}))
            return fail(DP_ERR_ARG, "dp_world_set_metrics: parameters must be finite");
        if (!(p->front >= 0) || !(p->rear >= 0) || !(p->half_width > 0) || !(p->corridor_half >= 0) || !(p->ttc_warn >= 0))
            return fail(DP_ERR_ARG, "dp_world_set_metrics: front, rear, corridor_half, ttc_warn >= 0 and half_width > 0");
        if (m) c->world.mp = *p;
    }
    c->world.met = m;
    return drop_episode_graph(c);
}
void dp_agent_model_default_params(dp_agent_model_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->a_max = 1.0; p->b = 1.5; p->b_max = 8.0; p->T = 1.5; p->s0 = 2.0; p->length = 4.5; p->ego_rear = 1.0; p->look = 100.0;
}
int dp_world_set_agent_model(dp_ctx* c, const dp_agent_model_params* p, const double* v0) {
    if (!c || (v0 && !p)) return fail(DP_ERR_ARG, "dp_world_set_agent_model: bad argument");
    if (p) {
        if (!all_finite({p->a_max, p->b, p->b_max, p->T, p->s0, p->length, p->ego_rear, p->look}))
            return fail(DP_ERR_ARG, "dp_world_set_agent_model: parameters must be finite");
        if (!(p->a_max > 0) || !(p->b > 0) || !(p->b_max > 0) || !(p->T > 0) || !(p->length > 0) || !(p->look > 0) || !(p->s0 >= 0) ||
            !(p->ego_rear >= 0))
            return fail(DP_ERR_ARG, "dp_world_set_agent_model: a_max, b, b_max, T, length, look > 0 and s0, ego_rear >= 0");
    }
    if (v0) {
        if (c->max_obs > DP_AGENT_MODEL_MAX_OBS)
            return fail(DP_ERR_ARG, "dp_world_set_agent_model: the context's max_obs exceeds DP_AGENT_MODEL_MAX_OBS");
        CK(cudaSetDevice(c->device));
        CK(dp_world_prepare());                             // function attributes are set before any launch or capture of the armed step
        c->world.amp = *p;
    }
    c->world.v0 = v0;
    if (!v0) c->world.lcs = nullptr;                        // lane changes run on the react phase
    return drop_episode_graph(c);
}
void dp_lane_change_default_params(dp_lane_change_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->politeness = 0.2; p->a_thr = 0.2; p->b_safe = 4.0; p->ego_b_safe = 4.0; p->ego_front = 4.0; p->lat_speed = 1.0;
    p->cooldown = 5.0; p->end_guard = 30.0;
}
int dp_world_set_lane_change(dp_ctx* c, const dp_lane_change_params* p, dp_lane_change_state* st) {
    if (!c || (st && !p)) return fail(DP_ERR_ARG, "dp_world_set_lane_change: bad argument");
    if (p) {
        if (!all_finite({p->politeness, p->a_thr, p->b_safe, p->ego_b_safe, p->ego_front, p->lat_speed, p->cooldown, p->end_guard}))
            return fail(DP_ERR_ARG, "dp_world_set_lane_change: parameters must be finite");
        if (!(p->lat_speed > 0) || !(p->b_safe > 0) || !(p->ego_b_safe > 0) || !(p->politeness >= 0) || !(p->cooldown >= 0) ||
            !(p->end_guard >= 0) || !(p->ego_front >= 0))
            return fail(DP_ERR_ARG, "dp_world_set_lane_change: lat_speed, b_safe, ego_b_safe > 0 and politeness, cooldown, end_guard, ego_front >= 0");
    }
    if (st) {
        if (!c->world.v0) return fail(DP_ERR_ARG, "dp_world_set_lane_change: the agent model is not armed (dp_world_set_agent_model)");
        CK(cudaSetDevice(c->device));
        CK(dp_world_prepare());                             // function attributes are set before any launch or capture of the armed step
        c->world.lcp = *p;
    }
    c->world.lcs = st;
    return drop_episode_graph(c);
}
int dp_world_set_v2x(dp_ctx* c, const dp_v2x_world_params* vp, int n, const dp_v2x_event_spec* spec, const double* wp_x, const double* wp_y,
                     int n_wp, dp_v2x_flags* flags, dp_v2x_episode_stats* stats) {
    if (!c) return fail(DP_ERR_ARG, "dp_world_set_v2x: bad argument");
    if (!spec) {
        c->v2x = DpV2xOpts{};
        return drop_episode_graph(c);
    }
    if (!vp || !stats || n < 0 || n_wp < 0 || (n_wp > 0 && (!wp_x || !wp_y)) || (vp->mode != 0 && vp->mode != 1) ||
        (vp->apply != 0 && vp->apply != 1))
        return fail(DP_ERR_ARG, "dp_world_set_v2x: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_world_set_v2x: map not uploaded");
    CK(cudaSetDevice(c->device));
    std::vector<dp_v2x_event_spec> h((size_t)n);
    if (n > 0) CK(cudaMemcpy(h.data(), spec, (size_t)n * sizeof(dp_v2x_event_spec), cudaMemcpyDeviceToHost));
    for (const dp_v2x_event_spec& e : h) {
        if (!all_finite({e.sig_cycle, e.sig_green, e.sig_yellow, e.sig_red, e.sig_offset, e.sig_range, e.ped_x, e.ped_y, e.ped_vx, e.ped_vy,
                         e.ped_t_on, e.ped_t_off, e.ped_range, e.rw_x, e.rw_y, e.rw_range}))
            return fail(DP_ERR_ARG, "dp_world_set_v2x: specifications must be finite");
        if (!(e.sig_range >= 0) || !(e.ped_range >= 0) || !(e.rw_range >= 0))
            return fail(DP_ERR_ARG, "dp_world_set_v2x: ranges must be >= 0");
        if (e.sig_road < 0 || e.sig_road > c->gmap.n_roads || e.sig_stop < -1)
            return fail(DP_ERR_ARG, "dp_world_set_v2x: sig_road outside [0, n_roads] or sig_stop < -1");
        if (e.sig_road > 0 && (!(e.sig_green > 0) || !(e.sig_yellow > 0) || !(e.sig_red > 0) || !(e.sig_cycle > 0) ||
                               !(std::fabs(e.sig_green + e.sig_yellow + e.sig_red - e.sig_cycle) <= 1e-9 * e.sig_cycle)))
            return fail(DP_ERR_ARG, "dp_world_set_v2x: signal durations must be > 0 and sum to the cycle");
        if (e.has_works && (e.wp_count < 0 || (e.wp_count > 0 && (e.wp_first < 0 || e.wp_first > n_wp - e.wp_count))))
            return fail(DP_ERR_ARG, "dp_world_set_v2x: warning-point slice out of range");
    }
    c->v2x.vp = *vp; c->v2x.spec = spec; c->v2x.wp_x = wp_x; c->v2x.wp_y = wp_y; c->v2x.flags = flags; c->v2x.stats = stats; c->v2x.n = n;
    return drop_episode_graph(c);
}
int dp_v2x_world_dev(dp_ctx* c, int first, int n, const dp_scene_hdr* hdr, dp_plan_record* rec, int cycle, void* stream) {
    if (!c || !hdr || n < 0 || first < 0 || first + n > c->max_scenes || cycle < 0) return fail(DP_ERR_ARG, "dp_v2x_world_dev: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_v2x_world_dev: map not uploaded");
    if (!c->v2x.spec) return fail(DP_ERR_STATE, "dp_v2x_world_dev: V2X is not armed (dp_world_set_v2x)");
    if (n > c->v2x.n) return fail(DP_ERR_ARG, "dp_v2x_world_dev: more scenes than the armed specifications");
    CK(cudaSetDevice(c->device));
    c->launches += n > 0 ? 1 : 0;
    CK(dp_launch_world_v2x(c->gmap, c->p, c->v2x, n, hdr, rec, cycle, (cudaStream_t)stream));
    return DP_OK;
}
int dp_world_step_dev(dp_ctx* c, int first, int n, dp_scene_hdr* hdr, dp_agent* agents, double* ox, double* oy, const dp_plan_record* rec,
                      void* stream) {
    if (!c || !hdr || !agents || !ox || !oy || n < 0 || first < 0 || first + n > c->max_scenes)
        return fail(DP_ERR_ARG, "dp_world_step_dev: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_world_step_dev: map not uploaded");
    CK(cudaSetDevice(c->device));
    c->launches += n > 0 ? 1 : 0;
    const DpWorldBufs b = {n, c->max_obs, hdr, agents, ox, oy, rec, c->d_last + (size_t)first * DP_PATH_POINTS};
    CK(dp_launch_world(c->gmap, c->p, c->world, b, (cudaStream_t)stream));
    return DP_OK;
}
namespace {
// the launches of one closed-loop episode, in order, on st (a capturing stream, or the caller's)
cudaError_t enqueue_closed_loop(dp_ctx* c, int first, int n, int cycles, dp_scene_hdr* hdr, dp_agent* agents, double* ox, double* oy,
                                dp_plan_record* rec, dp_scene_hdr* hdr_log, double* olx, double* oly, cudaStream_t st, bool rearm) {
    const size_t mo = (size_t)c->max_obs;
    DpWorldBufs b = {n, c->max_obs, hdr, agents, ox, oy, nullptr, c->d_last + (size_t)first * DP_PATH_POINTS};
    cudaError_t e;
    // a replayed graph re-uses its hand-off epochs: the per-scene Decision -> Planning flags start every replay from 0
    if (rearm && (e = cudaMemsetAsync(c->d_done + first, 0, (size_t)n * sizeof(unsigned), st)) != cudaSuccess) return e;
    c->launches += 1;
    if ((e = dp_launch_world(c->gmap, c->p, c->world, b, st)) != cudaSuccess) return e;
    for (int k = 0; k < cycles; ++k) {
        if (hdr_log && (e = cudaMemcpyAsync(hdr_log + (size_t)k * n, hdr, (size_t)n * sizeof(dp_scene_hdr), cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
        if (olx && (e = cudaMemcpyAsync(olx + (size_t)k * n * mo, ox, (size_t)n * mo * sizeof(double), cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
        if (oly && (e = cudaMemcpyAsync(oly + (size_t)k * n * mo, oy, (size_t)n * mo * sizeof(double), cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
        const DpIo io = make_io(c, first, nullptr);
        if ((e = run_cycle(c, first, n, hdr, ox, oy, rec + (size_t)k * n, nullptr, nullptr, nullptr, st, io)) != cudaSuccess) return e;
        if (c->v2x.spec) {                                  // V2X armed: the flags act on the records before the world step reads them
            c->launches += 1;
            if ((e = dp_launch_world_v2x(c->gmap, c->p, c->v2x, n, hdr, rec + (size_t)k * n, k, st)) != cudaSuccess) return e;
        }
        c->launches += 1;
        b.rec = rec + (size_t)k * n;
        if ((e = dp_launch_world(c->gmap, c->p, c->world, b, st)) != cudaSuccess) return e;
    }
    if (c->v2x.spec) {                                      // the tally: closes the red-crossing check of the last world step
        c->launches += 1;
        if ((e = dp_launch_world_v2x(c->gmap, c->p, c->v2x, n, hdr, nullptr, cycles, st)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}
}  // namespace
int dp_run_closed_loop_dev(dp_ctx* c, int first, int n, int cycles, dp_scene_hdr* hdr, dp_agent* agents, double* ox, double* oy,
                           dp_plan_record* rec, dp_scene_hdr* hdr_log, double* olx, double* oly, void* stream) {
    if (!c || !hdr || !agents || !ox || !oy || !rec || n < 0 || cycles < 0 || first < 0 || first + n > c->max_scenes)
        return fail(DP_ERR_ARG, "dp_run_closed_loop_dev: bad argument");
    if (!c->have_map) return fail(DP_ERR_STATE, "dp_run_closed_loop_dev: map not uploaded");
    if (c->submitted != c->waited) return fail(DP_ERR_STATE, "dp_run_closed_loop_dev: submitted cycles in flight, call dp_cycle_wait first");
    if (c->v2x.spec && n > c->v2x.n) return fail(DP_ERR_ARG, "dp_run_closed_loop_dev: more scenes than the armed V2X specifications");
    CK(cudaSetDevice(c->device));
    c->ep_last_graph = 0;
    if (n == 0) return DP_OK;
    // the graph holds the warp-kernel launches of a plain context (no gather armed, no record mirrors, no predicted tracks)
    const bool plain = c->kernel == 0 && c->tracks_T == 0 && !armed_any(c->armed);
    if (c->ep_graph && plain) {
        const void* key[8] = {hdr, agents, ox, oy, rec, hdr_log, olx, oly};
        const int dims[3] = {first, n, cycles};
        if (!c->ep_exec || memcmp(key, c->ep_key, sizeof(key)) != 0 || memcmp(dims, c->ep_dims, sizeof(dims)) != 0) {
            if (c->ep_exec) { cudaGraphExecDestroy(c->ep_exec); c->ep_exec = nullptr; }
            if (!c->ep_stream) CK(cudaStreamCreateWithFlags(&c->ep_stream, cudaStreamNonBlocking));
            dp_launch_prepare(c->lc);                       // function attributes are set outside the capture
            const long long before = c->launches;
            cudaGraph_t g = nullptr;
            cudaError_t e = cudaStreamBeginCapture(c->ep_stream, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess) {
                const cudaError_t e1 = enqueue_closed_loop(c, first, n, cycles, hdr, agents, ox, oy, rec, hdr_log, olx, oly, c->ep_stream, true);
                e = cudaStreamEndCapture(c->ep_stream, &g);
                if (e1 != cudaSuccess) e = e1;
            }
            if (e == cudaSuccess) e = cudaGraphInstantiate(&c->ep_exec, g, 0);
            if (g) cudaGraphDestroy(g);
            c->ep_launches = c->launches - before;
            c->launches = before;
            if (e != cudaSuccess) {                         // no graph on this driver / for these launches: enqueue them directly from now on
                cudaGetLastError();
                c->ep_exec = nullptr; c->ep_graph = 0;
            } else { memcpy(c->ep_key, key, sizeof(key)); memcpy(c->ep_dims, dims, sizeof(dims)); }
        }
        if (c->ep_exec) {
            CK(cudaGraphLaunch(c->ep_exec, (cudaStream_t)stream));
            c->launches += c->ep_launches;
            c->ep_last_graph = 1;
            return DP_OK;
        }
    }
    CK(enqueue_closed_loop(c, first, n, cycles, hdr, agents, ox, oy, rec, hdr_log, olx, oly, (cudaStream_t)stream, false));
    return DP_OK;
}
int dp_closed_loop_is_graph(dp_ctx* c) { return c ? c->ep_last_graph : 0; }

int64_t dp_launch_count(dp_ctx* c) { return c ? c->launches : 0; }

int dp_dev_alloc(dp_ctx* c, void** p, size_t bytes) {
    if (!c || !p) return fail(DP_ERR_ARG, "dp_dev_alloc");
    CK(cudaSetDevice(c->device));
    cudaError_t e = cudaMalloc(p, bytes ? bytes : 8);
    if (e != cudaSuccess) return fail(DP_ERR_NOMEM, "cudaMalloc", e);
    return DP_OK;
}
int dp_dev_free(dp_ctx* c, void* p) { if (c && p) { cudaSetDevice(c->device); cudaFree(p); } return DP_OK; }
int dp_memcpy_h2d(dp_ctx* c, void* dst, const void* src, size_t bytes, void* stream) {
    if (!c) return fail(DP_ERR_ARG, "dp_memcpy_h2d");
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return DP_OK;
}
int dp_memcpy_d2h(dp_ctx* c, void* dst, const void* src, size_t bytes, void* stream) {
    if (!c) return fail(DP_ERR_ARG, "dp_memcpy_d2h");
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return DP_OK;
}
int dp_stream_sync(dp_ctx* c, void* stream) {
    if (!c) return fail(DP_ERR_ARG, "dp_stream_sync");
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    return DP_OK;
}

}  // extern "C"
