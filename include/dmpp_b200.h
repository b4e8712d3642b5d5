/* include/dmpp_b200.h -- C ABI of the B200-native Decision/Planning hot path.
 *
 * One shared library (libdmpp_b200.so, built from decision-making-and-path-planning_b200/csrc/)
 * exports exactly the symbols declared here.  Plain C types, caller-owned buffers, int status
 * (0 = ok, negative = error; there is NO CPU fallback: every compute entry point fails with
 * DP_ERR_CUDA when no sm_100-class device is usable).  Each entry point cites the reference
 * interface (file:line in 123456jack/decision-making-and-path-planning) it replaces.
 *
 * Conventions (reference: SURVEY.md section 8): coordinates are double metres in the local
 * "global" frame; headings are degrees, 0 = east, CCW, [0,360) (Planning.cpp:712-750); speed is
 * km/h (Planning.cpp:258); periods are ms (Planning.cpp:77); lateral offsets passed to
 * search/create operators are RIGHT-of-travel positive (Decision.cpp:629,942).
 */
#ifndef DMPP_B200_H
#define DMPP_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DP_LANESUM 6          /* LANESUM      (Decision.h:79, Decision.cpp:498) */
#define DP_PATH_POINTS 200    /* local path   (Planning.h:33-34, Planning.cpp:115) */
#define DP_OUT_POINTS 100     /* PlanningOut  (Planning.cpp:180-183,205-212) */
#define DP_MAX_SWEEP 8        /* cap on K = #{i : i < (W - Vw)/0.6} per side (Decision.cpp:940) */
#define DP_NOT_FOUND 999.0    /* sentinel of SearchObstacle (Planning.cpp:161-162) */

enum {
    DP_OK = 0,
    DP_ERR_ARG = -1,          /* null pointer, size out of range */
    DP_ERR_CUDA = -2,         /* no device / CUDA runtime error (message via dp_last_error) */
    DP_ERR_STATE = -3,        /* map not uploaded, capacity exceeded */
    DP_ERR_NOMEM = -4
};

/* All constants the reference hides in the absent Share.h (SURVEY.md section 5 "config").
 * dp_default_params() returns the frozen values used by the oracle (oracle/compat/Share.h). */
typedef struct dp_params {
    double vehicle_width;            /* Vehicle_Width            Decision.cpp:370,811; 1.8 */
    double epsilon;                  /* EPSILON                  Planning.cpp:690;     1e-6 */
    double pi;                       /* PI                       Planning.cpp:728 */
    double road_faraim_max;          /* ROAD_FARAIM_MAX          Planning.cpp:260;     60 */
    double road_faraim_min;          /* ROAD_FARAIM_MIN          Planning.cpp:264;     15 */
    double pre_inter_faraim;         /* PRE_INTER_FARAIM         Planning.cpp:275;     20 */
    double inter_faraim;             /* INTER_FARAIM             Planning.cpp:283;     15 */
    double road_remain_distance;     /* ROAD_REMAIN_DISTANCE     Planning.cpp:821;     15 */
    double inter_remain_distance;    /* INTER_REMAIN_DISTANCE    Planning.cpp:826;     5 */
    double lat0, lng0, k_lat, k_lng; /* datum of GlobalToWGS84   Planning.cpp:209 */
    int32_t id_more;                 /* ID_MORE                  Decision.cpp:581;     8 */
    int32_t reserved;
} dp_params;

/* HD-map tables: app->decision_MapData[road][lane][id] / planning_MapData (Decision.cpp:562-578,
 * Planning.cpp:331-356) flattened to SoA, and the junction connectors
 * decision_InterMapData[last_road][next_road][last_lane][next_lane][id] (Decision.cpp:348,364). */
typedef struct dp_connector {
    uint16_t last_road, next_road, last_lane, next_lane; /* 1-based, as in LocationOut */
    int32_t lane;                                        /* index into lane_pt_off of its polyline */
} dp_connector;

typedef struct dp_map_desc {
    int32_t n_roads;
    const int32_t* road_lane_base;   /* [n_roads+1]: lanes of road r (1-based r) are base[r-1]..base[r]-1 */
    int32_t n_lanes;                 /* road lanes first, then one pseudo-lane per connector */
    const int32_t* lane_pt_off;      /* [n_lanes+1] offsets into the point arrays */
    int32_t n_conn;
    const dp_connector* conn;        /* [n_conn] */
    int64_t n_points;
    const double* x;                 /* [n_points] global_point.x */
    const double* y;
    const double* dir;               /* degrees */
    const uint16_t* lane_width;      /* cm  (Decision.cpp:578) */
    const uint16_t* lanechg_attr;    /* 0 none, 1 left, 2 right, 3 both (Decision.cpp:566) */
} dp_map_desc;

/* Per-scene, per-cycle input: LocationOut + the slice of RoadNavi the cycle reads
 * (Decision.cpp:155-169; Planning.cpp:95-112) + cycle period.  One 128-byte line per scene. */
typedef struct dp_scene_hdr {
    double x, y, dir;                /* LocationOut.globalpoint */
    double velocity;                 /* km/h */
    double period_ms;                /* z_period_last (Decision.cpp:137) */
    int32_t id[DP_LANESUM];          /* LocationOut.id[lane-1]: nearest map point per lane */
    uint16_t road_num, lane_num, pos, path_num;
    uint16_t last_roadnum, next_roadnum, last_lanenum, next_lanenum;
    uint16_t out_lane_no[DP_LANESUM];/* z_RoadNavi[path_num].out_lane_no (Decision.cpp:696) */
    uint16_t stub_attribute;         /* z_RoadNavi[path_num].stub_attribute (Decision.cpp:385) */
    uint16_t n_obs;                  /* obstacle points of this scene (<= ctx max_obs) */
    int32_t conn;                    /* connector index for pos 1/2, -1 otherwise */
    uint8_t pad[128 - 40 - 24 - 16 - 12 - 4 - 4];
} dp_scene_hdr;

/* Per-scene result of one Decision + Planning cycle: DecisionOut (Decision.cpp:187-196),
 * the public CPlanning fields (Planning.h:41-51) and PlanningOut scalars (Planning.cpp:189-201). */
typedef struct dp_plan_record {
    double velocity_expect;          /* DecisionOut.velocity_expect */
    double path_lat_dis, path_dir_err, remain_dis;   /* Planning.cpp:131 */
    double mindist_lat, mindist_lon; /* Planning.cpp:161-168 (brakedis = mindist_lon) */
    double brakespeed, des_acc;      /* Planning.cpp:171 */
    double radius;                   /* Planning.cpp:199 */
    double aim_x, aim_y, aim_dir;    /* aimpoint_far after Planning.cpp:121 */
    int32_t aim_id;
    uint16_t behavior, target_roadnum, target_lanenum, light, behavior_to_dlg;
    uint16_t afresh_cause;
    int16_t sweep_index;             /* avoid candidate picked this cycle: 0..K-1 = left i,
                                        K..2K-1 = right i, -1 = sweep not run or none feasible */
    int16_t path_near_id, path_front_near_id;
    int16_t ob_index;                /* obstacle that bounds the local path, -1 none */
    uint16_t ob_pathid;
    uint16_t n_traj;                 /* trajectories scored this cycle (SearchObstacle evaluations) */
    uint8_t afresh_planning, ob_flag, acc_flag, cnt;
} dp_plan_record;

/* Optional per-scene trace for parity tests: every SearchObstacle evaluation of the cycle. */
typedef struct dp_search_slot {
    double dis_lat, dis_lng;
    int16_t ob_index;
    uint16_t pathid;
    uint8_t evaluated, found;
    uint8_t pad[2];
} dp_search_slot;
typedef struct dp_trace_record {
    dp_search_slot region[6];        /* F, R, LF, LR, RF, RR   (Decision.cpp:811-842) */
    dp_search_slot sweep[2 * DP_MAX_SWEEP]; /* L0..L7, R0..R7 (Decision.cpp:940-974) */
    dp_search_slot junction;         /* Decision.cpp:370,455 */
    dp_search_slot local;            /* Planning.cpp:168 */
    double width_curlane, faraim_dis;
    uint32_t navi_lanechg, navi_lanechg_times; /* Decision.cpp:268 */
    uint16_t refpath_len;
    uint16_t ub_hits;                /* reference undefined-behaviour sites hit this cycle (clamped; see DESIGN.md) */
    uint32_t pts_scored;             /* sum of path points over the n_traj trajectories scored this cycle */
} dp_trace_record;

/* Cross-cycle state of one scene (SURVEY.md section 5 "checkpoint / resume"): the function
 * statics of Decision.cpp:915-917, the CDecision members of Decision.h:28-44, CPlanning's
 * his_behavior / count / aimpoint_far (Planning.h:22-23,49; Planning.cpp:51).  The last local
 * path (Planning.cpp:6) lives in a separate [scene][2][200] array. */
typedef struct dp_carry {
    double leftlight_time, rightlight_time, velocity_expect;
    double aim_x, aim_y, aim_dir;
    int32_t aim_id;
    uint32_t obsavoid_time, no_obsavoid_time, frontobs_time;
    int32_t plan_his_behavior;
    int32_t path_near_id;
    uint16_t behavior, target_roadnum, target_lanenum, light_status, behavior_to_dlg;
    uint16_t his_behavior, his_target_lanenum, his_light_status;
    uint8_t lanechg_status, obsavoid_status, plan_count, pad0;
    uint8_t pad[128 - 48 - 24 - 16 - 4];
} dp_carry;

/* A context belongs to one device and is NOT thread-safe: calls on one context must come from one thread at a time
 * (different contexts are independent; dp_last_error is per process). */
typedef struct dp_ctx dp_ctx;

const char* dp_last_error(void);
void dp_default_params(dp_params* p);

/* (1) context: replaces the singletons CDecision::Instance()/CPlanning::Instance()
 * (Decision.cpp:36-40, Planning.cpp:18-22) by an explicit, re-entrant handle. */
int dp_create(dp_ctx** out, int device, const dp_params* params, int max_scenes, int max_obs);
int dp_destroy(dp_ctx* ctx);

/* (2) map upload: replaces the app-owned tables read at Decision.cpp:562-666, Planning.cpp:331-374.
 * Precomputes per-point segment length and unit normal on the device, and the successor of every lane (section 9).  A connector
 * whose roads / lanes are not in the map, or whose `lane` is not a pseudo-lane (index >= road_lane_base[n_roads]), is DP_ERR_ARG. */
int dp_map_upload(dp_ctx* ctx, const dp_map_desc* map);

/* reset the carry of scenes [first, first+count) to the constructor state
 * (Decision.cpp:8-29, Planning.cpp:8-11,62).  dp_reset runs on the context's own stream and returns when done: it is ordered
 * with the host-pointer calls; cycles launched with dp_cycle_batch_dev on the CALLER's stream are not ordered with it -- use
 * dp_reset_dev(stream) there (enqueued on that stream, asynchronous) or synchronise the stream first. */
int dp_reset(dp_ctx* ctx, int first, int count);
int dp_reset_dev(dp_ctx* ctx, int first, int count, void* stream);
int dp_carry_download(dp_ctx* ctx, int first, int count, dp_carry* host_out, double* host_last_path);
int dp_carry_upload(dp_ctx* ctx, int first, int count, const dp_carry* host_in, const double* host_last_path);

/* (3)+(4) one fused Decision + Planning cycle for n_scenes scenes: replaces one iteration of
 * CDecisionThread (Decision.cpp:119-206) followed by one of CPlanningThread (Planning.cpp:64-226).
 * Device-pointer form: inputs/outputs already resident in HBM, launched on `stream`
 * (a cudaStream_t passed as void*), asynchronous.
 *   hdr[n_scenes]; obs_x/obs_y[n_scenes][max_obs];
 *   rec[n_scenes]; trace (nullable) [n_scenes]; path_xy (nullable) [n_scenes][2][200] = road_points;
 *   path_ll (nullable) [n_scenes][2][100] = PlanningOut.pnts (lat row, lng row).
 * scene i uses carry slot first_scene + i. */
int dp_cycle_batch_dev(dp_ctx* ctx, int first_scene, int n_scenes, const dp_scene_hdr* hdr,
                       const double* obs_x, const double* obs_y, dp_plan_record* rec,
                       dp_trace_record* trace, double* path_xy, double* path_ll, void* stream);

/* Whole scripted episodes with everything resident in HBM (replay / Monte-Carlo; SURVEY 8f rank 1, open loop): `cycles`
 * consecutive cycles of the same n_scenes scenes, hdr[cycles][n_scenes], obs_x/obs_y[cycles][n_scenes][max_obs],
 * rec[cycles][n_scenes], enqueued on `stream` in one call and asynchronous like dp_cycle_batch_dev.  The carry stays on the
 * device between cycles (the hysteresis counters and the carried path of Decision.cpp:915-917 / Planning.cpp:6 evolve as in
 * the reference) and nothing returns to the host until the caller synchronises the stream. */
int dp_run_episode_dev(dp_ctx* ctx, int first_scene, int n_scenes, int cycles, const dp_scene_hdr* hdr,
                       const double* obs_x, const double* obs_y, dp_plan_record* rec, void* stream);

/* Host-pointer form (the drop-in call): copies inputs host->device, runs the cycle, copies the
 * requested outputs device->host, and returns when they are valid.  Buffers may be pageable or
 * pinned; dp_host_alloc returns pinned memory. */
int dp_cycle_batch(dp_ctx* ctx, int first_scene, int n_scenes, const dp_scene_hdr* hdr,
                   const double* obs_x, const double* obs_y, dp_plan_record* rec,
                   dp_trace_record* trace, double* path_xy, double* path_ll);

/* Pipelined form of dp_cycle_batch for replay / Monte-Carlo hosts whose inputs of cycle k+1 do not depend on the
 * outputs of cycle k (the reference's two thread loops are already one cycle apart: CPlanningThread consumes the
 * DecisionOut of the previous wake-up, Planning.cpp:117-131).  dp_cycle_submit queues the host->device copies of one
 * cycle on a copy stream and its kernels on the compute stream and returns at once; dp_cycle_wait blocks until the
 * OLDEST submitted cycle has written its records into `rec`.  At most two cycles may be in flight; all four buffers
 * must be page-locked (dp_host_alloc) and must not be touched between submit and the matching wait; n_scenes is
 * limited to 32768 per call.  Cycles execute in submission order (each reads the carry the previous one wrote).  The inputs
 * are announced to the Decision warps by a flag that a four-byte copy raises behind the input DMAs, the Planning warps store
 * the records into `rec` themselves, and completion reaches the host as a flag in page-locked memory instead of a stream event.
 * dp_cycle_batch / dp_reset / dp_carry_* return DP_ERR_STATE while cycles are in flight. */
int dp_cycle_submit(dp_ctx* ctx, int first_scene, int n_scenes, const dp_scene_hdr* hdr,
                    const double* obs_x, const double* obs_y, dp_plan_record* rec);
int dp_cycle_wait(dp_ctx* ctx);
/* Record mirrors: from now on every finished plan record of scene slot s is ALSO stored at bases[k] + s for k < n
 * (n <= 8; n = 0 switches it off).  The bases must be addresses the device of `ctx` can store to: device memory of this
 * GPU, page-locked host memory, or -- the reason this exists -- the gathered-records buffers of the PEER GPUs mapped into
 * this process over NVLink (CUDA IPC / VMM / torch symmetric memory).  With one base per peer, pointing at this rank's slice of
 * the peer's buffer, the per-step all-gather of plan records (SURVEY 8e) happens inside the Planning launch as 128-byte
 * peer stores instead of a separate collective; the caller only needs a barrier before it reads the gathered buffer. */
int dp_set_record_mirrors(dp_ctx* ctx, int n, void* const* bases);
/* Fused gather of the plan records of a multi-GPU job (one process per GPU of one box; SURVEY 8e) through the C ABI alone -- no
 * collective library, no framework: every rank owns a buffer rec[depth][world][slots] + flags, the buffers are mapped into every
 * process over NVLink with CUDA IPC, and the cycle kernel itself stores each finished record into its rank's slice of EVERY
 * rank's buffer (dp_set_record_mirrors under the hood) and, when its last record is out, raises its flag on every rank.
 *   dp_gather_create   allocate my buffer, return its 64-byte IPC handle; the caller exchanges the handles (any transport)
 *   dp_gather_attach   handles[world][DP_IPC_BYTES] of all ranks (own entry ignored): map the peers
 *   dp_gather_arm      the NEXT cycle launch of ctx writes step `step` (>= 1, increasing): buffer step % depth, slice `rank`
 *   dp_gather_wait     enqueue on `stream` a wait for all `world` flags of that step in MY buffer; work that follows on the
 *                      stream may read dp_gather_buffer(step) = device pointer to rec[world][slots] of that step
 *   dp_gather_chain    fold that wait into the NEXT cycle launch instead of a launch of its own: after raising its own flags the
 *                      last warp of that launch waits for all flags of `prev_step` (0 = off) before the launch completes (and
 *                      before dp_cycle_wait's host flag): kernel of step s done => dp_gather_buffer(prev_step) is complete.
 *                      Deadlock-free as long as every rank launched prev_step before: no launch waits for a LATER step.
 * A rank may run ahead of a peer: with waits enqueued one step behind the launches (launch s, launch s+1, wait s, ...), depth 4
 * guarantees that a slice is never overwritten before every peer has waited for it. */
#define DP_IPC_BYTES 64
typedef struct dp_gather dp_gather;
int dp_gather_create(dp_ctx* ctx, int world, int rank, int slots_per_rank, int depth, dp_gather** out, void* my_handle_out);
int dp_gather_attach(dp_gather* g, const void* handles);
int dp_gather_arm(dp_gather* g, unsigned step);
int dp_gather_chain(dp_gather* g, unsigned prev_step);
/* Deferred variant -- the one a pipelined loop should use.  dp_gather_arm_deferred(g, s) before the launch of step s: that
 * launch keeps its own records local; instead its warps, AS THEY START, copy the records of the launch before (step s-1, armed
 * the same way, same slot range) into every rank's buffer, so the NVLink round trips hide under the cycle; the flags of s-1
 * go up when the last Decision warp retires and the launch's last warp waits for every rank's flag of s-1:
 *     launch of step s complete  =>  dp_gather_buffer(s-1) holds every rank's records of step s-1
 * (the contract of arm + chain, at about 1 us per step instead of 8).  One-shot: arm before every launch.
 * dp_gather_flush(g, stream) forwards, flags and awaits the LAST armed step (two small launches), at the end of a sequence.
 * dp_gather_set_lag(g, 2) (depth >= 4) relaxes the contract by one step -- launch of step s complete => buffer(s-2) complete --
 * which leaves a whole step of slack between the ranks instead of the ~20 us between the end of a Decision half and the end
 * of its launch: ranks whose steps differ by a few microseconds (different scenes) no longer wait for the slowest one at
 * every step.  dp_gather_flush then awaits the last two steps. */
int dp_gather_arm_deferred(dp_gather* g, unsigned step);
int dp_gather_set_lag(dp_gather* g, int lag);
int dp_gather_flush(dp_gather* g, void* stream);
int dp_gather_disarm(dp_gather* g);
int dp_gather_wait(dp_gather* g, unsigned step, void* stream);
const void* dp_gather_buffer(dp_gather* g, unsigned step);
int dp_gather_destroy(dp_gather* g);
int dp_host_alloc(void** p, size_t bytes);
int dp_host_free(void* p);

/* (5) dense candidate sweep for ONE scene (latency mode, BASELINE config 3): candidate c is the
 * lateral-offset copy (offset[c], RIGHT positive) of the first n_pts[c] points of the base
 * polyline base_x/base_y[n_base], scored by SearchObstacle against obstacle tracks
 * obs = o0 + j * dv for path point j (dv = 0 reproduces Decision.cpp:940-974).  cost =
 * feasibility {0, +inf} with threshold `clear_dis` (dis_lng > clear_dis, Decision.cpp:944);
 * best = lowest index among feasible, -1 if none.  Host pointers; out_dis_lng nullable. */
int dp_score_candidates(dp_ctx* ctx, const double* base_x, const double* base_y, int n_base,
                        const double* offset, const int32_t* n_pts, int n_cand,
                        const double* obs_x, const double* obs_y, const double* obs_dvx,
                        const double* obs_dvy, int n_obs, double lat_min, double lat_max,
                        double clear_dis, int32_t* best_index, double* best_dis_lng,
                        double* out_dis_lng);

/* Latency-mode session of (5): the candidate set (base line, offsets, point counts) is uploaded once; each
 * dp_sweep_score call is ONE kernel launch: the obstacle tracks travel in the kernel parameters, a thread-block cluster per
 * lateral offset scores all horizons of that offset, the grid's last CTA writes the winner into page-locked host memory, and
 * the call returns as soon as the host sees it (no stream synchronisation, no copies).  n_obs <= max_obs <= 192.
 * device_ms (nullable) = CUDA-event time around the launch; asking for it adds an event synchronisation to the call. */
typedef struct dp_sweep dp_sweep;
int dp_sweep_create(dp_ctx* ctx, dp_sweep** out, const double* base_x, const double* base_y, int n_base,
                    const double* offset, const int32_t* n_pts, int n_cand, int max_obs);
int dp_sweep_score(dp_sweep* s, const double* obs_x, const double* obs_y, const double* obs_dvx,
                   const double* obs_dvy, int n_obs, double lat_min, double lat_max, double clear_dis,
                   int32_t* best_index, double* best_dis_lng, float* device_ms);
int dp_sweep_destroy(dp_sweep* s);
/* The same session over SEVERAL base lines (distinct geometries): candidate c is the offset copy (offset[c]) of the first
 * n_pts[c] points of line cand_line[c]; lines_xy = [n_lines][2][n_base] (x row, y row per line).  Candidates that share
 * (line, offset) share one scan per obstacle, as in dp_sweep_create.  A row is cut into 16 parts (one warp each) when there are few rows, to shorten
 * the dependent chain, and into 4 when there are many (> 296) and the rows fill the machine. */
int dp_sweep_create_lines(dp_ctx* ctx, dp_sweep** out, const double* lines_xy, int n_lines, int n_base,
                          const int32_t* cand_line, const double* offset, const int32_t* n_pts, int n_cand, int max_obs);
/* ... whose lines are the 200-point local paths CShare::BezierPlanning draws (Planning.cpp:596-611, 863) from a start pose
 * to an aim pose: dp_sweep_set_bezier(poses[n_lines][6] = start x,y,dir, aim x,y,dir) rolls all lines out ON THE DEVICE
 * (two launches: the Bezier operator of dp_bezier_planning into the session's line buffer, then the rows' arclength
 * prefixes); the dp_sweep_score calls that follow score them.  A lateral x aim-distance grid of local paths, each with
 * its horizons, is this session with offset = 0.  dp_sweep_lines reads the lines back ([n_lines][2][200]). */
int dp_sweep_create_bezier(dp_ctx* ctx, dp_sweep** out, int n_lines, const int32_t* cand_line, const double* offset,
                           const int32_t* n_pts, int n_cand, int max_obs);
int dp_sweep_set_bezier(dp_sweep* s, const double* poses, float* device_ms);
int dp_sweep_lines(dp_sweep* s, double* lines_xy_out);
/* diagnostic: globaltimer stamps [n_rows][8] (ns) of the row-owner CTAs of the last dp_sweep_score: 0 start, 1 row pass done,
 * 2 groups selected, 3 reduced, 4 counted, 5 winner known, 6 system fence done (5, 6: last row only).  Only sessions created
 * with DP_SWEEP_DBG=1 in the environment record them (tools/sweep_probe.py). */
int dp_sweep_debug(dp_sweep* s, long long* out, int n_rows);

/* (6) operator-level batch calls, the CShare seam (SURVEY.md 8b).  Host pointers.
 * paths are [n_paths] polylines concatenated; path_off[n_paths+1]. */
/* CShare::SearchObstacle  (Planning.cpp:168; Decision.cpp:370,...,962) */
int dp_search_obstacle(dp_ctx* ctx, int n_paths, const int32_t* path_off, const double* px,
                       const double* py, const double* obs_x, const double* obs_y, int n_obs,
                       const double* lat_min, const double* lat_max, dp_search_slot* out);
/* CShare::CreateNewPath   (Decision.cpp:629,631,667,669,942,961) */
int dp_create_new_path(dp_ctx* ctx, int n_paths, const int32_t* path_off, const double* px,
                       const double* py, const double* offset, double* out_x, double* out_y);
/* CShare::BezierPlanning  (Planning.cpp:606,863): poses[n][6] = start x,y,dir, aim x,y,dir;
 * out[n][2][200] */
int dp_bezier_planning(dp_ctx* ctx, int n, const double* poses, double* out_xy);
/* CShare::NearestId       (Decision.cpp:1889,2074,2383; loop shape Planning.cpp:640-648): one query point per path;
 * out_id[i] = index of the path point nearest to (qx[i], qy[i]): lowest index among the points whose rounded distance
 * sqrt(dx*dx+dy*dy) is minimal, 0 when no distance is below 9999 */
int dp_nearest_id(dp_ctx* ctx, int n_paths, const int32_t* path_off, const double* px,
                  const double* py, const double* qx, const double* qy, int32_t* out_id);
/* CShare::MeanPoints      (Planning.cpp:872): out[n][2][200] */
int dp_mean_points(dp_ctx* ctx, int n_paths, const int32_t* path_off, const double* px,
                   const double* py, double* out_xy);

/* device properties + FMA micro-benchmark used as roofline denominator (SURVEY.md 8d):
 * returns measured FP64 / FP32 FMA throughput in TFLOP/s on the context's device. */
int dp_measure_fma_peak(dp_ctx* ctx, double* fp64_tflops, double* fp32_tflops);
/* Predicted agent tracks (BASELINE config 5; a generalisation: the reference has the members z_DynaObs_front/rear, Decision.h:14-15,
 * but their getters are commented out, Decision.cpp:162-163).  Every obstacle point gets a constant-turn-rate prediction of T
 * steps: position 0 = the obstacle point of the cycle call, position j+1 = position j + v_j, v_{j+1} = v_j rotated by dtheta
 * degrees, frozen after step T-1 (vx, vy: metres per step at step 0; operations pinned in oracle/cshare_spec.h rollout_ctr).
 * From then on the junction search of every cycle (Decision.cpp:370, :455: pos 1 / 2) runs against the moving agents -- agent o is
 * at its position j when the ego reaches path point j; the rollout is fused into the search, the track is never materialised --
 * while the lane-region, avoid and local-path searches keep the static positions, as in the reference.  Cycles then use the
 * group kernel whatever the context's kernel choice.  dp_clear_tracks switches back.
 *   dp_set_tracks     host arrays [n_scenes][max_obs] for carry slots first_scene .., copied into the context;
 *   dp_set_tracks_dev device arrays [max_scenes][max_obs] indexed by carry slot, referenced (not copied): they must stay valid,
 *                     and may be rewritten between cycles in stream order. */
int dp_set_tracks(dp_ctx* ctx, int first_scene, int n_scenes, int T, const double* vx, const double* vy, const double* dtheta_deg);
int dp_set_tracks_dev(dp_ctx* ctx, int T, const double* vx, const double* vy, const double* dtheta_deg);
int dp_clear_tracks(dp_ctx* ctx);

/* (8) Output stage (SURVEY.md 8f rank 3): the two frames CPlanningThread publishes at the end of every cycle, packed on the
 * device in a fixed little-endian layout (the reference's struct definitions are not in the reference; the field order
 * follows its assignments, every reserved byte is zero).  The path samples come from the carried local path of the carry
 * slot (= road_points of the cycle that just ran, Planning.cpp:217), so the call follows a cycle call in stream order and
 * needs none of that call's optional path outputs. */
typedef struct dp_ctrl_frame {       /* PlanningOut -> app->SetUdpSendCtrl (Planning.cpp:189-214) */
    uint8_t cnt;                     /* count % 100                 :189 */
    uint8_t apa;                     /* 0                           :190 */
    uint8_t desacc_vd;               /* acc_flag                    :193 */
    uint8_t desstr_vd;               /* false                       :197 */
    uint8_t road_type;               /* 0                           :200 */
    uint8_t sstop;                   /* TRUE                        :201 */
    uint16_t light;                  /* DecisionOut.light           :198 */
    double brakedis;                 /* mindist_lon                 :191 */
    double brake_speed;              /* 0                           :192 */
    double desacc;                   /* des_acc                     :194 */
    double desspd;                   /* brakespeed                  :195 */
    double desstr;                   /* 0                           :196 */
    double radius;                   /* CalculateRadius()           :199 */
    double pnts[DP_OUT_POINTS][2];   /* GlobalToWGS84(road_points[2 i]) as (lat, lng)  :203-212 */
} dp_ctrl_frame;                     /* 1656 bytes */
typedef struct dp_status_frame {     /* PlanningStatus -> app->SetPlanningStatus (Planning.cpp:173-186) */
    int32_t afresh_cause;            /* :174 */
    uint16_t trafficlight;           /* DecisionOut.light  :178 */
    uint16_t reserved;
    double near_ob_dist;             /* mindist_lon        :175 */
    double planspeed;                /* brakespeed         :176 */
    double planacc;                  /* des_acc            :177 */
    double path_points[DP_OUT_POINTS][2];   /* road_points[2 i] as (x, y)  :180-183 */
} dp_status_frame;                   /* 1632 bytes */
/* rec[n_scenes] = the records of the cycle that just ran for carry slots first_scene ..; ctrl / status nullable.
 * _dev: device pointers, asynchronous on `stream`; the other form takes host pointers and returns when the frames are valid. */
int dp_pack_frames_dev(dp_ctx* ctx, int first_scene, int n_scenes, const dp_plan_record* rec, dp_ctrl_frame* ctrl,
                       dp_status_frame* status, void* stream);
int dp_pack_frames(dp_ctx* ctx, int first_scene, int n_scenes, const dp_plan_record* rec, dp_ctrl_frame* ctrl,
                   dp_status_frame* status);

/* (9) Closed-loop episodes (SURVEY.md 8f rank 1): ego and agents advanced ON THE DEVICE between cycles, the carry (hysteresis
 * counters Decision.cpp:915-917, carried path Planning.cpp:6, his_behavior / count Planning.cpp:216-223) never leaves HBM, and
 * a whole episode is ONE CUDA graph launch.  The reference has no vehicle or traffic model (localisation, perception and
 * control are other modules of its application); the world step below is this library's, its arithmetic is frozen in
 * oracle/world_spec.h (junction transitions: tools/junction_oracle/world_junction.h) and the parity of this part is oracle-only by
 * construction.  Segment driving (pos 0) always; junctions
 * (pos 0 -> 1 -> 2 -> 0 through a connector) when dp_world_params.pre_junction_pts > 0.
 *
 * world step of one scene, given the record of the cycle that just ran (rec == NULL: place the agents and localise only):
 *   ego    target speed = rec.brakespeed [m/s, the unit of the planner's constants 3 / 10, Planning.cpp:888-990] * 3.6 km/h,
 *          approached with |dv| <= a_max * dt; distance = mean speed * dt, walked along the carried local path from
 *          rec.path_near_id (perfect tracking); heading = CalcGlobalDir of the segment it lands on; an ego whose lane index
 *          is within end_margin points of the lane end stops (with junctions on: only in pos 0 with no connector ahead);
 *   agents agent k moves v[k] * dt along its lane (index i, offset u into segment i -> i+1), keeps its lateral offset `lat`
 *          (LEFT positive) and stops at the lane end (with junctions on: continues on the lane's successor, see below); its
 *          obstacle point is written to obs_x / obs_y;
 *   localisation  hdr.id[l] = nearest point of lane l of the ego's road within [id[l] - loc_back, id[l] + loc_fwd]
 *          (squared distance, strict '<'), hdr.lane_num = the lane with the smallest such distance (lowest lane on ties),
 *          hdr.x / y / dir / velocity = the new ego state; everything else in the header is left as it is.
 *
 * junction transitions (pre_junction_pts = J > 0; J = 0 is the step above, bit for bit).  The ego's connector is the lowest c
 * with conn[c].(last_road, next_road, last_lane) = (road_num, next_roadnum, lane_num) and next_roadnum != road_num.  Nearest
 * points are searched as in the localisation (squared distance, strict '<', lowest index on ties); a pos other than 1 / 2 is 0.
 *   pos 0  localisation as above; then, when the ego has a connector c and id[lane_num-1] >= (points of its lane) - 1 - J:
 *          pos = 1, conn = c, last_roadnum = road_num, last_lanenum = lane_num, next_lanenum = conn[c].next_lane
 *          (also in the placement step);
 *   pos 1  localisation as above, then conn / last_roadnum / last_lanenum / next_lanenum re-picked from lane_num (no connector
 *          for that lane: back to pos 0, conn = -1); the connector is searched in [0, loc_fwd]; when its nearest point is
 *          strictly nearer than the nearest approach point: pos = 2, road_num = next_roadnum, lane_num = next_lanenum and
 *          id[l] = that connector index for every lane l of the approach road (Decision reads id[last_lanenum-1]);
 *   pos 2  the connector is searched in [id[last_lanenum-1] - loc_back, id[last_lanenum-1] + loc_fwd], every lane of the
 *          departure road (road_num) in [0, loc_fwd]; when the departure road's nearest point is strictly nearer than the
 *          connector's: pos = 0, conn = -1, path_num + 1, stub_attribute = 0, id[] / lane_num from the departure road; otherwise
 *          id[l] = the connector index as in pos 1.  An invalid conn or last_lanenum counts as a connector infinitely far away.
 *   agents an agent that walks past the end of a lane with a successor (lane_next, built by dp_map_upload: road lane -> the
 *          lowest connector leaving it, connector -> its next lane) continues on the successor from i = 0 with the leftover u
 *          (the gap between a lane end and its successor's start is jumped, not walked); at most 8 lanes per step. */
typedef struct dp_agent {
    double u;                        /* metres into segment i -> i+1 */
    double v;                        /* m/s along the lane */
    double lat;                      /* lateral offset from the lane centre line, LEFT positive, metres */
    int32_t lane;                    /* global lane index (road_lane_base[road - 1] + lane - 1) */
    int32_t i;                       /* map point index within the lane */
} dp_agent;                          /* 32 bytes; agents[n_scenes][max_obs], the first hdr.n_obs of a scene are used */
typedef struct dp_world_params {
    double a_max;                    /* m/s^2, default 3.0 (the planner's own braking command, Planning.cpp des_acc = -3) */
    int32_t loc_back, loc_fwd;       /* localisation window in map points, default 8 / 56 */
    int32_t end_margin;              /* default 160: the front region (120 points + ID_MORE) stays inside the lane */
    int32_t pre_junction_pts;        /* default 0 = junction transitions off; > 0: length of the pre-junction zone in map points
                                        (60 = the 30 m of Episodes(kind="junction"), >= 400 = kind="urban") */
} dp_world_params;
void dp_world_default_params(dp_world_params* p);
int dp_world_set_params(dp_ctx* ctx, const dp_world_params* p);
/* one world step for carry slots first_scene ..: hdr, agents, obs_x, obs_y are updated in place (device pointers) */
int dp_world_step_dev(dp_ctx* ctx, int first_scene, int n_scenes, dp_scene_hdr* hdr, dp_agent* agents, double* obs_x,
                      double* obs_y, const dp_plan_record* rec, void* stream);
/* `cycles` x (Decision + Planning cycle, world step) from the world in hdr / agents (placed and localised first), everything in
 * HBM, enqueued on `stream` as one graph launch (the graph is built on the first call and reused while the arguments stay the
 * same; DP_EPISODE_GRAPH=0 or a failed capture enqueues the same launches directly).  rec[cycles][n_scenes]; hdr_log
 * (nullable) [cycles][n_scenes] and obs_log_x / obs_log_y (nullable) [cycles][n_scenes][max_obs] receive the inputs every
 * cycle ran on -- replaying them through dp_run_episode_dev gives the same records.  hdr / agents / obs hold the final world. */
int dp_run_closed_loop_dev(dp_ctx* ctx, int first_scene, int n_scenes, int cycles, dp_scene_hdr* hdr, dp_agent* agents,
                           double* obs_x, double* obs_y, dp_plan_record* rec, dp_scene_hdr* hdr_log, double* obs_log_x,
                           double* obs_log_y, void* stream);
/* 1 when the last dp_run_closed_loop_dev call of this context was a graph launch, 0 when it enqueued the launches directly */
int dp_closed_loop_is_graph(dp_ctx* ctx);

/* (10) V2X event handlers (SURVEY.md 8f rank 4; Decision.cpp:1824-2434).  The reference evaluates them every segment cycle
 * (V2XEventDecision, Decision.cpp:283) and then discards the three flags; here they are a batch operator next to the cycle, one
 * warp per scene, with every quirk of the handlers kept (see oracle/v2x_oracle.cpp, which is pinned to the unmodified
 * reference's own private methods).  What a caller does with the flags is its business, as in the reference. */
typedef struct dp_v2x_data {         /* V2X_Data as the handlers read it + LocationOut.gpspoint + this scene's slice of the warning list */
    double ped_distance, ped_lat, ped_lng;     /* PedesDistance / PedesLatitude / PedesLongitude  Decision.cpp:1859-1861 */
    double rsi_lat, rsi_lng;                   /* RSILatitude / RSILongitude                       :2038, :2262 */
    double ego_lat, ego_lng;                   /* LocationOut.gpspoint                             :2257-2258 */
    int32_t ped_direction;                     /* PedesDirection    :1862 */
    int32_t spat_lane_occupied, spat_state;    /* SPATLaneOccupied / SPATState  :1979-1980 */
    int32_t warn_status;                       /* V2XWarnStatus: 3 signal, 4 road works, 5 pedestrian  :2149-2161 */
    int32_t wp_first, wp_count;                /* z_RSIWarningPointList = wp_lat / wp_lng[wp_first .. wp_first + wp_count) */
} dp_v2x_data;                       /* 80 bytes */
typedef struct dp_v2x_flags {
    uint16_t light_flag;             /* V2XLight_flag: 0 none, 1 red / yellow, 2 green   Decision.cpp:1984-1995 */
    uint8_t construction_flag;       /* :2124-2137, :2407-2425 */
    uint8_t pedestrian_flag;         /* :1935-1961 */
    uint8_t ub;                      /* the handler would have read its path vector out of bounds (empty path, nearest point = last point):
                                        the flags are then all 0 */
    uint8_t pad[3];
    double lng_distance;             /* pedestrian: lng_distance; road works: min_distance_construction (9999 when not computed) */
    double lat_distance;             /* pedestrian: lat_distance; road works: near_lat_distance         (9999 when not computed) */
} dp_v2x_flags;                      /* 24 bytes */
/* mode 0: V2XEventDecision as the reference calls it (status 4 -> V2XConstructionEvent); mode 1: status 4 ->
 * V2XConstructionEventTemporal (the alternative commented out at Decision.cpp:2156).  hdr[n] is the cycle's scene header
 * (road, lane, per-lane ids); wp_lat / wp_lng[n_wp] may be NULL when n_wp is 0.  Host pointers; _dev: device pointers, asynchronous. */
int dp_v2x_event_batch(dp_ctx* ctx, int n_scenes, const dp_scene_hdr* hdr, const dp_v2x_data* v2x, const double* wp_lat,
                       const double* wp_lng, int n_wp, int mode, dp_v2x_flags* out);
int dp_v2x_event_batch_dev(dp_ctx* ctx, int n_scenes, const dp_scene_hdr* hdr, const dp_v2x_data* v2x, const double* wp_lat,
                           const double* wp_lng, int mode, dp_v2x_flags* out, void* stream);
/* OPT-IN extension beyond the reference (which drops the flags, Decision.cpp:283-313): let the flags act on the speed command of
 * the records, in place, with the planner's own vocabulary (SpeedPlanning, Planning.cpp:888-990):
 *   pedestrian_flag or light_flag == 1 (red / yellow)  ->  brakespeed = 0, acc_flag = 1, des_acc = -3   (its "obstacle closer than 5 m" command)
 *   else construction_flag and brakespeed > 3          ->  brakespeed = 3                               (its creep speed)
 * Everything else in the record is left alone; lane choice is NOT touched.  A closed loop that steps the world with the adjusted
 * records (dp_world_step_dev) makes the ego actually stop.  Arithmetic-free, so parity is against oracle/v2x_oracle.cpp only. */
int dp_v2x_apply(dp_ctx* ctx, int n_scenes, const dp_v2x_flags* flags, dp_plan_record* rec);
int dp_v2x_apply_dev(dp_ctx* ctx, int n_scenes, const dp_v2x_flags* flags, dp_plan_record* rec, void* stream);

/* (11) Closed-loop episode metrics: one row per world, accumulated by the world step of section 9 in the warp that has just
 * moved the ego and the agents.  They only observe: no decision, record, world state or log changes with them, and with
 * metrics disarmed (the default) nothing is written.  The arithmetic is frozen in tools/junction_oracle/episode_metrics.h.
 *
 * When a row is written:
 *   placement step (rec == NULL, the first node of every episode): the row is initialised, also for a header that names no lane,
 *          so a replayed episode graph starts every episode from a clean row;
 *   every later step (rec != NULL) on a header that names a lane: the row is updated after the ego and the agents have moved (a
 *          header that names no lane leaves its row alone, as it leaves its world alone).
 * IEEE binary64, operations in the order written, no contraction; min / max updates are `if (x < m) m = x` / `if (x > m) m = x`.
 * Per step: v, vn = ego speed before / after the step (km/h); dt = period_ms / 1000; (c, s) = spec_sincos_deg(new dir);
 * ds = the step's distance (0 when the end_margin stop fired).  For every agent k < min(n_obs, max_obs), at its new obstacle
 * point (ox, oy), on map segment (ddx, ddy) of length L:
 *   dx = ox - x, dy = oy - y, lon = dx*c + dy*s, lat = dy*c - dx*s                      (ego frame, LEFT positive)
 *   inside    -rear <= lon <= front  &&  -half_width <= lat <= half_width
 *   clearance ex = lon > front ? lon - front : (lon < -rear ? -rear - lon : 0); ey = |lat| > half_width ? |lat| - half_width : 0;
 *             d = sqrt(ex*ex + ey*ey)
 *   lead      lon > front && |lat| <= corridor_half:  gap = lon - front,
 *             va = L == 0 ? 0 : v_agent * (ddx/L*c + ddy/L*s),  closing = vn/3.6 - va,  ttc = closing > 0 ? gap/closing : +inf
 * Fields (initial value):
 *   distance                 sum of ds in step order (0)
 *   min_clearance            min of d over steps and agents (+inf)
 *   min_lead_gap, min_ttc    min of gap / ttc over steps and lead agents (+inf)
 *   max_accel, min_accel     a = (vn - v) / 3.6 / dt, on steps with dt > 0 (-inf / +inf)
 *   max_abs_jerk             |a - last_accel| / dt on every step with an a after the first one (0)
 *   last_accel, accel_steps  the previous a (0) and the number of steps with an a (0)
 *   max_abs_lat_err / _dir_err  max of |rec.path_lat_dis| / |rec.path_dir_err| (0)
 *   steps                    steps accumulated (0)
 *   first_collision_step     1-based step of the first step with an agent inside, and the lowest such agent (-1 / -1)
 *   first_collision_agent
 *   collision_steps          steps with an agent inside; _front: with one inside at lon >= 0; _rear: with one inside at lon < 0
 *   collision_steps_front/_rear  (a step can count as both; unless the agents react (section 12), rear strikes are theirs)
 *   ttc_warn_steps           steps whose smallest ttc is < ttc_warn
 *   stopped_steps            steps with vn == 0;  end_stop_steps: steps on which the end_margin stop fired
 *   replans, aeb_steps       sum of rec.afresh_planning / rec.acc_flag
 *   behavior_steps[b]        steps with rec.behavior == b (b < 8)
 *   last_behavior            rec.behavior of the previous step (-1)
 *   behavior_switches        steps whose rec.behavior differs from the previous step's (the first step never counts) */
typedef struct dp_metrics_params {
    double front, rear;              /* ego box along its heading from the header's (x, y): default 4.0 (antenna to bumper,
                                        Planning.cpp:896) and 1.0 (this library's choice) */
    double half_width;               /* default 0.9 = Vehicle_Width / 2 */
    double corridor_half;            /* lead corridor, default 1.1 (the local-path corridor, Planning.cpp:168) */
    double ttc_warn;                 /* seconds, default 2.0 */
} dp_metrics_params;
typedef struct dp_episode_metrics {
    double distance, min_clearance, min_lead_gap, min_ttc;
    double max_accel, min_accel, max_abs_jerk, last_accel;
    double max_abs_lat_err, max_abs_dir_err;
    int32_t steps, first_collision_step, first_collision_agent;
    int32_t collision_steps, collision_steps_front, collision_steps_rear, ttc_warn_steps;
    int32_t stopped_steps, end_stop_steps, replans, aeb_steps;
    int32_t accel_steps, last_behavior, behavior_switches;
    uint32_t behavior_steps[8];
    uint32_t pad[6];                 /* zero */
} dp_episode_metrics;                /* 192 bytes */
void dp_metrics_default_params(dp_metrics_params* p);
/* m: device array indexed like hdr (the s-th scene of every later dp_world_step_dev / dp_run_closed_loop_dev call);
 * m == NULL disarms (p may then be NULL).  p must be finite with front, rear, corridor_half, ttc_warn >= 0 and half_width > 0,
 * else DP_ERR_ARG.  Context state like dp_world_set_params: the cached episode graph is rebuilt on its next call. */
int dp_world_set_metrics(dp_ctx* ctx, const dp_metrics_params* p, dp_episode_metrics* m);

/* (12) Reactive agents (opt-in): longitudinal car-following with the intelligent driver model.  Each agent adapts its speed to
 * the nearest vehicle ahead of it on its lane chain, the ego included.  The model only REWRITES EACH AGENT'S SPEED at the start
 * of a world step of section 9, from the state at the start of that step (Jacobi: every agent reads the old state of every
 * other agent and of the ego); the agent motion of section 9 then runs unchanged with the new v.  It runs on steps with
 * rec != NULL on headers that name a lane (the same early return as the step), for agents k < min(n_obs, max_obs).  With the
 * model disarmed (the default) nothing changes.  The arithmetic is frozen in tools/junction_oracle/agent_model.h.
 * Lane changes are section 13, on top of this model.  Out of scope: merges; yielding to a vehicle on a DIFFERENT connector that merges
 * into the same lane (it is seen only once it is on the chain); any change to how the ego moves.
 *
 * IEEE binary64, operations in the order written, no contraction; min updates are `if (x < m) m = x`.
 *   opt-out   !(v0[k] > 0) (0, negative, NaN): agent k keeps its speed (it moves exactly as in the disarmed step) but is still a
 *             leader for the others
 *   station   s = cump[off + i] + u, cump[off + i] = the sequential prefix (index order) of the lane's segment lengths
 *             sqrt(dx*dx + dy*dy) that dp_map_upload builds; len(l) = cump[off(l) + cnt(l) - 1]
 *   ego       pos as the step of section 9 reads it (0 when pre_junction_pts is 0), from the start-of-step header:
 *             pos 0 / 1: lane road_lane_base[road_num-1] + lane_num - 1, index id[lane_num-1];
 *             pos 2: lane conn[conn].lane, index id[last_lanenum-1] (an invalid conn or last_lanenum: no ego leader);
 *             the index clamped to [0, cnt-1], s_e = cump[off + index]; its speed is velocity / 3.6
 *   chain     l0 = the agent's lane, l1 = lane_next[l0], l2 = lane_next[l1] (stopping at -1; at most 2 hops);
 *             D1 = len(l0) - s_k, D2 = D1 + len(l1)
 *   candidate on l0: ds = s_j - s_k when s_j > s_k, or s_j == s_k && j > k (the ego: when s_e >= s_k);
 *             on l1: ds = D1 + s_j; on l2: ds = D2 + s_j; a lane that appears twice in the chain takes the smaller ds;
 *             only candidates with ds <= look count
 *   leader    g = ds - length (an agent) or ds - ego_rear (the ego); the candidate with the smallest g, the ego first on a tie,
 *             then the lowest agent index
 *   IDM       (delta = 4) with v = the agent's v, dt = period_ms / 1000:
 *               r = v / v0; fr = r * r; fr = fr * fr;
 *               leader:    dv = v - vl; z = v * T + v * dv / (2.0 * sqrt(a_max * b)); if (z < 0) z = 0; ss = s0 + z;
 *                          if (g > 0) { q = ss / g; acc = a_max * (1.0 - fr - q * q); } else acc = -b_max;
 *               no leader: acc = a_max * (1.0 - fr);
 *               if (acc < -b_max) acc = -b_max;
 *               vn = v + acc * dt; if (vn < 0) vn = 0;   v = vn */
typedef struct dp_agent_model_params {
    double a_max;                    /* IDM acceleration, m/s^2, default 1.0 */
    double b;                        /* comfortable deceleration, m/s^2, default 1.5 */
    double b_max;                    /* hardest deceleration, m/s^2, default 8.0 (the clamp, and the answer for an overlapping leader) */
    double T;                        /* time headway, s, default 1.5 */
    double s0;                       /* jam distance, m, default 2.0 */
    double length;                   /* point-to-point spacing subtracted for an agent leader, m, default 4.5 */
    double ego_rear;                 /* subtracted for the ego as leader, m, default 1.0 (= dp_metrics_params.rear) */
    double look;                     /* leader search horizon along the lane chain, m, default 100 */
} dp_agent_model_params;             /* 64 bytes */
/* the largest max_obs of a context that can arm the model: the world step stages 24 bytes per agent slot and world in shared memory */
#define DP_AGENT_MODEL_MAX_OBS 2048
void dp_agent_model_default_params(dp_agent_model_params* p);
/* v0: device array [n][max_obs] of desired speeds (m/s), indexed like hdr (the s-th scene of every later dp_world_step_dev /
 * dp_run_closed_loop_dev call); v0 == NULL disarms (p may then be NULL).  Context state like dp_world_set_metrics: the cached
 * episode graph is rebuilt on its next call.  DP_ERR_ARG for non-finite parameters, a_max, b, b_max, T, length, look <= 0,
 * s0, ego_rear < 0, or a context max_obs above DP_AGENT_MODEL_MAX_OBS. */
int dp_world_set_agent_model(dp_ctx* ctx, const dp_agent_model_params* p, const double* v0);

/* (13) Lane-changing agents (opt-in, on top of the reactive agents of section 12): MOBIL ("minimising overall braking induced
 * by lane changes", Kesting / Treiber / Helbing) with the IDM accelerations of section 12.  The model runs on the steps of
 * section 12 (rec != NULL, a header that names a lane), for agents k < min(n_obs, max_obs), from the same start-of-step state
 * (Jacobi): stations s, speeds v and lanes of every agent and the ego as section 12 reads them.  It may move an agent to a
 * neighbouring lane of its road where the map allows it (lanechg_attr), rewriting its lane / i / lat / v; the agent motion of
 * section 9 then runs unchanged.  Disarmed (the default) nothing changes.  The arithmetic is frozen in
 * tools/junction_oracle/lane_change.h.  Uses the agent model's parameters (a_max, b, b_max, T, s0, length, ego_rear, look) and
 * v0.  Two agents may pick the same gap in the same step (Jacobi): they are not arbitrated; the metrics see the outcome.
 * Out of scope: changes on connectors, merges between connectors, any change to how the ego moves.
 *
 * IEEE binary64, operations in the order written, no contraction.  Per agent k, with a_c = its clamped IDM acceleration of
 * section 12 (the value before vn = v + acc * dt), v = its start-of-step speed, st = its dp_lane_change_state:
 *   placement (rec == NULL, every scene, also a header that names no lane): st = {lat_goal = agents[k].lat, hold = 0, 0, 0}
 *   eligible  v0[k] > 0, l0 = its lane < road_lane_base[n_roads] (a road lane), lat == lat_goal, hold <= 0,
 *             len(l0) - s_k >= end_guard
 *   sides     road r with road_lane_base[r-1] <= l0 < road_lane_base[r] (binary search), lane number q = l0 - road_lane_base[r-1];
 *             attr = lanechg_attr[off(l0) + i]; left: m = l0 - 1 when q >= 1 and attr is 1 or 3; right: m = l0 + 1 when
 *             q + 1 < lanes of r and attr is 2 or 3.  Left is evaluated first.
 *   abeam     i_m = min(i, cnt(m) - 2), s_m = cump[off(m) + i_m] + u (exact for lanes sampled abeam, as scenes.Map builds
 *             them; an approximation for maps that are not); the side needs len(m) - s_m >= end_guard
 *   candidates on m alone (no chain): the ego (section 12's lane and s_e, when that lane is m) and every agent j with lane m;
 *             S == s_m for any of them: overlap, the side is unsafe; ahead (S > s_m) with ds = S - s_m <= look, behind (S < s_m)
 *             with ds = s_m - S <= look.  leader: the ahead candidate with the smallest g, g = ds - length (an agent) or
 *             ds - ego_rear (the ego); follower: the behind candidate with the smallest g, g = ds - length (an agent) or
 *             ds - ego_front (the ego); the ego first on a tie, then the lowest agent index (`if (g < best)` in index order)
 *   IDM       idm(v, v0, lead, g, vl) is section 12's acceleration, clamp at -b_max included (free road without a leader):
 *               r = v / v0; fr = r * r; fr = fr * fr; leader: dv = v - vl; z = v * T + v * dv / (2.0 * sqrt(a_max * b));
 *               if (z < 0) z = 0; ss = s0 + z; g > 0 ? a_max * (1.0 - fr - (ss / g) * (ss / g)) : -b_max;
 *               free: a_max * (1.0 - fr); then if (acc < -b_max) acc = -b_max
 *             the ego as follower knows no v0 and may stand: only the interaction term, with q = ss / g:
 *               g > 0 ? -a_max * (q * q) : -b_max, clamped at -b_max; 0 without a leader
 *   MOBIL     at_c = idm(v, v0[k], leader?, g_leader, v_leader)                                 (agent k on m)
 *             a_f  = the follower f behind the leader: gap S_l - S_f (stations subtracted directly) minus length (agent leader),
 *                    ego_rear (ego leader) or ego_front (ego follower); no leader: free road (ego: 0)
 *             at_f = the follower behind agent k: its own g above, leader speed v
 *             an agent follower with !(v0[f] > 0): a_f = at_f = 0; no follower: a_f = at_f = 0
 *             safe:      no overlap, (no leader or g_leader > 0), (no follower or g_follower > 0),
 *                        at_f >= -b_safe (agent follower) / >= -ego_b_safe (ego follower)
 *             incentive: delta = (at_c - a_c) + politeness * (at_f - a_f) > a_thr  (the old follower is deliberately left out)
 *             both sides safe and above threshold: the larger delta, left on a tie
 *   change    lane = m, i = i_m, u unchanged; P = point i of l0, Q / R = points i_m / i_m + 1 of m, (dx, dy) = R - Q,
 *             L = sqrt(dx*dx + dy*dy), d = L > 0 ? (P.x - Q.x) * (-(dy / L)) + (P.y - Q.y) * (dx / L) : 0; lat = lat + d
 *             (the obstacle point stays where it was); v = v + at_c * dt, if (v < 0) v = 0 (replaces section 12's speed);
 *             hold = cooldown; changes_left or changes_right += 1
 *   others    every agent k < min(n_obs, max_obs) that does not change this step (opted out, ineligible or not changing):
 *             hold = hold - dt; if (lat != lat_goal) { e = lat_goal - lat; w = lat_speed * dt;
 *             lat = fabs(e) <= w ? lat_goal : (e > 0 ? lat + w : lat - w); } */
typedef struct dp_lane_change_params {
    double politeness;               /* p, default 0.2 */
    double a_thr;                    /* incentive threshold, m/s^2, default 0.2 */
    double b_safe;                   /* an agent as the new follower must not need to brake harder than this, m/s^2, default 4.0 */
    double ego_b_safe;               /* the same test when the new follower is the ego, default 4.0: the lever for cut-ins */
    double ego_front;                /* ego box ahead of (x, y) when the ego is the follower, m, default 4.0 (= dp_metrics_params.front) */
    double lat_speed;                /* lateral speed back to lat_goal, m/s, default 1.0 */
    double cooldown;                 /* s between two changes of one agent, default 5.0 */
    double end_guard;                /* no change within this many metres of the end of the agent's lane or the target lane, default 30 */
} dp_lane_change_params;             /* 64 bytes */
typedef struct dp_lane_change_state {
    double lat_goal;                 /* the in-lane offset the agent returns to (its lat at placement) */
    double hold;                     /* seconds until the agent may start another change */
    int32_t changes_left, changes_right;
} dp_lane_change_state;              /* 24 bytes, [n][max_obs] indexed like hdr (the s-th scene of every later call) */
void dp_lane_change_default_params(dp_lane_change_params* p);
/* st == NULL disarms (p may then be NULL).  Context state like dp_world_set_agent_model: the cached episode graph is rebuilt on
 * its next call; disarming the agent model disarms lane changes too.  DP_ERR_ARG for non-finite parameters, lat_speed, b_safe,
 * ego_b_safe <= 0, politeness, cooldown, end_guard, ego_front < 0, or arming while the agent model is disarmed. */
int dp_world_set_lane_change(dp_ctx* ctx, const dp_lane_change_params* p, dp_lane_change_state* st);

/* (14) V2X events in closed-loop episodes (opt-in): each world carries one traffic signal, one crossing pedestrian and one
 * road-works zone, placed in map coordinates; every cycle a V2X launch between the cycle and the world step builds the cycle's
 * dp_v2x_data from the world, runs the handlers of section 10 on it (the same device code as dp_v2x_event_batch) and, with
 * apply = 1, lets the flags act on the cycle's record with the rule of dp_v2x_apply, so the world step of section 9 moves the
 * ego with the adjusted speed command.  Armed, an episode is: placement, then per cycle Decision + Planning -> V2X -> world
 * step, then one tally-only V2X launch (1 + cycles * 4 + 1 kernels).  Disarmed (the default) the episode is that of section 9,
 * launch for launch.  The rules are frozen in tools/junction_oracle/v2x_world.h.  Out of scope: agents that obey signals or
 * yield to pedestrians, pedestrians as obstacle points, V2X in pos 1 / 2.
 *
 * IEEE binary64, operations in the order written, no contraction.  World s at cycle k (k = 0 .. cycles-1 the cycle launches,
 * k = cycles the tally), with its cycle's header h (before the world step) and t = k * period_ms / 1000:
 *   row       the launch with k == 0 first initialises the world's row (also for a header that names no lane), so a replayed
 *             episode graph starts clean; a header that names no lane then gets zero flags and leaves its row alone
 *   GPS       GlobalToWGS84 as dp_frames_kernel: lat = fma(y, k_lat, lat0), lng = fma(x, k_lng, lng0)
 *   signal    sig_road > 0: phase ph = fmod(t + sig_offset, sig_cycle), ph += sig_cycle when ph < 0; state 6 (green) when
 *             ph < sig_green, else 7 (yellow) when ph < sig_green + sig_yellow, else 3 (red); sig_road == 0: state 0.
 *             on = sig_road > 0, h.road_num == sig_road and h.pos != 2 (the approach, pos 0 / 1); then on the ego's lane gl
 *             (off, cnt): stop = sig_stop < 0 || sig_stop > cnt - 1 ? cnt - 1 : sig_stop (-1: the stop line at the end of a
 *             junction approach), i = id[lane_num-1] clamped to [0, cnt-1], d = cump[off + stop] - cump[off + i]
 *             (cump: the prefix table of dp_map_upload, section 12); off the approach d = 0.
 *             spat_state = state, spat_lane_occupied = on && d >= 0 && d <= sig_range
 *   pedestrian ped_on = has_ped && ped_t_on <= t && t <= ped_t_off; then px = ped_x + ped_vx * (t - ped_t_on), py likewise;
 *             dx = px - h.x, dy = py - h.y, ped_distance = sqrt(dx * dx + dy * dy), (ped_lat, ped_lng) = GPS(px, py);
 *             otherwise ped_distance = ped_lat = ped_lng = 0.  ped_direction = the specification's
 *   road works has_works: (rsi_lat, rsi_lng) = GPS(rw_x, rw_y) when rw_rsi, else 0 / 0 (no RSI point: the warning list
 *             alone); wp_first / wp_count = the specification's slice of the caller's list, whose entries pass as
 *             GPS(wp_x, wp_y); rw_dx = rw_x - h.x, rw_dy = rw_y - h.y, near_works = sqrt(rw_dx * rw_dx + rw_dy * rw_dy) <= rw_range.
 *             !has_works: rsi 0 / 0, an empty slice, near_works false
 *   ego       (ego_lat, ego_lng) = GPS(h.x, h.y)
 *   warn_status  5 when ped_on && ped_distance <= ped_range, else 3 when on, else 4 when near_works, else 0
 *   handlers  only on headers with h.pos == 0 (SegmentDecision is their only caller, Decision.cpp:283) and k < cycles: the
 *             flags of section 10 with the world's mode; in pos 1 / 2 and on the tally the flags are zero (distances 9999)
 *   apply     stop  = pedestrian_flag || light_flag == 1; creep = !stop && construction_flag && rec.brakespeed > 3; with
 *             apply = 1 the record is adjusted as dp_v2x_apply does (stop: brakespeed 0, acc_flag 1, des_acc -3; creep:
 *             brakespeed 3); with apply = 0 the record is left alone and the row still counts both.  So with apply = 1,
 *             replaying hdr_log through dp_run_episode_dev gives the planner's own records, which differ from the logged ones
 *             in brakespeed / acc_flag / des_acc on the cycles with a stop or creep command, and nowhere else
 *   red crossing  a world step that starts with last_on && last_d >= 0 && last_phase == 3 and ends past the stop line: the
 *             header of the next launch has !on or d < 0.  The row carries (d, state, on) of the previous launch.
 * Row (initial value): min_ped_distance min of ped_distance over launches k < cycles with ped_on, any pos (+inf); cycles:
 * launches that ran the handlers; light_cycles[f] / construction_cycles[f] / pedestrian_cycles[f]: of those, the cycles with
 * that flag value; stop_cmds, creep_cmds, ub_cycles (flags.ub); red_crossings and first_red_crossing (k of the step, -1). */
typedef struct dp_v2x_event_spec {
    double sig_cycle, sig_green, sig_yellow, sig_red;  /* seconds; each > 0 and green + yellow + red == cycle (to 1e-9 of it) */
    double sig_offset;                 /* seconds added to t before the phase */
    double sig_range;                  /* metres before the stop index within which the approach counts as occupied */
    double ped_x, ped_y, ped_vx, ped_vy;               /* map metres at t = ped_t_on, m/s */
    double ped_t_on, ped_t_off;        /* active window, seconds */
    double ped_range;                  /* metres */
    double rw_x, rw_y, rw_range;       /* the road-works point (map metres) and its range */
    int32_t sig_road;                  /* governed road, 1-based; 0 = no signal */
    int32_t sig_stop;                  /* stop index on the governed road's lanes; -1 = the last point of the lane */
    int32_t has_ped, ped_direction;    /* ped_direction: PedesDirection as the handler reads it */
    int32_t has_works, rw_rsi;         /* rw_rsi: the RSI broadcasts (rw_x, rw_y) */
    int32_t wp_first, wp_count;        /* the zone's warning points: wp_x / wp_y[wp_first .. wp_first + wp_count) */
} dp_v2x_event_spec;                   /* 160 bytes */
typedef struct dp_v2x_world_params {
    int32_t mode;                      /* 0 / 1 as in dp_v2x_event_batch */
    int32_t apply;                     /* 1: the flags act on the records; 0: observe only (the row still counts) */
} dp_v2x_world_params;
typedef struct dp_v2x_episode_stats {
    double min_ped_distance;
    double last_d;                     /* carried from the previous launch (0) */
    int32_t cycles;
    int32_t light_cycles[3], construction_cycles[2], pedestrian_cycles[2];
    int32_t stop_cmds, creep_cmds, ub_cycles;
    int32_t red_crossings, first_red_crossing;
    int32_t last_phase, last_on;       /* carried from the previous launch (0 / 0) */
    int32_t pad;                       /* zero */
} dp_v2x_episode_stats;                /* 80 bytes */
/* spec[n] (device): one specification per world, indexed like hdr (the s-th scene of every later dp_run_closed_loop_dev /
 * dp_v2x_world_dev call, which may name at most n scenes); wp_x / wp_y[n_wp] (device, nullable when n_wp is 0): the warning
 * points; flags[n] (device, nullable): every V2X launch of a cycle stores the world's flags (the tally leaves them); stats[n] (device): the rows.  spec == NULL
 * disarms (everything else may then be NULL).  The setter copies the specifications to the host once to validate them:
 * DP_ERR_ARG for a mode other than 0 / 1, apply other than 0 / 1, non-finite values, signal durations that are not > 0 or do
 * not sum to the cycle, ranges < 0, sig_road outside [0, n_roads], sig_stop < -1, a warning-point slice outside [0, n_wp), or
 * NULL stats.  Context state like dp_world_set_metrics: the cached episode graph is rebuilt on its next call. */
int dp_world_set_v2x(dp_ctx* ctx, const dp_v2x_world_params* params, int n, const dp_v2x_event_spec* spec, const double* wp_x,
                     const double* wp_y, int n_wp, dp_v2x_flags* flags, dp_v2x_episode_stats* stats);
/* one V2X launch of cycle `cycle` for callers that step by hand: after dp_cycle_batch_dev wrote rec[n] for hdr[n], before
 * dp_world_step_dev(rec) moves the world; rec == NULL: the tally after the last world step (cycle = the number of cycles).
 * DP_ERR_STATE when V2X is disarmed. */
int dp_v2x_world_dev(dp_ctx* ctx, int first_scene, int n_scenes, const dp_scene_hdr* hdr, dp_plan_record* rec, int cycle,
                     void* stream);

/* diagnostic: phase time stamps (globaltimer, ns) of the most recent cycle launch, one row of 32 per CTA (row b = scenes
 * [b*g, (b+1)*g) of the batch; stamp 0 = CTA start, stamp i = end of phase i of csrc/dp_group.cuh).  Only contexts created
 * with DP_TIMELINE=1 in the environment record them; used by tools/group_timeline.py, never by the product path. */
int dp_debug_timeline(dp_ctx* ctx, long long* host_out, int n_blocks);
/* number of kernels this library has launched since dp_create (bench.py "gpu_launches") */
int64_t dp_launch_count(dp_ctx* ctx);
/* device pointer helpers so a Python/C++ caller can stage inputs for dp_cycle_batch_dev */
int dp_dev_alloc(dp_ctx* ctx, void** p, size_t bytes);
int dp_dev_free(dp_ctx* ctx, void* p);
int dp_memcpy_h2d(dp_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream);
int dp_memcpy_d2h(dp_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream);
int dp_stream_sync(dp_ctx* ctx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DMPP_B200_H */
