"""ctypes binding of libdmpp_b200.so (include/dmpp_b200.h) and the host-side mirror of the
reference's Decision/Planning interface for batches of scenes.

There is no CPU implementation behind this module: if the CUDA library is missing, or no
sm_100-class device is usable, construction raises -- it never falls back.
"""
import ctypes as C
import os

import numpy as np

from . import abi

_here = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_here, "libdmpp_b200.so")

# every symbol include/dmpp_b200.h declares (tests/test_abi.py checks the export table against the header)
SYMBOLS = [
    "dp_last_error", "dp_default_params", "dp_create", "dp_destroy", "dp_map_upload", "dp_reset", "dp_reset_dev",
    "dp_carry_download", "dp_carry_upload", "dp_cycle_batch_dev", "dp_cycle_batch", "dp_host_alloc",
    "dp_host_free", "dp_score_candidates", "dp_search_obstacle", "dp_create_new_path", "dp_bezier_planning",
    "dp_mean_points", "dp_measure_fma_peak", "dp_launch_count", "dp_dev_alloc", "dp_dev_free",
    "dp_memcpy_h2d", "dp_memcpy_d2h", "dp_stream_sync", "dp_sweep_create", "dp_sweep_score", "dp_sweep_destroy", "dp_sweep_debug", "dp_sweep_create_lines", "dp_sweep_create_bezier",
    "dp_sweep_set_bezier", "dp_sweep_lines",
    "dp_cycle_submit", "dp_cycle_wait", "dp_set_record_mirrors", "dp_nearest_id", "dp_run_episode_dev", "dp_debug_timeline",
    "dp_set_tracks", "dp_set_tracks_dev", "dp_clear_tracks",
    "dp_pack_frames_dev", "dp_pack_frames", "dp_world_default_params", "dp_world_set_params", "dp_world_step_dev",
    "dp_run_closed_loop_dev", "dp_closed_loop_is_graph", "dp_v2x_event_batch", "dp_v2x_event_batch_dev", "dp_v2x_apply", "dp_v2x_apply_dev",
    "dp_metrics_default_params", "dp_world_set_metrics", "dp_agent_model_default_params", "dp_world_set_agent_model",
    "dp_lane_change_default_params", "dp_world_set_lane_change", "dp_world_set_v2x", "dp_v2x_world_dev",
    "dp_v2x_traffic_default_params", "dp_world_set_v2x_traffic", "dp_v2x_obstacle_default_params", "dp_world_set_v2x_obstacles",
    "dp_v2x_obstacles_dev", "dp_run_closed_loop_part_dev", "dp_world_fork_dev", "dp_split_default_params", "dp_world_set_split",
    "dp_world_split_dev", "dp_world_split_map",
    "dp_gather_create", "dp_gather_attach", "dp_gather_arm", "dp_gather_chain", "dp_gather_arm_deferred", "dp_gather_set_lag", "dp_gather_flush", "dp_gather_disarm", "dp_gather_wait", "dp_gather_buffer", "dp_gather_destroy",
]

_lib = None


def load():
    """dlopen the product library (no CUDA call is made until dp_create)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'`" % LIB_PATH)
        _lib = C.CDLL(os.environ.get("DP_DEBUG_LIB") or LIB_PATH)   # DP_DEBUG_LIB: instrumented build for tools/ only
        _lib.dp_last_error.restype = C.c_char_p
        _lib.dp_launch_count.restype = C.c_int64
        _lib.dp_launch_count.argtypes = [C.c_void_p]
        vp, i = C.c_void_p, C.c_int
        _lib.dp_run_closed_loop_part_dev.argtypes = [vp, i, i, i, i, i] + [vp] * 10
        _lib.dp_world_fork_dev.argtypes = [vp, i, i, vp, i, i] + [vp] * 6
        _lib.dp_world_set_split.argtypes = [vp, vp, i, vp, vp]
        _lib.dp_world_split_dev.argtypes = [vp, i, i, i] + [vp] * 6
        _lib.dp_world_split_map.argtypes = [vp, i, vp, vp]
    return _lib


class DpError(RuntimeError):
    pass


def _ck(rc, what):
    if rc != 0:
        raise DpError("%s failed (%d): %s" % (what, rc, load().dp_last_error().decode()))


def metrics_params():
    """dp_metrics_default_params (no GPU needed)"""
    p = abi.MetricsParams()
    load().dp_metrics_default_params(C.byref(p))
    return p


def agent_model_params():
    """dp_agent_model_default_params (no GPU needed)"""
    p = abi.AgentModelParams()
    load().dp_agent_model_default_params(C.byref(p))
    return p


def lane_change_params():
    """dp_lane_change_default_params (no GPU needed)"""
    p = abi.LaneChangeParams()
    load().dp_lane_change_default_params(C.byref(p))
    return p


def v2x_traffic_params(**kw):
    """dp_v2x_traffic_default_params (no GPU needed), then the keyword fields"""
    p = abi.V2xTrafficParams()
    load().dp_v2x_traffic_default_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def v2x_obstacle_params(**kw):
    """dp_v2x_obstacle_default_params (no GPU needed), then the keyword fields"""
    p = abi.V2xObstacleParams()
    load().dp_v2x_obstacle_default_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def split_params(**kw):
    """dp_split_default_params (no GPU needed), then the keyword fields"""
    p = abi.SplitParams()
    load().dp_split_default_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def split_estimate(state):
    """the collision probability of every population (include/dmpp_b200.h section 18) from Episode.state() after the last part:
    p_g = norm_g * (1 / M) * sum_j [first_collision_step_j >= 0] / lw_j"""
    rows, groups = state["split_rows"], state["split_groups"]
    M = len(rows) // len(groups)
    hit = (state["metrics"]["first_collision_step"] >= 0).astype(np.float64)
    return groups["norm"] * (hit / rows["lw"]).reshape(-1, M).mean(axis=1)


def default_params():
    p = abi.Params()
    load().dp_default_params(C.byref(p))
    return p


class Planner:
    """Batched, explicit-state replacement for the CDecision + CPlanning singletons
    (Decision.h:105-107, Planning.h:38-40): one `cycle()` call runs one iteration of
    CDecisionThread followed by one of CPlanningThread for every scene of the batch."""

    def __init__(self, max_scenes, max_obs, device=0, params=None):
        self.lib = load()
        self.max_scenes, self.max_obs, self.device = int(max_scenes), int(max_obs), int(device)
        self.params = params if params is not None else default_params()
        self.ctx = C.c_void_p()
        _ck(self.lib.dp_create(C.byref(self.ctx), C.c_int(device), C.byref(self.params), C.c_int(self.max_scenes),
                               C.c_int(self.max_obs)), "dp_create")
        self._map = None

    def close(self):
        if self.ctx:
            self.lib.dp_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload_map(self, m):
        self._map = m
        d = m.desc()
        _ck(self.lib.dp_map_upload(self.ctx, C.byref(d)), "dp_map_upload")

    def reset(self, first=0, count=None):
        count = self.max_scenes - first if count is None else count
        _ck(self.lib.dp_reset(self.ctx, C.c_int(first), C.c_int(count)), "dp_reset")

    def reset_dev(self, first=0, count=None, stream=0):
        """stream-ordered reset for loops that launch cycle_dev on their own stream"""
        count = self.max_scenes - first if count is None else count
        _ck(self.lib.dp_reset_dev(self.ctx, C.c_int(first), C.c_int(count), C.c_void_p(stream)), "dp_reset_dev")

    def launch_count(self):
        return int(self.lib.dp_launch_count(self.ctx))

    # ---- the drop-in call: host buffers in, host buffers out ---------------------------------
    def cycle(self, hdr, ox, oy, first=0, trace=False, paths=False, out=None):
        n = hdr.shape[0]
        assert hdr.dtype == abi.scene_hdr and ox.shape == (n, self.max_obs) and oy.shape == (n, self.max_obs)
        o = out if out is not None else {}
        if "rec" not in o:
            o["rec"] = np.zeros(n, abi.plan_record)
        if trace and o.get("trace") is None:
            o["trace"] = np.zeros(n, abi.trace_record)
        if paths and o.get("path_xy") is None:
            o["path_xy"] = np.zeros((n, 2, abi.PATH_POINTS))
            o["path_ll"] = np.zeros((n, 2, abi.OUT_POINTS))
        _ck(self.lib.dp_cycle_batch(self.ctx, C.c_int(first), C.c_int(n), abi.ptr(hdr), abi.ptr(ox), abi.ptr(oy),
                                    abi.ptr(o["rec"]), abi.ptr(o.get("trace") if trace else None),
                                    abi.ptr(o.get("path_xy") if paths else None),
                                    abi.ptr(o.get("path_ll") if paths else None)), "dp_cycle_batch")
        return o

    # ---- predicted agent tracks (BASELINE config 5): constant-turn-rate parameters per obstacle point ----
    def set_tracks(self, vx, vy, dth, T, first=0):
        n = vx.shape[0]
        assert all(a.shape == (n, self.max_obs) for a in (vx, vy, dth))
        _ck(self.lib.dp_set_tracks(self.ctx, C.c_int(first), C.c_int(n), C.c_int(T), abi.ptr(vx), abi.ptr(vy), abi.ptr(dth)), "dp_set_tracks")

    def set_tracks_dev(self, T, d_vx, d_vy, d_dth):
        """device arrays [max_scenes][max_obs], referenced until clear_tracks / the next set"""
        _ck(self.lib.dp_set_tracks_dev(self.ctx, C.c_int(T), C.c_void_p(d_vx), C.c_void_p(d_vy), C.c_void_p(d_dth)), "dp_set_tracks_dev")

    def clear_tracks(self):
        _ck(self.lib.dp_clear_tracks(self.ctx), "dp_clear_tracks")

    def run_episodes_tracks(self, H, OX, OY, VX, VY, DTH, T, trace=True, paths=True):
        """run_episodes with a fresh track tile before every cycle"""
        cycles, n = H.shape
        self.reset(0, n)
        out = {"rec": np.zeros((cycles, n), abi.plan_record),
               "trace": np.zeros((cycles, n), abi.trace_record) if trace else None,
               "path_xy": np.zeros((cycles, n, 2, abi.PATH_POINTS)) if paths else None,
               "path_ll": np.zeros((cycles, n, 2, abi.OUT_POINTS)) if paths else None}
        for c in range(cycles):
            o = {"rec": out["rec"][c], "trace": out["trace"][c] if trace else None,
                 "path_xy": out["path_xy"][c] if paths else None, "path_ll": out["path_ll"][c] if paths else None}
            cc = np.ascontiguousarray
            self.set_tracks(cc(VX[c]), cc(VY[c]), cc(DTH[c]), T)
            self.cycle(cc(H[c]), cc(OX[c]), cc(OY[c]), trace=trace, paths=paths, out=o)
        self.clear_tracks()
        out["carry"], out["last_path"] = self.download_carry(0, n)
        return out

    def set_record_mirrors(self, bases):
        """bases: device-accessible addresses (ints); every finished record of slot s is also stored at base + 128 * s"""
        arr = (C.c_void_p * max(1, len(bases)))(*[C.c_void_p(int(b)) for b in bases])
        _ck(self.lib.dp_set_record_mirrors(self.ctx, C.c_int(len(bases)), arr), "dp_set_record_mirrors")

    def run_episode_dev(self, n, cycles, d_hdr, d_ox, d_oy, d_rec, first=0, stream=0):
        """`cycles` chained cycles of n scenes, all buffers device pointers: hdr[cycles][n], obs[cycles][n][max_obs], rec[cycles][n]"""
        _ck(self.lib.dp_run_episode_dev(self.ctx, C.c_int(first), C.c_int(n), C.c_int(cycles), C.c_void_p(d_hdr), C.c_void_p(d_ox),
                                        C.c_void_p(d_oy), C.c_void_p(d_rec), C.c_void_p(stream)), "dp_run_episode_dev")

    # ---- output stage: controller / status frames (include/dmpp_b200.h section 8) ----
    def pack_frames(self, rec, first=0, ctrl=True, status=True):
        """frames of the cycle that just ran for carry slots first ..: host records in, host frames out"""
        rec = np.ascontiguousarray(rec)
        n = rec.shape[0]
        cf = np.zeros(n, abi.ctrl_frame) if ctrl else None
        sf = np.zeros(n, abi.status_frame) if status else None
        _ck(self.lib.dp_pack_frames(self.ctx, C.c_int(first), C.c_int(n), abi.ptr(rec), abi.ptr(cf), abi.ptr(sf)), "dp_pack_frames")
        return cf, sf

    def pack_frames_dev(self, n, d_rec, d_ctrl, d_status, first=0, stream=0):
        _ck(self.lib.dp_pack_frames_dev(self.ctx, C.c_int(first), C.c_int(n), C.c_void_p(d_rec), C.c_void_p(d_ctrl or 0),
                                        C.c_void_p(d_status or 0), C.c_void_p(stream)), "dp_pack_frames_dev")

    # ---- V2X event handlers (include/dmpp_b200.h section 10) ----
    def v2x_event(self, hdr, v2x, wp_lat, wp_lng, mode=0):
        """V2XEventDecision (Decision.cpp:283) for every scene of the batch; mode 1: the Temporal road-works variant"""
        hdr, v2x = np.ascontiguousarray(hdr), np.ascontiguousarray(v2x)
        wl, wg = np.ascontiguousarray(wp_lat, np.float64), np.ascontiguousarray(wp_lng, np.float64)
        out = np.zeros(hdr.shape[0], abi.v2x_flags)
        _ck(self.lib.dp_v2x_event_batch(self.ctx, C.c_int(hdr.shape[0]), abi.ptr(hdr), abi.ptr(v2x), abi.ptr(wl) if wl.size else None,
                                        abi.ptr(wg) if wg.size else None, C.c_int(wl.size), C.c_int(mode), abi.ptr(out)), "dp_v2x_event_batch")
        return out

    def v2x_apply(self, flags, rec):
        """opt-in: the flags act on the speed command of the records (returns the adjusted copy)"""
        out = np.ascontiguousarray(rec).copy()
        _ck(self.lib.dp_v2x_apply(self.ctx, C.c_int(out.shape[0]), abi.ptr(np.ascontiguousarray(flags)), abi.ptr(out)), "dp_v2x_apply")
        return out

    def v2x_apply_dev(self, n, d_flags, d_rec, stream=0):
        _ck(self.lib.dp_v2x_apply_dev(self.ctx, C.c_int(n), C.c_void_p(d_flags), C.c_void_p(d_rec), C.c_void_p(stream)), "dp_v2x_apply_dev")

    def v2x_event_dev(self, n, d_hdr, d_v2x, d_wp_lat, d_wp_lng, d_out, mode=0, stream=0):
        _ck(self.lib.dp_v2x_event_batch_dev(self.ctx, C.c_int(n), C.c_void_p(d_hdr), C.c_void_p(d_v2x), C.c_void_p(d_wp_lat or 0),
                                            C.c_void_p(d_wp_lng or 0), C.c_int(mode), C.c_void_p(d_out), C.c_void_p(stream)),
            "dp_v2x_event_batch_dev")

    # ---- closed-loop episodes (include/dmpp_b200.h section 9) ----
    def world_params(self):
        wp = abi.WorldParams()
        self.lib.dp_world_default_params(C.byref(wp))
        return wp

    def set_world_params(self, wp):
        _ck(self.lib.dp_world_set_params(self.ctx, C.byref(wp)), "dp_world_set_params")

    def metrics_params(self):
        return metrics_params()

    def set_metrics(self, params, d_metrics):
        """arm the episode metrics (include/dmpp_b200.h section 11): d_metrics = device address of rows [n] indexed like hdr;
        d_metrics None / 0 disarms"""
        _ck(self.lib.dp_world_set_metrics(self.ctx, C.byref(params) if params is not None else None, C.c_void_p(d_metrics or 0)),
            "dp_world_set_metrics")

    def agent_model_params(self):
        return agent_model_params()

    def set_agent_model(self, params, d_v0):
        """arm the reactive agents (include/dmpp_b200.h section 12): d_v0 = device address of desired speeds [n][max_obs] (m/s)
        indexed like hdr; d_v0 None / 0 disarms"""
        _ck(self.lib.dp_world_set_agent_model(self.ctx, C.byref(params) if params is not None else None, C.c_void_p(d_v0 or 0)),
            "dp_world_set_agent_model")

    def lane_change_params(self):
        return lane_change_params()

    def set_lane_change(self, params, d_state):
        """arm the lane-changing agents (include/dmpp_b200.h section 13; the agent model must be armed): d_state = device address of
        dp_lane_change_state [n][max_obs] indexed like hdr, initialised by the placement step; d_state None / 0 disarms"""
        _ck(self.lib.dp_world_set_lane_change(self.ctx, C.byref(params) if params is not None else None, C.c_void_p(d_state or 0)),
            "dp_world_set_lane_change")

    def set_v2x_world(self, params, n, d_spec, d_wp_x=None, d_wp_y=None, n_wp=0, d_flags=None, d_stats=None):
        """arm the V2X events of closed-loop episodes (include/dmpp_b200.h section 14): params = V2xWorldParams (mode, apply);
        device addresses of spec[n] (dp_v2x_event_spec, indexed like hdr), the warning points wp_x / wp_y[n_wp], flags[n]
        (nullable) and stats[n]; d_spec None / 0 disarms"""
        _ck(self.lib.dp_world_set_v2x(self.ctx, C.byref(params) if params is not None else None, C.c_int(n), C.c_void_p(d_spec or 0),
                                      C.c_void_p(d_wp_x or 0), C.c_void_p(d_wp_y or 0), C.c_int(n_wp), C.c_void_p(d_flags or 0),
                                      C.c_void_p(d_stats or 0)), "dp_world_set_v2x")

    def set_v2x_traffic(self, params, d_stats):
        """let the agents obey the V2X events (include/dmpp_b200.h section 15; the agent model and the V2X events must be armed):
        d_stats = device address of dp_v2x_traffic_stats [n] indexed like hdr, initialised by the placement step; None / 0 disarms"""
        _ck(self.lib.dp_world_set_v2x_traffic(self.ctx, C.byref(params) if params is not None else None, C.c_void_p(d_stats or 0)),
            "dp_world_set_v2x_traffic")

    def set_v2x_obstacles(self, params, d_hdr_view, d_ox_view, d_oy_view, d_stats):
        """let the planner see the V2X road users (include/dmpp_b200.h section 16; the V2X events must be armed): device addresses of
        the views hdr_view[n] / ox_view / oy_view[n][max_obs] every cycle runs on and of dp_v2x_obstacle_stats [n], all indexed like
        hdr; d_stats None / 0 disarms"""
        _ck(self.lib.dp_world_set_v2x_obstacles(self.ctx, C.byref(params) if params is not None else None, C.c_void_p(d_hdr_view or 0),
                                                C.c_void_p(d_ox_view or 0), C.c_void_p(d_oy_view or 0), C.c_void_p(d_stats or 0)),
            "dp_world_set_v2x_obstacles")

    def v2x_obstacles_dev(self, n, d_hdr, d_ox, d_oy, d_prev_rec, cycle, tally=False, first=0, stream=0):
        """one obstacles launch of cycle `cycle` into the armed views, before cycle_dev runs on them; d_prev_rec = the records of cycle
        - 1 (None at cycle 0); tally=True: the row only, after the last world step and V2X tally"""
        _ck(self.lib.dp_v2x_obstacles_dev(self.ctx, C.c_int(first), C.c_int(n), C.c_void_p(d_hdr), C.c_void_p(d_ox), C.c_void_p(d_oy),
                                          C.c_void_p(d_prev_rec or 0), C.c_int(cycle), C.c_int(int(tally)), C.c_void_p(stream)),
            "dp_v2x_obstacles_dev")

    def v2x_world_dev(self, n, d_hdr, d_rec, cycle, first=0, stream=0):
        """one V2X launch of cycle `cycle` between cycle_dev and world_step_dev; d_rec None: the tally after the last step"""
        _ck(self.lib.dp_v2x_world_dev(self.ctx, C.c_int(first), C.c_int(n), C.c_void_p(d_hdr), C.c_void_p(d_rec or 0), C.c_int(cycle),
                                      C.c_void_p(stream)), "dp_v2x_world_dev")

    def world_step_dev(self, n, d_hdr, d_agents, d_ox, d_oy, d_rec=None, first=0, stream=0):
        _ck(self.lib.dp_world_step_dev(self.ctx, C.c_int(first), C.c_int(n), C.c_void_p(d_hdr), C.c_void_p(d_agents), C.c_void_p(d_ox),
                                       C.c_void_p(d_oy), C.c_void_p(d_rec or 0), C.c_void_p(stream)), "dp_world_step_dev")

    def run_closed_loop_dev(self, n, cycles, d_hdr, d_agents, d_ox, d_oy, d_rec, d_hdr_log=None, d_obs_log_x=None, d_obs_log_y=None,
                            first=0, stream=0):
        _ck(self.lib.dp_run_closed_loop_dev(self.ctx, C.c_int(first), C.c_int(n), C.c_int(cycles), C.c_void_p(d_hdr), C.c_void_p(d_agents),
                                            C.c_void_p(d_ox), C.c_void_p(d_oy), C.c_void_p(d_rec), C.c_void_p(d_hdr_log or 0),
                                            C.c_void_p(d_obs_log_x or 0), C.c_void_p(d_obs_log_y or 0), C.c_void_p(stream)),
            "dp_run_closed_loop_dev")

    def run_closed_loop_part_dev(self, n, k0, cycles, finish, d_hdr, d_agents, d_ox, d_oy, d_rec, d_prev_rec=None, d_hdr_log=None,
                                 d_obs_log_x=None, d_obs_log_y=None, first=0, stream=0):
        """cycles k0 .. k0 + cycles - 1 of an episode (include/dmpp_b200.h section 17); finish: the tallies after the last step"""
        _ck(self.lib.dp_run_closed_loop_part_dev(self.ctx, first, n, k0, cycles, int(finish), d_hdr, d_agents, d_ox, d_oy, d_prev_rec,
                                                 d_rec, d_hdr_log, d_obs_log_x, d_obs_log_y, stream), "dp_run_closed_loop_part_dev")

    def world_fork_dev(self, n, src, dst, d_hdr, d_agents, d_ox, d_oy, d_prev_rec=None, first=0, stream=0):
        """world dst + j becomes a copy of world src[j] in every per-world buffer (include/dmpp_b200.h section 17)"""
        src = np.ascontiguousarray(src, np.int32)
        _ck(self.lib.dp_world_fork_dev(self.ctx, first, n, src.ctypes.data if src.size else None, dst, src.size, d_hdr, d_agents, d_ox,
                                       d_oy, d_prev_rec, stream), "dp_world_fork_dev")

    def set_split(self, params, n, d_rows, d_groups):
        """arm splitting (include/dmpp_b200.h section 18) with rows[n] / groups[n / group] on the device; d_rows None disarms"""
        _ck(self.lib.dp_world_set_split(self.ctx, C.byref(params) if params is not None else None, n, d_rows, d_groups), "dp_world_set_split")

    def world_split_dev(self, n, level, d_hdr, d_agents, d_ox, d_oy, d_prev_rec=None, first=0, stream=0):
        """one split of worlds 0 .. n-1: select -> copy -> perturb (three launches)"""
        _ck(self.lib.dp_world_split_dev(self.ctx, first, n, level, d_hdr, d_agents, d_ox, d_oy, d_prev_rec, stream), "dp_world_split_dev")

    def split_map(self, n, stream=0):
        """the sources of the last split (copied on the split's stream and synchronised), -1 for the worlds that were not copied"""
        m = np.zeros(n, np.int32)
        _ck(self.lib.dp_world_split_map(self.ctx, n, m.ctypes.data, stream), "dp_world_split_map")
        return m

    def episode(self, hdr, agents, metrics=None, agent_model=None, lane_change=None, v2x=None, traffic=None, obstacles=None, split=None):
        """an episode to run in parts (Episode): the models are armed as run_closed_loop arms them, until Episode.close(); split:
        SplitParams (needs metrics) arms splitting between the parts (Episode.split)"""
        return Episode(self, hdr, agents, metrics, agent_model, lane_change, v2x, traffic, obstacles, split)

    def closed_loop_is_graph(self):
        return bool(self.lib.dp_closed_loop_is_graph(self.ctx))

    def run_closed_loop(self, hdr, agents, cycles, log=True, repeat=1, metrics=None, agent_model=None, lane_change=None, v2x=None,
                        traffic=None, obstacles=None):
        """host arrays in, host arrays out (the same dictionary as oracle.binding's run_closed_loop); `repeat` > 1 replays the
        episode from the same initial world (same device buffers, i.e. the cached graph) and returns the last run.
        metrics: None, or MetricsParams: the episode metrics are armed for this call (and disarmed after it) and the rows are
        returned under the key "metrics".  agent_model: None, or (AgentModelParams, v0[n][max_obs] desired speeds in m/s): the
        reactive agents are armed for this call (and disarmed after it).  lane_change: None, or LaneChangeParams (needs
        agent_model): the agents also change lanes for this call, and their final states are returned under "lane_change_state".
        v2x: None, or (V2xWorldParams, events) with events.spec[n] / wp_x / wp_y (scenes.V2xEvents): the V2X events are armed for
        this call, the rows are returned under "v2x_stats" and the flags of the last launch under "v2x_flags".  traffic: None, or
        V2xTrafficParams (needs agent_model and v2x): the agents obey the V2X events for this call, and their rows are returned
        under "v2x_traffic".  obstacles: None, or V2xObstacleParams (needs v2x): every cycle runs on a view of the world with the V2X
        road users in it for this call (the logs record the views), and the rows are returned under "v2x_obstacles".
        One Episode, one finishing part."""
        ep = self.episode(hdr, agents, metrics, agent_model, lane_change, v2x, traffic, obstacles)
        try:
            for r in range(repeat):
                if r:
                    ep.restart()
                o = ep.run(cycles, finish=True, log=log)
            st = ep.state()
            graph = st.pop("graph")
            o = {**{k: st.pop(k) for k in ("hdr", "agents", "ox", "oy")}, **o, **st}
            o["graph"] = graph
            return o
        finally:
            ep.close()

    # ---- pipelined form: at most two cycles in flight, buffers page-locked (see include/dmpp_b200.h) ----
    def submit(self, hdr, ox, oy, rec, first=0):
        n = hdr.shape[0]
        assert hdr.dtype == abi.scene_hdr and ox.shape == (n, self.max_obs) and oy.shape == (n, self.max_obs) and rec.shape == (n,)
        _ck(self.lib.dp_cycle_submit(self.ctx, C.c_int(first), C.c_int(n), abi.ptr(hdr), abi.ptr(ox), abi.ptr(oy), abi.ptr(rec)),
            "dp_cycle_submit")

    def submit_raw(self, first, n, hdr_ptr, ox_ptr, oy_ptr, rec_ptr):
        """dp_cycle_submit with addresses the caller has resolved once (a replay loop re-submits the same pinned buffers)"""
        _ck(self.lib.dp_cycle_submit(self.ctx, first, n, hdr_ptr, ox_ptr, oy_ptr, rec_ptr), "dp_cycle_submit")

    def wait(self):
        _ck(self.lib.dp_cycle_wait(self.ctx), "dp_cycle_wait")

    def run_episodes(self, H, OX, OY, trace=True, paths=True):
        """all cycles of [cycles][n] scripted episodes from a fresh carry; same layout as the oracle."""
        cycles, n = H.shape
        self.reset(0, n)
        out = {"rec": np.zeros((cycles, n), abi.plan_record),
               "trace": np.zeros((cycles, n), abi.trace_record) if trace else None,
               "path_xy": np.zeros((cycles, n, 2, abi.PATH_POINTS)) if paths else None,
               "path_ll": np.zeros((cycles, n, 2, abi.OUT_POINTS)) if paths else None}
        for c in range(cycles):
            o = {"rec": out["rec"][c], "trace": out["trace"][c] if trace else None,
                 "path_xy": out["path_xy"][c] if paths else None, "path_ll": out["path_ll"][c] if paths else None}
            self.cycle(np.ascontiguousarray(H[c]), np.ascontiguousarray(OX[c]), np.ascontiguousarray(OY[c]),
                       trace=trace, paths=paths, out=o)
        out["carry"], out["last_path"] = self.download_carry(0, n)
        return out

    def download_carry(self, first, count):
        c = np.zeros(count, abi.carry)
        lp = np.zeros((count, 2, abi.PATH_POINTS))
        _ck(self.lib.dp_carry_download(self.ctx, C.c_int(first), C.c_int(count), abi.ptr(c), abi.ptr(lp)), "dp_carry_download")
        return c, lp

    def upload_carry(self, first, carry, last_path):
        _ck(self.lib.dp_carry_upload(self.ctx, C.c_int(first), C.c_int(carry.shape[0]), abi.ptr(carry), abi.ptr(last_path)),
            "dp_carry_upload")

    # ---- device-pointer form (inputs resident in HBM; `stream` is a cudaStream_t value) ------
    def cycle_dev(self, n, d_hdr, d_ox, d_oy, d_rec, first=0, d_trace=None, d_path_xy=None, d_path_ll=None, stream=0):
        _ck(self.lib.dp_cycle_batch_dev(self.ctx, C.c_int(first), C.c_int(n), C.c_void_p(d_hdr), C.c_void_p(d_ox),
                                        C.c_void_p(d_oy), C.c_void_p(d_rec), C.c_void_p(d_trace or 0),
                                        C.c_void_p(d_path_xy or 0), C.c_void_p(d_path_ll or 0), C.c_void_p(stream)),
            "dp_cycle_batch_dev")

    # ---- operator level (the CShare seam) -----------------------------------------------------
    def search_obstacle(self, paths, ox, oy, lat_min, lat_max):
        """paths: list of (x[], y[]); one obstacle set; per-path windows."""
        off = np.zeros(len(paths) + 1, np.int32)
        off[1:] = np.cumsum([len(p[0]) for p in paths])
        px = np.ascontiguousarray(np.concatenate([np.asarray(p[0], np.float64) for p in paths]) if paths else np.zeros(0))
        py = np.ascontiguousarray(np.concatenate([np.asarray(p[1], np.float64) for p in paths]) if paths else np.zeros(0))
        ox, oy = np.ascontiguousarray(ox, np.float64), np.ascontiguousarray(oy, np.float64)
        lo = np.ascontiguousarray(np.broadcast_to(lat_min, len(paths)), np.float64)
        hi = np.ascontiguousarray(np.broadcast_to(lat_max, len(paths)), np.float64)
        out = np.zeros(len(paths), abi.search_slot)
        _ck(self.lib.dp_search_obstacle(self.ctx, C.c_int(len(paths)), abi.ptr(off), abi.ptr(px), abi.ptr(py), abi.ptr(ox),
                                        abi.ptr(oy), C.c_int(ox.size), abi.ptr(lo), abi.ptr(hi), abi.ptr(out)), "dp_search_obstacle")
        return out

    def create_new_path(self, paths, offsets):
        off = np.zeros(len(paths) + 1, np.int32)
        off[1:] = np.cumsum([len(p[0]) for p in paths])
        px = np.ascontiguousarray(np.concatenate([np.asarray(p[0], np.float64) for p in paths]))
        py = np.ascontiguousarray(np.concatenate([np.asarray(p[1], np.float64) for p in paths]))
        d = np.ascontiguousarray(offsets, np.float64)
        ox, oy = np.zeros_like(px), np.zeros_like(py)
        _ck(self.lib.dp_create_new_path(self.ctx, C.c_int(len(paths)), abi.ptr(off), abi.ptr(px), abi.ptr(py), abi.ptr(d),
                                        abi.ptr(ox), abi.ptr(oy)), "dp_create_new_path")
        return [(ox[off[i]:off[i + 1]], oy[off[i]:off[i + 1]]) for i in range(len(paths))]

    def bezier_planning(self, poses):
        poses = np.ascontiguousarray(poses, np.float64).reshape(-1, 6)
        out = np.zeros((poses.shape[0], 2, abi.PATH_POINTS))
        _ck(self.lib.dp_bezier_planning(self.ctx, C.c_int(poses.shape[0]), abi.ptr(poses), abi.ptr(out)), "dp_bezier_planning")
        return out

    def nearest_id(self, paths, qx, qy):
        """CShare::NearestId, one query point per path"""
        off = np.zeros(len(paths) + 1, np.int32)
        off[1:] = np.cumsum([len(p[0]) for p in paths])
        px = np.ascontiguousarray(np.concatenate([np.asarray(p[0], np.float64) for p in paths]))
        py = np.ascontiguousarray(np.concatenate([np.asarray(p[1], np.float64) for p in paths]))
        qx, qy = np.ascontiguousarray(qx, np.float64), np.ascontiguousarray(qy, np.float64)
        out = np.zeros(len(paths), np.int32)
        _ck(self.lib.dp_nearest_id(self.ctx, C.c_int(len(paths)), abi.ptr(off), abi.ptr(px), abi.ptr(py), abi.ptr(qx), abi.ptr(qy),
                                   abi.ptr(out)), "dp_nearest_id")
        return out

    def mean_points(self, paths):
        off = np.zeros(len(paths) + 1, np.int32)
        off[1:] = np.cumsum([len(p[0]) for p in paths])
        px = np.ascontiguousarray(np.concatenate([np.asarray(p[0], np.float64) for p in paths]))
        py = np.ascontiguousarray(np.concatenate([np.asarray(p[1], np.float64) for p in paths]))
        out = np.zeros((len(paths), 2, abi.PATH_POINTS))
        _ck(self.lib.dp_mean_points(self.ctx, C.c_int(len(paths)), abi.ptr(off), abi.ptr(px), abi.ptr(py), abi.ptr(out)), "dp_mean_points")
        return out

    def score_candidates(self, base_x, base_y, offset, n_pts, ox, oy, dvx=None, dvy=None, lat_min=-0.9, lat_max=0.9,
                         clear_dis=25.0, want_all=True):
        bx, by = np.ascontiguousarray(base_x, np.float64), np.ascontiguousarray(base_y, np.float64)
        off = np.ascontiguousarray(offset, np.float64)
        npt = np.ascontiguousarray(n_pts, np.int32)
        ox, oy = np.ascontiguousarray(ox, np.float64), np.ascontiguousarray(oy, np.float64)
        dvx = None if dvx is None else np.ascontiguousarray(dvx, np.float64)
        dvy = None if dvy is None else np.ascontiguousarray(dvy, np.float64)
        best = C.c_int32(-1)
        best_d = C.c_double(0)
        allv = np.zeros(off.size) if want_all else None
        _ck(self.lib.dp_score_candidates(self.ctx, abi.ptr(bx), abi.ptr(by), C.c_int(bx.size), abi.ptr(off), abi.ptr(npt),
                                         C.c_int(off.size), abi.ptr(ox), abi.ptr(oy), abi.ptr(dvx), abi.ptr(dvy), C.c_int(ox.size),
                                         C.c_double(lat_min), C.c_double(lat_max), C.c_double(clear_dis), C.byref(best),
                                         C.byref(best_d), abi.ptr(allv)), "dp_score_candidates")
        return best.value, best_d.value, allv

    def sweep_session(self, base_x, base_y, offset, n_pts, max_obs, **kw):
        return SweepSession(self, base_x, base_y, offset, n_pts, max_obs, **kw)

    def measure_fma_peak(self):
        a, b = C.c_double(0), C.c_double(0)
        _ck(self.lib.dp_measure_fma_peak(self.ctx, C.byref(a), C.byref(b)), "dp_measure_fma_peak")
        return a.value, b.value


class Episode:
    """a closed-loop episode run in parts (include/dmpp_b200.h section 17) on worlds 0 .. n-1 of a planner: owns the device buffers
    of the world and of the armed models, which stay armed until close().  run() continues the episode where the last part left
    it; fork() copies worlds on the device; state() downloads the world and the rows."""

    def __init__(self, planner, hdr, agents, metrics=None, agent_model=None, lane_change=None, v2x=None, traffic=None, obstacles=None,
                 split=None):
        n, mo = agents.shape
        assert split is None or (metrics is not None and n % split.group == 0), "the split scores the metrics rows of whole populations"
        assert lane_change is None or agent_model is not None, "lane changes run on the reactive agents"
        assert traffic is None or (agent_model is not None and v2x is not None), "the agents obey the V2X events on the reactive agents"
        assert obstacles is None or v2x is not None, "the planner sees the V2X road users of the armed V2X events"
        assert mo == planner.max_obs and hdr.shape == (n,) and n <= planner.max_scenes
        self.p, self.lib, self.n, self.mo = planner, planner.lib, n, mo
        self.models = dict(metrics=metrics, agent_model=agent_model, lane_change=lane_change, v2x=v2x, traffic=traffic, obstacles=obstacles,
                           split=split)
        self.h0, self.a0 = np.ascontiguousarray(hdr), np.ascontiguousarray(agents)
        sizes = {"hdr": n * 128, "agents": n * mo * 32, "ox": n * mo * 8, "oy": n * mo * 8, "prev_rec": n * 128}
        if metrics is not None:
            sizes["metrics"] = n * abi.episode_metrics.itemsize
        if agent_model is not None:
            am, v0 = agent_model
            v0 = np.ascontiguousarray(v0, np.float64)
            assert v0.shape == (n, mo)
            sizes["v0"] = n * mo * 8
        if lane_change is not None:
            sizes["lane_change_state"] = n * mo * abi.lane_change_state.itemsize
        if v2x is not None:
            vp, ev = v2x
            spec, wx, wy = np.ascontiguousarray(ev.spec), np.ascontiguousarray(ev.wp_x, np.float64), np.ascontiguousarray(ev.wp_y, np.float64)
            assert spec.dtype == abi.v2x_event_spec and spec.shape == (n,) and wx.shape == wy.shape
            sizes.update(v2x_spec=n * spec.itemsize, v2x_wp_x=max(wx.nbytes, 8), v2x_wp_y=max(wy.nbytes, 8),
                         v2x_flags=n * abi.v2x_flags.itemsize, v2x_stats=n * abi.v2x_episode_stats.itemsize)
        if traffic is not None:
            sizes["v2x_traffic"] = n * abi.v2x_traffic_stats.itemsize
        if obstacles is not None:
            sizes.update(v2x_hdr_view=n * 128, v2x_ox_view=n * mo * 8, v2x_oy_view=n * mo * 8, v2x_obstacles=n * abi.v2x_obstacle_stats.itemsize)
        if split is not None:
            sizes.update(split_rows=n * abi.split_row.itemsize, split_groups=n // split.group * abi.split_group.itemsize)
        self.sizes, self.d = sizes, {}
        self.k, self._cap = 0, {}                   # the next cycle of the episode; allocated part buffers: key -> (bytes, address)
        try:
            for k, b in sizes.items():
                self.d[k] = self._alloc(b)
            if metrics is not None:
                planner.set_metrics(metrics, self.d["metrics"])
            if agent_model is not None:
                self._h2d("v0", v0)
                planner.set_agent_model(am, self.d["v0"])
            if lane_change is not None:
                planner.set_lane_change(lane_change, self.d["lane_change_state"])
            if v2x is not None:
                for k, a in (("v2x_spec", spec), ("v2x_wp_x", wx), ("v2x_wp_y", wy)):
                    self._h2d(k, a)
                _ck(self.lib.dp_stream_sync(planner.ctx, None), "sync")
                planner.set_v2x_world(vp, n, self.d["v2x_spec"], self.d["v2x_wp_x"], self.d["v2x_wp_y"], wx.size, self.d["v2x_flags"],
                                      self.d["v2x_stats"])
            if traffic is not None:
                planner.set_v2x_traffic(traffic, self.d["v2x_traffic"])
            if obstacles is not None:
                planner.set_v2x_obstacles(obstacles, self.d["v2x_hdr_view"], self.d["v2x_ox_view"], self.d["v2x_oy_view"], self.d["v2x_obstacles"])
            if split is not None:
                planner.set_split(split, n, self.d["split_rows"], self.d["split_groups"])
            self.restart()
        except BaseException:
            self.close()
            raise

    def _alloc(self, b):
        p = C.c_void_p()
        _ck(self.lib.dp_dev_alloc(self.p.ctx, C.byref(p), C.c_size_t(b)), "dp_dev_alloc")
        return p.value

    def _h2d(self, k, a, offset=0):
        _ck(self.lib.dp_memcpy_h2d(self.p.ctx, C.c_void_p(self.d[k] + offset), abi.ptr(a), C.c_size_t(a.nbytes), None), "h2d")

    def _d2h(self, a, addr, nbytes):
        _ck(self.lib.dp_memcpy_d2h(self.p.ctx, abi.ptr(a), C.c_void_p(addr), C.c_size_t(nbytes), None), "d2h")

    def _part_buf(self, k, b):
        """a device buffer of at least b bytes for the parts' records / logs (grown when a longer part needs it)"""
        have = self._cap.get(k)
        if have is None or have[0] < b:
            if have is not None:
                self.lib.dp_dev_free(self.p.ctx, C.c_void_p(have[1]))
            self._cap[k] = have = (b, self._alloc(max(b, 8)))
        return have[1]

    def restart(self):
        """back to cycle 0 with the initial world (a fresh carry; the placement step of the next part initialises the rows)"""
        self.p.reset(0, self.n)
        self._h2d("hdr", self.h0)
        self._h2d("agents", self.a0)
        _ck(self.lib.dp_stream_sync(self.p.ctx, None), "sync")
        self.k = 0

    def run(self, cycles, finish=False, log=True):
        """cycles k .. k + cycles - 1 of the episode (k = the cycles run so far), then with finish the tallies.  Returns the part's
        records rec[cycles][n] and, with log, hdr_log / obs_log_x / obs_log_y [cycles][n](max_obs)"""
        n, mo, d = self.n, self.mo, self.d
        rec = self._part_buf("rec", cycles * n * 128)
        logs = {}
        if log:
            logs = {"hdr_log": self._part_buf("hdr_log", cycles * n * 128), "obs_log_x": self._part_buf("obs_log_x", cycles * n * mo * 8),
                    "obs_log_y": self._part_buf("obs_log_y", cycles * n * mo * 8)}
        self.p.run_closed_loop_part_dev(n, self.k, cycles, finish, d["hdr"], d["agents"], d["ox"], d["oy"], rec, d["prev_rec"],
                                        logs.get("hdr_log"), logs.get("obs_log_x"), logs.get("obs_log_y"))
        _ck(self.lib.dp_stream_sync(self.p.ctx, None), "sync")
        o = {"rec": np.zeros((cycles, n), abi.plan_record)}
        if log:
            o.update(hdr_log=np.zeros((cycles, n), abi.scene_hdr), obs_log_x=np.zeros((cycles, n, mo)), obs_log_y=np.zeros((cycles, n, mo)))
        self._d2h(o["rec"], rec, o["rec"].nbytes)
        for k in logs:
            self._d2h(o[k], logs[k], o[k].nbytes)
        if cycles > 0:                              # the next part's prev_rec (section 16 reads it; fork copies it)
            self._h2d("prev_rec", o["rec"][-1])
        _ck(self.lib.dp_stream_sync(self.p.ctx, None), "sync")
        self.k += cycles
        o["graph"] = self.p.closed_loop_is_graph()
        return o

    def fork(self, src, dst):
        """world dst + j becomes a copy of world src[j] (dp_world_fork_dev): world, carry, carried path, rows, states and inputs"""
        d = self.d
        self.p.world_fork_dev(self.n, src, dst, d["hdr"], d["agents"], d["ox"], d["oy"], d["prev_rec"])
        _ck(self.lib.dp_stream_sync(self.p.ctx, None), "sync")

    def split(self, level):
        """split the populations between two parts (dp_world_split_dev): level = the index of this split in the episode, from 0"""
        d = self.d
        self.p.world_split_dev(self.n, level, d["hdr"], d["agents"], d["ox"], d["oy"], d["prev_rec"])
        _ck(self.lib.dp_stream_sync(self.p.ctx, None), "sync")

    def state(self):
        """run_closed_loop's dictionary without the records and the logs: the world, the rows and states of the armed models, the
        carry and the carried path, and whether the last part ran as a graph"""
        n, mo, m = self.n, self.mo, self.models
        o = {"hdr": np.zeros(n, abi.scene_hdr), "agents": np.zeros((n, mo), abi.agent), "ox": np.zeros((n, mo)), "oy": np.zeros((n, mo))}
        if m["metrics"] is not None:
            o["metrics"] = np.zeros(n, abi.episode_metrics)
        if m["lane_change"] is not None:
            o["lane_change_state"] = np.zeros((n, mo), abi.lane_change_state)
        if m["v2x"] is not None:
            o["v2x_flags"], o["v2x_stats"] = np.zeros(n, abi.v2x_flags), np.zeros(n, abi.v2x_episode_stats)
        if m["traffic"] is not None:
            o["v2x_traffic"] = np.zeros(n, abi.v2x_traffic_stats)
        if m["obstacles"] is not None:
            o["v2x_obstacles"] = np.zeros(n, abi.v2x_obstacle_stats)
        if m["split"] is not None:
            o["split_rows"], o["split_groups"] = np.zeros(n, abi.split_row), np.zeros(n // m["split"].group, abi.split_group)
        for k in o:
            self._d2h(o[k], self.d[k], self.sizes[k])
        _ck(self.lib.dp_stream_sync(self.p.ctx, None), "sync")
        o["carry"], o["last_path"] = self.p.download_carry(0, n)
        o["graph"] = self.p.closed_loop_is_graph()
        return o

    def close(self):
        """disarm the models and free the buffers"""
        p, m = self.p, self.models
        if not p.ctx or self.d is None:
            return
        try:
            if m["split"] is not None:
                p.set_split(None, 0, None, None)
            if m["obstacles"] is not None:
                p.set_v2x_obstacles(None, None, None, None, None)
            if m["traffic"] is not None:
                p.set_v2x_traffic(None, None)
            if m["v2x"] is not None:
                p.set_v2x_world(None, 0, None)
            if m["metrics"] is not None:
                p.set_metrics(None, None)
            if m["lane_change"] is not None:
                p.set_lane_change(None, None)
            if m["agent_model"] is not None:
                p.set_agent_model(None, None)
        finally:
            for a in list(self.d.values()) + [v[1] for v in self._cap.values()]:
                self.lib.dp_dev_free(p.ctx, C.c_void_p(a))
            self.d, self._cap = None, {}


class Gather:
    """fused record gather across the GPUs of one box through the C ABI (CUDA IPC), see include/dmpp_b200.h dp_gather_*"""
    IPC_BYTES = 64

    def __init__(self, planner, world, rank, slots, depth=4):
        self.lib, self.planner, self.world, self.rank, self.slots = planner.lib, planner, world, rank, slots
        self.h = C.c_void_p()
        self.handle = (C.c_ubyte * self.IPC_BYTES)()
        _ck(self.lib.dp_gather_create(planner.ctx, C.c_int(world), C.c_int(rank), C.c_int(slots), C.c_int(depth), C.byref(self.h), self.handle),
            "dp_gather_create")
        self.lib.dp_gather_buffer.restype = C.c_void_p

    def my_handle(self):
        return bytes(self.handle)

    def attach(self, handles):
        """handles: list of `world` 64-byte handles, index = rank"""
        buf = (C.c_ubyte * (self.IPC_BYTES * self.world))(*b"".join(handles))
        _ck(self.lib.dp_gather_attach(self.h, buf), "dp_gather_attach")

    def arm(self, step):
        _ck(self.lib.dp_gather_arm(self.h, C.c_uint(step)), "dp_gather_arm")

    def chain(self, prev_step):
        """the next cycle launch also waits (in its last warp) for every rank's flag of prev_step; 0 = off"""
        _ck(self.lib.dp_gather_chain(self.h, C.c_uint(prev_step)), "dp_gather_chain")

    def arm_deferred(self, step):
        """the next cycle launch keeps its records local and forwards / flags / awaits the step armed before it"""
        _ck(self.lib.dp_gather_arm_deferred(self.h, C.c_uint(step)), "dp_gather_arm_deferred")

    def set_lag(self, lag):
        """deferred mode: a launch awaits the flags of the step `lag` launches back (1, or 2 with depth >= 4)"""
        _ck(self.lib.dp_gather_set_lag(self.h, C.c_int(lag)), "dp_gather_set_lag")

    def flush(self, stream=0):
        """forward, flag and await the last deferred step (end of a sequence)"""
        _ck(self.lib.dp_gather_flush(self.h, C.c_void_p(stream)), "dp_gather_flush")

    def disarm(self):
        _ck(self.lib.dp_gather_disarm(self.h), "dp_gather_disarm")

    def wait(self, step, stream=0):
        _ck(self.lib.dp_gather_wait(self.h, C.c_uint(step), C.c_void_p(stream)), "dp_gather_wait")

    def buffer(self, step):
        return int(self.lib.dp_gather_buffer(self.h, C.c_uint(step)))

    def close(self):
        if self.h:
            self.lib.dp_gather_destroy(self.h)
            self.h = C.c_void_p()


class SweepSession:
    """latency-mode dense candidate sweep (BASELINE config 3): candidate set resident on the device, one kernel launch per call
    (obstacles in the kernel parameters, winner written to page-locked memory by the grid's last CTA).
    base_x/base_y: ONE base line; or lines=[n_lines][2][n_base] + cand_line; or bezier_lines=n (lines drawn on the device by
    set_bezier(poses[n][6]))"""

    def __init__(self, planner, base_x, base_y, offset, n_pts, max_obs, lines=None, cand_line=None, bezier_lines=0):
        self.lib = planner.lib
        off, npt = np.ascontiguousarray(offset, np.float64), np.ascontiguousarray(n_pts, np.int32)
        self.h = C.c_void_p()
        self.n_lines, self.n_base = 1, 0
        if bezier_lines:
            cl = np.ascontiguousarray(cand_line, np.int32)
            self.n_lines, self.n_base = int(bezier_lines), 200
            _ck(self.lib.dp_sweep_create_bezier(planner.ctx, C.byref(self.h), C.c_int(self.n_lines), abi.ptr(cl), abi.ptr(off), abi.ptr(npt),
                                                C.c_int(off.size), C.c_int(max_obs)), "dp_sweep_create_bezier")
        elif lines is not None:
            ln, cl = np.ascontiguousarray(lines, np.float64), np.ascontiguousarray(cand_line, np.int32)
            self.n_lines, self.n_base = ln.shape[0], ln.shape[2]
            _ck(self.lib.dp_sweep_create_lines(planner.ctx, C.byref(self.h), abi.ptr(ln), C.c_int(ln.shape[0]), C.c_int(ln.shape[2]), abi.ptr(cl),
                                               abi.ptr(off), abi.ptr(npt), C.c_int(off.size), C.c_int(max_obs)), "dp_sweep_create_lines")
        else:
            bx, by = np.ascontiguousarray(base_x, np.float64), np.ascontiguousarray(base_y, np.float64)
            self.n_base = bx.size
            _ck(self.lib.dp_sweep_create(planner.ctx, C.byref(self.h), abi.ptr(bx), abi.ptr(by), C.c_int(bx.size), abi.ptr(off), abi.ptr(npt),
                                         C.c_int(off.size), C.c_int(max_obs)), "dp_sweep_create")
        self._ms = C.c_float(0)
        self._best = C.c_int32(-1)
        self._dis = C.c_double(0)

    def set_bezier(self, poses, want_ms=False):
        """poses[n_lines][6] = start x, y, dir, aim x, y, dir: the lines are rolled out on the device; returns device ms if asked"""
        ps = np.ascontiguousarray(poses, np.float64)
        assert ps.shape == (self.n_lines, 6)
        _ck(self.lib.dp_sweep_set_bezier(self.h, abi.ptr(ps), C.byref(self._ms) if want_ms else None), "dp_sweep_set_bezier")
        return self._ms.value if want_ms else None

    def lines(self):
        out = np.zeros((self.n_lines, 2, self.n_base))
        _ck(self.lib.dp_sweep_lines(self.h, abi.ptr(out)), "dp_sweep_lines")
        return out

    def score(self, ox, oy, dvx=None, dvy=None, lat_min=-0.9, lat_max=0.9, clear_dis=25.0, want_dis=True, want_ms=True):
        ox, oy = np.ascontiguousarray(ox, np.float64), np.ascontiguousarray(oy, np.float64)
        dvx = None if dvx is None else np.ascontiguousarray(dvx, np.float64)
        dvy = None if dvy is None else np.ascontiguousarray(dvy, np.float64)
        _ck(self.lib.dp_sweep_score(self.h, abi.ptr(ox), abi.ptr(oy), abi.ptr(dvx), abi.ptr(dvy), C.c_int(ox.size), C.c_double(lat_min),
                                    C.c_double(lat_max), C.c_double(clear_dis), C.byref(self._best),
                                    C.byref(self._dis) if want_dis else None, C.byref(self._ms) if want_ms else None), "dp_sweep_score")
        return self._best.value, self._dis.value, self._ms.value

    def close(self):
        if self.h:
            self.lib.dp_sweep_destroy(self.h)
            self.h = C.c_void_p()
