"""tools/junction_oracle/binding.py -- TEST INFRASTRUCTURE: ctypes loaders of the junction world-step oracle
(libjunction_oracle.so) and of the unmodified reference's closed loop with that step (libref_junction.so, where the reference
was built).  Same dictionaries as oracle.binding's run_closed_loop.  Imported by tests/ only."""
import ctypes as C
import os
import subprocess
import sys
import types

import numpy as np

_here = os.path.dirname(os.path.abspath(__file__))
_root = os.path.dirname(os.path.dirname(_here))
if _root not in sys.path:
    sys.path.insert(0, _root)
import dmpp_b200  # noqa: E402,F401
from dmpp_b200 import abi  # noqa: E402
from oracle import binding as ob  # noqa: E402


def build():
    subprocess.check_call(["make", "-s", "-C", _here, "all"])


class JunctionOracle:
    def __init__(self):
        build()
        self.lib = C.CDLL(os.path.join(_here, "libjunction_oracle.so"), mode=os.RTLD_NOW)
        self._base = ob.Oracle()
        self.params = self._base.params

    def set_map(self, m):
        self._keep = m
        self._desc = m.desc()
        assert self.lib.jo_set_map(C.byref(self._desc)) == 0
        self._n_lanes = m.n_lanes

    def world_params(self):
        return self._base.world_params()

    def lane_next(self):
        out = np.zeros(self._n_lanes, np.int32)
        assert self.lib.jo_lane_next(abi.ptr(out)) == 0
        return out

    def world_step(self, hdr, agents, ox, oy, rec=None, last_path=None, wp=None):
        """in place; rec None: place the agents and localise only"""
        wp = wp or self.world_params()
        n, max_obs = ox.shape
        assert self.lib.jo_world_step(C.byref(self.params), C.byref(wp), C.c_int(n), C.c_int(max_obs), abi.ptr(hdr), abi.ptr(agents),
                                      abi.ptr(ox), abi.ptr(oy), abi.ptr(rec), abi.ptr(last_path)) == 0

    def run_closed_loop(self, hdr, agents, cycles, wp=None, paths=False, threads=1, metrics=None, agent_model=None, lane_change=None,
                        v2x=None, traffic=None, obstacles=None):
        """hdr[n], agents[n][max_obs] (copied; the final world is returned), through jo_run_closed_loop; metrics = MetricsParams: the
        episode metrics of every world under "metrics"; agent_model = (AgentModelParams, v0[n][max_obs]): the reactive agents;
        lane_change = LaneChangeParams (with agent_model): their lane changes, the final states under "lane_change_state";
        v2x = (V2xWorldParams, events with spec / wp_x / wp_y): the V2X events, the rows under "v2x_stats" and the flags of the last
        launch under "v2x_flags"; traffic = V2xTrafficParams (with agent_model and v2x): the agents obey the V2X events, the rows
        under "v2x_traffic"; obstacles = V2xObstacleParams (with v2x): every cycle runs on the view of the V2X road users, the logs
        record the views, the rows under "v2x_obstacles"
        """
        assert lane_change is None or agent_model is not None
        assert traffic is None or (agent_model is not None and v2x is not None)
        assert obstacles is None or v2x is not None
        am, v0 = agent_model if agent_model is not None else (None, None)
        met = lcs = None
        if metrics is not None:
            met = np.frombuffer(np.full(hdr.shape[0] * abi.episode_metrics.itemsize, 0xAB, np.uint8).tobytes(), abi.episode_metrics).copy()
        if v0 is not None:
            v0 = np.ascontiguousarray(v0, np.float64)
            assert v0.shape == agents.shape
        if lane_change is not None:
            lcs = np.frombuffer(np.full(agents.size * abi.lane_change_state.itemsize, 0xAB, np.uint8).tobytes(),
                                abi.lane_change_state).reshape(agents.shape).copy()
        ref = lambda p: None if p is None else C.byref(p)
        models = (ref(metrics), abi.ptr(met), ref(am), abi.ptr(v0), ref(lane_change), abi.ptr(lcs))
        vflags = vstats = None
        if v2x is not None:
            vp, ev = v2x
            spec, wx, wy = self._v2x_inputs(ev)
            n = hdr.shape[0]
            assert spec.shape == (n,)
            vflags = np.frombuffer(np.full(n * abi.v2x_flags.itemsize, 0xAB, np.uint8).tobytes(), abi.v2x_flags).copy()
            vstats = np.frombuffer(np.full(n * abi.v2x_episode_stats.itemsize, 0xAB, np.uint8).tobytes(), abi.v2x_episode_stats).copy()
            models += (C.byref(vp), abi.ptr(spec), abi.ptr(wx), abi.ptr(wy), C.c_int(wx.size), abi.ptr(vflags), abi.ptr(vstats))
        else:
            models += (None,) * 4 + (C.c_int(0), None, None)
        tstats = None
        if traffic is not None:
            tstats = np.frombuffer(np.full(hdr.shape[0] * abi.v2x_traffic_stats.itemsize, 0xAB, np.uint8).tobytes(), abi.v2x_traffic_stats).copy()
        models += (ref(traffic), abi.ptr(tstats))
        ostats = None
        if obstacles is not None:
            ostats = np.frombuffer(np.full(hdr.shape[0] * abi.v2x_obstacle_stats.itemsize, 0xAB, np.uint8).tobytes(), abi.v2x_obstacle_stats).copy()
        models += (ref(obstacles), abi.ptr(ostats))
        f = self.lib.jo_run_closed_loop
        f.restype = C.c_longlong
        # ob._closed_loop passes the arrays every closed loop has; the model arguments follow them
        o = ob._closed_loop(types.SimpleNamespace(jo_run_closed_loop=lambda *a: f(*a, *models)), "jo_run_closed_loop", self.params,
                            wp or self.world_params(), hdr, agents, cycles, paths, threads)
        if met is not None:
            o["metrics"] = met
        if lcs is not None:
            o["lane_change_state"] = lcs
        if vstats is not None:
            o["v2x_flags"], o["v2x_stats"] = vflags, vstats
        if tstats is not None:
            o["v2x_traffic"] = tstats
        if ostats is not None:
            o["v2x_obstacles"] = ostats
        return o

    @staticmethod
    def closed_loop_state(hdr, agents, metrics=None, lane_change=None, v2x=None, traffic=None, obstacles=None):
        """the state run_closed_loop_part carries from part to part, fresh for k0 = 0: copies of hdr / agents, ox / oy, carry and
        last_path, and the rows and states of the armed models (0xAB-filled, as run_closed_loop hands them over) under
        run_closed_loop's keys"""
        n, max_obs = agents.shape

        def junk(dt, shape):
            return np.frombuffer(np.full(int(np.prod(shape)) * dt.itemsize, 0xAB, np.uint8).tobytes(), dt).reshape(shape).copy()

        st = {"hdr": hdr.copy(), "agents": agents.copy(), "ox": np.zeros((n, max_obs)), "oy": np.zeros((n, max_obs)),
              "carry": np.zeros(n, abi.carry), "last_path": np.zeros((n, 2, abi.PATH_POINTS))}
        if metrics is not None:
            st["metrics"] = junk(abi.episode_metrics, (n,))
        if lane_change is not None:
            st["lane_change_state"] = junk(abi.lane_change_state, agents.shape)
        if v2x is not None:
            st["v2x_flags"], st["v2x_stats"] = junk(abi.v2x_flags, (n,)), junk(abi.v2x_episode_stats, (n,))
        if traffic is not None:
            st["v2x_traffic"] = junk(abi.v2x_traffic_stats, (n,))
        if obstacles is not None:
            st["v2x_obstacles"] = junk(abi.v2x_obstacle_stats, (n,))
        return st

    def run_closed_loop_part(self, state, k0, cycles, finish=False, prev_rec=None, wp=None, paths=False, threads=1, metrics=None,
                             agent_model=None, lane_change=None, v2x=None, traffic=None, obstacles=None):
        """cycles k0 .. k0 + cycles - 1 of an episode (jo_run_closed_loop_part), on the state of closed_loop_state (k0 = 0) or of the
        previous part, in place; prev_rec[n] the records of cycle k0 - 1 (needed with obstacles when k0 > 0); finish: the tallies.
        The models as run_closed_loop takes them, their rows in the state.  Returns the part's rec, hdr_log, obs_log_x / obs_log_y
        (and path_xy) [cycles][n], ub_scene and status"""
        assert lane_change is None or agent_model is not None
        assert traffic is None or (agent_model is not None and v2x is not None)
        assert obstacles is None or v2x is not None
        st = state
        n, max_obs = st["agents"].shape
        am, v0 = agent_model if agent_model is not None else (None, None)
        if v0 is not None:
            v0 = np.ascontiguousarray(v0, np.float64)
            assert v0.shape == (n, max_obs)
        ref = lambda p: None if p is None else C.byref(p)
        get = lambda k, armed: abi.ptr(st[k]) if armed is not None else None
        models = (ref(metrics), get("metrics", metrics), ref(am), abi.ptr(v0), ref(lane_change), get("lane_change_state", lane_change))
        if v2x is not None:
            vp, ev = v2x
            spec, wx, wy = self._v2x_inputs(ev)
            assert spec.shape == (n,)
            models += (C.byref(vp), abi.ptr(spec), abi.ptr(wx), abi.ptr(wy), C.c_int(wx.size), abi.ptr(st["v2x_flags"]), abi.ptr(st["v2x_stats"]))
        else:
            models += (None,) * 4 + (C.c_int(0), None, None)
        models += (ref(traffic), get("v2x_traffic", traffic), ref(obstacles), get("v2x_obstacles", obstacles))
        prev_rec = None if prev_rec is None else np.ascontiguousarray(prev_rec)
        assert prev_rec is None or prev_rec.shape == (n,)
        o = {"rec": np.zeros((cycles, n), abi.plan_record), "hdr_log": np.zeros((cycles, n), abi.scene_hdr),
             "obs_log_x": np.zeros((cycles, n, max_obs)), "obs_log_y": np.zeros((cycles, n, max_obs)),
             "path_xy": np.zeros((cycles, n, 2, abi.PATH_POINTS)) if paths else None, "ub_scene": np.zeros(n, np.int32)}
        f = self.lib.jo_run_closed_loop_part
        f.restype = C.c_longlong
        rc = f(C.byref(self.params), C.byref(wp or self.world_params()), C.c_int(n), C.c_int(k0), C.c_int(cycles), C.c_int(int(finish)),
               C.c_int(max_obs), abi.ptr(st["hdr"]), abi.ptr(st["agents"]), abi.ptr(st["ox"]), abi.ptr(st["oy"]), abi.ptr(prev_rec),
               abi.ptr(o["rec"]), abi.ptr(o["hdr_log"]), abi.ptr(o["obs_log_x"]), abi.ptr(o["obs_log_y"]), abi.ptr(o["path_xy"]),
               abi.ptr(st["carry"]), abi.ptr(st["last_path"]), C.c_int(threads), abi.ptr(o["ub_scene"]), *models)
        if rc < 0:
            raise RuntimeError("jo_run_closed_loop_part failed: %d" % rc)
        o["status"] = rc
        return o

    def split_select(self, sp, level, met, rows, groups):
        """the select launch of a split (jo_world_split_select) for the populations of met[n]: rows[n] / groups[n / M] in place;
        returns map[n] (the source of every destination, -1 elsewhere)"""
        n = len(met)
        out = np.zeros(n, np.int32)
        assert self.lib.jo_world_split_select(C.byref(sp), C.c_int(n), C.c_int(level), abi.ptr(met), abi.ptr(rows), abi.ptr(groups),
                                              abi.ptr(out)) == 0
        return out

    def perturb(self, sp, level, hdr, agents, v0=None):
        """the perturb launch of a split (jo_world_perturb): agents[n][max_obs] and v0 (when given) in place"""
        n, max_obs = agents.shape
        assert v0 is None or (v0.shape == agents.shape and v0.dtype == np.float64 and v0.flags["C_CONTIGUOUS"])
        assert self.lib.jo_world_perturb(C.byref(sp), C.c_int(n), C.c_int(level), C.c_int(max_obs), abi.ptr(hdr), abi.ptr(agents),
                                         abi.ptr(v0)) == 0

    def spec_exp(self, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros_like(x)
        assert self.lib.jo_spec_exp(C.c_int(x.size), abi.ptr(x), abi.ptr(y)) == 0
        return y

    def split_sizeof(self, which):
        return self.lib.jo_split_sizeof(C.c_int(which))

    def v2x_obstacles_view(self, op, ev, hdr, ox, oy, k, stats, prev=None, tally=False, view=None):
        """one obstacles launch of cycle k for every world (jo_v2x_obstacles_view): stats in place; returns the view (hdr, ox, oy),
        built into `view` when given (slots beyond the view's n_obs keep what they held), fresh zero arrays otherwise"""
        spec, wx, wy = self._v2x_inputs(ev)
        hdr, ox, oy = np.ascontiguousarray(hdr), np.ascontiguousarray(ox, np.float64), np.ascontiguousarray(oy, np.float64)
        n, max_obs = ox.shape
        assert spec.shape == hdr.shape == (n,) and oy.shape == ox.shape and stats.dtype == abi.v2x_obstacle_stats and stats.shape == (n,)
        prev = None if prev is None else np.ascontiguousarray(prev)
        hv, vx, vy = view if view is not None else (np.zeros(n, abi.scene_hdr), np.zeros((n, max_obs)), np.zeros((n, max_obs)))
        assert self.lib.jo_v2x_obstacles_view(C.byref(op), C.c_int(max_obs), C.c_int(n), abi.ptr(spec), abi.ptr(wx), abi.ptr(wy), abi.ptr(hdr),
                                              abi.ptr(ox), abi.ptr(oy), abi.ptr(prev), C.c_int(k), C.c_int(int(tally)), abi.ptr(hv),
                                              abi.ptr(vx), abi.ptr(vy), abi.ptr(stats)) == 0
        return hv, vx, vy

    def v2x_obstacles_sizeof(self):
        """sizeof(dp_v2x_obstacle_params), sizeof(dp_v2x_obstacle_stats)"""
        return int(self.lib.jo_v2x_obstacles_sizeof(0)), int(self.lib.jo_v2x_obstacles_sizeof(1))

    def traffic_step(self, tp, ev, k, hdr, agents, ox, oy, v0, am, ts, rec=None, last_path=None, lp=None, lcs=None, wp=None):
        """one world step of cycle k with the agents obeying the V2X events (jo_traffic_step), everything in place; rec None: the
        placement step (the rows initialised); returns the leader kinds [n][max_obs]"""
        wp = wp or self.world_params()
        n, max_obs = agents.shape
        spec = np.ascontiguousarray(ev.spec)
        v0 = np.ascontiguousarray(v0, np.float64)
        assert spec.shape == (n,) and v0.shape == agents.shape and ts.dtype == abi.v2x_traffic_stats and ts.shape == (n,)
        assert (lp is None) == (lcs is None) and agents.flags["C_CONTIGUOUS"] and hdr.flags["C_CONTIGUOUS"]
        kinds = np.zeros((n, max_obs), np.int32)
        assert self.lib.jo_traffic_step(C.byref(self.params), C.byref(wp), C.byref(am), None if lp is None else C.byref(lp), C.byref(tp),
                                        C.c_int(n), C.c_int(max_obs), abi.ptr(spec), C.c_int(k), abi.ptr(hdr), abi.ptr(agents), abi.ptr(ox),
                                        abi.ptr(oy), abi.ptr(v0), abi.ptr(lcs), abi.ptr(rec), abi.ptr(last_path), abi.ptr(ts),
                                        abi.ptr(kinds)) == 0
        return kinds

    def traffic_leader(self, tp, am, spec, hdr, k, lanes, x, iv):
        """section 15's candidates after a vehicle scan (jo_traffic_leader): lanes[n][3] = (l0, l1, l2), x[n][6] = (D1, D2, sk, v, u,
        best), iv[n][2] = (i, lead) -> [n][3] = (best, lead, kind)"""
        n = len(spec)
        out = np.zeros((n, 3))
        args = [np.ascontiguousarray(a, t) for a, t in ((spec, abi.v2x_event_spec), (hdr, abi.scene_hdr), (k, np.int32), (lanes, np.int32),
                                                        (x, np.float64), (iv, np.int32))]
        assert self.lib.jo_traffic_leader(C.byref(tp), C.byref(am), C.c_int(n), *[abi.ptr(a) for a in args], abi.ptr(out)) == 0
        return out

    def traffic_side(self, tp, am, spec, hdr, k, lanes, x, lead):
        """... on a target lane (jo_traffic_side): lanes[n][2] = (m, i_m), x[n][4] = (s_m, u, v, g), lead[n] -> [n][3] = (g, lead, won)"""
        n = len(spec)
        out = np.zeros((n, 3))
        args = [np.ascontiguousarray(a, t) for a, t in ((spec, abi.v2x_event_spec), (hdr, abi.scene_hdr), (k, np.int32), (lanes, np.int32),
                                                        (x, np.float64), (lead, np.int32))]
        assert self.lib.jo_traffic_side(C.byref(tp), C.byref(am), C.c_int(n), *[abi.ptr(a) for a in args], abi.ptr(out)) == 0
        return out

    def traffic_sizeof(self):
        """sizeof(dp_v2x_traffic_params), sizeof(dp_v2x_traffic_stats)"""
        return int(self.lib.jo_traffic_sizeof(0)), int(self.lib.jo_traffic_sizeof(1))

    @staticmethod
    def _v2x_inputs(ev):
        spec, wx, wy = np.ascontiguousarray(ev.spec), np.ascontiguousarray(ev.wp_x, np.float64), np.ascontiguousarray(ev.wp_y, np.float64)
        assert spec.dtype == abi.v2x_event_spec and wx.shape == wy.shape
        return spec, wx, wy

    def v2x_data(self, spec, hdr, k):
        """the V2X data builder alone (jo_v2x_data): data[n], aux[n][3] = (d, spat_state, on + 2 * ped_on)"""
        spec, hdr = np.ascontiguousarray(spec), np.ascontiguousarray(hdr)
        n = hdr.shape[0]
        data, aux = np.zeros(n, abi.v2x_data), np.zeros((n, 3))
        assert self.lib.jo_v2x_data(C.byref(self.params), C.c_int(n), abi.ptr(spec), abi.ptr(hdr), C.c_int(k), abi.ptr(data), abi.ptr(aux)) == 0
        return data, aux

    def v2x_cycle(self, vp, ev, hdr, rec, k, stats):
        """one V2X launch for every world (jo_v2x_cycle): rec (adjusted in place; None: the tally) and stats in place, returns the flags"""
        spec, wx, wy = self._v2x_inputs(ev)
        hdr = np.ascontiguousarray(hdr)
        n = hdr.shape[0]
        assert stats.dtype == abi.v2x_episode_stats and stats.shape == (n,) and (rec is None or rec.flags["C_CONTIGUOUS"])
        flags = np.zeros(n, abi.v2x_flags)
        assert self.lib.jo_v2x_cycle(C.byref(self.params), C.byref(vp), C.c_int(n), abi.ptr(spec), abi.ptr(wx), abi.ptr(wy), C.c_int(wx.size),
                                     abi.ptr(hdr), abi.ptr(rec), C.c_int(k), abi.ptr(flags), abi.ptr(stats)) == 0
        return flags

    def gps(self, x, y):
        """GlobalToWGS84 of the points (x, y): (lat, lng)"""
        x, y = np.ascontiguousarray(x, np.float64), np.ascontiguousarray(y, np.float64)
        la, lo = np.zeros(x.size), np.zeros(x.size)
        self.lib.jo_gps(C.byref(self.params), C.c_int(x.size), abi.ptr(x), abi.ptr(y), abi.ptr(la), abi.ptr(lo))
        return la, lo

    def v2x_sizeof(self):
        """sizeof(dp_v2x_event_spec), sizeof(dp_v2x_episode_stats)"""
        return int(self.lib.jo_v2x_sizeof(0)), int(self.lib.jo_v2x_sizeof(1))

    def react_step(self, hdr, agents, v0, am, wp=None):
        """the react phase alone, agents[n][max_obs] in place (jo_react_step)"""
        wp = wp or self.world_params()
        n, max_obs = agents.shape
        v0 = np.ascontiguousarray(v0, np.float64)
        assert v0.shape == agents.shape and hdr.shape == (n,) and agents.flags["C_CONTIGUOUS"]
        assert self.lib.jo_react_step(C.byref(wp), C.byref(am), C.c_int(n), C.c_int(max_obs), abi.ptr(np.ascontiguousarray(hdr)),
                                      abi.ptr(agents), abi.ptr(v0)) == 0

    def lane_change_step(self, hdr, agents, v0, am, lp, lcs, wp=None):
        """the react and lane-change phases alone, agents and lcs [n][max_obs] in place (jo_lane_change_step)"""
        wp = wp or self.world_params()
        n, max_obs = agents.shape
        v0 = np.ascontiguousarray(v0, np.float64)
        assert v0.shape == agents.shape == lcs.shape and hdr.shape == (n,) and agents.flags["C_CONTIGUOUS"] and lcs.flags["C_CONTIGUOUS"]
        assert lcs.dtype == abi.lane_change_state
        assert self.lib.jo_lane_change_step(C.byref(wp), C.byref(am), C.byref(lp), C.c_int(n), C.c_int(max_obs),
                                            abi.ptr(np.ascontiguousarray(hdr)), abi.ptr(agents), abi.ptr(v0), abi.ptr(lcs)) == 0

    def lane_change_sizeof(self):
        """sizeof(dp_lane_change_params), sizeof(dp_lane_change_state)"""
        return int(self.lib.jo_lane_change_sizeof(0)), int(self.lib.jo_lane_change_sizeof(1))

    def agent_model_sizeof(self):
        return int(self.lib.jo_agent_model_sizeof())

    def metrics_step(self, hdr, agents, ox, oy, met, mp, rec=None, last_path=None, wp=None):
        """one world step plus its metric update, in place (jo_metrics_step)"""
        wp = wp or self.world_params()
        n, max_obs = ox.shape
        assert met.dtype == abi.episode_metrics and met.shape == (n,)
        assert self.lib.jo_metrics_step(C.byref(self.params), C.byref(wp), C.byref(mp), C.c_int(n), C.c_int(max_obs), abi.ptr(hdr),
                                        abi.ptr(agents), abi.ptr(ox), abi.ptr(oy), abi.ptr(rec), abi.ptr(last_path), abi.ptr(met)) == 0

    def metrics_sizeof(self):
        return int(self.lib.jo_metrics_sizeof())

    def sincos_deg(self, a):
        c, s = C.c_double(0), C.c_double(0)
        self.lib.jo_sincos_deg(C.c_double(a), C.byref(c), C.byref(s))
        return c.value, s.value


class JunctionReference:
    """needs an oracle.binding.Reference whose map is set (the loop reads the reference's own map tables)"""

    @staticmethod
    def available():
        return os.path.exists(os.path.join(_here, "libref_junction.so"))

    def __init__(self):
        self.lib = C.CDLL(os.path.join(_here, "libref_junction.so"), mode=os.RTLD_NOW)

    def run_closed_loop(self, params, wp, hdr, agents, cycles, paths=False):
        return ob._closed_loop(self.lib, "ref_run_closed_loop_junction", params, wp, hdr, agents, cycles, paths, None)
