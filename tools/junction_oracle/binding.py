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
                        v2x=None):
        """hdr[n], agents[n][max_obs] (copied; the final world is returned), through jo_run_closed_loop; metrics = MetricsParams: the
        episode metrics of every world under "metrics"; agent_model = (AgentModelParams, v0[n][max_obs]): the reactive agents;
        lane_change = LaneChangeParams (with agent_model): their lane changes, the final states under "lane_change_state";
        v2x = (V2xWorldParams, events with spec / wp_x / wp_y): the V2X events, the rows under "v2x_stats" and the flags of the last
        launch under "v2x_flags"
        """
        assert lane_change is None or agent_model is not None
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
        return o

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
