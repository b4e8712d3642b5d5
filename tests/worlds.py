"""Helpers of the closed-loop model tests (episode metrics, reactive agents, lane changes, junctions): the junction checker fixture,
worlds and their parameters, planners, the model parameters, a straight-road map and the GPU-against-checker comparison.  A plain
module: a test module imports what it uses, the `joracle` fixture included."""
import os

import numpy as np
import pytest

from conftest import assert_records_equal
from test_closed_loop import HDR as SEGMENT_HDR, check_closed_loop as check_segment_loop

HDR = SEGMENT_HDR + ["last_roadnum", "next_roadnum", "last_lanenum", "next_lanenum", "stub_attribute", "conn"]
WORLD = ("rec", "hdr_log", "hdr", "agents", "ox", "oy", "obs_log_x", "obs_log_y", "carry", "last_path")
DT = 0.1
W = 3.75


@pytest.fixture(scope="module")
def joracle(the_map):
    from tools.junction_oracle.binding import JunctionOracle
    j = JunctionOracle()
    j.set_map(the_map)
    return j


def jworld(the_map, seed0, n, kind="junction", n_obs=10):
    from dmpp_b200 import scenes
    return scenes.World(the_map, np.arange(seed0, seed0 + n), n_obs=n_obs, kind=kind)


def jparams(src, kind="junction"):
    from dmpp_b200 import scenes
    wp = src.world_params()
    wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]
    return wp


def planner_with(the_map, n, max_obs, J, env=None):
    from dmpp_b200.planner import Planner
    env = env or {}
    os.environ.update(env)
    try:
        p = Planner(max_scenes=n, max_obs=max_obs)
    finally:
        for k in env:
            del os.environ[k]
    p.upload_map(the_map)
    wp = p.world_params(); wp.pre_junction_pts = J
    p.set_world_params(wp)
    return p


def check_closed_loop(got, want, what):
    check_segment_loop(got, want, what)                     # records, logs, final world (every header byte), carry, last path
    assert_records_equal(got["hdr_log"], want["hdr_log"], HDR, what=what + " logged header")


def _with(p, kw):
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def mparams():
    from dmpp_b200 import planner
    return planner.metrics_params()


def amparams(**kw):
    from dmpp_b200 import planner
    return _with(planner.agent_model_params(), kw)


def lcparams(**kw):
    from dmpp_b200 import planner
    return _with(planner.lane_change_params(), kw)


def cump_of(m):
    """the sequential prefix of every lane's segment lengths (dp_map_prep_kernel), independently in numpy"""
    c = np.zeros(m.x.size)
    for gl in range(m.n_lanes):
        o, e = int(m.lane_pt_off[gl]), int(m.lane_pt_off[gl + 1])
        dx, dy = np.diff(m.x[o:e]), np.diff(m.y[o:e])
        c[o + 1:e] = np.add.accumulate(np.sqrt(dx * dx + dy * dy))
    return c


def idm(v, v0, p, g=None, vl=None, dt=DT):
    """the IDM step of section 12 in numpy float64, the operations in the order the header writes them"""
    v, v0 = np.float64(v), np.float64(v0)
    r = v / v0
    fr = r * r
    fr = fr * fr
    if g is None:
        acc = p.a_max * (1.0 - fr)
    else:
        dv = v - vl
        z = v * p.T + v * dv / (2.0 * np.sqrt(p.a_max * p.b))
        z = max(z, 0.0)
        ss = p.s0 + z
        acc = p.a_max * (1.0 - fr - (ss / g) * (ss / g)) if g > 0 else -p.b_max
    acc = max(acc, -p.b_max)
    return max(v + acc * np.float64(dt), 0.0)


class StraightRoad:
    """one road of `lanes` lanes W apart along +x, centred on y = 0 (lane 1 on the left), n points 0.5 m apart, lane-change
    attribute `attr`; with connector=True a further parallel pseudo-lane on the right (attribute 3) is a connector leaving the last
    lane"""

    def __init__(self, n=1000, lanes=1, attr=0, connector=False):
        from dmpp_b200 import abi
        ys = W * (lanes - 1) / 2 - W * np.arange(lanes + int(connector))
        self.n_roads, self.n_lanes = 1, len(ys)
        self.road_lane_base = np.array([0, lanes], np.int32)
        self.lane_pt_off = (n * np.arange(len(ys) + 1)).astype(np.int32)
        self.conn = np.array([(1, 1, 2, 2, 2)] if connector else [], abi.connector)
        self.x = np.tile(0.5 * np.arange(n), len(ys))
        self.y = np.repeat(ys, n).astype(np.float64)
        self.dir = np.zeros(self.x.size)
        self.lane_width = np.full(self.x.size, 375, np.uint16)
        self.lanechg_attr = np.full(self.x.size, attr, np.uint16)
        self.lanechg_attr[lanes * n:] = 3

    def desc(self):
        from dmpp_b200 import abi
        d = abi.MapDesc()
        d.n_roads, d.road_lane_base, d.n_lanes, d.lane_pt_off = self.n_roads, self.road_lane_base.ctypes.data, self.n_lanes, self.lane_pt_off.ctypes.data
        d.n_conn, d.conn, d.n_points = len(self.conn), self.conn.ctypes.data, self.x.size
        d.x, d.y, d.dir = self.x.ctypes.data, self.y.ctypes.data, self.dir.ctypes.data
        d.lane_width, d.lanechg_attr = self.lane_width.ctypes.data, self.lanechg_attr.ctypes.data
        return d


def first_strikes(the_map, w, met):
    """worlds with a collision, and where their first colliding agent started: on the ego's lane behind it (and of those, how many
    faster than the ego), ahead of it, or on another lane"""
    m = the_map
    cump = cump_of(m)
    h, a = w.hdr, w.agents
    s = np.nonzero(met["first_collision_step"] > 0)[0]
    gl = m.road_lane_base[h["road_num"][s].astype(int) - 1] + h["lane_num"][s].astype(int) - 1
    se = cump[m.lane_pt_off[gl] + h["id"][s, h["lane_num"][s].astype(int) - 1]]
    ag = a[s, met["first_collision_agent"][s]]
    sk = cump[m.lane_pt_off[ag["lane"]] + ag["i"]] + ag["u"]
    same_lane = ag["lane"] == gl
    behind = same_lane & (sk < se)
    return {"worlds": int(s.size), "behind": int(behind.sum()), "behind_faster": int((behind & (ag["v"] > h["velocity"][s] / 3.6)).sum()),
            "ahead": int((same_lane & ~behind).sum()), "other_lane": int((~same_lane).sum())}


def check_rows(got, want, what, rec=None):
    """byte for byte; with rec (the GPU's own records [cycles][n]): max_abs_dir_err is max |rec.path_dir_err| of those records, bit for
    bit, and within 1e-9 of the checker's -- the one record field the CUDA path reproduces to 1e-9 only (tests/test_closed_loop.py)"""
    from dmpp_b200 import abi
    assert got.dtype == want.dtype == abi.episode_metrics
    for f in abi.episode_metrics.names:
        if rec is not None and f == "max_abs_dir_err":
            assert (got[f] == np.abs(rec["path_dir_err"]).max(axis=0)).all(), what
            assert (np.abs(got[f] - want[f]) <= 1e-9).all(), what
            continue
        g, w = got[f].reshape(len(got), -1), want[f].reshape(len(want), -1)
        bad = (g.view(np.uint8).reshape(len(got), -1) != w.view(np.uint8).reshape(len(want), -1)).any(axis=1)
        assert not bad.any(), "%s: field %s differs in %d worlds, first %d: got %r want %r" % (
            what, f, bad.sum(), np.argmax(bad), got[f][np.argmax(bad)], want[f][np.argmax(bad)])


def gpu_vs_checker(joracle, the_map, kind, n, cycles, env=None, n_obs=10, repeat=1, metrics=True, lane_change=None):
    """the reactive agents, and with lane_change = LaneChangeParams their lane changes, metrics armed or not: the closed loop on the
    GPU against the checker, byte for byte"""
    from dmpp_b200 import scenes
    w = scenes.World(the_map, np.arange(n), n_obs=n_obs, kind=kind)
    mp = mparams() if metrics else None
    am = (amparams(), w.v0)
    want = joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=jparams(joracle, kind), threads=16, metrics=mp, agent_model=am,
                                   lane_change=lane_change)
    p = planner_with(the_map, n, n_obs, scenes.World.PRE_JUNCTION_PTS[kind], env)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, cycles, repeat=repeat, metrics=mp, agent_model=am, lane_change=lane_change)
    finally:
        p.close()
    what = "%s %r" % (kind, env)
    assert got["graph"] == (env is None and n_obs < 32), what   # (from 32 agents up the cycle runs on the group kernel)
    if metrics:
        check_rows(got["metrics"], want["metrics"], what, rec=got["rec"])
    check_closed_loop(got, want, what)
    if lane_change is None:
        assert (got["agents"]["v"] != w.agents["v"]).any()
    else:
        assert got["lane_change_state"].tobytes() == want["lane_change_state"].tobytes(), what
        st = got["lane_change_state"]
        assert (st["changes_left"] + st["changes_right"]).sum() > 0
    return got
