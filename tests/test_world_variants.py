"""Parity of the closed-loop world step, its agent models and the V2X operator on the maps and planner parameters of
tests/map_variants.py: jittered points with zero-length segments, UTM-like and scaled coordinates, a 6-lane and a 1-lane road, a
tight circle, a zig-zag and a hairpin, non-default dp_params.

Two maps are built here on top of those: `jitter_ends` (the jitter map whose highway lanes end in a duplicated point, so that an
agent that runs to the end of its lane stands on a zero-length segment) and `attrs6` (the shapes map whose 6-lane road carries
lane-change attributes 0-3 in blocks, so that the inner lanes allow a change to the right only or to the left only).

Without a GPU: the numpy restatements of the react and lane-change phases (test_reactive_agents / test_lane_change) and a new one
of the agent motion and its obstacle point against the checker (tools/junction_oracle) on agents placed on and just before
zero-length segments, at lane ends, on the outer lanes of the 6-lane road and around the circle; the checker's closed loop with
every option is not vacuous on any variant; with junctions on, highway worlds give what the segment-only oracle gives.
With a GPU (-m gpu): the full option set of the closed loop against the checker byte for byte (graph, direct launches, the group
kernel, 40 agents), the disarmed loop against the oracle and its log replayed open loop, single steps with first > 0 on the
hand-placed agents, the V2X operator and the output frames against the oracle."""
import math
import os

import numpy as np
import pytest

import map_variants as mv
from test_lane_change import restate as lc_restate
from test_map_variants import bound
from test_reactive_agents import restate as react_restate
from test_v2x_traffic import tparams, vparams
from worlds import WORLD, amparams, check_closed_loop, check_rows, cump_of, joracle, jparams, lcparams, mparams  # noqa: F401

CYCLES = {"highway": 25, "junction": 120}
WORLDS = {"highway": 1024, "junction": 512}
HOPS = 8                                                    # WORLD_MAX_HOPS: successor lanes an agent may enter in one step


# ---------------------------------------------------------------- the maps
def zero_segments(m, gl):
    """indices i of lane gl whose segment (i, i + 1) has no length"""
    o, e = int(m.lane_pt_off[gl]), int(m.lane_pt_off[gl + 1])
    return np.nonzero((np.diff(m.x[o:e]) == 0) & (np.diff(m.y[o:e]) == 0))[0]


def jitter_ends_map():
    roads, conns = mv.lanes_of(mv.variant("jitter").map)
    for road in roads[:5]:
        for ln in road:
            ln[0][-1], ln[1][-1] = ln[0][-2], ln[1][-2]     # the last segment of the lane has no length
    return mv.VariantMap(roads, conns)


def attrs6_map():
    """the 6-lane road's lane-change attributes in 40-point blocks: lane 1 {2, 0}, lanes 2-5 {1, 2, 3, 0} (shifted by lane),
    lane 6 {1, 0}"""
    roads, conns = mv.lanes_of(mv.variant("shapes").map)
    for l, ln in enumerate(roads[0]):
        cyc = [2, 0] if l == 0 else [1, 0] if l == 5 else list(np.roll([1, 2, 3, 0], l))
        b = np.arange(ln[0].size) // 40
        ln[4] = np.asarray(cyc, np.uint16)[(b + l) % len(cyc)]
    return mv.VariantMap(roads, conns)


_local = {}


def variant(name):
    if name in ("jitter_ends", "attrs6"):
        if name not in _local:
            _local[name] = mv.Variant(name, jitter_ends_map() if name == "jitter_ends" else attrs6_map(),
                                      sweep_roads=(2, 4, 5) if name == "attrs6" else (2, 4))
        return _local[name]
    return mv.variant(name)


def road_of(m, lanes):
    return np.searchsorted(m.road_lane_base, lanes, side="right")


# ---------------------------------------------------------------- hand-placed agents
LC_ROADS = {"jitter": (1, 3, 5), "jitter_ends": (1, 3, 5), "scaled": (1, 3, 5), "utm": (1, 3, 5), "shapes": (1, 2, 3), "attrs6": (1, 1, 3)}


def placed(v, n, seed, k=10):
    """(hdr[n], agents[n][k], v0[n][k]) on the highway roads LC_ROADS[name], one road per world with the ego on it (pos 0):
    agents on a zero-length segment (u = 0 or not) and one segment before one, at lane ends, on every lane of the road, fast
    enough to cross several segments per step; in half of the worlds agent 0 is stuck behind a slow agent 1 abeam of a
    zero-length segment of a neighbouring lane (where there is one), so that its lane change lands on it"""
    from dmpp_b200 import abi, scenes
    m = v.map
    rng = np.random.default_rng(seed)
    h = scenes.World(m, np.arange(seed, seed + n), kind="highway").hdr.copy()
    road = rng.choice(LC_ROADS[v.name], n)
    base, nl = m.road_lane_base[road - 1], m.road_lane_base[road] - m.road_lane_base[road - 1]
    lane = base[:, None] + rng.integers(0, 6, (n, k)) % nl[:, None]
    cnt = m.lane_pt_off[lane + 1] - m.lane_pt_off[lane]
    centre = rng.integers(150, 1750, n)
    i = np.clip(centre[:, None] + rng.integers(-100, 100, (n, k)), 0, cnt - 2)
    u = np.where(rng.random((n, k)) < 0.2, 0.0, rng.uniform(0, 0.45, (n, k)))
    v_ = np.where(rng.random((n, k)) < 0.1, 60.0, rng.uniform(0, 25, (n, k)))
    v0 = rng.uniform(-2, 30, (n, k))
    v0[rng.random((n, k)) < 0.05] = np.nan
    zs = {gl: zero_segments(m, gl) for gl in np.unique(lane)}
    for s in range(n):
        for j in range(k):
            z, r = zs[lane[s, j]], rng.random()
            if z.size and r < 0.4:
                d = int(z[np.argmin(np.abs(z - i[s, j]))])
                i[s, j] = d if r < 0.25 else max(d - 1, 0)          # on it, or on the segment before it
                if r < 0.12:
                    u[s, j] = 0.0
            elif r < 0.5:
                i[s, j] = cnt[s, j] - 2                             # at the lane end
                u[s, j] = 0.0 if r < 0.45 else 0.2
        if rng.random() < 0.5 and nl[s] > 1:                        # agent 0 behind a slow agent 1, a neighbour lane's zero segment abeam
            q = int(rng.integers(0, nl[s]))
            for ml in rng.permutation([base[s] + q - 1, base[s] + q + 1]):
                if not base[s] <= ml < base[s] + nl[s]:
                    continue
                z = zs.get(ml, zero_segments(m, ml))
                z = z[(z > 200) & (z < 1700)]
                d = int(z[rng.integers(0, z.size)]) if z.size else int(rng.integers(200, 1700))
                lane[s, :2], i[s, 0], i[s, 1], u[s, :2] = base[s] + q, d, d + 24, (0.0, 0.1)
                v_[s, :2], v0[s, :2] = (12.0, 1.0), (20.0, 1.0)
                break
    ag = np.zeros((n, k), abi.agent)
    ag["lane"], ag["i"], ag["u"], ag["v"] = lane, i, u, v_
    ag["lat"] = np.where(rng.random((n, k)) < 0.2, rng.uniform(-3, 3, (n, k)), rng.uniform(-0.5, 0.5, (n, k)))
    ag["lat"][:, :2] = 0.0
    el = 1 + rng.integers(0, 6, n) % nl
    gl = base + el - 1
    o = m.lane_pt_off[gl] + centre
    h["road_num"], h["lane_num"], h["next_roadnum"], h["pos"], h["conn"] = road, el, road, 0, -1
    h["id"] = centre[:, None]
    h["x"], h["y"], h["dir"] = m.x[o], m.y[o], m.dir[o]
    h["velocity"] = rng.uniform(0, 60, n)
    h["n_obs"] = np.maximum(rng.integers(0, k + 1, n), 2)
    return h, ag, v0


def check_placed(v, h, ag):
    """the placement reaches what it is for: agents on zero-length segments (jitter maps), at lane ends, on every lane"""
    m = v.map
    used = np.arange(ag.shape[1])[None, :] < h["n_obs"][:, None]
    a = ag[used]
    o = m.lane_pt_off[a["lane"]] + a["i"]
    zero = (m.x[o + 1] == m.x[o]) & (m.y[o + 1] == m.y[o])
    end = a["i"] == m.lane_pt_off[a["lane"] + 1] - m.lane_pt_off[a["lane"]] - 2
    if v.name.startswith("jitter"):
        assert (zero & (a["u"] == 0)).sum() > 50 and (zero & (a["u"] > 0)).sum() > 50
    assert end.sum() > 50
    r = LC_ROADS[v.name][0]
    assert set(np.unique(a["lane"]).tolist()) >= set(range(m.road_lane_base[r - 1], m.road_lane_base[r]))


def step_inputs(h):
    """a record and a carried straight path along the ego's heading for one world step"""
    from dmpp_b200 import abi
    n = h.shape[0]
    rng = np.random.default_rng(n)
    rec = np.zeros(n, abi.plan_record)
    rec["brakespeed"] = rng.uniform(0, 20, n)
    rec["afresh_planning"], rec["behavior"] = 1, 1
    lp = np.zeros((n, 2, 200))
    hr = np.radians(h["dir"])
    lp[:, 0] = h["x"][:, None] + 0.5 * np.arange(200) * np.cos(hr)[:, None]
    lp[:, 1] = h["y"][:, None] + 0.5 * np.arange(200) * np.sin(hr)[:, None]
    return rec, lp


# ---------------------------------------------------------------- CPU: independent restatements on the variant lanes
@pytest.mark.parametrize("name", ["jitter", "shapes", "attrs6"])
def test_react_restatement_on_variant_lanes(joracle, the_map, name):
    """section 12's react phase (test_reactive_agents.restate) against jo_react_step, byte for byte: the hand-placed agents, and
    on the jitter map also random agents on the junction approaches and connectors with egos in pos 0 / 1 / 2"""
    v = variant(name)
    m = v.map
    h, ag, v0 = placed(v, 600, 11)
    check_placed(v, h, ag)
    sets = [(h, ag, v0, jparams(joracle, "highway"))]
    if name == "jitter":
        rng = np.random.default_rng(12)
        hj, aj, v0j = placed(v, 400, 12)
        lanes = np.concatenate([np.arange(m.road_lane_base[5], m.road_lane_base[7]), m.conn["lane"].astype(np.int64)])
        aj["lane"] = rng.choice(lanes, aj.shape)
        cnt = m.lane_pt_off[aj["lane"] + 1] - m.lane_pt_off[aj["lane"]]
        aj["i"] = np.where(rng.random(aj.shape) < 0.2, cnt - 2, rng.integers(0, 1 << 30, aj.shape) % (cnt - 1))
        hj["road_num"], hj["lane_num"], hj["next_roadnum"] = 6, rng.integers(1, 3, 400), 7
        hj["pos"], hj["conn"], hj["last_lanenum"] = rng.integers(0, 3, 400), rng.integers(-1, len(m.conn) + 1, 400), rng.integers(0, 3, 400)
        hj["id"] = rng.integers(-20, 420, (400, 6))
        sets.append((hj, aj, v0j, jparams(joracle, "junction")))
    p = amparams(look=150.0)
    with bound(joracle, the_map, v):
        cump, nxt = cump_of(m), joracle.lane_next()
        for hh, aa, vv, wp in sets:
            got = aa.copy()
            joracle.react_step(hh, got, vv, p, wp=wp)
            want = np.stack([react_restate(m, cump, nxt, wp, p, hh[s], aa[s], vv[s]) for s in range(len(hh))])
            assert got["v"].tobytes() == want.tobytes(), name
            assert (got["v"] != aa["v"]).mean() > 0.3


@pytest.mark.parametrize("name", ["jitter", "shapes", "attrs6"])
def test_lane_change_restatement_on_variant_lanes(joracle, the_map, name):
    """section 13's phase (test_lane_change.restate) against jo_lane_change_step, byte for byte, on the hand-placed agents; the
    changes reach both sides, the outer lanes of the 6-lane road and (jitter) target segments without length"""
    from dmpp_b200 import abi
    v = variant(name)
    m = v.map
    h, ag, v0 = placed(v, 1000, 21)
    rng = np.random.default_rng(22)
    st = np.zeros(ag.shape, abi.lane_change_state)
    st["lat_goal"] = np.where(rng.random(ag.shape) < 0.15, ag["lat"] + rng.uniform(-1, 1, ag.shape), ag["lat"])
    st["hold"] = np.where(rng.random(ag.shape) < 0.15, rng.uniform(0, 0.3, ag.shape), rng.uniform(-3, 0, ag.shape))
    p, c = amparams(look=150.0), lcparams(politeness=0.3, a_thr=0.1, end_guard=20.0)
    with bound(joracle, the_map, v):
        assert (joracle.lane_next()[:m.road_lane_base[5]] < 0).all()   # the restatement's react phase has no successors to follow
        got, gst = ag.copy(), st.copy()
        joracle.lane_change_step(h, got, v0, p, c, gst, wp=jparams(joracle, "highway"))
    cump = cump_of(m)
    want = [lc_restate(m, cump, p, c, h[s], ag[s], v0[s], st[s]) for s in range(len(h))]
    assert got.tobytes() == np.stack([a for a, _ in want]).tobytes(), name
    assert gst.tobytes() == np.stack([s for _, s in want]).tobytes(), name
    moved = got["lane"] != ag["lane"]
    assert (got["lane"] < ag["lane"]).sum() > 20 and (got["lane"] > ag["lane"]).sum() > 20, name
    o = m.lane_pt_off[got["lane"]] + got["i"]
    onto_zero = moved & (m.x[o + 1] == m.x[o]) & (m.y[o + 1] == m.y[o])
    if name == "jitter":
        assert onto_zero.sum() > 20
    if name != "jitter":
        lanes6 = got["lane"][moved & (road_of(m, got["lane"]) == 1)] - m.road_lane_base[0]
        assert {0, 5} <= set(lanes6.tolist()) and (road_of(m, got["lane"][moved]) == 3).any()


def motion(m, nxt, junc, dt, a):
    """the agent's advance over one step and its obstacle point (include/dmpp_b200.h section 9, oracle/world_spec.cpp and
    tools/junction_oracle/world_junction.cpp) in plain Python float64: over the segments of its lane, clamped to the lane's last
    segment, and with junctions on into the lane's successor (at most HOPS of them)"""
    off, size = m.lane_pt_off, lambda gl: int(m.lane_pt_off[gl + 1] - m.lane_pt_off[gl])

    def seg(gl, i):
        o = int(off[gl]) + i
        dx, dy = float(m.x[o + 1]) - float(m.x[o]), float(m.y[o + 1]) - float(m.y[o])
        return math.sqrt(dx * dx + dy * dy), dx, dy
    lane, i, u = int(a["lane"]), int(a["i"]), float(a["u"]) + float(a["v"]) * dt
    hop = 0
    while True:
        cnt = size(lane)
        while i < cnt - 2 and not u < seg(lane, i)[0]:
            u -= seg(lane, i)[0]
            i += 1
        if i < cnt - 2:
            break
        i = cnt - 2
        L = seg(lane, i)[0]
        nx = int(nxt[lane]) if junc and hop < HOPS else -1
        if u < L or nx < 0:
            if u > L:
                u = L
            break
        u -= L
        lane, i, hop = nx, 0, hop + 1
    L, dx, dy = seg(lane, i)
    qx, qy = float(m.x[off[lane] + i]), float(m.y[off[lane] + i])
    if L > 0:
        t = u / L
        px, py = qx + t * dx, qy + t * dy
        qx, qy = px + float(a["lat"]) * (-(dy / L)), py + float(a["lat"]) * (dx / L)
    return lane, i, u, qx, qy, hop


@pytest.mark.parametrize("name", ["jitter", "jitter_ends", "scaled", "utm", "shapes"])
def test_motion_restatement_equals_checker(joracle, the_map, name):
    """jo_world_step's agents and obstacle points against `motion`, byte for byte, junctions off and on: the hand-placed agents,
    and agents on the junction approaches and connectors fast enough to hop over several lanes"""
    v = variant(name)
    m = v.map
    h, ag, _ = placed(v, 500, 31)
    rng = np.random.default_rng(32)
    lanes = np.concatenate([np.arange(m.road_lane_base[5], m.road_lane_base[7]), m.conn["lane"].astype(np.int64)])
    hop = rng.random(len(h)) < 0.4
    ag["lane"][hop] = rng.choice(lanes, (hop.sum(), ag.shape[1]))
    cnt = m.lane_pt_off[ag["lane"] + 1] - m.lane_pt_off[ag["lane"]]
    ag["i"][hop] = np.clip(cnt[hop] - 2 - rng.integers(0, 30, cnt[hop].shape), 0, None)
    ag["v"][hop] = np.where(rng.random(cnt[hop].shape) < 0.3, rng.uniform(100, 400, cnt[hop].shape), ag["v"][hop])
    rec, lp = step_inputs(h)
    hops = 0
    with bound(joracle, the_map, v):
        nxt = joracle.lane_next()
        for wp in (jparams(joracle, "highway"), jparams(joracle, "junction")):
            hh, got = h.copy(), ag.copy()
            ox, oy = np.zeros(ag.shape), np.zeros(ag.shape)
            joracle.world_step(hh, got, ox, oy, rec=rec, last_path=lp, wp=wp)
            for s in range(len(h)):
                dt = float(h["period_ms"][s]) / 1000.0
                for k in range(min(int(h["n_obs"][s]), ag.shape[1])):
                    lane, i, u, x, y, nh = motion(m, nxt, wp.pre_junction_pts > 0, dt, ag[s, k])
                    g = got[s, k]
                    assert (int(g["lane"]), int(g["i"])) == (lane, i) and g["u"].tobytes() == np.float64(u).tobytes(), (name, s, k)
                    assert ox[s, k].tobytes() == np.float64(x).tobytes() and oy[s, k].tobytes() == np.float64(y).tobytes(), (name, s, k)
                    hops += nh
                assert got[s, int(h["n_obs"][s]):].tobytes() == ag[s, int(h["n_obs"][s]):].tobytes()
    assert hops > 100


# ---------------------------------------------------------------- CPU: the checker's closed loop with every option
_runs = {}


def full(w, ev):
    return dict(metrics=mparams(), agent_model=(amparams(), w.v0), lane_change=lcparams(), v2x=(vparams(), ev), traffic=tparams())


def checker_run(joracle, the_map, name, kind, n_obs=10):
    """(world, events, the checker's closed loop) with metrics, reactive and lane-changing agents, V2X events and agents obeying
    them: WORLDS[kind] worlds of 10 agents, or 512 highway worlds of n_obs agents"""
    from dmpp_b200 import scenes
    key = (name, kind, n_obs)
    if key not in _runs:
        v = variant(name)
        n = WORLDS[kind] if n_obs == 10 else 512
        w = scenes.World(v.map, np.arange(n), n_obs=n_obs, kind=kind)
        ev = scenes.V2xEvents(w, np.arange(n))
        with bound(joracle, the_map, v):
            out = joracle.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(joracle, kind), threads=16, **full(w, ev))
        _runs[key] = (w, ev, out)
    return _runs[key]


def crossed_zero_segments(m, a0, a1):
    """agents that stayed on their lane and passed over at least one zero-length segment"""
    z = np.r_[(np.diff(m.x) == 0) & (np.diff(m.y) == 0), False]
    c = np.r_[0, np.cumsum(z)]
    g0, g1 = m.lane_pt_off[a0["lane"]] + a0["i"], m.lane_pt_off[a1["lane"]] + a1["i"]
    return int((((c[g1] - c[g0]) > 0) & (a0["lane"] == a1["lane"])).sum())


@pytest.mark.parametrize("name", mv.VARIANTS)
def test_closed_loop_is_not_vacuous(joracle, the_map, name):
    """the full option set reaches, on every variant: agents led by the signal line and by the pedestrian, junction positions 0, 1
    and 2, every value of every V2X flag, lane changes; jitter: agents crossing zero-length segments; shapes: changes to both sides
    on the 6-lane road, none from the 1-lane road, the ego's ids continuous around the circle"""
    v = variant(name)
    m = v.map
    runs = {kind: checker_run(joracle, the_map, name, kind) for kind in CYCLES}
    for kind, (w, _, o) in runs.items():
        assert not np.isnan(o["agents"]["u"]).any() and not np.isnan(o["hdr"]["x"]).any(), kind
    tr = np.concatenate([o["v2x_traffic"] for _, _, o in runs.values()])
    vs = np.concatenate([o["v2x_stats"] for _, _, o in runs.values()])
    assert tr["line_steps"].sum() > 1000 and tr["ped_steps"].sum() > 100, name
    # (on the x2 map the junction ego leaves pos 0 -- the handlers' only caller -- 60 m before the stop line, where the signal's
    # range of 25-60 m begins: the light flag stays 0 there, and test_v2x_operator_is_not_vacuous covers its values)
    assert (vs["light_cycles"].sum(axis=0) > 0).all() or (name == "scaled" and vs["light_cycles"][:, 0].sum() > 0), name
    assert (vs["pedestrian_cycles"].sum(axis=0) > 0).all(), name
    assert (vs["construction_cycles"].sum(axis=0) > 0).all(), name
    assert set(np.unique(runs["junction"][2]["hdr_log"]["pos"]).tolist()) == {0, 1, 2}, name
    w, _, o = runs["highway"]
    st = o["lane_change_state"]
    assert st["changes_left"].sum() > 50 and st["changes_right"].sum() > 50, name
    if name == "jitter":
        assert crossed_zero_segments(m, w.agents, o["agents"]) > 100
    if name == "shapes":
        road = road_of(m, o["agents"]["lane"])
        ch_l, ch_r = st["changes_left"], st["changes_right"]
        assert ch_l[road == 1].sum() > 20 and ch_r[road == 1].sum() > 20
        assert (ch_l[road == 2] + ch_r[road == 2]).sum() == 0 and (road == 2).sum() > 100
        assert set(np.unique(o["agents"]["lane"][road == 1]).tolist()) == set(range(m.road_lane_base[0], m.road_lane_base[1]))
        H, wp = o["hdr_log"], joracle.world_params()
        on = (H["road_num"][:-1] == 3) & (H["road_num"][1:] == 3)
        assert on.sum() > 500
        d = np.abs(H["id"][1:].astype(np.int64) - H["id"][:-1])[..., :3]
        assert (d[on] <= wp.loc_fwd).all()


@pytest.mark.parametrize("name", mv.VARIANTS)
def test_junction_option_on_highway_is_segment_loop(oracle, joracle, the_map, name):
    """junctions on or off, highway worlds (no connector anywhere) give what the segment-only loop of oracle/ gives, byte for byte"""
    from dmpp_b200 import scenes
    v = variant(name)
    w = scenes.World(v.map, np.arange(256))
    with bound(oracle, the_map, v), bound(joracle, the_map, v):
        off = oracle.run_closed_loop(w.hdr, w.agents, 60, threads=8)
        for J in (0, 60, 400):
            wp = joracle.world_params()
            wp.pre_junction_pts = J
            on = joracle.run_closed_loop(w.hdr, w.agents, 60, wp=wp, threads=8)
            for k in WORLD + ("obs_log_x", "obs_log_y"):
                assert on[k].tobytes() == off[k].tobytes(), (name, J, k)


# ---------------------------------------------------------------- CPU: the V2X operator's inputs
def v2x_inputs(v):
    """4096 highway headers with scenes.v2x_events, plus road-works scenes placed by hand in mode 1's reach: the ego on every lane
    of the multi-lane highway roads, the event point ahead of it, 1.9 m towards the left or right neighbour lane (nearer that
    lane than its own)"""
    from dmpp_b200 import abi, scenes
    m = v.map
    h = scenes.Episodes(m, np.arange(4096), cycles=1).hdr(0)
    vv, wl, wg = scenes.v2x_events(m, h, seed=1)
    p = mv.default_params()                                 # (scenes.v2x_events' datum: the default parameters)
    hs, xs = [], []
    for r in range(1, 6):
        b, nl = int(m.road_lane_base[r - 1]), int(m.road_lane_base[r] - m.road_lane_base[r - 1])
        for l in range(nl):
            for side in (-1, 1):
                if not 0 <= l + side < nl:
                    continue
                for idx in range(100, 1700, 37):
                    o, on = int(m.lane_pt_off[b + l]) + idx, int(m.lane_pt_off[b + l + side]) + idx
                    e = o + 16 + int(p.id_more)
                    en = on + 16 + int(p.id_more)
                    f = 1.9 / math.hypot(m.x[en] - m.x[e], m.y[en] - m.y[e])
                    wx, wy = m.x[e] + f * (m.x[en] - m.x[e]), m.y[e] + f * (m.y[en] - m.y[e])
                    hh = np.zeros(1, abi.scene_hdr)
                    hh["road_num"], hh["lane_num"], hh["id"], hh["x"], hh["y"] = r, l + 1, idx, m.x[o], m.y[o]
                    d = np.zeros(1, abi.v2x_data)
                    d["warn_status"] = 4
                    d["rsi_lat"], d["rsi_lng"] = p.lat0 + wy * p.k_lat, p.lng0 + wx * p.k_lng
                    d["ego_lat"], d["ego_lng"] = p.lat0 + m.y[o] * p.k_lat, p.lng0 + m.x[o] * p.k_lng
                    hs.append(hh); xs.append(d)
    return np.concatenate([h] + hs), np.concatenate([vv] + xs), wl, wg, h.size


V2X_NAMES = mv.VARIANTS + ["attrs6"]


@pytest.mark.parametrize("name", V2X_NAMES)
def test_v2x_operator_is_not_vacuous(oracle, the_map, name):
    """the oracle on the operator's inputs: every outcome of every handler in mode 0; in mode 1 the event points by the
    neighbour lanes raise the road-works flag on some scenes and not on others"""
    v = variant(name)
    h, vv, wl, wg, n0 = v2x_inputs(v)
    with bound(oracle, the_map, v):
        a, b = oracle.v2x_event(h, vv, wl, wg, 0), oracle.v2x_event(h, vv, wl, wg, 1)
    ok, st = a["ub"][:n0] == 0, vv["warn_status"][:n0]
    assert ok.mean() > 0.9
    assert set(np.unique(a["light_flag"][:n0][ok & (st == 3)]).tolist()) == {0, 1, 2}, name
    for s, f in ((4, "construction_flag"), (5, "pedestrian_flag")):
        hit = a[f][:n0][ok & (st == s)]
        assert 20 < hit.sum() < hit.size - 20, (name, s, f)
    crafted = b["construction_flag"][n0:]
    # (on the x2 map the lanes are 7.5 m apart: no event point is within the handler's 2 m of two lanes, every one flags)
    assert 20 < crafted.sum() and (crafted.sum() < crafted.size - 20 or name == "scaled"), name
    assert (b["construction_flag"][:n0] != a["construction_flag"][:n0]).any(), name


# ---------------------------------------------------------------- GPU
def planner_for(v, n, max_obs, J=None, env=None):
    from dmpp_b200.planner import Planner
    env = env or {}
    os.environ.update(env)
    try:
        p = Planner(max_scenes=n, max_obs=max_obs, params=v.params)
    finally:
        for k in env:
            del os.environ[k]
    p.upload_map(v.map)
    if J is not None:
        wp = p.world_params()
        wp.pre_junction_pts = J
        p.set_world_params(wp)
    return p


def gpu_vs_checker(joracle, the_map, name, kind, env=None, n_obs=10):
    """the full option set on the GPU against the checker: records, logs, final world, carry, metrics rows, lane-change states,
    V2X rows, flags and the agents' V2X rows"""
    from dmpp_b200 import scenes
    v = variant(name)
    w, ev, want = checker_run(joracle, the_map, name, kind, n_obs)
    p = planner_for(v, w.n, n_obs, scenes.World.PRE_JUNCTION_PTS[kind], env)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], **full(w, ev))
    finally:
        p.close()
    what = "%s %s %r %d agents" % (name, kind, env, n_obs)
    assert got["graph"] == (env is None and n_obs < 32), what   # (from 32 agents up the cycle runs on the group kernel)
    check_closed_loop(got, want, what)
    for k in ("lane_change_state", "v2x_stats", "v2x_flags", "v2x_traffic"):
        assert got[k].tobytes() == want[k].tobytes(), (what, k)
    check_rows(got["metrics"], want["metrics"], what, rec=got["rec"])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
@pytest.mark.parametrize("name", mv.VARIANTS)
def test_gpu_full_options_equal_checker(joracle, the_map, name, kind):
    """one graph launch: metrics, reactive and lane-changing agents, V2X events, agents obeying them"""
    gpu_vs_checker(joracle, the_map, name, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
@pytest.mark.parametrize("kind", list(CYCLES))
@pytest.mark.parametrize("name", ["jitter", "shapes", "utm"])
def test_gpu_direct_launches_and_group_kernel(joracle, the_map, name, kind, env):
    gpu_vs_checker(joracle, the_map, name, kind, env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["jitter", "shapes"])
def test_gpu_40_agents(joracle, the_map, name):
    """40 agents per world: the cycle runs on the group kernel by size, the world step's agent loops take two passes"""
    gpu_vs_checker(joracle, the_map, name, "highway", n_obs=40)


@pytest.mark.gpu
@pytest.mark.parametrize("name", mv.VARIANTS)
def test_gpu_disarmed_loop_equals_oracle_and_replays(oracle, joracle, the_map, name):
    """no model armed: highway worlds against the segment-only oracle, junction worlds against the checker; the logged inputs,
    replayed open loop, give the same records"""
    from dmpp_b200 import scenes
    v = variant(name)
    for kind in CYCLES:
        n = WORLDS[kind]
        w = scenes.World(v.map, np.arange(30_000, 30_000 + n), kind=kind)
        runner = oracle if kind == "highway" else joracle
        with bound(runner, the_map, v):
            kw = {} if kind == "highway" else dict(wp=jparams(joracle, kind))
            want = runner.run_closed_loop(w.hdr, w.agents, CYCLES[kind], threads=16, **kw)
        p = planner_for(v, n, 10, scenes.World.PRE_JUNCTION_PTS[kind])
        try:
            got = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind])
            rep = p.run_episodes(got["hdr_log"], got["obs_log_x"], got["obs_log_y"], trace=False, paths=False)
        finally:
            p.close()
        what = "%s %s disarmed" % (name, kind)
        assert got["graph"], what
        check_closed_loop(got, want, what)
        assert rep["rec"].tobytes() == got["rec"].tobytes(), what + " replay"


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def host(t, dtype, shape=None):
    a = np.frombuffer(t.cpu().numpy().tobytes(), dtype)
    return a if shape is None else a.reshape(shape)


def pedestrians(v, h, ag, seed):
    """a pedestrian standing in every world from t = 0, in the lane of agent 2 (2-8 m ahead of it, within 1.5 m of its lane) or,
    in a third of the worlds, at the end of agent 3's lane; a red signal on the ego's road in half of the worlds"""
    import types
    from dmpp_b200 import abi
    m = v.map
    n = h.shape[0]
    rng = np.random.default_rng(seed)
    s = np.zeros(n, abi.v2x_event_spec)
    s["has_ped"], s["ped_t_on"], s["ped_t_off"] = 1, 0.0, 1e9
    for w in range(n):
        k = 3 if rng.random() < 0.35 else 2
        gl = int(ag["lane"][w, k])
        o = int(m.lane_pt_off[gl])
        last = int(m.lane_pt_off[gl + 1]) - o - 1
        i = last if k == 3 else min(int(ag["i"][w, k]) + int(rng.integers(4, 16)), last)
        hd = math.radians(float(m.dir[o + i]))
        lat = float(rng.uniform(-1.5, 1.5))
        s["ped_x"][w], s["ped_y"][w] = m.x[o + i] - lat * math.sin(hd), m.y[o + i] + lat * math.cos(hd)
    red = rng.random(n) < 0.5
    s["sig_road"] = np.where(red, h["road_num"], 0)
    s["sig_stop"] = rng.integers(-1, 2000, n)
    s["sig_green"], s["sig_yellow"], s["sig_red"] = 1.0, 1.0, 100.0
    s["sig_cycle"], s["sig_offset"] = 102.0, 2.0
    return types.SimpleNamespace(spec=s, wp_x=np.zeros(0), wp_y=np.zeros(0))


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["react", "lanechg", "traffic"])
@pytest.mark.parametrize("name", ["jitter", "jitter_ends", "shapes"])
def test_gpu_single_steps_hand_placed(joracle, the_map, name, model):
    """dp_world_step_dev with first > 0 on the hand-placed agents (on and before zero-length segments, at lane ends, behind a slow
    leader abeam of a neighbour's zero-length segment, on the 6-lane road's outer lanes and the circle), 8 steps against
    jo_react_step / jo_lane_change_step + jo_world_step, or (traffic) jo_traffic_step with lane changes and a pedestrian standing
    by agents on zero-length segments: header, agents, obstacle points, lane-change states and V2X rows byte for byte"""
    import torch
    from dmpp_b200 import abi
    v = variant(name)
    n, first, k, steps = 700, 37, 10, 8
    h0, a0, v0 = placed(v, n, 41)
    check_placed(v, h0, a0)
    rec, lp = step_inputs(h0)
    am, lc = amparams(), lcparams(cooldown=0.15, lat_speed=10.0)
    ev = pedestrians(v, h0, a0, 42)
    tp = tparams(ped_half_width=1.5)
    st = np.zeros((n, k), abi.lane_change_state)
    ts = np.zeros(n, abi.v2x_traffic_stats)
    zero_hits = 0
    with bound(joracle, the_map, v):
        wp = jparams(joracle, "highway")
        h, ag, ox, oy = h0.copy(), a0.copy(), np.zeros((n, k)), np.zeros((n, k))
        if model == "traffic":
            joracle.traffic_step(tp, ev, 0, h, ag, ox, oy, v0, am, ts, lp=lc, lcs=st, wp=wp)
        else:
            joracle.world_step(h, ag, ox, oy, wp=wp)
            used = np.arange(k)[None, :] < h0["n_obs"][:, None]
            st[used] = 0
            st["lat_goal"][used] = a0["lat"][used]
        for c in range(steps):
            if model == "traffic":
                joracle.traffic_step(tp, ev, c, h, ag, ox, oy, v0, am, ts, rec=rec, last_path=lp, lp=lc, lcs=st, wp=wp)
                u_ = np.arange(k)[None, :] < h["n_obs"][:, None]
                o = v.map.lane_pt_off[ag["lane"]] + ag["i"]
                zero_hits += int((u_ & (v.map.x[o + 1] == v.map.x[o]) & (v.map.y[o + 1] == v.map.y[o])).sum())
            elif model == "lanechg":
                joracle.lane_change_step(h, ag, v0, am, lc, st, wp=wp)
                joracle.world_step(h, ag, ox, oy, rec=rec, last_path=lp, wp=wp)
            else:
                joracle.react_step(h, ag, v0, am, wp=wp)
                joracle.world_step(h, ag, ox, oy, rec=rec, last_path=lp, wp=wp)
    p = planner_for(v, first + n, k, 0)
    try:
        p.upload_carry(first, np.zeros(n, abi.carry), lp)
        d_h, d_a, d_v0, d_r = dev(h0), dev(a0), dev(v0), dev(rec)
        d_x, d_y = torch.zeros(n * k, dtype=torch.float64, device="cuda"), torch.zeros(n * k, dtype=torch.float64, device="cuda")
        d_st = dev(np.zeros((n, k), abi.lane_change_state))
        d_spec = dev(ev.spec)
        d_vs, d_ts = torch.zeros(n * 80, dtype=torch.uint8, device="cuda"), torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
        p.set_agent_model(am, d_v0.data_ptr())
        if model != "react":
            p.set_lane_change(lc, d_st.data_ptr())
        if model == "traffic":
            p.set_v2x_world(vparams(apply=0), n, d_spec.data_ptr(), None, None, 0, None, d_vs.data_ptr())
            p.set_v2x_traffic(tp, d_ts.data_ptr())
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None, first=first)
        for c in range(steps):
            if model == "traffic":
                p.v2x_world_dev(n, d_h.data_ptr(), None, c)     # the cycle the V2X events of this step belong to
            p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), first=first)
        torch.cuda.synchronize()
        p.set_v2x_traffic(None, None); p.set_v2x_world(None, 0, None); p.set_lane_change(None, None); p.set_agent_model(None, None)
    finally:
        p.close()
    what = "%s %s" % (name, model)
    used = np.arange(k)[None, :] < h0["n_obs"][:, None]
    assert host(d_h, abi.scene_hdr).tobytes() == h.tobytes(), what
    got = host(d_a, abi.agent, (n, k))
    assert got[used].tobytes() == ag[used].tobytes(), what
    assert got[~used].tobytes() == a0[~used].tobytes(), what
    gx, gy = host(d_x, np.float64, (n, k)), host(d_y, np.float64, (n, k))
    assert gx[used].tobytes() == ox[used].tobytes() and gy[used].tobytes() == oy[used].tobytes(), what
    assert (got["v"][used] != a0["v"][used]).mean() > 0.3, what
    if model != "react":
        assert host(d_st, abi.lane_change_state, (n, k))[used].tobytes() == st[used].tobytes(), what
        assert (got["lane"][used] != a0["lane"][used]).sum() > 20, what
    if model == "traffic":
        assert host(d_ts, abi.v2x_traffic_stats).tobytes() == ts.tobytes(), what
        assert ts["ped_steps"].sum() > 50 and ts["line_steps"].sum() > 50, what
        if name == "jitter_ends":
            assert zero_hits > 50, what                         # agents standing on zero-length lane ends with the pedestrian on


@pytest.mark.gpu
@pytest.mark.parametrize("name", V2X_NAMES)
def test_gpu_v2x_operator_equals_oracle(oracle, the_map, name):
    """dp_v2x_event_batch in modes 0 and 1 and dp_v2x_apply against the oracle, every byte"""
    from dmpp_b200 import scenes
    v = variant(name)
    h, vv, wl, wg, n0 = v2x_inputs(v)
    p = planner_for(v, 256, 10)
    try:
        with bound(oracle, the_map, v):
            for mode in (0, 1):
                want = oracle.v2x_event(h, vv, wl, wg, mode)
                got = p.v2x_event(h, vv, wl, wg, mode)
                assert got.tobytes() == want.tobytes(), (name, mode)
            ep = scenes.Episodes(v.map, np.arange(256), cycles=1)
            p.reset(0, 256)
            rec = p.cycle(np.ascontiguousarray(ep.hdr(0)), *ep.obstacles(0))["rec"]
            flags = want[:256]
            got = p.v2x_apply(flags, rec)
            assert got.tobytes() == oracle.v2x_apply(flags, rec).tobytes(), name
            assert (got.tobytes() != rec.tobytes())
    finally:
        p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["utm", "scaled"])
@pytest.mark.parametrize("kind,n,cycles", [("highway", 256, 25), ("junction", 64, 60)])
def test_gpu_frames_equal_oracle(oracle, the_map, name, kind, n, cycles):
    """dp_pack_frames (the GPS conversion of the path points included) against the oracle's frames, cycle by cycle"""
    from dmpp_b200 import scenes
    v = variant(name)
    ep = scenes.Episodes(v.map, np.arange(n), cycles=cycles, kind=kind)
    H, OX, OY = ep.all_cycles()
    with bound(oracle, the_map, v):
        want = oracle.run(H, OX, OY, exhaustive=False, threads=8)
        p = planner_for(v, n, OX.shape[2])
        try:
            p.reset(0, n)
            for c in range(cycles):
                o = p.cycle(np.ascontiguousarray(H[c]), np.ascontiguousarray(OX[c]), np.ascontiguousarray(OY[c]))
                ctrl, status = p.pack_frames(o["rec"])
                wc, ws = oracle.pack_frames(want["rec"][c], want["path_xy"][c])
                assert ctrl.tobytes() == wc.tobytes(), (name, kind, c)
                assert status.tobytes() == ws.tobytes(), (name, kind, c)
        finally:
            p.close()
