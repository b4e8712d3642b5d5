"""Lane-changing agents in closed-loop episodes (include/dmpp_b200.h section 13): on top of the reactive agents, an agent may move to
a neighbouring lane of its road where the map allows it, by MOBIL with the IDM accelerations of section 12.

The specification is tools/junction_oracle/lane_change.cpp.  CPU side: layout and defaults, known answers on a straight two-lane
road, identities (junction worlds, an unreachable threshold, opted-out agents), an independent numpy restatement of the phase,
invariants over 512 highway episodes and the effect (changes, cut-ins, collisions).  GPU side: the LANECHG instances of the world
step against the checker, byte for byte, lane-change states included."""
import ctypes as C

import numpy as np
import pytest

from worlds import (DT, WORLD, W, StraightRoad, amparams, cump_of, first_strikes, gpu_vs_checker, idm, joracle,  # noqa: F401
                    jparams, jworld, lcparams, mparams, planner_with)


# ---------------------------------------------------------------- CPU: layout and defaults
def test_layout_and_defaults(joracle):
    from dmpp_b200 import abi
    assert joracle.lane_change_sizeof() == (64, 24)
    assert C.sizeof(abi.LaneChangeParams) == 64 and abi.lane_change_state.itemsize == 24
    p = lcparams()                                          # through dp_lane_change_default_params: no GPU needed
    assert (p.politeness, p.a_thr, p.b_safe, p.ego_b_safe, p.ego_front, p.lat_speed, p.cooldown, p.end_guard) == \
        (0.2, 0.2, 4.0, 4.0, 4.0, 1.0, 5.0, 30.0)


# ---------------------------------------------------------------- CPU: known answers on a straight two-lane road
@pytest.fixture
def two_lane(joracle, the_map):
    def use(attr=3, connector=False):
        joracle.set_map(StraightRoad(6000, lanes=2, attr=attr, connector=connector))
        return joracle
    yield use
    joracle.set_map(the_map)


def scene2(ego, agents, v_kmh=0.0):
    """one world: the ego at (x, lane) heading +x; agents as (x, lane, v, lat); lanes are 0 / 1 (global) on the two-lane map"""
    from dmpp_b200 import abi
    ex, el = ego
    h = np.zeros(1, abi.scene_hdr)
    h["x"], h["y"], h["velocity"], h["period_ms"] = ex, W / 2 - W * el, v_kmh, 1000 * DT
    h["road_num"], h["lane_num"], h["next_roadnum"], h["conn"] = 1, el + 1, 1, -1
    h["id"][:, :2] = int(round(ex / 0.5))
    h["n_obs"] = len(agents)
    ag = np.zeros((1, len(agents)), abi.agent)
    for k, (x, lane, v, lat) in enumerate(agents):
        ag["i"][0, k] = int(x // 0.5)
        ag["u"][0, k] = x - 0.5 * int(x // 0.5)
        ag["lane"][0, k], ag["v"][0, k], ag["lat"][0, k] = lane, v, lat
    st = np.zeros((1, len(agents)), abi.lane_change_state)
    st["lat_goal"] = ag["lat"]
    return h, ag, st


SLOW = [(100.0, 1, 10.0, 0.25), (115.0, 1, 3.0, 0.0)]    # agent 0 on lane 2 behind a slow agent 1; lane 1 empty
SLOW_V0 = [15.0, 3.0]
FAR_EGO = (2500.0, 1)


def lc(o, h, ag, st, v0, am=None, lp=None):
    o.lane_change_step(h, ag, np.array([v0], np.float64), am or amparams(), lp or lcparams(), st)


def test_changes_left_past_a_slow_leader(two_lane):
    o, am = two_lane(), amparams()
    h, ag, st = scene2(FAR_EGO, SLOW)
    old = ag.copy()
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 0 and ag["i"][0, 0] == old["i"][0, 0] and ag["u"][0, 0] == old["u"][0, 0]
    assert ag["lat"][0, 0] == 0.25 - W
    assert ag["v"][0, 0] == idm(10.0, 15.0, am)             # free road on lane 1: at_c, not the braking of its own lane
    assert st["hold"][0, 0] == 5.0 and st["changes_left"][0, 0] == 1 and st["changes_right"][0, 0] == 0
    assert ag["lane"][0, 1] == 1 and st["changes_left"][0, 1] == 0   # the slow leader has no reason to move
    # back to lat_goal at lat_speed, snapping onto it; the speed follows the IDM on the new lane
    err = [abs(ag["lat"][0, 0] - 0.25)]
    for _ in range(40):
        v = ag["v"][0, 0]
        lc(o, h, ag, st, SLOW_V0)
        err.append(abs(ag["lat"][0, 0] - 0.25))
        assert ag["lane"][0, 0] == 0 and ag["v"][0, 0] == idm(v, 15.0, am)
    assert err[-1] == 0.0 and ag["lat"][0, 0] == 0.25
    steps = [e for e in err if e > 0]
    assert len(steps) == 38 and all(abs((a - b) - 0.1) < 1e-12 for a, b in zip(steps, steps[1:]))
    assert abs(st["hold"][0, 0] - (5.0 - 40 * DT)) < 1e-12 and st["changes_left"][0, 0] == 1


def test_close_follower_blocks_by_b_safe(two_lane):
    o = two_lane()
    agents = SLOW + [(90.0, 0, 15.0, 0.0)]                  # 10 m behind the abeam station on lane 1, closing at 5 m/s
    for b_safe, moves in ((4.0, False), (9.0, True)):
        h, ag, st = scene2(FAR_EGO, agents)
        lc(o, h, ag, st, SLOW_V0 + [15.0], lp=lcparams(b_safe=b_safe))
        assert (ag["lane"][0, 0] == 0) == moves, b_safe


def test_overlap_refuses_the_gap(two_lane):
    o = two_lane()
    h, ag, st = scene2(FAR_EGO, SLOW + [(100.0, 0, 10.0, 0.0)])   # abeam, the same station
    lc(o, h, ag, st, SLOW_V0 + [10.0], lp=lcparams(b_safe=100.0))
    assert ag["lane"][0, 0] == 1 and st["changes_left"][0, 0] == 0


def test_attribute_2_forbids_left(two_lane):
    o = two_lane(attr=2)
    h, ag, st = scene2(FAR_EGO, SLOW)
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 1
    o = two_lane(attr=1)                                    # ... and 1 allows it
    h, ag, st = scene2(FAR_EGO, SLOW)
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 0


def test_guards_cooldown_connectors_opt_out(two_lane):
    o = two_lane()
    n_end = 0.5 * 5999
    h, ag, st = scene2(FAR_EGO, [(n_end - 29.0, 1, 10.0, 0.0), (n_end - 25.0, 1, 3.0, 0.0)])   # within end_guard of the lane end
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 1
    h, ag, st = scene2(FAR_EGO, [(n_end - 29.0, 1, 10.0, 0.0), (n_end - 25.0, 1, 3.0, 0.0)])
    lc(o, h, ag, st, SLOW_V0, lp=lcparams(end_guard=20.0))
    assert ag["lane"][0, 0] == 0
    h, ag, st = scene2(FAR_EGO, SLOW)                       # cooldown: hold > 0 waits, hold <= 0 goes
    st["hold"][0, 0] = 0.15
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 1 and abs(st["hold"][0, 0] - 0.05) < 1e-15
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 1                            # 0.05 > 0
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 0
    h, ag, st = scene2(FAR_EGO, SLOW)                       # mid-manoeuvre (lat != lat_goal): no new change
    st["lat_goal"][0, 0] = 0.0
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 1 and ag["lat"][0, 0] == 0.15
    h, ag, st = scene2(FAR_EGO, SLOW)                       # opted out: keeps lane and speed
    lc(o, h, ag, st, [0.0, 3.0])
    assert ag["lane"][0, 0] == 1 and ag["v"][0, 0] == 10.0
    o = two_lane(connector=True)                            # on a connector (attribute 3, lanes on both sides): never
    h, ag, st = scene2(FAR_EGO, [(100.0, 2, 10.0, 0.0), (115.0, 2, 3.0, 0.0)])
    lc(o, h, ag, st, SLOW_V0)
    assert ag["lane"][0, 0] == 2 and st["changes_left"][0, 0] == st["changes_right"][0, 0] == 0


def test_ego_as_new_follower(two_lane):
    """the ego 12 m behind the abeam station on lane 1 at 54 km/h: ego_b_safe decides the cut-in"""
    o = two_lane()
    for ego_b_safe, moves in ((0.1, False), (100.0, True)):
        h, ag, st = scene2((88.0, 0), SLOW, v_kmh=54.0)
        lc(o, h, ag, st, SLOW_V0, lp=lcparams(ego_b_safe=ego_b_safe))
        assert (ag["lane"][0, 0] == 0) == moves, ego_b_safe


def test_politeness_switches_a_marginal_change_off(two_lane):
    o = two_lane()
    agents = [(100.0, 1, 10.0, 0.0), (150.0, 1, 7.0, 0.0), (60.0, 0, 12.0, 0.0)]
    v0 = [15.0, 7.0, 12.0]
    for p, moves in ((0.0, True), (0.2, True), (1.0, False)):
        h, ag, st = scene2(FAR_EGO, agents)
        lc(o, h, ag, st, v0, lp=lcparams(politeness=p))
        assert (ag["lane"][0, 0] == 0) == moves, p


# ---------------------------------------------------------------- CPU: identities
def closed(joracle, the_map, kind, n, cycles, v0=None, lp=None, seed0=0, metrics=True):
    from dmpp_b200 import scenes
    w = scenes.World(the_map, np.arange(seed0, seed0 + n), kind=kind)
    am = None if v0 is None else (amparams(), v0(w))
    return w, joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=jparams(joracle, kind), threads=8, metrics=mparams() if metrics else None,
                                      agent_model=am, lane_change=lp)


@pytest.mark.parametrize("kind,cycles,lp", [("junction", 120, {}), ("highway", 25, {"a_thr": 1e300})])
def test_armed_without_changes_is_react_only(joracle, the_map, kind, cycles, lp):
    """junction worlds (lane-change attribute 0 on roads 6 / 7) and an unreachable threshold: byte-identical to the reactive agents"""
    _, react = closed(joracle, the_map, kind, 256, cycles, lambda w: w.v0)
    _, on = closed(joracle, the_map, kind, 256, cycles, lambda w: w.v0, lcparams(**lp))
    for k in WORLD + ("metrics",):
        assert on[k].tobytes() == react[k].tobytes(), k
    st = on["lane_change_state"]
    assert (st["changes_left"] == 0).all() and (st["changes_right"] == 0).all()


def test_all_opted_out_is_the_disarmed_loop(joracle, the_map):
    _, off = closed(joracle, the_map, "highway", 256, 25)
    v0 = lambda w: np.where(np.arange(w.v0.size).reshape(w.v0.shape) % 3 == 0, np.nan, -w.v0 * (np.arange(w.v0.shape[1]) % 2))
    _, on = closed(joracle, the_map, "highway", 256, 25, v0, lcparams())
    for k in WORLD + ("metrics",):
        assert on[k].tobytes() == off[k].tobytes(), k


# ---------------------------------------------------------------- CPU: an independent restatement
def restate(m, cump, p, c, h, ag, v0, st):
    """the react (chain-free lanes: no successors on the highway roads) and lane-change phases in plain Python / numpy float64"""
    n = min(int(h["n_obs"]), ag.shape[0])
    off = m.lane_pt_off
    ag, st = ag.copy(), st.copy()
    L = [int(ag["lane"][k]) for k in range(n)]
    S = [cump[off[L[k]] + ag["i"][k]] + ag["u"][k] for k in range(n)]
    V = [ag["v"][k] for k in range(n)]
    length = lambda gl: cump[off[gl + 1] - 1]
    le = int(m.road_lane_base[h["road_num"] - 1] + h["lane_num"] - 1)
    se = cump[off[le] + min(max(int(h["id"][h["lane_num"] - 1]), 0), int(off[le + 1] - off[le]) - 1)]
    ve = h["velocity"] / 3.6
    dt = h["period_ms"] / 1000.0

    def best(cands):
        return min(cands, key=lambda t: (t[0], t[1])) if cands else None

    def acc_of(v, vd, lead):                                # lead = (g, order, vl) or None
        r = v / vd
        fr = (r * r) * (r * r)
        if lead is None:
            a = p.a_max * (1.0 - fr)
        else:
            z = max(v * p.T + v * (v - lead[2]) / (2.0 * np.sqrt(p.a_max * p.b)), 0.0)
            q = (p.s0 + z) / lead[0] if lead[0] > 0 else 0.0
            a = p.a_max * (1.0 - fr - q * q) if lead[0] > 0 else -p.b_max
        return max(a, -p.b_max)

    def ego_acc(lead):
        if lead is None:
            return 0.0
        z = max(ve * p.T + ve * (ve - lead[2]) / (2.0 * np.sqrt(p.a_max * p.b)), 0.0)
        q = (p.s0 + z) / lead[0] if lead[0] > 0 else 0.0
        a = -p.a_max * (q * q) if lead[0] > 0 else -p.b_max
        return max(a, -p.b_max)

    def relax(k):
        st["hold"][k] = st["hold"][k] - dt
        e, w = st["lat_goal"][k] - ag["lat"][k], c.lat_speed * dt
        if e != 0:
            ag["lat"][k] = st["lat_goal"][k] if abs(e) <= w else ag["lat"][k] + (w if e > 0 else -w)

    for k in range(n):
        if not v0[k] > 0:
            relax(k)
            continue
        own = [(se - S[k] - p.ego_rear, -1, ve)] if le == L[k] and se >= S[k] and se - S[k] <= p.look else []
        own += [(S[j] - S[k] - p.length, j, V[j]) for j in range(n)
                if j != k and L[j] == L[k] and (S[j] > S[k] or (S[j] == S[k] and j > k)) and S[j] - S[k] <= p.look]
        ac = acc_of(V[k], v0[k], best(own))
        vn = max(V[k] + ac * dt, 0.0)
        road = int(np.searchsorted(m.road_lane_base, L[k], side="right"))
        b0, nl = int(m.road_lane_base[road - 1]), m.lanes_of(road)
        q, i, u = L[k] - b0, int(ag["i"][k]), ag["u"][k]
        attr = int(m.lanechg_attr[off[L[k]] + i])
        choice = None
        if ag["lat"][k] == st["lat_goal"][k] and st["hold"][k] <= 0 and length(L[k]) - S[k] >= c.end_guard:
            for side, ok in ((-1, q >= 1 and attr in (1, 3)), (1, q + 1 < nl and attr in (2, 3))):
                if not ok:
                    continue
                ml = L[k] + side
                im = min(i, int(off[ml + 1] - off[ml]) - 2)
                sm = cump[off[ml] + im] + u
                if not length(ml) - sm >= c.end_guard:
                    continue
                vehicles = ([(se, -1, ve)] if le == ml else []) + [(S[j], j, V[j]) for j in range(n) if L[j] == ml]
                if any(s == sm for s, _, _ in vehicles):
                    continue
                ahead = [(s - sm - (p.ego_rear if j < 0 else p.length), j, v, s) for s, j, v in vehicles if s > sm and s - sm <= p.look]
                behind = [(sm - s - (c.ego_front if j < 0 else p.length), j, v, s) for s, j, v in vehicles if s < sm and sm - s <= p.look]
                ld, fl = best(ahead), best(behind)
                if (ld is not None and not ld[0] > 0) or (fl is not None and not fl[0] > 0):
                    continue
                atc = acc_of(V[k], v0[k], ld)
                af = atf = 0.0
                if fl is not None and fl[1] < 0:
                    af = ego_acc(None if ld is None else ((ld[3] - fl[3]) - c.ego_front, 0, ld[2]))
                    atf = ego_acc((fl[0], 0, V[k]))
                    if not atf >= -c.ego_b_safe:
                        continue
                elif fl is not None:
                    vdf = v0[fl[1]]
                    if vdf > 0:
                        gap = None if ld is None else ((ld[3] - fl[3]) - (p.ego_rear if ld[1] < 0 else p.length), 0, ld[2])
                        af = acc_of(fl[2], vdf, gap)
                        atf = acc_of(fl[2], vdf, (fl[0], 0, V[k]))
                    if not atf >= -c.b_safe:
                        continue
                delta = (atc - ac) + c.politeness * (atf - af)
                if delta > c.a_thr and (choice is None or delta > choice[0]):
                    choice = (delta, side, ml, im, atc)
        if choice is None:
            ag["v"][k] = vn
            relax(k)
            continue
        _, side, ml, im, atc = choice
        P = np.array([m.x[off[L[k]] + i], m.y[off[L[k]] + i]])
        Q = np.array([m.x[off[ml] + im], m.y[off[ml] + im]])
        R = np.array([m.x[off[ml] + im + 1], m.y[off[ml] + im + 1]])
        dx, dy = R - Q
        Ls = np.sqrt(dx * dx + dy * dy)
        d = (P[0] - Q[0]) * (-(dy / Ls)) + (P[1] - Q[1]) * (dx / Ls) if Ls > 0 else 0.0
        ag["lat"][k] = ag["lat"][k] + d
        ag["lane"][k], ag["i"][k] = ml, im
        ag["v"][k] = max(V[k] + atc * dt, 0.0)
        st["hold"][k] = c.cooldown
        st["changes_left" if side < 0 else "changes_right"][k] += 1
    return ag, st


def test_numpy_restatement_equals_checker(joracle, the_map):
    """10 000 random agent states on the three-lane road 1 and the two-lane road 5 of the highway map: agents bunched within 120 m
    of each other and of the ego, at lane ends, abeam of each other, mid-manoeuvre, in their cooldown and opted out"""
    from dmpp_b200 import abi
    m = the_map
    rng = np.random.default_rng(13)
    n, k = 1000, 10
    w = jworld(m, 0, n, kind="highway")
    h, ag = w.hdr.copy(), w.agents.copy()
    road = np.where(rng.random(n) < 0.5, 1, 5)
    nl = m.road_lane_base[road] - m.road_lane_base[road - 1]
    base = m.road_lane_base[road - 1]
    ag["lane"] = base[:, None] + rng.integers(0, 3, (n, k)) % nl[:, None]
    cnt = m.lane_pt_off[ag["lane"] + 1] - m.lane_pt_off[ag["lane"]]
    centre = rng.integers(0, 2400, n)
    centre[rng.random(n) < 0.1] = 2350
    ag["i"] = np.clip(centre[:, None] + rng.integers(-120, 120, (n, k)), 0, cnt - 2)
    ag["u"] = np.where(rng.random((n, k)) < 0.2, 0.0, rng.uniform(0, 0.5, (n, k)))
    ab = rng.random(n) < 0.3                                # agent 3 abeam of agent 1 (or on its spot)
    ag[ab, 3] = ag[ab, 1]
    ag["lane"][ab, 3] = base[ab] + rng.integers(0, 3, ab.sum()) % nl[ab]
    ag["v"] = np.where(rng.random((n, k)) < 0.1, 0.0, rng.uniform(0, 25, (n, k)))
    ag["lat"] = np.where(rng.random((n, k)) < 0.2, rng.uniform(-3, 3, (n, k)), rng.uniform(-0.5, 0.5, (n, k)))
    st = np.zeros((n, k), abi.lane_change_state)
    st["lat_goal"] = np.where(rng.random((n, k)) < 0.2, ag["lat"] + rng.uniform(-1, 1, (n, k)), ag["lat"])
    st["hold"] = np.where(rng.random((n, k)) < 0.2, rng.uniform(0, 0.3, (n, k)), rng.uniform(-3, 0, (n, k)))
    st["changes_left"] = rng.integers(0, 3, (n, k))
    v0 = rng.uniform(-2, 30, (n, k))
    v0[rng.random((n, k)) < 0.05] = np.nan
    h["road_num"], h["lane_num"] = road, 1 + rng.integers(0, 3, n) % nl
    h["id"] = np.clip(centre[:, None] + rng.integers(-60, 60, (n, 6)), 0, 2400)
    h["n_obs"] = rng.integers(0, k + 1, n)
    h["velocity"] = rng.uniform(0, 90, n)
    h["pos"] = 0
    p, c = amparams(look=150.0), lcparams(politeness=0.3, a_thr=0.1, end_guard=20.0)
    got, gst = ag.copy(), st.copy()
    joracle.lane_change_step(h, got, v0, p, c, gst, wp=jparams(joracle, "highway"))
    cump = cump_of(m)
    want = [restate(m, cump, p, c, h[s], ag[s], v0[s], st[s]) for s in range(n)]
    assert got.tobytes() == np.stack([a for a, _ in want]).tobytes()
    assert gst.tobytes() == np.stack([s for _, s in want]).tobytes()
    moved = got["lane"] != ag["lane"]
    print("changes", moved.sum(), "left", (got["lane"] < ag["lane"]).sum())
    assert moved.sum() > 150 and (got["lane"] < ag["lane"]).any() and (got["lane"] > ag["lane"]).any()


# ---------------------------------------------------------------- CPU: invariants and effect over 512 highway episodes
@pytest.fixture(scope="module")
def highway_steps(joracle, the_map):
    """highway seeds 0-511: the world after every cycle 1 .. 25 with lane changes (one closed loop per length), and the 25-cycle runs
    react-only and with lane changes"""
    from dmpp_b200 import scenes
    w = scenes.World(the_map, np.arange(512), kind="highway")
    wp = jparams(joracle, "highway")
    am, lp, mp = (amparams(), w.v0), lcparams(), mparams()
    states = [(w.agents, None)]
    for c in range(1, 26):
        o = joracle.run_closed_loop(w.hdr, w.agents, c, wp=wp, threads=16, agent_model=am, lane_change=lp)
        states.append((o["agents"], o["lane_change_state"]))
    react = joracle.run_closed_loop(w.hdr, w.agents, 25, wp=wp, threads=16, metrics=mp, agent_model=am)
    on = joracle.run_closed_loop(w.hdr, w.agents, 25, wp=wp, threads=16, metrics=mp, agent_model=am, lane_change=lp)
    return w, states, react, on


def road_of(m, lanes):
    return np.searchsorted(m.road_lane_base, lanes, side="right")


def test_invariants_over_highway_episodes(the_map, highway_steps):
    w, states, _, on = highway_steps
    m = the_map
    goal = states[1][1]["lat_goal"]
    assert goal.tobytes() == np.ascontiguousarray(w.agents["lat"]).tobytes()
    assert states[-1][0].tobytes() == on["agents"].tobytes() and states[-1][1].tobytes() == on["lane_change_state"].tobytes()
    left = np.zeros(w.agents.shape, np.int64)
    right = np.zeros(w.agents.shape, np.int64)
    for (a0, _), (a1, s1) in zip(states, states[1:]):
        assert (road_of(m, a1["lane"]) == road_of(m, w.agents["lane"])).all()
        d = a1["lane"].astype(np.int64) - a0["lane"]
        assert np.isin(d, (-1, 0, 1)).all()
        left += d == -1
        right += d == 1
        grew = np.abs(a1["lat"] - goal) > np.abs(a0["lat"] - goal)
        assert not (grew & (d == 0)).any()
        assert (s1["changes_left"] == left).all() and (s1["changes_right"] == right).all()
        assert (s1["lat_goal"] == goal).all()


def cut_ins(m, hdr_log, states, ahead=30.0):
    """(world, step) pairs where an agent moved into the ego's lane with its station 0 .. `ahead` m in front of the ego's"""
    cump = cump_of(m)
    out = set()
    for c, ((a0, _), (a1, _)) in enumerate(zip(states, states[1:])):
        h = hdr_log[c]
        le = m.road_lane_base[h["road_num"].astype(int) - 1] + h["lane_num"].astype(int) - 1
        se = cump[m.lane_pt_off[le] + h["id"][np.arange(len(h)), h["lane_num"].astype(int) - 1]]
        sk = cump[m.lane_pt_off[a1["lane"]] + a1["i"]] + a1["u"]
        hit = (a1["lane"] != a0["lane"]) & (a1["lane"] == le[:, None]) & (sk >= se[:, None]) & (sk - se[:, None] <= ahead)
        out |= {(int(s), c) for s in np.nonzero(hit.any(axis=1))[0]}
    return out


def test_lane_changes_happen(the_map, highway_steps):
    """findings, not claims: how many worlds change lanes, the cut-ins in front of the ego, and the collision table of DESIGN.md §5;
    asserted is only that changes and cut-ins happen"""
    w, states, react, on = highway_steps
    st = on["lane_change_state"]
    n_ch = st["changes_left"] + st["changes_right"]
    ci = cut_ins(the_map, on["hdr_log"], states)
    print("worlds with a change", int((n_ch.sum(axis=1) > 0).sum()), "changes", int(n_ch.sum()), "left", int(st["changes_left"].sum()),
          "right", int(st["changes_right"].sum()), "cut-ins within 30 m", len(ci), "in worlds", len({s for s, _ in ci}))
    for name, o in (("react-only", react), ("react + lane change", on)):
        print(name, first_strikes(the_map, w, o["metrics"]), "aeb steps", int(o["metrics"]["aeb_steps"].sum()))
    assert (n_ch.sum(axis=1) > 0).sum() > 50 and len(ci) > 0


@pytest.mark.parametrize("kind", ["highway"])
def test_lane_change_log_replays_open_loop(oracle, highway_steps, kind):
    _, _, _, on = highway_steps
    rep = oracle.run(on["hdr_log"], on["obs_log_x"], on["obs_log_y"], exhaustive=False, threads=8)
    assert rep["rec"].tobytes() == on["rec"].tobytes()


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_graph_equals_checker(joracle, the_map):
    """4096 highway worlds as ONE graph launch, replayed three times from the same initial world; metrics armed too"""
    gpu_vs_checker(joracle, the_map, "highway", 4096, 25, repeat=3, lane_change=lcparams())


@pytest.mark.gpu
@pytest.mark.parametrize("env,metrics", [({"DP_EPISODE_GRAPH": "0"}, False), ({"DP_KERNEL": "group"}, True)])
def test_gpu_direct_launches_and_group_kernel(joracle, the_map, env, metrics):
    gpu_vs_checker(joracle, the_map, "highway", 4096, 25, env=env, metrics=metrics, lane_change=lcparams())


@pytest.mark.gpu
def test_gpu_highway_200_agents(joracle, the_map):
    gpu_vs_checker(joracle, the_map, "highway", 1024, 25, n_obs=200, lane_change=lcparams())


@pytest.mark.gpu
def test_gpu_single_steps_ragged(joracle, the_map):
    """dp_world_step_dev with first > 0: ragged n_obs, agents at lane ends, abeam of each other, mid-manoeuvre and in their cooldown,
    mixed opt-out agents, against jo_lane_change_step + the checker's world step; the placement step initialises the states"""
    import torch
    from dmpp_b200 import abi
    n, first = 600, 37
    m = the_map
    w = jworld(m, 123, n, kind="highway")
    rng = np.random.default_rng(9)
    w.hdr["n_obs"] = rng.integers(0, 11, n)
    ends = (m.lane_pt_off[w.agents["lane"] + 1] - m.lane_pt_off[w.agents["lane"]]) - 2
    w.agents["i"][::3] = ends[::3] - rng.integers(0, 80, (len(w.agents[::3]), 10))
    dup = rng.random(n) < 0.3
    w.agents[dup, 4] = w.agents[dup, 2]
    v0 = np.where(rng.random(w.v0.shape) < 0.2, 0.0, w.v0 + rng.uniform(-2, 8, w.v0.shape))
    rec = np.zeros(n, abi.plan_record)
    rec["brakespeed"] = rng.uniform(0, 20, n)
    rec["afresh_planning"], rec["behavior"] = 1, 1
    lp_ = np.zeros((n, 2, 200))
    hr = np.radians(w.hdr["dir"])
    lp_[:, 0] = w.hdr["x"][:, None] + 0.5 * np.arange(200) * np.cos(hr)[:, None]
    lp_[:, 1] = w.hdr["y"][:, None] + 0.5 * np.arange(200) * np.sin(hr)[:, None]
    # a short cooldown and a quick return to lat_goal (3.75 m in 4 steps): within 12 steps agents are caught mid-manoeuvre and
    # some change lanes twice
    wp, am, lc = jparams(joracle, "highway"), amparams(), lcparams(cooldown=0.15, lat_speed=10.0)
    p = planner_with(m, first + n, 10, 0)
    try:
        p.upload_carry(first, np.zeros(n, abi.carry), lp_)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()
        st = np.zeros((n, 10), abi.lane_change_state)
        st["hold"] = 77.0                                   # overwritten by the placement step
        d_h, d_a, d_v0, d_r, d_st = dev(w.hdr), dev(w.agents), dev(v0), dev(rec), dev(st)
        d_x, d_y = torch.zeros(n * 10, dtype=torch.float64, device="cuda"), torch.zeros(n * 10, dtype=torch.float64, device="cuda")
        p.set_agent_model(am, d_v0.data_ptr())
        p.set_lane_change(lc, d_st.data_ptr())
        h, ag, ox, oy = w.hdr.copy(), w.agents.copy(), np.zeros((n, 10)), np.zeros((n, 10))
        joracle.world_step(h, ag, ox, oy, wp=wp)
        used = np.arange(10)[None, :] < w.hdr["n_obs"][:, None]
        st[used] = 0
        st["lat_goal"][used] = w.agents["lat"][used]
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None, first=first)
        for _ in range(12):
            joracle.lane_change_step(h, ag, v0, am, lc, st, wp=wp)
            joracle.world_step(h, ag, ox, oy, rec=rec, last_path=lp_, wp=wp)
            p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), first=first)
        torch.cuda.synchronize()
        assert np.frombuffer(d_h.cpu().numpy().tobytes(), abi.scene_hdr).tobytes() == h.tobytes()
        got = np.frombuffer(d_a.cpu().numpy().tobytes(), abi.agent).reshape(n, 10)
        gst = np.frombuffer(d_st.cpu().numpy().tobytes(), abi.lane_change_state).reshape(n, 10)
        assert got[used].tobytes() == ag[used].tobytes()
        assert got[~used].tobytes() == w.agents[~used].tobytes()
        assert gst[used].tobytes() == st[used].tobytes()
        assert (gst["hold"][~used] == 77.0).all()
        assert (got["lane"][used] != w.agents["lane"][used]).sum() > 10 and (gst["changes_left"][used] > 1).any()
    finally:
        p.set_agent_model(None, None)
        p.close()


@pytest.mark.gpu
def test_gpu_arm_disarm_rearm(the_map):
    """on one context: react-only episodes after lane changes are byte-identical to a context that never armed them; re-arming
    repeats the armed run"""
    n = 1024
    w = jworld(the_map, 700, n, kind="highway")
    am = (amparams(), w.v0)
    never = planner_with(the_map, n, 10, 0)
    try:
        ref = never.run_closed_loop(w.hdr, w.agents, 25, agent_model=am)
    finally:
        never.close()
    p = planner_with(the_map, n, 10, 0)
    try:
        a = p.run_closed_loop(w.hdr, w.agents, 25, agent_model=am, lane_change=lcparams())
        b = p.run_closed_loop(w.hdr, w.agents, 25, agent_model=am)
        c = p.run_closed_loop(w.hdr, w.agents, 25, agent_model=am, lane_change=lcparams())
    finally:
        p.close()
    assert a["graph"] and b["graph"] and c["graph"]
    for k in WORLD:
        assert b[k].tobytes() == ref[k].tobytes(), k
        assert c[k].tobytes() == a[k].tobytes(), k
    assert a["lane_change_state"].tobytes() == c["lane_change_state"].tobytes()
    assert a["agents"].tobytes() != ref["agents"].tobytes()


@pytest.mark.gpu
def test_gpu_bad_params(the_map):
    from dmpp_b200 import planner
    p = planner_with(the_map, 16, 10, 0)
    lib = p.lib
    try:
        assert lib.dp_world_set_lane_change(p.ctx, C.byref(lcparams()), C.c_void_p(16)) == -1   # the agent model is not armed
        assert lib.dp_world_set_agent_model(p.ctx, C.byref(amparams()), C.c_void_p(16)) == 0
        for field, bad in (("lat_speed", 0.0), ("b_safe", 0.0), ("ego_b_safe", -1.0), ("politeness", -0.1), ("cooldown", -1.0),
                           ("end_guard", -1.0), ("ego_front", -0.5), ("a_thr", float("nan")), ("politeness", float("inf"))):
            assert lib.dp_world_set_lane_change(p.ctx, C.byref(lcparams(**{field: bad})), C.c_void_p(16)) == -1, field
        assert lib.dp_world_set_lane_change(p.ctx, None, C.c_void_p(16)) == -1
        assert lib.dp_world_set_lane_change(p.ctx, C.byref(lcparams(politeness=0.0, cooldown=0.0, end_guard=0.0, ego_front=0.0,
                                                                    a_thr=-1.0)), C.c_void_p(16)) == 0
        assert lib.dp_world_set_lane_change(p.ctx, None, None) == 0
        with pytest.raises(planner.DpError):
            p.set_lane_change(lcparams(lat_speed=float("nan")), 16)
        assert lib.dp_world_set_agent_model(p.ctx, None, None) == 0
    finally:
        p.close()
