"""Agents obey the V2X events in closed-loop episodes (include/dmpp_b200.h section 15; arithmetic frozen in
tools/junction_oracle/v2x_traffic.h): the stop line of a red or yellow signal and the active pedestrian are two more leaders of the
reactive agents, standing still, and of their lane changes' target lane.

CPU side: layout and defaults; a numpy restatement of the candidates and of the leader choice against the checker on random states;
known answers on a straight road; obey = 0 against the model disarmed; the effect on seeds 0-511.
GPU side: the TRAFFIC instances of the world step against the checker byte for byte (graph replays, direct launches, the group
kernel, metrics and lane changes armed or not), arm / disarm / re-arm, stepping by hand, bad arguments."""
import ctypes as C
import types

import numpy as np
import pytest

from worlds import (WORLD, StraightRoad, amparams, check_closed_loop, check_rows, cump_of, first_strikes, jparams, jworld,  # noqa: F401
                    joracle, lcparams, mparams, planner_with)

CYCLES = {"highway": 25, "junction": 120}


def tparams(**kw):
    from dmpp_b200 import planner
    return planner.v2x_traffic_params(**kw)


def vparams(mode=0, apply=1):
    from dmpp_b200 import abi
    return abi.V2xWorldParams(mode, apply)


def test_layouts_and_defaults(joracle):
    from dmpp_b200 import abi
    assert joracle.traffic_sizeof() == (C.sizeof(abi.V2xTrafficParams), abi.v2x_traffic_stats.itemsize) == (24, 32)
    p = tparams()                                           # through dp_v2x_traffic_default_params: no GPU needed
    assert (p.b_commit, p.ped_half_width, p.obey, p.pad) == (4.0, 2.0, 1, 0)
    assert p.b_commit == lcparams().b_safe


# ---------------------------------------------------------------- CPU: the candidates, restated
def world_of(m, cump, tp, s, h, k):
    """section 15's world in Python float64: (state, ped_on, px, py, governed lanes, S(l))"""
    t = float(k) * float(h["period_ms"]) / 1000.0
    state = 0
    if s["sig_road"] > 0:
        ph = float(np.fmod(t + float(s["sig_offset"]), float(s["sig_cycle"])))
        if ph < 0:
            ph += float(s["sig_cycle"])
        state = 6 if ph < s["sig_green"] else (7 if ph < float(s["sig_green"]) + float(s["sig_yellow"]) else 3)
    ped_on = bool(s["has_ped"] and s["ped_t_on"] <= t <= s["ped_t_off"])
    px = py = 0.0
    if ped_on:
        tp_ = t - float(s["ped_t_on"])
        px, py = float(s["ped_x"]) + float(s["ped_vx"]) * tp_, float(s["ped_y"]) + float(s["ped_vy"]) * tp_
    gb = ge = 0
    if s["sig_road"] > 0:
        gb, ge = int(m.road_lane_base[s["sig_road"] - 1]), int(m.road_lane_base[s["sig_road"]])

    def S(l):
        off, cnt = int(m.lane_pt_off[l]), int(m.lane_pt_off[l + 1] - m.lane_pt_off[l])
        stop = cnt - 1 if (s["sig_stop"] < 0 or s["sig_stop"] > cnt - 1) else int(s["sig_stop"])
        return float(cump[off + stop])
    return types.SimpleNamespace(line=state in (3, 7), ped_on=ped_on, px=px, py=py, gov=lambda l: gb <= l < ge, S=S, state=state)


def line_gap(tp, am, ds, v):
    if not ds <= am.look:
        return None
    g = ds - am.length
    return g if (g > 0 and v * v <= 2.0 * tp.b_commit * g) else None


def ped_gap(m, w, tp, am, l, i, u):
    if not w.ped_on:
        return None
    o = int(m.lane_pt_off[l])
    qx, qy, rx, ry = float(m.x[o + i]), float(m.y[o + i]), float(m.x[o + i + 1]), float(m.y[o + i + 1])
    dx, dy = rx - qx, ry - qy
    L = float(np.sqrt(dx * dx + dy * dy))
    if not L > 0:
        return None
    q = u / L
    Px, Py, tx, ty = qx + q * dx, qy + q * dy, dx / L, dy / L
    ex, ey = w.px - Px, w.py - Py
    lon, lat = ex * tx + ey * ty, ey * tx - ex * ty
    return lon - am.length if (0 < lon <= am.look and abs(lat) <= tp.ped_half_width) else None


def line_ds(w, l0, l1, l2, D1, D2, sk):
    """the line's distance along the chain (None: no line), the first governed lane deciding"""
    if not w.line:
        return None
    if w.gov(l0):
        return w.S(l0) - sk if w.S(l0) > sk else None
    if l1 >= 0 and w.gov(l1):
        return D1 + w.S(l1)
    if l2 >= 0 and w.gov(l2):
        return D2 + w.S(l2)
    return None


def leader_of(m, w, tp, am, l0, l1, l2, D1, D2, sk, v, i, u, lead, best):
    kind = 0
    if w.line:
        ds = line_ds(w, l0, l1, l2, D1, D2, sk)
        g = None if ds is None else line_gap(tp, am, ds, v)
        if g is not None and (not lead or g < best):
            best, lead, kind = g, True, 1
    g = ped_gap(m, w, tp, am, l0, i, u)
    if g is not None and (not lead or g < best):
        best, lead, kind = g, True, 2
    return best, lead, kind


def side_of(m, w, tp, am, ml, im, sm, u, v, lead, g):
    won = False
    if w.line and w.gov(ml) and w.S(ml) > sm:
        c = line_gap(tp, am, w.S(ml) - sm, v)
        if c is not None and (not lead or c < g):
            g, lead, won = c, True, True
    c = ped_gap(m, w, tp, am, ml, im, u)
    if c is not None and (not lead or c < g):
        g, lead, won = c, True, True
    return g, lead, won


def random_states(m, cump, n, rng):
    """specifications and agents that reach every clause: the line on l0 / l1 / l2 and nowhere, commit pass and fail, states 0 / 3 / 6
    / 7, the pedestrian inside and outside the band, behind and beyond look, ties with the vehicle leader"""
    from dmpp_b200 import abi
    road = rng.integers(1, m.n_roads + 1, n)
    h = np.zeros(n, abi.scene_hdr)
    h["period_ms"] = rng.choice([100.0, 80.0, 120.0], n)
    k = rng.integers(0, 300, n).astype(np.int32)
    s = np.zeros(n, abi.v2x_event_spec)
    s["sig_road"] = np.where(rng.random(n) < 0.85, road, 0)
    g, yl, r = rng.uniform(1, 20, n), rng.uniform(0.5, 4, n), rng.uniform(1, 20, n)
    s["sig_green"], s["sig_yellow"], s["sig_red"], s["sig_cycle"] = g, yl, r, g + yl + r
    s["sig_offset"] = rng.uniform(-60, 60, n)
    base, top = m.road_lane_base[road - 1], m.road_lane_base[road]
    gov = base + (rng.random(n) * (top - base)).astype(np.int64)
    other = rng.integers(0, m.n_lanes, n)
    # chain: where the first governed lane sits (0, 1, 2 or nowhere)
    where = rng.integers(0, 4, n)
    lanes = np.stack([np.where(where == 0, gov, other), np.where(where == 1, gov, np.where(rng.random(n) < 0.2, -1, other)),
                      np.where(where == 2, gov, other)], axis=1)
    lanes[:, 2] = np.where(lanes[:, 1] < 0, -1, lanes[:, 2])
    notgov = (lanes < base[:, None]) | (lanes >= top[:, None])
    lanes[:, 1] = np.where((where == 2) & ~notgov[:, 1], -1, lanes[:, 1])           # keep the first governed lane where it is meant
    lanes[:, 2] = np.where(lanes[:, 1] < 0, -1, lanes[:, 2])
    l0 = lanes[:, 0]
    cnt = m.lane_pt_off[l0 + 1] - m.lane_pt_off[l0]
    i = (rng.random(n) * (cnt - 1)).astype(np.int64)
    # stop lines within reach: around the agent on l0, near the start of l1 / l2; sometimes the lane's last point
    stop = np.where(where == 0, i + rng.integers(-20, 220, n), rng.integers(0, 150, n))
    s["sig_stop"] = np.where(rng.random(n) < 0.1, -1, np.maximum(stop, 0))
    u = rng.uniform(0, 0.5, n)
    sk = cump[m.lane_pt_off[l0] + i] + u
    x = np.zeros((n, 6))
    x[:, 0] = rng.uniform(0, 60, n)                         # D1
    x[:, 1] = x[:, 0] + rng.uniform(0, 60, n)               # D2
    x[:, 2], x[:, 3], x[:, 4] = sk, rng.uniform(0, 20, n), u
    x[:, 5] = rng.uniform(-5, 100, n)                       # the vehicle leader's g
    iv = np.stack([i, rng.random(n) < 0.5], axis=1).astype(np.int32)
    # the pedestrian in the agent's segment frame: lon -10 .. 110, lat -3 .. 3
    o = m.lane_pt_off[l0] + i
    dx, dy = m.x[o + 1] - m.x[o], m.y[o + 1] - m.y[o]
    L = np.sqrt(dx * dx + dy * dy)
    tx, ty = dx / L, dy / L
    lon, lat = rng.uniform(-10, 110, n), rng.uniform(-3, 3, n)
    px, py = m.x[o] + u / L * dx, m.y[o] + u / L * dy
    s["ped_x"], s["ped_y"] = px + lon * tx - lat * ty, py + lon * ty + lat * tx
    s["has_ped"] = rng.random(n) < 0.6
    t = k * h["period_ms"] / 1000.0
    s["ped_t_on"] = np.where(rng.random(n) < 0.8, t - rng.uniform(0, 5, n), t + 1.0)
    s["ped_t_off"] = s["ped_t_on"] + rng.uniform(0, 20, n)
    return h, s, k, lanes.astype(np.int32), x, iv


def test_numpy_candidates_equal_checker(joracle, the_map):
    """10 000 random agents: section 12's leader after the vehicle scan (best, lead, kind) and the target lane's leader (g, lead, won),
    every byte, with ties forced against the vehicle leader"""
    m, cump = the_map, cump_of(the_map)
    rng = np.random.default_rng(15)
    n = 10000
    h, s, k, lanes, x, iv = random_states(m, cump, n, rng)
    am = amparams()
    tp = tparams(b_commit=float(rng.uniform(2, 6)), ped_half_width=1.5)
    # ties: half of the agents with a vehicle leader get exactly the candidate's g
    ws = [world_of(m, cump, tp, s[j], h[j], int(k[j])) for j in range(n)]
    for j in range(n):
        l0, l1, l2 = (int(v) for v in lanes[j])
        b, lead, kind = leader_of(m, ws[j], tp, am, l0, l1, l2, *x[j, :4], int(iv[j, 0]), float(x[j, 4]), False, 0.0)
        if kind and rng.random() < 0.5:
            x[j, 5], iv[j, 1] = b, 1
    got = joracle.traffic_leader(tp, am, s, h, k, lanes, x, iv)
    want = np.zeros((n, 3))
    for j in range(n):
        l0, l1, l2 = (int(v) for v in lanes[j])
        want[j] = leader_of(m, ws[j], tp, am, l0, l1, l2, *x[j, :4], int(iv[j, 0]), float(x[j, 4]), bool(iv[j, 1]), float(x[j, 5]))
    assert got.tobytes() == want.tobytes()
    kind = want[:, 2]
    states = np.array([w.state for w in ws])
    print({"kinds": np.bincount(kind.astype(int)).tolist(), "states": np.bincount(states).tolist()})
    assert (np.bincount(kind.astype(int), minlength=3) > 500).all() and {0, 3, 6, 7} <= set(states.tolist())
    # the line decided on each chain position, and the commit test failing
    line = (kind == 1)
    for pos in range(3):
        gov = np.array([ws[j].gov(int(lanes[j, pos])) and (pos == 0 or not any(ws[j].gov(int(lanes[j, q])) for q in range(pos)))
                        for j in range(n)])
        assert (line & gov).sum() > 50, pos
    ds = [line_ds(ws[j], *(int(v) for v in lanes[j]), *x[j, :3]) for j in range(n)]
    fail = np.array([d is not None and d <= am.look and d - am.length > 0 and line_gap(tp, am, d, x[j, 3]) is None for j, d in enumerate(ds)])
    assert fail.sum() > 200
    # pedestrian: in the band, out of it, behind
    ped_in = np.array([ped_gap(m, ws[j], tp, am, int(lanes[j, 0]), int(iv[j, 0]), x[j, 4]) is not None for j in range(n)])
    assert ped_in.sum() > 500 and ((s["has_ped"] == 1) & ~ped_in).sum() > 500
    tie = (iv[:, 1] == 1) & (x[:, 5] == want[:, 0])
    assert (tie & (kind == 0)).sum() > 200                  # a tie keeps the vehicle
    # the target lane: m = l0 abeam, safe (g > 0) and unsafe (g <= 0)
    sl = np.stack([lanes[:, 0], iv[:, 0]], axis=1)
    xs = np.stack([x[:, 2], x[:, 4], x[:, 3], x[:, 5]], axis=1)
    got = joracle.traffic_side(tp, am, s, h, k, sl, xs, iv[:, 1])
    want = np.array([side_of(m, ws[j], tp, am, int(sl[j, 0]), int(sl[j, 1]), *xs[j, :3], bool(iv[j, 1]), float(xs[j, 3]))
                     for j in range(n)], np.float64)
    assert got.tobytes() == want.tobytes()
    won, g = want[:, 2] == 1, want[:, 0]
    assert (won & (g > 0)).sum() > 300 and (won & (g <= 0)).sum() > 30    # unsafe: the pedestrian within length


# ---------------------------------------------------------------- CPU: known answers on a straight road
@pytest.fixture
def road(joracle, the_map):
    def use(lanes=1, attr=0):
        joracle.set_map(StraightRoad(6000, lanes=lanes, attr=attr))
        return joracle
    yield use
    joracle.set_map(the_map)


DT = 0.1
W = 3.75


def scene(agents, lanes=1):
    """one world on StraightRoad: the ego standing far ahead on lane 1; agents as (x, lane, v, lat)"""
    from dmpp_b200 import abi
    h = np.zeros(1, abi.scene_hdr)
    h["x"], h["y"], h["period_ms"] = 2900.0, W * (lanes - 1) / 2, 1000 * DT
    h["road_num"], h["lane_num"], h["next_roadnum"], h["conn"] = 1, 1, 1, -1
    h["id"][:, :lanes] = 5800
    h["n_obs"] = len(agents)
    ag = np.zeros((1, len(agents)), abi.agent)
    for k, (x, lane, v, lat) in enumerate(agents):
        ag["i"][0, k] = int(x // 0.5)
        ag["u"][0, k] = x - 0.5 * int(x // 0.5)
        ag["lane"][0, k], ag["v"][0, k], ag["lat"][0, k] = lane, v, lat
    return h, ag


def signal(stop=400, green=10.0, yellow=3.0, red=1000.0, offset=13.0):
    """a signal on road 1 at point `stop` (station stop / 2 m); by default red for the first 1000 s"""
    from dmpp_b200 import abi
    s = np.zeros(1, abi.v2x_event_spec)
    s["sig_road"], s["sig_stop"] = 1, stop
    s["sig_green"], s["sig_yellow"], s["sig_red"], s["sig_cycle"] = green, yellow, red, green + yellow + red
    s["sig_offset"] = offset
    return types.SimpleNamespace(spec=s, wp_x=np.zeros(0), wp_y=np.zeros(0))


def pedestrian(x, y):
    from dmpp_b200 import abi
    s = np.zeros(1, abi.v2x_event_spec)
    s["has_ped"], s["ped_x"], s["ped_y"], s["ped_t_off"] = 1, x, y, 1e6
    return types.SimpleNamespace(spec=s, wp_x=np.zeros(0), wp_y=np.zeros(0))


def episode(o, ev, agents, v0, steps, tp=None, lanes=1, lp=None):
    """`steps` world steps of the checker with the ego standing; returns the agents' (x, v, lane) per step, the row, the kinds and the
    final lane-change states"""
    from dmpp_b200 import abi
    h, ag = scene(agents, lanes)
    n = ag.shape[1]
    ox, oy = np.zeros((1, n)), np.zeros((1, n))
    ts = np.zeros(1, abi.v2x_traffic_stats)
    lcs = None if lp is None else np.zeros((1, n), abi.lane_change_state)
    v0 = np.array([v0], np.float64)
    tp, am = tp or tparams(), amparams()
    rec, lpath = np.zeros(1, abi.plan_record), np.zeros((1, 400))
    o.traffic_step(tp, ev, 0, h, ag, ox, oy, v0, am, ts, lp=lp, lcs=lcs)
    xs, vs, ls, kinds = [], [], [], []
    for k in range(steps):
        kinds.append(o.traffic_step(tp, ev, k, h, ag, ox, oy, v0, am, ts, rec=rec, last_path=lpath, lp=lp, lcs=lcs)[0])
        xs.append(0.5 * ag["i"][0] + ag["u"][0]); vs.append(ag["v"][0].copy()); ls.append(ag["lane"][0].copy())
    return np.array(xs), np.array(vs), np.array(ls), ts[0], np.array(kinds), lcs


def test_red_line_stops_the_agent(road):
    o = road()
    xs, vs, _, r, kinds, _ = episode(o, signal(), [(100.0, 0, 10.0, 0.0)], [15.0], 600)
    assert xs[:, 0].max() < 200.0 - 4.5 and vs[-1, 0] == 0.0 and xs[-1, 0] > 200.0 - 4.5 - 3.0
    assert r["red_runs"] == 0 and r["line_steps"] == (kinds[:, 0] == 1).sum() > 100 and r["ped_steps"] == 0
    # obey = 0: counted, but the agent drives through and the run is counted once
    xs, vs, _, r0, kinds0, _ = episode(o, signal(), [(100.0, 0, 10.0, 0.0)], [15.0], 600, tp=tparams(obey=0))
    assert xs[-1, 0] > 300.0 and r0["red_runs"] == 1 and r0["line_steps"] == (kinds0[:, 0] == 1).sum() > 0
    # yellow stops it too when it can stop; green does not
    xs, *_ = episode(o, signal(green=100.0, yellow=1000.0, red=10.0, offset=100.0), [(100.0, 0, 10.0, 0.0)], [15.0], 600)
    assert xs[:, 0].max() < 200.0 - 4.5
    xs, _, _, r, *_ = episode(o, signal(green=1000.0, offset=0.0), [(100.0, 0, 10.0, 0.0)], [15.0], 300)
    assert xs[-1, 0] > 300.0 and r["red_runs"] == 0 and r["line_steps"] == 0


def test_too_fast_at_yellow_continues_and_runs_the_red(road):
    """10 m before the line at 15 m/s: g = 5.5 m, 15^2 > 2 * 4 * 5.5, so it does not commit; the light turns red 0.2 s later"""
    o = road()
    ev = signal(green=10.0, yellow=3.0, red=20.0, offset=12.8)
    xs, vs, _, r, kinds, _ = episode(o, ev, [(190.0, 0, 15.0, 0.0)], [15.0], 30)
    assert (vs[:, 0] == 15.0).all() and xs[-1, 0] > 200.0
    assert r["red_runs"] == 1 and r["line_steps"] == 0 and (kinds == 0).all()
    # with b_commit = 25 it commits and brakes, but the IDM's hardest braking (b_max = 8) cannot stop it in 5.5 m: it runs all the same
    _, vs, _, r, *_ = episode(o, ev, [(190.0, 0, 15.0, 0.0)], [15.0], 30, tp=tparams(b_commit=25.0))
    assert vs[1, 0] < 15.0 and r["line_steps"] > 0 and r["red_runs"] == 1


def test_pedestrian_in_the_lane_stops_the_agent(road):
    o = road()
    xs, vs, _, r, kinds, _ = episode(o, pedestrian(150.0, 0.0), [(100.0, 0, 10.0, 0.0)], [15.0], 400)
    assert xs[:, 0].max() < 150.0 - 4.5 and vs[-1, 0] == 0.0
    assert r["ped_hits"] == 0 and r["ped_steps"] == (kinds[:, 0] == 2).sum() > 100 and r["line_steps"] == 0
    assert r["min_ped_dist"] == np.abs(150.0 - xs[:, 0]).min() > 4.5
    xs, _, _, r0, *_ = episode(o, pedestrian(150.0, 0.0), [(100.0, 0, 10.0, 0.0)], [15.0], 400, tp=tparams(obey=0))
    assert xs[-1, 0] > 200.0 and r0["ped_hits"] >= 4 and r0["min_ped_dist"] < 0.5 and r0["ped_steps"] > 0


def test_pedestrian_beyond_the_band_does_not(road):
    o = road()
    free, *_ = episode(o, signal(green=1000.0, offset=0.0), [(100.0, 0, 10.0, 0.0)], [15.0], 200)
    for y, w in ((2.01, 2.0), (-2.5, 2.0), (1.0, 0.9)):
        xs, _, _, r, kinds, _ = episode(o, pedestrian(150.0, y), [(100.0, 0, 10.0, 0.0)], [15.0], 200, tp=tparams(ped_half_width=w))
        assert xs.tobytes() == free.tobytes() and r["ped_steps"] == 0 and (kinds == 0).all(), y
        assert r["ped_hits"] == 0 and abs(y) <= r["min_ped_dist"] <= np.hypot(y, 1.0)   # (sampled at the ends of 1 m steps)
    xs, *_ = episode(o, pedestrian(150.0, 1.99), [(100.0, 0, 10.0, 0.0)], [15.0], 200)
    assert xs[:, 0].max() < 150.0 - 4.5


def test_no_lane_change_to_pass_a_red_line(road):
    """two governed lanes, changes allowed.  One agent 20 m before the red line on lane 2, braking for it: lane 1 is free road up to the
    same line, so without the target lane's line MOBIL would see an incentive of about 1 + 8 m/s^2 and change; with it the target
    lane offers the same leader and the agent stays.  A queue of agents behind slower ones may change lanes, but nobody runs the line"""
    o = road(lanes=2, attr=3)
    xs, vs, ls, r, _, st = episode(o, signal(), [(180.0, 1, 5.0, 0.0)], [15.0], 200, lanes=2, lp=lcparams())
    assert (ls == 1).all() and (st["changes_left"] + st["changes_right"]).sum() == 0 and vs[0, 0] < 5.0
    assert r["red_runs"] == 0 and xs.max() < 200.0 - 4.5 and vs[-1, 0] == 0.0
    queue = [(60.0 + 15.0 * j, 1, 10.0 - j, 0.0) for j in range(6)]
    xs, vs, ls, r, _, st = episode(o, signal(), queue, [15.0] * 6, 600, lanes=2, lp=lcparams())
    assert r["red_runs"] == 0 and xs.max() < 200.0 - 4.5 and (vs[-1] == 0).all() and r["line_steps"] > 0
    # the same queue without the signal changes lanes, and with obey = 0 it runs the line
    _, _, _, _, _, st = episode(o, signal(green=1000.0, offset=0.0), queue, [15.0] * 6, 100, lanes=2, lp=lcparams())
    assert (st["changes_left"] + st["changes_right"]).sum() > 0
    _, _, _, r, _, _ = episode(o, signal(), queue, [15.0] * 6, 600, lanes=2, lp=lcparams(), tp=tparams(obey=0))
    assert r["red_runs"] == 6


# ---------------------------------------------------------------- CPU: the checker on the seeded worlds
def closed(o, the_map, kind, n, traffic, seed0=0, lane_change=False):
    from dmpp_b200 import scenes
    w = jworld(the_map, seed0, n, kind=kind)
    ev = scenes.V2xEvents(w, np.arange(seed0, seed0 + n))
    kw = dict(lane_change=lcparams()) if lane_change else {}
    return w, ev, o.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(o, kind), threads=16, metrics=mparams(),
                                    agent_model=(amparams(), w.v0), v2x=(vparams(), ev), traffic=traffic, **kw)


@pytest.fixture(scope="module")
def runs(joracle, the_map):
    out = {}
    for kind in CYCLES:
        for obey in (None, 0, 1):
            out[kind, obey] = closed(joracle, the_map, kind, 512, None if obey is None else tparams(obey=obey))
    return out


@pytest.mark.parametrize("kind", list(CYCLES))
def test_obey_0_is_the_model_disarmed(joracle, the_map, runs, kind):
    """obey = 0: records, logs, world, carry, metrics and V2X rows byte-identical to the model disarmed (and with lane changes);
    obey = 1 changes them"""
    off, obs, on = runs[kind, None][2], runs[kind, 0][2], runs[kind, 1][2]
    for k in WORLD + ("metrics", "v2x_stats", "v2x_flags"):
        assert obs[k].tobytes() == off[k].tobytes(), k
    assert on["agents"].tobytes() != off["agents"].tobytes()
    a, b = closed(joracle, the_map, kind, 128, None, 700, True)[2], closed(joracle, the_map, kind, 128, tparams(obey=0), 700, True)[2]
    for k in WORLD + ("metrics", "v2x_stats", "lane_change_state"):
        assert a[k].tobytes() == b[k].tobytes(), k
    assert (b["v2x_traffic"]["line_steps"] + b["v2x_traffic"]["ped_steps"]).sum() > 0


def effect(the_map, runs):
    """the effect figures of DESIGN.md section 5 (obey 0 -> 1)"""
    out = {}
    for obey in (0, 1):
        w, ev, o = runs["junction", obey]
        ts, vs, met = o["v2x_traffic"], o["v2x_stats"], o["metrics"]
        out["junction", obey] = dict(red_runs=int(ts["red_runs"].sum()), line_steps=int(ts["line_steps"].sum()),
                                     ego_red_crossings=int(vs["red_crossings"].sum()), ego_stopped_steps=int(met["stopped_steps"].sum()),
                                     first_strikes=first_strikes(the_map, w, met))
        w, ev, o = runs["highway", obey]
        ts, met = o["v2x_traffic"], o["metrics"]
        ped = ev.spec["has_ped"] == 1
        out["highway", obey] = dict(ped_hits=int(ts["ped_hits"].sum()), ped_steps=int(ts["ped_steps"].sum()),
                                    hit_worlds=int((ts["ped_hits"] > 0).sum()), min_ped_dist_below_2m=int((ts["min_ped_dist"][ped] < 2.0).sum()),
                                    min_ped_dist_median=round(float(np.median(ts["min_ped_dist"][ped])), 3),
                                    collision_worlds=int((met["first_collision_step"] > 0).sum()),
                                    collision_steps=int(met["collision_steps"].sum()))
    return out


def test_effect_on_seeds_0_511(the_map, runs):
    """the effect table of DESIGN.md section 5, from the checker (apply = 1, reactive agents, obey 0 against 1)"""
    e = effect(the_map, runs)
    print(e)
    j0, j1, h0, h1 = e["junction", 0], e["junction", 1], e["highway", 0], e["highway", 1]
    assert (j0["red_runs"], j1["red_runs"]) == (765, 299) and (j0["ego_red_crossings"], j1["ego_red_crossings"]) == (151, 113)
    assert (j0["ego_stopped_steps"], j1["ego_stopped_steps"]) == (10109, 13556)
    assert j0["first_strikes"] == {"worlds": 272, "behind": 50, "behind_faster": 45, "ahead": 122, "other_lane": 100}
    assert j1["first_strikes"] == {"worlds": 254, "behind": 42, "behind_faster": 38, "ahead": 129, "other_lane": 83}
    assert (h0["ped_hits"], h1["ped_hits"]) == (424, 403) and (h0["hit_worlds"], h1["hit_worlds"]) == (86, 57)
    assert (h0["min_ped_dist_below_2m"], h1["min_ped_dist_below_2m"]) == (127, 76)
    assert (h0["collision_worlds"], h1["collision_worlds"]) == (208, 218)
    for kind in CYCLES:                                     # the row counts the same candidates whether they are obeyed or not
        assert (runs[kind, 0][2]["v2x_traffic"]["line_steps"].sum() + runs[kind, 0][2]["v2x_traffic"]["ped_steps"].sum()) > 0


# ---------------------------------------------------------------- GPU
def gpu_vs_checker(joracle, the_map, kind, n, tp, env=None, repeat=1, metrics=True, lane_change=False, seed0=0):
    from dmpp_b200 import scenes
    w = jworld(the_map, seed0, n, kind=kind)
    ev = scenes.V2xEvents(w, np.arange(seed0, seed0 + n))
    kw = dict(metrics=mparams() if metrics else None, agent_model=(amparams(), w.v0), v2x=(vparams(), ev), traffic=tp,
              lane_change=lcparams() if lane_change else None)
    want = joracle.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(joracle, kind), threads=16, **kw)
    p = planner_with(the_map, n, 10, scenes.World.PRE_JUNCTION_PTS[kind], env)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], repeat=repeat, **kw)
    finally:
        p.close()
    what = "%s %r obey %d" % (kind, env, tp.obey)
    assert got["graph"] == (env is None), what
    check_closed_loop(got, want, what)
    for k in ("v2x_stats", "v2x_flags", "v2x_traffic") + (("lane_change_state",) if lane_change else ()):
        assert got[k].tobytes() == want[k].tobytes(), (what, k)
    if metrics:
        check_rows(got["metrics"], want["metrics"], what, rec=got["rec"])
    t = got["v2x_traffic"]
    assert (t["line_steps"] + t["ped_steps"]).sum() > 0, what
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
def test_gpu_graph_equals_checker(joracle, the_map, kind):
    """4096 worlds as ONE graph launch, replayed three times from the same initial world; obey 1 and 0"""
    gpu_vs_checker(joracle, the_map, kind, 4096, tparams(), repeat=3)
    gpu_vs_checker(joracle, the_map, kind, 4096, tparams(obey=0), metrics=False)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
def test_gpu_direct_launches_and_group_kernel(joracle, the_map, kind, env):
    gpu_vs_checker(joracle, the_map, kind, 4096, tparams(b_commit=3.0, ped_half_width=1.5), env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
def test_gpu_with_lane_changes(joracle, the_map, kind):
    """the LANECHG instances, metrics armed and not"""
    gpu_vs_checker(joracle, the_map, kind, 4096, tparams(), lane_change=True)
    gpu_vs_checker(joracle, the_map, kind, 1024, tparams(obey=0), lane_change=True, metrics=False, seed0=3000)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def host(t, dtype, shape=None):
    a = np.frombuffer(t.cpu().numpy().tobytes(), dtype)
    return a if shape is None else a.reshape(shape)


@pytest.mark.gpu
def test_gpu_arm_disarm_rearm(joracle, the_map):
    """on one context: armed, disarmed (the run without the model, launch for launch), re-armed (the armed run again); disarming the
    V2X events or the agent model underneath disarms it"""
    from dmpp_b200 import scenes
    import torch
    n, kind = 2048, "junction"
    cycles = CYCLES[kind]
    w = jworld(the_map, 900, n, kind=kind)
    ev = scenes.V2xEvents(w, np.arange(900, 900 + n))
    base = dict(agent_model=(amparams(), w.v0), v2x=(vparams(), ev))
    p = planner_with(the_map, n, 10, 60)
    try:
        c0 = p.launch_count(); off = p.run_closed_loop(w.hdr, w.agents, cycles, **base); n_off = p.launch_count() - c0
        c0 = p.launch_count(); a = p.run_closed_loop(w.hdr, w.agents, cycles, traffic=tparams(), **base); n_on = p.launch_count() - c0
        b = p.run_closed_loop(w.hdr, w.agents, cycles, **base)
        c = p.run_closed_loop(w.hdr, w.agents, cycles, traffic=tparams(), **base)
        # disarming underneath: V2X, then the agent model
        d_ts = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
        d_v0, d_spec = dev(w.v0), dev(ev.spec)
        d_s = torch.zeros(n * 80, dtype=torch.uint8, device="cuda")
        p.set_agent_model(amparams(), d_v0.data_ptr())
        p.set_v2x_world(vparams(), n, d_spec.data_ptr(), None, None, 0, None, d_s.data_ptr())
        p.set_v2x_traffic(tparams(), d_ts.data_ptr())
        p.set_v2x_world(None, 0, None)
        p.set_v2x_world(vparams(), n, d_spec.data_ptr(), None, None, 0, None, d_s.data_ptr())
        d_h, d_a = dev(w.hdr), dev(w.agents)
        d_x, d_y = torch.zeros(n * 10, dtype=torch.float64, device="cuda"), torch.zeros(n * 10, dtype=torch.float64, device="cuda")
        d_ts.fill_(0xAB)
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None)   # placement: the rows are not touched
        torch.cuda.synchronize()
        untouched_v2x = (d_ts == 0xAB).all().item()
        p.set_v2x_traffic(tparams(), d_ts.data_ptr())
        p.set_agent_model(None, None)
        p.set_agent_model(amparams(), d_v0.data_ptr())
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None)
        torch.cuda.synchronize()
        untouched_am = (d_ts == 0xAB).all().item()
        p.set_v2x_traffic(tparams(), d_ts.data_ptr())       # armed again: the placement step initialises the rows
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None)
        torch.cuda.synchronize()
        rows = host(d_ts, __import__("dmpp_b200").abi.v2x_traffic_stats)
        p.set_agent_model(None, None); p.set_v2x_world(None, 0, None)
    finally:
        p.close()
    assert a["graph"] and b["graph"] and c["graph"] and off["graph"] and n_on == n_off
    for k in WORLD + ("v2x_stats",):
        assert b[k].tobytes() == off[k].tobytes(), k
        assert c[k].tobytes() == a[k].tobytes(), k
    assert c["v2x_traffic"].tobytes() == a["v2x_traffic"].tobytes() and a["agents"].tobytes() != off["agents"].tobytes()
    assert untouched_v2x and untouched_am
    assert (rows["red_runs"] == 0).all() and np.isinf(rows["min_ped_dist"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
def test_gpu_stepping_by_hand_equals_graph(joracle, the_map, kind):
    """placement, then per cycle dp_cycle_batch_dev -> dp_v2x_world_dev -> dp_world_step_dev (whose t is the cycle of that V2X
    launch), then the tally: the graph's result"""
    import torch
    from dmpp_b200 import abi, scenes
    n, cycles = 1024, CYCLES[kind]
    w = jworld(the_map, 300, n, kind=kind)
    ev = scenes.V2xEvents(w, np.arange(300, 300 + n))
    p = planner_with(the_map, n, 10, scenes.World.PRE_JUNCTION_PTS[kind])
    try:
        graph = p.run_closed_loop(w.hdr, w.agents, cycles, agent_model=(amparams(), w.v0), v2x=(vparams(), ev), traffic=tparams())
        d_h, d_a, d_v0 = dev(w.hdr), dev(w.agents), dev(w.v0)
        d_x, d_y = torch.zeros(n * 10, dtype=torch.float64, device="cuda"), torch.zeros(n * 10, dtype=torch.float64, device="cuda")
        d_rec = torch.zeros(cycles * n * 128, dtype=torch.uint8, device="cuda")
        d_spec, d_wx, d_wy = dev(ev.spec), dev(np.append(ev.wp_x, 0.0)), dev(np.append(ev.wp_y, 0.0))
        d_s = torch.zeros(n * 80, dtype=torch.uint8, device="cuda")
        d_ts = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
        p.set_agent_model(amparams(), d_v0.data_ptr())
        p.set_v2x_world(vparams(), n, d_spec.data_ptr(), d_wx.data_ptr(), d_wy.data_ptr(), ev.wp_x.size, None, d_s.data_ptr())
        p.set_v2x_traffic(tparams(), d_ts.data_ptr())
        p.reset(0, n)
        torch.cuda.synchronize()
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None)
        for k in range(cycles):
            r = d_rec.data_ptr() + k * n * 128
            p.cycle_dev(n, d_h.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), r)
            p.v2x_world_dev(n, d_h.data_ptr(), r, k)
            p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), r)
        p.v2x_world_dev(n, d_h.data_ptr(), None, cycles)
        torch.cuda.synchronize()
        p.set_v2x_traffic(None, None); p.set_v2x_world(None, 0, None); p.set_agent_model(None, None)
    finally:
        p.close()
    assert host(d_rec, abi.plan_record, (cycles, n)).tobytes() == graph["rec"].tobytes()
    assert host(d_h, abi.scene_hdr).tobytes() == graph["hdr"].tobytes()
    assert host(d_a, abi.agent, (n, 10)).tobytes() == graph["agents"].tobytes()
    assert host(d_s, abi.v2x_episode_stats).tobytes() == graph["v2x_stats"].tobytes()
    assert host(d_ts, abi.v2x_traffic_stats).tobytes() == graph["v2x_traffic"].tobytes()


@pytest.mark.gpu
def test_gpu_bad_arguments(the_map):
    import torch
    from dmpp_b200 import scenes
    n = 16
    w = jworld(the_map, 0, n, kind="junction")
    ev = scenes.V2xEvents(w, np.arange(n))
    p = planner_with(the_map, n, 10, 60)
    lib = p.lib
    try:
        d_ts = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
        d_v0, d_spec = dev(w.v0), dev(ev.spec)
        d_s = torch.zeros(n * 80, dtype=torch.uint8, device="cuda")

        def arm(tp):
            return lib.dp_world_set_v2x_traffic(p.ctx, C.byref(tp), C.c_void_p(d_ts.data_ptr()))

        assert arm(tparams()) == -1                         # neither the agent model nor V2X armed
        p.set_agent_model(amparams(), d_v0.data_ptr())
        assert arm(tparams()) == -1                         # V2X not armed
        p.set_agent_model(None, None)
        p.set_v2x_world(vparams(), n, d_spec.data_ptr(), None, None, 0, None, d_s.data_ptr())
        assert arm(tparams()) == -1                         # the agent model not armed
        p.set_agent_model(amparams(), d_v0.data_ptr())
        for kw in (dict(b_commit=0.0), dict(b_commit=-1.0), dict(b_commit=float("nan")), dict(ped_half_width=-0.1),
                   dict(ped_half_width=float("inf")), dict(obey=2), dict(obey=-1)):
            assert arm(tparams(**kw)) == -1, kw
        assert lib.dp_world_set_v2x_traffic(p.ctx, None, C.c_void_p(d_ts.data_ptr())) == -1
        assert arm(tparams(ped_half_width=0.0)) == 0 and arm(tparams(obey=0)) == 0
        d_h, d_a = dev(w.hdr), dev(w.agents)
        d_x, d_y = torch.zeros((n + 1) * 10, dtype=torch.float64, device="cuda"), torch.zeros((n + 1) * 10, dtype=torch.float64, device="cuda")
        assert lib.dp_world_step_dev(p.ctx, 0, n + 1, C.c_void_p(d_h.data_ptr()), C.c_void_p(d_a.data_ptr()), C.c_void_p(d_x.data_ptr()),
                                     C.c_void_p(d_y.data_ptr()), None, None) == -1   # more scenes than the armed specifications
        assert lib.dp_world_set_v2x_traffic(p.ctx, None, None) == 0                   # disarm
        with pytest.raises(AssertionError):
            p.run_closed_loop(w.hdr, w.agents, 4, traffic=tparams())
    finally:
        p.close()
