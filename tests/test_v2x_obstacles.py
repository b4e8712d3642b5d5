"""The planner sees the V2X road users (include/dmpp_b200.h section 16; rules frozen in tools/junction_oracle/v2x_obstacles.h).

CPU side: layouts and defaults; a numpy restatement of the view and the row against the checker on random states (capacity drops
and headers that name no lane included); known answers on a straight road; what = 0 against the model disarmed; the logged views
replayed through the open-loop oracle; the effect on the seeded highway worlds.
GPU side: the closed loop with the model armed against the checker byte for byte (graph replays, direct launches, the group kernel,
200-agent urban worlds, every other world option armed), what = 0 against the model disarmed, stepping by hand, arm / disarm /
re-arm, the launch count, bad arguments."""
import ctypes as C
import types

import numpy as np
import pytest

from worlds import W, WORLD, StraightRoad, amparams, check_closed_loop, check_rows, jparams, joracle, lcparams, mparams, planner_with  # noqa: F401

CYCLES = {"highway": 25, "junction": 120, "urban": 120}
N_OBS, MAX_OBS = 10, 14            # the seeded worlds' agents, and room for a pedestrian or a works point and 3 warning points


def vparams(mode=0, apply=1):
    from dmpp_b200 import abi
    return abi.V2xWorldParams(mode, apply)


def oparams(**kw):
    from dmpp_b200 import planner
    return planner.v2x_obstacle_params(**kw)


def tparams(**kw):
    from dmpp_b200 import planner
    return planner.v2x_traffic_params(**kw)


def world(the_map, seed0, n, kind="highway", n_obs=N_OBS, max_obs=MAX_OBS):
    from dmpp_b200 import scenes
    return scenes.World(the_map, np.arange(seed0, seed0 + n), n_obs=n_obs, kind=kind, max_obs=max_obs)


def events(w, seed0=0):
    from dmpp_b200 import scenes
    return scenes.V2xEvents(w, np.arange(seed0, seed0 + w.n))


def used(log, hdr_log):
    """the slots of an obstacle log [cycles][n][max_obs] that the logged views name (the rest are not written)"""
    return np.arange(log.shape[2])[None, None, :] < hdr_log["n_obs"][:, :, None]


def check_views(got, want, what):
    """the logged views: every header byte (check_closed_loop compares named fields), every used slot bit for bit"""
    assert got["hdr_log"].tobytes() == want["hdr_log"].tobytes(), what + " logged views"
    u = used(got["obs_log_x"], want["hdr_log"])
    for k in ("obs_log_x", "obs_log_y"):
        assert (got[k].view(np.uint64)[u] == want[k].view(np.uint64)[u]).all(), what + " " + k


def same_world(a, b, what):
    """two GPU episodes: every WORLD array byte for byte, the final points and the logs over the slots that are written"""
    for k in WORLD:
        if k not in ("ox", "oy", "obs_log_x", "obs_log_y"):
            assert a[k].tobytes() == b[k].tobytes(), what + " " + k
    n_obs = a["hdr"]["n_obs"].max()
    for k in ("ox", "oy"):
        assert a[k][:, :n_obs].tobytes() == b[k][:, :n_obs].tobytes(), what + " " + k
    check_views(a, b, what)


def test_layouts_and_defaults(joracle):
    from dmpp_b200 import abi
    assert joracle.v2x_obstacles_sizeof() == (C.sizeof(abi.V2xObstacleParams), abi.v2x_obstacle_stats.itemsize) == (40, 80)
    p = oparams()
    assert (p.range, p.front, p.rear, p.half_width, p.what, p.pad) == (100.0, 4.0, 1.0, 0.9, 7, 0)
    m = mparams()
    assert (p.front, p.rear, p.half_width) == (m.front, m.rear, m.half_width)            # the metrics' ego box
    assert oparams(what=0, range=5.0).what == 0 and oparams(range=5.0).range == 5.0


# ---------------------------------------------------------------- CPU: the rules, restated
def restate(m, op, max_obs, s, wx, wy, h, ox, oy, prev, k, tally, r, sincos):
    """one obstacles launch of section 16 in Python float64, the operations in the order the header writes them: returns the view
    (header, points of the used slots) or None on the tally, and updates the row r (a numpy record) in place"""
    from dmpp_b200 import abi
    inf = float("inf")
    if k == 0:
        for f in abi.v2x_obstacle_stats.names:
            r[f] = 0
        r["min_ped_clearance"] = r["min_works_clearance"] = inf
        r["first_ped_hit"] = r["first_works_hit"] = r["last_ped_slot"] = -1
    na = min(int(h["n_obs"]), max_obs)
    view = None if tally else (h.copy(), list(ox[:na]), list(oy[:na]))
    road, lane = int(h["road_num"]), int(h["lane_num"])
    if road < 1 or road > m.n_roads or lane < 1 or lane > m.road_lane_base[road] - m.road_lane_base[road - 1] or lane > abi.LANESUM:
        return view
    t = float(k) * float(h["period_ms"]) / 1000.0
    c, sn = sincos(float(h["dir"]))
    x, y = float(h["x"]), float(h["y"])

    def box(px, py):
        dx, dy = px - x, py - y
        lon, lat = dx * c + dy * sn, dy * c - dx * sn
        ex = lon - op.front if lon > op.front else (-op.rear - lon if lon < -op.rear else 0.0)
        ey = abs(lat) - op.half_width if abs(lat) > op.half_width else 0.0
        return (-op.rear <= lon <= op.front and -op.half_width <= lat <= op.half_width), float(np.sqrt(ex * ex + ey * ey))

    def near(px, py):
        dx, dy = px - x, py - y
        return float(np.sqrt(dx * dx + dy * dy)) <= op.range

    if prev is not None and prev["ob_flag"]:
        oi = int(prev["ob_index"])
        r["ped_bound_cycles"] += int(r["last_ped_slot"] >= 0 and oi == r["last_ped_slot"])
        r["works_bound_cycles"] += int(r["last_works_first"] <= oi < r["last_works_end"])
    ped_on = bool(s["has_ped"] and s["ped_t_on"] <= t <= s["ped_t_off"])
    if ped_on:
        tp = t - float(s["ped_t_on"])
        px, py = float(s["ped_x"]) + float(s["ped_vx"]) * tp, float(s["ped_y"]) + float(s["ped_vy"]) * tp
        hit, d = box(px, py)
        if hit:
            r["ped_hits"] += 1
            if r["first_ped_hit"] < 0:
                r["first_ped_hit"] = k
        if d < r["min_ped_clearance"]:
            r["min_ped_clearance"] = d
    wps = [(float(wx[int(s["wp_first"]) + i]), float(wy[int(s["wp_first"]) + i])) for i in range(int(s["wp_count"]))] if s["has_works"] else []
    if s["has_works"]:
        hits = []
        for px_, py_ in [(float(s["rw_x"]), float(s["rw_y"]))] + wps:
            hit, d = box(px_, py_)
            hits.append(hit)
            if d < r["min_works_clearance"]:
                r["min_works_clearance"] = d
        if any(hits):
            r["works_hits"] += 1
            if r["first_works_hit"] < 0:
                r["first_works_hit"] = k
    if tally:
        return None
    hv, vx, vy = view
    cand = []
    if op.what & 1 and ped_on and near(px, py):
        cand.append(("ped", px, py))
    if s["has_works"]:
        if op.what & 2 and near(float(s["rw_x"]), float(s["rw_y"])):
            cand.append(("works", float(s["rw_x"]), float(s["rw_y"])))
        if op.what & 4:
            cand += [("works", a, b) for a, b in wps if near(a, b)]
    ped_slot, dropped, wf = -1, 0, None
    for kind, a, b in cand:
        if kind == "works" and wf is None:
            wf = len(vx)
        if len(vx) < max_obs:
            if kind == "ped":
                ped_slot = len(vx)
            vx.append(a)
            vy.append(b)
        else:
            dropped += 1
    if wf is None:
        wf = len(vx)
    r["views"] += 1
    r["ped_cycles"] += int(ped_slot >= 0)
    r["works_cycles"] += int(len(vx) > wf)
    r["dropped"] += dropped
    r["last_ped_slot"], r["last_works_first"], r["last_works_end"] = ped_slot, wf, len(vx)
    if len(vx) > na:
        hv["n_obs"] = len(vx)
    return hv, vx, vy


def random_states(the_map, n, max_obs, rng):
    """headers that name a lane (and 10 % that do not), random n_obs (also above max_obs), specifications with and without each
    event, warning points and pedestrians near the ego (inside its box too), previous records, carried rows"""
    from dmpp_b200 import abi
    from test_v2x_world import random_states as v2x_states
    h, s, k = v2x_states(the_map, n, rng)
    h["dir"] = rng.uniform(-180, 360, n)
    bad = rng.random(n) < 0.1
    h["road_num"] = np.where(bad & (rng.random(n) < 0.5), 0, h["road_num"])
    h["lane_num"] = np.where(bad, 7, h["lane_num"])
    h["n_obs"] = rng.integers(0, max_obs + 3, n)
    s["ped_x"], s["ped_y"] = h["x"] + rng.normal(0, 4, n), h["y"] + rng.normal(0, 2, n)
    s["ped_t_on"] = np.where(rng.random(n) < 0.5, 0.0, s["ped_t_on"])
    s["rw_x"], s["rw_y"] = h["x"] + rng.normal(0, 30, n), h["y"] + rng.normal(0, 3, n)
    s["wp_first"] = rng.integers(0, 20, n)
    n_wp = 40
    wx, wy = np.zeros((n, n_wp)), np.zeros((n, n_wp))
    wx[:] = h["x"][:, None] + rng.normal(0, 20, (n, n_wp))
    wy[:] = h["y"][:, None] + rng.normal(0, 2, (n, n_wp))
    prev = np.zeros(n, abi.plan_record)
    prev["ob_flag"] = rng.random(n) < 0.7
    prev["ob_index"] = rng.integers(-1, max_obs, n)
    r = np.zeros(n, abi.v2x_obstacle_stats)
    r["last_ped_slot"] = rng.integers(-1, max_obs, n)
    r["last_works_first"] = rng.integers(0, max_obs, n)
    r["last_works_end"] = r["last_works_first"] + rng.integers(0, 4, n)
    r["min_ped_clearance"] = np.where(rng.random(n) < 0.5, np.inf, rng.uniform(0, 5, n))
    r["min_works_clearance"] = np.where(rng.random(n) < 0.5, np.inf, rng.uniform(0, 5, n))
    r["first_ped_hit"] = np.where(rng.random(n) < 0.5, -1, 2)
    r["first_works_hit"] = np.where(rng.random(n) < 0.5, -1, 3)
    k = np.where(rng.random(n) < 0.1, 0, k)
    return h, s, k, wx, wy, prev, r


def test_numpy_view_and_row_equal_checker(joracle, the_map):
    """10 000 random states: the view (header bytes, used slots) and every byte of the row, for random parameters, cycles (0 too),
    tallies and previous records"""
    from dmpp_b200 import abi
    rng = np.random.default_rng(16)
    n, max_obs = 10000, 8
    h, s, k, wx, wy, prev, r0 = random_states(the_map, n, max_obs, rng)
    ox, oy = rng.normal(0, 100, (n, max_obs)), rng.normal(0, 100, (n, max_obs))
    seen = dict(drop=0, ped=0, works=0, noname=0, tally=0, pb=0, wb=0, ph=0, wh=0)
    for i in range(n):
        op = oparams(what=int(rng.integers(0, 8)), range=float(rng.choice([0.0, 15.0, 40.0, 100.0])),
                     front=float(rng.uniform(0, 6)), rear=float(rng.uniform(0, 2)), half_width=float(rng.uniform(0.3, 2)))
        tally = bool(rng.random() < 0.1)
        pv = prev[i:i + 1] if (k[i] > 0 and rng.random() < 0.9) else None
        ev = types.SimpleNamespace(spec=s[i:i + 1], wp_x=wx[i], wp_y=wy[i])
        got = r0[i:i + 1].copy()
        view = (np.zeros(1, abi.scene_hdr), np.full((1, max_obs), -7.0), np.full((1, max_obs), -7.0))
        gv = joracle.v2x_obstacles_view(op, ev, h[i:i + 1], ox[i:i + 1], oy[i:i + 1], int(k[i]), got, prev=pv, tally=tally, view=view)
        want = r0[i:i + 1].copy()
        wv = restate(the_map, op, max_obs, s[i], wx[i], wy[i], h[i], ox[i], oy[i], None if pv is None else pv[0], int(k[i]), tally, want[0],
                     joracle.sincos_deg)
        assert got.tobytes() == want.tobytes(), (i, got, want)
        if tally:
            seen["tally"] += 1
            assert (gv[1] == -7.0).all() and gv[0].tobytes() == np.zeros(1, abi.scene_hdr).tobytes()
            continue
        hv, vx, vy = wv
        assert gv[0][0].tobytes() == hv.tobytes(), i
        nv = len(vx)
        assert (gv[1][0, :nv] == vx).all() and (gv[2][0, :nv] == vy).all() and (gv[1][0, nv:] == -7.0).all(), i
        seen["drop"] += int(want["dropped"][0] > r0["dropped"][i])
        seen["ped"] += int(want["ped_cycles"][0] > r0["ped_cycles"][i])
        seen["works"] += int(want["works_cycles"][0] > r0["works_cycles"][i])
        seen["noname"] += int(want["views"][0] == r0["views"][i] and k[i] > 0)
        seen["pb"] += int(want["ped_bound_cycles"][0] > r0["ped_bound_cycles"][i])
        seen["wb"] += int(want["works_bound_cycles"][0] > r0["works_bound_cycles"][i])
        seen["ph"] += int(want["ped_hits"][0] > r0["ped_hits"][i])
        seen["wh"] += int(want["works_hits"][0] > r0["works_hits"][i])
    print(seen)
    assert all(v >= 50 for v in seen.values()), seen


# ---------------------------------------------------------------- CPU: known answers on a straight road
@pytest.fixture
def road(joracle, the_map):
    def use(lanes=1, attr=0):
        joracle.set_map(StraightRoad(2000, lanes=lanes, attr=attr))
        return joracle
    yield use
    joracle.set_map(the_map)


def straight_world(lanes):
    """one world on StraightRoad: the ego on lane 1 at x = 100 m, 30 km/h, 100 ms cycles, no agents (room for 6 points)"""
    from dmpp_b200 import abi
    h = np.zeros(1, abi.scene_hdr)
    h["x"], h["y"], h["velocity"], h["period_ms"] = 100.0, W * (lanes - 1) / 2, 30.0, 100.0
    h["road_num"], h["lane_num"], h["next_roadnum"], h["conn"] = 1, 1, 1, -1
    h["id"][:, :lanes] = 200
    return h, np.zeros((1, 6), abi.agent)


def test_standing_pedestrian_ahead_stops_the_ego(road):
    """a pedestrian standing in the ego's lane 40 m ahead, V2X flags not applied: perceived, the cycle's local path is bounded by the
    pedestrian's slot and the ego stops short of it; not perceived (what = 0), it drives into it"""
    from dmpp_b200 import abi
    o = road()
    h, ag = straight_world(1)
    s = np.zeros(1, abi.v2x_event_spec)
    s["has_ped"], s["ped_x"], s["ped_t_off"] = 1, 140.0, 1e6
    ev = types.SimpleNamespace(spec=s, wp_x=np.zeros(0), wp_y=np.zeros(0))
    seen = o.run_closed_loop(h, ag, 100, v2x=(vparams(apply=0), ev), obstacles=oparams())
    blind = o.run_closed_loop(h, ag, 100, v2x=(vparams(apply=0), ev), obstacles=oparams(what=0))
    r, rb = seen["v2x_obstacles"][0], blind["v2x_obstacles"][0]
    assert (seen["hdr_log"]["n_obs"] == 1).all() and (seen["obs_log_x"][:, 0, 0] == 140.0).all()
    flagged = seen["rec"]["ob_flag"] == 1
    assert (seen["rec"]["ob_index"][flagged] == 0).all() and flagged.sum() >= 95                 # slot 0: the pedestrian
    # every record is checked once: cycle k - 1's by launch k, the last one by the tally
    assert r["ped_bound_cycles"] == seen["rec"]["ob_flag"].sum() and r["ped_cycles"] == 100 and r["views"] == 100 and r["last_ped_slot"] == 0
    assert seen["hdr"]["velocity"][0] == 0.0 and 140.0 - 4.0 - 5.0 < seen["hdr"]["x"][0] < 140.0 - 4.0
    assert r["ped_hits"] == 0 and r["first_ped_hit"] == -1 and r["min_ped_clearance"] > 1.0
    assert (blind["hdr_log"]["n_obs"] == 0).all() and (blind["rec"]["ob_flag"] == 0).all()
    assert blind["hdr"]["x"][0] > 180.0 and rb["ped_hits"] > 0 and rb["min_ped_clearance"] == 0.0 and rb["ped_bound_cycles"] == 0
    assert rb["ped_cycles"] == 0 and rb["last_ped_slot"] == -1


def test_warning_points_on_the_ego_lane(road):
    """a road-works zone on lane 1 of a two-lane road with lane changes allowed (works point and three warning points 5 m apart): the
    ego leaves the lane or stops before them; without the points it drives through"""
    from dmpp_b200 import abi
    o = road(lanes=2, attr=3)
    h, ag = straight_world(2)
    s = np.zeros(1, abi.v2x_event_spec)
    s["has_works"], s["rw_x"], s["rw_y"], s["wp_count"] = 1, 140.0, W / 2, 3
    ev = types.SimpleNamespace(spec=s, wp_x=np.array([140.0, 145.0, 150.0]), wp_y=np.full(3, W / 2))
    seen = o.run_closed_loop(h, ag, 100, v2x=(vparams(apply=0), ev), obstacles=oparams())
    blind = o.run_closed_loop(h, ag, 100, v2x=(vparams(apply=0), ev), obstacles=oparams(what=0))
    r, rb = seen["v2x_obstacles"][0], blind["v2x_obstacles"][0]
    left_lane = seen["hdr"]["lane_num"][0] != 1
    stopped = seen["hdr"]["velocity"][0] == 0.0 and seen["hdr"]["x"][0] < 140.0 - 4.0
    assert left_lane or stopped
    assert r["works_hits"] == 0 and r["min_works_clearance"] > 1.0 and r["works_bound_cycles"] > 50 and r["works_cycles"] == 100
    assert (seen["hdr_log"]["n_obs"] == 4).all() and r["last_works_first"] == 0 and r["last_works_end"] == 4
    assert blind["hdr"]["x"][0] > 180.0 and rb["works_hits"] > 0 and rb["min_works_clearance"] == 0.0


# ---------------------------------------------------------------- CPU: the checker on the seeded worlds
@pytest.fixture(scope="module")
def runs(joracle, the_map):
    """highway seeds 0-511 x 25 cycles, metrics armed: V2X apply {0, 1} x what {off, 0, 7}"""
    w = world(the_map, 0, 512)
    ev = events(w)
    out = {"w": w, "ev": ev}
    for apply in (0, 1):
        for what in (None, 0, 7):
            out[apply, what] = joracle.run_closed_loop(w.hdr, w.agents, 25, threads=16, metrics=mparams(), v2x=(vparams(0, apply), ev),
                                                       obstacles=None if what is None else oparams(what=what))
    return out


def test_what_0_is_the_model_disarmed(runs):
    for apply in (0, 1):
        off, obs = runs[apply, None], runs[apply, 0]
        for k in WORLD + ("metrics", "v2x_stats", "v2x_flags"):
            assert obs[k].tobytes() == off[k].tobytes(), (apply, k)
        r = obs["v2x_obstacles"]
        assert (r["views"] == 25).all() and r["ped_cycles"].sum() == r["works_cycles"].sum() == r["ped_bound_cycles"].sum() == 0
        assert r["ped_hits"].sum() > 0
        assert runs[apply, 7]["rec"].tobytes() != off["rec"].tobytes()


def test_logged_views_replay_through_the_open_loop_oracle(oracle, runs):
    """apply = 0: the records are the planner's own, so replaying the logged views (hdr_log, obs logs) gives them again"""
    o = runs[0, 7]
    rep = oracle.run(o["hdr_log"], o["obs_log_x"], o["obs_log_y"], exhaustive=True)
    assert rep["rec"].tobytes() == o["rec"].tobytes()
    assert (o["hdr_log"]["n_obs"] > N_OBS).sum() > 1000


def effect(runs, apply, what):
    ev, o = runs["ev"], runs[apply, what]
    r, met = o["v2x_obstacles"], o["metrics"]
    ped, wk = ev.spec["has_ped"] == 1, ev.spec["has_works"] == 1
    clr = r["min_ped_clearance"][ped]
    return dict(ped_hit_worlds=int((r["ped_hits"][ped] > 0).sum()), ped_clear_median=round(float(np.median(clr)), 2),
                ped_clear_min=round(float(clr.min()), 2), ped_under_1m=int((clr < 1.0).sum()),
                works_hit_worlds=int((r["works_hits"][wk] > 0).sum()), works_clear_min=round(float(r["min_works_clearance"][wk].min()), 2),
                b4=int(met["behavior_steps"][:, 4].sum()), b5=int(met["behavior_steps"][:, 5].sum()),
                lane_changes=int(met["behavior_steps"][:, 2:4].sum()), ped_bound=int(r["ped_bound_cycles"].sum()),
                works_bound=int(r["works_bound_cycles"].sum()), collisions=int((met["collision_steps"] > 0).sum()))


def test_effect_on_seeds_0_511(runs):
    """the effect table of DESIGN.md section 5, from the checker (286 pedestrian worlds, 226 road-works worlds)"""
    ev = runs["ev"]
    assert (int(ev.spec["has_ped"].sum()), int(ev.spec["has_works"].sum())) == (286, 226)
    got = {(a, w): effect(runs, a, w) for a in (0, 1) for w in (0, 7)}
    for k, v in got.items():
        print(k, v)
    assert got == EFFECT


# (apply, what) -> the effect figures; collisions = worlds with an agent inside the ego box at some step (section 11)
EFFECT = {
    (0, 0): dict(ped_hit_worlds=31, ped_clear_median=14.37, ped_clear_min=0.0, ped_under_1m=54, works_hit_worlds=7, works_clear_min=0.0,
                 b4=861, b5=776, lane_changes=149, ped_bound=0, works_bound=0, collisions=207),
    (0, 7): dict(ped_hit_worlds=29, ped_clear_median=14.37, ped_clear_min=0.0, ped_under_1m=52, works_hit_worlds=7, works_clear_min=0.0,
                 b4=893, b5=825, lane_changes=134, ped_bound=677, works_bound=284, collisions=209),
    (1, 0): dict(ped_hit_worlds=28, ped_clear_median=15.95, ped_clear_min=0.0, ped_under_1m=50, works_hit_worlds=7, works_clear_min=0.0,
                 b4=859, b5=781, lane_changes=149, ped_bound=0, works_bound=0, collisions=211),
    (1, 7): dict(ped_hit_worlds=28, ped_clear_median=15.95, ped_clear_min=0.0, ped_under_1m=50, works_hit_worlds=7, works_clear_min=0.0,
                 b4=890, b5=830, lane_changes=134, ped_bound=671, works_bound=284, collisions=211),
}


# ---------------------------------------------------------------- GPU
def gpu_vs_checker(joracle, the_map, kind, n, op, vp=None, env=None, repeat=1, models=False, seed0=0, n_obs=N_OBS, max_obs=MAX_OBS):
    """the closed loop with the V2X road users armed, on the GPU against the checker, byte for byte: records, views, world, carry,
    V2X rows and flags, the new rows; with models: metrics, reactive and lane-changing agents, and agents that obey the events"""
    from dmpp_b200 import scenes
    vp = vp or vparams(0, 1)
    w = world(the_map, seed0, n, kind=kind, n_obs=n_obs, max_obs=max_obs)
    ev = events(w, seed0)
    kw = dict(metrics=mparams(), agent_model=(amparams(), w.v0), lane_change=lcparams(), traffic=tparams()) if models else {}
    want = joracle.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(joracle, kind), threads=16, v2x=(vp, ev), obstacles=op, **kw)
    p = planner_with(the_map, n, max_obs, scenes.World.PRE_JUNCTION_PTS[kind], env)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], repeat=repeat, v2x=(vp, ev), obstacles=op, **kw)
    finally:
        p.close()
    what = "%s %r what=%d" % (kind, env, op.what)
    assert got["graph"] == (env is None and max_obs < 32), what   # (from 32 obstacle slots up the cycle runs on the group kernel)
    check_closed_loop(got, want, what)
    check_views(got, want, what)
    for k in ("v2x_stats", "v2x_flags", "v2x_obstacles"):
        assert got[k].tobytes() == want[k].tobytes(), what + " " + k
    if models:
        check_rows(got["metrics"], want["metrics"], what, rec=got["rec"])
        assert got["v2x_traffic"].tobytes() == want["v2x_traffic"].tobytes(), what
        # (the state of a slot beyond the world's agents is never written)
        assert got["lane_change_state"][:, :n_obs].tobytes() == want["lane_change_state"][:, :n_obs].tobytes(), what
    r = got["v2x_obstacles"]
    assert (r["views"] > 0).all()
    if kind == "highway" and op.what == 7:
        assert r["ped_cycles"].sum() > 0 and r["works_cycles"].sum() > 0 and r["ped_bound_cycles"].sum() > 0 and r["works_bound_cycles"].sum() > 0
    return w, ev, got


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["highway", "junction"])
def test_gpu_graph_equals_checker(joracle, the_map, kind):
    """4096 worlds as ONE graph launch, replayed three times from the same initial world"""
    gpu_vs_checker(joracle, the_map, kind, 4096, oparams(), repeat=3)


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
def test_gpu_direct_launches_and_group_kernel(joracle, the_map, env):
    """highway worlds with 12 slots for 10 agents, so that points are dropped; mode 1"""
    _, _, got = gpu_vs_checker(joracle, the_map, "highway", 4096, oparams(), vp=vparams(1, 1), env=env, max_obs=12)
    assert got["v2x_obstacles"]["dropped"].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["highway", "junction"])
def test_gpu_with_every_world_option(joracle, the_map, kind):
    """metrics, reactive and lane-changing agents and agents that obey the V2X events, armed with the road users; observe-only too"""
    gpu_vs_checker(joracle, the_map, kind, 4096, oparams(), models=True)
    gpu_vs_checker(joracle, the_map, kind, 1024, oparams(what=0, range=60.0), vp=vparams(0, 0), models=True, seed0=5000)


@pytest.mark.gpu
def test_gpu_urban_200_agents(joracle, the_map):
    """200 agents per world (the group kernel runs the cycle), urban junction worlds"""
    gpu_vs_checker(joracle, the_map, "urban", 256, oparams(), n_obs=200, max_obs=204)


@pytest.mark.gpu
def test_gpu_what_0_is_the_model_disarmed(joracle, the_map):
    """observe-only: records, views (= the world), world, carry and every other row byte for byte those of the model disarmed"""
    from dmpp_b200 import scenes
    n, kind = 4096, "highway"
    w = world(the_map, 0, n)
    ev = events(w)
    kw = dict(metrics=mparams(), agent_model=(amparams(), w.v0), lane_change=lcparams(), traffic=tparams(), v2x=(vparams(0, 1), ev))
    p = planner_with(the_map, n, MAX_OBS, scenes.World.PRE_JUNCTION_PTS[kind])
    try:
        off = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], **kw)
        obs = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], obstacles=oparams(what=0), **kw)
    finally:
        p.close()
    for k in ("rec", "hdr", "agents", "carry", "last_path", "hdr_log", "metrics", "v2x_stats", "v2x_flags", "v2x_traffic"):
        assert obs[k].tobytes() == off[k].tobytes(), k
    assert obs["lane_change_state"][:, :N_OBS].tobytes() == off["lane_change_state"][:, :N_OBS].tobytes()
    same_world(obs, off, "what 0")
    assert obs["v2x_obstacles"]["ped_hits"].sum() > 0


@pytest.mark.gpu
def test_gpu_arm_disarm_rearm_and_launch_count(joracle, the_map):
    """on one context: V2X alone takes 1 + cycles * 4 + 1 kernels (plus the carry reset), with the road users 1 + cycles * 5 + 2;
    disarming gives the V2X-only episode back, re-arming repeats the armed one; disarming V2X disarms the road users"""
    n, kind = 2048, "highway"
    cycles = CYCLES[kind]
    w = world(the_map, 900, n)
    ev = events(w, 900)
    want = joracle.run_closed_loop(w.hdr, w.agents, cycles, threads=16, v2x=(vparams(), ev), obstacles=oparams())
    p = planner_with(the_map, n, MAX_OBS, 0)
    try:
        c0 = p.launch_count(); p.reset(0, n); reset = p.launch_count() - c0
        c0 = p.launch_count(); v = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev)); v_only = p.launch_count() - c0
        c0 = p.launch_count(); a = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev), obstacles=oparams()); armed = p.launch_count() - c0
        b = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev))
        c = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev), obstacles=oparams())
    finally:
        p.close()
    assert a["graph"] and b["graph"] and c["graph"] and v["graph"]
    assert v_only == reset + 1 + cycles * 4 + 1 and armed == reset + 1 + cycles * 5 + 2, (reset, v_only, armed)
    check_closed_loop(a, want, "armed")
    check_views(a, want, "armed")
    assert a["v2x_obstacles"].tobytes() == want["v2x_obstacles"].tobytes()
    same_world(b, v, "disarmed")
    same_world(c, a, "re-armed")
    assert c["v2x_obstacles"].tobytes() == a["v2x_obstacles"].tobytes()
    assert a["rec"].tobytes() != v["rec"].tobytes()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def host(t, dtype, shape=None):
    a = np.frombuffer(t.cpu().numpy().tobytes(), dtype)
    return a if shape is None else a.reshape(shape)


@pytest.mark.gpu
def test_gpu_stepping_by_hand_equals_graph(joracle, the_map):
    """placement, then per cycle dp_v2x_obstacles_dev -> dp_cycle_batch_dev on the view -> dp_v2x_world_dev -> dp_world_step_dev,
    then the V2X tally and the obstacles tally: the graph's result"""
    import torch
    from dmpp_b200 import abi
    n, cycles, mo = 1024, CYCLES["highway"], MAX_OBS
    w = world(the_map, 300, n)
    ev = events(w, 300)
    p = planner_with(the_map, n, mo, 0)
    try:
        graph = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev), obstacles=oparams())
        d_h, d_a = dev(w.hdr), dev(w.agents)
        z = lambda b: torch.zeros(b, dtype=torch.uint8, device="cuda")
        d_x, d_y = z(n * mo * 8), z(n * mo * 8)
        d_hv, d_vx, d_vy, d_os = z(n * 128), z(n * mo * 8), z(n * mo * 8), z(n * 80)
        d_rec = z(cycles * n * 128)
        d_spec, d_wx, d_wy = dev(ev.spec), dev(np.append(ev.wp_x, 0.0)), dev(np.append(ev.wp_y, 0.0))
        d_f, d_s = z(n * 24), z(n * 80)
        p.set_v2x_world(vparams(), n, d_spec.data_ptr(), d_wx.data_ptr(), d_wy.data_ptr(), ev.wp_x.size, d_f.data_ptr(), d_s.data_ptr())
        p.set_v2x_obstacles(oparams(), d_hv.data_ptr(), d_vx.data_ptr(), d_vy.data_ptr(), d_os.data_ptr())
        p.reset(0, n)
        torch.cuda.synchronize()
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None)
        for k in range(cycles):
            r = d_rec.data_ptr() + k * n * 128
            p.v2x_obstacles_dev(n, d_h.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), r - n * 128 if k > 0 else None, k)
            p.cycle_dev(n, d_hv.data_ptr(), d_vx.data_ptr(), d_vy.data_ptr(), r)
            p.v2x_world_dev(n, d_h.data_ptr(), r, k)
            p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), r)
        p.v2x_world_dev(n, d_h.data_ptr(), None, cycles)
        p.v2x_obstacles_dev(n, d_h.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_rec.data_ptr() + (cycles - 1) * n * 128, cycles, tally=True)
        torch.cuda.synchronize()
        p.set_v2x_world(None, 0, None)
    finally:
        p.close()
    assert host(d_rec, abi.plan_record, (cycles, n)).tobytes() == graph["rec"].tobytes()
    assert host(d_h, abi.scene_hdr).tobytes() == graph["hdr"].tobytes()
    assert host(d_s, abi.v2x_episode_stats).tobytes() == graph["v2x_stats"].tobytes()
    assert host(d_os, abi.v2x_obstacle_stats).tobytes() == graph["v2x_obstacles"].tobytes()
    assert host(d_hv, abi.scene_hdr).tobytes() == graph["hdr_log"][-1].tobytes()     # the last view


@pytest.mark.gpu
def test_gpu_bad_arguments(the_map):
    import torch
    from dmpp_b200 import abi
    n, mo = 16, MAX_OBS
    w = world(the_map, 0, n)
    ev = events(w)
    p = planner_with(the_map, n, mo, 0)
    lib = p.lib
    try:
        z = lambda b: torch.zeros(b, dtype=torch.uint8, device="cuda")
        d_hv, d_vx, d_vy, d_os, d_s = z(n * 128), z(n * mo * 8), z(n * mo * 8), z(n * 80), z(n * 80)
        d_h, d_x = dev(w.hdr), z(n * mo * 8)

        def arm(op=None, hv=True, stats=True):
            return lib.dp_world_set_v2x_obstacles(p.ctx, C.byref(op or oparams()), C.c_void_p(d_hv.data_ptr() if hv else 0),
                                                  C.c_void_p(d_vx.data_ptr()), C.c_void_p(d_vy.data_ptr()),
                                                  C.c_void_p(d_os.data_ptr() if stats else 0))

        def step(count=n, cycle=1, tally=0, hdr=True):
            return lib.dp_v2x_obstacles_dev(p.ctx, 0, count, C.c_void_p(d_h.data_ptr() if hdr else 0), C.c_void_p(d_x.data_ptr()),
                                            C.c_void_p(d_x.data_ptr()), None, C.c_int(cycle), C.c_int(tally), None)

        assert arm() == -1                                                  # V2X not armed
        assert step() == -3                                                 # the model not armed
        d_spec, d_wx, d_wy = dev(ev.spec), dev(np.append(ev.wp_x, 0.0)), dev(np.append(ev.wp_y, 0.0))
        assert lib.dp_world_set_v2x(p.ctx, C.byref(vparams()), C.c_int(n), C.c_void_p(d_spec.data_ptr()), C.c_void_p(d_wx.data_ptr()),
                                    C.c_void_p(d_wy.data_ptr()), C.c_int(ev.wp_x.size), None, C.c_void_p(d_s.data_ptr())) == 0
        for kw in (dict(range=float("nan")), dict(front=float("inf")), dict(range=-1.0), dict(half_width=0.0), dict(front=-0.1),
                   dict(rear=-1.0), dict(what=8), dict(what=-1)):
            assert arm(oparams(**kw)) == -1, kw
        assert arm(hv=False) == -1
        assert arm() == 0 and arm(stats=False) == 0 and arm() == 0                           # arm, disarm (stats NULL), re-arm
        assert step() == 0 and step(tally=1) == 0
        assert step(count=n + 1) == -1 and step(cycle=-1) == -1 and step(tally=2) == -1 and step(hdr=False) == -1
        torch.cuda.synchronize()
        # predicted tracks: the setter refuses them, and so does the episode runner
        vx = np.zeros((n, mo))
        p.set_tracks(vx, vx, vx, 4)
        assert arm() == -3
        p.clear_tracks()
        assert arm() == 0
        p.set_tracks(vx, vx, vx, 4)
        d_ag, d_rec = dev(w.agents), z(4 * n * 128)
        assert lib.dp_run_closed_loop_dev(p.ctx, 0, n, 4, C.c_void_p(d_h.data_ptr()), C.c_void_p(d_ag.data_ptr()), C.c_void_p(d_x.data_ptr()),
                                          C.c_void_p(d_x.data_ptr()), C.c_void_p(d_rec.data_ptr()), None, None, None, None) == -3
        p.clear_tracks()
        # disarming V2X disarms the road users
        assert lib.dp_world_set_v2x(p.ctx, None, 0, None, None, None, 0, None, None) == 0
        assert step() == -3
        with pytest.raises(Exception):
            p.run_closed_loop(w.hdr, w.agents, 4, obstacles=oparams())
    finally:
        p.close()
