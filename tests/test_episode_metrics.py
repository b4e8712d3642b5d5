"""Closed-loop episode metrics (include/dmpp_b200.h section 11): one 192-byte row per world, accumulated by the world step after
the ego and the agents have moved -- collisions, clearance, lead gap, time to collision, ride comfort, replans.

The specification is tools/junction_oracle/episode_metrics.cpp.  CPU side: layout and defaults, known answers on a straight
one-road map, the metrics only observe, and the rows recomputed independently in numpy from the logs.  GPU side: the armed world
step against the checker, byte for byte."""
import ctypes as C

import numpy as np
import pytest

from worlds import WORLD, StraightRoad, check_closed_loop, check_rows, joracle, jparams, jworld, mparams, planner_with  # noqa: F401


# ---------------------------------------------------------------- CPU: layout and defaults
def test_layout_and_defaults(joracle):
    from dmpp_b200 import abi
    assert joracle.metrics_sizeof() == abi.episode_metrics.itemsize == 192
    assert C.sizeof(abi.MetricsParams) == 40
    p = mparams()                                           # through dp_metrics_default_params: no GPU needed
    assert (p.front, p.rear, p.half_width, p.corridor_half, p.ttc_warn) == (4.0, 1.0, 0.9, 1.1, 2.0)
    assert joracle.sincos_deg(0.0) == (1.0, 0.0)


# ---------------------------------------------------------------- CPU: known answers on a straight road
@pytest.fixture
def straight(joracle, the_map):
    joracle.set_map(StraightRoad(1000))
    yield joracle
    joracle.set_map(the_map)


def straight_scene(n, v_kmh, brakespeed):
    """n egos at x = 100 (point 200), heading 0, 100 ms; records that keep (or command) the speed; a straight carried path"""
    from dmpp_b200 import abi
    h = np.zeros(n, abi.scene_hdr)
    h["x"], h["dir"], h["velocity"], h["period_ms"] = 100.0, 0.0, v_kmh, 100.0
    h["road_num"], h["lane_num"], h["next_roadnum"], h["conn"] = 1, 1, 1, -1
    h["id"][:, 0] = 200
    rec = np.zeros(n, abi.plan_record)
    rec["brakespeed"], rec["afresh_planning"], rec["behavior"] = brakespeed, 1, 1
    lp = np.zeros((n, 2, 200))
    lp[:, 0] = 100.0 + 0.5 * np.arange(200)
    return h, rec, lp


def agents_at(xs, lat=0.0, v=0.0):
    from dmpp_b200 import abi
    ag = np.zeros((len(xs), 1), abi.agent)
    for s, x in enumerate(xs):
        ag["i"][s, 0] = int(x // 0.5)
        ag["u"][s, 0] = x - 0.5 * int(x // 0.5)
    ag["lat"], ag["v"] = lat, v
    return ag


def step(o, h, ag, rec, lp, met, mp=None):
    n = h.shape[0]
    h["n_obs"] = ag.shape[1]
    o.metrics_step(h, ag, np.zeros((n, ag.shape[1])), np.zeros((n, ag.shape[1])), met, mp or mparams(), rec=rec, last_path=lp)


def fresh(o, h, ag):
    from dmpp_b200 import abi
    met = np.zeros(h.shape[0], abi.episode_metrics)
    h["n_obs"] = ag.shape[1]
    o.metrics_step(h, ag, np.zeros(ag.shape, np.float64), np.zeros(ag.shape, np.float64), met, mparams())   # placement
    return met


def test_known_answers_standing_ego(straight):
    """standing ego at x = 100: agents at 102 (inside, ahead), 99.5 (inside, behind), 97 (3 m behind), 110 with lat 1.5 (no lead)"""
    o = straight
    h, rec, lp = straight_scene(4, 0.0, 0.0)
    ag = agents_at([102.0, 99.5, 97.0, 110.0])
    ag["lat"][3, 0] = 1.5
    met = fresh(o, h, ag)
    assert (met["steps"] == 0).all() and np.isinf(met["min_clearance"]).all() and (met["last_behavior"] == -1).all()
    step(o, h, ag, rec, lp, met)
    assert (h["x"] == 100.0).all() and (met["stopped_steps"] == 1).all() and (met["steps"] == 1).all()
    a, b, d, e = met
    assert (a["collision_steps"], a["collision_steps_front"], a["collision_steps_rear"]) == (1, 1, 0)
    assert (a["first_collision_step"], a["first_collision_agent"], a["min_clearance"]) == (1, 0, 0.0)
    assert (b["collision_steps"], b["collision_steps_front"], b["collision_steps_rear"]) == (1, 0, 1)
    assert d["collision_steps"] == 0 and d["first_collision_step"] == -1 and d["min_clearance"] == 2.0
    assert np.isinf(d["min_lead_gap"]) and np.isinf(d["min_ttc"])
    assert e["collision_steps"] == 0 and np.isinf(e["min_lead_gap"]) and e["min_clearance"] == np.sqrt(6.0 * 6.0 + 0.6 * 0.6)
    assert (met["max_accel"] == 0).all() and (met["max_abs_jerk"] == 0).all() and (met["behavior_steps"][:, 1] == 1).all()


def test_known_answers_lead_and_ttc(straight):
    """ego at 36 km/h walks 1 m to x = 101; an agent at 4 m/s walks from 110.6 to 111: gap 6, closing 6 m/s, ttc 1 s"""
    o = straight
    h, rec, lp = straight_scene(1, 36.0, 10.0)
    ag = agents_at([110.6], v=4.0)
    met = fresh(o, h, ag)
    step(o, h, ag, rec, lp, met)
    assert h["x"][0] == 101.0 and h["velocity"][0] == 36.0
    m = met[0]
    assert m["min_lead_gap"] == 6.0 and m["min_ttc"] == 1.0 and m["ttc_warn_steps"] == 1
    assert m["distance"] == 1.0 and m["min_clearance"] == 6.0 and m["collision_steps"] == 0 and m["stopped_steps"] == 0


def test_known_answers_accel_and_jerk(straight):
    """three steps of a speed command clipped by a_max: up, up, down -- against numpy evaluating the same operations"""
    o = straight
    h, rec, lp = straight_scene(1, 0.0, 10.0)
    ag = agents_at([300.0])
    met = fresh(o, h, ag)
    dvm = 3.0 * 3.6 * 0.1
    v = [0.0]
    for bs in (10.0, 10.0, 0.0):
        rec["brakespeed"] = bs
        rec["behavior"] = 1 if bs else 3
        step(o, h, ag, rec, lp, met)
        v.append(max(v[-1] + (dvm if bs * 3.6 > v[-1] else -dvm), 0.0))
    a = [(v[k + 1] - v[k]) / 3.6 / 0.1 for k in range(3)]
    m = met[0]
    assert h["velocity"][0] == v[-1]
    assert m["max_accel"] == max(a) and m["min_accel"] == min(a) and m["min_accel"] < 0
    assert m["max_abs_jerk"] == max(abs(a[1] - a[0]) / 0.1, abs(a[2] - a[1]) / 0.1)
    assert m["last_accel"] == a[2] and m["accel_steps"] == 3 and m["behavior_switches"] == 1
    assert m["behavior_steps"][1] == 2 and m["behavior_steps"][3] == 1 and m["last_behavior"] == 3


def test_placement_resets_dirty_rows(straight):
    from dmpp_b200 import abi
    o = straight
    h, rec, lp = straight_scene(2, 0.0, 0.0)
    h["road_num"][1] = 9                                    # names no road of the map
    ag = agents_at([102.0, 102.0])
    met = np.frombuffer(np.full(2 * 192, 0x5A, np.uint8).tobytes(), abi.episode_metrics).copy()
    want = np.zeros(2, abi.episode_metrics)
    met2 = fresh(o, h.copy(), ag.copy())
    h["n_obs"] = 1
    o.metrics_step(h, ag, np.zeros((2, 1)), np.zeros((2, 1)), met, mparams())
    assert met.tobytes() == met2.tobytes()
    assert (met["pad"] == 0).all() and (met["first_collision_step"] == -1).all() and (met["max_accel"] == -np.inf).all()
    want[:] = met
    step(o, h, ag, rec, lp, met)                            # a step: the invalid header's row (and world) stay as they are
    assert met[1].tobytes() == want[1].tobytes() and met[0]["steps"] == 1


# ---------------------------------------------------------------- CPU: observation only, independent recomputation
@pytest.fixture(scope="module")
def runs_512(joracle, the_map):
    from dmpp_b200 import scenes
    out = {}
    for kind, cycles in (("junction", 120), ("highway", 60)):
        w = jworld(the_map, 0, 512, kind=kind) if kind != "highway" else scenes.World(the_map, np.arange(512))
        wp = jparams(joracle, kind)
        on = joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=wp, threads=8, metrics=mparams())
        out[kind] = (w, wp, on)
    return out


@pytest.mark.parametrize("kind", ["junction", "highway"])
def test_metrics_only_observe(joracle, runs_512, kind):
    w, wp, on = runs_512[kind]
    off = joracle.run_closed_loop(w.hdr, w.agents, on["rec"].shape[0], wp=wp, threads=8)
    for k in WORLD:
        assert on[k].tobytes() == off[k].tobytes(), k


def recompute(the_map, joracle, w, wp, o):
    """every field but min_ttc / ttc_warn_steps (they need the agents' speeds, which are not logged), from the logs alone"""
    mp = mparams()
    m = the_map
    H, OX, OY, R = o["hdr_log"], o["obs_log_x"], o["obs_log_y"], o["rec"]
    cycles, n = H.shape
    after = np.concatenate([H[1:], o["hdr"][None]])
    AX, AY = np.concatenate([OX[1:], o["ox"][None]]), np.concatenate([OY[1:], o["oy"][None]])
    lane_size = np.diff(m.lane_pt_off)
    conn = m.conn
    f = {k: np.zeros(n) for k in ("distance", "max_abs_jerk", "last_accel", "max_abs_lat_err", "max_abs_dir_err")}
    f.update(min_clearance=np.full(n, np.inf), min_lead_gap=np.full(n, np.inf), max_accel=np.full(n, -np.inf), min_accel=np.full(n, np.inf))
    ints = ("steps", "collision_steps", "collision_steps_front", "collision_steps_rear", "stopped_steps", "end_stop_steps", "replans",
            "aeb_steps", "accel_steps", "behavior_switches")
    f.update({k: np.zeros(n, np.int64) for k in ints})
    f["first_collision_step"], f["first_collision_agent"], f["last_behavior"] = np.full(n, -1), np.full(n, -1), np.full(n, -1)
    f["behavior_steps"] = np.zeros((n, 8), np.int64)
    sincos = {}
    k_obs = np.arange(OX.shape[2])
    for c in range(cycles):
        h0, h1, r = H[c], after[c], R[c]
        v, vn, dt = h0["velocity"], h1["velocity"], h0["period_ms"] / 1000.0
        gl = m.road_lane_base[h0["road_num"].astype(int) - 1] + h0["lane_num"].astype(int) - 1
        pos = np.where((wp.pre_junction_pts > 0) & ((h0["pos"] == 1) | (h0["pos"] == 2)), h0["pos"], 0)
        has_conn = np.array([((conn["last_road"] == h0["road_num"][s]) & (conn["next_road"] == h0["next_roadnum"][s]) &
                              (conn["last_lane"] == h0["lane_num"][s])).any() and h0["next_roadnum"][s] != h0["road_num"][s] for s in range(n)])
        stop_zone = (wp.pre_junction_pts <= 0) | ((pos == 0) & ~has_conn)
        at_end = stop_zone & (h0["id"][np.arange(n), h0["lane_num"].astype(int) - 1] >= lane_size[gl] - wp.end_margin)
        ds = np.where(at_end, 0.0, (v + vn) * 0.5 / 3.6 * dt)
        for d in np.unique(h1["dir"]):
            if d not in sincos:
                sincos[d] = joracle.sincos_deg(float(d))
        cs = np.array([sincos[d] for d in h1["dir"]])
        cc, ss = cs[:, 0:1], cs[:, 1:2]
        dx, dy = AX[c] - h1["x"][:, None], AY[c] - h1["y"][:, None]
        lon, lat = dx * cc + dy * ss, dy * cc - dx * ss
        alat = np.abs(lat)
        used = k_obs[None, :] < h0["n_obs"][:, None].astype(int)
        inside = used & (-mp.rear <= lon) & (lon <= mp.front) & (-mp.half_width <= lat) & (lat <= mp.half_width)
        ex = np.where(lon > mp.front, lon - mp.front, np.where(lon < -mp.rear, -mp.rear - lon, 0.0))
        ey = np.where(alat > mp.half_width, alat - mp.half_width, 0.0)
        d = np.where(used, np.sqrt(ex * ex + ey * ey), np.inf).min(axis=1)
        lead = used & (lon > mp.front) & (alat <= mp.corridor_half)
        gap = np.where(lead, lon - mp.front, np.inf).min(axis=1)
        f["distance"] = f["distance"] + ds
        f["min_clearance"] = np.minimum(f["min_clearance"], d)
        f["min_lead_gap"] = np.minimum(f["min_lead_gap"], gap)
        a = (vn - v) / 3.6 / dt
        ok = dt > 0
        f["max_accel"] = np.where(ok, np.maximum(f["max_accel"], a), f["max_accel"])
        f["min_accel"] = np.where(ok, np.minimum(f["min_accel"], a), f["min_accel"])
        j = np.abs(a - f["last_accel"]) / dt
        f["max_abs_jerk"] = np.where(ok & (f["accel_steps"] > 0), np.maximum(f["max_abs_jerk"], j), f["max_abs_jerk"])
        f["last_accel"] = np.where(ok, a, f["last_accel"])
        f["accel_steps"] += ok
        f["max_abs_lat_err"] = np.maximum(f["max_abs_lat_err"], np.abs(r["path_lat_dis"]))
        f["max_abs_dir_err"] = np.maximum(f["max_abs_dir_err"], np.abs(r["path_dir_err"]))
        hit = inside.any(axis=1)
        first = np.where(hit, np.argmax(inside, axis=1), -1)
        new = hit & (f["first_collision_step"] < 0)
        f["first_collision_step"] = np.where(new, c + 1, f["first_collision_step"])
        f["first_collision_agent"] = np.where(new, first, f["first_collision_agent"])
        f["collision_steps"] += hit
        f["collision_steps_front"] += (inside & (lon >= 0)).any(axis=1)
        f["collision_steps_rear"] += (inside & (lon < 0)).any(axis=1)
        f["stopped_steps"] += vn == 0
        f["end_stop_steps"] += at_end
        f["replans"] += r["afresh_planning"]
        f["aeb_steps"] += r["acc_flag"]
        b = r["behavior"].astype(int)
        f["behavior_steps"][np.arange(n)[b < 8], b[b < 8]] += 1
        f["behavior_switches"] += (f["steps"] > 0) & (b != f["last_behavior"])
        f["last_behavior"] = b
        f["steps"] += 1
    return f


@pytest.mark.parametrize("kind", ["junction", "highway"])
def test_rows_recomputed_from_logs(the_map, joracle, runs_512, kind):
    w, wp, on = runs_512[kind]
    got = on["metrics"]
    want = recompute(the_map, joracle, w, wp, on)
    for k, v in want.items():
        g = got[k]
        assert (g == v).all(), (kind, k, np.argwhere(g != v)[:3].tolist())


def test_metrics_find_things(runs_512):
    w, wp, on = runs_512["junction"]
    M = on["metrics"]
    print("512 junction worlds x 120 cycles: %d with a collision (%d front, %d rear), %d with a ttc warning, min clearance %.3f m, "
          "%d end stops" % ((M["collision_steps"] > 0).sum(), (M["collision_steps_front"] > 0).sum(), (M["collision_steps_rear"] > 0).sum(),
                            (M["ttc_warn_steps"] > 0).sum(), M["min_clearance"].min(), (M["end_stop_steps"] > 0).sum()))
    assert (M["collision_steps"] > 0).any() and (M["ttc_warn_steps"] > 0).any()
    assert np.isfinite(M["min_clearance"][w.hdr["n_obs"] > 0]).all()
    assert (M["steps"] == 120).all() and (M["first_collision_step"][M["collision_steps"] > 0] >= 1).all()


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,cycles,env", [("highway", 4096, 60, None), ("junction", 4096, 120, None),
                                               ("junction", 4096, 120, {"DP_EPISODE_GRAPH": "0"}),
                                               ("junction", 4096, 120, {"DP_KERNEL": "group"})])
def test_gpu_rows_equal_checker(joracle, the_map, kind, n, cycles, env):
    from dmpp_b200 import scenes
    w = scenes.World(the_map, np.arange(n)) if kind == "highway" else jworld(the_map, 0, n)
    want = joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=jparams(joracle, kind), threads=16, metrics=mparams())
    p = planner_with(the_map, n, 10, scenes.World.PRE_JUNCTION_PTS[kind], env)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, cycles, metrics=mparams())
    finally:
        p.close()
    assert got["graph"] == (env is None)
    check_rows(got["metrics"], want["metrics"], "%s %r" % (kind, env), rec=got["rec"])
    check_closed_loop(got, want, "%s %r" % (kind, env))


@pytest.mark.gpu
def test_gpu_urban_200_agents(joracle, the_map):
    w = jworld(the_map, 0, 256, kind="urban", n_obs=200)
    want = joracle.run_closed_loop(w.hdr, w.agents, 120, wp=jparams(joracle, "urban"), threads=16, metrics=mparams())
    p = planner_with(the_map, 256, 200, 400)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, 120, metrics=mparams())
    finally:
        p.close()
    check_rows(got["metrics"], want["metrics"], "urban", rec=got["rec"])
    check_closed_loop(got, want, "urban")
    assert (got["metrics"]["collision_steps"] > 0).any()


@pytest.mark.gpu
def test_gpu_observation_only_and_replays(the_map):
    w = jworld(the_map, 300, 2048)
    p = planner_with(the_map, 2048, 10, 60)
    try:
        off = p.run_closed_loop(w.hdr, w.agents, 120)
        on = p.run_closed_loop(w.hdr, w.agents, 120, metrics=mparams())
        on3 = p.run_closed_loop(w.hdr, w.agents, 120, repeat=3, metrics=mparams())
    finally:
        p.close()
    for k in WORLD:
        assert on[k].tobytes() == off[k].tobytes() == on3[k].tobytes(), k
    assert on["graph"] and on3["graph"] and on["metrics"].tobytes() == on3["metrics"].tobytes()


@pytest.mark.gpu
def test_gpu_arm_run_disarm_run(the_map):
    import torch
    from dmpp_b200 import abi
    n = 1024
    w = jworld(the_map, 700, n)
    p = planner_with(the_map, n, 10, 60)
    bufs = [torch.full((n * 192,), 0xA5, dtype=torch.uint8, device="cuda") for _ in range(2)]
    rows = lambda b: np.frombuffer(b.cpu().numpy().tobytes(), abi.episode_metrics)
    try:
        p.set_metrics(mparams(), bufs[0].data_ptr())
        a = p.run_closed_loop(w.hdr, w.agents, 40)
        first = rows(bufs[0])
        assert a["graph"] and (first["steps"] == 40).all()
        p.set_metrics(None, None)
        bufs[0].fill_(0x3C)
        torch.cuda.synchronize()
        b = p.run_closed_loop(w.hdr, w.agents, 40)
        assert b["graph"] and (bufs[0] == 0x3C).all().item(), "a disarmed episode wrote metrics"
        assert a["rec"].tobytes() == b["rec"].tobytes()
        p.set_metrics(mparams(), bufs[1].data_ptr())
        p.run_closed_loop(w.hdr, w.agents, 40)
        assert rows(bufs[1]).tobytes() == first.tobytes() and (bufs[0] == 0x3C).all().item()
    finally:
        p.set_metrics(None, None)
        p.close()


@pytest.mark.gpu
def test_gpu_single_steps_ragged(joracle, the_map):
    """dp_world_step_dev with first > 0, mixed n_obs, agents at lane and connector ends, invalid headers, against jo_metrics_step"""
    import torch
    from dmpp_b200 import abi
    n, first = 600, 37
    w = jworld(the_map, 123, n)
    rng = np.random.default_rng(9)
    m = the_map
    w.hdr["n_obs"] = rng.integers(0, 11, n)
    ends = (m.lane_pt_off[w.agents["lane"] + 1] - m.lane_pt_off[w.agents["lane"]]) - 2
    w.agents["i"][::3] = ends[::3]
    c1 = int(m.conn["lane"][1])
    w.agents["lane"][::7, 0] = c1
    w.agents["i"][::7, 0] = int(m.lane_pt_off[c1 + 1] - m.lane_pt_off[c1]) - 2
    w.hdr["road_num"][::11] = 0
    w.hdr["lane_num"][5::13] = 7
    rec = np.zeros(n, abi.plan_record)
    rec["brakespeed"] = rng.uniform(0, 20, n)
    rec["afresh_planning"], rec["behavior"] = 1, rng.integers(0, 9, n)
    rec["path_lat_dis"], rec["acc_flag"] = rng.normal(0, 0.5, n), rng.integers(0, 2, n)
    lp = np.zeros((n, 2, 200))
    lp[:, 0] = w.hdr["x"][:, None] + 0.5 * np.arange(200)
    lp[:, 1] = w.hdr["y"][:, None]
    wp = jparams(joracle)
    mp = mparams()
    p = planner_with(the_map, first + n, 10, 60)
    try:
        p.upload_carry(first, np.zeros(n, abi.carry), lp)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()
        d_h, d_a = dev(w.hdr), dev(w.agents)
        d_x, d_y = torch.zeros(n * 10, dtype=torch.float64, device="cuda"), torch.zeros(n * 10, dtype=torch.float64, device="cuda")
        d_r = dev(rec)
        d_m = torch.full((n * 192,), 0x77, dtype=torch.uint8, device="cuda")
        p.set_metrics(mp, d_m.data_ptr())
        h, ag, ox, oy = w.hdr.copy(), w.agents.copy(), np.zeros((n, 10)), np.zeros((n, 10))
        met = np.frombuffer(np.full(n * 192, 0x77, np.uint8).tobytes(), abi.episode_metrics).copy()
        joracle.metrics_step(h, ag, ox, oy, met, mp, wp=wp)
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None, first=first)
        for _ in range(3):
            joracle.metrics_step(h, ag, ox, oy, met, mp, rec=rec, last_path=lp, wp=wp)
            p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), first=first)
        torch.cuda.synchronize()
        got = np.frombuffer(d_m.cpu().numpy().tobytes(), abi.episode_metrics)
        check_rows(got, met, "single steps")
        assert np.frombuffer(d_h.cpu().numpy().tobytes(), abi.scene_hdr).tobytes() == h.tobytes()
        assert (got["steps"][w.hdr["road_num"] == 0] == 0).all() and (got["steps"] == 3).sum() > n // 2
    finally:
        p.set_metrics(None, None)
        p.close()


@pytest.mark.gpu
def test_gpu_bad_params(the_map):
    from dmpp_b200 import planner
    p = planner_with(the_map, 16, 10, 0)
    lib = p.lib
    try:
        for field, bad in (("front", float("nan")), ("half_width", -0.5), ("half_width", 0.0), ("ttc_warn", float("inf")), ("rear", -1.0)):
            mp = mparams()
            setattr(mp, field, bad)
            assert lib.dp_world_set_metrics(p.ctx, C.byref(mp), C.c_void_p(16)) == -1, field
        assert lib.dp_world_set_metrics(p.ctx, None, C.c_void_p(16)) == -1
        assert lib.dp_world_set_metrics(p.ctx, None, None) == 0
        with pytest.raises(planner.DpError):
            mp = mparams(); mp.corridor_half = float("nan")
            p.set_metrics(mp, 16)
    finally:
        p.close()
