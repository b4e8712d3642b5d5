"""V2X events in closed-loop episodes (include/dmpp_b200.h section 14; rules frozen in tools/junction_oracle/v2x_world.h).

CPU side: a numpy restatement of the data builder and of the red-crossing rule against the checker on random states; the checker's
flags against oracle/v2x_oracle.cpp (pinned to the unmodified reference by tests/test_v2x.py) on the data it built; the checker's
closed loop with V2X disarmed against today's loop; every flag value and warn_status on the seeded worlds.
GPU side: the closed loop with V2X armed against the checker byte for byte (graph, direct launches, group kernel, every other world
option armed), stepping by hand, arm / disarm / re-arm, the launch count, the replay of the logged headers, bad arguments."""
import ctypes as C
import types
from fractions import Fraction

import numpy as np
import pytest

from worlds import WORLD, amparams, check_closed_loop, check_rows, cump_of, jparams, jworld, joracle, lcparams, mparams, planner_with  # noqa: F401

CYCLES = {"highway": 25, "junction": 120}


def vparams(mode=0, apply=1):
    from dmpp_b200 import abi
    return abi.V2xWorldParams(mode, apply)


def events(the_map, w, seed0=0):
    from dmpp_b200 import scenes
    return scenes.V2xEvents(w, np.arange(seed0, seed0 + w.n))


def closed(joracle, the_map, kind, n, vp, seed0=0):
    w = jworld(the_map, seed0, n, kind=kind)
    ev = events(the_map, w, seed0)
    return w, ev, joracle.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(joracle, kind), threads=16,
                                          v2x=None if vp is None else (vp, ev))


def test_layouts(joracle):
    from dmpp_b200 import abi
    assert joracle.v2x_sizeof() == (abi.v2x_event_spec.itemsize, abi.v2x_episode_stats.itemsize) == (160, 80)
    assert C.sizeof(abi.V2xWorldParams) == 8


# ---------------------------------------------------------------- CPU: the rules, restated
def fma(a, b, c):
    """correctly rounded a * b + c (float(Fraction) rounds once)"""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def restate(m, cump, p, s, h, k):
    """the data builder of section 14 in Python float64, the operations in the order the header writes them; returns
    (fields of dp_v2x_data, d, state, on, ped_on)"""
    t = float(k) * float(h["period_ms"]) / 1000.0
    road, lane, pos = int(h["road_num"]), int(h["lane_num"]), int(h["pos"])
    state = 0
    if s["sig_road"] > 0:
        ph = float(np.fmod(t + float(s["sig_offset"]), float(s["sig_cycle"])))
        if ph < 0:
            ph += float(s["sig_cycle"])
        state = 6 if ph < s["sig_green"] else (7 if ph < float(s["sig_green"]) + float(s["sig_yellow"]) else 3)
    on = bool(s["sig_road"] > 0 and road == s["sig_road"] and pos != 2)
    d = 0.0
    if on:
        gl = m.lane_index(road, lane)
        off, cnt = int(m.lane_pt_off[gl]), int(m.lane_pt_off[gl + 1] - m.lane_pt_off[gl])
        stop = cnt - 1 if (s["sig_stop"] < 0 or s["sig_stop"] > cnt - 1) else int(s["sig_stop"])
        i = min(max(int(h["id"][lane - 1]), 0), cnt - 1)
        d = float(cump[off + stop]) - float(cump[off + i])
    v = dict(spat_state=state, spat_lane_occupied=int(on and d >= 0 and d <= s["sig_range"]), ped_distance=0.0, ped_lat=0.0, ped_lng=0.0,
             ped_direction=int(s["ped_direction"]), rsi_lat=0.0, rsi_lng=0.0, wp_first=0, wp_count=0)
    ped_on = bool(s["has_ped"] and s["ped_t_on"] <= t <= s["ped_t_off"])
    x, y = float(h["x"]), float(h["y"])
    if ped_on:
        tp = t - float(s["ped_t_on"])
        px, py = float(s["ped_x"]) + float(s["ped_vx"]) * tp, float(s["ped_y"]) + float(s["ped_vy"]) * tp
        dx, dy = px - x, py - y
        v.update(ped_distance=float(np.sqrt(dx * dx + dy * dy)), ped_lat=fma(py, p.k_lat, p.lat0), ped_lng=fma(px, p.k_lng, p.lng0))
    near = False
    if s["has_works"]:
        if s["rw_rsi"]:
            v.update(rsi_lat=fma(float(s["rw_y"]), p.k_lat, p.lat0), rsi_lng=fma(float(s["rw_x"]), p.k_lng, p.lng0))
        v.update(wp_first=int(s["wp_first"]), wp_count=int(s["wp_count"]))
        dx, dy = float(s["rw_x"]) - x, float(s["rw_y"]) - y
        near = float(np.sqrt(dx * dx + dy * dy)) <= s["rw_range"]
    v.update(ego_lat=fma(y, p.k_lat, p.lat0), ego_lng=fma(x, p.k_lng, p.lng0))
    v["warn_status"] = 5 if (ped_on and v["ped_distance"] <= s["ped_range"]) else 3 if on else 4 if near else 0
    return v, d, state, on, ped_on


def random_states(the_map, n, rng):
    """headers that name a lane of the map (pos 0 / 1 / 2, indices also outside the lane), specifications with and without each
    event, cycles 1 .. 300"""
    from dmpp_b200 import abi
    m = the_map
    h = np.zeros(n, abi.scene_hdr)
    road = rng.integers(1, m.n_roads + 1, n)
    nl = m.road_lane_base[road] - m.road_lane_base[road - 1]
    lane = 1 + (rng.random(n) * nl).astype(np.int64)
    gl = m.road_lane_base[road - 1] + lane - 1
    cnt = m.lane_pt_off[gl + 1] - m.lane_pt_off[gl]
    idx = (rng.random(n) * (cnt + 20)).astype(np.int64) - 10
    h["road_num"], h["lane_num"], h["pos"] = road, lane, rng.integers(0, 3, n)
    for l in range(abi.LANESUM):
        h["id"][:, l] = idx
    pt = m.lane_pt_off[gl] + np.clip(idx, 0, cnt - 1)
    h["x"], h["y"] = m.x[pt] + rng.normal(0, 3, n), m.y[pt] + rng.normal(0, 3, n)
    h["period_ms"] = rng.integers(80, 121, n).astype(np.float64)
    s = np.zeros(n, abi.v2x_event_spec)
    s["sig_road"] = np.where(rng.random(n) < 0.6, road, np.where(rng.random(n) < 0.5, 0, rng.integers(1, m.n_roads + 1, n)))
    s["sig_stop"] = np.where(rng.random(n) < 0.5, -1, (rng.random(n) * (cnt + 50)).astype(np.int64))
    g, yl, r = rng.uniform(1, 20, n), rng.uniform(0.5, 4, n), rng.uniform(1, 20, n)
    s["sig_green"], s["sig_yellow"], s["sig_red"], s["sig_cycle"] = g, yl, r, g + yl + r
    s["sig_offset"] = rng.uniform(-60, 60, n)
    s["sig_range"] = rng.uniform(0, 300, n)
    s["has_ped"], s["ped_direction"] = rng.random(n) < 0.7, rng.random(n) < 0.5
    s["ped_x"], s["ped_y"] = h["x"] + rng.normal(0, 30, n), h["y"] + rng.normal(0, 30, n)
    s["ped_vx"], s["ped_vy"] = rng.normal(0, 2, n), rng.normal(0, 2, n)
    s["ped_t_on"] = rng.uniform(0, 20, n)
    s["ped_t_off"] = s["ped_t_on"] + rng.uniform(0, 20, n)
    s["ped_range"] = rng.uniform(0, 80, n)
    s["has_works"], s["rw_rsi"] = rng.random(n) < 0.7, rng.random(n) < 0.6
    s["rw_x"], s["rw_y"] = h["x"] + rng.normal(0, 60, n), h["y"] + rng.normal(0, 60, n)
    s["rw_range"] = rng.uniform(0, 100, n)
    s["wp_count"] = rng.integers(0, 4, n)
    s["wp_first"] = rng.integers(0, 20, n)
    return h, s, rng.integers(1, 301, n)


def test_numpy_data_builder_and_red_crossing_equal_checker(joracle, the_map):
    """10 000 random states: every byte of dp_v2x_data, d, the signal state, on / ped_on; and the red-crossing rule of the tally
    from random carried (last_d, last_phase, last_on)"""
    from dmpp_b200 import abi
    rng = np.random.default_rng(14)
    n = 10000
    h, s, k = random_states(the_map, n, rng)
    cump, p = cump_of(the_map), joracle.params
    want = np.zeros(n, abi.v2x_data)
    aux = np.zeros((n, 3))
    for i in range(n):
        v, d, state, on, ped_on = restate(the_map, cump, p, s[i], h[i], int(k[i]))
        for f, x in v.items():
            want[f][i] = x
        aux[i] = d, state, int(on) + 2 * int(ped_on)
        got, gaux = joracle.v2x_data(s[i:i + 1], h[i:i + 1], int(k[i]))
        assert got.tobytes() == want[i:i + 1].tobytes(), (i, got, want[i])
        assert gaux.tobytes() == aux[i:i + 1].tobytes(), (i, gaux, aux[i])
    for f in ("warn_status", "spat_state", "spat_lane_occupied"):
        assert len(np.unique(want[f])) >= (4 if f == "warn_status" else 2), f
    assert (aux[:, 2] % 2 == 1).sum() > 1000 and (aux[:, 2] >= 2).sum() > 1000 and (aux[:, 0] < 0).any()
    # the red-crossing rule: the tally closes the step that started with the carried state
    st = np.zeros(n, abi.v2x_episode_stats)
    st["last_on"] = rng.random(n) < 0.7
    st["last_d"] = np.where(rng.random(n) < 0.1, 0.0, rng.uniform(-5, 40, n))
    st["last_phase"] = rng.choice([0, 3, 3, 6, 7], n)
    st["first_red_crossing"] = np.where(rng.random(n) < 0.5, -1, 3)
    ev = types.SimpleNamespace(spec=s, wp_x=np.zeros(30), wp_y=np.zeros(30))
    got = st.copy()
    joracle.v2x_cycle(vparams(), ev, h, None, 7, got)
    _, aux7 = joracle.v2x_data(s, h, 7)
    cross = st["last_on"].astype(bool) & (st["last_d"] >= 0) & (st["last_phase"] == 3) & ((aux7[:, 2] % 2 == 0) | (aux7[:, 0] < 0))
    assert (got["red_crossings"] == st["red_crossings"] + cross).all()
    assert (got["first_red_crossing"] == np.where(cross & (st["first_red_crossing"] < 0), 6, st["first_red_crossing"])).all()
    assert 500 < cross.sum() < n - 500
    rest = [f for f in abi.v2x_episode_stats.names if f not in ("red_crossings", "first_red_crossing")]
    for f in rest:                                                # the tally changes nothing else
        assert got[f].tobytes() == st[f].tobytes(), f


# ---------------------------------------------------------------- CPU: the checker on the seeded worlds
@pytest.fixture(scope="module")
def runs(joracle, the_map):
    out = {}
    for kind in CYCLES:
        for mode in (0, 1):
            for apply in (0, 1):
                out[kind, mode, apply] = closed(joracle, the_map, kind, 512, vparams(mode, apply))
        out[kind, None] = closed(joracle, the_map, kind, 512, None)
    return out


@pytest.mark.parametrize("kind", list(CYCLES))
@pytest.mark.parametrize("mode", [0, 1])
def test_checker_flags_equal_oracle(oracle, joracle, runs, kind, mode):
    """every logged cycle: the checker's flags are oracle.v2x_event on the data the checker built (pos 0), zero elsewhere"""
    from dmpp_b200 import abi
    w, ev, o = runs[kind, mode, 1]
    wl, wg = joracle.gps(ev.wp_x, ev.wp_y)
    zero = np.zeros(w.n, abi.v2x_flags)
    zero["lng_distance"] = zero["lat_distance"] = 9999
    seen = 0
    for k in range(CYCLES[kind]):
        h = o["hdr_log"][k]
        rec = np.zeros(w.n, abi.plan_record)
        flags = joracle.v2x_cycle(vparams(mode, 0), ev, h, rec, k, np.zeros(w.n, abi.v2x_episode_stats))
        data, _ = joracle.v2x_data(ev.spec, h, k)
        want = oracle.v2x_event(h, data, wl, wg, mode)
        p0 = h["pos"] == 0
        assert flags[p0].tobytes() == want[p0].tobytes(), k
        assert flags[~p0].tobytes() == zero[~p0].tobytes(), k
        seen += p0.sum()
    assert seen > 1000


@pytest.mark.parametrize("kind", list(CYCLES))
def test_checker_disarmed_is_todays_loop(oracle, joracle, runs, kind):
    """V2X disarmed: the checker's loop is the loop it was (against oracle/'s segment-only loop on the highway); observe-only
    (apply = 0) changes nothing either; apply = 1 does"""
    w, _, off = runs[kind, None]
    if kind == "highway":
        want = oracle.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(oracle, kind), threads=16)
        for k in WORLD:
            assert off[k].tobytes() == want[k].tobytes(), k
    for mode in (0, 1):
        obs, on = runs[kind, mode, 0][2], runs[kind, mode, 1][2]
        for k in WORLD:
            assert obs[k].tobytes() == off[k].tobytes(), k
        assert on["rec"].tobytes() != off["rec"].tobytes() and on["hdr"].tobytes() != off["hdr"].tobytes()


def test_every_flag_value_and_warn_status(joracle, runs):
    seen = {"light_cycles": np.zeros(3, int), "construction_cycles": np.zeros(2, int), "pedestrian_cycles": np.zeros(2, int)}
    warn = set()
    for kind in CYCLES:
        for mode in (0, 1):
            w, ev, o = runs[kind, mode, 1]
            st = o["v2x_stats"]
            for f in seen:
                seen[f] += st[f].sum(axis=0)
            assert (st["cycles"] == st["light_cycles"].sum(axis=1)).all() and st["ub_cycles"].sum() == 0
            for k in range(CYCLES[kind]):
                data, _ = joracle.v2x_data(ev.spec, o["hdr_log"][k], k)
                warn |= set(np.unique(data["warn_status"][o["hdr_log"][k]["pos"] == 0]).tolist())
            if kind == "junction":
                assert st["red_crossings"].sum() > 0 and st["stop_cmds"].sum() > 0
            else:
                assert np.isfinite(st["min_ped_distance"]).sum() > 100 and st["creep_cmds"].sum() > 0
    print(seen, warn)
    for f, v in seen.items():
        assert (v > 0).all(), (f, v)
    assert warn == {0, 3, 4, 5}


def test_effect_on_seeds_0_511(runs):
    """the effect table of DESIGN.md section 5, from the checker (mode 0, apply 0 against 1): junction red crossings 188 -> 165 and
    stop commands 2851 -> 5243; highway worlds whose pedestrian comes within 2 m of the ego 41 -> 35"""
    j0, j1 = runs["junction", 0, 0][2]["v2x_stats"], runs["junction", 0, 1][2]["v2x_stats"]
    assert (j0["red_crossings"].sum(), j1["red_crossings"].sum()) == (188, 165)
    assert (j0["stop_cmds"].sum(), j1["stop_cmds"].sum()) == (2851, 5243)
    w, ev, _ = runs["highway", 0, 0]
    ped = ev.spec["has_ped"] == 1
    near = [int((runs["highway", 0, a][2]["v2x_stats"]["min_ped_distance"][ped] < 2.0).sum()) for a in (0, 1)]
    assert near == [41, 35]


# ---------------------------------------------------------------- GPU
def gpu_vs_checker(joracle, the_map, kind, n, vp, env=None, repeat=1, models=False, seed0=0):
    from dmpp_b200 import scenes
    w = jworld(the_map, seed0, n, kind=kind)
    ev = events(the_map, w, seed0)
    kw = dict(metrics=mparams(), agent_model=(amparams(), w.v0), lane_change=lcparams()) if models else {}
    want = joracle.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(joracle, kind), threads=16, v2x=(vp, ev), **kw)
    p = planner_with(the_map, n, 10, scenes.World.PRE_JUNCTION_PTS[kind], env)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], repeat=repeat, v2x=(vp, ev), **kw)
    finally:
        p.close()
    what = "%s %r" % (kind, env)
    assert got["graph"] == (env is None), what
    check_closed_loop(got, want, what)
    assert got["v2x_stats"].tobytes() == want["v2x_stats"].tobytes(), what
    assert got["v2x_flags"].tobytes() == want["v2x_flags"].tobytes(), what
    if models:
        check_rows(got["metrics"], want["metrics"], what, rec=got["rec"])
        assert got["lane_change_state"].tobytes() == want["lane_change_state"].tobytes(), what
    assert got["v2x_stats"]["stop_cmds"].sum() > 0
    return w, ev, got


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
def test_gpu_graph_equals_checker(joracle, the_map, kind):
    """4096 worlds as ONE graph launch, replayed three times from the same initial world"""
    gpu_vs_checker(joracle, the_map, kind, 4096, vparams(0, 1), repeat=3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
def test_gpu_direct_launches_and_group_kernel(joracle, the_map, kind, env):
    gpu_vs_checker(joracle, the_map, kind, 4096, vparams(1, 1), env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
def test_gpu_with_every_world_option(joracle, the_map, kind):
    """metrics, reactive and lane-changing agents armed with the V2X events; mode 1, and observe-only"""
    gpu_vs_checker(joracle, the_map, kind, 4096, vparams(1, 1), models=True)
    gpu_vs_checker(joracle, the_map, kind, 1024, vparams(0, 0), models=True, seed0=5000)


@pytest.mark.gpu
def test_gpu_arm_disarm_rearm_and_launch_count(joracle, the_map):
    """on one context: disarmed episodes are byte-identical to the checker's loop without V2X and take 1 + cycles * 3 kernels (plus
    the carry reset); armed, one more per cycle and the tally; re-arming repeats the armed run"""
    n, kind = 2048, "junction"
    cycles = CYCLES[kind]
    w = jworld(the_map, 900, n, kind=kind)
    ev = events(the_map, w, 900)
    want = joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=jparams(joracle, kind), threads=16)
    p = planner_with(the_map, n, 10, 60)
    try:
        c0 = p.launch_count(); p.reset(0, n); reset = p.launch_count() - c0
        c0 = p.launch_count(); b0 = p.run_closed_loop(w.hdr, w.agents, cycles); off = p.launch_count() - c0
        c0 = p.launch_count(); a = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev)); armed = p.launch_count() - c0
        b = p.run_closed_loop(w.hdr, w.agents, cycles)
        c = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev))
    finally:
        p.close()
    assert a["graph"] and b["graph"] and c["graph"] and b0["graph"]
    assert off == reset + 1 + cycles * 3 and armed == off + cycles + 1, (reset, off, armed)
    check_closed_loop(b0, want, "disarmed")
    for k in WORLD:
        assert b[k].tobytes() == b0[k].tobytes(), k
        assert c[k].tobytes() == a[k].tobytes(), k
    assert c["v2x_stats"].tobytes() == a["v2x_stats"].tobytes()
    assert a["rec"].tobytes() != b0["rec"].tobytes()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def host(t, dtype, shape=None):
    a = np.frombuffer(t.cpu().numpy().tobytes(), dtype)
    return a if shape is None else a.reshape(shape)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
def test_gpu_stepping_by_hand_equals_graph(joracle, the_map, kind):
    """placement, then per cycle dp_cycle_batch_dev -> dp_v2x_world_dev -> dp_world_step_dev, then the tally: the graph's result"""
    import torch
    from dmpp_b200 import abi, scenes
    n, cycles = 1024, CYCLES[kind]
    w = jworld(the_map, 300, n, kind=kind)
    ev = events(the_map, w, 300)
    p = planner_with(the_map, n, 10, scenes.World.PRE_JUNCTION_PTS[kind])
    try:
        graph = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev))
        d_h, d_a = dev(w.hdr), dev(w.agents)
        d_x, d_y = torch.zeros(n * 10, dtype=torch.float64, device="cuda"), torch.zeros(n * 10, dtype=torch.float64, device="cuda")
        d_rec = torch.zeros(cycles * n * 128, dtype=torch.uint8, device="cuda")
        d_spec, d_wx, d_wy = dev(ev.spec), dev(np.append(ev.wp_x, 0.0)), dev(np.append(ev.wp_y, 0.0))
        d_f = torch.zeros(n * 24, dtype=torch.uint8, device="cuda")
        d_s = torch.zeros(n * 80, dtype=torch.uint8, device="cuda")
        p.set_v2x_world(vparams(), n, d_spec.data_ptr(), d_wx.data_ptr(), d_wy.data_ptr(), ev.wp_x.size, d_f.data_ptr(), d_s.data_ptr())
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
        p.set_v2x_world(None, 0, None)
    finally:
        p.close()
    assert host(d_rec, abi.plan_record, (cycles, n)).tobytes() == graph["rec"].tobytes()
    assert host(d_h, abi.scene_hdr).tobytes() == graph["hdr"].tobytes()
    assert host(d_s, abi.v2x_episode_stats).tobytes() == graph["v2x_stats"].tobytes()
    assert host(d_f, abi.v2x_flags).tobytes() == graph["v2x_flags"].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CYCLES))
def test_gpu_log_replay_gives_the_planners_records(joracle, the_map, kind):
    """hdr_log / obs logs through dp_run_episode_dev: the planner's own records; the logged ones differ from them only in brakespeed /
    acc_flag / des_acc, only on the cycles with a stop or creep command, and there as the apply rule says"""
    import torch
    from dmpp_b200 import abi, scenes
    n, cycles = 2048, CYCLES[kind]
    w = jworld(the_map, 0, n, kind=kind)
    ev = events(the_map, w)
    p = planner_with(the_map, n, 10, scenes.World.PRE_JUNCTION_PTS[kind])
    try:
        o = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(vparams(), ev))
        d_h, d_x, d_y = dev(o["hdr_log"]), dev(o["obs_log_x"]), dev(o["obs_log_y"])
        d_r = torch.zeros(cycles * n * 128, dtype=torch.uint8, device="cuda")
        p.reset(0, n)
        p.run_episode_dev(n, cycles, d_h.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr())
        torch.cuda.synchronize()
        rep = host(d_r, abi.plan_record, (cycles, n))
    finally:
        p.close()
    cmd = np.zeros((cycles, n), bool)
    st = np.zeros(n, abi.v2x_episode_stats)
    for k in range(cycles):
        r = rep[k].copy()
        f = joracle.v2x_cycle(vparams(), ev, o["hdr_log"][k], r, k, st)
        stop = (f["pedestrian_flag"] == 1) | (f["light_flag"] == 1)
        cmd[k] = stop | ((f["construction_flag"] == 1) & (rep[k]["brakespeed"] > 3.0))
        assert r.tobytes() == o["rec"][k].tobytes(), k             # logged = the apply rule on the planner's record
    assert rep[~cmd].tobytes() == o["rec"][~cmd].tobytes()
    others = [f for f in abi.plan_record.names if f not in ("brakespeed", "acc_flag", "des_acc")]
    for f in others:
        assert rep[f].tobytes() == o["rec"][f].tobytes(), f
    assert cmd.sum() > 50 and (rep[cmd]["brakespeed"] != o["rec"][cmd]["brakespeed"]).any()


@pytest.mark.gpu
def test_gpu_bad_arguments(the_map):
    import torch
    from dmpp_b200 import abi, scenes
    n = 16
    w = jworld(the_map, 0, n, kind="junction")
    ev = scenes.V2xEvents(w, np.arange(n))
    p = planner_with(the_map, n, 10, 60)
    lib = p.lib
    try:
        d_s = torch.zeros(n * 80, dtype=torch.uint8, device="cuda")
        d_h = dev(w.hdr)

        def arm(spec, vp=vparams(), n_wp=0, stats=True, count=n):
            d_spec = dev(spec)
            return lib.dp_world_set_v2x(p.ctx, C.byref(vp), C.c_int(count), C.c_void_p(d_spec.data_ptr()), None, None, C.c_int(n_wp), None,
                                        C.c_void_p(d_s.data_ptr() if stats else 0))

        assert arm(ev.spec) == 0
        assert lib.dp_v2x_world_dev(p.ctx, 0, n + 1, C.c_void_p(d_h.data_ptr()), None, 1, None) == -1     # more scenes than armed
        assert lib.dp_v2x_world_dev(p.ctx, 0, n, C.c_void_p(d_h.data_ptr()), None, -1, None) == -1
        assert lib.dp_v2x_world_dev(p.ctx, 0, n, None, None, 1, None) == -1
        for field, bad in (("sig_cycle", 15.0), ("sig_green", 0.0), ("sig_red", -6.0), ("sig_offset", float("nan")), ("sig_range", -1.0),
                           ("ped_range", -0.5), ("rw_range", float("inf")), ("ped_x", float("nan")), ("sig_road", 9), ("sig_road", -1),
                           ("sig_stop", -2)):
            s = ev.spec.copy()
            s[field][5] = bad
            assert arm(s) == -1, field
        s = ev.spec.copy()
        s["has_works"][3], s["wp_first"][3], s["wp_count"][3] = 1, 0, 1
        assert arm(s) == -1 and arm(s, n_wp=0) == -1
        assert arm(ev.spec, vp=vparams(2, 1)) == -1 and arm(ev.spec, vp=vparams(0, 2)) == -1
        assert arm(ev.spec, stats=False) == -1 and arm(ev.spec, count=-1) == -1
        assert lib.dp_world_set_v2x(p.ctx, None, 0, None, None, None, 0, None, None) == 0               # disarm
        assert lib.dp_v2x_world_dev(p.ctx, 0, n, C.c_void_p(d_h.data_ptr()), None, 1, None) == -3        # not armed
        with pytest.raises(Exception):
            p.run_closed_loop(w.hdr, w.agents, 4, v2x=(vparams(), types.SimpleNamespace(spec=s, wp_x=np.zeros(0), wp_y=np.zeros(0))))
        assert abi.v2x_event_spec.itemsize == 160
    finally:
        p.close()
