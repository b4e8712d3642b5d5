"""Reactive agents in closed-loop episodes (include/dmpp_b200.h section 12): at the start of every world step each agent adapts
its speed to the nearest vehicle ahead of it on its lane chain, the ego included, with the intelligent driver model.

The specification is tools/junction_oracle/agent_model.cpp.  CPU side: layout and defaults, known answers on a straight one-lane
road and across a connector, opt-out agents and identity with the model disarmed, an independent numpy restatement of the react
phase, and the effect the model is for (fewer agents driving into the ego from behind).  GPU side: the REACT instances of the
world step against the checker, byte for byte."""
import ctypes as C

import numpy as np
import pytest

from worlds import (DT, WORLD, StraightRoad, amparams, cump_of, first_strikes, gpu_vs_checker, idm, joracle, jparams,  # noqa: F401
                    jworld, mparams, planner_with)


# ---------------------------------------------------------------- CPU: layout and defaults
def test_layout_and_defaults(joracle):
    from dmpp_b200 import abi
    assert joracle.agent_model_sizeof() == C.sizeof(abi.AgentModelParams) == 64
    p = amparams()                                          # through dp_agent_model_default_params: no GPU needed
    assert (p.a_max, p.b, p.b_max, p.T, p.s0, p.length, p.ego_rear, p.look) == (1.0, 1.5, 8.0, 1.5, 2.0, 4.5, 1.0, 100.0)


# ---------------------------------------------------------------- CPU: known answers on a straight lane
@pytest.fixture
def straight(joracle, the_map):
    joracle.set_map(StraightRoad(6000))
    yield joracle
    joracle.set_map(the_map)


def scene(ego_x, xs, vs, v_kmh=0.0):
    """one world: a standing (or moving) ego at ego_x heading +x, agents at xs with speeds vs; a straight carried path"""
    from dmpp_b200 import abi
    h = np.zeros(1, abi.scene_hdr)
    h["x"], h["dir"], h["velocity"], h["period_ms"] = ego_x, 0.0, v_kmh, 1000 * DT
    h["road_num"], h["lane_num"], h["next_roadnum"], h["conn"] = 1, 1, 1, -1
    h["id"][:, 0] = int(round(ego_x / 0.5))
    h["n_obs"] = len(xs)
    ag = np.zeros((1, len(xs)), abi.agent)
    for k, x in enumerate(xs):
        ag["i"][0, k] = int(x // 0.5)
        ag["u"][0, k] = x - 0.5 * int(x // 0.5)
    ag["v"][0] = vs
    rec = np.zeros(1, abi.plan_record)
    rec["brakespeed"], rec["afresh_planning"], rec["behavior"] = v_kmh / 3.6, 1, 1
    lp = np.zeros((1, 2, 200))
    lp[:, 0] = ego_x + 0.5 * np.arange(200)
    return h, ag, rec, lp


def station(ag, k):
    return 0.5 * ag["i"][0, k] + ag["u"][0, k]             # exact on this map: every segment is 0.5 m


def test_free_agent_gains_idm_acceleration(straight):
    o, p = straight, amparams()
    h, ag, _, _ = scene(10.0, [200.0, 350.0], [9.0, 12.0])   # 150 m apart: beyond `look`
    v0 = np.array([[13.5, 12.0]])
    o.react_step(h, ag, v0, p)
    assert ag["v"][0, 0] == idm(9.0, 13.5, p)
    assert abs(ag["v"][0, 0] - (9.0 + p.a_max * (1.0 - (9.0 / 13.5) ** 4) * DT)) < 1e-12
    assert ag["v"][0, 1] == 12.0                            # at its desired speed: keeps it


def test_stops_behind_standing_ego(straight):
    """an agent 40 m behind a standing ego at 10 m/s: it stops with its point behind the ego's rear by >= s0 - 0.5 m and never
    enters the metrics box in 600 steps"""
    from dmpp_b200 import abi
    o, p, mp = straight, amparams(), mparams()
    h, ag, rec, lp = scene(100.0, [60.0], [10.0])
    met = np.zeros(1, abi.episode_metrics)
    ox, oy = np.zeros((1, 1)), np.zeros((1, 1))
    o.metrics_step(h, ag, ox, oy, met, mp)                  # placement
    for _ in range(600):
        o.react_step(h, ag, np.array([[10.0]]), p)
        o.metrics_step(h, ag, ox, oy, met, mp, rec=rec, last_path=lp)
    assert h["x"][0] == 100.0 and ag["v"][0, 0] == 0.0
    assert ox[0, 0] <= 100.0 - mp.rear - (p.s0 - 0.5)
    assert met["collision_steps"][0] == 0 and met["steps"][0] == 600


def test_follower_settles_at_equilibrium_spacing(straight):
    """a follower behind a leader cruising at v < v0 settles to (s0 + v T) / sqrt(1 - (v/v0)^4) + length, within 1 %"""
    o, p = straight, amparams()
    v, v0 = 5.0, 15.0
    h, ag, rec, lp = scene(5.0, [40.0, 80.0], [v, v])       # the ego stands behind both: it is nobody's leader
    speeds = np.array([[v0, v]])                            # the leader is at its desired speed
    ox, oy = np.zeros((1, 2)), np.zeros((1, 2))
    for _ in range(1500):
        o.react_step(h, ag, speeds, p)
        o.world_step(h, ag, ox, oy, rec=rec, last_path=lp)
    want = (p.s0 + v * p.T) / np.sqrt(1 - (v / v0) ** 4) + p.length
    got = station(ag, 1) - station(ag, 0)
    assert ag["v"][0, 1] == v and abs(ag["v"][0, 0] - v) < 1e-3
    assert abs(got - want) <= 0.01 * want, (got, want)


def test_overlapping_leader_gives_hardest_braking(straight):
    o, p = straight, amparams()
    h, ag, _, _ = scene(10.0, [200.0, 203.0], [10.0, 10.0])   # 3 m apart: g = 3 - 4.5 <= 0
    o.react_step(h, ag, np.array([[10.0, 10.0]]), p)
    assert ag["v"][0, 0] == 10.0 - p.b_max * DT == idm(10.0, 10.0, p, g=-1.5, vl=10.0)
    assert ag["v"][0, 1] == 10.0


def test_ties_in_station(straight):
    """equal stations: the higher index is ahead of the lower one; equal gaps: the ego wins, then the lowest agent index"""
    o, p = straight, amparams()
    h, ag, _, _ = scene(10.0, [200.0, 200.0], [10.0, 10.0])
    o.react_step(h, ag, np.array([[12.0, 12.0]]), p)
    assert ag["v"][0, 0] == idm(10.0, 12.0, p, g=-p.length, vl=10.0)   # agent 1 counts as its leader, 0 m ahead
    assert ag["v"][0, 1] == idm(10.0, 12.0, p)                         # agent 0 does not count for agent 1
    # ego at 100 (g = 50 - 1.0) against agent 1 at 103.5 (g = 53.5 - 4.5): the ego leads
    h, ag, _, _ = scene(100.0, [50.0, 103.5], [10.0, 3.0])
    o.react_step(h, ag, np.array([[12.0, 0.0]]), p)
    assert ag["v"][0, 0] == idm(10.0, 12.0, p, g=49.0, vl=0.0) != idm(10.0, 12.0, p, g=49.0, vl=3.0)
    # two agents at the same gap: the lower index leads
    h, ag, _, _ = scene(10.0, [50.0, 80.0, 80.0], [10.0, 4.0, 6.0])
    o.react_step(h, ag, np.array([[12.0, 0.0, 0.0]]), p)
    assert ag["v"][0, 0] == idm(10.0, 12.0, p, g=30.0 - p.length, vl=4.0)
    # the ego at the agent's own station counts (s_e >= s_k); beyond `look` nothing counts
    h, ag, _, _ = scene(200.0, [200.0, 20.0], [10.0, 10.0])
    o.react_step(h, ag, np.array([[12.0, 12.0]]), p)
    assert ag["v"][0, 0] == idm(10.0, 12.0, p, g=-p.ego_rear, vl=0.0) and ag["v"][0, 1] == idm(10.0, 12.0, p)


# ---------------------------------------------------------------- CPU: across a connector
def connector_case(the_map):
    """an approach lane gl with the connector c that follows it (lane_next), and the connector's index cc"""
    m = the_map
    cc = 0
    c = int(m.conn["lane"][cc])
    gl = int(m.road_lane_base[m.conn["last_road"][cc] - 1] + m.conn["last_lane"][cc] - 1)
    return gl, c, cc


def test_brakes_for_agent_and_ego_on_the_next_connector(joracle, the_map):
    from dmpp_b200 import abi
    m, p = the_map, amparams()
    gl, c, cc = connector_case(the_map)
    assert joracle.lane_next()[gl] == c
    cump = cump_of(m)
    cnt = int(m.lane_pt_off[gl + 1] - m.lane_pt_off[gl])
    wp = jparams(joracle)
    w = jworld(the_map, 0, 1)
    h = w.hdr.copy()
    h["road_num"], h["lane_num"], h["pos"], h["n_obs"] = 7, 1, 0, 2   # the ego far away on the departure road
    h["id"][0] = 300
    ag = np.zeros((1, 2), abi.agent)
    ag["lane"], ag["i"], ag["u"], ag["v"] = [[gl, c]], [[cnt - 10, 6]], [[0.1, 0.0]], [[10.0, 0.0]]
    v0 = np.array([[10.0, 0.0]])
    a1 = ag.copy()
    dt = h["period_ms"][0] / 1000.0
    joracle.react_step(h, a1, v0, p, wp=wp)
    sk = cump[m.lane_pt_off[gl] + cnt - 10] + 0.1
    ds = (cump[m.lane_pt_off[gl] + cnt - 1] - sk) + cump[m.lane_pt_off[c] + 6]
    assert ds < p.look and a1["v"][0, 0] == idm(10.0, 10.0, p, g=ds - p.length, vl=0.0, dt=dt) < 10.0
    assert a1["v"][0, 1] == 0.0
    # the ego in pos 2 on that connector, at index 6 (id[last_lanenum-1]), the agent on the connector opted out and moved away
    h2 = h.copy()
    h2["pos"], h2["conn"], h2["last_lanenum"], h2["last_roadnum"] = 2, cc, m.conn["last_lane"][cc], m.conn["last_road"][cc]
    h2["id"][0, :] = 6
    h2["velocity"] = 18.0
    a2 = ag.copy()
    a2["lane"][0, 1] = gl
    a2["i"][0, 1] = 0
    joracle.react_step(h2, a2, v0, p, wp=wp)
    assert a2["v"][0, 0] == idm(10.0, 10.0, p, g=ds - p.ego_rear, vl=18.0 / 3.6, dt=dt) < 10.0
    # the same header with junctions off reads pos 0: the ego is on lane 1 of road 7 at index 6, two hops down the chain
    le = int(m.road_lane_base[6])
    assert joracle.lane_next()[c] == le
    a3 = ag.copy()
    a3["lane"][0, 1], a3["i"][0, 1] = gl, 0
    joracle.react_step(h2, a3, v0, p, wp=jparams(joracle, "highway"))
    d2 = ds - cump[m.lane_pt_off[c] + 6] + cump[m.lane_pt_off[c + 1] - 1]
    assert a3["v"][0, 0] == idm(10.0, 10.0, p, g=(d2 + cump[m.lane_pt_off[le] + 6]) - p.ego_rear, vl=18.0 / 3.6, dt=dt) != a2["v"][0, 0]


# ---------------------------------------------------------------- CPU: opt-out and identity
def closed(joracle, the_map, kind, n, cycles, v0=None, seed0=0):
    from dmpp_b200 import scenes
    w = scenes.World(the_map, np.arange(seed0, seed0 + n), kind=kind)
    wp = jparams(joracle, kind)
    am = None if v0 is None else (amparams(), v0(w))
    return w, joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=wp, threads=8, metrics=mparams(), agent_model=am)


@pytest.mark.parametrize("kind,cycles", [("highway", 25), ("junction", 120)])
def test_all_opted_out_is_the_disarmed_loop(joracle, the_map, kind, cycles):
    _, off = closed(joracle, the_map, kind, 256, cycles)
    v0 = lambda w: np.where(np.arange(w.v0.size).reshape(w.v0.shape) % 3 == 0, np.nan, -w.v0 * (np.arange(w.v0.shape[1]) % 2))
    _, on = closed(joracle, the_map, kind, 256, cycles, v0)
    for k in WORLD + ("metrics",):
        assert on[k].tobytes() == off[k].tobytes(), k


def test_opted_out_agents_keep_their_speed(joracle, the_map):
    def v0(w):
        v = w.v0.copy()
        v[:, ::2] = 0.0
        return v
    w, on = closed(joracle, the_map, "junction", 256, 120, v0)
    assert on["agents"]["v"][:, ::2].tobytes() == w.agents["v"][:, ::2].tobytes()
    assert (on["agents"]["v"][:, 1::2] != w.agents["v"][:, 1::2]).mean() > 0.5


# ---------------------------------------------------------------- CPU: an independent restatement
def restate(m, cump, nxt, wp, p, h, ag, v0):
    """the react phase of section 12 in plain Python / numpy float64, one scene"""
    n = min(int(h["n_obs"]), ag.shape[0])
    off = m.lane_pt_off
    L = [int(ag["lane"][k]) for k in range(n)]
    S = [cump[off[L[k]] + ag["i"][k]] + ag["u"][k] for k in range(n)]
    V = [ag["v"][k] for k in range(n)]
    length = lambda gl: cump[off[gl + 1] - 1]
    pos = int(h["pos"]) if wp.pre_junction_pts > 0 and h["pos"] in (1, 2) else 0
    le = None
    if pos != 2:
        le, idx = int(m.road_lane_base[h["road_num"] - 1] + h["lane_num"] - 1), int(h["id"][h["lane_num"] - 1])
    elif 0 <= h["conn"] < len(m.conn) and 1 <= h["last_lanenum"] <= 6:
        le, idx = int(m.conn["lane"][h["conn"]]), int(h["id"][h["last_lanenum"] - 1])
    if le is not None:
        cnt = int(off[le + 1] - off[le])
        se = cump[off[le] + min(max(idx, 0), cnt - 1)]
    out = ag["v"].copy()
    for k in range(n):
        if not v0[k] > 0:
            continue
        chain = [(L[k], None)]
        l1 = int(nxt[L[k]])
        if l1 >= 0:
            d1 = length(L[k]) - S[k]
            chain.append((l1, d1))
            l2 = int(nxt[l1])
            if l2 >= 0:
                chain.append((l2, d1 + length(l1)))

        def dist(lane, s, ahead_on_own):
            best = None
            for cl, base in chain:
                if cl != lane:
                    continue
                d = (s - S[k] if ahead_on_own else None) if base is None else base + s
                if d is not None and (best is None or d < best):
                    best = d
            return best
        cands = []                                          # (g, order, speed): the ego is order -1
        if le is not None:
            d = dist(le, se, se >= S[k])
            if d is not None and d <= p.look:
                cands.append((d - p.ego_rear, -1, h["velocity"] / 3.6))
        for j in range(n):
            if j == k:
                continue
            d = dist(L[j], S[j], S[j] > S[k] or (S[j] == S[k] and j > k))
            if d is not None and d <= p.look:
                cands.append((d - p.length, j, V[j]))
        dt = h["period_ms"] / 1000.0
        if cands:
            g, _, vl = min(cands, key=lambda c: (c[0], c[1]))
            out[k] = idm(V[k], v0[k], p, g=g, vl=vl, dt=dt)
        else:
            out[k] = idm(V[k], v0[k], p, dt=dt)
    return out


def test_numpy_restatement_equals_checker(joracle, the_map):
    """10 000 random agent states on the junction map: lanes with and without successors, agents at lane ends, equal stations,
    opted-out agents, egos in pos 0 / 1 / 2 with valid and invalid connectors"""
    m = the_map
    rng = np.random.default_rng(12)
    n, k = 1000, 10
    w = jworld(m, 4000, n)
    h, ag = w.hdr.copy(), w.agents.copy()
    lanes = np.concatenate([np.arange(m.road_lane_base[5], m.road_lane_base[7]), m.conn["lane"].astype(np.int64)])
    ag["lane"] = rng.choice(lanes, (n, k))
    cnt = m.lane_pt_off[ag["lane"] + 1] - m.lane_pt_off[ag["lane"]]
    ag["i"] = np.where(rng.random((n, k)) < 0.2, cnt - 2, rng.integers(0, 1 << 30, (n, k)) % (cnt - 1))
    ag["u"] = np.where(rng.random((n, k)) < 0.2, 0.0, rng.uniform(0, 0.5, (n, k)))
    ag["v"] = np.where(rng.random((n, k)) < 0.1, 0.0, rng.uniform(0, 20, (n, k)))
    dup = rng.random(n) < 0.3                               # equal stations: agent 3 on agent 1's spot
    ag[dup, 3] = ag[dup, 1]
    v0 = rng.uniform(-2, 25, (n, k))
    v0[rng.random((n, k)) < 0.05] = np.nan
    h["n_obs"] = rng.integers(0, k + 1, n)
    h["pos"] = rng.integers(0, 3, n)
    h["conn"] = rng.integers(-1, len(m.conn) + 1, n)
    h["last_lanenum"] = rng.integers(0, 4, n)
    h["id"] = rng.integers(-20, 500, (n, 6))
    h["velocity"] = rng.uniform(0, 60, n)
    wp = jparams(joracle)
    p = amparams(look=150.0)
    got = ag.copy()
    joracle.react_step(h, got, v0, p, wp=wp)
    cump, nxt = cump_of(m), joracle.lane_next()
    want = np.stack([restate(m, cump, nxt, wp, p, h[s], ag[s], v0[s]) for s in range(n)])
    assert got["v"].tobytes() == want.tobytes()
    for f in ("u", "lane", "i", "lat"):
        assert got[f].tobytes() == ag[f].tobytes()
    changed = got["v"] != ag["v"]
    assert changed.mean() > 0.3 and (got["v"] == 0).any()


# ---------------------------------------------------------------- CPU: what the model is for
@pytest.fixture(scope="module")
def runs_512(joracle, the_map):
    out = {}
    for kind, cycles in (("highway", 25), ("junction", 120)):
        w, off = closed(joracle, the_map, kind, 512, cycles)
        _, on = closed(joracle, the_map, kind, 512, cycles, lambda w: w.v0)
        out[kind] = (w, off, on)
    return out


def test_fewer_strikes_from_behind(the_map, runs_512):
    """seeds 0-511, default metrics: the checker counts 71 (highway, 25 cycles) and 163 (junction, 120 cycles) worlds whose first
    collision is with an agent that started behind the ego on its lane; with the model on, 22 and 51"""
    got = {}
    for kind, (w, off, on) in runs_512.items():
        got[kind] = (first_strikes(the_map, w, off["metrics"]), first_strikes(the_map, w, on["metrics"]))
        print(kind, "off", got[kind][0], "on", got[kind][1])
    assert got["highway"][0]["behind"] == 71 and got["junction"][0]["behind"] == 163
    assert got["highway"][1]["behind"] <= 30 and got["junction"][1]["behind"] <= 70


@pytest.mark.parametrize("kind", ["highway", "junction"])
def test_reactive_log_replays_open_loop(oracle, runs_512, kind):
    _, _, on = runs_512[kind]
    rep = oracle.run(on["hdr_log"], on["obs_log_x"], on["obs_log_y"], exhaustive=False, threads=8)
    assert rep["rec"].tobytes() == on["rec"].tobytes()


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind,cycles", [("highway", 25), ("junction", 120)])
def test_gpu_graph_equals_checker(joracle, the_map, kind, cycles):
    """4096 worlds as ONE graph launch, replayed three times from the same initial world; metrics armed too"""
    gpu_vs_checker(joracle, the_map, kind, 4096, cycles, repeat=3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,cycles", [("highway", 25), ("junction", 120)])
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
def test_gpu_direct_launches_and_group_kernel(joracle, the_map, kind, cycles, env):
    gpu_vs_checker(joracle, the_map, kind, 4096, cycles, env=env, metrics=kind == "junction")


@pytest.mark.gpu
def test_gpu_urban_200_agents(joracle, the_map):
    gpu_vs_checker(joracle, the_map, "urban", 256, 120, n_obs=200)


@pytest.mark.gpu
def test_gpu_single_steps_ragged(joracle, the_map):
    """dp_world_step_dev with first > 0: ragged n_obs, agents at lane and connector ends, hop chains, equal stations, mixed opt-out
    agents, egos in pos 0 / 1 / 2, against jo_react_step + the checker's world step"""
    import torch
    from dmpp_b200 import abi
    n, first = 600, 37
    m = the_map
    w = jworld(m, 123, n)
    rng = np.random.default_rng(9)
    w.hdr["n_obs"] = rng.integers(0, 11, n)
    ends = (m.lane_pt_off[w.agents["lane"] + 1] - m.lane_pt_off[w.agents["lane"]]) - 2
    w.agents["i"][::3] = ends[::3]
    c1 = int(m.conn["lane"][1])
    w.agents["lane"][::7, 0] = c1
    w.agents["i"][::7, 0] = int(m.lane_pt_off[c1 + 1] - m.lane_pt_off[c1]) - 2
    w.agents["v"][::5] = 40.0
    dup = rng.random(n) < 0.3
    w.agents[dup, 4] = w.agents[dup, 2]
    q = np.arange(1, n, 4)                                 # egos in pos 2, on connector q % n_conn at index 5
    cq = m.conn[q % len(m.conn)]
    w.hdr["pos"][q], w.hdr["conn"][q] = 2, q % len(m.conn)
    w.hdr["last_roadnum"][q], w.hdr["last_lanenum"][q] = cq["last_road"], cq["last_lane"]
    w.hdr["road_num"][q], w.hdr["lane_num"][q], w.hdr["next_lanenum"][q] = cq["next_road"], cq["next_lane"], cq["next_lane"]
    w.hdr["id"][q] = 5
    v0 = np.where(rng.random(w.v0.shape) < 0.2, 0.0, w.v0 + rng.uniform(-2, 4, w.v0.shape))
    rec = np.zeros(n, abi.plan_record)
    rec["brakespeed"] = rng.uniform(0, 20, n)
    rec["afresh_planning"], rec["behavior"] = 1, 1
    lp = np.zeros((n, 2, 200))
    lp[:, 0] = w.hdr["x"][:, None] + 0.5 * np.arange(200)
    lp[:, 1] = w.hdr["y"][:, None]
    wp, am = jparams(joracle), amparams()
    p = planner_with(m, first + n, 10, 60)
    try:
        p.upload_carry(first, np.zeros(n, abi.carry), lp)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()
        d_h, d_a, d_v0, d_r = dev(w.hdr), dev(w.agents), dev(v0), dev(rec)
        d_x, d_y = torch.zeros(n * 10, dtype=torch.float64, device="cuda"), torch.zeros(n * 10, dtype=torch.float64, device="cuda")
        p.set_agent_model(am, d_v0.data_ptr())
        h, ag, ox, oy = w.hdr.copy(), w.agents.copy(), np.zeros((n, 10)), np.zeros((n, 10))
        joracle.world_step(h, ag, ox, oy, wp=wp)
        p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), None, first=first)
        for _ in range(6):
            joracle.react_step(h, ag, v0, am, wp=wp)
            joracle.world_step(h, ag, ox, oy, rec=rec, last_path=lp, wp=wp)
            p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), first=first)
        torch.cuda.synchronize()
        assert np.frombuffer(d_h.cpu().numpy().tobytes(), abi.scene_hdr).tobytes() == h.tobytes()
        got = np.frombuffer(d_a.cpu().numpy().tobytes(), abi.agent).reshape(n, 10)
        used = np.arange(10)[None, :] < w.hdr["n_obs"][:, None]
        assert got[used].tobytes() == ag[used].tobytes()
        assert (got[~used].tobytes() == w.agents[~used].tobytes())
        assert (got["v"][used] != w.agents["v"][used]).mean() > 0.3 and (h["pos"] == 2).any()
    finally:
        p.set_agent_model(None, None)
        p.close()


@pytest.mark.gpu
def test_gpu_arm_disarm_rearm(the_map):
    """on one context: disarmed episodes are byte-identical to a context that never armed the model; re-arming repeats the armed run"""
    n = 1024
    w = jworld(the_map, 700, n)
    never = planner_with(the_map, n, 10, 60)
    try:
        ref = never.run_closed_loop(w.hdr, w.agents, 60)
    finally:
        never.close()
    p = planner_with(the_map, n, 10, 60)
    try:
        a = p.run_closed_loop(w.hdr, w.agents, 60, agent_model=(amparams(), w.v0))
        b = p.run_closed_loop(w.hdr, w.agents, 60)
        c = p.run_closed_loop(w.hdr, w.agents, 60, agent_model=(amparams(), w.v0))
    finally:
        p.close()
    assert a["graph"] and b["graph"] and c["graph"]
    for k in WORLD:
        assert b[k].tobytes() == ref[k].tobytes(), k
        assert c[k].tobytes() == a[k].tobytes(), k
    assert a["agents"].tobytes() != ref["agents"].tobytes()


@pytest.mark.gpu
def test_gpu_bad_params(the_map):
    from dmpp_b200 import planner
    p = planner_with(the_map, 16, 10, 0)
    lib = p.lib
    try:
        for field, bad in (("a_max", 0.0), ("b", -1.0), ("b_max", float("nan")), ("T", 0.0), ("length", 0.0), ("look", float("inf")),
                           ("s0", -0.1), ("ego_rear", -1.0)):
            assert lib.dp_world_set_agent_model(p.ctx, C.byref(amparams(**{field: bad})), C.c_void_p(16)) == -1, field
        assert lib.dp_world_set_agent_model(p.ctx, None, C.c_void_p(16)) == -1
        assert lib.dp_world_set_agent_model(p.ctx, C.byref(amparams(s0=0.0, ego_rear=0.0)), None) == 0
        assert lib.dp_world_set_agent_model(p.ctx, None, None) == 0
        with pytest.raises(planner.DpError):
            p.set_agent_model(amparams(T=float("nan")), 16)
    finally:
        p.close()
    big = planner.Planner(max_scenes=4, max_obs=2049)
    try:
        assert big.lib.dp_world_set_agent_model(big.ctx, C.byref(amparams()), C.c_void_p(16)) == -1
    finally:
        big.close()
