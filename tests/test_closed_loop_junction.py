"""Closed-loop episodes through junctions (include/dmpp_b200.h section 9, dp_world_params.pre_junction_pts > 0): the world step
takes the ego through pos 0 -> 1 -> 2 -> 0 along a connector and the agents into the successors of their lanes.

The specification is the junction oracle of tools/junction_oracle (the cycle restatement of oracle/ with the junction world step
between its cycles; with the option off its step IS oracle/world_spec.cpp's).  CPU side: known answers on the synthetic map, the
option switched off is the segment-only step, the loop is alive, and the junction oracle against the UNMODIFIED reference driven
the same way.  GPU side: dp_run_closed_loop_dev against the junction oracle, bit for bit."""
import numpy as np
import pytest

from conftest import assert_records_equal, same
from test_oracle_vs_ref import CARRY, REC
from worlds import HDR, check_closed_loop, joracle, jparams, jworld, planner_with  # noqa: F401  (joracle: the module fixture)


def compressed(seq):
    return [int(seq[0])] + [int(v) for i, v in enumerate(seq[1:]) if v != seq[i]]


# ---------------------------------------------------------------- CPU: known answers
def test_lane_successors(joracle, the_map):
    """approach lane -> its connector (the lowest one leaving it), connector -> its next lane, every other lane -> none"""
    m, o = the_map, joracle
    c = m.conn
    assert [int(x) for x in c["lane"]] == [m.n_lanes - 2, m.n_lanes - 1]
    assert c["next_lane"].tolist() == [1, 2]
    nx = np.full(m.n_lanes, -1)
    nx[m.lane_index(6, 1)], nx[m.lane_index(6, 2)] = c["lane"][0], c["lane"][1]
    nx[c["lane"][0]], nx[c["lane"][1]] = m.lane_index(7, 1), m.lane_index(7, 2)
    assert o.lane_next().tolist() == nx.tolist()
    # through the world step: an agent past the end of every lane lands on the successor (or stays: no successor)
    from dmpp_b200 import abi
    lanes = list(range(m.n_lanes))
    h = np.zeros(len(lanes), abi.scene_hdr)
    h["road_num"], h["lane_num"], h["n_obs"], h["period_ms"] = 1, 1, 1, 100.0
    h["next_roadnum"] = 1
    ag = np.zeros((len(lanes), 1), abi.agent)
    ag["lane"][:, 0] = lanes
    ag["i"][:, 0] = (m.lane_pt_off[1:] - m.lane_pt_off[:-1]) - 2
    ag["v"] = 1.0                                           # 0.1 m past a lane end: never past a whole segment of the next lane
    ag["u"][:, 0] = [np.hypot(*(np.array([m.x[k + 1] - m.x[k], m.y[k + 1] - m.y[k]]))) for k in m.lane_pt_off[1:] - 2]
    wp = o.world_params(); wp.pre_junction_pts = 60
    rec = np.zeros(len(lanes), abi.plan_record)
    o.world_step(h, ag, np.zeros((len(lanes), 1)), np.zeros((len(lanes), 1)), rec=rec, last_path=np.zeros((len(lanes), 2, 200)), wp=wp)
    want = np.array(lanes)
    want[m.lane_index(6, 1)], want[m.lane_index(6, 2)] = c["lane"][0], c["lane"][1]
    want[c["lane"][0]], want[c["lane"][1]] = m.lane_index(7, 1), m.lane_index(7, 2)
    assert ag["lane"][:, 0].tolist() == want.tolist()
    moved = want != np.array(lanes)
    assert (ag["i"][moved, 0] == 0).all() and (np.abs(ag["u"][moved, 0] - 0.1) < 1e-12).all()


def test_junction_step_known_answers(joracle, the_map):
    """one ego placed by hand on approach lane 1 of road 6 (standing: speed 0, so only the placement moves it) and two agents:
    pos 0 -> 1 at id 339 = 400 - 1 - 60, 1 -> 2 on the connector, 2 -> 0 on road 7; the agents jump the connector gaps"""
    from dmpp_b200 import abi
    m = the_map
    oracle = joracle
    wp = oracle.world_params(); wp.pre_junction_pts = 60
    g61, g72 = m.lane_index(6, 1), m.lane_index(7, 2)
    c0 = int(m.conn["lane"][0])
    P = lambda gl, i: (m.x[m.lane_pt_off[gl] + i], m.y[m.lane_pt_off[gl] + i])
    h = np.zeros(1, abi.scene_hdr)
    h["x"], h["y"] = P(g61, 300)
    h["dir"], h["velocity"], h["period_ms"] = 90.0, 0.0, 100.0
    h["road_num"], h["lane_num"], h["n_obs"], h["conn"] = 6, 1, 2, -1
    h["last_roadnum"], h["next_roadnum"], h["last_lanenum"], h["next_lanenum"] = 6, 7, 1, 1
    h["id"][0, :2] = 300
    h["stub_attribute"] = 2
    n_c = int(m.lane_pt_off[c0 + 1] - m.lane_pt_off[c0])
    ag = np.zeros((1, 2), abi.agent)
    seg = lambda gl, i: float(np.hypot(P(gl, i + 1)[0] - P(gl, i)[0], P(gl, i + 1)[1] - P(gl, i)[1]))
    # agent 0: 0.3 m before the end of approach lane 1 at 5 m/s; agent 1: 0.1 m before the end of connector 0 at 5 m/s
    ag["lane"] = [[g61, c0]]
    ag["i"] = [[398, n_c - 2]]
    ag["u"] = [[seg(g61, 398) - 0.3, seg(c0, n_c - 2) - 0.1]]
    ag["v"] = 5.0
    ox, oy = np.zeros((1, 2)), np.zeros((1, 2))
    oracle.world_step(h, ag, ox, oy, wp=wp)                                          # placement: id 300 < 339, pos stays 0
    assert h["pos"][0] == 0 and h["id"][0, 0] == 300
    ox0, oy0 = ox.copy(), oy.copy()
    rec = np.zeros(1, abi.plan_record)
    lp = np.zeros((1, 2, 200))

    def step(gl=None, i=None):
        if gl is not None:
            h["x"], h["y"] = P(gl, i)
        oracle.world_step(h, ag, ox, oy, rec=rec, last_path=lp, wp=wp)

    step()
    # agents: 0.3 + 0.5 m -> 0.2 m into segment 0 of the connector / 0.4 m into the departure lane
    u0 = (seg(g61, 398) - 0.3 + 5.0 * 0.1) - seg(g61, 398)
    u1 = (seg(c0, n_c - 2) - 0.1 + 5.0 * 0.1) - seg(c0, n_c - 2)
    assert ag["lane"][0].tolist() == [c0, m.lane_index(7, 1)] and ag["i"][0].tolist() == [0, 0]
    assert ag["u"][0, 0] == u0 and ag["u"][0, 1] == u1
    # ... and jump the gaps: connector 0 starts 3.25 m beside approach lane 1 and ends at the start of departure lane 2
    assert np.hypot(ox[0, 0] - ox0[0, 0], oy[0, 0] - oy0[0, 0]) > 3.0
    assert np.hypot(ox[0, 1] - ox0[0, 1], oy[0, 1] - oy0[0, 1]) > 3.0
    assert h["pos"][0] == 0 and h["x"][0] == P(g61, 300)[0]                        # standing ego
    step(g61, 338)
    assert h["pos"][0] == 0 and h["id"][0, 0] == 338
    step(g61, 339)                                                                   # the pre-junction zone: 339 >= 400 - 1 - 60
    assert (h["pos"][0], h["conn"][0], h["last_roadnum"][0], h["last_lanenum"][0], h["next_lanenum"][0]) == (1, 0, 6, 1, 1)
    assert h["road_num"][0] == 6 and h["id"][0, 0] == 339
    step(g61, 399)                                                                   # the approach end: still nearer than the connector
    assert h["pos"][0] == 1 and h["id"][0, 0] == 395                                 # (the window ends at 339 + 56)
    step(c0, 20)                                                                     # on the connector, nearer to lane 1 than to lane 2
    assert (h["pos"][0], h["road_num"][0], h["lane_num"][0], h["conn"][0]) == (2, 7, 1, 0)
    assert h["id"][0, :2].tolist() == [20, 20] and h["path_num"][0] == 0
    step(c0, 40)
    assert h["pos"][0] == 2 and h["id"][0, :2].tolist() == [40, 40]
    step(c0, n_c - 1)                                                                # connector end = start of departure lane 2: a tie stays
    assert h["pos"][0] == 2
    step(g72, 10)                                                                    # on road 7
    assert (h["pos"][0], h["road_num"][0], h["lane_num"][0], h["conn"][0]) == (0, 7, 2, -1)
    assert h["path_num"][0] == 1 and h["stub_attribute"][0] == 0 and h["id"][0, 1] == 10
    step(g72, 30)                                                                    # segment driving again, no connector ahead
    assert h["pos"][0] == 0 and h["id"][0, 1] == 30 and h["path_num"][0] == 1


# ---------------------------------------------------------------- CPU: the option switched off is today's step
def test_option_off_junction_ego_stays_frozen(oracle, joracle, the_map):
    """pre_junction_pts = 0: a junction world's ego stops at the approach road's end margin, as with the segment-only step of
    oracle/ -- which gives the same bytes"""
    w = jworld(the_map, 0, 256)
    wp = joracle.world_params()
    assert wp.pre_junction_pts == 0
    a = joracle.run_closed_loop(w.hdr, w.agents, 20, threads=4)
    H = a["hdr_log"]
    assert (H["x"] == H["x"][0]).all() and (H["y"] == H["y"][0]).all() and (H["velocity"][1:] == 0).all()
    assert (H["pos"] == H["pos"][0]).all() and (H["road_num"] == 6).all() and (H["path_num"] == 0).all()
    assert (a["agents"]["lane"] == w.agents["lane"]).all()                         # agents stop at their lane ends
    b = oracle.run_closed_loop(w.hdr, w.agents, 20, threads=4)
    for k in ("rec", "hdr_log", "hdr", "agents", "ox", "oy", "carry", "last_path"):
        assert a[k].tobytes() == b[k].tobytes(), k


@pytest.mark.parametrize("seed0,n,cycles", [(0, 256, 60), (31000, 96, 120)])
def test_option_on_highway_is_unchanged(oracle, joracle, the_map, seed0, n, cycles):
    """option on or off, highway worlds (no connector anywhere) give what the segment-only step of oracle/ gives, byte for byte"""
    from dmpp_b200 import scenes
    w = scenes.World(the_map, np.arange(seed0, seed0 + n))
    off = oracle.run_closed_loop(w.hdr, w.agents, cycles, threads=4)
    for J in (0, 60, 400):
        wp = joracle.world_params(); wp.pre_junction_pts = J
        on = joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=wp, threads=4)
        for k in ("rec", "hdr_log", "hdr", "agents", "ox", "oy", "obs_log_x", "obs_log_y", "carry", "last_path"):
            assert on[k].tobytes() == off[k].tobytes(), (J, k)


# ---------------------------------------------------------------- CPU: the loop is alive
@pytest.fixture(scope="module")
def junction_512(joracle, the_map):
    w = jworld(the_map, 0, 512)
    return w, joracle.run_closed_loop(w.hdr, w.agents, 120, wp=jparams(joracle), threads=8)


def test_junction_loop_is_alive(junction_512):
    w, a = junction_512
    H = a["hdr_log"]
    pos, road, path = H["pos"].astype(int), H["road_num"].astype(int), H["path_num"].astype(int)
    allowed = {(0,), (1,), (2,), (0, 1), (1, 2), (2, 0), (0, 1, 2), (1, 2, 0), (0, 1, 2, 0)}
    for s in range(w.n):
        assert tuple(compressed(pos[:, s])) in allowed, (s, compressed(pos[:, s]))
    # road 6 before the connector, road 7 in it (the header names the NEXT road, Decision.cpp:417) and after it;
    # path_num 0 -> 1 and stub_attribute -> 0 exactly at the 2 -> 0 step
    before = (path == 0) & (pos != 2)
    assert (road[before] == 6).all() and (road[~before] == 7).all()
    p_step = np.diff(path, axis=0)
    assert set(np.unique(p_step).tolist()) <= {0, 1}
    at = p_step == 1
    assert (pos[:-1][at] == 2).all() and (pos[1:][at] == 0).all() and (H["stub_attribute"][1:][at] == 0).all()
    left = (pos[:-1] == 2) & (pos[1:] == 0)
    assert (at == left).all()
    share = (a["hdr"]["path_num"] == 1).mean()
    print("share of junction worlds on road 7 after 120 cycles: %.3f" % share)
    assert share > 0.5
    r = a["rec"]
    inj = (pos == 1) | (pos == 2)
    assert (r["behavior_to_dlg"][inj] == 13).any()
    assert (r["afresh_cause"][inj] == 4).any()
    # the ego follows the junction speed command: it slows down behind agents in the junction and moves again
    assert (H["velocity"][inj] < 5).any() and (np.diff(H["velocity"], axis=0)[inj[1:]] > 0).any()
    assert (a["agents"]["lane"] != w.agents["lane"]).any()                         # agents crossed into successor lanes


def test_junction_log_replays_open_loop(oracle, junction_512):
    w, a = junction_512
    rep = oracle.run(a["hdr_log"], a["obs_log_x"], a["obs_log_y"], exhaustive=False, threads=8)
    assert rep["rec"].tobytes() == a["rec"].tobytes()


def test_urban_loop_is_alive(joracle, the_map):
    w = jworld(the_map, 0, 256, kind="urban")
    a = joracle.run_closed_loop(w.hdr, w.agents, 120, wp=jparams(joracle, "urban"), threads=8)
    pos = a["hdr_log"]["pos"].astype(int)
    assert (pos[0] == 1).all() and (pos == 2).any() and (a["hdr"]["path_num"] == 1).any()


# ---------------------------------------------------------------- CPU: oracle vs the unmodified reference
@pytest.mark.parametrize("kind,seed0,n,cycles", [("junction", 0, 128, 120), ("urban", 500, 48, 120)])
def test_junction_closed_loop_oracle_equals_unmodified_reference(joracle, reference, the_map, kind, seed0, n, cycles):
    from tools.junction_oracle.binding import JunctionReference
    if not JunctionReference.available():
        pytest.skip("tools/junction_oracle/libref_junction.so not built (needs oracle/_ref/libref.so)")
    w = jworld(the_map, seed0, n, kind=kind)
    wp = jparams(joracle, kind)
    a = joracle.run_closed_loop(w.hdr, w.agents, cycles, wp=wp, paths=True, threads=4)
    b = JunctionReference().run_closed_loop(joracle.params, wp, w.hdr, w.agents, cycles, paths=True)
    assert b["status"] == 0
    clean = a["ub_scene"] == 0
    assert clean.mean() > 0.95
    assert_records_equal(a["rec"][:, clean], b["rec"][:, clean], REC, what="record")
    assert_records_equal(a["hdr_log"][:, clean], b["hdr_log"][:, clean], HDR, what="logged header")
    for k in ("obs_log_x", "obs_log_y", "path_xy"):
        assert same(a[k][:, clean], b[k][:, clean]).all(), k
    assert a["agents"][clean].tobytes() == b["agents"][clean].tobytes()
    assert_records_equal(a["carry"][clean], b["carry"][clean], CARRY, what="final state")
    assert (a["hdr"]["path_num"][clean] == 1).any()


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def jplanner(the_map):
    p = planner_with(the_map, 4096, 10, 60)
    yield p
    p.close()


@pytest.fixture(scope="module")
def junction_4096(joracle, the_map):
    w = jworld(the_map, 0, 4096)
    return w, joracle.run_closed_loop(w.hdr, w.agents, 120, wp=jparams(joracle), threads=16)


@pytest.mark.gpu
def test_gpu_junction_closed_loop_equals_oracle(jplanner, junction_4096):
    """4096 junction worlds x 120 cycles in ONE graph launch, replayed three times from the same initial world"""
    w, want = junction_4096
    got = jplanner.run_closed_loop(w.hdr, w.agents, 120, repeat=3)
    assert got["graph"], "the episode did not run as a CUDA graph"
    check_closed_loop(got, want, "junction graph")
    assert (got["hdr"]["path_num"] == 1).mean() > 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
def test_gpu_junction_direct_launches_and_group_kernel(the_map, junction_4096, env):
    w, want = junction_4096
    p = planner_with(the_map, 4096, 10, 60, env)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, 120)
        assert not got["graph"]
        check_closed_loop(got, want, str(env))
    finally:
        p.close()


@pytest.mark.gpu
def test_gpu_urban_200_agents_equals_oracle(joracle, the_map):
    """BASELINE config 5 worlds: the whole approach is the pre-junction zone, 200 agents each (group kernel)"""
    w = jworld(the_map, 0, 256, kind="urban", n_obs=200)
    want = joracle.run_closed_loop(w.hdr, w.agents, 120, wp=jparams(joracle, "urban"), threads=16)
    p = planner_with(the_map, 256, 200, 400)
    try:
        got = p.run_closed_loop(w.hdr, w.agents, 120)
        check_closed_loop(got, want, "urban")
    finally:
        p.close()
    assert (want["hdr_log"]["pos"] == 2).any()


@pytest.mark.gpu
def test_gpu_junction_log_replays_open_loop(jplanner, the_map):
    w = jworld(the_map, 9000, 1024)
    got = jplanner.run_closed_loop(w.hdr, w.agents, 120)
    assert (got["hdr_log"]["pos"] == 2).any() and (got["hdr"]["path_num"] == 1).any()
    rep = jplanner.run_episodes(got["hdr_log"], got["obs_log_x"], got["obs_log_y"], trace=False, paths=False)
    assert rep["rec"].tobytes() == got["rec"].tobytes()


@pytest.mark.gpu
def test_gpu_junction_steps_ragged_and_windows(jplanner, joracle, the_map):
    """ragged obstacle counts, agents at lane and connector ends, other window sizes and zone lengths"""
    w = jworld(the_map, 123, 600)
    rng = np.random.default_rng(5)
    w.hdr["n_obs"] = rng.integers(0, 11, 600)
    m = the_map
    ends = (m.lane_pt_off[w.agents["lane"] + 1] - m.lane_pt_off[w.agents["lane"]]) - 2
    w.agents["i"][::3] = ends[::3]
    w.agents["v"][::5] = 40.0
    c1 = int(m.conn["lane"][1])
    w.agents["lane"][::7, 0] = c1
    w.agents["i"][::7, 0] = int(m.lane_pt_off[c1 + 1] - m.lane_pt_off[c1]) - 2
    for loc_back, loc_fwd, a_max, J in ((3, 17, 1.5, 60), (8, 56, 3.0, 120), (0, 40, 3.0, 400)):
        wp = jplanner.world_params()
        wp.loc_back, wp.loc_fwd, wp.a_max, wp.pre_junction_pts = loc_back, loc_fwd, a_max, J
        jplanner.set_world_params(wp)
        try:
            want = joracle.run_closed_loop(w.hdr, w.agents, 24, wp=wp, threads=8)
            got = jplanner.run_closed_loop(w.hdr, w.agents, 24)
            check_closed_loop(got, want, "ragged %r" % ((loc_back, loc_fwd, a_max, J),))
        finally:
            jplanner.set_world_params(jparams(jplanner))


@pytest.mark.gpu
def test_gpu_highway_option_on_equals_option_off(the_map):
    from dmpp_b200 import scenes
    w = scenes.World(the_map, np.arange(2048))
    runs = []
    for J in (0, 60):
        p = planner_with(the_map, 2048, 10, J)
        try:
            runs.append(p.run_closed_loop(w.hdr, w.agents, 40))
        finally:
            p.close()
    for k in ("rec", "hdr_log", "hdr", "agents", "ox", "oy", "obs_log_x", "obs_log_y", "carry", "last_path"):
        assert runs[0][k].tobytes() == runs[1][k].tobytes(), k
