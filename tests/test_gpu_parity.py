"""GPU parity proper: the CUDA path (through the C ABI, libdmpp_b200.so) against the CPU oracle on
the same seeded inputs.  Discrete outputs AND continuous outputs are compared bit for bit
(the operator specification is IEEE-exact on both sides); the only toleranced field is
path_dir_err, where the reference calls libm atan (Planning.cpp:737) and the device evaluates
the specification's polynomial: |diff| <= 1e-9 degrees."""
import numpy as np
import pytest

from conftest import assert_records_equal, same

pytestmark = pytest.mark.gpu

REC_EXACT = ["velocity_expect", "path_lat_dis", "remain_dis", "mindist_lat", "mindist_lon", "brakespeed", "des_acc",
             "radius", "aim_x", "aim_y", "aim_dir", "aim_id", "behavior", "target_roadnum", "target_lanenum", "light",
             "behavior_to_dlg", "afresh_cause", "sweep_index", "path_near_id", "path_front_near_id", "ob_index",
             "ob_pathid", "n_traj", "afresh_planning", "ob_flag", "acc_flag", "cnt", "path_dir_err"]
DIR_ERR_TOL = {"path_dir_err": 1e-9}
CARRY = ["leftlight_time", "rightlight_time", "velocity_expect", "aim_x", "aim_y", "aim_dir", "aim_id", "obsavoid_time",
         "no_obsavoid_time", "frontobs_time", "plan_his_behavior", "path_near_id", "behavior", "target_roadnum",
         "target_lanenum", "light_status", "behavior_to_dlg", "his_behavior", "his_target_lanenum", "his_light_status",
         "lanechg_status", "obsavoid_status", "plan_count"]
SLOT = ["dis_lat", "dis_lng", "ob_index", "pathid", "evaluated", "found"]


@pytest.fixture(scope="module")
def planner(the_map):
    from dmpp_b200.planner import Planner
    p = Planner(max_scenes=4096, max_obs=64)
    p.upload_map(the_map)
    yield p
    p.close()


def pad_obs(OX, OY, max_obs):
    c, n, k = OX.shape
    X = np.zeros((c, n, max_obs)); Y = np.zeros((c, n, max_obs))
    X[:, :, :k] = OX; Y[:, :, :k] = OY
    return X, Y


def run_both(planner, oracle, the_map, seeds, kind, cycles, n_obs):
    from dmpp_b200 import scenes
    ep = scenes.Episodes(the_map, seeds, cycles=cycles, kind=kind, n_obs=n_obs)
    H, OX, OY = ep.all_cycles()
    want = oracle.run(H, OX, OY, exhaustive=True, threads=8)
    PX, PY = pad_obs(OX, OY, planner.max_obs)
    got = planner.run_episodes(H, PX, PY)
    return H, got, want


def check(got, want, what):
    clean = want["trace"]["ub_hits"] == 0                       # reference-UB cycles are defined by clamping; still compared
    assert_records_equal(got["rec"], want["rec"], REC_EXACT, close=DIR_ERR_TOL, what=what + " rec")
    assert np.array_equal(got["trace"]["ub_hits"] > 0, ~clean), what + " ub flags"
    for grp in ("region", "sweep"):
        for f in SLOT:
            ok = same(got["trace"][grp][f], want["trace"][grp][f])
            assert ok.all(), "%s trace.%s.%s mismatch at %s" % (what, grp, f, np.argwhere(~ok)[0])
    for grp in ("junction", "local"):
        assert_records_equal(got["trace"][grp], want["trace"][grp], SLOT, what=what + " trace." + grp)
    assert_records_equal(got["trace"], want["trace"], ["width_curlane", "faraim_dis", "navi_lanechg", "navi_lanechg_times",
                                                        "refpath_len", "pts_scored"], what=what + " trace")
    assert same(got["path_xy"], want["path_xy"]).all(), what + " road_points"
    assert same(got["path_ll"], want["path_ll"]).all(), what + " PlanningOut.pnts"
    assert_records_equal(got["carry"], want["carry"], CARRY, what=what + " carry")
    assert same(got["last_path"], want["last_path"]).all(), what + " last_Bpoints"


def test_highway_default_set(planner, oracle, the_map):
    """BASELINE config 2 shape: 4096 seeded highway scenes x 25 cycles, ego + 10 vehicles."""
    H, got, want = run_both(planner, oracle, the_map, np.arange(4096), "highway", 25, 10)
    check(got, want, "highway")
    beh = np.unique(got["rec"]["behavior"])
    assert set(beh.tolist()) >= {1, 2, 4, 5}, beh            # the episode mix really exercises the rule tree
    assert (got["rec"]["sweep_index"] >= 0).any()


def test_junction(planner, oracle, the_map):
    H, got, want = run_both(planner, oracle, the_map, np.arange(100000, 100512), "junction", 80, 10)
    check(got, want, "junction")
    assert set(np.unique(H["pos"]).tolist()) == {0, 1, 2}


@pytest.mark.parametrize("n_obs", [1, 3, 31, 32, 33, 50])
def test_obstacle_counts(planner, oracle, the_map, n_obs):
    """chunked (N < 32) and grouped (N >= 32) lane mappings of the nearest-point search"""
    H, got, want = run_both(planner, oracle, the_map, np.arange(7000, 7000 + 192), "highway", 12, n_obs)
    check(got, want, "n_obs=%d" % n_obs)


def test_urban_junction_200_agents(oracle, the_map):
    """BASELINE config 5 shape: junction episodes (pos 0 -> 1 -> 2 -> 0), 200 agents per scene"""
    from dmpp_b200 import scenes
    from dmpp_b200.planner import Planner
    ep = scenes.Episodes(the_map, np.arange(880000, 880000 + 96), cycles=70, kind="junction", n_obs=200)
    H, OX, OY = ep.all_cycles()
    want = oracle.run(H, OX, OY, exhaustive=True, threads=8)
    p = Planner(max_scenes=96, max_obs=200)
    p.upload_map(the_map)
    got = p.run_episodes(H, OX, OY)
    p.close()
    check(got, want, "junction-200")
    assert set(np.unique(H["pos"]).tolist()) == {0, 1, 2}


@pytest.mark.parametrize("n_obs,n", [(200, 96), (10, 256)])
def test_urban_predicted_tracks(oracle, the_map, n_obs, n):
    """BASELINE config 5: ~400-point lane + connector reference paths, every agent with a constant-turn-rate track of T = 400
    steps rolled out on the device (dp_set_tracks); the junction search runs against the moving agents.  Bit-exact vs the
    oracle's tile search; N = 10 goes through a context that would otherwise use the warp kernel."""
    from dmpp_b200 import scenes
    from dmpp_b200.planner import Planner
    ep = scenes.Episodes(the_map, np.arange(40_000, 40_000 + n), cycles=40, kind="urban", n_obs=n_obs)
    H, OX, OY, VX, VY, DTH = ep.all_cycles_tracks()
    want = oracle.run_tracks(H, OX, OY, VX, VY, DTH, ep.TRACK_T, threads=8)
    p = Planner(max_scenes=n, max_obs=n_obs)
    p.upload_map(the_map)
    got = p.run_episodes_tracks(H, OX, OY, VX, VY, DTH, ep.TRACK_T)
    check(got, want, "urban tracks N=%d" % n_obs)
    static = p.run_episodes(H, OX, OY)                      # tracks cleared: the reference's static semantics again
    p.close()
    check(static, oracle.run(H, OX, OY, threads=8), "urban static N=%d" % n_obs)
    assert (got["trace"]["junction"]["pathid"] != static["trace"]["junction"]["pathid"]).mean() > 0.3


def test_zero_obstacles_and_ragged(planner, oracle, the_map):
    from dmpp_b200 import scenes
    ep = scenes.Episodes(the_map, np.arange(300, 300 + 256), cycles=8, n_obs=12)
    H, OX, OY = ep.all_cycles()
    H["n_obs"] = (np.arange(256) % 13)[None, :]                # ragged: 0..12 obstacles per scene
    want = oracle.run(H, OX, OY, exhaustive=True)
    PX, PY = pad_obs(OX, OY, planner.max_obs)
    got = planner.run_episodes(H, PX, PY)
    check(got, want, "ragged")


def test_operator_parity(planner, oracle, the_map):
    rng = np.random.default_rng(5)
    # SearchObstacle / CreateNewPath on random curved polylines, incl. P = 2, 3 and P > one tile
    paths, wins = [], []
    for P in (2, 3, 17, 120, 128, 129, 300, 700):
        t = np.linspace(0, 1, P)
        x = 50 * t * (1 + rng.random()) + rng.normal(0, 0.01, P)
        y = 8 * np.sin(3 * t + rng.random()) + rng.normal(0, 0.01, P)
        paths.append((x, y)); wins.append((-rng.random() * 2, rng.random() * 2))
    for n_obs in (1, 10, 40):
        ox = rng.uniform(-5, 105, n_obs); oy = rng.uniform(-10, 10, n_obs)
        got = planner.search_obstacle(paths, ox, oy, [w[0] for w in wins], [w[1] for w in wins])
        for i, (p, w) in enumerate(zip(paths, wins)):
            want = oracle.search_obstacle(p[0], p[1], ox, oy, w[0], w[1])
            for f in ("dis_lat", "dis_lng", "ob_index", "pathid", "found"):
                assert same(got[i][f], want[f]), (i, n_obs, f, got[i], want)
    offs = rng.uniform(-4, 4, len(paths))
    got = planner.create_new_path(paths, offs)
    for i, p in enumerate(paths):
        wx, wy = oracle.create_new_path(p[0], p[1], offs[i])
        assert np.array_equal(got[i][0], wx) and np.array_equal(got[i][1], wy)
    poses = np.column_stack([rng.uniform(-1000, 1000, 64), rng.uniform(-1000, 1000, 64), rng.uniform(0, 360, 64),
                             rng.uniform(-1000, 1000, 64), rng.uniform(-1000, 1000, 64), rng.uniform(0, 360, 64)])
    got = planner.bezier_planning(poses)
    for i in range(64):
        assert np.array_equal(got[i], oracle.bezier(poses[i]))
    mp = [p for p in paths if len(p[0]) <= 200] + [(np.array([1.0, 1.0, 2.0]), np.array([0.0, 0.0, 0.0]))]
    got = planner.mean_points(mp)
    for i, p in enumerate(mp):
        assert np.array_equal(got[i], oracle.mean_points(p[0], p[1]))


def test_dense_sweep(planner, oracle, the_map):
    """BASELINE config 3 shape, reduced grid for the CPU oracle: lateral x aim distance x horizon candidates,
    50 obstacles with constant-velocity tracks; lowest-index feasible candidate and every dis_lng bit-exact."""
    rng = np.random.default_rng(11)
    gl = the_map.lane_index(3, 2)
    o = the_map.lane_pt_off[gl] + 300
    bx, by = the_map.x[o:o + 256], the_map.y[o:o + 256]
    lat = np.arange(-3.15, 3.16, 0.1)
    hor = np.arange(8, 257, 8)
    offset = np.repeat(lat, len(hor)); n_pts = np.tile(hor, len(lat)).astype(np.int32)
    ox = bx[rng.integers(10, 250, 50)] + rng.normal(0, 2.0, 50); oy = by[rng.integers(10, 250, 50)] + rng.normal(0, 2.0, 50)
    for dv in (None, (rng.normal(0, 0.05, 50), rng.normal(0, 0.05, 50))):
        dvx, dvy = (None, None) if dv is None else dv
        best, best_d, allv = planner.score_candidates(bx, by, offset, n_pts, ox, oy, dvx, dvy)
        wbest, wall = oracle.score_candidates(bx, by, offset, n_pts, ox, oy, dvx, dvy)
        assert best == wbest
        assert np.array_equal(allv, wall)
        if best >= 0:
            assert best_d == wall[best]


def test_dense_sweep_session_full_grid(planner, oracle, the_map):
    """BASELINE config 3 at full size through the latency-mode session: 64 lateral offsets x 32 aim distances x 32
    horizons = 65 536 candidates, 50 obstacle tracks.  The CPU oracle scores the full grid once (a few seconds);
    repeated graph replays with moved obstacles are checked on the winner only."""
    rng = np.random.default_rng(2024)
    gl = the_map.lane_index(3, 2)
    o = the_map.lane_pt_off[gl] + 900
    bx, by = the_map.x[o:o + 256], the_map.y[o:o + 256]
    lat = -3.15 + 0.1 * np.arange(64)
    aim = 10.0 + 2.5 * np.arange(32)
    hor = 8 * (1 + np.arange(32))
    # enumeration order lateral-major; the candidate's point count is min(horizon, points within the aim distance)
    L, A, Hh = np.meshgrid(lat, aim, hor, indexing="ij")
    n_pts = np.minimum(Hh, np.maximum(2, (A / 0.5).astype(np.int64))).astype(np.int32).ravel()
    offset = L.ravel()
    assert offset.size == 65536
    ox = bx[rng.integers(5, 250, 50)] + rng.normal(0, 1.5, 50); oy = by[rng.integers(5, 250, 50)] + rng.normal(0, 1.5, 50)
    dvx, dvy = rng.normal(0, 0.04, 50), rng.normal(0, 0.04, 50)
    sess = planner.sweep_session(bx, by, offset, n_pts, 64)
    best, dis, ms = sess.score(ox, oy, dvx, dvy)
    wbest, wall = oracle.score_candidates(bx, by, offset, n_pts, ox, oy, dvx, dvy)
    assert best == wbest and (best < 0 or dis == wall[best])
    b2, d2, all2 = planner.score_candidates(bx, by, offset, n_pts, ox, oy, dvx, dvy)
    assert b2 == wbest and np.array_equal(all2, wall)
    for it in range(20):                                     # graph replays: idempotent for equal inputs
        assert sess.score(ox, oy, dvx, dvy)[:2] == (best, dis)
    sess.close()


@pytest.mark.parametrize("n_obs", [0, 1, 31, 33, 64])
def test_dense_sweep_session_shapes(planner, oracle, the_map, n_obs):
    """the one-launch session against the oracle over obstacle counts around the 32-lane blocks, ragged candidate sets (a
    candidate with fewer than 2 points is never found: dis_lng = 999 > clear_dis makes it feasible, Decision.cpp:944), changing
    corridor / clearance arguments and obstacles that move between calls"""
    rng = np.random.default_rng(100 + n_obs)
    gl = the_map.lane_index(3, 2)
    o = the_map.lane_pt_off[gl] + 500
    bx, by = the_map.x[o:o + 200], the_map.y[o:o + 200]
    offset = rng.choice(-2.0 + 0.25 * np.arange(17), 600)
    n_pts = rng.integers(2, 201, 600).astype(np.int32)
    n_pts[rng.integers(0, 600, 5)] = 200
    sess = planner.sweep_session(bx, by, offset, n_pts, 64)
    n_pts1 = n_pts.copy(); n_pts1[[400, 17]] = [1, 0]        # two candidates without a path, behind many ordinary ones
    sess1 = planner.sweep_session(bx, by, offset, n_pts1, 64)
    for it in range(6):
        idx = rng.integers(5, 195, n_obs)
        ox, oy = bx[idx] + rng.normal(0, 1.2, n_obs), by[idx] + rng.normal(0, 1.2, n_obs)
        dvx, dvy = rng.normal(0, 0.05, n_obs), rng.normal(0, 0.05, n_obs)
        lo, hi, clear = (-0.9, 0.9, 25.0) if it % 2 == 0 else (-1.4, 0.6, 60.0 + it)
        for s_, npt in ((sess, n_pts), (sess1, n_pts1)):
            wbest, wall = oracle.score_candidates(bx, by, offset, npt, ox, oy, dvx, dvy, lat_min=lo, lat_max=hi, clear_dis=clear)
            best, dis, _ = s_.score(ox, oy, dvx, dvy, lat_min=lo, lat_max=hi, clear_dis=clear)
            assert best == wbest, (it, best, wbest)
            assert best < 0 or dis == wall[best]
            assert s_.score(ox, oy, dvx, dvy, lat_min=lo, lat_max=hi, clear_dis=clear, want_ms=False)[:2] == (best, dis)
    sess.close(); sess1.close()


def bezier_grid(the_map, n_lat, n_aim, n_hor, seed=7):
    """lateral x aim-distance grid of local paths (Planning.cpp:596-611): ego pose on a lane, aim poses at arclength a on the
    laterally shifted lane; every (lateral, aim) pair is its own Bezier line, its horizons are prefixes of that line"""
    gl = the_map.lane_index(3, 2)
    o = the_map.lane_pt_off[gl] + 700
    lx, ly, ld = the_map.x[o:o + 400], the_map.y[o:o + 400], the_map.dir[o:o + 400]
    lat = np.linspace(-3.0, 3.0, n_lat)
    aim_id = np.linspace(40, 200, n_aim).astype(int)        # 20 .. 100 m ahead at 0.5 m spacing
    poses = np.zeros((n_lat * n_aim, 6))
    for i, d in enumerate(lat):
        for k, a in enumerate(aim_id):
            h = np.deg2rad(ld[a])
            # map headings are degrees from +x, counter-clockwise (scenes.Map.add_lane): (sin h, -cos h) is the right normal
            poses[i * n_aim + k] = (lx[0], ly[0], ld[0], lx[a] + d * np.sin(h), ly[a] - d * np.cos(h), ld[a])
    hor = np.linspace(8, 200, n_hor).astype(np.int32)
    cand_line = np.repeat(np.arange(n_lat * n_aim), n_hor).astype(np.int32)
    n_pts = np.tile(hor, n_lat * n_aim).astype(np.int32)
    return poses, cand_line, n_pts, (lx, ly)


def test_dense_sweep_bezier_lines(planner, oracle, the_map):
    """distinct-geometry grid: every (lateral, aim distance) pair is its own Bezier local path drawn ON THE DEVICE
    (dp_sweep_set_bezier), every horizon a prefix of it.  Lines == the BezierPlanning operator bit for bit; winner and its
    dis_lng == the oracle scoring each line's horizons alone (lowest candidate index over all lines), for the latency shape
    (few rows, 16 parts per row) and the throughput shape (> 296 rows, 4 parts per row)."""
    rng = np.random.default_rng(5)
    for n_lat, n_aim, n_hor in ((6, 5, 7), (20, 16, 4)):
        poses, cand_line, n_pts, (lx, ly) = bezier_grid(the_map, n_lat, n_aim, n_hor)
        n_lines = n_lat * n_aim
        off = np.zeros(cand_line.size)
        sess = planner.sweep_session(None, None, off, n_pts, 64, cand_line=cand_line, bezier_lines=n_lines)
        sess.set_bezier(poses)
        lines = sess.lines()
        want_lines = planner.bezier_planning(poses)
        assert np.array_equal(lines.reshape(n_lines, 400), np.asarray(want_lines).reshape(n_lines, 400))
        for it in range(3):
            N = 50
            idx = rng.integers(10, 200, N)
            ox, oy = lx[idx] + rng.normal(0, 2.0, N), ly[idx] + rng.normal(0, 2.0, N)
            dvx, dvy = rng.normal(0, 0.03, N), rng.normal(0, 0.03, N)
            clear = (25.0, 60.0, 5.0)[it]
            wbest, wdis = -1, None
            for ln in range(n_lines):                       # candidates of a line are contiguous, lines ascend: first feasible overall
                sel = np.nonzero(cand_line == ln)[0]
                b, dall = oracle.score_candidates(lines[ln, 0], lines[ln, 1], off[sel], n_pts[sel], ox, oy, dvx, dvy, clear_dis=clear)
                if b >= 0:
                    wbest, wdis = int(sel[b]), dall[b]
                    break
            best, dis, _ = sess.score(ox, oy, dvx, dvy, clear_dis=clear)
            assert best == wbest, (n_lat, it, best, wbest)
            assert best < 0 or dis == wdis
        # the same lines uploaded from the host (dp_sweep_create_lines) score identically
        sess2 = planner.sweep_session(None, None, off, n_pts, 64, lines=lines, cand_line=cand_line)
        assert sess2.score(ox, oy, dvx, dvy, clear_dis=clear)[:2] == (best, dis)
        sess.close(); sess2.close()


def test_reset_and_carry_roundtrip(planner, oracle, the_map):
    """checkpoint/resume: episodes split in two halves with the carry downloaded and re-uploaded in
    between give the same result as one uninterrupted run (idempotent state hand-off)."""
    from dmpp_b200 import scenes
    ep = scenes.Episodes(the_map, np.arange(900, 900 + 128), cycles=20, n_obs=10)
    H, OX, OY = ep.all_cycles()
    PX, PY = pad_obs(OX, OY, planner.max_obs)
    full = planner.run_episodes(H, PX, PY)
    planner.reset(0, 128)
    for c in range(10):
        planner.cycle(np.ascontiguousarray(H[c]), PX[c], PY[c])
    carry, lp = planner.download_carry(0, 128)
    planner.reset(0, 128)
    planner.upload_carry(0, carry, lp)
    for c in range(10, 20):
        o = planner.cycle(np.ascontiguousarray(H[c]), PX[c], PY[c])
        assert (o["rec"].tobytes() == full["rec"][c].tobytes())


def test_reset_dev_is_ordered_with_the_callers_stream(planner, oracle, the_map):
    """dp_reset_dev enqueues the reset on the caller's stream: back-to-back episodes launched without any host synchronisation
    (the loop shape of bench.py's latency histogram) repeat the first episode bit for bit"""
    import torch
    from dmpp_b200 import scenes
    n, cycles = 256, 8
    ep = scenes.Episodes(the_map, np.arange(7000, 7000 + n), cycles=cycles, n_obs=10)
    H, OX, OY = ep.all_cycles()
    PX, PY = pad_obs(OX, OY, planner.max_obs)
    dev = torch.device("cuda", 0)
    d_hdr = torch.from_numpy(H.view(np.uint8).reshape(cycles, n, 128)).to(dev)
    d_ox, d_oy = torch.from_numpy(PX).to(dev), torch.from_numpy(PY).to(dev)
    d_rec = torch.empty((3, cycles, n, 128), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    torch.cuda.synchronize()
    for e in range(3):
        planner.reset_dev(0, n, stream=st.cuda_stream)
        for c in range(cycles):
            planner.cycle_dev(n, d_hdr[c].data_ptr(), d_ox[c].data_ptr(), d_oy[c].data_ptr(), d_rec[e, c].data_ptr(), stream=st.cuda_stream)
    torch.cuda.synchronize()
    r = d_rec.cpu().numpy()
    want = oracle.run(H, OX, OY, exhaustive=False, threads=4, paths=False, calls=False, trace=False)["rec"]
    for e in range(3):
        assert r[e].tobytes() == r[0].tobytes(), e
    got = r[0].view(want.dtype).reshape(cycles, n)
    for f in ("behavior", "n_traj", "sweep_index", "path_near_id", "afresh_planning"):
        assert np.array_equal(got[f], want[f]), f


def test_library_is_the_cuda_path(planner):
    """the calls above really launched kernels from libdmpp_b200.so"""
    assert planner.launch_count() > 100
    fp64, fp32 = planner.measure_fma_peak()
    assert fp64 > 5 and fp32 > 20, (fp64, fp32)


def test_pinned_host_paths(planner, oracle, the_map):
    """dp_cycle_batch with PINNED host buffers (three input DMAs, records stored straight into the caller's buffer) must give
    byte-identical records to the staged-copy route used with pageable buffers."""
    import torch
    from dmpp_b200 import abi, scenes
    n, cycles = 512, 12
    ep = scenes.Episodes(the_map, np.arange(4242, 4242 + n), cycles=cycles, n_obs=10)
    H, OX, OY = ep.all_cycles()
    PX, PY = pad_obs(OX, OY, planner.max_obs)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    Hp = pin(H.view(np.uint8).reshape(cycles, n, 128)).view(abi.scene_hdr).reshape(cycles, n)
    PXp, PYp = pin(PX), pin(PY)
    rec_p = torch.empty((n, 128), dtype=torch.uint8).pin_memory().numpy().view(abi.plan_record).reshape(n)
    planner.reset(0, n)
    got = []
    for c in range(cycles):
        planner.cycle(Hp[c], PXp[c], PYp[c], out={"rec": rec_p})
        got.append(rec_p.copy())
    planner.reset(0, n)
    for c in range(cycles):
        o = planner.cycle(np.ascontiguousarray(H[c]), PX[c], PY[c])
        assert o["rec"].tobytes() == got[c].tobytes(), "cycle %d" % c
    want = oracle.run(H, OX, OY, paths=False, calls=False, trace=False, exhaustive=False)
    assert_records_equal(np.stack(got), want["rec"], REC_EXACT, close=DIR_ERR_TOL, what="pinned")


def test_pipelined_submit_wait(planner, oracle, the_map):
    """dp_cycle_submit / dp_cycle_wait with two cycles in flight: records byte-identical to the synchronous call, in
    submission order; the state errors the header promises."""
    import torch
    from dmpp_b200 import abi, scenes
    from dmpp_b200.planner import DpError
    n, cycles = 512, 12
    ep = scenes.Episodes(the_map, np.arange(777, 777 + n), cycles=cycles, n_obs=10)
    H, OX, OY = ep.all_cycles()
    PX, PY = pad_obs(OX, OY, planner.max_obs)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    Hp = pin(H.view(np.uint8).reshape(cycles, n, 128)).view(abi.scene_hdr).reshape(cycles, n)
    PXp, PYp = pin(PX), pin(PY)
    recs = [torch.empty((n, 128), dtype=torch.uint8).pin_memory().numpy().view(abi.plan_record).reshape(n) for _ in range(2)]
    planner.reset(0, n)
    with pytest.raises(DpError):
        planner.wait()                                           # nothing in flight
    got = []
    planner.submit(Hp[0], PXp[0], PYp[0], recs[0])
    for c in range(1, cycles):
        planner.submit(Hp[c], PXp[c], PYp[c], recs[c & 1])
        if c == 1:
            with pytest.raises(DpError):
                planner.submit(Hp[c], PXp[c], PYp[c], recs[0])   # a third cycle in flight is refused
            with pytest.raises(DpError):
                planner.reset(0, n)                              # state calls are refused while cycles are in flight
        planner.wait()
        got.append(recs[(c - 1) & 1].copy())
    planner.wait()
    got.append(recs[(cycles - 1) & 1].copy())
    with pytest.raises(DpError):
        planner.submit(np.ascontiguousarray(H[0]), PX[0], PY[0], recs[0])   # pageable inputs are refused
    want = oracle.run(H, OX, OY, paths=False, calls=False, trace=False, exhaustive=False)
    assert_records_equal(np.stack(got), want["rec"], REC_EXACT, close=DIR_ERR_TOL, what="pipelined")
    planner.reset(0, n)
    for c in range(cycles):
        o = planner.cycle(np.ascontiguousarray(H[c]), PX[c], PY[c])
        assert o["rec"].tobytes() == got[c].tobytes(), "cycle %d" % c


def test_pipelined_submit_wait_one_wave(oracle, the_map):
    """the pipelined pair on a context of its own, 512 scenes and 4096 scenes (one full wave: the Decision CTAs waiting for the
    input flag and the Planning launch compete for the slots).  Same records as the oracle."""
    import torch
    from dmpp_b200 import abi, scenes
    from dmpp_b200.planner import Planner
    for n, cycles in ((512, 10), (4096, 6)):
        p = Planner(n, 10)
        p.upload_map(the_map)
        ep = scenes.Episodes(the_map, np.arange(31000, 31000 + n), cycles=cycles, n_obs=10)
        H, OX, OY = ep.all_cycles()
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
        Hp = pin(H.view(np.uint8).reshape(cycles, n, 128)).view(abi.scene_hdr).reshape(cycles, n)
        PXp, PYp = pin(OX), pin(OY)
        recs = [torch.empty((n, 128), dtype=torch.uint8).pin_memory().numpy().view(abi.plan_record).reshape(n) for _ in range(2)]
        p.reset(0, n)
        got, pend = [], []
        for c in range(cycles):
            if len(pend) == 2:
                p.wait(); got.append(recs[pend.pop(0) & 1].copy())
            p.submit(Hp[c], PXp[c], PYp[c], recs[c & 1])
            pend.append(c)
        while pend:
            p.wait(); got.append(recs[pend.pop(0) & 1].copy())
        want = oracle.run(H, OX, OY, paths=False, calls=False, trace=False, exhaustive=False)
        assert_records_equal(np.stack(got), want["rec"], REC_EXACT, close=DIR_ERR_TOL, what="pipelined, %d scenes" % n)
        p.close()


def test_record_mirrors(planner, the_map):
    """dp_set_record_mirrors: every finished record is also stored at base[k] + slot (the hook the multi-GPU gather uses
    with peer-mapped buffers); here two device buffers on the same GPU and a non-zero first slot."""
    import torch
    from dmpp_b200 import abi, scenes
    n, first, cycles = 300, 40, 6
    ep = scenes.Episodes(the_map, np.arange(9000, 9000 + n), cycles=cycles, n_obs=10)
    H, OX, OY = ep.all_cycles()
    PX, PY = pad_obs(OX, OY, planner.max_obs)
    dev = torch.device("cuda", 0)
    m1 = torch.zeros((first + n + 8, 128), dtype=torch.uint8, device=dev)
    m2 = torch.zeros((first + n + 8, 128), dtype=torch.uint8, device=dev)
    planner.reset(first, n)
    planner.set_record_mirrors([m1.data_ptr(), m2.data_ptr()])
    try:
        for c in range(cycles):
            o = planner.cycle(np.ascontiguousarray(H[c]), PX[c], PY[c], first=first)
            torch.cuda.synchronize()
            for m in (m1, m2):
                got = m.cpu().numpy()
                assert got[first:first + n].tobytes() == o["rec"].tobytes(), "cycle %d" % c
                assert not got[:first].any() and not got[first + n:].any(), "stores outside the slot range"
    finally:
        planner.set_record_mirrors([])


def test_nearest_id_operator_and_near_ties(planner, oracle):
    """CShare::NearestId on the GPU compares SQUARED distances and falls back to the reference's sqrt loop when two different
    squared distances lie within 2^-49 of each other.  Random paths, exact ties (duplicate points), and crafted near ties where
    two squared distances differ by one ulp (so their sqrt may or may not round to the same double), in both index orders."""
    rng = np.random.default_rng(11)
    paths, qx, qy = [], [], []
    for P in (1, 2, 31, 32, 33, 200, 257):
        for _ in range(6):
            paths.append((rng.uniform(-50, 50, P), rng.uniform(-50, 50, P))); qx.append(rng.uniform(-60, 60)); qy.append(rng.uniform(-60, 60))
    x = rng.uniform(-5, 5, 200); y = rng.uniform(-5, 5, 200)
    x[150] = x[20]; y[150] = y[20]; x[77] = x[20]; y[77] = y[20]          # exact ties: lowest index wins
    paths.append((x, y)); qx.append(x[20] + 1e-3); qy.append(y[20] - 2e-3)
    paths.append((np.full(200, 1e5), np.full(200, 1e5))); qx.append(0.0); qy.append(0.0)   # nothing closer than 9999 -> 0
    for base in (1.0, 3.0, 0.75, 123.456, 1e-3, 777.0):
        for lo_first in (True, False):
            # query at the origin; point A at (2b, b) -> e = 5 b^2; point B at (2b, b') with b' = nextafter(b): e one or two ulps up
            b = base; b2 = np.nextafter(b, np.inf)
            x = np.full(64, 50.0 * b + 100.0); y = np.full(64, 50.0 * b + 100.0)
            ia, ib = (5, 40) if lo_first else (40, 5)
            x[ia] = 2 * b; y[ia] = b; x[ib] = 2 * b; y[ib] = b2
            paths.append((x, y)); qx.append(0.0); qy.append(0.0)
    got = planner.nearest_id(paths, qx, qy)
    for i, p in enumerate(paths):
        want = oracle.nearest_id(qx[i], qy[i], p[0], p[1])
        assert int(got[i]) == want, (i, len(p[0]), int(got[i]), want)


def test_multi_wave_batch_one_warp_ctas(oracle, the_map):
    """Batches above one wave (> 4144 scenes on a B200) run the one-warp-per-CTA instantiation of the cycle kernels with the
    overlapped launch; same parity bar: every record, trace slot, path sample and the final carry against the oracle."""
    from dmpp_b200.planner import Planner
    n = 6000
    p = Planner(max_scenes=n, max_obs=12)
    p.upload_map(the_map)
    try:
        H, got, want = run_both(p, oracle, the_map, np.arange(50_000, 50_000 + n), "highway", 10, 10)
        check(got, want, "6000 scenes")
        H, got, want = run_both(p, oracle, the_map, np.arange(70_000, 70_000 + n), "junction", 8, 10)
        check(got, want, "6000 junction scenes")
    finally:
        p.close()


@pytest.mark.parametrize("split", ["warp", "group", "group1", "group2"])
def test_launch_modes_agree(planner, the_map, monkeypatch, split):
    """Every way the cycle can be launched must produce the same bytes (records, traces, paths, carried state) as the
    module's default planner: the warp-per-scene kernel, and the group kernel in its three CTA shapes (DP_GROUP_CFG 0/1/2)."""
    from dmpp_b200 import scenes
    from dmpp_b200.planner import Planner
    n, cycles = 384, 10
    for kind, seed0 in (("highway", 31_000), ("junction", 32_000)):
        ep = scenes.Episodes(the_map, np.arange(seed0, seed0 + n), cycles=cycles, kind=kind, n_obs=10)
        H, OX, OY = ep.all_cycles()
        PX, PY = pad_obs(OX, OY, planner.max_obs)
        want = planner.run_episodes(H, PX, PY)
        env = {"warp": {"DP_KERNEL": "warp"}, "group": {"DP_KERNEL": "group"}, "group1": {"DP_KERNEL": "group", "DP_GROUP_CFG": "1"},
               "group2": {"DP_KERNEL": "group", "DP_GROUP_CFG": "2"}}[split]
        for k, v in env.items():
            monkeypatch.setenv(k, v)                           # read by dp_create (DP_GROUP_CFG: at the first group launch of the process)
        alt = Planner(max_scenes=n, max_obs=planner.max_obs)
        for k in env:
            monkeypatch.delenv(k)
        alt.upload_map(the_map)
        got = alt.run_episodes(H, PX, PY)
        alt.close()
        for k in ("rec", "trace", "path_xy", "path_ll", "carry", "last_path"):
            assert got[k].tobytes() == want[k].tobytes(), (kind, split, k)


def test_error_behaviour(planner, the_map):
    """every entry point reports a negative status + dp_last_error instead of failing silently (INTEGRATION.md)"""
    from dmpp_b200 import abi
    from dmpp_b200.planner import DpError, Planner
    fresh = Planner(max_scenes=8, max_obs=4)
    h = np.zeros(4, abi.scene_hdr); ox = np.zeros((4, 4)); oy = np.zeros((4, 4))
    with pytest.raises(DpError, match="map not uploaded"):
        fresh.cycle(h, ox, oy)
    fresh.upload_map(the_map)
    with pytest.raises(DpError):
        fresh.cycle(np.zeros(16, abi.scene_hdr), np.zeros((16, 4)), np.zeros((16, 4)))      # more scenes than the context holds
    with pytest.raises(DpError):
        fresh.reset(4, 8)                                                                 # slot range out of bounds
    with pytest.raises(DpError):
        fresh.set_record_mirrors([0x1000] * 9)                                            # more mirrors than supported
    fresh.close()


def test_run_episode_dev(planner, the_map):
    """dp_run_episode_dev: whole episodes resident in HBM, one call -- records of every cycle and the final carry must be the
    bytes the cycle-by-cycle host path produces."""
    import torch
    from dmpp_b200 import abi, scenes
    n, cycles = 1500, 14
    for kind, seed0 in (("highway", 61_000), ("junction", 62_000)):
        ep = scenes.Episodes(the_map, np.arange(seed0, seed0 + n), cycles=cycles, kind=kind, n_obs=10)
        H, OX, OY = ep.all_cycles()
        PX, PY = pad_obs(OX, OY, planner.max_obs)
        want = planner.run_episodes(H, PX, PY, trace=False, paths=False)
        dev = torch.device("cuda", 0)
        d_h = torch.from_numpy(H.view(np.uint8).reshape(cycles, n, 128)).to(dev)
        d_x, d_y = torch.from_numpy(PX).to(dev), torch.from_numpy(PY).to(dev)
        d_r = torch.zeros((cycles, n, 128), dtype=torch.uint8, device=dev)
        planner.reset(0, n)
        torch.cuda.synchronize()
        planner.run_episode_dev(n, cycles, d_h.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(),
                                stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = d_r.cpu().numpy().view(abi.plan_record).reshape(cycles, n)
        assert got.tobytes() == want["rec"].tobytes(), kind
        carry, last = planner.download_carry(0, n)
        assert carry.tobytes() == want["carry"].tobytes() and last.tobytes() == want["last_path"].tobytes(), kind


@pytest.mark.parametrize("kind,n,cycles,n_obs,seed0", [("highway", 4096, 25, 7, 200_000), ("highway", 3000, 40, 16, 300_000),
                                                       ("junction", 2000, 30, 3, 400_000), ("highway", 1024, 25, 33, 500_000)])
def test_soak_other_seeds_and_obstacle_counts(planner, oracle, the_map, kind, n, cycles, n_obs, seed0):
    """more of the same bar on other seeds, episode lengths and obstacle counts (7: three candidates per sweep pass with two idle
    lanes; 16: two per pass; 3: eight per pass; 33: the grouped N >= 32 path inside the cycle kernel)"""
    H, got, want = run_both(planner, oracle, the_map, np.arange(seed0, seed0 + n), kind, cycles, n_obs)
    check(got, want, "%s n=%d N=%d" % (kind, n, n_obs))
