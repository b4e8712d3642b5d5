"""Parity of the plan cycle on maps and parameters other than the built-in ones (tests/map_variants.py): lane widths at every
avoid-sweep size K = 0..8, jittered points with duplicates, UTM-like and scaled coordinates, 6-lane / 1-lane roads, a tight
circle, a zig-zag and a hairpin, and non-default dp_params.

Without a GPU: the group-kernel emulation (tools/emu) against the oracle for CTA group sizes 7, 14 and 16, the oracle against
the unmodified reference where it is built, and checks that the comparison is not vacuous (the episodes reach the avoid sweep
on both sides, every K, the outer lanes of the 6-lane road).  With a GPU (-m gpu): the real library -- warp kernel, group
kernel, the one-warp CTAs of a batch above one wave, the device map prep and dp_map_upload's width check -- against the
oracle with the full bar of test_gpu_parity.check, and the dense sweep on base paths from the irregular lanes."""
import contextlib

import numpy as np
import pytest

import map_variants as mv
from conftest import assert_records_equal, same
from test_gpu_parity import check, pad_obs
from test_oracle_vs_ref import CALL, CARRY as REF_CARRY, REC as REF_REC

SCENES = 256
SWEEP_SCENES = 384


@contextlib.contextmanager
def bound(runner, the_map, v):
    """the oracle / emulator / reference hold one map (and the first two one parameter set) per process: use the variant's,
    then give the built-in map and the defaults back to the rest of the suite"""
    params = getattr(runner, "params", None)
    runner.set_map(v.map)
    if params is not None:
        runner.params = v.params if v.params is not None else mv.default_params()
    try:
        yield runner
    finally:
        runner.set_map(the_map)
        if params is not None:
            runner.params = params


_sets = {}


def episode_sets(v):
    """(label, H, OX, OY): the highway mix of roads 1-5, the sweep roads with an obstacle wall beside the blocker (the avoid sweep
    on both sides; 15 obstacles, so the warp kernel deals the candidates out to lanes), and junction episodes (roads 6/7 and a
    connector, pos 0 -> 1 -> 2 -> 0)"""
    from dmpp_b200 import scenes
    if v.name not in _sets:
        m = v.map
        _sets[v.name] = [
            ("highway",) + scenes.Episodes(m, np.arange(SCENES), cycles=25, n_obs=10).all_cycles(),
            ("sweep",) + mv.walled(scenes.Episodes(m, np.arange(10_000, 10_000 + SWEEP_SCENES), cycles=25, n_obs=9, roads=v.sweep_roads)),
            ("junction",) + scenes.Episodes(m, np.arange(100_000, 100_000 + 96), cycles=60, kind="junction", n_obs=10).all_cycles(),
        ]
    return _sets[v.name]


_want = {}


def oracle_runs(oracle, the_map, v):
    if v.name not in _want:
        with bound(oracle, the_map, v):
            _want[v.name] = [oracle.run(H, OX, OY, exhaustive=True, threads=8) for _, H, OX, OY in episode_sets(v)]
    return _want[v.name]


@pytest.fixture(scope="module")
def emu(the_map):
    from tools.emu.binding import Emu
    e = Emu()
    e.set_map(the_map)
    return e


# ---- without a GPU ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("group", [7, 14, 16])
@pytest.mark.parametrize("name", mv.VARIANTS)
def test_emulated_group_kernel_matches_oracle(emu, oracle, the_map, name, group):
    v = mv.variant(name)
    wants = oracle_runs(oracle, the_map, v)
    with bound(emu, the_map, v):
        for (label, H, OX, OY), want in zip(episode_sets(v), wants):
            got = emu.run(H, OX, OY, group=group)
            check(got, want, "%s %s G=%d" % (name, label, group))
            fast = emu.run(H, OX, OY, group=group, trace=False, paths=False)    # the untraced path: the same records
            assert fast["rec"].tobytes() == got["rec"].tobytes(), (name, label, group)


# share of cycles on which the reference itself reads out of bounds (defined by the oracle, excluded from the comparison as in
# test_oracle_vs_ref): below 0.1 % everywhere but on the x2 map, where the junction episodes reach 0.25 %
MAX_UB = {"scaled": 0.003}


@pytest.mark.parametrize("name", mv.MAP_VARIANTS)
def test_oracle_matches_unmodified_reference(oracle, the_map, name):
    """test_oracle_vs_ref on the variant maps: records, the SearchObstacle call log (every candidate the reference scores, so
    every avoid-sweep candidate at K != 4), paths, final state and trajectory count.  The reference has dp_params compiled
    in: the parameter variants cannot run here."""
    from oracle import binding
    if not binding.Reference.available():
        pytest.skip("oracle/_ref/libref.so not built (needs the reference sources at build time)")
    v = mv.variant(name)
    ref = binding.Reference()
    with bound(oracle, the_map, v), bound(ref, the_map, v):
        for label, H, OX, OY in episode_sets(v):
            what = "%s %s" % (name, label)
            a = oracle.run(H, OX, OY, exhaustive=False, threads=8)
            b = ref.run(H, OX, OY)
            assert b["msgbox"] == 0
            clean = a["trace"]["ub_hits"] == 0
            assert clean.mean() > 1.0 - MAX_UB.get(name, 0.001), (what, clean.mean())
            assert_records_equal(a["rec"], b["rec"], REF_REC, mask=clean, what=what + " record")
            assert np.array_equal(a["n_calls"], b["n_calls"]), what
            assert_records_equal(a["calls"], b["calls"], CALL, what=what + " SearchObstacle call log")
            assert (same(a["path_xy"], b["path_xy"]) | ~clean[..., None, None]).all(), what
            assert (same(a["path_ll"], b["path_ll"]) | ~clean[..., None, None]).all(), what
            assert_records_equal(a["carry"], b["carry"], REF_CARRY, what=what + " final state")
            assert same(a["last_path"], b["last_path"]).all(), what
            assert a["traj"] == b["traj"], what


@pytest.mark.parametrize("name", mv.VARIANTS)
def test_variant_is_not_vacuous(oracle, the_map, name):
    """every variant reaches the avoid sweep on both sides (behaviours 4 and 5) and the junction positions; a parameter variant
    changes the oracle's records, so the parameter is really read"""
    v = mv.variant(name)
    wants = oracle_runs(oracle, the_map, v)
    rec = np.concatenate([w["rec"].ravel() for w in wants])
    assert set(np.unique(rec["behavior"]).tolist()) >= {1, 4, 5}, name
    assert (rec["sweep_index"] >= 0).sum() > 50, name
    assert set(np.unique(episode_sets(v)[2][1]["pos"]).tolist()) == {0, 1, 2}
    if v.params is not None:
        base = oracle_runs(oracle, the_map, mv.Variant("builtin", the_map))
        for label, w, b in zip(("highway", "sweep", "junction"), wants, base):
            assert w["rec"].tobytes() != b["rec"].tobytes(), (name, label)


def test_widths_reach_every_sweep_size(oracle, the_map):
    """K = #{i : i < (W - Vw) / 0.6} avoid candidates per side: the episodes run cycles at every K from 0 to 8, the exhaustive
    trace holds exactly the 2K candidates of the cycle's K, and the sweep picks a candidate on either side for every K >= 2.
    (With K = 1 the only candidate per side is the lane itself under the window the front check has just found blocked.)"""
    v = mv.variant("widths")
    for (label, H, OX, OY), w in zip(episode_sets(v), oracle_runs(oracle, the_map, v)):
        if label != "sweep":
            continue
        rec, tr = w["rec"], w["trace"]
        K = np.vectorize(mv.sweep_k)(tr["width_curlane"])
        ev = tr["sweep"]["evaluated"] != 0                                  # [cycles][n][2 * DP_MAX_SWEEP]
        swept = ev.any(axis=2)
        si = rec["sweep_index"]
        for k in range(9):
            at = K == k
            assert at.any(), k
            if k == 0:
                assert not (swept & at).any()
                continue
            want = np.zeros(2 * mv.MAX_SWEEP, bool); want[:k] = True; want[mv.MAX_SWEEP:mv.MAX_SWEEP + k] = True
            assert (ev[swept & at] == want).all(), k
            assert (swept & at).sum() > 10, k
            if k >= 2:
                assert ((si >= 0) & (si < k) & at).any(), ("left", k)
                assert ((si >= k) & at).any(), ("right", k)


def test_shapes_put_egos_on_the_outer_and_single_lanes():
    v = mv.variant("shapes")
    (_, H, _, _), (_, Hs, _, _) = episode_sets(v)[:2]
    assert {1, 6} <= set(np.unique(H["lane_num"][H["road_num"] == 1]).tolist())          # both edges of the 6-lane road
    for h in (H, Hs):
        assert set(np.unique(h["lane_num"][h["road_num"] == 2]).tolist()) == {1}         # the 1-lane road
    assert set(np.unique(np.concatenate([H["road_num"].ravel(), Hs["road_num"].ravel()])).tolist()) == {1, 2, 3, 4, 5}


# ---- on the GPU ------------------------------------------------------------------------------------------------------------------

# obstacle counts of the highway episodes on the GPU: the warp kernel deals the shifted avoid candidates out to (candidate,
# obstacle) lanes up to 16 obstacles (min(8, 32 / M) candidates per pass for M relevant ones) and scores them one at a time above;
# 33 also takes the grouped nearest-point scans.  The widths variant, whose K varies, runs three counts that reach the deal-out.
HIGHWAY_OBS = {name: ((1, 3, 7, 16, 17, 33)[i % 6],) for i, name in enumerate(mv.VARIANTS)}
HIGHWAY_OBS["widths"] = (3, 7, 16)


def planner_for(v, n, max_obs, kernel, monkeypatch):
    from dmpp_b200.planner import Planner
    monkeypatch.setenv("DP_KERNEL", kernel)                 # read by dp_create
    p = Planner(max_scenes=n, max_obs=max_obs, params=v.params)
    monkeypatch.delenv("DP_KERNEL")
    p.upload_map(v.map)
    return p


def gpu_vs_oracle(p, oracle, the_map, v, sets, what):
    """every set against the oracle with the full check; the untraced run (the production path: the sums of the exactly pruned
    scans stop early, the sweep stops at its first feasible candidate) gives the same records"""
    with bound(oracle, the_map, v):
        for label, H, OX, OY in sets:
            want = oracle.run(H, OX, OY, exhaustive=True, threads=8)
            PX, PY = pad_obs(OX, OY, p.max_obs)
            got = p.run_episodes(H, PX, PY)
            check(got, want, "%s %s" % (what, label))
            fast = p.run_episodes(H, PX, PY, trace=False, paths=False)
            assert fast["rec"].tobytes() == got["rec"].tobytes(), (what, label, "untraced")


def highway_sets(v, seed0, n, cycles):
    from dmpp_b200 import scenes
    return [("highway %d obs" % k,) + scenes.Episodes(v.map, np.arange(seed0, seed0 + n), cycles=cycles, n_obs=k).all_cycles()
            for k in HIGHWAY_OBS[v.name]]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["warp", "group"])
@pytest.mark.parametrize("name", mv.VARIANTS)
def test_cycle_kernels_match_oracle(oracle, the_map, monkeypatch, name, kernel):
    """records, traces, paths, carry and last_path of both cycle kernels and the device map prep against the oracle: highway
    episodes at the variant's obstacle counts, the walled sweep episodes (15 obstacles: both sides of the sweep through the
    deal-out) and junction episodes"""
    v = mv.variant(name)
    p = planner_for(v, 512, 33, kernel, monkeypatch)
    try:
        gpu_vs_oracle(p, oracle, the_map, v, highway_sets(v, 20_000, 512, 20) + episode_sets(v)[1:], "%s %s" % (name, kernel))
    finally:
        p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", mv.VARIANTS)
def test_one_warp_ctas_match_oracle(oracle, the_map, monkeypatch, name):
    """a batch above one wave (> 4144 scenes on a B200) runs the one-warp-per-CTA instantiation of the warp kernel: walled
    episodes on all highway roads (15 obstacles) and the variant's highway obstacle counts"""
    from dmpp_b200 import scenes
    v = mv.variant(name)
    n = 4400
    p = planner_for(v, n, 33, "warp", monkeypatch)
    try:
        walls = ("walled",) + mv.walled(scenes.Episodes(v.map, np.arange(60_000, 60_000 + n), cycles=8, n_obs=9,
                                                        roads=[1, 2, 3, 4, 5] + v.sweep_roads))
        gpu_vs_oracle(p, oracle, the_map, v, [walls] + highway_sets(v, 70_000, n, 6), "%s %d scenes" % (name, n))
    finally:
        p.close()


@pytest.mark.gpu
def test_upload_rejects_the_first_width_with_a_ninth_candidate(the_map):
    """dp_map_upload refuses a lane on which the avoid sweep would enumerate more than DP_MAX_SWEEP candidates per side: for
    each vehicle width the first refused width (in cm) is the first at which the oracle's loop would reach a ninth candidate"""
    from dmpp_b200.planner import DpError, Planner
    for vw in (1.8, 0.5, 1.23):
        first = next(w for w in range(100, 65536) if mv.sweep_k(w / 100.0, vw) > mv.MAX_SWEEP)
        assert mv.sweep_k((first - 1) / 100.0, vw) == mv.MAX_SWEEP
        p = Planner(max_scenes=8, max_obs=4, params=mv.params_with(vehicle_width=vw))
        try:
            roads, conns = mv.lanes_of(the_map)
            roads[1][2][3][777] = first - 1
            p.upload_map(mv.VariantMap(roads, conns))
            roads[1][2][3][777] = first
            with pytest.raises(DpError, match="too wide"):
                p.upload_map(mv.VariantMap(roads, conns))
        finally:
            p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,road,lane,start", [("jitter", 3, 2, 300), ("utm", 4, 1, 500), ("shapes", 5, 1, 800),
                                                  ("shapes", 3, 1, 100)])
def test_dense_sweep_on_variant_lanes(oracle, name, road, lane, start):
    """score_candidates and a sweep session on base paths taken from the jittered lanes (duplicate points included), from
    UTM-like coordinates, across the hairpin and around the tight circle: winner and every dis_lng bit-exact"""
    from dmpp_b200.planner import Planner
    v = mv.variant(name)
    m = v.map
    o = m.lane_pt_off[m.lane_index(road, lane)] + start
    bx, by = m.x[o:o + 200], m.y[o:o + 200]
    if name == "jitter":
        assert (np.hypot(np.diff(bx), np.diff(by)) == 0).any()                  # a duplicated point inside the base path
    rng = np.random.default_rng(road * 10 + lane)
    offset = rng.choice(-2.0 + 0.25 * np.arange(17), 500)
    n_pts = rng.integers(2, 201, 500).astype(np.int32)
    p = Planner(max_scenes=8, max_obs=64)
    sess = p.sweep_session(bx, by, offset, n_pts, 64)
    try:
        for it, n_obs in enumerate((1, 17, 33, 50)):
            idx = rng.integers(5, 195, n_obs)
            ox, oy = bx[idx] + rng.normal(0, 1.2, n_obs), by[idx] + rng.normal(0, 1.2, n_obs)
            dvx, dvy = rng.normal(0, 0.05, n_obs), rng.normal(0, 0.05, n_obs)
            clear = (25.0, 40.0, 10.0, 60.0)[it]
            wbest, wall = oracle.score_candidates(bx, by, offset, n_pts, ox, oy, dvx, dvy, clear_dis=clear)
            best, best_d, allv = p.score_candidates(bx, by, offset, n_pts, ox, oy, dvx, dvy, clear_dis=clear)
            assert best == wbest and np.array_equal(allv, wall), (name, it)
            sb, sd, _ = sess.score(ox, oy, dvx, dvy, clear_dis=clear)
            assert sb == wbest and (sb < 0 or sd == wall[sb]), (name, it, sb, wbest)
    finally:
        sess.close()
        p.close()
