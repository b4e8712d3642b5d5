"""Closed-loop episodes in parts and forked worlds (include/dmpp_b200.h section 17).

CPU side: the checker in parts equals the checker in one call, byte for byte (records, concatenated logs, final world, carry, last
path, every row, state and flag), on highway and junction worlds with every option set and seams inside pos 1 / 2, and on 200-agent
urban worlds; a fork on the checker (every array and the carry gathered on the host) continues every copy as its source.
GPU side: CUDA in parts equals CUDA in one call and both equal the checker in parts (graph updates, direct launches, the group
kernel); the launch count of a part; forks mid-episode against a host gather, their continuations against their sources and the
checker; a fork of more than 4096 worlds; bad arguments."""
import types

import numpy as np
import pytest

from worlds import amparams, jparams, joracle, lcparams, mparams  # noqa: F401

CYCLES = {"highway": 25, "junction": 120, "urban": 120}
SPLITS = {"highway": [(10, 15), (1, 1, 23), (25, 0)], "junction": [(30, 30, 30, 30), (1, 59, 60)], "urban": [(1, 59, 60)]}
N_OBS, MAX_OBS = 10, 14
OPTIONS = ("none", "agents", "v2x0", "v2x1", "all")
ROWS = ("metrics", "lane_change_state", "v2x_flags", "v2x_stats", "v2x_traffic", "v2x_obstacles")


def world(the_map, n, kind, seed0=0, n_obs=N_OBS, max_obs=MAX_OBS):
    from dmpp_b200 import scenes
    return scenes.World(the_map, np.arange(seed0, seed0 + n), n_obs=n_obs, kind=kind, max_obs=max_obs)


def options(w, which, seed0=0):
    """the model keywords of an option set: nothing; metrics + reactive + lane-changing agents; V2X (apply 0 / 1) + agents that obey
    it + the road users the planner sees; everything"""
    from dmpp_b200 import abi, planner, scenes
    if which == "none":
        return {}
    kw = dict(agent_model=(amparams(), w.v0))
    if which in ("agents", "all"):
        kw.update(metrics=mparams(), lane_change=lcparams())
    if which != "agents":
        ev = scenes.V2xEvents(w, np.arange(seed0, seed0 + w.n))
        kw.update(v2x=(abi.V2xWorldParams(0, 0 if which == "v2x0" else 1), ev), traffic=planner.v2x_traffic_params(),
                  obstacles=planner.v2x_obstacle_params())
    return kw


def rows_of(kw):
    return {k: kw.get(k) for k in ("metrics", "lane_change", "v2x", "traffic", "obstacles")}


def checker_parts(jo, w, kind, kw, split, threads=16):
    """the checker in parts: the concatenated records and logs, and the final state"""
    st = jo.closed_loop_state(w.hdr, w.agents, **rows_of(kw))
    outs, k0, prev = [], 0, None
    for i, c in enumerate(split):
        o = jo.run_closed_loop_part(st, k0, c, finish=i == len(split) - 1, prev_rec=prev, wp=jparams(jo, kind), threads=threads, **kw)
        outs.append(o)
        k0 += c
        if c:
            prev = o["rec"][-1]
    cat = {k: np.concatenate([o[k] for o in outs]) for k in ("rec", "hdr_log", "obs_log_x", "obs_log_y")}
    return {**st, **cat}


def used(log, hdr_log):
    return np.arange(log.shape[2])[None, None, :] < hdr_log["n_obs"][:, :, None]


def same_episode(got, want, what, checker=False, whole=True):
    """byte for byte: records, logged headers, final world, carry, last path and every row present in both; the obstacle slots that
    are written (the logs: those the logged header names -- with the road users armed the checker's view buffers start each part from
    zeros --, the final points and lane-change states: the world's agents).  checker: `want` is the checker's, and the records'
    path_dir_err and the metrics' max_abs_dir_err agree to 1e-9 (worlds.check_closed_loop, worlds.check_rows; whole: the records cover the
    whole episode, so max_abs_dir_err is also their maximum)"""
    from worlds import check_closed_loop, check_rows
    rows = [k for k in ROWS if k in got and k in want]
    if checker:
        check_closed_loop(got, want, what)
        if "metrics" in rows:
            if whole:
                check_rows(got["metrics"], want["metrics"], what, rec=got["rec"])
            else:                                           # (the records of the last part only)
                g, w = got["metrics"].copy(), want["metrics"].copy()
                assert (np.abs(g["max_abs_dir_err"] - w["max_abs_dir_err"]) <= 1e-9).all(), what
                g["max_abs_dir_err"] = w["max_abs_dir_err"] = 0
                assert g.tobytes() == w.tobytes(), what + ": metrics"
            rows.remove("metrics")
    else:
        for k in ("rec", "hdr_log", "hdr", "agents", "carry", "last_path"):
            assert got[k].tobytes() == want[k].tobytes(), "%s: %s" % (what, k)
    agents = np.arange(got["ox"].shape[1])[None, :] < want["hdr"]["n_obs"][:, None]
    for k in rows:
        if k == "lane_change_state":
            assert (got[k].view(np.uint8).reshape(agents.shape + (-1,)) == want[k].view(np.uint8).reshape(agents.shape + (-1,)))[agents].all(), \
                "%s: %s" % (what, k)
        else:
            assert got[k].tobytes() == want[k].tobytes(), "%s: %s" % (what, k)
    for k in ("ox", "oy"):
        assert (got[k].view(np.uint64) == want[k].view(np.uint64))[agents].all(), "%s: %s" % (what, k)
    u = used(got["obs_log_x"], want["hdr_log"])
    for k in ("obs_log_x", "obs_log_y"):
        assert (got[k].view(np.uint64)[u] == want[k].view(np.uint64)[u]).all(), "%s: %s" % (what, k)


# ---------------------------------------------------------------- CPU: the checker
@pytest.mark.parametrize("which", OPTIONS)
@pytest.mark.parametrize("kind", ["highway", "junction"])
def test_checker_parts_equal_one_call(joracle, the_map, kind, which):
    w = world(the_map, 256, kind)
    kw = options(w, which)
    one = joracle.run_closed_loop(w.hdr, w.agents, CYCLES[kind], wp=jparams(joracle, kind), threads=16, **kw)
    assert (one["rec"]["brakespeed"] != 0).any()
    if kind == "junction":                                  # the seams fall inside the junction passage
        pos = one["hdr_log"]["pos"]
        assert ((pos[29] > 0) | (pos[59] > 0) | (pos[89] > 0)).any()
    for split in SPLITS[kind]:
        same_episode(checker_parts(joracle, w, kind, kw, split), one, "%s %s %r" % (kind, which, split))


def test_checker_parts_urban_200_agents(joracle, the_map):
    w = world(the_map, 16, "urban", n_obs=200, max_obs=204)
    kw = options(w, "all")
    one = joracle.run_closed_loop(w.hdr, w.agents, CYCLES["urban"], wp=jparams(joracle, "urban"), threads=16, **kw)
    same_episode(checker_parts(joracle, w, "urban", kw, SPLITS["urban"][0]), one, "urban")


def host_fork(arrays, src, dst):
    """array[dst + j] = array[src[j]] along the world axis, for every array"""
    for a in arrays:
        a[dst:dst + len(src)] = a[src]


def forked_inputs(kw, src, dst):
    """copies of the per-world inputs of the option set (v0, the V2X specifications) with the fork applied"""
    kw = dict(kw)
    if "agent_model" in kw:
        am, v0 = kw["agent_model"]
        v0 = v0.copy()
        host_fork([v0], src, dst)
        kw["agent_model"] = (am, v0)
    if "v2x" in kw:
        vp, ev = kw["v2x"]
        spec = ev.spec.copy()
        host_fork([spec], src, dst)
        kw["v2x"] = (vp, types.SimpleNamespace(spec=spec, wp_x=ev.wp_x, wp_y=ev.wp_y))
    return kw


@pytest.mark.parametrize("kind,k1", [("highway", 10), ("junction", 50)])
def test_checker_fork_continues_as_the_source(joracle, the_map, kind, k1):
    """part 1 on 2m worlds, a host fork of worlds src (a permutation of 0..m-1, with repeats) into m .. 2m-1, then the rest: every
    copy's continuation equals its source's"""
    m = 128
    w = world(the_map, 2 * m, kind)
    kw = options(w, "all")
    wp = jparams(joracle, kind)
    st = joracle.closed_loop_state(w.hdr, w.agents, **rows_of(kw))
    a = joracle.run_closed_loop_part(st, 0, k1, wp=wp, threads=16, **kw)
    rng = np.random.default_rng(7)
    src = rng.integers(0, m, m)
    prev = a["rec"][-1].copy()
    host_fork(list(st.values()) + [prev], src, m)
    kw2 = forked_inputs(kw, src, m)
    b = joracle.run_closed_loop_part(st, k1, CYCLES[kind] - k1, finish=True, prev_rec=prev, wp=wp, threads=16, **kw2)
    for k in ("rec", "hdr_log"):
        assert b[k][:, m:].tobytes() == b[k][:, src].tobytes(), k
    for k, v in st.items():
        assert v[m:].tobytes() == v[src].tobytes(), k
    if kind == "junction":
        assert (a["hdr_log"]["pos"][-1] > 0).any()


# ---------------------------------------------------------------- GPU
def planner_for(the_map, n, kind, max_obs=MAX_OBS, env=None):
    from dmpp_b200 import scenes
    from worlds import planner_with
    return planner_with(the_map, n, max_obs, scenes.World.PRE_JUNCTION_PTS[kind], env)


def cuda_parts(p, w, kw, split, log=True):
    ep = p.episode(w.hdr, w.agents, **kw)
    try:
        outs = [ep.run(c, finish=i == len(split) - 1, log=log) for i, c in enumerate(split)]
        st = ep.state()
    finally:
        ep.close()
    keys = ("rec", "hdr_log", "obs_log_x", "obs_log_y") if log else ("rec",)
    return {**st, **{k: np.concatenate([o[k] for o in outs]) for k in keys}, "graphs": [o["graph"] for o in outs]}


@pytest.mark.gpu
@pytest.mark.parametrize("which", OPTIONS)
@pytest.mark.parametrize("kind", ["highway", "junction"])
def test_gpu_parts_equal_one_call_and_checker(joracle, the_map, kind, which):
    """4096 worlds: the graph (replayed and updated part by part) in every split against one call and the checker in parts"""
    n = 4096
    w = world(the_map, n, kind)
    kw = options(w, which)
    want = checker_parts(joracle, w, kind, kw, SPLITS[kind][-1])
    p = planner_for(the_map, n, kind)
    try:
        one = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], repeat=2, **kw)
        assert one["graph"]
        same_episode(one, want, "%s %s one call" % (kind, which), checker=True)
        for split in SPLITS[kind]:
            got = cuda_parts(p, w, kw, split)
            what = "%s %s %r" % (kind, which, split)
            assert all(got["graphs"]), what
            same_episode(got, one, what)
            same_episode(got, want, what + " checker", checker=True)
    finally:
        p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
@pytest.mark.parametrize("kind", ["highway", "junction"])
def test_gpu_parts_direct_launches_and_group_kernel(joracle, the_map, kind, env):
    n = 4096
    w = world(the_map, n, kind)
    kw = options(w, "all")
    want = checker_parts(joracle, w, kind, kw, SPLITS[kind][0])
    p = planner_for(the_map, n, kind, env=env)
    try:
        one = p.run_closed_loop(w.hdr, w.agents, CYCLES[kind], **kw)
        assert not one["graph"]
        for split in SPLITS[kind]:
            got = cuda_parts(p, w, kw, split)
            assert not any(got["graphs"])
            same_episode(got, one, "%s %r %r" % (kind, env, split))
            same_episode(got, want, "%s %r %r checker" % (kind, env, split), checker=True)
    finally:
        p.close()


@pytest.mark.gpu
def test_gpu_parts_urban_200_agents(joracle, the_map):
    w = world(the_map, 256, "urban", n_obs=200, max_obs=204)
    kw = options(w, "all")
    want = checker_parts(joracle, w, "urban", kw, (60, 60))
    p = planner_for(the_map, 256, "urban", max_obs=204)
    try:
        got = cuda_parts(p, w, kw, SPLITS["urban"][0])
    finally:
        p.close()
    same_episode(got, want, "urban", checker=True)


def dev_buf(p, nbytes):
    import ctypes as C
    a = C.c_void_p()
    assert p.lib.dp_dev_alloc(p.ctx, C.byref(a), C.c_size_t(nbytes)) == 0
    return a.value


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["none", "v2x1"])
def test_gpu_launch_counts(the_map, which):
    """(k0 == 0) + cycles * (3 + V2X + obstacles) + finish * (V2X + obstacles); k0 = 0, finish = 1 is dp_run_closed_loop_dev launch
    for launch and byte for byte"""
    n, kind = 1024, "highway"
    w = world(the_map, n, kind)
    kw = options(w, which)
    extra = 2 if which != "none" else 0
    p = planner_for(the_map, n, kind)
    try:
        ep = p.episode(w.hdr, w.agents, **kw)
        try:
            d = ep.d
            rec = dev_buf(p, 25 * n * 128)
            c0 = p.launch_count()
            p.run_closed_loop_dev(n, 25, d["hdr"], d["agents"], d["ox"], d["oy"], rec)
            one = p.launch_count() - c0
            st_one = ep.state()
            ep.restart()
            counts, prev = [], None
            for k0, cycles, finish in ((0, 10, 0), (10, 1, 0), (11, 14, 0), (25, 0, 1)):
                c0 = p.launch_count()
                p.run_closed_loop_part_dev(n, k0, cycles, finish, d["hdr"], d["agents"], d["ox"], d["oy"], rec, prev)
                counts.append(p.launch_count() - c0)
                assert p.closed_loop_is_graph()
                prev = rec + (cycles - 1) * n * 128 if cycles else prev   # (rec reused as a ring: its last row is the next prev_rec)
            st_parts = ep.state()
            ep.restart()
            c0 = p.launch_count()
            p.run_closed_loop_part_dev(n, 0, 25, 1, d["hdr"], d["agents"], d["ox"], d["oy"], rec)
            zero_one = p.launch_count() - c0
            st_zero_one = ep.state()
            p.lib.dp_dev_free(p.ctx, rec)
        finally:
            ep.close()
    finally:
        p.close()
    per = 3 + extra
    assert one == zero_one == 1 + 25 * per + extra, (one, zero_one)
    assert counts == [1 + 10 * per, per, 14 * per, extra], counts
    for k in st_one:
        if k != "graph":
            assert st_parts[k].tobytes() == st_one[k].tobytes() == st_zero_one[k].tobytes(), k


def gather(st, src, dst):
    """the host gather a fork must equal: copies of every per-world array with array[dst + j] = array[src[j]]"""
    out = {k: v.copy() for k, v in st.items() if k != "graph"}
    host_fork(list(out.values()), src, dst)
    return out


def device_inputs(ep):
    """the Episode's device-only per-world buffers: v0, the V2X specifications, prev_rec"""
    from dmpp_b200 import abi
    n, mo, o = ep.n, ep.mo, {}
    for k, dt, shape in (("v0", np.float64, (n, mo)), ("v2x_spec", abi.v2x_event_spec, (n,)), ("prev_rec", abi.plan_record, (n,))):
        if k in ep.d:
            o[k] = np.zeros(shape, dt)
            ep._d2h(o[k], ep.d[k], o[k].nbytes)
    ep.p.lib.dp_stream_sync(ep.p.ctx, None)
    return o


@pytest.mark.gpu
def test_gpu_fork_mid_junction_episode(joracle, the_map):
    """512 junction worlds forked into 512 more in pos 1 / 2 with every model armed: the fork equals a host gather of every buffer
    and the carry, worlds outside dst are untouched, every copy's next part equals its source's, and the checker continued from the
    forked state equals CUDA"""
    m, kind, k1 = 512, "junction", 50
    w = world(the_map, 2 * m, kind)
    kw = options(w, "all")
    rng = np.random.default_rng(3)
    src = rng.permutation(m)[: m - 16]
    src = np.concatenate([src, src[:16]]).astype(np.int32)   # (repeated sources)
    p = planner_for(the_map, 2 * m, kind)
    try:
        ep = p.episode(w.hdr, w.agents, **kw)
        try:
            a = ep.run(k1, log=False)
            before, inp_before = ep.state(), device_inputs(ep)
            assert (before["hdr"]["pos"][:m] > 0).sum() > 50
            ep.fork(src, m)
            after, inp_after = ep.state(), device_inputs(ep)
            want, want_inp = gather(before, src, m), gather(inp_before, src, m)
            for k in want:
                assert after[k].tobytes() == want[k].tobytes(), k
            for k in want_inp:
                assert inp_after[k].tobytes() == want_inp[k].tobytes(), k
            b = ep.run(CYCLES[kind] - k1, finish=True)
            end = ep.state()
        finally:
            ep.close()
    finally:
        p.close()
    assert (inp_after["prev_rec"][:m].tobytes() == a["rec"][-1][:m].tobytes())
    for k in ("rec", "hdr_log"):
        assert b[k][:, m:].tobytes() == b[k][:, src].tobytes(), k
    for k, v in end.items():
        if k != "graph":
            assert v[m:].tobytes() == v[src].tobytes(), k
    st = {k: v for k, v in after.items() if k != "graph"}
    kw2 = forked_inputs(kw, src, m)
    c = joracle.run_closed_loop_part(st, k1, CYCLES[kind] - k1, finish=True, prev_rec=inp_after["prev_rec"], wp=jparams(joracle, kind),
                                     threads=16, **kw2)
    same_episode({**end, **b}, {**st, **c}, "checker from the fork", checker=True, whole=False)


@pytest.mark.gpu
def test_gpu_fork_of_more_than_4096_worlds(the_map):
    """odd max_obs (8-byte rows), 4100 sources: two launches"""
    m, kind = 4100, "highway"
    w = world(the_map, 2 * m, kind, max_obs=11)
    kw = options(w, "agents")
    src = np.arange(m, dtype=np.int32)[::-1].copy()
    p = planner_for(the_map, 2 * m, kind, max_obs=11)
    try:
        ep = p.episode(w.hdr, w.agents, **kw)
        try:
            ep.run(5, log=False)
            before, inp_before = ep.state(), device_inputs(ep)
            c0 = p.launch_count()
            ep.fork(src, m)
            assert p.launch_count() - c0 == 2
            after, inp_after = ep.state(), device_inputs(ep)
            b = ep.run(5, finish=True, log=False)
            end = ep.state()
        finally:
            ep.close()
    finally:
        p.close()
    want, want_inp = gather(before, src, m), gather(inp_before, src, m)
    for k in want:
        assert after[k].tobytes() == want[k].tobytes(), k
    for k in want_inp:
        assert inp_after[k].tobytes() == want_inp[k].tobytes(), k
    assert b["rec"][:, m:].tobytes() == b["rec"][:, src].tobytes()
    assert end["metrics"][m:].tobytes() == end["metrics"][src].tobytes()


@pytest.mark.gpu
def test_gpu_bad_arguments(the_map):
    import ctypes as C
    from dmpp_b200.planner import DpError
    n, kind = 64, "highway"
    w = world(the_map, n, kind)
    kw = options(w, "all")
    p = planner_for(the_map, n, kind)
    try:
        ep = p.episode(w.hdr, w.agents, **kw)
        try:
            d = ep.d
            rec = dev_buf(p, 4 * n * 128)
            run = lambda k0=1, cycles=1, finish=0, prev=d["prev_rec"]: p.run_closed_loop_part_dev(
                n, k0, cycles, finish, d["hdr"], d["agents"], d["ox"], d["oy"], rec, prev)
            run(k0=0)
            for bad in (dict(k0=-1), dict(finish=2), dict(finish=-1), dict(prev=None)):
                with pytest.raises(DpError):
                    run(**bad)
            fork = lambda src=(0, 1), dst=2, prev=d["prev_rec"], nn=n: p.world_fork_dev(nn, np.array(src), dst, d["hdr"], d["agents"],
                                                                                      d["ox"], d["oy"], prev)
            fork()
            fork(src=(), dst=n)                             # count 0: nothing
            for bad in (dict(src=(0, n)), dict(src=(-1,)), dict(src=(2,)), dict(src=(0, 3)), dict(dst=-1), dict(dst=n - 1),
                        dict(prev=None), dict(nn=n + 1)):
                with pytest.raises(DpError):
                    fork(**bad)
            rc = p.lib.dp_world_fork_dev(p.ctx, 1, n, np.array([0], np.int32).ctypes.data, 1, 1, d["hdr"], d["agents"], d["ox"], d["oy"],
                                         d["prev_rec"], None)
            assert rc != 0                                  # first + n > max_scenes
            z = np.zeros((n, ep.mo))
            p.set_tracks(z, z, z, 5)
            with pytest.raises(DpError):
                fork()
            p.clear_tracks()
            p.lib.dp_dev_free(p.ctx, C.c_void_p(rec))
        finally:
            ep.close()
    finally:
        p.close()
