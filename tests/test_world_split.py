"""Splitting worlds between the parts of an episode (include/dmpp_b200.h section 18).

CPU side: layouts and defaults; spec_exp against math.exp; a numpy restatement of the select and the perturbation against the checker
on 10 000 random populations; the invariants of the assignment; the estimator on a Gaussian random walk with a known answer; checker
episodes in which every copy continues as its source, and beta = 0 as parts plus perturbation.
GPU side: byte parity with the checker in parts with splits (graph, direct launches, group kernel); beta = 0 with no noise against
the same parts without splits, and the launch count; a 131 072-world split; the fork copies the split rows; arm / disarm / re-arm and
bad arguments; the beta = 0 and beta > 0 estimates of one source agree."""
import math

import numpy as np
import pytest

from test_episode_parts import options, planner_for, rows_of, same_episode, world
from worlds import jparams, joracle  # noqa: F401

MASK = (1 << 64) - 1
HI = 1 << 63


# ---------------------------------------------------------------- a numpy restatement of the rules
def mix(z):
    z ^= z >> 30; z = (z * 0xbf58476d1ce4e5b9) & MASK
    z ^= z >> 27; z = (z * 0x94d049bb133111eb) & MASK
    return z ^ (z >> 31)


def key(seed, level, a, b):
    return mix(mix(mix(mix(seed) ^ level) ^ a) ^ b)


def u01(h):
    return float(h >> 11) * 2.0 ** -53


def select_np(jo, sp, M, g, level, c, rows, grp):
    """population g: clearances c[M], rows[M] / grp (a 0-d split_group) in place; returns N and map (relative to the population)"""
    if level == 0:
        rows["v_prev"], rows["lw"], rows["root"], rows["pad"] = -sp.c_max, 1.0, np.arange(M), 0
        grp["norm"], grp["levels"], grp["copies"], grp["roots_alive"], grp["pad"] = 1.0, 0, 0, M, 0
    V = -np.where(c < sp.c_max, c, sp.c_max)
    w = jo.spec_exp(sp.beta * (V - rows["v_prev"]))
    C = np.zeros(M)
    acc = 0.0
    for j in range(M):                                      # (sequential: the order the rules fix)
        acc = acc + w[j]
        C[j] = acc
    W = C[-1]
    u = u01(key(sp.seed, level, HI | g, 0))
    A = np.clip(np.ceil((M * C) / W - u), 0, M).astype(np.int64)
    A[-1] = M
    N = np.diff(np.concatenate([[0], A]))
    rows["lw"] = rows["lw"] * w
    rows["v_prev"] = V
    grp["norm"] = grp["norm"] * (W / M)
    grp["levels"] += 1
    m = np.full(M, -1, np.int32)
    m[np.flatnonzero(N == 0)] = np.repeat(np.arange(M), np.maximum(N - 1, 0))
    grp["copies"] += np.maximum(N - 1, 0).sum()
    grp["roots_alive"] = len(np.unique(rows["root"][np.where(m >= 0, m, np.arange(M))]))
    return N, m


def perturb_np(sp, level, hdr, agents, v0=None):
    n, mo = agents.shape
    for i in range(n):
        for k in range(min(int(hdr["n_obs"][i]), mo)):
            f = 1.0 + sp.amp_v * (2.0 * u01(key(sp.seed, level, i, 2 * k)) - 1.0)
            agents["v"][i, k] = agents["v"][i, k] * f
            if v0 is not None:
                v0[i, k] = v0[i, k] * (1.0 + sp.amp_v0 * (2.0 * u01(key(sp.seed, level, i, 2 * k + 1)) - 1.0))


def split_params(**kw):
    from dmpp_b200 import planner
    return planner.split_params(**kw)


def gather(arrays, m):
    """array[i] = array[m[i]] where m[i] >= 0, along the world axis, for every array"""
    d = np.flatnonzero(m >= 0)
    for a in arrays:
        a[d] = a[m[d]]


# ---------------------------------------------------------------- CPU
def test_layouts_and_defaults(joracle):
    from dmpp_b200 import abi
    import ctypes as C
    assert C.sizeof(abi.SplitParams) == joracle.split_sizeof(0) == 48
    assert abi.split_row.itemsize == joracle.split_sizeof(1) == 24
    assert abi.split_group.itemsize == joracle.split_sizeof(2) == 24
    sp = split_params()
    assert (sp.group, sp.pad, sp.beta, sp.c_max, sp.amp_v, sp.amp_v0, sp.seed) == (256, 0, 0.5, 10.0, 0.1, 0.0, 0)


def test_spec_exp(joracle):
    x = np.random.default_rng(5).uniform(-50, 50, 10 ** 6)
    y = joracle.spec_exp(x)
    want = np.array([math.exp(v) for v in x])
    assert (np.abs(y - want) <= 2 * np.spacing(want)).all()
    assert joracle.spec_exp([0.0])[0] == 1.0 and joracle.spec_exp([-0.0])[0] == 1.0


def test_select_and_perturb_restated(joracle):
    """10 000 random populations (M in 1 .. 1024, tied, zero and +inf clearances, beta = 0 on every tenth) over two levels"""
    from dmpp_b200 import abi
    rng = np.random.default_rng(11)
    for t in range(10000):
        M = int(rng.integers(1, 1025)) if t % 50 else 1024
        sp = split_params(group=M, beta=0.0 if t % 10 == 0 else float(rng.uniform(0, 5)), c_max=float(rng.uniform(0.5, 10)),
                          seed=int(rng.integers(0, 2 ** 63)))
        rows, grp = np.zeros(M, abi.split_row), np.zeros(1, abi.split_group)
        rows_np, grp_np = rows.copy(), grp.copy()
        for level in (0, int(rng.integers(1, 40))):
            c = rng.choice([0.0, np.inf, 1.5, sp.c_max], M) if t % 3 == 0 else rng.uniform(0, 12, M)
            met = np.zeros(M, abi.episode_metrics)
            met["min_clearance"] = c
            m = joracle.split_select(sp, level, met, rows, grp)
            N, m_np = select_np(joracle, sp, M, 0, level, c, rows_np, grp_np[0])
            assert m.tobytes() == m_np.tobytes(), (t, level)
            assert rows.tobytes() == rows_np.tobytes() and grp.tobytes() == grp_np.tobytes(), (t, level)
            # invariants: sum N = M, survivors keep their slots, sources and destinations are disjoint
            assert N.sum() == M and (N >= 0).all()
            assert ((m >= 0) == (N == 0)).all()
            assert not np.isin(m[m >= 0], np.flatnonzero(m >= 0)).any()
            assert (N[m[m >= 0]] >= 2).all()
            if sp.beta == 0:
                assert (m == -1).all() and (rows["lw"] == 1).all() and grp["norm"][0] == 1.0
            gather([rows, rows_np], m)
    hdr = np.zeros(64, abi.scene_hdr)
    hdr["n_obs"] = rng.integers(0, 14, 64)
    agents = np.zeros((64, 12), abi.agent)
    agents["v"] = rng.uniform(0, 30, agents.shape)
    v0 = rng.uniform(0, 30, agents.shape)
    for sp in (split_params(amp_v=0.3, amp_v0=0.2, seed=9), split_params(amp_v=0.0, amp_v0=0.0)):
        a1, a2, w1, w2 = agents.copy(), agents.copy(), v0.copy(), v0.copy()
        joracle.perturb(sp, 3, hdr, a1, w1)
        perturb_np(sp, 3, hdr, a2, w2)
        assert a1.tobytes() == a2.tobytes() and w1.tobytes() == w2.tobytes()
        if sp.amp_v == 0:
            assert a1.tobytes() == agents.tobytes() and w1.tobytes() == v0.tobytes()
        else:
            assert (a1["v"] != agents["v"]).any() and (w1 != v0).any()


def random_walk_split(joracle, beta, P, M, T, every, a, seed):
    """P populations of M Gaussian random walks of T steps; a split every `every` steps; the score is section 11's row with
    min_clearance = a - running max (c_max = a) and the walk's fresh increments as the perturbation.  Returns p_g per population"""
    from dmpp_b200 import abi, planner
    n = P * M
    sp = split_params(group=M, beta=beta, c_max=a, seed=seed)
    rng = np.random.default_rng(seed)
    s, top = np.zeros(n), np.zeros(n)
    met = np.zeros(n, abi.episode_metrics)
    rows, groups = np.zeros(n, abi.split_row), np.zeros(P, abi.split_group)
    for k in range(T):
        s += rng.standard_normal(n)
        top = np.maximum(top, s)
        if (k + 1) % every == 0 and k + 1 < T:
            met["min_clearance"] = a - top
            m = joracle.split_select(sp, (k + 1) // every - 1, met, rows, groups)
            gather([s, top, rows], m)
    met["min_clearance"] = a - top
    met["first_collision_step"] = np.where(top >= a, 1, -1)
    return planner.split_estimate({"metrics": met, "split_rows": rows, "split_groups": groups})


def test_estimator_on_a_random_walk(joracle):
    """P(max of a 50-step Gaussian walk >= a) at about 1e-3 from 10^6 plain samples; the split estimate (mean over populations) lies
    within 4 standard errors of it, and beta > 0 has the smaller standard error at the same budget"""
    T, a = 50, 21.0
    rng = np.random.default_rng(123)
    hits = 0
    for _ in range(10):
        hits += (np.cumsum(rng.standard_normal((100000, T)), axis=1).max(axis=1) >= a).sum()
    p = hits / 1e6
    assert 3e-4 < p < 3e-3, p
    P, M = 64, 256
    est = {}
    for beta in (0.0, 0.2):
        g = random_walk_split(joracle, beta, P, M, T, 5, a, seed=77)
        est[beta] = (g.mean(), g.std(ddof=1) / math.sqrt(P))
    for beta, (mean, se) in est.items():
        sd = math.hypot(se, math.sqrt(p * (1 - p) / 1e6))
        assert abs(mean - p) <= 4 * sd, (beta, mean, se, p)
    assert est[0.2][1] < est[0.0][1], est


def checker_split_parts(jo, w, kind, kw, sp, cycles, every, perturb_only=False):
    """the checker in parts of `every` cycles with a split (select -> host gather -> perturb) at every seam; with perturb_only the
    seams only perturb.  Returns the concatenated records and logs, the final state with the split rows, the per-split maps, the
    inputs (v0, the V2X specifications) as the splits left them, every part's outputs and the state after every part"""
    from dmpp_b200 import abi
    kw = dict(kw)
    v0 = None
    if "agent_model" in kw:
        am, v0 = kw["agent_model"]
        v0 = v0.copy()
        kw["agent_model"] = (am, v0)
    spec = None
    if "v2x" in kw:
        import types
        vp, ev = kw["v2x"]
        spec = ev.spec.copy()
        kw["v2x"] = (vp, types.SimpleNamespace(spec=spec, wp_x=ev.wp_x, wp_y=ev.wp_y))
    st = jo.closed_loop_state(w.hdr, w.agents, **rows_of(kw))
    n = w.n
    rows, groups = np.zeros(n, abi.split_row), np.zeros(n // sp.group, abi.split_group)
    outs, maps, states, k0, prev = [], [], [], 0, None
    while k0 < cycles:
        c = min(every, cycles - k0)
        o = jo.run_closed_loop_part(st, k0, c, finish=k0 + c == cycles, prev_rec=prev, wp=jparams(jo, kind), threads=16, **kw)
        outs.append(o)
        prev = o["rec"][-1].copy()
        k0 += c
        states.append({**{k: v.copy() for k, v in st.items()}, "prev_rec": prev.copy(), "split_rows": rows.copy(),
                       **({"v0": v0.copy()} if v0 is not None else {})})
        if k0 < cycles:
            level = k0 // every - 1
            if not perturb_only:
                m = jo.split_select(sp, level, st["metrics"], rows, groups)
                gather(list(st.values()) + [prev, rows] + [x for x in (v0, spec) if x is not None], m)
                maps.append(m)
            jo.perturb(sp, level, st["hdr"], st["agents"], v0)
    cat = {k: np.concatenate([o[k] for o in outs]) for k in ("rec", "hdr_log", "obs_log_x", "obs_log_y")}
    return {**st, **cat, "split_rows": rows, "split_groups": groups, "maps": maps, "v0": v0, "v2x_spec": spec, "prev_rec": prev,
            "parts": outs, "states": states}


def test_checker_copies_continue_as_their_sources(joracle, the_map):
    """4 populations of M = 64 highway worlds, 25 cycles, a split every 5 with no noise: every copy's next part (records, logs) and
    its world, carry, rows, states, inputs and split row after that part equal its source's"""
    M, kind = 64, "highway"
    w = world(the_map, 4 * M, kind)
    kw = options(w, "agents")
    sp = split_params(group=M, beta=2.0, amp_v=0.0, seed=4)
    got = checker_split_parts(joracle, w, kind, kw, sp, 25, 5)
    assert sum((m >= 0).sum() for m in got["maps"]) > 0
    for i, m in enumerate(got["maps"]):
        d = np.flatnonzero(m >= 0)
        nxt = got["parts"][i + 1]
        for k in ("rec", "hdr_log"):
            assert nxt[k][:, d].tobytes() == nxt[k][:, m[d]].tobytes(), (i, k)
        after = got["states"][i + 1]
        assert {"hdr", "agents", "ox", "oy", "carry", "last_path", "metrics", "lane_change_state", "v0", "split_rows"} <= set(after)
        for k, v in after.items():
            assert v[d].tobytes() == v[m[d]].tobytes(), (i, k)
    assert (got["split_groups"]["levels"] == 4).all()
    assert (got["split_groups"]["copies"] > 0).all()


def test_checker_beta_zero_is_parts_plus_perturbation(joracle, the_map):
    kind = "highway"
    w = world(the_map, 128, kind)
    kw = options(w, "agents")
    sp = split_params(group=32, beta=0.0, amp_v=0.1, amp_v0=0.05, seed=2)
    a = checker_split_parts(joracle, w, kind, kw, sp, 25, 5)
    b = checker_split_parts(joracle, w, kind, kw, sp, 25, 5, perturb_only=True)
    assert all((m == -1).all() for m in a["maps"])
    for k in ("rec", "hdr", "agents", "metrics", "v0"):
        assert a[k].tobytes() == b[k].tobytes(), k
    assert (a["split_rows"]["lw"] == 1).all() and (a["split_groups"]["norm"] == 1).all()
    assert (a["rec"] != checker_split_parts(joracle, w, kind, kw, split_params(group=32, beta=0.0, amp_v=0.0), 25, 5)["rec"]).any()


# ---------------------------------------------------------------- GPU
def device_inputs(ep):
    from dmpp_b200 import abi
    n, mo, o = ep.n, ep.mo, {}
    for k, dt, shape in (("v0", np.float64, (n, mo)), ("v2x_spec", abi.v2x_event_spec, (n,)), ("prev_rec", abi.plan_record, (n,))):
        if k in ep.d:
            o[k] = np.zeros(shape, dt)
            ep._d2h(o[k], ep.d[k], o[k].nbytes)
    ep.p.lib.dp_stream_sync(ep.p.ctx, None)
    return o


def cuda_split_parts(p, w, kw, sp, cycles, every, splits=True):
    ep = p.episode(w.hdr, w.agents, split=sp, **kw)
    try:
        outs, maps, k0, counts = [], [], 0, []
        while k0 < cycles:
            c = min(every, cycles - k0)
            outs.append(ep.run(c, finish=k0 + c == cycles))
            k0 += c
            if k0 < cycles and splits:
                c0 = p.launch_count()
                ep.split(k0 // every - 1)
                counts.append(p.launch_count() - c0)
                maps.append(p.split_map(w.n))
        st = ep.state()
        st.update(device_inputs(ep))
    finally:
        ep.close()
    cat = {k: np.concatenate([o[k] for o in outs]) for k in ("rec", "hdr_log", "obs_log_x", "obs_log_y")}
    return {**st, **cat, "maps": maps, "counts": counts, "graphs": [o["graph"] for o in outs]}


def check_split_parity(got, want, what):
    same_episode(got, want, what, checker=True, whole=False)     # (prev_rec is the last part's last row of records: compared there)
    for k in ("split_rows", "split_groups", "v0", "v2x_spec"):
        if want.get(k) is not None:
            assert got[k].tobytes() == want[k].tobytes(), "%s: %s" % (what, k)
    assert len(got["maps"]) == len(want["maps"])
    for a, b in zip(got["maps"], want["maps"]):
        assert a.tobytes() == b.tobytes(), what + ": map"


@pytest.mark.gpu
@pytest.mark.parametrize("kind,cycles,every", [("highway", 25, 5), ("junction", 120, 10)])
def test_gpu_split_parity_with_checker(joracle, the_map, kind, cycles, every):
    """4096 worlds (16 populations of 256), every model armed, a split at every seam: byte parity with the checker"""
    n = 4096
    w = world(the_map, n, kind)
    kw = options(w, "all")
    sp = split_params(group=256, beta=0.4, amp_v=0.1, amp_v0=0.05, seed=17)
    want = checker_split_parts(joracle, w, kind, kw, sp, cycles, every)
    assert sum((m >= 0).sum() for m in want["maps"]) > 0
    p = planner_for(the_map, n, kind)
    try:
        got = cuda_split_parts(p, w, kw, sp, cycles, every)
    finally:
        p.close()
    assert all(got["graphs"])
    check_split_parity(got, want, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DP_EPISODE_GRAPH": "0"}, {"DP_KERNEL": "group"}])
def test_gpu_split_direct_launches_and_group_kernel(joracle, the_map, env):
    n, kind = 4096, "highway"
    w = world(the_map, n, kind)
    kw = options(w, "all")
    sp = split_params(group=256, beta=0.4, amp_v=0.1, seed=5)
    want = checker_split_parts(joracle, w, kind, kw, sp, 25, 5)
    p = planner_for(the_map, n, kind, env=env)
    try:
        got = cuda_split_parts(p, w, kw, sp, 25, 5)
    finally:
        p.close()
    assert not any(got["graphs"])
    check_split_parity(got, want, repr(env))


@pytest.mark.gpu
def test_gpu_identity_and_launch_count(the_map):
    """beta = 0 and both amplitudes 0: everything but the split rows equals the same parts without splits; 3 launches per split"""
    n, kind = 4096, "junction"
    w = world(the_map, n, kind)
    kw = options(w, "all")
    sp = split_params(group=256, beta=0.0, amp_v=0.0, amp_v0=0.0)
    p = planner_for(the_map, n, kind)
    try:
        a = cuda_split_parts(p, w, kw, sp, 120, 10)
        b = cuda_split_parts(p, w, kw, sp, 120, 10, splits=False)
    finally:
        p.close()
    assert a["counts"] == [3] * 11
    assert all((m == -1).all() for m in a["maps"])
    same_episode(a, b, "identity")
    for k in ("v0", "v2x_spec", "prev_rec"):
        assert a[k].tobytes() == b[k].tobytes(), k
    assert (a["split_rows"]["lw"] == 1).all() and (a["split_groups"]["norm"] == 1).all() and (a["split_groups"]["levels"] == 11).all()


@pytest.mark.gpu
def test_gpu_split_of_131072_worlds(joracle, the_map):
    """512 populations of 256 after 5 cycles: the select against the checker's, the copy against a host gather, the perturbation
    against the checker's"""
    n, kind = 131072, "highway"
    w = world(the_map, n, kind, max_obs=10)
    kw = options(w, "agents")
    sp = split_params(group=256, beta=0.8, amp_v=0.1, amp_v0=0.1, seed=8)
    p = planner_for(the_map, n, kind, max_obs=10)
    try:
        ep = p.episode(w.hdr, w.agents, split=sp, **kw)
        try:
            ep.run(5, log=False)
            before = ep.state()
            before.update(device_inputs(ep))
            ep.split(0)
            m = p.split_map(n)
            after = ep.state()
            after.update(device_inputs(ep))
        finally:
            ep.close()
    finally:
        p.close()
    from dmpp_b200 import abi
    rows, groups = np.zeros(n, abi.split_row), np.zeros(n // 256, abi.split_group)
    want_m = joracle.split_select(sp, 0, before["metrics"], rows, groups)
    assert m.tobytes() == want_m.tobytes() and (m >= 0).sum() > 1000
    assert after["split_groups"].tobytes() == groups.tobytes()
    want = {k: v.copy() for k, v in before.items() if k not in ("graph", "split_rows", "split_groups")}
    gather(list(want.values()) + [rows], m)
    joracle.perturb(sp, 0, want["hdr"], want["agents"], want["v0"])
    assert after["split_rows"].tobytes() == rows.tobytes()
    for k in want:
        assert after[k].tobytes() == want[k].tobytes(), k


@pytest.mark.gpu
def test_gpu_fork_copies_the_split_rows_and_bad_arguments(the_map):
    from dmpp_b200.planner import DpError
    n, kind = 256, "highway"
    w = world(the_map, n, kind)
    kw = options(w, "all")
    sp = split_params(group=64, beta=1.0, seed=3)
    p = planner_for(the_map, n, kind)
    try:
        ep = p.episode(w.hdr, w.agents, split=sp, **kw)
        try:
            d = ep.d
            ep.run(5)
            ep.split(0)
            before = ep.state()
            src = np.arange(0, 64, dtype=np.int32)
            ep.fork(src, 128)
            after = ep.state()
            assert after["split_rows"][128:192].tobytes() == before["split_rows"][:64].tobytes()
            split = lambda nn=n, level=1, prev=d["prev_rec"]: p.world_split_dev(nn, level, d["hdr"], d["agents"], d["ox"], d["oy"], prev)
            for bad in (dict(nn=n - 1), dict(nn=n + 64), dict(level=-1), dict(prev=None)):
                with pytest.raises(DpError):
                    split(**bad)
            for bad in (dict(group=0), dict(group=1025), dict(group=7), dict(beta=-1.0), dict(beta=6.0), dict(c_max=0.0),
                        dict(amp_v=1.0), dict(amp_v0=-0.1), dict(beta=float("nan"))):
                with pytest.raises(DpError):
                    p.set_split(split_params(**{"group": 64, **bad}), n, d["split_rows"], d["split_groups"])
            z = np.zeros((n, ep.mo))
            p.set_tracks(z, z, z, 5)
            with pytest.raises(DpError):
                split()
            p.clear_tracks()
            p.set_metrics(None, None)                       # the score is the metrics row
            with pytest.raises(DpError):
                split()
            p.set_metrics(kw["metrics"], d["metrics"])
            p.set_split(None, 0, None, None)                # disarmed: the fork leaves the rows alone, the split refuses
            rows = ep.state()["split_rows"]
            ep.fork(np.arange(64, 128, dtype=np.int32), 128)
            assert ep.state()["split_rows"].tobytes() == rows.tobytes()
            with pytest.raises(DpError):
                split()
            p.set_split(sp, n, d["split_rows"], d["split_groups"])   # re-armed
            split()
            split(level=0)
            g = ep.state()["split_groups"]
            assert (g["levels"] == 1).all()
        finally:
            ep.close()
    finally:
        p.close()


def effect_run(p, w, kw, sp, cycles=120, every=10):
    from dmpp_b200 import planner
    ep = p.episode(w.hdr, w.agents, split=sp, **kw)
    try:
        for k0 in range(0, cycles, every):
            ep.run(every, finish=k0 + every == cycles, log=False)
            if k0 + every < cycles:
                ep.split(k0 // every)
        return planner.split_estimate(ep.state())
    finally:
        ep.close()


def junction_copies(the_map, seed, P, M):
    from dmpp_b200 import scenes
    return scenes.World(the_map, np.full(P * M, seed), n_obs=10, kind="junction", max_obs=14)


@pytest.mark.gpu
def test_gpu_effect_estimates_agree(the_map):
    """16 populations of 256 copies of one junction source, amp_v = 0.1, a split every 10 cycles: the first source among seeds
    0 .. 63 whose beta = 0 estimate lies in (0.05, 0.5) has beta = 0 and beta > 0 estimates within 4 combined standard errors"""
    P, M = 16, 256
    p = planner_for(the_map, P * M, "junction")
    try:
        for seed in range(64):
            w = junction_copies(the_map, seed, P, M)
            kw = options(w, "agents")
            g0 = effect_run(p, w, kw, split_params(group=M, beta=0.0, amp_v=0.1, seed=seed))
            if 0.05 < g0.mean() < 0.5:
                g1 = effect_run(p, w, kw, split_params(group=M, beta=0.3, amp_v=0.1, seed=seed + 1000))
                se = math.hypot(g0.std(ddof=1), g1.std(ddof=1)) / math.sqrt(P)
                assert abs(g0.mean() - g1.mean()) <= 4 * se, (seed, g0.mean(), g1.mean(), se)
                return
        pytest.fail("no junction source among seeds 0 .. 63 with 0.05 < p < 0.5")
    finally:
        p.close()
