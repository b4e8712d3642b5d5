"""The batched class facade (host/BatchFacade.h: dmpp::CDecision / dmpp::CPlanning with the reference's public surface,
forwarding to dp_cycle_batch through host/PlannerBatch.h) compiled as a C++ program and run against the oracle's records."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_cpp_facade_matches_oracle(oracle, the_map, tmp_path):
    from dmpp_b200 import scenes
    n, cycles, n_obs = 96, 25, 10
    ep = scenes.Episodes(the_map, np.arange(60_000, 60_000 + n), cycles=cycles, n_obs=n_obs)
    H, OX, OY = ep.all_cycles()
    want = oracle.run(H, OX, OY, exhaustive=False, threads=4)
    ctrl, status = oracle.pack_frames(want["rec"].reshape(-1), want["path_xy"].reshape(-1, 2, 200))
    v, wl, wg = scenes.v2x_events(the_map, H[0], seed=5)
    f0, f1 = oracle.v2x_event(H[0], v, wl, wg, 0), oracle.v2x_event(H[0], v, wl, wg, 1)
    m = the_map
    exe = str(tmp_path / "dmpp_facade_main")                 # (per-test directory: never a file another user left behind)
    pkg = os.path.join(ROOT, "decision-making-and-path-planning_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-o", exe, os.path.join(ROOT, "tests", "cpp", "facade_main.cpp"),
                           "-L" + pkg, "-ldmpp_b200", "-Wl,-rpath," + pkg])
    with tempfile.NamedTemporaryFile(suffix=".bin", delete=False) as f:
        np.array([m.n_roads, m.n_lanes, len(m.conn), m.x.size, n, cycles, n_obs, wl.size], np.int32).tofile(f)
        for a in (m.road_lane_base, m.lane_pt_off, m.conn, m.x, m.y, m.dir, m.lane_width, m.lanechg_attr, H, OX, OY, want["rec"], ctrl, status, v, wl, wg, f0, f1):
            np.ascontiguousarray(a).tofile(f)
        dump = f.name
    try:
        out = subprocess.run([exe, dump], capture_output=True, text=True, timeout=300)
    finally:
        os.unlink(dump)
    assert out.returncode == 0 and "FACADE OK" in out.stdout, out.stdout + out.stderr
