"""Golden vectors: outputs of the UNMODIFIED reference frozen by tests/golden/make_golden.py.  The CPU
oracle is checked against them here (no GPU); the CUDA path is checked against the same files in
test_golden_gpu (marked gpu)."""
import glob
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_records_equal, same
from test_oracle_vs_ref import CARRY

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from make_golden import episodes, sig  # noqa: E402

FILES = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz")))
REC = ["velocity_expect", "path_lat_dis", "remain_dis", "mindist_lon", "brakespeed", "des_acc", "radius", "aim_x", "aim_y",
       "aim_dir", "aim_id", "behavior", "target_roadnum", "target_lanenum", "light", "behavior_to_dlg", "afresh_cause",
       "path_near_id", "path_front_near_id", "n_traj", "afresh_planning", "acc_flag", "cnt"]


def load(path, the_map):
    g = np.load(path)
    s0, n, cyc, nobs = (int(v) for v in g["meta"])
    ep = episodes(the_map, str(g["kind"]), np.arange(s0, s0 + n), cyc, nobs)
    H, OX, OY = ep.all_cycles()
    inp = np.array([np.frombuffer(H.tobytes(), np.uint8).astype(np.uint64).sum(), OX.sum(), OY.sum()])
    assert np.array_equal(inp, g["inputs"]), "scene generator drifted: regenerate the fixtures deliberately"
    return g, H, OX, OY


def test_fixtures_exist():
    assert len(FILES) >= 5


@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
def test_oracle_matches_golden(path, oracle, the_map):
    g, H, OX, OY = load(path, the_map)
    a = oracle.run(H, OX, OY, exhaustive=False)
    clean = a["trace"]["ub_hits"] == 0
    assert_records_equal(a["rec"], g["rec"], REC + ["path_dir_err"], mask=clean, what="record")
    assert (same(sig(a["path_xy"], 2), g["path_sig"]) | ~clean).all()
    assert (same(sig(a["path_ll"], 2), g["path_ll_sig"]) | ~clean).all()
    assert np.array_equal(a["n_calls"], g["n_calls"])
    assert np.array_equal(sig(a["calls"], 2), g["calls_sig"])
    assert_records_equal(a["carry"], g["carry"], CARRY, what="final state")
    assert np.array_equal(sig(a["last_path"], 1), g["last_path_sig"])


@pytest.mark.gpu
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
def test_cuda_matches_golden(path, the_map):
    from dmpp_b200.planner import Planner
    g, H, OX, OY = load(path, the_map)
    p = Planner(H.shape[1], OX.shape[2])
    p.upload_map(the_map)
    a = p.run_episodes(H, OX, OY)
    p.close()
    clean = a["trace"]["ub_hits"] == 0
    assert_records_equal(a["rec"], g["rec"], REC, mask=clean, what="record")
    assert (np.abs(a["rec"]["path_dir_err"] - g["rec"]["path_dir_err"]) <= 1e-9)[clean].all()
    assert (same(sig(a["path_xy"], 2), g["path_sig"]) | ~clean).all()
    assert (same(sig(a["path_ll"], 2), g["path_ll_sig"]) | ~clean).all()
    assert_records_equal(a["carry"], g["carry"], CARRY, what="final state")
    assert np.array_equal(sig(a["last_path"], 1), g["last_path_sig"])
