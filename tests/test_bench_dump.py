"""bench.py --dump-outputs: the files hold the plan records of the LAST timed step (warmup + steps cycles into the episode),
field for field what the oracle computes for that cycle, and --steps sets how many steps are timed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_records_equal
from test_gpu_parity import DIR_ERR_TOL, REC_EXACT

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_timed_step(oracle, the_map, tmp_path):
    from dmpp_b200 import abi, scenes
    warmup, steps, n = 3, 4, 512
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                          "--scenes", str(n), "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    assert sorted(os.listdir(tmp_path)) == sorted(f + ".npy" for f in ("scene",) + abi.plan_record.names)
    got = np.zeros(n, abi.plan_record)
    for f in abi.plan_record.names:
        a = np.load(os.path.join(tmp_path, f + ".npy"))
        assert a.dtype == np.float64 and a.shape == (n,), f
        got[f] = a
    assert np.array_equal(np.load(os.path.join(tmp_path, "scene.npy")), np.arange(n))
    import bench
    cycles = warmup + steps                                  # the last step is this many cycles into the bench's episode
    assert cycles < bench.EPISODE
    H, OX, OY = scenes.Episodes(the_map, np.arange(n), cycles=bench.EPISODE, n_obs=bench.N_OBS).all_cycles()   # (the script depends on the length)
    want = oracle.run(H[:cycles].copy(), OX[:cycles].copy(), OY[:cycles].copy(), threads=8)["rec"][-1]
    assert_records_equal(got, want, REC_EXACT, close=DIR_ERR_TOL, what="dumped record")
