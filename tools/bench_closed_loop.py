"""closed-loop episodes (dp_run_closed_loop_dev: ONE graph launch per episode) against the same launches enqueued one by one,
for a full batch and for a single scene (where the launch latency is the cycle), 4096 junction worlds x 120 cycles through the
connector (dp_world_params.pre_junction_pts = 60), the world step alone (highway against junction worlds), and the output-frame
kernel against the HBM copy peak.  CUDA events on the launching stream; prints one JSON line with the card's name and power
limit read in the same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import dmpp_b200  # noqa: E402,F401
from dmpp_b200 import abi, scenes  # noqa: E402
from dmpp_b200.planner import Planner  # noqa: E402

cycles = int(sys.argv[1]) if len(sys.argv) > 1 else 25
reps = 12
dev = torch.device("cuda", 0)
m = scenes.Map()
peaks = {}
try:
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
except OSError:
    pass
hbm_peak = float(peaks.get("hbm_gbs", 6549.4))


def u8(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)


def planner(n, kind):
    p = Planner(n, 10); p.upload_map(m)
    wp = p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]
    p.set_world_params(wp)
    return p, scenes.World(m, np.arange(n), 10, kind=kind)


def episode(n, graph, kind="highway", cycles=cycles):
    os.environ["DP_EPISODE_GRAPH"] = "1" if graph else "0"
    p, w = planner(n, kind)
    h0, a0 = u8(w.hdr), u8(w.agents)
    d_h, d_a = torch.empty_like(h0), torch.empty_like(a0)
    d_x = torch.zeros((n, 10), dtype=torch.float64, device=dev); d_y = torch.zeros_like(d_x)
    d_r = torch.zeros((cycles, n, 128), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms, wall = [], []
    for r in range(reps):
        d_h.copy_(h0); d_a.copy_(a0)
        p.reset_dev(0, n, stream=st.cuda_stream); torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record(st)
        p.run_closed_loop_dev(n, cycles, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
        ms.append(e0.elapsed_time(e1))
    assert p.closed_loop_is_graph() == graph
    rec = np.frombuffer(d_r.cpu().numpy().tobytes(), abi.plan_record).reshape(cycles, n)
    best, bw = float(np.median(ms[3:])), float(np.median(wall[3:]))
    out = {"ms_per_episode": best, "us_per_cycle": best / cycles * 1e3, "wall_us_per_cycle": bw / cycles * 1e3,
           "plan_cycles_per_s": n * cycles / (best * 1e-3), "trajectories_per_s": float(rec["n_traj"].sum()) / (best * 1e-3),
           "launches_per_episode": 3 * cycles + 1}
    if kind != "highway":
        hdr = np.frombuffer(d_h.cpu().numpy().tobytes(), abi.scene_hdr)
        out["share_through_junction"] = float((hdr["path_num"] == 1).mean())
    p.close()
    return out, rec


def world_step(n, kind, launches=50):
    """dp_world_step_dev alone on the world and records left by a 20-cycle episode; the world is restored before every timed
    window of `launches` back-to-back steps (the steps move it in place)"""
    os.environ["DP_EPISODE_GRAPH"] = "1"
    p, w = planner(n, kind)
    d_h, d_a = u8(w.hdr), u8(w.agents)
    d_x = torch.zeros((n, 10), dtype=torch.float64, device=dev); d_y = torch.zeros_like(d_x)
    d_r = torch.zeros((20, n, 128), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    p.reset_dev(0, n, stream=st.cuda_stream)
    p.run_closed_loop_dev(n, 20, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), stream=st.cuda_stream)
    torch.cuda.synchronize()
    h0, a0 = d_h.clone(), d_a.clone()
    rec = d_r[-1].contiguous()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    us = []
    for r in range(reps):
        d_h.copy_(h0); d_a.copy_(a0)
        e0.record(st)
        for _ in range(launches):
            p.world_step_dev(n, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), rec.data_ptr(), stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        us.append(e0.elapsed_time(e1) * 1e3 / launches)
    p.close()
    return {"scenes": n, "kind": kind, "us_per_step": float(np.median(us[3:])), "us_min": float(np.min(us[3:])),
            "us_max": float(np.max(us[3:])), "launches_per_window": launches, "windows": reps - 3}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def frames(n):
    p = Planner(n, 10); p.upload_map(m)
    ep = scenes.Episodes(m, np.arange(n), cycles=2, n_obs=10)
    H, OX, OY = ep.all_cycles()
    d_h, d_x, d_y = u8(H[0]), torch.from_numpy(OX[0]).to(dev), torch.from_numpy(OY[0]).to(dev)
    d_r = torch.zeros((n, 128), dtype=torch.uint8, device=dev)
    d_c = torch.zeros((n, 1656), dtype=torch.uint8, device=dev); d_s = torch.zeros((n, 1632), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    p.reset_dev(0, n, stream=st.cuda_stream)
    p.cycle_dev(n, d_h.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), stream=st.cuda_stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for r in range(20):
        flush.fill_(r)
        e0.record(st)
        p.pack_frames_dev(n, d_r.data_ptr(), d_c.data_ptr(), d_s.data_ptr(), stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = float(np.median(ms[3:]))
    by = n * (128 + 3200 + 1656 + 1632)                   # record + carried path in, both frames out
    p.close()
    return {"scenes": n, "us": t * 1e3, "algorithmic_bytes": by, "gb_per_s": by / (t * 1e-3) / 1e9, "frac_of_hbm_peak": by / (t * 1e-3) / 1e9 / hbm_peak,
            "hbm_peak_gb_per_s": hbm_peak, "l2": "256 MiB written before every launch"}


out = {"cycles": cycles, "card": card()}
for n in (4096, 1):
    g, rg = episode(n, True)
    d, rd = episode(n, False)
    assert rg.tobytes() == rd.tobytes(), "graph and direct launches disagree"
    out["scenes_%d" % n] = {"graph": g, "direct": d}
jg, rjg = episode(4096, True, "junction", 120)
jd, rjd = episode(4096, False, "junction", 120)
assert rjg.tobytes() == rjd.tobytes(), "junction: graph and direct launches disagree"
out["junction_4096x120"] = {"graph": jg, "direct": jd}
out["world_step_4096"] = [world_step(4096, k) for k in ("highway", "junction", "highway", "junction")]   # alternated
out["frames"] = [frames(4096), frames(131072)]
print(json.dumps(out))
