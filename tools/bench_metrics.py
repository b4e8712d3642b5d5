"""closed-loop episode metrics (include/dmpp_b200.h section 11): cost of arming them.  In one run, alternated four times:
4096 highway worlds x 25 cycles and 4096 junction worlds x 120 cycles as ONE graph launch each, metrics off against on; and
dp_world_step_dev alone (4096 junction worlds), off against on.  The records of both arms must be byte-identical.  CUDA events
on the launching stream; prints one JSON line with the card's name, power limit and max SM clock read in the same run."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import dmpp_b200  # noqa: E402,F401
from dmpp_b200 import abi, planner as pl, scenes  # noqa: E402
from dmpp_b200.planner import Planner  # noqa: E402

N, REPS, ROUNDS = 4096, 10, 4
dev = torch.device("cuda", 0)
m = scenes.Map()


def u8(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)


class Arm:
    """one planner + world of one kind; metrics armed or not"""

    def __init__(self, kind, cycles, metrics):
        self.p = Planner(N, 10); self.p.upload_map(m)
        wp = self.p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]
        self.p.set_world_params(wp)
        w = scenes.World(m, np.arange(N), 10, kind=kind)
        self.cycles = cycles
        self.h0, self.a0 = u8(w.hdr), u8(w.agents)
        self.d_h, self.d_a = torch.empty_like(self.h0), torch.empty_like(self.a0)
        self.d_x = torch.zeros((N, 10), dtype=torch.float64, device=dev); self.d_y = torch.zeros_like(self.d_x)
        self.d_r = torch.zeros((cycles, N, 128), dtype=torch.uint8, device=dev)
        self.d_m = torch.zeros((N, 192), dtype=torch.uint8, device=dev)
        if metrics:
            self.p.set_metrics(pl.metrics_params(), self.d_m.data_ptr())

    def episode_ms(self):
        st = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.d_h.copy_(self.h0); self.d_a.copy_(self.a0)
        self.p.reset_dev(0, N, stream=st.cuda_stream); torch.cuda.synchronize()
        e0.record(st)
        self.p.run_closed_loop_dev(N, self.cycles, self.d_h.data_ptr(), self.d_a.data_ptr(), self.d_x.data_ptr(), self.d_y.data_ptr(),
                                   self.d_r.data_ptr(), stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        assert self.p.closed_loop_is_graph()
        return e0.elapsed_time(e1)

    def step_us(self, launches=50):
        """dp_world_step_dev alone on the world and records the last episode left (the world restored before every window)"""
        st = torch.cuda.current_stream()
        h, a, rec = self.d_h.clone(), self.d_a.clone(), self.d_r[-1].contiguous()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.d_h.copy_(h); self.d_a.copy_(a)
        e0.record(st)
        for _ in range(launches):
            self.p.world_step_dev(N, self.d_h.data_ptr(), self.d_a.data_ptr(), self.d_x.data_ptr(), self.d_y.data_ptr(), rec.data_ptr(),
                                  stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        self.d_h.copy_(h); self.d_a.copy_(a)
        return e0.elapsed_time(e1) * 1e3 / launches


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "n": len(xs)}


out = {"scenes": N, "card": card(), "episode": {}, "world_step_junction": {}}
for kind, cycles in (("highway", 25), ("junction", 120)):
    arms = {"off": Arm(kind, cycles, False), "on": Arm(kind, cycles, True)}
    for a in arms.values():                                 # warm-up: graph build and first launches
        a.episode_ms(); a.episode_ms()
    ep = {"off": [], "on": []}
    st = {"off": [], "on": []}
    for r in range(ROUNDS):                                 # alternated, the order flipped every round
        for name in (("off", "on") if r % 2 == 0 else ("on", "off")):
            ep[name] += [arms[name].episode_ms() for _ in range(REPS)]
            if kind == "junction":
                st[name] += [arms[name].step_us() for _ in range(REPS)]
    assert arms["off"].d_r.cpu().numpy().tobytes() == arms["on"].d_r.cpu().numpy().tobytes(), kind + ": records differ"
    rows = np.frombuffer(arms["on"].d_m.cpu().numpy().tobytes(), abi.episode_metrics)
    res = {"cycles": cycles, "ms_per_episode_off": summary(ep["off"]), "ms_per_episode_on": summary(ep["on"]),
           "on_over_off": float(np.median(ep["on"]) / np.median(ep["off"])), "records_identical": True,
           "worlds_with_collision": int((rows["collision_steps"] > 0).sum()), "worlds_with_ttc_warning": int((rows["ttc_warn_steps"] > 0).sum())}
    out["episode"]["%s_%dx%d" % (kind, N, cycles)] = res
    if kind == "junction":
        out["world_step_junction"] = {"us_per_step_off": summary(st["off"]), "us_per_step_on": summary(st["on"]),
                                      "on_over_off": float(np.median(st["on"]) / np.median(st["off"])), "launches_per_window": 50}
    for a in arms.values():
        a.p.set_metrics(None, None); a.p.close()
print(json.dumps(out))
