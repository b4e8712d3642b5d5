"""lane-changing agents (include/dmpp_b200.h section 13): cost of arming them on top of the reactive agents (section 12).  In one
run, alternated four times: 4096 highway worlds x 25 cycles as ONE graph launch, react-only against react + lane changes; and
dp_world_step_dev alone, on the same world state and records (4096 highway worlds with 10 agents, 1024 highway worlds with 200
agents).  With lane changes on the obstacles move differently, so the records differ and the episode delta mixes the kernel's
cost with a changed planner workload; the world-step timing is the clean cost figure.  Also counts, with metrics armed in both
arms, the worlds with a collision and where their first colliding agent started, and the worlds with a lane change.  CUDA events
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

REPS, ROUNDS = 10, 4
dev = torch.device("cuda", 0)
m = scenes.Map()


def u8(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)


def cump_of():
    c = np.zeros(m.x.size)
    for gl in range(m.n_lanes):
        o, e = int(m.lane_pt_off[gl]), int(m.lane_pt_off[gl + 1])
        dx, dy = np.diff(m.x[o:e]), np.diff(m.y[o:e])
        c[o + 1:e] = np.add.accumulate(np.sqrt(dx * dx + dy * dy))
    return c


class Arm:
    """one planner + world of one kind; the agent model armed or not, and optionally the episode metrics"""

    def __init__(self, kind, n, n_obs, cycles, react, metrics=False):
        self.n = n
        self.p = Planner(n, n_obs); self.p.upload_map(m)
        wp = self.p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]
        self.p.set_world_params(wp)
        self.w = scenes.World(m, np.arange(n), n_obs, kind=kind)
        self.cycles = cycles
        self.h0, self.a0 = u8(self.w.hdr), u8(self.w.agents)
        self.d_h, self.d_a = torch.empty_like(self.h0), torch.empty_like(self.a0)
        self.d_x = torch.zeros((n, n_obs), dtype=torch.float64, device=dev); self.d_y = torch.zeros_like(self.d_x)
        self.d_r = torch.zeros((cycles, n, 128), dtype=torch.uint8, device=dev)
        self.d_v0 = u8(self.w.v0)
        self.d_m = torch.zeros((n, 192), dtype=torch.uint8, device=dev)
        if metrics:
            self.p.set_metrics(pl.metrics_params(), self.d_m.data_ptr())
        if react:
            self.p.set_agent_model(pl.agent_model_params(), self.d_v0.data_ptr())

    def episode_ms(self, graph=True):
        st = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.d_h.copy_(self.h0); self.d_a.copy_(self.a0)
        self.p.reset_dev(0, self.n, stream=st.cuda_stream); torch.cuda.synchronize()
        e0.record(st)
        self.p.run_closed_loop_dev(self.n, self.cycles, self.d_h.data_ptr(), self.d_a.data_ptr(), self.d_x.data_ptr(), self.d_y.data_ptr(),
                                   self.d_r.data_ptr(), stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        assert self.p.closed_loop_is_graph() or not graph
        return e0.elapsed_time(e1)

    def step_us(self, h, a, rec, launches=50):
        """dp_world_step_dev alone from world state (h, a) with records rec (the world restored before every window)"""
        st = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.d_h.copy_(h); self.d_a.copy_(a)
        e0.record(st)
        for _ in range(launches):
            self.p.world_step_dev(self.n, self.d_h.data_ptr(), self.d_a.data_ptr(), self.d_x.data_ptr(), self.d_y.data_ptr(), rec.data_ptr(),
                                  stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / launches

    def close(self):
        self.p.set_agent_model(None, None); self.p.set_metrics(None, None); self.p.close()


def first_strikes(w, met, cump):
    h, a = w.hdr, w.agents
    s = np.nonzero(met["first_collision_step"] > 0)[0]
    gl = m.road_lane_base[h["road_num"][s].astype(int) - 1] + h["lane_num"][s].astype(int) - 1
    se = cump[m.lane_pt_off[gl] + h["id"][s, h["lane_num"][s].astype(int) - 1]]
    ag = a[s, met["first_collision_agent"][s]]
    sk = cump[m.lane_pt_off[ag["lane"]] + ag["i"]] + ag["u"]
    same_lane = ag["lane"] == gl
    behind = same_lane & (sk < se)
    return {"worlds_with_collision": int(s.size), "first_agent_behind_on_ego_lane": int(behind.sum()),
            "of_them_faster_than_ego": int((behind & (ag["v"] > h["velocity"][s] / 3.6)).sum()),
            "first_agent_ahead_on_ego_lane": int((same_lane & ~behind).sum()), "first_agent_on_other_lane": int((~same_lane).sum())}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "n": len(xs)}


class LcArm(Arm):
    """Arm with the reactive agents armed, and lane changes on top when lanechg"""

    def __init__(self, n, n_obs, cycles, lanechg, metrics=False):
        super().__init__("highway", n, n_obs, cycles, True, metrics)
        self.d_s = torch.zeros((n, n_obs, abi.lane_change_state.itemsize), dtype=torch.uint8, device=self.d_h.device)
        if lanechg:
            self.p.set_lane_change(pl.lane_change_params(), self.d_s.data_ptr())

    def step_us(self, h, a, rec, s=None, launches=50):
        if s is not None:
            self.d_s.copy_(s)
        return super().step_us(h, a, rec, launches)

    def close(self):
        self.p.set_lane_change(None, None)
        super().close()


out = {"card": card(), "episode": {}, "world_step": {}, "collisions": {}, "lane_changes": {}}
cump = cump_of()
arms = {"react": LcArm(4096, 10, 25, False), "lanechg": LcArm(4096, 10, 25, True)}
for a in arms.values():                                     # warm-up: graph build and first launches
    a.episode_ms(); a.episode_ms()
ep = {"react": [], "lanechg": []}
for r in range(ROUNDS):                                     # alternated, the order flipped every round
    for name in (("react", "lanechg") if r % 2 == 0 else ("lanechg", "react")):
        ep[name] += [arms[name].episode_ms() for _ in range(REPS)]
out["episode"]["highway_4096x25"] = {
    "cycles": 25, "ms_per_episode_react": summary(ep["react"]), "ms_per_episode_lanechg": summary(ep["lanechg"]),
    "lanechg_over_react": float(np.median(ep["lanechg"]) / np.median(ep["react"])),
    "records_identical": arms["react"].d_r.cpu().numpy().tobytes() == arms["lanechg"].d_r.cpu().numpy().tobytes()}
for a in arms.values():
    a.close()

for n in (512, 4096):                                       # the collision table, metrics armed in both arms
    tab = {}
    for name, lanechg in (("react", False), ("lanechg", True)):
        a = LcArm(n, 10, 25, lanechg, metrics=True)
        a.episode_ms()
        tab[name] = first_strikes(a.w, np.frombuffer(a.d_m.cpu().numpy().tobytes(), abi.episode_metrics), cump)
        if lanechg:
            st = np.frombuffer(a.d_s.cpu().numpy().tobytes(), abi.lane_change_state).reshape(n, 10)
            ch = st["changes_left"] + st["changes_right"]
            out["lane_changes"]["highway_%dx25" % n] = {"worlds_with_a_change": int((ch.sum(axis=1) > 0).sum()), "changes": int(ch.sum()),
                                                        "left": int(st["changes_left"].sum()), "right": int(st["changes_right"].sum())}
        a.close()
    out["collisions"]["highway_%dx25" % n] = tab

for n, n_obs in ((4096, 10), (1024, 200)):
    arms = {"react": LcArm(n, n_obs, 25, False), "lanechg": LcArm(n, n_obs, 25, True)}
    src = arms["lanechg"]
    src.episode_ms(graph=False)                             # one armed episode (200 agents: group kernel, no graph): the state
                                                            # both arms step from, placement done
    h, a, rec, s = src.d_h.clone(), src.d_a.clone(), src.d_r[-1].contiguous(), src.d_s.clone()
    for x in arms.values():
        x.step_us(h, a, rec, s)
    st = {"react": [], "lanechg": []}
    for r in range(ROUNDS):
        for name in (("react", "lanechg") if r % 2 == 0 else ("lanechg", "react")):
            st[name] += [arms[name].step_us(h, a, rec, s) for _ in range(REPS)]
    out["world_step"]["highway_%dx%d_agents" % (n, n_obs)] = {
        "us_per_step_react": summary(st["react"]), "us_per_step_lanechg": summary(st["lanechg"]),
        "lanechg_over_react": float(np.median(st["lanechg"]) / np.median(st["react"])), "launches_per_window": 50}
    for x in arms.values():
        x.close()
print(json.dumps(out))
