"""cost of arming the world step's models, one sub-command per model; every measurement alternates the arms four times, the order
flipped every round, with CUDA events on the launching stream, and prints one JSON line with the card's name, power limit and max
SM clock read in the same run.

  metrics      episode metrics (include/dmpp_b200.h section 11): 4096 highway worlds x 25 cycles and 4096 junction worlds x 120
               cycles as ONE graph launch each, metrics off against on; and dp_world_step_dev alone (4096 junction worlds), off
               against on.  The records of both arms must be byte-identical.
  agents       reactive agents (section 12): the same two episodes, model off against on; and dp_world_step_dev alone, off against
               on, on the same world state and records (4096 junction worlds with 10 agents, 1024 urban worlds with 200 agents).
               With the model on the obstacles move differently, so the records differ and the episode delta mixes the kernel's cost
               with a changed planner workload; the world-step timing is the clean cost figure.  Also counts, with metrics armed in
               both arms, the worlds with a collision and where their first colliding agent started (the ego's lane behind / ahead
               of it, another lane).
  lane_change  lane changes (section 13) on top of the reactive agents, against the reactive agents alone: the highway episode,
               the collision table and the lane changes made, and dp_world_step_dev alone (4096 highway worlds with 10 agents, 1024
               with 200).
  v2x          V2X events in closed-loop episodes (section 14): the highway and junction episodes (4096 worlds) disarmed, observe-only
               (apply = 0: the records must equal the disarmed ones, the delta is the V2X launches alone) and applied; the V2X launch
               alone (dp_v2x_world_dev, 4096 worlds, apply = 0, on the world and records the last episode left); and the effect of
               applying the flags on seeds 0-511 (red crossings, stop cycles, worlds that stopped on a red and left on green, the
               minimum ego-pedestrian distance while the pedestrian is active)."""
import argparse
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
    """one planner + world of one kind, with the models asked for armed"""

    def __init__(self, kind, n, n_obs, cycles, metrics=False, react=False, lanechg=False, v2x=None):
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
        self.d_s = torch.zeros((n, n_obs, abi.lane_change_state.itemsize), dtype=torch.uint8, device=dev)
        if metrics:
            self.p.set_metrics(pl.metrics_params(), self.d_m.data_ptr())
        if react:
            self.p.set_agent_model(pl.agent_model_params(), self.d_v0.data_ptr())
        if lanechg:
            self.p.set_lane_change(pl.lane_change_params(), self.d_s.data_ptr())
        if v2x is not None:                                 # v2x = apply (0 / 1)
            self.ev = scenes.V2xEvents(self.w, np.arange(n))
            self.d_spec, self.d_wx, self.d_wy = u8(self.ev.spec), u8(np.append(self.ev.wp_x, 0.0)), u8(np.append(self.ev.wp_y, 0.0))
            self.d_vf = torch.zeros((n, abi.v2x_flags.itemsize), dtype=torch.uint8, device=dev)
            self.d_vs = torch.zeros((n, abi.v2x_episode_stats.itemsize), dtype=torch.uint8, device=dev)
            self.p.set_v2x_world(abi.V2xWorldParams(0, v2x), n, self.d_spec.data_ptr(), self.d_wx.data_ptr(), self.d_wy.data_ptr(),
                                 self.ev.wp_x.size, self.d_vf.data_ptr(), self.d_vs.data_ptr())

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

    def state(self):
        """the world, the last records and the lane-change states the last episode left"""
        return self.d_h.clone(), self.d_a.clone(), self.d_r[-1].contiguous(), self.d_s.clone()

    def step_us(self, h, a, rec, s, launches=50):
        """dp_world_step_dev alone from world state (h, a, lane-change states s) with records rec; the world is restored after the
        window, so that every window starts from the same state"""
        st = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.d_h.copy_(h); self.d_a.copy_(a); self.d_s.copy_(s)
        e0.record(st)
        for _ in range(launches):
            self.p.world_step_dev(self.n, self.d_h.data_ptr(), self.d_a.data_ptr(), self.d_x.data_ptr(), self.d_y.data_ptr(), rec.data_ptr(),
                                  stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        self.d_h.copy_(h); self.d_a.copy_(a); self.d_s.copy_(s)
        return e0.elapsed_time(e1) * 1e3 / launches

    def v2x_us(self, launches=50):
        """dp_v2x_world_dev alone (cycle 5) on the world and the last records the last episode left"""
        st = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(launches):
            self.p.v2x_world_dev(self.n, self.d_h.data_ptr(), self.d_r[-1].data_ptr(), 5, stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / launches

    def close(self):
        self.p.set_v2x_world(None, 0, None); self.p.set_lane_change(None, None); self.p.set_agent_model(None, None); self.p.set_metrics(None, None); self.p.close()


def alternate(arms, *measures):
    """REPS samples of every measure per arm and round, ROUNDS rounds, the order of the arms flipped every round"""
    out = [{k: [] for k in arms} for _ in measures]
    for r in range(ROUNDS):
        for name in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            for res, f in zip(out, measures):
                res[name] += [f(arms[name]) for _ in range(REPS)]
    return out


def warm(arms):
    for a in arms.values():                                 # graph build and first launches
        a.episode_ms(); a.episode_ms()


def close(arms):
    for a in arms.values():
        a.close()


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


def metrics_of(a):
    return np.frombuffer(a.d_m.cpu().numpy().tobytes(), abi.episode_metrics)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "n": len(xs)}


def ratio(xs, ys):
    return float(np.median(xs) / np.median(ys))


def records_identical(arms):
    a, b = arms.values()
    return a.d_r.cpu().numpy().tobytes() == b.d_r.cpu().numpy().tobytes()


def bench_metrics():
    N = 4096
    out = {"scenes": N, "card": card(), "episode": {}, "world_step_junction": {}}
    for kind, cycles in (("highway", 25), ("junction", 120)):
        arms = {"off": Arm(kind, N, 10, cycles), "on": Arm(kind, N, 10, cycles, metrics=True)}
        warm(arms)
        if kind == "junction":                              # the world-step windows run on the world and records the last episode left
            ep, st = alternate(arms, Arm.episode_ms, lambda a: a.step_us(*a.state()))
        else:
            ep, = alternate(arms, Arm.episode_ms)
        assert records_identical(arms), kind + ": records differ"
        rows = metrics_of(arms["on"])
        out["episode"]["%s_%dx%d" % (kind, N, cycles)] = {
            "cycles": cycles, "ms_per_episode_off": summary(ep["off"]), "ms_per_episode_on": summary(ep["on"]),
            "on_over_off": ratio(ep["on"], ep["off"]), "records_identical": True,
            "worlds_with_collision": int((rows["collision_steps"] > 0).sum()), "worlds_with_ttc_warning": int((rows["ttc_warn_steps"] > 0).sum())}
        if kind == "junction":
            out["world_step_junction"] = {"us_per_step_off": summary(st["off"]), "us_per_step_on": summary(st["on"]),
                                          "on_over_off": ratio(st["on"], st["off"]), "launches_per_window": 50}
        close(arms)
    return out


def bench_agents():
    out = {"card": card(), "episode": {}, "world_step": {}, "collisions": {}}
    cump = cump_of()
    for kind, cycles in (("highway", 25), ("junction", 120)):
        arms = {"off": Arm(kind, 4096, 10, cycles), "on": Arm(kind, 4096, 10, cycles, react=True)}
        warm(arms)
        ep, = alternate(arms, Arm.episode_ms)
        out["episode"]["%s_4096x%d" % (kind, cycles)] = {
            "cycles": cycles, "ms_per_episode_off": summary(ep["off"]), "ms_per_episode_on": summary(ep["on"]),
            "on_over_off": ratio(ep["on"], ep["off"]), "records_identical": records_identical(arms)}
        close(arms)
        for n in (512, 4096):                               # the collision table, metrics armed in both arms
            tab = {}
            for name, react in (("off", False), ("on", True)):
                a = Arm(kind, n, 10, cycles, metrics=True, react=react)
                a.episode_ms()
                tab[name] = first_strikes(a.w, metrics_of(a), cump)
                a.close()
            out["collisions"]["%s_%dx%d" % (kind, n, cycles)] = tab
    for kind, n, n_obs in (("junction", 4096, 10), ("urban", 1024, 200)):
        arms = {"off": Arm(kind, n, n_obs, 120), "on": Arm(kind, n, n_obs, 120, react=True)}
        arms["off"].episode_ms(graph=False)                 # one disarmed episode: the world state and records both arms step from
        s = arms["off"].state()
        for x in arms.values():
            x.step_us(*s)
        st, = alternate(arms, lambda x: x.step_us(*s))
        out["world_step"]["%s_%dx%d_agents" % (kind, n, n_obs)] = {
            "us_per_step_off": summary(st["off"]), "us_per_step_on": summary(st["on"]), "on_over_off": ratio(st["on"], st["off"]),
            "launches_per_window": 50}
        close(arms)
    return out


def bench_lane_change():
    out = {"card": card(), "episode": {}, "world_step": {}, "collisions": {}, "lane_changes": {}}
    cump = cump_of()
    arm = lambda n, n_obs, lanechg, metrics=False: Arm("highway", n, n_obs, 25, metrics=metrics, react=True, lanechg=lanechg)
    arms = {"react": arm(4096, 10, False), "lanechg": arm(4096, 10, True)}
    warm(arms)
    ep, = alternate(arms, Arm.episode_ms)
    out["episode"]["highway_4096x25"] = {
        "cycles": 25, "ms_per_episode_react": summary(ep["react"]), "ms_per_episode_lanechg": summary(ep["lanechg"]),
        "lanechg_over_react": ratio(ep["lanechg"], ep["react"]), "records_identical": records_identical(arms)}
    close(arms)
    for n in (512, 4096):                                   # the collision table, metrics armed in both arms
        tab = {}
        for name, lanechg in (("react", False), ("lanechg", True)):
            a = arm(n, 10, lanechg, metrics=True)
            a.episode_ms()
            tab[name] = first_strikes(a.w, metrics_of(a), cump)
            if lanechg:
                st = np.frombuffer(a.d_s.cpu().numpy().tobytes(), abi.lane_change_state).reshape(n, 10)
                ch = st["changes_left"] + st["changes_right"]
                out["lane_changes"]["highway_%dx25" % n] = {"worlds_with_a_change": int((ch.sum(axis=1) > 0).sum()), "changes": int(ch.sum()),
                                                            "left": int(st["changes_left"].sum()), "right": int(st["changes_right"].sum())}
            a.close()
        out["collisions"]["highway_%dx25" % n] = tab
    for n, n_obs in ((4096, 10), (1024, 200)):
        arms = {"react": arm(n, n_obs, False), "lanechg": arm(n, n_obs, True)}
        arms["lanechg"].episode_ms(graph=False)             # one armed episode (200 agents: group kernel, no graph): the state
        s = arms["lanechg"].state()                         # both arms step from, placement done
        for x in arms.values():
            x.step_us(*s)
        st, = alternate(arms, lambda x: x.step_us(*s))
        out["world_step"]["highway_%dx%d_agents" % (n, n_obs)] = {
            "us_per_step_react": summary(st["react"]), "us_per_step_lanechg": summary(st["lanechg"]),
            "lanechg_over_react": ratio(st["lanechg"], st["react"]), "launches_per_window": 50}
        close(arms)
    return out


def v2x_effect(kind, cycles, n=512):
    """seeds 0 .. n-1, apply 0 against 1: what the flags do to the episode"""
    out = {}
    w = scenes.World(m, np.arange(n), 10, kind=kind)
    ev = scenes.V2xEvents(w, np.arange(n))
    for apply in (0, 1):
        p = Planner(n, 10); p.upload_map(m)
        wp = p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]; p.set_world_params(wp)
        o = p.run_closed_loop(w.hdr, w.agents, cycles, v2x=(abi.V2xWorldParams(0, apply), ev))
        p.close()
        st, hl = o["v2x_stats"], o["hdr_log"]
        r = {"stop_cycles": int(st["stop_cmds"].sum()), "creep_cycles": int(st["creep_cmds"].sum()),
             "worlds_with_a_stop_command": int((st["stop_cmds"] > 0).sum()), "handler_cycles": int(st["cycles"].sum())}
        if kind == "junction":
            s = ev.spec
            t = np.arange(cycles)[:, None] * hl["period_ms"] / 1000.0
            ph = np.fmod(t + s["sig_offset"][None, :], s["sig_cycle"][None, :])
            ph = np.where(ph < 0, ph + s["sig_cycle"][None, :], ph)
            state = np.where(ph < s["sig_green"], 6, np.where(ph < s["sig_green"] + s["sig_yellow"], 7, 3))
            on = (hl["road_num"] == 6) & (hl["pos"] != 2)
            stopped_red = on & (hl["velocity"] == 0) & (state == 3)
            left = on[:-1] & ~on[1:]                           # the step from cycle k left the approach
            left_green = left & (state[:-1] == 6)
            sr = stopped_red.any(axis=0)
            later_green = np.array([left_green[np.argmax(stopped_red[:, i]):, i].any() if sr[i] else False for i in range(n)])
            r.update(red_crossings=int(st["red_crossings"].sum()), worlds_crossing_on_red=int((st["red_crossings"] > 0).sum()),
                     worlds_stopped_on_red=int(sr.sum()), worlds_stopped_on_red_then_left_on_green=int(later_green.sum()),
                     worlds_crossed=int(left.any(axis=0).sum()))
        else:
            d = st["min_ped_distance"][ev.spec["has_ped"] == 1]
            r.update(worlds_with_pedestrian=int(d.size), min_ped_distance_median=float(np.median(d)), min_ped_distance_min=float(d.min()),
                     worlds_within_1m=int((d < 1.0).sum()), worlds_within_2m=int((d < 2.0).sum()))
        out["apply_%d" % apply] = r
    return out


def bench_v2x():
    N = 4096
    out = {"scenes": N, "card": card(), "episode": {}, "v2x_launch": {}, "effect": {}}
    for kind, cycles in (("highway", 25), ("junction", 120)):
        arms = {"off": Arm(kind, N, 10, cycles), "observe": Arm(kind, N, 10, cycles, v2x=0), "apply": Arm(kind, N, 10, cycles, v2x=1)}
        warm(arms)
        ep, = alternate(arms, Arm.episode_ms)
        same = arms["off"].d_r.cpu().numpy().tobytes() == arms["observe"].d_r.cpu().numpy().tobytes()
        assert same, kind + ": observe-only records differ from the disarmed ones"
        out["episode"]["%s_%dx%d" % (kind, N, cycles)] = {
            "cycles": cycles, "ms_off": summary(ep["off"]), "ms_observe": summary(ep["observe"]), "ms_apply": summary(ep["apply"]),
            "observe_over_off": ratio(ep["observe"], ep["off"]), "apply_over_off": ratio(ep["apply"], ep["off"]),
            "records_identical_off_observe": same}
        a = arms["observe"]
        a.v2x_us()
        us = [a.v2x_us() for _ in range(REPS * ROUNDS)]
        out["v2x_launch"]["%s_%d" % (kind, N)] = {"us_per_launch": summary(us), "launches_per_window": 50}
        close(arms)
        out["effect"]["%s_512x%d" % (kind, cycles)] = v2x_effect(kind, cycles)
    return out


if __name__ == "__main__":
    benches = {"metrics": bench_metrics, "agents": bench_agents, "lane_change": bench_lane_change, "v2x": bench_v2x}
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("model", choices=list(benches))
    print(json.dumps(benches[ap.parse_args().model]()))
