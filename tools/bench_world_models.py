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
               minimum ego-pedestrian distance while the pedestrian is active).
  traffic      agents that obey the V2X events (section 15), with the reactive agents and the V2X events (apply = 1) armed in every
               arm: disarmed, obey = 0 (the records must equal the disarmed ones: the delta is the candidates' cost alone) and
               obey = 1, for the highway and junction episodes (4096 worlds) and dp_world_step_dev alone (4096 junction worlds with 10
               agents, 1024 urban worlds with 200); and the effect of obey 0 -> 1 on seeds 0-511 (agent red runs, ego red crossings,
               collisions and where they started, ego stopped steps; pedestrian hits and distances, ego collisions).
  obstacles    the planner sees the V2X road users (section 16), with the V2X events (apply = 1) armed in every arm and 14 obstacle
               slots for 10 agents: disarmed, what = 0 (the view is the world: the records must equal the disarmed ones, the delta is
               the obstacles launches alone) and what = 7, for 4096 highway worlds x 25 cycles as ONE graph launch; and
               dp_v2x_obstacles_dev alone (4096 worlds, what = 0 and 7, on the world and records the last episode left).  The effect
               on seeds 0-511 is the checker's, in tests/test_v2x_obstacles.py.
  parts        episodes in parts and forked worlds (section 17): 4096 junction worlds x 120 cycles as 1 x 120, 4 x 30 and 12 x 10
               parts with nothing armed and with every model armed (14 slots for 10 agents), the host not synchronising between parts
               and the records reused as a ring; the host time per part (capture + graph update or instantiate); the fork kernel
               (131 072 worlds, max_obs 10, every model armed, 0..65535 -> 65536..) against a cudaMemcpyAsync device-to-device copy
               of the same byte count, and a 4096-world fork; and the effect of perturbing the agents' v0 in forked copies of the
               highway worlds (seeds 0-511, metrics + reactive + lane-changing agents): 10 cycles, 7 copies per world with v0 scaled
               by a seeded uniform factor in [0.9, 1.1] per agent, 15 more cycles."""
import argparse
import json
import os
import subprocess
import sys
import time

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

    def __init__(self, kind, n, n_obs, cycles, metrics=False, react=False, lanechg=False, v2x=None, traffic=None, obstacles=None,
                 max_obs=None):
        self.n = n
        mo = max_obs or n_obs
        self.p = Planner(n, mo); self.p.upload_map(m)
        wp = self.p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]
        self.p.set_world_params(wp)
        self.w = scenes.World(m, np.arange(n), n_obs, kind=kind, max_obs=mo)
        self.cycles = cycles
        self.h0, self.a0 = u8(self.w.hdr), u8(self.w.agents)
        self.d_h, self.d_a = torch.empty_like(self.h0), torch.empty_like(self.a0)
        self.d_x = torch.zeros((n, mo), dtype=torch.float64, device=dev); self.d_y = torch.zeros_like(self.d_x)
        self.d_r = torch.zeros((cycles, n, 128), dtype=torch.uint8, device=dev)
        self.d_v0 = u8(self.w.v0)
        self.d_m = torch.zeros((n, 192), dtype=torch.uint8, device=dev)
        self.d_s = torch.zeros((n, mo, abi.lane_change_state.itemsize), dtype=torch.uint8, device=dev)
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
        if traffic is not None:                             # traffic = obey (0 / 1)
            self.d_ts = torch.zeros((n, abi.v2x_traffic_stats.itemsize), dtype=torch.uint8, device=dev)
            self.p.set_v2x_traffic(pl.v2x_traffic_params(obey=traffic), self.d_ts.data_ptr())
        if obstacles is not None:                           # obstacles = what (0 .. 7)
            self.d_hv = torch.zeros((n, 128), dtype=torch.uint8, device=dev)
            self.d_vx, self.d_vy = torch.zeros_like(self.d_x), torch.zeros_like(self.d_x)
            self.d_os = torch.zeros((n, abi.v2x_obstacle_stats.itemsize), dtype=torch.uint8, device=dev)
            self.p.set_v2x_obstacles(pl.v2x_obstacle_params(what=obstacles), self.d_hv.data_ptr(), self.d_vx.data_ptr(), self.d_vy.data_ptr(),
                                     self.d_os.data_ptr())

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

    def obstacles_us(self, launches=50):
        """dp_v2x_obstacles_dev alone (cycle 5) on the world and the last records the last episode left"""
        st = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(launches):
            self.p.v2x_obstacles_dev(self.n, self.d_h.data_ptr(), self.d_x.data_ptr(), self.d_y.data_ptr(), self.d_r[-1].data_ptr(), 5,
                                     stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / launches

    def close(self):
        self.p.set_v2x_obstacles(None, None, None, None, None); self.p.set_v2x_traffic(None, None); self.p.set_v2x_world(None, 0, None); self.p.set_lane_change(None, None); self.p.set_agent_model(None, None); self.p.set_metrics(None, None); self.p.close()


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


def traffic_effect(kind, cycles, n=512):
    """seeds 0 .. n-1 with metrics, reactive agents and V2X (apply = 1) armed, obey 0 against 1"""
    out, cump = {}, cump_of()
    w = scenes.World(m, np.arange(n), 10, kind=kind)
    ev = scenes.V2xEvents(w, np.arange(n))
    for obey in (0, 1):
        p = Planner(n, 10); p.upload_map(m)
        wp = p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]; p.set_world_params(wp)
        o = p.run_closed_loop(w.hdr, w.agents, cycles, metrics=pl.metrics_params(), agent_model=(pl.agent_model_params(), w.v0),
                              v2x=(abi.V2xWorldParams(0, 1), ev), traffic=pl.v2x_traffic_params(obey=obey))
        p.close()
        ts, vs, met = o["v2x_traffic"], o["v2x_stats"], o["metrics"]
        r = {"line_steps": int(ts["line_steps"].sum()), "ped_steps": int(ts["ped_steps"].sum())}
        if kind == "junction":
            r.update(agent_red_runs=int(ts["red_runs"].sum()), worlds_with_agent_red_run=int((ts["red_runs"] > 0).sum()),
                     ego_red_crossings=int(vs["red_crossings"].sum()), ego_stopped_steps=int(met["stopped_steps"].sum()),
                     first_strikes=first_strikes(w, met, cump))
        else:
            ped = ev.spec["has_ped"] == 1
            d = ts["min_ped_dist"][ped]
            r.update(ped_hits=int(ts["ped_hits"].sum()), worlds_with_ped_hit=int((ts["ped_hits"] > 0).sum()), worlds_with_pedestrian=int(d.size),
                     min_ped_dist_median=float(np.median(d)), worlds_min_ped_dist_below_2m=int((d < 2.0).sum()),
                     ego_collision_worlds=int((met["first_collision_step"] > 0).sum()), ego_collision_steps=int(met["collision_steps"].sum()))
        out["obey_%d" % obey] = r
    return out


def bench_traffic():
    out = {"card": card(), "episode": {}, "world_step": {}, "effect": {}}
    for kind, cycles in (("highway", 25), ("junction", 120)):
        N = 4096
        mk = lambda t: Arm(kind, N, 10, cycles, react=True, v2x=1, traffic=t)   # noqa: E731
        arms = {"off": mk(None), "obey0": mk(0), "obey1": mk(1)}
        warm(arms)
        ep, = alternate(arms, Arm.episode_ms)
        same = arms["off"].d_r.cpu().numpy().tobytes() == arms["obey0"].d_r.cpu().numpy().tobytes()
        assert same, kind + ": obey = 0 records differ from the disarmed ones"
        out["episode"]["%s_%dx%d" % (kind, N, cycles)] = {
            "cycles": cycles, "ms_off": summary(ep["off"]), "ms_obey0": summary(ep["obey0"]), "ms_obey1": summary(ep["obey1"]),
            "obey0_over_off": ratio(ep["obey0"], ep["off"]), "obey1_over_off": ratio(ep["obey1"], ep["off"]),
            "records_identical_off_obey0": same}
        close(arms)
    for kind, N, n_obs in (("junction", 4096, 10), ("urban", 1024, 200)):
        mk = lambda t: Arm(kind, N, n_obs, 2, react=True, v2x=1, traffic=t)    # noqa: E731
        arms = {"off": mk(None), "obey0": mk(0), "obey1": mk(1)}
        for a in arms.values():                             # (from 32 agents up the cycle runs on the group kernel: no graph)
            a.episode_ms(graph=n_obs < 32)
        h, a_, rec, s = arms["off"].state()
        for a in arms.values():                             # the V2X launch that sets the hand-stepped cycle (section 15's t)
            a.p.v2x_world_dev(N, h.data_ptr(), rec.data_ptr(), 40)
            a.step_us(h, a_, rec, s)
        st, = alternate(arms, lambda x: x.step_us(h, a_, rec, s))
        out["world_step"]["%s_%dx%d" % (kind, N, n_obs)] = {
            "us_off": summary(st["off"]), "us_obey0": summary(st["obey0"]), "us_obey1": summary(st["obey1"]),
            "obey0_over_off": ratio(st["obey0"], st["off"]), "obey1_over_off": ratio(st["obey1"], st["off"]), "launches_per_window": 50}
        close(arms)
    for kind, cycles in (("junction", 120), ("highway", 25)):
        out["effect"]["%s_512x%d" % (kind, cycles)] = traffic_effect(kind, cycles)
    return out


def bench_obstacles():
    N, kind, cycles = 4096, "highway", 25
    out = {"scenes": N, "max_obs": 14, "agents": 10, "card": card(), "episode": {}, "obstacles_launch": {}}
    mk = lambda what: Arm(kind, N, 10, cycles, v2x=1, obstacles=what, max_obs=14)   # noqa: E731
    arms = {"off": mk(None), "what0": mk(0), "what7": mk(7)}
    warm(arms)
    ep, = alternate(arms, Arm.episode_ms)
    same = arms["off"].d_r.cpu().numpy().tobytes() == arms["what0"].d_r.cpu().numpy().tobytes()
    assert same, "what = 0 records differ from the disarmed ones"
    differ = arms["off"].d_r.cpu().numpy().tobytes() != arms["what7"].d_r.cpu().numpy().tobytes()
    out["episode"]["%s_%dx%d" % (kind, N, cycles)] = {
        "cycles": cycles, "ms_off": summary(ep["off"]), "ms_what0": summary(ep["what0"]), "ms_what7": summary(ep["what7"]),
        "what0_over_off": ratio(ep["what0"], ep["off"]), "what7_over_off": ratio(ep["what7"], ep["off"]),
        "records_identical_off_what0": same, "records_differ_off_what7": differ, "target_what0_over_off": 1.05,
        "target_met": ratio(ep["what0"], ep["off"]) <= 1.05}
    for name in ("what0", "what7"):
        a = arms[name]
        a.obstacles_us()
        us = [a.obstacles_us() for _ in range(REPS * ROUNDS)]
        out["obstacles_launch"]["%s_%s_%d" % (name, kind, N)] = {"us_per_launch": summary(us), "launches_per_window": 50}
    close(arms)
    return out


def parts_ms(a, split, host_ms):
    """one episode of a.cycles cycles as the parts of `split` (the records a ring of the longest part), the host not synchronising
    between parts: device time from before the first part to after the last; the host time of every part call into host_ms"""
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.d_h.copy_(a.h0); a.d_a.copy_(a.a0)
    a.p.reset_dev(0, a.n, stream=st.cuda_stream); torch.cuda.synchronize()
    ring = a.d_r[:max(split)]
    e0.record(st)
    k0, prev = 0, None
    for i, c in enumerate(split):
        t = time.perf_counter()
        a.p.run_closed_loop_part_dev(a.n, k0, c, i == len(split) - 1, a.d_h.data_ptr(), a.d_a.data_ptr(), a.d_x.data_ptr(), a.d_y.data_ptr(),
                                     ring.data_ptr(), prev, stream=st.cuda_stream)
        host_ms.append((time.perf_counter() - t) * 1e3)
        assert a.p.closed_loop_is_graph()
        k0, prev = k0 + c, ring[c - 1].data_ptr()           # (read by the next part before its cycles overwrite the ring)
    e1.record(st); torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def fork_bench():
    """the fork kernel on 131 072 worlds with every model armed against a cudaMemcpyAsync of the same bytes"""
    N, mo, half = 131072, 10, 65536
    p = Planner(N, mo); p.upload_map(m)
    z = lambda b: torch.randint(0, 255, (N * b,), dtype=torch.uint8, device=dev)   # noqa: E731
    buf = {"hdr": z(128), "agents": z(32 * mo), "ox": z(8 * mo), "oy": z(8 * mo), "prev_rec": z(128), "met": z(192), "v0": z(8 * mo),
           "lcs": z(24 * mo), "spec": torch.zeros(N * 160, dtype=torch.uint8, device=dev), "vstats": z(80), "vflags": z(24), "ts": z(32),
           "os": z(80), "hv": z(128), "vx": z(8 * mo), "vy": z(8 * mo)}
    wx = torch.zeros(1, dtype=torch.float64, device=dev)
    p.set_metrics(pl.metrics_params(), buf["met"].data_ptr())
    p.set_agent_model(pl.agent_model_params(), buf["v0"].data_ptr())
    p.set_lane_change(pl.lane_change_params(), buf["lcs"].data_ptr())
    p.set_v2x_world(abi.V2xWorldParams(0, 1), N, buf["spec"].data_ptr(), wx.data_ptr(), wx.data_ptr(), 0, buf["vflags"].data_ptr(),
                    buf["vstats"].data_ptr())
    p.set_v2x_traffic(pl.v2x_traffic_params(), buf["ts"].data_ptr())
    p.set_v2x_obstacles(pl.v2x_obstacle_params(), buf["hv"].data_ptr(), buf["vx"].data_ptr(), buf["vy"].data_ptr(), buf["os"].data_ptr())
    per_world = sum(buf[k].numel() // N for k in buf if k not in ("hv", "vx", "vy")) + 128 + 3200   # + the carry slot and carried path
    st = torch.cuda.current_stream()
    src_big = torch.empty(half * per_world, dtype=torch.uint8, device=dev); dst_big = torch.empty_like(src_big)
    launches = 20

    def fork_us(count):
        src = np.arange(count, dtype=np.int32)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(launches):
            p.world_fork_dev(N, src, half, buf["hdr"].data_ptr(), buf["agents"].data_ptr(), buf["ox"].data_ptr(), buf["oy"].data_ptr(),
                             buf["prev_rec"].data_ptr(), stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / launches

    def copy_us():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(launches):
            dst_big.copy_(src_big)                           # (contiguous, same dtype and device: cudaMemcpyAsync device to device)
        e1.record(st); torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / launches

    fork_us(half); copy_us(); fork_us(4096)
    f, c = [], []
    for r in range(ROUNDS):
        for which in ((0, 1) if r % 2 == 0 else (1, 0)):
            (f if which == 0 else c).extend(fork_us(half) if which == 0 else copy_us() for _ in range(REPS))
    small = [fork_us(4096) for _ in range(REPS * ROUNDS)]
    p.set_v2x_obstacles(None, None, None, None, None); p.set_v2x_traffic(None, None); p.set_v2x_world(None, 0, None)
    p.set_lane_change(None, None); p.set_agent_model(None, None); p.set_metrics(None, None); p.close()
    moved = 2 * half * per_world                             # read + written
    return {"worlds": N, "max_obs": mo, "forked": half, "bytes_per_world": per_world, "launches_per_window": launches,
            "fork_us": summary(f), "memcpy_us": summary(c), "fork_TBps": moved / np.median(f) / 1e6, "memcpy_TBps": moved / np.median(c) / 1e6,
            "fork_over_memcpy_bandwidth": float(np.median(c) / np.median(f)), "target": 0.8,
            "target_met": bool(np.median(c) / np.median(f) >= 0.8),
            "fork_4096_us": summary(small), "fork_4096_note": "20 MB moved: L2-resident after the first launch of the window"}


def fork_effect():
    """highway seeds 0-511 x 8 (n = 4096), metrics + reactive + lane-changing agents: 10 cycles, then worlds 0-511 forked into 7
    copies each with v0 scaled per agent by a seeded uniform factor in [0.9, 1.1], then 15 cycles; the sources against one
    25-cycle call"""
    n0, copies, k1, cycles = 512, 7, 10, 25
    w = scenes.World(m, np.arange(n0), 10, kind="highway")
    kw = dict(metrics=pl.metrics_params(), lane_change=pl.lane_change_params())
    p1 = Planner(n0, 10); p1.upload_map(m)
    one = p1.run_closed_loop(w.hdr, w.agents, cycles, log=False, agent_model=(pl.agent_model_params(), w.v0), **kw)
    p1.close()
    n = n0 * (copies + 1)
    tile = lambda a: np.ascontiguousarray(np.concatenate([a] * (copies + 1)))   # noqa: E731
    p = Planner(n, 10); p.upload_map(m)
    ep = p.episode(tile(w.hdr), tile(w.agents), agent_model=(pl.agent_model_params(), tile(w.v0)), **kw)
    try:
        ep.run(k1, log=False)
        early = ep.state()["metrics"][:n0]
        src = np.tile(np.arange(n0, dtype=np.int32), copies)
        ep.fork(src, n0)
        v0 = np.zeros((n, 10)); ep._d2h(v0, ep.d["v0"], v0.nbytes); p.lib.dp_stream_sync(p.ctx, None)
        v0[n0:] *= np.random.default_rng(2026).uniform(0.9, 1.1, (n - n0, 10))
        ep._h2d("v0", v0); p.lib.dp_stream_sync(p.ctx, None)
        ep.run(cycles - k1, finish=True, log=False)
        met = ep.state()["metrics"]
        agents = ep.state()["agents"]
    finally:
        ep.close(); p.close()
    assert met[:n0].tobytes() == one["metrics"].tobytes(), "the unperturbed sources differ from the one-call episode"
    moved = (agents[n0:].reshape(copies, n0, 10)["u"] != agents[:n0]["u"][None]).any(axis=2)   # the perturbation took effect
    src_hit = met["collision_steps"][:n0] > 0
    copy_hit = (met["collision_steps"][n0:] > 0).reshape(copies, n0)
    late = (early["collision_steps"] == 0)
    cump = cump_of()
    h, a = w.hdr, w.agents
    klass = np.full(n0, "none", object)
    s = np.nonzero(met["first_collision_step"][:n0] > 0)[0]
    gl = m.road_lane_base[h["road_num"][s].astype(int) - 1] + h["lane_num"][s].astype(int) - 1
    se = cump[m.lane_pt_off[gl] + h["id"][s, h["lane_num"][s].astype(int) - 1]]
    ag = a[s, met["first_collision_agent"][:n0][s]]
    sk = cump[m.lane_pt_off[ag["lane"]] + ag["i"]] + ag["u"]
    klass[s] = np.where(ag["lane"] != gl, "other_lane", np.where(sk < se, "behind", "ahead"))
    table = {}
    for name in ("behind", "ahead", "other_lane"):
        sel = late & src_hit & (klass == name)
        table["collide_after_step_10_first_agent_" + name] = {"worlds": int(sel.sum()), "copies_that_still_collide": float(copy_hit[:, sel].mean()) if sel.any() else None}
    sel = late & ~src_hit
    table["no_collision"] = {"worlds": int(sel.sum()), "copies_that_collide": float(copy_hit[:, sel].mean()) if sel.any() else None}
    return {"worlds": n0, "copies": copies, "fork_after_cycle": k1, "cycles": cycles, "v0_factor": [0.9, 1.1], "seed": 2026,
            "sources_equal_one_call": True, "copies_whose_agents_end_elsewhere_than_their_source": float(moved.mean()), "worlds_with_collision": int(src_hit.sum()), "worlds_colliding_in_first_10_steps": int((~late).sum()),
            "table": table}


def bench_parts():
    N, kind, cycles = 4096, "junction", 120
    out = {"scenes": N, "cycles": cycles, "card": card(), "episode": {}}
    splits = {"1x120": [120], "4x30": [30] * 4, "12x10": [10] * 12}
    for arm_name, kw in (("nothing", {}), ("everything", dict(metrics=True, react=True, lanechg=True, v2x=1, traffic=1, obstacles=7, max_obs=14))):
        a = Arm(kind, N, 10, cycles, **kw)
        host = {k: [] for k in splits}
        for k, sp in splits.items():                        # warm every split's graphs
            parts_ms(a, sp, []); parts_ms(a, sp, [])
        res = {k: [] for k in splits}
        for r in range(ROUNDS):
            for k in (list(splits) if r % 2 == 0 else list(splits)[::-1]):
                res[k] += [parts_ms(a, splits[k], host[k]) for _ in range(REPS)]
        a.close()
        out["episode"][arm_name] = {k: {"ms_per_episode": summary(res[k]), "over_1x120": ratio(res[k], res["1x120"]),
                                        "host_ms_per_part": summary(host[k])} for k in splits}
        r430 = ratio(res["4x30"], res["1x120"])
        out["episode"][arm_name]["target_4x30_over_1x120"] = 1.03
        out["episode"][arm_name]["target_met"] = bool(r430 <= 1.03)
    out["fork"] = fork_bench()
    out["effect_highway_512"] = fork_effect()
    return out


def split_worlds(kind, n, seeds=None, everything=True):
    """an Episode of n worlds with every model armed (metrics only with everything False) and splitting armed"""
    seeds = np.arange(n) if seeds is None else seeds
    w = scenes.World(m, seeds, 10, kind=kind, max_obs=14)
    kw = dict(metrics=pl.metrics_params(), agent_model=(pl.agent_model_params(), w.v0), lane_change=pl.lane_change_params())
    if everything:
        kw.update(v2x=(abi.V2xWorldParams(0, 1), scenes.V2xEvents(w, seeds)), traffic=pl.v2x_traffic_params(), obstacles=pl.v2x_obstacle_params())
    return w, kw


def split_cost(kind, n, M):
    """dp_world_split_dev alone after 10 cycles, every model armed.  Every split of the ladder and every timed split is a level-0
    split (the rows start afresh) on the metrics rows of cycle 10, restored before each call: a copy overwrites the metrics row of
    its destination, so without the restore later calls would resample ever fewer distinct worlds.  (beta, c_max) is the rung of
    the ladder whose copied fraction is closest to one half; the copied fraction of every timed call is recorded"""
    p = Planner(n, 14); p.upload_map(m)
    wp = p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]; p.set_world_params(wp)
    w, kw = split_worlds(kind, n)
    ep = p.episode(w.hdr, w.agents, split=pl.split_params(group=M), **kw)
    st = torch.cuda.current_stream()
    d = ep.d
    try:
        ep.run(10, log=False)
        met0 = ep.state()["metrics"]

        def restore():
            ep._h2d("metrics", met0); p.lib.dp_stream_sync(p.ctx, None)

        frac = {}
        for c_max in (10.0, 50.0):
            for beta in (0.1, 0.25, 0.5, 1.0, 2.0, 5.0):
                if beta * c_max > 50:
                    continue
                restore()
                p.set_split(pl.split_params(group=M, beta=beta, c_max=c_max), n, d["split_rows"], d["split_groups"])
                ep.split(0)
                frac["beta=%g,c_max=%g" % (beta, c_max)] = (beta, c_max, float((p.split_map(n) >= 0).mean()))
        rung = min(frac, key=lambda k: abs(frac[k][2] - 0.5))
        beta, c_max, _ = frac[rung]
        p.set_split(pl.split_params(group=M, beta=beta, c_max=c_max), n, d["split_rows"], d["split_groups"])

        def one_split():
            """device time of one split: the stream is held by a spin so that the three launches queue up behind the first event"""
            restore()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(2_000_000)
            e0.record(st)
            p.world_split_dev(n, 0, d["hdr"], d["agents"], d["ox"], d["oy"], d["prev_rec"], stream=st.cuda_stream)
            e1.record(st); torch.cuda.synchronize()
            copied.append(float((p.split_map(n) >= 0).mean()))
            return e0.elapsed_time(e1) * 1e3
        copied = []
        one_split(); one_split()
        copied = []
        xs = [one_split() for _ in range(REPS * ROUNDS)]
    finally:
        ep.close(); p.close()
    return {"kind": kind, "worlds": n, "group": M, "every_model_armed": True, "level": 0, "beta": beta, "c_max": c_max,
            "copied_fraction_by_rung": {k: v[2] for k, v in frac.items()},
            "copied_fraction_of_timed_splits": summary(copied), "split_us": summary(xs)}


def split_overhead():
    """4096 junction worlds x 120 cycles as 12 x 10 parts, a split at each of the 11 seams (beta = 0, no noise) against none"""
    N, kind, cycles, every = 4096, "junction", 120, 10
    p = Planner(N, 14); p.upload_map(m)
    wp = p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]; p.set_world_params(wp)
    w, kw = split_worlds(kind, N)
    ep = p.episode(w.hdr, w.agents, split=pl.split_params(group=256, beta=0.0, amp_v=0.0), **kw)
    st = torch.cuda.current_stream()
    d = ep.d
    ring = torch.empty(every * N * 128, dtype=torch.uint8, device=dev)

    def episode_ms(splits):
        ep.restart()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        prev = None
        for k0 in range(0, cycles, every):
            p.run_closed_loop_part_dev(N, k0, every, k0 + every == cycles, d["hdr"], d["agents"], d["ox"], d["oy"], ring.data_ptr(), prev,
                                       stream=st.cuda_stream)
            prev = ring.data_ptr() + (every - 1) * N * 128  # (the ring's last row: read by the next part before its cycles overwrite it)
            if splits and k0 + every < cycles:
                p.world_split_dev(N, k0 // every, d["hdr"], d["agents"], d["ox"], d["oy"], prev, stream=st.cuda_stream)
        e1.record(st); torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    try:
        arms = {"no_split": False, "split": True}
        finals = {}
        for k, v in arms.items():
            episode_ms(v); episode_ms(v)
            finals[k] = {x: y for x, y in ep.state().items() if x not in ("graph", "split_rows", "split_groups", "ox", "oy", "lane_change_state")}
        res = {k: [] for k in arms}
        for r in range(ROUNDS):
            for k in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
                res[k] += [episode_ms(arms[k]) for _ in range(REPS)]
    finally:
        ep.close(); p.close()
    same = all(finals["split"][k].tobytes() == finals["no_split"][k].tobytes() for k in finals["split"])
    r = ratio(res["split"], res["no_split"])
    return {"worlds": N, "cycles": cycles, "parts": "12x10", "splits": 11, "every_model_armed": True,
            "ms_per_episode": {k: summary(v) for k, v in res.items()}, "split_over_no_split": r, "target": 1.03,
            "target_met": bool(r <= 1.03), "final_states_identical": same}


def split_effect(max_sources=32):
    """junction sources among seeds 0-511 that do not collide in 120 cycles (metrics, reactive agents, lane changes); per source 16
    populations of 256 copies, amp_v = 0.1, a split every 10 cycles, beta = 0 against beta = 0.3 at the same budget"""
    kind, cycles, every, P, M, beta = "junction", 120, 10, 16, 256, 0.3
    p = Planner(P * M, 14); p.upload_map(m)
    wp = p.world_params(); wp.pre_junction_pts = scenes.World.PRE_JUNCTION_PTS[kind]; p.set_world_params(wp)
    w, kw = split_worlds(kind, 512, everything=False)
    one = p.run_closed_loop(w.hdr, w.agents, cycles, log=False, **kw)
    quiet = np.nonzero(one["metrics"]["first_collision_step"] < 0)[0]
    rows = []
    try:
        for s in quiet[:max_sources]:
            wc, kwc = split_worlds(kind, P * M, seeds=np.full(P * M, s), everything=False)
            row = {"seed": int(s)}
            for name, b in (("beta0", 0.0), ("beta%g" % beta, beta)):
                ep = p.episode(wc.hdr, wc.agents, split=pl.split_params(group=M, beta=b, amp_v=0.1, seed=int(s)), **kwc)
                try:
                    for k0 in range(0, cycles, every):
                        ep.run(every, finish=k0 + every == cycles, log=False)
                        if k0 + every < cycles:
                            ep.split(k0 // every)
                    stt = ep.state()
                finally:
                    ep.close()
                g = pl.split_estimate(stt)
                row[name] = {"p": float(g.mean()), "se": float(g.std(ddof=1) / np.sqrt(P)),
                             "raw_collision_fraction": float((stt["metrics"]["first_collision_step"] >= 0).mean()),
                             "roots_alive_mean": float(stt["split_groups"]["roots_alive"].mean())}
            rows.append(row)
    finally:
        p.close()
    bname = "beta%g" % beta
    return {"sources_checked": 512, "non_colliding_sources": int(quiet.size), "sources_run": len(rows), "populations": P, "group": M,
            "amp_v": 0.1, "split_every": every, "cycles": cycles, "beta": beta,
            "sources_with_p_gt_0": {"beta0": sum(r["beta0"]["p"] > 0 for r in rows), bname: sum(r[bname]["p"] > 0 for r in rows)},
            "per_source": rows}


def bench_split():
    return {"card": card(), "split_4096_junction": split_cost("junction", 4096, 256), "split_131072_highway": split_cost("highway", 131072, 256),
            "targets_us": {"4096": 20, "131072": 400}, "episode_overhead": split_overhead(), "effect": split_effect()}


if __name__ == "__main__":
    benches = {"metrics": bench_metrics, "agents": bench_agents, "lane_change": bench_lane_change, "v2x": bench_v2x, "traffic": bench_traffic,
               "obstacles": bench_obstacles, "parts": bench_parts, "split": bench_split}
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("model", choices=list(benches))
    print(json.dumps(benches[ap.parse_args().model]()))
