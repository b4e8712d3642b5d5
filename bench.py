#!/usr/bin/env python
"""bench.py -- headline benchmark of the Decision/Planning hot path (BASELINE.json metric:
trajectories scored / s and plan cycles / s).

Workload (BASELINE config 2, SURVEY.md 8d): 4096 independent synthetic highway scenes per GPU, ego + 10
vehicles, reference-derived default candidate set, 25-cycle scripted episodes.  One "step" = one
Decision+Planning cycle for every scene of the batch (the Decision and the Planning launch of dp_cycle_kernel, overlapped).

  python bench.py [--gpus N] [--steps K] [--warmup W]          our CUDA path (one rank per GPU)
  python bench.py [...] --dump-outputs DIR                     ... and the plan records of its last timed step, as .npy files
  python bench.py --impl reference [...]                       the reference's own CPU code (oracle/_ref)

Prints ONE JSON line (rank 0).  See DESIGN.md section 6 for how each number is obtained.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import dmpp_b200  # noqa: E402,F401
from dmpp_b200 import abi, scenes  # noqa: E402

SCENES = 4096
N_OBS = 10
EPISODE = 25
METRIC = "trajectories_scored_per_s"
UNIT = "trajectories/s"


def workload_desc(world):
    return {"workload": ("config2" if SCENES == 4096 else "config4 shard") + ": %d highway scenes/GPU x default candidate set (6 lane regions + 2K avoid offsets + 1 local path), "
                        "ego + %d vehicles, %d-cycle scripted episodes" % (SCENES, N_OBS, EPISODE),
            "scenes_per_gpu": SCENES, "obstacles": N_OBS, "episode_cycles": EPISODE,
            "parallelism": "scenes sharded %d-way, no data-path collective in the compute phase; when N>1 every rank's plan records are "
                           "gathered on every rank each step: GATHER_KIND; step i+1 is complete when its kernels AND the gather of step i-1 are, "
                           "the gathers of the last two steps (dp_gather_flush) are exposed and counted" % world,
            "l2": "256 MiB buffer written between timed steps (L2 flush); inputs resident in HBM for `value`"}


def alg_flops(pts, ntraj, n_obs):
    """SURVEY.md 8d: F(P,N) = 18 P + N (5 P + 12) summed over the trajectories actually scored."""
    return 18.0 * pts + n_obs * (5.0 * pts + 12.0 * ntraj)


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the UNMODIFIED reference (oracle/_ref/libref.so), one process per core
# ------------------------------------------------------------------------------------------------
_W = {}


def _worker_init(seed0, n, cycles):
    from oracle import binding
    m = scenes.Map()
    if binding.Reference.available():
        r = binding.Reference(); kind = "reference"
    else:
        r = binding.Oracle(); kind = "port"
    r.set_map(m)
    ep = scenes.Episodes(m, np.arange(seed0, seed0 + n), cycles=cycles, n_obs=N_OBS)
    _W.update(r=r, kind=kind, data=ep.all_cycles())
    return kind


def _worker_run(_):
    H, OX, OY = _W["data"]
    if H.size == 0:
        return 0, 0.0, 0
    if _W["kind"] == "reference":
        o = _W["r"].run(H, OX, OY, paths=False, calls=False)
    else:
        o = _W["r"].run(H, OX, OY, paths=False, calls=False, trace=False, exhaustive=False, threads=1)
    return int(o["traj"]), float(o["seconds"]), int(H.size)


class CpuArm:
    """P worker processes, each owning a private copy of the (non re-entrant) reference and a scene slice."""

    def __init__(self, total_scenes, cycles, procs):
        import multiprocessing as mp
        self.procs = procs
        self.ctx = mp.get_context("spawn")
        per = (total_scenes + procs - 1) // procs
        self.pools = [self.ctx.Pool(1) for _ in range(procs)]
        # the SAME scenes the GPU arm scores (seeds 0 .. total_scenes-1, rank-major), split into one contiguous range per core
        kinds = [p.apply_async(_worker_init, (i * per, max(0, min(per, total_scenes - i * per)), cycles)) for i, p in enumerate(self.pools)]
        self.kind = kinds[0].get()
        for k in kinds:
            k.get()

    def step(self):
        t0 = time.perf_counter()
        res = [p.apply_async(_worker_run, (0,)) for p in self.pools]
        res = [r.get() for r in res]
        dt = time.perf_counter() - t0
        return sum(r[0] for r in res), dt, sum(r[2] for r in res)

    def close(self):
        for p in self.pools:                                 # let the workers exit normally (their loaded libraries stay visible to
            p.close()                                        # whoever inspects the process at exit), do not terminate() them
        for p in self.pools:
            p.join()


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = host_cores()
    total = min(SCENES, 4096) * max(1, world)               # the GPU arm's scenes: SCENES per rank, seeds rank-major
    arm = CpuArm(total, EPISODE, cores)
    for _ in range(max(1, min(args.warmup, 2))):
        arm.step()
    traj = 0; secs = 0.0; cyc = 0
    steps = args.steps
    for _ in range(steps):
        t, dt, c = arm.step()
        traj += t; secs += dt; cyc += c
    arm.close()
    val = traj / secs
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": secs / cyc * total * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_desc(max(1, world)),
            "same_config": True, "scenes_total": total,
            "plan_cycles_per_s": cyc / secs,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": arm.kind, "per_core": val / max(cores, 1),
                             "sample": "%d steps, each = %d scenes (seeds 0..%d, the GPU arm's own) x %d cycles (whole episodes), one process "
                                       "per core running the unmodified Decision.cpp/Planning.cpp objects" % (steps, total, total - 1, EPISODE)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "ms_per_step is normalised to one plan cycle of %d scenes" % total}
    emit(line)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index; self.stop = False; self.sm = []; self.reasons = set(); self.max_sm = None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}
            while not self.stop:
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.002)
        except Exception as e:  # noqa: BLE001
            self.reasons.add("sampler_error:%s" % type(e).__name__)

    def result(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from dmpp_b200.planner import Planner

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # the record gather runs beside the next step's kernels: keep its footprint to a few CTAs so that the one-wave
        # Decision launch (1024 CTAs on 1036 slots) still fits
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "4")
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, args.warmup
    m = scenes.Map()
    ep = scenes.Episodes(m, np.arange(rank * SCENES, (rank + 1) * SCENES), cycles=EPISODE, n_obs=N_OBS)
    H, OX, OY = ep.all_cycles()
    planner = Planner(max_scenes=SCENES, max_obs=N_OBS, device=local_rank)
    planner.upload_map(m)

    # ---- untimed replay with the trace on: trajectories and path points scored per cycle (deterministic) ----
    rep = planner.run_episodes(H, OX, OY, trace=True, paths=False)
    traj_c = rep["rec"]["n_traj"].astype(np.int64).sum(axis=1)
    pts_c = rep["trace"]["pts_scored"].astype(np.int64).sum(axis=1)
    flops_c = alg_flops(pts_c.astype(np.float64), traj_c.astype(np.float64), N_OBS)

    # ---- inputs resident in HBM ----
    d_hdr = torch.from_numpy(H.view(np.uint8).reshape(EPISODE, SCENES, 128)).to(dev)
    d_ox = torch.from_numpy(OX).to(dev)
    d_oy = torch.from_numpy(OY).to(dev)
    d_recs = [torch.empty((SCENES, 128), dtype=torch.uint8, device=dev) for _ in range(3)]   # plan records, rotated per step
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(W + K)]
    # N > 1: the records of every rank are gathered on every rank each step.  The gather is fused into the Planning launch:
    # each rank's kernel stores its finished records straight into its slice of every peer's gathered buffer over NVLink
    # (torch symmetric memory gives the peer mappings, dp_set_record_mirrors hands them to the kernel); what is left of the
    # collective is a barrier, run on a side stream beside the next step's kernels.  Three gathered buffers rotate so that a
    # step never overwrites records a peer may still be reading.
    comm = torch.cuda.Stream(device=dev) if world > 1 else None
    gath = hdl = gat = None
    gather_kind = "none"
    if world > 1 and not os.environ.get("DP_BENCH_NO_IPC"):
        try:   # the C ABI's own fused gather: CUDA IPC peer mapping, records + completion flags stored by the cycle kernel
            from dmpp_b200.planner import Gather
            gat = Gather(planner, world, rank, SCENES, depth=4)
            gat.set_lag(int(os.environ.get("DP_GATHER_LAG", "2")))   # a launch awaits the gather two steps back: a whole step of slack between ranks
            hs = [None] * world
            dist.all_gather_object(hs, gat.my_handle())
            gat.attach(hs)
            gather_kind = ("dp_gather_* (C ABI, CUDA IPC mapping), deferred: the cycle kernel of step i+1 forwards step i's records to every "
                           "rank over NVLink as its warps start, raises that step's completion flags and waits for every rank's flags of step i-1 (lag 2)")
        except Exception as e:  # noqa: BLE001
            print("dp_gather unavailable (%s): falling back to torch symmetric memory" % e, file=sys.stderr)
            gat = None
    if world > 1 and gat is None:
        try:
            if os.environ.get("DP_BENCH_NO_SYMM"):
                raise RuntimeError("disabled by DP_BENCH_NO_SYMM")
            import torch.distributed._symmetric_memory as symm
            gath = [symm.empty((world * SCENES, 128), dtype=torch.uint8, device=dev) for _ in range(3)]
            hdl = [symm.rendezvous(g, dist.group.WORLD) for g in gath]
            for g in gath:
                g.zero_()
            gather_kind = "peer stores from the Planning launch (NVLink, symmetric memory) + barrier on a side stream"
        except Exception as e:  # noqa: BLE001 -- no peer mapping on this box: fall back to NCCL's all_gather
            print("symmetric memory unavailable (%s): using all_gather_into_tensor" % e, file=sys.stderr)
            gath = [torch.empty((world * SCENES, 128), dtype=torch.uint8, device=dev) for _ in range(3)]
            hdl = None
            gather_kind = "all_gather_into_tensor on a side stream"

    sampler = ClockSampler(local_rank)
    sampler.start()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    tail_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def finish_gather(i, rec_i):
        """what is left of step i's gather after its kernels: a barrier (peer stores) or the whole all_gather (fallback)"""
        if hdl is not None:
            hdl[i % 3].barrier()
        else:
            dist.all_gather_into_tensor(gath[i % 3], rec_i)

    def dev_loop(first, count):
        """N > 1: the gather of step i is finished on a side stream concurrently with the kernels of step i+1 (it is
        released by the start event of step i+1, so it cannot hide inside the untimed L2 flush); a step is complete when
        its kernels AND the previous step's gather are done; the last one is timed on its own."""
        pending = None                                       # (step, records) whose gather is not finished yet
        for i in range(first, first + count):
            c = i % EPISODE
            if c == 0:
                torch.cuda.synchronize()
                planner.reset(0, SCENES)
            flush.zero_()
            rec_i = d_recs[i % 3]
            if gat is not None:
                # step i+1 of the fused gather, deferred: this launch forwards the records of the launch before to every rank as its
                # warps start, raises that step's flags when its Decision half retires and waits for every rank's flag in its
                # last warp (depth 4: nobody overwrites a slice a peer still reads)
                gat.arm_deferred(i + 1)
                ev[i][0].record(stream)
                planner.cycle_dev(SCENES, d_hdr[c].data_ptr(), d_ox[c].data_ptr(), d_oy[c].data_ptr(), rec_i.data_ptr(),
                                  stream=stream.cuda_stream)
                ev[i][1].record(stream)
                ev[i][2].record(stream)
                pending = (i, rec_i)
                continue
            if hdl is not None:                              # this step's records go to slice `rank` of every rank's buffer i % 3
                planner.set_record_mirrors([p + rank * SCENES * 128 for p in hdl[i % 3].buffer_ptrs])
            ev[i][0].record(stream)
            if pending is not None:
                comm.wait_event(ev[i][0])
                with torch.cuda.stream(comm):
                    finish_gather(*pending)
                    gdone = torch.cuda.Event()
                    gdone.record(comm)
            planner.cycle_dev(SCENES, d_hdr[c].data_ptr(), d_ox[c].data_ptr(), d_oy[c].data_ptr(), rec_i.data_ptr(),
                              stream=stream.cuda_stream)
            ev[i][1].record(stream)
            if pending is not None:
                stream.wait_event(gdone)
            ev[i][2].record(stream)
            pending = (i, rec_i) if world > 1 else None
        if world > 1:
            tail_ev[0].record(stream)
            if gat is not None:
                gat.flush(stream=stream.cuda_stream)         # the last step's records: forwarded, flagged and awaited
            else:
                finish_gather(*pending)
            tail_ev[1].record(stream)
        return pending

    barrier()
    dev_loop(0, W)
    barrier()
    l0 = planner.launch_count()
    last = dev_loop(W, K)
    barrier()
    if world > 1 and gat is not None:                        # my gathered buffer of the last step holds every rank's records
        import ctypes as C_
        host = np.zeros((world, SCENES, 128), np.uint8)
        assert planner.lib.dp_memcpy_d2h(planner.ctx, abi.ptr(host), C_.c_void_p(gat.buffer(last[0] + 1)), C_.c_size_t(host.nbytes),
                                         C_.c_void_p(stream.cuda_stream)) == 0
        torch.cuda.synchronize()
        mine = last[1].cpu().numpy()
        assert np.array_equal(host[rank], mine), "own slice of the gathered records differs"
        allrec = [torch.zeros_like(last[1]) for _ in range(world)]
        dist.all_gather(allrec, last[1])
        for r in range(world):
            assert np.array_equal(host[r], allrec[r].cpu().numpy()), "gathered slice of rank %d differs" % r
        gat.disarm()
    elif world > 1:                                          # the gathered buffer of the last step holds every rank's records
        g = gath[last[0] % 3].view(world, SCENES, 128)
        assert torch.equal(g[rank], last[1]), "own slice of the gathered records differs"
        chk = torch.tensor([float(last[1][:, :].sum(dtype=torch.int64).item())], dtype=torch.float64, device=dev)
        allchk = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allchk, chk)
        for r in range(world):
            assert float(g[r].sum(dtype=torch.int64).item()) == float(allchk[r].item()), "gathered slice of rank %d differs" % r
        planner.set_record_mirrors([])
    dump = None
    if args.dump_outputs:                                    # copied now: the loops below write into d_recs again
        mine = d_recs[(W + K - 1) % 3]
        parts = [torch.empty_like(mine) for _ in range(world)] if world > 1 else [mine]
        if world > 1:
            dist.all_gather(parts, mine)
        dump = np.concatenate([t.cpu().numpy() for t in parts]).view(abi.plan_record).reshape(-1)
    launches = planner.launch_count() - l0 - sum(1 for i in range(W, W + K) if i % EPISODE == 0)
    kern_ms = np.array([ev[i][0].elapsed_time(ev[i][1]) for i in range(W, W + K)])
    step_ms = np.array([ev[i][0].elapsed_time(ev[i][2]) for i in range(W, W + K)])
    tail_ms = tail_ev[0].elapsed_time(tail_ev[1]) if world > 1 else 0.0
    cyc_idx = np.array([i % EPISODE for i in range(W, W + K)])
    total_ms = torch.tensor([step_ms.sum() + tail_ms], dtype=torch.float64, device=dev)
    traj = torch.tensor([float(traj_c[cyc_idx].sum())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(traj, op=dist.ReduceOp.SUM)
    total_s = float(total_ms.item()) * 1e-3
    value = float(traj.item()) / total_s

    # ---- cycle-latency histogram (BASELINE metric "p99 cycle latency"): LAT_N more cycles of the same workload, each one
    #      bracketed by CUDA events on the launching stream, L2 flushed before each, no gather; >= 10 000 samples for a real p99 ----
    lat = None
    if not args.no_extras:
        LAT_N = 10000
        lev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(LAT_N)]
        planner.set_record_mirrors([])
        for i in range(LAT_N):
            c = i % EPISODE
            if c == 0:
                planner.reset_dev(0, SCENES, stream=stream.cuda_stream)   # ON the launching stream: dp_reset runs on the context's own
            flush.zero_()
            lev[i][0].record(stream)
            planner.cycle_dev(SCENES, d_hdr[c].data_ptr(), d_ox[c].data_ptr(), d_oy[c].data_ptr(), d_recs[0].data_ptr(), stream=stream.cuda_stream)
            lev[i][1].record(stream)
        torch.cuda.synchronize()
        lms = np.array([a.elapsed_time(b) for a, b in lev])
        steady = lms[np.arange(LAT_N) % EPISODE != 0]        # without the first cycle of an episode (InitialPlanning for every scene)
        hist, edges = np.histogram(lms, bins=20)
        lat = {"samples": LAT_N, "p50": float(np.percentile(lms, 50)), "p90": float(np.percentile(lms, 90)), "p99": float(np.percentile(lms, 99)),
               "p99.9": float(np.percentile(lms, 99.9)), "max": float(lms.max()), "mean": float(lms.mean()),
               "steady": {"samples": int(steady.size), "p50": float(np.percentile(steady, 50)), "p99": float(np.percentile(steady, 99)),
                          "p99.9": float(np.percentile(steady, 99.9)), "max": float(steady.max()),
                          "what": "the same without the first cycle of each %d-cycle episode, where every scene runs InitialPlanning and "
                                  "writes its whole carried path (Planning.cpp:124-128)" % EPISODE},
               "histogram": {"edges_ms": [float(e) for e in edges], "counts": [int(h) for h in hist]},
               "p50_by_cycle_of_episode": [float(np.percentile(lms[np.arange(LAT_N) % EPISODE == c_], 50)) for c_ in range(EPISODE)],
               "what": "device time of one Decision+Planning cycle of %d scenes, CUDA events, cold L2 (256 MiB flush before every cycle)" % SCENES}
        barrier()

    # ---- end to end through the host-pointer C ABI: pinned host inputs, H2D + kernel + D2H every step ----
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()  # noqa: E731
    Hh = pin(H.view(np.uint8).reshape(EPISODE, SCENES, 128)).view(abi.scene_hdr).reshape(EPISODE, SCENES)
    OXh, OYh = pin(OX), pin(OY)
    rec_h = torch.empty((SCENES, 128), dtype=torch.uint8).pin_memory().numpy().view(abi.plan_record).reshape(SCENES)
    out = {"rec": rec_h}
    e2e_t = np.zeros(W + K)
    # N > 1: the end-to-end loops keep the gather: every record also goes to every peer's gathered buffer (mirrors set once,
    # buffer 0) and each step ends with the barrier that makes the gathered buffer readable
    if world > 1 and gat is None and hdl is not None:
        torch.cuda.synchronize()
        planner.set_record_mirrors([p + rank * SCENES * 128 for p in hdl[0].buffer_ptrs])
    gstep = [W + K + 1]                                      # fused-gather step numbers continue after the device loops

    def arm_gather(deferred=False):
        if gat is not None:
            gstep[0] += 1
            if deferred:
                gat.arm_deferred(gstep[0])                   # pipelined: this launch forwards / flags / awaits the step before
            else:
                gat.arm(gstep[0]); gat.chain(0)

    def step_gather():
        if world > 1:
            if gat is not None:
                gat.wait(gstep[0], stream=stream.cuda_stream)
            elif hdl is not None:
                hdl[0].barrier()
            else:
                dist.all_gather_into_tensor(gath[0], d_recs[0])
            torch.cuda.current_stream().synchronize()

    barrier()
    for i in range(W + K):
        c = i % EPISODE
        if c == 0:
            planner.reset(0, SCENES)
        if i == W:
            barrier()
        t0 = time.perf_counter()
        arm_gather()
        planner.cycle(Hh[c], OXh[c], OYh[c], out=out)
        step_gather()
        e2e_t[i] = time.perf_counter() - t0
    barrier()
    e2e_s = torch.tensor([e2e_t[W:].sum()], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_sync_val = float(traj.item()) / float(e2e_s.item())
    assert int(rec_h["n_traj"].astype(np.int64).sum()) == int(traj_c[(W + K - 1) % EPISODE]), "e2e result differs from replay"

    # ---- the same, pipelined: dp_cycle_submit / dp_cycle_wait, two cycles in flight.  Every step still moves its own
    #      inputs host->device and its records device->host inside the timed region; the region ends after the last wait. ----
    # THREE record buffers for two cycles in flight: the records of step s are read on the host AFTER step s+2 has been
    # submitted (it writes another buffer), so the read is off the wait(s) -> submit(s+2) turnaround that feeds the GPU
    recs2 = [rec_h] + [torch.empty((SCENES, 128), dtype=torch.uint8).pin_memory().numpy().view(abi.plan_record).reshape(SCENES) for _ in range(2)]
    import ctypes as C_

    CH = 32768                                               # dp_cycle_submit takes at most 32768 scenes per call
    chunks = [(s0, min(SCENES, s0 + CH)) for s0 in range(0, SCENES, CH)]
    vp = lambda a: C_.c_void_p(a.ctypes.data)                # noqa: E731  (addresses resolved once: the loop re-submits the same pinned buffers)
    in_ptr = [[(C_.c_int(s0), C_.c_int(s1 - s0), vp(Hh[c, s0:s1]), vp(OXh[c, s0:s1]), vp(OYh[c, s0:s1])) for s0, s1 in chunks] for c in range(EPISODE)]
    rec_ptr = [[vp(recs2[b][s0:s1]) for s0, s1 in chunks] for b in range(3)]

    def pipe_loop(first, count):
        got = 0; pend = []; k = 0                            # record slices in flight (at most two); k = submit counter
        for i in range(first, first + count):
            c = i % EPISODE
            if c == 0:
                while pend:
                    planner.wait(); got += int(pend.pop(0)["n_traj"].sum(dtype=np.int64))
                planner.reset(0, SCENES)
            for j, (s0, s1) in enumerate(chunks):
                done = None
                if len(pend) == 2:
                    planner.wait(); done = pend.pop(0)
                arm_gather(deferred=True)
                b = k % 3; k += 1
                planner.submit_raw(*in_ptr[c][j], rec_ptr[b][j])
                pend.append(recs2[b][s0:s1])
                if done is not None:
                    got += int(done["n_traj"].sum(dtype=np.int64))
        while pend:
            planner.wait(); got += int(pend.pop(0)["n_traj"].sum(dtype=np.int64))
        if gat is not None:
            gat.flush(stream=stream.cuda_stream)             # the last step's records; every earlier step was complete when its successor was
            torch.cuda.current_stream().synchronize()
        else:
            step_gather()
        return got

    barrier()
    pipe_loop(0, W)
    barrier()
    t0 = time.perf_counter()
    got = pipe_loop(W, K)
    pipe_t = time.perf_counter() - t0
    barrier()
    assert got == int(traj_c[cyc_idx].sum()), "pipelined e2e results differ from replay"
    e2e_p = torch.tensor([pipe_t], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_p, op=dist.ReduceOp.MAX)
    e2e_val = float(traj.item()) / float(e2e_p.item())
    if world > 1:
        torch.cuda.synchronize()
        if gat is not None:
            gat.disarm()
        planner.set_record_mirrors([])

    # ---- the other BASELINE configs (extra keys of the same line) ----
    extras = {}
    if not args.no_extras:
        from dmpp_b200.planner import Planner as P_

        def extra(key, fn, *a):
            """every extra key is measured on its own: one that fails reports its error and the others still run"""
            try:
                extras[key] = fn(*a)
            except Exception as e:  # noqa: BLE001
                extras[key] = {"error": repr(e)}

        if world == 1:
            extra("config3", config3_line, P_, m)
            extra("config3_distinct_geometry", config3_bezier_line, P_, m)
            extra("config4_shard", config4_line, torch, dist, P_, m, dev, rank, world, local_rank, 131072)
        else:
            extra("config4", config4_line, torch, dist, P_, m, dev, rank, world, local_rank, 1048576)
            extra("config3_split", config3_split_line, torch, dist, P_, m, dev, rank, world, local_rank)
        extra("config5", config5_line, torch, dist, P_, m, dev, rank, world, local_rank)
        extra("closed_loop", closed_loop_line, torch, dist, P_, m, dev, rank, world, local_rank)
        if world == 1:
            extra("output_frames", frames_line, torch, P_, m, dev, local_rank)
    sampler.stop = True
    sampler.join(timeout=2)

    if gat is not None:                                      # every rank is done with the peers' buffers before anyone unmaps them
        torch.cuda.synchronize()
        dist.barrier()
        gat.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    fp64_tf, fp32_tf = planner.measure_fma_peak()
    achieved = float(flops_c[cyc_idx].sum()) / (kern_ms.sum() * 1e-3) / 1e12
    bytes_scene = 128 + N_OBS * 16 + 2 * 128 + 3200 + 128        # hdr + obstacles + carry r/w + last path read + record
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic = None
    try:   # DRAM bytes per launch of dp_cycle_kernel from the committed `ncu --set full` capture of tools/profile_cycle.py
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_r2.json")))["dp_cycle_kernel"]["dram_bytes_per_launch"]
    except Exception:  # noqa: BLE001
        pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": float(step_ms.mean()), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": {k: (v.replace("GATHER_KIND", gather_kind) if isinstance(v, str) else v)
                                                        for k, v in workload_desc(world).items()},
        "plan_cycles_per_s": world * SCENES * K / total_s,
        "trajectories_per_step_per_gpu": float(traj_c[cyc_idx].mean()),
        "cycle_latency_ms": {"p50": float(np.percentile(step_ms, 50)), "p99": float(np.percentile(step_ms, 99)),
                             "max": float(step_ms.max()), "samples": int(K), "what": "device time of one Decision+Planning cycle of %d scenes (the K timed steps)" % SCENES},
        "e2e": {"value": e2e_val, "unit": UNIT,
                "h2d_bytes_per_step": SCENES * (128 + 2 * N_OBS * 8), "d2h_bytes_per_step": SCENES * 128,
                "ms_per_step": float(e2e_p.item()) / K * 1e3, "plan_cycles_per_s": world * SCENES * K / float(e2e_p.item()),
                "api": "dp_cycle_submit + dp_cycle_wait (host pointers, pinned; two cycles in flight: the inputs of step i+1 cross "
                       "PCIe while step i computes; every step's records land in one of three pinned buffers and are read on the host right after "
                       "step i+2 has been submitted; timed region ends after the last wait and the last read)",
                "synchronous": {"value": e2e_sync_val, "ms_per_step": float(e2e_t[W:].mean() * 1e3),
                                "plan_cycles_per_s": world * SCENES * K / float(e2e_s.item()),
                                "api": "dp_cycle_batch (host pointers, pinned; returns when the records are valid)"}},
        "gpu_launches": int(launches),
        "roofline": {"bound": "fp64", "kernel": "dp_cycle_kernel", "achieved": achieved, "peak": fp64_tf, "unit": "TFLOP/s",
                     "frac": achieved / fp64_tf if fp64_tf else None, "traffic": traffic,
                     "peak_source": "FP64 FMA micro-benchmark run in this process (dp_measure_fma_peak); MEASURED_PEAKS.json has no "
                                    "CUDA-core FP64 figure. fp32 FMA peak measured the same way: %.1f TFLOP/s" % fp32_tf,
                     "algorithmic_flops_per_launch": float(flops_c[cyc_idx].mean()),
                     "kernel_ms": float(kern_ms.mean()),
                     "hbm": {"achieved": SCENES * bytes_scene / (kern_ms.mean() * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "algorithmic_bytes_per_launch": SCENES * bytes_scene,
                             "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s"}},
        "clocks": sampler.result(),
    }
    if lat is not None:
        line["cycle_latency_ms"] = lat
    line.update(extras)
    if world > 1:
        line["e2e"]["gather"] = "included: every record is also stored into every peer's gathered buffer by the kernel, a barrier follows each synchronous step / the last pipelined wait"
    if world == 1 and not args.no_cpu_baseline:
        try:   # baseline (ii) of BASELINE.md section 3: the re-entrant restatement (oracle port) over all host cores, std::thread
            from oracle import binding as ob
            orc = ob.Oracle(); orc.set_map(m)
            cores = host_cores()
            t_traj = 0; t_s = 0.0; n = 0
            orc.run(H, OX, OY, paths=False, calls=False, trace=False, exhaustive=False, threads=cores)
            while t_s < 3.0 and n < 40:
                o_ = orc.run(H, OX, OY, paths=False, calls=False, trace=False, exhaustive=False, threads=cores)
                t_traj += int(o_["traj"]); t_s += float(o_["seconds"]); n += 1
            line["cpu_baseline_port"] = {"value": t_traj / t_s, "unit": UNIT, "cores": cores, "kind": "port", "per_core": t_traj / t_s / max(cores, 1),
                                         "sample": "%d passes over the GPU arm's %d scenes x %d cycles, re-entrant oracle restatement, one std::thread "
                                                   "per core (baseline (ii) of BASELINE.md section 3)" % (n, SCENES, EPISODE)}
            o1 = orc.run(np.ascontiguousarray(H[:, :256]), np.ascontiguousarray(OX[:, :256]), np.ascontiguousarray(OY[:, :256]), paths=False,
                         calls=False, trace=False, exhaustive=False, threads=1)
            line["cpu_baseline_port"]["one_thread"] = int(o1["traj"]) / float(o1["seconds"])
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline_port"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
        try:
            cores = host_cores()
            arm = CpuArm(min(SCENES, 4096), EPISODE, cores)
            arm.step()
            t_traj = 0; t_s = 0.0; n = 0
            while t_s < 4.0 and n < 40:
                t, dt, _ = arm.step()
                t_traj += t; t_s += dt; n += 1
            arm.close()
            line["cpu_baseline"] = {"value": t_traj / t_s, "unit": UNIT, "cores": cores, "kind": arm.kind, "per_core": t_traj / t_s / max(cores, 1),
                                    "sample": "%d passes over %d scenes x %d cycles, one process per core (unmodified reference "
                                              "objects when kind=reference)" % (n, min(SCENES, 4096), EPISODE)}
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
    emit(line)
    if dump is not None:
        dump_records(args.dump_outputs, dump)
    planner.close()
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_records(path, rec):
    """one float64 array per plan-record field, plus `scene`: the global scene index (= seed) of each row.  When all
    scenes would pass DUMP_MAX_BYTES, a fixed seeded sample of them, the same for every build of the project."""
    os.makedirs(path, exist_ok=True)
    names = ("scene",) + rec.dtype.names
    cap = DUMP_MAX_BYTES // (8 * len(names)) - 16             # (16 x 8 bytes: the .npy header of each file)
    idx = np.arange(rec.size) if rec.size <= cap else np.sort(np.random.default_rng(0).choice(rec.size, cap, replace=False))
    for f in names:
        a = idx if f == "scene" else rec[f][idx]
        np.save(os.path.join(path, f + ".npy"), a.astype(np.float64))
    print("plan records of the last timed step: %d of %d scenes written to %s" % (idx.size, rec.size, path), file=sys.stderr)


# ------------------------------------------------------------------------------------------------
# the other BASELINE configs, as extra keys of the same JSON line
# ------------------------------------------------------------------------------------------------
N_TRAJ_OFF = abi.plan_record.fields["n_traj"][1]             # byte offset of the uint16 trajectory count inside a plan record


def traj_of(torch, d_rec):
    """sum of plan_record.n_traj over a device buffer of records [n][128] uint8"""
    v = d_rec.view(torch.int16)[:, N_TRAJ_OFF // 2].to(torch.int64) & 0xffff
    return int(v.sum().item())


def device_cycles(torch, planner, n, d_hdr, d_ox, d_oy, d_rec, episode, warmup, steps, flush=None, after=None, before=None):
    """`warmup + steps` cycles of n scenes with inputs resident in HBM; per-step device ms (CUDA events on the launching
    stream) of the timed ones and the trajectories they scored.  `after(i)`: work enqueued after the cycle inside the timed
    region (the record gather of a multi-GPU run)."""
    st = torch.cuda.current_stream()
    ms, traj = [], 0
    for i in range(warmup + steps):
        c = i % episode
        if c == 0:
            torch.cuda.synchronize()
            planner.reset(0, n)
        if flush is not None:
            flush.zero_()
        if before is not None:
            before(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        planner.cycle_dev(n, d_hdr[c].data_ptr(), d_ox[c].data_ptr(), d_oy[c].data_ptr(), d_rec.data_ptr(), stream=st.cuda_stream)
        if after is not None:
            after(i)
        e1.record(st)
        if i >= warmup:
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
            traj += traj_of(torch, d_rec)
    return np.array(ms), traj


def config3_line(planner_cls, m, calls=10000):
    """BASELINE config 3: one scene, 65 536 candidates (64 lateral offsets x 32 aim distances x 32 horizons), 50 obstacle
    tracks, latency mode: one kernel launch per call, p50 / p99 over `calls` calls (host buffers in, winner out); device time
    (CUDA events around the launch) from a second loop so that the event synchronisation is not in the wall-clock figure."""
    bx, by, offset, n_pts, ox0, oy0, dvx, dvy = config3_grid(m)
    N = ox0.size
    p = planner_cls(16, 64)
    p.upload_map(m)
    sess = p.sweep_session(bx, by, offset, n_pts, 64)
    wall, dev = np.zeros(calls), np.zeros(calls)
    for i in range(50):
        sess.score(ox0, oy0, dvx, dvy, want_dis=False)
    l0 = p.launch_count()
    for i in range(calls):
        ox = ox0 + 0.01 * (i % 97)                            # the obstacles move between calls
        t0 = time.perf_counter()
        sess.score(ox, oy0, dvx, dvy, want_ms=False)
        wall[i] = time.perf_counter() - t0
    launches = p.launch_count() - l0
    for i in range(calls):
        dev[i] = sess.score(ox0 + 0.01 * (i % 97), oy0, dvx, dvy, want_dis=False)[2]
    rows = 0.0; groups = 0
    for off in np.unique(offset):
        ps = np.unique(n_pts[offset == off])
        rows += float(ps.max()); groups += ps.size
    flops = 18.0 * rows + N * (5.0 * rows + 12.0 * groups)
    pts_naive = float(n_pts.astype(np.int64).sum())
    fp64, _ = p.measure_fma_peak()
    sess.close(); p.close()
    return {"workload": "config3: 1 scene, 65536 candidates (64 lateral x 32 aim distances x 32 horizons), 50 obstacle tracks, one kernel launch per call",
            "calls": calls, "gpu_launches": int(launches),
            "latency_ms": {"p50": float(np.percentile(wall, 50) * 1e3), "p99": float(np.percentile(wall, 99) * 1e3), "max": float(wall.max() * 1e3),
                           "what": "wall clock of dp_sweep_score: host obstacle buffers in, winner index and its dis_lng on the host"},
            "latency_ms_device": {"p50": float(np.percentile(dev, 50)), "p99": float(np.percentile(dev, 99))},
            "candidates_per_s": offset.size / float(np.median(wall)),
            "roofline": {"bound": "fp64", "kernel": "sweep_rows_kernel", "unit": "TFLOP/s", "achieved": flops / (np.median(dev) * 1e-3) / 1e12,
                         "peak": fp64, "frac": flops / (np.median(dev) * 1e-3) / 1e12 / fp64, "algorithmic_flops_per_call": flops,
                         "flops_if_every_candidate_were_scored_alone": 18.0 * pts_naive + N * (5.0 * pts_naive + 12.0 * offset.size),
                         "note": "row-sharing formulation: candidates of one lateral offset share one pass per obstacle (3136 distinct (offset, "
                                 "horizon) groups, 64 rows); latency mode is bound by the dependent chain of one (row, obstacle) pass and the "
                                 "launch latency, not by the FMA roofline"}}


def config3_bezier_line(planner_cls, m, calls=2000):
    """config 3 with a longitudinal axis that changes GEOMETRY: 64 lateral offsets x 32 aim distances = 2048 distinct Bezier local
    paths (Planning.cpp:596-611: ego pose -> aim pose on the laterally shifted lane), each with 32 horizons (prefixes of ITS line)
    = 65 536 candidates, 50 obstacle tracks.  Per planning cycle: dp_sweep_set_bezier (all lines drawn on the device, arclength
    prefixes) once, then dp_sweep_score; both timed, each over `calls` calls."""
    rng = np.random.default_rng(77)
    gl = m.lane_index(3, 2)
    o = m.lane_pt_off[gl] + 700
    lx, ly, ld = m.x[o:o + 400], m.y[o:o + 400], m.dir[o:o + 400]
    n_lat, n_aim, n_hor = 64, 32, 32
    lat = np.linspace(-3.15, 3.15, n_lat)
    aim_id = np.linspace(40, 200, n_aim).astype(int)          # aim point 20 .. 100 m ahead
    poses = np.zeros((n_lat * n_aim, 6))
    for i, d in enumerate(lat):
        for k, a in enumerate(aim_id):
            h = np.deg2rad(ld[a])
            poses[i * n_aim + k] = (lx[0], ly[0], ld[0], lx[a] + d * np.sin(h), ly[a] - d * np.cos(h), ld[a])
    hor = np.linspace(8, 200, n_hor).astype(np.int32)
    cand_line = np.repeat(np.arange(n_lat * n_aim), n_hor).astype(np.int32)
    n_pts = np.tile(hor, n_lat * n_aim).astype(np.int32)
    off = np.zeros(cand_line.size)
    N = 50
    idx = rng.integers(10, 200, N)
    ox0, oy0 = lx[idx] + rng.normal(0, 2.0, N), ly[idx] + rng.normal(0, 2.0, N)
    dvx, dvy = rng.normal(0, 0.03, N), rng.normal(0, 0.03, N)
    p = planner_cls(16, 64)
    p.upload_map(m)
    sess = p.sweep_session(None, None, off, n_pts, 64, cand_line=cand_line, bezier_lines=n_lat * n_aim)
    sess.set_bezier(poses)
    for i in range(30):
        sess.score(ox0, oy0, dvx, dvy)
    wall, dev, setw, setd = np.zeros(calls), np.zeros(calls), np.zeros(calls), np.zeros(calls)
    l0 = p.launch_count()
    for i in range(calls):
        ps = poses.copy(); ps[:, 0] += 0.01 * (i % 50)          # the ego moves: new lines every cycle
        t0 = time.perf_counter()
        sess.set_bezier(ps)
        t1 = time.perf_counter()
        sess.score(ox0 + 0.01 * (i % 97), oy0, dvx, dvy, want_ms=False)
        t2 = time.perf_counter()
        setw[i], wall[i] = t1 - t0, t2 - t1                    # (set_bezier only enqueues; its device time is inside the score wall time)
    launches = p.launch_count() - l0
    for i in range(calls):
        setd[i] = sess.set_bezier(poses, want_ms=True)
        dev[i] = sess.score(ox0 + 0.01 * (i % 97), oy0, dvx, dvy, want_dis=False)[2]
    rows_pts = float(n_lat * n_aim * 200)
    groups = float(n_lat * n_aim * n_hor)
    flops = 18.0 * rows_pts + N * (5.0 * rows_pts + 12.0 * groups)
    fp64, _ = p.measure_fma_peak()
    sess.close(); p.close()
    pc = lambda a, q: float(np.percentile(a, q))              # noqa: E731
    return {"workload": "config3, distinct geometry: 2048 Bezier local paths (64 lateral x 32 aim distances) x 32 horizons = 65536 candidates, "
                        "50 obstacle tracks; lines re-drawn on the device every cycle",
            "calls": calls, "gpu_launches": int(launches),
            "cycle_latency_ms": {"p50": pc(setw + wall, 50) * 1e3, "p99": pc(setw + wall, 99) * 1e3,
                                 "what": "wall clock of dp_sweep_set_bezier + dp_sweep_score: poses and obstacles in, winner on the host"},
            "score_latency_ms_device": {"p50": pc(dev, 50), "p99": pc(dev, 99)},
            "set_bezier_ms_device": {"p50": pc(setd, 50), "p99": pc(setd, 99)},
            "candidates_per_s": cand_line.size / float(np.median(setw + wall)),
            "roofline": {"bound": "fp64", "kernel": "sweep_rows_kernel", "unit": "TFLOP/s", "achieved": flops / (np.median(dev) * 1e-3) / 1e12,
                         "peak": fp64, "frac": flops / (np.median(dev) * 1e-3) / 1e12 / fp64, "algorithmic_flops_per_call": flops,
                         "note": "2048 rows x 2 obstacle blocks x 4 parts of a row per warp (throughput shape of the same kernel)"}}


def config3_grid(m):
    rng = np.random.default_rng(2024)
    gl = m.lane_index(3, 2)
    o = m.lane_pt_off[gl] + 900
    bx, by = m.x[o:o + 256], m.y[o:o + 256]
    lat = -3.15 + 0.1 * np.arange(64)
    aim = 10.0 + 2.5 * np.arange(32)
    hor = 8 * (1 + np.arange(32))
    L, A, Hh = np.meshgrid(lat, aim, hor, indexing="ij")
    n_pts = np.minimum(Hh, np.maximum(2, (A / 0.5).astype(np.int64))).astype(np.int32).ravel()
    offset = L.ravel()
    N = 50
    idx = rng.integers(5, 250, N)
    ox0, oy0 = bx[idx] + rng.normal(0, 1.5, N), by[idx] + rng.normal(0, 1.5, N)
    dvx, dvy = rng.normal(0, 0.04, N), rng.normal(0, 0.04, N)
    return bx, by, offset, n_pts, ox0, oy0, dvx, dvy


def config3_split_line(torch, dist, planner_cls, m, dev, rank, world, local_rank, calls=2000):
    """cross-GPU argmin (SURVEY.md 8e): ONE scene's 65 536 candidates split over the ranks by contiguous index ranges; every
    rank scores its range (dp_sweep_score), the winners meet in a packed (cost bits << 32 | global index) int64 MIN all-reduce
    over NCCL: lowest cost first, lowest global index on ties -- the reference's first feasible candidate."""
    from dmpp_b200 import parallel
    bx, by, offset, n_pts, ox0, oy0, dvx, dvy = config3_grid(m)
    lo, hi = parallel.scene_range(offset.size, rank, world)
    p = planner_cls(16, 64, device=local_rank)
    p.upload_map(m)
    sess = p.sweep_session(bx, by, np.ascontiguousarray(offset[lo:hi]), np.ascontiguousarray(n_pts[lo:hi]), 64)
    full = p.sweep_session(bx, by, offset, n_pts, 64) if rank == 0 else None
    wall = np.zeros(calls)
    agree = True
    for i in range(calls + 20):
        ox = ox0 + 0.01 * (i % 97) - (2.0 if i % 5 == 0 else 0.0)           # the obstacles move between calls
        torch.cuda.synchronize(); dist.barrier()
        t0 = time.perf_counter()
        best, _, _ = sess.score(ox, oy0, dvx, dvy, want_dis=False)
        cost, win = parallel.global_argmin(0.0 if best >= 0 else float("inf"), (best + lo) if best >= 0 else 0xFFFFFFFF, device=dev)
        if i >= 20:
            wall[i - 20] = time.perf_counter() - t0
        if rank == 0 and i % 50 == 0:
            fb, _, _ = full.score(ox, oy0, dvx, dvy, want_dis=False)
            agree = agree and ((fb < 0 and cost == float("inf")) or (fb >= 0 and cost == 0.0 and win == fb))
    sess.close()
    if full is not None:
        full.close()
    p.close()
    return {"workload": "config3 split %d-way: 65536 candidates of ONE scene by contiguous index ranges, packed int64 MIN all-reduce (NCCL) of the winners" % world,
            "calls": calls, "latency_ms": {"p50": float(np.percentile(wall, 50) * 1e3), "p99": float(np.percentile(wall, 99) * 1e3)},
            "winner_equals_single_gpu": bool(agree)}


def config4_line(torch, dist, planner_cls, m, dev, rank, world, local_rank, total_scenes, episode=12, warmup=2, steps=10):
    """BASELINE config 4: the Monte-Carlo scene sweep (default candidate set), total_scenes split over the ranks by contiguous
    seed ranges; when world > 1 every rank's plan records are stored into every rank's gathered buffer by the kernel itself
    (NVLink peer stores, dp_set_record_mirrors) and a barrier closes each step inside the timed region."""
    n = total_scenes // world
    seeds = np.arange(rank * n, (rank + 1) * n)
    ep = scenes.Episodes(m, seeds, cycles=episode, n_obs=N_OBS)
    H, OX, OY = ep.all_cycles()
    p = planner_cls(max_scenes=n, max_obs=N_OBS, device=local_rank)
    p.upload_map(m)
    d_hdr = torch.from_numpy(H.view(np.uint8).reshape(episode, n, 128)).to(dev)
    d_ox = torch.from_numpy(OX).to(dev); d_oy = torch.from_numpy(OY).to(dev)
    d_rec = torch.empty((n, 128), dtype=torch.uint8, device=dev)
    gather = "none"; after = None; hdl = None; gat = None
    if world > 1 and not os.environ.get("DP_BENCH_NO_IPC"):
        try:
            from dmpp_b200.planner import Gather
            gat = Gather(p, world, rank, n, depth=4)
            gat.set_lag(2)
            hs = [None] * world
            dist.all_gather_object(hs, gat.my_handle())
            gat.attach(hs)
            st_ = torch.cuda.current_stream()
            cnt = [0]

            # many waves per launch: the eager variant (records stored on every rank as each Planning warp ends) measured cheaper than
            # the deferred one (131072 scenes per GPU, 2 GPUs: 1.95 ms without a gather, 2.04 eager, 2.14 deferred; tools/config4_probe.py)
            mode4 = os.environ.get("DP_CFG4_GATHER", "eager")

            def before(i):
                cnt[0] += 1
                if mode4 == "deferred":
                    gat.arm_deferred(cnt[0])
                elif mode4 == "eager":
                    gat.arm(cnt[0])
            after = (lambda i: gat.wait(cnt[0], stream=st_.cuda_stream)) if mode4 == "eager" else None
            gather = {"deferred": "dp_gather_* (C ABI, CUDA IPC), deferred: the launch of step i+1 forwards step i's records to every rank, raises the "
                                  "flags and awaits every rank's flags of step i-1; the last two steps' gathers (dp_gather_flush) are timed and added",
                      "eager": "dp_gather_* (C ABI, CUDA IPC), eager: peer stores + flags from the kernel as it ends, wait for every rank's flag inside the timed step",
                      "none": "NO gather (experiment)"}[mode4]
        except Exception as e:  # noqa: BLE001
            gat = None
            gather = "dp_gather failed (%s)" % type(e).__name__
    if world > 1 and gat is None:
        try:
            import torch.distributed._symmetric_memory as symm
            g = symm.empty((world * n, 128), dtype=torch.uint8, device=dev)
            hdl = symm.rendezvous(g, dist.group.WORLD)
            p.set_record_mirrors([q + rank * n * 128 for q in hdl.buffer_ptrs])
            after = lambda i: hdl.barrier()                  # noqa: E731
            gather = "peer stores from the kernel (NVLink, symmetric memory) + barrier, inside the timed step"
        except Exception as e:  # noqa: BLE001
            gbuf = torch.empty((world * n, 128), dtype=torch.uint8, device=dev)
            after = lambda i: dist.all_gather_into_tensor(gbuf, d_rec)   # noqa: E731
            gather = "all_gather_into_tensor inside the timed step (%s)" % type(e).__name__
    l0 = p.launch_count()
    ms, traj = device_cycles(torch, p, n, d_hdr, d_ox, d_oy, d_rec, episode, warmup, steps, after=after, before=before if gat is not None else None)
    tail = 0.0
    if gat is not None:                                      # the gathers still in flight belong to the timed work
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        st_ = torch.cuda.current_stream()
        e0.record(st_); gat.flush(stream=st_.cuda_stream); e1.record(st_)
        torch.cuda.synchronize()
        tail = e0.elapsed_time(e1)
    launches = p.launch_count() - l0
    t = torch.tensor([ms.sum() + tail], dtype=torch.float64, device=dev)
    tr = torch.tensor([float(traj)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tr, op=dist.ReduceOp.SUM)
        if gat is not None:
            gat.close()
        p.set_record_mirrors([])
    p.close()
    secs = float(t.item()) * 1e-3
    return {"workload": "config4: %d scenes (seeds 0..%d) x default candidate set, sharded %d-way by contiguous seed ranges, %d-cycle episodes"
                        % (n * world, n * world - 1, world, episode),
            "scenes_total": n * world, "scenes_per_gpu": n, "steps": steps, "warmup": warmup, "gather": gather,
            "value": float(tr.item()) / secs, "unit": UNIT, "plan_cycles_per_s": n * world * steps / secs,
            "ms_per_step": secs / steps * 1e3, "ns_per_scene_cycle": secs / steps / (n * world) * 1e9 * world,
            "gpu_launches": int(launches), "scaling": "strong" if world > 1 else "single GPU shard",
            "l2": "inputs (%.0f MB per cycle per GPU) exceed the 126 MB L2; no flush needed" % ((128 + 16 * N_OBS) * n / 1e6)}


def config5_line(torch, dist, planner_cls, m, dev, rank, world, local_rank, n=1024, n_obs=200, episode=40, warmup=3, steps=20):
    """BASELINE config 5: urban junction scenes (reference path = lane + connector, ~400 points, pos 1 / 2), 200 agents per scene
    with constant-turn-rate predicted tracks, T = 400 steps of 0.02 s (8 s horizon): one launch of the group kernel per step --
    track rollout fused into the junction search against the moving agents (never materialised), Decision rule tree, Planning.
    Weak scaling: n scenes per GPU."""
    seeds = np.arange(7_000_000 + rank * n, 7_000_000 + (rank + 1) * n)
    ep = scenes.Episodes(m, seeds, cycles=episode, n_obs=n_obs, kind="urban")
    H, OX, OY, VX, VY, DTH = ep.all_cycles_tracks()
    T = ep.TRACK_T
    p = planner_cls(max_scenes=n, max_obs=n_obs, device=local_rank)
    p.upload_map(m)
    d_hdr = torch.from_numpy(H.view(np.uint8).reshape(episode, n, 128)).to(dev)
    d_ox = torch.from_numpy(OX).to(dev); d_oy = torch.from_numpy(OY).to(dev)
    d_vx = torch.from_numpy(VX).to(dev); d_vy = torch.from_numpy(VY).to(dev); d_dth = torch.from_numpy(DTH).to(dev)
    d_rec = torch.empty((n, 128), dtype=torch.uint8, device=dev)
    d_tr = torch.zeros((n, abi.trace_record.itemsize), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    ms, traj, pts = [], 0, 0
    l0 = p.launch_count()
    for i in range(warmup + steps):
        c = i % episode
        if c == 0:
            torch.cuda.synchronize()
            p.reset(0, n)
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        p.set_tracks_dev(T, d_vx[c].data_ptr(), d_vy[c].data_ptr(), d_dth[c].data_ptr())
        p.cycle_dev(n, d_hdr[c].data_ptr(), d_ox[c].data_ptr(), d_oy[c].data_ptr(), d_rec.data_ptr(), d_trace=d_tr.data_ptr(), stream=st.cuda_stream)
        e1.record(st)
        if i >= warmup:
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
            traj += traj_of(torch, d_rec)
            pts += int(d_tr.view(torch.int32)[:, abi.trace_record.fields["pts_scored"][1] // 4].to(torch.int64).sum().item())
    launches = p.launch_count() - l0
    ms = np.array(ms)
    t = torch.tensor([ms.sum()], dtype=torch.float64, device=dev)
    tr = torch.tensor([float(traj), float(pts)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tr, op=dist.ReduceOp.SUM)
    fp64, _ = p.measure_fma_peak()
    p.close()
    secs = float(t.item()) * 1e-3
    flops = alg_flops(float(tr[1].item()), float(tr[0].item()), n_obs)
    return {"workload": "config5: %d urban junction scenes/GPU x %d agents with constant-turn-rate tracks (T = %d x 0.02 s), lane + connector "
                        "reference path (~400 points), %d-cycle episodes; one group-kernel launch per step" % (n, n_obs, T, episode),
            "scenes_per_gpu": n, "agents": n_obs, "track_steps": T, "steps": steps, "warmup": warmup,
            "value": float(tr[0].item()) / secs, "unit": UNIT, "plan_cycles_per_s": n * world * steps / secs,
            "agent_checks_per_s": float(tr[0].item()) * n_obs / secs, "path_points_per_trajectory": float(tr[1].item()) / max(float(tr[0].item()), 1.0),
            "ms_per_step": secs / steps * 1e3, "p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99)),
            "gpu_launches": int(launches), "scaling": "weak", "l2": "256 MiB buffer written between timed steps",
            "roofline": {"bound": "fp64", "kernel": "dp_group_kernel", "unit": "TFLOP/s", "achieved": flops / secs / 1e12 / world, "peak": fp64,
                         "frac": flops / secs / 1e12 / world / fp64, "note": "algorithmic flops F(P,N) = 18 P + N (5 P + 12) of the trajectories scored "
                         "(SURVEY.md 8d), per GPU; the pruned search evaluates a fraction of the P x N pairs, so this is work done per second, "
                         "not FMA-pipe utilisation"},
            "tracks": "constant-turn-rate rollout fused into the search: T x N positions per scene exist only in registers"}


def measured_hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback 6650 GB/s"


def closed_loop_line(torch, dist, planner_cls, m, dev, rank, world, local_rank, n=4096, cycles=25, reps=10):
    """SURVEY.md 8f rank 1: closed-loop episodes.  Ego, agents and localisation are advanced on the device between cycles
    (dp_world_kernel), the carry never leaves HBM, and a whole episode of `cycles` x (Decision + Planning launch pair, world step)
    is ONE CUDA graph launch (dp_run_closed_loop_dev).  Weak scaling: n worlds per GPU, no exchange between ranks.  Warm L2 (the
    episode is one launch: nothing can be flushed in between), CUDA events around the whole episode."""
    w = scenes.World(m, np.arange(9_000_000 + rank * n, 9_000_000 + (rank + 1) * n), 10)
    p = planner_cls(max_scenes=n, max_obs=10, device=local_rank)
    p.upload_map(m)
    h0 = torch.from_numpy(w.hdr.view(np.uint8).reshape(n, 128)).to(dev)
    a0 = torch.from_numpy(w.agents.view(np.uint8).reshape(n, 320)).to(dev)
    d_h, d_a = torch.empty_like(h0), torch.empty_like(a0)
    d_x = torch.zeros((n, 10), dtype=torch.float64, device=dev); d_y = torch.zeros_like(d_x)
    d_r = torch.zeros((cycles, n, 128), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    ms, traj = [], 0
    l0 = p.launch_count()
    for r in range(reps):
        d_h.copy_(h0); d_a.copy_(a0)
        p.reset_dev(0, n, stream=st.cuda_stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        p.run_closed_loop_dev(n, cycles, d_h.data_ptr(), d_a.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), stream=st.cuda_stream)
        e1.record(st)
        torch.cuda.synchronize()
        if r >= 3:
            ms.append(e0.elapsed_time(e1))
            traj += traj_of(torch, d_r.reshape(cycles * n, 128))
    launches = p.launch_count() - l0
    graph = p.closed_loop_is_graph()
    p.close()
    ms = np.array(ms)
    t = torch.tensor([ms.sum()], dtype=torch.float64, device=dev)
    tr = torch.tensor([float(traj)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tr, op=dist.ReduceOp.SUM)
    secs = float(t.item()) * 1e-3
    eps = len(ms)
    return {"workload": "closed loop: %d worlds/GPU (the config-2 scene draw at cycle 0, then nothing scripted) x %d cycles; ego walked "
                        "along its own plan, agents along their lanes, windowed re-localisation, all on the device" % (n, cycles),
            "worlds_per_gpu": n, "cycles": cycles, "episodes_timed": eps, "one_graph_launch_per_episode": bool(graph),
            "value": float(tr[0].item()) / secs, "unit": UNIT, "plan_cycles_per_s": n * world * cycles * eps / secs,
            "ms_per_episode": secs / eps * 1e3, "us_per_cycle": secs / eps / cycles * 1e6, "p50_ms_per_episode": float(np.percentile(ms, 50)),
            "gpu_launches": int(launches), "kernels_per_episode": 3 * cycles + 1, "scaling": "weak", "l2": "warm (one launch per episode)"}


def frames_line(torch, planner_cls, m, dev, local_rank, n=131072, reps=20):
    """SURVEY.md 8f rank 3: the output stage.  dp_frames_kernel packs PlanningOut (1656 B) and PlanningStatus (1632 B) per scene
    from the 128-byte plan record and the carried 3200-byte local path: byte work bound by HBM, measured against the copy peak
    of MEASURED_PEAKS.json with a cold L2."""
    ep = scenes.Episodes(m, np.arange(n), cycles=1, n_obs=10)
    H, OX, OY = ep.all_cycles()
    p = planner_cls(max_scenes=n, max_obs=10, device=local_rank)
    p.upload_map(m)
    d_h = torch.from_numpy(H[0].view(np.uint8).reshape(n, 128)).to(dev)
    d_x, d_y = torch.from_numpy(OX[0]).to(dev), torch.from_numpy(OY[0]).to(dev)
    d_r = torch.zeros((n, 128), dtype=torch.uint8, device=dev)
    d_c = torch.zeros((n, abi.ctrl_frame.itemsize), dtype=torch.uint8, device=dev)
    d_s = torch.zeros((n, abi.status_frame.itemsize), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    p.reset_dev(0, n, stream=st.cuda_stream)
    p.cycle_dev(n, d_h.data_ptr(), d_x.data_ptr(), d_y.data_ptr(), d_r.data_ptr(), stream=st.cuda_stream)
    ms = []
    for r in range(reps):
        flush.fill_(r & 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        p.pack_frames_dev(n, d_r.data_ptr(), d_c.data_ptr(), d_s.data_ptr(), stream=st.cuda_stream)
        e1.record(st)
        torch.cuda.synchronize()
        if r >= 3:
            ms.append(e0.elapsed_time(e1))
    p.close()
    peak, src = measured_hbm_peak()
    t = float(np.median(ms)) * 1e-3
    by = n * (128 + 3200 + abi.ctrl_frame.itemsize + abi.status_frame.itemsize)
    return {"workload": "PlanningOut + PlanningStatus frames of %d scenes, one launch" % n, "scenes": n, "ms": t * 1e3,
            "frames_per_s": 2 * n / t, "gpu_launches": reps,
            "roofline": {"bound": "hbm", "kernel": "dp_frames_kernel", "unit": "GB/s", "achieved": by / t / 1e9, "peak": peak,
                         "frac": by / t / 1e9 / peak, "algorithmic_bytes_per_launch": by, "peak_source": src,
                         "note": "bytes = scenes x (128 record + 3200 carried path in, 1656 + 1632 frames out)"},
            "l2": "256 MiB buffer written before every launch"}


_OUT_FD = None


def emit(line):
    """the ONE JSON line goes to the real stdout; everything else any library prints (NCCL's version banner ...) was
    redirected to stderr in main()"""
    data = (json.dumps(line) + "\n").encode()
    if _OUT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_OUT_FD, data)


def main():
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)                                            # C-level and Python-level stdout -> stderr from here on
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the latency histogram and the config 3 / 4 / 5 keys")
    ap.add_argument("--scenes", type=int, default=SCENES,
                    help="scenes per GPU (default = BASELINE config 2; 131072 x 8 GPUs = config 4, the 1M-scene sweep)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the plan records of the last one (every rank's) as DIR/<field>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: use it with --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    globals()["SCENES"] = args.scenes
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
