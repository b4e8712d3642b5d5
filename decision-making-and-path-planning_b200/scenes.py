"""Deterministic synthetic HD map + scripted scene episodes (SURVEY.md section 8d).

Neutral input generation: the same arrays feed the unmodified reference (oracle/_ref), the CPU
restatement (oracle/) and the CUDA path, so nothing here is part of either side of a parity check.
Randomness is a stateless SplitMix64 hash of (scene seed, stream, index): scene s of any batch is
always the same scene, whatever the batch size or the rank that generates it.

Map (all lanes 2000 points, ~0.5 m spacing; lane 1 is the LEFTMOST lane, as in the reference where
the left neighbour of lane n is lane n-1, Decision.cpp:602-604):
  road 1  straight, heading 0 deg,   3 lanes, lanechg_attribute {2,3,1}   (lane changes allowed)
  road 2  straight, heading 30 deg,  3 lanes, attribute 0                 (in-lane avoid sweep)
  road 3  arc R=400 m (left turn),   3 lanes, attribute {2,3,1}
  road 4  S-curve,                   3 lanes, attribute 0 up to id 700, {2,3,1} to 1500, 0 after
  road 5  straight, heading 200 deg, 2 lanes, attribute {3,2}: both neighbours are virtual
                                     (CreateNewPath(+-W), Decision.cpp:629-631,667-669)
  road 6  approach,  heading 90 deg, 2 lanes, 400 points, attribute 0     (junction scenes)
  road 7  departure, heading 180 deg,2 lanes, 400 points, attribute 0
  road 8  straight, heading 75 deg,  3 lanes, attribute of lanes 1 and 2: 2 at every 128th point, 3 elsewhere; lane 3: 1
                                     (the only shape on which the obstacle-motivated RIGHT change of Decision.cpp:1296-1424
                                     can fire: attribute exactly 2 at the ego's point, odd attributes ahead, quirk 1)
  connectors 6->7: lane 1->1 and lane 2->2, quarter circle left turn

`Episodes` draws seeded scenes; `Directed` scripts the scene families that the random mix (almost) never reaches -- the
right lane change (behaviour 3) sites of the rule tree.
"""
import ctypes as C
import math

import numpy as np

from . import abi

LANE_W = 3.75
SPACING = 0.5
N_PTS = 2000
MASK = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x):
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = x + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def rnd(seed, stream, k=0):
    """uniform [0,1) double, stateless in (seed, stream, k); all arguments broadcast."""
    with np.errstate(over="ignore"):
        s = (np.asarray(seed, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
             + np.asarray(stream, dtype=np.uint64) * np.uint64(0xD1B54A32D192ED03)
             + np.asarray(k, dtype=np.uint64) * np.uint64(0x8CB92BA72F3D8DD7))
    return (splitmix64(splitmix64(s)) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


class Map:
    """SoA map tables + the dp_map_desc view of them."""

    def __init__(self):
        xs, ys, dirs, widths, attrs = [], [], [], [], []
        self.road_lane_base = [0]
        self.lane_pt_off = [0]
        self.lane_road = []
        conns = []

        def add_lane(cx, cy, hd, d_left, attr):
            # offset the centre line by d_left metres to the LEFT of travel
            h = np.radians(hd)
            x = cx - d_left * np.sin(h)
            y = cy + d_left * np.cos(h)
            xs.append(x); ys.append(y); dirs.append(np.mod(hd, 360.0))
            widths.append(np.full(x.shape, int(round(LANE_W * 100)), np.uint16))
            attrs.append(np.broadcast_to(np.asarray(attr, np.uint16), x.shape).copy())
            self.lane_pt_off.append(self.lane_pt_off[-1] + x.size)

        def add_road(cx, cy, hd, lane_attrs):
            n = len(lane_attrs)
            for l in range(n):                      # lane 1 leftmost
                d_left = (0.5 * (n - 1) - l) * LANE_W
                add_lane(cx, cy, hd, d_left, lane_attrs[l])
                self.lane_road.append(len(self.road_lane_base))
            self.road_lane_base.append(self.road_lane_base[-1] + n)

        s = np.arange(N_PTS) * SPACING
        # road 1: straight east
        add_road(100.0 + s, 50.0 + 0 * s, np.zeros(N_PTS), [2, 3, 1])
        # road 2: straight, heading 30 deg
        c30, s30 = math.cos(math.radians(30.0)), math.sin(math.radians(30.0))
        add_road(-500.0 + s * c30, 200.0 + s * s30, np.full(N_PTS, 30.0), [0, 0, 0])
        # road 3: arc, radius 400 m, turning left, starting heading 10 deg
        R = 400.0
        th = np.radians(10.0) + s / R
        add_road(2000.0 + R * (np.sin(th) - math.sin(math.radians(10.0))),
                 -300.0 - R * (np.cos(th) - math.cos(math.radians(10.0))), np.degrees(th), [2, 3, 1])
        # road 4: S-curve y = A sin(2 pi x / Lw)
        A, Lw = 12.0, 400.0
        x4 = s
        y4 = A * np.sin(2 * np.pi * x4 / Lw)
        hd4 = np.degrees(np.arctan2(A * 2 * np.pi / Lw * np.cos(2 * np.pi * x4 / Lw), 1.0))
        ids = np.arange(N_PTS)
        seg = lambda a: np.where(ids < 700, 0, np.where(ids < 1500, a, 0))
        add_road(-1500.0 + x4, -800.0 + y4, hd4, [seg(2), seg(3), seg(1)])
        # road 5: straight heading 200 deg, 2 lanes with virtual neighbours
        c2, s2 = math.cos(math.radians(200.0)), math.sin(math.radians(200.0))
        add_road(800.0 + s * c2, 1500.0 + s * s2, np.full(N_PTS, 200.0), [3, 2])
        # roads 6/7 + connectors (junction)
        n_j = 400
        sj = np.arange(n_j) * SPACING
        jx, jy = 3000.0, 1000.0                      # stop line of the approach (north-bound)
        add_road(jx + 0 * sj, jy - (n_j - 1) * SPACING + sj, np.full(n_j, 90.0), [0, 0])
        Rc = 14.0                                    # left turn: north -> west
        add_road(jx - Rc - 0.5 - sj, jy + Rc + 0.5 + 0 * sj, np.full(n_j, 180.0), [0, 0])
        # road 8: straight heading 75 deg; lanes 1/2 carry attribute 2 on isolated points, 3 in between
        c8, s8 = math.cos(math.radians(75.0)), math.sin(math.radians(75.0))
        a23 = np.where(ids % 128 == 0, 2, 3)
        add_road(-2500.0 + s * c8, 900.0 + s * s8, np.full(N_PTS, 75.0), [a23, a23, 1])
        self.n_road_lanes = self.road_lane_base[-1]
        for l in (0, 1):                             # connector lane l+1 -> lane l+1
            r_l = Rc + (0.5 - l) * LANE_W            # left lane (l=0) has the smaller radius
            n_c = int(r_l * (math.pi / 2) / SPACING) + 2
            a = np.linspace(0.0, math.pi / 2, n_c)
            # centre of the turn is (jx - Rc - 0.5, jy + 0.5); start heading north at angle 0
            ccx, ccy = jx - Rc - 0.5, jy + 0.5
            px = ccx + r_l * np.cos(a)
            py = ccy + r_l * np.sin(a)
            xs.append(px); ys.append(py); dirs.append(np.mod(90.0 + np.degrees(a), 360.0))
            widths.append(np.full(px.shape, int(round(LANE_W * 100)), np.uint16))
            attrs.append(np.zeros(px.shape, np.uint16))
            self.lane_pt_off.append(self.lane_pt_off[-1] + px.size)
            conns.append((6, 7, l + 1, l + 1, len(self.lane_pt_off) - 2))

        self.x = np.ascontiguousarray(np.concatenate(xs), np.float64)
        self.y = np.ascontiguousarray(np.concatenate(ys), np.float64)
        self.dir = np.ascontiguousarray(np.concatenate(dirs), np.float64)
        self.lane_width = np.ascontiguousarray(np.concatenate(widths), np.uint16)
        self.lanechg_attr = np.ascontiguousarray(np.concatenate(attrs), np.uint16)
        self.road_lane_base = np.asarray(self.road_lane_base, np.int32)
        self.lane_pt_off = np.asarray(self.lane_pt_off, np.int32)
        self.conn = np.array(conns, dtype=abi.connector)
        self.n_roads = len(self.road_lane_base) - 1
        self.n_lanes = len(self.lane_pt_off) - 1

    def lanes_of(self, road):
        return int(self.road_lane_base[road] - self.road_lane_base[road - 1])

    def lane_index(self, road, lane):
        return int(self.road_lane_base[road - 1]) + lane - 1

    def desc(self):
        d = abi.MapDesc()
        d.n_roads = self.n_roads
        d.road_lane_base = self.road_lane_base.ctypes.data
        d.n_lanes = self.n_lanes
        d.lane_pt_off = self.lane_pt_off.ctypes.data
        d.n_conn = len(self.conn)
        d.conn = self.conn.ctypes.data
        d.n_points = self.x.size
        d.x = self.x.ctypes.data
        d.y = self.y.ctypes.data
        d.dir = self.dir.ctypes.data
        d.lane_width = self.lane_width.ctypes.data
        d.lanechg_attr = self.lanechg_attr.ctypes.data
        return d


# streams of the per-scene hash
(S_ROAD, S_LANE, S_ID0, S_SPEED, S_WOB_A, S_WOB_W, S_NAV, S_NAVL, S_CHG, S_CHG_T, S_CHG_D, S_YAW,
 S_PERIOD, S_OB_LANE, S_OB_S, S_OB_V, S_OB_LAT, S_KIND, S_OB_NEAR) = range(19)


class Episodes:
    """Scripted (open-loop) episodes: `hdr(c)`, `obstacles(c)` give the inputs of cycle c for all scenes.

    kind: 'highway' (roads 1-5, pos 0), 'junction' (roads 6/7 + connector, pos 0 -> 1 -> 2 -> 0) or 'urban' (BASELINE config 5:
    the same junction approached from far away with the whole approach treated as the pre-junction zone, so the reference
    path lane + connector has ~400 points; `tracks(c)` gives every agent a constant-turn-rate prediction, T = 400 steps of 0.02 s).
    """
    TRACK_T = 400
    TRACK_DT = 0.02

    def __init__(self, m: Map, seeds, n_obs=10, kind="highway", cycles=25, roads=None):
        self.m = m
        self.seeds = np.asarray(seeds, dtype=np.uint64)
        self.n = self.seeds.size
        self.n_obs = int(n_obs)
        self.kind = kind
        self.cycles = cycles
        sd = self.seeds
        if kind == "highway":
            roads = np.asarray(roads if roads is not None else [1, 2, 3, 4, 5], np.int32)
            self.road = roads[(rnd(sd, S_ROAD) * len(roads)).astype(np.int64)]
            nl = (m.road_lane_base[self.road] - m.road_lane_base[self.road - 1]).astype(np.int64)
            self.lane0 = 1 + (rnd(sd, S_LANE) * nl).astype(np.int64)
            self.nl = nl
            self.s0 = 60.0 + rnd(sd, S_ID0) * 820.0           # metres along the lane
            # a few scenes start close to the lane end (shortened front path, Decision.cpp:581)
            near_end = rnd(sd, S_KIND) < 0.04
            self.s0 = np.where(near_end, 925.0 + rnd(sd, S_ID0) * 30.0, self.s0)
            self.v = 15.0 + rnd(sd, S_SPEED) * 60.0           # km/h
        else:
            self.road = np.full(self.n, 6, np.int32)
            self.nl = np.full(self.n, 2, np.int64)
            self.lane0 = 1 + (rnd(sd, S_LANE) * 2).astype(np.int64)
            self.s0 = 150.0 + rnd(sd, S_ID0) * 35.0           # 14.5 .. 49.5 m before the stop line
            if kind == "urban":                               # 70 % of the scenes start 170-190 m before it
                self.s0 = np.where(rnd(sd, S_KIND) < 0.7, 10.0 + rnd(sd, S_ID0) * 20.0, self.s0)
            self.v = 12.0 + rnd(sd, S_SPEED) * 25.0
        self.wob_a = rnd(sd, S_WOB_A) * 0.3
        self.wob_w = 0.2 + rnd(sd, S_WOB_W) * 0.6
        # scripted ego lane change: direction +-1 at cycle t, only where a real neighbour exists
        chg = rnd(sd, S_CHG) < (0.3 if kind == "highway" else 0.0)
        d = np.where(rnd(sd, S_CHG_D) < 0.5, -1, 1)
        ok = (self.lane0 + d >= 1) & (self.lane0 + d <= self.nl)
        self.chg_dir = np.where(chg & ok, d, 0)
        self.chg_t = 3 + (rnd(sd, S_CHG_T) * max(1, cycles - 6)).astype(np.int64)
        # navigation: 0.55 no demand (all lanes exit), else a single exit lane
        nav_all = rnd(sd, S_NAV) < 0.55
        self.nav_lane = np.where(nav_all, 0, 1 + (rnd(sd, S_NAVL) * self.nl).astype(np.int64))
        # obstacles: lane, start offset relative to ego (m), speed (m/s), lateral jitter (m)
        k = np.arange(self.n_obs, dtype=np.uint64)[None, :]
        s2 = sd[:, None]
        self.ob_lane = 1 + (rnd(s2, S_OB_LANE, k) * self.nl[:, None]).astype(np.int64)
        rel = -25.0 + rnd(s2, S_OB_S, k) * 125.0
        # make the first obstacle a near in-lane blocker in 45 % of the scenes (arms avoid / lane change)
        near = (rnd(sd, S_OB_NEAR) < 0.45)
        rel[:, 0] = np.where(near, 6.0 + rnd(sd, S_OB_S, 1000) * 16.0, rel[:, 0])
        self.ob_lane[:, 0] = np.where(near, self.lane0, self.ob_lane[:, 0])
        self.ob_s0 = self.s0[:, None] + rel
        self.ob_v = rnd(s2, S_OB_V, k) * 18.0
        self.ob_v[:, 0] = np.where(near, self.v / 3.6 * (0.5 + 0.5 * rnd(sd, S_OB_V, 1000)), self.ob_v[:, 0])
        self.ob_lat = (rnd(s2, S_OB_LAT, k) - 0.5) * 1.2
        self.t = np.zeros(self.n)                               # elapsed ms, advanced by hdr()
        self._t_cache = {}

    # ---- helpers ------------------------------------------------------------------------------
    def period_ticks(self, c):
        return 80 + (rnd(self.seeds, S_PERIOD, c) * 41.0).astype(np.int64)

    def elapsed_s(self, c):
        """scripted time at the START of cycle c (sum of the periods of cycles < c), seconds."""
        if c not in self._t_cache:
            t = np.zeros(self.n)
            for i in range(c):
                t = t + self.period_ticks(i) / 1000.0
            self._t_cache[c] = t
        return self._t_cache[c]

    def _lane_xy(self, lane_idx, s):
        """point at arclength-parameter s (metres, index = s / SPACING) of global lane lane_idx."""
        m = self.m
        off = m.lane_pt_off[lane_idx].astype(np.int64)
        cnt = (m.lane_pt_off[lane_idx + 1] - m.lane_pt_off[lane_idx]).astype(np.int64)
        f = np.clip(s / SPACING, 0.0, (cnt - 1) - 1e-9)
        i = np.floor(f).astype(np.int64)
        t = f - i
        x = m.x[off + i] * (1 - t) + m.x[off + i + 1] * t
        y = m.y[off + i] * (1 - t) + m.y[off + i + 1] * t
        hd = m.dir[off + i]
        idn = np.rint(f).astype(np.int64)
        return x, y, hd, idn

    def hdr(self, c):
        m = self.m
        h = np.zeros(self.n, dtype=abi.scene_hdr)
        ticks = self.period_ticks(c)
        h["period_ms"] = ticks.astype(np.float64) / 1000.0 * 1000.0      # == what the reference computes
        t = self.elapsed_s(c)
        s = self.s0 + self.v / 3.6 * t
        if self.kind == "highway":
            s = np.minimum(s, 985.0)        # keep id + ID_MORE inside the lane (no OOB map reads, Decision.cpp:590-594)
        h["velocity"] = self.v
        h["n_obs"] = self.n_obs
        h["conn"] = -1
        h["last_roadnum"] = 1; h["next_roadnum"] = 1; h["last_lanenum"] = 1; h["next_lanenum"] = 1
        wob = self.wob_a * np.sin(self.wob_w * c)
        yaw = (rnd(self.seeds, S_YAW, c) - 0.5) * 4.0
        if self.kind == "highway":
            # scripted lane change: lateral blend over 8 cycles centred on chg_t
            prog = np.clip((c - self.chg_t + 4) / 8.0, 0.0, 1.0) * (self.chg_dir != 0)
            lane = np.where(prog >= 0.5, self.lane0 + self.chg_dir, self.lane0)
            lat_from_lane0 = -prog * self.chg_dir * LANE_W      # metres to the LEFT (+) of lane0 centre
            lat_left = np.where(prog >= 0.5, lat_from_lane0 + self.chg_dir * LANE_W, lat_from_lane0) + wob
            gl = m.road_lane_base[self.road - 1].astype(np.int64) + lane - 1
            x, y, hd, idn = self._lane_xy(gl, s)
            hr = np.radians(hd)
            h["x"] = x - lat_left * np.sin(hr)
            h["y"] = y + lat_left * np.cos(hr)
            h["dir"] = np.mod(hd + yaw + 360.0, 360.0)
            h["road_num"] = self.road
            h["lane_num"] = lane
            h["pos"] = 0
            h["path_num"] = 0
            for l in range(abi.LANESUM):
                h["id"][:, l] = np.where(l < self.nl, idn, 0)
            out = np.zeros((self.n, abi.LANESUM), np.uint16)
            allm = self.nav_lane == 0
            for l in range(abi.LANESUM):
                out[:, l] = np.where(allm & (l < self.nl), l + 1, 0)
            out[:, 0] = np.where(allm, out[:, 0], self.nav_lane)
            h["out_lane_no"] = out
            h["stub_attribute"] = 0
        else:
            lane = self.lane0
            app_len = 399 * SPACING
            gl6 = m.road_lane_base[5].astype(np.int64) + lane - 1
            gl7 = m.road_lane_base[6].astype(np.int64) + lane - 1
            cidx = lane - 1                                         # connector index == lane-1
            gc = m.conn["lane"][cidx].astype(np.int64)
            clen = (m.lane_pt_off[gc + 1] - m.lane_pt_off[gc] - 1) * SPACING
            in_app = s < app_len
            in_con = (~in_app) & (s < app_len + clen)
            in_dep = ~(in_app | in_con)
            xa, ya, ha, ia = self._lane_xy(gl6, np.minimum(s, app_len))
            xc, yc, hc, ic = self._lane_xy(gc, np.clip(s - app_len, 0.0, clen))
            xd, yd, hdd, idd = self._lane_xy(gl7, np.maximum(s - app_len - clen, 0.0))
            x = np.where(in_app, xa, np.where(in_con, xc, xd))
            y = np.where(in_app, ya, np.where(in_con, yc, yd))
            hd = np.where(in_app, ha, np.where(in_con, hc, hdd))
            hr = np.radians(hd)
            h["x"] = x - wob * np.sin(hr)
            h["y"] = y + wob * np.cos(hr)
            h["dir"] = np.mod(hd + yaw + 360.0, 360.0)
            pre = in_app & ((s > app_len - 30.0) | (self.kind == "urban"))   # pre-junction zone: last 30 m (urban: the whole approach)
            h["pos"] = np.where(in_con, 2, np.where(pre, 1, 0))
            h["road_num"] = np.where(in_app, 6, 7)                 # in the junction: NEXT road (Decision.cpp:417)
            h["lane_num"] = lane
            h["path_num"] = np.where(in_dep, 1, 0)
            h["last_roadnum"] = 6; h["next_roadnum"] = 7
            h["last_lanenum"] = lane; h["next_lanenum"] = lane
            h["conn"] = cidx
            idv = np.where(in_app, ia, np.where(in_con, ic, idd))
            for l in range(abi.LANESUM):
                h["id"][:, l] = np.where(l < 2, idv, 0)
            out = np.zeros((self.n, abi.LANESUM), np.uint16)
            out[:, 0] = 1; out[:, 1] = 2
            h["out_lane_no"] = out
            h["stub_attribute"] = np.where(in_dep, 0, 1 + (self.seeds % np.uint64(3)).astype(np.int64))
        return h

    def obstacles(self, c):
        """(obs_x, obs_y) of cycle c, each [n, n_obs] C-contiguous."""
        m = self.m
        t = self.elapsed_s(c)[:, None]
        s = self.ob_s0 + self.ob_v * t
        if self.kind == "highway":
            gl = m.road_lane_base[self.road - 1].astype(np.int64)[:, None] + self.ob_lane - 1
            x, y, hd, _ = self._lane_xy(gl, s)
        else:
            # agents spread over approach lanes, connector and departure lanes by arclength
            app_len = 399 * SPACING
            gl6 = m.road_lane_base[5].astype(np.int64) + self.ob_lane - 1
            gl7 = m.road_lane_base[6].astype(np.int64) + self.ob_lane - 1
            gc = m.conn["lane"][self.ob_lane - 1].astype(np.int64)
            clen = (m.lane_pt_off[gc + 1] - m.lane_pt_off[gc] - 1) * SPACING
            in_app = s < app_len
            in_con = (~in_app) & (s < app_len + clen)
            xa, ya, ha, _ = self._lane_xy(gl6, np.clip(s, 0.0, app_len))
            xc, yc, hc, _ = self._lane_xy(gc, np.clip(s - app_len, 0.0, clen))
            xd, yd, hdd, _ = self._lane_xy(gl7, np.maximum(s - app_len - clen, 0.0))
            x = np.where(in_app, xa, np.where(in_con, xc, xd))
            y = np.where(in_app, ya, np.where(in_con, yc, yd))
            hd = np.where(in_app, ha, np.where(in_con, hc, hdd))
        hr = np.radians(hd)
        ox = x - self.ob_lat * np.sin(hr)
        oy = y + self.ob_lat * np.cos(hr)
        return np.ascontiguousarray(ox), np.ascontiguousarray(oy)

    def all_cycles(self):
        """[cycles][n] hdr and [cycles][n][n_obs] obstacle arrays (cycle-major)."""
        H = np.zeros((self.cycles, self.n), dtype=abi.scene_hdr)
        OX = np.zeros((self.cycles, self.n, self.n_obs))
        OY = np.zeros((self.cycles, self.n, self.n_obs))
        for c in range(self.cycles):
            H[c] = self.hdr(c)
            OX[c], OY[c] = self.obstacles(c)
        return H, OX, OY

    def tracks(self, c):
        """constant-turn-rate prediction of every agent at cycle c: per-step displacement (vx, vy) [m per 0.02 s step] along the
        heading of the lane it is on, and a small constant heading change per step [deg]; each [n, n_obs]."""
        m = self.m
        t = self.elapsed_s(c)[:, None]
        s = self.ob_s0 + self.ob_v * t
        app_len = 399 * SPACING
        gl6 = m.road_lane_base[5].astype(np.int64) + self.ob_lane - 1
        gl7 = m.road_lane_base[6].astype(np.int64) + self.ob_lane - 1
        gc = m.conn["lane"][self.ob_lane - 1].astype(np.int64)
        clen = (m.lane_pt_off[gc + 1] - m.lane_pt_off[gc] - 1) * SPACING
        in_app = s < app_len
        in_con = (~in_app) & (s < app_len + clen)
        _, _, ha, _ = self._lane_xy(gl6, np.clip(s, 0.0, app_len))
        _, _, hc, _ = self._lane_xy(gc, np.clip(s - app_len, 0.0, clen))
        _, _, hdd, _ = self._lane_xy(gl7, np.maximum(s - app_len - clen, 0.0))
        hr = np.radians(np.where(in_app, ha, np.where(in_con, hc, hdd)))
        step = self.ob_v * self.TRACK_DT
        k = np.arange(self.n_obs, dtype=np.uint64)[None, :]
        dth = (rnd(self.seeds[:, None], S_YAW, k + np.uint64(7000)) - 0.5) * 0.1
        return np.ascontiguousarray(step * np.cos(hr)), np.ascontiguousarray(step * np.sin(hr)), np.ascontiguousarray(dth)

    def all_cycles_tracks(self):
        """all_cycles() plus the track parameters VX, VY, DTH, each [cycles][n][n_obs]"""
        H, OX, OY = self.all_cycles()
        VX = np.zeros_like(OX); VY = np.zeros_like(OX); DTH = np.zeros_like(OX)
        for c in range(self.cycles):
            VX[c], VY[c], DTH[c] = self.tracks(c)
        return H, OX, OY, VX, VY, DTH


class World:
    """Initial worlds for the closed-loop episode runner (include/dmpp_b200.h section 9): the scene drawn by
    `Episodes(kind=kind)` at cycle 0 -- ego pose, speed, navigation slice -- plus one `dp_agent` per obstacle (lane, map
    index, offset into the segment, speed, lateral offset).  From there on nothing is scripted: the library advances ego,
    agents and localisation itself.  The cycle period is a whole number of milliseconds per scene, fixed over the episode.
    kind 'junction' / 'urban': the agents sit on the approach lane, the connector or the departure lane by arclength, as
    `Episodes.obstacles` spreads them; the ego crosses the junction only with dp_world_params.pre_junction_pts > 0
    (`PRE_JUNCTION_PTS[kind]` matches the scripted episodes).  `v0`: the agents' desired speeds for the reactive agents of
    include/dmpp_b200.h section 12, by default their initial speeds.  `max_obs` (default n_obs): the width of `agents` / `v0`,
    zero-padded beyond the n_obs agents (hdr.n_obs stays n_obs), for contexts with room for more obstacle points than agents --
    the V2X road users of include/dmpp_b200.h section 16 are appended in those slots."""
    PRE_JUNCTION_PTS = {"highway": 0, "junction": 60, "urban": 400}

    def __init__(self, m: Map, seeds, n_obs=10, roads=None, kind="highway", max_obs=None):
        ep = Episodes(m, seeds, n_obs=n_obs, kind=kind, cycles=1, roads=roads)
        self.m, self.n, self.n_obs, self.kind = m, ep.n, int(n_obs), kind
        self.hdr = ep.hdr(0)
        self.hdr["period_ms"] = ep.period_ticks(0).astype(np.float64)
        a = np.zeros((self.n, self.n_obs), abi.agent)
        s = ep.ob_s0
        if kind == "highway":
            gl = m.road_lane_base[ep.road - 1].astype(np.int64)[:, None] + ep.ob_lane - 1
        else:
            app_len = 399 * SPACING
            gl6 = m.road_lane_base[5].astype(np.int64) + ep.ob_lane - 1
            gl7 = m.road_lane_base[6].astype(np.int64) + ep.ob_lane - 1
            gc = m.conn["lane"][ep.ob_lane - 1].astype(np.int64)
            clen = (m.lane_pt_off[gc + 1] - m.lane_pt_off[gc] - 1) * SPACING
            in_app = s < app_len
            in_con = (~in_app) & (s < app_len + clen)
            gl = np.where(in_app, gl6, np.where(in_con, gc, gl7))
            s = np.where(in_app, s, np.where(in_con, s - app_len, s - app_len - clen))
        cnt = (m.lane_pt_off[gl + 1] - m.lane_pt_off[gl]).astype(np.int64)
        f = np.clip(s / SPACING, 0.0, cnt - 2.0)
        i = np.floor(f).astype(np.int64)
        a["lane"] = gl
        a["i"] = i
        a["u"] = (f - i) * SPACING
        a["v"] = ep.ob_v
        a["lat"] = ep.ob_lat
        if max_obs is not None and int(max_obs) != self.n_obs:
            assert int(max_obs) > self.n_obs
            pad = np.zeros((self.n, int(max_obs)), abi.agent)
            pad[:, :self.n_obs] = a
            a = pad
        self.agents = np.ascontiguousarray(a)
        self.v0 = np.ascontiguousarray(a["v"])


def v2x_events(m: Map, hdr, seed=0, p_far=0.12):
    """Seeded V2X inputs for the scenes of `hdr` (highway headers): a pedestrian, a signal phase, a road-works event point and a
    list of warning points per scene, placed relative to the ego's lane so that every branch of the handlers
    (Decision.cpp:1824-2434) is reached: ahead of / behind the ego, left / right of / on its path, on the neighbour lanes,
    beyond 100 m.  Returns (v2x[n] as abi.v2x_data, wp_lat, wp_lng); positions go through the equirectangular datum of the
    default parameters."""
    n = hdr.shape[0]
    sd = np.arange(n, dtype=np.uint64) + np.uint64(seed) * np.uint64(1000003)
    lat0, lng0, k_lat, k_lng = 23.0, 113.0, 1.0 / 110574.0, 1.0 / 102470.0
    lane = hdr["lane_num"].astype(np.int64)
    gl = m.road_lane_base[hdr["road_num"].astype(np.int64) - 1].astype(np.int64) + lane - 1
    off = m.lane_pt_off[gl].astype(np.int64)
    cnt = (m.lane_pt_off[gl + 1] - m.lane_pt_off[gl]).astype(np.int64)
    eid = np.take_along_axis(hdr["id"].astype(np.int64), (lane - 1)[:, None], axis=1)[:, 0]

    def place(k, stream, lat_span):
        """a point `ahead` map points in front of the ego (sometimes behind / far), `d` metres to the LEFT of its lane"""
        ahead = (rnd(sd, stream, k) * 180.0).astype(np.int64) + 2
        far = rnd(sd, stream + 1, k) < p_far
        ahead = np.where(far, np.where(rnd(sd, stream + 2, k) < 0.5, -30, 260), ahead)
        i = np.clip(eid + ahead, 0, cnt - 2)
        d = (rnd(sd, stream + 3, k) - 0.45) * lat_span
        x0, y0 = m.x[off + i], m.y[off + i]
        hr = np.radians(m.dir[off + i])
        x, y = x0 - d * np.sin(hr), y0 + d * np.cos(hr)
        return lat0 + y * k_lat, lng0 + x * k_lng

    v = np.zeros(n, abi.v2x_data)
    v["warn_status"] = np.array([3, 4, 5, 4, 5, 0, 4, 5])[(rnd(sd, 200) * 8).astype(np.int64)]
    v["ped_lat"], v["ped_lng"] = place(0, 210, 14.0)
    v["ped_distance"] = -10.0 + rnd(sd, 201) * 125.0
    v["ped_direction"] = (rnd(sd, 202) < 0.3).astype(np.int32)
    v["spat_lane_occupied"] = (rnd(sd, 203) < 0.7).astype(np.int32)
    v["spat_state"] = np.array([3, 6, 7, 1, 0])[(rnd(sd, 204) * 5).astype(np.int64)]
    v["rsi_lat"], v["rsi_lng"] = place(1, 220, 9.0)
    none = rnd(sd, 205) < 0.1
    v["rsi_lat"] = np.where(none, 0.0, v["rsi_lat"])
    v["ego_lat"], v["ego_lng"] = lat0 + hdr["y"] * k_lat, lng0 + hdr["x"] * k_lng
    cntw = (rnd(sd, 206) * 6).astype(np.int64)
    v["wp_count"] = cntw
    v["wp_first"] = np.concatenate([[0], np.cumsum(cntw)[:-1]])
    cols = [place(10 + k, 230, 5.0) for k in range(6)]         # entry k of every scene's list; kept where k < its count
    la, lo = np.stack([c[0] for c in cols], axis=1), np.stack([c[1] for c in cols], axis=1)
    keep = np.arange(6)[None, :] < cntw[:, None]
    return v, np.ascontiguousarray(la[keep]), np.ascontiguousarray(lo[keep])


# streams of the V2X events of closed-loop worlds
(V_OFF, V_RANGE, V_KIND, V_PED_S, V_PED_D, V_PED_V, V_PED_T, V_PED_R, V_PED_DIR, V_RW_LANE, V_RW_S, V_RW_D, V_RW_RSI,
 V_RW_N) = range(300, 314)


class V2xEvents:
    """Seeded V2X events for the closed-loop worlds of `World` (include/dmpp_b200.h section 14), one dp_v2x_event_spec per world in
    map coordinates: `spec[n]`, and the warning points `wp_x` / `wp_y` the road-works zones index.  `seeds` are the worlds' seeds.
      junction / urban worlds: a signal at the end of the approach (road 6, stop index -1) with a seeded phase offset, cycle
          SIGNAL = (cycle, green, yellow, red) seconds, and a seeded range of 25-60 m, so that some worlds start beyond it;
      highway worlds: half of them a pedestrian who crosses the ego's road from its right at a seeded station 15-70 m ahead of the
          ego's start, from 4 m right to 1 m left of its lane at 0.8-2 m/s, active from a seeded instant in the first second, with
          a seeded range of 40-120 m; the other half a road-works zone 20-90 m ahead on a seeded lane of the ego's road, up to
          1.5 m off its centre line, an RSI point in 70 % of them and 0-3 warning points 5 m apart along that lane.
    Between them the seeded worlds reach every flag value of the handlers and every warn_status."""
    SIGNAL = (14.0, 6.0, 2.0, 6.0)

    def __init__(self, world, seeds, seed=0):
        m, h, n = world.m, world.hdr, world.n
        sd = np.asarray(seeds, np.uint64) + np.uint64(seed) * np.uint64(1000003)
        assert sd.shape == (n,)
        spec = np.zeros(n, abi.v2x_event_spec)
        self.wp_x, self.wp_y = np.zeros(0), np.zeros(0)
        if world.kind != "highway":
            cyc, g, y, r = self.SIGNAL
            spec["sig_road"], spec["sig_stop"] = 6, -1
            spec["sig_cycle"], spec["sig_green"], spec["sig_yellow"], spec["sig_red"] = cyc, g, y, r
            spec["sig_offset"] = rnd(sd, V_OFF) * cyc
            spec["sig_range"] = 25.0 + rnd(sd, V_RANGE) * 35.0
            self.spec = spec
            return
        road, lane = h["road_num"].astype(np.int64), h["lane_num"].astype(np.int64)
        base = m.road_lane_base[road - 1].astype(np.int64)
        nl = (m.road_lane_base[road] - m.road_lane_base[road - 1]).astype(np.int64)
        eid = np.take_along_axis(h["id"].astype(np.int64), (lane - 1)[:, None], axis=1)[:, 0]

        def point(gl, ahead_m, left_m):
            off, cnt = m.lane_pt_off[gl].astype(np.int64), (m.lane_pt_off[gl + 1] - m.lane_pt_off[gl]).astype(np.int64)
            i = np.clip(eid + np.rint(ahead_m / SPACING).astype(np.int64), 0, cnt - 2)
            hr = np.radians(m.dir[off + i])
            nx, ny = -np.sin(hr), np.cos(hr)                # left normal of the lane
            return m.x[off + i] + left_m * nx, m.y[off + i] + left_m * ny, nx, ny

        ped = rnd(sd, V_KIND) < 0.5
        x, y, nx, ny = point(base + lane - 1, 15.0 + rnd(sd, V_PED_S) * 55.0, -4.0 + rnd(sd, V_PED_D) * 5.0)
        v = 0.8 + rnd(sd, V_PED_V) * 1.2
        spec["has_ped"] = ped
        spec["ped_x"], spec["ped_y"], spec["ped_vx"], spec["ped_vy"] = x, y, v * nx, v * ny
        spec["ped_t_on"] = rnd(sd, V_PED_T)
        spec["ped_t_off"] = spec["ped_t_on"] + 30.0
        spec["ped_range"] = 40.0 + rnd(sd, V_PED_R) * 80.0
        spec["ped_direction"] = rnd(sd, V_PED_DIR) < 0.3
        gw = base + (rnd(sd, V_RW_LANE) * nl).astype(np.int64)
        ahead = 20.0 + rnd(sd, V_RW_S) * 70.0
        rx, ry, _, _ = point(gw, ahead, -0.5 + rnd(sd, V_RW_D) * 2.0)
        works = ~ped
        spec["has_works"], spec["rw_rsi"] = works, works & (rnd(sd, V_RW_RSI) < 0.7)
        spec["rw_x"], spec["rw_y"], spec["rw_range"] = rx, ry, 150.0
        cnt = np.where(works, (rnd(sd, V_RW_N) * 4).astype(np.int64), 0)
        spec["wp_count"], spec["wp_first"] = cnt, np.concatenate([[0], np.cumsum(cnt)[:-1]])
        cols = [point(gw, ahead + 5.0 * k, 0.0)[:2] for k in range(3)]
        keep = np.arange(3)[None, :] < cnt[:, None]
        self.wp_x = np.ascontiguousarray(np.stack([c[0] for c in cols], axis=1)[keep])
        self.wp_y = np.ascontiguousarray(np.stack([c[1] for c in cols], axis=1)[keep])
        self.spec = spec


# streams of the directed families
(D_FAM, D_LANE, D_ID, D_GAP, D_LAT, D_SPEED, D_NAV, D_STALL, D_YAW, D_PERIOD, D_OTHER_S, D_OTHER_L, D_MOVE, D_WOB) = range(100, 114)


class Directed:
    """Scripted scene families that reach the RIGHT lane change of the rule tree (behaviour 3).  Same interface as
    `Episodes` (hdr(c), obstacles(c), all_cycles()); every quantity is a stateless hash of (seed, stream, index).

    family 'right_obstacle' -- Decision.cpp:1296-1424 (commit at :1382) and the right-lane aim walk with its loop-bound quirk
        (Planning.cpp:473-501): road 8, ego STANDING on a point whose attribute is exactly 2 (the run of odd attributes ahead
        is > 50 m), a standing vehicle 8-20 m ahead in its lane, right neighbour lane mostly clear; the signal timer passes
        1500 ms after ~16 cycles.  Lane 1 scenes take the no-way-back branch (light 2, 50 m), lane 2 scenes the other one
        (light 1, 10 m) and walk the right lane for the aim point.  At cycle `move_t` the ego appears on the target lane.
    family 'right_nav' -- Decision.cpp:1086-1143 (commit at :1108): the navigation asks for a right change on a lane whose
        attribute is 2.  The signal timer of that branch restarts every cycle unless light_status is already 2 (quirk 3), so
        the commit needs either (a) ONE cycle period >= 2000 ms (a stalled cycle: `stall` sub-family, roads 1 and 3, lane 1),
        or (b) light 2 carried over from an avoid-right manoeuvre on an attribute-0 stretch that ends (`carry` sub-family:
        road 4 lane 1 crossing id 700 behind a vehicle that sits left of the lane centre).
    """

    def __init__(self, m: Map, seeds, family="right_obstacle", n_obs=10, cycles=40):
        self.m, self.family, self.n_obs, self.cycles = m, family, int(n_obs), int(cycles)
        self.seeds = np.asarray(seeds, dtype=np.uint64)
        self.n = self.seeds.size
        sd = self.seeds
        n = self.n
        self.lat_wob = (rnd(sd, D_WOB) - 0.5) * 0.16
        if family == "right_obstacle":
            self.road = np.full(n, 8, np.int64)
            self.lane0 = 1 + (rnd(sd, D_LANE) * 2).astype(np.int64)             # lane 1 or 2
            self.id0 = 128 * (2 + (rnd(sd, D_ID) * 10).astype(np.int64))        # attribute 2 exactly here
            self.v = np.zeros(n)
            self.gap = 8.0 + rnd(sd, D_GAP) * 12.0
            self.lead_lat = (rnd(sd, D_LAT) - 0.5) * 1.0
            self.lead_v = np.zeros(n)
            self.move_t = 24 + (rnd(sd, D_MOVE) * 12).astype(np.int64)
            self.nav = np.zeros((n, abi.LANESUM), np.uint16)
            self.nav[:, :3] = [1, 2, 3]
            self.stall_t = np.full(n, -1, np.int64)
        elif family == "right_nav":
            sub = rnd(sd, D_FAM) < 0.5                                          # True: stall, False: carry
            self.sub_stall = sub
            self.road = np.where(sub, np.where(rnd(sd, D_LANE) < 0.5, 1, 3), 4).astype(np.int64)
            self.lane0 = np.ones(n, np.int64)
            self.v = 25.0 + rnd(sd, D_SPEED) * 15.0
            self.id0 = np.where(sub, 200 + (rnd(sd, D_ID) * 1200).astype(np.int64), 660 + (rnd(sd, D_ID) * 30).astype(np.int64))
            self.gap = np.where(sub, 30.0 + rnd(sd, D_GAP) * 40.0, 9.0 + rnd(sd, D_GAP) * 4.0)
            self.lead_lat = np.where(sub, (rnd(sd, D_LAT) - 0.5) * 0.6, 0.45 + rnd(sd, D_LAT) * 0.15)
            self.lead_v = self.v / 3.6
            self.move_t = np.full(n, 10 ** 6, np.int64)
            self.nav = np.zeros((n, abi.LANESUM), np.uint16)
            self.nav[:, 0] = 2 + (rnd(sd, D_NAV) * 2).astype(np.int64)          # exit lane 2 or 3: lane 1 must go right
            self.stall_t = np.where(sub, 4 + (rnd(sd, D_STALL) * (cycles - 8)).astype(np.int64), -1)
        else:
            raise ValueError(family)
        self.nl = (m.road_lane_base[self.road] - m.road_lane_base[self.road - 1]).astype(np.int64)
        k = np.arange(1, self.n_obs, dtype=np.uint64)[None, :]
        s2 = sd[:, None]
        # the other vehicles: far lanes / far behind, a few in the right neighbour lane (then the change may never commit)
        self.other_rel = -80.0 + rnd(s2, D_OTHER_S, k) * 200.0
        ol = rnd(s2, D_OTHER_L, k)
        self.other_lane = np.where(ol < 0.12, np.minimum(self.lane0[:, None] + 1, self.nl[:, None]), self.nl[:, None])
        self.other_lane = np.where(ol > 0.9, self.lane0[:, None], self.other_lane)
        self.other_rel = np.where(self.other_lane == self.lane0[:, None], -90.0 - rnd(s2, D_OTHER_S, k + np.uint64(500)) * 60.0, self.other_rel)
        self._t_cache = {}

    period_ticks_base = Episodes.period_ticks
    _lane_xy = Episodes._lane_xy

    def period_ticks(self, c):
        t = 80 + (rnd(self.seeds, D_PERIOD, c) * 41.0).astype(np.int64)
        return np.where(self.stall_t == c, 2000 + (rnd(self.seeds, D_STALL, 7) * 1000.0).astype(np.int64), t)

    def elapsed_s(self, c):
        if c not in self._t_cache:
            t = np.zeros(self.n)
            for i in range(c):
                t = t + self.period_ticks(i) / 1000.0
            self._t_cache[c] = t
        return self._t_cache[c]

    def hdr(self, c):
        m = self.m
        h = np.zeros(self.n, dtype=abi.scene_hdr)
        h["period_ms"] = self.period_ticks(c).astype(np.float64) / 1000.0 * 1000.0        # == what the reference computes
        t = self.elapsed_s(c)
        s = self.id0 * SPACING + self.v / 3.6 * t
        lane = np.where(c >= self.move_t, np.minimum(self.lane0 + 1, self.nl), self.lane0)
        gl = m.road_lane_base[self.road - 1].astype(np.int64) + lane - 1
        x, y, hd, idn = self._lane_xy(gl, s)
        hr = np.radians(hd)
        lat = self.lat_wob * np.sin(0.4 * c)
        h["x"] = x - lat * np.sin(hr)
        h["y"] = y + lat * np.cos(hr)
        h["dir"] = np.mod(hd + (rnd(self.seeds, D_YAW, c) - 0.5) * 3.0 + 360.0, 360.0)
        h["velocity"] = self.v
        h["n_obs"] = self.n_obs
        h["conn"] = -1
        h["road_num"] = self.road
        h["lane_num"] = lane
        h["last_roadnum"] = 1; h["next_roadnum"] = 1; h["last_lanenum"] = 1; h["next_lanenum"] = 1
        for l in range(abi.LANESUM):
            h["id"][:, l] = np.where(l < self.nl, idn, 0)
        h["out_lane_no"] = self.nav
        return h

    def obstacles(self, c):
        m = self.m
        t = self.elapsed_s(c)
        S = np.zeros((self.n, self.n_obs)); L = np.zeros((self.n, self.n_obs), np.int64); LAT = np.zeros((self.n, self.n_obs))
        S[:, 0] = self.id0 * SPACING + self.gap + self.lead_v * t
        L[:, 0] = self.lane0
        LAT[:, 0] = self.lead_lat
        if self.n_obs > 1:
            S[:, 1:] = (self.id0 * SPACING + self.v / 3.6 * t)[:, None] + self.other_rel
            L[:, 1:] = self.other_lane
        gl = m.road_lane_base[self.road - 1].astype(np.int64)[:, None] + L - 1
        x, y, hd, _ = self._lane_xy(gl, S)
        hr = np.radians(hd)
        return np.ascontiguousarray(x - LAT * np.sin(hr)), np.ascontiguousarray(y + LAT * np.cos(hr))

    def all_cycles(self):
        H = np.zeros((self.cycles, self.n), dtype=abi.scene_hdr)
        OX = np.zeros((self.cycles, self.n, self.n_obs))
        OY = np.zeros((self.cycles, self.n, self.n_obs))
        for c in range(self.cycles):
            H[c] = self.hdr(c)
            OX[c], OY[c] = self.obstacles(c)
        return H, OX, OY
