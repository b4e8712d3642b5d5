"""Maps and planner parameters other than the built-in ones, for the parity suites of tests/test_map_variants.py.

The built-in map (scenes.Map) is regular in ways the reference does not require: every lane is 375 cm wide, roads have 2 or 3
lanes, points are ~0.5 m apart without duplicates, curves are gentle and the coordinates lie near the origin.  The cycle kernels
have logic that depends on exactly these things (the avoid-sweep size K = #{i : i < (W - Vw) / 0.6}, the map-derived pruning
bounds lane_hmax / lane_hmin / lane_dnmax, the prefix tables cump / lane_cerr / run_end), so each variant here moves one of them:

  widths   the built-in map with per-lane and per-point lane widths covering every K from 0 to 8: the boundary widths
           Vw + 0.6 k, 1 cm either side of them, and 660 cm (K = 8, the widest lane dp_map_upload accepts at Vw = 1.8 m)
  jitter   points moved along the tangent by up to +-0.22 m (segments of 0.06-0.94 m, up to 1.43 m after a duplicate), small
           lateral noise, and about one duplicated point per 150 (lane_hmin = 0: the pruning bound switches off)
  utm      the whole map moved to UTM-like coordinates (x ~ 6e5, y ~ 2.5e6, non-dyadic offsets)
  scaled   the whole map scaled x2 (1 m spacing)
  shapes   roads 1-5 rebuilt: a 6-lane straight road (attributes {2,3,3,3,3,1}), a 1-lane road, a 3-lane circle (lane radii
           12.25-19.75 m: every lane passes the same place ~8 times), a 2-lane zig-zag (35 degree kinks every 40 points) and a
           2-lane hairpin (R = 6 m) between two straights; roads 6-8 and the junction connectors are the built-in ones
  params   the built-in map with non-default dp_params: vehicle width, ID_MORE, the far-aim distances, the remaining distances

Every variant is deterministic: the random ones draw from scenes.rnd (a stateless hash of seed, stream and index).  A variant's
`map` has the fields, desc() and helpers of scenes.Map, so scenes.Episodes, the oracle, the emulator and Planner.upload_map
take it unchanged; its `params` (None: the defaults) goes to Planner(params=...), the oracle and the emulator alike.
`walled` adds obstacles beside the in-lane blocker of highway episodes, so that the avoid sweep also picks on the right."""
import ctypes as C
import math

import numpy as np

from dmpp_b200 import abi, scenes

SEED = 20261021
VW = 1.8                                   # dp_params.vehicle_width default (Decision.cpp Vehicle_Width)
MAX_SWEEP = 8                              # DP_MAX_SWEEP


def sweep_k(width_m, vw=VW):
    """avoid candidates per side the oracle enumerates for lane width W (Decision.cpp:940), uncapped: the same double
    arithmetic as the kernels (Python floats are IEEE doubles)"""
    k = 0
    while k < 64 and k < (width_m - vw) / 0.6:
        k += 1
    return k


def boundary_widths(vw=VW):
    """lane widths in cm at every K boundary W = Vw + 0.6 k (k = 0..8) and 1 cm either side, within what the library accepts"""
    out = set()
    for k in range(MAX_SWEEP + 1):
        c = int(round(100 * (vw + 0.6 * k)))
        out.update(w for w in (c - 1, c, c + 1) if 100 <= w and sweep_k(w / 100.0, vw) <= MAX_SWEEP)
    return np.array(sorted(out), np.uint16)


class VariantMap(scenes.Map):
    """scenes.Map assembled from explicit lanes: roads[r-1] = [(x, y, dir, width_cm, attr), ...] (lane 1 first), connectors =
    [((last_road, next_road, last_lane, next_lane), (x, y, dir, width_cm, attr)), ...]"""

    def __init__(self, roads, connectors):
        lanes = [ln for road in roads for ln in road] + [ln for _, ln in connectors]
        self.road_lane_base = np.concatenate([[0], np.cumsum([len(r) for r in roads])]).astype(np.int32)
        self.lane_pt_off = np.concatenate([[0], np.cumsum([ln[0].size for ln in lanes])]).astype(np.int32)
        self.lane_road = [r + 1 for r, road in enumerate(roads) for _ in road]
        self.n_road_lanes = int(self.road_lane_base[-1])
        cat = lambda k, t: np.ascontiguousarray(np.concatenate([np.asarray(ln[k]) for ln in lanes]), t)   # noqa: E731
        self.x, self.y, self.dir = cat(0, np.float64), cat(1, np.float64), cat(2, np.float64)
        self.lane_width, self.lanechg_attr = cat(3, np.uint16), cat(4, np.uint16)
        self.conn = np.array([(*key, self.n_road_lanes + i) for i, (key, _) in enumerate(connectors)], dtype=abi.connector)
        self.n_roads = len(roads)
        self.n_lanes = len(lanes)


def lanes_of(m):
    """(roads, connectors) of a map in VariantMap's layout, arrays copied"""
    def lane(g):
        a, b = m.lane_pt_off[g], m.lane_pt_off[g + 1]
        return [m.x[a:b].copy(), m.y[a:b].copy(), m.dir[a:b].copy(), m.lane_width[a:b].copy(), m.lanechg_attr[a:b].copy()]
    roads = [[lane(g) for g in range(m.road_lane_base[r], m.road_lane_base[r + 1])] for r in range(m.n_roads)]
    conns = [(tuple(int(c[f]) for f in ("last_road", "next_road", "last_lane", "next_lane")), lane(int(c["lane"]))) for c in m.conn]
    return roads, conns


def road_from_centre(cx, cy, hd, attrs, width_cm=375):
    """lanes of a road around centre line (cx, cy, heading hd in degrees per point), lane 1 leftmost, as scenes.Map.add_road"""
    n = len(attrs)
    h = np.radians(hd)
    out = []
    for l in range(n):
        d_left = (0.5 * (n - 1) - l) * scenes.LANE_W
        x, y = cx - d_left * np.sin(h), cy + d_left * np.cos(h)
        out.append([x, y, np.mod(hd, 360.0), np.full(x.size, width_cm, np.uint16),
                    np.broadcast_to(np.asarray(attrs[l], np.uint16), x.shape).copy()])
    return out


def polyline(x0, y0, seg_hd):
    """centre line from segment headings (degrees, one per segment): points 0.5 m apart; a point's heading is that of the
    segment leaving it (the last point keeps the last segment's)"""
    h = np.radians(seg_hd)
    x = x0 + np.concatenate([[0.0], np.cumsum(scenes.SPACING * np.cos(h))])
    y = y0 + np.concatenate([[0.0], np.cumsum(scenes.SPACING * np.sin(h))])
    return x, y, np.concatenate([seg_hd, seg_hd[-1:]])


# ---- the variants -------------------------------------------------------------------------------------------------------------

def widths_map(base):
    roads, conns = lanes_of(base)
    bw = boundary_widths()
    k = 0
    for r, road in enumerate(roads):
        for l, ln in enumerate(road):
            n = ln[0].size
            u = scenes.rnd(SEED, 1, np.arange(n // 80 + 1) + 1000 * (10 * r + l))
            if r in (1, 3):
                # roads 2 and 4 run the in-lane avoid sweep (attribute 0): 40 m blocks cycling through every boundary width
                blocks = bw[(np.arange(n // 80 + 1) + 7 * (10 * r + l)) % bw.size]
            else:
                # elsewhere per-lane widths, a third of the lanes with per-point blocks of any width 150-660 cm
                blocks = np.full(n // 80 + 1, bw[(k * 5) % bw.size])
                if l % 3 == 1:
                    blocks = (150 + u * 511).astype(np.uint16)
                k += 1
            ln[3] = np.repeat(blocks, 80)[:n].astype(np.uint16)
    for i, (_, ln) in enumerate(conns):
        ln[3] = np.full(ln[0].size, bw[(3 * i + 4) % bw.size], np.uint16)
    return VariantMap(roads, conns)


def jitter_map(base):
    roads, conns = lanes_of(base)
    g = 0
    for ln in [ln for road in roads for ln in road] + [ln for _, ln in conns]:
        n = ln[0].size
        i = np.arange(n)
        h = np.radians(ln[2])
        t = (scenes.rnd(SEED, 2, i + 10_000 * g) - 0.5) * 0.44            # along the tangent, +-0.22 m
        d = (scenes.rnd(SEED, 3, i + 10_000 * g) - 0.5) * 0.04            # across it, +-2 cm
        ln[0] = ln[0] + t * np.cos(h) - d * np.sin(h)
        ln[1] = ln[1] + t * np.sin(h) + d * np.cos(h)
        dup = np.nonzero(scenes.rnd(SEED, 4, i[:-1] + 10_000 * g) < 1.0 / 150)[0]
        ln[0][dup + 1] = ln[0][dup]; ln[1][dup + 1] = ln[1][dup]            # point i+1 repeats point i: a zero-length segment
        g += 1
    return VariantMap(roads, conns)


def affine_map(base, scale=1.0, dx=0.0, dy=0.0):
    roads, conns = lanes_of(base)
    for ln in [ln for road in roads for ln in road] + [ln for _, ln in conns]:
        ln[0] = ln[0] * scale + dx
        ln[1] = ln[1] * scale + dy
    return VariantMap(roads, conns)


def shapes_map(base):
    roads, conns = lanes_of(base)
    n = scenes.N_PTS
    s = np.arange(n) * scenes.SPACING
    # road 1: 6-lane straight, heading 15 deg
    r1 = road_from_centre(400.0 + s * math.cos(math.radians(15)), -2000.0 + s * math.sin(math.radians(15)), np.full(n, 15.0),
                          [2, 3, 3, 3, 3, 1])
    # road 2: 1-lane straight, heading 120 deg, in-lane avoid sweep
    r2 = road_from_centre(-3000.0 + s * math.cos(math.radians(120)), -1000.0 + s * math.sin(math.radians(120)), np.full(n, 120.0), [0])
    # road 3: 3-lane circle, centre-line radius 16 m (lanes 12.25 / 16 / 19.75 m), turning left: ~10 laps of the centre lane
    R = 16.0
    a = s / R
    r3 = road_from_centre(4000.0 + R * np.sin(a), 3000.0 - R * np.cos(a), np.degrees(a), [2, 3, 1])
    # road 4: 2-lane zig-zag, the heading alternating +-17.5 deg every 40 points (a 35 degree kink each time), attribute 0
    zz = np.where((np.arange(n - 1) // 40) % 2 == 0, 17.5, -17.5)
    x4, y4, h4 = polyline(-4000.0, 3000.0, zz)
    r4 = road_from_centre(x4, y4, h4, [0, 0])
    # road 5: 2-lane hairpin: 900 points east, a left half turn of R = 6 m (lanes 4.125 / 7.875 m), then west
    nt = int(round(math.pi * 6.0 / scenes.SPACING))
    hp = np.concatenate([np.zeros(900), 180.0 * (np.arange(nt) + 0.5) / nt, np.full(n - 1 - 900 - nt, 180.0)])
    x5, y5, h5 = polyline(5000.0, -4000.0, hp)
    r5 = road_from_centre(x5, y5, h5, [0, 0])
    return VariantMap([r1, r2, r3, r4, r5] + roads[5:], conns)


def default_params():
    """dp_params defaults (the oracle's copy, the same values as dp_default_params; needs no GPU)"""
    from oracle import binding
    p = abi.Params()
    binding.Oracle().lib.oracle_default_params(C.byref(p))
    return p


def params_with(**kw):
    p = default_params()
    for k, v in kw.items():
        setattr(p, k, v)
    return p


PARAM_SETS = {
    "vw050": dict(vehicle_width=0.5),
    "vw120": dict(vehicle_width=1.2),
    "vw220": dict(vehicle_width=2.2),
    "idmore5": dict(id_more=5),
    "idmore12": dict(id_more=12),
    "faraim": dict(road_faraim_max=42.0, road_faraim_min=9.5, pre_inter_faraim=27.0, inter_faraim=11.0),
    "remain": dict(road_remain_distance=9.0, inter_remain_distance=8.5),
}
MAP_VARIANTS = ["widths", "jitter", "utm", "scaled", "shapes"]
VARIANTS = MAP_VARIANTS + ["params_" + k for k in PARAM_SETS]


def walled(ep, n_wall=6, step=0.35):
    """all_cycles() of highway episodes plus `n_wall` obstacle slots beside the first obstacle (the near in-lane blocker of 45 %
    of the scenes), so that the avoid sweep picks on either side at every K and has several obstacles near the lane at once:
      - half the scenes keep the blocker where Episodes put it (|lat| <= 0.6 m) and build the wall towards the left: the left
        candidates are blocked as well, and the sweep picks on the right;
      - the other half move the blocker 0.6-0.9 m off the centre, to the left or to the right, and build the wall on that side:
        the candidate shifted 0.3 m the other way is clear (a pick at K = 2), the ones on the wall side are not.
    A scene uses 2..n_wall of the slots, 0.35 m apart; the others stand 40 m to the side, out of every search's reach, so the
    number of obstacles near the lane varies from scene to scene.  Obstacle 0 of every scene becomes the near in-lane blocker
    (as Episodes makes it in 45 % of the scenes: 6-22 m ahead, slower than the ego).  n_obs grows by n_wall."""
    m, sd = ep.m, ep.seeds
    ep.ob_lane[:, 0] = ep.lane0
    ep.ob_s0[:, 0] = ep.s0 + 6.0 + scenes.rnd(sd, scenes.S_OB_S, 1000) * 16.0
    ep.ob_v[:, 0] = ep.v / 3.6 * (0.5 + 0.5 * scenes.rnd(sd, scenes.S_OB_V, 1000))
    H, OX, OY = ep.all_cycles()
    t = np.stack([ep.elapsed_s(c) for c in range(ep.cycles)])                       # [cycles][n]
    s = ep.ob_s0[None, :, 0] + ep.ob_v[None, :, 0] * t
    gl = np.broadcast_to(m.road_lane_base[ep.road - 1].astype(np.int64) + ep.ob_lane[:, 0] - 1, s.shape)
    x, y, hd, _ = ep._lane_xy(gl, s)
    hr = np.radians(hd)
    moved = scenes.rnd(sd, 900) < 0.5
    side = np.where(moved & (scenes.rnd(sd, 901) < 0.5), -1.0, 1.0)                 # +1: the wall grows to the left
    lat0 = np.where(moved, side * (0.6 + 0.3 * scenes.rnd(sd, 902)), ep.ob_lat[:, 0])  # metres to the left of the lane centre
    OX[:, :, 0] = np.where(moved, x - lat0 * np.sin(hr), OX[:, :, 0])
    OY[:, :, 0] = np.where(moved, y + lat0 * np.cos(hr), OY[:, :, 0])
    j = np.arange(1, n_wall + 1)
    used = 2 + (scenes.rnd(sd, 903) * (n_wall - 1)).astype(np.int64)                # 2 .. n_wall slots next to the blocker
    lat = np.where(j <= used[:, None], lat0[:, None] + side[:, None] * step * j, 40.0)[None]
    OX = np.ascontiguousarray(np.concatenate([OX, x[..., None] - lat * np.sin(hr)[..., None]], 2))
    OY = np.ascontiguousarray(np.concatenate([OY, y[..., None] + lat * np.cos(hr)[..., None]], 2))
    H["n_obs"] += n_wall
    return H, OX, OY


class Variant:
    """`sweep_roads`: the roads of the map whose lanes run the in-lane avoid sweep (lane-change attribute 0)"""

    def __init__(self, name, m, params=None, sweep_roads=(2, 4)):
        self.name, self.map, self.params, self.sweep_roads = name, m, params, list(sweep_roads)

    def __repr__(self):
        return "Variant(%s)" % self.name


_cache = {}


def variant(name):
    """the named variant, built once per process"""
    if name not in _cache:
        base = scenes.Map()
        if name.startswith("params_"):
            v = Variant(name, base, params_with(**PARAM_SETS[name[len("params_"):]]))
        else:
            m = {"widths": widths_map, "jitter": jitter_map, "shapes": shapes_map,
                 "utm": lambda b: affine_map(b, dx=600_000.37, dy=2_500_000.91),
                 "scaled": lambda b: affine_map(b, scale=2.0)}[name](base)
            v = Variant(name, m, sweep_roads=(2, 4, 5) if name == "shapes" else (2, 4))
        _cache[name] = v
    return _cache[name]
