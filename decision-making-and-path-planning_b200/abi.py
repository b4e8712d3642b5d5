"""numpy / ctypes mirrors of the C ABI structs in include/dmpp_b200.h (and oracle/ref_api.h).

Every dtype here is checked against sizeof() reported by the loaded libraries in tests/test_abi.py.
"""
import ctypes as C

import numpy as np

LANESUM = 6
PATH_POINTS = 200
OUT_POINTS = 100
MAX_SWEEP = 8
NOT_FOUND = 999.0

scene_hdr = np.dtype(
    [
        ("x", "<f8"), ("y", "<f8"), ("dir", "<f8"), ("velocity", "<f8"), ("period_ms", "<f8"),
        ("id", "<i4", (LANESUM,)),
        ("road_num", "<u2"), ("lane_num", "<u2"), ("pos", "<u2"), ("path_num", "<u2"),
        ("last_roadnum", "<u2"), ("next_roadnum", "<u2"), ("last_lanenum", "<u2"), ("next_lanenum", "<u2"),
        ("out_lane_no", "<u2", (LANESUM,)),
        ("stub_attribute", "<u2"), ("n_obs", "<u2"),
        ("conn", "<i4"),
        ("pad", "u1", (28,)),
    ],
    align=False,
)
assert scene_hdr.itemsize == 128

plan_record = np.dtype(
    [
        ("velocity_expect", "<f8"), ("path_lat_dis", "<f8"), ("path_dir_err", "<f8"), ("remain_dis", "<f8"),
        ("mindist_lat", "<f8"), ("mindist_lon", "<f8"), ("brakespeed", "<f8"), ("des_acc", "<f8"),
        ("radius", "<f8"), ("aim_x", "<f8"), ("aim_y", "<f8"), ("aim_dir", "<f8"),
        ("aim_id", "<i4"),
        ("behavior", "<u2"), ("target_roadnum", "<u2"), ("target_lanenum", "<u2"), ("light", "<u2"),
        ("behavior_to_dlg", "<u2"), ("afresh_cause", "<u2"),
        ("sweep_index", "<i2"), ("path_near_id", "<i2"), ("path_front_near_id", "<i2"), ("ob_index", "<i2"),
        ("ob_pathid", "<u2"), ("n_traj", "<u2"),
        ("afresh_planning", "u1"), ("ob_flag", "u1"), ("acc_flag", "u1"), ("cnt", "u1"),
    ]
)
assert plan_record.itemsize == 128

search_slot = np.dtype(
    [("dis_lat", "<f8"), ("dis_lng", "<f8"), ("ob_index", "<i2"), ("pathid", "<u2"),
     ("evaluated", "u1"), ("found", "u1"), ("pad", "u1", (2,))]
)
assert search_slot.itemsize == 24

trace_record = np.dtype(
    [
        ("region", search_slot, (6,)), ("sweep", search_slot, (2 * MAX_SWEEP,)),
        ("junction", search_slot), ("local", search_slot),
        ("width_curlane", "<f8"), ("faraim_dis", "<f8"),
        ("navi_lanechg", "<u4"), ("navi_lanechg_times", "<u4"),
        ("refpath_len", "<u2"), ("ub_hits", "<u2"), ("pts_scored", "<u4"),
    ]
)
assert trace_record.itemsize == 608

carry = np.dtype(
    [
        ("leftlight_time", "<f8"), ("rightlight_time", "<f8"), ("velocity_expect", "<f8"),
        ("aim_x", "<f8"), ("aim_y", "<f8"), ("aim_dir", "<f8"),
        ("aim_id", "<i4"), ("obsavoid_time", "<u4"), ("no_obsavoid_time", "<u4"), ("frontobs_time", "<u4"),
        ("plan_his_behavior", "<i4"), ("path_near_id", "<i4"),
        ("behavior", "<u2"), ("target_roadnum", "<u2"), ("target_lanenum", "<u2"), ("light_status", "<u2"),
        ("behavior_to_dlg", "<u2"), ("his_behavior", "<u2"), ("his_target_lanenum", "<u2"),
        ("his_light_status", "<u2"),
        ("lanechg_status", "u1"), ("obsavoid_status", "u1"), ("plan_count", "u1"), ("pad0", "u1"),
        ("pad", "u1", (36,)),
    ]
)
assert carry.itemsize == 128

ref_call = np.dtype(
    [("lat_min", "<f8"), ("lat_max", "<f8"), ("dis_lat", "<f8"), ("dis_lng", "<f8"), ("n_path", "<i4"),
     ("ob_index", "<i2"), ("pathid", "<u2"), ("found", "u1"), ("pad", "u1", (7,))]
)
assert ref_call.itemsize == 48

ctrl_frame = np.dtype(
    [("cnt", "u1"), ("apa", "u1"), ("desacc_vd", "u1"), ("desstr_vd", "u1"), ("road_type", "u1"), ("sstop", "u1"), ("light", "<u2"),
     ("brakedis", "<f8"), ("brake_speed", "<f8"), ("desacc", "<f8"), ("desspd", "<f8"), ("desstr", "<f8"), ("radius", "<f8"),
     ("pnts", "<f8", (OUT_POINTS, 2))]
)
assert ctrl_frame.itemsize == 1656

status_frame = np.dtype(
    [("afresh_cause", "<i4"), ("trafficlight", "<u2"), ("reserved", "<u2"), ("near_ob_dist", "<f8"), ("planspeed", "<f8"),
     ("planacc", "<f8"), ("path_points", "<f8", (OUT_POINTS, 2))]
)
assert status_frame.itemsize == 1632

agent = np.dtype([("u", "<f8"), ("v", "<f8"), ("lat", "<f8"), ("lane", "<i4"), ("i", "<i4")])
assert agent.itemsize == 32

v2x_data = np.dtype(
    [("ped_distance", "<f8"), ("ped_lat", "<f8"), ("ped_lng", "<f8"), ("rsi_lat", "<f8"), ("rsi_lng", "<f8"), ("ego_lat", "<f8"),
     ("ego_lng", "<f8"), ("ped_direction", "<i4"), ("spat_lane_occupied", "<i4"), ("spat_state", "<i4"), ("warn_status", "<i4"),
     ("wp_first", "<i4"), ("wp_count", "<i4")]
)
assert v2x_data.itemsize == 80

v2x_flags = np.dtype(
    [("light_flag", "<u2"), ("construction_flag", "u1"), ("pedestrian_flag", "u1"), ("ub", "u1"), ("pad", "u1", (3,)),
     ("lng_distance", "<f8"), ("lat_distance", "<f8")]
)
assert v2x_flags.itemsize == 24

connector = np.dtype(
    [("last_road", "<u2"), ("next_road", "<u2"), ("last_lane", "<u2"), ("next_lane", "<u2"), ("lane", "<i4")]
)
assert connector.itemsize == 12


class Params(C.Structure):
    _fields_ = [
        ("vehicle_width", C.c_double), ("epsilon", C.c_double), ("pi", C.c_double),
        ("road_faraim_max", C.c_double), ("road_faraim_min", C.c_double),
        ("pre_inter_faraim", C.c_double), ("inter_faraim", C.c_double),
        ("road_remain_distance", C.c_double), ("inter_remain_distance", C.c_double),
        ("lat0", C.c_double), ("lng0", C.c_double), ("k_lat", C.c_double), ("k_lng", C.c_double),
        ("id_more", C.c_int32), ("reserved", C.c_int32),
    ]


class WorldParams(C.Structure):
    _fields_ = [("a_max", C.c_double), ("loc_back", C.c_int32), ("loc_fwd", C.c_int32), ("end_margin", C.c_int32),
                ("pre_junction_pts", C.c_int32)]


episode_metrics = np.dtype(
    [
        ("distance", "<f8"), ("min_clearance", "<f8"), ("min_lead_gap", "<f8"), ("min_ttc", "<f8"),
        ("max_accel", "<f8"), ("min_accel", "<f8"), ("max_abs_jerk", "<f8"), ("last_accel", "<f8"),
        ("max_abs_lat_err", "<f8"), ("max_abs_dir_err", "<f8"),
        ("steps", "<i4"), ("first_collision_step", "<i4"), ("first_collision_agent", "<i4"),
        ("collision_steps", "<i4"), ("collision_steps_front", "<i4"), ("collision_steps_rear", "<i4"), ("ttc_warn_steps", "<i4"),
        ("stopped_steps", "<i4"), ("end_stop_steps", "<i4"), ("replans", "<i4"), ("aeb_steps", "<i4"),
        ("accel_steps", "<i4"), ("last_behavior", "<i4"), ("behavior_switches", "<i4"),
        ("behavior_steps", "<u4", (8,)), ("pad", "<u4", (6,)),
    ]
)
assert episode_metrics.itemsize == 192


class MetricsParams(C.Structure):
    _fields_ = [("front", C.c_double), ("rear", C.c_double), ("half_width", C.c_double), ("corridor_half", C.c_double),
                ("ttc_warn", C.c_double)]


class AgentModelParams(C.Structure):
    _fields_ = [("a_max", C.c_double), ("b", C.c_double), ("b_max", C.c_double), ("T", C.c_double), ("s0", C.c_double),
                ("length", C.c_double), ("ego_rear", C.c_double), ("look", C.c_double)]


class LaneChangeParams(C.Structure):
    _fields_ = [("politeness", C.c_double), ("a_thr", C.c_double), ("b_safe", C.c_double), ("ego_b_safe", C.c_double),
                ("ego_front", C.c_double), ("lat_speed", C.c_double), ("cooldown", C.c_double), ("end_guard", C.c_double)]


lane_change_state = np.dtype([("lat_goal", "<f8"), ("hold", "<f8"), ("changes_left", "<i4"), ("changes_right", "<i4")])
assert lane_change_state.itemsize == 24


v2x_event_spec = np.dtype(
    [
        ("sig_cycle", "<f8"), ("sig_green", "<f8"), ("sig_yellow", "<f8"), ("sig_red", "<f8"), ("sig_offset", "<f8"), ("sig_range", "<f8"),
        ("ped_x", "<f8"), ("ped_y", "<f8"), ("ped_vx", "<f8"), ("ped_vy", "<f8"), ("ped_t_on", "<f8"), ("ped_t_off", "<f8"),
        ("ped_range", "<f8"), ("rw_x", "<f8"), ("rw_y", "<f8"), ("rw_range", "<f8"),
        ("sig_road", "<i4"), ("sig_stop", "<i4"), ("has_ped", "<i4"), ("ped_direction", "<i4"), ("has_works", "<i4"), ("rw_rsi", "<i4"),
        ("wp_first", "<i4"), ("wp_count", "<i4"),
    ]
)
assert v2x_event_spec.itemsize == 160

v2x_episode_stats = np.dtype(
    [
        ("min_ped_distance", "<f8"), ("last_d", "<f8"), ("cycles", "<i4"), ("light_cycles", "<i4", (3,)),
        ("construction_cycles", "<i4", (2,)), ("pedestrian_cycles", "<i4", (2,)), ("stop_cmds", "<i4"), ("creep_cmds", "<i4"),
        ("ub_cycles", "<i4"), ("red_crossings", "<i4"), ("first_red_crossing", "<i4"), ("last_phase", "<i4"), ("last_on", "<i4"),
        ("pad", "<i4"),
    ]
)
assert v2x_episode_stats.itemsize == 80


class V2xWorldParams(C.Structure):
    _fields_ = [("mode", C.c_int32), ("apply", C.c_int32)]


class MapDesc(C.Structure):
    _fields_ = [
        ("n_roads", C.c_int32), ("road_lane_base", C.c_void_p),
        ("n_lanes", C.c_int32), ("lane_pt_off", C.c_void_p),
        ("n_conn", C.c_int32), ("conn", C.c_void_p),
        ("n_points", C.c_int64),
        ("x", C.c_void_p), ("y", C.c_void_p), ("dir", C.c_void_p),
        ("lane_width", C.c_void_p), ("lanechg_attr", C.c_void_p),
    ]


def ptr(a):
    """void* of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"], "array must be C-contiguous"
    return C.c_void_p(a.ctypes.data)
