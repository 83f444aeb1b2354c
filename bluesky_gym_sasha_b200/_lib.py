"""ctypes binding of libbsg_b200.so (include/bsg.h).  Loading fails loudly: there is no CPU fallback.

The structures mirror include/bsg.h field by field; tests/test_abi.py checks that every symbol the
header declares is exported and that the struct sizes agree with what the library reports.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BSG_B200_LIB", os.path.join(_HERE, "libbsg_b200.so"))    # override: A/B builds

BSG_OK, BSG_EINVAL, BSG_ECUDA, BSG_ESTATE, BSG_ENOMEM = 0, -1, -2, -3, -4
ENV_DESCENT, ENV_HORIZONTAL_CR, ENV_SECTOR_CR, ENV_MERGE, ENV_PLAN_WAYPOINT, ENV_VERTICAL_CR, ENV_STATIC_OBSTACLE = 0, 1, 2, 3, 4, 5, 6
AUTORESET_DISABLED, AUTORESET_NEXT_STEP, AUTORESET_SAME_STEP = 0, 1, 2
CD_LON_WRAP, CD_SYMMETRIC, CD_CULL, CD_ALLTILES = 1, 2, 4, 8
# CD record storage [tile][field][CD_TILE] (BSG_CD_TILE, BSG_CD_REC_*)
CD_TILE = 256
CD_REC_X, CD_REC_Y, CD_REC_CH, CD_REC_SH, CD_REC_U, CD_REC_V, CD_REC_ALT, CD_REC_VS, CD_REC_FIELDS = range(9)

# indices into the per-env records (include/bsg.h)
F64_WPT_LAT, F64_WPT_LON, F64_TARGET_ALT, F64_POLY_AREA, F64_WPTS, F64_COUNT = 0, 1, 2, 3, 4, 16
F32_TOTAL_REWARD, F32_DRIFT_SUM, F32_FINAL_ALT, F32_LAST_HDG, F32_LAST_WDIST, F32_LAST_DRIFT, F32_COUNT = 0, 1, 2, 3, 4, 5, 8
(I32_STEP, I32_EPISODE, I32_SIMK, I32_WPT_REACH, I32_DRIFT_N, I32_INTRUSIONS, I32_NUM_AC, I32_NVERT,
 I32_NEEDS_RESET, I32_FAF, I32_NCONF, I32_NLOS, I32_RESET_FLAGS, I32_NPAIRS) = range(14)
PAIR_CONF_IJ, PAIR_CONF_JI, PAIR_LOS, PAIR_ATTR_COUNT = 1 << 16, 1 << 17, 1 << 18, 6
I32_COUNT = 16
FL_ALIVE, FL_LNAV, FL_LASTWP, FL_WPSHIFT = 1, 2, 4, 8


class Perf(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("vminto", "vmaxic", "vminer", "vmaxer", "vminap", "vmaxap",
                                         "vsmin", "vsmax", "hmax", "mmo", "axmax_gd", "axmax_air")]


class Config(C.Structure):
    _fields_ = [("env_type", C.c_int32), ("num_envs", C.c_int32), ("n_intruders", C.c_int32),
                ("cd_enabled", C.c_int32), ("autoreset_mode", C.c_int32), ("max_episode_steps", C.c_int32),
                ("default_hdg_random", C.c_int32), ("device", C.c_int32), ("seed", C.c_uint64),
                ("env_id_offset", C.c_int64), ("rpz", C.c_float), ("hpz", C.c_float),
                ("dtlookahead", C.c_float), ("perf", Perf), ("wind_obs", C.c_int32),
                ("sector_density_uniform", C.c_int32), ("init_alt", C.c_float), ("cd_pair_cap", C.c_int32)]


class Wind(C.Structure):
    _fields_ = [("n_points", C.c_int32), ("n_alt", C.c_int32), ("alt_step", C.c_float),
                ("d_lat", C.c_void_p), ("d_lon", C.c_void_p), ("d_vn", C.c_void_p), ("d_ve", C.c_void_p),
                ("d_gs", C.c_void_p)]


class AcState(C.Structure):
    _fields_ = [("n", C.c_int32)] + [(k, C.c_void_p) for k in (
        "lat", "lon", "alt", "tas", "hdg", "vs", "selspd", "selalt", "selvs", "ap_trk", "cas", "ax", "curlegdir",
        "swlnav", "iactwp", "env_f64", "env_f32", "env_i32", "poly")]


class CdLists(C.Structure):
    _fields_ = [("d_conf_pairs", C.c_void_p), ("d_conf_attr", C.c_void_p), ("conf_cap", C.c_int64),
                ("d_los_pairs", C.c_void_p), ("los_cap", C.c_int64), ("d_npairs", C.c_void_p)]


CD_ATTR = ("qdr", "dist", "dcpa", "tcpa", "tinconf")          # BSG_CD_ATTR_* columns of d_conf_attr

# single-airspace traffic (bsg_traf_*): BSG_TF_* flag bits, BSG_TRAF_* sizes
(TF_ALIVE, TF_LNAV, TF_VNAV, TF_VNAVSPD, TF_LASTWP, TF_ASAS, TF_RESOOFF, TF_PH_GD, TF_PH_AP, TF_ACTIVATE) = (1 << b for b in range(10))
TF_IWP_SHIFT, TF_NWP_SHIFT, TRAF_PARTNERS, TRAF_CTR_COUNT = 16, 24, 8, 4
# conflict / LoS event tracking (bsg_traf_events_*): BSG_EV_CTR_* slots of the counter array
(EV_CTR_NCONF_TOTAL, EV_CTR_NLOS_TOTAL, EV_CTR_NCONF_ACTIVE, EV_CTR_NLOS_ACTIVE, EV_CTR_LOG_OVERFLOW, EV_CTR_TRUNCATED) = range(6)
EV_CTR_COUNT = 8
PRIM_LINE, PRIM_RING, PRIM_RECT, PRIM_EDGE, PRIM_EDGE_END, PRIM_FLOATS = 1, 2, 3, 4, 5, 8      # bsg_render records


class TrafConfig(C.Structure):
    _fields_ = [("n", C.c_int64), ("max_wpts", C.c_int32), ("reso", C.c_int32), ("reso_mode", C.c_int32), ("simdt", C.c_float),
                ("rpz", C.c_float), ("hpz", C.c_float), ("dtlookahead", C.c_float), ("resofach", C.c_float),
                ("resofacv", C.c_float), ("perf", Perf), ("lat0", C.c_double), ("lon0", C.c_double), ("row0", C.c_int64)]


class TrafTensors(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("pos", "kin", "cmd", "aux", "actwp", "vnav1", "vnav2", "asas", "flags", "partners",
                                          "rt_pos", "rt_con", "rt_dir", "counters")]


class TrafEvents(C.Structure):
    _fields_ = [("d_cur", C.c_void_p), ("d_prev", C.c_void_p), ("set_bytes", C.c_int64), ("d_conf_log", C.c_void_p),
                ("d_los_log", C.c_void_p), ("d_los_sev", C.c_void_p), ("conf_log_cap", C.c_int64), ("los_log_cap", C.c_int64),
                ("d_counters", C.c_void_p)]


class Layout(C.Structure):
    _fields_ = [("slots", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("info_dim", C.c_int32),
                ("n_sub", C.c_int32), ("env_f64", C.c_int32), ("env_f32", C.c_int32), ("env_i32", C.c_int32),
                ("poly_f64", C.c_int32), ("simdt", C.c_float)]


TENSOR_FIELDS = ("pos", "kin", "cmd", "aux", "flags", "tcpamax", "inconf", "env_f64", "env_f32", "env_i32",
                 "poly", "obs", "final_obs", "final_ids", "final_count", "reward", "terminated", "truncated", "info", "actions_staging",
                 "cd_pairs", "cd_attr")


class TensorTable(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in TENSOR_FIELDS]


SYMBOLS = ("bsg_abi_version", "bsg_abi_struct_size", "bsg_last_error", "bsg_device_count", "bsg_query_layout", "bsg_create",
           "bsg_destroy", "bsg_bind_state", "bsg_reset", "bsg_step", "bsg_step_host", "bsg_step_host_block", "bsg_step_host_copy", "bsg_step_host_begin", "bsg_step_host_wait", "bsg_host_copy", "bsg_host_widen", "bsg_set_obs_noise", "bsg_get_noise_calls", "bsg_set_noise_calls", "bsg_load_state", "bsg_set_seed", "bsg_set_wind", "bsg_traf_update",
           "bsg_cd_padded", "bsg_cd_pack", "bsg_cd_order_workspace", "bsg_cd_pack_ordered", "bsg_cd_detect", "bsg_cd_cull_workspace", "bsg_cd_detect_culled", "bsg_cd_detect_peers", "bsg_cd_unpermute", "bsg_probe_fp32",
           "bsg_traf_pack", "bsg_traf_order_workspace", "bsg_traf_pack_ordered", "bsg_traf_activate", "bsg_traf_workspace", "bsg_traf_substep", "bsg_traf_events_workspace",
           "bsg_traf_events_update", "bsg_render")

_lib = None


class BsgError(RuntimeError):
    pass


def load():
    """Loads the CUDA extension; raises if it has not been built (python -m bluesky_gym_sasha_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BsgError(f"{LIB_PATH} is missing: build it with `python -m bluesky_gym_sasha_b200.build` "
                       "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, f32, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_float, C.c_double
    lib.bsg_abi_version.restype = C.c_int
    lib.bsg_last_error.restype = C.c_char_p
    lib.bsg_device_count.restype = C.c_int
    lib.bsg_query_layout.argtypes = [C.POINTER(Config), C.POINTER(Layout)]
    lib.bsg_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    lib.bsg_destroy.argtypes = [vp]
    lib.bsg_destroy.restype = None
    lib.bsg_bind_state.argtypes = [vp, C.POINTER(TensorTable)]
    lib.bsg_reset.argtypes = [vp, vp, vp]
    lib.bsg_step.argtypes = [vp, vp, vp]
    lib.bsg_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.bsg_step_host_block.argtypes = [vp, vp, vp, C.c_size_t, vp]
    lib.bsg_step_host_begin.argtypes = [vp, vp, vp, C.c_size_t, vp]
    lib.bsg_step_host_begin.restype = C.c_int
    lib.bsg_step_host_wait.argtypes = [vp, vp, vp, C.c_size_t]
    lib.bsg_step_host_wait.restype = C.c_int
    lib.bsg_set_obs_noise.argtypes = [vp, f32]
    lib.bsg_set_obs_noise.restype = C.c_int
    lib.bsg_set_seed.argtypes = [vp, C.c_uint64]
    lib.bsg_set_seed.restype = C.c_int
    lib.bsg_set_wind.argtypes = [vp, C.POINTER(Wind)]
    lib.bsg_set_wind.restype = C.c_int
    lib.bsg_load_state.argtypes = [vp, i32, C.POINTER(AcState), vp]
    lib.bsg_load_state.restype = C.c_int
    lib.bsg_get_noise_calls.argtypes = [vp, C.POINTER(u32)]
    lib.bsg_get_noise_calls.restype = C.c_int
    lib.bsg_set_noise_calls.argtypes = [vp, u32]
    lib.bsg_set_noise_calls.restype = C.c_int
    lib.bsg_host_copy.argtypes = [vp, vp, C.c_size_t]
    lib.bsg_host_copy.restype = C.c_int
    lib.bsg_host_widen.argtypes = [vp, vp, C.c_size_t]
    lib.bsg_host_widen.restype = C.c_int
    lib.bsg_step_host_copy.argtypes = [vp, vp, vp, C.c_size_t, vp, C.c_size_t, vp]
    lib.bsg_traf_update.argtypes = [vp, i32, vp]
    lib.bsg_render.argtypes = [vp, i32, i32, i32, u32, vp, vp]
    lib.bsg_render.restype = C.c_int
    lib.bsg_traf_pack.argtypes = [C.POINTER(TrafConfig), C.POINTER(TrafTensors), vp, vp]
    lib.bsg_traf_order_workspace.argtypes = [i64]
    lib.bsg_traf_order_workspace.restype = i64
    lib.bsg_traf_pack_ordered.argtypes = [C.POINTER(TrafConfig), C.POINTER(TrafTensors), i32, vp, vp, vp, vp, i64, vp]
    lib.bsg_traf_activate.argtypes = [C.POINTER(TrafConfig), C.POINTER(TrafTensors), vp]
    lib.bsg_traf_substep.argtypes = [C.POINTER(TrafConfig), C.POINTER(TrafTensors), vp, i32, vp, vp, vp, vp, i64, vp, i64, vp]
    lib.bsg_traf_workspace.argtypes = [i64, i64]
    lib.bsg_traf_workspace.restype = i64
    lib.bsg_traf_events_workspace.argtypes = [i64, i64]
    lib.bsg_traf_events_workspace.restype = i64
    lib.bsg_traf_events_update.argtypes = [C.POINTER(TrafEvents), vp, C.POINTER(CdLists), i64, vp]
    lib.bsg_cd_padded.argtypes = [i64]
    lib.bsg_cd_padded.restype = i64
    lib.bsg_cd_pack.argtypes = [vp, vp, vp, vp, vp, vp, i64, f64, f64, vp, vp]
    lib.bsg_cd_order_workspace.argtypes = [i64]
    lib.bsg_cd_order_workspace.restype = i64
    lib.bsg_cd_pack_ordered.argtypes = [vp, vp, vp, vp, vp, vp, i64, f64, f64, vp, vp, vp, i64, vp]
    lib.bsg_cd_detect.argtypes = [vp, i64, i64, i64, f32, f32, f32, u32, vp, vp, vp, vp, C.POINTER(CdLists), vp]
    lib.bsg_cd_cull_workspace.argtypes = [i64, i64]
    lib.bsg_cd_cull_workspace.restype = i64
    lib.bsg_cd_detect_culled.argtypes = [vp, i64, i64, i64, f32, f32, f32, u32, vp, vp, vp, vp, C.POINTER(CdLists), vp, i64, vp]
    lib.bsg_cd_detect_peers.argtypes = [C.POINTER(vp), i32, i32, i64, f32, f32, f32, u32, vp, vp, vp, vp, C.POINTER(CdLists), vp, i64, vp]
    lib.bsg_cd_unpermute.argtypes = [vp, i64, C.POINTER(CdLists), vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.bsg_probe_fp32.argtypes = [i32, C.POINTER(f64)]
    lib.bsg_abi_struct_size.argtypes = [C.c_int]
    lib.bsg_abi_struct_size.restype = C.c_int
    for name in ("bsg_query_layout", "bsg_create", "bsg_bind_state", "bsg_reset", "bsg_step", "bsg_step_host", "bsg_step_host_block", "bsg_step_host_copy",
                 "bsg_traf_update", "bsg_traf_pack", "bsg_traf_pack_ordered", "bsg_traf_activate", "bsg_traf_substep", "bsg_traf_events_update", "bsg_cd_pack", "bsg_cd_pack_ordered",
                 "bsg_cd_detect", "bsg_cd_detect_culled", "bsg_cd_detect_peers", "bsg_cd_unpermute", "bsg_probe_fp32"):
        getattr(lib, name).restype = C.c_int
    for which, st in enumerate((Config, Layout, TensorTable, Wind, Perf, AcState, CdLists, TrafConfig, TrafTensors, TrafEvents)):
        if lib.bsg_abi_struct_size(which) != C.sizeof(st):
            raise BsgError(f"{LIB_PATH}: sizeof({st.__name__}) is {lib.bsg_abi_struct_size(which)} in the library, "
                           f"{C.sizeof(st)} in bluesky_gym_sasha_b200/_lib.py (include/bsg.h changed: rebuild / update the binding)")
    _lib = lib
    return lib


def check(rc):
    if rc != BSG_OK:
        msg = load().bsg_last_error().decode("utf-8", "replace")
        raise BsgError(f"libbsg_b200 error {rc}: {msg}")


def query_layout(cfg: Config) -> Layout:
    lay = Layout()
    check(load().bsg_query_layout(C.byref(cfg), C.byref(lay)))
    return lay
