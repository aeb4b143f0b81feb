"""ctypes binding of the C ABI in include/ekf_slam_b200.h (the same stub a maintainer of the reference
would write, see INTEGRATION.md).  The shared library is built in-tree by build.sh / __graft_entry__.build();
there is no fallback of any kind: a missing library or a missing GPU raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# EKF_B200_LIB: development aid (a differently-built copy of the same library); never a fallback
LIB_PATH = os.environ.get("EKF_B200_LIB") or os.path.join(_HERE, "libekfslam_b200.so")

c_double_p = ctypes.POINTER(ctypes.c_double)
c_float_p = ctypes.POINTER(ctypes.c_float)
c_u8_p = ctypes.POINTER(ctypes.c_uint8)
c_i32_p = ctypes.POINTER(ctypes.c_int32)
c_i64_p = ctypes.POINTER(ctypes.c_int64)
c_u64_p = ctypes.POINTER(ctypes.c_uint64)
c_void_pp = ctypes.POINTER(ctypes.c_void_p)


class EkfError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"ekf_slam_b200 error {code}: {message}")
        self.code = code


# name -> (restype, argtypes); every symbol include/ekf_slam_b200.h and include/circle_fit_b200.h declare
SIGNATURES = {
    "ekf_version": (ctypes.c_char_p, []),
    "ekf_last_error": (ctypes.c_char_p, []),
    "ekf_device_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)]),
    "ekf_host_alloc": (ctypes.c_int, [c_void_pp, ctypes.c_uint64]),
    "ekf_host_free": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_void_pp]),
    "ekf_create_ex": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void_pp]),
    "ekf_clone": (ctypes.c_int, [ctypes.c_void_p, c_void_pp]),
    "ekf_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_num_landmarks": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_engine": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_predict": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_double, ctypes.c_double]),
    "ekf_measurement": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_u8_p]),
    "ekf_data_association": (ctypes.c_int, [ctypes.c_void_p, c_double_p, ctypes.c_int, c_u8_p, c_i32_p,
                                            c_double_p, c_double_p, c_u8_p]),
    "ekf_maha": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_int, c_double_p]),
    "ekf_get_pose": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "ekf_get_landmarks": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "ekf_get_state": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "ekf_set_state": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "ekf_association_log_open": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p]),
    "ekf_get_sigma": (ctypes.c_int, [ctypes.c_void_p, c_double_p, ctypes.c_int64]),
    "ekf_get_sigma_rows": (ctypes.c_int, [ctypes.c_void_p, c_i64_p, ctypes.c_int, c_double_p, ctypes.c_int64]),
    "ekf_get_sigma_diag": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "ekf_set_sigma": (ctypes.c_int, [ctypes.c_void_p, c_double_p, ctypes.c_int64]),
    "ekf_get_init_flag": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int)]),
    "ekf_set_init_flag": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "ekf_update_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_device_pointers": (ctypes.c_int, [ctypes.c_void_p, c_void_pp, c_i64_p, c_void_pp]),
    "ekf_stream": (ctypes.c_void_p, [ctypes.c_void_p]),
    "ekf_launch_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_sweep_count": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]),
    "ekf_set_carry_pending": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "ekf_set_max_pending": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "ekf_batch_create": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, c_void_pp]),
    "ekf_batch_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_batch_size": (ctypes.c_int64, [ctypes.c_void_p]),
    "ekf_batch_engine": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_batch_sweep_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_batch_step_known": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_batch_step_unknown": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                              ctypes.c_int, ctypes.c_void_p]),
    "ekf_batch_step_known_sparse": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                   ctypes.c_void_p, ctypes.c_int64]),
    "ekf_batch_step_known_sparse_dev": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                       ctypes.c_void_p, ctypes.c_int64]),
    "ekf_batch_step_known_dev": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_batch_step_unknown_dev": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                  ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    "ekf_batch_get_poses": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_batch_get_poses_async": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_batch_get_states": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "ekf_batch_get_sigma": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, c_double_p, ctypes.c_int64]),
    "ekf_batch_checkpoint_size": (ctypes.c_int, [ctypes.c_void_p, c_i64_p, c_i64_p]),
    "ekf_batch_export": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_batch_import": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_void_p, ctypes.c_uint64]),
    "ekf_batch_get_known": (ctypes.c_int, [ctypes.c_void_p, c_u8_p]),
    "ekf_batch_set_known": (ctypes.c_int, [ctypes.c_void_p, c_u8_p]),
    "ekf_batch_update_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_batch_pose_error": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p]),
    "ekf_batch_get_marginals": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_batch_nees": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                      ctypes.c_void_p]),
    "ekf_batch_nees_dev": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                          ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_batch_set_nis": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "ekf_batch_nis": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]),
    "ekf_batch_nis_dev": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]),
    "ekf_batch_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_batch_device_pointers": (ctypes.c_int, [ctypes.c_void_p, c_void_pp, c_i64_p, c_void_pp, c_i64_p]),
    "ekf_batch_stream": (ctypes.c_void_p, [ctypes.c_void_p]),
    "ekf_timer_start": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_timer_stop": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]),
    "ekf_batch_timer_start": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_batch_timer_stop": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]),
    "ekf_batch_launch_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_normalize_angles": (ctypes.c_int, [c_double_p, c_double_p, ctypes.c_int64, ctypes.c_int]),
    "ekf_update_pose": (ctypes.c_int, [ctypes.c_double, ctypes.c_double, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p]),
    "ekf_body_twist": (ctypes.c_int, [ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, c_double_p]),
    # include/circle_fit_b200.h
    "circles_last_error": (ctypes.c_char_p, []),
    "circles_max_clusters": (ctypes.c_int, []),
    "circles_max_beams": (ctypes.c_int, []),
    "circles_create": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void_pp]),
    "circles_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "circles_run_f32": (ctypes.c_int, [ctypes.c_void_p, c_float_p, ctypes.c_int64, c_double_p, c_i32_p]),
    "circles_run_f64": (ctypes.c_int, [ctypes.c_void_p, c_double_p, ctypes.c_int64, c_double_p, c_i32_p]),
    "circles_run_dev_f32": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]),
    "circles_device_outputs": (ctypes.c_int, [ctypes.c_void_p, c_void_pp, c_void_pp]),
    "circles_last_clusters": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, c_i32_p, c_i32_p, c_double_p, c_u8_p,
                                             c_double_p]),
    "circles_fit_clusters": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_i32_p, ctypes.c_int, c_double_p, c_u8_p]),
    "circles_set_centres_only": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "circles_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "circles_timer_start": (ctypes.c_int, [ctypes.c_void_p]),
    "circles_timer_stop": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]),
    "circles_launch_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    # include/tube_world_b200.h
    "tubeworld_last_error": (ctypes.c_char_p, []),
    "tubeworld_create": (ctypes.c_int, [ctypes.c_int64, ctypes.c_void_p, c_double_p, c_double_p, ctypes.c_int, ctypes.c_uint64,
                                        ctypes.c_int64, ctypes.c_int, c_void_pp]),
    "tubeworld_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "tubeworld_step_known": (ctypes.c_int, [ctypes.c_void_p]),
    "tubeworld_step_scan": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "tubeworld_outputs": (ctypes.c_int, [ctypes.c_void_p, c_void_pp, c_void_pp, c_void_pp, c_void_pp, c_void_pp]),
    "tubeworld_download": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p, c_u8_p, c_double_p, c_float_p]),
    "tubeworld_odometry": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "tubeworld_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "tubeworld_stream": (ctypes.c_void_p, [ctypes.c_void_p]),
    "tubeworld_set_stream": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
}

# include/ekf_sharded_b200.h (separate library: it links NCCL)
SHARDED_LIB_PATH = os.environ.get("EKF_B200_SHARDED_LIB") or os.path.join(_HERE, "libekfslam_sharded_b200.so")
SIGNATURES_SHARDED = {
    "ekf_sharded_last_error": (ctypes.c_char_p, []),
    "ekf_sharded_unique_id": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_sharded_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, c_void_pp]),
    "ekf_sharded_create_local": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void_pp]),
    "ekf_sharded_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_sharded_predict": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_double, ctypes.c_double]),
    "ekf_sharded_measurement": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ekf_sharded_data_association": (ctypes.c_int, [ctypes.c_void_p, c_double_p, ctypes.c_int, c_u8_p, c_i32_p,
                                                    c_double_p, c_double_p, c_u8_p]),
    "ekf_sharded_get_state": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "ekf_sharded_set_max_pending": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "ekf_sharded_exchange_bytes": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_sharded_attach_exchange": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_u64_p, ctypes.c_uint64]),
    "ekf_sharded_rows": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_i64_p, c_i64_p]),
    "ekf_sharded_get_sigma_rows": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_double_p, ctypes.c_int64]),
    "ekf_sharded_get_sigma_row_list": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_i64_p, ctypes.c_int, c_double_p,
                                                      ctypes.c_int64]),
    "ekf_sharded_update_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_sharded_sweep_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_sharded_set_carry_pending": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "ekf_sharded_launch_count": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ekf_sharded_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_sharded_timer_start": (ctypes.c_int, [ctypes.c_void_p]),
    "ekf_sharded_timer_stop": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]),
}

_lib = None
_lib_sharded = None


def _preload_bundled_nccl():
    """libekfslam_sharded_b200.so needs `libnccl.so.2`.  If the process later imports torch, torch insists on the NCCL
    it was built with (a newer one than the system's), and whichever libnccl.so.2 is mapped first wins: so map the
    wheel-bundled one first when there is one.  Without it the dynamic loader falls back to the system library."""
    import importlib.util
    import sys
    if "torch" in sys.modules:
        return  # torch already mapped its own
    spec = importlib.util.find_spec("nvidia.nccl") if importlib.util.find_spec("nvidia") else None
    for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
        cand = os.path.join(base, "lib", "libnccl.so.2")
        if os.path.exists(cand):
            try:
                ctypes.CDLL(cand, mode=ctypes.RTLD_GLOBAL)
            except OSError:
                pass
            return


def load_sharded():
    """Load the row-sharded engine's library (once).  Raises if it has not been built or NCCL cannot be resolved."""
    global _lib_sharded
    if _lib_sharded is not None:
        return _lib_sharded
    if not os.path.exists(SHARDED_LIB_PATH):
        raise ImportError(f"{SHARDED_LIB_PATH} is missing: run ./build.sh")
    _preload_bundled_nccl()
    lib = ctypes.CDLL(SHARDED_LIB_PATH)
    for name, (res, args) in SIGNATURES_SHARDED.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib_sharded = lib
    return lib


def load():
    """Load the product library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: run ./build.sh (or __graft_entry__.build()). "
            "There is no CPU fallback for the EKF-SLAM hot path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header and library out of step
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise EkfError(rc, load().ekf_last_error().decode("utf-8", "replace"))


def device_count():
    c = ctypes.c_int(0)
    rc = load().ekf_device_count(ctypes.byref(c))
    return c.value if rc == 0 else 0
