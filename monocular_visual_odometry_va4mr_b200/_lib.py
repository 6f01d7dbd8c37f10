"""ctypes binding of ``csrc/libb200vo.so`` (C ABI declared in ``include/b200vo.h``).

The library is the product: if it is missing or no B200 is present every call raises --
there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(CSRC, "libb200vo.so")

c_u8p = C.POINTER(C.c_uint8)
c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
c_i32p = C.POINTER(C.c_int32)
c_intp = C.POINTER(C.c_int)


class BatchCfg(C.Structure):
    _fields_ = [
        ("rows", C.c_int), ("cols", C.c_int),
        ("win_w", C.c_int), ("win_h", C.c_int), ("max_level", C.c_int),
        ("crit_type", C.c_int), ("crit_max_count", C.c_int),
        ("crit_eps", C.c_double), ("min_eig_thr", C.c_double),
        ("pnp_iters", C.c_int), ("pnp_reproj_err", C.c_float), ("pnp_conf", C.c_double),
        ("K", C.c_double * 9),
        ("max_landmarks", C.c_int), ("max_candidates", C.c_int),
    ]


class LoopCfg(C.Structure):
    _fields_ = [
        ("batch", BatchCfg),
        ("min_dist_landmarks", C.c_double), ("max_dist_landmarks", C.c_double), ("min_baseline_angle_deg", C.c_double),
        ("min_baseline_frames", C.c_int),
        ("max_corners", C.c_int), ("quality_level", C.c_double), ("feature_min_dist", C.c_double),
        ("max_frames", C.c_int),
    ]


# name -> (restype, argtypes); mirrors include/b200vo.h one to one
SIGNATURES = {
    "b200vo_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "b200vo_destroy": (None, [C.c_void_p]),
    "b200vo_last_error": (C.c_char_p, [C.c_void_p]),
    "b200vo_version": (C.c_int, [c_intp]),
    "b200vo_launch_count": (C.c_longlong, [C.c_void_p]),
    "b200vo_last_gpu_ms": (C.c_float, [C.c_void_p]),
    "b200vo_calc_optical_flow_pyr_lk": (C.c_int, [
        C.c_void_p, c_u8p, c_u8p, C.c_int, C.c_int, C.c_size_t, C.c_size_t, c_f32p, C.c_int,
        C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double,
        c_f32p, c_u8p, c_f32p]),
    "b200vo_frame_upload": (C.c_int, [C.c_void_p, C.c_int, c_u8p, C.c_int, C.c_int, C.c_size_t,
                                      C.c_int, C.c_int, C.c_int]),
    "b200vo_klt_slots": (C.c_int, [
        C.c_void_p, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
        C.c_double, C.c_int, C.c_double, c_f32p, c_u8p, c_f32p]),
    "b200vo_frame_download_level": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_u8p, c_intp, c_intp, c_intp]),
    "b200vo_good_features_to_track": (C.c_int, [
        C.c_void_p, c_u8p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_double, C.c_double, C.c_int,
        c_f32p, c_intp]),
    "b200vo_knn2_ratio": (C.c_int, [
        C.c_void_p, c_f32p, C.c_int, c_f32p, C.c_int, C.c_int, C.c_double, c_i32p, c_f32p, c_u8p]),
    "b200vo_find_essential_mat_ransac": (C.c_int, [
        C.c_void_p, c_f32p, c_f32p, C.c_int, c_f64p, C.c_double, C.c_double, C.c_int, c_f64p, c_u8p, c_intp]),
    "b200vo_find_essential_mat_ransac_samples": (C.c_int, [
        C.c_void_p, c_f32p, c_f32p, C.c_int, c_f64p, c_i32p, C.c_int, C.c_double, C.c_double, c_f64p, c_u8p, c_intp,
        c_i32p, c_i32p, c_f64p, c_intp, c_intp]),
    # device-pointer forms: every array argument is a raw device address (int)
    "b200vo_calc_optical_flow_pyr_lk_dev": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p, C.c_int,
        C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200vo_good_features_to_track_dev": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_void_p]),
    "b200vo_knn2_ratio_dev": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200vo_find_essential_mat_ransac_dev": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, c_f64p, C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200vo_solve_pnp_ransac_p3p_dev": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, c_f64p, C.c_int, C.c_float, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
        C.c_void_p]),
    "b200vo_debug_pose_phases": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, c_f64p, C.c_int, C.c_float, C.c_double, C.POINTER(C.c_longlong), c_f32p]),
    "b200vo_sift_detect_and_compute": (C.c_int, [C.c_void_p, c_u8p, C.c_int, C.c_int, C.c_size_t, C.c_int, c_f32p, c_f32p, c_i32p]),
    "b200vo_recover_pose": (C.c_int, [C.c_void_p, c_f64p, c_f32p, c_f32p, C.c_int, c_f64p, C.c_double, c_f64p, c_f64p, c_u8p, c_intp]),
    "b200vo_min_distance_mask": (C.c_int, [C.c_void_p, c_f32p, C.c_int, c_f32p, C.c_int, C.c_float, c_u8p]),
    "b200vo_triangulate_landmarks": (C.c_int, [
        C.c_void_p, c_f64p, C.c_double, C.c_double, C.c_double, C.c_int, c_f32p, c_f32p, c_i32p, C.c_int, c_f64p, C.c_int,
        c_f64p, c_u8p, c_f32p, c_f32p, c_intp]),
    "b200vo_batch_min_distance_mask": (C.c_int, [C.c_void_p, C.c_int, c_f32p, c_i32p, C.c_int, c_f32p, c_i32p, C.c_int, C.c_float, c_u8p]),
    "b200vo_batch_triangulate_landmarks": (C.c_int, [
        C.c_void_p, c_f64p, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_i32p, c_i32p, c_f64p,
        c_i32p, C.c_int, c_f64p, c_u8p, c_f32p, c_f32p, c_i32p]),
    "b200vo_solve_pnp_ransac_p3p": (C.c_int, [
        C.c_void_p, c_f32p, c_f32p, C.c_int, c_f64p, C.c_int, C.c_float, C.c_double, c_f64p, c_f64p,
        c_i32p, c_intp, c_intp]),
    "b200vo_solve_pnp_ransac_p3p_samples": (C.c_int, [
        C.c_void_p, c_f32p, c_f32p, C.c_int, c_f64p, c_i32p, C.c_int, C.c_float, C.c_double, c_f64p,
        c_f64p, c_i32p, c_intp, c_intp, c_i32p, c_intp, c_intp]),
    "b200vo_batch_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(BatchCfg), C.POINTER(C.c_void_p)]),
    "b200vo_batch_destroy": (None, [C.c_void_p]),
    "b200vo_batch_set_intrinsics": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_f64p]),
    "b200vo_batch_set_frame_size": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_i32p, c_i32p]),
    "b200vo_batch_prime": (C.c_int, [C.c_void_p, c_u8p]),
    "b200vo_batch_submit_frames": (C.c_int, [C.c_void_p, c_u8p]),
    "b200vo_batch_submit_frames_dev": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200vo_batch_good_features": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, c_f32p, c_i32p]),
    "b200vo_batch_step": (C.c_int, [
        C.c_void_p, c_u8p, c_f32p, c_f32p, c_i32p, c_f32p, c_i32p, c_f32p, c_u8p, c_f32p, c_u8p,
        c_f64p, c_u8p, c_u8p, c_i32p]),
    "b200vo_batch_step_dev": (C.c_int, [C.c_void_p] + [C.c_void_p] * 14),
    "b200vo_batch_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "b200vo_batch_profile_read": (C.c_int, [C.c_void_p, c_f32p, c_intp]),
    "b200vo_loop_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(LoopCfg), C.POINTER(C.c_void_p)]),
    "b200vo_loop_destroy": (None, [C.c_void_p]),
    "b200vo_loop_set_intrinsics": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_f64p]),
    "b200vo_loop_set_frame_size": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_i32p, c_i32p]),
    "b200vo_loop_load": (C.c_int, [C.c_void_p, C.c_int, c_u8p, c_f32p, c_f32p, C.c_int, c_f32p, c_f32p, c_i32p, C.c_int, c_f64p,
                                   C.c_int]),
    "b200vo_loop_read_state": (C.c_int, [C.c_void_p, C.c_int, c_f32p, c_f32p, c_i32p, c_f32p, c_f32p, c_i32p, c_i32p, c_f64p, c_i32p,
                                         c_i32p]),
    "b200vo_loop_bootstrap": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_u8p, c_u8p, C.c_double, c_i32p, c_i32p, c_i32p, c_i32p]),
    "b200vo_loop_submit_frames": (C.c_int, [C.c_void_p, c_u8p]),
    "b200vo_loop_submit_frames_dev": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200vo_loop_step": (C.c_int, [C.c_void_p, c_u8p, c_i32p, c_i32p, c_i32p, c_i32p, c_f64p]),
    "b200vo_loop_step_dev": (C.c_int, [C.c_void_p] + [C.c_void_p] * 6),
    "b200vo_loop_step_seqs": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_u8p, c_i32p, c_i32p, c_i32p, c_i32p, c_f64p]),
    "b200vo_loop_step_seqs_dev": (C.c_int, [C.c_void_p, C.c_int, c_i32p] + [C.c_void_p] * 6),
    "b200vo_loop_submit_frames_seqs": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_u8p]),
    "b200vo_loop_submit_frames_seqs_dev": (C.c_int, [C.c_void_p, C.c_int, c_i32p, C.c_void_p]),
    "b200vo_sync": (C.c_int, [C.c_void_p]),
    "b200vo_host_alloc": (C.c_void_p, [C.c_void_p, C.c_size_t]),
    "b200vo_host_free": (None, [C.c_void_p, C.c_void_p]),
    "b200vo_stream": (C.c_void_p, [C.c_void_p]),
}


def build(force: bool = False) -> str:
    """Compile libb200vo.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    if force:
        subprocess.check_call(["make", "-C", CSRC, "-s", "clean"])
    subprocess.check_call(["make", "-C", CSRC, "-s", "-j8"])
    return SO_PATH


_lib = None


def load():
    """Load the shared library and bind every declared symbol.  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class B200VOError(RuntimeError):
    pass


class Context:
    """One CUDA device + stream + buffer pool (``b200vo_ctx``)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.b200vo_create(device, C.byref(h))
        if rc != 0 or not h:
            raise B200VOError(
                f"b200vo_create(device={device}) failed with code {rc}: a B200 (sm_100) GPU is required; "
                "this package has no CPU fallback")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.b200vo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def last_error(self) -> str:
        return (self.lib.b200vo_last_error(self.h) or b"").decode()

    def launch_count(self) -> int:
        return int(self.lib.b200vo_launch_count(self.h))

    def last_gpu_ms(self) -> float:
        return float(self.lib.b200vo_last_gpu_ms(self.h))

    def sync(self):
        self.lib.b200vo_sync(self.h)

    def stream(self) -> int:
        return int(self.lib.b200vo_stream(self.h) or 0)


_default_ctx: dict[int, Context] = {}


def default_context(device: int = 0) -> Context:
    ctx = _default_ctx.get(device)
    if ctx is None:
        ctx = _default_ctx[device] = Context(device)
    return ctx
