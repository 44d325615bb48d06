"""ctypes binding of include/gut_b200.h (libgut_b200.so).  There is NO CPU or PyTorch fallback: if the CUDA
extension cannot be built/loaded, or no GPU is present when a context is created, this raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libgut_b200.so")
_LIB = None


class Camera(C.Structure):
    """gutb200_camera"""

    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("principal", C.c_float * 2), ("focal", C.c_float * 2),
        ("radial", C.c_float * 6), ("tangential", C.c_float * 2), ("thin_prism", C.c_float * 4),
        ("pose_start", C.c_float * 7), ("pose_end", C.c_float * 7),
        ("model", C.c_int32), ("max_angle", C.c_float),
        ("ftheta_reference_poly", C.c_int32), ("ftheta_bw", C.c_float * 6), ("ftheta_fw", C.c_float * 6), ("ftheta_cde", C.c_float * 3),
        ("rolling_shutter", C.c_int32),
    ]


class Config(C.Structure):
    """gutb200_config"""

    _fields_ = [
        ("kernel_degree", C.c_int32), ("min_kernel_density", C.c_float), ("min_alpha", C.c_float),
        ("max_alpha", C.c_float), ("min_transmittance", C.c_float),
        ("ut_alpha", C.c_float), ("ut_beta", C.c_float), ("ut_kappa", C.c_float), ("ut_delta", C.c_float),
        ("ut_margin", C.c_float),
        ("rect_bounding", C.c_int32), ("tight_opacity_bounding", C.c_int32), ("tile_culling", C.c_int32),
        ("global_z_order", C.c_int32), ("enable_timings", C.c_int32), ("n_rolling_shutter_iterations", C.c_int32),
        ("k_buffer_size", C.c_int32), ("subtile_culling", C.c_int32),
    ]


EXPORTS = [
    "gutb200_version", "gutb200_default_config", "gutb200_create", "gutb200_destroy", "gutb200_last_error",
    "gutb200_forward", "gutb200_backward", "gutb200_forward_host", "gutb200_backward_host", "gutb200_last_stats",
    "gutb200_debug_copy", "gutb200_collect_times", "gutb200_collect_stage_times", "gutb200_set_timings", "gutb200_launch_count",
    "gutb200_backward_compact", "gutb200_sph_grad_from_views", "gutb200_camera_position",
    "gutb200_debug_work_counters", "gutb200_debug_fma_peak",
    "gutb200_selective_adam_update", "gutb200_gaussian_adam_step", "gutb200_gaussian_adam_step_reg",  # bound in optimizers/__init__.py
    "gutb200_image_loss_scratch_bytes", "gutb200_image_loss",  # bound in losses.py
]

def camera_position(cam):
    """Sensor position in world space as the kernels compute it (gutb200_camera_position): numpy float32 [3]."""
    import numpy as np

    out = np.zeros(3, np.float32)
    if load().gutb200_camera_position(C.byref(cam), out.ctypes.data) != 0:
        raise RuntimeError("gutb200_camera_position failed")
    return out


DBG_TILES_COUNT, DBG_SORTED_KEYS, DBG_SORTED_VALUES, DBG_TILE_RANGES, DBG_DEPTH, DBG_RGB, DBG_PROJ = range(7)


def lib_path() -> str:
    return _SO


def load():
    """Load (building in-tree if sources are newer) the sm_100a shared library."""
    global _LIB
    if _LIB is not None:
        return _LIB
    import build as _build  # 3dgrut_b200/build.py

    if _build.needs_build():
        _build.build()
    if not os.path.exists(_SO):
        raise RuntimeError(f"{_SO} is missing: the CUDA extension was not built (no fallback path exists)")
    lib = C.CDLL(_SO)
    lib.gutb200_version.restype = C.c_char_p
    lib.gutb200_last_error.restype = C.c_char_p
    lib.gutb200_last_error.argtypes = [C.c_void_p]
    lib.gutb200_launch_count.restype = C.c_int64
    lib.gutb200_launch_count.argtypes = [C.c_void_p]
    lib.gutb200_create.argtypes = [C.POINTER(Config), C.c_int, C.POINTER(C.c_void_p)]
    lib.gutb200_destroy.argtypes = [C.c_void_p]
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    cam = C.POINTER(Camera)
    lib.gutb200_forward.argtypes = [vp, vp, cam, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.gutb200_backward.argtypes = [vp, vp, cam, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.gutb200_backward_compact.argtypes = [vp, vp, cam, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.gutb200_sph_grad_from_views.argtypes = [vp, vp, i64, vp, i32, i32, vp, vp, vp]
    lib.gutb200_camera_position.argtypes = [cam, vp]
    lib.gutb200_forward_host.argtypes = [vp, cam, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.gutb200_backward_host.argtypes = [vp, cam, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.gutb200_last_stats.argtypes = [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    lib.gutb200_debug_copy.argtypes = [vp, C.c_int, vp, C.c_size_t]
    lib.gutb200_collect_times.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.gutb200_collect_stage_times.argtypes = [vp, C.POINTER(C.c_float)]
    lib.gutb200_set_timings.argtypes = [vp, C.c_int]
    lib.gutb200_debug_work_counters.argtypes = [vp, vp, vp, vp, vp]
    lib.gutb200_debug_fma_peak.argtypes = [vp, C.c_int, C.POINTER(C.c_float)]
    _LIB = lib
    return lib


def default_config() -> Config:
    cfg = Config()
    load().gutb200_default_config(C.byref(cfg))
    return cfg


class Context:
    """Owning wrapper of a gutb200_ctx*."""

    def __init__(self, cfg: Config, device: int = 0):
        self._lib = load()
        self._h = C.c_void_p()
        rc = self._lib.gutb200_create(C.byref(cfg), int(device), C.byref(self._h))
        if rc != 0 or not self._h:
            raise RuntimeError(f"gutb200_create failed (rc={rc}): a CUDA device is required, there is no CPU path")
        self.cfg = cfg

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gutb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise RuntimeError(f"{what} failed: {self._lib.gutb200_last_error(self._h).decode()}")

    def forward(self, stream, cam, n, particles, sph, sph_degree, rays_o, rays_d, out_rgba, out_dist, out_hits, visibility):
        self._check(self._lib.gutb200_forward(self._h, stream, C.byref(cam), n, particles, sph, sph_degree, rays_o, rays_d,
                                              out_rgba, out_dist, out_hits, visibility), "gutb200_forward")

    def backward(self, stream, cam, n, particles, sph, sph_degree, rays_o, rays_d, out_rgba, d_rgba, out_dist, d_dist,
                 d_particles, d_sph):
        self._check(self._lib.gutb200_backward(self._h, stream, C.byref(cam), n, particles, sph, sph_degree, rays_o, rays_d,
                                               out_rgba, d_rgba, out_dist, d_dist, d_particles, d_sph), "gutb200_backward")

    def backward_compact(self, stream, cam, n, particles, sph, sph_degree, rays_o, rays_d, out_rgba, d_rgba, out_dist, d_dist,
                         d_particles, d_radiance):
        """Like backward, but emits the [N,4] masked radiance gradient instead of the [N,48] SH gradient (view-parallel exchange)."""
        self._check(self._lib.gutb200_backward_compact(self._h, stream, C.byref(cam), n, particles, sph, sph_degree, rays_o, rays_d,
                                                       out_rgba, d_rgba, out_dist, d_dist, d_particles, d_radiance), "gutb200_backward_compact")

    def sph_grad_from_views(self, stream, n, particles, sph_degree, view_positions, d_radiance_all, d_sph):
        """view_positions: float32 numpy [views,3] (host); d_radiance_all: device [views,N,4]; d_sph: device [N,48]."""
        import numpy as np

        vp_ = np.ascontiguousarray(view_positions, dtype=np.float32)
        self._check(self._lib.gutb200_sph_grad_from_views(self._h, stream, n, particles, sph_degree, int(vp_.shape[0]), vp_.ctypes.data,
                                                          d_radiance_all, d_sph), "gutb200_sph_grad_from_views")

    def forward_host(self, cam, n, particles, sph, sph_degree, rays_o, rays_d, out_rgba, out_dist, out_hits, visibility):
        self._check(self._lib.gutb200_forward_host(self._h, C.byref(cam), n, particles, sph, sph_degree, rays_o, rays_d,
                                                   out_rgba, out_dist, out_hits, visibility), "gutb200_forward_host")

    def backward_host(self, cam, n, particles, sph, sph_degree, rays_o, rays_d, out_rgba, d_rgba, out_dist, d_dist,
                      d_particles, d_sph):
        self._check(self._lib.gutb200_backward_host(self._h, C.byref(cam), n, particles, sph, sph_degree, rays_o, rays_d,
                                                    out_rgba, d_rgba, out_dist, d_dist, d_particles, d_sph), "gutb200_backward_host")

    def stats(self):
        n, i, v, t = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        self._check(self._lib.gutb200_last_stats(self._h, C.byref(n), C.byref(i), C.byref(v), C.byref(t)), "gutb200_last_stats")
        return {"N": n.value, "I": i.value, "V": v.value, "T": t.value}

    def debug_copy(self, what: int):
        import numpy as np

        st = self.stats()
        shape, dt = {
            DBG_TILES_COUNT: ((st["N"],), np.uint32), DBG_SORTED_KEYS: ((st["I"],), np.uint64),
            DBG_SORTED_VALUES: ((st["I"],), np.uint32), DBG_TILE_RANGES: ((st["T"], 2), np.uint32),
            DBG_DEPTH: ((st["N"],), np.float32), DBG_RGB: ((st["N"], 3), np.float32), DBG_PROJ: ((st["N"], 8), np.float32),
        }[what]
        out = np.zeros(shape, dt)
        self._check(self._lib.gutb200_debug_copy(self._h, what, out.ctypes.data, out.nbytes), "gutb200_debug_copy")
        return out

    def collect_times(self):
        f, b = C.c_float(), C.c_float()
        self._check(self._lib.gutb200_collect_times(self._h, C.byref(f), C.byref(b)), "gutb200_collect_times")
        return f.value, b.value

    STAGES = ("project", "scan", "expand", "sort", "tile_ranges", "render", "render_backward", "project_backward")

    def collect_stage_times(self):
        arr = (C.c_float * 8)()
        self._check(self._lib.gutb200_collect_stage_times(self._h, arr), "gutb200_collect_stage_times")
        return dict(zip(self.STAGES, [float(v) for v in arr]))

    def set_timings(self, level: int):
        self._check(self._lib.gutb200_set_timings(self._h, int(level)), "gutb200_set_timings")

    def launch_count(self) -> int:
        return int(self._lib.gutb200_launch_count(self._h))

    COUNTERS = ("tests_ref", "tests_exec", "hits", "fwd_iters", "hit_iters", "screens", "bwd_lanes", "iters16", "iters8", "sub16_hits", "sub8_hits")

    def work_counters(self, particles, rays_o, rays_d):
        """Work counters of the last forward (device pointers as passed to it): dict of ints (gutb200_debug_work_counters)."""
        arr = (C.c_uint64 * 16)()
        self._check(self._lib.gutb200_debug_work_counters(self._h, particles, rays_o, rays_d, arr), "gutb200_debug_work_counters")
        return dict(zip(self.COUNTERS, [int(v) for v in arr]))

    def fma_peak_tflops(self, repeats: int = 5) -> float:
        v = C.c_float()
        self._check(self._lib.gutb200_debug_fma_peak(self._h, int(repeats), C.byref(v)), "gutb200_debug_fma_peak")
        return float(v.value)


# ---------------------------------------------------------------------------------------------------------------
# include/grt_b200.h (3DGRT: LBVH build + ordered ray tracing), same shared library

class GrtConfig(C.Structure):
    """grtb200_config"""

    _fields_ = [("kernel_degree", C.c_int32), ("min_response", C.c_float), ("min_alpha", C.c_float), ("max_alpha", C.c_float),
                ("density_clamping", C.c_int32)]


GRT_EXPORTS = ["grtb200_default_config", "grtb200_create", "grtb200_destroy", "grtb200_last_error", "grtb200_build_bvh", "grtb200_trace",
               "grtb200_trace_bwd", "grtb200_scene_aabb", "grtb200_launch_count", "grtb200_debug_trace_counters", "grtb200_set_replay"]


def _grt_lib():
    lib = load()
    if not getattr(lib, "_grt_ready", False):
        vp, i64, i32, f32 = C.c_void_p, C.c_int64, C.c_int32, C.c_float
        lib.grtb200_last_error.restype = C.c_char_p
        lib.grtb200_last_error.argtypes = [vp]
        lib.grtb200_launch_count.restype = i64
        lib.grtb200_launch_count.argtypes = [vp]
        lib.grtb200_create.argtypes = [C.POINTER(GrtConfig), C.c_int, C.POINTER(vp)]
        lib.grtb200_destroy.argtypes = [vp]
        lib.grtb200_build_bvh.argtypes = [vp, vp, i64, vp, vp, vp, vp, i32, i32]
        lib.grtb200_trace.argtypes = [vp, vp, i64, vp, vp, i32, f32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.grtb200_trace_bwd.argtypes = [vp, vp, i64, vp, vp, i32, f32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.grtb200_scene_aabb.argtypes = [vp, vp]
        lib.grtb200_set_replay.argtypes = [vp, i32]
        lib.grtb200_debug_trace_counters.argtypes = [vp, vp, i64, vp, vp, i32, f32, i32, i32, i32, vp, vp, vp, vp, vp]
        lib._grt_ready = True
    return lib


def grt_default_config() -> GrtConfig:
    cfg = GrtConfig()
    _grt_lib().grtb200_default_config(C.byref(cfg))
    return cfg


class GrtContext:
    """Owning wrapper of a grtb200_ctx*."""

    def __init__(self, cfg: GrtConfig, device: int = 0):
        self._lib = _grt_lib()
        self._h = C.c_void_p()
        rc = self._lib.grtb200_create(C.byref(cfg), int(device), C.byref(self._h))
        if rc != 0 or not self._h:
            raise RuntimeError(f"grtb200_create failed (rc={rc}): a CUDA device is required, there is no CPU path")
        self.cfg = cfg

    def close(self):
        if getattr(self, "_h", None):
            self._lib.grtb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed: {self._lib.grtb200_last_error(self._h).decode()}")

    def build_bvh(self, stream, n, pos, rot, scl, dns, rebuild=True, allow_update=False):
        self._check(self._lib.grtb200_build_bvh(self._h, stream, n, pos, rot, scl, dns, int(rebuild), int(allow_update)), "grtb200_build_bvh")

    def trace(self, stream, n, particles, sph, sph_degree, min_t, batch, height, width, rays_o, rays_d, r2w_host, out_rgb, out_alpha,
              out_dist, out_hits, visibility):
        self._check(self._lib.grtb200_trace(self._h, stream, n, particles, sph, sph_degree, min_t, batch, height, width, rays_o, rays_d,
                                            r2w_host, out_rgb, out_alpha, out_dist, out_hits, visibility), "grtb200_trace")

    def trace_bwd(self, stream, n, particles, sph, sph_degree, min_t, batch, height, width, rays_o, rays_d, r2w_host, out_rgb, out_alpha,
                  out_dist, d_rgb, d_alpha, d_dist, d_particles, d_sph):
        self._check(self._lib.grtb200_trace_bwd(self._h, stream, n, particles, sph, sph_degree, min_t, batch, height, width, rays_o, rays_d,
                                                r2w_host, out_rgb, out_alpha, out_dist, d_rgb, d_alpha, d_dist, d_particles, d_sph),
                    "grtb200_trace_bwd")

    def scene_aabb(self):
        import numpy as np

        out = np.zeros(6, np.float32)
        self._check(self._lib.grtb200_scene_aabb(self._h, out.ctypes.data), "grtb200_scene_aabb")
        return out

    def set_replay(self, enable: bool):
        """Record hit lists in the forward for the backward's replay (default on); off frees the cache (inference-only rendering)."""
        self._check(self._lib.grtb200_set_replay(self._h, int(bool(enable))), "grtb200_set_replay")

    TRACE_COUNTERS = ("rays", "queries", "node_visits", "box_tests", "proxy_tests", "candidate_hits", "accepted_hits", "packet_rays")

    def trace_counters(self, stream, n, particles, sph, sph_degree, min_t, batch, height, width, rays_o, rays_d, r2w_host, visibility_scratch):
        """Work counters of one forward trace (debug; synchronises): dict of ints."""
        arr = (C.c_uint64 * 8)()
        self._check(self._lib.grtb200_debug_trace_counters(self._h, stream, n, particles, sph, sph_degree, min_t, batch, height, width, rays_o, rays_d,
                                                           r2w_host, visibility_scratch, arr), "grtb200_debug_trace_counters")
        return dict(zip(self.TRACE_COUNTERS, [int(v) for v in arr]))

    def launch_count(self) -> int:
        return int(self._lib.grtb200_launch_count(self._h))
