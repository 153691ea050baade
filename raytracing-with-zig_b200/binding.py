"""ctypes binding of librtz.so (include/rtz.h).  The product path: no oracle, no CPU fallback.

If the shared library is missing this module raises at import of `lib()` — loudly — instead of
degrading to anything else.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
import os

# RTZ_LIB=<path> loads another build of the same ABI (A/B timing of kernel changes inside one GPU call)
LIB_PATH = Path(os.environ["RTZ_LIB"]) if os.environ.get("RTZ_LIB") else PKG / "csrc" / "librtz.so"

D3 = C.c_double * 3


class rtz_sphere(C.Structure):
    """reference Sphere{center,radius,mat} (src/sphere.zig:13-17) with the Material inlined."""
    _fields_ = [("center", D3), ("radius", C.c_double), ("mat_type", C.c_int32), ("reserved", C.c_int32),
                ("albedo", D3), ("fuzz", C.c_double), ("refraction_index", C.c_double)]


class rtz_camera(C.Structure):
    """the fields of reference Camera (src/camera.zig:82-103) that render() reads."""
    _fields_ = [("width", C.c_uint64), ("height", C.c_uint64), ("center", D3), ("pixel0", D3), ("du", D3),
                ("dv", D3), ("defocus_disk_u", D3), ("defocus_disk_v", D3), ("defocus_angle", C.c_double),
                ("samples_per_pixel", C.c_uint64), ("bounce_max", C.c_uint64), ("pixel_samples_scale", C.c_double),
                ("t_min", C.c_double), ("t_max", C.c_double), ("seed", C.c_uint64), ("has_seed", C.c_int32),
                ("mode", C.c_int32)]


class rtz_shard(C.Structure):
    _fields_ = [("rank", C.c_uint32), ("world", C.c_uint32), ("tile_w", C.c_uint32), ("tile_h", C.c_uint32)]


class rtz_stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("segments", C.c_uint64), ("sphere_tests", C.c_uint64),
                ("depth_capped", C.c_uint64), ("absorbed", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("trace_ms", C.c_double), ("resolve_ms", C.c_double), ("total_ms", C.c_double),
                ("seed_used", C.c_uint64), ("nan_samples", C.c_uint64), ("gpus", C.c_uint32), ("gather", C.c_uint32),
                ("gather_ms", C.c_double)]


class rtz_denoise_params(C.Structure):
    """à-trous levels and edge scales of rtz_denoise (include/rtz.h); NULL / None = the library's defaults."""
    _fields_ = [("levels", C.c_uint32), ("reserved", C.c_uint32), ("sigma_color", C.c_double),
                ("sigma_normal", C.c_double), ("sigma_albedo", C.c_double)]


class rtz_hit(C.Structure):
    _fields_ = [("hit", C.c_int32), ("index", C.c_int32), ("front", C.c_int32), ("reserved", C.c_int32),
                ("t", C.c_double), ("point", D3), ("normal", D3)]


class rtz_scatter(C.Structure):
    _fields_ = [("scattered", C.c_int32), ("reserved", C.c_int32), ("origin", D3), ("direction", D3),
                ("attenuation", D3)]


RTZ_OK = 0
SCENE_FINAL, SCENE_CHAPTER13, SCENE_SWEEP = 0, 1, 2
MODE_PATH, MODE_PATH_BVH = 0, 4   # MODE_PATH_BVH: extension, same image through a BVH (include/rtz.h)
ERR_NAMES = {1: "RTZ_ERR_BAD_ARG", 2: "RTZ_ERR_NO_DEVICE", 3: "RTZ_ERR_CUDA", 4: "RTZ_ERR_IO",
             5: "RTZ_ERR_TOO_MANY_SPHERES", 6: "RTZ_ERR_ARCH", 7: "RTZ_ERR_NCCL"}
GATHER_AUTO, GATHER_P2P, GATHER_NCCL = 0, 1, 2
ABI_VERSION = 2
# rtz_probe_sweeps kinds (include/rtz.h)
(SWEEP_CONST, SWEEP_CULL, SWEEP_SKIP_SELF, SWEEP_SMEM, SWEEP_GLOBAL, SWEEP_COOP, SWEEP_COOP_REGROUPED,
 SWEEP_BVH, SWEEP_WAVE4) = range(9)
BVH_HOST, BVH_DEVICE = 0, 1   # rtz_probe_bvh builders

# every symbol include/rtz.h declares, with its signature
_u8p, _f64p, _f32p = C.POINTER(C.c_uint8), C.POINTER(C.c_double), C.POINTER(C.c_float)
_vp, _u64, _u32, _i32, _f64 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_double
SIGNATURES = {
    "rtz_render": (_i32, [C.POINTER(rtz_camera), C.POINTER(rtz_sphere), _u64, _u8p, C.POINTER(rtz_stats)]),
    "rtz_render_linear": (_i32, [C.POINTER(rtz_camera), C.POINTER(rtz_sphere), _u64, _u8p, _f64p, C.POINTER(rtz_stats)]),
    "rtz_write_ppm": (_i32, [C.c_char_p, _u64, _u64, _u8p]),
    "rtz_context_create": (_i32, [_i32, _vp, C.POINTER(_vp)]),
    "rtz_context_destroy": (_i32, [_vp]),
    "rtz_scene_upload": (_i32, [_vp, C.POINTER(rtz_sphere), _u64]),
    "rtz_scene_upload_device": (_i32, [_vp, _vp, _u64]),
    "rtz_scene_generate": (_i32, [_vp, _i32, _u64, _u64, C.POINTER(rtz_sphere), _u64, C.POINTER(_u64), C.POINTER(_u64)]),
    "rtz_shard_pixels": (_u64, [_u64, _u64, C.POINTER(rtz_shard)]),
    "rtz_render_resident": (_i32, [_vp, C.POINTER(rtz_camera), C.POINTER(rtz_shard), _vp, C.POINTER(rtz_stats)]),
    "rtz_render_resident_linear": (_i32, [_vp, C.POINTER(rtz_camera), C.POINTER(rtz_shard), _vp, _vp,
                                          C.POINTER(rtz_stats)]),
    "rtz_render_guides": (_i32, [_vp, C.POINTER(rtz_camera), _u64, _vp, _vp, C.POINTER(rtz_stats)]),
    "rtz_render_guides_sharded": (_i32, [_vp, C.POINTER(rtz_camera), C.POINTER(rtz_shard), _u64, _vp, _vp,
                                         C.POINTER(rtz_stats)]),
    "rtz_denoise": (_i32, [_vp, _u64, _u64, _vp, _vp, _vp, C.POINTER(rtz_denoise_params), _vp, _vp,
                           C.POINTER(rtz_stats)]),
    "rtz_render_denoised": (_i32, [C.POINTER(rtz_camera), C.POINTER(rtz_sphere), _u64, _u64,
                                   C.POINTER(rtz_denoise_params), _u8p, _f32p, C.POINTER(rtz_stats)]),
    "rtz_deinterleave": (_i32, [_vp, _u64, _u64, _u32, _u32, _u32, _vp, _vp]),
    "rtz_deinterleave_f32": (_i32, [_vp, _u64, _u64, _u32, _u32, _u32, _vp, _vp]),
    "rtz_multi_create": (_i32, [_i32, C.POINTER(_i32), _u32, _u32, _i32, C.POINTER(_vp)]),
    "rtz_multi_destroy": (_i32, [_vp]),
    "rtz_multi_gpus": (_i32, [_vp]),
    "rtz_multi_gather": (_i32, [_vp]),
    "rtz_multi_scene_upload": (_i32, [_vp, C.POINTER(rtz_sphere), _u64]),
    "rtz_multi_render": (_i32, [_vp, C.POINTER(rtz_camera), _u8p, C.POINTER(_vp), C.POINTER(rtz_stats)]),
    "rtz_render_multi": (_i32, [C.POINTER(rtz_camera), C.POINTER(rtz_sphere), _u64, _i32, _u8p, C.POINTER(rtz_stats)]),
    "rtz_multi_render_denoised": (_i32, [_vp, C.POINTER(rtz_camera), _u64, C.POINTER(rtz_denoise_params), _u8p, _f32p,
                                         C.POINTER(rtz_stats)]),
    "rtz_render_multi_denoised": (_i32, [C.POINTER(rtz_camera), C.POINTER(rtz_sphere), _u64, _i32, _u64,
                                         C.POINTER(rtz_denoise_params), _u8p, _f32p, C.POINTER(rtz_stats)]),
    "rtz_probe_hit": (_i32, [C.POINTER(rtz_sphere), _u64, D3, D3, _f64, _f64, C.POINTER(rtz_hit)]),
    "rtz_probe_scatter": (_i32, [C.POINTER(rtz_sphere), _u64, _i32, D3, D3, _u64, _u32, _u32, _u32,
                                 C.POINTER(rtz_scatter)]),
    "rtz_probe_hits": (_i32, [C.POINTER(rtz_sphere), _u64, _vp, _u64, _f64, _f64, _vp]),
    "rtz_probe_scatters": (_i32, [C.POINTER(rtz_sphere), _u64, _vp, _u64, _u64, _vp]),
    "rtz_probe_to_rgb": (_i32, [_f64p, _u64, _u8p]),
    "rtz_probe_sweep_order": (_i32, [C.POINTER(rtz_sphere), _u64, C.POINTER(_i32)]),
    "rtz_probe_cull_bounds": (_i32, [C.POINTER(rtz_sphere), _u64, _f32p, _f32p, C.POINTER(_i32)]),
    "rtz_probe_sweeps": (_i32, [C.POINTER(rtz_sphere), _u64, _vp, _u64, _f64, _f64, _i32, _i32, _vp]),
    "rtz_probe_scene_rows": (_i32, [_vp, _vp, _u64, C.POINTER(_u64)]),
    "rtz_probe_bvh": (_i32, [_vp, _i32, _vp, _u64, C.POINTER(_i32), _f32p, C.POINTER(_u64)]),
    "rtz_probe_uniform": (_i32, [_u64, _u32, _u32, _u32, _u64, _f32p]),
    "rtz_probe_camera_ray": (_i32, [C.POINTER(rtz_camera), _u64, _u64, _u64, _u64, _f32p, _f32p, _f32p]),
    "rtz_strerror": (C.c_char_p, [_i32]),
    "rtz_last_error": (C.c_char_p, []),
    "rtz_abi_version": (_i32, []),
    "rtz_device_count": (_i32, [C.POINTER(_i32)]),
    "rtz_measure_fp32_peak": (_i32, [_i32, _i32, _f64p]),
}

_lib = None


class RtzError(RuntimeError):
    def __init__(self, status: int, detail: str = ""):
        self.status = status
        super().__init__(f"{ERR_NAMES.get(status, status)}: {detail}")


def lib() -> C.CDLL:
    """Load librtz.so.  Raises (never falls back) when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(f"{LIB_PATH} is missing: run `python -m __graft_entry__` / build.py first. "
                              "This package has no CPU or PyTorch fallback.")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(l, name)  # AttributeError if the .so does not export a declared symbol
            except AttributeError:
                if os.environ.get("RTZ_LIB"):   # A/B timing against an older build of the ABI: tolerate what it lacks
                    continue
                raise
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(status: int) -> None:
    if status != RTZ_OK:
        l = lib()
        raise RtzError(status, (l.rtz_strerror(status) or b"").decode() + " | " + (l.rtz_last_error() or b"").decode())
