"""ctypes mirrors of include/rtz.h plus loaders for the oracle and the product library.

Used by the tests, by bench.py's cpu_baseline / --impl reference legs (oracle side) and by
__graft_entry__.smoke().  The product Python layer has its OWN ctypes binding in
raytracing-with-zig_b200/ and never touches the oracle.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
GOLDEN = Path(__file__).resolve().parent / "golden"

D3 = C.c_double * 3


class Sphere(C.Structure):
    _fields_ = [
        ("center", D3),
        ("radius", C.c_double),
        ("mat_type", C.c_int32),
        ("reserved", C.c_int32),
        ("albedo", D3),
        ("fuzz", C.c_double),
        ("refraction_index", C.c_double),
    ]


class Camera(C.Structure):
    _fields_ = [
        ("width", C.c_uint64),
        ("height", C.c_uint64),
        ("center", D3),
        ("pixel0", D3),
        ("du", D3),
        ("dv", D3),
        ("defocus_disk_u", D3),
        ("defocus_disk_v", D3),
        ("defocus_angle", C.c_double),
        ("samples_per_pixel", C.c_uint64),
        ("bounce_max", C.c_uint64),
        ("pixel_samples_scale", C.c_double),
        ("t_min", C.c_double),
        ("t_max", C.c_double),
        ("seed", C.c_uint64),
        ("has_seed", C.c_int32),
        ("mode", C.c_int32),
    ]


class Shard(C.Structure):
    _fields_ = [("rank", C.c_uint32), ("world", C.c_uint32), ("tile_w", C.c_uint32), ("tile_h", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [
        ("samples", C.c_uint64),
        ("segments", C.c_uint64),
        ("sphere_tests", C.c_uint64),
        ("depth_capped", C.c_uint64),
        ("absorbed", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("trace_ms", C.c_double),
        ("resolve_ms", C.c_double),
        ("total_ms", C.c_double),
        ("seed_used", C.c_uint64),
        ("nan_samples", C.c_uint64),
        ("gpus", C.c_uint32),
        ("gather", C.c_uint32),
        ("gather_ms", C.c_double),
    ]


class Hit(C.Structure):
    _fields_ = [
        ("hit", C.c_int32),
        ("index", C.c_int32),
        ("front", C.c_int32),
        ("reserved", C.c_int32),
        ("t", C.c_double),
        ("point", D3),
        ("normal", D3),
    ]


class Scatter(C.Structure):
    _fields_ = [
        ("scattered", C.c_int32),
        ("reserved", C.c_int32),
        ("origin", D3),
        ("direction", D3),
        ("attenuation", D3),
    ]


MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC = 0, 1, 2
MODE_PATH, MODE_LEGACY_SKY, MODE_LEGACY_FLAT, MODE_LEGACY_NORMAL, MODE_PATH_BVH = 0, 1, 2, 3, 4


def d3(v):
    return D3(*[float(x) for x in v])


def make_sphere(center, radius, mat, albedo=(1, 1, 1), fuzz=0.0, ior=1.0) -> Sphere:
    """Hittable.init(.sphere, ...) + Material.init defaults (reference src/material.zig:119-124)."""
    s = Sphere()
    s.center = d3(center)
    s.radius = max(0.0, float(radius))
    s.mat_type = mat
    s.albedo = d3(albedo)
    s.fuzz = float(fuzz)
    s.refraction_index = float(ior)
    return s


def sphere_array(spheres):
    arr = (Sphere * len(spheres))()
    for i, s in enumerate(spheres):
        arr[i] = s
    return arr


# --------------------------------------------------------------------------------------------
# oracle
# --------------------------------------------------------------------------------------------
_oracle = None


def build_oracle(force: bool = False) -> Path:
    so = ORACLE_DIR / "liboracle.so"
    srcs = list(ORACLE_DIR.glob("*.cpp")) + list(ORACLE_DIR.glob("*.h")) + [ROOT / "include" / "rtz.h"]

    def stale():
        return force or not so.exists() or any(s.stat().st_mtime > so.stat().st_mtime for s in srcs)

    if not stale():   # nothing to write: a built tree may be read-only
        return so
    import fcntl
    with open(ORACLE_DIR / ".build.lock", "w") as lock:   # N ranks / xdist workers may race here
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if stale():
                subprocess.run(["make", "-C", str(ORACLE_DIR), "-B", "liboracle.so"], check=True, capture_output=True)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return so


def oracle():
    """Load (building if needed) the CPU oracle.  Test infrastructure only."""
    global _oracle
    if _oracle is not None:
        return _oracle
    lib = C.CDLL(str(build_oracle()))
    vp, u64, f64, i32 = C.c_void_p, C.c_uint64, C.c_double, C.c_int32
    P = C.POINTER
    sig = {
        "orc_prng_new": (vp, [u64]),
        "orc_prng_free": (None, [vp]),
        "orc_prng_next": (u64, [vp]),
        "orc_prng_float": (f64, [vp]),
        "orc_prng_draws": (u64, [vp]),
        "orc_prng_state": (None, [vp, P(u64)]),
        "orc_generate_world": (u64, [vp, P(Sphere), u64]),
        "orc_generate_chapter13": (u64, [P(Sphere), u64]),
        "orc_generate_sweep": (u64, [vp, u64, P(Sphere)]),
        "orc_image_height": (u64, [u64, f64]),
        "orc_viewport": (None, [u64, u64, f64, f64, P(f64), P(f64)]),
        "orc_camera_build": (i32, [u64, f64, D3, D3, D3, f64, f64, f64, f64, u64, u64, P(Camera)]),
        "orc_camera_legacy": (None, [u64, f64, i32, P(Camera)]),
        "orc_render_reference": (i32, [P(Camera), P(Sphere), u64, vp, P(C.c_uint8), P(f64), P(Stats)]),
        "orc_render_philox64": (i32, [P(Camera), P(Sphere), u64, u64, i32, P(C.c_uint8), P(f64), P(Stats)]),
        "orc_render_legacy": (i32, [P(Camera), P(Sphere), u64, P(C.c_uint8), P(f64), P(Stats)]),
        "orc_write_ppm": (i32, [C.c_char_p, u64, u64, P(C.c_uint8)]),
        "orc_write_ppm_ascii": (i32, [C.c_char_p, u64, u64, P(C.c_uint8)]),
        "orc_to_rgb": (None, [P(f64), u64, P(C.c_uint8)]),
        "orc_linear_to_gamma": (f64, [f64]),
        "orc_sphere_hit": (None, [P(Sphere), D3, D3, f64, f64, P(Hit)]),
        "orc_list_hit": (None, [P(Sphere), u64, D3, D3, f64, f64, P(Hit)]),
        "orc_scatter": (None, [P(Sphere), D3, D3, P(Hit), vp, P(Scatter)]),
        "orc_vec_unit": (None, [D3, D3]),
        "orc_vec_cross": (None, [D3, D3, D3]),
        "orc_vec_dot": (f64, [D3, D3]),
        "orc_vec_len": (f64, [D3]),
        "orc_vec_near_zero": (i32, [D3]),
        "orc_vec_reflect": (None, [D3, D3, D3]),
        "orc_vec_refract": (None, [D3, D3, f64, D3]),
        "orc_vec_div_scalar": (None, [D3, f64, D3]),
        "orc_random_unit_vec": (None, [vp, D3]),
        "orc_random_in_unit_disk": (None, [vp, D3]),
        "orc_random_double_range": (f64, [f64, f64, vp]),
        "orc_interval_surrounds": (i32, [f64, f64, f64]),
        "orc_interval_contains": (i32, [f64, f64, f64]),
        "orc_interval_clamp": (f64, [f64, f64, f64]),
        "orc_reflectance": (f64, [f64, f64]),
        "orc_philox": (None, [P(C.c_uint32), P(C.c_uint32), P(C.c_uint32)]),
        "orc_hardware_threads": (i32, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    # optional: the f32 device mirror (oracle/rtz_mirror.cpp)
    if hasattr(lib, "orc_render_mirror"):
        lib.orc_render_mirror.restype = i32
        lib.orc_render_mirror.argtypes = [P(Camera), P(Sphere), u64, u64, i32, P(Shard), P(C.c_uint8), P(f64), P(Stats)]
    if hasattr(lib, "orc_mirror_camera_ray"):
        lib.orc_mirror_camera_ray.restype = None
        lib.orc_mirror_camera_ray.argtypes = [P(Camera), u64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                              P(C.c_float), P(C.c_float), P(C.c_float)]
    _oracle = lib
    return lib


# --------------------------------------------------------------------------------------------
# small helpers shared by tests
# --------------------------------------------------------------------------------------------
def read_ppm(path) -> tuple[int, int, bytes, bytes]:
    """Return (w, h, pixel bytes, whole file bytes) of a binary P6 file."""
    raw = Path(path).read_bytes()
    assert raw[:3] == b"P6\n", raw[:8]
    parts = raw.split(b"\n", 3)
    w, h = (int(x) for x in parts[1].split())
    assert parts[2] == b"255"
    body = parts[3]
    return w, h, body[: 3 * w * h], raw


def final_scene(seed: int):
    """Scene.init(seed) + generateWorld(): returns (prng handle, Sphere array, n)."""
    o = oracle()
    prng = o.orc_prng_new(seed)
    buf = (Sphere * 600)()
    n = o.orc_generate_world(prng, buf, 600)
    return prng, buf, int(n)


def chapter13_scene():
    o = oracle()
    buf = (Sphere * 5)()
    n = o.orc_generate_chapter13(buf, 5)
    return buf, int(n)


def build_camera(width, aspect, look_from, look_at, vfov, *, vup=(0, 1, 0), viewport_focus=10.0, focus=10.0,
                 defocus=0.0, spp=100, bounce_max=50, seed=None) -> Camera:
    cam = Camera()
    rc = oracle().orc_camera_build(width, aspect, d3(look_from), d3(look_at), d3(vup), vfov, viewport_focus, focus,
                                   defocus, spp, bounce_max, C.byref(cam))
    assert rc == 0
    if seed is not None:
        cam.seed, cam.has_seed = seed, 1
    return cam


def main_camera(width, spp, seed=None) -> Camera:
    """The camera of reference src/main.zig:23-31 (setDefocusAngle(.6), setFocusDist(10), setViewport(...))."""
    return build_camera(width, 16.0 / 9.0, (13, 2, 3), (0, 0, 0), 20, viewport_focus=10.0, focus=10.0, defocus=0.6,
                        spp=spp, seed=seed)
