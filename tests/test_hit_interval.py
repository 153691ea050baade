"""The hit interval (t_min, t_max) across its range, ray by ray and in whole renders.

The other parity tests hold the interval at the book's (1e-3, inf), with a finite t_max only in probe calls.  Yet
Scene.interval is the caller's: the early chapters of the book use (0, inf).  Two exactness arguments of the sweeps
depend on it (DESIGN.md §4):
  * the culled sweep tests its block boxes over [0, closest], a superset of (t_min |d|, closest) only for t_min >= 0;
  * the wavefront sweeps drop the sphere a ray leaves, whose roots with the exact c = 0 are h -/+ |h| <= 0.  The
    roots are formed from |h| itself: sqrt(h * h) exceeds |h| where h * h underflows (|h| < 2^-63), and at t_min = 0
    it put a root of a leaving ray at h + sqrt(h * h) > 0, a re-hit the wavefront sweeps never report.
So t_min < 0 is refused by every render entry point and by the sweep probe (-0.0 is accepted and renders as 0.0
does); the one-ray hit probe, HittableList.hit for the reference's unit tests, keeps taking any interval.  Every sweep
must equal the mirror bit for bit at every accepted interval: t_min 0, -0.0, 1e-30, 1e-3, 0.75 against t_max inf, 20, 1, 0, and an
interval with t_max < t_min.  The new family of rays ("underflowing self roots") starts on a sphere at c +- r e_a and
leaves it, outwards or inwards, with a direction whose a component is +-(1 .. 2) 2^e, e = -90 .. -56.
"""
import ctypes as C

import numpy as np
import pytest

import rtzlib as R
from test_block_regroup import _scene as _tie_scene
from test_guides import _check as _check_guides
from test_guides import guide_mirror  # noqa: F401  (the fixture)
from test_ray_parity import (CH13_CAMERAS, HIT, RAY, _camera_rays, _check, _mirror_hits, _moved_camera, _ptr,
                             _secondary, _translated)
from test_sweep_parity import NAMES, _c3_rays, _pad128, _same, _scene, _self_family, _tie_rays

TMINS = [0.0, -0.0, 1e-30, 1e-3, 0.75]
TMAXS = [np.inf, 20.0, 1.0, 0.0]
GRID = [(a, b) for a in TMINS for b in TMAXS] + [(0.75, 0.5)]
U8 = C.POINTER(C.c_uint8)
F64 = C.POINTER(C.c_double)


# ------------------------------------------------------------------------------------------------ rays and scenes
def _underflow_family(sp, n, rng, count=16, per=3):
    """Rays from c + s r e_a (rounded to f32; s = +-1, every axis a) of `count` spheres, with self set, whose a
    component is +-(1 .. 2) 2^e (e = -90 .. -56, `per` draws each) and whose other two components are a random unit
    pair: |h| is about r 2^e.  Returns the rays and whether each leaves its sphere outwards."""
    idx = rng.choice(n, size=min(n, count), replace=False)
    o, d, self_, out = [], [], [], []
    for i in idx:
        c, r = np.array(sp[i].center[:]), float(np.float32(sp[i].radius))
        for a in range(3):
            j, k = [x for x in range(3) if x != a]
            for s in (-1.0, 1.0):
                oo = np.float32(c).astype(float)
                oo[a] = float(np.float32(c[a] + s * r))
                for outwards in (True, False):
                    for _ in range(per):
                        e = int(rng.integers(-90, -55))
                        dd = np.zeros(3)
                        dd[a] = (s if outwards else -s) * rng.uniform(1.0, 2.0) * 2.0 ** e
                        phi = rng.uniform(0, 2 * np.pi)
                        dd[j], dd[k] = np.cos(phi), np.sin(phi)
                        o.append(oo), d.append(dd), self_.append(i), out.append(outwards)
    rays = np.zeros(len(o), RAY)
    rays["orig"], rays["dir"], rays["self"] = np.float32(o), np.float32(d), self_
    return rays, np.array(out)


def _chapter13(T=(0.0, 0.0, 0.0)):
    sp, n = R.chapter13_scene()
    return _translated(sp, n, np.array(T)), n


def _scenes(orc):
    """(label, spheres, n, translation) of the CPU checks: chapter 13, the final scene at 0 and moved by 10^3, a
    sweep scene."""
    return [("ch13", *_chapter13(), (0.0, 0.0, 0.0)),
            ("final", _scene(orc, 485), 485, (0.0, 0.0, 0.0)),
            ("final T=1e3", _scene(orc, 485, (1e3, 1e3, 1e3)), 485, (1e3, 1e3, 1e3)),
            ("sweep-128", _scene(orc, 128), 128, (0.0, 0.0, 0.0))]


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("tmin", [0.0, -0.0, 1e-30, 1e-3])
def test_a_ray_leaving_its_sphere_never_hits_it(orc, tmin):
    """The mirror on the underflow family: an outward ray never returns the sphere it leaves, with the candidate gate
    on or off."""
    rng = np.random.default_rng(29)
    for label, sp, n, _ in _scenes(orc):
        rays, out = _underflow_family(sp, n, rng)
        got = _mirror_hits(orc, sp, n, rays, tmin)
        nogate = _mirror_hits(orc, sp, n, rays, tmin, gate=False)
        assert got.tobytes() == nogate.tobytes(), label
        back = np.flatnonzero(out & (got["best"] == rays["self"]))
        assert len(back) == 0, (label, len(back), rays[back[:4]], got[back[:4]])


# explained disagreements with the f64 reference, on these seeds at most 27 % (underflow, final scene, (0, inf)),
# 44 % (self, 128 spheres, (0, 1)) and none (camera): at t_min = 0 the reference re-hits the sphere a ray leaves at
# its f64 near root, the f32 origin's offset from the surface, which _classify's self_hit explains
BOUNDS = {"underflow": 0.35, "self": 0.55, "camera": 0.01}


@pytest.mark.parametrize("tmin,tmax", GRID, ids=[f"{a!r}-{b!r}" for a, b in GRID])
def test_interval_grid_stays_in_the_error_model(orc, tmin, tmax):
    """The mirror at every interval of the grid against the f64 reference: no unexplained disagreement, roots within
    their error bounds, explained ones within the measured rates, the gate only filters (_check)."""
    rng = np.random.default_rng(31)
    for label, sp, n, T in _scenes(orc):
        under, _ = _underflow_family(sp, n, rng, count=8, per=2)
        _check(orc, sp, n, under, tmin, tmax, BOUNDS["underflow"], f"{label} underflow")
        if n == 5:
            cam = _camera_rays(orc, _moved_camera(160, np.array(T), **CH13_CAMERAS["ch12"]), 7, 60, 4, rng)
        else:
            cam = _c3_rays(orc, T, rng, pixels=60)
        _check(orc, sp, n, cam, tmin, tmax, BOUNDS["camera"], f"{label} camera")
        _check(orc, sp, n, _self_family(orc, sp, n, cam, rng), tmin, tmax, BOUNDS["self"], f"{label} self")


def _camera(**kw):
    return R.build_camera(64, 16.0 / 9.0, (-2, 2, 1), (0, 0, -1), 20, spp=2, seed=1, **kw)


def test_negative_t_min_is_refused_before_any_device_work(pkg):
    """t_min = -1e-3 and -1e-300 (and a NaN t_max) are refused with RTZ_ERR_BAD_ARG by the renders and the sweep
    probe, which check the camera or the interval before they touch a device."""
    l = pkg.lib()
    sp, n = R.chapter13_scene()
    P = C.POINTER(pkg.rtz_sphere)
    rays = np.zeros(128, RAY)
    rays["dir"][:, 2] = -1.0
    rays["self"] = -1
    out = np.zeros(128, HIT)
    o3 = np.zeros(3, np.float32)
    for bad in (-1e-3, -1e-300):
        cam = _camera()
        cam.t_min = bad
        pc = C.cast(C.pointer(cam), C.POINTER(pkg.rtz_camera))
        rgb = np.zeros(cam.width * cam.height * 3, np.uint8)
        lin = np.zeros(cam.width * cam.height * 3)
        st = pkg.rtz_stats()
        assert l.rtz_render(pc, C.cast(sp, P), n, rgb.ctypes.data_as(U8), C.byref(st)) == 1, bad
        assert l.rtz_render_linear(pc, C.cast(sp, P), n, rgb.ctypes.data_as(U8), lin.ctypes.data_as(F64),
                                   C.byref(st)) == 1, bad
        assert b"t_min" in l.rtz_last_error()
        for kind in range(len(NAMES)):
            assert l.rtz_probe_sweeps(C.cast(sp, P), n, _ptr(rays), 128, bad, np.inf, kind, 16, _ptr(out)) == 1, kind
        assert b"t_min" in l.rtz_last_error()
        assert l.rtz_probe_camera_ray(pc, 0, 0, 0, 1, o3.ctypes.data_as(C.POINTER(C.c_float)),
                                      o3.ctypes.data_as(C.POINTER(C.c_float)), None) == 1
        for call in (lambda: pkg.render_host(cam, sp, n), lambda: pkg.render_host_denoised(cam, sp, n),
                     lambda: pkg.render_host_multi(cam, sp, n, num_gpus=1)):
            with pytest.raises(pkg.RtzError) as e:
                call()
            assert e.value.status == 1, bad
    cam = _camera()
    cam.t_max = float("nan")
    rgb = np.zeros(cam.width * cam.height * 3, np.uint8)
    assert l.rtz_render(C.cast(C.pointer(cam), C.POINTER(pkg.rtz_camera)), C.cast(sp, P), n, rgb.ctypes.data_as(U8),
                        None) == 1


# ------------------------------------------------------------------------------------------------ GPU: ray by ray
def _gpu_scene(orc, n):
    if n == 5:
        return _chapter13()[0]
    return _scene(orc, n)


def _families_for(orc, sp, n, rng):
    """(label, rays) of every family on one scene: underflowing self roots, camera, secondary, self."""
    if n == 5:
        cam = _camera_rays(orc, _moved_camera(160, np.zeros(3), **CH13_CAMERAS["ch12"]), 7, 64, 4, rng)
    else:
        cam = _c3_rays(orc, (0.0, 0.0, 0.0), rng, pixels=48)
    under, _ = _underflow_family(sp, n, rng, count=12, per=2)
    return [("underflow", under), ("camera", cam), ("secondary", _secondary(orc, sp, n, cam, rng)),
            ("self", _self_family(orc, sp, n, cam, rng))]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5, 64, 128, 200, 485, 512, 4096, 8192])
def test_interval_grid_in_every_sweep(pkg, gpu, orc, n):
    """Every sweep that serves the scene size (WAVE4 included up to 512 spheres; the culled sweep at split_max 0,
    16 and 64) equals the mirror bit for bit on every family at every interval of the grid."""
    rng = np.random.default_rng(n + 5)
    sp = _gpu_scene(orc, n)
    rays = _pad128(np.concatenate([r for _, r in _families_for(orc, sp, n, rng)]))
    bad = []
    for tmin, tmax in GRID:
        bad += _same(pkg, orc, sp, n, rays, f"n={n} ({tmin!r}, {tmax!r})", tmin=tmin, tmax=tmax, splits=(0, 16, 64))
    assert not bad, "\n".join(bad[:20])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5, 485])
def test_hit_probe_takes_any_interval(pkg, gpu, orc, n):
    """rtz_probe_hits is HittableList.hit for the reference's unit tests, which take Interval(-6, 6): it accepts a
    negative t_min (its scalar sweep has no t_min >= 0 shortcut) and equals the mirror bit for bit there too, as on
    the grid."""
    rng = np.random.default_rng(n + 17)
    sp = _gpu_scene(orc, n)
    rays = np.concatenate([r for _, r in _families_for(orc, sp, n, rng)])
    P = C.POINTER(pkg.rtz_sphere)
    bad = []
    for tmin, tmax in [(-6.0, 6.0), (-1e-3, np.inf), (-1e-300, 20.0), (-0.0, 1.0)] + GRID:
        want = _mirror_hits(orc, sp, n, rays, tmin, tmax)
        got = np.zeros(len(rays), HIT)
        assert pkg.lib().rtz_probe_hits(C.cast(sp, P), n, _ptr(rays), len(rays), tmin, tmax, _ptr(got)) == 0
        if got.tobytes() != want.tobytes():
            bad.append(f"({tmin!r}, {tmax!r}): {int((got != want).sum())} of {len(rays)} rays")
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_interval_grid_on_exact_ties(pkg, gpu, orc):
    rng = np.random.default_rng(8)
    bad = []
    for ground_first in (True, False):
        spt, pairs = _tie_scene(ground_first)
        arr = R.sphere_array(spt)
        rays = _tie_rays(rng, pairs)
        for tmin, tmax in GRID:
            bad += _same(pkg, orc, arr, len(spt), rays, f"ties {ground_first} ({tmin!r}, {tmax!r})", tmin=tmin,
                         tmax=tmax, splits=(0, 16, 64))
    assert not bad, "\n".join(bad[:20])


# ------------------------------------------------------------------------------------------------ GPU: renders
INTERVALS = [(0.0, np.inf), (1e-3, 3.0), (0.5, np.inf), (1e-3, 0.0), (0.0, 2.5)]


def _mirror(orc, cam, sp, n, shard=None):
    pixels = cam.width * cam.height
    if shard is not None:
        tiles = -(-cam.width // shard.tile_w) * -(-cam.height // shard.tile_h)
        pixels = -(-tiles // shard.world) * shard.tile_w * shard.tile_h
    rgb, lin, st = np.zeros((pixels, 3), np.uint8), np.zeros((pixels, 3)), R.Stats()
    sh = C.byref(R.Shard(shard.rank, shard.world, shard.tile_w, shard.tile_h)) if shard is not None else None
    assert orc.orc_render_mirror(C.byref(cam), sp, n, cam.seed, max(1, orc.orc_hardware_threads()), sh,
                                 rgb.ctypes.data_as(U8), lin.ctypes.data_as(F64), C.byref(st)) == 0
    return rgb, lin, st


def _stats(st):
    return st.samples, st.segments, st.depth_capped, st.absorbed, st.nan_samples


def _render_cases():
    """(scene size, environment, BVH too): each size's default kernel, the kernel variants on 128 spheres."""
    c = [(5, {}, True), (64, {}, False), (128, {}, True), (513, {}, False), (4096, {}, False), (8192, {}, False)]
    c += [(485, {"RTZ_SPLIT": s}, s == "16") for s in ("0", "16", "64")]
    c += [(128, {"RTZ_VARIANT": v}, False) for v in ("8", "11", "12", "4")]
    c += [(5, {"RTZ_DRAIN": "0"}, False), (128, {"RTZ_DRAIN": "0"}, False), (485, {"RTZ_DRAIN": "0"}, False)]
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("n,env,bvh", _render_cases(),
                         ids=[f"{n}-{','.join(f'{k}={v}' for k, v in e.items()) or 'default'}"
                              for n, e, _ in _render_cases()])
def test_renders_across_the_interval(pkg, orc, monkeypatch, n, env, bvh):
    """A small frame at each interval through the kernel the scene size or the environment selects (the BVH mode
    beside it where marked, one shard of three on the default kernels): bytes, f32 linear colour and counters,
    NaN samples included, equal the mirror's."""
    sp = _gpu_scene(orc, n)
    if n == 5:
        cam = R.build_camera(96, 16.0 / 9.0, (-2, 2, 1), (0, 0, -1), 20, spp=16, seed=0x1A7)
    else:
        cam = R.build_camera(96 if n < 4096 else 64, 16.0 / 9.0, (13, 2, 3), (0, 0, 0), 20, defocus=0.6, spp=8,
                             seed=0x1A7)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    r = pkg.Renderer(0)
    try:
        r.upload(sp, n)
        for tmin, tmax in INTERVALS:
            cam.t_min, cam.t_max = tmin, tmax
            cam.mode = R.MODE_PATH
            mrgb, mlin, mst = _mirror(orc, cam, sp, n)
            for mode in (R.MODE_PATH, R.MODE_PATH_BVH) if bvh else (R.MODE_PATH,):
                cam.mode = mode
                img, lin32, st = r.render_linear(cam)
                label = (env, mode, tmin, tmax)
                assert np.array_equal(img.cpu().numpy().reshape(-1, 3), mrgb), label
                assert np.array_equal(lin32.cpu().numpy().reshape(-1, 3), mlin.astype(np.float32)), label
                assert _stats(st) == _stats(mst), (label, _stats(st), _stats(mst))
            cam.mode = R.MODE_PATH
            if not env or "RTZ_SPLIT" in env:
                shard = pkg.rtz_shard(1, 3, 7, 5)
                srgb, slin, sst = _mirror(orc, cam, sp, n, shard)
                img, lin32, st = r.render_linear(cam, shard)
                assert np.array_equal(img.cpu().numpy().reshape(-1, 3), srgb), (env, "shard", tmin, tmax)
                assert np.array_equal(lin32.cpu().numpy().reshape(-1, 3), slin.astype(np.float32)), (env, tmin, tmax)
                assert _stats(st) == _stats(sst), (env, "shard", tmin, tmax)
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("interval", [(0.0, np.inf), (0.5, 3.0)], ids=["0-inf", "0.5-3"])
def test_guides_across_the_interval(gpu, guide_mirror, orc, interval):  # noqa: F811
    for sp, n, cam in ((*R.chapter13_scene(), R.build_camera(160, 16.0 / 9.0, (-2, 2, 1), (0, 0, -1), 20, spp=8,
                                                            seed=0xDEADBEEF)),
                       (_scene(orc, 485), 485, R.build_camera(96, 16.0 / 9.0, (13, 2, 3), (0, 0, 0), 20, defocus=0.6,
                                                              spp=8, seed=0xDEADBEEF))):
        cam.t_min, cam.t_max = interval
        _check_guides(gpu, guide_mirror, cam, sp, n, 3)


@pytest.mark.gpu
def test_negative_t_min_is_refused_everywhere_and_minus_zero_is_zero(pkg, gpu):
    """The device-side entry points refuse t_min < 0 (the resident renders, guides, the multi-GPU renderer) and leave
    the installed scene as it was; t_min = -0.0 renders the bytes of 0.0 in every call."""
    sp, n = R.chapter13_scene()
    gpu.upload(sp, n)
    multi = pkg.MultiRenderer(1)
    multi.upload(sp, n)
    try:
        zero = _camera()
        zero.t_min = 0.0
        good, _ = pkg.render_host(zero, sp, n)
        for bad in (-1e-3, -1e-300):
            cam = _camera()
            cam.t_min = bad
            for call in (lambda: gpu.render(cam), lambda: gpu.render_linear(cam), lambda: gpu.render_guides(cam, 2),
                         lambda: multi.render(cam), lambda: gpu.render(cam, pkg.rtz_shard(1, 3, 7, 5))):
                with pytest.raises(pkg.RtzError) as e:
                    call()
                assert e.value.status == 1, bad
        neg = _camera()
        neg.t_min = -0.0
        assert np.array_equal(pkg.render_host(neg, sp, n)[0], good)
        assert np.array_equal(gpu.render(neg)[0].cpu().numpy(), good)
        assert np.array_equal(gpu.render(zero)[0].cpu().numpy(), good)
        assert np.array_equal(multi.render(neg)[0], good)
        alb0, nrm0, _ = gpu.render_guides(zero, 2)
        alb1, nrm1, _ = gpu.render_guides(neg, 2)
        assert np.array_equal(alb0.cpu().numpy(), alb1.cpu().numpy())
        assert np.array_equal(nrm0.cpu().numpy(), nrm1.cpu().numpy())
        assert np.array_equal(pkg.render_host_denoised(neg, sp, n)[0], pkg.render_host_denoised(zero, sp, n)[0])
    finally:
        multi.close()
