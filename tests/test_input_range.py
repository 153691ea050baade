"""The render at the edges of its input range.

Materials.  The scenes of the other parity tests have the book's materials (albedo in [0, 1), fuzz <= 0.5, ior 1.5
or 1/1.5).  Here the edge set goes to the ends: albedo exactly 0 and 1 (and -0.0), fuzz 4 and 1 (metal rays that
scatter into the surface are absorbed: 5 to 12 % of the samples, against 0.2 % in the book's scenes), glass of
ior 0.5 holding glass of ior 1.0.  The mirror must stay within the statistical gates of the f64 restatement, and
the device must equal the mirror bit for bit in every trace kernel.  Albedos outside [0, 1] are refused at upload
(include/rtz.h): the fixed-point pixel sums clamp each sample at 0, where the reference clamps the mean.

Sample bookkeeping.  In an empty world the blue channel of every sample is exactly 1.0f (the sky's
fmaf(a, 1, 1 - a) rounds back to 1), so a pixel's blue sum is (samples traced for it) x 2^32 and its f64 linear
value is exactly 1.0, for every spp up to 2^31 - 1.  A chunk of samples lost, doubled or credited to the wrong
pixel moves that pixel's blue value off 1.0.  This is checked at the top of the sample range (a 1x1 frame at
2^31 - 1 spp), on both sides of the 2^32-chunk limit of the wavefront kernels' chunk bookkeeping, and on the C4
frame, whole and in shards.
"""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import rtzlib as R

ROOT = Path(__file__).resolve().parent.parent
L, M, D = R.MAT_LAMBERTIAN, R.MAT_METAL, R.MAT_DIELECTRIC

EDGE = [R.make_sphere((0, -100.5, -1), 100, L, (1.0, 1.0, 1.0)),
        R.make_sphere((0, 0, -1.2), 0.5, L, (1.0, 0.0, -0.0)),
        R.make_sphere((-1, 0, -1), 0.5, D, ior=0.5),
        R.make_sphere((-1, 0, -1), 0.4, D, ior=1.0),
        R.make_sphere((1, 0, -1), 0.5, M, (1.0, 1.0, 1.0), fuzz=4.0),
        R.make_sphere((0.4, -0.35, -0.6), 0.15, M, (0.0, 1.0, 0.5), fuzz=1.0),
        R.make_sphere((-0.4, -0.35, -0.6), 0.15, M, (0.9, 0.9, 0.9), fuzz=0.0)]
VIEWS = {"ch12": dict(look_from=(-2, 2, 1), look_at=(0, 0, -1), vfov=20),
         "wide": dict(look_from=(0, 0, 0.5), look_at=(0, 0, -1), vfov=90)}
U8 = C.POINTER(C.c_uint8)
F64 = C.POINTER(C.c_double)


def _threads(orc):
    return max(1, orc.orc_hardware_threads())


def _mirror(orc, cam, sp, n, seed, linear=True):
    rgb = np.zeros((cam.height * cam.width, 3), np.uint8)
    lin = np.zeros((cam.height * cam.width, 3)) if linear else None
    st = R.Stats()
    assert orc.orc_render_mirror(C.byref(cam), sp, n, seed, _threads(orc), None, rgb.ctypes.data_as(U8),
                                 lin.ctypes.data_as(F64) if linear else None, C.byref(st)) == 0
    return rgb, lin, st


def _reference(orc, cam, sp, n, seed):
    rgb = np.zeros((cam.height * cam.width, 3), np.uint8)
    st = R.Stats()
    assert orc.orc_render_philox64(C.byref(cam), sp, n, seed, _threads(orc), rgb.ctypes.data_as(U8), None,
                                   C.byref(st)) == 0
    return rgb, st


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("spp", [64, 256])
@pytest.mark.parametrize("view", list(VIEWS))
def test_edge_materials_mirror_vs_f64(orc, view, spp):
    """The edge set: the f32 mirror (the device's bit-exact twin) against the f64 restatement of the reference,
    with the gates of test_oracle_stat.py (RMSE within 1.25x the reference's seed-to-seed floor, |bias| <= 0.25
    level) and the path statistics: segments per sample within 1 %, the absorbed fraction within 2 %."""
    sp = R.sphere_array(EDGE)
    cam = R.build_camera(160, 16.0 / 9.0, spp=spp, seed=0x5EED, **VIEWS[view])
    m, _, mst = _mirror(orc, cam, sp, len(EDGE), 0x5EED, linear=False)
    a, ast = _reference(orc, cam, sp, len(EDGE), 1)
    b, _ = _reference(orc, cam, sp, len(EDGE), 2)
    m, a, b = (x.astype(float) for x in (m, a, b))
    floor, err = np.sqrt(np.mean((a - b) ** 2)), np.sqrt(np.mean((m - a) ** 2))
    bias = (m - a).mean(axis=0)
    assert err <= 1.25 * floor, (err, floor)
    assert np.abs(bias).max() <= 0.25, bias
    assert mst.samples == ast.samples == cam.width * cam.height * spp
    seg_m, seg_a = mst.segments / mst.samples, ast.segments / ast.samples
    assert abs(seg_m - seg_a) <= 0.01 * seg_a, (seg_m, seg_a)
    abs_m, abs_a = mst.absorbed / mst.samples, ast.absorbed / ast.samples
    assert abs_a > 0.02 and abs(abs_m - abs_a) <= 0.02 * abs_a, (abs_m, abs_a)
    assert mst.depth_capped / mst.samples <= 5e-4 and ast.depth_capped / ast.samples <= 5e-4


BLUE_VIEWS = {"170": dict(vfov=170), "90-defocus": dict(vfov=90, defocus=10.0), "20": dict(vfov=20)}


@pytest.mark.parametrize("spp", [1, 3, 1000])
@pytest.mark.parametrize("view", list(BLUE_VIEWS))
def test_empty_world_blue_is_exactly_one_on_the_mirror(orc, view, spp):
    """The known answer the GPU bookkeeping tests below rely on, on the mirror: every pixel's blue linear value is
    exactly 1.0, red and green lie in [0, 1], one segment per sample."""
    cam = R.build_camera(64, 16.0 / 9.0, (0, 0, 0), (0, 0, -1), spp=spp, seed=0xB1E, **BLUE_VIEWS[view])
    _, lin, st = _mirror(orc, cam, (R.Sphere * 1)(), 0, 0xB1E)
    assert (lin[:, 2] == 1.0).all(), np.unique(lin[:, 2])
    assert lin[:, :2].min() >= 0.0 and lin[:, :2].max() <= 1.0
    assert st.samples == st.segments == cam.width * cam.height * spp


# ------------------------------------------------------------------------------------------------ GPU: refusals
BAD_ALBEDO = [-1e-30, -0.5, 1.0 + 2.0 ** -52, 1.5, 4.0]
OK_ALBEDO = [0.0, -0.0, 1.0]


def _with_albedo(sp, n, i, channel, value):
    arr = (R.Sphere * n)()
    for k in range(n):
        arr[k] = sp[k]
    alb = list(arr[i].albedo)
    alb[channel] = value
    arr[i].albedo = R.d3(alb)
    return arr


@pytest.mark.gpu
def test_albedo_outside_unit_interval_is_refused(pkg, gpu):
    """Every entry point that takes spheres refuses a lambertian or metal albedo component outside [0, 1] with
    RTZ_ERR_BAD_ARG and names the sphere; a refused upload leaves the installed scene as it was.  0, -0.0 and 1
    are accepted (-0.0 renders as 0 does), and so is any dielectric albedo, which nothing reads."""
    sp, n = R.chapter13_scene()
    cam = R.build_camera(64, 16.0 / 9.0, (-2, 2, 1), (0, 0, -1), 20, spp=2, seed=1)
    good, _ = pkg.render_host(cam, sp, n)
    gpu.upload(sp, n)
    multi = pkg.MultiRenderer(1)
    multi.upload(sp, n)
    l = pkg.lib()
    P = C.POINTER(pkg.rtz_sphere)
    hit, scat = pkg.binding.rtz_hit(), pkg.binding.rtz_scatter()
    try:
        for i in (1, 4):   # the lambertian centre sphere, the metal right sphere
            assert sp[i].mat_type == (L if i == 1 else M)
            for channel in range(3):
                for value in BAD_ALBEDO:
                    arr = _with_albedo(sp, n, i, channel, value)
                    label = (i, channel, value)
                    calls = [lambda: pkg.render_host(cam, arr, n), lambda: gpu.upload(arr, n),
                             lambda: pkg.render_host_denoised(cam, arr, n), lambda: multi.upload(arr, n),
                             lambda: pkg.render_host_multi(cam, arr, n, num_gpus=1)]
                    for call in calls:
                        with pytest.raises(pkg.RtzError) as e:
                            call()
                        assert e.value.status == 1, label
                        assert f"sphere {i}: albedo[{channel}]" in str(e.value), (label, str(e.value))
                    assert l.rtz_probe_hit(C.cast(arr, P), n, R.d3((0, 0, 0)), R.d3((0, 0, -1)), 1e-3, np.inf,
                                           C.byref(hit)) == 1, label
                    assert l.rtz_probe_scatter(C.cast(arr, P), n, i, R.d3((0, 0, 0)), R.d3((0, 0, -1)), 1, 0, 0, 0,
                                               C.byref(scat)) == 1, label
                    img, _ = gpu.render(cam)
                    assert np.array_equal(img.cpu().numpy(), good), label
                    mimg, _ = multi.render(cam)
                    assert np.array_equal(mimg, good), label
                imgs = []
                for value in OK_ALBEDO:
                    arr = _with_albedo(sp, n, i, channel, value)
                    rgb, st = pkg.render_host(cam, arr, n)
                    assert st.samples == cam.width * cam.height * 2
                    imgs.append(rgb)
                    gpu.upload(arr, n)
                    multi.upload(arr, n)
                assert np.array_equal(imgs[0], imgs[1]), (i, channel)   # +0.0 and -0.0
                gpu.upload(sp, n)
                multi.upload(sp, n)
        glass = sp
        for i in (2, 3):
            glass = _with_albedo(glass, n, i, 0, 7.0)
            glass = _with_albedo(glass, n, i, 1, 7.0)
            glass = _with_albedo(glass, n, i, 2, 7.0)
        rgb, _ = pkg.render_host(cam, glass, n)
        assert np.array_equal(rgb, good)
    finally:
        multi.close()


# ------------------------------------------------------------------------------------------------ GPU: edge materials
def _sweep_scene(orc, n):
    prng = orc.orc_prng_new(0xDEADBEEF)
    sp = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, sp) == n
    orc.orc_prng_free(prng)
    return sp


def _edge_materials(sp, n):
    """Sphere i takes the material of edge-set entry i mod 7, geometry unchanged."""
    for i in range(n):
        e = EDGE[i % len(EDGE)]
        sp[i].mat_type, sp[i].albedo, sp[i].fuzz, sp[i].refraction_index = e.mat_type, e.albedo, e.fuzz, e.refraction_index
    return sp


@pytest.mark.gpu
@pytest.mark.parametrize("n_spheres", [7, 47, 207, 407, 607, 8192])
def test_edge_materials_equal_mirror_in_every_kernel(pkg, gpu, orc, monkeypatch, n_spheres):
    """The sweep scene with the edge set's materials, through every trace kernel that serves its size: 7 and 47
    spheres the wavefront kernels with the per-thread drain, 207 the four-path wavefront kernel with the per-warp
    drain, 407 the culled constant-bank kernel, 607 shared memory, 8192 global memory; RTZ_VARIANT=11 the lockstep
    kernels, RTZ_DRAIN=0 no drain.  Bytes, linear colour and counters equal the mirror's."""
    n = n_spheres
    sp = _edge_materials(_sweep_scene(orc, n), n)
    cam = R.build_camera(96 if n < 4096 else 64, 16.0 / 9.0, (13, 2, 3), (0, 0, 0), 20, defocus=0.6, spp=8,
                         seed=0x5EED)
    mrgb, mlin, mst = _mirror(orc, cam, sp, n, 0x5EED)
    want = (mst.samples, mst.segments, mst.depth_capped, mst.absorbed, 0)
    assert mst.absorbed > 0
    envs = [{}, {"RTZ_DRAIN": "0"}, {"RTZ_VARIANT": "11"}]
    if n <= 256:
        envs += [{"RTZ_VARIANT": "8"}, {"RTZ_VARIANT": "12"}]
    for env in envs:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        r = pkg.Renderer(0)
        try:
            r.upload(sp, n)
            for mode in (R.MODE_PATH, R.MODE_PATH_BVH) if not env else (R.MODE_PATH,):
                cam.mode = mode
                img, lin32, st = r.render_linear(cam)
                assert np.array_equal(img.cpu().numpy().reshape(-1, 3), mrgb), (env, mode)
                assert np.array_equal(lin32.cpu().numpy().reshape(-1, 3), mlin.astype(np.float32)), (env, mode)
                assert (st.samples, st.segments, st.depth_capped, st.absorbed, st.nan_samples) == want, (env, mode)
            cam.mode = R.MODE_PATH
        finally:
            r.close()
        for k in env:
            monkeypatch.delenv(k)
    for env in ({}, {"RTZ_DRAIN": "0"}):   # read per frame: the one-shot call's cached context follows it
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        rgb, st, lin = pkg.render_host(cam, sp, n, want_linear=True)
        assert np.array_equal(lin.reshape(-1, 3), mlin) and np.array_equal(rgb.reshape(-1, 3), mrgb), env
        assert (st.samples, st.segments, st.depth_capped, st.absorbed, st.nan_samples) == want, env
        for k in env:
            monkeypatch.delenv(k)


# ------------------------------------------------------------------------------------------------ GPU: bookkeeping
# rtz_render_linear (the f64 linear colour) renders on a context cached per process, and the kernel variant and the
# constant-bank switch are read when a context is created: each setting renders in a process of its own.
_WORKER = r'''
import importlib, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
pkg = importlib.import_module("raytracing-with-zig_b200")
raw = open(sys.argv[2], "rb").read()
size = len(bytes(pkg.rtz_camera()))
out = {}
for k in range(len(raw) // size):
    cam = pkg.rtz_camera.from_buffer_copy(raw[k * size:(k + 1) * size])
    rgb, st, lin = pkg.render_host(cam, (pkg.rtz_sphere * 1)(), 0, want_linear=True)
    out[f"lin{k}"] = lin
    out[f"st{k}"] = np.array([st.samples, st.segments, st.sphere_tests, st.depth_capped, st.absorbed, st.nan_samples],
                             np.uint64)
np.savez(sys.argv[3], **out)
'''


def _empty_world_in_fresh_process(tmp_path, env, cams):
    """Render each camera over an empty world through rtz_render_linear in a new process with `env` set; returns
    [(f64 linear [H, W, 3], (samples, segments, sphere_tests, depth_capped, absorbed, nan_samples))]."""
    cam_file, out_file = tmp_path / "cams.bin", tmp_path / "out.npz"
    cam_file.write_bytes(b"".join(bytes(c) for c in cams))
    r = subprocess.run([sys.executable, "-c", _WORKER, str(ROOT), str(cam_file), str(out_file)],
                       env=dict(os.environ, **env), capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, (env, r.stdout[-2000:] + r.stderr[-4000:])
    res = np.load(out_file)
    return [(res[f"lin{k}"], tuple(int(x) for x in res[f"st{k}"])) for k in range(len(cams))]


def _check_blue(lin, st, pixels, spp, label):
    assert st[:3] == (pixels * spp, pixels * spp, 0) and st[3:] == (0, 0, 0), (label, st)
    lin = lin.reshape(-1, 3)
    bad = np.flatnonzero(lin[:, 2] != 1.0)
    assert len(bad) == 0, (label, len(bad), bad[:8], lin[bad[:8], 2])
    assert lin[:, :2].min() >= 0.0 and lin[:, :2].max() <= 1.0, label


def _known_answer(cam):
    spp = cam.samples_per_pixel
    assert (float(spp * 2 ** 32) * 2.0 ** -32) * cam.pixel_samples_scale == 1.0


@pytest.mark.gpu
@pytest.mark.timeout(1200)
def test_samples_at_the_top_of_the_spp_range(pkg, tmp_path):
    """A 1x1 frame at the largest accepted spp, 2^31 - 1: the pixel's blue sum is (2^31 - 1) x 2^32, within 2^32 of
    2^63.  Through the default kernel (the wavefront kernel, drain on), the lockstep kernel (RTZ_VARIANT=11),
    without the drain, through the shared-memory kernel (RTZ_GEO_CONST=0) and through the BVH."""
    spp = 2 ** 31 - 1
    cam = R.build_camera(1, 1.0, (0, 0, 0), (0, 0, -1), 90, defocus=10.0, spp=spp, seed=0x70F)
    assert (cam.width, cam.height) == (1, 1)
    _known_answer(cam)
    bvh = R.Camera.from_buffer_copy(bytes(cam))
    bvh.mode = R.MODE_PATH_BVH
    for env, cams in (({}, [cam, bvh]), ({"RTZ_VARIANT": "11"}, [cam]), ({"RTZ_DRAIN": "0"}, [cam]),
                      ({"RTZ_GEO_CONST": "0"}, [cam])):
        for k, (lin, st) in enumerate(_empty_world_in_fresh_process(tmp_path, env, cams)):
            _check_blue(lin, st, 1, spp, (env, cams[k].mode))


@pytest.mark.gpu
@pytest.mark.timeout(1200)
def test_chunk_count_at_the_wavefront_limit(pkg, tmp_path):
    """RTZ_CHUNK=1 makes every sample a chunk.  255 x 1 pixels at 16 843 009 spp are 2^32 - 1 chunks, the largest
    frame the wavefront kernel takes (its chunk -> pixel division is a 64-bit reciprocal, exact below 2^32);
    256 x 1 at 2^24 spp are 2^32 chunks, the first frame handed to the lockstep kernel."""
    cams = [R.build_camera(255, 255.0, (0, 0, 0), (0, 0, -1), 170, spp=16843009, seed=0xC4A),
            R.build_camera(256, 256.0, (0, 0, 0), (0, 0, -1), 170, spp=2 ** 24, seed=0xC4B)]
    assert [(c.width, c.height, c.width * c.samples_per_pixel) for c in cams] == [(255, 1, 2 ** 32 - 1),
                                                                                  (256, 1, 2 ** 32)]
    for c in cams:
        _known_answer(c)
    for c, (lin, st) in zip(cams, _empty_world_in_fresh_process(tmp_path, {"RTZ_CHUNK": "1"}, cams)):
        _check_blue(lin, st, c.width, c.samples_per_pixel, c.width)


@pytest.mark.gpu
@pytest.mark.timeout(1200)
def test_c4_frame_bookkeeping_whole_and_sharded(pkg, gpu):
    """The C4 frame (3840 x 2160, 64 spp) over an empty world: whole through rtz_render_linear (f64), and as 8 shards
    of 4 x 4 tiles and 3 shards of 7 x 5 tiles through render_linear (f32).  Every shard slot of a pixel holds
    (float) of the whole frame's value, and tile padding reads 0."""
    spp = 64
    cam = R.build_camera(3840, 16.0 / 9.0, (0, 0, 0), (0, 0, -1), 90, spp=spp, seed=0xC4)
    W, H = cam.width, cam.height
    assert (W, H) == (3840, 2160)
    rgb, st, lin = pkg.render_host(cam, (R.Sphere * 1)(), 0, want_linear=True)
    _check_blue(lin, (st.samples, st.segments, st.sphere_tests, st.depth_capped, st.absorbed, st.nan_samples),
                W * H, spp, "whole")
    lin32 = lin.reshape(-1, 3).astype(np.float32)
    gpu.upload((R.Sphere * 1)(), 0)
    for world, (tw, th) in ((8, (4, 4)), (3, (7, 5))):
        per_rank, idx = pkg.tile_index_map(W, H, world, tw, th)
        idx = idx.reshape(-1)
        samples = 0
        for rank in range(world):
            img, part, pst = gpu.render_linear(cam, pkg.rtz_shard(rank, world, tw, th))
            part = part.cpu().numpy()
            assert part.shape == (per_rank, 3)
            mine = (idx >= rank * per_rank) & (idx < (rank + 1) * per_rank)
            slot = idx[mine] - rank * per_rank
            got = np.zeros_like(part)
            got[slot] = lin32[mine]
            assert np.array_equal(part, got), (world, rank, int((part != got).any(1).sum()))
            assert int(mine.sum()) * spp == pst.samples == pst.segments and pst.sphere_tests == 0, (world, rank)
            assert (pst.depth_capped, pst.absorbed, pst.nan_samples) == (0, 0, 0)
            samples += pst.samples
        assert samples == W * H * spp
