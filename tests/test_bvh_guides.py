"""First-hit guides of RTZ_MODE_PATH_BVH frames through the hierarchy (guides_kernel_bvh).

A BVH-mode frame of a scene beyond the constant bank (more than 512 padded spheres) finds its guide hits through the
BVH; every other frame keeps the brute-force guide kernels.  Either way the buffers are those of RTZ_MODE_PATH bit for
bit, because the traversal returns the (t, original index) minimum the brute-force sweep returns.  Which kernel ran
shows in the stats: the brute-force kernels report rays * n sphere tests, the BVH kernel the tests it made.
"""
import ctypes as C
import importlib
import re
import subprocess

import numpy as np
import pytest

import rtzlib as R

F32P = C.POINTER(C.c_float)
SEED = 0xDEADBEEF


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def guide_mirror(tmp_path_factory):
    """tests/guide_mirror.cpp built with the oracle's flags into a temporary directory."""
    so = tmp_path_factory.mktemp("bvh_guide_mirror") / "libguide_mirror.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-pthread",
                    "-shared", "-o", str(so), str(R.ROOT / "tests" / "guide_mirror.cpp")], check=True,
                   capture_output=True)
    lib = C.CDLL(str(so))
    lib.orc_mirror_guides.restype = C.c_int32
    lib.orc_mirror_guides.argtypes = [C.POINTER(R.Camera), C.POINTER(R.Sphere), C.c_uint64, C.c_uint64, C.c_uint64,
                                      F32P, F32P]
    return lib


def mirror_guides(lib, cam, sp, n, g):
    H, W = int(cam.height), int(cam.width)
    alb, nrm = np.zeros((H, W, 3), np.float32), np.zeros((H, W, 3), np.float32)
    assert lib.orc_mirror_guides(C.byref(cam), C.cast(sp, C.POINTER(R.Sphere)), n, cam.seed, g,
                                 alb.ctypes.data_as(F32P), nrm.ctypes.data_as(F32P)) == 0
    return alb, nrm


def sweep_scene(n):
    orc = R.oracle()
    prng = orc.orc_prng_new(7)
    buf = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, buf) == n
    orc.orc_prng_free(prng)
    return buf


def tie_scene():
    """600 sweep spheres, each followed by an exact copy of another colour and material: every hit is an exact tie in
    t, which the lower index (the original) must win."""
    sp = sweep_scene(600)
    out = []
    for s in sp:
        d = R.Sphere.from_buffer_copy(bytes(s))
        d.mat_type, d.albedo, d.fuzz = R.MAT_METAL, R.d3((0.11, 0.22, 0.33)), 0.0
        out += [s, d]
    return R.sphere_array(out), len(out)


def nested_scene():
    """Hollow glass: 200 glass shells of radius 0.2 with a glass sphere of radius 0.18 and a lambertian core of radius
    0.05 at the same centre, over the 600 sweep spheres."""
    rng = np.random.default_rng(11)
    out = list(sweep_scene(600))
    for _ in range(200):
        c = (rng.uniform(-11, 11), 0.2, rng.uniform(-11, 11))
        out += [R.make_sphere(c, 0.2, R.MAT_DIELECTRIC, ior=1.5), R.make_sphere(c, 0.18, R.MAT_DIELECTRIC, ior=1 / 1.5),
                R.make_sphere(c, 0.05, R.MAT_LAMBERTIAN, albedo=tuple(rng.uniform(0, 1, 3)))]
    return R.sphere_array(out), len(out)


def guides(gpu, cam, sp, n, g, mode, shard=None):
    c = R.Camera.from_buffer_copy(bytes(cam))
    c.mode = mode
    gpu.upload(sp, n)
    alb, nrm, st = gpu.render_guides(c, g, shard=shard)
    return alb.cpu().numpy(), nrm.cpu().numpy(), st


def check_bvh(gpu, cam, sp, n, g, mirror=None):
    """BVH-mode guides == RTZ_MODE_PATH guides (== the guide mirror when given), and the stats of each kernel."""
    a0, n0, st0 = guides(gpu, cam, sp, n, g, R.MODE_PATH)
    a1, n1, st1 = guides(gpu, cam, sp, n, g, R.MODE_PATH_BVH)
    assert np.array_equal(bits(a1), bits(a0)), f"{np.count_nonzero(bits(a1) != bits(a0))} albedo words differ"
    assert np.array_equal(bits(n1), bits(n0)), f"{np.count_nonzero(bits(n1) != bits(n0))} normal words differ"
    if mirror is not None:
        ma, mn = mirror_guides(mirror, cam, sp, n, g)
        assert np.array_equal(bits(a1), bits(ma)) and np.array_equal(bits(n1), bits(mn))
    rays = int(cam.width) * int(cam.height) * g
    assert (st0.samples, st0.segments, st0.sphere_tests, st0.kernel_launches) == (rays, rays, rays * n, 1)
    assert (st1.samples, st1.segments, st1.kernel_launches, st1.seed_used) == (rays, rays, 1, cam.seed)
    assert st1.trace_ms > 0 and st1.total_ms == st1.trace_ms
    return a1, n1, st1


# ------------------------------------------------------------------ no GPU
def test_bvh_guide_kernel_keeps_to_registers():
    """Codegen guard (no GPU needed): the BVH guide kernel does not spill (STL / LDL)."""
    lib = R.ROOT / "raytracing-with-zig_b200" / "csrc" / "librtz.so"
    importlib.import_module("raytracing-with-zig_b200.build").build_all()
    out = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    want = [k for k in body if "guides_kernel_bvh" in k]
    assert len(want) == 1, want
    assert not re.search(r"\b(STL|LDL)\b", "\n".join(body[want[0]]))


# ------------------------------------------------------------------ one GPU
@pytest.mark.gpu
@pytest.mark.parametrize("n,width", [(513, 48), (4096, 40), (16384, 32)])
@pytest.mark.parametrize("g", [1, 3, 64, 65])
def test_sweep_scene_bvh_guides(gpu, guide_mirror, n, width, g):
    sp = sweep_scene(n)
    cam = R.main_camera(width, 65, seed=0x5EED + n)
    affordable = n * width * width * 9 // 16 * g <= 4096 * 40 * 23 * 65
    _, nrm, st = check_bvh(gpu, cam, sp, n, g, guide_mirror if affordable else None)
    rays = int(cam.width) * int(cam.height) * g
    assert 0 < st.sphere_tests < rays * n
    assert (nrm == 0).all(-1).any() and (nrm != 0).any(-1).any()  # sky and spheres


@pytest.mark.gpu
@pytest.mark.parametrize("g", [1, 5])
def test_exact_ties_keep_the_lower_index(gpu, guide_mirror, g):
    sp, n = tie_scene()
    cam = R.main_camera(64, 8, seed=3)
    alb, _, _ = check_bvh(gpu, cam, sp, n, g, guide_mirror)
    assert not np.isclose(alb, np.float32(0.11)).any()  # no pixel took a copy


@pytest.mark.gpu
def test_nested_glass_spheres(gpu, guide_mirror):
    sp, n = nested_scene()
    cam = R.build_camera(80, 16.0 / 9.0, (13, 2, 3), (0, 0, 0), 30, spp=4, seed=9)
    alb, _, _ = check_bvh(gpu, cam, sp, n, 4, guide_mirror)
    assert (alb == 1).all(-1).any()  # glass is seen


@pytest.mark.gpu
def test_far_camera(gpu, guide_mirror):
    """A camera 10^5 from a scene of radius ~10 (10^4 scene radii): the traversal widens each box for the far origin
    (hit_box<true>)."""
    rng = np.random.default_rng(5)
    sp = R.sphere_array([R.make_sphere(rng.uniform(-8, 8, 3), rng.uniform(0.2, 1.5), int(rng.integers(0, 3)),
                                       albedo=tuple(rng.uniform(0, 1, 3)), fuzz=0.1, ior=1.5) for _ in range(700)])
    d = 1e5
    cam = R.build_camera(64, 16.0 / 9.0, (d * 0.6, d * 0.48, d * 0.64), (0, 0, 0), 0.014, viewport_focus=d, focus=d,
                         spp=4, seed=21)
    _, nrm, _ = check_bvh(gpu, cam, sp, 700, 4, guide_mirror)
    assert (nrm != 0).any(-1).mean() > 0.2  # the scene fills a good part of the frame


@pytest.mark.gpu
def test_threshold_at_the_constant_bank(gpu):
    """513 spheres (n_pad 544) take the BVH kernel; 512 keep the constant-bank sweep, which reports rays * n tests."""
    cam = R.main_camera(48, 8, seed=17)
    rays = int(cam.width) * int(cam.height) * 8
    _, _, st = check_bvh(gpu, cam, sweep_scene(513), 513, 8)
    assert st.sphere_tests < rays * 513
    _, _, st = check_bvh(gpu, cam, sweep_scene(512), 512, 8)
    assert st.sphere_tests == rays * 512
    # and a BVH frame of the final scene (485 spheres) keeps the culled constant-bank kernel
    _, sp, n = R.final_scene(SEED)
    _, _, st = check_bvh(gpu, cam, sp, n, 8)
    assert st.sphere_tests == rays * n


def _shard(rank, world, tile):
    B = importlib.import_module("raytracing-with-zig_b200.binding")
    return B.rtz_shard(rank, world, tile[0], tile[1])


@pytest.mark.gpu
@pytest.mark.parametrize("tile", [(4, 4), (7, 5)])
@pytest.mark.parametrize("g", [3, 64])
def test_sharded_bvh_guides_deinterleave_to_the_whole_frame(gpu, tile, g):
    import torch
    sp = sweep_scene(4096)
    cam = R.main_camera(61, 64, seed=SEED)
    cam.mode = R.MODE_PATH_BVH
    W, H = int(cam.width), int(cam.height)
    gpu.upload(sp, 4096)
    wa, wn, _ = gpu.render_guides(cam, g)
    dist = importlib.import_module("raytracing-with-zig_b200.distributed")
    per_rank, idx = dist.tile_index_map(W, H, 3, *tile)
    pad = np.ones(3 * per_rank, bool)
    pad[idx.reshape(-1)] = False
    alb, nrm, tot = [], [], 0
    for rank in range(3):
        a, nn, st = gpu.render_guides(cam, g, shard=_shard(rank, 3, tile))
        alb.append(a), nrm.append(nn)
        assert st.kernel_launches == 1 and 0 < st.sphere_tests
        tot += st.samples
    assert tot == W * H * g
    for parts, whole in ((alb, wa), (nrm, wn)):
        cat = torch.cat(parts)
        assert bits(cat.cpu().numpy()[pad]).max(initial=0) == 0  # +0 padding
        img = gpu.deinterleave(cat, W, H, 3, *tile)
        assert np.array_equal(bits(img.cpu().numpy()), bits(whole.cpu().numpy())), (tile, g)


@pytest.mark.gpu
def test_bvh_render_denoised_equals_the_resident_composition(pkg, gpu):
    sp = sweep_scene(4096)
    cam = R.main_camera(96, 16, seed=SEED)
    cam.mode = R.MODE_PATH_BVH
    params = pkg.rtz_denoise_params(3, 0, 0.5, 0.125, 1.0)
    rgb, lin, st = pkg.render_host_denoised(cam, sp, 4096, 0, params)
    assert rgb.std() > 10
    gpu.upload(sp, 4096)
    _, l0, _ = gpu.render_linear(cam)
    a0, n0, _ = gpu.render_guides(cam, 16)
    r0, o0, _ = gpu.denoise(l0, a0, n0, params=params)
    assert np.array_equal(rgb, r0.cpu().numpy()) and np.array_equal(bits(lin), bits(o0.cpu().numpy()))
    # the RTZ_MODE_PATH frame is the same frame
    cam.mode = R.MODE_PATH
    rgb_p, lin_p, _ = pkg.render_host_denoised(cam, sp, 4096, 0, params)
    assert np.array_equal(rgb, rgb_p) and np.array_equal(bits(lin), bits(lin_p))
    # the one-device multi path
    cam.mode = R.MODE_PATH_BVH
    m = pkg.MultiRenderer(1)
    m.upload(sp, 4096)
    rgb_m, lin_m, _ = m.render_denoised(cam, 0, params)
    m.close()
    assert np.array_equal(rgb, rgb_m) and np.array_equal(bits(lin), bits(lin_m))


# ------------------------------------------------------------------ two or more GPUs
@pytest.mark.gpu
@pytest.mark.parametrize("gather", ["p2p", "nccl"])
def test_multi_gpu_bvh_denoised_equals_single_gpu(pkg, gather):
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    sp = sweep_scene(4096)
    cam = R.main_camera(97, 16, seed=SEED)
    cam.mode = R.MODE_PATH_BVH
    ref_rgb, ref_lin, _ = pkg.render_host_denoised(cam, sp, 4096)
    for world in sorted({2, ngpu}):
        for tile in ((4, 4), (7, 5)):
            m = pkg.MultiRenderer(world, tile=tile, gather=gather)
            m.upload(sp, 4096)
            rgb, lin, st = m.render_denoised(cam)
            m.close()
            assert np.array_equal(rgb, ref_rgb) and np.array_equal(bits(lin), bits(ref_lin)), (world, tile, gather)
