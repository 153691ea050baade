"""Edge-avoiding à-trous denoiser (rtz_denoise, rtz_render_denoised; DESIGN.md §5 K7).

Chain of custody:
    device denoise == denoise mirror (tests/denoise_mirror.cpp), bit for bit, linear colour and bytes  (GPU tests)
    denoise mirror == a numpy restatement (f32 arithmetic, exact fmaf), bit for bit                    (CPU tests)
    denoise mirror against a high-spp render of another seed: RMSE and bias gates                      (CPU tests)
"""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import rtzlib as R
from test_guides import CH13_DEFOCUS, bits, fmaf

F32P = C.POINTER(C.c_float)
MIRROR_SRC = R.ROOT / "tests" / "denoise_mirror.cpp"
DEFAULTS = (5, 0.25, 0.25, 0.25)   # levels, sigma_color, sigma_normal, sigma_albedo of include/rtz.h
CUSTOM = (3, 0.6, 0.4, 0.15)


@pytest.fixture(scope="session")
def dmirror(tmp_path_factory):
    """tests/denoise_mirror.cpp (render mirror + guide mirror + denoise mirror) built with the oracle's flags."""
    so = tmp_path_factory.mktemp("denoise_mirror") / "libdenoise_mirror.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-pthread",
                    "-shared", "-o", str(so), str(MIRROR_SRC)], check=True, capture_output=True)
    lib = C.CDLL(str(so))
    lib.orc_mirror_denoise.restype = C.c_int32
    lib.orc_mirror_denoise.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                       C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p]
    lib.orc_mirror_guides.restype = C.c_int32
    lib.orc_mirror_guides.argtypes = [C.POINTER(R.Camera), C.POINTER(R.Sphere), C.c_uint64, C.c_uint64, C.c_uint64,
                                      F32P, F32P]
    lib.orc_render_mirror.restype = C.c_int32
    lib.orc_render_mirror.argtypes = [C.POINTER(R.Camera), C.POINTER(R.Sphere), C.c_uint64, C.c_uint64, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def mirror_denoise(lib, c, a, n, levels, sc, sn, sa):
    c, a, n = (np.ascontiguousarray(x, np.float32) for x in (c, a, n))
    H, W = c.shape[:2]
    lin, rgb = np.zeros((H, W, 3), np.float32), np.zeros((H, W, 3), np.uint8)
    assert lib.orc_mirror_denoise(W, H, c.ctypes.data, a.ctypes.data, n.ctypes.data, levels, sc, sn, sa,
                                  lin.ctypes.data, rgb.ctypes.data) == 0
    return lin, rgb


def mirror_render(lib, cam, sp, n, seed):
    """The f32 render mirror's linear colour as the device stores it: (float) of the f64 value."""
    H, W = int(cam.height), int(cam.width)
    lin = np.zeros((H, W, 3), np.float64)
    rgb = np.zeros((H, W, 3), np.uint8)
    assert lib.orc_render_mirror(C.byref(cam), C.cast(sp, C.POINTER(R.Sphere)), n, seed, 8, None, rgb.ctypes.data,
                                 lin.ctypes.data, None) == 0
    return lin, rgb


def mirror_guides(lib, cam, sp, n, g):
    H, W = int(cam.height), int(cam.width)
    alb, nrm = np.zeros((H, W, 3), np.float32), np.zeros((H, W, 3), np.float32)
    assert lib.orc_mirror_guides(C.byref(cam), C.cast(sp, C.POINTER(R.Sphere)), n, cam.seed, g,
                                 alb.ctypes.data_as(F32P), nrm.ctypes.data_as(F32P)) == 0
    return alb, nrm


def to_rgb(orc, lin):
    out = np.zeros(lin.shape, np.uint8)
    flat = np.ascontiguousarray(lin, np.float64)
    orc.orc_to_rgb(flat.ctypes.data_as(C.POINTER(C.c_double)), flat.size // 3, out.ctypes.data_as(C.POINTER(C.c_uint8)))
    return out


# ------------------------------------------------------------------ numpy restatement (f32, exact fmaf)
def _dist2(q, p):
    d = q - p
    return fmaf(d[..., 2], d[..., 2], fmaf(d[..., 1], d[..., 1], d[..., 0] * d[..., 0]))


def _edge(x):
    t = np.fmax(fmaf(x, np.float32(-2.0 ** -6), np.float32(1)), np.float32(0))
    for _ in range(6):
        t = t * t
    return t


def numpy_denoise(c, a, n, levels, sc, sn, sa):
    f = np.float32
    if levels == 0:
        return c.copy()
    H, W = c.shape[:2]
    m = np.fmax(a, f(2.0 ** -8))
    e = c / m
    ic, inn, ia = f(1.0 / (sc * sc)), f(1.0 / (sn * sn)), f(1.0 / (sa * sa))
    h1 = np.array([1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16], f)
    for lvl in range(levels):
        s = 1 << lvl
        num, den = np.zeros_like(e), np.zeros((H, W), f)
        for i in range(5):
            dy = (i - 2) * s
            for j in range(5):
                dx = (j - 2) * s
                y0, y1, x0, x1 = max(0, -dy), min(H, H - dy), max(0, -dx), min(W, W - dx)
                if y0 >= y1 or x0 >= x1:
                    continue
                P = (slice(y0, y1), slice(x0, x1))
                Q = (slice(y0 + dy, y1 + dy), slice(x0 + dx, x1 + dx))
                w = (h1[i] * h1[j]) * _edge(_dist2(e[Q], e[P]) * ic)
                w = w * _edge(_dist2(n[Q], n[P]) * inn)
                w = w * _edge(_dist2(a[Q], a[P]) * ia)
                for k in range(3):
                    num[P + (k,)] = fmaf(w, e[Q + (k,)] - e[P + (k,)], num[P + (k,)])
                den[P] = den[P] + w
        e = e + num / den[..., None]
        ic = ic * f(4)
    return e * m


def random_inputs(W, H, seed):
    """Colour in [0, 2), albedo with zero pixels and zero channels, averaged (non-unit) normals and zero (sky) ones."""
    rng = np.random.default_rng(seed)
    f = np.float32
    c = (rng.random((H, W, 3)) * 2).astype(f)
    a = rng.random((H, W, 3)).astype(f)
    a[rng.random((H, W)) < 0.15] = 0
    a[rng.random((H, W, 3)) < 0.1] = 0
    u = rng.normal(size=(2, H, W, 3))
    u /= np.linalg.norm(u, axis=-1, keepdims=True)
    n = ((u[0] + u[1]) * 0.5).astype(f)
    unit = rng.random((H, W)) < 0.5
    n[unit] = u[0][unit]
    n[rng.random((H, W)) < 0.15] = 0
    return c, a, n


SIZES = [(1, 1), (1, 9), (9, 1), (7, 3), (33, 17), (64, 48)]


@pytest.mark.parametrize("levels", [0, 1, 2, 3, 4, 5])
@pytest.mark.parametrize("W,H", SIZES)
def test_mirror_equals_a_numpy_restatement(dmirror, W, H, levels):
    c, a, n = random_inputs(W, H, 1000 * W + H)
    for prm in ((levels,) + DEFAULTS[1:], (levels,) + CUSTOM[1:]):
        lin, _ = mirror_denoise(dmirror, c, a, n, *prm)
        assert np.array_equal(bits(lin), bits(numpy_denoise(c, a, n, *prm))), prm


def test_constant_region_comes_back_bit_for_bit(dmirror):
    H, W = 21, 37
    c = np.broadcast_to(np.array([0.3, 0.7, 1.9], np.float32), (H, W, 3))
    a = np.ones((H, W, 3), np.float32)
    n = np.broadcast_to(np.array([0.0, 0.6, 0.8], np.float32), (H, W, 3))
    for levels in range(9):
        for prm in (DEFAULTS[1:], CUSTOM[1:]):
            lin, _ = mirror_denoise(dmirror, c, a, n, levels, *prm)
            assert np.array_equal(bits(lin), bits(c)), (levels, prm)


def test_nothing_crosses_a_hard_normal_edge(dmirror):
    """Normals (0,0,1) left, (0,1,0) right: |dn|^2 * in = 2 * 64 >= 64 at sigma_normal = 1/8, so each side is its own
    denoise run alone, bit for bit, at every level (steps up to 128 reach across)."""
    c, a, _ = random_inputs(50, 19, 7)
    n = np.zeros_like(c)
    n[:, :20] = (0, 0, 1)
    n[:, 20:] = (0, 1, 0)
    for levels in (1, 3, 8):
        prm = (levels, 0.25, 0.125, 0.25)
        whole, _ = mirror_denoise(dmirror, c, a, n, *prm)
        for cols in (slice(0, 20), slice(20, 50)):
            alone, _ = mirror_denoise(dmirror, c[:, cols], a[:, cols], n[:, cols], *prm)
            assert np.array_equal(bits(whole[:, cols]), bits(alone)), (levels, cols)


def test_zero_levels_is_a_copy(dmirror, orc):
    c, a, n = random_inputs(33, 17, 3)
    c[0, 0] = (0.0, 1.5, 0.999 ** 2)
    lin, rgb = mirror_denoise(dmirror, c, a, n, 0, *DEFAULTS[1:])
    assert np.array_equal(bits(lin), bits(c))
    assert np.array_equal(rgb, to_rgb(orc, c))


# ------------------------------------------------------------------ quality on the mirror
QUALITY_SCENES = ("final", "ch13")
REF_SEED = 0x5EED1


def _quality_case(orc, lib, scene, width, spp, ref_spp, ref_seed):
    """Noisy `spp` render + guides at g = 16 (seed 0xDEADBEEF) and a `ref_spp` reference of another seed: with the
    same seed the counter-based streams would share samples 0 .. 15 and flatter the noisy image."""
    if scene == "final":
        _, sp, n = R.final_scene(0xDEADBEEF)
        mk = lambda s, seed: R.main_camera(width, s, seed=seed)  # noqa: E731
    else:
        sp, n = R.chapter13_scene()
        mk = lambda s, seed: R.build_camera(width, 16.0 / 9.0, spp=s, seed=seed, **CH13_DEFOCUS)  # noqa: E731
    cam = mk(spp, 0xDEADBEEF)
    lin, _ = mirror_render(lib, cam, sp, n, cam.seed)
    alb, nrm = mirror_guides(lib, cam, sp, n, 16)
    ref, ref_rgb = mirror_render(lib, mk(ref_spp, ref_seed), sp, n, ref_seed)
    return lin.astype(np.float32), alb, nrm, ref, ref_rgb


def quality(noisy, den_lin, den_rgb, ref, ref_rgb):
    """(denoised RMSE / noisy RMSE in linear colour, per-channel mean byte bias of the denoised frame)."""
    rmse = lambda x: np.sqrt(np.mean((x.astype(np.float64) - ref) ** 2))  # noqa: E731
    bias = (den_rgb.astype(np.float64) - ref_rgb).reshape(-1, 3).mean(0)
    return rmse(den_lin) / rmse(noisy), bias


@pytest.fixture(scope="module")
def mirror_quality(orc, dmirror):
    out = {}
    for scene in QUALITY_SCENES:
        lin, alb, nrm, ref, ref_rgb = _quality_case(orc, dmirror, scene, 160, 16, 1024, REF_SEED)
        dl, dr = mirror_denoise(dmirror, lin, alb, nrm, *DEFAULTS)
        out[scene] = quality(lin, dl, dr, ref, ref_rgb)
    return out


@pytest.mark.parametrize("scene", QUALITY_SCENES)
def test_mirror_denoise_lowers_error_without_bias(mirror_quality, scene):
    """16 spp at 160x90, defaults, against 1 024 spp of another seed: the error drops and the mean byte bias stays
    within a quarter of an 8-bit level per channel (measured: DESIGN.md §5 K7)."""
    ratio, bias = mirror_quality[scene]
    assert ratio < 0.9, ratio
    assert np.abs(bias).max() <= 0.25, bias


@pytest.mark.parametrize("scene", [
    pytest.param("final", marks=pytest.mark.xfail(strict=True, reason="the gate misses on the final scene: denoised "
                                                  "RMSE 0.83 x the noisy one at the defaults (DESIGN.md §5 K7)")),
    "ch13"])
def test_mirror_denoise_halves_the_error(mirror_quality, scene):
    ratio, _ = mirror_quality[scene]
    assert ratio <= 0.5, ratio


def test_denoise_kernels_keep_to_registers():
    """Codegen guard (no GPU needed): the three denoise kernels do not spill (STL / LDL)."""
    import importlib
    importlib.import_module("raytracing-with-zig_b200.build").build_all()
    lib = R.ROOT / "raytracing-with-zig_b200" / "csrc" / "librtz.so"
    out = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    kernels = [k for k in body if "denoise_" in k]
    assert len(kernels) == 3, kernels
    for k in kernels:
        assert not re.search(r"\b(STL|LDL)\b", "\n".join(body[k])), k


# ------------------------------------------------------------------ on the GPU
def _params(pkg, prm):
    return pkg.rtz_denoise_params(prm[0], 0, prm[1], prm[2], prm[3])


def _device_inputs(gpu, cam, sp, n, g):
    gpu.upload(sp, n)
    _, lin, _ = gpu.render_linear(cam)
    alb, nrm, _ = gpu.render_guides(cam, g)
    return lin, alb, nrm


def _check_device(pkg, gpu, dmirror, lin, alb, nrm, prm, default=False):
    import torch
    rgb, out, st = gpu.denoise(lin, alb, nrm, params=None if default else _params(pkg, prm))
    ml, mr = mirror_denoise(dmirror, lin.cpu().numpy(), alb.cpu().numpy(), nrm.cpu().numpy(), *prm)
    got = out.cpu().numpy()
    assert np.array_equal(bits(got), bits(ml)), f"{np.count_nonzero(bits(got) != bits(ml))} linear words differ"
    assert np.array_equal(rgb.cpu().numpy(), mr)
    assert st.kernel_launches == (prm[0] + 2 if prm[0] else 1) and st.total_ms > 0
    assert (st.samples, st.segments, st.trace_ms, st.seed_used) == (0, 0, 0.0, 0)
    torch.cuda.synchronize()
    return got, rgb


@pytest.mark.gpu
@pytest.mark.parametrize("levels", [1, 3, 5])
@pytest.mark.parametrize("spp,g", [(8, 1), (64, 1), (64, 16)])
def test_device_denoise_matches_mirror(pkg, gpu, dmirror, spp, g, levels):
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(160, spp, seed=0xDEADBEEF)
    lin, alb, nrm = _device_inputs(gpu, cam, sp, n, g)
    if levels == DEFAULTS[0]:
        _check_device(pkg, gpu, dmirror, lin, alb, nrm, DEFAULTS, default=True)
    _check_device(pkg, gpu, dmirror, lin, alb, nrm, (levels,) + DEFAULTS[1:])
    _check_device(pkg, gpu, dmirror, lin, alb, nrm, (levels,) + CUSTOM[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(1, 1), (7, 3), (33, 17)])
def test_device_denoise_matches_mirror_on_odd_sizes(pkg, gpu, dmirror, W, H):
    import torch
    c, a, n = random_inputs(W, H, 11 * W + H)
    t = [torch.from_numpy(x).cuda() for x in (c, a, n)]
    for levels in (0, 1, 3, 5, 8):
        _check_device(pkg, gpu, dmirror, *t, (levels,) + CUSTOM[1:])


@pytest.mark.gpu
def test_device_denoise_matches_mirror_at_c3_size(pkg, gpu, dmirror):
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(1200, 16, seed=0xDEADBEEF)
    lin, alb, nrm = _device_inputs(gpu, cam, sp, n, 16)
    assert tuple(lin.shape) == (675, 1200, 3)
    _check_device(pkg, gpu, dmirror, lin, alb, nrm, DEFAULTS, default=True)


@pytest.mark.gpu
def test_one_shot_equals_the_resident_composition(pkg, gpu):
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(160, 32, seed=0xDEADBEEF)
    for g, prm in ((0, None), (4, CUSTOM)):
        params = None if prm is None else _params(pkg, prm)
        rgb, lin, st = pkg.render_host_denoised(cam, sp, n, guide_samples=g, params=params)
        l, a, nr = _device_inputs(gpu, cam, sp, n, g or 16)
        drgb, dlin, dst = gpu.denoise(l, a, nr, params=params)
        assert np.array_equal(rgb, drgb.cpu().numpy()) and np.array_equal(bits(lin), bits(dlin.cpu().numpy()))
        _, rst = gpu.render(cam)
        assert (st.samples, st.segments, st.sphere_tests, st.seed_used) == (rst.samples, rst.segments,
                                                                            rst.sphere_tests, cam.seed)
        assert st.kernel_launches == rst.kernel_launches + 1 + dst.kernel_launches
        assert st.total_ms >= st.trace_ms > 0
    # no seed: one drawn seed keys the render and the guides, and reproduces the frame through the composition
    free = R.Camera.from_buffer_copy(bytes(cam))
    free.has_seed, free.seed = 0, 0
    rgb, lin, st = pkg.render_host_denoised(free, sp, n)
    cam.seed = st.seed_used
    l, a, nr = _device_inputs(gpu, cam, sp, n, 16)
    drgb, dlin, _ = gpu.denoise(l, a, nr)
    assert np.array_equal(rgb, drgb.cpu().numpy()) and np.array_equal(bits(lin), bits(dlin.cpu().numpy()))


@pytest.fixture(scope="module")
def device_quality(pkg, gpu):
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(400, 16, seed=0xDEADBEEF)
    lin, alb, nrm = _device_inputs(gpu, cam, sp, n, 16)
    rgb, out, _ = gpu.denoise(lin, alb, nrm)
    ref_rgb, _, ref = pkg.render_host(R.main_camera(400, 2048, seed=0x5EED2), sp, n, want_linear=True)
    return quality(lin.cpu().numpy(), out.cpu().numpy(), rgb.cpu().numpy(), ref, ref_rgb)


@pytest.mark.gpu
def test_device_denoise_lowers_error_without_bias(device_quality):
    """The final scene at 400x225, 16 spp denoised at the defaults, against 2 048 spp of another seed."""
    ratio, bias = device_quality
    assert ratio < 0.9, ratio
    assert np.abs(bias).max() <= 0.25, bias


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="the gate misses on the final scene (DESIGN.md §5 K7)")
def test_device_denoise_halves_the_error(device_quality):
    ratio, _ = device_quality
    assert ratio <= 0.5, ratio


@pytest.mark.gpu
def test_denoise_refusals(pkg, gpu):
    import torch
    l = pkg.lib()
    H, W = 8, 12
    bufs = [torch.zeros((H, W, 3), dtype=torch.float32, device="cuda:0") for _ in range(4)]
    img = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda:0")
    col, alb, nrm, out = (C.c_void_p(b.data_ptr()) for b in bufs)
    rgb = C.c_void_p(img.data_ptr())

    def dn(w=W, h=H, c=col, a=alb, n=nrm, prm=None, lo=out, ro=rgb, ctx=gpu._ctx):
        p = None if prm is None else C.byref(_params(pkg, prm) if isinstance(prm, tuple) else prm)
        return l.rtz_denoise(ctx, w, h, c, a, n, p, lo, ro, None)

    assert dn() == 0 and dn(lo=None) == 0 and dn(ro=None) == 0
    assert dn(ctx=None) == 1
    assert dn(c=None) == 1 and dn(a=None) == 1 and dn(n=None) == 1
    assert dn(lo=None, ro=None) == 1
    assert dn(lo=col) == 1 and dn(lo=nrm) == 1                              # an output on an input
    assert dn(lo=C.c_void_p(bufs[1].data_ptr() - 4)) == 1                   # ... or overlapping one by a word
    assert dn(ro=C.c_void_p(bufs[2].data_ptr() + 100)) == 1
    assert dn(ro=C.c_void_p(bufs[3].data_ptr() + 8)) == 1                    # the outputs on each other
    assert dn(w=0) == 1 and dn(h=0) == 1
    assert dn(w=1 << 16, h=1 << 15) == 1                                     # 2^31 pixels
    assert dn(prm=(8, 0.5, 0.5, 0.5)) == 0 and dn(prm=(9, 0.5, 0.5, 0.5)) == 1
    bad = pkg.rtz_denoise_params(2, 1, 0.5, 0.5, 0.5)
    assert dn(prm=bad) == 1                                                  # reserved != 0
    for k in range(1, 4):
        for v in (0.0, -1.0, float("nan"), float("inf")):
            prm = [3, 0.5, 0.5, 0.5]
            prm[k] = v
            assert dn(prm=tuple(prm)) == 1, prm
    assert dn(prm=(1, 1e-18, 0.5, 0.5)) == 0 and dn(prm=(8, 1e-18, 0.5, 0.5)) == 1  # 4^7 / sigma^2 overflows f32
    # the one-shot
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(32, 8, seed=1)
    h = int(cam.height)
    hr = np.zeros((h, 32, 3), np.uint8)
    hl = np.zeros((h, 32, 3), np.float32)
    bsp = C.cast(sp, C.POINTER(pkg.rtz_sphere))

    def one(c=cam, g=0, prm=None, ro=hr.ctypes.data_as(C.POINTER(C.c_uint8)), lo=hl.ctypes.data_as(F32P), s=bsp, cnt=n):
        p = None if prm is None else C.byref(_params(pkg, prm))
        return l.rtz_render_denoised(C.byref(pkg.rtz_camera.from_buffer_copy(bytes(c))), s, cnt, g, p, ro, lo, None)

    def variant(**kw):
        c = R.Camera.from_buffer_copy(bytes(cam))
        for k, v in kw.items():
            setattr(c, k, v)
        return c

    assert one() == 0 and one(g=8) == 0 and one(ro=None) == 0 and one(lo=None) == 0
    assert one(g=9) == 1
    assert one(ro=None, lo=None) == 1
    assert one(s=None) == 1
    assert one(prm=(9, 0.5, 0.5, 0.5)) == 1 and one(prm=(3, 0.0, 0.5, 0.5)) == 1
    assert one(c=variant(mode=R.MODE_LEGACY_NORMAL, samples_per_pixel=1)) == 1
    assert one(c=variant(width=0)) == 1
    assert one(c=variant(width=1 << 16, height=1 << 15)) == 1
    with pytest.raises(pkg.RtzError):
        gpu.denoise(bufs[0], bufs[1], bufs[2], params=pkg.rtz_denoise_params(3, 0, -1.0, 0.5, 0.5))
