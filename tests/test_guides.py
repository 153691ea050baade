"""First-hit denoiser guides (rtz_render_guides) and the f32 linear colour (rtz_render_resident_linear).

Chain of custody of the guides:
    device guides == guide mirror (tests/guide_mirror.cpp: the f32 device mirror's cameraRay / sweep + the guide
                     loop), bit for bit                                                           (GPU tests)
    guide mirror  == a numpy restatement on the mirror's camera rays, bit for bit                 (CPU test)
    device guides == per-sample values from the device probes rtz_probe_camera_ray + rtz_probe_hits (GPU test)
The linear colour is (float) of the f64 value rtz_render_linear reports, which the mirror pins already.
"""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import rtzlib as R

F32P = C.POINTER(C.c_float)
MIRROR_SRC = R.ROOT / "tests" / "guide_mirror.cpp"


@pytest.fixture(scope="session")
def guide_mirror(tmp_path_factory):
    """tests/guide_mirror.cpp built with the oracle's flags (oracle/Makefile) into a temporary directory."""
    so = tmp_path_factory.mktemp("guide_mirror") / "libguide_mirror.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-pthread",
                    "-shared", "-o", str(so), str(MIRROR_SRC)], check=True, capture_output=True)
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


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ------------------------------------------------------------------ numpy restatement (f32, exact fma)
def fmaf(a, b, c):
    """fmaf in f32, correctly rounded: the product of two floats is exact in f64, TwoSum gives the exact error e of
    the f64 sum s, and rounding s to f32 differs from rounding s + e only when s is a tie between two floats and
    e != 0; then the exact value lies on e's side."""
    a, b, c = np.broadcast_arrays(*(np.asarray(x, np.float32) for x in (a, b, c)))
    p = a.astype(np.float64) * b.astype(np.float64)
    c64 = c.astype(np.float64)
    s = p + c64
    z = s - p
    e = (p - (s - z)) + (c64 - z)
    r = s.astype(np.float32)
    r64 = r.astype(np.float64)
    other = np.nextafter(r, np.where(s > r64, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
    tie = (r64 != s) & ((r64 + other.astype(np.float64)) * 0.5 == s) & (e != 0)
    return np.where(tie, np.where(e > 0, np.maximum(r, other), np.minimum(r, other)), r)


def sphere_table(sp, n):
    """The device's per-sphere f32 rows, as rtz_scene_upload forms them."""
    c = np.array([list(sp[i].center) for i in range(n)], np.float64).astype(np.float32)
    r = np.array([max(sp[i].radius, 0.0) for i in range(n)], np.float64).astype(np.float32)
    c2 = (c.astype(np.float64) ** 2).sum(1)
    nq = -((c2 - r.astype(np.float64) ** 2) - float(np.float32(2.0 ** -18)) * c2).astype(np.float32)
    mat = np.array([sp[i].mat_type for i in range(n)])
    alb = np.array([list(sp[i].albedo) for i in range(n)], np.float64).astype(np.float32)
    alb[mat == R.MAT_DIELECTRIC] = 1.0
    return dict(c=c, r2=r * r, nq=nq, inv_r=np.float32(1.0) / r, alb=alb)


def numpy_values(o, d, ln, T, tmin, tmax):
    """Per ray (rows of o, d, ln): the six guide values, restating the mirror's sweep (gate, direct-form root, strict
    nearer, ascending order) and the sky / HitRecord expressions."""
    f = np.float32
    ox, oy, oz = o.T
    dx, dy, dz = d.T
    tmin_d, closest = f(tmin) * ln, f(tmax) * ln
    best = np.full(len(o), -1)
    k1 = -fmaf(dz, oz, fmaf(dy, oy, dx * ox))
    nk2 = -fmaf(oz, oz, fmaf(oy, oy, ox * ox)) * (f(1) - f(2.0 ** -18))
    tx, ty, tz = f(2) * ox, f(2) * oy, f(2) * oz
    for i, (cx, cy, cz) in enumerate(T["c"]):
        he = fmaf(dz, cz, fmaf(dy, cy, fmaf(dx, cx, k1)))
        w = fmaf(tz, cz, fmaf(ty, cy, fmaf(tx, cx, nk2))) + T["nq"][i]
        gate = ~np.signbit(fmaf(he, he, w))
        ocx, ocy, ocz = cx - ox, cy - oy, cz - oz
        h = fmaf(dz, ocz, fmaf(dy, ocy, dx * ocx))
        cc = fmaf(ocz, ocz, fmaf(ocy, ocy, fmaf(ocx, ocx, -T["r2"][i])))
        disc = fmaf(h, h, -cc)
        ok = gate & (disc >= 0)
        sq = np.sqrt(np.where(ok, disc, f(0)))
        t1, t2 = h - sq, h + sq
        a1 = ok & (t1 > tmin_d) & (t1 < closest)
        a2 = ok & ~a1 & (t2 > tmin_d) & (t2 < closest)
        upd = a1 | a2
        closest = np.where(upd, np.where(a1, t1, t2), closest)
        best = np.where(upd, i, best)
    v = np.zeros((len(o), 6), np.float32)
    miss = best < 0
    a = f(0.5) * (dy + f(1))
    w = f(1) - a
    sky = np.stack([fmaf(a, f(0.5), w), fmaf(a, f(0.7), w), fmaf(a, f(1.0), w)], 1)
    hit = ~miss
    b = best[hit]
    t = closest[hit]
    p = np.stack([fmaf(t, dx[hit], ox[hit]), fmaf(t, dy[hit], oy[hit]), fmaf(t, dz[hit], oz[hit])], 1)
    nrm = (p - T["c"][b]) * T["inv_r"][b][:, None]
    dn = fmaf(dz[hit], nrm[:, 2], fmaf(dy[hit], nrm[:, 1], dx[hit] * nrm[:, 0]))
    nrm = np.where((dn < 0)[:, None], nrm, -nrm)
    v[miss, :3] = sky[miss]
    v[hit, :3] = T["alb"][b]
    v[hit, 3:] = nrm
    return v


def fold(vals):
    """vals [pixels, g, 6] -> [pixels, 6]: ascending samples from +0 in f32, one division by g."""
    acc = np.zeros((vals.shape[0], 6), np.float32)
    for s in range(vals.shape[1]):
        acc = acc + vals[:, s]
    return acc / np.float32(vals.shape[1])


CH13_DEFOCUS = dict(look_from=(-2, 2, 1), look_at=(0, 0, -1), vfov=20, defocus=10.0, viewport_focus=3.4, focus=3.4)


@pytest.mark.parametrize("g", [1, 5, 70])
def test_mirror_guides_equal_a_numpy_restatement(orc, guide_mirror, g):
    """orc_mirror_guides == a numpy restatement of the sweep and the guide values (fmaf formed exactly: the f64
    product with a TwoSum tie correction, sky pixels included) on the mirror's own camera rays, folded in order."""
    sp, n = R.chapter13_scene()
    cam = R.build_camera(14, 16.0 / 9.0, spp=70, seed=0xDEADBEEF, **dict(CH13_DEFOCUS, vfov=60))  # sky in view too
    H, W = int(cam.height), int(cam.width)
    o, d, ln = np.zeros((H * W, g, 3), np.float32), np.zeros((H * W, g, 3), np.float32), np.zeros((H * W, g), np.float32)
    for j in range(H):
        for i in range(W):
            k = j * W + i
            orc.orc_mirror_camera_ray(C.byref(cam), cam.seed, i, j, 0, g, o[k].ctypes.data_as(F32P),
                                      d[k].ctypes.data_as(F32P), ln[k].ctypes.data_as(F32P))
    v = numpy_values(o.reshape(-1, 3), d.reshape(-1, 3), ln.reshape(-1), sphere_table(sp, n), cam.t_min, cam.t_max)
    exp = fold(v.reshape(H * W, g, 6))
    alb, nrm = mirror_guides(guide_mirror, cam, sp, n, g)
    assert np.array_equal(bits(alb.reshape(-1, 3)), bits(exp[:, :3]))
    assert np.array_equal(bits(nrm.reshape(-1, 3)), bits(exp[:, 3:]))
    miss = (v[:, 3:] == 0).all(1)
    assert 0 < miss.sum() < len(v)  # both the sky and the spheres are covered


def test_guide_kernels_keep_to_registers():
    """Codegen guard (no GPU needed): the guide kernels neither spill (STL / LDL) nor guard a vote with BRA.DIV."""
    lib = R.ROOT / "raytracing-with-zig_b200" / "csrc" / "librtz.so"
    import importlib
    importlib.import_module("raytracing-with-zig_b200.build").build_all()
    out = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    guides = [k for k in body if "guide_kernel" in k]
    assert len(guides) == 3, guides
    for k in guides:
        sass = "\n".join(body[k])
        assert not re.search(r"\b(STL|LDL)\b", sass), k
        assert "BRA.DIV" not in sass, k
        assert "FFMA2" in sass, k


# ------------------------------------------------------------------ on the GPU
CH13_CAMERAS = {
    "ch11": dict(look_from=(0, 0, 0), look_at=(0, 0, -1), vfov=90),
    "ch12": dict(look_from=(-2, 2, 1), look_at=(0, 0, -1), vfov=20),
    "ch13": CH13_DEFOCUS,
}


def _sweep_scene(orc, n):
    prng = orc.orc_prng_new(7)
    buf = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, buf) == n
    orc.orc_prng_free(prng)
    return buf


def _device_guides(gpu, cam, sp, n, g):
    gpu.upload(sp, n)
    alb, nrm, st = gpu.render_guides(cam, g)
    return alb.cpu().numpy(), nrm.cpu().numpy(), st


def _check(gpu, guide_mirror, cam, sp, n, g):
    alb, nrm, st = _device_guides(gpu, cam, sp, n, g)
    malb, mnrm = mirror_guides(guide_mirror, cam, sp, n, g)
    assert np.array_equal(bits(alb), bits(malb)), f"{np.count_nonzero(bits(alb) != bits(malb))} albedo words differ"
    assert np.array_equal(bits(nrm), bits(mnrm)), f"{np.count_nonzero(bits(nrm) != bits(mnrm))} normal words differ"
    rays = int(cam.width) * int(cam.height) * g
    assert (st.samples, st.segments, st.sphere_tests, st.kernel_launches, st.seed_used) == (rays, rays, rays * n, 1, cam.seed)
    assert (st.depth_capped, st.absorbed, st.nan_samples, st.resolve_ms) == (0, 0, 0, 0.0)
    assert st.trace_ms > 0 and st.total_ms == st.trace_ms
    return alb, nrm


@pytest.mark.gpu
@pytest.mark.parametrize("preset", list(CH13_CAMERAS))
@pytest.mark.parametrize("g", [1, 3, 64])
def test_chapter13_guides_match_mirror(gpu, guide_mirror, preset, g):
    sp, n = R.chapter13_scene()
    cam = R.build_camera(160, 16.0 / 9.0, spp=64, seed=0xDEADBEEF, **CH13_CAMERAS[preset])
    _check(gpu, guide_mirror, cam, sp, n, g)


@pytest.mark.gpu
@pytest.mark.parametrize("g", [1, 7, 64, 65, 130])
def test_final_scene_guides_match_mirror(gpu, guide_mirror, g):
    """The book's final scene: the culled constant-bank sweep over the regrouped rows (ties on the original index)."""
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(160, 130, seed=0xDEADBEEF)
    alb, nrm = _check(gpu, guide_mirror, cam, sp, n, g)
    if g == 1:  # glass and sky pixels occur; the normal of one hit is unit up to the f32 hit point (grazing hits on
        # the radius-1000 ground sphere lose a few 1e-3 of the length: the render shades with the same normal)
        assert (alb == 1.0).all(-1).any() and (nrm == 0).all(-1).any()
        hit = ~(nrm == 0).all(-1)
        assert np.abs(np.linalg.norm(nrm[hit], axis=-1) - 1).max() < 1e-2


@pytest.mark.gpu
@pytest.mark.parametrize("n,width,g", [(16, 96, 5), (513, 64, 3), (4096, 48, 2), (8192, 32, 3)])
def test_sweep_scene_guides_match_mirror(gpu, guide_mirror, orc, n, width, g):
    """16 spheres: the plain constant-bank sweep; 513 and more: the plain rows from global memory (the render stages
    513 and 4096 in shared memory and reads 8 192 from global memory: the guides read global memory for all)."""
    sp = _sweep_scene(orc, n)
    cam = R.main_camera(width, 8, seed=0x5EED + n)
    _check(gpu, guide_mirror, cam, sp, n, g)


@pytest.mark.gpu
def test_empty_world_guides_are_the_sky(gpu, guide_mirror):
    sp = (R.Sphere * 1)()
    for defocus in (0.0, 0.6):
        cam = R.build_camera(64, 16.0 / 9.0, (13, 2, 3), (0, 0, 0), 20, defocus=defocus, spp=4, seed=3)
        alb, nrm = _check(gpu, guide_mirror, cam, sp, 0, 4)
        assert (nrm == 0).all() and (alb > 0).all()


@pytest.mark.gpu
def test_bvh_mode_gives_the_same_guides(gpu, orc):
    _, sp, n = R.final_scene(0xDEADBEEF)
    for cam, sps, cnt in ((R.main_camera(120, 9, seed=5), sp, n), (R.main_camera(64, 9, seed=6), _sweep_scene(orc, 600), 600)):
        a0, n0, _ = _device_guides(gpu, cam, sps, cnt, 9)
        cam.mode = R.MODE_PATH_BVH
        a1, n1, _ = _device_guides(gpu, cam, sps, cnt, 9)
        assert np.array_equal(bits(a0), bits(a1)) and np.array_equal(bits(n0), bits(n1))


RAY = np.dtype([("orig", "<f4", 3), ("dir", "<f4", 3), ("self", "<i4")])
RAY_HIT = np.dtype([("best", "<i4"), ("front", "<i4"), ("t", "<f4"), ("len", "<f4"), ("point", "<f4", 3),
                    ("normal", "<f4", 3)])


@pytest.mark.gpu
def test_guides_tie_to_the_device_probes(pkg, gpu):
    """For sampled pixels of a one-sample guide frame: the camera ray from rtz_probe_camera_ray, its hit from
    rtz_probe_hits and the sphere table give the guide values.  rtz_probe_hits normalises the direction it is given
    again, which changes a unit direction unless its length rounds to exactly 1, so only those rays are compared (the
    probe's t_min * 1 instead of t_min * |d| cannot matter: no sphere is nearer than 0.01 to the camera)."""
    l = pkg.lib()
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(160, 4, seed=0xDEADBEEF)
    alb, nrm, _ = _device_guides(gpu, cam, sp, n, 1)
    bcam = pkg.rtz_camera.from_buffer_copy(bytes(cam))
    rng = np.random.default_rng(1)
    W, H = int(cam.width), int(cam.height)
    pix = rng.choice(W * H, 600, replace=False)
    rays = np.zeros(len(pix), RAY)
    o, d, ln = np.zeros(3, np.float32), np.zeros(3, np.float32), np.zeros(1, np.float32)
    for k, p in enumerate(pix):
        pkg.binding.check(l.rtz_probe_camera_ray(C.byref(bcam), int(p % W), int(p // W), 0, 1, o.ctypes.data_as(F32P),
                                                 d.ctypes.data_as(F32P), ln.ctypes.data_as(F32P)))
        rays[k] = (o, d, -1)
    hits = np.zeros(len(pix), RAY_HIT)
    pkg.binding.check(l.rtz_probe_hits(C.cast(sp, C.POINTER(pkg.rtz_sphere)), n, rays.ctypes.data, len(rays),
                                       cam.t_min, cam.t_max, hits.ctypes.data))
    keep = hits["len"] == np.float32(1)
    assert keep.sum() >= 200, keep.sum()
    T = sphere_table(sp, n)
    hit = hits["best"] >= 0
    exp = np.zeros((len(pix), 6), np.float32)
    dy = rays["dir"][:, 1]
    a = np.float32(0.5) * (dy + np.float32(1))
    w = np.float32(1) - a
    exp[~hit, 0], exp[~hit, 1], exp[~hit, 2] = (fmaf(a, np.float32(c), w)[~hit] for c in (0.5, 0.7, 1.0))
    exp[hit, :3] = T["alb"][hits["best"][hit]]
    exp[hit, 3:] = hits["normal"][hit]
    exp = fold(exp[:, None, :])
    assert hit[keep].any() and (~hit[keep]).any()
    got = np.concatenate([alb.reshape(-1, 3)[pix], nrm.reshape(-1, 3)[pix]], 1)
    assert np.array_equal(bits(got[keep]), bits(exp[keep]))


@pytest.mark.gpu
def test_linear_colour_whole_frame_and_shard(pkg, gpu, orc):
    _, sp, n = R.final_scene(0xDEADBEEF)
    cam = R.main_camera(200, 12, seed=0xDEADBEEF)
    rgb_h, _, lin64 = pkg.render_host(cam, sp, n, want_linear=True)   # rtz_render_linear: f64
    gpu.upload(sp, n)
    img, lin, st = gpu.render_linear(cam)
    img0, st0 = gpu.render(cam)
    assert np.array_equal(lin.cpu().numpy().view(np.uint32), lin64.astype(np.float32).view(np.uint32))
    assert np.array_equal(img.cpu().numpy(), img0.cpu().numpy()) and np.array_equal(img.cpu().numpy(), rgb_h)
    assert (st.samples, st.segments) == (st0.samples, st0.segments)
    # one rank's tiles: the compact layout, against the mirror's f64 linear colour of the same shard
    shard = R.Shard(1, 3, 8, 4)
    bshard = pkg.rtz_shard(1, 3, 8, 4)
    simg, slin, _ = gpu.render_linear(cam, shard=bshard)
    npix = gpu.shard_pixels(cam.width, cam.height, bshard)
    mrgb, mlin = np.zeros((npix, 3), np.uint8), np.zeros((npix, 3), np.float64)
    assert orc.orc_render_mirror(C.byref(cam), sp, n, cam.seed, 8, C.byref(shard), mrgb.ctypes.data_as(C.POINTER(C.c_uint8)),
                                 mlin.ctypes.data_as(C.POINTER(C.c_double)), None) == 0
    assert np.array_equal(slin.cpu().numpy().view(np.uint32), mlin.astype(np.float32).view(np.uint32))
    assert np.array_equal(simg.cpu().numpy(), mrgb)
    sref, _ = gpu.render(cam, shard=bshard)
    assert np.array_equal(simg.cpu().numpy(), sref.cpu().numpy())


@pytest.mark.gpu
def test_guides_and_linear_refusals(pkg, gpu):
    import torch
    l = pkg.lib()
    _, sp, n = R.final_scene(0xDEADBEEF)
    gpu.upload(sp, n)
    cam = R.main_camera(32, 8, seed=1)
    buf = torch.empty((int(cam.height), int(cam.width), 3), dtype=torch.float32, device="cuda:0")
    p = C.c_void_p(buf.data_ptr())

    def guides(c, g=2, alb=p, nrm=p, ctx=gpu._ctx):
        return l.rtz_render_guides(ctx, C.byref(pkg.rtz_camera.from_buffer_copy(bytes(c))), g, alb, nrm, None)

    def variant(**kw):
        c = R.Camera.from_buffer_copy(bytes(cam))
        for k, v in kw.items():
            setattr(c, k, v)
        return c

    assert guides(cam) == 0
    assert guides(cam, alb=None) == 0 and guides(cam, nrm=None) == 0
    assert guides(cam, alb=None, nrm=None) == 1
    assert guides(cam, ctx=None) == 1
    assert guides(cam, g=0) == 1 and guides(cam, g=9) == 1 and guides(cam, g=8) == 0
    assert guides(variant(has_seed=0)) == 1
    assert guides(variant(width=0)) == 1
    assert guides(variant(mode=R.MODE_LEGACY_NORMAL, samples_per_pixel=1), g=1) == 1
    # the f32 linear colour: required, and not for the legacy modes
    img = torch.empty((int(cam.height), int(cam.width), 3), dtype=torch.uint8, device="cuda:0")
    bcam = pkg.rtz_camera.from_buffer_copy(bytes(cam))
    assert l.rtz_render_resident_linear(gpu._ctx, C.byref(bcam), None, C.c_void_p(img.data_ptr()), None, None) == 1
    lcam = pkg.rtz_camera.from_buffer_copy(bytes(variant(mode=R.MODE_LEGACY_NORMAL, samples_per_pixel=1)))
    assert l.rtz_render_resident_linear(gpu._ctx, C.byref(lcam), None, C.c_void_p(img.data_ptr()), p, None) == 1
    with pytest.raises(pkg.RtzError):
        gpu.render_guides(variant(has_seed=0), 1)
