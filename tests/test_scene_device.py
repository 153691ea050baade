"""Scenes installed from device memory (rtz_scene_upload_device) and the BVH built on the device.

A list uploaded from a CUDA tensor must leave the context exactly as the host upload of the same list does (every row,
compared through rtz_probe_scene_rows), so every frame kind is the same bytes with the same counters.  The device BVH
builder must give the host builder's tree node for node (rtz_probe_bvh), with the same set of spheres in every leaf.
Refusals name the same first sphere with the same status and message.
"""
import ctypes as C
import importlib
import re
import subprocess

import numpy as np
import pytest

import rtzlib as R

SEED = 0xDEADBEEF
MODE_LEGACY_NORMAL = 3
STAT_FIELDS = ("samples", "segments", "sphere_tests", "depth_capped", "absorbed", "nan_samples", "kernel_launches")


def binding():
    return importlib.import_module("raytracing-with-zig_b200.binding")


def sweep_scene(n, seed=7):
    orc = R.oracle()
    prng = orc.orc_prng_new(seed)
    buf = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, buf) == n
    orc.orc_prng_free(prng)
    return buf


def random_scene(n, seed):
    rng = np.random.default_rng(seed)
    return R.sphere_array([R.make_sphere(rng.uniform(-3, 3, 3), rng.uniform(0.1, 0.8), int(rng.integers(0, 3)),
                                         albedo=tuple(rng.uniform(0, 1, 3)), fuzz=0.2, ior=1.5) for _ in range(n)])


def equal_axis_scene():
    """1 200 spheres, most sharing x = 1.0 exactly and half of those sharing y too: every split meets runs of equal keys."""
    rng = np.random.default_rng(3)
    out = [R.make_sphere((0, -1000, 0), 1000, R.MAT_LAMBERTIAN, albedo=(0.5, 0.5, 0.5))]
    for k in range(1199):
        y = 0.5 if k % 2 else rng.uniform(0, 20)
        out.append(R.make_sphere((1.0 if k % 5 else rng.uniform(-30, 30), y, rng.uniform(-30, 30)), 0.2,
                                 k % 3, albedo=(0.3, 0.6, 0.9), fuzz=0.1, ior=1.5))
    return R.sphere_array(out)


def signed_zero_scene():
    """900 spheres whose centres hold +0.0 and -0.0 on every axis: equal keys that must fall back to the index."""
    rng = np.random.default_rng(4)
    out = []
    for k in range(900):
        c = [rng.choice([0.0, -0.0, rng.uniform(-5, 5)]) for _ in range(3)]
        out.append(R.make_sphere(c, 0.05 + 0.01 * (k % 7), k % 3, albedo=(0.8, 0.4, 0.2), fuzz=0.0, ior=1.5))
    return R.sphere_array(out)


def nested_glass_scene():
    rng = np.random.default_rng(11)
    out = list(sweep_scene(600))
    for _ in range(200):
        c = (rng.uniform(-11, 11), 0.2, rng.uniform(-11, 11))
        out += [R.make_sphere(c, 0.2, R.MAT_DIELECTRIC, ior=1.5), R.make_sphere(c, 0.18, R.MAT_DIELECTRIC, ior=1 / 1.5),
                R.make_sphere(c, 0.05, R.MAT_LAMBERTIAN, albedo=tuple(rng.uniform(0, 1, 3)))]
    return R.sphere_array(out)


def far_sphere_scene():
    out = list(sweep_scene(700))
    out.append(R.make_sphere((1e4, 3.0, -2e3), 5.0, R.MAT_METAL, albedo=(0.9, 0.9, 0.9), fuzz=0.0))
    return R.sphere_array(out)


def as_tensor(sp, n, device=0):
    import torch
    raw = np.frombuffer(bytes(sp)[: n * C.sizeof(R.Sphere)], dtype=np.float64).reshape(n, 10).copy()
    return torch.from_numpy(raw).to(f"cuda:{device}")


def scene_rows(r):
    l, size = r.lib, C.c_uint64(0)
    assert l.rtz_probe_scene_rows(r._ctx, None, 0, C.byref(size)) == 0
    buf = (C.c_uint8 * size.value)()
    assert l.rtz_probe_scene_rows(r._ctx, buf, size.value, C.byref(size)) == 0
    return bytes(buf)


def probe_bvh(r, builder):
    l, cnt = r.lib, C.c_uint64(0)
    B = binding()
    binding().check(l.rtz_probe_bvh(r._ctx, builder, None, 0, None, None, C.byref(cnt)))
    nodes = np.zeros(cnt.value * 16, np.uint32)
    order = np.zeros(max(r.n_spheres, 1), np.int32)
    r2 = C.c_float(0)
    B.check(l.rtz_probe_bvh(r._ctx, builder, nodes.ctypes.data_as(C.c_void_p), cnt.value,
                            order.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(r2), C.byref(cnt)))
    return nodes.reshape(-1, 16), order[: r.n_spheres], np.float32(r2.value)


def leaf_sets(nodes, order):
    """order sorted inside every leaf range (the leaves partition 0 .. n-1)"""
    kids = nodes[:, 12:14].view(np.int32).reshape(-1)
    codes = -1 - kids[(kids < 0)]
    first, cnt = codes >> 3, codes & 7
    assert cnt.sum() == len(order)
    out = order.copy()
    key = np.zeros(len(order), np.int64)
    key[first] = 1
    leaf = np.cumsum(key)
    idx = np.lexsort((order, leaf))
    return out[idx]


def check_same_tree(r):
    hn, ho, hr2 = probe_bvh(r, binding().BVH_HOST)
    dn, do, dr2 = probe_bvh(r, binding().BVH_DEVICE)
    assert hn.shape == dn.shape
    diff = np.nonzero((hn != dn).any(1))[0]
    assert diff.size == 0, f"{diff.size} of {len(hn)} nodes differ, first {diff[:5]}"
    assert hr2.view(np.uint32) == dr2.view(np.uint32)
    assert np.array_equal(leaf_sets(hn, ho), leaf_sets(dn, do))
    assert np.array_equal(np.sort(do), np.arange(r.n_spheres))


def stats(st):
    return tuple(getattr(st, f) for f in STAT_FIELDS)


def frames(r, n, width, spp):
    """Every frame kind of the resident API over the installed scene: bytes and counters."""
    out = {}
    cam = R.main_camera(width, spp, seed=SEED + n)
    for mode in (R.MODE_PATH, R.MODE_PATH_BVH):
        cam.mode = mode
        img, st = r.render(cam)
        out[f"rgb{mode}"] = (img.cpu().numpy().tobytes(), stats(st))
        _, lin, st = r.render_linear(cam)
        out[f"lin{mode}"] = (lin.cpu().numpy().tobytes(), stats(st))
        alb, nrm, st = r.render_guides(cam, min(spp, 4))
        out[f"guides{mode}"] = (alb.cpu().numpy().tobytes() + nrm.cpu().numpy().tobytes(), stats(st))
        if mode == R.MODE_PATH:
            rgb, dl, _ = r.denoise(lin, alb, nrm)
            out["denoised"] = (rgb.cpu().numpy().tobytes() + dl.cpu().numpy().tobytes(), ())
    legacy = R.Camera()
    R.oracle().orc_camera_legacy(width, 16.0 / 9.0, MODE_LEGACY_NORMAL, C.byref(legacy))
    img, st = r.render(legacy)
    out["legacy"] = (img.cpu().numpy().tobytes(), stats(st))
    return out


def check_both_uploads(r, sp, n, width=48, spp=8, tree=True):
    """host upload vs device upload of one list: rows, every frame, and the device tree against the host tree"""
    r.upload(sp, n)
    rows_h, fr_h = scene_rows(r), frames(r, n, width, spp)
    r.upload(as_tensor(sp, n))
    rows_d = scene_rows(r)
    assert rows_d == rows_h, f"rows differ at byte {next(i for i in range(len(rows_h)) if rows_h[i] != rows_d[i])}" \
        if len(rows_d) == len(rows_h) else (len(rows_d), len(rows_h))
    fr_d = frames(r, n, width, spp)
    for k in fr_h:
        assert fr_d[k][0] == fr_h[k][0], f"{k}: frames differ"
        assert fr_d[k][1] == fr_h[k][1], (k, fr_d[k][1], fr_h[k][1])
    if tree:
        check_same_tree(r)
    return fr_h


# ------------------------------------------------------------------ no GPU
def test_new_kernels_keep_to_registers():
    """Codegen guard (no GPU needed): the install and BVH build kernels are sm_100a code that does not spill."""
    lib = R.ROOT / "raytracing-with-zig_b200" / "csrc" / "librtz.so"
    importlib.import_module("raytracing-with-zig_b200.build").build_all()
    out = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    names = ["scene_check_kernel", "scene_flatten_kernel", "bvh_reach_kernel", "bvh_boxes_kernel", "bvh_init_kernel",
             "bvh_ranges_kernel", "bvh_reduce_kernel", "bvh_node_kernel", "bvh_keys_index_kernel",
             "bvh_keys_axis_kernel", "bvh_descend_kernel"]
    for nm in names:
        want = [k for k in body if nm in k]
        assert len(want) == 1, (nm, want)
        assert not re.search(r"\b(STL|LDL)\b", "\n".join(body[want[0]])), nm


def test_pack_spheres_round_trips_on_the_host(pkg):
    import torch
    sp = random_scene(37, 1)
    arr, n = pkg.renderer._as_sphere_array(sp)
    raw = np.frombuffer(bytes(arr), np.float64).reshape(n, 10).copy()
    words = raw.view(np.int32)
    t = pkg.pack_spheres(torch.from_numpy(raw[:, 0:3].copy()), raw[:, 3], torch.from_numpy(words[:, 8].copy()),
                         raw[:, 5:8], raw[:, 8], raw[:, 9])
    assert t.dtype == torch.float64 and t.shape == (n, 10) and t.is_contiguous()
    assert t.numpy().tobytes() == bytes(arr)


# ------------------------------------------------------------------ one GPU
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 4, 5, 8, 9, 33])
def test_small_scenes(gpu, n):
    check_both_uploads(gpu, random_scene(n, n), n)


@pytest.mark.gpu
def test_final_scene(gpu):
    _, sp, n = R.final_scene(SEED)
    check_both_uploads(gpu, sp, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [512, 513, 7200, 7201, 16384])
def test_sweep_scenes(gpu, n):
    check_both_uploads(gpu, sweep_scene(n), n, width=48 if n < 7200 else 32, spp=8 if n < 7200 else 4)


@pytest.mark.gpu
def test_sweep_scene_of_2_20_spheres(gpu):
    n = 1 << 20
    sp, cnt, _ = gpu.generate(binding().SCENE_SWEEP, 7, n)
    assert cnt == n
    check_both_uploads(gpu, sp, n, width=16, spp=2)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", [equal_axis_scene, signed_zero_scene, nested_glass_scene, far_sphere_scene])
def test_adversarial_scenes(gpu, scene):
    sp = scene()
    check_both_uploads(gpu, sp, len(sp), width=40, spp=4)


BAD = {
    "mat_type": lambda s: setattr(s, "mat_type", 7),
    "radius0": lambda s: setattr(s, "radius", 0.0),
    "nonfinite": lambda s: s.center.__setitem__(1, float("nan")),
    "albedo": lambda s: s.albedo.__setitem__(2, 1.5),
}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [100, 1000])
@pytest.mark.parametrize("kind", sorted(BAD))
def test_refusals_match_the_host_upload(pkg, n, kind):
    B = binding()
    empty = None
    for where in (0, n // 2, n - 1):
        sp = random_scene(n, 5)
        sp[where].mat_type = R.MAT_LAMBERTIAN
        BAD[kind](sp[where])
        r = pkg.Renderer(0)
        if empty is None:
            r.upload(R.sphere_array([]), 0)
            empty = frames(r, 0, 16, 2)["rgb0"]
        with pytest.raises(B.RtzError) as eh:
            r.upload(sp, n)
        rows_h = scene_rows(r)
        with pytest.raises(B.RtzError) as ed:
            r.upload(as_tensor(sp, n))
        assert (ed.value.status, str(ed.value)) == (eh.value.status, str(eh.value)), (where, kind)
        if kind != "mat_type":
            assert f"sphere {where}:" in str(ed.value)
        assert scene_rows(r) == rows_h
        assert frames(r, 0, 16, 2)["rgb0"] == empty  # an empty world
        # a refused list leaves an installed scene as it was
        good = random_scene(n, 6)
        r.upload(as_tensor(good, n))
        rows_good = scene_rows(r)
        with pytest.raises(B.RtzError):
            r.upload(as_tensor(sp, n))
        assert scene_rows(r) == rows_good
        r.close()


@pytest.mark.gpu
def test_refused_pointers_and_sizes(gpu):
    import torch
    l, ctx = gpu.lib, gpu._ctx
    t = as_tensor(random_scene(8, 2), 8)
    assert l.rtz_scene_upload_device(ctx, C.c_void_p(t.data_ptr()), (1 << 20) + 1) == 1
    assert l.rtz_scene_upload_device(ctx, None, 8) == 1
    host = np.zeros((8, 10))
    assert l.rtz_scene_upload_device(ctx, C.c_void_p(host.ctypes.data), 8) == 1
    assert b"device" in l.rtz_last_error()
    pinned = torch.zeros((8, 10), dtype=torch.float64).pin_memory()
    assert l.rtz_scene_upload_device(ctx, C.c_void_p(pinned.data_ptr()), 8) == 1
    with pytest.raises(ValueError):
        gpu.upload(t.cpu())
    with pytest.raises(ValueError):
        gpu.upload(t.float())
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            gpu.upload(t.to("cuda:1"))


@pytest.mark.gpu
def test_device_host_device_on_one_context(pkg, gpu):
    scenes = [sweep_scene(9000, 1), sweep_scene(8000, 2), sweep_scene(700, 3)]
    ref = pkg.Renderer(0)
    cam = R.main_camera(32, 4, seed=SEED)
    cam.mode = R.MODE_PATH_BVH
    for k, sp in enumerate(scenes):
        n = len(sp)
        gpu.upload(as_tensor(sp, n) if k != 1 else sp, n)
        img, st = gpu.render(cam)
        ref.upload(sp, n)
        rimg, rst = ref.render(cam)
        assert np.array_equal(img.cpu().numpy(), rimg.cpu().numpy()) and stats(st) == stats(rst), k
        check_same_tree(gpu)
    ref.close()


@pytest.mark.gpu
def test_tensor_written_by_torch_without_a_synchronise(pkg, gpu):
    import torch
    n = 5000
    g = torch.Generator(device="cuda:0").manual_seed(1)
    for _ in range(3):
        center = torch.rand((n, 3), generator=g, device="cuda:0", dtype=torch.float64) * 40 - 20
        center[:, 1] = center[:, 1].abs() * 0.05
        radius = torch.rand(n, generator=g, device="cuda:0", dtype=torch.float64) * 0.3 + 0.05
        mat = torch.randint(0, 3, (n,), generator=g, device="cuda:0", dtype=torch.int32)
        albedo = torch.rand((n, 3), generator=g, device="cuda:0", dtype=torch.float64)
        t = pkg.pack_spheres(center, radius, mat, albedo, 0.1, 1.5)
        gpu.upload(t)  # no synchronise: the renderer's stream waits for torch's
        rows_d = scene_rows(gpu)
        host = t.cpu().numpy()
        arr = (R.Sphere * n).from_buffer_copy(host.tobytes())
        gpu.upload(arr, n)
        assert scene_rows(gpu) == rows_d
    # pack_spheres writes the records _as_sphere_array writes
    sp = random_scene(20, 9)
    raw = np.frombuffer(bytes(sp), np.float64).reshape(20, 10)
    t = pkg.pack_spheres(torch.tensor(raw[:, 0:3], device="cuda:0"), torch.tensor(raw[:, 3], device="cuda:0"),
                         torch.tensor(raw.view(np.int32)[:, 8], device="cuda:0"), torch.tensor(raw[:, 5:8], device="cuda:0"),
                         torch.tensor(raw[:, 8], device="cuda:0"), torch.tensor(raw[:, 9], device="cuda:0"))
    assert t.cpu().numpy().tobytes() == bytes(pkg.renderer._as_sphere_array(sp)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [513, 16384, 1 << 20])
def test_generated_scene_installs_from_the_device(pkg, gpu, n):
    sp, cnt, _ = gpu.generate(binding().SCENE_SWEEP, 0x5EED, n)
    assert cnt == n
    rows_gen = scene_rows(gpu)
    gen = probe_bvh(gpu, binding().BVH_DEVICE)
    ref = pkg.Renderer(0)
    ref.upload(sp, n)
    assert scene_rows(ref) == rows_gen
    host = probe_bvh(ref, binding().BVH_HOST)
    ref.close()
    assert np.array_equal(gen[0], host[0]) and gen[2].view(np.uint32) == host[2].view(np.uint32)
    assert np.array_equal(leaf_sets(gen[0], gen[1]), leaf_sets(host[0], host[1]))
