"""Denoised frames from shards and from N GPUs: rtz_render_guides_sharded, rtz_deinterleave_f32,
rtz_multi_render_denoised / rtz_render_multi_denoised and distributed.render_sharded_denoised.

The rule every path keeps: the denoised frame of a sharded or N-GPU render equals rtz_render_denoised on one GPU with
the same seed, guide samples and params, bit for bit in the f32 linear colour and byte for byte in the RGB.  It holds
because the linear colour comes from integer pixel sums, each guide pixel folds its own samples in order keyed by its
global pixel index, and the filter runs unchanged over the whole frame on one device.
"""
import ctypes as C
import importlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import rtzlib as R

SEED = 0xDEADBEEF
WORLDS = (1, 2, 3, 8)
TILES = ((4, 4), (16, 16), (7, 5))
GS = (1, 5, 16, 64, 100)
SPP = 100


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _camera(size, spp=SPP, seed=SEED):
    """161x97 (odd: partial tiles on both edges) or 160x90, the reference's main camera otherwise."""
    w, h = size
    cam = R.build_camera(w, w / (h + 0.5), (13, 2, 3), (0, 0, 0), 20, defocus=0.6, spp=spp, seed=seed)
    assert (int(cam.width), int(cam.height)) == size
    return cam


def _sweep_scene(n):
    orc = R.oracle()
    prng = orc.orc_prng_new(7)
    buf = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, buf) == n
    orc.orc_prng_free(prng)
    return buf


def _scene(kind):
    """(spheres, n, mode, whether the constant-bank kernels cull it).  final: the culled constant-bank guide kernel;
    sweep48: the plain constant-bank one; sweep600: the global-memory one; final_bvh: RTZ_MODE_PATH_BVH."""
    if kind in ("final", "final_bvh"):
        _, sp, n = R.final_scene(SEED)
        return sp, n, R.MODE_PATH_BVH if kind == "final_bvh" else R.MODE_PATH, True
    n = {"sweep48": 48, "sweep600": 600}[kind]
    return _sweep_scene(n), n, R.MODE_PATH, False


SCENES = ("final", "sweep48", "sweep600", "final_bvh")


def _bcam(pkg, cam):
    return pkg.rtz_camera.from_buffer_copy(bytes(cam))


def _shard_guides(gpu, cam, g, world, tile):
    """Every rank's compact guides (albedo and normal lists, in rank order)."""
    alb, nrm = [], []
    for rank in range(world):
        a, nn, _ = gpu.render_guides(cam, g, shard=_shard(rank, world, tile))
        alb.append(a), nrm.append(nn)
    return alb, nrm


def _shard(rank, world, tile):
    B = importlib.import_module("raytracing-with-zig_b200.binding")
    return B.rtz_shard(rank, world, tile[0], tile[1])


def _padding_mask(cam, world, tile):
    """[world * per_rank] True where the concatenated compact buffers hold tile padding."""
    dist = importlib.import_module("raytracing-with-zig_b200.distributed")
    per_rank, idx = dist.tile_index_map(int(cam.width), int(cam.height), world, *tile)
    pad = np.ones(world * per_rank, bool)
    pad[idx.reshape(-1)] = False
    return pad


# ------------------------------------------------------------------ no GPU
def test_new_exchange_kernels_keep_to_registers():
    """Codegen guard (no GPU needed): the f32 de-interleave and the resolve that scatters bytes and f32 linear colour
    into device 0's row-major planes do not spill."""
    lib = R.ROOT / "raytracing-with-zig_b200" / "csrc" / "librtz.so"
    importlib.import_module("raytracing-with-zig_b200.build").build_all()
    out = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    want = [k for k in body if "deinterleave_kernelIfE" in k or "resolve_scatter_kernel" in k]
    assert len(want) == 2, want
    for k in want:
        assert not re.search(r"\b(STL|LDL)\b", "\n".join(body[k])), k


# ------------------------------------------------------------------ one GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind", SCENES)
def test_sharded_guides_deinterleave_to_the_whole_frame(pkg, gpu, kind):
    """For every world, tile size, frame size and g: the ranks' compact guides, de-interleaved, are the whole-frame
    guides bit for bit, and the compact padding pixels are 0."""
    import torch
    sp, n, mode, culls = _scene(kind)
    host_culls = C.c_int32(-1)
    boxes = np.zeros(6 * 64, np.float32)
    r2 = C.c_float()
    pkg.binding.check(pkg.lib().rtz_probe_cull_bounds(C.cast(sp, C.POINTER(pkg.rtz_sphere)), n,
                                                      boxes.ctypes.data_as(C.POINTER(C.c_float)), C.byref(r2),
                                                      C.byref(host_culls)))
    assert bool(host_culls.value) == culls
    gpu.upload(sp, n)
    for size in ((161, 97), (160, 90)):
        cam = _camera(size)
        cam.mode = mode
        W, H = size
        for g in GS:
            wa, wn, wst = gpu.render_guides(cam, g)
            wa, wn = bits(wa.cpu().numpy()), bits(wn.cpu().numpy())
            for world in WORLDS:
                for tile in TILES:
                    alb, nrm = _shard_guides(gpu, cam, g, world, tile)
                    pad = _padding_mask(cam, world, tile)
                    for parts, whole in ((alb, wa), (nrm, wn)):
                        cat = torch.cat(parts)
                        assert (cat.cpu().numpy()[pad] == 0).all()
                        assert bits(cat.cpu().numpy()[pad]).max(initial=0) == 0  # +0, not -0
                        img = gpu.deinterleave(cat, W, H, world, *tile)
                        assert np.array_equal(bits(img.cpu().numpy()), whole), (kind, size, g, world, tile)
            # the shards' stats count their own pixels, padding excluded: they add up to the frame's
            tot = 0
            for rank in range(3):
                _, _, st = gpu.render_guides(cam, g, shard=_shard(rank, 3, (7, 5)))
                assert st.kernel_launches == 1 and st.seed_used == SEED
                tot += st.samples
            assert tot == wst.samples == W * H * g


@pytest.mark.gpu
@pytest.mark.parametrize("kind", SCENES)
def test_sharded_linear_colour_deinterleaves_to_the_whole_frame(pkg, gpu, kind):
    import torch
    sp, n, mode, _ = _scene(kind)
    gpu.upload(sp, n)
    for size in ((161, 97), (160, 90)):
        cam = _camera(size, spp=24)
        cam.mode = mode
        W, H = size
        rgb, lin, _ = gpu.render_linear(cam)
        for world in WORLDS:
            for tile in TILES:
                parts = [gpu.render_linear(cam, shard=_shard(r, world, tile)) for r in range(world)]
                img = gpu.deinterleave(torch.cat([p[1] for p in parts]), W, H, world, *tile)
                assert np.array_equal(bits(img.cpu().numpy()), bits(lin.cpu().numpy())), (kind, size, world, tile)
                b = gpu.deinterleave(torch.cat([p[0] for p in parts]), W, H, world, *tile)
                assert torch.equal(b, rgb)


def _sharded_denoise_on_one_device(gpu, cam, g, params, world, tile):
    """The torchrun composition, rank by rank on one device: render_linear + render_guides(shard), concatenated as
    gather_tiles leaves them, de-interleaved and denoised."""
    import torch
    W, H = int(cam.width), int(cam.height)
    lin, alb, nrm = [], [], []
    for r in range(world):
        shard = _shard(r, world, tile)
        lin.append(gpu.render_linear(cam, shard=shard)[1])
        a, nn, _ = gpu.render_guides(cam, g, shard=shard)
        alb.append(a), nrm.append(nn)
    planes = [gpu.deinterleave(torch.cat(p), W, H, world, *tile) for p in (lin, alb, nrm)]
    rgb, out, _ = gpu.denoise(*planes, params=params)
    return rgb.cpu().numpy(), out.cpu().numpy()


def _custom_params(pkg):
    return pkg.rtz_denoise_params(3, 0, 0.5, 0.125, 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", SCENES)
def test_sharded_denoise_equals_render_denoised(pkg, gpu, kind):
    sp, n, mode, _ = _scene(kind)
    gpu.upload(sp, n)
    for size in ((161, 97), (160, 90)):
        cam = _camera(size, spp=16)
        cam.mode = mode
        for params in (None, _custom_params(pkg)):
            ref_rgb, ref_lin, _ = pkg.render_host_denoised(cam, sp, n, 0, params)
            assert ref_rgb.std() > 10
            for world, tile in ((2, (4, 4)), (3, (7, 5)), (8, (16, 16))):
                rgb, lin = _sharded_denoise_on_one_device(gpu, cam, 16, params, world, tile)
                assert np.array_equal(rgb, ref_rgb) and np.array_equal(bits(lin), bits(ref_lin)), (kind, size, world)
    # distributed.render_sharded_denoised without a process group: world 1, tiles de-interleaved on this rank
    cam = _camera((160, 90), spp=16)
    cam.mode = mode
    rgb, lin, st = pkg.render_sharded_denoised(gpu, cam, 5, _custom_params(pkg), tile=(7, 5))
    ref_rgb, ref_lin, ref_st = pkg.render_host_denoised(cam, sp, n, 5, _custom_params(pkg))
    assert np.array_equal(rgb.cpu().numpy(), ref_rgb) and np.array_equal(bits(lin.cpu().numpy()), bits(ref_lin))
    assert (st.samples, st.segments) == (ref_st.samples, ref_st.segments)
    cam.has_seed = 0
    with pytest.raises(ValueError):
        pkg.render_sharded_denoised(gpu, cam)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("final", "final_bvh"))
def test_multi_on_one_device_equals_render_denoised(pkg, kind):
    sp, n, mode, _ = _scene(kind)
    cam = _camera((161, 97), spp=16)
    cam.mode = mode
    for g, params in ((0, None), (7, _custom_params(pkg))):
        ref_rgb, ref_lin, ref = pkg.render_host_denoised(cam, sp, n, g, params)
        m = pkg.MultiRenderer(1)
        m.upload(sp, n)
        for _ in range(2):
            rgb, lin, st = m.render_denoised(cam, g, params)
            assert np.array_equal(rgb, ref_rgb) and np.array_equal(bits(lin), bits(ref_lin))
            assert (st.samples, st.segments, st.sphere_tests, st.kernel_launches, st.gpus, st.seed_used) == \
                (ref.samples, ref.segments, ref.sphere_tests, ref.kernel_launches, 1, SEED)
        m.close()
        rgb, lin, st = pkg.render_host_multi_denoised(cam, sp, n, num_gpus=1, guide_samples=g, params=params)
        assert np.array_equal(rgb, ref_rgb) and np.array_equal(bits(lin), bits(ref_lin)) and st.gpus == 1
    # no seed: one is drawn for the frame and reported; rendering with it gives the same frame
    free = R.Camera.from_buffer_copy(bytes(cam))
    free.has_seed, free.seed = 0, 0
    rgb, lin, st = pkg.render_host_multi_denoised(free, sp, n, num_gpus=1)
    free.has_seed, free.seed = 1, st.seed_used
    rgb2, lin2, _ = pkg.render_host_denoised(free, sp, n)
    assert np.array_equal(rgb, rgb2) and np.array_equal(bits(lin), bits(lin2))


@pytest.mark.gpu
def test_refusals(pkg, gpu):
    import torch
    l = pkg.lib()
    _, sp, n = R.final_scene(SEED)
    gpu.upload(sp, n)
    cam = _camera((160, 90), spp=8)
    buf = torch.empty(160 * 90 * 3 * 4, dtype=torch.float32, device="cuda:0")
    p = C.c_void_p(buf.data_ptr())
    q = C.c_void_p(buf.data_ptr() + 160 * 90 * 3 * 4)

    def variant(**kw):
        c = R.Camera.from_buffer_copy(bytes(cam))
        for k, v in kw.items():
            setattr(c, k, v)
        return _bcam(pkg, c)

    def guides(c=None, shard=(1, 3, 4, 4), g=2, alb=p, nrm=q, ctx=gpu._ctx):
        sh = C.byref(pkg.rtz_shard(*shard)) if shard is not None else None
        return l.rtz_render_guides_sharded(ctx, C.byref(c or _bcam(pkg, cam)), sh, g, alb, nrm, None)

    assert guides() == 0 and guides(shard=None) == 0 and guides(alb=None) == 0 and guides(nrm=None) == 0
    assert guides(alb=None, nrm=None) == 1 and guides(ctx=None) == 1
    assert guides(shard=(3, 3, 4, 4)) == 1 and guides(shard=(0, 0, 4, 4)) == 1
    assert guides(shard=(0, 2, 0, 4)) == 1 and guides(shard=(0, 2, 4, 0)) == 1
    assert guides(variant(mode=R.MODE_LEGACY_NORMAL, samples_per_pixel=1), g=1) == 1
    assert guides(variant(has_seed=0)) == 1
    assert guides(g=0) == 1 and guides(g=9) == 1 and guides(g=8) == 0
    assert guides(variant(t_min=-1e-3)) == 1
    # 2^31 pixels at g >= 64: one work item each, one past the grid's limit (refused before any launch)
    big = variant(width=1 << 16, height=1 << 15, samples_per_pixel=64)
    assert guides(big, shard=None, g=64) == 1 and guides(big, shard=(0, 1, 1 << 16, 1), g=64) == 1
    # rtz_deinterleave_f32 mirrors rtz_deinterleave
    def deint(ctx=gpu._ctx, W=160, H=90, world=2, tw=4, th=4, src=p, dst=q):
        return l.rtz_deinterleave_f32(ctx, W, H, world, tw, th, src, dst)
    assert deint() == 0
    assert deint(ctx=None) == 1 and deint(src=None) == 1 and deint(dst=None) == 1
    assert deint(world=0) == 1 and deint(tw=0) == 1 and deint(th=0) == 1 and deint(W=0) == 1
    # the denoised N-GPU frame: rtz_render_denoised's refusals
    m = pkg.MultiRenderer(1)
    m.upload(sp, n)
    rgb = np.empty(160 * 90 * 3, np.uint8)
    lin = np.empty(160 * 90 * 3, np.float32)
    rp, lp = rgb.ctypes.data_as(C.POINTER(C.c_uint8)), lin.ctypes.data_as(C.POINTER(C.c_float))
    spp_ = C.cast(sp, C.POINTER(pkg.rtz_sphere))

    def multi(c=None, g=0, prm=None, r=rp, li=lp, mm=m._m):
        return l.rtz_multi_render_denoised(mm, C.byref(c or _bcam(pkg, cam)), g, prm, r, li, None)

    def one_shot(c=None, g=0, prm=None, r=rp, li=lp):
        return l.rtz_render_multi_denoised(C.byref(c or _bcam(pkg, cam)), spp_, n, 1, g, prm, r, li, None)

    for fn in (multi, one_shot):
        assert fn() == 0 and fn(r=None) == 0 and fn(li=None) == 0
        assert fn(r=None, li=None) == 1
        assert fn(variant(mode=R.MODE_LEGACY_NORMAL, samples_per_pixel=1)) == 1
        assert fn(g=9) == 1 and fn(g=8) == 0
        assert fn(variant(t_min=-1e-3)) == 1
        for bad in ((9, 0, 1, 1, 1), (3, 1, 1, 1, 1), (3, 0, 0, 1, 1), (3, 0, 1, float("inf"), 1), (3, 0, 1, 1, -1),
                    (8, 0, 1e-37, 1, 1)):
            assert fn(prm=C.byref(pkg.rtz_denoise_params(*bad))) == 1, bad
        assert fn(variant(width=1 << 16, height=1 << 15)) == 1  # 2^31 pixels: one past the denoiser's limit
    assert multi(mm=None) == 1
    assert l.rtz_render_multi_denoised(C.byref(_bcam(pkg, cam)), None, n, 1, 0, None, rp, lp, None) == 1
    m.close()


# ------------------------------------------------------------------ two or more GPUs
def _ngpu():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.parametrize("gather", ["p2p", "nccl"])
def test_multi_gpu_denoised_equals_single_gpu(pkg, gather):
    ngpu = _ngpu()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    _, sp, n = R.final_scene(SEED)
    cam = _camera((161, 97), spp=16)
    params = _custom_params(pkg)
    ref_rgb, ref_lin, ref = pkg.render_host_denoised(cam, sp, n, 0, params)
    for world in sorted({2, min(ngpu, 3), ngpu}):
        for tile in TILES:
            m = pkg.MultiRenderer(world, tile=tile, gather=gather)
            assert (m.gpus, m.gather) == (world, gather)
            m.upload(sp, n)
            for _ in range(2):  # twice: buffers are reused from frame to frame
                rgb, lin, st = m.render_denoised(cam, 0, params)
                assert np.array_equal(rgb, ref_rgb) and np.array_equal(bits(lin), bits(ref_lin)), (world, tile, gather)
                assert (st.samples, st.segments, st.sphere_tests, st.depth_capped, st.absorbed, st.nan_samples) == \
                    (ref.samples, ref.segments, ref.sphere_tests, ref.depth_capped, ref.absorbed, ref.nan_samples)
                assert (st.gpus, st.gather, st.seed_used) == (world, m.lib.rtz_multi_gather(m._m), SEED)
                assert st.total_ms >= st.trace_ms > 0
            m.close()
    m = pkg.MultiRenderer(2, devices=[1, 0], gather=gather)
    m.upload(sp, n)
    rgb, lin, _ = m.render_denoised(cam, 0, params)
    assert np.array_equal(rgb, ref_rgb) and np.array_equal(bits(lin), bits(ref_lin))
    m.close()
    rgb, lin, st = pkg.render_host_multi_denoised(cam, sp, n, num_gpus=0, params=params)
    assert np.array_equal(rgb, ref_rgb) and np.array_equal(bits(lin), bits(ref_lin)) and st.gpus == ngpu


WORKER = r'''
import importlib, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["RTZ_ROOT"])
sys.path.insert(0, os.path.join(os.environ["RTZ_ROOT"], "tests"))
import rtzlib as R
rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device(f"cuda:{lr}"))
pkg = importlib.import_module("raytracing-with-zig_b200")
_, sp, n = R.final_scene(0xDEADBEEF)
cam = R.build_camera(161, 161 / 97.5, (13, 2, 3), (0, 0, 0), 20, defocus=0.6, spp=16, seed=0xDEADBEEF)
r = pkg.Renderer(lr)
r.upload(sp, n)
rgb, lin, st = pkg.render_sharded_denoised(r, cam, 0, None, (7, 5))
if rank == 0:
    ref_rgb, ref_lin, _ = pkg.render_host_denoised(cam, sp, n)
    assert np.array_equal(rgb.cpu().numpy(), ref_rgb), "sharded denoised bytes differ from the 1-GPU frame"
    assert np.array_equal(lin.cpu().numpy().view(np.uint32), ref_lin.view(np.uint32)), "linear colour differs"
    np.save(os.environ["RTZ_OUT"], rgb.cpu().numpy())
else:
    assert rgb is None and lin is None
dist.barrier()
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_torchrun_sharded_denoised_equals_single_gpu(tmp_path):
    ngpu = _ngpu()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = tmp_path / "rgb.npy"
    env = dict(os.environ, RTZ_ROOT=str(R.ROOT), RTZ_OUT=str(out))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(ngpu, 8)}",
                        "--master-addr", "127.0.0.1", "--master-port", "29543", str(script)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert np.load(out).shape == (97, 161, 3)
