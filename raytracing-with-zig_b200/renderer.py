"""Resident renderer: scene and frame stay in HBM; PyTorch supplies device memory and the stream.

`Renderer.render` is the Python face of `Camera.render` (reference src/camera.zig:123-145) on one
GPU; the arithmetic happens in csrc/ (hand-written sm_100a kernels) behind include/rtz.h.
"""
from __future__ import annotations

import ctypes as C

from . import binding as B


def _as_sphere_array(spheres):
    if isinstance(spheres, C.Array):
        return spheres, len(spheres)
    arr = (B.rtz_sphere * len(spheres))()
    for i, s in enumerate(spheres):
        C.memmove(C.byref(arr, i * C.sizeof(B.rtz_sphere)), C.byref(s), C.sizeof(B.rtz_sphere))
    return arr, len(spheres)


def pack_spheres(center, radius, mat_type, albedo, fuzz, refraction_index):
    """`rtz_sphere` records built on the device with torch ops: a contiguous float64 [n, 10] tensor on the device of
    `center` (column 4 holds the int32 pair (mat_type, reserved = 0)), what `Renderer.upload` installs without a host
    round trip.  center, albedo: [n, 3]; radius, mat_type, fuzz, refraction_index: [n] (or anything that broadcasts)."""
    import torch

    center = torch.as_tensor(center)
    n, dev = center.shape[0], center.device
    out = torch.empty((n, 10), dtype=torch.float64, device=dev)
    f64 = dict(dtype=torch.float64, device=dev)
    out[:, 0:3] = torch.as_tensor(center, **f64)
    out[:, 3] = torch.as_tensor(radius, **f64)
    out[:, 5:8] = torch.as_tensor(albedo, **f64)
    out[:, 8] = torch.as_tensor(fuzz, **f64)
    out[:, 9] = torch.as_tensor(refraction_index, **f64)
    words = out.view(torch.int32)  # [n, 20]: column 4 is words 8 (mat_type) and 9 (reserved)
    words[:, 8] = torch.as_tensor(mat_type, dtype=torch.int32, device=dev)
    words[:, 9] = 0
    return out


def _cast_camera(cam) -> B.rtz_camera:
    """Accept any ctypes struct with the rtz_camera layout (tests use their own mirror class)."""
    if isinstance(cam, B.rtz_camera):
        return cam
    assert C.sizeof(cam) == C.sizeof(B.rtz_camera)
    out = B.rtz_camera()
    C.memmove(C.byref(out), C.byref(cam), C.sizeof(out))
    return out


class Renderer:
    """One rtz_context bound to a CUDA device and to a torch stream of its own on it.

    Stream ordering: the library launches everything on `self.stream` (a real `torch.cuda.Stream`, so its
    handle is never the NULL that `rtz_context_create` reads as "make your own stream").  Every call first
    makes that stream wait for torch's current stream (`_order_after_torch`), so tensors produced by torch or
    by a collective (the NCCL tile gather makes the current stream wait for its result) are complete before
    the library reads them; every library call blocks until its own work is done, so results are complete
    for whatever torch does next."""

    def __init__(self, device: int | None = None):
        import torch

        if not torch.cuda.is_available():
            raise B.RtzError(2, "no CUDA device: raytracing-with-zig_b200 has no CPU fallback")
        self.torch = torch
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.lib = B.lib()
        self.stream = torch.cuda.Stream(device=self.device)
        assert self.stream.cuda_stream != 0
        self._ctx = C.c_void_p()
        B.check(self.lib.rtz_context_create(self.device, C.c_void_p(self.stream.cuda_stream), C.byref(self._ctx)))
        self.n_spheres = 0

    def _order_after_torch(self):
        self.stream.wait_stream(self.torch.cuda.current_stream(self.device))

    def close(self):
        if self._ctx:
            self.lib.rtz_context_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, spheres, n: int | None = None):
        """HittableList.add for the whole list: flatten to the device SoA and copy to HBM.  A CUDA tensor of
        `rtz_sphere` records (float64 [n, 10], contiguous, on this renderer's device: `pack_spheres`) is installed
        from device memory (`rtz_scene_upload_device`), ordered after torch's current stream."""
        torch = self.torch
        if isinstance(spheres, torch.Tensor):
            t = spheres
            if not t.is_cuda or t.device.index != self.device:
                raise ValueError(f"spheres on {t.device}: this renderer installs device tensors of cuda:{self.device}")
            if t.dtype != torch.float64 or t.dim() != 2 or t.shape[1] != 10 or not t.is_contiguous():
                raise ValueError("spheres must be a contiguous float64 [n, 10] tensor of rtz_sphere records")
            n = t.shape[0] if n is None else int(n)
            if n > t.shape[0]:
                raise ValueError(f"n = {n} but the tensor holds {t.shape[0]} spheres")
            self._order_after_torch()
            B.check(self.lib.rtz_scene_upload_device(self._ctx, C.c_void_p(t.data_ptr() if n else 0), n))
            self.n_spheres = n
            return
        arr, cnt = _as_sphere_array(spheres)
        n = cnt if n is None else int(n)
        ptr = C.cast(arr, C.POINTER(B.rtz_sphere))
        B.check(self.lib.rtz_scene_upload(self._ctx, ptr, n))
        self.n_spheres = n

    def generate(self, kind: int, seed: int, n: int = 0):
        """Scene.init(seed) + generateWorld / generateChapter13 / the config-5 sweep scene, generated on the
        device with the reference's PRNG stream and installed as this renderer's scene.
        Returns (spheres, count, prng_state): the f64 spheres in list order and Scene.prng after generation."""
        cap = int(n) if kind == B.SCENE_SWEEP else 22 * 22 + 4
        arr = (B.rtz_sphere * max(cap, 1))()
        cnt = C.c_uint64(0)
        state = (C.c_uint64 * 4)()
        B.check(self.lib.rtz_scene_generate(self._ctx, int(kind), C.c_uint64(seed), C.c_uint64(n), arr, cap,
                                            C.byref(cnt), state))
        self.n_spheres = int(cnt.value)
        return arr, int(cnt.value), [int(x) for x in state]

    def shard_pixels(self, width: int, height: int, shard: B.rtz_shard | None) -> int:
        return int(self.lib.rtz_shard_pixels(width, height, C.byref(shard) if shard is not None else None))

    def render(self, camera, shard: B.rtz_shard | None = None, out=None):
        """Render the frame (or this rank's tiles) into a device uint8 tensor; returns (tensor, stats)."""
        torch = self.torch
        cam = _cast_camera(camera)
        if shard is None:
            shape = (int(cam.height), int(cam.width), 3)
        else:
            shape = (self.shard_pixels(cam.width, cam.height, shard), 3)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=f"cuda:{self.device}")
        assert out.is_cuda and out.is_contiguous() and out.dtype == torch.uint8 and out.numel() == shape[0] * shape[1] * (shape[2] if len(shape) == 3 else 1)
        st = B.rtz_stats()
        self._order_after_torch()
        B.check(self.lib.rtz_render_resident(self._ctx, C.byref(cam), C.byref(shard) if shard is not None else None,
                                             C.c_void_p(out.data_ptr()), C.byref(st)))
        return out, st

    def render_linear(self, camera, shard: B.rtz_shard | None = None, out=None, linear=None):
        """`render`, plus the linear colour before gamma and quantisation (the noisy input of a denoiser) as a
        float32 device tensor of the same shape; returns (uint8 tensor, float32 tensor, stats)."""
        torch = self.torch
        cam = _cast_camera(camera)
        if shard is None:
            shape = (int(cam.height), int(cam.width), 3)
        else:
            shape = (self.shard_pixels(cam.width, cam.height, shard), 3)
        dev = f"cuda:{self.device}"
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=dev)
        if linear is None:
            linear = torch.empty(shape, dtype=torch.float32, device=dev)
        for t, dt in ((out, torch.uint8), (linear, torch.float32)):
            assert t.is_cuda and t.is_contiguous() and t.dtype == dt and tuple(t.shape) == shape, (t.shape, t.dtype)
        st = B.rtz_stats()
        self._order_after_torch()
        B.check(self.lib.rtz_render_resident_linear(self._ctx, C.byref(cam),
                                                    C.byref(shard) if shard is not None else None,
                                                    C.c_void_p(out.data_ptr()), C.c_void_p(linear.data_ptr()),
                                                    C.byref(st)))
        return out, linear, st

    def render_guides(self, camera, samples: int, albedo=None, normal=None, shard: B.rtz_shard | None = None):
        """First-hit denoiser guides of the frame's camera rays, samples 0 .. samples-1 of every pixel (the camera
        needs its seed): float32 [H, W, 3] device tensors (albedo, normal), or [shard_pixels, 3] in the compact tile
        layout for a shard; returns (albedo, normal, stats)."""
        torch = self.torch
        cam = _cast_camera(camera)
        if shard is None:
            shape = (int(cam.height), int(cam.width), 3)
        else:
            shape = (self.shard_pixels(cam.width, cam.height, shard), 3)
        dev = f"cuda:{self.device}"
        if albedo is None:
            albedo = torch.empty(shape, dtype=torch.float32, device=dev)
        if normal is None:
            normal = torch.empty(shape, dtype=torch.float32, device=dev)
        for t in (albedo, normal):
            assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float32 and tuple(t.shape) == shape, (t.shape, t.dtype)
        st = B.rtz_stats()
        self._order_after_torch()
        a, n = C.c_void_p(albedo.data_ptr()), C.c_void_p(normal.data_ptr())
        if shard is None:
            B.check(self.lib.rtz_render_guides(self._ctx, C.byref(cam), int(samples), a, n, C.byref(st)))
        else:
            B.check(self.lib.rtz_render_guides_sharded(self._ctx, C.byref(cam), C.byref(shard), int(samples), a, n,
                                                       C.byref(st)))
        return albedo, normal, st

    def denoise(self, linear, albedo, normal, params: B.rtz_denoise_params | None = None, out_linear=None,
                out_rgb=None):
        """Denoise a whole frame (`rtz_denoise`): the float32 [H, W, 3] device tensors of `render_linear` and
        `render_guides`; returns (uint8 tensor, float32 tensor, stats) of the denoised frame."""
        torch = self.torch
        shape = tuple(linear.shape)
        assert len(shape) == 3 and shape[2] == 3, shape
        dev = f"cuda:{self.device}"
        if out_linear is None:
            out_linear = torch.empty(shape, dtype=torch.float32, device=dev)
        if out_rgb is None:
            out_rgb = torch.empty(shape, dtype=torch.uint8, device=dev)
        for t, dt in ((linear, torch.float32), (albedo, torch.float32), (normal, torch.float32),
                      (out_linear, torch.float32), (out_rgb, torch.uint8)):
            assert t.is_cuda and t.is_contiguous() and t.dtype == dt and tuple(t.shape) == shape, (t.shape, t.dtype)
        st = B.rtz_stats()
        self._order_after_torch()
        B.check(self.lib.rtz_denoise(self._ctx, shape[1], shape[0], C.c_void_p(linear.data_ptr()),
                                     C.c_void_p(albedo.data_ptr()), C.c_void_p(normal.data_ptr()),
                                     C.byref(params) if params is not None else None,
                                     C.c_void_p(out_linear.data_ptr()), C.c_void_p(out_rgb.data_ptr()), C.byref(st)))
        return out_rgb, out_linear, st

    def deinterleave(self, gathered, width: int, height: int, world: int, tile_w: int, tile_h: int, out=None):
        """`world` compact tile buffers back to back -> the row-major [H, W, 3] frame: uint8 (the bytes) or float32
        (linear colour, guides)."""
        torch = self.torch
        fn = {torch.uint8: self.lib.rtz_deinterleave, torch.float32: self.lib.rtz_deinterleave_f32}[gathered.dtype]
        assert gathered.is_cuda and gathered.is_contiguous()
        if out is None:
            out = torch.empty((height, width, 3), dtype=gathered.dtype, device=gathered.device)
        assert out.dtype == gathered.dtype and out.is_contiguous() and out.numel() == height * width * 3
        self._order_after_torch()   # `gathered` may still be in flight on torch's / NCCL's streams
        B.check(fn(self._ctx, width, height, world, tile_w, tile_h, C.c_void_p(gathered.data_ptr()),
                   C.c_void_p(out.data_ptr())))
        return out


class MultiRenderer:
    """`rtz_multi`: ONE process driving N GPUs of the box behind the C ABI (no torchrun, no torch.distributed).

    The frame is cut into interleaved tiles, every device traces its tiles, and the bytes reach device 0 either
    through the fused resolve + peer-memory store (`gather="p2p"`) or a grouped ncclSend/ncclRecv (`"nccl"`)."""

    def __init__(self, num_gpus: int = 0, devices=None, tile=(4, 4), gather: str = "auto"):
        self.lib = B.lib()
        self._m = C.c_void_p()
        devs = (C.c_int32 * len(devices))(*devices) if devices else None
        g = {"auto": B.GATHER_AUTO, "p2p": B.GATHER_P2P, "nccl": B.GATHER_NCCL}[gather]
        B.check(self.lib.rtz_multi_create(int(num_gpus), devs, int(tile[0]), int(tile[1]), g, C.byref(self._m)))
        self.gpus = int(self.lib.rtz_multi_gpus(self._m))
        self.gather = {B.GATHER_P2P: "p2p", B.GATHER_NCCL: "nccl"}[int(self.lib.rtz_multi_gather(self._m))]

    def close(self):
        if self._m:
            self.lib.rtz_multi_destroy(self._m)
            self._m = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, spheres, n: int | None = None):
        arr, cnt = _as_sphere_array(spheres)
        n = cnt if n is None else int(n)
        B.check(self.lib.rtz_multi_scene_upload(self._m, C.cast(arr, C.POINTER(B.rtz_sphere)), n))

    def render(self, camera, to_host: bool = True):
        """Returns (numpy uint8 [H,W,3] or None, stats); the image also stays resident on device 0."""
        import numpy as np

        cam = _cast_camera(camera)
        H, W = int(cam.height), int(cam.width)
        rgb = np.empty((H, W, 3), dtype=np.uint8) if to_host else None
        st = B.rtz_stats()
        ptr = rgb.ctypes.data_as(C.POINTER(C.c_uint8)) if to_host else None
        B.check(self.lib.rtz_multi_render(self._m, C.byref(cam), ptr, None, C.byref(st)))
        return rgb, st

    def render_denoised(self, camera, guide_samples: int = 0, params: B.rtz_denoise_params | None = None):
        """`rtz_multi_render_denoised`: the frame on every device, denoised on device 0 — the bytes and linear
        colour of `render_host_denoised`.  Returns (numpy uint8 [H,W,3], numpy float32 [H,W,3], stats)."""
        import numpy as np

        cam = _cast_camera(camera)
        H, W = int(cam.height), int(cam.width)
        rgb = np.empty((H, W, 3), dtype=np.uint8)
        lin = np.empty((H, W, 3), dtype=np.float32)
        st = B.rtz_stats()
        B.check(self.lib.rtz_multi_render_denoised(self._m, C.byref(cam), int(guide_samples),
                                                   C.byref(params) if params is not None else None,
                                                   rgb.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                   lin.ctypes.data_as(C.POINTER(C.c_float)), C.byref(st)))
        return rgb, lin, st


def render_host_multi(camera, spheres, n: int | None = None, num_gpus: int = 0):
    """`rtz_render_multi`: the one-shot C-ABI call with HOST buffers on `num_gpus` devices (0 = all)."""
    import numpy as np

    l = B.lib()
    cam = _cast_camera(camera)
    arr, cnt = _as_sphere_array(spheres)
    n = cnt if n is None else int(n)
    rgb = np.empty((int(cam.height), int(cam.width), 3), dtype=np.uint8)
    st = B.rtz_stats()
    B.check(l.rtz_render_multi(C.byref(cam), C.cast(arr, C.POINTER(B.rtz_sphere)), n, int(num_gpus),
                               rgb.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(st)))
    return rgb, st


def render_host_multi_denoised(camera, spheres, n: int | None = None, num_gpus: int = 0, guide_samples: int = 0,
                               params: B.rtz_denoise_params | None = None):
    """`rtz_render_multi_denoised`: `render_host_denoised` on `num_gpus` devices (0 = all), denoised on the first.
    Returns (numpy uint8 [H,W,3], numpy float32 [H,W,3], stats)."""
    import numpy as np

    l = B.lib()
    cam = _cast_camera(camera)
    arr, cnt = _as_sphere_array(spheres)
    n = cnt if n is None else int(n)
    H, W = int(cam.height), int(cam.width)
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    lin = np.empty((H, W, 3), dtype=np.float32)
    st = B.rtz_stats()
    B.check(l.rtz_render_multi_denoised(C.byref(cam), C.cast(arr, C.POINTER(B.rtz_sphere)), n, int(num_gpus),
                                        int(guide_samples), C.byref(params) if params is not None else None,
                                        rgb.ctypes.data_as(C.POINTER(C.c_uint8)),
                                        lin.ctypes.data_as(C.POINTER(C.c_float)), C.byref(st)))
    return rgb, lin, st


def render_host_denoised(camera, spheres, n: int | None = None, guide_samples: int = 0,
                         params: B.rtz_denoise_params | None = None):
    """`rtz_render_denoised`: the one-shot C-ABI call with HOST buffers, render + guides + denoise.
    Returns (numpy uint8 [H,W,3], numpy float32 [H,W,3] denoised linear colour, stats)."""
    import numpy as np

    l = B.lib()
    cam = _cast_camera(camera)
    arr, cnt = _as_sphere_array(spheres)
    n = cnt if n is None else int(n)
    H, W = int(cam.height), int(cam.width)
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    lin = np.empty((H, W, 3), dtype=np.float32)
    st = B.rtz_stats()
    B.check(l.rtz_render_denoised(C.byref(cam), C.cast(arr, C.POINTER(B.rtz_sphere)), n, int(guide_samples),
                                  C.byref(params) if params is not None else None,
                                  rgb.ctypes.data_as(C.POINTER(C.c_uint8)), lin.ctypes.data_as(C.POINTER(C.c_float)),
                                  C.byref(st)))
    return rgb, lin, st


def render_host(camera, spheres, n: int | None = None, want_linear: bool = False):
    """The one-shot C-ABI call with HOST buffers (`rtz_render`): what a Zig/C host would call.

    Returns (numpy uint8 [H,W,3], stats[, numpy float64 [H,W,3]]).  Host->device copy of the scene
    and device->host copy of the image happen inside the call."""
    import numpy as np

    l = B.lib()
    cam = _cast_camera(camera)
    arr, cnt = _as_sphere_array(spheres)
    n = cnt if n is None else int(n)
    H, W = int(cam.height), int(cam.width)
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    st = B.rtz_stats()
    sp = C.cast(arr, C.POINTER(B.rtz_sphere))
    if want_linear:
        lin = np.empty((H, W, 3), dtype=np.float64)
        B.check(l.rtz_render_linear(C.byref(cam), sp, n, rgb.ctypes.data_as(C.POINTER(C.c_uint8)),
                                    lin.ctypes.data_as(C.POINTER(C.c_double)), C.byref(st)))
        return rgb, st, lin
    B.check(l.rtz_render(C.byref(cam), sp, n, rgb.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(st)))
    return rgb, st
