"""raytracing-with-zig_b200 — B200-native `Camera.render` for AndrewJarrett/raytracing-with-zig.

Only what the hot path needs:
  csrc/            hand-written sm_100a CUDA kernels + the C ABI (include/rtz.h) -> librtz.so
  host/            C++ mirror of the reference's Scene/Camera/Hittable/Material/PPM API above the ABI
  zig/             the Zig glue a reference maintainer would drop in (see INTEGRATION.md)
  binding.py       ctypes view of the ABI (raises when librtz.so is missing: no fallback)
  renderer.py      resident renderer on torch device memory / streams (render, denoiser inputs, denoise); MultiRenderer = N GPUs in one process (rtz_multi)
  distributed.py   interleaved-tile sharding + NCCL gather (one process per GPU)
"""
from .binding import RtzError, lib, rtz_camera, rtz_denoise_params, rtz_shard, rtz_sphere, rtz_stats  # noqa: F401
from .renderer import (MultiRenderer, Renderer, pack_spheres, render_host, render_host_denoised,  # noqa: F401
                       render_host_multi, render_host_multi_denoised)
from .distributed import render_sharded, render_sharded_denoised, tile_index_map  # noqa: F401
