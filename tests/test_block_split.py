"""The culled sweep's sphere-parallel pass against the f32 mirror, bit for bit.

A culled 32-sphere block that at most `split_max` of the warp's 64 paths reach is swept sphere-parallel: lane l
takes sphere base + l, and only the paths whose own box test admits the block are tested, one broadcast ray at a
time.  Every other block keeps the packed two-sphere sweep.  RTZ_SPLIT (read for each frame) overrides
the threshold: 0 is the packed sweep alone, 64 splits every reached block.  The image, the pixel sums and every
work counter must not depend on it.  The scenes are those that press on the cull (grazing rows, axis-parallel
rays, a camera inside a block's box, a large sphere among small ones, duplicates, equal-t ties across regrouped
blocks), a last block of fewer than 32 spheres, and a camera beyond the padding's radius R, where every block is
needed.  Each is rendered with the drain kernel on and off, whole and as one shard of three.
"""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import rtzlib as R
from test_block_cull import CAMERAS, _grid_scene
from test_block_regroup import _reversed_pair, _scene

SPLITS = ["0", "64", None]  # None: the built-in threshold


def test_split_kernel_keeps_its_registers_and_the_uniform_sweep(pkg):
    """Codegen guard (no GPU needed): the sphere-parallel branch must not make the culled kernel spill, and the
    packed loop must keep its sphere operands in uniform registers."""
    out = subprocess.run(["cuobjdump", "-sass", str(pkg.binding.LIB_PATH)], capture_output=True, text=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    culled = [k for k in body if "trace_kernel_const_cullILi128ELi6" in k]
    assert len(culled) == 1, culled
    sass = "\n".join(body[culled[0]])
    assert not re.search(r"\b(STL|LDL)\b", sass), "the culled kernel spills to local memory"
    assert len(re.findall(r"FFMA2 [^;]*UR\d+\.F32x2", sass)) >= 48
    assert "BRA.DIV" not in sass


def _cases():
    c = []
    for view in CAMERAS:
        c.append(("plain", view))
    c += [("big", "inside"), ("big", "final"), ("duplicates", "grazing"), ("duplicates", "final"),
          ("plain", "beyond_r"), ("ties_ground_first", None), ("ties_ground_later", None)]
    return c


def _setup(pkg, kind, view):
    if kind.startswith("ties"):
        sp, pairs = _scene(kind == "ties_ground_first")
        first, second, x0, z0 = _reversed_pair(pkg, sp, pairs)
        cam = R.build_camera(8, 1.0, (x0, 1.0, z0 + 30.0), (x0, 1.0, z0), 0.0, spp=256, seed=0xBEEF)
        return R.sphere_array(sp), len(sp), cam
    sp, n = _grid_scene(big=kind == "big", duplicates=kind == "duplicates")
    if view == "beyond_r":
        # the ground reaches 2000 from the world origin: primary rays start beyond the padded radius
        cam = R.build_camera(96, 16.0 / 9.0, (0.0, 40.0, 6000.0), (0.0, 0.0, 0.0), 0.3, spp=16, seed=0xC0FFEE)
    else:
        cam = R.build_camera(96, 16.0 / 9.0, spp=16, seed=0xC0FFEE, **CAMERAS[view])
    return sp, n, cam


def _mirror(orc, cam, sp, n, seed, shard=None):
    if shard is None:
        npix = cam.width * cam.height
    else:
        tiles_x = (cam.width + shard.tile_w - 1) // shard.tile_w
        tiles_y = (cam.height + shard.tile_h - 1) // shard.tile_h
        npix = ((tiles_x * tiles_y + shard.world - 1) // shard.world) * shard.tile_w * shard.tile_h
    rgb = np.zeros((npix, 3), np.uint8)
    lin = np.zeros((npix, 3), np.float64)
    st = R.Stats()
    assert orc.orc_render_mirror(C.byref(cam), sp, n, seed, 8, C.byref(shard) if shard is not None else None,
                                 rgb.ctypes.data_as(C.POINTER(C.c_uint8)), lin.ctypes.data_as(C.POINTER(C.c_double)),
                                 C.byref(st)) == 0
    return rgb, lin, st


def _key(st):
    return st.samples, st.segments, st.depth_capped, st.absorbed, st.nan_samples


@pytest.mark.gpu
@pytest.mark.parametrize("kind,view", _cases(), ids=[f"{k}-{v}" if v else k for k, v in _cases()])
def test_split_sweep_matches_mirror_bit_exact(pkg, gpu, orc, monkeypatch, kind, view):
    sp, n, cam = _setup(pkg, kind, view)
    assert 257 <= n <= 512
    if not kind.startswith("ties"):
        assert (n + 7) // 8 * 8 % 32 != 0  # the grid scenes end on a block of fewer than 32 spheres
    mrgb, mlin, mst = _mirror(orc, cam, sp, n, cam.seed)
    msh = R.Shard(1, 3, 4, 4)
    srgb, _, sst = _mirror(orc, cam, sp, n, cam.seed, msh)
    sh = pkg.rtz_shard(1, 3, 4, 4)
    gpu.upload(sp, n)
    for split in SPLITS:
        for drain in ("1", "0"):
            if split is None:
                monkeypatch.delenv("RTZ_SPLIT", raising=False)
            else:
                monkeypatch.setenv("RTZ_SPLIT", split)
            monkeypatch.setenv("RTZ_DRAIN", drain)
            what = f"RTZ_SPLIT={split} RTZ_DRAIN={drain}"
            rgb, st, lin = pkg.render_host(cam, sp, n, want_linear=True)
            assert _key(st) == _key(mst), what
            assert st.sphere_tests == st.segments * n == mst.sphere_tests, what
            assert np.array_equal(lin.reshape(-1, 3), mlin), f"{what}: {np.count_nonzero(lin.reshape(-1, 3) != mlin)} sums differ"
            assert np.array_equal(rgb.reshape(-1, 3), mrgb), what
            img, st = gpu.render(cam, sh)
            assert np.array_equal(img.cpu().numpy().reshape(-1, 3), srgb), what
            assert _key(st) == _key(sst), what
