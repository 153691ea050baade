"""The culled constant-bank sweep (trace_kernel_const<128,6,true>) against the f32 mirror, bit for bit.

The kernel skips a block of 32 spheres when no path of the warp can reach the block's padded box over
(0, closest]; a skip that dropped an accepted root would change a pixel or a counter.  The scenes below have
257-512 spheres laid out like the book's final scene (a ground sphere first, then small spheres row by row, so
that every block is a compact strip and the host turns the cull on), with the cases that press on the bound:
spheres at the extremes of their rows (tangent to their block's box faces) seen by grazing camera rays, rays
nearly parallel to the axes (huge reciprocals), a camera inside a block's box, a large sphere inside a block of
small ones, and exact duplicates of spheres in later blocks (ties in t, where the earlier sphere must win).
"""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import rtzlib as R


def test_culled_sweep_stays_on_the_uniform_datapath(pkg):
    """Codegen guard (no GPU needed): the block vote must not cost the culled kernel the packed sweep on uniform
    registers fed by LDCU, nor put a vote behind BRA.DIV."""
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
    assert len(re.findall(r"FFMA2 [^;]*UR\d+\.F32x2", sass)) >= 48, "sweep operands are no longer uniform registers"
    assert "BRA.DIV" not in sass and "LDCU.64" in sass


def _grid_scene(big=False, duplicates=False):
    rng = np.random.default_rng(7)
    sp = [R.make_sphere((0, -1000, 0), 1000, R.MAT_LAMBERTIAN, (0.5, 0.5, 0.5))]
    for a in range(-10, 10):
        for b in range(-10, 10):
            # every fourth row sits at the extremes of its cell: its spheres touch the faces of the block's box
            jx, jz = (0.0, 0.8 * (b % 2)) if a % 4 == 0 else tuple(0.8 * rng.random(2))
            kind = rng.random()
            c = (a + 0.1 + jx, 0.2, b + 0.1 + jz)
            if kind < 0.6:
                sp.append(R.make_sphere(c, 0.2, R.MAT_LAMBERTIAN, tuple(0.2 + 0.6 * rng.random(3))))
            elif kind < 0.85:
                sp.append(R.make_sphere(c, 0.2, R.MAT_METAL, tuple(0.5 + 0.5 * rng.random(3)), fuzz=0.0 if kind < 0.7 else 0.3))
            else:
                sp.append(R.make_sphere(c, 0.2, R.MAT_DIELECTRIC, ior=1.5))
    if big:  # a large sphere in the middle of a block of small ones
        sp[200] = R.make_sphere((sp[200].center[0], 1.5, sp[200].center[2]), 1.5, R.MAT_METAL, (0.7, 0.6, 0.5))
    if duplicates:  # exact copies in later blocks: equal roots, the lower index must win
        for i in (5, 40, 77, 150, 233):
            s = sp[i]
            sp.append(R.make_sphere(tuple(s.center), s.radius, R.MAT_LAMBERTIAN, (0.9, 0.1, 0.1)))
    return R.sphere_array(sp), len(sp)


CAMERAS = {
    # grazing: the eye at the height of the small spheres' tops, looking along a row
    "grazing": dict(look_from=(14.0, 0.4, 0.5), look_at=(0.0, 0.4, 0.5), vfov=30),
    # nearly axis-parallel rays (reciprocals of order 1e4): a narrow field of view straight down -z
    "axis": dict(look_from=(0.5, 0.2, 30.0), look_at=(0.5, 0.2, 0.0), vfov=0.01),
    # the eye inside the slab of small spheres, i.e. inside a block's box
    "inside": dict(look_from=(0.5, 0.3, 0.55), look_at=(6.0, 0.1, 4.0), vfov=60),
    # the book's view, with defocus
    "final": dict(look_from=(13, 2, 3), look_at=(0, 0, 0), vfov=20, defocus=0.6),
}


def _mirror(orc, cam, sp, n, seed):
    npix = cam.width * cam.height
    rgb = np.zeros((npix, 3), np.uint8)
    lin = np.zeros((npix, 3), np.float64)
    st = R.Stats()
    assert orc.orc_render_mirror(C.byref(cam), sp, n, seed, 8, None, rgb.ctypes.data_as(C.POINTER(C.c_uint8)),
                                 lin.ctypes.data_as(C.POINTER(C.c_double)), C.byref(st)) == 0
    return rgb, lin, st


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["plain", "big", "duplicates"])
@pytest.mark.parametrize("view", list(CAMERAS))
def test_culled_sweep_matches_mirror_bit_exact(pkg, gpu, orc, scene, view):
    sp, n = _grid_scene(big=scene == "big", duplicates=scene == "duplicates")
    assert 257 <= n <= 512
    cam = R.build_camera(160, 16.0 / 9.0, spp=24, seed=0xC0FFEE, **CAMERAS[view])
    rgb, st, lin = pkg.render_host(cam, sp, n, want_linear=True)
    mrgb, mlin, mst = _mirror(orc, cam, sp, n, 0xC0FFEE)
    assert (st.samples, st.segments, st.depth_capped, st.absorbed, st.nan_samples) == (
        mst.samples, mst.segments, mst.depth_capped, mst.absorbed, mst.nan_samples)
    assert st.sphere_tests == st.segments * n == mst.sphere_tests  # the brute-force count, culled or not
    assert np.array_equal(lin.reshape(-1, 3), mlin), f"{np.count_nonzero(lin.reshape(-1, 3) != mlin)} sums differ"
    assert np.array_equal(rgb.reshape(-1, 3), mrgb)
