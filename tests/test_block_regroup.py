"""The culled sweep on regrouped blocks: the order it visits the spheres in, and its image against the f32 mirror.

At upload the culled constant-bank kernel gets its own copy of the sweep rows with the spheres regrouped into
compact 32-sphere blocks (sphere 0 kept in slot 0, median splits of the centres for the rest).  The reference
keeps, among equal roots, the sphere listed first; the regrouped sweep must pick the same one, so its ties go by
original index.  The scenes below list their small spheres in shuffled order, so the regrouping is far from the
identity, and add pairs of spheres that every camera ray of a zero-width view hits at bit-equal t while the
regrouping puts the higher-indexed sphere of the pair in an earlier block.
"""
import ctypes as C

import numpy as np
import pytest

import rtzlib as R
from test_block_cull import CAMERAS, _mirror


def _sweep_order(pkg, sp, n):
    out = (C.c_int32 * max(n, 1))()
    assert pkg.lib().rtz_probe_sweep_order(C.cast(sp, C.POINTER(pkg.rtz_sphere)), n, out) == 0
    return np.array(out[:n], dtype=np.int64)


def _reference_order(centres):
    """The regrouping written out independently: sphere 0 in slot 0, then median splits along the longest axis of
    the centres (f32), ties by index, each cut on a multiple of 32 slots, every final block sorted by index."""
    c = np.asarray(centres, dtype=np.float32)

    def split(idx, slot0):
        blocks = (slot0 + len(idx) + 31) // 32 - slot0 // 32
        if blocks <= 1:
            return sorted(idx)
        span = c[idx].max(axis=0) - c[idx].min(axis=0)
        axis = int(np.argmax(span))  # first axis on equal spans, as the product's strict '>'
        cut = (slot0 // 32 + blocks // 2) * 32
        ordered = sorted(idx, key=lambda i: (float(c[i, axis]), i))
        return split(ordered[:cut - slot0], slot0) + split(ordered[cut - slot0:], cut)

    return [0] + split(list(range(1, len(c))), 1) if len(c) else []


def _scene(ground_first=True, seed=11):
    """Ground + a 20 x 20 grid of small spheres in shuffled order, then tie pairs: at four places (x0, 1, z0) a red
    sphere centred 1.5 to the right of x0 and, later in the list, a blue metal one 1.5 to the left.  A ray
    straight down -z through x = x0, y = 1 meets both at the same t, bit for bit (its x component is exactly 0),
    and no other pair."""
    rng = np.random.default_rng(seed)
    small = []
    for a in range(-10, 10):
        for b in range(-10, 10):
            c = (a + 0.1 + 0.8 * rng.random(), 0.2, b + 0.1 + 0.8 * rng.random())
            kind = rng.random()
            if kind < 0.6:
                small.append(R.make_sphere(c, 0.2, R.MAT_LAMBERTIAN, tuple(0.2 + 0.6 * rng.random(3))))
            elif kind < 0.85:
                small.append(R.make_sphere(c, 0.2, R.MAT_METAL, tuple(0.5 + 0.5 * rng.random(3)), fuzz=0.3))
            else:
                small.append(R.make_sphere(c, 0.2, R.MAT_DIELECTRIC, ior=1.5))
    small = [small[i] for i in rng.permutation(len(small))]
    ground = R.make_sphere((0, -1000, 0), 1000, R.MAT_LAMBERTIAN, (0.5, 0.5, 0.5))
    sp = [ground] + small if ground_first else small[:150] + [ground] + small[150:]
    pairs = []
    for x0, z0 in ((-7.5, -6.0), (-2.5, 5.0), (2.5, -2.0), (7.5, 3.0)):
        pairs.append((len(sp), len(sp) + 1, x0, z0))
        sp.append(R.make_sphere((x0 + 1.5, 1.0, z0), 1.7, R.MAT_LAMBERTIAN, (0.9, 0.1, 0.1)))
        sp.append(R.make_sphere((x0 - 1.5, 1.0, z0), 1.7, R.MAT_METAL, (0.1, 0.2, 0.9), fuzz=0.0))
    return sp, pairs


def _reversed_pair(pkg, sp, pairs):
    """A tie pair (first, second) whose second sphere the regrouping sweeps in an earlier block than the first."""
    order = _sweep_order(pkg, R.sphere_array(sp), len(sp))
    slot = np.empty_like(order)
    slot[order] = np.arange(len(order))
    rev = [p for p in pairs if slot[p[1]] // 32 < slot[p[0]] // 32]
    assert rev, "no tie pair is reversed by the regrouping: the tie test would test nothing"
    return rev[0]


def test_sweep_order_is_the_blocked_median_split(pkg):
    for ground_first in (True, False):
        sp, _ = _scene(ground_first)
        arr, n = R.sphere_array(sp), len(sp)
        order = _sweep_order(pkg, arr, n)
        assert sorted(order) == list(range(n)) and order[0] == 0      # a bijection; sphere 0 stays in slot 0
        assert np.array_equal(order, _sweep_order(pkg, arr, n))        # deterministic
        assert list(order) == _reference_order([s.center[:] for s in sp])
    # the book's scene: the regrouped blocks are compact, the reference's are strips about 22 units long
    _, arr, n = R.final_scene(0xDEADBEEF)
    order = _sweep_order(pkg, arr, n)
    c = np.array([arr[i].center[:] for i in range(n)])

    def mean_block_length(o):
        return np.mean([np.ptp(c[o[b:b + 32]], axis=0).max() for b in range(32, n - 31, 32)])

    assert mean_block_length(np.arange(n)) > 20 and mean_block_length(order) < 0.5 * mean_block_length(np.arange(n))
    assert pkg.lib().rtz_probe_sweep_order(None, 0, None) == 0


def test_tie_pairs_are_reversed_by_the_regrouping(pkg):
    for ground_first in (True, False):
        sp, pairs = _scene(ground_first)
        _reversed_pair(pkg, sp, pairs)


def _check(pkg, orc, sp, cam, seed):
    arr, n = R.sphere_array(sp), len(sp)
    assert 257 <= n <= 512
    rgb, st, lin = pkg.render_host(cam, arr, n, want_linear=True)
    mrgb, mlin, mst = _mirror(orc, cam, arr, n, seed)
    assert (st.samples, st.segments, st.depth_capped, st.absorbed, st.nan_samples) == (
        mst.samples, mst.segments, mst.depth_capped, mst.absorbed, mst.nan_samples)
    assert st.sphere_tests == st.segments * n == mst.sphere_tests
    assert np.array_equal(lin.reshape(-1, 3), mlin), f"{np.count_nonzero(lin.reshape(-1, 3) != mlin)} sums differ"
    assert np.array_equal(rgb.reshape(-1, 3), mrgb)


@pytest.mark.gpu
@pytest.mark.parametrize("ground_first", [True, False], ids=["ground_first", "ground_later"])
@pytest.mark.parametrize("view", list(CAMERAS))
def test_regrouped_sweep_matches_mirror_bit_exact(pkg, gpu, orc, ground_first, view):
    sp, _ = _scene(ground_first)
    cam = R.build_camera(160, 16.0 / 9.0, spp=24, seed=0xC0FFEE, **CAMERAS[view])
    _check(pkg, orc, sp, cam, 0xC0FFEE)


@pytest.mark.gpu
@pytest.mark.parametrize("ground_first", [True, False], ids=["ground_first", "ground_later"])
def test_cross_block_ties_keep_the_first_listed_sphere(pkg, gpu, orc, ground_first):
    """A zero-width view straight down -z onto a reversed tie pair: every camera ray hits both spheres at the
    same t, and the red one (listed first) must win, in the trace kernel and in the drain.  The frame is small and
    deep (8 x 8 pixels, 512 samples), so the trace kernel's queue runs dry with paths in flight and the drain
    kernel finishes them."""
    sp, pairs = _scene(ground_first)
    first, second, x0, z0 = _reversed_pair(pkg, sp, pairs)
    cam = R.build_camera(8, 1.0, (x0, 1.0, z0 + 30.0), (x0, 1.0, z0), 0.0, spp=512, seed=0xBEEF)
    assert tuple(cam.du) == (0.0, 0.0, 0.0) and tuple(cam.dv) == (0.0, 0.0, 0.0)
    # the tie is real: alone, each sphere of the pair is hit at the same t by the camera ray
    ts = []
    for i in (first, second):
        h = pkg.binding.rtz_hit()
        one = C.cast(R.sphere_array([sp[i]]), C.POINTER(pkg.rtz_sphere))
        assert pkg.lib().rtz_probe_hit(one, 1, R.d3((x0, 1.0, z0 + 30.0)), R.d3((0, 0, -1)), 0.001, float("inf"),
                                       C.byref(h)) == 0
        assert h.hit
        ts.append(h.t)
    assert ts[0] == ts[1]
    _check(pkg, orc, sp, cam, 0xBEEF)
