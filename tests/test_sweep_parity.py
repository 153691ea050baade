"""Ray by ray: every production sweep against the f32 mirror, on chosen rays.

test_ray_parity.py ties the mirror to the f64 reference ray by ray, and the device's scalar probe sweep to the
mirror.  The render kernels find their closest hits with other code: the packed two-path sweep over the constant
bank, shared memory or global memory; its culled form (padded block boxes, regrouped rows, the sphere-parallel
pass); the wavefront kernels' sweeps that drop the sphere a ray leaves (two paths per lane, and the four-path kernel's
own sweep over 128 paths per warp); the drain's warp-cooperative sweep; the BVH
traversal.  rtz_probe_sweeps runs each of them, with the render kernel's template arguments, on rays the tests
choose, and every result must equal the mirror's bit for bit.

The rays are those a render rarely or never produces: axis-parallel directions (exact +-0 and subnormal components,
whose reciprocals are infinite) on the planes of the block boxes, one ulp either side, on their edges and corners and
on the tangent and centre planes of spheres; origins at R (1 +- 2^-k) around the padding's radius and far beyond it;
warps in which exactly k of the 64 paths reach a block, at sphere-parallel thresholds 0, 16 and 64; exact ties across
regrouped blocks; rays leaving a sphere, outwards, inwards and along its tangent plane; a finite t_max.  The CPU tests
check that each new family stays within the f64 error model on the mirror, so that "device == mirror" also means
"within the error model", and that rtz_probe_cull_bounds gives the documented block boxes.
"""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import rtzlib as R
from test_block_regroup import _scene as _tie_scene
from test_ray_parity import (HIT, RAY, TMIN, TRANSLATIONS, _camera_rays, _check, _families, _mirror_hits,
                             _moved_camera, _ptr, _rays, _secondary, _sweep_scene, _translated, _unit)

CONST, CULL, SKIP_SELF, SMEM, GLOBAL, COOP, COOP_REGROUPED, BVH, WAVE4 = range(9)
NAMES = ["CONST", "CULL", "SKIP_SELF", "SMEM", "GLOBAL", "COOP", "COOP_REGROUPED", "BVH", "WAVE4"]
CULL_SIZES = [65, 200, 257, 485, 511, 512]  # 485 is the book's final scene; the rest sweep scenes
F32 = np.float32


# ------------------------------------------------------------------------------------------------ scenes
def _scene(orc, n, T=(0.0, 0.0, 0.0)):
    if n == 485:
        _, sp, n = R.final_scene(0xDEADBEEF)
        return _translated(sp, n, np.array(T))
    return _sweep_scene(orc, n, T)


def _order(pkg, sp, n):
    out = (C.c_int32 * n)()
    assert pkg.lib().rtz_probe_sweep_order(C.cast(sp, C.POINTER(pkg.rtz_sphere)), n, out) == 0
    return np.array(out[:], dtype=np.int64)


def _bounds(pkg, sp, n):
    """rtz_probe_cull_bounds: (boxes [blocks, 6] = lo.x hi.x lo.y hi.y lo.z hi.z, cull_r2, host culls)."""
    nb = ((n + 7) // 8 * 8 + 31) // 32
    boxes = np.zeros((max(nb, 1), 6), np.float32)
    r2, culls = C.c_float(), C.c_int32()
    rc = pkg.lib().rtz_probe_cull_bounds(C.cast(sp, C.POINTER(pkg.rtz_sphere)), n,
                                         boxes.ctypes.data_as(C.POINTER(C.c_float)), C.byref(r2), C.byref(culls))
    assert rc == 0, rc
    return boxes[:nb], np.float32(r2.value), culls.value


def _rows(sp, n):
    """The f32 centres and radii the device holds, and the radius sqrt(r^2) the bounds are built from."""
    c = np.array([sp[i].center[:] for i in range(n)], float).astype(F32)
    r = np.array([sp[i].radius for i in range(n)], float).astype(F32)
    return c, r, np.sqrt((r * r).astype(float))


def _restated_bounds(pkg, sp, n):
    """DESIGN.md §5's rule, written out: on the regrouped order, R = 2 max(|c| + r) outside block 0, and for every
    sphere of block b >= 1 the pad 1e-4 (1 + r + |c|_1) + 1e-6 (1.001 R + |c|)^2 / r around c +- r, the block's hull
    rounded outwards to f32 with nextafter; the host culls when the block volumes average under a quarter of their
    joint hull's (and the scene fits the constant bank)."""
    order = _order(pkg, sp, n)
    c32, _, r = _rows(sp, n)
    c = c32.astype(float)
    n_pad = (n + 7) // 8 * 8
    nb = (n_pad + 31) // 32
    rest = order[32:]
    norm = lambda v: np.sqrt(v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2])
    R_ = 2.0 * max((norm(c[rest]) + r[rest]).max(), 0.0) if len(rest) else 0.0
    boxes = np.zeros((nb, 6), np.float32)
    lo_all, hi_all, vols, pads = np.full(3, np.inf), np.full(3, -np.inf), [], {}
    for b in range(1, nb):
        idx = order[32 * b:min(n, 32 * b + 32)]
        cb, rb = c[idx], r[idx]
        X = 1.001 * R_ + norm(cb)
        with np.errstate(divide="ignore"):
            pad = 1e-4 * (1.0 + rb + np.abs(cb[:, 0]) + np.abs(cb[:, 1]) + np.abs(cb[:, 2])) + 1e-6 * X * X / rb
        lo = (cb - rb[:, None] - pad[:, None]).min(0)
        hi = (cb + rb[:, None] + pad[:, None]).max(0)
        fl = np.nextafter(lo.astype(F32), F32(-np.inf))
        fh = np.nextafter(hi.astype(F32), F32(np.inf))
        boxes[b] = [fl[0], fh[0], fl[1], fh[1], fl[2], fh[2]]
        lo_all, hi_all = np.minimum(lo_all, lo), np.maximum(hi_all, hi)
        vols.append((hi[0] - lo[0]) * (hi[1] - lo[1]) * (hi[2] - lo[2]))
        pads[b] = (idx, pad)
    vol_all = (hi_all[0] - lo_all[0]) * (hi_all[1] - lo_all[1]) * (hi_all[2] - lo_all[2])
    culls = int(n_pad <= 512 and len(vols) > 0 and np.isfinite(R_) and sum(vols) < 0.25 * len(vols) * vol_all)
    return boxes, F32(R_ * R_), culls, pads


# ------------------------------------------------------------------------------------------------ box_reach in numpy
def _box_reach(box, o, d, closest):
    """box_reach (rtz_kernels.cuh) in f32 for rays o, d (unit, f32): the slab test over [0, closest] with fminf /
    fmaxf dropping NaN, and NaN reciprocals for origins beyond cull_r2 left to the caller."""
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = (F32(1) / d.astype(F32)).astype(F32)
        t = [((F32(box[2 * a + s]) + (-o[:, a]).astype(F32)).astype(F32) * inv[:, a]).astype(F32)
             for a in range(3) for s in (0, 1)]
    tn = np.fmax(np.fmax(np.fmin(t[0], t[1]), np.fmin(t[2], t[3])), np.fmax(np.fmin(t[4], t[5]), F32(0)))
    tf = np.fmin(np.fmin(np.fmax(t[0], t[1]), np.fmax(t[2], t[3])), np.fmin(np.fmax(t[4], t[5]), F32(closest)))
    return tn <= tf


def _unit32(d):
    """set_direction's unit vector, for the numpy box test (one rounding of each step, as the device does)."""
    d = d.astype(F32)
    ln = np.sqrt(np.float32(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]))
    return (d * (F32(1) / ln)[:, None]).astype(F32)


# ------------------------------------------------------------------------------------------------ new ray families
def _pick(rng, sp, order, b, n):
    """Caller's index and f64 centre / radius of a random sphere of regrouped block b."""
    slots = np.arange(32 * b, min(n, 32 * b + 32))
    i = int(order[rng.choice(slots)])
    return i, np.array(sp[i].center[:]), float(sp[i].radius)


def _axis_family(pkg, orc, sp, n, rng, blocks):
    """Axis-parallel rays on box planes (exact, +-1 ulp), on box edges and corners, and on the tangent and centre
    planes of spheres, aimed along the plane at spheres of the block and of its neighbours.  Direction components
    that are not aimed are +0, -0, 1e-38 or the smallest subnormal."""
    boxes, _, _ = _bounds(pkg, sp, n)
    order = _order(pkg, sp, n)
    nb = len(boxes)
    tiny = [0.0, -0.0, 1e-38, -1e-38, float(np.float32(1.4e-45)), -float(np.float32(1.4e-45))]
    o, d = [], []
    for b in blocks:
        box = boxes[b]
        for tb in {max(b - 1, 1), b, min(b + 1, nb - 1)}:
            for _ in range(3):
                _, c, r = _pick(rng, sp, order, tb, n)
                for a in range(3):
                    j, k = [x for x in range(3) if x != a]
                    planes = [box[2 * a], box[2 * a + 1]]
                    planes += [np.nextafter(F32(p), F32(s * np.inf)) for p in planes for s in (-1, 1)]
                    planes += [F32(c[a] - r), F32(c[a] + r), F32(c[a])]
                    for p in planes:
                        # one zero component: in the plane, aimed at the centre from 3r to 6r away
                        u = _unit(rng, 1)[0]
                        u[a] = 0.0
                        u /= np.linalg.norm(u)
                        oo = c - (3 + 3 * rng.random()) * max(r, 1e-3) * u
                        oo[a] = p
                        dd = c - oo
                        dd[a] = tiny[rng.integers(len(tiny))]
                        o.append(oo), d.append(dd)
                        # two zero components: along axis j, on the plane and on an edge with a plane of axis k
                        for ok in (c[k], box[2 * k], box[2 * k + 1]):
                            oo = c.copy()
                            oo[a], oo[k] = p, ok
                            oo[j] = c[j] - rng.choice([-1, 1]) * (2 + rng.random()) * max(r, 1e-3)
                            dd = np.zeros(3)
                            dd[j] = np.sign(c[j] - oo[j])
                            dd[a], dd[k] = tiny[rng.integers(len(tiny))], tiny[rng.integers(len(tiny))]
                            o.append(oo), d.append(dd)
            # corners of the box: axis-parallel and aimed at a sphere of the block
            for corner in range(8):
                oo = np.array([box[2 * a + ((corner >> a) & 1)] for a in range(3)], float)
                _, c, _ = _pick(rng, sp, order, tb, n)
                o.append(oo), d.append(c - oo)
                for a in range(3):
                    dd = np.array([tiny[rng.integers(len(tiny))] for _ in range(3)])
                    dd[a] = 1.0 if c[a] > oo[a] else -1.0
                    o.append(oo), d.append(dd)
    return _rays(np.array(o), np.array(d))


def _radius_family(pkg, orc, sp, n, rng):
    """Origins at |o| = R (1 +- 2^-k), k = 1 .. 22, at 10 R and 10^4 R, each aimed at a random sphere of a culled
    block; and rays leaving the ground sphere (slot 0, block 0) beyond R towards culled blocks."""
    _, r2, _ = _bounds(pkg, sp, n)
    order = _order(pkg, sp, n)
    nb = ((n + 7) // 8 * 8 + 31) // 32
    Rr = float(np.sqrt(np.float64(r2)))
    scales = [1 + s * 2.0 ** -k for k in range(1, 23) for s in (-1, 1)] + [10.0, 1e4]
    o, d = [], []
    for s in scales:
        for u in _unit(rng, 6):
            _, c, _ = _pick(rng, sp, order, int(rng.integers(1, nb)), n)
            oo = np.float32(u * Rr * s).astype(float)
            o.append(oo), d.append(c - oo)
    rays = _rays(np.array(o), np.array(d))
    # ground points beyond R (where the ground reaches beyond it): straight down onto sphere 0, then towards culled
    # spheres
    g0, r0 = np.array(sp[0].center[:]), float(sp[0].radius)
    top = []
    for _ in range(48):
        v = _unit(rng, 1)[0]
        v[1] = 0.0
        top.append(g0 + v / np.linalg.norm(v) * r0 * rng.uniform(0.05, 0.95) + np.array([0.0, r0 + 5.0, 0.0]))
    down = _mirror_hits(orc, sp, n, _rays(np.array(top), np.tile([0.0, -1.0, 0.0], (len(top), 1))))
    p = down["point"][down["best"] == 0].astype(float)
    p = p[(p * p).sum(1) > Rr * Rr]
    if not len(p):
        return rays
    tgt = np.array([_pick(rng, sp, order, int(rng.integers(1, nb)), n)[1] for _ in range(len(p))])
    ground = _rays(p, tgt - p, np.zeros(len(p), int))
    return np.concatenate([rays, ground])


def _reaching(box, c, r, rng):
    """An origin inside `box` near a sphere (centre c, radius r) of its block: every box test reaches the block."""
    for _ in range(100):
        oo = c + (1.2 + rng.random()) * r * _unit(rng, 1)[0]
        if all(box[2 * a] < oo[a] < box[2 * a + 1] for a in range(3)):
            return oo
    return c + 0.0


def _warp(pkg, orc, sp, n, rng, b, k):
    """64 rays, of which exactly k reach block b's box (origins inside it, aimed at its spheres) and 64 - k cannot
    (origins outside it and within R, pointing away), in a random arrangement of lanes and slots.  Confirmed with
    the numpy box test."""
    boxes, r2, _ = _bounds(pkg, sp, n)
    order = _order(pkg, sp, n)
    box = boxes[b]
    mid = np.array([(box[2 * a] + box[2 * a + 1]) / 2 for a in range(3)], float)
    half = np.array([(box[2 * a + 1] - box[2 * a]) / 2 for a in range(3)], float)
    o, d = [], []
    for _ in range(k):
        _, c, r = _pick(rng, sp, order, b, n)
        oo = _reaching(box, c, r, rng)
        o.append(oo), d.append(c - oo + 0.3 * r * _unit(rng, 1)[0])
    while len(o) < 64:
        u = _unit(rng, 1)[0]
        oo = mid + u * (np.linalg.norm(half) * 1.05 + 0.01)
        o.append(oo), d.append(u + 0.2 * _unit(rng, 1)[0])
    o, d = np.array(o), np.array(d)
    rays = _rays(o, d)
    oo32, du32 = rays["orig"], _unit32(rays["dir"])
    inside = np.array([all(box[2 * a] < oo32[q, a] < box[2 * a + 1] for a in range(3)) for q in range(64)])
    within = (oo32.astype(float) ** 2).sum(1) * (1 - 2.0 ** -18) < float(r2) * 0.999
    reach = _box_reach(box, oo32, du32, np.inf)
    assert inside[:k].all() and reach[:k].all() and within.all(), (b, k)
    assert not reach[k:].any(), (b, k, int(reach[k:].sum()))
    return rays[rng.permutation(64)]


def _self_family(orc, sp, n, cam_rays, rng):
    """Rays leaving real surface points with self set: outwards, inwards (_secondary), and along the tangent plane
    with h exactly 0 (origin c + r e_x in f32, direction with a zero x component)."""
    sec = _secondary(orc, sp, n, cam_rays, rng)
    idx = rng.choice(n, size=min(n, 64), replace=False)
    o, d = [], []
    for i in idx:
        c, r = np.array(sp[i].center[:]), float(np.float32(sp[i].radius))
        for s in (-1.0, 1.0):
            oo = np.float32(c).astype(float)
            oo[0] = float(np.float32(np.float32(c[0]) + np.float32(s * r)))
            dd = np.array([0.0, *_unit(rng, 1)[0][:2]])
            o.append(oo), d.append(dd)
    tang = _rays(np.array(o), np.array(d), np.repeat(idx, 2))
    return np.concatenate([sec, tang])


def _tie_rays(rng, pairs):
    """Rays straight down -z through x = x0 (exact) of test_block_regroup's tie pairs, at many heights and depths:
    both spheres of a pair are hit at bit-equal t."""
    o = []
    for _, _, x0, z0 in pairs:
        for _ in range(32):
            o.append((x0, 1.0 + rng.uniform(-0.75, 0.75), z0 + rng.uniform(5, 40)))
    o = np.array(o)
    return _rays(o, np.tile([0.0, 0.0, -1.0], (len(o), 1)))


def _dup_scene(orc):
    """The first 256 spheres of the final scene listed twice: every hit is an exact tie, the copy of the ground
    (sphere 256) lands in another regrouped block than sphere 0, and the lower index must win."""
    _, sp, _ = R.final_scene(0xDEADBEEF)
    both = (R.Sphere * 512)()
    for i in range(256):
        both[i] = both[256 + i] = sp[i]
    return both, 512


def _c3_rays(orc, T, rng, pixels=120, per=4):
    cam = _moved_camera(300, np.array(T), look_from=(13, 2, 3), look_at=(0, 0, 0), vfov=20, defocus=0.6)
    return _camera_rays(orc, cam, 5, pixels, per, rng)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("T", [(0.0, 0.0, 0.0), (1e3, 1e3, 1e3)], ids=lambda T: "T=%g,%g,%g" % T)
def test_new_families_stay_in_the_error_model(pkg, orc, T):
    """The mirror on every new family: no unexplained disagreement with the f64 reference, explained ones within
    each family's bound, and the candidate gate only filters."""
    rng = np.random.default_rng(41)
    sp, n = _scene(orc, 485, T), 485
    _check(orc, sp, n, _axis_family(pkg, orc, sp, n, rng, [1, 7, 15]), max_explained=0.5, label="axis")
    # at 10 R and 10^4 R from a scene moved by 10^3 the error model's bounds are wide, and many rays ambiguous
    _check(orc, sp, n, _radius_family(pkg, orc, sp, n, rng), max_explained=0.5, label="radius")
    for b, k in ((1, 17), (8, 63), (15, 1)):
        _check(orc, sp, n, _warp(pkg, orc, sp, n, rng, b, k), max_explained=0.05, label=f"warp b={b} k={k}")
    cam = _c3_rays(orc, T, rng)
    _check(orc, sp, n, _self_family(orc, sp, n, cam, rng), tmax=50.0, max_explained=0.2, label="self")
    dup, nd = _dup_scene(orc)
    dup = _translated(dup, nd, np.array(T))
    _check(orc, dup, nd, _c3_rays(orc, T, rng), tmax=60.0, max_explained=0.01, label="duplicates")
    spt, pairs = _tie_scene(True)
    arr = _translated(R.sphere_array(spt), len(spt), np.zeros(3))
    got = _check(orc, arr, len(spt), _tie_rays(rng, pairs), max_explained=0.01, label="ties")
    assert (got["best"] >= 0).all()


def _radius_zero_scene(orc, r):
    sp = _sweep_scene(orc, 65, (0.0, 0.0, 0.0))
    sp[40].radius = r
    return sp


@pytest.mark.parametrize("case", CULL_SIZES + [4096, "T=1e4", "duplicates", "r^2=0", "r=0"])
def test_cull_bounds_equal_the_documented_rule(pkg, orc, case):
    """rtz_probe_cull_bounds against the numpy restatement, bit for bit; every sphere of block b inside its box with
    at least its padding to spare.  A sphere of radius 0 is refused as the upload refuses it; one of radius 1e-30,
    whose f32 square is 0, gets an infinite pad and so an infinite box (the block is always swept)."""
    if case == "r=0":
        sp, n = _radius_zero_scene(orc, 0.0), 65
        out = np.zeros(6 * 3, np.float32)
        r2, culls = C.c_float(), C.c_int32()
        assert pkg.lib().rtz_probe_cull_bounds(C.cast(sp, C.POINTER(pkg.rtz_sphere)), n,
                                               out.ctypes.data_as(C.POINTER(C.c_float)), C.byref(r2), C.byref(culls)) == 1
        return
    if case == "r^2=0":
        sp, n = _radius_zero_scene(orc, 1e-30), 65
    elif case == "T=1e4":
        sp, n = _scene(orc, 485, (1e4, -1e4, 1e4)), 485
    elif case == "duplicates":
        sp, n = _dup_scene(orc)
    else:
        sp, n = _scene(orc, case), case
    boxes, r2, culls = _bounds(pkg, sp, n)
    want, wr2, wculls, pads = _restated_bounds(pkg, sp, n)
    assert boxes.tobytes() == want.tobytes()
    assert r2 == wr2 and culls == wculls
    if case in (485, "duplicates"):
        assert culls == 1
    if case == "r^2=0":
        assert np.isinf(boxes).sum() >= 6
    c, r, _ = _rows(sp, n)
    for b, (idx, pad) in pads.items():
        box = boxes[b].astype(float)
        for a in range(3):
            assert (box[2 * a] <= c[idx, a] - r[idx].astype(float) - pad).all(), (b, a)
            assert (c[idx, a] + r[idx].astype(float) + pad <= box[2 * a + 1]).all(), (b, a)


def test_cull_bounds_refusals(pkg):
    l = pkg.lib()
    sp, n = R.chapter13_scene()
    P = C.cast(sp, C.POINTER(pkg.rtz_sphere))
    box = np.zeros(6, np.float32).ctypes.data_as(C.POINTER(C.c_float))
    r2, culls = C.c_float(), C.c_int32()
    assert l.rtz_probe_cull_bounds(None, n, box, C.byref(r2), C.byref(culls)) == 1
    assert l.rtz_probe_cull_bounds(P, n, None, C.byref(r2), C.byref(culls)) == 1
    assert l.rtz_probe_cull_bounds(P, n, box, None, C.byref(culls)) == 1
    assert l.rtz_probe_cull_bounds(P, n, box, C.byref(r2), None) == 1
    assert l.rtz_probe_cull_bounds(P, (1 << 20) + 1, box, C.byref(r2), C.byref(culls)) == 1
    bad = R.sphere_array([R.make_sphere((0, 0, 0), 1.0, R.MAT_LAMBERTIAN, (1.5, 0.5, 0.5))])
    assert l.rtz_probe_cull_bounds(C.cast(bad, C.POINTER(pkg.rtz_sphere)), 1, box, C.byref(r2), C.byref(culls)) == 1
    assert l.rtz_probe_cull_bounds(None, 0, None, C.byref(r2), C.byref(culls)) == 0 and culls.value == 0
    assert l.rtz_probe_cull_bounds(P, n, box, C.byref(r2), C.byref(culls)) == 0 and culls.value == 0


# ------------------------------------------------------------------------------------------------ GPU
def _probe(pkg, sp, n, rays, kind, tmin=TMIN, tmax=np.inf, split=16):
    out = np.zeros(len(rays), HIT)
    l = pkg.lib()
    rc = l.rtz_probe_sweeps(C.cast(sp, C.POINTER(pkg.rtz_sphere)), n, _ptr(rays), len(rays), tmin, tmax, kind, split,
                            _ptr(out))
    assert rc == 0, (NAMES[kind], rc, l.rtz_last_error())
    return out


def _pad128(rays):
    """Whole warps for every kind: 64 rays for the two-path sweeps, 128 for WAVE4."""
    k = (-len(rays)) % 128
    return np.concatenate([rays, np.resize(rays, k)]) if k else rays


def _kinds(n):
    k = [GLOBAL, COOP, COOP_REGROUPED, BVH]
    if n <= 512:
        k = [CONST, CULL, SKIP_SELF, WAVE4] + k
    if n <= 6000:
        k.append(SMEM)
    return k


def _same(pkg, orc, sp, n, rays, label, kinds=None, tmin=TMIN, tmax=np.inf, splits=(16,)):
    """Every kind equals the mirror bit for bit; returns the list of disagreements."""
    rays = _pad128(rays)
    want = _mirror_hits(orc, sp, n, rays, tmin, tmax)
    bad = []
    for kind in kinds if kinds is not None else _kinds(n):
        for split in splits if kind == CULL else (16,):
            got = _probe(pkg, sp, n, rays, kind, tmin, tmax, split)
            if got.tobytes() != want.tobytes():
                diff = np.flatnonzero(got != want)
                bad.append(f"{label} {NAMES[kind]} split={split}: {len(diff)} of {len(rays)} rays, first {diff[0]}: "
                           f"{rays[diff[0]]} got {got[diff[0]]} want {want[diff[0]]}")
    return bad


def _with_sphere(sp_scene, n_scene, one, at=100):
    """The scene with sphere `one` inserted at index `at`."""
    out = (R.Sphere * (n_scene + 1))()
    for i in range(at):
        out[i] = sp_scene[i]
    out[at] = one
    for i in range(at, n_scene):
        out[i + 1] = sp_scene[i]
    return out, n_scene + 1


@pytest.mark.gpu
@pytest.mark.parametrize("T", [TRANSLATIONS[0], TRANSLATIONS[5], TRANSLATIONS[11], TRANSLATIONS[8]],
                         ids=lambda T: "T=%g,%g,%g" % T)
def test_ray_parity_families_in_every_sweep(pkg, gpu, orc, T):
    rng = np.random.default_rng(23)
    bad = []
    final, nf = _scene(orc, 485, T), 485
    for label, sp, n, rays, tmin, tmax, _ in _families(orc, np.array(T), rng):
        bad += _same(pkg, orc, sp, n, rays, label, tmin=tmin, tmax=tmax)
        if n == 1:  # into a culled block of the final scene
            both, nb = _with_sphere(final, nf, sp[0])
            slot = int(np.flatnonzero(_order(pkg, both, nb) == 100)[0])
            assert slot >= 32, (label, slot)
            bad += _same(pkg, orc, both, nb, rays, label + " in the final scene", [CULL, COOP_REGROUPED, CONST],
                         tmin, tmax, splits=(0, 16, 64))
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("n", CULL_SIZES)
def test_axis_parallel_rays_on_box_planes(pkg, gpu, orc, n):
    rng = np.random.default_rng(n)
    bad = []
    for T in [(0.0, 0.0, 0.0), (1e3, 1e3, 1e3)]:
        sp = _scene(orc, n, T)
        nb = ((n + 7) // 8 * 8 + 31) // 32
        rays = _axis_family(pkg, orc, sp, n, rng, sorted({1, nb // 2, nb - 1}))
        bad += _same(pkg, orc, sp, n, rays, f"axis T={T}", splits=(0, 16, 64))
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [200, 485, 512])
def test_origins_around_the_padding_radius(pkg, gpu, orc, n):
    rng = np.random.default_rng(7 * n)
    bad = []
    for T in [(0.0, 0.0, 0.0), (1e3, 0.0, 0.0)]:
        sp = _scene(orc, n, T)
        rays = _radius_family(pkg, orc, sp, n, rng)
        bad += _same(pkg, orc, sp, n, rays, f"radius T={T}", splits=(0, 16, 64))
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("n", CULL_SIZES)
def test_warp_compositions_at_every_split(pkg, gpu, orc, n):
    """For several blocks, warps in which exactly k of the 64 paths reach the block, k around the sphere-parallel
    thresholds, swept at split_max 0, 16 and 64 (the last block of most of these scenes is partial)."""
    rng = np.random.default_rng(11 * n)
    sp = _scene(orc, n, (0.0, 0.0, 0.0))
    nb = ((n + 7) // 8 * 8 + 31) // 32
    warps = [_warp(pkg, orc, sp, n, rng, b, k) for b in sorted({1, nb // 2, nb - 1})
             for k in (0, 1, 15, 16, 17, 32, 63, 64)]
    bad = _same(pkg, orc, sp, n, np.concatenate(warps), "warps", [CULL, CONST, COOP_REGROUPED], splits=(0, 16, 64))
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_ties_and_self_with_a_finite_t_max(pkg, gpu, orc):
    rng = np.random.default_rng(5)
    bad = []
    for T in [(0.0, 0.0, 0.0), (1e3, 1e3, 1e3)]:
        sp, n = _scene(orc, 485, T), 485
        cam = _c3_rays(orc, T, rng)
        bad += _same(pkg, orc, sp, n, _self_family(orc, sp, n, cam, rng), f"self T={T}", tmax=50.0,
                     splits=(0, 16, 64))
        dup, nd = _dup_scene(orc)
        dup = _translated(dup, nd, np.array(T))
        bad += _same(pkg, orc, dup, nd, np.concatenate([_c3_rays(orc, T, rng), _self_family(orc, dup, nd, cam, rng)]),
                     f"duplicates T={T}", tmax=60.0, splits=(0, 16, 64))
    for ground_first in (True, False):
        spt, pairs = _tie_scene(ground_first)
        arr = R.sphere_array(spt)
        rays = _tie_rays(rng, pairs)
        bad += _same(pkg, orc, arr, len(spt), rays, f"ties ground_first={ground_first}", tmax=80.0, splits=(0, 16, 64))
    assert not bad, "\n".join(bad)


SIZES = {CONST: [65, 200, 257, 485, 511, 512], SKIP_SELF: [65, 200, 257, 485, 511, 512],
         CULL: [65, 200, 257, 485, 511, 512], SMEM: [513, 4096, 6000], GLOBAL: [8192, 16384],
         COOP: [1, 31, 33, 64, 485], COOP_REGROUPED: [1, 31, 33, 64, 485],
         WAVE4: [33, 64, 65, 128, 200, 256, 257, 512]}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [(k, n) for k, ns in SIZES.items() for n in ns],
                         ids=[f"{NAMES[k]}-{n}" for k, ns in SIZES.items() for n in ns])
def test_scene_sizes_of_each_sweep(pkg, gpu, orc, kind, n):
    rng = np.random.default_rng(n + 1000 * kind)
    if n < 4:
        sp = R.sphere_array([R.make_sphere((0.0, 0.0, -1.0), 0.5, R.MAT_LAMBERTIAN, (0.5, 0.5, 0.5))])
    else:
        sp = _scene(orc, n, (0.0, 0.0, 0.0))
    cam = _c3_rays(orc, (0.0, 0.0, 0.0), rng, pixels=64)
    rays = np.concatenate([cam, _secondary(orc, sp, n, cam, rng)])
    bad = _same(pkg, orc, sp, n, rays, "camera+secondary", [kind], splits=(0, 16, 64))
    bad += _same(pkg, orc, sp, n, rays, "camera+secondary t_max=20", [kind], tmax=20.0)
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5, 485, 4096, 16384])
def test_bvh_on_duplicated_scenes(pkg, gpu, orc, n):
    """Every sphere listed twice: deep trees, and every hit a tie that the lower index must win."""
    rng = np.random.default_rng(n)
    sp = R.chapter13_scene()[0] if n == 5 else _scene(orc, n, (0.0, 0.0, 0.0))
    both = (R.Sphere * (2 * n))()
    for i in range(n):
        both[i] = both[n + i] = sp[i]
    cam = _c3_rays(orc, (0.0, 0.0, 0.0), rng, pixels=64)
    rays = np.concatenate([cam, _secondary(orc, both, 2 * n, cam, rng)])
    bad = _same(pkg, orc, both, 2 * n, rays, "duplicated", [BVH])
    bad += _same(pkg, orc, both, 2 * n, rays, "duplicated t_max=20", [BVH], tmax=20.0)
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_malformed_calls_are_refused(pkg, gpu, orc):
    import torch
    l = pkg.lib()
    P = C.POINTER(pkg.rtz_sphere)
    sp, n = _scene(orc, 485), 485
    rng = np.random.default_rng(3)
    rays = _pad128(_c3_rays(orc, (0.0, 0.0, 0.0), rng, pixels=16))
    out = np.zeros(len(rays), HIT)
    ok = (C.cast(sp, P), n, _ptr(rays), len(rays), TMIN, np.inf, CONST, 16, _ptr(out))

    def call(**kw):
        args = list(ok)
        for k, v in kw.items():
            args[["sp", "n", "rays", "m", "tmin", "tmax", "kind", "split", "out"].index(k)] = v
        return l.rtz_probe_sweeps(*args)

    assert call() == 0
    refused = [dict(sp=None), dict(n=0), dict(rays=None), dict(out=None), dict(m=(1 << 31) + 64), dict(kind=-1),
               dict(kind=9), dict(split=-1), dict(split=65), dict(m=63), dict(m=32, kind=GLOBAL),
               dict(m=64, kind=WAVE4)]
    big = _scene(orc, 513)
    refused += [dict(sp=C.cast(big, P), n=513, kind=k) for k in (CONST, CULL, SKIP_SELF, WAVE4)]
    for r in refused:
        assert call(**r) == 1, r
    selfish = rays.copy()
    for s in (-2, n):
        selfish["self"][5] = s
        for kind in (SKIP_SELF, CULL, COOP_REGROUPED, WAVE4):
            assert call(rays=_ptr(selfish), kind=kind) == 1, (s, kind)
    assert b"self" in l.rtz_last_error()
    bad = R.sphere_array([R.make_sphere((0, 0, 0), 0.0, R.MAT_LAMBERTIAN)])
    assert call(sp=C.cast(bad, P), n=1, kind=COOP) == 1
    # the shared-memory kind is refused where the render would read the rows from global memory
    huge = _scene(orc, 7000)
    assert call(sp=C.cast(huge, P), n=7000, kind=SMEM) == 1 and b"shared memory" in l.rtz_last_error()
    # m = 0 runs nothing; the COOP and BVH kinds take any m
    assert call(m=0) == 0 and call(m=37, kind=COOP) == 0 and call(m=37, kind=BVH) == 0
    # a refused call leaves no context behind: contexts that are never destroyed hold device memory, refused calls
    # (the last one refused after its upload) must not
    torch.cuda.synchronize()

    def drop(fn, times=24):
        free0 = torch.cuda.mem_get_info()[0]
        fn(times)
        return free0 - torch.cuda.mem_get_info()[0]

    leaked = []

    def leak(times):
        for _ in range(times):
            c = C.c_void_p()
            assert l.rtz_context_create(0, None, C.byref(c)) == 0
            assert l.rtz_scene_upload(c, C.cast(huge, P), 7000) == 0
            leaked.append(c)

    def refuse(times):
        for _ in range(times):
            assert call(sp=C.cast(huge, P), n=7000, kind=SMEM) == 1

    held = drop(leak)
    for c in leaked:
        l.rtz_context_destroy(c)
    assert held > 0
    assert min(drop(refuse) for _ in range(3)) < held / 2


def test_four_path_wavefront_kernel_keeps_its_registers_and_the_uniform_sweep(pkg):
    """Codegen guard (no GPU needed): the four-path wavefront kernel, whose sweep RTZ_SWEEP_WAVE4 probes through the
    same inlined function, must not spill, must keep its sphere operands in uniform registers and must not diverge."""
    out = subprocess.run(["cuobjdump", "-sass", str(pkg.binding.LIB_PATH)], capture_output=True, text=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    wave = [k for k in body if "trace_kernel_wave_nILi4ELi128ELi6" in k]
    assert len(wave) == 1, wave
    sass = "\n".join(body[wave[0]])
    assert not re.search(r"\b(STL|LDL)\b", sass), "the four-path wavefront kernel spills to local memory"
    assert len(re.findall(r"FFMA2 [^;]*UR\d+\.F32x2", sass)) >= 48
    assert "BRA.DIV" not in sass
