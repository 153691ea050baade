"""Ray by ray: the device's per-ray arithmetic against an f64 restatement of the reference, and the sphere gate.

The whole-image tests (test_oracle_stat.py) see an arithmetic error only when it is large and common enough to
move an image.  Here single rays of seeded families go through the f32 mirror's sweep / shade (the twins of the
batched device probes rtz_probe_hits / rtz_probe_scatters, which the GPU tests below match bit for bit) and are
compared with the f64 reference on the SAME f32-rounded inputs: spheres and rays are built in f64, translated in
f64, then rounded to f32 once.

Error model of a hit (eps = 2^-24, unit direction, distance units, per ray and sphere i with oc = c_i - o):
  * delta_i = K eps max(|oc|^2, r_i^2) bounds the f32 error of the direct form's discriminant
    disc = h^2 - (|oc|^2 - r^2), h = d.oc (with the margin of the candidate gate, DESIGN.md §4, the gate never
    rejects what the direct form accepts, so the direct form's error is the only one that matters);
  * a root h -/+ sqrt(disc) is then off by at most e_i = min(sqrt(delta_i), delta_i / (2 sqrt|disc|)) + K eps |h|.
A ray whose hit sphere (or hit versus miss) differs from the reference is EXPLAINED only if its f64 ray is
ambiguous: the discriminant of one of the two spheres lies within delta of 0, the two spheres' roots lie within
their errors of each other, or a root lies within its error of t_min |d| or t_max |d|.  Unexplained disagreements
must be zero; where the sphere agrees, |t - t*| <= e_i (plus, on the sphere the ray starts on, the f64 near root:
DESIGN.md §4's exact c = 0 for that sphere moves the far root by it).  K = 32 (the derivation gives about 17 for the direct
form; the rest is slack for the direction's normalisation).

Scatters compare the mirror's shade with a numpy f64 restatement of material.zig fed the same Philox words,
starting from the f64 hit point of the same ray.  Branches (reflect / refract, absorbed, nearZero) must agree
unless the f64 quantity lies within its error of the threshold; directions agree within an angle of about
K eps (1 + |p| / r) plus the root's error over r (the hit point moves along the ray); attenuations are exact.
"""
import ctypes as C

import numpy as np
import pytest

import rtzlib as R

EPS = 2.0 ** -24
K = 32.0
TMIN = 0.001

RAY = np.dtype([("orig", "<f4", 3), ("dir", "<f4", 3), ("self", "<i4")])
HIT = np.dtype([("best", "<i4"), ("front", "<i4"), ("t", "<f4"), ("len", "<f4"), ("point", "<f4", 3),
                ("normal", "<f4", 3)])
BOUNCE = np.dtype([("sphere", "<i4"), ("orig", "<f4", 3), ("dir", "<f4", 3), ("pixel", "<u4"), ("sample", "<u4"),
                   ("bounce", "<u4")])
SCAT = np.dtype([("term", "<i4"), ("orig", "<f4", 3), ("dir", "<f4", 3), ("len", "<f4"), ("attenuation", "<f4", 3)])

AXES = {"x": (1, 0, 0), "y": (0, 1, 0), "z": (0, 0, 1), "xyz": (1, 1, 1)}
TRANSLATIONS = [(0.0, 0.0, 0.0)] + [tuple(s * np.array(a, float)) for s in (1e2, 1e3, 1e4) for a in AXES.values()]
CH13_CAMERAS = {
    "ch11": dict(look_from=(0, 0, 0), look_at=(0, 0, -1), vfov=90),
    "ch12": dict(look_from=(-2, 2, 1), look_at=(0, 0, -1), vfov=20),
    "ch13": dict(look_from=(-2, 2, 1), look_at=(0, 0, -1), vfov=20, defocus=10.0, viewport_focus=3.4, focus=3.4),
}


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ------------------------------------------------------------------------------------------------ scenes and rays
def _translated(sp, n, T):
    """Copy of n spheres moved by T in f64, centres and radii rounded to f32 (the inputs every side then shares)."""
    out = (R.Sphere * n)()
    for i in range(n):
        out[i] = sp[i]
        out[i].center = R.d3(np.float32(np.array(sp[i].center[:]) + T).astype(float))
        out[i].radius = float(np.float32(sp[i].radius))
    return out


def _geometry(sp, n):
    cen = np.array([sp[i].center[:] for i in range(n)], float)
    rad = np.array([max(sp[i].radius, 0.0) for i in range(n)], float)
    return cen, rad


def _rays(o, d, self_=None):
    r = np.zeros(len(o), RAY)
    r["orig"], r["dir"] = np.float32(o), np.float32(d)
    r["self"] = -1 if self_ is None else self_
    return r


def _camera_rays(orc, cam, seed, pixels, per_pixel, rng):
    o = np.zeros((pixels * per_pixel, 3), np.float32)
    d = np.zeros_like(o)
    F = C.POINTER(C.c_float)
    for k in range(pixels):
        i, j = int(rng.integers(cam.width)), int(rng.integers(cam.height))
        sl = slice(k * per_pixel, (k + 1) * per_pixel)
        orc.orc_mirror_camera_ray(C.byref(cam), seed, i, j, k, per_pixel, o[sl].ctypes.data_as(F),
                                  d[sl].ctypes.data_as(F), None)
    return _rays(o, d)


def _moved_camera(width, T, **kw):
    kw = dict(kw)
    kw["look_from"] = tuple(np.array(kw["look_from"], float) + T)
    kw["look_at"] = tuple(np.array(kw["look_at"], float) + T)
    return R.build_camera(width, 16.0 / 9.0, spp=1, **kw)


def _unit(rng, m):
    v = rng.normal(size=(m, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _mirror_hits(orc, sp, n, rays, tmin=TMIN, tmax=np.inf, gate=True):
    out = np.zeros(len(rays), HIT)
    orc.orc_mirror_set_gate(1 if gate else 0)
    try:
        orc.orc_mirror_hits(sp, n, _ptr(rays), len(rays), tmin, tmax, _ptr(out))
    finally:
        orc.orc_mirror_set_gate(1)
    return out


def _secondary(orc, sp, n, cam_rays, rng):
    """Rays that leave real surface points (the mirror's f32 hit points) with `self` set: scattered outwards
    (normal + unit vector) and inwards (against the normal, as a refraction goes)."""
    h = _mirror_hits(orc, sp, n, cam_rays)
    ok = h["best"] >= 0
    p, nrm, best = h["point"][ok], h["normal"][ok].astype(float), h["best"][ok]
    u = _unit(rng, len(p))
    out_dir = nrm + u
    in_dir = -nrm + 0.9 * u
    return _rays(np.concatenate([p, p]), np.concatenate([out_dir, in_dir]), np.concatenate([best, best]))


def _tangent_family(rng, r, T, m_per_k=12):
    """One sphere of radius r; rays passing at r (1 +- 2^-k) from its centre, k = 4..22, from 3r away, with
    direction lengths from 1e-3 to 1e3."""
    sp = R.sphere_array([R.make_sphere((0.3 * r, -0.2 * r, 0.1 * r), r, R.MAT_LAMBERTIAN, (0.5, 0.5, 0.5))])
    sp = _translated(sp, 1, T)
    c = np.array(sp[0].center[:])
    o, d = [], []
    for k in range(4, 23):
        for sgn in (-1.0, 1.0):
            u = _unit(rng, m_per_k)
            v = np.cross(u, _unit(rng, m_per_k))
            v /= np.linalg.norm(v, axis=1, keepdims=True)
            b = float(np.float32(r)) * (1.0 + sgn * 2.0 ** -k)
            o.append(c + b * v - 3.0 * r * u)
            d.append(u * 10.0 ** rng.uniform(-3, 3, size=(m_per_k, 1)))
    return sp, 1, _rays(np.concatenate(o), np.concatenate(d))


def _edge_family(rng, T, tmax, m=600):
    """A unit sphere; origins placed so that the entry root sits within a few ulps of t_min |d| (tmax = inf) or of
    a finite t_max |d|, direction lengths from 1e-3 to 1e3."""
    sp = R.sphere_array([R.make_sphere((0.0, 0.0, 0.0), 1.0, R.MAT_METAL, (0.7, 0.6, 0.5))])
    sp = _translated(sp, 1, T)
    c = np.array(sp[0].center[:])
    u = _unit(rng, m)
    w = np.cross(u, _unit(rng, m))
    w /= np.linalg.norm(w, axis=1, keepdims=True)
    b = rng.uniform(0, 0.9, size=(m, 1))
    entry = c + b * w - np.sqrt(1 - b * b) * u
    L = 10.0 ** rng.uniform(-3, 3, size=(m, 1))
    edge = TMIN if np.isinf(tmax) else tmax
    j = rng.integers(-8, 9, size=(m, 1))
    o = entry - u * (edge * L * (1.0 + j * 2.0 ** -23))
    return sp, 1, _rays(o, u * L)


# ------------------------------------------------------------------------------------------------ the f64 reference
def _reference(orc, sp, n, rays, tmin, tmax):
    """orc_list_hit (HittableList.hit in f64) per ray: (best, t in distance units)."""
    m = len(rays)
    best, t = np.full(m, -1), np.full(m, np.nan)
    hit = R.Hit()
    o64, d64 = rays["orig"].astype(float), rays["dir"].astype(float)
    L = np.linalg.norm(d64, axis=1)
    for k in range(m):
        orc.orc_list_hit(sp, n, R.d3(o64[k]), R.d3(d64[k]), tmin, tmax, C.byref(hit))
        if hit.hit:
            best[k], t[k] = hit.index, hit.t * L[k]
    return best, t


def _sphere_terms(o, du, cen, rad, idx):
    """f64 discriminant, both roots, delta and root error of sphere idx[k] for ray k (distance units)."""
    oc = cen[idx] - o
    h = np.einsum("ij,ij->i", du, oc)
    oc2 = np.einsum("ij,ij->i", oc, oc)
    disc = h * h - (oc2 - rad[idx] ** 2)
    delta = K * EPS * np.maximum(oc2, rad[idx] ** 2)
    sq = np.sqrt(np.maximum(disc, 0.0))
    err = np.minimum(np.sqrt(delta), delta / (2 * np.maximum(np.sqrt(np.abs(disc)), 1e-300))) + K * EPS * np.abs(h)
    return disc, np.stack([h - sq, h + sq], 1), delta, err


def _classify(orc, sp, n, rays, got, tmin=TMIN, tmax=np.inf):
    """Compare device-arithmetic hits with the f64 reference.  Returns (unexplained ray indices, explained count,
    bad-t ray indices)."""
    ref_best, ref_t = _reference(orc, sp, n, rays, tmin, tmax)
    cen, rad = _geometry(sp, n)
    o = rays["orig"].astype(float)
    d = rays["dir"].astype(float)
    L = np.linalg.norm(d, axis=1)
    du = d / L[:, None]
    lo, hi = tmin * L, tmax * L
    dev_best, dev_t = got["best"].astype(int), got["t"].astype(float)

    def ambiguous(idx, mask):
        disc, roots, delta, err = _sphere_terms(o, du, cen, rad, np.where(idx >= 0, idx, 0))
        near_edge = ((np.abs(roots - lo[:, None]) <= err[:, None]) | (np.abs(roots - hi[:, None]) <= err[:, None])).any(1)
        return mask & (idx >= 0) & ((np.abs(disc) <= delta) | near_edge), roots, err

    same = ref_best == dev_best
    amb_r, roots_r, err_r = ambiguous(ref_best, np.ones(len(rays), bool))
    amb_d, roots_d, err_d = ambiguous(dev_best, np.ones(len(rays), bool))
    both = (ref_best >= 0) & (dev_best >= 0)
    # the device's sphere has an f64 root within the two errors of the reference's root: a near tie
    close = both & (np.abs(roots_d - ref_t[:, None]) <= (err_r + err_d)[:, None] + 1e-300).any(1)
    # the sphere the ray starts on: the reference re-hits it at its f64 near root (the f32 origin's offset from the
    # surface, up to an ulp of |o|) where the exact c = 0 puts that root at 0
    sidx = rays["self"].astype(int)
    _, roots_s, _, err_s = _sphere_terms(o, du, cen, rad, np.maximum(sidx, 0))
    near = np.abs(roots_s).min(1)
    self_hit = (sidx >= 0) & ((ref_best == sidx) | (dev_best == sidx)) & (near + err_s >= lo)
    explained = ~same & (amb_r | amb_d | close | self_hit)
    unexplained = np.flatnonzero(~same & ~explained)
    # where the sphere agrees the root must be within its error, unless a root sits at an interval edge; on the
    # sphere the ray starts on, c := 0 moves the far root by the f64 near root (the f32 origin's offset from the
    # surface)
    hit = same & (ref_best >= 0)
    err_t = err_r + 4 * EPS * np.abs(ref_t) + np.where(rays["self"] == ref_best, np.abs(roots_r).min(1), 0.0)
    bad_t = np.flatnonzero(hit & ~(np.abs(dev_t - ref_t) <= err_t) & ~amb_r & ~self_hit)
    return unexplained, int(explained.sum()), bad_t


def _check(orc, sp, n, rays, tmin=TMIN, tmax=np.inf, max_explained=0.0, label=""):
    got = _mirror_hits(orc, sp, n, rays, tmin, tmax)
    nogate = _mirror_hits(orc, sp, n, rays, tmin, tmax, gate=False)
    assert got.tobytes() == nogate.tobytes(), f"{label}: the gate dropped a sphere the direct form accepts"
    unexplained, explained, bad_t = _classify(orc, sp, n, rays, got, tmin, tmax)
    assert len(unexplained) == 0, f"{label}: {len(unexplained)} of {len(rays)} rays disagree unexplained"
    assert len(bad_t) == 0, f"{label}: {len(bad_t)} roots outside their error bound"
    assert explained <= max_explained * len(rays), f"{label}: {explained} of {len(rays)} explained disagreements"
    return got


# ------------------------------------------------------------------------------------------------ hit families
def _families(orc, T, rng):
    """(label, spheres, n, rays, t_min, t_max, explained-rate bound) of every family at translation T."""
    out = []
    sp13, n13 = R.chapter13_scene()
    sp13 = _translated(sp13, n13, T)
    for name, kw in CH13_CAMERAS.items():
        cam = _moved_camera(160, T, **kw)
        cam_rays = _camera_rays(orc, cam, 7, 250, 8, rng)
        out.append((f"camera-{name}", sp13, n13, cam_rays, TMIN, np.inf, 0.002))
        # explained here mostly by the reference re-hitting the sphere a ray leaves (DESIGN.md §4's exact c = 0)
        out.append((f"secondary-{name}", sp13, n13, _secondary(orc, sp13, n13, cam_rays, rng), TMIN, np.inf, 0.05))
    prng, spf, nf = R.final_scene(0xDEADBEEF)
    spf = _translated(spf, nf, T)
    cam = _moved_camera(300, T, look_from=(13, 2, 3), look_at=(0, 0, 0), vfov=20, defocus=0.6)
    cam_rays = _camera_rays(orc, cam, 5, 150, 4, rng)
    out.append(("camera-c3", spf, nf, cam_rays, TMIN, np.inf, 0.002))
    out.append(("secondary-c3", spf, nf, _secondary(orc, spf, nf, cam_rays, rng), TMIN, np.inf, 0.05))
    for r in (1e-3, 0.2, 1000.0):
        out.append((f"tangent-r{r:g}",) + _tangent_family(rng, r, T) + (TMIN, np.inf, 0.5))
    out.append(("edge-tmin",) + _edge_family(rng, T, np.inf) + (TMIN, np.inf, 1.0))
    out.append(("edge-tmax",) + _edge_family(rng, T, 2.0) + (TMIN, 2.0, 1.0))
    return out


@pytest.mark.parametrize("T", TRANSLATIONS, ids=lambda T: "T=%g,%g,%g" % T)
def test_hits_match_f64_reference_ray_by_ray(orc, T):
    rng = np.random.default_rng(abs(hash(T)) % 2**32)
    for label, sp, n, rays, tmin, tmax, bound in _families(orc, np.array(T), rng):
        _check(orc, sp, n, rays, tmin, tmax, bound, f"{label} T={T}")


@pytest.mark.parametrize("T", [(0.0, 0.0, 0.0), (1e3, 1e3, 1e3)])
def test_duplicate_spheres_lower_index_wins(orc, T):
    """Exact copies of every chapter-13 sphere listed after the originals: every hit is a tie in t, which the
    sphere listed first wins, in f64 and in the device arithmetic."""
    sp13, n13 = R.chapter13_scene()
    both = (R.Sphere * (2 * n13))()
    for i in range(n13):
        both[i] = both[n13 + i] = sp13[i]
        both[n13 + i].albedo = R.d3((0.9, 0.1, 0.1))
    sp = _translated(both, 2 * n13, np.array(T))
    rng = np.random.default_rng(3)
    rays = _camera_rays(orc, _moved_camera(160, np.array(T), **CH13_CAMERAS["ch12"]), 9, 300, 4, rng)
    got = _check(orc, sp, 2 * n13, rays, max_explained=0.01, label="duplicates")
    assert (got["best"] < n13).all()
    ref_best, _ = _reference(orc, sp, 2 * n13, rays, TMIN, np.inf)
    assert (ref_best < n13).all()


def test_inside_grazing_deviation_stays_in_its_band(orc):
    """DESIGN.md §4: a ray travelling inside the sphere it starts on at near-grazing incidence can miss its exit,
    because the exact c = 0 is applied behind the rounded gate disc >= 0 of the direct form.  On the radius-100
    ground of chapter 13 that happens where h^2 is below the rounding error of c (about eps r^2): rays leaving the
    surface inwards at 2^-k below the tangent plane.  Every such miss is explained by the error model, and they
    stay confined to the grazing band: none above an angle of 2^-6, and not all of those below."""
    rng = np.random.default_rng(11)
    c0 = np.array([0.0, -100.5, -1.0])
    sp = R.sphere_array([R.make_sphere(tuple(c0), 100.0, R.MAT_LAMBERTIAN, (0.8, 0.8, 0.0))])
    m = 20000
    nrm = _unit(rng, m)
    p = c0 + 100.0 * nrm
    t = np.cross(nrm, _unit(rng, m))
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    k = rng.integers(4, 17, size=m)
    rays = _rays(p, t - (2.0 ** -k)[:, None] * nrm, np.zeros(m, int))
    got = _check(orc, sp, 1, rays, max_explained=0.5, label="inside-grazing")
    ref_best, _ = _reference(orc, sp, 1, rays, TMIN, np.inf)
    missed = (ref_best == 0) & (got["best"] < 0)
    rate = [missed[k == j].mean() for j in range(4, 17)]
    assert max(rate[:3]) == 0.0, rate
    assert max(rate) < 1.0, rate


# ------------------------------------------------------------------------------------------------ scatters
def _philox_uniforms(orc, seed, pixel, sample, bounce):
    ctr = (C.c_uint32 * 4)(pixel, sample, bounce, 0)
    key = (C.c_uint32 * 2)(seed & 0xFFFFFFFF, seed >> 32)
    out = (C.c_uint32 * 4)()
    orc.orc_philox(ctr, key, out)
    return np.array([(x >> 8) * 2.0 ** -24 for x in out])


def _scatter_f64(orc, sp, rec, seed):
    """material.zig in f64 from the f64 hit of the record's ray: (term, unit direction, attenuation, margins)."""
    s = sp[rec["sphere"]]
    c, r = np.array(s.center[:]), s.radius
    o, d = rec["orig"].astype(float), rec["dir"].astype(float)
    du = d / np.linalg.norm(d)
    oc = c - o
    h = du @ oc
    disc = h * h - (oc @ oc - r * r)
    if disc < 0:
        return None, disc, K * EPS * max(oc @ oc, r * r)
    t = h - np.sqrt(disc) if h - np.sqrt(disc) > TMIN * np.linalg.norm(d) else h + np.sqrt(disc)
    p = o + t * du
    n = (p - c) / r
    front = du @ n < 0
    if not front:
        n = -n
    u = _philox_uniforms(orc, seed, int(rec["pixel"]), int(rec["sample"]), int(rec["bounce"]) + 1)
    # the hit point's rounding, and the root's own error moving it along the ray (large at grazing incidence),
    # both turn the normal by about their size over r
    delta = K * EPS * max(oc @ oc, r * r)
    root_err = min(np.sqrt(delta), delta / (2 * max(np.sqrt(disc), 1e-300))) + K * EPS * abs(h)
    tol = K * EPS * (1 + np.linalg.norm(p) / r) + root_err / r
    if s.mat_type == R.MAT_DIELECTRIC:
        ri = 1.0 / s.refraction_index if front else s.refraction_index
        cos_t = min(-(du @ n), 1.0)
        sin_t = np.sqrt(1.0 - cos_t * cos_t)
        q = ((1 - ri) / (1 + ri)) ** 2
        refl = q + (1 - q) * (1 - cos_t) ** 5
        margin = min(abs(ri * sin_t - 1), abs(refl - u[0]))
        if ri * sin_t > 1 or refl > u[0]:
            nd = du - 2 * (du @ n) * n
        else:
            perp = ri * (du + cos_t * n)
            nd = perp - np.sqrt(abs(1 - perp @ perp)) * n
        return -1, nd / np.linalg.norm(nd), np.ones(3), margin, tol / max(np.sqrt(abs(1 - (ri * sin_t) ** 2)), np.sqrt(tol)), tol
    z = 1 - 2 * u[1]
    uv = np.array([np.sqrt(1 - z * z) * np.cos(2 * np.pi * u[2]), np.sqrt(1 - z * z) * np.sin(2 * np.pi * u[2]), z])
    alb = np.float32(np.array(s.albedo[:]))
    if s.mat_type == R.MAT_LAMBERTIAN:
        nd = n + uv
        margin = abs(nd - 1e-8).min()
        if (nd < 1e-8).all():
            nd = n
        return -1, nd / np.linalg.norm(nd), alb, margin, tol / max(np.linalg.norm(nd), np.sqrt(tol)), tol
    nd = du - 2 * (du @ n) * n + s.fuzz * uv
    margin = abs(nd @ n) / max(np.linalg.norm(nd), 1e-30)
    if not nd @ n > 0:
        return 1, None, None, margin, 0.0, tol
    return -1, nd / np.linalg.norm(nd), alb, margin, tol / max(np.linalg.norm(nd), np.sqrt(tol)), tol


def _scatter_records(rng, T):
    """Lambertian, metal (fuzz 0, 0.3, 1.5) and dielectric (ior 1.5, 1/1.5, 1, 2.4) spheres; rays hitting them from
    outside (front) and from inside (back, dielectrics), at angles from head-on to 1e-6 rad from grazing."""
    mats = [R.make_sphere((0, 0, 0), 0.5, R.MAT_LAMBERTIAN, (0.8, 0.3, 0.1))]
    mats += [R.make_sphere((0, 0, 0), 0.5, R.MAT_METAL, (0.7, 0.6, 0.5), fuzz=f) for f in (0.0, 0.3, 1.5)]
    mats += [R.make_sphere((0, 0, 0), 0.5, R.MAT_DIELECTRIC, ior=e) for e in (1.5, 1 / 1.5, 1.0, 2.4)]
    sp = _translated(R.sphere_array(mats), len(mats), T)
    recs = []
    m = 400
    for i in range(len(mats)):
        c = np.array(sp[i].center[:])
        for inside in ((False, True) if mats[i].mat_type == R.MAT_DIELECTRIC else (False,)):
            nrm = _unit(rng, m)
            tan = np.cross(nrm, _unit(rng, m))
            tan /= np.linalg.norm(tan, axis=1, keepdims=True)
            # incidence angle from the normal: head-on .. 1e-6 rad from grazing, dense around 40-45 degrees
            ang = np.concatenate([rng.uniform(0, np.pi / 2 - 1e-6, m // 2), np.pi / 2 - 10.0 ** rng.uniform(-6, -1, m // 4),
                                  rng.uniform(np.radians(38), np.radians(46), m - m // 2 - m // 4)])
            d = -np.cos(ang)[:, None] * nrm + np.sin(ang)[:, None] * tan
            p = c + 0.5 * nrm
            if inside:  # from inside, exiting at p; short directions keep t_min |d| below half the chord
                d = (np.cos(ang)[:, None] * nrm + np.sin(ang)[:, None] * tan) * 1e-4
                o = p - d * (0.5 * np.cos(ang) * 1e4)[:, None]
            else:
                o = p - d * 2.0
            for k in range(m):
                recs.append((i, np.float32(o[k]), np.float32(d[k]), int(rng.integers(1 << 20)), k, int(rng.integers(8))))
    out = np.zeros(len(recs), BOUNCE)
    for k, (i, o, d, px, smp, b) in enumerate(recs):
        out[k] = (i, o, d, px, smp, b)
    return sp, len(mats), out


@pytest.mark.parametrize("T", [(0.0, 0.0, 0.0), (1e2, 0.0, 0.0), (0.0, 0.0, 1e3), (1e4, 1e4, 1e4)],
                         ids=lambda T: "T=%g,%g,%g" % T)
def test_scatters_match_f64_material(orc, T):
    rng = np.random.default_rng(17)
    seed = 0xABADCAFE12345678
    sp, n, recs = _scatter_records(rng, np.array(T))
    got = np.zeros(len(recs), SCAT)
    orc.orc_mirror_scatters(sp, n, _ptr(recs), len(recs), seed, _ptr(got))
    bad_branch, bad_dir, bad_att, misses = [], [], [], 0
    for k in range(len(recs)):
        ref = _scatter_f64(orc, sp, recs[k], seed)
        if ref[0] is None or got["term"][k] == -2:  # a miss: both, or one where the ray is tangent in f64
            if (ref[0] is None) != (got["term"][k] == -2):
                misses += 1
                o, d = recs["orig"][k].astype(float), recs["dir"][k].astype(float)
                du = d / np.linalg.norm(d)
                oc = np.array(sp[recs["sphere"][k]].center[:]) - o
                h, r = du @ oc, sp[recs["sphere"][k]].radius
                assert abs(h * h - (oc @ oc - r * r)) <= K * EPS * max(oc @ oc, r * r), recs[k]
            continue
        term, nd, att, margin, ang_tol, tol = ref
        if term != got["term"][k]:
            if margin > 4 * tol:
                bad_branch.append(k)
            continue
        if term != -1:
            continue
        gd = got["dir"][k].astype(float)
        cosang = np.clip(gd @ nd / np.linalg.norm(gd), -1, 1)
        if np.arccos(cosang) > 4 * ang_tol + 1e-6 and margin > 4 * tol:
            bad_dir.append(k)
        if not np.array_equal(got["attenuation"][k], np.float32(att)):
            bad_att.append(k)
    assert misses <= 0.1 * len(recs), misses  # a quarter of the records graze their sphere
    assert not bad_branch, (len(bad_branch), recs[bad_branch[:3]])
    assert not bad_dir, (len(bad_dir), recs[bad_dir[:3]])
    assert not bad_att, (len(bad_att), recs[bad_att[:3]])


def test_sampling_over_all_uniforms(orc):
    """cosSin2Pi over all 2^24 uniforms against f64 (DESIGN.md §4: |err| < 2e-7); the unit vector's norm within a
    few ulps of 1; lens points in the closed unit disk."""
    N = 1 << 24
    c, s = np.zeros(N, np.float32), np.zeros(N, np.float32)
    F = C.POINTER(C.c_float)
    orc.orc_mirror_cos_sin_all(c.ctypes.data_as(F), s.ctypes.data_as(F))
    a = 2 * np.pi * np.arange(N, dtype=np.float64) * 2.0 ** -24
    assert np.abs(c - np.cos(a)).max() < 2e-7
    assert np.abs(s - np.sin(a)).max() < 2e-7
    rng = np.random.default_rng(5)
    idx = rng.integers(N, size=1 << 20)
    z = np.float32(1.0) - np.float32(2.0) * np.float32(rng.integers(N, size=1 << 20) * 2.0 ** -24)
    rad = np.sqrt(np.float32(1.0) - z * z)
    v = np.stack([rad * c[idx], rad * s[idx], z], 1).astype(np.float64)
    assert np.abs(np.linalg.norm(v, axis=1) - 1).max() < 8 * 2.0 ** -24
    r = np.sqrt(np.float32(rng.integers(N, size=1 << 20) * 2.0 ** -24))
    disk = np.hypot((r * c[idx]).astype(float), (r * s[idx]).astype(float))
    assert disk.max() <= 1.0


# ------------------------------------------------------------------------------------------------ whole renders
def _render(orc, fn, cam, sp, n, seed, linear=False):
    rgb = np.zeros((cam.height, cam.width, 3), np.uint8)
    lin = np.zeros((cam.height * cam.width, 3)) if linear else None
    st = R.Stats()
    u8 = rgb.ctypes.data_as(C.POINTER(C.c_uint8))
    lp = lin.ctypes.data_as(C.POINTER(C.c_double)) if linear else None
    if fn == "mirror":
        assert orc.orc_render_mirror(C.byref(cam), sp, n, seed, 8, None, u8, lp, C.byref(st)) == 0
    else:
        assert orc.orc_render_philox64(C.byref(cam), sp, n, seed, 8, u8, lp, C.byref(st)) == 0
    return rgb, lin, st


def _mirror_no_gate(orc, cam, sp, n, seed):
    orc.orc_mirror_set_gate(0)
    try:
        return _render(orc, "mirror", cam, sp, n, seed, linear=True)
    finally:
        orc.orc_mirror_set_gate(1)


@pytest.mark.parametrize("T", [(300.0, 0.0, 0.0), (0.0, 0.0, 1000.0), (3000.0, 3000.0, 0.0)],
                         ids=lambda T: "T=%g,%g,%g" % T)
def test_translated_chapter13_mirror_vs_f64(orc, T):
    """The chapter-13 scene and ch12 camera moved by T: the mirror stays within the statistical gates of
    test_oracle_stat.py, and equals the mirror without the candidate gate bit for bit."""
    sp, n = R.chapter13_scene()
    sp = _translated(sp, n, np.array(T))
    cam = _moved_camera(200, np.array(T), **CH13_CAMERAS["ch12"])
    cam.samples_per_pixel, cam.pixel_samples_scale = 64, 1.0 / 64
    m, mlin, mst = _render(orc, "mirror", cam, sp, n, 7, linear=True)
    _, glin, gst = _mirror_no_gate(orc, cam, sp, n, 7)
    assert np.array_equal(mlin, glin) and (mst.segments, mst.absorbed) == (gst.segments, gst.absorbed)
    a, _, ast = _render(orc, "ref", cam, sp, n, 1)
    b, _, _ = _render(orc, "ref", cam, sp, n, 2)
    m, a, b = (x.astype(float) for x in (m, a, b))
    floor, rm = np.sqrt(np.mean((a - b) ** 2)), np.sqrt(np.mean((m - a) ** 2))
    bias = (m - a).mean(axis=(0, 1))
    assert rm <= 1.25 * floor, (rm, floor)
    assert np.abs(bias).max() <= 0.25, bias
    seg_m, seg_a = mst.segments / mst.samples, ast.segments / ast.samples
    assert abs(seg_m - seg_a) / seg_a < 0.02, (seg_m, seg_a)


@pytest.mark.parametrize("T", [(0.0, 0.0, 0.0), (1000.0, 0.0, 1000.0)], ids=lambda T: "T=%g,%g,%g" % T)
def test_final_scene_gate_only_filters(orc, T):
    """The book's final scene: the mirror with the candidate gate equals the mirror without it (every sphere sent
    to the direct form), bit for bit; moved by T it also stays within the statistical gates."""
    prng, sp, n = R.final_scene(0xDEADBEEF)
    sp = _translated(sp, n, np.array(T))
    cam = _moved_camera(160, np.array(T), look_from=(13, 2, 3), look_at=(0, 0, 0), vfov=20, defocus=0.6)
    cam.samples_per_pixel, cam.pixel_samples_scale = 32, 1.0 / 32
    m, mlin, mst = _render(orc, "mirror", cam, sp, n, 0xDEADBEEF, linear=True)
    _, glin, gst = _mirror_no_gate(orc, cam, sp, n, 0xDEADBEEF)
    assert np.array_equal(mlin, glin) and (mst.segments, mst.absorbed) == (gst.segments, gst.absorbed)
    if any(T):
        a, _, ast = _render(orc, "ref", cam, sp, n, 1)
        b, _, _ = _render(orc, "ref", cam, sp, n, 2)
        m, a, b = (x.astype(float) for x in (m, a, b))
        floor, rm = np.sqrt(np.mean((a - b) ** 2)), np.sqrt(np.mean((m - a) ** 2))
        assert rm <= 1.25 * floor, (rm, floor)
        assert np.abs((m - a).mean(axis=(0, 1))).max() <= 0.25
        assert abs(mst.segments / mst.samples - ast.segments / ast.samples) / (ast.segments / ast.samples) < 0.02


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_probes_equal_mirror_twins_bit_exact(pkg, orc):
    l = pkg.lib()
    P = C.POINTER(pkg.rtz_sphere)
    rng = np.random.default_rng(23)
    for T in [TRANSLATIONS[0], TRANSLATIONS[4], TRANSLATIONS[9], TRANSLATIONS[12]]:
        for label, sp, n, rays, tmin, tmax, _ in _families(orc, np.array(T), rng):
            want = _mirror_hits(orc, sp, n, rays, tmin, tmax)
            got = np.zeros(len(rays), HIT)
            assert l.rtz_probe_hits(C.cast(sp, P), n, _ptr(rays), len(rays), tmin, tmax, _ptr(got)) == 0
            assert got.tobytes() == want.tobytes(), (label, T, int((got != want).sum()))
        sp, n, recs = _scatter_records(rng, np.array(T))
        want = np.zeros(len(recs), SCAT)
        orc.orc_mirror_scatters(sp, n, _ptr(recs), len(recs), 99, _ptr(want))
        got = np.zeros(len(recs), SCAT)
        assert l.rtz_probe_scatters(C.cast(sp, P), n, _ptr(recs), len(recs), 99, _ptr(got)) == 0
        assert got.tobytes() == want.tobytes(), (T, int((got != want).sum()))
    bad = np.zeros(1, BOUNCE)
    bad["sphere"] = 99
    assert l.rtz_probe_scatters(C.cast(sp, P), n, _ptr(bad), 1, 0, _ptr(np.zeros(1, SCAT))) == 1


def _sweep_scene(orc, n, T):
    prng = orc.orc_prng_new(0xDEADBEEF)
    sp = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, sp) == n
    orc.orc_prng_free(prng)
    return _translated(sp, n, np.array(T))


@pytest.mark.gpu
@pytest.mark.parametrize("n_spheres", [4, 9, 16, 32, 33, 64, 65, 200, 256, 257, 485, 513, 4096, 8192])
def test_translated_scene_equals_mirror_in_every_kernel(pkg, gpu, orc, monkeypatch, n_spheres):
    """A sweep scene moved to (1000, 1000, 1000) (and the final scene, at 485, so that the culled kernel runs)
    through every trace kernel that serves its size: bytes, fixed-point sums and counters equal the mirror's."""
    T = np.array((1000.0, 1000.0, 1000.0))
    if n_spheres == 485:
        prng, sp, n = R.final_scene(0xDEADBEEF)
        sp = _translated(sp, n, T)
    else:
        sp, n = _sweep_scene(orc, n_spheres, T), n_spheres
    cam = _moved_camera(96 if n < 4096 else 64, T, look_from=(13, 2, 3), look_at=(0, 0, 0), vfov=20, defocus=0.6)
    cam.samples_per_pixel, cam.pixel_samples_scale, cam.seed, cam.has_seed = 8, 1.0 / 8, 0x5EED, 1
    mrgb, mlin, mst = _render(orc, "mirror", cam, sp, n, 0x5EED, linear=True)
    envs = [{}, {"RTZ_DRAIN": "0"}, {"RTZ_VARIANT": "11"}, {"RTZ_VARIANT": "11", "RTZ_DRAIN": "0"},
            {"RTZ_VARIANT": "1"}, {"RTZ_VARIANT": "2"}, {"RTZ_VARIANT": "3"}]
    if n <= 256:
        envs += [{"RTZ_VARIANT": "8"}, {"RTZ_VARIANT": "12"}, {"RTZ_VARIANT": "12", "RTZ_DRAIN": "0"}]
    for env in envs:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        r = pkg.Renderer(0)
        try:
            r.upload(sp, n)
            for mode in (R.MODE_PATH, R.MODE_PATH_BVH) if not env else (R.MODE_PATH,):
                cam.mode = mode
                img, st = r.render(cam)
                assert np.array_equal(img.cpu().numpy().reshape(-1, 3), mrgb.reshape(-1, 3)), (env, mode)
                assert (st.samples, st.segments, st.depth_capped, st.absorbed) == (
                    mst.samples, mst.segments, mst.depth_capped, mst.absorbed), (env, mode)
            cam.mode = R.MODE_PATH
        finally:
            r.close()
        for k in env:
            monkeypatch.delenv(k)
    rgb, st, lin = pkg.render_host(cam, sp, n, want_linear=True)
    assert np.array_equal(lin.reshape(-1, 3), mlin)
