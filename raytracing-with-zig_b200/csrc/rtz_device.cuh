// rtz_device.cuh — device functions of the B200 path tracer (sm_100a).
//
// These are the GPU restatements of the reference's per-sample functions:
//   getRay / sampleSquare / defocusDiskSample   reference src/camera.zig:187-215
//   HittableList.hit + Sphere.hit                reference src/hittable.zig:64-77, src/sphere.zig:26-54
//   Lambertian / Metal / Dielectric .scatter     reference src/material.zig:27-110
//   Vec.reflect / refract / nearZero             reference src/vec.zig:26-29,103-112
//
// ARITHMETIC CONTRACT (DESIGN.md §4).  Everything is FP32 with IEEE round-to-nearest +, -, *,
// /, sqrt and EXPLICIT fmaf(); the translation unit is compiled with -fmad=false so the
// compiler never contracts on its own.  No approximate intrinsics.  The CPU oracle keeps an
// independent mirror of this contract (oracle/rtz_mirror.cpp) and the parity tests require the
// two to agree BIT FOR BIT on the fixed-point pixel sums.
//
// Differences from the reference's formulation, all distribution-preserving:
//   * the ray direction is normalised once per segment (a = |d|^2 = 1 in Sphere.hit); t_min is
//     rescaled by |d| so the (t_min, inf) interval keeps its reference meaning (Q7/Q8);
//   * |d|^2 and r^2 are hoisted out of the sphere sweep (17 algorithmic FLOP / test, SURVEY §8d);
//   * the per-test miss/hit decision uses the discriminant expanded around per-ray constants,
//         h = d.c - d.o ,   c' = (|c|^2 - r^2) - 2 c.o + |o|^2 ,   disc = h^2 - c'
//     (8 fused ops per test instead of 10, and no 1e6-sized cancellation for the radius-1000
//     ground sphere); the ROOT of a candidate is then computed from the reference's direct form
//     oc = c - o, exactly as Sphere.hit writes it;
//   * the sphere the ray starts on ("self") is intersected with c = |oc|^2 - r^2 := 0, the exact
//     value, instead of the FP32-rounded one: this removes the self-intersection bias of a
//     naive FP32 port (SURVEY §7 risk 5) without touching any other sphere;
//   * RNG is Philox4x32-10 keyed (seed) with counter (pixel, sample, bounce, 0) instead of
//     one shared sequential Xoshiro stream (north_star); unit vectors and lens points are drawn in
//     CLOSED FORM (z uniform + angle; sqrt(u) + angle; sine / cosine from FP32 minimax polynomials)
//     instead of the reference's rejection loops (accept pi/6 and pi/4): same uniform distributions,
//     no data-dependent loop, exactly one Philox block per camera ray and per scatter.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rtz {

// Material type tags live in the .w lane of the aux float4 as integer bits.
constexpr int kLambertian = 0, kMetal = 1, kDielectric = 2;

struct DevCamera {
    float p0x, p0y, p0z;     // pixel0
    float dux, duy, duz;     // du
    float dvx, dvy, dvz;     // dv
    float cx, cy, cz;        // center
    float uux, uuy, uuz;     // defocusDiskU
    float vvx, vvy, vvz;     // defocusDiskV
    float tmin, tmax;        // Scene.interval (src/Scene.zig:21): (1e-3, +inf) by default
    int defocus;             // defocusAngle > 0
    uint32_t width, height, spp, bounce_max;
    uint32_t key0, key1;     // Philox key = seed
    uint32_t rk0[10], rk1[10];  // its ten round keys (key + r * Weyl constants), precomputed on the host: the kernels
                                // read them as constant-bank operands of the XORs instead of bumping the key per round
};

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11).  10 rounds, 2 x (IMAD.HI + IMAD.LO) each.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0, c1 = lo1, c2 = n2, c3 = lo0;
        k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// the same with the round keys taken from the camera block (kernel parameter = constant bank)
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const DevCamera& cam) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ cam.rk0[r], n2 = hi0 ^ c3 ^ cam.rk1[r];
        c0 = n0, c1 = lo1, c2 = n2, c3 = lo0;
    }
    return make_uint4(c0, c1, c2, c3);
}

// uniform in [0,1): top 24 bits, exact in FP32
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * 0x1p-24f; }

struct RngKey {
    uint32_t k0, k1, pixel, sample;
};

// (cos 2*pi*u, sin 2*pi*u) for the 24-bit uniform u = (x >> 8) * 2^-24.  The top two bits of u pick the quarter
// turn exactly; the other 22 are the fraction f of that quarter, and sin(pi/2 f) = f S(f^2), cos(pi/2 f) = C(f^2)
// with degree-4 minimax polynomials (|error| < 2e-7, measured over all 2^22 arguments).  Only IEEE multiplies and
// explicit fmaf: the CPU mirror reproduces it bit for bit, and there is no rejection loop — every sample costs
// the same instructions in every lane, and a camera ray / a scatter consumes exactly ONE Philox block.
__device__ __forceinline__ void cos_sin_2pi(uint32_t x, float& c, float& s) {
    const uint32_t q = x >> 30;
    const float f = (float)((x >> 8) & 0x3FFFFFu) * 0x1p-22f;
    const float z = f * f;
    float sp = fmaf(z, 0x1.3e7abap-13f, -0x1.3259fap-8f);
    sp = fmaf(z, sp, 0x1.46693cp-4f);
    sp = fmaf(z, sp, -0x1.4abbc6p-1f);
    sp = fmaf(z, sp, 0x1.921fb6p+0f);
    sp = sp * f;
    float cp = fmaf(z, 0x1.c29b9cp-11f, -0x1.550192p-6f);
    cp = fmaf(z, cp, 0x1.03bd86p-2f);
    cp = fmaf(z, cp, -0x1.3bd3aep+0f);
    cp = fmaf(z, cp, 1.0f);
    const float a = (q & 1u) ? sp : cp;  // |cos|, |sin| after q quarter turns
    const float b = (q & 1u) ? cp : sp;
    c = (q == 1u || q == 2u) ? -a : a;
    s = (q >= 2u) ? -b : b;
}

// Vec.randomInUnitDisk (src/vec.zig:82-92): uniform in the unit disk.  The reference rejects from the square;
// here the same distribution in closed form: radius sqrt(u1), angle 2*pi*u2.
__device__ __forceinline__ void sample_disk(uint32_t x1, uint32_t x2, float& a, float& b) {
    const float rad = sqrtf(u01(x1));
    float c, s;
    cos_sin_2pi(x2, c, s);
    a = rad * c, b = rad * s;
}

// Vec.randomUnitVec (src/vec.zig:71-80): uniform on the unit sphere.  The reference rejects from the cube and
// normalises; here the same distribution in closed form (Archimedes): z uniform in (-1, 1], angle 2*pi*u2.
__device__ __forceinline__ void random_unit_vec(uint32_t x1, uint32_t x2, float& ux, float& uy, float& uz) {
    const float z = fmaf(-2.0f, u01(x1), 1.0f);
    const float rad = sqrtf(fmaf(-z, z, 1.0f));
    float c, s;
    cos_sin_2pi(x2, c, s);
    ux = rad * c, uy = rad * s, uz = z;
}

// ---------------------------------------------------------------------------------------------
// Per-lane path state
// ---------------------------------------------------------------------------------------------
struct Path {
    float ox, oy, oz;   // ray origin
    float dx, dy, dz;   // ray direction, UNIT length
    float tr, tg, tb;   // throughput (returnColor of rayColor)
    float len;          // |d| before normalisation: the hit interval in distance units is (t_min*len, t_max*len)
    int self;           // sphere the origin lies on, -1 for camera rays
    uint32_t bounce;    // scatters so far
};

// Store an un-normalised direction: normalise and keep its length, which rescales Scene.interval (Q7/Q8).
__device__ __forceinline__ void set_direction(Path& p, float dx, float dy, float dz) {
    const float len2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
    const float len = sqrtf(len2);
    const float inv = 1.0f / len;
    p.dx = dx * inv, p.dy = dy * inv, p.dz = dz * inv;
    p.len = len;
}

// Camera.getRay (src/camera.zig:187-200) for pixel (i,j), sample k.sample.
__device__ __forceinline__ void camera_ray(const DevCamera& c, const RngKey& k, uint32_t i, uint32_t j, Path& p) {
    const uint4 r = philox4x32_10(k.pixel, k.sample, 0u, 0u, c);
    const float sx = (float)i + (u01(r.x) - 0.5f);  // sampleSquare (:203-209)
    const float sy = (float)j + (u01(r.y) - 0.5f);
    const float psx = fmaf(c.dvx, sy, fmaf(c.dux, sx, c.p0x));
    const float psy = fmaf(c.dvy, sy, fmaf(c.duy, sx, c.p0y));
    const float psz = fmaf(c.dvz, sy, fmaf(c.duz, sx, c.p0z));
    p.ox = c.cx, p.oy = c.cy, p.oz = c.cz;
    if (c.defocus) {  // defocusDiskSample (:212-215)
        float a, b;
        sample_disk(r.z, r.w, a, b);
        p.ox = fmaf(c.vvx, b, fmaf(c.uux, a, c.cx));
        p.oy = fmaf(c.vvy, b, fmaf(c.uuy, a, c.cy));
        p.oz = fmaf(c.vvz, b, fmaf(c.uuz, a, c.cz));
    }
    set_direction(p, psx - p.ox, psy - p.oy, psz - p.oz);
    p.tr = p.tg = p.tb = 1.0f;
    p.self = -1;
    p.bounce = 0;
}

// ---------------------------------------------------------------------------------------------
// HittableList.hit: brute-force closest hit over all spheres (src/hittable.zig:64-77), with
// Sphere.hit's half-b quadratic (src/sphere.zig:26-43) for a unit direction.
// Algorithmic cost per test: 17 FLOP (miss path of src/sphere.zig:27-33, |d|^2 and r^2 hoisted);
// executed: 7 FFMA + 1 FADD on the expanded form.  The root is only evaluated for candidates.
// ---------------------------------------------------------------------------------------------
// Does root t of sphere i replace the running closest hit (closest, best)?  The ascending loop's rule is "strictly
// nearer", so an exact tie keeps the earlier sphere.  A sweep that visits the spheres in another order (the culled
// kernel's regrouped blocks) passes `orig`, slot -> index in the caller's list: a tie then goes to the lower
// original index, which is the sphere the ascending loop keeps.  best < 0 (closest = t_max) never ties.
__device__ __forceinline__ bool nearer(float t, int i, float closest, int best, const int* __restrict__ orig) {
    return t < closest || (orig && t == closest && best >= 0 && __ldg(orig + i) < __ldg(orig + best));
}
__device__ __forceinline__ void slow_path(float h, float disc, int i, int self, float tmin_d, float& closest,
                                          int& best, const int* __restrict__ orig = nullptr) {
    if (i == self) disc = h * h;  // exact c = 0 for the sphere we stand on
    const float sq = sqrtf(disc);
    float t = h - sq;  // (h - sqrtd)/a with a = 1
    if (!(t > tmin_d && nearer(t, i, closest, best, orig))) {  // Interval.surrounds is strict (src/interval.zig:36-38)
        t = h + sq;
        if (!(t > tmin_d && nearer(t, i, closest, best, orig))) return;
    }
    closest = t;  // shrinking t_max; ties keep the earlier sphere
    best = i;
}

// per-ray constants of the expanded discriminant
struct RayK {
    float k1;             // -(d.o)
    float nk2;            // -|o|^2
    float tx, ty, tz;     // 2*o
};
__device__ __forceinline__ RayK ray_constants(const Path& p) {
    RayK k;
    k.k1 = -fmaf(p.dz, p.oz, fmaf(p.dy, p.oy, p.dx * p.ox));
    k.nk2 = -fmaf(p.oz, p.oz, fmaf(p.oy, p.oy, p.ox * p.ox));
    k.tx = 2.0f * p.ox, k.ty = 2.0f * p.oy, k.tz = 2.0f * p.oz;
    return k;
}
// candidate test: sign of the expanded discriminant; cw = -(|c|^2 - r^2) from the host
__device__ __forceinline__ float expanded_disc(float cx, float cy, float cz, float cw, const Path& p, const RayK& k) {
    const float h = fmaf(p.dz, cz, fmaf(p.dy, cy, fmaf(p.dx, cx, k.k1)));
    const float w = fmaf(k.tz, cz, fmaf(k.ty, cy, fmaf(k.tx, cx, k.nk2))) + cw;
    return fmaf(h, h, w);
}
// root of a candidate from the direct form (src/sphere.zig:27-42); g = {cx, cy, cz, -r^2}
__device__ __forceinline__ void candidate_root(const float4 g, float nr2, int i, const Path& p, float tmin_d,
                                               float& closest, int& best, const int* __restrict__ orig = nullptr) {
    const float ocx = g.x - p.ox, ocy = g.y - p.oy, ocz = g.z - p.oz;
    const float h = fmaf(p.dz, ocz, fmaf(p.dy, ocy, p.dx * ocx));
    const float c = fmaf(ocz, ocz, fmaf(ocy, ocy, fmaf(ocx, ocx, nr2)));
    const float disc = fmaf(h, h, -c);
    if (disc >= 0.0f) slow_path(h, disc, i, p.self, tmin_d, closest, best, orig);
}

// scalar sweep over plain rows {cx, cy, cz, -r^2} + the pair layout's w: serves the one-ray probes;
// the render kernel runs the same arithmetic on sphere pairs (sweep2 in rtz_kernels.cuh)
__device__ __forceinline__ float pair_w(const float4* __restrict__ pairs, int i) {
    const float4 p1 = pairs[(i & ~1) + 1];
    return (i & 1) ? p1.w : p1.z;
}
__device__ __forceinline__ void sweep_rows(const float4* __restrict__ geo, const float4* __restrict__ pairs, int first,
                                           int n, const Path& p, float tmin, float tmax, float& t_out, int& best_out) {
    const float tmin_d = tmin * p.len;
    float closest = tmax * p.len;  // Interval(t_min, t_max) in distance units; +inf stays +inf
    int best = -1;
    const RayK k = ray_constants(p);
    for (int i = first; i < first + n; ++i) {
        const float4 g = geo[i];
        const float d = expanded_disc(g.x, g.y, g.z, pair_w(pairs, i), p, k);
        if (!(__float_as_uint(d) >> 31)) candidate_root(g, g.w, i, p, tmin_d, closest, best);
    }
    t_out = closest;
    best_out = best;
}

// ---------------------------------------------------------------------------------------------
// Shading of one finished segment.  Returns true when the sample is finished; then (sr,sg,sb)
// is its colour.  `term` reports why: 0 sky, 1 absorbed, 2 depth cap.
//   aux[i]    = {r, 1/r, fuzz | ior, type bits}
//   albedo[i] = {r, g, b, 1/ior}
// ---------------------------------------------------------------------------------------------
// kFlagSelf (the wavefront kernel): a scattered ray that LEAVES the sphere it starts on cannot hit it — with the
// exact c = 0 its roots are h - |h| and h + |h|, both <= 0 when h = d.(centre - origin) <= 0 — so the sweep may drop
// that sphere from its candidates.  The flag (bit 30 of `self`) is set from the very h candidate_root would form.
constexpr int kSelfLeaves = 0x40000000;
template <bool kFlagSelf = false>
__device__ __forceinline__ bool shade(const DevCamera& cam, const RngKey& k, const float4* __restrict__ geo,
                                      const float4* __restrict__ aux, const float4* __restrict__ albedo, Path& p,
                                      float t, int best, float& sr, float& sg, float& sb, int& term) {
    if (best < 0) {
        // sky (src/camera.zig:171-177): a = 0.5*(unit(dir).y + 1); white*(1-a) + blue*a
        const float a = 0.5f * (p.dy + 1.0f);
        const float w = 1.0f - a;
        sr = p.tr * fmaf(a, 0.5f, w);
        sg = p.tg * fmaf(a, 0.7f, w);
        sb = p.tb * fmaf(a, 1.0f, w);
        term = 0;
        return true;
    }
    const float4 gc = geo[best];
    const float gx = gc.x, gy = gc.y, gz = gc.z;
    const float4 ax = __ldg(aux + best);
    const float4 al = __ldg(albedo + best);
    // HitRecord (src/sphere.zig:44-53)
    const float px = fmaf(t, p.dx, p.ox), py = fmaf(t, p.dy, p.oy), pz = fmaf(t, p.dz, p.oz);
    float nx = (px - gx) * ax.y, ny = (py - gy) * ax.y, nz = (pz - gz) * ax.y;
    float dn = fmaf(p.dz, nz, fmaf(p.dy, ny, p.dx * nx));
    const bool front = dn < 0.0f;
    if (!front) nx = -nx, ny = -ny, nz = -nz, dn = -dn;
    const int type = __float_as_int(ax.w);
    const uint32_t stream = p.bounce + 1u;  // stream 0 belongs to the camera ray
    const uint4 r0 = philox4x32_10(k.pixel, k.sample, stream, 0u, cam);
    float ndx, ndy, ndz;
    if (type == kDielectric) {
        // Dielectric.scatter (src/material.zig:82-103)
        const float ri = front ? al.w : ax.z;
        const float cosT = fminf(-dn, 1.0f);
        const float sinT = sqrtf(fmaf(-cosT, cosT, 1.0f));
        const bool cannot = ri * sinT > 1.0f;
        float q = (1.0f - ri) / (1.0f + ri);
        q = q * q;
        const float x = 1.0f - cosT;
        const float x2 = x * x;
        const float refl = fmaf(1.0f - q, x * (x2 * x2), q);  // Schlick (:106-110)
        if (cannot || refl > u01(r0.x)) {
            const float kk = -2.0f * dn;  // Vec.reflect (src/vec.zig:103-105)
            ndx = fmaf(kk, nx, p.dx), ndy = fmaf(kk, ny, p.dy), ndz = fmaf(kk, nz, p.dz);
        } else {  // Vec.refract (src/vec.zig:107-112)
            const float ex = ri * fmaf(cosT, nx, p.dx), ey = ri * fmaf(cosT, ny, p.dy), ez = ri * fmaf(cosT, nz, p.dz);
            const float kk = -sqrtf(fabsf(1.0f - fmaf(ez, ez, fmaf(ey, ey, ex * ex))));
            ndx = fmaf(kk, nx, ex), ndy = fmaf(kk, ny, ey), ndz = fmaf(kk, nz, ez);
        }
    } else {
        float ux, uy, uz;
        random_unit_vec(r0.y, r0.z, ux, uy, uz);
        if (type == kLambertian) {
            // Lambertian.scatter (src/material.zig:27-39) incl. nearZero WITHOUT abs (Q1)
            ndx = nx + ux, ndy = ny + uy, ndz = nz + uz;
            if (ndx < 1e-8f && ndy < 1e-8f && ndz < 1e-8f) ndx = nx, ndy = ny, ndz = nz;
        } else {
            // Metal.scatter (src/material.zig:55-68): reflect + fuzz * unit vector; absorbed
            // when the fuzzed direction points into the surface.  fuzz is not clamped (Q5).
            const float kk = -2.0f * dn;
            ndx = fmaf(ax.z, ux, fmaf(kk, nx, p.dx));
            ndy = fmaf(ax.z, uy, fmaf(kk, ny, p.dy));
            ndz = fmaf(ax.z, uz, fmaf(kk, nz, p.dz));
            if (!(fmaf(ndz, nz, fmaf(ndy, ny, ndx * nx)) > 0.0f)) {
                sr = sg = sb = 0.0f;
                term = 1;
                return true;
            }
        }
        p.tr *= al.x, p.tg *= al.y, p.tb *= al.z;
    }
    p.bounce += 1u;
    if (p.bounce >= cam.bounce_max) {  // src/camera.zig:153,181 (Q9)
        sr = sg = sb = 0.0f;
        term = 2;
        return true;
    }
    p.ox = px, p.oy = py, p.oz = pz;
    set_direction(p, ndx, ndy, ndz);
    p.self = best;
    if (kFlagSelf) {
        const float ocx = gx - px, ocy = gy - py, ocz = gz - pz;
        const float h = fmaf(p.dz, ocz, fmaf(p.dy, ocy, p.dx * ocx));
        if (!(h > 0.0f)) p.self = best | kSelfLeaves;
    }
    return false;
}

// Sample colour -> unsigned 32.32 fixed point.  Integer accumulation makes the pixel sum
// independent of which lane / warp / GPU traced which sample.
__device__ __forceinline__ unsigned long long to_fixed(float c) {
    c = (c >= 0.0f) ? c : 0.0f;  // also maps NaN to 0
    return __float2ull_rn(c * 4294967296.0f);
}

}  // namespace rtz
