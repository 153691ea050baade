// rtz_mirror.cpp — CPU ORACLE, part 2 (test infrastructure, NOT product code).
//
// An independent CPU restatement of the DEVICE arithmetic contract (DESIGN.md §4): the same
// reference functions as rtz_oracle.cpp (getRay, HittableList.hit, Sphere.hit, Material.scatter,
// Color.toRgb — reference src/camera.zig:148-215, src/hittable.zig:64-77, src/sphere.zig:26-54,
// src/material.zig:27-110, src/color.zig:63-80), but evaluated the way the B200 kernels
// evaluate them: FP32, explicit fmaf, unit ray directions, candidate test on the discriminant
// expanded around per-ray constants, roots from the direct form, exact c = 0 for the sphere the ray
// starts on, Philox4x32-10 keyed (seed; pixel, sample, bounce, 0), closed-form unit vectors and lens
// points (polynomial sine / cosine), 32.32 fixed-point pixel sums, f64 resolve.
//
// Because every operation is an IEEE-754 correctly rounded +,-,*,/,sqrt or fma, the GPU must
// reproduce these numbers BIT FOR BIT; tests/test_gpu_parity.py asserts exactly that on the
// fixed-point sums' images.  The chain of custody for stochastic scenes is therefore
//   GPU  ==(bit-exact)==  this mirror  ~~(statistical: RMSE / bias / segments-per-sample)~~
//   f64 reference restatement (rtz_oracle.cpp)  ==(byte-exact)==  test-files/chapter14.ppm.
//
// Build: with rtz_oracle.cpp, g++ -O2 -ffp-contract=off -mfma (std::fmaf -> one vfmadd; the
// compiler itself never contracts).
#include <cmath>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include "../include/rtz.h"
#include "philox_ref.h"

namespace {

struct F3 {
    float x, y, z;
};

struct MSphere {  // the device SoA, one element
    float cx, cy, cz, r2;      // geom
    float nq;                  // -(|c|^2 - r^2), evaluated in f64 on the FP32-rounded sphere
    float r, inv_r, param;     // aux (param = fuzz | ior)
    int type;
    float ar, ag, ab, inv_ior;  // albedo
};

struct MCamera {
    F3 p0, du, dv, c, uu, vv;
    float tmin, tmax;
    bool defocus;
    uint32_t W, H, spp, bounce_max, k0, k1;
};

struct Rng {
    uint32_t key[2], pixel, sample;
    void block(uint32_t bounce, uint32_t blk, uint32_t out[4]) const {
        const uint32_t ctr[4] = {pixel, sample, bounce, blk};
        philox4x32_10(ctr, key, out);
    }
};

inline float u01(uint32_t x) { return (float)(x >> 8) * 0x1p-24f; }

// (cos 2*pi*u, sin 2*pi*u), u = (x >> 8) * 2^-24: quarter turn from the top two bits, degree-4 minimax
// polynomials in the fraction of the quarter (the device's cos_sin_2pi, operation for operation)
inline void cosSin2Pi(uint32_t x, float& c, float& s) {
    const uint32_t q = x >> 30;
    const float f = (float)((x >> 8) & 0x3FFFFFu) * 0x1p-22f;
    const float z = f * f;
    float sp = std::fmaf(z, 0x1.3e7abap-13f, -0x1.3259fap-8f);
    sp = std::fmaf(z, sp, 0x1.46693cp-4f);
    sp = std::fmaf(z, sp, -0x1.4abbc6p-1f);
    sp = std::fmaf(z, sp, 0x1.921fb6p+0f);
    sp = sp * f;
    float cp = std::fmaf(z, 0x1.c29b9cp-11f, -0x1.550192p-6f);
    cp = std::fmaf(z, cp, 0x1.03bd86p-2f);
    cp = std::fmaf(z, cp, -0x1.3bd3aep+0f);
    cp = std::fmaf(z, cp, 1.0f);
    const float a = (q & 1u) ? sp : cp;
    const float b = (q & 1u) ? cp : sp;
    c = (q == 1u || q == 2u) ? -a : a;
    s = (q >= 2u) ? -b : b;
}

// uniform in the unit disk, closed form: radius sqrt(u1), angle 2*pi*u2
inline void sampleDisk(uint32_t x1, uint32_t x2, float& a, float& b) {
    const float rad = std::sqrt(u01(x1));
    float c, s;
    cosSin2Pi(x2, c, s);
    a = rad * c, b = rad * s;
}

// uniform on the unit sphere, closed form: z uniform in (-1, 1], angle 2*pi*u2
inline F3 randomUnitVec(uint32_t x1, uint32_t x2) {
    const float z = std::fmaf(-2.0f, u01(x1), 1.0f);
    const float rad = std::sqrt(std::fmaf(-z, z, 1.0f));
    float c, s;
    cosSin2Pi(x2, c, s);
    return {rad * c, rad * s, z};
}

struct Path {
    F3 o, d;
    float tr, tg, tb, len;
    int self;
    uint32_t bounce;
};

inline void setDirection(Path& p, float dx, float dy, float dz) {
    const float len2 = std::fmaf(dz, dz, std::fmaf(dy, dy, dx * dx));
    const float len = std::sqrt(len2);
    const float inv = 1.0f / len;
    p.d = {dx * inv, dy * inv, dz * inv};
    p.len = len;
}

inline void cameraRay(const MCamera& c, const Rng& g, uint32_t i, uint32_t j, Path& p) {
    uint32_t r[4];
    g.block(0, 0, r);
    const float sx = (float)i + (u01(r[0]) - 0.5f);
    const float sy = (float)j + (u01(r[1]) - 0.5f);
    const float psx = std::fmaf(c.dv.x, sy, std::fmaf(c.du.x, sx, c.p0.x));
    const float psy = std::fmaf(c.dv.y, sy, std::fmaf(c.du.y, sx, c.p0.y));
    const float psz = std::fmaf(c.dv.z, sy, std::fmaf(c.du.z, sx, c.p0.z));
    p.o = c.c;
    if (c.defocus) {
        float a, b;
        sampleDisk(r[2], r[3], a, b);
        p.o = {std::fmaf(c.vv.x, b, std::fmaf(c.uu.x, a, c.c.x)), std::fmaf(c.vv.y, b, std::fmaf(c.uu.y, a, c.c.y)),
               std::fmaf(c.vv.z, b, std::fmaf(c.uu.z, a, c.c.z))};
    }
    setDirection(p, psx - p.o.x, psy - p.o.y, psz - p.o.z);
    p.tr = p.tg = p.tb = 1.0f;
    p.self = -1;
    p.bounce = 0;
}

// The candidate gate's margin (the device's kGateSlack, DESIGN.md §4): the gate tests
// disc + 64 eps (|o|^2 + |c|^2) >= 0, the per-ray half folded into -|o|^2, the per-sphere half into nq.
constexpr float kGateSlack = 0x1p-18f;
inline float gate_nk2(const F3& o) { return -std::fmaf(o.z, o.z, std::fmaf(o.y, o.y, o.x * o.x)) * (1.0f - kGateSlack); }

inline MSphere mirror_sphere(const rtz_sphere& s) {
    MSphere m;
    const float r = (float)(s.radius < 0 ? 0.0 : s.radius);
    m.cx = (float)s.center[0], m.cy = (float)s.center[1], m.cz = (float)s.center[2], m.r2 = r * r;
    const double c2 = (double)m.cx * m.cx + (double)m.cy * m.cy + (double)m.cz * m.cz;
    m.nq = -(float)((c2 - (double)r * r) - (double)kGateSlack * c2);
    m.r = r, m.inv_r = 1.0f / r;
    m.param = s.mat_type == RTZ_MAT_METAL ? (float)s.fuzz : (float)s.refraction_index;
    m.type = s.mat_type;
    m.ar = (float)s.albedo[0], m.ag = (float)s.albedo[1], m.ab = (float)s.albedo[2];
    m.inv_ior = 1.0f / (float)s.refraction_index;
    return m;
}

// Test-only: false sends every sphere to the direct form (orc_mirror_set_gate).  A conservative gate only filters,
// so the mirror's results must not depend on it.
bool g_gate = true;

inline void sweep(const std::vector<MSphere>& sp, const Path& p, float tmin, float tmax, float& t_out, int& best_out) {
    const float tmin_d = tmin * p.len;  // Scene.interval in distance units
    float closest = tmax * p.len;
    int best = -1;
    const int n = (int)sp.size();
    // per-ray constants of the expanded discriminant
    const float k1 = -std::fmaf(p.d.z, p.o.z, std::fmaf(p.d.y, p.o.y, p.d.x * p.o.x));
    const float nk2 = gate_nk2(p.o);
    const float tx = 2.0f * p.o.x, ty = 2.0f * p.o.y, tz = 2.0f * p.o.z;
    const bool gate = g_gate;
    for (int i = 0; i < n; ++i) {
        const MSphere& s = sp[i];
        // candidate test: h = d.c - d.o ; w = (2 o.c - |o|^2) - (|c|^2 - r^2) - margin ; disc = h^2 + w
        const float he = std::fmaf(p.d.z, s.cz, std::fmaf(p.d.y, s.cy, std::fmaf(p.d.x, s.cx, k1)));
        const float w = std::fmaf(tz, s.cz, std::fmaf(ty, s.cy, std::fmaf(tx, s.cx, nk2))) + s.nq;
        const float de = std::fmaf(he, he, w);
        if (gate && std::signbit(de)) continue;
        // root from the direct form (reference src/sphere.zig:27-42, unit direction)
        const float ocx = s.cx - p.o.x, ocy = s.cy - p.o.y, ocz = s.cz - p.o.z;
        const float h = std::fmaf(p.d.z, ocz, std::fmaf(p.d.y, ocy, p.d.x * ocx));
        const float c = std::fmaf(ocz, ocz, std::fmaf(ocy, ocy, std::fmaf(ocx, ocx, -s.r2)));
        const float disc = std::fmaf(h, h, -c);
        if (!(disc >= 0.0f)) continue;
        // exact c = 0 on the sphere the ray starts on: roots h -/+ |h| (not sqrt(h * h), which exceeds |h| where h * h
        // underflows)
        const float sq = i == p.self ? std::fabs(h) : std::sqrt(disc);
        float t = h - sq;
        if (!(t > tmin_d && t < closest)) {
            t = h + sq;
            if (!(t > tmin_d && t < closest)) continue;
        }
        closest = t;
        best = i;
    }
    t_out = closest;
    best_out = best;
}

// returns true when the sample is finished; term 0 sky, 1 absorbed, 2 depth cap
inline bool shade(const MCamera& cam, const Rng& g, const std::vector<MSphere>& sp, Path& p, float t, int best,
                  float& sr, float& sg, float& sb, int& term) {
    if (best < 0) {
        const float a = 0.5f * (p.d.y + 1.0f);
        const float w = 1.0f - a;
        sr = p.tr * std::fmaf(a, 0.5f, w);
        sg = p.tg * std::fmaf(a, 0.7f, w);
        sb = p.tb * std::fmaf(a, 1.0f, w);
        term = 0;
        return true;
    }
    const MSphere& s = sp[best];
    const float px = std::fmaf(t, p.d.x, p.o.x), py = std::fmaf(t, p.d.y, p.o.y), pz = std::fmaf(t, p.d.z, p.o.z);
    float nx = (px - s.cx) * s.inv_r, ny = (py - s.cy) * s.inv_r, nz = (pz - s.cz) * s.inv_r;
    float dn = std::fmaf(p.d.z, nz, std::fmaf(p.d.y, ny, p.d.x * nx));
    const bool front = dn < 0.0f;
    if (!front) nx = -nx, ny = -ny, nz = -nz, dn = -dn;
    const uint32_t stream = p.bounce + 1u;
    uint32_t r0[4];
    g.block(stream, 0, r0);
    float ndx, ndy, ndz;
    if (s.type == RTZ_MAT_DIELECTRIC) {
        const float ri = front ? s.inv_ior : s.param;
        const float cosT = std::fmin(-dn, 1.0f);
        const float sinT = std::sqrt(std::fmaf(-cosT, cosT, 1.0f));
        const bool cannot = ri * sinT > 1.0f;
        float q = (1.0f - ri) / (1.0f + ri);
        q = q * q;
        const float x = 1.0f - cosT;
        const float x2 = x * x;
        const float refl = std::fmaf(1.0f - q, x * (x2 * x2), q);
        if (cannot || refl > u01(r0[0])) {
            const float kk = -2.0f * dn;
            ndx = std::fmaf(kk, nx, p.d.x), ndy = std::fmaf(kk, ny, p.d.y), ndz = std::fmaf(kk, nz, p.d.z);
        } else {
            const float ex = ri * std::fmaf(cosT, nx, p.d.x), ey = ri * std::fmaf(cosT, ny, p.d.y),
                        ez = ri * std::fmaf(cosT, nz, p.d.z);
            const float kk = -std::sqrt(std::fabs(1.0f - std::fmaf(ez, ez, std::fmaf(ey, ey, ex * ex))));
            ndx = std::fmaf(kk, nx, ex), ndy = std::fmaf(kk, ny, ey), ndz = std::fmaf(kk, nz, ez);
        }
    } else {
        const F3 u = randomUnitVec(r0[1], r0[2]);
        if (s.type == RTZ_MAT_LAMBERTIAN) {
            ndx = nx + u.x, ndy = ny + u.y, ndz = nz + u.z;
            if (ndx < 1e-8f && ndy < 1e-8f && ndz < 1e-8f) ndx = nx, ndy = ny, ndz = nz;
        } else {
            const float kk = -2.0f * dn;
            ndx = std::fmaf(s.param, u.x, std::fmaf(kk, nx, p.d.x));
            ndy = std::fmaf(s.param, u.y, std::fmaf(kk, ny, p.d.y));
            ndz = std::fmaf(s.param, u.z, std::fmaf(kk, nz, p.d.z));
            if (!(std::fmaf(ndz, nz, std::fmaf(ndy, ny, ndx * nx)) > 0.0f)) {
                sr = sg = sb = 0.0f;
                term = 1;
                return true;
            }
        }
        p.tr *= s.ar, p.tg *= s.ag, p.tb *= s.ab;
    }
    p.bounce += 1u;
    if (p.bounce >= cam.bounce_max) {
        sr = sg = sb = 0.0f;
        term = 2;
        return true;
    }
    p.o = {px, py, pz};
    setDirection(p, ndx, ndy, ndz);
    p.self = best;
    return false;
}

inline uint64_t toFixed(float c) {
    c = (c >= 0.0f) ? c : 0.0f;
    // samples lie in [0, 1] (rtz_scene_upload refuses albedos outside it): c * 2^32 is exact and at most 2^32, and
    // llrint rounds it half to even as __float2ull_rn does
    return (uint64_t)std::llrint((double)(c * 4294967296.0f));
}

inline uint8_t toByte(double lin) {
    double g = lin > 0.0 ? std::sqrt(lin) : 0.0;
    g = g < 0.0 ? 0.0 : (g > 0.999 ? 0.999 : g);
    return (uint8_t)(256.0 * g);
}

inline F3 f3(const double* p) { return {(float)p[0], (float)p[1], (float)p[2]}; }

}  // namespace

extern "C" {

// Render this rank's tiles (shard == NULL: the whole frame, row-major) exactly as the device
// does.  Output layout = rtz_render_resident's compact tile layout; padded pixels are 0.
int orc_render_mirror(const rtz_camera* cam, const rtz_sphere* sp, uint64_t n, uint64_t seed, int threads,
                      const rtz_shard* shard, uint8_t* rgb, double* linear, rtz_stats* st) {
    if (!cam || !sp || cam->mode != RTZ_MODE_PATH) return RTZ_ERR_BAD_ARG;
    if (threads < 1) threads = 1;
    std::vector<MSphere> ms(n);
    for (uint64_t i = 0; i < n; ++i) ms[i] = mirror_sphere(sp[i]);
    MCamera c;
    c.p0 = f3(cam->pixel0), c.du = f3(cam->du), c.dv = f3(cam->dv), c.c = f3(cam->center);
    c.uu = f3(cam->defocus_disk_u), c.vv = f3(cam->defocus_disk_v);
    c.tmin = (float)cam->t_min;
    c.tmax = (float)cam->t_max;
    c.defocus = cam->defocus_angle > 0;
    c.W = (uint32_t)cam->width, c.H = (uint32_t)cam->height;
    c.spp = (uint32_t)cam->samples_per_pixel, c.bounce_max = (uint32_t)cam->bounce_max;
    c.k0 = (uint32_t)seed, c.k1 = (uint32_t)(seed >> 32);

    rtz_shard sh{0, 1, c.W, 1};
    if (shard) sh = *shard;
    const uint32_t tiles_x = (c.W + sh.tile_w - 1) / sh.tile_w, tiles_y = (c.H + sh.tile_h - 1) / sh.tile_h;
    const uint64_t tiles = (uint64_t)tiles_x * tiles_y;
    const uint32_t n_local_tiles = (uint32_t)((tiles + sh.world - 1) / sh.world);
    const uint32_t tile_pixels = sh.tile_w * sh.tile_h;
    const uint64_t n_local = (uint64_t)n_local_tiles * tile_pixels;

    struct K {
        uint64_t samples = 0, segments = 0, capped = 0, absorbed = 0;
    };
    std::vector<K> ks(threads);
    auto work = [&](int tid) {
        K& k = ks[tid];
        for (uint64_t lp = tid; lp < n_local; lp += threads) {
            const uint32_t lt = (uint32_t)(lp / tile_pixels), within = (uint32_t)(lp - (uint64_t)lt * tile_pixels);
            const uint64_t gt = (uint64_t)lt * sh.world + sh.rank;
            const uint32_t ty = (uint32_t)(gt / tiles_x), tx = (uint32_t)(gt - (uint64_t)ty * tiles_x);
            const uint32_t x = tx * sh.tile_w + within % sh.tile_w, y = ty * sh.tile_h + within / sh.tile_w;
            uint64_t acc[3] = {0, 0, 0};
            if (x < c.W && y < c.H && ty < tiles_y) {
                for (uint32_t s = 0; s < c.spp; ++s) {
                    if (c.bounce_max == 0) {  // rayColor's loop never runs: black, no hit test (camera.zig:153,181)
                        ++k.samples;
                        continue;
                    }
                    Rng g{{c.k0, c.k1}, y * c.W + x, s};
                    Path p;
                    cameraRay(c, g, x, y, p);
                    for (;;) {
                        float t;
                        int best;
                        sweep(ms, p, c.tmin, c.tmax, t, best);
                        ++k.segments;
                        float sr, sg, sb;
                        int term;
                        if (shade(c, g, ms, p, t, best, sr, sg, sb, term)) {
                            acc[0] += toFixed(sr), acc[1] += toFixed(sg), acc[2] += toFixed(sb);
                            ++k.samples;
                            k.capped += term == 2, k.absorbed += term == 1;
                            break;
                        }
                    }
                }
            }
            for (int ch = 0; ch < 3; ++ch) {
                const double lin = ((double)acc[ch] * 0x1p-32) * cam->pixel_samples_scale;
                if (rgb) rgb[3 * lp + ch] = toByte(lin);
                if (linear) linear[3 * lp + ch] = lin;
            }
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < threads; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& t : th) t.join();
    if (st) {
        std::memset(st, 0, sizeof(*st));
        for (auto& k : ks)
            st->samples += k.samples, st->segments += k.segments, st->depth_capped += k.capped, st->absorbed += k.absorbed;
        st->sphere_tests = st->segments * n;
        st->seed_used = seed;
    }
    return RTZ_OK;
}

// Camera.getRay as the device evaluates it (mirror of rtz_probe_camera_ray): n rays of pixel (i, j)
void orc_mirror_camera_ray(const rtz_camera* cam, uint64_t seed, uint32_t i, uint32_t j, uint32_t sample0, uint32_t n,
                           float* o, float* d, float* len) {
    MCamera c;
    c.p0 = f3(cam->pixel0), c.du = f3(cam->du), c.dv = f3(cam->dv), c.c = f3(cam->center);
    c.uu = f3(cam->defocus_disk_u), c.vv = f3(cam->defocus_disk_v);
    c.tmin = (float)cam->t_min, c.tmax = (float)cam->t_max;
    c.defocus = cam->defocus_angle > 0;
    c.W = (uint32_t)cam->width, c.H = (uint32_t)cam->height;
    c.spp = (uint32_t)cam->samples_per_pixel, c.bounce_max = (uint32_t)cam->bounce_max;
    c.k0 = (uint32_t)seed, c.k1 = (uint32_t)(seed >> 32);
    for (uint32_t k = 0; k < n; ++k) {
        Rng g{{c.k0, c.k1}, j * c.W + i, sample0 + k};
        Path p;
        cameraRay(c, g, i, j, p);
        o[3 * k] = p.o.x, o[3 * k + 1] = p.o.y, o[3 * k + 2] = p.o.z;
        d[3 * k] = p.d.x, d[3 * k + 1] = p.d.y, d[3 * k + 2] = p.d.z;
        if (len) len[k] = p.len;
    }
}

// Test-only: on = 0 sends every sphere to the direct form in the mirror's renders and probes.
void orc_mirror_set_gate(int on) { g_gate = on != 0; }

// twin of rtz_probe_hits: the mirror's sweep for m rays
void orc_mirror_hits(const rtz_sphere* sp, uint64_t n, const rtz_probe_ray* rays, uint64_t m, double tmin, double tmax,
                     rtz_ray_hit* out) {
    std::vector<MSphere> ms(n);
    for (uint64_t i = 0; i < n; ++i) ms[i] = mirror_sphere(sp[i]);
    for (uint64_t k = 0; k < m; ++k) {
        const rtz_probe_ray& r = rays[k];
        Path p;
        p.o = {r.orig[0], r.orig[1], r.orig[2]}, p.self = r.self, p.bounce = 0, p.tr = p.tg = p.tb = 1.0f;
        setDirection(p, r.dir[0], r.dir[1], r.dir[2]);
        float t;
        int best;
        sweep(ms, p, (float)tmin, (float)tmax, t, best);
        rtz_ray_hit h = {best, 0, t, p.len, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
        if (best >= 0) {
            const MSphere& s = ms[best];
            const float px = std::fmaf(t, p.d.x, p.o.x), py = std::fmaf(t, p.d.y, p.o.y), pz = std::fmaf(t, p.d.z, p.o.z);
            float nx = (px - s.cx) * s.inv_r, ny = (py - s.cy) * s.inv_r, nz = (pz - s.cz) * s.inv_r;
            const bool front = std::fmaf(p.d.z, nz, std::fmaf(p.d.y, ny, p.d.x * nx)) < 0.0f;
            if (!front) nx = -nx, ny = -ny, nz = -nz;
            h.front = front, h.point[0] = px, h.point[1] = py, h.point[2] = pz;
            h.normal[0] = nx, h.normal[1] = ny, h.normal[2] = nz;
        }
        out[k] = h;
    }
}

// twin of rtz_probe_scatters: Sphere.hit on the record's sphere, then the mirror's shade
void orc_mirror_scatters(const rtz_sphere* sp, uint64_t n, const rtz_probe_bounce* recs, uint64_t m, uint64_t seed,
                         rtz_ray_scatter* out) {
    std::vector<MSphere> ms(n);
    for (uint64_t i = 0; i < n; ++i) ms[i] = mirror_sphere(sp[i]);
    MCamera c{};
    c.tmin = 1e-3f, c.tmax = INFINITY, c.bounce_max = 0xFFFFFFFFu;
    c.k0 = (uint32_t)seed, c.k1 = (uint32_t)(seed >> 32);
    for (uint64_t k = 0; k < m; ++k) {
        const rtz_probe_bounce& r = recs[k];
        Path p;
        p.o = {r.orig[0], r.orig[1], r.orig[2]}, p.self = -1, p.bounce = r.bounce, p.tr = p.tg = p.tb = 1.0f;
        setDirection(p, r.dir[0], r.dir[1], r.dir[2]);
        const std::vector<MSphere> one{ms[r.sphere]};
        float t;
        int best;
        sweep(one, p, c.tmin, c.tmax, t, best);
        rtz_ray_scatter s = {-2, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, 0.f, {0.f, 0.f, 0.f}};
        if (best >= 0) {
            const Rng g{{c.k0, c.k1}, r.pixel, r.sample};
            float sr, sg, sb;
            int term = -1;
            if (shade(c, g, ms, p, t, r.sphere, sr, sg, sb, term)) {
                s.term = term;
            } else {
                s.term = -1;
                s.orig[0] = p.o.x, s.orig[1] = p.o.y, s.orig[2] = p.o.z;
                s.dir[0] = p.d.x, s.dir[1] = p.d.y, s.dir[2] = p.d.z, s.len = p.len;
                s.attenuation[0] = p.tr, s.attenuation[1] = p.tg, s.attenuation[2] = p.tb;
            }
        }
        out[k] = s;
    }
}

// the mirror's (cos 2 pi u, sin 2 pi u) for the 2^24 uniforms u = i * 2^-24, i = 0 .. 2^24 - 1
void orc_mirror_cos_sin_all(float* c, float* s) {
    for (uint32_t i = 0; i < (1u << 24); ++i) cosSin2Pi(i << 8, c[i], s[i]);
}

// one-ray mirrors of the device probes
void orc_mirror_uniform(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, uint64_t n, float* out) {
    Rng g{{(uint32_t)seed, (uint32_t)(seed >> 32)}, pixel, sample};
    for (uint64_t b = 0; 4 * b < n; ++b) {
        uint32_t r[4];
        g.block(bounce, (uint32_t)b, r);
        for (int q = 0; q < 4 && 4 * b + q < n; ++q) out[4 * b + q] = u01(r[q]);
    }
}

}  // extern "C"
