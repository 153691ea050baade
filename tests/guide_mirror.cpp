// guide_mirror.cpp — CPU restatement of rtz_render_guides (test infrastructure, not product code).
//
// It is the f32 device mirror's translation unit plus the guide loop, so the guides are built from the mirror's own
// cameraRay, sweep and sphere table: the very rays and first hits of the mirror's render.  tests/test_guides.py
// compiles it next to the oracle (same flags) and compares the device guides with it bit for bit.
#include <algorithm>

#include "../oracle/rtz_mirror.cpp"

extern "C" {

// Guides of the whole frame (row-major, 3 floats per pixel each; either output may be NULL), samples 0 .. g-1 of every
// pixel: per sample the albedo / normal of the camera ray's closest hit (sky colour / 0 on a miss), added per pixel in
// ascending sample order from +0 in f32, then divided by (float)g once.
int orc_mirror_guides(const rtz_camera* cam, const rtz_sphere* sp, uint64_t n, uint64_t seed, uint64_t g, float* albedo,
                      float* normal) {
    if (!cam || (!sp && n) || g == 0) return RTZ_ERR_BAD_ARG;
    std::vector<MSphere> ms(n);
    for (uint64_t i = 0; i < n; ++i) ms[i] = mirror_sphere(sp[i]);
    MCamera c;
    c.p0 = f3(cam->pixel0), c.du = f3(cam->du), c.dv = f3(cam->dv), c.c = f3(cam->center);
    c.uu = f3(cam->defocus_disk_u), c.vv = f3(cam->defocus_disk_v);
    c.tmin = (float)cam->t_min, c.tmax = (float)cam->t_max;
    c.defocus = cam->defocus_angle > 0;
    c.W = (uint32_t)cam->width, c.H = (uint32_t)cam->height;
    c.spp = (uint32_t)cam->samples_per_pixel, c.bounce_max = (uint32_t)cam->bounce_max;
    c.k0 = (uint32_t)seed, c.k1 = (uint32_t)(seed >> 32);
    const uint64_t n_pix = (uint64_t)c.W * c.H;
    auto work = [&](uint64_t first, uint64_t step) {
        for (uint64_t px = first; px < n_pix; px += step) {
            const uint32_t y = (uint32_t)(px / c.W), x = (uint32_t)(px - (uint64_t)y * c.W);
            float acc[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
            for (uint64_t s = 0; s < g; ++s) {
                Rng rng{{c.k0, c.k1}, (uint32_t)px, (uint32_t)s};
                Path p;
                cameraRay(c, rng, x, y, p);
                float t;
                int best;
                sweep(ms, p, c.tmin, c.tmax, t, best);
                float v[6];
                if (best < 0) {  // shade's sky at throughput 1
                    const float a = 0.5f * (p.d.y + 1.0f);
                    const float w = 1.0f - a;
                    v[0] = std::fmaf(a, 0.5f, w), v[1] = std::fmaf(a, 0.7f, w), v[2] = std::fmaf(a, 1.0f, w);
                    v[3] = v[4] = v[5] = 0.0f;
                } else {  // HitRecord normal, against the ray
                    const MSphere& m = ms[best];
                    const float hx = std::fmaf(t, p.d.x, p.o.x), hy = std::fmaf(t, p.d.y, p.o.y), hz = std::fmaf(t, p.d.z, p.o.z);
                    float nx = (hx - m.cx) * m.inv_r, ny = (hy - m.cy) * m.inv_r, nz = (hz - m.cz) * m.inv_r;
                    if (!(std::fmaf(p.d.z, nz, std::fmaf(p.d.y, ny, p.d.x * nx)) < 0.0f)) nx = -nx, ny = -ny, nz = -nz;
                    const bool glass = m.type == RTZ_MAT_DIELECTRIC;
                    v[0] = glass ? 1.0f : m.ar, v[1] = glass ? 1.0f : m.ag, v[2] = glass ? 1.0f : m.ab;
                    v[3] = nx, v[4] = ny, v[5] = nz;
                }
                for (int k = 0; k < 6; ++k) acc[k] += v[k];
            }
            for (int k = 0; k < 3; ++k) {
                if (albedo) albedo[3 * px + k] = acc[k] / (float)g;
                if (normal) normal[3 * px + k] = acc[3 + k] / (float)g;
            }
        }
    };
    const unsigned threads = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<std::thread> th;
    for (unsigned t = 1; t < threads; ++t) th.emplace_back(work, t, threads);
    work(0, threads);
    for (auto& t : th) t.join();
    return RTZ_OK;
}

}  // extern "C"
