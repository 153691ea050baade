// block_cull_estimate.cpp — CPU estimate of what warp-uniform block culling would save in the constant-bank sweep.
//
// Replays the C3 frame's segments (the f32 mirror's arithmetic, oracle/rtz_mirror.cpp, included unchanged) through
// the lockstep kernel's warp schedule (trace_body: 64 slots per warp, chunks of 256 samples of one pixel, free
// A-slots refilled before B-slots in lane order, one sweep per iteration, blocks of 32 spheres in order, each
// path's running closest hit updated after every block) and reports the fraction of sphere tests a warp still
// executes when it skips every block whose padded bound none of its live paths can reach over (0, closest].
// Three block orders (the reference's; the spatial regrouping the culled kernel sweeps, sweep_order in
// csrc/rtz_api.cu; the same blocks swept near to far from the camera) times two bounds (axis-aligned boxes,
// bounding spheres).  With boxes on the regrouped order it also reports what each path would execute if it swept
// only the blocks its own bound admits, how many of the warp's paths reach each swept culled block, and the cost
// of sweeping a block sphere-parallel over its k reaching paths (min(64, a k + 2) path-units against the packed
// sweep's 64, for a = 1.5 / 2 / 3: sweep2's split branch).
//
// Build and run (a few seconds per 100 pixels on one core):
//   g++ -O2 -std=c++17 -ffp-contract=off -mfma -pthread -o /tmp/bce tools/block_cull_estimate.cpp oracle/rtz_oracle.cpp
//   /tmp/bce [pixels=1000] [samples=256]
#include "../oracle/rtz_mirror.cpp"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <random>

extern "C" {
void* orc_prng_new(uint64_t seed);
void orc_prng_free(void* p);
uint64_t orc_generate_world(void* prng, rtz_sphere* out, uint64_t cap);
int orc_camera_build(uint64_t width, double aspect, const double lookFrom[3], const double lookAt[3],
                     const double vUp[3], double vfov, double viewport_focus_dist, double focus_dist,
                     double defocus_angle, uint64_t spp, uint64_t bounce_max, rtz_camera* out);
}

namespace {

struct Seg {
    Path p;
    float t;   // the mirror's closest hit (distance units)
    int best;
};

// Sphere.hit of one sphere with the mirror's arithmetic and closest = +inf: the root the ascending loop would
// accept, or +inf.  With a finite running closest the loop accepts that same root iff it lies below closest.
float accepted_root(const MSphere& s, int i, const Path& p, float tmin_d) {
    const float k1 = -std::fmaf(p.d.z, p.o.z, std::fmaf(p.d.y, p.o.y, p.d.x * p.o.x));
    const float nk2 = gate_nk2(p.o);
    const float he = std::fmaf(p.d.z, s.cz, std::fmaf(p.d.y, s.cy, std::fmaf(p.d.x, s.cx, k1)));
    const float w = std::fmaf(2.0f * p.o.z, s.cz, std::fmaf(2.0f * p.o.y, s.cy, std::fmaf(2.0f * p.o.x, s.cx, nk2))) + s.nq;
    if (std::signbit(std::fmaf(he, he, w))) return INFINITY;
    const float ocx = s.cx - p.o.x, ocy = s.cy - p.o.y, ocz = s.cz - p.o.z;
    const float h = std::fmaf(p.d.z, ocz, std::fmaf(p.d.y, ocy, p.d.x * ocx));
    const float c = std::fmaf(ocz, ocz, std::fmaf(ocy, ocy, std::fmaf(ocx, ocx, -s.r2)));
    const float disc = std::fmaf(h, h, -c);
    if (!(disc >= 0.0f)) return INFINITY;
    const float sq = i == p.self ? std::fabs(h) : std::sqrt(disc);
    float t = h - sq;
    if (t > tmin_d) return t;
    t = h + sq;
    return t > tmin_d ? t : INFINITY;
}

struct Bound {
    float lo[3], hi[3];   // box
    float c[3], r;        // sphere
    bool all;             // always swept (holds a sphere too large to bound usefully)
};

bool box_needed(const Bound& b, const Path& p, float closest) {
    const float o[3] = {p.o.x, p.o.y, p.o.z}, d[3] = {p.d.x, p.d.y, p.d.z};
    float tn = 0.0f, tf = closest;
    for (int a = 0; a < 3; ++a) {
        const float inv = 1.0f / d[a];
        const float t0 = (b.lo[a] - o[a]) * inv, t1 = (b.hi[a] - o[a]) * inv;
        tn = std::fmax(tn, std::fmin(t0, t1));
        tf = std::fmin(tf, std::fmax(t0, t1));
    }
    return tn <= tf;
}

bool sphere_needed(const Bound& b, const Path& p, float closest) {
    const float ox = b.c[0] - p.o.x, oy = b.c[1] - p.o.y, oz = b.c[2] - p.o.z;
    const float h = p.d.x * ox + p.d.y * oy + p.d.z * oz;
    const float c = ox * ox + oy * oy + oz * oz - b.r * b.r;
    const float disc = h * h - c;
    if (disc < 0.0f) return false;
    const float sq = std::sqrt(disc);
    return h + sq >= 0.0f && h - sq <= closest;
}

std::vector<Bound> make_bounds(const std::vector<MSphere>& ms, const std::vector<int>& order, int n_pad) {
    std::vector<Bound> out;
    for (int base = 0; base < n_pad; base += 32) {
        Bound b{{INFINITY, INFINITY, INFINITY}, {-INFINITY, -INFINITY, -INFINITY}, {0, 0, 0}, 0, false};
        for (int q = base; q < std::min(base + 32, (int)order.size()); ++q) {
            const MSphere& s = ms[order[q]];
            if (s.r > 100.0f) b.all = true;
            const float c[3] = {s.cx, s.cy, s.cz};
            const float pad = 1e-4f * (1.0f + s.r + std::fabs(s.cx) + std::fabs(s.cy) + std::fabs(s.cz));
            for (int a = 0; a < 3; ++a)
                b.lo[a] = std::min(b.lo[a], c[a] - s.r - pad), b.hi[a] = std::max(b.hi[a], c[a] + s.r + pad);
        }
        for (int a = 0; a < 3; ++a) b.c[a] = 0.5f * (b.lo[a] + b.hi[a]);
        for (int q = base; q < std::min(base + 32, (int)order.size()); ++q) {
            const MSphere& s = ms[order[q]];
            const float dx = s.cx - b.c[0], dy = s.cy - b.c[1], dz = s.cz - b.c[2];
            const float pad = 1e-4f * (1.0f + s.r + std::fabs(s.cx) + std::fabs(s.cy) + std::fabs(s.cz));
            b.r = std::max(b.r, std::sqrt(dx * dx + dy * dy + dz * dz) + s.r + pad);
        }
        out.push_back(b);
    }
    return out;
}

// median splits along the longest axis of the centres, cut at multiples of 32 (offset by the ground in slot 0),
// final blocks sorted by index: the product's regroup() in csrc/rtz_api.cu
void kd_order(const std::vector<MSphere>& ms, std::vector<int>& idx, int first, int cnt, int slot0) {
    const int end_slot = slot0 + cnt;
    const int blocks = (end_slot + 31) / 32 - slot0 / 32;
    if (blocks <= 1) {
        std::sort(idx.begin() + first, idx.begin() + first + cnt);
        return;
    }
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int q = first; q < first + cnt; ++q) {
        const MSphere& s = ms[idx[q]];
        const float c[3] = {s.cx, s.cy, s.cz};
        for (int a = 0; a < 3; ++a) lo[a] = std::min(lo[a], c[a]), hi[a] = std::max(hi[a], c[a]);
    }
    int axis = 0;
    for (int a = 1; a < 3; ++a)
        if (hi[a] - lo[a] > hi[axis] - lo[axis]) axis = a;
    const int cut_slot = (slot0 / 32 + blocks / 2) * 32;
    const int left = cut_slot - slot0;
    auto key = [&](int i) { return axis == 0 ? ms[i].cx : axis == 1 ? ms[i].cy : ms[i].cz; };
    std::nth_element(idx.begin() + first, idx.begin() + first + left, idx.begin() + first + cnt,
                     [&](int x, int y) { return key(x) < key(y) || (key(x) == key(y) && x < y); });
    kd_order(ms, idx, first, left, slot0);
    kd_order(ms, idx, first + left, cnt - left, cut_slot);
}

struct Result {
    double executed = 0, total = 0, bound_tests = 0, iters = 0;
    double per_path = 0;             // tests if each live path swept only block 0 and the blocks its own bound admits
    double split[3] = {0, 0, 0};     // tests-equivalent of the split sweep for kSplitCost[j] (see main)
    double hist[65] = {};            // swept culled blocks by the number of paths of the warp that reach them
    double always = 0;               // tests of the blocks swept without a bound test (block 0)
};
// cost of a sphere-parallel pass per reaching path, in units of one path of the packed sweep
constexpr double kSplitCost[3] = {1.5, 2.0, 3.0};

// one warp runs all chunks in sequence (each chunk = the samples of one pixel)
// `seq`: the order in which the blocks are swept (block 0 first)
Result replay(const std::vector<std::vector<std::vector<Seg>>>& chunks, const std::vector<MSphere>& ms,
              const std::vector<int>& order, int n_pad, const std::vector<Bound>& bounds, const std::vector<int>& seq,
              int kind, float tmin) {
    const int nb = (int)bounds.size();
    struct SlotState {
        int chunk = -1, sample = 0, seg = 0;
        bool alive = false;
    } slot[64];
    Result R;
    size_t ci = 0, si = 0;  // next sample to hand out
    std::vector<float> root(nb);
    for (;;) {
        for (int s = 0; s < 64; ++s) {  // A-slots (0..31) before B-slots (32..63), lane order
            if (slot[s].alive) continue;
            while (ci < chunks.size() && si >= chunks[ci].size()) ++ci, si = 0;
            if (ci >= chunks.size()) break;
            slot[s] = {(int)ci, (int)si++, 0, true};
        }
        int live = 0;
        for (auto& s : slot) live += s.alive;
        if (!live) break;
        R.iters += 1;
        float closest[64];
        std::vector<std::vector<float>> rb(64);
        for (int s = 0; s < 64; ++s) {
            closest[s] = INFINITY;
            if (!slot[s].alive) continue;
            const Seg& g = chunks[slot[s].chunk][slot[s].sample][slot[s].seg];
            rb[s].assign(nb, INFINITY);
            const float tmin_d = tmin * g.p.len;
            for (int q = 0; q < (int)order.size(); ++q) {
                const float t = accepted_root(ms[order[q]], order[q], g.p, tmin_d);
                if (t < rb[s][q / 32]) rb[s][q / 32] = t;
            }
        }
        for (int b : seq) {
            const int cnt = std::min(32, n_pad - 32 * b);
            R.total += cnt;
            bool need = bounds[b].all;
            int reach = 0;  // paths whose own bound admits the block (every live path for block 0)
            if (!need) {
                R.bound_tests += 1;
                for (int s = 0; s < 64; ++s) {
                    if (!slot[s].alive) continue;
                    const Path& p = chunks[slot[s].chunk][slot[s].sample][slot[s].seg].p;
                    reach += kind == 0 ? box_needed(bounds[b], p, closest[s]) : sphere_needed(bounds[b], p, closest[s]);
                }
                need = reach > 0;
                if (need) R.hist[reach] += 1;
                // split sweep: a sphere-parallel pass costs a * k + 2 path-units (k broadcast rays, the lane's sphere
                // loads and the mask conversion), the packed sweep 64; the kernel takes the cheaper of the two
                for (int j = 0; j < 3; ++j)
                    if (need) R.split[j] += cnt * std::min(64.0, kSplitCost[j] * reach + 2.0) / 64.0;
            } else {
                reach = live;
                R.always += cnt;
                for (int j = 0; j < 3; ++j) R.split[j] += cnt;
            }
            R.per_path += cnt * reach / 64.0;
            for (int s = 0; s < 64; ++s) {
                if (!slot[s].alive) continue;
                if (!need && rb[s][b] < closest[s]) {
                    std::fprintf(stderr, "NOT CONSERVATIVE: block %d skipped, root %.9g < closest %.9g\n", b, rb[s][b], closest[s]);
                    std::exit(1);
                }
                if (need) closest[s] = std::min(closest[s], rb[s][b]);
            }
            if (need) R.executed += cnt;
        }
        for (int s = 0; s < 64; ++s) {
            if (!slot[s].alive) continue;
            const auto& smp = chunks[slot[s].chunk][slot[s].sample];
            const Seg& g = smp[slot[s].seg];
            if (closest[s] != g.t && !(std::isinf(closest[s]) && std::isinf(g.t))) {
                std::fprintf(stderr, "replay disagrees with the mirror: %.9g vs %.9g\n", closest[s], g.t);
                std::exit(1);
            }
            if (++slot[s].seg >= (int)smp.size()) slot[s].alive = false;
        }
    }
    return R;
}

}  // namespace

int main(int argc, char** argv) {
    const int n_pixels = argc > 1 ? std::atoi(argv[1]) : 1000;
    const int n_samples = argc > 2 ? std::atoi(argv[2]) : 256;
    // C3: final scene (Xoshiro seed 0xdeadbeef), camera of src/main.zig, 1200 px wide, depth 50, Philox seed 0xdeadbeef
    void* prng = orc_prng_new(0xdeadbeefull);
    std::vector<rtz_sphere> sp(600);
    sp.resize(orc_generate_world(prng, sp.data(), sp.size()));
    orc_prng_free(prng);
    rtz_camera cam;
    const double from[3] = {13, 2, 3}, at[3] = {0, 0, 0}, up[3] = {0, 1, 0};
    orc_camera_build(1200, 16.0 / 9.0, from, at, up, 20, 10.0, 10.0, 0.6, 500, 50, &cam);
    const int n = (int)sp.size(), n_pad = (n + 7) & ~7;

    std::vector<MSphere> ms(n);
    for (int i = 0; i < n; ++i) ms[i] = mirror_sphere(sp[i]);
    MCamera c;
    c.p0 = f3(cam.pixel0), c.du = f3(cam.du), c.dv = f3(cam.dv), c.c = f3(cam.center);
    c.uu = f3(cam.defocus_disk_u), c.vv = f3(cam.defocus_disk_v);
    c.tmin = (float)cam.t_min, c.tmax = (float)cam.t_max;
    c.defocus = cam.defocus_angle > 0;
    c.W = (uint32_t)cam.width, c.H = (uint32_t)cam.height;
    c.spp = (uint32_t)cam.samples_per_pixel, c.bounce_max = (uint32_t)cam.bounce_max;
    const uint64_t seed = 0xDEADBEEFull;
    c.k0 = (uint32_t)seed, c.k1 = (uint32_t)(seed >> 32);

    // record every segment of n_samples samples of n_pixels random pixels
    std::mt19937 rng(12345);
    std::vector<std::vector<std::vector<Seg>>> chunks(n_pixels);
    double segments = 0;
    for (int k = 0; k < n_pixels; ++k) {
        const uint32_t x = rng() % c.W, y = rng() % c.H;
        chunks[k].resize(n_samples);
        for (int s = 0; s < n_samples; ++s) {
            Rng g{{c.k0, c.k1}, y * c.W + x, (uint32_t)s};
            Path p;
            cameraRay(c, g, x, y, p);
            for (;;) {
                float t;
                int best;
                sweep(ms, p, c.tmin, c.tmax, t, best);
                chunks[k][s].push_back({p, t, best});
                segments += 1;
                float sr, sg, sb;
                int term;
                if (shade(c, g, ms, p, t, best, sr, sg, sb, term)) break;
            }
        }
    }
    std::printf("C3 scene: %d spheres (%d padded, %d blocks of 32); %d pixels x %d samples, %.0f segments (%.4f per sample)\n",
                n, n_pad, (n_pad + 31) / 32, n_pixels, n_samples, segments, segments / ((double)n_pixels * n_samples));

    std::vector<int> ref(n), kd(n);
    for (int i = 0; i < n; ++i) ref[i] = kd[i] = i;
    kd_order(ms, kd, 1, n - 1, 1);  // the ground stays in slot 0
    const char* order_name[3] = {"reference order", "spatial regrouping", "regrouped, near first"};
    const char* bound_name[2] = {"boxes", "spheres"};
    std::printf("%-22s %-8s %10s %12s\n", "block order", "bound", "executed", "bound tests");
    for (int o = 0; o < 3; ++o) {
        const std::vector<int>& order = o == 0 ? ref : kd;
        const auto bounds = make_bounds(ms, order, n_pad);
        std::vector<int> seq(bounds.size());
        for (int b = 0; b < (int)seq.size(); ++b) seq[b] = b;
        if (o == 2) {  // blocks 1.. by the distance from the camera to the centre of their box
            auto dist = [&](int b) {
                const Bound& B = bounds[b];
                double d2 = 0.0;
                for (int a = 0; a < 3; ++a) d2 += std::pow(0.5 * (B.lo[a] + B.hi[a]) - from[a], 2);
                return d2;
            };
            std::stable_sort(seq.begin() + 1, seq.end(), [&](int x, int y) { return dist(x) < dist(y); });
        }
        for (int kind = 0; kind < 2; ++kind) {
            const Result R = replay(chunks, ms, order, n_pad, bounds, seq, kind, c.tmin);
            const double frac = R.executed / R.total;
            // bound tests per path and iteration, in units of the sweep's n_pad tests per path and iteration
            const double bt = R.bound_tests / R.iters / n_pad;
            std::printf("%-22s %-8s %9.1f%% %12.3f", order_name[o], bound_name[kind], 100.0 * frac, R.bound_tests / R.iters);
            // predicted step time relative to today: the sweep is 87.7 % of the kernel's warp-instructions
            for (double cb : {1.0, 1.5, 3.0}) {
                const double rel = (1.0 - 0.877) + 0.877 * (frac + cb * bt);
                std::printf("   c_b=%.1f: x%.3f (%.1f%% less time)", cb, 1.0 / rel, 100.0 * (1.0 - rel));
            }
            std::printf("\n");
            if (kind != 0 || o == 0) continue;
            // boxes on the regrouped order: what sweeping each path's own blocks would execute, how many paths reach
            // the culled blocks that are swept, and the split sweep's cost model
            std::printf("%-31s %9.1f%%\n", "  per path (own box_reach)", 100.0 * R.per_path / R.total);
            double swept = 0;
            for (int k = 1; k <= 64; ++k) swept += R.hist[k];
            std::printf("  paths reaching a swept culled block, cumulative share:");
            double acc = 0;
            for (int k = 1, c = 0; k <= 64; ++k) {
                acc += R.hist[k];
                const int marks[6] = {4, 8, 16, 24, 32, 48};
                if (c < 6 && k == marks[c]) std::printf("  <=%d: %.0f%%", k, 100.0 * acc / swept), ++c;
            }
            std::printf("\n");
            for (int j = 0; j < 3; ++j)
                std::printf("  split sweep, a = %.1f: %9.1f%% of brute force, culled blocks at %.2f of the packed sweep\n",
                            kSplitCost[j], 100.0 * R.split[j] / R.total,
                            (R.split[j] - R.always) / (R.executed - R.always));
        }
    }
    return 0;
}
