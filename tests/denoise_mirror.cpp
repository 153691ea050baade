// denoise_mirror.cpp — CPU restatement of rtz_denoise (test infrastructure, not product code).
//
// It is the guide mirror's translation unit (and so the f32 render mirror's) plus the à-trous filter of
// csrc/rtz_denoise.cuh, written out again from its contract: the same f32 operations in the same order, explicit
// std::fmaf and std::fmax only.  tests/test_denoise.py compiles it with the oracle's flags (-ffp-contract=off -mfma)
// and compares the device with it bit for bit; the same library renders the noisy inputs, the guides and the
// high-spp references of the CPU quality test.
#include "guide_mirror.cpp"

namespace {

inline float dn_modulus(float a) { return std::fmax(a, 0x1p-8f); }

inline float dn_edge(float x) {  // max(0, 1 - x/64)^64
    float t = std::fmax(std::fmaf(x, -0x1p-6f, 1.0f), 0.0f);
    for (int i = 0; i < 6; ++i) t = t * t;
    return t;
}

inline float dn_dist2(const float* q, const float* p) {
    const float d0 = q[0] - p[0], d1 = q[1] - p[1], d2 = q[2] - p[2];
    return std::fmaf(d2, d2, std::fmaf(d1, d1, d0 * d0));
}

template <class F>
void dn_rows(uint64_t H, F body) {
    const unsigned threads = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<std::thread> th;
    for (unsigned t = 1; t < threads; ++t)
        th.emplace_back([&, t] {
            for (uint64_t y = t; y < H; y += threads) body(y);
        });
    for (uint64_t y = 0; y < H; y += threads) body(y);
    for (auto& t : th) t.join();
}

}  // namespace

extern "C" {

// rtz_denoise on host buffers (whole frame, row-major, 3 f32 per pixel); either output may be NULL.
int orc_mirror_denoise(uint64_t W, uint64_t H, const float* c, const float* a, const float* n, uint32_t levels,
                       double sigma_color, double sigma_normal, double sigma_albedo, float* linear_out,
                       uint8_t* rgb_out) {
    if (!c || !a || !n || W == 0 || H == 0) return RTZ_ERR_BAD_ARG;
    const uint64_t np = W * H;
    std::vector<float> out(3 * np);
    if (levels == 0) {
        std::copy(c, c + 3 * np, out.begin());
    } else {
        float ic = (float)(1.0 / (sigma_color * sigma_color));
        const float in = (float)(1.0 / (sigma_normal * sigma_normal));
        const float ia = (float)(1.0 / (sigma_albedo * sigma_albedo));
        std::vector<float> e(3 * np), e2(3 * np);
        for (uint64_t i = 0; i < 3 * np; ++i) e[i] = c[i] / dn_modulus(a[i]);
        const float h1[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};
        for (uint32_t l = 0; l < levels; ++l) {
            const int64_t s = (int64_t)1 << l;
            dn_rows(H, [&](uint64_t y) {
                for (uint64_t x = 0; x < W; ++x) {
                    const uint64_t p = y * W + x;
                    const float* ep = &e[3 * p];
                    float num[3] = {0.0f, 0.0f, 0.0f}, den = 0.0f;
                    for (int i = 0; i < 5; ++i) {
                        const int64_t qy = (int64_t)y + (i - 2) * s;
                        if (qy < 0 || qy >= (int64_t)H) continue;
                        for (int j = 0; j < 5; ++j) {
                            const int64_t qx = (int64_t)x + (j - 2) * s;
                            if (qx < 0 || qx >= (int64_t)W) continue;
                            const uint64_t q = (uint64_t)qy * W + (uint64_t)qx;
                            const float* eq = &e[3 * q];
                            const float w = ((h1[i] * h1[j]) * dn_edge(dn_dist2(eq, ep) * ic)) *
                                            dn_edge(dn_dist2(&n[3 * q], &n[3 * p]) * in) *
                                            dn_edge(dn_dist2(&a[3 * q], &a[3 * p]) * ia);
                            for (int k = 0; k < 3; ++k) num[k] = std::fmaf(w, eq[k] - ep[k], num[k]);
                            den = den + w;
                        }
                    }
                    for (int k = 0; k < 3; ++k) e2[3 * p + k] = ep[k] + num[k] / den;
                }
            });
            e.swap(e2);
            ic = ic * 4.0f;
        }
        for (uint64_t i = 0; i < 3 * np; ++i) out[i] = e[i] * dn_modulus(a[i]);
    }
    for (uint64_t i = 0; i < 3 * np; ++i) {
        if (linear_out) linear_out[i] = out[i];
        if (rgb_out) rgb_out[i] = toByte((double)out[i]);
    }
    return RTZ_OK;
}

}  // extern "C"
