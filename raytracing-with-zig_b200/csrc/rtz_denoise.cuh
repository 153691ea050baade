// rtz_denoise.cuh — edge-avoiding à-trous denoiser (Dammertz et al. 2010) over a whole row-major frame (sm_100a):
// the linear colour, demodulated by the first-hit albedo, filtered under the guidance of that albedo and the first-hit
// normal (rtz_render_guides), then remodulated and quantised as the resolve does.
//
// Per pixel p, with colour c, albedo a and normal n (3 f32 each):
//   demodulate   m = max(a, 2^-8) per channel, e = c / m;
//   level k      (k = 0 .. L-1, step s = 2^k) over the taps (dx, dy) in {-2..2}^2 * s that lie in the image, visited
//                dy-major then dx, both ascending, with the B3-spline weight h = h1[dy] * h1[dx],
//                h1 = (1/16, 1/4, 3/8, 1/4, 1/16) (exact dyadic products):
//                  w_q = ((h * E(|e_q - e_p|^2 * ic_k)) * E(|n_q - n_p|^2 * in)) * E(|a_q - a_p|^2 * ia),
//                  |v|^2 = fmaf(v2, v2, fmaf(v1, v1, v0 * v0)),
//                  E(x) = max(0, 1 - x 2^-6)^64: one fmaf, one fmaxf, six squarings (exactly 0 from x = 64 on),
//                  num_c = fmaf(w_q, e_q,c - e_p,c, num_c), den = den + w_q (both from +0, in tap order),
//                  e'_p,c = e_p,c + num_c / den      (the centre tap has w = 9/64, so den > 0);
//                ic_k = ic_0 * 4^k, ic_0 = (float)(1 / sigma_c^2), in, ia likewise: formed on the host;
//   remodulate   out = e^(L) * m; the bytes are Color.toRgb of (double)out (to_byte, the resolve's quantiser).
// L = 0 is a copy: out = c.  Only IEEE + - * / and explicit fmaf / fmaxf, no atomics, a fixed order: a CPU
// restatement (tests/denoise_mirror.cpp) agrees bit for bit.
//
// The difference form makes two things exact: a region constant in e and in the guides comes back unchanged, and a
// tap at guide distance x >= 64 adds exactly 0 to both sums, so nothing crosses a hard normal or albedo edge.
#pragma once
#include "rtz_kernels.cuh"

namespace rtz {

constexpr int kDenoiseMaxLevels = 8;
constexpr unsigned kDenoiseBlockX = 32, kDenoiseBlockY = 8;  // a 32 x 8 tile of pixels per block: taps share lines

// the packed planes of the context's scratch buffer: e (ping, pong), normal, albedo; one float4 per pixel each
struct DenoiseLevelParams {
    const float4* __restrict__ e_in;
    float4* __restrict__ e_out;
    const float4* __restrict__ nrm;
    const float4* __restrict__ alb;
    uint32_t width, height, tiles_x, step;
    float ic, in, ia;  // 1/sigma^2 of colour (this level), normal, albedo
};

__device__ __forceinline__ float denoise_modulus(float a) { return fmaxf(a, 0x1p-8f); }

// E(x) = max(0, 1 - x/64)^64
__device__ __forceinline__ float denoise_edge(float x) {
    float t = fmaxf(fmaf(x, -0x1p-6f, 1.0f), 0.0f);
    t = t * t, t = t * t, t = t * t, t = t * t, t = t * t, t = t * t;
    return t;
}

__device__ __forceinline__ float denoise_dist2(float4 q, float4 p) {
    const float d0 = q.x - p.x, d1 = q.y - p.y, d2 = q.z - p.z;
    return fmaf(d2, d2, fmaf(d1, d1, d0 * d0));
}

// pixel of this thread in the block's 32 x 8 tile (a 1-D grid of tiles: any frame of < 2^31 pixels fits)
__device__ __forceinline__ bool denoise_pixel(uint32_t width, uint32_t height, uint32_t tiles_x, uint32_t& x,
                                              uint32_t& y) {
    const uint32_t ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    x = tx * kDenoiseBlockX + threadIdx.x, y = ty * kDenoiseBlockY + threadIdx.y;
    return x < width && y < height;
}

// demodulate and pack: e = c / max(a, 2^-8), and the guides, one float4 per pixel each
__global__ void __launch_bounds__(256) denoise_prepare_kernel(const float* __restrict__ color,
                                                              const float* __restrict__ albedo,
                                                              const float* __restrict__ normal, float4* __restrict__ e,
                                                              float4* __restrict__ nrm, float4* __restrict__ alb,
                                                              uint32_t width, uint32_t height, uint32_t tiles_x) {
    uint32_t x, y;
    if (!denoise_pixel(width, height, tiles_x, x, y)) return;
    const uint32_t p = y * width + x;
    const size_t p3 = 3ull * p;  // 3 * pixels may pass 2^32
    const float c0 = color[p3], c1 = color[p3 + 1], c2 = color[p3 + 2];
    const float a0 = albedo[p3], a1 = albedo[p3 + 1], a2 = albedo[p3 + 2];
    e[p] = make_float4(c0 / denoise_modulus(a0), c1 / denoise_modulus(a1), c2 / denoise_modulus(a2), 0.0f);
    alb[p] = make_float4(a0, a1, a2, 0.0f);
    nrm[p] = make_float4(normal[p3], normal[p3 + 1], normal[p3 + 2], 0.0f);
}

// one à-trous level at step P.step
__global__ void __launch_bounds__(256) denoise_level_kernel(const DenoiseLevelParams P) {
    uint32_t x, y;
    if (!denoise_pixel(P.width, P.height, P.tiles_x, x, y)) return;
    const float h1[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};
    const uint32_t p = y * P.width + x;
    const float4 ep = P.e_in[p], np = P.nrm[p], ap = P.alb[p];
    float num0 = 0.0f, num1 = 0.0f, num2 = 0.0f, den = 0.0f;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        // unsigned wrap-around: a row above the image wraps past 2^31 > height and is skipped like one below it
        const uint32_t qy = y + (uint32_t)(i - 2) * P.step;
        if (qy >= P.height) continue;
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const uint32_t qx = x + (uint32_t)(j - 2) * P.step;
            if (qx >= P.width) continue;
            const uint32_t q = qy * P.width + qx;
            const float4 eq = __ldg(P.e_in + q), nq = __ldg(P.nrm + q), aq = __ldg(P.alb + q);
            const float w = ((h1[i] * h1[j]) * denoise_edge(denoise_dist2(eq, ep) * P.ic)) *
                                denoise_edge(denoise_dist2(nq, np) * P.in) * denoise_edge(denoise_dist2(aq, ap) * P.ia);
            num0 = fmaf(w, eq.x - ep.x, num0), num1 = fmaf(w, eq.y - ep.y, num1), num2 = fmaf(w, eq.z - ep.z, num2);
            den = den + w;
        }
    }
    P.e_out[p] = make_float4(ep.x + num0 / den, ep.y + num1 / den, ep.z + num2 / den, 0.0f);
}

// remodulate (e == null: levels = 0, the colour itself), then the optional f32 store and the bytes
__global__ void __launch_bounds__(256) denoise_finish_kernel(const float4* __restrict__ e,
                                                             const float* __restrict__ color,
                                                             const float* __restrict__ albedo,
                                                             float* __restrict__ linear_out, uint8_t* __restrict__ rgb,
                                                             uint32_t width, uint32_t height, uint32_t tiles_x) {
    uint32_t x, y;
    if (!denoise_pixel(width, height, tiles_x, x, y)) return;
    const uint32_t p = y * width + x;
    const size_t p3 = 3ull * p;
    float v[3];
    if (e) {
        const float4 ev = e[p];
        v[0] = ev.x * denoise_modulus(albedo[p3]);
        v[1] = ev.y * denoise_modulus(albedo[p3 + 1]);
        v[2] = ev.z * denoise_modulus(albedo[p3 + 2]);
    } else {
        v[0] = color[p3], v[1] = color[p3 + 1], v[2] = color[p3 + 2];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        if (linear_out) linear_out[p3 + c] = v[c];
        if (rgb) rgb[p3 + c] = to_byte((double)v[c]);
    }
}

}  // namespace rtz
