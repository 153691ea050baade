// rtz_guides.cuh — first-hit guide buffers for a denoiser (sm_100a): the albedo and the normal that the camera rays
// of a frame see at their closest hit.
//
// The guide kernel does not share a launch with the render.  It regenerates the frame's camera rays (camera_ray with
// the key (seed, j*W + i, s), bounce 0: the render's first ray of sample s, bit for bit) and finds their closest hit
// with the render's own sweep (sweep2, unchanged), so its hits are the ones the render's first world.hit returns:
// the (t, original index) minimum over Scene.interval, with the same gate and roots.  RTZ_MODE_PATH_BVH scenes beyond
// the constant bank find that minimum through the hierarchy instead (guides_kernel_bvh): the same buffers bit for bit.
//
// Per ray, six f32 values:
//   albedo  hit: the sphere's albedo for lambertian and metal (the attenuation scatter applies), (1, 1, 1) for
//                dielectric; miss: the sky colour of shade's miss branch at throughput 1, which is what the render
//                returns for that ray (so colour / albedo = 1 on the sky);
//   normal  hit: the HitRecord normal (p - c) * (1/r), flipped against the ray on a back face; miss: (0, 0, 0).
// Per pixel and channel, the values of samples 0 .. g-1 are added in ascending sample order, each in f32 to a running
// sum that starts at +0, and the sum is divided by (float)g once.  Normals are averaged, not renormalised.  A CPU
// restatement of this order (tests/guide_mirror.cpp) must agree bit for bit.
//
// Work: a warp sweeps 64 camera rays at a time, two per lane, as the render does.  Its work item is whole pixels:
// floor(64 / g) of them for g < 64 (so g = 1 still fills all 64 slots), one for g >= 64, swept in rounds of 64 of its
// samples.  A pixel never spans two warps, so its sums keep their order: after each sweep the six values of every ray
// are staged in shared memory and each (pixel, channel) is folded by one lane.
//
// Shards: the items run over the local pixels of a rank's tiles (ShardGeom, the compact layout of the render), each
// mapped to its global pixel (x, y) by local_to_global_rcp once per item (guide_slot: mapped per ray and per stored
// channel, with divisions, the whole-frame kernel ran 4-15 % longer on a B200) and keyed by y*W + x, so a pixel's guides do not depend on the
// shard that computes them.  The whole frame is the shard {0, 1, W, 1}, whose compact layout is the row-major image.
// A tile-padding pixel still sweeps rays (those of pixel (min(x, W-1), min(y, H-1))) so that every lane takes part in
// the sweep's votes; its sums are never stored into a real pixel.
#pragma once
#include "rtz_bvh.cuh"
#include "rtz_kernels.cuh"

namespace rtz {

struct GuideParams {
    DevCamera cam;
    const float4* pairs;     // sweep layout in global memory (guide_kernel_global; the constant-bank kernel has its own)
    const float4* geom;      // per-lane rows {cx, cy, cz, -r^2}: candidate roots, hit records
    const float4* aux;       // {r, 1/r, fuzz|ior, type}
    const float4* albedo;    // {r, g, b, 1/ior}
    const float* wexp;       // w of the pair layout as a plain row
    const int* orig;         // culled sweep: slot -> index in the caller's list (ties in t), else null
    int n_pad;
    uint32_t g;              // guide samples per pixel
    uint32_t pix_per_item;   // whole pixels per warp: floor(64 / g), 1 for g >= 64
    uint32_t n_items;
    ShardGeom sh;            // the pixels the items run over
    unsigned long long rcp_tile_pixels, rcp_tiles_x, rcp_tile_w;  // its divisors as reciprocals (local_to_global_rcp)
    uint32_t n_local;        // sh.n_local_tiles * sh.tile_pixels
    uint32_t row_major;      // 0: outputs in the compact layout, padding written as 0; 1: at y*W + x of row-major
                             // planes (possibly device 0's memory through peer access), padding not written
    float* albedo_out;       // 3 f32 per pixel, or null
    float* normal_out;       // 3 f32 per pixel, or null
};

// the constant-bank form: the rows the render's constant-bank kernels sweep (plain, or regrouped with their boxes)
struct GuideParamsConst {
    GuideParams p;
    float4 pairs[kMaxConstSpheres];
    float4 boxes[2 * (kMaxConstSpheres / 32)];
    float cull_r2;
    int split_max;
};

constexpr int kGuideStageFloats = 6 * 64;  // per warp: the six values of 64 rays

// Ray slot j of a work item (lane j % 32, first or second path): its local pixel pix0 + j / g (a slot past the item's
// last ray takes ray 0 of the item and its result is not folded; for g >= 64 every slot is the item's one pixel), that
// pixel's (x, y) (tile padding: clamped into the frame, a valid ray whose sums are never stored into a real pixel) and
// the first sample index of the slot's pixel among the item's rays.  Mapped once per item, not per round.
struct GuideSlot {
    uint32_t x, y, base;
};

// where slot j's pixel is stored (low 32 bits: pixel index in the output, compact or row-major) | kGuidePadding
constexpr unsigned long long kGuidePadding = 1ull << 32;

__device__ __forceinline__ GuideSlot guide_slot(const GuideParams& P, uint32_t pix0, uint32_t j, uint32_t rays,
                                                unsigned long long& dest) {
    const DevCamera& cam = P.cam;
    const uint32_t pl = (j < rays ? j : 0) / P.g;
    GuideSlot s;
    const bool inside = local_to_global_rcp(P.sh, P.rcp_tile_pixels, P.rcp_tiles_x, P.rcp_tile_w, cam.width, cam.height,
                                            pix0 + pl, s.x, s.y);
    dest = (inside ? 0ull : kGuidePadding) | (P.row_major ? (inside ? s.y * cam.width + s.x : 0u) : pix0 + pl);
    s.x = min(s.x, cam.width - 1), s.y = min(s.y, cam.height - 1);
    s.base = pl * P.g;
    return s;
}

// the slot's camera ray in the round that starts at ray r0 of the item (pixel y*W + x, sample r - base)
__device__ __forceinline__ void guide_ray(const DevCamera& cam, const GuideSlot& s, uint32_t r, uint32_t rays, Path& p) {
    if (r >= rays) r = 0;
    camera_ray(cam, RngKey{cam.key0, cam.key1, s.y * cam.width + s.x, r - s.base}, s.x, s.y, p);
}

// the six values of one swept ray into its column `j` of the staging rows (row c = channel c: albedo rgb, normal xyz)
__device__ __forceinline__ void guide_values(const GuideParams& P, const Path& p, float t, int best, float* stage,
                                             uint32_t j) {
    float v[6];
    if (best < 0) {
        // shade's sky (src/camera.zig:171-177) at throughput 1
        const float a = 0.5f * (p.dy + 1.0f);
        const float w = 1.0f - a;
        v[0] = fmaf(a, 0.5f, w), v[1] = fmaf(a, 0.7f, w), v[2] = fmaf(a, 1.0f, w);
        v[3] = v[4] = v[5] = 0.0f;
    } else {
        const float4 ax = __ldg(P.aux + best);
        float px, py, pz;
        hit_record(P.geom[best], ax.y, p, t, px, py, pz, v[3], v[4], v[5]);
        if (__float_as_int(ax.w) == kDielectric) {
            v[0] = v[1] = v[2] = 1.0f;
        } else {
            const float4 al = __ldg(P.albedo + best);
            v[0] = al.x, v[1] = al.y, v[2] = al.z;
        }
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) stage[c * 64 + j] = v[c];
}

// channel c of the pixel at `dest` (guide_slot): compact padding is stored as +0, row-major padding not at all
__device__ __forceinline__ void guide_store(const GuideParams& P, unsigned long long dest, uint32_t c, float value) {
    float* out = c < 3 ? P.albedo_out : P.normal_out;
    if (!out || (dest >= kGuidePadding && P.row_major)) return;
    out[3ull * (uint32_t)dest + (c < 3 ? c : c - 3)] = dest >= kGuidePadding ? 0.0f : value;
}

// The work split and fold of every guide kernel, over its staging rows (kGuideStageFloats or more).
// sweep(P, a, b, ta, ia, tb, ib, stage) finds the closest hits of the lane's two rays, called by the whole (converged)
// warp; it may use the staging rows as scratch until it returns.
template <class Sweep>
__device__ __forceinline__ void guide_body(const GuideParams& P, float* __restrict__ stage_mem, Sweep sweep) {
    float* const stage = stage_mem;
    // one warp per block, so that the work item is visibly warp-uniform to ptxas: with the item derived from the warp
    // index inside a wider block, it guards the sweep's votes with divergent-branch checks (BRA.DIV)
    const uint32_t item = blockIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    const DevCamera& cam = P.cam;
    const uint32_t g = P.g;
    const uint32_t pix0 = item * P.pix_per_item;
    const uint32_t n_here = min(P.pix_per_item, P.n_local - pix0);  // the last item may hold fewer
    const uint32_t rays = n_here * g;
    __shared__ unsigned long long dest[64];  // per slot: where its pixel is stored (the fold reads slot pl * g's)
    const GuideSlot sa = guide_slot(P, pix0, lane, rays, dest[lane]);
    const GuideSlot sb = guide_slot(P, pix0, 32 + lane, rays, dest[32 + lane]);
    float acc = 0.0f;  // g >= 64: lane c < 6 holds the running sum of channel c of the item's one pixel
    for (uint32_t r0 = 0; r0 < rays; r0 += 64) {
        Path a, b;
        guide_ray(cam, sa, r0 + lane, rays, a);
        guide_ray(cam, sb, r0 + 32 + lane, rays, b);
        __syncwarp();  // converged before the sweep's votes
        float ta = 0.f, tb = 0.f;
        int ia = -1, ib = -1;
        sweep(P, a, b, ta, ia, tb, ib, stage);
        __syncwarp();  // the culled sweep reads its staging rows (the same memory) until it returns
        guide_values(P, a, ta, ia, stage, lane);
        guide_values(P, b, tb, ib, stage, 32 + lane);
        __syncwarp();
        if (g < 64) {  // one round: fold every (pixel, channel) of the item, samples in ascending order
            for (uint32_t q = lane; q < 6 * n_here; q += 32) {
                const uint32_t pl = q / 6, c = q - 6 * pl;
                const float* row = stage + c * 64 + pl * g;
                float sum = 0.0f;
                for (uint32_t s = 0; s < g; ++s) sum += row[s];
                guide_store(P, dest[pl * g], c, sum / (float)g);
            }
        } else if (lane < 6) {
            const uint32_t m = min(64u, rays - r0);
            for (uint32_t s = 0; s < m; ++s) acc += stage[lane * 64 + s];
        }
        __syncwarp();  // the next round rewrites the rows
    }
    if (g >= 64 && lane < 6) guide_store(P, dest[0], lane, acc / (float)g);
}

// The render's brute-force sweep (sweep2) over the rows it reads from the constant bank (n_pad <= kMaxConstSpheres):
// the same rows, through the same uniform loads; kCull = the culled kernel's regrouped rows, boxes and sphere-parallel
// split.
template <bool kCull>
struct GuideSweepConst {
    const GuideParamsConst& C;
    __device__ __forceinline__ void operator()(const GuideParams& P, const Path& a, const Path& b, float& ta, int& ia,
                                               float& tb, int& ib, float* stage) const {
        sweep2<true, false, kCull>(C.pairs, P.geom, P.n_pad, P.cam.tmin, P.cam.tmax, a, b, ta, ia, tb, ib, C.boxes,
                                   C.cull_r2, P.orig, P.wexp, C.split_max, reinterpret_cast<float4*>(stage));
    }
};

// ... and over the plain pair rows in global memory (L1 / L2, warp-uniform addresses), for larger scenes
struct GuideSweepGlobal {
    const float4* __restrict__ pairs;
    __device__ __forceinline__ void operator()(const GuideParams& P, const Path& a, const Path& b, float& ta, int& ia,
                                               float& tb, int& ib, float* stage) const {
        sweep2<false, false, false>(pairs, P.geom, P.n_pad, P.cam.tmin, P.cam.tmax, a, b, ta, ia, tb, ib, nullptr,
                                    0.0f, P.orig, P.wexp, 0, reinterpret_cast<float4*>(stage));
    }
};

template <bool kCull>
__global__ void __launch_bounds__(32, 24) guide_kernel_const(const __grid_constant__ GuideParamsConst C) {
    __shared__ __align__(16) float stage[kCull ? kCullStageFloats : kGuideStageFloats];
    guide_body(C.p, stage, GuideSweepConst<kCull>{C});
}

__global__ void __launch_bounds__(32, 24) guide_kernel_global(const __grid_constant__ GuideParams P) {
    __shared__ __align__(16) float stage[kGuideStageFloats];
    guide_body(P, stage, GuideSweepGlobal{P.pairs});
}

// The BVH form: BvhParams' fields around the guide parameters (bvh_closest_hit reads them by name).
struct GuideParamsBvh {
    GuideParams p;               // geom: the plain rows, which the hierarchy's `order` indexes
    const BvhNode* nodes;
    const int* order;
    const float* wexp;
    float r2;
    unsigned long long* tests;   // += the sphere tests the traversal makes (every slot's, padding included)
};

// The lane's two rays through the hierarchy, one after the other, on trace_kernel_bvh's shared-memory stacks
struct GuideSweepBvh {
    const GuideParamsBvh& B;
    int* stack;
    float* tstack;
    unsigned long long& n_tests;
    __device__ __forceinline__ void operator()(const GuideParams& P, const Path& a, const Path& b, float& ta, int& ia,
                                               float& tb, int& ib, float*) const {
        bvh_closest_hit<32>(B, a, P.cam.tmin, P.cam.tmax, stack, tstack, ta, ia, n_tests);
        bvh_closest_hit<32>(B, b, P.cam.tmin, P.cam.tmax, stack, tstack, tb, ib, n_tests);
    }
};

// RTZ_MODE_PATH_BVH scenes beyond the constant bank (n_pad > kMaxConstSpheres), where guide_kernel_global would read
// every sphere for every ray.  The traversal returns the (t, original index) minimum, which is the brute-force
// sweep's answer, so the buffers are guide_kernel_global's bit for bit.
__global__ void __launch_bounds__(32, 24) guides_kernel_bvh(const __grid_constant__ GuideParamsBvh B) {
    __shared__ __align__(16) float stage[kGuideStageFloats];
    __shared__ int s_stack[kBvhMaxDepth * 32];
    __shared__ float s_tstack[kBvhMaxDepth * 32];
    unsigned long long n_tests = 0;
    guide_body(B.p, stage, GuideSweepBvh{B, s_stack + threadIdx.x, s_tstack + threadIdx.x, n_tests});
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n_tests += __shfl_xor_sync(0xFFFFFFFFu, n_tests, o);
    if (threadIdx.x == 0) atomicAdd(B.tests, n_tests);
}

}  // namespace rtz
