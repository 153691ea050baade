// rtz_bvh.cuh — EXTENSION, not in the reference (SURVEY §8f row 4): RTZ_MODE_PATH_BVH.
//
// The reference's HittableList.hit is brute force over all spheres (src/hittable.zig:64-77) and that is what
// the product's default mode, the benchmark and the roofline are about.  This mode answers the same question —
// the closest hit of a ray — through a bounding-volume hierarchy over the spheres, and is held to the same
// image BIT FOR BIT: every sphere it does test goes through exactly the arithmetic of the brute-force path
// (sign of the expanded discriminant, then the root from the reference's direct form), and the closest hit
// is the minimum over (t, sphere index) in lexicographic order, which is what "first sphere wins a tie" of
// the ascending brute-force loop means.  The boxes are padded, so the traversal can only visit MORE spheres
// than the ray touches, never fewer.  `rtz_stats.sphere_tests` counts the tests actually made in this mode.
#pragma once
#include "rtz_kernels.cuh"

namespace rtz {

// One inner node: the boxes of its two children and where they lead.  child >= 0: inner node index;
// child < 0: leaf, -1 - (first * 8 + count) into `order` (count <= 4 spheres); kBvhEmpty: nothing there.
struct BvhNode {
    float lo0[3], hi0[3], lo1[3], hi1[3];
    int child0, child1;
    float inv_r0, inv_r1;  // the largest 1 / r among each child's spheres (hit_box's slack)
};
static_assert(sizeof(BvhNode) == 64, "BvhNode is four float4");
constexpr int kBvhEmpty = 0x7fffffff;
constexpr int kBvhMaxDepth = 24;  // median split, leaves of <= 4: 2^20 spheres need 19 levels

struct BvhParams {
    TraceParams p;
    const BvhNode* nodes;
    const int* order;     // leaf ranges: original sphere indices
    const float* wexp;    // [n] w = -(|c|^2 - r^2) of the expanded discriminant, as in the sweep layout
    float r2;             // the squared origin radius the boxes' padding covers (hit_box)
};

// Sphere.hit for one sphere through the brute-force arithmetic, closest hit kept as min over (t, index).
__device__ __forceinline__ void test_sphere_lex(const float4 g, float w, int i, const Path& p, const RayK& k, float tmin_d,
                                                float& closest, int& best) {
    const float de = expanded_disc(g.x, g.y, g.z, w, p, k);
    if (__float_as_uint(de) >> 31) return;  // the sweep's candidate test: sign bit of the expanded discriminant
    const float ocx = g.x - p.ox, ocy = g.y - p.oy, ocz = g.z - p.oz;
    const float h = fmaf(p.dz, ocz, fmaf(p.dy, ocy, p.dx * ocx));
    const float c = fmaf(ocz, ocz, fmaf(ocy, ocy, fmaf(ocx, ocx, g.w)));
    const float disc = fmaf(h, h, -c);
    if (!(disc >= 0.0f)) return;
    const float sq = (i == p.self) ? fabsf(h) : sqrtf(disc);  // slow_path's exact roots h -/+ |h| on the self sphere
    // the root the ascending loop would accept: the near one if it lies beyond t_min, else the far one
    float t = h - sq;
    if (!(t > tmin_d)) {
        t = h + sq;
        if (!(t > tmin_d)) return;
    }
    if (t < closest || (t == closest && i < best)) closest = t, best = i;
}

// slab test of one box against the ray segment (t_lo, t_hi); fminf/fmaxf drop the NaN of 0 * inf.
// The direct form accepts a root of sphere (c, r) at a point up to 12 eps |c - o|^2 / r outside the sphere (box_reach
// in rtz_kernels.cuh).  The builder pads every sphere by 1e-6 (1.001 R + |c|)^2 / r, which covers origins with
// |o|^2 <= r2 = R^2 (the origin test reads |o|^2 (1 - 2^-18)).  A ray from farther out (kFar) widens each box by
// s = 1e-6 (|m - o| + |h|)^2 max(1/r) instead (m the box's centre, h its half diagonal: |c - o| <= |m - o| + |h|).
template <bool kFar>
__device__ __forceinline__ bool hit_box(const float* lo, const float* hi, float inv_r, const Path& p, float ix, float iy,
                                        float iz, float t_lo, float t_hi, float& t_near) {
    float s = 0.0f;
    if (kFar) {
        const float mx = 0.5f * (lo[0] + hi[0]) - p.ox, my = 0.5f * (lo[1] + hi[1]) - p.oy, mz = 0.5f * (lo[2] + hi[2]) - p.oz;
        const float hx = 0.5f * (hi[0] - lo[0]), hy = 0.5f * (hi[1] - lo[1]), hz = 0.5f * (hi[2] - lo[2]);
        const float dist = sqrtf(fmaf(mz, mz, fmaf(my, my, mx * mx))) + sqrtf(fmaf(hz, hz, fmaf(hy, hy, hx * hx)));
        s = 1e-6f * (dist * dist) * inv_r;
    }
    const float ax = (lo[0] - s - p.ox) * ix, bx = (hi[0] + s - p.ox) * ix;
    const float ay = (lo[1] - s - p.oy) * iy, by = (hi[1] + s - p.oy) * iy;
    const float az = (lo[2] - s - p.oz) * iz, bz = (hi[2] + s - p.oz) * iz;
    const float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), t_lo));
    const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), t_hi));
    t_near = tn;
    return tn <= tf;
}

constexpr int kBvhDone = (int)0x80000000;
template <int kBlock, bool kFar>
__device__ __forceinline__ void bvh_walk(const BvhParams& B, const Path& p, const RayK& k, float tmin_d, float& closest,
                                         int& best, int* stack, float* tstack, unsigned long long& n_tests) {
    const float ix = 1.0f / p.dx, iy = 1.0f / p.dy, iz = 1.0f / p.dz;
    const float4* geom = B.p.geom;
    int sp = 0;
    int node = 0;
    auto pop = [&]() {
        while (sp > 0) {
            --sp;
            if (tstack[sp * kBlock] <= closest) return stack[sp * kBlock];
        }
        return kBvhDone;
    };
    for (;;) {
        while (node >= 0) {  // inner nodes
            const float4* np = reinterpret_cast<const float4*>(B.nodes + node);
            const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3);
            const float lo0[3] = {n0.x, n0.y, n0.z}, hi0[3] = {n0.w, n1.x, n1.y};
            const float lo1[3] = {n1.z, n1.w, n2.x}, hi1[3] = {n2.y, n2.z, n2.w};
            const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
            float t0, t1;
            const bool h0 = c0 != kBvhEmpty && hit_box<kFar>(lo0, hi0, n3.z, p, ix, iy, iz, tmin_d, closest, t0);
            const bool h1 = c1 != kBvhEmpty && hit_box<kFar>(lo1, hi1, n3.w, p, ix, iy, iz, tmin_d, closest, t1);
            if (h0 && h1) {  // nearer child first, the other on the stack with its entry distance
                const bool swap = t1 < t0;
                stack[sp * kBlock] = swap ? c0 : c1;
                tstack[sp * kBlock] = swap ? t0 : t1;
                ++sp;
                node = swap ? c1 : c0;
            } else if (h0 || h1) {
                node = h0 ? c0 : c1;
            } else {
                node = pop();
            }
        }
        if (node == kBvhDone) break;
        const int code = -1 - node, first = code >> 3, cnt = code & 7;  // a leaf
        for (int q = 0; q < cnt; ++q) {
            const int i = __ldg(B.order + first + q);
            test_sphere_lex(__ldg(geom + i), __ldg(B.wexp + i), i, p, k, tmin_d, closest, best);
        }
        n_tests += (unsigned)cnt;
        node = pop();
    }
}

// Closest hit through the hierarchy.  "While-while" traversal: a warp first walks inner nodes until every lane
// holds a leaf (or is done), then all lanes test their leaves together, so that box tests and sphere tests
// are not interleaved lane by lane.  A popped entry whose box lies beyond the current closest hit is skipped.
template <int kBlock>
__device__ __forceinline__ void bvh_closest_hit(const BvhParams& B, const Path& p, float tmin, float tmax, int* stack,
                                                float* tstack, float& t_out, int& best_out, unsigned long long& n_tests) {
    const RayK k = ray_constants(p);
    const float tmin_d = tmin * p.len;
    float closest = tmax * p.len;
    int best = -1;
    if (-k.nk2 <= B.r2)
        bvh_walk<kBlock, false>(B, p, k, tmin_d, closest, best, stack, tstack, n_tests);
    else
        bvh_walk<kBlock, true>(B, p, k, tmin_d, closest, best, stack, tstack, n_tests);
    t_out = closest, best_out = best;
}

// Persistent path-trace kernel of the BVH mode: one path per thread, otherwise the organisation of trace_body
// (chunks of one pixel from a global queue, regeneration, integer accumulation, the same camera_ray / shade).
template <int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_bvh(const __grid_constant__ BvhParams B) {
    __shared__ int s_stack[kBvhMaxDepth * kBlock];
    __shared__ float s_tstack[kBvhMaxDepth * kBlock];
    const TraceParams& P = B.p;
    int* stack = s_stack + threadIdx.x;
    float* tstack = s_tstack + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DevCamera& cam = P.cam;
    Slot S;
    S.alive = false, S.lp = 0;
    S.key = RngKey{cam.key0, cam.key1, 0u, 0u};
    S.path.ox = S.path.oy = S.path.oz = 0.f, S.path.dx = S.path.dy = 0.f, S.path.dz = 1.f;
    S.path.tr = S.path.tg = S.path.tb = 0.f, S.path.len = 1.f, S.path.self = -1, S.path.bounce = 0;
    uint32_t ch_lp = 0, ch_x = 0, ch_y = 0, ch_next = 0, ch_end = 0;
    bool exhausted = false;
    unsigned long long n_seg = 0, n_tests = 0;
    uint32_t n_samp = 0, n_cap = 0, n_abs = 0;
    for (;;) {
        unsigned need = __ballot_sync(0xFFFFFFFFu, !S.alive);
        while (need && !exhausted) {
            if (ch_next >= ch_end) {
                unsigned long long cid = 0;
                if (lane == 0) cid = atomicAdd(P.counter, 1ULL);
                cid = __shfl_sync(0xFFFFFFFFu, cid, 0);
                if (__any_sync(0xFFFFFFFFu, cid >= P.n_chunks)) {
                    exhausted = true;
                    break;
                }
                ch_lp = (uint32_t)(cid / P.chunks_per_pixel);
                const uint32_t part = (uint32_t)(cid - (unsigned long long)ch_lp * P.chunks_per_pixel);
                const bool inside = local_to_global(P.sh, cam.width, cam.height, ch_lp, ch_x, ch_y);
                if (__any_sync(0xFFFFFFFFu, !inside)) continue;  // tile padding
                ch_next = part * P.chunk;
                ch_end = min(ch_next + P.chunk, cam.spp);
            }
            const uint32_t avail = ch_end - ch_next;
            const uint32_t rank = __popc(need & lt_mask);
            if (((need >> lane) & 1u) && rank < avail) {
                S.lp = ch_lp;
                S.key.pixel = ch_y * cam.width + ch_x, S.key.sample = ch_next + rank;
                camera_ray(cam, S.key, ch_x, ch_y, S.path);
                S.alive = true;
            }
            ch_next += min((uint32_t)__popc(need), avail);
            need = __ballot_sync(0xFFFFFFFFu, !S.alive);
        }
        if (__ballot_sync(0xFFFFFFFFu, S.alive) == 0u) break;
        if (S.alive) {
            float t;
            int best;
            bvh_closest_hit<kBlock>(B, S.path, cam.tmin, cam.tmax, stack, tstack, t, best, n_tests);
            finish_or_continue(P, P.geom, P.aux, P.albedo, S, t, best, n_seg, n_samp, n_cap, n_abs);
        }
        __syncwarp();
    }
    unsigned long long v0 = n_samp, v1 = n_seg, v2 = n_cap, v3 = n_abs, v4 = n_tests;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v0 += __shfl_xor_sync(0xFFFFFFFFu, v0, o);
        v1 += __shfl_xor_sync(0xFFFFFFFFu, v1, o);
        v2 += __shfl_xor_sync(0xFFFFFFFFu, v2, o);
        v3 += __shfl_xor_sync(0xFFFFFFFFu, v3, o);
        v4 += __shfl_xor_sync(0xFFFFFFFFu, v4, o);
    }
    if (lane == 0) {
        atomicAdd(P.stats + 0, v0);
        atomicAdd(P.stats + 1, v1);
        atomicAdd(P.stats + 2, v2);
        atomicAdd(P.stats + 3, v3);
        atomicAdd(P.stats + 4, v4);
    }
}

// RTZ_SWEEP_BVH (rtz_probe_sweeps): one ray per thread through bvh_closest_hit, with trace_kernel_bvh's stacks
__global__ void __launch_bounds__(128) probe_bvh_kernel(const __grid_constant__ BvhParams B, const SweepProbeIO io) {
    __shared__ int s_stack[kBvhMaxDepth * 128];
    __shared__ float s_tstack[kBvhMaxDepth * 128];
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= io.m) return;
    Path p;
    probe_path(io.rays[k], p);
    float t;
    int best;
    unsigned long long n_tests = 0;
    bvh_closest_hit<128>(B, p, io.tmin, io.tmax, s_stack + threadIdx.x, s_tstack + threadIdx.x, t, best, n_tests);
    probe_store(io, k, p, t, best);
}

}  // namespace rtz
