// rtz_bvh_build.cuh — scenes installed from device memory (rtz_scene_upload_device) and the BVH of
// RTZ_MODE_PATH_BVH built on the device.  Both give what the host paths give, bit for bit:
//   - scene_check_kernel / scene_flatten_kernel: host_scene's tests and rows, with its arithmetic (f64 -> f32 casts
//     round to nearest, q in f64 with the same association, no contraction: the build passes -fmad=false);
//   - the bvh_*_kernels: BvhBuilder's tree node for node (DESIGN.md §5 K8).  Its topology depends on n alone (a range
//     of cnt > 4 splits into cnt / 2 and cnt - cnt / 2, numbered in pre-order), so every level is built at once: the
//     centroid bounds of each range choose the axis, and a stable two-pass radix sort over (range, index) then
//     (range, key) puts the cnt / 2 smallest spheres under (key, index) on the left, the set std::nth_element leaves
//     there.  Boxes are order-independent f32 min / max over a range of per-sphere boxes computed as
//     BvhBuilder::bounds computes them.
#pragma once
#include <cub/device/device_radix_sort.cuh>

#include "../../include/rtz.h"
#include "rtz_bvh.cuh"

namespace rtz {

// ---- device scene install ----------------------------------------------------------------------------------------

__device__ __forceinline__ bool finite3_d(const double v[3]) { return isfinite(v[0]) && isfinite(v[1]) && isfinite(v[2]); }

// Whether host_scene accepts the sphere: its tests, in any order (the host names the refused sphere).
__device__ __forceinline__ bool sphere_ok(const rtz_sphere& s) {
    if (s.mat_type < RTZ_MAT_LAMBERTIAN || s.mat_type > RTZ_MAT_DIELECTRIC) return false;
    const float r = (float)(s.radius < 0 ? 0.0 : s.radius);
    const bool mat_ok = s.mat_type == RTZ_MAT_DIELECTRIC
                            ? (isfinite(s.refraction_index) && (float)s.refraction_index != 0.0f)
                            : (finite3_d(s.albedo) && (s.mat_type != RTZ_MAT_METAL || isfinite(s.fuzz)));
    if (!finite3_d(s.center) || !isfinite(s.radius) || !(r > 0.0f) || !mat_ok) return false;
    if (s.mat_type != RTZ_MAT_DIELECTRIC)
        for (int k = 0; k < 3; ++k)
            if (!(s.albedo[k] >= 0.0 && s.albedo[k] <= 1.0)) return false;
    return true;
}

// *first_bad = the lowest index of a refused sphere (stays ~0 when every sphere is accepted)
__global__ void __launch_bounds__(256) scene_check_kernel(const rtz_sphere* sp, uint64_t n, unsigned long long* first_bad) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !sphere_ok(sp[i])) atomicMin(first_bad, (unsigned long long)i);
}

struct SceneRowsOut {
    float4 *geom, *pairs, *aux, *albedo;
    float* wexp;
    DSphere* ds;
};

__device__ __forceinline__ void flatten_sphere(const rtz_sphere* sp, uint64_t n, uint64_t i, const SceneRowsOut& o,
                                               float4& g, float& w) {
    if (i < n) {
        const rtz_sphere s = sp[i];
        const float r = (float)(s.radius < 0 ? 0.0 : s.radius);
        const float cx = (float)s.center[0], cy = (float)s.center[1], cz = (float)s.center[2];
        const double c2 = (double)cx * cx + (double)cy * cy + (double)cz * cz;
        const double q = (c2 - (double)r * r) - (double)kGateSlack * c2;
        g = make_float4(cx, cy, cz, -(r * r));
        w = -(float)q;
        const float param = s.mat_type == RTZ_MAT_METAL ? (float)s.fuzz : (float)s.refraction_index;
        o.aux[i] = make_float4(r, 1.0f / r, param, __int_as_float(s.mat_type));
        o.albedo[i] = make_float4((float)s.albedo[0], (float)s.albedo[1], (float)s.albedo[2], 1.0f / (float)s.refraction_index);
        o.ds[i] = DSphere{s.center[0], s.center[1], s.center[2], s.radius < 0 ? 0.0 : s.radius};
    } else {  // padding: w = -inf, never a candidate
        g = make_float4(0.f, 0.f, 0.f, -0.f);
        w = -INFINITY;
        o.aux[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        o.albedo[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    o.geom[i] = g;
    o.wexp[i] = w;
}

// One thread per pair of spheres: their rows and the two float4 of the pair layout (pair_rows).
__global__ void __launch_bounds__(256) scene_flatten_kernel(const rtz_sphere* sp, uint64_t n, uint32_t n_pad,
                                                            const SceneRowsOut o) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pad / 2) return;
    float4 A, B;
    float wa, wb;
    flatten_sphere(sp, n, 2ull * p, o, A, wa);
    flatten_sphere(sp, n, 2ull * p + 1, o, B, wb);
    o.pairs[2 * p] = make_float4(A.x, B.x, A.y, B.y);
    o.pairs[2 * p + 1] = make_float4(A.z, B.z, wa, wb);
}

// ---- the BVH on the device -----------------------------------------------------------------------------------------

// Inner nodes of BvhBuilder's tree over a range of c spheres.  At depth d the (hypothetical, fully halved) ranges
// have q = c >> d or q + 1 spheres, c - q 2^d of them q + 1; a range is an inner node iff it holds more than 4.
__host__ __device__ inline int bvh_inner_nodes(int c) {
    int total = 0;
    for (int d = 0; (c >> d) >= 4; ++d) {
        const int q = c >> d;
        total += q > 4 ? (1 << d) : c - (q << d);
    }
    return total;
}

// Whether depth d of the tree over c spheres has an inner node (a range of more than 4 spheres)
__host__ __device__ inline bool bvh_level_splits(int c, int d) {
    const int q = c >> d;
    return q > 4 || (q == 4 && c > (q << d));
}

// One range of `order` at the level being built.  cnt == 0: no range (below a leaf).  node: its inner node's index,
// or -1 for a leaf; parent: the inner node whose child it is (-1 for the root), as child (k & 1) for range k.
struct BuildRange {
    int first, cnt, node, parent;
};
constexpr int kBuildAcc = 13;  // per range: centroid min[3], max[3]; box lo[3], hi[3]; max 1/r (ordered uint32)

__device__ __forceinline__ unsigned f2o(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float o2f(unsigned o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }

__device__ __forceinline__ void init_acc(unsigned* a) {
#pragma unroll
    for (int j = 0; j < kBuildAcc; ++j) a[j] = (j < 3 || (j >= 6 && j < 9)) ? 0xFFFFFFFFu : 0u;
}

// twice the farthest point of a sphere other than sphere 0 (BvhBuilder's R): the f64 max as uint64 bits (>= 0)
__global__ void __launch_bounds__(256) bvh_reach_kernel(const float4* g, int n, unsigned long long* reach_bits) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double v = 0.0;
    if (i >= 1 && i < n) {
        const float4 s = g[i];
        v = sqrt((double)s.x * s.x + (double)s.y * s.y + (double)s.z * s.z) + sqrt(-(double)s.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reach_bits, (unsigned long long)__double_as_longlong(v));
}

// per sphere: the padded box (lo.xyz, 1 / r) and (hi.xyz) of BvhBuilder::bounds
__global__ void __launch_bounds__(256) bvh_boxes_kernel(const float4* g, int n, const unsigned long long* reach_bits,
                                                        float4* lo_ir, float4* hi) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double R = 2.0 * __longlong_as_double((long long)*reach_bits);
    const float4 s = g[i];
    const float r = sqrtf(-s.w);
    const double cn = sqrt((double)s.x * s.x + (double)s.y * s.y + (double)s.z * s.z);
    const float pad = 1e-4f * (1.0f + r + fabsf(s.x) + fabsf(s.y) + fabsf(s.z)) +
                      (float)(1e-6 * (1.001 * R + cn) * (1.001 * R + cn) / r);
    lo_ir[i] = make_float4(s.x - r - pad, s.y - r - pad, s.z - r - pad, 1.0f / r);
    hi[i] = make_float4(s.x + r + pad, s.y + r + pad, s.z + r + pad, 0.f);
}

// depth 0: order = identity, every sphere in range 0 = the whole list (node 0)
__global__ void __launch_bounds__(256) bvh_init_kernel(int n, int* order, int* seg, BuildRange* rg, unsigned* acc) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) order[p] = p, seg[p] = 0;
    if (p == 0) rg[0] = BuildRange{0, n, 0, -1}, init_acc(acc);
}

// the ranges of depth d + 1 from those of depth d (range k splits into 2k and 2k + 1), accumulators reset
__global__ void __launch_bounds__(256) bvh_ranges_kernel(const BuildRange* prev, int nr, BuildRange* next, unsigned* acc) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nr) return;
    const BuildRange P = prev[k >> 1];
    BuildRange C{0, 0, -1, -1};
    if (P.cnt > 4) {
        const int half = P.cnt / 2;
        if (k & 1)
            C = BuildRange{P.first + half, P.cnt - half, P.cnt - half > 4 ? P.node + 1 + bvh_inner_nodes(half) : -1, P.node};
        else
            C = BuildRange{P.first, half, half > 4 ? P.node + 1 : -1, P.node};
    }
    next[k] = C;
    init_acc(acc + (size_t)kBuildAcc * k);
}

// Centroid bounds, box and max 1 / r of every range new at this depth: a segmented scan over each warp's lanes (the
// ranges are runs of positions), then one set of atomics per run.
__global__ void __launch_bounds__(256) bvh_reduce_kernel(const int* order, const int* seg, const BuildRange* rg,
                                                         const float4* g, const float4* lo_ir, const float4* hi, int n,
                                                         unsigned* acc) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    int r = -1;
    unsigned v[kBuildAcc];
    init_acc(v);
    if (p < n) {
        r = seg[p];
        if (rg[r].cnt == 0) {
            r = -1;
        } else {
            const int i = order[p];
            const float4 s = g[i], l = lo_ir[i], h = hi[i];
            v[0] = v[3] = f2o(s.x), v[1] = v[4] = f2o(s.y), v[2] = v[5] = f2o(s.z);
            v[6] = f2o(l.x), v[7] = f2o(l.y), v[8] = f2o(l.z);
            v[9] = f2o(h.x), v[10] = f2o(h.y), v[11] = f2o(h.z);
            v[12] = f2o(l.w);
        }
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int ro = __shfl_up_sync(0xFFFFFFFFu, r, o);
        const bool take = lane >= (unsigned)o && ro == r;
#pragma unroll
        for (int j = 0; j < kBuildAcc; ++j) {
            const unsigned u = __shfl_up_sync(0xFFFFFFFFu, v[j], o);
            if (take) v[j] = (j < 3 || (j >= 6 && j < 9)) ? min(v[j], u) : max(v[j], u);
        }
    }
    const int rn = __shfl_down_sync(0xFFFFFFFFu, r, 1);
    if (r >= 0 && (lane == 31 || rn != r)) {
        unsigned* a = acc + (size_t)kBuildAcc * r;
#pragma unroll
        for (int j = 0; j < kBuildAcc; ++j) {
            if (j < 3 || (j >= 6 && j < 9))
                atomicMin(a + j, v[j]);
            else
                atomicMax(a + j, v[j]);
        }
    }
}

// Every range new at this depth fills its slot of its parent node (box, 1 / r, child reference); an inner range
// chooses its split axis: the largest centroid extent, ties to the lower axis.
__global__ void __launch_bounds__(256) bvh_node_kernel(const BuildRange* rg, int nr, const unsigned* acc, BvhNode* nodes,
                                                       int* axis) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nr) return;
    const BuildRange R = rg[k];
    if (R.cnt == 0) return;
    const unsigned* a = acc + (size_t)kBuildAcc * k;
    if (R.parent >= 0) {
        BvhNode& nd = nodes[R.parent];
        float* lo = (k & 1) ? nd.lo1 : nd.lo0;
        float* hi = (k & 1) ? nd.hi1 : nd.hi0;
        for (int j = 0; j < 3; ++j) lo[j] = o2f(a[6 + j]), hi[j] = o2f(a[9 + j]);
        const int child = R.cnt > 4 ? R.node : -1 - (R.first * 8 + R.cnt);
        if (k & 1)
            nd.inv_r1 = o2f(a[12]), nd.child1 = child;
        else
            nd.inv_r0 = o2f(a[12]), nd.child0 = child;
    }
    if (R.cnt > 4) {
        float ext[3];
        for (int j = 0; j < 3; ++j) ext[j] = o2f(a[3 + j]) - o2f(a[j]);
        int ax = 0;
        for (int j = 1; j < 3; ++j)
            if (ext[j] > ext[ax]) ax = j;
        axis[k] = ax;
    }
}

// pass 1 keys: (range, sphere index)
__global__ void __launch_bounds__(256) bvh_keys_index_kernel(const int* order, const int* seg, int n,
                                                             unsigned long long* keys) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) keys[p] = ((unsigned long long)seg[p] << 20) | (unsigned)order[p];
}

// pass 2 keys: (range, centre on the range's axis as an orderable integer, -0.0 as +0.0 so that the host's `<` and
// the index decide equal keys); ranges that do not split keep key 0 (their set is all that matters)
__global__ void __launch_bounds__(256) bvh_keys_axis_kernel(const unsigned long long* by_index, const BuildRange* rg,
                                                            const int* axis, const float4* g, int n,
                                                            unsigned long long* keys, int* idx) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const unsigned long long ka = by_index[p];
    const int i = (int)(ka & 0xFFFFFu), r = (int)(ka >> 20);
    unsigned key = 0;
    if (rg[r].cnt > 4) {
        const float4 s = g[i];
        const int ax = axis[r];
        float c = ax == 0 ? s.x : ax == 1 ? s.y : s.z;
        if (c == 0.0f) c = 0.0f;
        key = f2o(c);
    }
    keys[p] = ((unsigned long long)r << 32) | key;
    idx[p] = i;
}

// position p's range one level down: the left or right part of a range that split, the left part (never a new
// range) of one that did not, so that range ids stay ordered like the positions
__global__ void __launch_bounds__(256) bvh_descend_kernel(const BuildRange* rg, int n, int* seg) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int r = seg[p];
    const BuildRange R = rg[r];
    seg[p] = 2 * r + ((R.cnt > 4 && p >= R.first + R.cnt / 2) ? 1 : 0);
}

}  // namespace rtz
