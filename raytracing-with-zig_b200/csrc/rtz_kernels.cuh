// rtz_kernels.cuh — the kernels of librtz (sm_100a).
//   K1 trace_kernel     : persistent path-trace megakernel (Camera.render's loop nest,
//                         reference src/camera.zig:128-140 with rayColor :148-183 inlined)
//   K2 legacy_kernel    : deterministic f64 primary-ray kernel for the chapter4/5/6 goldens
//   K3 resolve_kernel   : 1/spp scale + gamma + clamp + 8-bit pack (src/camera.zig:137,
//                         src/color.zig:63-80, src/ppm.zig:51-56)
//   K4 deinterleave_kernel : rank-0 side of the multi-GPU tile gather
//   probe kernels       : one-ray versions of sweep / shade / toRgb for the unit KATs
//   ffma_peak_kernel    : FP32 pipe micro-benchmark for the roofline denominator
#pragma once
#include "rtz_device.cuh"

namespace rtz {

struct ShardGeom {
    uint32_t rank, world, tile_w, tile_h, tiles_x, tiles_y, n_local_tiles, tile_pixels;
};

struct TraceParams {
    DevCamera cam;
    ShardGeom sh;
    const float4* pairs;    // [n_pad]   sweep layout, spheres in pairs (A=2p, B=2p+1):
                            //           [2p] = {cxA,cxB,cyA,cyB}  [2p+1] = {czA,czB,wA,wB},  w = -(|c|^2 - r^2)
    const float4* geom;     // [n_pad]   per-lane lookups: {cx, cy, cz, -r^2}
    const float4* aux;      // [n_pad] {r, 1/r, fuzz|ior, type}
    const float4* albedo;   // [n_pad] {r,g,b,1/ior}
    const float* wexp;      // [n_pad] w of the pair layout as a plain row (per-lane lookups: coop_hit, the BVH extension)
    // The culled kernel and its drain sweep the spheres regrouped into compact blocks (rtz_scene_upload): the rows
    // above then hold that order, and orig[slot] is the sphere's index in the caller's list, which breaks exact ties
    // in t.  Null for every other kernel: slot = index.
    const int* orig;
    int n_spheres;
    int n_pad;              // n rounded up to a multiple of 8 (padding spheres can never be hit)
    // Work chunks = runs of `chunk` samples of ONE pixel (a warp's 64 paths then share their camera geometry: warps
    // fed with samples of different pixels measured 7-16 % slower), handed out by the global queue in index order.
    uint32_t chunk;         // samples per work chunk
    uint32_t chunks_per_pixel;
    uint32_t n_local_pixels;
    uint64_t n_chunks;      // n_local_pixels(padded) * chunks_per_pixel
    unsigned long long* accum;    // [n_local_pixels*3] 32.32 fixed-point colour sums
    unsigned long long* counter;  // work-queue head
    unsigned long long* stats;    // {samples, segments, depth_capped, absorbed, (BVH tests), NaN samples}
    // The drain pool.  A warp that needs new work after the queue has run dry does not keep sweeping all N spheres
    // for the few long paths it has left (64 slots for them, and nobody to share them with): it parks its live
    // paths here and retires; drain_kernel then finishes every parked path, one warp per path, spheres across lanes.
    float4* pool;                 // [pool_cap][4]: {o, |d|} {d, self} {throughput, bounce} {pixel, sample, local pixel, -}
    unsigned int* pool_count;     // paths parked (trace kernel) ; pool_count[1] = next path to hand out (drain kernel)
    unsigned long long* timeline; // diagnostics (RTZ_TIMELINE=1), else null: per warp {start, queue ran dry, done} in ns, SM id
    // trace_kernel_wave only: a shading / regeneration pass over fewer than this many paths is put off to the next
    // iteration (1 = never put off, 32 = full passes only); the host derives both from the cost of a sweep
    uint32_t wave_shade_min, wave_regen_min;
    // ... and the divisors of its chunk bookkeeping as 64-bit reciprocals (ceil(2^64 / d), 0 for d = 1): a chunk of a
    // 64-spp frame lasts two regeneration passes, and four 32-bit divisions per chunk were 5 % of the kernel
    unsigned long long rcp_tile_pixels, rcp_tiles_x, rcp_tile_w, rcp_chunks_per_pixel;
};

// Scenes of up to kMaxConstSpheres spheres travel as a __grid_constant__ kernel parameter: the
// sweep then reads them through the constant bank with uniform loads (LDCU -> uniform registers
// -> UR operands of FADD2/FFMA2), which needs no LDS, no vector registers and no shared memory.
constexpr int kMaxConstSpheres = 512;  // 8 KiB: what the constant cache serves at full rate (1024 spheres already thrash it: measured)
struct TraceParamsConst {
    TraceParams p;
    float4 pairs[kMaxConstSpheres];
    // trace_kernel_const<.., true> only: the padded box of every 32-sphere block of the sweep,
    // [2b] = {lo.x, hi.x, lo.y, hi.y}, [2b+1] = {lo.z, hi.z, 0, 0} (block 0 is always swept), and the squared
    // distance from the world origin beyond which a ray origin was not accounted for in the padding
    float4 boxes[2 * (kMaxConstSpheres / 32)];
    float cull_r2;
    // a culled block that at most this many of the warp's 64 paths reach is swept sphere-parallel (sweep2)
    int split_max;
};
constexpr int kSplitMax = 16;

// local (compact, padded) pixel index -> global pixel; false for tile padding
__device__ __forceinline__ bool local_to_global(const ShardGeom& s, uint32_t W, uint32_t H, uint32_t lp, uint32_t& x,
                                                uint32_t& y) {
    const uint32_t lt = lp / s.tile_pixels, within = lp - lt * s.tile_pixels;
    const uint32_t gt = lt * s.world + s.rank;
    const uint32_t ty = gt / s.tiles_x, tx = gt - ty * s.tiles_x;
    const uint32_t wy = within / s.tile_w, wx = within - wy * s.tile_w;
    x = tx * s.tile_w + wx, y = ty * s.tile_h + wy;
    return x < W && y < H && ty < s.tiles_y;
}

// the same with the divisions by launch constants done as multiplications: for n, d < 2^32 and M = ceil(2^64 / d),
// floor(n / d) = floor(n * M / 2^64) exactly (the excess n * (M - 2^64 / d) / 2^64 is below 2^-32 < 1 / d)
__device__ __forceinline__ uint32_t div_by(uint32_t n, unsigned long long rcp) {
    return rcp ? (uint32_t)__umul64hi((unsigned long long)n, rcp) : n;
}
__device__ __forceinline__ bool local_to_global_rcp(const ShardGeom& s, unsigned long long rcp_tile_pixels,
                                                    unsigned long long rcp_tiles_x, unsigned long long rcp_tile_w, uint32_t W,
                                                    uint32_t H, uint32_t lp, uint32_t& x, uint32_t& y) {
    const uint32_t lt = div_by(lp, rcp_tile_pixels), within = lp - lt * s.tile_pixels;
    const uint32_t gt = lt * s.world + s.rank;
    const uint32_t ty = div_by(gt, rcp_tiles_x), tx = gt - ty * s.tiles_x;
    const uint32_t wy = div_by(within, rcp_tile_w), wx = within - wy * s.tile_w;
    x = tx * s.tile_w + wx, y = ty * s.tile_h + wy;
    return x < W && y < H && ty < s.tiles_y;
}

// --- 1-D TMA (cp.async.bulk) staging of the scene into shared memory ---------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(phase)
        : "memory");
}

// ---------------------------------------------------------------------------------------------
// K1: persistent path-trace megakernel.
//
// Work = the rank's (pixel, sample) pairs, pixel-major, cut into chunks of <= P.chunk samples of
// ONE pixel; chunks are handed out by a global atomic queue.  Every thread keeps TWO paths in
// flight (slots A and B), so a warp advances 64 paths in lockstep: one loop iteration is one
// world.hit for every live path.  A path that ended takes the next sample of the warp's current
// chunk at once (path regeneration), so the sphere sweep — 99 % of the work — always runs with
// full warps except while the queue drains.
//
// The sweep tests ONE path against a PAIR of spheres per packed FP32x2 instruction (FFMA2 / FADD2, new on
// sm_100): per sphere pair and path 7 FFMA2 + 1 FADD2 + 2 funnel shifts that append the discriminants'
// sign bits to the path's candidate mask, plus 4 uniform loads (LDCU.64) shared by the paths of the
// thread.  Measured on B200 (tools/ubench/sweep_ops.cu, shadow.cu, ldcu_cost.cu): a packed op holds the
// FMA pipe for 2.06 cycles and every other instruction of the loop still costs 0.3-0.75 issue cycles in
// its shadow, so the loop runs at 10.4 cycles per ray-sphere test against 8 for the packed ops alone.
// Roots are only evaluated for the mask's candidates, in ascending sphere order, after each block of
// 32 spheres.
//
// Finished samples are converted to 32.32 fixed point and added to the pixel with 64-bit integer
// REDs; integer addition commutes, so the image is bit-identical for any schedule, tile size or
// GPU count.
// ---------------------------------------------------------------------------------------------
struct Slot {
    Path path;
    RngKey key;
    uint32_t lp;  // local pixel (accumulator index)
    bool alive;
};


// evaluate the candidates of one 32-sphere block for one path: Sphere.hit's root selection
// (src/sphere.zig:35-42) with the shrinking t_max of HittableList.hit (src/hittable.zig:66-73).
// `gather[i]` = {cx, cy, cz, -r^2} serves the per-lane (divergent) lookups.
__device__ __forceinline__ void resolve_candidates(const float4* __restrict__ gather, unsigned cand, int base, int cnt,
                                                   const Path& p, float tmin_d, float& closest, int& best,
                                                   const int* __restrict__ orig = nullptr) {
    while (cand) {
        const int bit = 31 - __clz(cand);  // highest bit = lowest sphere index: ascending order
        cand &= ~(1u << bit);
        const int i = base + (cnt - 1 - bit);
        const float4 g = gather[i];
        candidate_root(g, g.w, i, p, tmin_d, closest, best, orig);
    }
}

// One path against one PAIR of spheres: 7 FFMA2 + 1 FADD2 = two ray-sphere tests (17 algorithmic
// FLOP each).  The ray constants are scalar-broadcast operands (R.F32), the sphere pair is the
// packed operand; this orientation needs fewer register-file reads per FFMA2 than packing two rays
// (tools/ubench/sweep_shapes.cu), and on sm_100 the register file, not the FMA pipe, is what bounds
// a packed instruction with several distinct register operands (tools/ubench/ffma2_patterns.cu).
__device__ __forceinline__ void test_pair(const float4 p0, const float4 p1, const Path& p, const RayK& k,
                                          unsigned& mask) {
    const float2 cx = make_float2(p0.x, p0.y), cy = make_float2(p0.z, p0.w);
    const float2 cz = make_float2(p1.x, p1.y), cw = make_float2(p1.z, p1.w);
    float2 h = __ffma2_rn(make_float2(p.dx, p.dx), cx, make_float2(k.k1, k.k1));
    h = __ffma2_rn(make_float2(p.dy, p.dy), cy, h);
    h = __ffma2_rn(make_float2(p.dz, p.dz), cz, h);
    float2 w = __ffma2_rn(make_float2(k.tx, k.tx), cx, make_float2(k.nk2, k.nk2));
    w = __ffma2_rn(make_float2(k.ty, k.ty), cy, w);
    w = __ffma2_rn(make_float2(k.tz, k.tz), cz, w);
    w = __fadd2_rn(w, cw);
    const float2 disc = __ffma2_rn(h, h, w);
    mask = __funnelshift_l(__float_as_uint(disc.x), mask, 1);  // append sign(disc): sphere 2p ...
    mask = __funnelshift_l(__float_as_uint(disc.y), mask, 1);  // ... then sphere 2p+1
}

// Can the segment (0, closest] of a path reach the padded box of a block?  Slab test; `ix, iy, iz` = 1 / d.
//
// Exactness contract of the block cull: a lane may report "no" only if the FP32 pipeline (sign of the expanded
// discriminant, then the direct-form root in (t_min * |d|, closest)) would accept no sphere of the block.
//  * An accepted root lies inside the padded box.  Acceptance is decided by the direct form, whose disc is off by at
//    most about 12 eps |c - o|^2 (eps = 2^-24); the expanded gate in front of it only filters and, with its margin
//    (kGateSlack), never rejects what the direct form accepts.  So an accepted point p = o + t d — a self hit,
//    o + 2 h d, included — has |p - c|^2 <= r^2 + 24 eps |c - o|^2: |p - c| <= r + 12 eps |c - o|^2 / r.  The host
//    pads every sphere by 1e-6 (1.001 R + |c|)^2 / r for |o| <= R (1e-6 > 16 eps) on top of the BVH builder's
//    1e-4 (1 + r + |c|_1); a ray starting farther out than R (|o|^2 > cull_r2) needs every block.  The origin test
//    reads -nk2 = |o|^2 (1 - 2^-18), i.e. it admits |o| up to R (1 + 2e-6), well inside the 1.001 R of the padding.
//  * The test itself errs towards "yes": the interval is [0, closest], a superset of (t_min |d|, closest), and
//    compared with <=, never strictly; an accepted point sits at least the padding inside every face, far beyond
//    the few ulps of (lo - o) * (1 / d); fminf / fmaxf drop the NaN of 0 * inf (an axis-parallel ray in the plane
//    of a face), which is then outside the box by the padding; an origin inside the box gives t_near = 0 <= t_far.
// The contract is per path, so sweep2 may leave a path out of a block whose box it does not reach: the sphere-parallel
// pass tests only the paths that reach the block, and the packed sweep tests every path of the warp, and both give
// the same hits.  The two evaluate the same candidate gate (expanded_disc is test_pair's FMA sequence, one sphere at a
// time) and resolve the candidates with resolve_candidates in ascending slot order, so the hit is still the
// (t, original index) minimum whichever of the two swept a block.
__device__ __forceinline__ bool box_reach(const float4 b0, const float4 b1, const Path& p, float ix, float iy, float iz,
                                          float closest) {
    const float2 tx = __fmul2_rn(__fadd2_rn(make_float2(b0.x, b0.y), make_float2(-p.ox, -p.ox)), make_float2(ix, ix));
    const float2 ty = __fmul2_rn(__fadd2_rn(make_float2(b0.z, b0.w), make_float2(-p.oy, -p.oy)), make_float2(iy, iy));
    const float2 tz = __fmul2_rn(__fadd2_rn(make_float2(b1.x, b1.y), make_float2(-p.oz, -p.oz)), make_float2(iz, iz));
    const float tn = fmaxf(fmaxf(fminf(tx.x, tx.y), fminf(ty.x, ty.y)), fmaxf(fminf(tz.x, tz.y), 0.0f));
    const float tf = fminf(fminf(fmaxf(tx.x, tx.y), fmaxf(ty.x, ty.y)), fminf(fmaxf(tz.x, tz.y), closest));
    return tn <= tf;
}

// a shared-memory load the compiler cannot forward from an earlier store (so the stored value need not stay live)
__device__ __forceinline__ float4 lds_opaque(const float4* p) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p))
                 : "memory");
    return v;
}

// The sphere-parallel candidate test of one block: lane l holds sphere base + l ({cx, cy, cz} of `g`, and w), and
// each path in `need` (bit l = the path of lane l) is read back from `stage` (its ray constants and direction, two
// float4 at a uniform address) and tested against all of them at once.  The path's lane gets the ballot of the
// spheres that pass the gate: bit l = sphere base + l.
__device__ __forceinline__ unsigned split_candidates(const float4* __restrict__ stage, unsigned need, const float4 g,
                                                     float w, unsigned lane) {
    unsigned cand = 0u;
    while (need) {
        const unsigned src = __ffs(need) - 1;
        need &= need - 1u;
        const float4 s0 = stage[2 * src], s1 = stage[2 * src + 1];
        Path q;
        q.dx = s1.y, q.dy = s1.z, q.dz = s1.w;
        const RayK k{s0.x, s0.y, s0.z, s0.w, s1.x};
        const float d = expanded_disc(g.x, g.y, g.z, w, q, k);
        const unsigned pass = __ballot_sync(0xFFFFFFFFu, !(__float_as_uint(d) >> 31));
        if (lane == src) cand = pass;
    }
    return cand;
}

// HittableList.hit for the two paths of a thread.  `pairs` is warp-uniform storage (shared memory
// or the constant bank): per sphere pair 2 LDS.128 + 2 x (7 FFMA2 + 1 FADD2 + 2 SHF) for FOUR tests.
// n_pad is a multiple of 8; padding spheres have w = -inf -> disc = -inf -> never a candidate.
// kConstBank selects two register-allocation nudges that were measured per kernel (same arithmetic):
// the constant-bank kernel pins 2*o (+0.8 %), the shared-memory kernel forms t_min*len late (+4 % at N = 1024).
// (Deferring the candidates of several blocks to per-lane lists and resolving them together was built twice and
// measured on one box: +3.7 % warp-instructions, +0.4 % time.  The 64 paths of a warp come from one pixel, so
// their candidates coincide and one pass per non-empty block already serves all lanes.)
// kCull (constant-bank lockstep kernel): a block of 32 spheres that no path of the warp can reach over (0, closest]
// is skipped as a whole — a warp-uniform branch, so the loop stays on the uniform datapath.  Block 0 (the ground of
// the book's scenes) is always swept first, which gives most paths a short closest hit before the bounds are tested.
// The packed sweep costs the same whether 1 or 64 paths reach a block.  So a culled block that at most `split_max` of
// the warp's 64 paths reach is swept sphere-parallel instead: lane l takes sphere base + l, and each reaching path's
// ray constants are broadcast from the warp's staging rows (`stage`, written once per call) for one expanded_disc
// and one ballot, which the path's lane keeps as its candidate mask.
template <bool kConstBank, bool kSkipSelf = false, bool kCull = false>
__device__ __forceinline__ void sweep2(const float4* __restrict__ pairs, const float4* __restrict__ gather, int n_pad,
                                       float tmin, float tmax, const Path& a, const Path& b, float& ta, int& ia,
                                       float& tb, int& ib, const float4* __restrict__ boxes = nullptr,
                                       float cull_r2 = 0.0f, const int* __restrict__ orig = nullptr,
                                       const float* __restrict__ wexp = nullptr, int split_max = 0,
                                       float4* __restrict__ stage = nullptr) {
    RayK ka = ray_constants(a), kb = ray_constants(b);
    // pin 2*o in registers: left alone, ptxas keeps o and re-adds it for every block of 32 spheres (not in the culled
    // sweep: its six reciprocals need those registers, and with the pin it spills under the 80-register cap)
    if (kConstBank && !kCull) asm volatile("" : "+f"(ka.tx), "+f"(ka.ty), "+f"(ka.tz), "+f"(kb.tx), "+f"(kb.ty), "+f"(kb.tz));
    // Interval(t_min, t_max) of Scene.interval in distance units (directions are unit length)
    float ca = tmax * a.len, cb = tmax * b.len;
    int ba = -1, bb = -1;
    float iax = 0.f, iay = 0.f, iaz = 0.f, ibx = 0.f, iby = 0.f, ibz = 0.f;
    if (kCull) {
        // an origin the padding does not cover (|o|^2 > cull_r2) gets NaN reciprocals: box_reach then sees the whole
        // segment [0, closest] and the path needs every block (no predicate register held across the sweep)
        iax = 1.0f / a.dx, iay = 1.0f / a.dy, iaz = 1.0f / a.dz;
        ibx = 1.0f / b.dx, iby = 1.0f / b.dy, ibz = 1.0f / b.dz;
        if (!(-ka.nk2 <= cull_r2)) iax = iay = iaz = __int_as_float(0x7fffffff);
        if (!(-kb.nk2 <= cull_r2)) ibx = iby = ibz = __int_as_float(0x7fffffff);
    }
    if (kCull) {
        // the warp's staging rows: path j (32 + lane for slot B) at stage[2j], stage[2j + 1], which the sphere-parallel
        // pass broadcasts, and the lane's reciprocals at stage[128 + 2 lane], stage[129 + 2 lane]
        const unsigned lane = threadIdx.x & 31u;
        stage[2 * lane] = make_float4(ka.k1, ka.nk2, ka.tx, ka.ty);
        stage[2 * lane + 1] = make_float4(ka.tz, a.dx, a.dy, a.dz);
        stage[2 * lane + 64] = make_float4(kb.k1, kb.nk2, kb.tx, kb.ty);
        stage[2 * lane + 65] = make_float4(kb.tz, b.dx, b.dy, b.dz);
        stage[2 * lane + 128] = make_float4(iax, iay, iaz, 0.f);
        stage[2 * lane + 129] = make_float4(ibx, iby, ibz, 0.f);
        __syncwarp();
    }
    for (int base = 0; base < n_pad; base += 32) {
        unsigned canda, candb;
        unsigned need_a = 0u, need_b = 0u;
        if (kCull && base > 0) {
            const float4 b0 = boxes[base >> 4], b1 = boxes[(base >> 4) + 1];
            need_a = __ballot_sync(0xFFFFFFFFu, box_reach(b0, b1, a, iax, iay, iaz, ca));
            need_b = __ballot_sync(0xFFFFFFFFu, box_reach(b0, b1, b, ibx, iby, ibz, cb));
            if ((need_a | need_b) == 0u) continue;
        }
        const int cnt = min(32, n_pad - base);
        if (kCull && base > 0 && __popc(need_a) + __popc(need_b) <= split_max) {
            const unsigned lane = threadIdx.x & 31u;
            // lanes >= cnt (the last block of a scene whose n_pad is not a multiple of 32) test a repeated sphere:
            // their ballot bits are shifted out below
            const int i = min(base + (int)lane, n_pad - 1);
            const float4 g = gather[i];
            const float w = __ldg(wexp + i);
            canda = split_candidates(stage, need_a, g, w, lane);
            candb = split_candidates(stage + 64, need_b, g, w, lane);
            canda = __brev(canda) >> (32 - cnt);  // sphere base + i at bit cnt - 1 - i, as the packed sweep leaves it
            candb = __brev(candb) >> (32 - cnt);
            // the lane's own ray constants and reciprocals are read back instead of being held across this branch
            // (the kernel runs at 80 registers)
            const float4 a0 = lds_opaque(stage + 2 * lane), a1 = lds_opaque(stage + 2 * lane + 1);
            const float4 b0 = lds_opaque(stage + 2 * lane + 64), b1 = lds_opaque(stage + 2 * lane + 65);
            const float4 ra = lds_opaque(stage + 2 * lane + 128), rb = lds_opaque(stage + 2 * lane + 129);
            ka = RayK{a0.x, a0.y, a0.z, a0.w, a1.x}, kb = RayK{b0.x, b0.y, b0.z, b0.w, b1.x};
            iax = ra.x, iay = ra.y, iaz = ra.z, ibx = rb.x, iby = rb.y, ibz = rb.z;
        } else {
            unsigned ma = 0xFFFFFFFFu, mb = 0xFFFFFFFFu;  // 1 = miss
            const float4* g = pairs + base;
#pragma unroll 1
            for (int k = 0; k < cnt; k += 8) {
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    const float4 p0 = g[k + u], p1 = g[k + u + 1];
                    test_pair(p0, p1, a, ka, ma);
                    test_pair(p0, p1, b, kb, mb);
                }
            }
            canda = ~ma, candb = ~mb;
        }
        if (kSkipSelf) {  // a ray that leaves its sphere outwards (shade<true> flagged it) cannot hit it: not a candidate
            const unsigned ra = (unsigned)(a.self & ~kSelfLeaves) - (unsigned)base, rb = (unsigned)(b.self & ~kSelfLeaves) - (unsigned)base;
            if ((a.self >> 30) == 1 && ra < (unsigned)cnt) canda &= ~(1u << (cnt - 1 - (int)ra));
            if ((b.self >> 30) == 1 && rb < (unsigned)cnt) candb &= ~(1u << (cnt - 1 - (int)rb));
        }
        if (canda | candb) {
            // t_min * len is formed HERE, behind an opaque copy, so that it does not occupy two more
            // registers across the whole sweep of the shared-memory kernel (96 registers at 5 CTAs per SM)
            float la = a.len, lb = b.len;
            if (!kConstBank) asm volatile("" : "+f"(la), "+f"(lb));
            resolve_candidates(gather, canda, base, cnt, a, tmin * la, ca, ba, orig);
            resolve_candidates(gather, candb, base, cnt, b, tmin * lb, cb, bb, orig);
        }
    }
    ta = ca, ia = ba, tb = cb, ib = bb;
}

__device__ __forceinline__ void finish_or_continue(const TraceParams& P, const float4* gather, const float4* s_aux,
                                                   const float4* s_alb, Slot& s, float t, int best,
                                                   unsigned long long& n_seg, uint32_t& n_samp, uint32_t& n_cap,
                                                   uint32_t& n_abs) {
    ++n_seg;
    float sr, sg, sb;
    int term;
    if (shade(P.cam, s.key, gather, s_aux, s_alb, s.path, t, best, sr, sg, sb, term)) {
        const unsigned long long fr = to_fixed(sr), fg = to_fixed(sg), fb = to_fixed(sb);
        unsigned long long* px = P.accum + 3ull * s.lp;
        if (fr) atomicAdd(px + 0, fr);
        if (fg) atomicAdd(px + 1, fg);
        if (fb) atomicAdd(px + 2, fb);
        if (sr != sr || sg != sg || sb != sb) atomicAdd(P.stats + 5, 1ULL);  // NaN sample: adds 0, but is counted
        ++n_samp;
        n_cap += (term == 2), n_abs += (term == 1);
        s.alive = false;
    }
}

// The same for trace_body, which keeps no per-lane work counters (every register counts at 80 per thread):
// segments and samples are counted per warp from the live-slot votes, the two rare endings go straight to global
// memory.
__device__ __forceinline__ void finish_or_continue(const TraceParams& P, const float4* gather, const float4* s_aux,
                                                   const float4* s_alb, Slot& s, float t, int best) {
    float sr, sg, sb;
    int term;
    if (shade(P.cam, s.key, gather, s_aux, s_alb, s.path, t, best, sr, sg, sb, term)) {
        const unsigned long long fr = to_fixed(sr), fg = to_fixed(sg), fb = to_fixed(sb);
        unsigned long long* px = P.accum + 3ull * s.lp;
        if (fr) atomicAdd(px + 0, fr);
        if (fg) atomicAdd(px + 1, fg);
        if (fb) atomicAdd(px + 2, fb);
        if (sr != sr || sg != sg || sb != sb) atomicAdd(P.stats + 5, 1ULL);  // NaN sample: adds 0, but is counted
        if (term == 2) atomicAdd(P.stats + 2, 1ULL);  // depth cap: 0.02 % of the samples
        if (term == 1) atomicAdd(P.stats + 3, 1ULL);  // absorbed by a metal: 0.2 %
        s.alive = false;
    }
}

// The body shared by the two kernels below.  `geo` is the warp-uniform geometry the sweep reads,
// `gather` the copy for per-lane lookups (candidate roots, hit records).
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// HittableList.hit for ONE path by the whole warp: lane l tests spheres l, l + 32, ... with the arithmetic of the
// sweep (sign of the expanded discriminant, then the direct-form root, ascending within the lane), and the
// closest hit is the warp's minimum over (t, sphere index).  That is the hit of the ascending loop: a sphere is
// accepted iff its root beats every earlier one strictly, so the winner is the smallest t and, among equal t, the
// smallest index — independent of how the spheres are dealt to the lanes (the BVH extension relies on the same
// fact).  Used while the queue drains: a warp that is down to a few live paths would otherwise sweep all N
// spheres with 64 slots for them, 6.5 us per bounce on an empty SM (measured with RTZ_TIMELINE: the last 1 % of
// the warps used to finish 0.4 ms after the other 99 %).  The discriminants of 8 spheres per lane are evaluated
// back to back so that their loads overlap (the rows are cold in L1: the sweep reads the constant bank).
// `orig` (null = identity): the rows are in another order than the caller's list; ties go by original index.
template <bool kUniform = false>  // kUniform: every lane already holds the path and wants the result
__device__ __forceinline__ void coop_hit(const float4* __restrict__ geom, const float* __restrict__ wexp,
                                         const int* __restrict__ orig, int n, float tmin, float tmax, const Path& mine,
                                         int src, unsigned lane, float& t_out, int& best_out) {
    Path q = mine;
    if (!kUniform) {
        q.ox = __shfl_sync(0xFFFFFFFFu, mine.ox, src), q.oy = __shfl_sync(0xFFFFFFFFu, mine.oy, src);
        q.oz = __shfl_sync(0xFFFFFFFFu, mine.oz, src), q.dx = __shfl_sync(0xFFFFFFFFu, mine.dx, src);
        q.dy = __shfl_sync(0xFFFFFFFFu, mine.dy, src), q.dz = __shfl_sync(0xFFFFFFFFu, mine.dz, src);
        q.len = __shfl_sync(0xFFFFFFFFu, mine.len, src), q.self = __shfl_sync(0xFFFFFFFFu, mine.self, src);
    }
    const float tmin_d = tmin * q.len;
    float closest = tmax * q.len;
    int best = -1;
    const RayK k = ray_constants(q);
    for (int base = (int)lane; base < n; base += 256) {  // 8 spheres per lane and round
        unsigned cand = 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = base + 32 * j;
            if (i < n) {
                const float4 g = __ldg(geom + i);
                const float d = expanded_disc(g.x, g.y, g.z, __ldg(wexp + i), q, k);
                cand |= (__float_as_uint(d) >> 31 ^ 1u) << j;
            }
        }
        while (cand) {  // ascending
            const int j = __ffs(cand) - 1;
            cand &= cand - 1u;
            const int i = base + 32 * j;
            const float4 g = __ldg(geom + i);
            candidate_root(g, g.w, i, q, tmin_d, closest, best, orig);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float t2 = __shfl_xor_sync(0xFFFFFFFFu, closest, o);
        const int b2 = __shfl_xor_sync(0xFFFFFFFFu, best, o);
        // on equal t the lower (original) index wins; -1 = none loses
        const bool tie_won = t2 == closest && b2 >= 0 && (best < 0 || (orig ? __ldg(orig + b2) < __ldg(orig + best) : b2 < best));
        if (t2 < closest || tie_won) closest = t2, best = b2;
    }
    if (kUniform || (int)lane == src) t_out = closest, best_out = best;
}

__device__ __forceinline__ void park_path(float4* __restrict__ e, const Slot& s) {
    const Path& p = s.path;
    e[0] = make_float4(p.ox, p.oy, p.oz, p.len);
    e[1] = make_float4(p.dx, p.dy, p.dz, __int_as_float(p.self));
    e[2] = make_float4(p.tr, p.tg, p.tb, __uint_as_float(p.bounce));
    e[3] = make_float4(__uint_as_float(s.key.pixel), __uint_as_float(s.key.sample), __uint_as_float(s.lp), 0.f);
}
__device__ __forceinline__ void unpark_path(const float4* __restrict__ e, uint32_t k0, uint32_t k1, Slot& s) {
    const float4 a = e[0], b = e[1], c = e[2], d = e[3];
    Path& p = s.path;
    p.ox = a.x, p.oy = a.y, p.oz = a.z, p.len = a.w;
    p.dx = b.x, p.dy = b.y, p.dz = b.z, p.self = __float_as_int(b.w);
    p.tr = c.x, p.tg = c.y, p.tb = c.z, p.bounce = __float_as_uint(c.w);
    s.key = RngKey{k0, k1, __float_as_uint(d.x), __float_as_uint(d.y)};
    s.lp = __float_as_uint(d.z);
    s.alive = true;
}

// a staged camera ray (trace_body's warp-cooperative regeneration): origin, unit direction, |direction|
__device__ __forceinline__ void take_camera_ray(const float* stage, uint32_t j, Path& p) {
    p.ox = stage[0 * 64 + j], p.oy = stage[1 * 64 + j], p.oz = stage[2 * 64 + j];
    p.dx = stage[3 * 64 + j], p.dy = stage[4 * 64 + j], p.dz = stage[5 * 64 + j];
    p.len = stage[6 * 64 + j];
    p.tr = p.tg = p.tb = 1.0f;
    p.self = -1;
    p.bounce = 0;
}
constexpr int kStageFloats = 7 * 64;  // per warp: 7 rows (origin, unit direction, |direction|) of 64 rays (two slots per lane)
// the culled kernel's rows also hold, during the sweep, the 8 ray constants of each of the 64 paths and the 6
// reciprocals of each lane (sweep2)
constexpr int kCullStageFloats = 12 * 64;

// the warp's diagnostics row of P.timeline, formed where it is written: the opaque read of the block index keeps the
// compiler from holding the 64-bit pointer in registers across the whole trace loop
template <int kBlock>
__device__ __forceinline__ unsigned long long* timeline_row(const TraceParams& P) {
    unsigned cta;
    asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(cta));
    return P.timeline + 4ull * ((unsigned long long)cta * (kBlock / 32) + (threadIdx.x >> 5));
}

template <bool kConstBank, int kBlock, bool kCull = false>
__device__ __forceinline__ void trace_body(const TraceParams& P, const float4* __restrict__ pairs,
                                           const float4* __restrict__ gather, float* __restrict__ stage_mem,
                                           const float4* __restrict__ boxes = nullptr, float cull_r2 = 0.0f,
                                           int split_max = 0) {
    float* const stage = stage_mem + (threadIdx.x >> 5) * (kCull ? kCullStageFloats : kStageFloats);
    if (P.timeline && (threadIdx.x & 31u) == 0u) timeline_row<kBlock>(P)[0] = globaltimer_ns();
    // material rows are touched once per HIT (not per test): they stay in global memory / L1
    const float4* s_aux = P.aux;
    const float4* s_alb = P.albedo;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DevCamera& cam = P.cam;

    Slot A, B;
    A.alive = B.alive = false;
    A.lp = B.lp = 0;
    A.key = B.key = RngKey{cam.key0, cam.key1, 0u, 0u};
    A.path.ox = A.path.oy = A.path.oz = 0.f, A.path.dx = A.path.dy = 0.f, A.path.dz = 1.f;
    A.path.tr = A.path.tg = A.path.tb = 0.f, A.path.len = 1.f, A.path.self = -1, A.path.bounce = 0;
    B.path = A.path;

    // warp-uniform chunk state (parking it in shared memory between regenerations was tried: ptxas then no longer
    // treats the branches on it as uniform and the sweep leaves the uniform datapath)
    uint32_t ch_lp = 0, ch_x = 0, ch_y = 0, ch_next = 0, ch_end = 0;
    bool exhausted = false;

    // work counters, per warp, from the votes: a slot that was live and is free now has finished a sample
    unsigned long long n_seg = 0;
    uint32_t n_samp = 0;
    unsigned prev_a = 0u, prev_b = 0u;

    for (;;) {
        unsigned need_a = __ballot_sync(0xFFFFFFFFu, !A.alive);
        unsigned need_b = __ballot_sync(0xFFFFFFFFu, !B.alive);
        n_samp += __popc(prev_a & need_a) + __popc(prev_b & need_b);
        if (need_a | need_b) {
            while ((need_a | need_b) && !exhausted) {
                if (ch_next >= ch_end) {
                    unsigned long long cid = 0;
                    if (lane == 0) cid = atomicAdd(P.counter, 1ULL);
                    cid = __shfl_sync(0xFFFFFFFFu, cid, 0);
                    // the conditions below are the same in every lane; voting on them makes that
                    // visible to ptxas (uniform branches keep the warp provably converged)
                    if (__any_sync(0xFFFFFFFFu, cid >= P.n_chunks)) {
                        exhausted = true;
                        if (P.timeline && lane == 0u) timeline_row<kBlock>(P)[1] = globaltimer_ns();
                        break;
                    }
                    // (the chunk is committed only behind the `continue`: written the other way round ptxas no
                    // longer proves the loop converged and the sweep leaves the uniform datapath)
                    const uint32_t lp = (uint32_t)(cid / P.chunks_per_pixel);
                    const uint32_t part = (uint32_t)(cid - (unsigned long long)lp * P.chunks_per_pixel);
                    uint32_t x, y;
                    const bool inside = local_to_global(P.sh, cam.width, cam.height, lp, x, y);
                    if (__any_sync(0xFFFFFFFFu, !inside)) continue;  // tile padding
                    ch_lp = lp, ch_x = x, ch_y = y;
                    ch_next = part * P.chunk;
                    ch_end = min(ch_next + P.chunk, cam.spp);
                }
                const uint32_t avail = ch_end - ch_next;
                const uint32_t na = __popc(need_a);
                const uint32_t rank_a = __popc(need_a & lt_mask);
                const uint32_t rank_b = na + __popc(need_b & lt_mask);
                const uint32_t n_gen = min(na + (uint32_t)__popc(need_b), avail);
                // Camera rays, warp-cooperative: the chunk's next n_gen samples are generated 32 at a time by ALL
                // lanes into the warp's staging rows and then picked up by the lanes that own the free slots.
                // Which lane computes a ray does not matter — its random numbers depend on (pixel, sample) only —
                // and one full-width pass replaces two passes of ~7 active lanes each (ncu: 28 % of the kernel's
                // warp-instructions at 16 spheres, profiles/r2_*).
                const uint32_t pix = ch_y * cam.width + ch_x;
                for (uint32_t j0 = 0; j0 < n_gen; j0 += 32u) {
                    const uint32_t j = j0 + lane;
                    if (j < n_gen) {
                        const RngKey key{cam.key0, cam.key1, pix, ch_next + j};
                        Path t;
                        camera_ray(cam, key, ch_x, ch_y, t);
                        stage[0 * 64 + j] = t.ox, stage[1 * 64 + j] = t.oy, stage[2 * 64 + j] = t.oz;
                        stage[3 * 64 + j] = t.dx, stage[4 * 64 + j] = t.dy, stage[5 * 64 + j] = t.dz;
                        stage[6 * 64 + j] = t.len;
                    }
                }
                __syncwarp();
                if (((need_a >> lane) & 1u) && rank_a < n_gen) {
                    A.lp = ch_lp;
                    A.key.pixel = pix, A.key.sample = ch_next + rank_a;
                    take_camera_ray(stage, rank_a, A.path);
                    A.alive = true;
                }
                if (((need_b >> lane) & 1u) && rank_b < n_gen) {
                    B.lp = ch_lp;
                    B.key.pixel = pix, B.key.sample = ch_next + rank_b;
                    take_camera_ray(stage, rank_b, B.path);
                    B.alive = true;
                }
                __syncwarp();  // the rows are rewritten by the next round
                ch_next += n_gen;
                need_a = __ballot_sync(0xFFFFFFFFu, !A.alive);
                need_b = __ballot_sync(0xFFFFFFFFu, !B.alive);
            }
        }
        if (exhausted && P.pool) {
            // no more work to hand out: park what is still in flight for drain_kernel and retire
            const unsigned pa = __ballot_sync(0xFFFFFFFFu, A.alive), pb = __ballot_sync(0xFFFFFFFFu, B.alive);
            unsigned base = 0u;
            if (lane == 0u) base = atomicAdd(P.pool_count, (unsigned)(__popc(pa) + __popc(pb)));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (A.alive) park_path(P.pool + 4ull * (base + __popc(pa & lt_mask)), A);
            if (B.alive) park_path(P.pool + 4ull * (base + __popc(pa) + __popc(pb & lt_mask)), B);
            break;
        }
        // loop exit on a FRESH warp vote: the condition is warp-uniform by construction, which lets
        // ptxas keep the sweep below on the uniform datapath (uniform loads / UR operands)
        const unsigned live_a = __ballot_sync(0xFFFFFFFFu, A.alive), live_b = __ballot_sync(0xFFFFFFFFu, B.alive);
        if ((live_a | live_b) == 0u) break;  // queue drained, every path finished
        n_seg += (unsigned)(__popc(live_a) + __popc(live_b));
        prev_a = live_a, prev_b = live_b;
        float ta = 0.f, tb = 0.f;
        int ia = -1, ib = -1;
        sweep2<kConstBank, false, kCull>(pairs, gather, P.n_pad, cam.tmin, cam.tmax, A.path, B.path, ta, ia, tb, ib,
                                         boxes, cull_r2, kCull ? P.orig : nullptr, P.wexp, split_max,
                                         reinterpret_cast<float4*>(stage));
        if (A.alive) finish_or_continue(P, gather, s_aux, s_alb, A, ta, ia);
        if (B.alive) finish_or_continue(P, gather, s_aux, s_alb, B, tb, ib);
        // explicit reconvergence point: with it ptxas proves the loop top converged (no BRA.DIV before
        // the votes) and keeps the sweep's addressing / constant-bank operands on the uniform datapath
        __syncwarp();
    }
    if (P.timeline && lane == 0u) {
        unsigned long long* const tl = timeline_row<kBlock>(P);
        unsigned smid;
        asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
        tl[2] = globaltimer_ns(), tl[3] = smid;
    }
    if (lane == 0u) {  // one atomic per warp and counter
        atomicAdd(P.stats + 0, (unsigned long long)n_samp);
        atomicAdd(P.stats + 1, n_seg);
    }
}

// ---------------------------------------------------------------------------------------------
// K1 with R paths per thread and the path state PARKED in shared memory.
//
// EXPERIMENTAL (RTZ_VARIANT=4; the two-path register kernel below stays the default).  The four LDCU.64
// of a sphere pair are shared by the R paths of a thread, so R = 4 brings the sweep loop from 10.4 to 9.7
// cycles per test in isolation.  Four paths need 4 x 8 sweep constants in registers, so everything the
// sweep does not read (origin, throughput, RNG counter, pixel, bounce) lives in shared memory, one word
// per (field, slot, thread): bank = thread, never a conflict, and the slot index may be a per-lane
// variable.  Shading runs ONE slot at a time through a single copy of its code; camera rays are
// generated by all lanes of the warp for whichever lane owns the free slot.  Measured on C3: the same
// 159 ms as the register kernel (the extra shared-memory traffic eats the saving of the loop), and the
// same bytes: tests/test_gpu_parity.py::test_image_is_independent_of_the_schedule.
// ---------------------------------------------------------------------------------------------
enum ParkField { kOx, kOy, kOz, kDx, kDy, kDz, kTr, kTg, kTb, kLen, kSelf, kBounce, kPixel, kSample, kLp, kParkFields };

template <int R, int kBlock>
struct Park {
    float* base;  // [kParkFields][R][kBlock]
    __device__ __forceinline__ float& f(int field, int slot) const {
        return base[(field * R + slot) * kBlock + threadIdx.x];
    }
    __device__ __forceinline__ uint32_t& u(int field, int slot) const {
        return reinterpret_cast<uint32_t*>(base)[(field * R + slot) * kBlock + threadIdx.x];
    }
    // re-read a parked word inside a rarely executed branch: `volatile` keeps the compiler from
    // holding the value in a register across the sweep instead
    __device__ __forceinline__ float fv(int field, int slot) const {
        return *reinterpret_cast<volatile float*>(&base[(field * R + slot) * kBlock + threadIdx.x]);
    }
    __device__ __forceinline__ void store_ray(int s, const Path& p) const {
        f(kOx, s) = p.ox, f(kOy, s) = p.oy, f(kOz, s) = p.oz;
        f(kDx, s) = p.dx, f(kDy, s) = p.dy, f(kDz, s) = p.dz;
        f(kTr, s) = p.tr, f(kTg, s) = p.tg, f(kTb, s) = p.tb;
        f(kLen, s) = p.len, u(kSelf, s) = (uint32_t)p.self, u(kBounce, s) = p.bounce;
    }
    __device__ __forceinline__ void load_ray(int s, Path& p) const {
        p.ox = f(kOx, s), p.oy = f(kOy, s), p.oz = f(kOz, s);
        p.dx = f(kDx, s), p.dy = f(kDy, s), p.dz = f(kDz, s);
        p.tr = f(kTr, s), p.tg = f(kTg, s), p.tb = f(kTb, s);
        p.len = f(kLen, s), p.self = (int)u(kSelf, s), p.bounce = u(kBounce, s);
    }
};

// what the sweep keeps in registers per path
struct Hot {
    float dx, dy, dz, k1, tx, ty, tz, nk2;
};

__device__ __forceinline__ void test_pair_hot(const float4 p0, const float4 p1, const Hot& q, unsigned& mask) {
    const float2 cx = make_float2(p0.x, p0.y), cy = make_float2(p0.z, p0.w);
    const float2 cz = make_float2(p1.x, p1.y), cw = make_float2(p1.z, p1.w);
    float2 h = __ffma2_rn(make_float2(q.dx, q.dx), cx, make_float2(q.k1, q.k1));
    h = __ffma2_rn(make_float2(q.dy, q.dy), cy, h);
    h = __ffma2_rn(make_float2(q.dz, q.dz), cz, h);
    float2 w = __ffma2_rn(make_float2(q.tx, q.tx), cx, make_float2(q.nk2, q.nk2));
    w = __ffma2_rn(make_float2(q.ty, q.ty), cy, w);
    w = __ffma2_rn(make_float2(q.tz, q.tz), cz, w);
    w = __fadd2_rn(w, cw);
    const float2 disc = __ffma2_rn(h, h, w);
    mask = __funnelshift_l(__float_as_uint(disc.x), mask, 1);
    mask = __funnelshift_l(__float_as_uint(disc.y), mask, 1);
}

template <int R, int kBlock>
__device__ __forceinline__ void trace_body_parked(const TraceParams& P, const float4* __restrict__ pairs,
                                                  const float4* __restrict__ gather, float* park_mem,
                                                  uint8_t* todo_mem) {
    const Park<R, kBlock> park{park_mem};
    uint8_t* todo = todo_mem + (threadIdx.x >> 5) * (32 * R);  // this warp's list of free slots
    const float4* s_aux = P.aux;
    const float4* s_alb = P.albedo;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DevCamera& cam = P.cam;
    constexpr unsigned kFull = (1u << R) - 1u;

    unsigned alive = 0;  // bit s = slot s carries a live path
    {
        Path idle;  // what a slot without a path sweeps (its result is ignored)
        idle.ox = idle.oy = idle.oz = 0.f, idle.dx = idle.dy = 0.f, idle.dz = 1.f;
        idle.tr = idle.tg = idle.tb = 0.f, idle.len = 1.f, idle.self = -1, idle.bounce = 0;
#pragma unroll
        for (int s = 0; s < R; ++s) park.store_ray(s, idle);
    }

    uint32_t ch_lp = 0, ch_x = 0, ch_y = 0, ch_next = 0, ch_end = 0;  // warp-uniform chunk state
    bool exhausted = false;
    unsigned long long n_seg = 0;
    uint32_t n_samp = 0, n_cap = 0, n_abs = 0;

    for (;;) {
        // ---- path regeneration, warp-cooperative: the free slots of the whole warp are ranked (slot-
        // major), published in `todo`, and the camera rays of the chunk's next samples are generated
        // 32 at a time by ALL lanes, each writing into the owner's parked slot.  Which lane computes a
        // ray does not matter: its random numbers depend on (pixel, sample) only.
        for (;;) {
            const unsigned dead = ~alive & kFull;
            unsigned bal[R];
            uint32_t total = 0;
#pragma unroll
            for (int s = 0; s < R; ++s) {
                bal[s] = __ballot_sync(0xFFFFFFFFu, (dead >> s) & 1u);
                total += __popc(bal[s]);
            }
            if (total == 0u || exhausted) break;
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
            const uint32_t n = min(total, ch_end - ch_next);
            uint32_t before = 0;
#pragma unroll
            for (int s = 0; s < R; ++s) {
                const uint32_t r = before + __popc(bal[s] & lt_mask);
                if (((dead >> s) & 1u) && r < n) {
                    todo[r] = (uint8_t)(lane | (s << 5));
                    alive |= 1u << s;
                }
                before += __popc(bal[s]);
            }
            __syncwarp();
            for (uint32_t j = lane; j < n; j += 32u) {
                const unsigned id = todo[j];
                const int owner = (int)(id & 31u) - (int)lane, s = (int)(id >> 5);  // owner as an offset from this thread
                const RngKey key{cam.key0, cam.key1, ch_y * cam.width + ch_x, ch_next + j};
                Path p;
                camera_ray(cam, key, ch_x, ch_y, p);
                const Park<R, kBlock> dst{park_mem + owner};
                dst.store_ray(s, p);
                dst.u(kPixel, s) = key.pixel, dst.u(kSample, s) = key.sample, dst.u(kLp, s) = ch_lp;
            }
            ch_next += n;
            __syncwarp();
        }
        if (__ballot_sync(0xFFFFFFFFu, alive != 0u) == 0u) break;  // queue drained, every path finished

        // ---- HittableList.hit for the R paths of the thread ----
        Hot hot[R];
        float closest[R];
        int best[R];
#pragma unroll
        for (int s = 0; s < R; ++s) {
            Path p;
            p.ox = park.f(kOx, s), p.oy = park.f(kOy, s), p.oz = park.f(kOz, s);
            p.dx = park.f(kDx, s), p.dy = park.f(kDy, s), p.dz = park.f(kDz, s);
            RayK k = ray_constants(p);
            // pin 2*o in registers: left alone, ptxas keeps o and re-adds it inside the sweep loop
            asm volatile("" : "+f"(k.tx), "+f"(k.ty), "+f"(k.tz));
            hot[s] = Hot{p.dx, p.dy, p.dz, k.k1, k.tx, k.ty, k.tz, k.nk2};
            closest[s] = cam.tmax * park.f(kLen, s);
            best[s] = -1;
        }
        for (int base = 0; base < P.n_pad; base += 32) {
            const int cnt = min(32, P.n_pad - base);
            unsigned m[R];
#pragma unroll
            for (int s = 0; s < R; ++s) m[s] = 0xFFFFFFFFu;  // 1 = miss
            const float4* g = pairs + base;
#pragma unroll 1
            for (int k = 0; k < cnt; k += 8) {
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    const float4 p0 = g[k + u], p1 = g[k + u + 1];
#pragma unroll
                    for (int s = 0; s < R; ++s) test_pair_hot(p0, p1, hot[s], m[s]);
                }
            }
            unsigned any = 0;
#pragma unroll
            for (int s = 0; s < R; ++s) any |= ~m[s];
            if (any) {
#pragma unroll
                for (int s = 0; s < R; ++s) {
                    if (~m[s]) {
                        Path p;
                        p.ox = park.fv(kOx, s), p.oy = park.fv(kOy, s), p.oz = park.fv(kOz, s);
                        p.dx = hot[s].dx, p.dy = hot[s].dy, p.dz = hot[s].dz;
                        p.self = __float_as_int(park.fv(kSelf, s));
                        const float tmin_d = cam.tmin * park.fv(kLen, s);
                        resolve_candidates(gather, ~m[s], base, cnt, p, tmin_d, closest[s], best[s]);
                    }
                }
            }
        }

        // ---- shading, one slot at a time through one copy of the code ----
#pragma unroll 1
        for (int s = 0; s < R; ++s) {
            float t = closest[0];
            int b = best[0];
#pragma unroll
            for (int q = 1; q < R; ++q)
                if (s == q) t = closest[q], b = best[q];
            if ((alive >> s) & 1u) {
                ++n_seg;
                Path p;
                park.load_ray(s, p);
                const RngKey key{cam.key0, cam.key1, park.u(kPixel, s), park.u(kSample, s)};
                float sr, sg, sb;
                int term;
                if (shade(cam, key, gather, s_aux, s_alb, p, t, b, sr, sg, sb, term)) {
                    const unsigned long long fr = to_fixed(sr), fg = to_fixed(sg), fb = to_fixed(sb);
                    unsigned long long* px = P.accum + 3ull * park.u(kLp, s);
                    if (fr) atomicAdd(px + 0, fr);
                    if (fg) atomicAdd(px + 1, fg);
                    if (fb) atomicAdd(px + 2, fb);
                    if (sr != sr || sg != sg || sb != sb) atomicAdd(P.stats + 5, 1ULL);
                    ++n_samp;
                    n_cap += (term == 2), n_abs += (term == 1);
                    alive &= ~(1u << s);
                } else {
                    park.store_ray(s, p);
                }
            }
            __syncwarp();
        }
    }
    unsigned long long v0 = n_samp, v1 = n_seg, v2 = n_cap, v3 = n_abs;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v0 += __shfl_xor_sync(0xFFFFFFFFu, v0, o);
        v1 += __shfl_xor_sync(0xFFFFFFFFu, v1, o);
        v2 += __shfl_xor_sync(0xFFFFFFFFu, v2, o);
        v3 += __shfl_xor_sync(0xFFFFFFFFu, v3, o);
    }
    if (lane == 0) {
        atomicAdd(P.stats + 0, v0);
        atomicAdd(P.stats + 1, v1);
        atomicAdd(P.stats + 2, v2);
        atomicAdd(P.stats + 3, v3);
    }
}

template <int R, int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_const_parked(const __grid_constant__ TraceParamsConst C) {
    __shared__ float park_mem[kParkFields * R * kBlock];
    __shared__ uint8_t todo_mem[kBlock * R];
    trace_body_parked<R, kBlock>(C.p, C.pairs, C.p.geom, park_mem, todo_mem);
}

// K1a: geometry in the constant bank (kernel parameter): the default for scenes of up to
// kMaxConstSpheres spheres.  The sweep's sphere operands are uniform registers fed by LDCU; they cost
// no register-file bandwidth, which is what bounds FFMA2 on sm_100.  No shared memory at all.
template <int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_const(const __grid_constant__ TraceParamsConst C) {
    __shared__ float stage[(kBlock / 32) * kStageFloats];
    trace_body<true, kBlock>(C.p, C.pairs, C.p.geom, stage);
}

// K1a with block culling: the same body, but a block of 32 spheres whose padded box (C.boxes) no path of the warp
// can reach is skipped.  The host takes it for scenes whose blocks are compact against the scene's extent.
template <int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_const_cull(const __grid_constant__ TraceParamsConst C) {
    __shared__ __align__(16) float stage[(kBlock / 32) * kCullStageFloats];
    trace_body<true, kBlock, true>(C.p, C.pairs, C.p.geom, stage, C.boxes, C.cull_r2, C.split_max);
}

// K1b: geometry staged into shared memory by 1-D TMA bulk copies (cp.async.bulk + mbarrier): scenes
// too large for the parameter space; 32 B of shared memory per sphere (up to ~7 200 spheres in 227 KiB).
template <int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_smem(const __grid_constant__ TraceParams P) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4* s_pairs = reinterpret_cast<float4*>(smem_raw);  // [n_pad] sweep layout
    float4* s_geom = s_pairs + P.n_pad;                      // [n_pad] per-lane lookups
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ float stage[(kBlock / 32) * kStageFloats];
    if (threadIdx.x == 0) {
        mbar_init(&s_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t bytes = (uint32_t)P.n_pad * 16u;
        mbar_expect_tx(&s_bar, 2u * bytes);
        bulk_g2s(s_pairs, P.pairs, bytes, &s_bar);
        bulk_g2s(s_geom, P.geom, bytes, &s_bar);
    }
    mbar_wait(&s_bar, 0);
    trace_body<false, kBlock>(P, s_pairs, s_geom, stage);
}

// K1c: geometry read from global memory (L1 / L2, warp-uniform addresses): scenes whose 32 B per sphere do
// not fit the shared memory of an SM (more than ~7 200 spheres).  The reference's HittableList has no size
// limit (src/hittable.zig:43-62), so neither has the drop-in; the sweep just loses its staging.
template <int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_global(const __grid_constant__ TraceParams P) {
    __shared__ float stage[(kBlock / 32) * kStageFloats];
    trace_body<false, kBlock>(P, P.pairs, P.geom, stage);
}

// ---------------------------------------------------------------------------------------------
// K1w: the warp-level WAVEFRONT organisation of the same work, for shading-bound scenes (few spheres).
//
// In the lockstep kernel above a lane shades the two paths it sweeps, so Material.scatter runs once per slot with
// whichever lanes happen to hold a hit (ncu at 16 spheres: 20.7 of 32 threads active over the kernel, 13 in
// shading), and a sweep of 16 spheres is only a tenth of the instructions.  Here the 64 paths of a warp live in
// SHARED memory, one word per (field, path), and every stage picks the paths it applies to from a compacted list,
// 32 at a time, whichever lane they were swept by:
//     sweep   lane l sweeps paths l and l + 32 (the packed two-sphere sweep, unchanged)        -> t, best
//     sky     misses are finished where they were swept (a dozen instructions + the three REDs)
//     shade   the hits of all 64 paths, compacted: one full-width pass of Material.scatter per 32 hits
//     regen   the free paths, compacted: one full-width pass of Camera.getRay per 32 new samples
// A pass that would run with fewer than wave_*_min paths is put off: its paths simply stay as they are for one
// more iteration (a hit that is swept again yields the same hit; a free path sweeps a stale ray whose result is
// ignored), which costs 1/64 of a sweep per path instead of a nearly empty pass — the host sets the thresholds
// from the sweep's length.  Work is counted where a segment is shaded, so nothing is counted twice.
// The image cannot depend on any of this: a sample's random numbers are a function of (pixel, sample, bounce)
// and the pixel sums are integers.  tests/test_gpu_parity.py compares this kernel with the mirror bit for bit.
// ---------------------------------------------------------------------------------------------
enum WaveField { wOx, wOy, wOz, wDx, wDy, wDz, wLen, wSelf, wTr, wTg, wTb, wBounce, wSample, wPixel, wLp, wT, wBest, kWaveFields };
constexpr int kMaxWaveSpheres = 256;  // beyond, the sweep dominates and the lockstep kernel's register-resident paths win (measured)
constexpr int kWaveWords = kWaveFields * 64 + 32;  // per warp: the fields of 64 paths + two 64-byte index lists

// the sky colour of a path that missed everything (src/camera.zig:171-177), added to its pixel
__device__ __forceinline__ void wave_add_sky(const TraceParams& P, const float* w, const uint32_t* wu, uint32_t s) {
    const float al = 0.5f * (w[wDy * 64 + s] + 1.0f);
    const float wh = 1.0f - al;
    const float sr = w[wTr * 64 + s] * fmaf(al, 0.5f, wh);
    const float sg = w[wTg * 64 + s] * fmaf(al, 0.7f, wh);
    const float sb = w[wTb * 64 + s] * fmaf(al, 1.0f, wh);
    const unsigned long long fr = to_fixed(sr), fg = to_fixed(sg), fb = to_fixed(sb);
    unsigned long long* px = P.accum + 3ull * wu[wLp * 64 + s];
    if (fr) atomicAdd(px + 0, fr);
    if (fg) atomicAdd(px + 1, fg);
    if (fb) atomicAdd(px + 2, fb);
    if (sr != sr || sg != sg || sb != sb) atomicAdd(P.stats + 5, 1ULL);  // NaN sample: adds 0, but is counted
}
constexpr uint32_t kWaveSky = 0xFFFFFFFFu;    // wBest of a free path whose sky colour has not been added yet
constexpr uint32_t kWaveEnded = 0xFFFFFFFEu;  // wBest of a free path that owes nothing

template <int kBlock>
__device__ __forceinline__ void trace_body_wave(const TraceParams& P, const float4* __restrict__ pairs,
                                                const float4* __restrict__ gather, float* __restrict__ wave_mem) {
    float* const w = wave_mem + (threadIdx.x >> 5) * kWaveWords;
    uint32_t* const wu = reinterpret_cast<uint32_t*>(w);
    uint8_t* const hit_list = reinterpret_cast<uint8_t*>(w + kWaveFields * 64);
    uint8_t* const free_list = hit_list + 64;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DevCamera& cam = P.cam;
    const uint32_t sa = lane, sb = lane + 32u;  // the two paths this lane sweeps

    // what a path without a sample sweeps (its result is ignored)
    w[wOx * 64 + sa] = w[wOy * 64 + sa] = w[wOz * 64 + sa] = 0.f, w[wDx * 64 + sa] = w[wDy * 64 + sa] = 0.f;
    w[wDz * 64 + sa] = 1.f, w[wLen * 64 + sa] = 1.f, wu[wSelf * 64 + sa] = 0xFFFFFFFFu;
    w[wOx * 64 + sb] = w[wOy * 64 + sb] = w[wOz * 64 + sb] = 0.f, w[wDx * 64 + sb] = w[wDy * 64 + sb] = 0.f;
    w[wDz * 64 + sb] = 1.f, w[wLen * 64 + sb] = 1.f, wu[wSelf * 64 + sb] = 0xFFFFFFFFu;
    wu[wBest * 64 + sa] = kWaveEnded, wu[wBest * 64 + sb] = kWaveEnded;
    __syncwarp();

    bool alive_a = false, alive_b = false;
    uint32_t ch_lp = 0, ch_x = 0, ch_y = 0, ch_next = 0, ch_end = 0;  // warp-uniform chunk state
    bool exhausted = false;
    unsigned long long n_seg = 0;
    uint32_t n_samp = 0, flip = 0;

    for (;;) {
        // ---- regen: Camera.getRay for the free paths, 32 new samples per pass, whichever lane owns the path ----
        if (!exhausted) {
            const unsigned fa = __ballot_sync(0xFFFFFFFFu, !alive_a), fb = __ballot_sync(0xFFFFFFFFu, !alive_b);
            const uint32_t nfa = __popc(fa), n_free = nfa + __popc(fb);
            const uint32_t rem = n_free & 31u;
            const uint32_t n_fill = (n_free - rem) + (rem >= P.wave_regen_min ? rem : 0u);
            if (n_fill) {
                const uint32_t rank_a = __popc(fa & lt_mask), rank_b = nfa + __popc(fb & lt_mask);
                if (!alive_a) free_list[rank_a] = (uint8_t)sa;
                if (!alive_b) free_list[rank_b] = (uint8_t)sb;
                __syncwarp();
                uint32_t done = 0;
                while (done < n_fill && !exhausted) {
                    const uint32_t n_batch = min(32u, n_fill - done);
                    // the batch takes the next n_batch samples of the queue; it may run over the end of a chunk
                    // into the next pixel, so pixel and sample are per-lane values here
                    uint32_t filled = 0, my_x = 0, my_y = 0, my_lp = 0, my_sample = 0;
                    bool have = false;
                    while (filled < n_batch) {
                        if (ch_next >= ch_end) {
                            unsigned long long cid = 0;
                            if (lane == 0) cid = atomicAdd(P.counter, 1ULL);
                            cid = __shfl_sync(0xFFFFFFFFu, cid, 0);
                            if (__any_sync(0xFFFFFFFFu, cid >= P.n_chunks)) {
                                exhausted = true;
                                break;
                            }
                            // (the host launches this kernel only for frames of fewer than 2^32 chunks)
                            const uint32_t lp = div_by((uint32_t)cid, P.rcp_chunks_per_pixel);
                            const uint32_t part = (uint32_t)cid - lp * P.chunks_per_pixel;
                            uint32_t x, y;
                            const bool inside = local_to_global_rcp(P.sh, P.rcp_tile_pixels, P.rcp_tiles_x, P.rcp_tile_w,
                                                                    cam.width, cam.height, lp, x, y);
                            if (__any_sync(0xFFFFFFFFu, !inside)) continue;  // tile padding
                            ch_lp = lp, ch_x = x, ch_y = y;
                            ch_next = part * P.chunk;
                            ch_end = min(ch_next + P.chunk, cam.spp);
                        }
                        const uint32_t take = min(n_batch - filled, ch_end - ch_next);
                        if (lane - filled < take) {  // filled <= lane < filled + take
                            my_x = ch_x, my_y = ch_y, my_lp = ch_lp, my_sample = ch_next + (lane - filled);
                            have = true;
                        }
                        filled += take, ch_next += take;
                    }
                    if (lane < n_batch) {
                        // the pass first retires the path that held the slot: a miss still owes its sky colour
                        const uint32_t s = free_list[done + lane];
                        if (wu[wBest * 64 + s] == kWaveSky) {
                            wave_add_sky(P, w, wu, s);
                            wu[wBest * 64 + s] = kWaveEnded;
                        }
                    }
                    if (have) {
                        const uint32_t pix = my_y * cam.width + my_x;
                        const RngKey key{cam.key0, cam.key1, pix, my_sample};
                        Path t;
                        camera_ray(cam, key, my_x, my_y, t);
                        const uint32_t s = free_list[done + lane];
                        w[wOx * 64 + s] = t.ox, w[wOy * 64 + s] = t.oy, w[wOz * 64 + s] = t.oz;
                        w[wDx * 64 + s] = t.dx, w[wDy * 64 + s] = t.dy, w[wDz * 64 + s] = t.dz;
                        w[wLen * 64 + s] = t.len, wu[wSelf * 64 + s] = 0xFFFFFFFFu;
                        w[wTr * 64 + s] = 1.0f, w[wTg * 64 + s] = 1.0f, w[wTb * 64 + s] = 1.0f;
                        wu[wBounce * 64 + s] = 0u, wu[wSample * 64 + s] = my_sample, wu[wPixel * 64 + s] = pix;
                        wu[wLp * 64 + s] = my_lp;
                    }
                    done += filled;
                }
                __syncwarp();
                if (!alive_a && rank_a < done) alive_a = true;
                if (!alive_b && rank_b < done) alive_b = true;
            }
        }
        if (exhausted) {  // no regeneration pass will retire the free paths any more: add what they owe
            if (!alive_a && wu[wBest * 64 + sa] == kWaveSky) wave_add_sky(P, w, wu, sa), wu[wBest * 64 + sa] = kWaveEnded;
            if (!alive_b && wu[wBest * 64 + sb] == kWaveSky) wave_add_sky(P, w, wu, sb), wu[wBest * 64 + sb] = kWaveEnded;
        }
        if (exhausted && P.pool) {
            // no more work to hand out: park what is still in flight for drain_kernel and retire (a hit that was
            // put off is parked as it was before its sweep; the drain sweeps it again)
            const unsigned pa = __ballot_sync(0xFFFFFFFFu, alive_a), pb = __ballot_sync(0xFFFFFFFFu, alive_b);
            unsigned base = 0u;
            if (lane == 0u) base = atomicAdd(P.pool_count, (unsigned)(__popc(pa) + __popc(pb)));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const uint32_t s = h ? sb : sa;
                if (h ? alive_b : alive_a) {
                    float4* e = P.pool + 4ull * (base + (h ? __popc(pa) + __popc(pb & lt_mask) : __popc(pa & lt_mask)));
                    e[0] = make_float4(w[wOx * 64 + s], w[wOy * 64 + s], w[wOz * 64 + s], w[wLen * 64 + s]);
                    const int self = (int)wu[wSelf * 64 + s];  // the drain does not know the flag; without it the same hit is found
                    e[1] = make_float4(w[wDx * 64 + s], w[wDy * 64 + s], w[wDz * 64 + s],
                                       __int_as_float((self >> 30) == 1 ? self & ~kSelfLeaves : self));
                    e[2] = make_float4(w[wTr * 64 + s], w[wTg * 64 + s], w[wTb * 64 + s], w[wBounce * 64 + s]);
                    e[3] = make_float4(w[wPixel * 64 + s], w[wSample * 64 + s], w[wLp * 64 + s], 0.f);
                }
            }
            break;
        }
        const unsigned live_a = __ballot_sync(0xFFFFFFFFu, alive_a), live_b = __ballot_sync(0xFFFFFFFFu, alive_b);
        if ((live_a | live_b) == 0u) break;  // queue drained, every path finished

        // ---- sweep: HittableList.hit for the lane's two paths ----
        Path a, b;
        a.ox = w[wOx * 64 + sa], a.oy = w[wOy * 64 + sa], a.oz = w[wOz * 64 + sa];
        a.dx = w[wDx * 64 + sa], a.dy = w[wDy * 64 + sa], a.dz = w[wDz * 64 + sa];
        a.len = w[wLen * 64 + sa], a.self = (int)wu[wSelf * 64 + sa];
        b.ox = w[wOx * 64 + sb], b.oy = w[wOy * 64 + sb], b.oz = w[wOz * 64 + sb];
        b.dx = w[wDx * 64 + sb], b.dy = w[wDy * 64 + sb], b.dz = w[wDz * 64 + sb];
        b.len = w[wLen * 64 + sb], b.self = (int)wu[wSelf * 64 + sb];
        float ta = 0.f, tb = 0.f;
        int ia = -1, ib = -1;
        sweep2<true, true>(pairs, gather, P.n_pad, cam.tmin, cam.tmax, a, b, ta, ia, tb, ib);
        const bool hit_a = alive_a && ia >= 0, hit_b = alive_b && ib >= 0;
        if (hit_a) w[wT * 64 + sa] = ta, wu[wBest * 64 + sa] = (uint32_t)ia;
        if (hit_b) w[wT * 64 + sb] = tb, wu[wBest * 64 + sb] = (uint32_t)ib;

        // ---- sky: a miss ends the sample; its colour is added by the pass that reuses the slot ----
        if (alive_a && ia < 0) wu[wBest * 64 + sa] = kWaveSky, alive_a = false;
        if (alive_b && ib < 0) wu[wBest * 64 + sb] = kWaveSky, alive_b = false;
        {
            const unsigned still_a = __ballot_sync(0xFFFFFFFFu, alive_a), still_b = __ballot_sync(0xFFFFFFFFu, alive_b);
            const uint32_t n_sky = __popc(live_a & ~still_a) + __popc(live_b & ~still_b);
            n_seg += n_sky, n_samp += n_sky;
        }

        // ---- shade: Material.scatter for the hits of all 64 paths, compacted, 32 per pass ----
        const unsigned ha = __ballot_sync(0xFFFFFFFFu, hit_a), hb = __ballot_sync(0xFFFFFFFFu, hit_b);
        const uint32_t nha = __popc(ha), n_hit = nha + __popc(hb);
        const uint32_t hrem = n_hit & 31u;
        const uint32_t n_proc = (n_hit - hrem) + (hrem >= (exhausted ? 1u : P.wave_shade_min) ? hrem : 0u);
        if (n_proc) {
            // the order of the list alternates, so that the hits put off by one iteration lead the next
            uint32_t rank_a = __popc(ha & lt_mask), rank_b = nha + __popc(hb & lt_mask);
            if (flip) rank_a = n_hit - 1u - rank_a, rank_b = n_hit - 1u - rank_b;
            if (hit_a) hit_list[rank_a] = (uint8_t)sa;
            if (hit_b) hit_list[rank_b] = (uint8_t)sb;
            __syncwarp();
            uint32_t n_end = 0;
            for (uint32_t j0 = 0; j0 < n_proc; j0 += 32u) {
                const uint32_t j = j0 + lane;
                bool ended = false;
                if (j < n_proc) {
                    const uint32_t s = hit_list[j];
                    Path p;
                    p.ox = w[wOx * 64 + s], p.oy = w[wOy * 64 + s], p.oz = w[wOz * 64 + s];
                    p.dx = w[wDx * 64 + s], p.dy = w[wDy * 64 + s], p.dz = w[wDz * 64 + s];
                    p.tr = w[wTr * 64 + s], p.tg = w[wTg * 64 + s], p.tb = w[wTb * 64 + s];
                    p.len = 1.f, p.self = -1, p.bounce = wu[wBounce * 64 + s];
                    const RngKey key{cam.key0, cam.key1, wu[wPixel * 64 + s], wu[wSample * 64 + s]};
                    const float t = w[wT * 64 + s];
                    const int best = (int)wu[wBest * 64 + s];
                    float sr, sg, sbl;
                    int term;
                    if (shade<true>(cam, key, gather, P.aux, P.albedo, p, t, best, sr, sg, sbl, term)) {
                        // a hit ends a sample black (absorbed by a metal, depth cap): nothing to add
                        if (term == 2) atomicAdd(P.stats + 2, 1ULL);
                        if (term == 1) atomicAdd(P.stats + 3, 1ULL);
                        wu[wBest * 64 + s] = kWaveEnded;  // tells the lane that sweeps this path that it is free
                        ended = true;
                    } else {
                        w[wOx * 64 + s] = p.ox, w[wOy * 64 + s] = p.oy, w[wOz * 64 + s] = p.oz;
                        w[wDx * 64 + s] = p.dx, w[wDy * 64 + s] = p.dy, w[wDz * 64 + s] = p.dz;
                        w[wTr * 64 + s] = p.tr, w[wTg * 64 + s] = p.tg, w[wTb * 64 + s] = p.tb;
                        w[wLen * 64 + s] = p.len, wu[wSelf * 64 + s] = (uint32_t)p.self, wu[wBounce * 64 + s] = p.bounce;
                    }
                }
                n_end += __popc(__ballot_sync(0xFFFFFFFFu, ended));
            }
            n_seg += n_proc, n_samp += n_end;
            __syncwarp();
            if (hit_a && rank_a < n_proc && wu[wBest * 64 + sa] == kWaveEnded) alive_a = false;
            if (hit_b && rank_b < n_proc && wu[wBest * 64 + sb] == kWaveEnded) alive_b = false;
        }
        flip ^= 1u;
        __syncwarp();
    }
    if (lane == 0u) {  // one atomic per warp and counter
        atomicAdd(P.stats + 0, (unsigned long long)n_samp);
        atomicAdd(P.stats + 1, n_seg);
    }
}

template <int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_wave(const __grid_constant__ TraceParamsConst C) {
    __shared__ float wave_mem[(kBlock / 32) * kWaveWords];
    trace_body_wave<kBlock>(C.p, C.pairs, C.p.geom, wave_mem);
}

// ---------------------------------------------------------------------------------------------
// K1w with S paths per lane (S = 4, 128 paths per warp: the default for 33..256 spheres; RTZ_VARIANT=12 forces it).  The same stages as
// trace_body_wave over 32 * S paths: the ballots, lists and chunk bookkeeping of an iteration and the uniform loads
// of the sweep are shared by twice as many paths, and a partial pass is a smaller share of the passes.  The sweep keeps
// only what the packed loop reads (direction + the five constants of the expanded discriminant per path) in
// registers; origin, |d| and self are re-read from shared memory where a candidate is resolved.
// ---------------------------------------------------------------------------------------------
template <int S>
struct WaveN {
    static constexpr int kPaths = 32 * S;
    static constexpr int kWords = kWaveFields * kPaths + 2 * kPaths / 4;  // fields + two byte lists of kPaths entries
};

template <int S>
__device__ __forceinline__ void wave_add_sky_n(const TraceParams& P, const float* w, const uint32_t* wu, uint32_t s) {
    constexpr int N = WaveN<S>::kPaths;
    const float al = 0.5f * (w[wDy * N + s] + 1.0f);
    const float wh = 1.0f - al;
    const float sr = w[wTr * N + s] * fmaf(al, 0.5f, wh);
    const float sg = w[wTg * N + s] * fmaf(al, 0.7f, wh);
    const float sb = w[wTb * N + s] * fmaf(al, 1.0f, wh);
    const unsigned long long fr = to_fixed(sr), fg = to_fixed(sg), fb = to_fixed(sb);
    unsigned long long* px = P.accum + 3ull * wu[wLp * N + s];
    if (fr) atomicAdd(px + 0, fr);
    if (fg) atomicAdd(px + 1, fg);
    if (fb) atomicAdd(px + 2, fb);
    if (sr != sr || sg != sg || sb != sb) atomicAdd(P.stats + 5, 1ULL);
}

template <int S, int kBlock>
__device__ __forceinline__ void trace_body_wave_n(const TraceParams& P, const float4* __restrict__ pairs,
                                                  const float4* __restrict__ gather, float* __restrict__ wave_mem) {
    constexpr int N = WaveN<S>::kPaths;
    float* const w = wave_mem + (threadIdx.x >> 5) * WaveN<S>::kWords;
    uint32_t* const wu = reinterpret_cast<uint32_t*>(w);
    uint8_t* const hit_list = reinterpret_cast<uint8_t*>(w + kWaveFields * N);
    uint8_t* const free_list = hit_list + N;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DevCamera& cam = P.cam;

#pragma unroll
    for (int h = 0; h < S; ++h) {  // what a path without a sample sweeps (its result is ignored)
        const uint32_t s = lane + 32u * h;
        w[wOx * N + s] = w[wOy * N + s] = w[wOz * N + s] = 0.f, w[wDx * N + s] = w[wDy * N + s] = 0.f;
        w[wDz * N + s] = 1.f, w[wLen * N + s] = 1.f, wu[wSelf * N + s] = 0xFFFFFFFFu, wu[wBest * N + s] = kWaveEnded;
    }
    __syncwarp();

    unsigned alive = 0u;  // bit h: path lane + 32 h carries a sample
    uint32_t ch_lp = 0, ch_x = 0, ch_y = 0, ch_next = 0, ch_end = 0;  // warp-uniform chunk state
    bool exhausted = false;
    unsigned long long n_seg = 0;
    uint32_t n_samp = 0, flip = 0;

    for (;;) {
        // ---- regen ----
        if (!exhausted) {
            unsigned fb[S];
            uint32_t n_free = 0;
#pragma unroll
            for (int h = 0; h < S; ++h) fb[h] = __ballot_sync(0xFFFFFFFFu, !((alive >> h) & 1u)), n_free += __popc(fb[h]);
            const uint32_t rem = n_free & 31u;
            const uint32_t n_fill = (n_free - rem) + (rem >= P.wave_regen_min ? rem : 0u);
            if (n_fill) {
                uint32_t rank[S], before = 0;
#pragma unroll
                for (int h = 0; h < S; ++h) {
                    rank[h] = before + __popc(fb[h] & lt_mask);
                    before += __popc(fb[h]);
                    if (!((alive >> h) & 1u)) free_list[rank[h]] = (uint8_t)(lane + 32u * h);
                }
                __syncwarp();
                uint32_t done = 0;
                while (done < n_fill && !exhausted) {
                    const uint32_t n_batch = min(32u, n_fill - done);
                    uint32_t filled = 0, my_x = 0, my_y = 0, my_lp = 0, my_sample = 0;
                    bool have = false;
                    while (filled < n_batch) {
                        if (ch_next >= ch_end) {
                            unsigned long long cid = 0;
                            if (lane == 0) cid = atomicAdd(P.counter, 1ULL);
                            cid = __shfl_sync(0xFFFFFFFFu, cid, 0);
                            if (__any_sync(0xFFFFFFFFu, cid >= P.n_chunks)) {
                                exhausted = true;
                                break;
                            }
                            const uint32_t lp = div_by((uint32_t)cid, P.rcp_chunks_per_pixel);
                            const uint32_t part = (uint32_t)cid - lp * P.chunks_per_pixel;
                            uint32_t x, y;
                            const bool inside = local_to_global_rcp(P.sh, P.rcp_tile_pixels, P.rcp_tiles_x, P.rcp_tile_w,
                                                                    cam.width, cam.height, lp, x, y);
                            if (__any_sync(0xFFFFFFFFu, !inside)) continue;  // tile padding
                            ch_lp = lp, ch_x = x, ch_y = y;
                            ch_next = part * P.chunk;
                            ch_end = min(ch_next + P.chunk, cam.spp);
                        }
                        const uint32_t take = min(n_batch - filled, ch_end - ch_next);
                        if (lane - filled < take) {
                            my_x = ch_x, my_y = ch_y, my_lp = ch_lp, my_sample = ch_next + (lane - filled);
                            have = true;
                        }
                        filled += take, ch_next += take;
                    }
                    if (lane < n_batch) {
                        const uint32_t s = free_list[done + lane];
                        if (wu[wBest * N + s] == kWaveSky) {
                            wave_add_sky_n<S>(P, w, wu, s);
                            wu[wBest * N + s] = kWaveEnded;
                        }
                    }
                    if (have) {
                        const uint32_t pix = my_y * cam.width + my_x;
                        const RngKey key{cam.key0, cam.key1, pix, my_sample};
                        Path t;
                        camera_ray(cam, key, my_x, my_y, t);
                        const uint32_t s = free_list[done + lane];
                        w[wOx * N + s] = t.ox, w[wOy * N + s] = t.oy, w[wOz * N + s] = t.oz;
                        w[wDx * N + s] = t.dx, w[wDy * N + s] = t.dy, w[wDz * N + s] = t.dz;
                        w[wLen * N + s] = t.len, wu[wSelf * N + s] = 0xFFFFFFFFu;
                        w[wTr * N + s] = 1.0f, w[wTg * N + s] = 1.0f, w[wTb * N + s] = 1.0f;
                        wu[wBounce * N + s] = 0u, wu[wSample * N + s] = my_sample, wu[wPixel * N + s] = pix;
                        wu[wLp * N + s] = my_lp;
                    }
                    done += filled;
                }
                __syncwarp();
#pragma unroll
                for (int h = 0; h < S; ++h)
                    if (!((alive >> h) & 1u) && rank[h] < done) alive |= 1u << h;
            }
        }
        if (exhausted) {
#pragma unroll
            for (int h = 0; h < S; ++h) {
                const uint32_t s = lane + 32u * h;
                if (!((alive >> h) & 1u) && wu[wBest * N + s] == kWaveSky) wave_add_sky_n<S>(P, w, wu, s), wu[wBest * N + s] = kWaveEnded;
            }
        }
        if (exhausted && P.pool) {
            unsigned pb[S];
            uint32_t total = 0;
#pragma unroll
            for (int h = 0; h < S; ++h) pb[h] = __ballot_sync(0xFFFFFFFFu, (alive >> h) & 1u), total += __popc(pb[h]);
            unsigned base = 0u;
            if (lane == 0u) base = atomicAdd(P.pool_count, total);
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
#pragma unroll
            for (int h = 0; h < S; ++h) {
                const uint32_t s = lane + 32u * h;
                if ((alive >> h) & 1u) {
                    float4* e = P.pool + 4ull * (base + __popc(pb[h] & lt_mask));
                    e[0] = make_float4(w[wOx * N + s], w[wOy * N + s], w[wOz * N + s], w[wLen * N + s]);
                    const int self = (int)wu[wSelf * N + s];
                    e[1] = make_float4(w[wDx * N + s], w[wDy * N + s], w[wDz * N + s],
                                       __int_as_float((self >> 30) == 1 ? self & ~kSelfLeaves : self));
                    e[2] = make_float4(w[wTr * N + s], w[wTg * N + s], w[wTb * N + s], w[wBounce * N + s]);
                    e[3] = make_float4(w[wPixel * N + s], w[wSample * N + s], w[wLp * N + s], 0.f);
                }
                base += __popc(pb[h]);
            }
            break;
        }
        unsigned live[S], any_live = 0;
#pragma unroll
        for (int h = 0; h < S; ++h) live[h] = __ballot_sync(0xFFFFFFFFu, (alive >> h) & 1u), any_live |= live[h];
        if (any_live == 0u) break;

        // ---- sweep ----
        float dx[S], dy[S], dz[S], closest[S];
        RayK k[S];
        int best[S];
#pragma unroll
        for (int h = 0; h < S; ++h) {
            const uint32_t s = lane + 32u * h;
            Path q;
            q.ox = w[wOx * N + s], q.oy = w[wOy * N + s], q.oz = w[wOz * N + s];
            q.dx = dx[h] = w[wDx * N + s], q.dy = dy[h] = w[wDy * N + s], q.dz = dz[h] = w[wDz * N + s];
            k[h] = ray_constants(q);
            asm volatile("" : "+f"(k[h].tx), "+f"(k[h].ty), "+f"(k[h].tz));
            closest[h] = cam.tmax * w[wLen * N + s];
            best[h] = -1;
        }
        for (int base = 0; base < P.n_pad; base += 32) {
            const int cnt = min(32, P.n_pad - base);
            unsigned m[S];
#pragma unroll
            for (int h = 0; h < S; ++h) m[h] = 0xFFFFFFFFu;  // 1 = miss
            const float4* g = pairs + base;
#pragma unroll 1
            for (int q0 = 0; q0 < cnt; q0 += 8) {
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    const float4 p0 = g[q0 + u], p1 = g[q0 + u + 1];
#pragma unroll
                    for (int h = 0; h < S; ++h) {
                        Path q;
                        q.dx = dx[h], q.dy = dy[h], q.dz = dz[h];
                        test_pair(p0, p1, q, k[h], m[h]);
                    }
                }
            }
            unsigned any = 0;
#pragma unroll
            for (int h = 0; h < S; ++h) m[h] = ~m[h], any |= m[h];
            if (any) {
#pragma unroll
                for (int h = 0; h < S; ++h) {
                    if (m[h]) {
                        const uint32_t s = lane + 32u * h;
                        const volatile float* wv = w;  // re-read here, not held in registers across the packed loop
                        const volatile uint32_t* wuv = wu;
                        Path q;
                        q.ox = wv[wOx * N + s], q.oy = wv[wOy * N + s], q.oz = wv[wOz * N + s];
                        q.dx = dx[h], q.dy = dy[h], q.dz = dz[h];
                        q.self = (int)wuv[wSelf * N + s];
                        unsigned c = m[h];
                        const unsigned rel = (unsigned)(q.self & ~kSelfLeaves) - (unsigned)base;
                        if ((q.self >> 30) == 1 && rel < (unsigned)cnt) c &= ~(1u << (cnt - 1 - (int)rel));
                        resolve_candidates(gather, c, base, cnt, q, cam.tmin * wv[wLen * N + s], closest[h], best[h]);
                    }
                }
            }
        }
        unsigned hit = 0u;
#pragma unroll
        for (int h = 0; h < S; ++h) {
            const uint32_t s = lane + 32u * h;
            if ((alive >> h) & 1u) {
                if (best[h] >= 0) {
                    w[wT * N + s] = closest[h], wu[wBest * N + s] = (uint32_t)best[h];
                    hit |= 1u << h;
                } else {  // sky: the colour is added by the pass that reuses the slot
                    wu[wBest * N + s] = kWaveSky;
                    alive &= ~(1u << h);
                }
            }
        }
        {
            uint32_t n_sky = 0;
#pragma unroll
            for (int h = 0; h < S; ++h) n_sky += __popc(live[h] & ~__ballot_sync(0xFFFFFFFFu, (alive >> h) & 1u));
            n_seg += n_sky, n_samp += n_sky;
        }

        // ---- shade ----
        unsigned hb[S];
        uint32_t n_hit = 0;
#pragma unroll
        for (int h = 0; h < S; ++h) hb[h] = __ballot_sync(0xFFFFFFFFu, (hit >> h) & 1u), n_hit += __popc(hb[h]);
        const uint32_t hrem = n_hit & 31u;
        const uint32_t n_proc = (n_hit - hrem) + (hrem >= (exhausted ? 1u : P.wave_shade_min) ? hrem : 0u);
        if (n_proc) {
            uint32_t rank[S], before = 0;
#pragma unroll
            for (int h = 0; h < S; ++h) {
                rank[h] = before + __popc(hb[h] & lt_mask);
                before += __popc(hb[h]);
                if (flip) rank[h] = n_hit - 1u - rank[h];
                if ((hit >> h) & 1u) hit_list[rank[h]] = (uint8_t)(lane + 32u * h);
            }
            __syncwarp();
            uint32_t n_end = 0;
            for (uint32_t j0 = 0; j0 < n_proc; j0 += 32u) {
                const uint32_t j = j0 + lane;
                bool ended = false;
                if (j < n_proc) {
                    const uint32_t s = hit_list[j];
                    Path p;
                    p.ox = w[wOx * N + s], p.oy = w[wOy * N + s], p.oz = w[wOz * N + s];
                    p.dx = w[wDx * N + s], p.dy = w[wDy * N + s], p.dz = w[wDz * N + s];
                    p.tr = w[wTr * N + s], p.tg = w[wTg * N + s], p.tb = w[wTb * N + s];
                    p.len = 1.f, p.self = -1, p.bounce = wu[wBounce * N + s];
                    const RngKey key{cam.key0, cam.key1, wu[wPixel * N + s], wu[wSample * N + s]};
                    const float t = w[wT * N + s];
                    const int bst = (int)wu[wBest * N + s];
                    float sr, sg, sbl;
                    int term;
                    if (shade<true>(cam, key, gather, P.aux, P.albedo, p, t, bst, sr, sg, sbl, term)) {
                        if (term == 2) atomicAdd(P.stats + 2, 1ULL);
                        if (term == 1) atomicAdd(P.stats + 3, 1ULL);
                        wu[wBest * N + s] = kWaveEnded;
                        ended = true;
                    } else {
                        w[wOx * N + s] = p.ox, w[wOy * N + s] = p.oy, w[wOz * N + s] = p.oz;
                        w[wDx * N + s] = p.dx, w[wDy * N + s] = p.dy, w[wDz * N + s] = p.dz;
                        w[wTr * N + s] = p.tr, w[wTg * N + s] = p.tg, w[wTb * N + s] = p.tb;
                        w[wLen * N + s] = p.len, wu[wSelf * N + s] = (uint32_t)p.self, wu[wBounce * N + s] = p.bounce;
                    }
                }
                n_end += __popc(__ballot_sync(0xFFFFFFFFu, ended));
            }
            n_seg += n_proc, n_samp += n_end;
            __syncwarp();
#pragma unroll
            for (int h = 0; h < S; ++h)
                if (((hit >> h) & 1u) && rank[h] < n_proc && wu[wBest * N + lane + 32u * h] == kWaveEnded) alive &= ~(1u << h);
        }
        flip ^= 1u;
        __syncwarp();
    }
    if (lane == 0u) {
        atomicAdd(P.stats + 0, (unsigned long long)n_samp);
        atomicAdd(P.stats + 1, n_seg);
    }
}

template <int S, int kBlock, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) trace_kernel_wave_n(const __grid_constant__ TraceParamsConst C) {
    __shared__ float wave_mem[(kBlock / 32) * WaveN<S>::kWords];
    trace_body_wave_n<S, kBlock>(C.p, C.pairs, C.p.geom, wave_mem);
}

// ---------------------------------------------------------------------------------------------
// K1d: the drain.  Finishes the paths the trace kernel parked when its queue ran dry.  A warp holds up to 32
// parked paths, one per lane.  Per bounce the closest hit of every live path is found by the WHOLE warp — the
// path is broadcast, lane l tests spheres l, l + 32, ... (coop_hit) — and then all lanes shade their own paths
// together; lanes whose path ended take the next parked one.  A bounce costs ~N/32 tests per lane and live path
// instead of the N a lockstep warp pays for however few paths it has left, so the frame no longer ends with a
// millisecond of nearly empty warps (RTZ_TIMELINE, DESIGN.md §5).  Same arithmetic, same closest hit (minimum
// over (t, index)): same image.
// kWarp == false (scenes of fewer spheres than a warp has lanes): every thread sweeps its own path's spheres.
// ---------------------------------------------------------------------------------------------
template <bool kWarp>
__global__ void __launch_bounds__(128) drain_kernel(const __grid_constant__ TraceParams P) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned n_parked = *P.pool_count;
    const DevCamera& cam = P.cam;
    Slot s;
    s.alive = false, s.lp = 0;
    s.key = RngKey{cam.key0, cam.key1, 0u, 0u};
    s.path.ox = s.path.oy = s.path.oz = 0.f, s.path.dx = s.path.dy = 0.f, s.path.dz = 1.f;
    s.path.tr = s.path.tg = s.path.tb = 0.f, s.path.len = 1.f, s.path.self = -1, s.path.bounce = 0;
    bool empty = false;  // warp-uniform: the pool has nothing left to hand out
    unsigned long long n_seg = 0;
    unsigned n_samp = 0;
    for (;;) {
        const unsigned need = __ballot_sync(0xFFFFFFFFu, !s.alive);
        if (need && !empty) {
            unsigned base = 0u;
            if (lane == 0u) base = atomicAdd(P.pool_count + 1, (unsigned)__popc(need));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            const unsigned idx = base + __popc(need & lt_mask);
            if (((need >> lane) & 1u) && idx < n_parked) unpark_path(P.pool + 4ull * idx, cam.key0, cam.key1, s);
            empty = base + (unsigned)__popc(need) >= n_parked;
        }
        const unsigned live = __ballot_sync(0xFFFFFFFFu, s.alive);
        if (live == 0u) break;
        float t = 0.f;
        int best = -1;
        if (kWarp) {
            for (unsigned m = live; m; m &= m - 1u)
                coop_hit<false>(P.geom, P.wexp, P.orig, P.n_spheres, cam.tmin, cam.tmax, s.path, __ffs(m) - 1, lane, t, best);
        } else if (s.alive) {
            sweep_rows(P.geom, P.pairs, 0, P.n_spheres, s.path, cam.tmin, cam.tmax, t, best);
        }
        n_seg += (unsigned)__popc(live);
        if (s.alive) {
            float sr, sg, sb;
            int term;
            if (shade(cam, s.key, P.geom, P.aux, P.albedo, s.path, t, best, sr, sg, sb, term)) {
                const unsigned long long fr = to_fixed(sr), fg = to_fixed(sg), fb = to_fixed(sb);
                unsigned long long* px = P.accum + 3ull * s.lp;
                if (fr) atomicAdd(px + 0, fr);
                if (fg) atomicAdd(px + 1, fg);
                if (fb) atomicAdd(px + 2, fb);
                if (sr != sr || sg != sg || sb != sb) atomicAdd(P.stats + 5, 1ULL);
                if (term == 2) atomicAdd(P.stats + 2, 1ULL);
                if (term == 1) atomicAdd(P.stats + 3, 1ULL);
                s.alive = false;
            }
        }
        n_samp += (unsigned)__popc(live & __ballot_sync(0xFFFFFFFFu, !s.alive));
    }
    if (lane == 0u && n_seg) {
        atomicAdd(P.stats + 0, (unsigned long long)n_samp);
        atomicAdd(P.stats + 1, n_seg);
    }
}

// ---------------------------------------------------------------------------------------------
// K3: resolve.  pixelColor * pixelSamplesScale (src/camera.zig:137), then Color.toRgb
// (src/color.zig:63-80): sqrt if > 0, clamp [0, .999], trunc(256 x).  f64 like the reference
// (one sqrt per channel per pixel; the kernel is bound by its 27 B/pixel of HBM traffic).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint8_t to_byte(double lin) {
    double g = lin > 0.0 ? sqrt(lin) : 0.0;
    g = g < 0.0 ? 0.0 : (g > 0.999 ? 0.999 : g);  // Interval.clamp (src/interval.zig:40-47)
    return (uint8_t)(256.0 * g);
}

__global__ void resolve_kernel(const unsigned long long* __restrict__ accum, uint64_t n_pixels, double scale,
                               uint8_t* __restrict__ rgb, double* __restrict__ linear) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per channel
    if (i >= 3 * n_pixels) return;
    const double lin = ((double)accum[i] * 0x1p-32) * scale;
    rgb[i] = to_byte(lin);
    if (linear) linear[i] = lin;
}

// K3 fused with the multi-GPU tile exchange (rtz_multi_*, RTZ_GATHER_P2P): the same resolve, but every channel
// is stored at its place in the ROW-MAJOR image, which lives on device 0 — peer memory over NVLink for the
// other devices.  A device's resolve IS its half of the gather: no staging buffer, no de-interleave pass.
__global__ void resolve_scatter_kernel(const unsigned long long* __restrict__ accum, const ShardGeom sh, uint32_t W,
                                       uint32_t H, double scale, uint8_t* __restrict__ image) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per channel
    if (i >= 3ull * sh.n_local_tiles * sh.tile_pixels) return;
    const uint32_t lp = (uint32_t)(i / 3), ch = (uint32_t)(i - 3ull * lp);
    uint32_t x, y;
    if (!local_to_global(sh, W, H, lp, x, y)) return;  // tile padding
    image[3ull * ((uint64_t)y * W + x) + ch] = to_byte(((double)accum[i] * 0x1p-32) * scale);
}

// ---------------------------------------------------------------------------------------------
// K2: legacy deterministic pipelines behind test-files/chapter{4,5,6}.ppm.  f64, reference
// operation order (the file is compiled with -fmad=false, so nothing is contracted): one ray
// through the pixel centre, Sphere.hit as written (a = |d|^2 kept, division by a), no gamma,
// trunc(255.999 c).
// ---------------------------------------------------------------------------------------------
struct DSphere {
    double cx, cy, cz, r;
};
struct LegacyParams {
    double p0[3], du[3], dv[3], c[3];
    double tmin, tmax;
    uint32_t width, height;
    int mode;
    int n;
    const DSphere* spheres;
};
__device__ __forceinline__ double ddot(double ax, double ay, double az, double bx, double by, double bz) {
    return (ax * bx + ay * by) + az * bz;
}
__global__ void legacy_kernel(const __grid_constant__ LegacyParams P, uint8_t* __restrict__ rgb,
                              double* __restrict__ linear) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P.width * P.height) return;
    const uint32_t j = idx / P.width, i = idx - j * P.width;
    const double fi = (double)i, fj = (double)j;
    const double pcx = (P.p0[0] + P.du[0] * fi) + P.dv[0] * fj;
    const double pcy = (P.p0[1] + P.du[1] * fi) + P.dv[1] * fj;
    const double pcz = (P.p0[2] + P.du[2] * fi) + P.dv[2] * fj;
    const double ox = P.c[0], oy = P.c[1], oz = P.c[2];
    const double dx = pcx - ox, dy = pcy - oy, dz = pcz - oz;
    bool hit = false;
    double nx = 0, ny = 0, nz = 0;
    if (P.mode != 1) {
        double closest = P.tmax;
        for (int s = 0; s < P.n; ++s) {
            const DSphere sp = P.spheres[s];
            const double ocx = sp.cx - ox, ocy = sp.cy - oy, ocz = sp.cz - oz;
            const double a = ddot(dx, dy, dz, dx, dy, dz);
            const double h = ddot(dx, dy, dz, ocx, ocy, ocz);
            const double c = ddot(ocx, ocy, ocz, ocx, ocy, ocz) - sp.r * sp.r;
            const double disc = h * h - a * c;
            if (disc < 0) continue;
            const double sq = sqrt(disc);
            double root = (h - sq) / a;
            if (!(P.tmin < root && root < closest)) {
                root = (h + sq) / a;
                if (!(P.tmin < root && root < closest)) continue;
            }
            closest = root;
            hit = true;
            const double px = ox + dx * root, py = oy + dy * root, pz = oz + dz * root;
            const double inv = 1.0 / sp.r;  // divScalar = multiply by reciprocal (Q2)
            nx = (px - sp.cx) * inv, ny = (py - sp.cy) * inv, nz = (pz - sp.cz) * inv;
            if (!(ddot(dx, dy, dz, nx, ny, nz) < 0)) nx = -nx, ny = -ny, nz = -nz;
        }
    }
    double r, g, b;
    if (hit && P.mode == 2) {
        r = 1, g = 0, b = 0;
    } else if (hit) {
        r = (nx + 1.0) * 0.5, g = (ny + 1.0) * 0.5, b = (nz + 1.0) * 0.5;
    } else {
        const double inv = 1.0 / sqrt(ddot(dx, dy, dz, dx, dy, dz));
        const double a = 0.5 * (dy * inv + 1.0);
        r = 1.0 * (1.0 - a) + 0.5 * a, g = 1.0 * (1.0 - a) + 0.7 * a, b = 1.0 * (1.0 - a) + 1.0 * a;
    }
    rgb[3 * idx + 0] = (uint8_t)(255.999 * r);
    rgb[3 * idx + 1] = (uint8_t)(255.999 * g);
    rgb[3 * idx + 2] = (uint8_t)(255.999 * b);
    if (linear) linear[3 * idx + 0] = r, linear[3 * idx + 1] = g, linear[3 * idx + 2] = b;
}

// ---------------------------------------------------------------------------------------------
// K4: de-interleave `world` equal-sized compact tile buffers into the row-major image.
// ---------------------------------------------------------------------------------------------
__global__ void deinterleave_kernel(const uint8_t* __restrict__ gathered, uint64_t per_rank_pixels, uint32_t W,
                                    uint32_t H, uint32_t world, uint32_t tw, uint32_t th, uint32_t tiles_x,
                                    uint8_t* __restrict__ out) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint64_t)W * H) return;
    const uint32_t y = (uint32_t)(idx / W), x = (uint32_t)(idx - (uint64_t)y * W);
    const uint32_t tx = x / tw, ty = y / th;
    const uint32_t gt = ty * tiles_x + tx;
    const uint32_t rank = gt % world, lt = gt / world;
    const uint64_t lp = (uint64_t)lt * (tw * th) + (y - ty * th) * tw + (x - tx * tw);
    const uint8_t* src = gathered + 3ull * ((uint64_t)rank * per_rank_pixels + lp);
    out[3 * idx + 0] = src[0], out[3 * idx + 1] = src[1], out[3 * idx + 2] = src[2];
}

// ---------------------------------------------------------------------------------------------
// probes: one thread per record, the same device functions the render kernel inlines
// ---------------------------------------------------------------------------------------------
__global__ void probe_hits_kernel(const float4* geom, const float4* pairs, const float4* aux, int n_pad,
                                  const rtz_probe_ray* rays, uint64_t m, float tmin, float tmax, rtz_ray_hit* out) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const rtz_probe_ray r = rays[k];
    Path p;
    p.ox = r.orig[0], p.oy = r.orig[1], p.oz = r.orig[2], p.self = r.self, p.bounce = 0, p.tr = p.tg = p.tb = 1.f;
    set_direction(p, r.dir[0], r.dir[1], r.dir[2]);
    float t;
    int best;
    sweep_rows(geom, pairs, 0, n_pad, p, tmin, tmax, t, best);
    rtz_ray_hit h = {best, 0, t, p.len, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    if (best >= 0) {
        const float gx = geom[best].x, gy = geom[best].y, gz = geom[best].z;
        const float px = fmaf(t, p.dx, p.ox), py = fmaf(t, p.dy, p.oy), pz = fmaf(t, p.dz, p.oz);
        float nx = (px - gx) * aux[best].y, ny = (py - gy) * aux[best].y, nz = (pz - gz) * aux[best].y;
        const bool front = fmaf(p.dz, nz, fmaf(p.dy, ny, p.dx * nx)) < 0.f;
        if (!front) nx = -nx, ny = -ny, nz = -nz;
        h.front = front, h.point[0] = px, h.point[1] = py, h.point[2] = pz, h.normal[0] = nx, h.normal[1] = ny, h.normal[2] = nz;
    }
    out[k] = h;
}

__global__ void probe_scatters_kernel(DevCamera cam, const float4* geom, const float4* pairs, const float4* aux,
                                      const float4* albedo, const rtz_probe_bounce* recs, uint64_t m,
                                      rtz_ray_scatter* out) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const rtz_probe_bounce r = recs[k];
    Path p;
    p.ox = r.orig[0], p.oy = r.orig[1], p.oz = r.orig[2], p.self = -1, p.bounce = r.bounce, p.tr = p.tg = p.tb = 1.f;
    set_direction(p, r.dir[0], r.dir[1], r.dir[2]);
    float t;
    int best;
    sweep_rows(geom, pairs, r.sphere, 1, p, cam.tmin, cam.tmax, t, best);  // Sphere.hit on that one sphere
    rtz_ray_scatter s = {-2, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, 0.f, {0.f, 0.f, 0.f}};
    if (best >= 0) {
        const RngKey key{cam.key0, cam.key1, r.pixel, r.sample};
        float sr, sg, sb;
        int term = -1;
        if (shade(cam, key, geom, aux, albedo, p, t, best, sr, sg, sb, term)) {
            s.term = term;
        } else {
            s.term = -1;
            s.orig[0] = p.ox, s.orig[1] = p.oy, s.orig[2] = p.oz;
            s.dir[0] = p.dx, s.dir[1] = p.dy, s.dir[2] = p.dz, s.len = p.len;
            s.attenuation[0] = p.tr, s.attenuation[1] = p.tg, s.attenuation[2] = p.tb;
        }
    }
    out[k] = s;
}

__global__ void probe_camera_ray_kernel(DevCamera cam, uint32_t i, uint32_t j, uint32_t sample0, uint32_t n, float* o,
                                        float* d, float* len) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const RngKey key{cam.key0, cam.key1, j * cam.width + i, sample0 + k};
    Path p;
    camera_ray(cam, key, i, j, p);
    o[3 * k + 0] = p.ox, o[3 * k + 1] = p.oy, o[3 * k + 2] = p.oz;
    d[3 * k + 0] = p.dx, d[3 * k + 1] = p.dy, d[3 * k + 2] = p.dz;
    if (len) len[k] = p.len;
}

__global__ void probe_to_rgb_kernel(const double* lin, uint64_t n3, uint8_t* out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n3) out[i] = to_byte(lin[i]);
}

__global__ void probe_uniform_kernel(uint32_t k0, uint32_t k1, uint32_t pixel, uint32_t sample, uint32_t bounce,
                                     uint64_t n, float* out) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * b >= n) return;
    const uint4 r = philox4x32_10(pixel, sample, bounce, (uint32_t)b, k0, k1);
    const float v[4] = {u01(r.x), u01(r.y), u01(r.z), u01(r.w)};
    for (int q = 0; q < 4 && 4 * b + q < n; ++q) out[4 * b + q] = v[q];
}

// ---------------------------------------------------------------------------------------------
// FP32 pipe peak: independent FMA chains, no memory traffic.
// ---------------------------------------------------------------------------------------------
template <int kVariant>
__global__ void __launch_bounds__(256) ffma_peak_kernel(float a, float b, int iters, float* sink) {
    constexpr int C = 16;
    float x[C];
#pragma unroll
    for (int i = 0; i < C; ++i) x[i] = (float)(threadIdx.x + i) * 1e-3f;
    if (kVariant == 0) {  // scalar FFMA, 16 independent chains
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < C; ++i) x[i] = fmaf(x[i], a, b);
        }
    } else if (kVariant == 1) {  // packed FFMA2, all operands packed
        float2 aa = make_float2(a, a), bb = make_float2(b, b);
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < C; i += 2) {
                float2 v = __ffma2_rn(make_float2(x[i], x[i + 1]), aa, bb);
                x[i] = v.x, x[i + 1] = v.y;
            }
        }
    } else {  // packed FFMA2 with one scalar-broadcast operand (R.F32), as the sweep uses it
        float2 bb = make_float2(b, b);
        float s = a;
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < C; i += 2) {
                float2 v = __ffma2_rn(make_float2(x[i], x[i + 1]), make_float2(s, s), bb);
                x[i] = v.x, x[i + 1] = v.y;
            }
            s = __int_as_float(__float_as_int(s) ^ (it & 1));  // keep the scalar in a vector register
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < C; ++i) s += x[i];
    if (s == 123.456f) *sink = s;
}

}  // namespace rtz
