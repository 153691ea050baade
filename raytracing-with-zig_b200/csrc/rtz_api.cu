// rtz_api.cu — host side of librtz.so: the C ABI declared in include/rtz.h.
// Replaces the body of Camera.render (reference src/camera.zig:123-145) and PPM.saveBinary
// (src/ppm.zig:42-60).  There is no CPU fallback anywhere in this file: every compute entry
// point needs a CUDA device and fails with RTZ_ERR_NO_DEVICE / RTZ_ERR_CUDA otherwise.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only: libnccl.so.2 is dlopen()ed on first use (rtz_multi_*, RTZ_GATHER_NCCL)

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <map>
#include <mutex>
#include <thread>
#include <memory>
#include <string>
#include <vector>

#include "../../include/rtz.h"
#include "rtz_kernels.cuh"
#include "rtz_bvh.cuh"
#include "rtz_scene.cuh"

namespace {

thread_local std::string g_last_error;

#define RTZ_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) {                                                                    \
            g_last_error = std::string(#call) + ": " + cudaGetErrorString(e_);                      \
            return (e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver) ? RTZ_ERR_NO_DEVICE \
                                                                                  : RTZ_ERR_CUDA;   \
        }                                                                                           \
    } while (0)

uint64_t os_seed() {  // Scene.init with seed == null draws from getrandom (src/Scene.zig:33-36)
    uint64_t s = 0;
    FILE* f = std::fopen("/dev/urandom", "rb");
    if (f) {
        if (std::fread(&s, 1, sizeof(s), f) != sizeof(s)) s = 0x9e3779b97f4a7c15ULL;
        std::fclose(f);
    }
    return s;
}

inline float bits_to_float(int32_t v) {
    float f;
    std::memcpy(&f, &v, 4);
    return f;
}

// Entry points select the context's device; the caller's current device is restored on return.
struct DeviceGuard {
    int saved = -1;
    DeviceGuard() {
        if (cudaGetDevice(&saved) != cudaSuccess) saved = -1;
    }
    ~DeviceGuard() {
        if (saved >= 0) cudaSetDevice(saved);
    }
};

inline bool finite3(const double v[3]) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); }

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr, cap = 0;
        cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr, cap = 0;
    }
};

}  // namespace

struct rtz_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    size_t smem_optin = 0;
    int variant = 0;
    bool geo_const = true;   // scenes that fit the kernel-parameter space use the constant-bank kernel;
                             // RTZ_GEO_CONST=0 forces the TMA + shared-memory kernel
    // scene (device SoA f32 + the f64 copy the legacy kernel reads)
    DevBuf<float4> geom, pairs, aux, albedo;
    DevBuf<float> wexp;  // w of the pair layout as a plain row
    DevBuf<rtz::DSphere> dspheres;
    std::vector<float4> h_pairs;
    // padded boxes of the 32-sphere blocks (TraceParamsConst::boxes) and whether the constant-bank kernel culls with them
    std::vector<float4> h_boxes;
    float cull_r2 = 0.0f;
    bool cull = false;
    // ... and the rows that kernel and its drain read: the spheres regrouped into compact blocks (sweep_order), slot s
    // holding sphere rg_orig[s] of the caller's list.  Uploaded only for a scene that is culled.
    DevBuf<float4> rg_geom, rg_aux, rg_albedo;
    DevBuf<float> rg_wexp;
    DevBuf<int> rg_orig;
    std::vector<float4> h_rg_pairs;
    // RTZ_MODE_PATH_BVH (extension): hierarchy over the same FP32 spheres, built on the first render that
    // asks for it (h_geom / h_w are the host copies it is built from)
    DevBuf<rtz::BvhNode> bvh_nodes;
    DevBuf<int> bvh_order;
    std::vector<float4> h_geom;
    std::vector<float> h_w;
    bool bvh_ready = false;
    int n_spheres = 0, n_pad = 0;
    // frame state
    DevBuf<unsigned long long> accum;
    DevBuf<unsigned long long> counters;  // [0] queue head, [1..4] stats, [5] BVH tests, [6] NaN samples, [8] drain pool {parked, next}
    DevBuf<float4> pool;                  // drain pool: 4 float4 per parked path, 64 paths per resident warp
    uint64_t frame_launches = 0;          // kernels launched for the frame in flight
    DevBuf<unsigned long long> timeline;  // RTZ_TIMELINE=1: per-warp {start, queue dry, done} stamps of the last frame
    DevBuf<uint8_t> rgb;                  // used by the host-buffer entry points
    DevBuf<double> linear;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    unsigned long long* h_counters = nullptr;  // pinned
};

namespace {

int32_t shard_geom(uint64_t W, uint64_t H, const rtz_shard* s, rtz::ShardGeom& g) {
    rtz_shard d{0, 1, (uint32_t)W, 1};  // whole frame: tiles are rows -> compact layout == row-major image
    if (s) d = *s;
    if (d.world == 0 || d.rank >= d.world || d.tile_w == 0 || d.tile_h == 0) return RTZ_ERR_BAD_ARG;
    g.rank = d.rank, g.world = d.world, g.tile_w = d.tile_w, g.tile_h = d.tile_h;
    g.tiles_x = (uint32_t)((W + d.tile_w - 1) / d.tile_w);
    g.tiles_y = (uint32_t)((H + d.tile_h - 1) / d.tile_h);
    const uint64_t tiles = (uint64_t)g.tiles_x * g.tiles_y;
    // every rank gets the size of rank 0 (the largest) so gathered buffers are equal-sized
    g.n_local_tiles = (uint32_t)((tiles + d.world - 1) / d.world);
    const uint64_t tile_pixels = (uint64_t)d.tile_w * d.tile_h;
    if (tile_pixels > 0xFFFFFFFFull || (uint64_t)g.n_local_tiles * tile_pixels > 0xFFFFFFFFull) return RTZ_ERR_BAD_ARG;
    g.tile_pixels = (uint32_t)tile_pixels;
    return RTZ_OK;
}

int32_t check_camera(const rtz_camera* c) {
    if (!c || c->width == 0 || c->height == 0) return RTZ_ERR_BAD_ARG;
    if (c->width > 0xFFFFFFFFull || c->height > 0xFFFFFFFFull || c->width * c->height > 0xFFFFFFFFull) return RTZ_ERR_BAD_ARG;
    // a NaN / infinite camera would only produce NaN samples: refuse it up front (t_max may be +inf, Scene.zig:21)
    if (!finite3(c->center) || !finite3(c->pixel0) || !finite3(c->du) || !finite3(c->dv) || !finite3(c->defocus_disk_u) ||
        !finite3(c->defocus_disk_v) || !std::isfinite(c->defocus_angle) || !std::isfinite(c->pixel_samples_scale) ||
        !std::isfinite(c->t_min) || std::isnan(c->t_max)) {
        g_last_error = "camera has a non-finite field";
        return RTZ_ERR_BAD_ARG;
    }
    if (c->mode < RTZ_MODE_PATH || c->mode > RTZ_MODE_PATH_BVH) return RTZ_ERR_BAD_ARG;
    if (c->samples_per_pixel == 0 || c->samples_per_pixel > 0x7FFFFFFFull) return RTZ_ERR_BAD_ARG;
    if (c->mode != RTZ_MODE_PATH && c->mode != RTZ_MODE_PATH_BVH && c->samples_per_pixel != 1) return RTZ_ERR_BAD_ARG;
    if (c->bounce_max > 0xFFFFFFFFull) return RTZ_ERR_BAD_ARG;
    return RTZ_OK;
}

rtz::DevCamera to_dev_camera(const rtz_camera& c, uint64_t seed) {
    rtz::DevCamera d;
    d.p0x = (float)c.pixel0[0], d.p0y = (float)c.pixel0[1], d.p0z = (float)c.pixel0[2];
    d.dux = (float)c.du[0], d.duy = (float)c.du[1], d.duz = (float)c.du[2];
    d.dvx = (float)c.dv[0], d.dvy = (float)c.dv[1], d.dvz = (float)c.dv[2];
    d.cx = (float)c.center[0], d.cy = (float)c.center[1], d.cz = (float)c.center[2];
    d.uux = (float)c.defocus_disk_u[0], d.uuy = (float)c.defocus_disk_u[1], d.uuz = (float)c.defocus_disk_u[2];
    d.vvx = (float)c.defocus_disk_v[0], d.vvy = (float)c.defocus_disk_v[1], d.vvz = (float)c.defocus_disk_v[2];
    d.tmin = (float)c.t_min;
    d.tmax = (float)c.t_max;
    d.defocus = c.defocus_angle > 0 ? 1 : 0;  // src/camera.zig:191
    d.width = (uint32_t)c.width, d.height = (uint32_t)c.height;
    d.spp = (uint32_t)c.samples_per_pixel, d.bounce_max = (uint32_t)c.bounce_max;
    d.key0 = (uint32_t)seed, d.key1 = (uint32_t)(seed >> 32);
    for (uint32_t r = 0; r < 10; ++r) d.rk0[r] = d.key0 + r * 0x9E3779B9u, d.rk1[r] = d.key1 + r * 0xBB67AE85u;
    return d;
}

// Work chunks: runs of <= 128 samples of ONE pixel (RTZ_CHUNK overrides the cap: experiments; the image does not
// depend on it).  A warp keeps its chunk until it is used up, so the chunk bounds how long the last warps run on
// after the queue is dry: measured on 1/8 shards of C3, 128 beats 256 (19.79 vs 19.95 ms) and 64 (19.88 ms).  Schedules that cut the END of the queue into small or across-pixel chunks, reorder it (pixels
// that look into glass first) or let drained warps sweep sphere-parallel were built and measured in round 2
// (DESIGN.md §5): with the drain kernel none of them is needed, and the reordering even costs 2 %.
void pick_chunks(const rtz_context* ctx, rtz::TraceParams& P, uint64_t n_local_pixels) {
    // long frames (>= 128 big chunks per resident warp: C3 whole, C4) take 256, where the per-chunk bookkeeping still
    // shows (155.1 vs 155.9 ms on C3); short ones (a 1/8 shard of C3: 57 per warp) take 128 for the shorter tail
    const uint64_t big_chunks_per_warp = n_local_pixels * P.cam.spp / (256ull * (uint64_t)ctx->sm_count * 24);
    uint32_t cap = big_chunks_per_warp >= 128 ? 256u : 128u;
    if (const char* e = std::getenv("RTZ_CHUNK")) cap = (uint32_t)std::max(1, std::atoi(e));
    P.chunk = P.cam.spp < cap ? P.cam.spp : cap;
    P.chunks_per_pixel = (P.cam.spp + P.chunk - 1) / P.chunk;
    P.n_local_pixels = (uint32_t)n_local_pixels;
    P.n_chunks = n_local_pixels * P.chunks_per_pixel;
}

template <class Kern, class Params>
int32_t launch_trace(rtz_context* ctx, Kern kern, const Params& P, uint64_t n_chunks, int block, size_t smem) {
    if (smem) RTZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    RTZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, block, smem));
    if (per_sm < 1) {
        g_last_error = "scene does not fit in shared memory";
        return RTZ_ERR_TOO_MANY_SPHERES;
    }
    // persistent grid: every SM full, but never more warps than chunks of work
    uint64_t blocks = (uint64_t)ctx->sm_count * per_sm;
    const uint64_t max_useful = (n_chunks + (block / 32) - 1) / (block / 32);
    if (blocks > max_useful) blocks = max_useful ? max_useful : 1;
    kern<<<(unsigned)blocks, block, smem, ctx->stream>>>(P);
    RTZ_CUDA(cudaGetLastError());
    return RTZ_OK;
}

// RTZ_MODE_PATH_BVH (extension) needs the hierarchy: built on the host from the FP32 spheres the first time a
// render asks for it, so that plain uploads (and every brute-force frame) never pay for it.
int32_t ensure_bvh(rtz_context* c);

// What one device contributes to a frame.  `image` set: the resolve stores every channel at its place in the
// ROW-MAJOR image (possibly peer memory of device 0) instead of the compact tile buffer `d_rgb`.
struct FrameTarget {
    uint8_t* d_rgb = nullptr;
    double* d_linear = nullptr;
    uint8_t* image = nullptr;
};

// Enqueue the frame (memsets, trace kernel, resolve, counter read-back) on the context's stream; no host wait.
int32_t enqueue_path(rtz_context* ctx, const rtz_camera* cam, const rtz::ShardGeom& sg, const FrameTarget& out,
                     uint64_t seed) {
    if (ctx->n_spheres < 0) return RTZ_ERR_BAD_ARG;  // an empty world is a valid HittableList: every ray sees the sky
    const uint64_t n_local_pixels = (uint64_t)sg.n_local_tiles * sg.tile_pixels;
    if (n_local_pixels > 0xFFFFFFFFull) return RTZ_ERR_BAD_ARG;
    if (cam->mode == RTZ_MODE_PATH_BVH) {
        const int32_t rc = ensure_bvh(ctx);
        if (rc != RTZ_OK) return rc;
    }
    RTZ_CUDA(ctx->accum.reserve(3 * n_local_pixels));
    rtz::TraceParams P;
    P.cam = to_dev_camera(*cam, seed);
    P.sh = sg;
    P.geom = ctx->geom.p, P.pairs = ctx->pairs.p, P.aux = ctx->aux.p, P.albedo = ctx->albedo.p, P.wexp = ctx->wexp.p;
    P.orig = nullptr;
    P.n_spheres = ctx->n_spheres, P.n_pad = ctx->n_pad;
    pick_chunks(ctx, P, n_local_pixels);
    P.accum = ctx->accum.p;
    P.counter = ctx->counters.p;
    P.stats = ctx->counters.p + 1;
    {
        // wavefront kernel: a shading or camera-ray pass over r < 32 paths is worth running when it costs less than
        // sweeping those r paths once more (r/64 of a sweep); measured optimum (same-box A/B, profiles/r2_wave_ab.txt):
        // 16 of 32 lanes up to 32 spheres, 12 at 64, 8 from 128 on
        P.wave_shade_min = P.wave_regen_min = ctx->n_pad <= 32 ? 16u : ctx->n_pad <= 64 ? 12u : 8u;
        auto rcp = [](uint64_t d) -> unsigned long long {  // ceil(2^64 / d); 0 stands for d = 1
            return d <= 1 ? 0ull : (unsigned long long)(((unsigned __int128)1 << 64) / d) + 1ull;  // d never divides 2^64 unless a power of two: then +1 overshoots by one ulp, still exact for n < 2^32
        };
        P.rcp_tile_pixels = rcp(sg.tile_pixels), P.rcp_tiles_x = rcp(sg.tiles_x), P.rcp_tile_w = rcp(sg.tile_w);
        P.rcp_chunks_per_pixel = rcp(P.chunks_per_pixel);
        if (const char* e = std::getenv("RTZ_WAVE_SHADE_MIN")) P.wave_shade_min = (uint32_t)std::min(32, std::max(1, std::atoi(e)));
        if (const char* e = std::getenv("RTZ_WAVE_REGEN_MIN")) P.wave_regen_min = (uint32_t)std::min(32, std::max(1, std::atoi(e)));
    }
    P.timeline = nullptr;
    if (const char* e = std::getenv("RTZ_TIMELINE")) {  // diagnostics: tools/tail_timeline.py reads the file back
        if (e[0] == '1') {
            RTZ_CUDA(ctx->timeline.reserve(4 * 65536));
            RTZ_CUDA(cudaMemsetAsync(ctx->timeline.p, 0, 4 * 65536 * sizeof(unsigned long long), ctx->stream));
            P.timeline = ctx->timeline.p;
        }
    }
    // drain pool (RTZ_DRAIN=0: the warps finish their own paths in lockstep, as in round 1)
    P.pool = nullptr, P.pool_count = reinterpret_cast<unsigned int*>(ctx->counters.p + 8);
    const char* de = std::getenv("RTZ_DRAIN");
    const bool drain = cam->mode == RTZ_MODE_PATH && ctx->variant != 4 && P.cam.bounce_max > 0 && !(de && de[0] == '0');
    if (drain) {
        RTZ_CUDA(ctx->pool.reserve(4ull * 64 * 32 * (size_t)ctx->sm_count * 2));  // 64 paths per warp, <= 64 warps per SM
        P.pool = ctx->pool.p;
    }
    const bool use_const = ctx->n_pad <= rtz::kMaxConstSpheres && ctx->geo_const;
    const size_t smem = use_const ? 0 : (size_t)ctx->n_pad * 32;  // pair layout + per-lane rows
    // too large to stage next to the kernel's own static shared memory (ray staging rows): read it from L1/L2
    cudaFuncAttributes fa{};
    RTZ_CUDA(cudaFuncGetAttributes(&fa, rtz::trace_kernel_smem<512, 1>));
    const bool use_global = !use_const && smem + fa.sharedSizeBytes + 1024 > ctx->smem_optin;
    RTZ_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    RTZ_CUDA(cudaMemsetAsync(ctx->accum.p, 0, 3 * n_local_pixels * sizeof(unsigned long long), ctx->stream));
    RTZ_CUDA(cudaMemsetAsync(ctx->counters.p, 0, 16 * sizeof(unsigned long long), ctx->stream));
    RTZ_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    ctx->frame_launches = P.cam.bounce_max == 0 ? 1 : 2;
    int32_t rc = RTZ_OK;
    if (P.cam.bounce_max == 0) {
        // `while (bounces < bounceMax)` never runs (src/camera.zig:153): every sample is black and no
        // world.hit is made.  Nothing to trace; the zeroed sums resolve to zeros.
    } else if (cam->mode == RTZ_MODE_PATH_BVH) {
        rtz::BvhParams B{P, ctx->bvh_nodes.p, ctx->bvh_order.p, ctx->wexp.p};
        rc = launch_trace(ctx, rtz::trace_kernel_bvh<128, 6>, B, P.n_chunks, 128, 0);
    } else if (use_const) {
        static thread_local rtz::TraceParamsConst C;  // 8 KiB: keep it off the stack
        C.p = P;
        std::memcpy(C.pairs, ctx->h_pairs.data(), (size_t)ctx->n_pad * sizeof(float4));
        // <128,6> (80 registers, 24 warps/SM) is the measured best; the uniform loads want occupancy
        const bool wave_ok = P.n_chunks <= 0xFFFFFFFFull;  // the wavefront kernel's chunk bookkeeping is 32-bit
        if (ctx->variant == 4)  // experimental: 4 paths per thread, path state parked in shared memory (DESIGN.md §5)
            rc = launch_trace(ctx, rtz::trace_kernel_const_parked<4, 128, 6>, C, P.n_chunks, 128, 0);
        else if (ctx->variant == 1)
            rc = launch_trace(ctx, rtz::trace_kernel_const<256, 3>, C, P.n_chunks, 256, 0);
        else if (ctx->variant == 2)
            rc = launch_trace(ctx, rtz::trace_kernel_const<128, 5>, C, P.n_chunks, 128, 0);
        else if (ctx->variant == 6)  // 28 warps per SM at 72 registers (experiment)
            rc = launch_trace(ctx, rtz::trace_kernel_const<128, 7>, C, P.n_chunks, 128, 0);
        else if (ctx->variant == 7)  // 32 warps per SM at 64 registers (experiment)
            rc = launch_trace(ctx, rtz::trace_kernel_const<128, 8>, C, P.n_chunks, 128, 0);
        else if (ctx->variant == 9 && wave_ok)  // wavefront kernel at 40 / 36 warps per SM (experiments: no faster than 32)
            rc = launch_trace(ctx, rtz::trace_kernel_wave<128, 10>, C, P.n_chunks, 128, 0);
        else if (ctx->variant == 10 && wave_ok)
            rc = launch_trace(ctx, rtz::trace_kernel_wave<128, 9>, C, P.n_chunks, 128, 0);
        else if (wave_ok && (ctx->variant == 8 || (ctx->variant == 0 && ctx->n_pad <= 32)))
            // shading-bound scenes: the warp-level wavefront organisation (compacted shading / camera-ray passes), 64
            // paths per warp.  Same-box A/B against the lockstep kernel: 1.18x at 16 spheres, 1.14x at 32
            // (profiles/r2_wave_ab.txt).  RTZ_VARIANT=11 forces the lockstep kernel, 8 / 12 the two wavefront kernels.
            rc = launch_trace(ctx, rtz::trace_kernel_wave<128, 8>, C, P.n_chunks, 128, 0);
        else if (wave_ok && (ctx->variant == 12 || (ctx->variant == 0 && ctx->n_pad <= rtz::kMaxWaveSpheres)))
            // ... with 128 paths per warp (four per lane) where the sweep is a third to two thirds of the work: 1.10x at
            // 64 spheres, 1.06x at 128, 1.015x at 256; 0.99x at 512 and on C3, where the lockstep kernel stays
            rc = launch_trace(ctx, rtz::trace_kernel_wave_n<4, 128, 6>, C, P.n_chunks, 128, 0);
        else if (ctx->n_pad <= 64)
            // lockstep kernel on a shading-bound scene: warps, not registers (<128,8>: 64 registers, 32 warps per SM)
            rc = launch_trace(ctx, rtz::trace_kernel_const<128, 8>, C, P.n_chunks, 128, 0);
        else if (ctx->cull) {
            // the culled kernel, and the drain after it, work on the regrouped rows: sphere indices (hits, Path.self,
            // parked paths) are slots throughout, and only exact ties in t look up the original index.  The device
            // pair rows have no reader here (the sweep reads C.pairs, the drain the plain rows).
            P.geom = ctx->rg_geom.p, P.aux = ctx->rg_aux.p, P.albedo = ctx->rg_albedo.p, P.wexp = ctx->rg_wexp.p;
            P.orig = ctx->rg_orig.p, P.pairs = nullptr;
            C.p = P;
            std::memcpy(C.pairs, ctx->h_rg_pairs.data(), (size_t)ctx->n_pad * sizeof(float4));
            std::memcpy(C.boxes, ctx->h_boxes.data(), ctx->h_boxes.size() * sizeof(float4));
            C.cull_r2 = ctx->cull_r2;
            // culled blocks that at most this many of a warp's 64 paths reach are swept sphere-parallel (sweep2);
            // RTZ_SPLIT overrides it for tests and A/B runs (0: the packed sweep alone, 64: every reached block
            // sphere-parallel).  The image does not depend on it.
            C.split_max = rtz::kSplitMax;
            if (const char* e = std::getenv("RTZ_SPLIT")) C.split_max = std::atoi(e);
            rc = launch_trace(ctx, rtz::trace_kernel_const_cull<128, 6>, C, P.n_chunks, 128, 0);
        } else
            rc = launch_trace(ctx, rtz::trace_kernel_const<128, 6>, C, P.n_chunks, 128, 0);
    } else if (use_global) {
        rc = launch_trace(ctx, rtz::trace_kernel_global<128, 5>, P, P.n_chunks, 128, 0);
    } else {
        // Launch shape: the one that keeps most warps resident for this scene's shared-memory
        // footprint.  <128,5> (94 registers, 20 warps/SM) is the measured best while five CTAs fit;
        // large scenes trade CTAs for wider CTAs.  RTZ_VARIANT=1..3 forces a shape (experiments).
        int occ[3] = {0, 0, 0};
        RTZ_CUDA(cudaFuncSetAttribute(rtz::trace_kernel_smem<128, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        RTZ_CUDA(cudaFuncSetAttribute(rtz::trace_kernel_smem<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        RTZ_CUDA(cudaFuncSetAttribute(rtz::trace_kernel_smem<512, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        RTZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[0], rtz::trace_kernel_smem<128, 5>, 128, smem));
        RTZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[1], rtz::trace_kernel_smem<256, 2>, 256, smem));
        RTZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[2], rtz::trace_kernel_smem<512, 1>, 512, smem));
        const int warps[3] = {occ[0] * 4, occ[1] * 8, occ[2] * 16};
        int shape = 0;
        for (int k = 1; k < 3; ++k)
            if (warps[k] > warps[shape]) shape = k;
        if (ctx->variant >= 1 && ctx->variant <= 3) shape = ctx->variant - 1;
        switch (shape) {
            case 1: rc = launch_trace(ctx, rtz::trace_kernel_smem<256, 2>, P, P.n_chunks, 256, smem); break;
            case 2: rc = launch_trace(ctx, rtz::trace_kernel_smem<512, 1>, P, P.n_chunks, 512, smem); break;
            default: rc = launch_trace(ctx, rtz::trace_kernel_smem<128, 5>, P, P.n_chunks, 128, smem); break;
        }
    }
    if (rc != RTZ_OK) return rc;
    if (drain) {  // finish what the trace kernel parked: persistent grid, one warp (or, below 64 spheres, one thread) per path
        const unsigned blocks = (unsigned)ctx->sm_count * 8;
        if (ctx->n_spheres >= 64)
            rtz::drain_kernel<true><<<blocks, 128, 0, ctx->stream>>>(P);
        else
            rtz::drain_kernel<false><<<blocks, 128, 0, ctx->stream>>>(P);
        RTZ_CUDA(cudaGetLastError());
        ctx->frame_launches += 1;
    }
    RTZ_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    const uint64_t n3 = 3 * n_local_pixels;
    if (out.image)
        rtz::resolve_scatter_kernel<<<(unsigned)((n3 + 255) / 256), 256, 0, ctx->stream>>>(
            ctx->accum.p, sg, (uint32_t)cam->width, (uint32_t)cam->height, cam->pixel_samples_scale, out.image);
    else
        rtz::resolve_kernel<<<(unsigned)((n3 + 255) / 256), 256, 0, ctx->stream>>>(
            ctx->accum.p, n_local_pixels, cam->pixel_samples_scale, out.d_rgb, out.d_linear);
    RTZ_CUDA(cudaGetLastError());
    RTZ_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
    RTZ_CUDA(cudaMemcpyAsync(ctx->h_counters, ctx->counters.p, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                             ctx->stream));
    return RTZ_OK;
}

// Wait for the frame enqueued by enqueue_path and report the work it did.
int32_t collect_path(rtz_context* ctx, const rtz_camera* cam, const rtz::ShardGeom& sg, rtz_stats* st, uint64_t seed) {
    RTZ_CUDA(cudaStreamSynchronize(ctx->stream));
    if (const char* path = std::getenv("RTZ_TIMELINE_OUT")) {
        if (ctx->timeline.p && std::getenv("RTZ_TIMELINE") && std::getenv("RTZ_TIMELINE")[0] == '1') {
            std::vector<unsigned long long> h(4 * 65536);
            RTZ_CUDA(cudaMemcpy(h.data(), ctx->timeline.p, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            if (FILE* f = std::fopen(path, "wb")) {
                std::fwrite(h.data(), sizeof(unsigned long long), h.size(), f);
                std::fclose(f);
            }
        }
    }
    if (st) {
        std::memset(st, 0, sizeof(*st));
        st->samples = ctx->h_counters[1], st->segments = ctx->h_counters[2];
        if (cam->bounce_max == 0) {  // counted on the host: the kernel did not run
            uint64_t px = 0;
            for (uint32_t t = sg.rank; t < (uint64_t)sg.tiles_x * sg.tiles_y; t += sg.world) {
                const uint32_t ty = t / sg.tiles_x, tx = t - ty * sg.tiles_x;
                const uint64_t w = std::min<uint64_t>(sg.tile_w, cam->width - (uint64_t)tx * sg.tile_w);
                const uint64_t h = std::min<uint64_t>(sg.tile_h, cam->height - (uint64_t)ty * sg.tile_h);
                px += w * h;
            }
            st->samples = px * cam->samples_per_pixel;
        }
        st->depth_capped = ctx->h_counters[3], st->absorbed = ctx->h_counters[4];
        st->sphere_tests = cam->mode == RTZ_MODE_PATH_BVH ? ctx->h_counters[5] : st->segments * (uint64_t)ctx->n_spheres;
        st->nan_samples = ctx->h_counters[6];
        st->kernel_launches = ctx->frame_launches;
        st->gpus = 1;
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2]), st->trace_ms = ms;
        cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]), st->resolve_ms = ms;
        cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[3]), st->total_ms = ms;
        st->seed_used = seed;
    }
    return RTZ_OK;
}

int32_t render_path(rtz_context* ctx, const rtz_camera* cam, const rtz::ShardGeom& sg, uint8_t* d_rgb,
                    double* d_linear, rtz_stats* st, uint64_t seed) {
    FrameTarget out;
    out.d_rgb = d_rgb, out.d_linear = d_linear;
    const int32_t rc = enqueue_path(ctx, cam, sg, out, seed);
    if (rc != RTZ_OK) return rc;
    return collect_path(ctx, cam, sg, st, seed);
}

int32_t render_legacy(rtz_context* ctx, const rtz_camera* cam, uint8_t* d_rgb, double* d_linear, rtz_stats* st) {
    rtz::LegacyParams P;
    for (int k = 0; k < 3; ++k) P.p0[k] = cam->pixel0[k], P.du[k] = cam->du[k], P.dv[k] = cam->dv[k], P.c[k] = cam->center[k];
    P.tmin = cam->t_min, P.tmax = cam->t_max;
    P.width = (uint32_t)cam->width, P.height = (uint32_t)cam->height;
    P.mode = cam->mode, P.n = ctx->n_spheres, P.spheres = ctx->dspheres.p;
    const uint32_t n = P.width * P.height;
    RTZ_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    rtz::legacy_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(P, d_rgb, d_linear);
    RTZ_CUDA(cudaGetLastError());
    RTZ_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
    RTZ_CUDA(cudaStreamSynchronize(ctx->stream));
    if (st) {
        std::memset(st, 0, sizeof(*st));
        st->samples = n;
        st->segments = cam->mode == RTZ_MODE_LEGACY_SKY ? 0 : n;
        st->sphere_tests = st->segments * (uint64_t)ctx->n_spheres;
        st->kernel_launches = 1;
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[3]), st->trace_ms = st->total_ms = ms;
    }
    return RTZ_OK;
}

struct ScopedCtx {  // context for the one-shot entry points
    rtz_context* c = nullptr;
    ~ScopedCtx() {
        if (c) rtz_context_destroy(c);
    }
};

}  // namespace

// =================================================================================================
extern "C" {

int32_t rtz_abi_version(void) { return RTZ_ABI_VERSION; }

const char* rtz_strerror(int32_t s) {
    switch (s) {
        case RTZ_OK: return "ok";
        case RTZ_ERR_BAD_ARG: return "bad argument";
        case RTZ_ERR_NO_DEVICE: return "no CUDA device (librtz has no CPU fallback)";
        case RTZ_ERR_CUDA: return "CUDA error";
        case RTZ_ERR_IO: return "I/O error";
        case RTZ_ERR_TOO_MANY_SPHERES: return "scene does not fit in shared memory";
        case RTZ_ERR_ARCH: return "device is not sm_100 (librtz ships sm_100a code only)";
        case RTZ_ERR_NCCL: return "NCCL error (libnccl.so.2 missing or a collective failed)";
        default: return "unknown status";
    }
}
const char* rtz_last_error(void) { return g_last_error.c_str(); }

int32_t rtz_device_count(int32_t* count_out) {
    if (!count_out) return RTZ_ERR_BAD_ARG;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        g_last_error = cudaGetErrorString(e);
        *count_out = 0;
        return RTZ_ERR_NO_DEVICE;
    }
    *count_out = n;
    return n > 0 ? RTZ_OK : RTZ_ERR_NO_DEVICE;
}

int32_t rtz_context_create(int32_t device, void* stream, rtz_context** out) {
    if (!out) return RTZ_ERR_BAD_ARG;
    *out = nullptr;
    int n = 0;
    int32_t rc = rtz_device_count(&n);
    if (rc != RTZ_OK) return rc;
    DeviceGuard guard;
    if (device < 0) RTZ_CUDA(cudaGetDevice(&device));
    if (device >= n) return RTZ_ERR_BAD_ARG;
    RTZ_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RTZ_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10 || prop.minor != 0) {  // sm_100a SASS only runs on compute capability 10.0
        g_last_error = std::string("device ") + prop.name + " is sm_" + std::to_string(prop.major * 10 + prop.minor);
        return RTZ_ERR_ARCH;
    }
    rtz_context* c = new rtz_context();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    if (const char* e = std::getenv("RTZ_GEO_CONST")) c->geo_const = e[0] == '1';
    if (const char* e = std::getenv("RTZ_VARIANT")) c->variant = std::atoi(e);
    if (stream) {
        c->stream = (cudaStream_t)stream;
    } else {
        cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            delete c;
            g_last_error = cudaGetErrorString(e);
            return RTZ_ERR_CUDA;
        }
        c->own_stream = true;
    }
    for (auto& e : c->ev) cudaEventCreate(&e);
    cudaMallocHost(&c->h_counters, 8 * sizeof(unsigned long long));
    if (c->counters.reserve(16) != cudaSuccess || !c->h_counters) {
        rtz_context_destroy(c);
        g_last_error = "allocation failed";
        return RTZ_ERR_CUDA;
    }
    *out = c;
    return RTZ_OK;
}

int32_t rtz_context_destroy(rtz_context* c) {
    if (!c) return RTZ_ERR_BAD_ARG;
    DeviceGuard guard;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    c->geom.release(), c->pairs.release(), c->aux.release(), c->albedo.release(), c->dspheres.release();
    c->accum.release(), c->counters.release(), c->rgb.release(), c->linear.release(), c->timeline.release(), c->pool.release();
    c->bvh_nodes.release(), c->bvh_order.release(), c->wexp.release();
    c->rg_geom.release(), c->rg_aux.release(), c->rg_albedo.release(), c->rg_wexp.release(), c->rg_orig.release();
    for (auto& e : c->ev)
        if (e) cudaEventDestroy(e);
    if (c->h_counters) cudaFreeHost(c->h_counters);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return RTZ_OK;
}

namespace {
// The order in which the culled kernel sweeps the spheres: slot -> index in the caller's list.  Sphere 0 (the
// ground of the book's scenes) keeps slot 0, since block 0 is always swept first; the others are split
// recursively at the median of the longest axis of their centres, with every cut on a multiple of 32 slots, so
// that each 32-sphere block is a compact cluster with a small box.  Equal coordinates are ordered by index and
// every final block is sorted by index: the order depends on the FP32 centres alone, the same on every device.
void regroup(const std::vector<float4>& g, std::vector<int>& idx, int first, int cnt, int slot0) {
    const int blocks = (slot0 + cnt + 31) / 32 - slot0 / 32;
    if (blocks <= 1) {
        std::sort(idx.begin() + first, idx.begin() + first + cnt);
        return;
    }
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int q = first; q < first + cnt; ++q) {
        const float c[3] = {g[idx[q]].x, g[idx[q]].y, g[idx[q]].z};
        for (int a = 0; a < 3; ++a) lo[a] = std::min(lo[a], c[a]), hi[a] = std::max(hi[a], c[a]);
    }
    int axis = 0;
    for (int a = 1; a < 3; ++a)
        if (hi[a] - lo[a] > hi[axis] - lo[axis]) axis = a;
    const int cut_slot = (slot0 / 32 + blocks / 2) * 32;
    const int left = cut_slot - slot0;
    auto key = [&](int i) { return axis == 0 ? g[i].x : axis == 1 ? g[i].y : g[i].z; };
    std::nth_element(idx.begin() + first, idx.begin() + first + left, idx.begin() + first + cnt,
                     [&](int x, int y) { return key(x) < key(y) || (key(x) == key(y) && x < y); });
    regroup(g, idx, first, left, slot0);
    regroup(g, idx, first + left, cnt - left, cut_slot);
}
std::vector<int> sweep_order(const std::vector<float4>& g, int n) {
    std::vector<int> idx(n);
    for (int i = 0; i < n; ++i) idx[i] = i;
    if (n > 1) regroup(g, idx, 1, n - 1, 1);
    return idx;
}

// sweep layout of the rows g / w: one FFMA2 = one ray x the two spheres of a pair
std::vector<float4> pair_rows(const std::vector<float4>& g, const std::vector<float>& w, int n_pad) {
    std::vector<float4> pr(std::max(n_pad, 1));
    for (int p = 0; p < n_pad / 2; ++p) {
        const float4 A = g[2 * p], B = g[2 * p + 1];
        pr[2 * p] = make_float4(A.x, B.x, A.y, B.y);
        pr[2 * p + 1] = make_float4(A.z, B.z, w[2 * p], w[2 * p + 1]);
    }
    return pr;
}

// Median-split BVH over the FP32 spheres {cx, cy, cz, -r^2} (RTZ_MODE_PATH_BVH).  Boxes are padded well beyond
// the rounding of the slab test and of the hit point, so the traversal is conservative.
struct BvhBuilder {
    const std::vector<float4>& g;
    std::vector<rtz::BvhNode> nodes;
    std::vector<int> order;
    explicit BvhBuilder(const std::vector<float4>& geom, int n) : g(geom), order(n) {
        for (int i = 0; i < n; ++i) order[i] = i;
    }
    void bounds(int first, int cnt, float lo[3], float hi[3]) const {
        for (int a = 0; a < 3; ++a) lo[a] = INFINITY, hi[a] = -INFINITY;
        for (int q = first; q < first + cnt; ++q) {
            const float4 s = g[order[q]];
            const float c[3] = {s.x, s.y, s.z};
            const float r = std::sqrt(-s.w);
            const float pad = 1e-4f * (1.0f + r + std::fabs(s.x) + std::fabs(s.y) + std::fabs(s.z));
            for (int a = 0; a < 3; ++a) lo[a] = std::min(lo[a], c[a] - r - pad), hi[a] = std::max(hi[a], c[a] + r + pad);
        }
    }
    // returns the child reference of the range: leaf code (< 0) or the index of a new inner node (>= 0)
    int build(int first, int cnt) {
        if (cnt <= 4) return -1 - (first * 8 + cnt);
        float clo[3] = {INFINITY, INFINITY, INFINITY}, chi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (int q = first; q < first + cnt; ++q) {
            const float4 s = g[order[q]];
            const float c[3] = {s.x, s.y, s.z};
            for (int a = 0; a < 3; ++a) clo[a] = std::min(clo[a], c[a]), chi[a] = std::max(chi[a], c[a]);
        }
        int axis = 0;
        for (int a = 1; a < 3; ++a)
            if (chi[a] - clo[a] > chi[axis] - clo[axis]) axis = a;
        const int half = cnt / 2;
        std::nth_element(order.begin() + first, order.begin() + first + half, order.begin() + first + cnt, [&](int x, int y) {
            const float cx = axis == 0 ? g[x].x : axis == 1 ? g[x].y : g[x].z;
            const float cy = axis == 0 ? g[y].x : axis == 1 ? g[y].y : g[y].z;
            return cx < cy || (cx == cy && x < y);
        });
        const int me = (int)nodes.size();
        nodes.emplace_back();
        const int c0 = build(first, half), c1 = build(first + half, cnt - half);
        rtz::BvhNode& nd = nodes[me];
        bounds(first, half, nd.lo0, nd.hi0);
        bounds(first + half, cnt - half, nd.lo1, nd.hi1);
        nd.child0 = c0, nd.child1 = c1, nd.pad0 = nd.pad1 = 0;
        return me;
    }
    void run() {
        const int n = (int)order.size();
        nodes.reserve(n / 2 + 2);
        const int root = n > 0 ? build(0, n) : rtz::kBvhEmpty;
        if (root != 0) {  // fewer than five spheres (or none): a root whose first child is the only leaf
            rtz::BvhNode nd{};
            if (n > 0) bounds(0, n, nd.lo0, nd.hi0);
            nd.child0 = root, nd.child1 = rtz::kBvhEmpty;
            nodes.insert(nodes.begin(), nd);
        }
    }
};
}  // namespace

int32_t rtz_scene_upload(rtz_context* c, const rtz_sphere* sp, uint64_t n) {
    if (!c || (!sp && n) || n > (1u << 20)) return RTZ_ERR_BAD_ARG;
    DeviceGuard guard;
    RTZ_CUDA(cudaSetDevice(c->device));
    const int n_pad = (int)((n + 7) & ~7ull);
    std::vector<float4> g(n_pad ? n_pad : 1), a(n_pad ? n_pad : 1), al(n_pad ? n_pad : 1);
    std::vector<float> w(n_pad ? n_pad : 1);
    std::vector<rtz::DSphere> ds(n ? n : 1);
    for (uint64_t i = 0; i < n; ++i) {
        const rtz_sphere& s = sp[i];
        if (s.mat_type < RTZ_MAT_LAMBERTIAN || s.mat_type > RTZ_MAT_DIELECTRIC) return RTZ_ERR_BAD_ARG;
        const float r = (float)(s.radius < 0 ? 0.0 : s.radius);  // Sphere.init clamp (src/sphere.zig:21)
        // A radius-0 sphere makes the reference panic in Vec.divScalar (src/vec.zig:39-45) when it is hit, and
        // NaN / infinite geometry only yields NaN samples: both are refused here instead of rendered wrongly.
        const bool mat_ok = s.mat_type == RTZ_MAT_DIELECTRIC
                                ? (std::isfinite(s.refraction_index) && (float)s.refraction_index != 0.0f)
                                : (finite3(s.albedo) && (s.mat_type != RTZ_MAT_METAL || std::isfinite(s.fuzz)));
        if (!finite3(s.center) || !std::isfinite(s.radius) || !(r > 0.0f) || !mat_ok) {
            g_last_error = "sphere " + std::to_string(i) + ": radius must be > 0 and every field of its material finite";
            return RTZ_ERR_BAD_ARG;
        }
        const float cx = (float)s.center[0], cy = (float)s.center[1], cz = (float)s.center[2];
        // q = |c|^2 - r^2 of the FP32-rounded sphere less the per-sphere half of the gate's margin (kGateSlack at
        // ray_constants), evaluated in f64 and rounded once
        const double c2 = (double)cx * cx + (double)cy * cy + (double)cz * cz;
        const double q = (c2 - (double)r * r) - (double)rtz::kGateSlack * c2;
        g[i] = make_float4(cx, cy, cz, -(r * r));
        w[i] = -(float)q;
        const float param = s.mat_type == RTZ_MAT_METAL ? (float)s.fuzz : (float)s.refraction_index;
        a[i] = make_float4(r, 1.0f / r, param, bits_to_float(s.mat_type));
        al[i] = make_float4((float)s.albedo[0], (float)s.albedo[1], (float)s.albedo[2],
                            1.0f / (float)s.refraction_index);
        ds[i] = rtz::DSphere{s.center[0], s.center[1], s.center[2], s.radius < 0 ? 0.0 : s.radius};
    }
    for (int i = (int)n; i < n_pad; ++i) {  // padding: w = -inf  ->  disc = -inf (never a candidate)
        g[i] = make_float4(0.f, 0.f, 0.f, -0.f);
        w[i] = -INFINITY;
        a[i] = make_float4(0.f, 0.f, 0.f, bits_to_float(0));
        al[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    std::vector<float4> pr = pair_rows(g, w, n_pad);
    // Bounds of the culled kernel's 32-sphere blocks, on its regrouped order (box_reach in rtz_kernels.cuh states
    // the exactness contract these paddings serve).  R covers every ray origin within twice the farthest point of
    // a sphere outside block 0; block 0 (the ground of the book's scenes) has no box: it is always swept.
    const std::vector<int> order = sweep_order(g, (int)n);
    const int n_blocks = (n_pad + 31) / 32;
    std::vector<float4> bx(2 * (size_t)std::max(n_blocks, 1), make_float4(0.f, 0.f, 0.f, 0.f));
    double reach = 0.0;
    for (uint64_t q = 32; q < n; ++q) {
        const float4 s = g[order[q]];
        reach = std::max(reach, std::sqrt((double)s.x * s.x + (double)s.y * s.y + (double)s.z * s.z) + std::sqrt(-(double)s.w));
    }
    const double R = 2.0 * reach;
    double lo_all[3] = {INFINITY, INFINITY, INFINITY}, hi_all[3] = {-INFINITY, -INFINITY, -INFINITY}, vol_sum = 0.0;
    std::vector<double> vols;
    for (int b = 1; b < n_blocks; ++b) {
        double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (uint64_t q = 32ull * b; q < std::min<uint64_t>(n, 32ull * b + 32); ++q) {
            const float4 s = g[order[q]];
            const double c[3] = {s.x, s.y, s.z}, r = std::sqrt(-(double)s.w);
            const double cn = std::sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
            const double pad = 1e-4 * (1.0 + r + std::fabs(c[0]) + std::fabs(c[1]) + std::fabs(c[2])) +
                               1e-6 * (1.001 * R + cn) * (1.001 * R + cn) / r;
            for (int a = 0; a < 3; ++a) lo[a] = std::min(lo[a], c[a] - r - pad), hi[a] = std::max(hi[a], c[a] + r + pad);
        }
        float fl[3], fh[3];  // rounded outwards
        for (int a = 0; a < 3; ++a) {
            fl[a] = std::nextafter((float)lo[a], -INFINITY), fh[a] = std::nextafter((float)hi[a], INFINITY);
            lo_all[a] = std::min(lo_all[a], lo[a]), hi_all[a] = std::max(hi_all[a], hi[a]);
        }
        bx[2 * b] = make_float4(fl[0], fh[0], fl[1], fh[1]);
        bx[2 * b + 1] = make_float4(fl[2], fh[2], 0.f, 0.f);
        vols.push_back((hi[0] - lo[0]) * (hi[1] - lo[1]) * (hi[2] - lo[2]));
    }
    // Culling pays where the blocks are small against the region they share; where every block spans the scene the
    // box tests would be pure overhead, so the plain sweep runs.  Regrouped, even a uniform cloud of spheres has
    // compact blocks (485 in a cube: about 7 % each), and it is faster culled (DESIGN.md §5).
    for (double v : vols) vol_sum += v;
    const double vol_all = (hi_all[0] - lo_all[0]) * (hi_all[1] - lo_all[1]) * (hi_all[2] - lo_all[2]);
    const bool cull = n_pad <= rtz::kMaxConstSpheres && !vols.empty() && std::isfinite(R) &&
                      vol_sum < 0.25 * vols.size() * vol_all;
    // the rows of the culled kernel in its order; padding stays in slots n .. n_pad-1
    std::vector<float4> rg(cull ? n_pad : 0), ra(cull ? n_pad : 0), ral(cull ? n_pad : 0), rpr;
    std::vector<float> rw(cull ? n_pad : 0);
    std::vector<int> ro(cull ? n_pad : 0);
    if (cull) {
        for (int q = 0; q < n_pad; ++q) {
            const int i = q < (int)n ? order[q] : q;
            rg[q] = g[i], ra[q] = a[i], ral[q] = al[i], rw[q] = w[i], ro[q] = i;
        }
        rpr = pair_rows(rg, rw, n_pad);
    }
    // Not failure-atomic by itself (growing a buffer frees the old one), so the context holds NO scene from here
    // until every copy has been enqueued: a failed upload leaves an empty world behind, never stale geometry.
    c->n_spheres = c->n_pad = 0;
    c->h_pairs.clear(), c->h_rg_pairs.clear(), c->h_geom.clear(), c->h_w.clear();
    c->cull = false;
    c->bvh_ready = false;
    if (n_pad) {
        RTZ_CUDA(c->geom.reserve(n_pad));
        RTZ_CUDA(c->pairs.reserve(n_pad));
        RTZ_CUDA(c->aux.reserve(n_pad));
        RTZ_CUDA(c->albedo.reserve(n_pad));
        RTZ_CUDA(c->wexp.reserve(n_pad));
        RTZ_CUDA(cudaMemcpyAsync(c->wexp.p, w.data(), n_pad * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        // pageable sources: cudaMemcpyAsync returns once the bytes are staged, so the vectors may die at return
        RTZ_CUDA(cudaMemcpyAsync(c->geom.p, g.data(), n_pad * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RTZ_CUDA(cudaMemcpyAsync(c->pairs.p, pr.data(), n_pad * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RTZ_CUDA(cudaMemcpyAsync(c->aux.p, a.data(), n_pad * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RTZ_CUDA(cudaMemcpyAsync(c->albedo.p, al.data(), n_pad * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    }
    if (cull) {
        RTZ_CUDA(c->rg_geom.reserve(n_pad));
        RTZ_CUDA(c->rg_aux.reserve(n_pad));
        RTZ_CUDA(c->rg_albedo.reserve(n_pad));
        RTZ_CUDA(c->rg_wexp.reserve(n_pad));
        RTZ_CUDA(c->rg_orig.reserve(n_pad));
        RTZ_CUDA(cudaMemcpyAsync(c->rg_geom.p, rg.data(), n_pad * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RTZ_CUDA(cudaMemcpyAsync(c->rg_aux.p, ra.data(), n_pad * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RTZ_CUDA(cudaMemcpyAsync(c->rg_albedo.p, ral.data(), n_pad * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RTZ_CUDA(cudaMemcpyAsync(c->rg_wexp.p, rw.data(), n_pad * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        RTZ_CUDA(cudaMemcpyAsync(c->rg_orig.p, ro.data(), n_pad * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    RTZ_CUDA(c->dspheres.reserve(ds.size()));
    RTZ_CUDA(cudaMemcpyAsync(c->dspheres.p, ds.data(), ds.size() * sizeof(rtz::DSphere), cudaMemcpyHostToDevice,
                             c->stream));
    c->h_pairs.swap(pr);  // host copy: small scenes travel to the kernel as a __grid_constant__ parameter
    c->h_rg_pairs.swap(rpr);
    c->h_boxes.swap(bx);
    c->cull_r2 = (float)(R * R);
    c->cull = cull;
    g.resize(n), w.resize(n);
    c->h_geom.swap(g), c->h_w.swap(w);  // what the BVH extension is built from, if it is ever asked for
    c->n_spheres = (int)n, c->n_pad = n_pad;
    return RTZ_OK;
}

}  // extern "C"

namespace {
int32_t ensure_bvh(rtz_context* c) {
    if (c->bvh_ready) return RTZ_OK;
    const size_t n = (size_t)c->n_spheres;
    BvhBuilder bvh(c->h_geom, (int)n);
    bvh.run();
    RTZ_CUDA(c->bvh_nodes.reserve(bvh.nodes.size()));
    RTZ_CUDA(c->bvh_order.reserve(std::max<size_t>(1, bvh.order.size())));
    RTZ_CUDA(cudaMemcpyAsync(c->bvh_nodes.p, bvh.nodes.data(), bvh.nodes.size() * sizeof(rtz::BvhNode), cudaMemcpyHostToDevice, c->stream));
    if (n) {
        RTZ_CUDA(cudaMemcpyAsync(c->bvh_order.p, bvh.order.data(), n * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    RTZ_CUDA(cudaStreamSynchronize(c->stream));
    c->bvh_ready = true;
    return RTZ_OK;
}
}  // namespace

extern "C" {

int32_t rtz_scene_generate(rtz_context* c, int32_t kind, uint64_t seed, uint64_t n_spheres, rtz_sphere* out,
                           uint64_t cap, uint64_t* n_out, uint64_t state_out[4]) {
    if (!c || kind < RTZ_SCENE_FINAL || kind > RTZ_SCENE_SWEEP) return RTZ_ERR_BAD_ARG;
    if (kind == RTZ_SCENE_SWEEP && (n_spheres < 4 || n_spheres > (1u << 20))) return RTZ_ERR_BAD_ARG;
    DeviceGuard guard;
    RTZ_CUDA(cudaSetDevice(c->device));
    // capacity of the device list: the final scene has at most 22*22 + 4 spheres, the sweep exactly n
    const uint64_t dev_cap = kind == RTZ_SCENE_SWEEP ? n_spheres : 22 * 22 + 4;
    rtz_sphere* d_sp = nullptr;
    rtz::SceneGenOut* d_res = nullptr;
    RTZ_CUDA(cudaMalloc(&d_sp, dev_cap * sizeof(rtz_sphere)));
    if (cudaMalloc(&d_res, sizeof(rtz::SceneGenOut)) != cudaSuccess) {
        cudaFree(d_sp);
        return RTZ_ERR_CUDA;
    }
    rtz::scene_kernel<<<1, 1, 0, c->stream>>>(kind, seed, n_spheres, d_sp, dev_cap, d_res);
    rtz::SceneGenOut res{};
    std::vector<rtz_sphere> host;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(&res, d_res, sizeof res, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess && res.count > 0 && res.count <= dev_cap) {
        host.resize(res.count);
        e = cudaMemcpyAsync(host.data(), d_sp, res.count * sizeof(rtz_sphere), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    }
    cudaFree(d_sp), cudaFree(d_res);
    if (e != cudaSuccess) {
        g_last_error = cudaGetErrorString(e);
        return RTZ_ERR_CUDA;
    }
    if (res.count == 0 || res.count > dev_cap) return RTZ_ERR_BAD_ARG;  // the sweep could not reach n spheres
    if (n_out) *n_out = res.count;
    if (state_out) std::memcpy(state_out, res.state, sizeof res.state);
    if (out)
        for (uint64_t i = 0; i < res.count && i < cap; ++i) out[i] = host[i];
    return rtz_scene_upload(c, host.data(), res.count);
}

uint64_t rtz_shard_pixels(uint64_t W, uint64_t H, const rtz_shard* s) {
    rtz::ShardGeom g;
    if (shard_geom(W, H, s, g) != RTZ_OK) return 0;
    return (uint64_t)g.n_local_tiles * g.tile_pixels;
}

static int32_t render_resident_impl(rtz_context* c, const rtz_camera* cam, const rtz_shard* shard, uint8_t* d_rgb,
                                    double* d_linear, rtz_stats* st) {
    if (!c || !d_rgb) return RTZ_ERR_BAD_ARG;
    int32_t rc = check_camera(cam);
    if (rc != RTZ_OK) return rc;
    DeviceGuard guard;
    RTZ_CUDA(cudaSetDevice(c->device));
    if (cam->mode != RTZ_MODE_PATH && cam->mode != RTZ_MODE_PATH_BVH) {
        if (shard && shard->world != 1) return RTZ_ERR_BAD_ARG;  // the legacy modes are whole-frame only
        return render_legacy(c, cam, d_rgb, d_linear, st);
    }
    rtz::ShardGeom g;
    rc = shard_geom(cam->width, cam->height, shard, g);
    if (rc != RTZ_OK) return rc;
    const uint64_t seed = cam->has_seed ? cam->seed : os_seed();
    return render_path(c, cam, g, d_rgb, d_linear, st, seed);
}

int32_t rtz_render_resident(rtz_context* c, const rtz_camera* cam, const rtz_shard* shard, uint8_t* d_rgb,
                            rtz_stats* st) {
    return render_resident_impl(c, cam, shard, d_rgb, nullptr, st);
}

int32_t rtz_deinterleave(rtz_context* c, uint64_t W, uint64_t H, uint32_t world, uint32_t tw, uint32_t th,
                         const uint8_t* d_gathered, uint8_t* d_rgb) {
    if (!c || !d_gathered || !d_rgb || !W || !H) return RTZ_ERR_BAD_ARG;
    rtz_shard s{0, world, tw, th};
    rtz::ShardGeom g;
    int32_t rc = shard_geom(W, H, &s, g);
    if (rc != RTZ_OK) return rc;
    if (W > 0xFFFFFFFFull || H > 0xFFFFFFFFull || W * H > 0xFFFFFFFFull) return RTZ_ERR_BAD_ARG;
    DeviceGuard guard;
    RTZ_CUDA(cudaSetDevice(c->device));
    const uint64_t n = W * H;
    rtz::deinterleave_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(
        d_gathered, (uint64_t)g.n_local_tiles * g.tile_pixels, (uint32_t)W, (uint32_t)H, world, tw, th, g.tiles_x, d_rgb);
    RTZ_CUDA(cudaGetLastError());
    RTZ_CUDA(cudaStreamSynchronize(c->stream));
    return RTZ_OK;
}

// The host-buffer entry points keep ONE lazily created context per DEVICE (buffers and stream are reused
// from frame to frame; nothing of the caller's is retained).  A call renders on the caller's current device.
static std::mutex g_default_mu;
static std::map<int, rtz_context*> g_default_ctx;

int32_t rtz_render_linear(const rtz_camera* cam, const rtz_sphere* sp, uint64_t n, uint8_t* rgb_out,
                          double* linear_out, rtz_stats* st) {
    if (!rgb_out || (!sp && n)) return RTZ_ERR_BAD_ARG;
    int32_t rc = check_camera(cam);
    if (rc != RTZ_OK) return rc;
    int cnt = 0;
    rc = rtz_device_count(&cnt);
    if (rc != RTZ_OK) return rc;
    std::lock_guard<std::mutex> lock(g_default_mu);
    DeviceGuard guard;
    int dev = 0;
    RTZ_CUDA(cudaGetDevice(&dev));
    rtz_context*& slot = g_default_ctx[dev];
    if (!slot) {
        rc = rtz_context_create(dev, nullptr, &slot);
        if (rc != RTZ_OK) return rc;
    }
    rtz_context* c = slot;
    rc = rtz_scene_upload(c, sp, n);
    if (rc != RTZ_OK) return rc;
    RTZ_CUDA(cudaSetDevice(c->device));
    const uint64_t px = cam->width * cam->height;
    RTZ_CUDA(c->rgb.reserve(3 * px));
    if (linear_out) RTZ_CUDA(c->linear.reserve(3 * px));
    rc = render_resident_impl(c, cam, nullptr, c->rgb.p, linear_out ? c->linear.p : nullptr, st);
    if (rc != RTZ_OK) return rc;
    RTZ_CUDA(cudaSetDevice(c->device));
    RTZ_CUDA(cudaMemcpyAsync(rgb_out, c->rgb.p, 3 * px, cudaMemcpyDeviceToHost, c->stream));
    if (linear_out)
        RTZ_CUDA(cudaMemcpyAsync(linear_out, c->linear.p, 3 * px * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    RTZ_CUDA(cudaStreamSynchronize(c->stream));
    return RTZ_OK;
}

int32_t rtz_render(const rtz_camera* cam, const rtz_sphere* sp, uint64_t n, uint8_t* rgb_out, rtz_stats* st) {
    return rtz_render_linear(cam, sp, n, rgb_out, nullptr, st);
}

int32_t rtz_write_ppm(const char* path, uint64_t w, uint64_t h, const uint8_t* rgb) {
    if (!path || w > 0xFFFFFFFFull || h > 0xFFFFFFFFull || (!rgb && w * h)) return RTZ_ERR_BAD_ARG;
    if (w && h > (SIZE_MAX / 3) / w) return RTZ_ERR_BAD_ARG;  // 3 * w * h must fit a size_t
    FILE* f = std::fopen(path, "wb");
    if (!f) {
        g_last_error = std::string(path) + ": " + std::strerror(errno);
        return RTZ_ERR_IO;
    }
    bool ok = std::fprintf(f, "P6\n%llu %llu\n255\n", (unsigned long long)w, (unsigned long long)h) > 0;
    const size_t nb = (size_t)(3 * w * h);
    ok = ok && std::fwrite(rgb, 1, nb, f) == nb;
    ok = ok && std::fputc('\n', f) != EOF;  // trailing newline (src/ppm.zig:57)
    ok = (std::fclose(f) == 0) && ok;
    return ok ? RTZ_OK : RTZ_ERR_IO;
}

}  // extern "C" (first part)

// ---- N GPUs of one box behind the same call ----------------------------------------------------------
namespace {

// NCCL entry points, resolved from libnccl.so.2 at run time so that single-GPU users need no NCCL at all.
struct NcclApi {
    void* handle = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    bool load() {
        if (handle) return true;
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (handle) break;
        }
        if (!handle) {
            g_last_error = std::string("dlopen(libnccl.so.2): ") + dlerror();
            return false;
        }
#define RTZ_NCCL_SYM(field, sym)                                              \
    field = reinterpret_cast<decltype(field)>(dlsym(handle, #sym));            \
    if (!field) {                                                              \
        g_last_error = "libnccl.so.2 lacks " #sym;                             \
        return false;                                                          \
    }
        RTZ_NCCL_SYM(CommInitAll, ncclCommInitAll)
        RTZ_NCCL_SYM(CommDestroy, ncclCommDestroy)
        RTZ_NCCL_SYM(Send, ncclSend)
        RTZ_NCCL_SYM(Recv, ncclRecv)
        RTZ_NCCL_SYM(GroupStart, ncclGroupStart)
        RTZ_NCCL_SYM(GroupEnd, ncclGroupEnd)
        RTZ_NCCL_SYM(GetErrorString, ncclGetErrorString)
#undef RTZ_NCCL_SYM
        return true;
    }
};
NcclApi g_nccl;

#define RTZ_NCCL(call)                                                                  \
    do {                                                                                \
        ncclResult_t r_ = (call);                                                       \
        if (r_ != ncclSuccess) {                                                        \
            g_last_error = std::string(#call) + ": " + g_nccl.GetErrorString(r_);       \
            return RTZ_ERR_NCCL;                                                        \
        }                                                                               \
    } while (0)

}  // namespace

// One host thread per extra device: uploads and launches for the N devices of an rtz_multi are issued concurrently
// (one thread walking eight devices costs ~0.1 ms per device per frame, 4 % of a 21 ms frame).  The caller's thread
// serves device 0 itself; the ABI stays synchronous and single-entry.
struct MultiWorker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<int32_t()> job;
    bool has_job = false, done = true, quit = false;
    int32_t rc = RTZ_OK;
    std::string err;
    void loop() {
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv.wait(lk, [&] { return has_job || quit; });
            if (quit) return;
            has_job = false;
            lk.unlock();
            g_last_error.clear();
            const int32_t r = job();
            lk.lock();
            rc = r, err = g_last_error, done = true;
            cv.notify_all();
        }
    }
    void post(std::function<int32_t()> f) {
        std::lock_guard<std::mutex> lk(mu);
        job = std::move(f), has_job = true, done = false;
        cv.notify_all();
    }
    int32_t wait() {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return done; });
        if (rc != RTZ_OK) g_last_error = err;
        return rc;
    }
    void stop() {
        {
            std::lock_guard<std::mutex> lk(mu);
            quit = true;
            cv.notify_all();
        }
        if (th.joinable()) th.join();
    }
};

struct rtz_multi {
    std::vector<std::unique_ptr<MultiWorker>> workers;  // [r] for r >= 1
    std::vector<int> dev;
    std::vector<rtz_context*> ctx;
    std::vector<cudaEvent_t> done;        // per device: its resolve has finished
    uint32_t tile_w = 4, tile_h = 4;
    int gather = RTZ_GATHER_P2P;
    std::vector<ncclComm_t> comms;        // RTZ_GATHER_NCCL
    std::vector<uint8_t*> local;          // RTZ_GATHER_NCCL: per-device compact tile buffer (device r), r >= 1
    std::vector<size_t> local_cap;
    DevBuf<uint8_t> gathered;             // RTZ_GATHER_NCCL, device 0: `world` compact buffers back to back
    DevBuf<uint8_t> image;                // device 0: the row-major frame
    cudaEvent_t ev_start = nullptr, ev_traced = nullptr, ev_end = nullptr;  // device 0's stream
};

namespace {
// fn(r) for every device of the group, concurrently; the first failure is reported
int32_t on_every_device(rtz_multi* m, const std::function<int32_t(int)>& fn) {
    const int world = (int)m->ctx.size();
    for (int r = 1; r < world; ++r) m->workers[r]->post([&fn, r] { return fn(r); });
    int32_t rc = fn(0);
    for (int r = 1; r < world; ++r) {
        const int32_t w = m->workers[r]->wait();
        if (rc == RTZ_OK) rc = w;
    }
    return rc;
}
}  // namespace

extern "C" {

int32_t rtz_multi_destroy(rtz_multi* m) {
    if (!m) return RTZ_ERR_BAD_ARG;
    DeviceGuard guard;
    for (auto& w : m->workers)
        if (w) w->stop();
    for (size_t r = 0; r < m->ctx.size(); ++r) {
        if (!m->ctx[r]) continue;
        cudaSetDevice(m->dev[r]);
        cudaStreamSynchronize(m->ctx[r]->stream);
        if (r < m->local.size() && m->local[r]) cudaFree(m->local[r]);
        if (r < m->done.size() && m->done[r]) cudaEventDestroy(m->done[r]);
    }
    for (ncclComm_t c : m->comms)
        if (c && g_nccl.CommDestroy) g_nccl.CommDestroy(c);
    if (!m->dev.empty()) {
        cudaSetDevice(m->dev[0]);
        m->gathered.release(), m->image.release();
        for (cudaEvent_t e : {m->ev_start, m->ev_traced, m->ev_end})
            if (e) cudaEventDestroy(e);
    }
    for (rtz_context* c : m->ctx)
        if (c) rtz_context_destroy(c);
    delete m;
    return RTZ_OK;
}

int32_t rtz_multi_create(int32_t num_gpus, const int32_t* devices, uint32_t tile_w, uint32_t tile_h, int32_t gather,
                         rtz_multi** out) {
    if (!out || gather < RTZ_GATHER_AUTO || gather > RTZ_GATHER_NCCL) return RTZ_ERR_BAD_ARG;
    *out = nullptr;
    int visible = 0;
    int32_t rc = rtz_device_count(&visible);
    if (rc != RTZ_OK) return rc;
    if (num_gpus <= 0) num_gpus = visible;
    if (num_gpus > visible) {
        g_last_error = "asked for " + std::to_string(num_gpus) + " GPUs, " + std::to_string(visible) + " visible";
        return RTZ_ERR_BAD_ARG;
    }
    DeviceGuard guard;
    rtz_multi* m = new rtz_multi();
    m->tile_w = tile_w ? tile_w : 4, m->tile_h = tile_h ? tile_h : 4;
    m->dev.resize(num_gpus), m->ctx.assign(num_gpus, nullptr), m->done.assign(num_gpus, nullptr);
    m->local.assign(num_gpus, nullptr), m->local_cap.assign(num_gpus, 0);
    for (int r = 0; r < num_gpus; ++r) {
        m->dev[r] = devices ? devices[r] : r;
        for (int q = 0; q < r; ++q)
            if (m->dev[q] == m->dev[r]) rc = RTZ_ERR_BAD_ARG;  // a device may appear once
        if (rc == RTZ_OK) rc = rtz_context_create(m->dev[r], nullptr, &m->ctx[r]);
        if (rc != RTZ_OK) {
            rtz_multi_destroy(m);
            return rc;
        }
        cudaSetDevice(m->dev[r]);
        cudaEventCreateWithFlags(&m->done[r], cudaEventDisableTiming);
    }
    m->workers.resize(num_gpus);
    for (int r = 1; r < num_gpus; ++r) {
        m->workers[r] = std::make_unique<MultiWorker>();
        MultiWorker* w = m->workers[r].get();
        w->th = std::thread([w] { w->loop(); });
    }
    cudaSetDevice(m->dev[0]);
    cudaEventCreate(&m->ev_start), cudaEventCreate(&m->ev_traced), cudaEventCreate(&m->ev_end);
    if (const char* e = std::getenv("RTZ_GATHER")) {
        if (!std::strcmp(e, "p2p")) gather = RTZ_GATHER_P2P;
        if (!std::strcmp(e, "nccl")) gather = RTZ_GATHER_NCCL;
    }
    // peer mapping of device 0's memory into every other device (the fused resolve + gather writes through it)
    bool p2p_ok = true;
    if (gather != RTZ_GATHER_NCCL) {
        for (int r = 1; r < num_gpus && p2p_ok; ++r) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, m->dev[r], m->dev[0]);
            if (!can) {
                p2p_ok = false;
                break;
            }
            cudaSetDevice(m->dev[r]);
            const cudaError_t e = cudaDeviceEnablePeerAccess(m->dev[0], 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (e != cudaSuccess) p2p_ok = false, cudaGetLastError();
        }
        if (!p2p_ok && gather == RTZ_GATHER_P2P) {
            g_last_error = "RTZ_GATHER_P2P: device 0's memory cannot be mapped into every other device";
            rtz_multi_destroy(m);
            return RTZ_ERR_CUDA;
        }
    }
    m->gather = (gather == RTZ_GATHER_NCCL || !p2p_ok) ? RTZ_GATHER_NCCL : RTZ_GATHER_P2P;
    if (m->gather == RTZ_GATHER_NCCL && num_gpus > 1) {
        if (!g_nccl.load()) {
            rtz_multi_destroy(m);
            return RTZ_ERR_NCCL;
        }
        m->comms.assign(num_gpus, nullptr);
        const ncclResult_t r = g_nccl.CommInitAll(m->comms.data(), num_gpus, m->dev.data());
        if (r != ncclSuccess) {
            g_last_error = std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(r);
            m->comms.clear();
            rtz_multi_destroy(m);
            return RTZ_ERR_NCCL;
        }
    }
    *out = m;
    return RTZ_OK;
}

int32_t rtz_multi_gpus(const rtz_multi* m) { return m ? (int32_t)m->ctx.size() : -1; }
int32_t rtz_multi_gather(const rtz_multi* m) { return m ? m->gather : -1; }

int32_t rtz_multi_scene_upload(rtz_multi* m, const rtz_sphere* sp, uint64_t n) {
    if (!m) return RTZ_ERR_BAD_ARG;
    return on_every_device(m, [&](int r) { return rtz_scene_upload(m->ctx[r], sp, n); });
}

int32_t rtz_multi_render(rtz_multi* m, const rtz_camera* cam, uint8_t* rgb_out, uint8_t** d_rgb_out, rtz_stats* st) {
    if (!m) return RTZ_ERR_BAD_ARG;
    int32_t rc = check_camera(cam);
    if (rc != RTZ_OK) return rc;
    DeviceGuard guard;
    const int world = (int)m->ctx.size();
    rtz_context* c0 = m->ctx[0];
    const uint64_t px = cam->width * cam->height;
    RTZ_CUDA(cudaSetDevice(m->dev[0]));
    RTZ_CUDA(m->image.reserve(3 * px));
    if (d_rgb_out) *d_rgb_out = m->image.p;
    const bool path_mode = cam->mode == RTZ_MODE_PATH || cam->mode == RTZ_MODE_PATH_BVH;
    if (!path_mode || world == 1) {
        // the deterministic legacy modes are 90 000 rays: one device; and one device needs no exchange
        rc = render_resident_impl(c0, cam, nullptr, m->image.p, nullptr, st);
        if (rc != RTZ_OK) return rc;
        RTZ_CUDA(cudaSetDevice(m->dev[0]));
        if (rgb_out) {
            RTZ_CUDA(cudaMemcpyAsync(rgb_out, m->image.p, 3 * px, cudaMemcpyDeviceToHost, c0->stream));
            RTZ_CUDA(cudaStreamSynchronize(c0->stream));
        }
        return RTZ_OK;
    }
    const uint64_t seed = cam->has_seed ? cam->seed : os_seed();  // ONE key for the whole frame
    std::vector<rtz::ShardGeom> sg(world);
    for (int r = 0; r < world; ++r) {
        const rtz_shard sh{(uint32_t)r, (uint32_t)world, m->tile_w, m->tile_h};
        rc = shard_geom(cam->width, cam->height, &sh, sg[r]);
        if (rc != RTZ_OK) return rc;
    }
    const size_t per_rank = 3 * (size_t)sg[0].n_local_tiles * sg[0].tile_pixels;  // equal on every rank
    const bool nccl = m->gather == RTZ_GATHER_NCCL;
    if (nccl) {
        RTZ_CUDA(m->gathered.reserve(per_rank * world));
        for (int r = 1; r < world; ++r) {
            if (m->local_cap[r] >= per_rank) continue;
            RTZ_CUDA(cudaSetDevice(m->dev[r]));
            if (m->local[r]) cudaFree(m->local[r]);
            m->local[r] = nullptr, m->local_cap[r] = 0;
            RTZ_CUDA(cudaMalloc(&m->local[r], per_rank));
            m->local_cap[r] = per_rank;
        }
        RTZ_CUDA(cudaSetDevice(m->dev[0]));
    }
    RTZ_CUDA(cudaEventRecord(m->ev_start, c0->stream));
    // every device's frame is enqueued (by its own host thread) before the first wait
    rc = on_every_device(m, [&](int r) -> int32_t {
        RTZ_CUDA(cudaSetDevice(m->dev[r]));
        FrameTarget out;
        if (nccl)
            out.d_rgb = r == 0 ? m->gathered.p : m->local[r];
        else
            out.image = m->image.p;  // peer memory for r >= 1
        const int32_t e = enqueue_path(m->ctx[r], cam, sg[r], out, seed);
        if (e != RTZ_OK) return e;
        RTZ_CUDA(cudaEventRecord(m->done[r], m->ctx[r]->stream));
        return RTZ_OK;
    });
    if (rc != RTZ_OK) return rc;
    RTZ_CUDA(cudaSetDevice(m->dev[0]));
    RTZ_CUDA(cudaEventRecord(m->ev_traced, c0->stream));
    if (nccl) {
        RTZ_NCCL(g_nccl.GroupStart());
        for (int r = 1; r < world; ++r) {
            RTZ_NCCL(g_nccl.Send(m->local[r], per_rank, ncclUint8, 0, m->comms[r], m->ctx[r]->stream));
            RTZ_NCCL(g_nccl.Recv(m->gathered.p + per_rank * r, per_rank, ncclUint8, r, m->comms[0], c0->stream));
        }
        RTZ_NCCL(g_nccl.GroupEnd());
        RTZ_CUDA(cudaSetDevice(m->dev[0]));
        rtz::deinterleave_kernel<<<(unsigned)((px + 255) / 256), 256, 0, c0->stream>>>(
            m->gathered.p, (uint64_t)sg[0].n_local_tiles * sg[0].tile_pixels, (uint32_t)cam->width, (uint32_t)cam->height,
            (uint32_t)world, m->tile_w, m->tile_h, sg[0].tiles_x, m->image.p);
        RTZ_CUDA(cudaGetLastError());
    } else {
        for (int r = 1; r < world; ++r) RTZ_CUDA(cudaStreamWaitEvent(c0->stream, m->done[r], 0));
    }
    RTZ_CUDA(cudaEventRecord(m->ev_end, c0->stream));
    if (rgb_out) RTZ_CUDA(cudaMemcpyAsync(rgb_out, m->image.p, 3 * px, cudaMemcpyDeviceToHost, c0->stream));
    rtz_stats total;
    std::memset(&total, 0, sizeof total);
    for (int r = 0; r < world; ++r) {
        RTZ_CUDA(cudaSetDevice(m->dev[r]));
        rtz_stats one;
        rc = collect_path(m->ctx[r], cam, sg[r], &one, seed);
        if (rc != RTZ_OK) return rc;
        total.samples += one.samples, total.segments += one.segments, total.sphere_tests += one.sphere_tests;
        total.depth_capped += one.depth_capped, total.absorbed += one.absorbed, total.nan_samples += one.nan_samples;
        total.kernel_launches += one.kernel_launches;
        total.trace_ms = std::max(total.trace_ms, one.trace_ms);
        total.resolve_ms = std::max(total.resolve_ms, one.resolve_ms);
    }
    RTZ_CUDA(cudaSetDevice(m->dev[0]));
    RTZ_CUDA(cudaStreamSynchronize(c0->stream));
    if (st) {
        float ms = 0;
        cudaEventElapsedTime(&ms, m->ev_start, m->ev_end), total.total_ms = ms;
        total.gather_ms = std::max(0.0, total.total_ms - total.trace_ms);
        total.kernel_launches += nccl ? 1 : 0;
        total.gpus = (uint32_t)world;
        total.gather = (uint32_t)m->gather;
        total.seed_used = seed;
        *st = total;
    }
    return RTZ_OK;
}

// one lazily created rtz_multi per device count for the one-shot form
static std::mutex g_multi_mu;
static std::map<int, rtz_multi*> g_multi;

int32_t rtz_render_multi(const rtz_camera* cam, const rtz_sphere* sp, uint64_t n, int32_t num_gpus, uint8_t* rgb_out,
                         rtz_stats* st) {
    if (!rgb_out || (!sp && n)) return RTZ_ERR_BAD_ARG;
    int32_t rc = check_camera(cam);
    if (rc != RTZ_OK) return rc;
    int visible = 0;
    rc = rtz_device_count(&visible);
    if (rc != RTZ_OK) return rc;
    if (num_gpus <= 0) num_gpus = visible;
    std::lock_guard<std::mutex> lock(g_multi_mu);
    rtz_multi*& slot = g_multi[num_gpus];
    if (!slot) {
        rc = rtz_multi_create(num_gpus, nullptr, 0, 0, RTZ_GATHER_AUTO, &slot);
        if (rc != RTZ_OK) return rc;
    }
    rc = rtz_multi_scene_upload(slot, sp, n);
    if (rc != RTZ_OK) return rc;
    return rtz_multi_render(slot, cam, rgb_out, nullptr, st);
}

}  // extern "C"

extern "C" {

// ---- probes -------------------------------------------------------------------------------------
}  // extern "C"

namespace {
// Upload the scene to a fresh context, copy the m records in, run `launch(ctx, in, out)` and copy the m results out.
template <class In, class Out, class Launch>
int32_t run_probe(const rtz_sphere* sp, uint64_t n, const In* in, uint64_t m, Out* out, Launch launch) {
    ScopedCtx sc;
    int32_t rc = rtz_context_create(-1, nullptr, &sc.c);
    if (rc != RTZ_OK) return rc;
    rc = rtz_scene_upload(sc.c, sp, n);
    if (rc != RTZ_OK) return rc;
    In* din = nullptr;
    Out* dout = nullptr;
    cudaError_t e = cudaMalloc(&din, m * sizeof(In));
    if (e == cudaSuccess) e = cudaMalloc(&dout, m * sizeof(Out));
    if (e == cudaSuccess) e = cudaMemcpyAsync(din, in, m * sizeof(In), cudaMemcpyHostToDevice, sc.c->stream);
    if (e == cudaSuccess) {
        launch(sc.c, din, dout, (unsigned)((m + 127) / 128));
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, m * sizeof(Out), cudaMemcpyDeviceToHost, sc.c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(sc.c->stream);
    cudaFree(din);
    cudaFree(dout);
    RTZ_CUDA(e);
    return RTZ_OK;
}
}  // namespace

extern "C" {

int32_t rtz_probe_hits(const rtz_sphere* sp, uint64_t n, const rtz_probe_ray* rays, uint64_t m, double tmin,
                       double tmax, rtz_ray_hit* out) {
    if (!sp || !n || (!rays && m) || (!out && m) || m > (1ull << 31)) return RTZ_ERR_BAD_ARG;
    if (!m) return RTZ_OK;
    return run_probe(sp, n, rays, m, out, [&](rtz_context* c, const rtz_probe_ray* din, rtz_ray_hit* dout, unsigned blocks) {
        rtz::probe_hits_kernel<<<blocks, 128, 0, c->stream>>>(c->geom.p, c->pairs.p, c->aux.p, c->n_pad, din, m,
                                                             (float)tmin, (float)tmax, dout);
    });
}

int32_t rtz_probe_scatters(const rtz_sphere* sp, uint64_t n, const rtz_probe_bounce* recs, uint64_t m, uint64_t seed,
                           rtz_ray_scatter* out) {
    if (!sp || !n || (!recs && m) || (!out && m) || m > (1ull << 31)) return RTZ_ERR_BAD_ARG;
    for (uint64_t k = 0; k < m; ++k)
        if (recs[k].sphere < 0 || (uint64_t)recs[k].sphere >= n) return RTZ_ERR_BAD_ARG;
    if (!m) return RTZ_OK;
    rtz_camera cam;
    std::memset(&cam, 0, sizeof(cam));
    cam.t_min = 1e-3, cam.t_max = INFINITY, cam.bounce_max = 0xFFFFFFFFull, cam.samples_per_pixel = 1, cam.width = cam.height = 1;
    const rtz::DevCamera dc = to_dev_camera(cam, seed);
    return run_probe(sp, n, recs, m, out, [&](rtz_context* c, const rtz_probe_bounce* din, rtz_ray_scatter* dout, unsigned blocks) {
        rtz::probe_scatters_kernel<<<blocks, 128, 0, c->stream>>>(dc, c->geom.p, c->pairs.p, c->aux.p, c->albedo.p, din, m,
                                                                 dout);
    });
}

int32_t rtz_probe_hit(const rtz_sphere* sp, uint64_t n, const double o[3], const double d[3], double tmin, double tmax,
                      rtz_hit* out) {
    if (!sp || !n || !o || !d || !out) return RTZ_ERR_BAD_ARG;
    const rtz_probe_ray r = {{(float)o[0], (float)o[1], (float)o[2]}, {(float)d[0], (float)d[1], (float)d[2]}, -1};
    rtz_ray_hit h;
    const int32_t rc = rtz_probe_hits(sp, n, &r, 1, tmin, tmax, &h);
    if (rc != RTZ_OK) return rc;
    std::memset(out, 0, sizeof(*out));
    out->hit = h.best >= 0;
    if (h.best >= 0) {
        out->index = h.best, out->front = h.front;
        out->t = (double)h.t / (double)h.len;  // back to the reference's units of |dir|
        for (int k = 0; k < 3; ++k) out->point[k] = h.point[k], out->normal[k] = h.normal[k];
    }
    return RTZ_OK;
}

int32_t rtz_probe_scatter(const rtz_sphere* sp, uint64_t n, int32_t index, const double o[3], const double d[3],
                          uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, rtz_scatter* out) {
    if (!sp || !n || index < 0 || (uint64_t)index >= n || !o || !d || !out) return RTZ_ERR_BAD_ARG;
    const rtz_probe_bounce r = {index, {(float)o[0], (float)o[1], (float)o[2]}, {(float)d[0], (float)d[1], (float)d[2]},
                                pixel, sample, bounce};
    rtz_ray_scatter h;
    const int32_t rc = rtz_probe_scatters(sp, n, &r, 1, seed, &h);
    if (rc != RTZ_OK) return rc;
    std::memset(out, 0, sizeof(*out));
    out->scattered = h.term == -1;
    if (h.term == -1)
        for (int k = 0; k < 3; ++k) {
            out->origin[k] = h.orig[k];
            out->direction[k] = (double)h.dir[k] * (double)h.len;
            out->attenuation[k] = h.attenuation[k];
        }
    return RTZ_OK;
}

int32_t rtz_probe_sweep_order(const rtz_sphere* sp, uint64_t n, int32_t* order_out) {
    if ((!sp || !order_out) && n) return RTZ_ERR_BAD_ARG;
    if (n > (1u << 20)) return RTZ_ERR_BAD_ARG;
    std::vector<float4> g(n);
    for (uint64_t i = 0; i < n; ++i) {
        if (!finite3(sp[i].center)) return RTZ_ERR_BAD_ARG;
        g[i] = make_float4((float)sp[i].center[0], (float)sp[i].center[1], (float)sp[i].center[2], 0.f);
    }
    const std::vector<int> order = sweep_order(g, (int)n);
    std::copy(order.begin(), order.end(), order_out);
    return RTZ_OK;
}

int32_t rtz_probe_to_rgb(const double* lin, uint64_t n, uint8_t* rgb_out) {
    if (!lin || !rgb_out || !n) return RTZ_ERR_BAD_ARG;
    ScopedCtx sc;
    int32_t rc = rtz_context_create(-1, nullptr, &sc.c);
    if (rc != RTZ_OK) return rc;
    double* dl = nullptr;
    uint8_t* dr = nullptr;
    if (n > (1ull << 32)) return RTZ_ERR_BAD_ARG;
    RTZ_CUDA(cudaMalloc(&dl, 3 * n * sizeof(double)));
    cudaError_t e = cudaMalloc(&dr, 3 * n);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dl, lin, 3 * n * sizeof(double), cudaMemcpyHostToDevice, sc.c->stream);
    if (e == cudaSuccess) {
        rtz::probe_to_rgb_kernel<<<(unsigned)((3 * n + 255) / 256), 256, 0, sc.c->stream>>>(dl, 3 * n, dr);
        e = cudaMemcpyAsync(rgb_out, dr, 3 * n, cudaMemcpyDeviceToHost, sc.c->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(sc.c->stream);
    cudaFree(dl), cudaFree(dr);
    RTZ_CUDA(e);
    return RTZ_OK;
}

int32_t rtz_probe_camera_ray(const rtz_camera* cam, uint64_t i, uint64_t j, uint64_t sample0, uint64_t n, float* o_out,
                             float* d_out, float* len_out) {
    if (!o_out || !d_out || !n || n > (1u << 24)) return RTZ_ERR_BAD_ARG;
    int32_t rc = check_camera(cam);
    if (rc != RTZ_OK) return rc;
    if (i >= cam->width || j >= cam->height) return RTZ_ERR_BAD_ARG;
    ScopedCtx sc;
    rc = rtz_context_create(-1, nullptr, &sc.c);
    if (rc != RTZ_OK) return rc;
    const rtz::DevCamera dc = to_dev_camera(*cam, cam->has_seed ? cam->seed : os_seed());
    float* buf;
    RTZ_CUDA(cudaMalloc(&buf, n * 7 * sizeof(float)));
    float *d_o = buf, *d_d = buf + 3 * n, *d_l = buf + 6 * n;
    rtz::probe_camera_ray_kernel<<<(unsigned)((n + 127) / 128), 128, 0, sc.c->stream>>>(
        dc, (uint32_t)i, (uint32_t)j, (uint32_t)sample0, (uint32_t)n, d_o, d_d, d_l);
    cudaError_t e = cudaMemcpyAsync(o_out, d_o, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, sc.c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_out, d_d, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, sc.c->stream);
    if (e == cudaSuccess && len_out) e = cudaMemcpyAsync(len_out, d_l, n * sizeof(float), cudaMemcpyDeviceToHost, sc.c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(sc.c->stream);
    cudaFree(buf);
    RTZ_CUDA(e);
    return RTZ_OK;
}

int32_t rtz_probe_uniform(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, uint64_t n, float* out) {
    if (!out || !n) return RTZ_ERR_BAD_ARG;
    ScopedCtx sc;
    int32_t rc = rtz_context_create(-1, nullptr, &sc.c);
    if (rc != RTZ_OK) return rc;
    float* dout;
    RTZ_CUDA(cudaMalloc(&dout, n * sizeof(float)));
    const uint64_t blocks = (n + 3) / 4;
    rtz::probe_uniform_kernel<<<(unsigned)((blocks + 127) / 128), 128, 0, sc.c->stream>>>(
        (uint32_t)seed, (uint32_t)(seed >> 32), pixel, sample, bounce, n, dout);
    cudaError_t e = cudaMemcpyAsync(out, dout, n * sizeof(float), cudaMemcpyDeviceToHost, sc.c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(sc.c->stream);
    cudaFree(dout);
    RTZ_CUDA(e);
    return RTZ_OK;
}

int32_t rtz_measure_fp32_peak(int32_t device, int32_t variant, double* tflops_out) {
    if (!tflops_out || variant < 0 || variant > 2) return RTZ_ERR_BAD_ARG;
    ScopedCtx sc;
    int32_t rc = rtz_context_create(device, nullptr, &sc.c);
    if (rc != RTZ_OK) return rc;
    rtz_context* c = sc.c;
    float* sink;
    RTZ_CUDA(cudaMalloc(&sink, 4));
    const int iters = 1 << 14, blocks = c->sm_count * 8, threads = 256;
    float best_ms = 1e30f;
    cudaError_t e = cudaSuccess;
    for (int rep = 0; rep < 6 && e == cudaSuccess; ++rep) {
        cudaEventRecord(c->ev[0], c->stream);
        if (variant == 0)
            rtz::ffma_peak_kernel<0><<<blocks, threads, 0, c->stream>>>(1.0000001f, 1e-7f, iters, sink);
        else if (variant == 1)
            rtz::ffma_peak_kernel<1><<<blocks, threads, 0, c->stream>>>(1.0000001f, 1e-7f, iters, sink);
        else if (variant == 2)
            rtz::ffma_peak_kernel<2><<<blocks, threads, 0, c->stream>>>(1.0000001f, 1e-7f, iters, sink);
        cudaEventRecord(c->ev[1], c->stream);
        e = cudaStreamSynchronize(c->stream);
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
        if (rep > 0 && ms < best_ms) best_ms = ms;
    }
    cudaFree(sink);
    RTZ_CUDA(e);
    double flops = 2.0 * 16 * (double)iters * (double)blocks * threads;
    *tflops_out = flops / (best_ms * 1e-3) / 1e12;
    return RTZ_OK;
}

}  // extern "C"
