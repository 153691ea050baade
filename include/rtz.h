/*
 * rtz.h — C ABI of librtz.so, the B200-native replacement for the body of
 * `Camera.render` in AndrewJarrett/raytracing-with-zig.
 *
 * The reference has no FFI today: it is one statically linked Zig executable and
 * `pub fn render(self: Camera) !void` (reference src/camera.zig:123-145) is the seam.
 * Everything above that seam (Scene construction, CameraBuilder maths, the PPM file)
 * stays on the host in f64; everything inside its loop nest — getRay
 * (src/camera.zig:187-215), rayColor (:148-183), HittableList.hit
 * (src/hittable.zig:64-77), Sphere.hit (src/sphere.zig:26-54), Material.scatter
 * (src/material.zig:27-110) and Color.toRgb (src/color.zig:63-80) — runs on the GPU
 * behind the entry points declared here.
 *
 * Conventions (inherited from the reference, SURVEY.md §8b):
 *   - the caller owns every buffer; the library copies in and keeps nothing after a
 *     call returns, except inside an explicit rtz_context;
 *   - calls are synchronous and blocking; a context must not be used from two host
 *     threads at once;
 *   - every function returns an int32 status, 0 = RTZ_OK.  There is NO CPU fallback:
 *     without a usable CUDA device the calls fail with RTZ_ERR_NO_DEVICE.
 *   - all structs are plain `extern struct`-compatible PODs (fixed-width ints, f64).
 */
#ifndef RTZ_H
#define RTZ_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTZ_ABI_VERSION 2   /* 2: rtz_stats grew (nan_samples, gpus, gather_ms); rtz_multi_* / rtz_render_multi added */

/* ---- status codes --------------------------------------------------------------- */
#define RTZ_OK 0
#define RTZ_ERR_BAD_ARG 1      /* null pointer, zero-sized image, unknown mode/material ... */
#define RTZ_ERR_NO_DEVICE 2    /* no CUDA device / driver: the product has no CPU path        */
#define RTZ_ERR_CUDA 3         /* a CUDA runtime call or a kernel failed; see rtz_last_error  */
#define RTZ_ERR_IO 4           /* rtz_write_ppm could not create / write the file             */
#define RTZ_ERR_TOO_MANY_SPHERES 5 /* more than 2^20 spheres (larger scenes than shared memory   */
                                   /* holds are swept from global memory, they are not an error) */
#define RTZ_ERR_ARCH 6         /* device is not sm_100 (the library ships sm_100a code only)  */
#define RTZ_ERR_NCCL 7         /* libnccl.so.2 could not be loaded or an NCCL call failed      */

/* ---- material tags: reference src/material.zig:113-117 (MaterialType) ------------ */
#define RTZ_MAT_LAMBERTIAN 0
#define RTZ_MAT_METAL 1
#define RTZ_MAT_DIELECTRIC 2

/* ---- render modes ----------------------------------------------------------------
 * RTZ_MODE_PATH is the current reference source: jittered samples, defocus disk,
 * bounded path loop, gamma-2, clamp[0,.999], trunc(256x)  (src/camera.zig:123-215,
 * src/color.zig:63-80).
 * The LEGACY modes are the deterministic pipelines that produced the reference's
 * golden images test-files/chapter4.ppm / chapter5.ppm / chapter6.ppm (earlier
 * revisions of the same program; SURVEY.md §4.3): one ray through the pixel centre,
 * no RNG, no scatter, no gamma, quantiser trunc(255.999*c), hit interval (0, inf).
 * They are explicit so that nothing about them is silent behaviour.  They compute in
 * f64 on the device (90 000 rays) so the pre-quantisation values match the CPU
 * reference to the last bit; samples_per_pixel must be 1. */
#define RTZ_MODE_PATH 0
#define RTZ_MODE_LEGACY_SKY 1     /* chapter4: sky gradient only                              */
#define RTZ_MODE_LEGACY_FLAT 2    /* chapter5: any hit -> flat red (1,0,0), else sky          */
#define RTZ_MODE_LEGACY_NORMAL 3  /* chapter6: closest hit -> 0.5*(normal+1), else sky        */
#define RTZ_MODE_PATH_BVH 4       /* EXTENSION, not in the reference: RTZ_MODE_PATH with the   */
                                  /* closest hit found through a BVH over the spheres instead  */
                                  /* of the brute-force list; the image is bit-identical,      */
                                  /* rtz_stats.sphere_tests counts the tests actually made     */

/* One sphere with its material inlined.
 * reference: Sphere{center,radius,mat} src/sphere.zig:13-17; Material union
 * src/material.zig:126-129 with Lambertian{albedo} :16-19, Metal{albedo,fuzz} :42-46,
 * Dielectric{refractionIndex} :71-74; defaults of MaterialArgs :119-124. */
typedef struct rtz_sphere {
    double center[3];
    double radius;            /* > 0 and finite.  Sphere.init clamps negatives to 0 (:18-24); a    */
                              /* radius-0 sphere makes the reference panic in Vec.divScalar        */
                              /* (src/vec.zig:39-45) the moment it is hit, so the library refuses  */
                              /* it (and any non-finite field) with RTZ_ERR_BAD_ARG at upload      */
    int32_t mat_type;         /* RTZ_MAT_*                                                    */
    int32_t reserved;         /* must be 0                                                    */
    double albedo[3];         /* lambertian, metal                                            */
    double fuzz;              /* metal; NOT clamped to <= 1 (reference does not clamp)        */
    double refraction_index;  /* dielectric                                                   */
} rtz_sphere;

/* The fields of the reference `Camera` that `render` reads, by value.
 * reference: Camera struct src/camera.zig:82-103; Image :26-29; Scene.interval and
 * Scene.seed src/Scene.zig:19-21. */
typedef struct rtz_camera {
    uint64_t width, height;           /* Image.width/height                                   */
    double center[3];                 /* Camera.center  (:87)                                 */
    double pixel0[3];                 /* location of pixel (0,0)  (:103)                      */
    double du[3], dv[3];              /* pixel-to-pixel offsets  (:101-102)                   */
    double defocus_disk_u[3];         /* (:98)                                                */
    double defocus_disk_v[3];         /* (:99)                                                */
    double defocus_angle;             /* (:100); <= 0 disables the thin lens (:191)           */
    uint64_t samples_per_pixel;       /* (:88)                                                */
    uint64_t bounce_max;              /* (:90), reference default 50 (:221)                   */
    double pixel_samples_scale;       /* 1/spp (:89), applied as a multiply (:137)            */
    double t_min, t_max;              /* Scene.interval, (1e-3, +inf)  (src/Scene.zig:21)     */
    uint64_t seed;                    /* Scene.seed: key of the counter-based RNG             */
    int32_t has_seed;                 /* 0: the library draws a key from the OS, like         */
                                      /*    Scene.init does with getrandom (src/Scene.zig:33) */
    int32_t mode;                     /* RTZ_MODE_*                                           */
} rtz_camera;

/* Image-space sharding of one frame over `world` GPUs by interleaved tiles
 * (north_star; SURVEY.md §8e).  Tiles are tile_w x tile_h pixels, numbered row-major
 * over the image; tile k belongs to rank k % world.  A rank's pixels are stored
 * compactly, tile after tile (local tile j = global tile j*world + rank), each tile
 * row-major and padded to tile_w*tile_h pixels.  world = 1 reproduces the plain image
 * only through rtz_deinterleave / the whole-frame calls. */
typedef struct rtz_shard {
    uint32_t rank, world;
    uint32_t tile_w, tile_h;
} rtz_shard;

/* Work actually done, counted by the kernels (SURVEY.md §8d: measured, not assumed). */
typedef struct rtz_stats {
    uint64_t samples;          /* camera rays traced to termination                           */
    uint64_t segments;         /* world.hit calls (src/camera.zig:154)                        */
    uint64_t sphere_tests;     /* segments * n_spheres (brute force, src/hittable.zig:68)     */
    uint64_t depth_capped;     /* samples that ran out of bounces (src/camera.zig:181)        */
    uint64_t absorbed;         /* samples ended by a non-scattering metal hit (:163)          */
    uint64_t kernel_launches;  /* kernels launched by this call                               */
    double trace_ms;           /* path-trace kernel, CUDA events on the launching stream      */
    double resolve_ms;         /* resolve / pack kernel                                       */
    double total_ms;           /* first launch -> packed bytes ready on the device            */
    uint64_t seed_used;        /* RNG key actually used (== camera.seed when has_seed)        */
    uint64_t nan_samples;      /* samples whose colour was NaN (a zero-length scattered direction, */
                               /* src/vec.zig:126-128 unit of a zero vector); they add 0 to the    */
                               /* pixel instead of poisoning it, and are COUNTED here, not hidden  */
    uint32_t gpus;             /* devices that rendered this frame (1 unless rtz_multi_*)          */
    uint32_t gather;           /* RTZ_GATHER_P2P / RTZ_GATHER_NCCL when gpus > 1, else 0           */
    double gather_ms;          /* multi-GPU: end of the slowest trace kernel -> whole image on     */
                               /* device 0 (tile exchange over NVLink + de-interleave)             */
} rtz_stats;

/* ---- whole-frame, host buffers (the drop-in for the body of Camera.render) --------
 * Renders on the CURRENT CUDA device (one cached context per device; the caller's current device is
 * left as it was) and writes width*height*3 bytes, row-major,
 * top row first, r,g,b — exactly the bytes PPM.saveBinary emits between header and
 * trailer (src/ppm.zig:51-56).  `stats_out` may be NULL. */
int32_t rtz_render(const rtz_camera* camera, const rtz_sphere* spheres, uint64_t n_spheres,
                   uint8_t* rgb_out, rtz_stats* stats_out);

/* Same, additionally returning the per-pixel linear colour BEFORE gamma/quantisation
 * (f64, 3 per pixel): pixelColor * pixelSamplesScale of src/camera.zig:137.  Used by the
 * parity tests ("floats agree before quantisation").  `linear_out` may be NULL. */
int32_t rtz_render_linear(const rtz_camera* camera, const rtz_sphere* spheres, uint64_t n_spheres,
                          uint8_t* rgb_out, double* linear_out, rtz_stats* stats_out);

/* PPM.saveBinary (src/ppm.zig:42-60): "P6\n{w} {h}\n255\n" + 3*w*h bytes + "\n". */
int32_t rtz_write_ppm(const char* path, uint64_t width, uint64_t height, const uint8_t* rgb);

/* ---- resident API: scene and frame stay in HBM (bench `value`, multi-GPU ranks) ---- */
typedef struct rtz_context rtz_context;

/* device < 0: use the current device.  stream: a cudaStream_t passed as void*.
 * NULL = the context creates its OWN non-blocking stream, which is NOT ordered against any other
 * stream of the caller: device buffers handed to rtz_render_resident / rtz_deinterleave must be
 * complete before the call (every call blocks until its own work is done, so results are complete
 * on return).  To order the library's work with the CUDA legacy default stream or the per-thread
 * default stream pass RTZ_STREAM_LEGACY / RTZ_STREAM_PER_THREAD (CUDA's own handle values). */
#define RTZ_STREAM_LEGACY ((void*)0x1)
#define RTZ_STREAM_PER_THREAD ((void*)0x2)
int32_t rtz_context_create(int32_t device, void* stream, rtz_context** ctx_out);
int32_t rtz_context_destroy(rtz_context* ctx);

/* Flatten AoS f64 spheres to the device SoA f32 layout and upload (HittableList.add,
 * src/hittable.zig:60-62, for the whole list at once). */
int32_t rtz_scene_upload(rtz_context* ctx, const rtz_sphere* spheres, uint64_t n_spheres);

/* Scene.init(seed) followed by Scene.generateWorld / generateChapter13 (src/Scene.zig:23-46, 48-134,
 * 136-182), or BASELINE config 5's generalised final scene of exactly n_spheres spheres, generated ON THE
 * DEVICE by one thread with the reference's exact PRNG stream (Zig std DefaultPrng = Xoshiro256++ seeded by
 * SplitMix64, Random.float(f64)), then installed as the context's scene like rtz_scene_upload does.
 * spheres_out (optional, host, `cap` entries) receives the f64 spheres in list order, *n_out their number,
 * prng_state_out (optional) the four words of Scene.prng after generation.  (SURVEY.md 8f row 2.) */
#define RTZ_SCENE_FINAL 0      /* generateWorld: ~485 spheres                                  */
#define RTZ_SCENE_CHAPTER13 1  /* generateChapter13: 5 spheres, no random draws                */
#define RTZ_SCENE_SWEEP 2      /* config 5: exactly n_spheres (>= 4) spheres                   */
int32_t rtz_scene_generate(rtz_context* ctx, int32_t kind, uint64_t seed, uint64_t n_spheres,
                           rtz_sphere* spheres_out, uint64_t cap, uint64_t* n_out, uint64_t prng_state_out[4]);

/* Number of pixels (padded) in rank's compact tile buffer for this image. */
uint64_t rtz_shard_pixels(uint64_t width, uint64_t height, const rtz_shard* shard);

/* Render this rank's tiles of the frame.  `d_rgb_out` is a DEVICE pointer to
 * 3*rtz_shard_pixels(...) bytes in the compact tile layout described at rtz_shard.
 * shard == NULL means {0,1,...}: the whole frame, and then d_rgb_out is the plain
 * row-major image (3*width*height bytes).  The call enqueues on the context's stream
 * and synchronises it before returning (stats need the counters). */
int32_t rtz_render_resident(rtz_context* ctx, const rtz_camera* camera, const rtz_shard* shard,
                            uint8_t* d_rgb_out, rtz_stats* stats_out);

/* Rank-0 side of the tile gather: `d_gathered` holds `world` compact buffers of equal
 * size (rtz_shard_pixels of rank 0, the largest) back to back, as an all-gather /
 * gather leaves them; writes the plain row-major image to `d_rgb_out` (device). */
int32_t rtz_deinterleave(rtz_context* ctx, uint64_t width, uint64_t height, uint32_t world,
                         uint32_t tile_w, uint32_t tile_h, const uint8_t* d_gathered,
                         uint8_t* d_rgb_out);

/* ---- N GPUs of ONE box behind the same call (north_star: "rendered on 8xB200" as a drop-in for
 * Camera.render; SURVEY.md 8b `num_gpus`, 8e "single process ... no host MPI").  ONE host process, no
 * launcher: the library drives every device itself.  The frame is cut into interleaved tile_w x tile_h
 * tiles (tile k -> device k % gpus, rtz_shard), every device traces its tiles, and the packed bytes
 * travel to device 0 over NVLink either
 *   RTZ_GATHER_P2P   fused into the resolve kernel: each device's resolve writes its pixels straight
 *                    into device 0's row-major image through peer memory (no staging, no second kernel), or
 *   RTZ_GATHER_NCCL  ncclCommInitAll + one grouped ncclSend/ncclRecv of the compact tile buffers,
 *                    then rtz_deinterleave on device 0 (libnccl.so.2 is loaded on first use).
 * RTZ_GATHER_AUTO picks P2P when every device can map device 0's memory, NCCL otherwise (env RTZ_GATHER=
 * p2p|nccl overrides).  The image is the single-GPU image BYTE FOR BYTE for any device count and tile
 * size (integer accumulation, counter-based RNG). */
#define RTZ_GATHER_AUTO 0
#define RTZ_GATHER_P2P 1
#define RTZ_GATHER_NCCL 2
typedef struct rtz_multi rtz_multi;

/* num_gpus <= 0: every visible device.  devices: num_gpus ordinals, or NULL for 0..num_gpus-1;
 * devices[0] is "rank 0", where the image lands.  tile_w/tile_h = 0: the default 4x4. */
int32_t rtz_multi_create(int32_t num_gpus, const int32_t* devices, uint32_t tile_w, uint32_t tile_h,
                         int32_t gather, rtz_multi** multi_out);
int32_t rtz_multi_destroy(rtz_multi* multi);
int32_t rtz_multi_gpus(const rtz_multi* multi);              /* devices in use, or -1            */
int32_t rtz_multi_gather(const rtz_multi* multi);            /* RTZ_GATHER_P2P or RTZ_GATHER_NCCL */
/* HittableList for every device (rtz_scene_upload on each). */
int32_t rtz_multi_scene_upload(rtz_multi* multi, const rtz_sphere* spheres, uint64_t n_spheres);
/* Camera.render on all devices: launches are enqueued on every device before the first wait.  The
 * row-major image stays resident on device 0 (*d_rgb_out, optional, receives that DEVICE pointer, valid
 * until the next call on `multi`); rgb_out (optional, HOST, 3*width*height bytes) receives a copy.
 * stats_out: work counters summed over the devices, trace_ms = slowest device, total_ms = first launch
 * -> image complete on device 0 (events on device 0's stream). */
int32_t rtz_multi_render(rtz_multi* multi, const rtz_camera* camera, uint8_t* rgb_out, uint8_t** d_rgb_out,
                         rtz_stats* stats_out);
/* One-shot form with HOST buffers — rtz_render on num_gpus devices (<= 0: all).  Keeps one lazily
 * created rtz_multi per device count, like rtz_render keeps one context. */
int32_t rtz_render_multi(const rtz_camera* camera, const rtz_sphere* spheres, uint64_t n_spheres,
                         int32_t num_gpus, uint8_t* rgb_out, rtz_stats* stats_out);

/* ---- device-side unit probes (one ray; used by the KATs that mirror the reference's
 * own unit tests, src/sphere.zig:76-136, src/hittable.zig:185-209,
 * src/material.zig:168-281).  They run the SAME device functions the render kernel
 * inlines, on the GPU. ---------------------------------------------------------------- */
typedef struct rtz_hit {
    int32_t hit;           /* 0 = miss (null HitRecord)                                       */
    int32_t index;         /* index of the sphere hit                                         */
    int32_t front;         /* HitRecord.front                                                 */
    int32_t reserved;
    double t;              /* in units of |dir|, as the reference reports it                  */
    double point[3];
    double normal[3];
} rtz_hit;

/* HittableList.hit(ray, Interval(t_min, t_max)) — src/hittable.zig:64-77. */
int32_t rtz_probe_hit(const rtz_sphere* spheres, uint64_t n_spheres, const double orig[3],
                      const double dir[3], double t_min, double t_max, rtz_hit* out);

typedef struct rtz_scatter {
    int32_t scattered;     /* 0 = absorbed (null Scatter)                                     */
    int32_t reserved;
    double origin[3];
    double direction[3];
    double attenuation[3];
} rtz_scatter;

/* Material.scatter(ray, rec) — src/material.zig:145-151 — for sphere `index` of the list,
 * with the counter-based RNG at (seed, pixel, sample, bounce). */
int32_t rtz_probe_scatter(const rtz_sphere* spheres, uint64_t n_spheres, int32_t index,
                          const double orig[3], const double dir[3], uint64_t seed, uint32_t pixel,
                          uint32_t sample, uint32_t bounce, rtz_scatter* out);

/* The order in which the culled constant-bank sweep visits the spheres (host only, no device needed):
 * order_out[slot] = index of the sphere in the list, for the n slots.  Sphere 0 stays in slot 0; the others are
 * regrouped by median splits of their centres into compact blocks of 32 slots. */
int32_t rtz_probe_sweep_order(const rtz_sphere* spheres, uint64_t n_spheres, int32_t* order_out);

/* Color.toRgb (src/color.zig:63-80) on the device for `n` colours (3 f64 each). */
int32_t rtz_probe_to_rgb(const double* linear, uint64_t n, uint8_t* rgb_out);

/* Counter-based RNG stream as the kernels see it: fills `out` with `n` uniform floats in
 * [0,1) from Philox4x32-10 blocks (key = seed, counter = (pixel, sample, bounce, block)). */
int32_t rtz_probe_uniform(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce,
                          uint64_t n, float* out);

/* ---- diagnostics ------------------------------------------------------------------ */
/* Camera.getRay(i, j) for sample `sample` of pixel (i, j) (src/camera.zig:187-215: sampleSquare jitter,
 * defocusDiskSample origin), evaluated by the DEVICE code of the render kernel: n rays for samples
 * sample0 .. sample0+n-1.  origin_out / dir_out receive 3 floats per ray (dir is the UNIT direction),
 * len_out (optional) the length of the un-normalised `pixelSample - origin` the reference stores. */
int32_t rtz_probe_camera_ray(const rtz_camera* camera, uint64_t i, uint64_t j, uint64_t sample0, uint64_t n,
                             float* origin_out, float* dir_out, float* len_out);

const char* rtz_strerror(int32_t status);
const char* rtz_last_error(void);   /* detail of the last RTZ_ERR_CUDA on this thread        */
int32_t rtz_abi_version(void);
int32_t rtz_device_count(int32_t* count_out);

/* Measured FP32 pipe peak for the roofline denominator (SURVEY.md §8d asks for a measured
 * FFMA-chain figure next to the nominal 148*128*2*f_clk): runs an unrolled independent
 * FFMA-chain kernel on the device and returns TFLOP/s.  variant 0 = scalar FFMA,
 * 1 = packed FFMA2 (fma.rn.f32x2), 2 = FFMA2 with a scalar-broadcast operand.  (The sweep loop's
 * own ceiling is measured by tools/ubench/sweep_shapes.cu.) */
int32_t rtz_measure_fp32_peak(int32_t device, int32_t variant, double* tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* RTZ_H */
