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
    double albedo[3];         /* lambertian, metal: every component in [0, 1] (-0.0 included), */
                              /* else RTZ_ERR_BAD_ARG at upload.  Samples then lie in [0, 1].   */
                              /* Each is clamped at 0 and added to an unsigned 32.32 fixed-     */
                              /* point pixel sum, which agrees with the reference (it sums      */
                              /* signed samples and clamps the mean) only for samples >= 0, and */
                              /* a sum stays <= spp * 2^32 < 2^63: exact for every accepted     */
                              /* spp.  Unchecked for a dielectric: its scatter never reads it.  */
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
    double t_min, t_max;              /* Scene.interval, (1e-3, +inf)  (src/Scene.zig:21);    */
                                      /* t_min < 0 is refused by the renders (RTZ_ERR_BAD_ARG;*/
                                      /* -0.0 renders as 0), t_max may be anything but NaN     */
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

/* rtz_scene_upload of a list that is already in DEVICE memory: d_spheres holds n_spheres records, in device or
 * managed memory usable from the context's device (else RTZ_ERR_BAD_ARG).  They are read on the context's stream, so
 * the caller orders them like any other input of the resident API; the call returns once they have been read and
 * keeps nothing of them.  The context's state afterwards is that of rtz_scene_upload of the same list, bit for bit,
 * and so are its refusals: the same status and rtz_last_error for the same first refused sphere, the installed scene
 * left as it was.  Up to 512 padded spheres the list comes to the host (<= 40 KiB) and takes rtz_scene_upload's path;
 * larger lists are checked and flattened on the device, without the host pass rtz_scene_upload makes. */
int32_t rtz_scene_upload_device(rtz_context* ctx, const rtz_sphere* d_spheres, uint64_t n_spheres);

/* Scene.init(seed) followed by Scene.generateWorld / generateChapter13 (src/Scene.zig:23-46, 48-134,
 * 136-182), or BASELINE config 5's generalised final scene of exactly n_spheres spheres, generated ON THE
 * DEVICE by one thread with the reference's exact PRNG stream (Zig std DefaultPrng = Xoshiro256++ seeded by
 * SplitMix64, Random.float(f64)), then installed from device memory as the context's scene (rtz_scene_upload_device).
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

/* rtz_render_resident, plus the linear colour before gamma/quantisation as f32 (3 per pixel, same layout as
 * d_rgb_out: compact tiles for a shard, row-major for the whole frame): (float) of rtz_render_linear's value.
 * The bytes are rtz_render_resident's.  d_linear_out (DEVICE) is required; the legacy modes are refused. */
int32_t rtz_render_resident_linear(rtz_context* ctx, const rtz_camera* camera, const rtz_shard* shard,
                                   uint8_t* d_rgb_out, float* d_linear_out, rtz_stats* stats_out);

/* First-hit guides of the frame's camera rays, samples 0 .. guide_samples-1 of every pixel (whole frame,
 * row-major, top row first, 3 f32 per pixel each).  Either output may be NULL, not both.
 * For each sample the ray is the frame's own camera ray (the counter-based RNG at (seed, pixel, sample, 0)) and
 * its closest hit the render's first hit.  albedo: the sphere's albedo (lambertian, metal), (1,1,1) (dielectric),
 * the sky colour the render returns for that ray on a miss; normal: the unit normal against the ray, (0,0,0) on a
 * miss.  Per pixel, the samples' f32 values are added in ascending sample order from +0 and divided by
 * guide_samples once; normals are not renormalised.  Guides do not depend on bounce_max, and RTZ_MODE_PATH_BVH
 * gives the buffers of RTZ_MODE_PATH.  In RTZ_MODE_PATH_BVH, for a scene of more than 512 spheres (padded to
 * whole 32-sphere blocks), the hits are found through the BVH (built on first use, as for a BVH render); the buffers
 * are still those of RTZ_MODE_PATH, bit for bit.  RTZ_ERR_BAD_ARG for a legacy mode, has_seed == 0 (an OS-drawn seed would
 * give other rays than the frame's), guide_samples == 0 or > samples_per_pixel, both outputs NULL, or more than
 * 2^31 - 1 work items (pixels for guide_samples >= 64).
 * stats: samples = segments = width*height*guide_samples, sphere_tests, kernel_launches, trace_ms = total_ms
 * (the guide kernel), seed_used; the rest 0.  sphere_tests is segments * n for the brute-force sweeps and, through
 * the BVH, the tests actually made (the rays that fill a warp's last 64 slots included).  Blocks like
 * rtz_render_resident. */
int32_t rtz_render_guides(rtz_context* ctx, const rtz_camera* camera, uint64_t guide_samples,
                          float* d_albedo_out, float* d_normal_out, rtz_stats* stats_out);

/* rtz_render_guides for this rank's tiles (rtz_shard): the outputs are DEVICE buffers of 3 f32 per pixel for
 * rtz_shard_pixels(...) pixels in the compact tile layout of rtz_render_resident, tile-padding pixels 0.  Every pixel's
 * values are the whole frame's (its rays are keyed by its global index y*width + x), so the shards' buffers, gathered
 * and passed through rtz_deinterleave_f32, equal rtz_render_guides bit for bit.  shard == NULL is rtz_render_guides.
 * RTZ_ERR_BAD_ARG as rtz_render_guides (the 2^31 - 1 work items count the shard's padded pixels), and for a shard
 * with rank >= world or a zero tile size.  stats as rtz_render_guides, samples = segments = the shard's pixels
 * (padding excluded) * guide_samples. */
int32_t rtz_render_guides_sharded(rtz_context* ctx, const rtz_camera* camera, const rtz_shard* shard,
                                  uint64_t guide_samples, float* d_albedo_out, float* d_normal_out, rtz_stats* stats_out);

/* ---- denoiser: edge-avoiding à-trous wavelet filter (Dammertz et al. 2010) over the linear colour, guided by the
 * first-hit albedo and normal above ---------------------------------------------------------------------------
 * Per pixel the colour is demodulated by the albedo (e = c / max(a, 2^-8)), filtered in `levels` passes of 5x5 taps
 * at steps 1, 2, 4 ... with B3-spline weights times three edge-stopping factors E(x) = max(0, 1 - x/64)^64 of the
 * squared differences of e (scaled by 4^k / sigma_color^2 at level k), of the normal (1 / sigma_normal^2) and of the
 * albedo (1 / sigma_albedo^2), then remodulated; a tap at x >= 64 contributes nothing.  The bytes are Color.toRgb of
 * the f32 result, as the resolve forms them.  IEEE f32 arithmetic in a fixed order (DESIGN.md §5 K7): the output is
 * reproducible bit for bit.  The filter runs on one device over the whole frame; a sharded or multi-GPU frame brings
 * its linear colour and guides to that device first (rtz_deinterleave_f32, rtz_multi_render_denoised). */
typedef struct rtz_denoise_params {
    uint32_t levels;       /* à-trous levels, step 2^k for k < levels; 0 = copy; <= 8                       */
    uint32_t reserved;     /* must be 0                                                                     */
    double sigma_color;    /* > 0, finite: edge scale of the demodulated colour at level 0                  */
    double sigma_normal;   /* > 0, finite                                                                   */
    double sigma_albedo;   /* > 0, finite                                                                   */
} rtz_denoise_params;
/* params NULL: levels 5, sigma_color 0.25, sigma_normal 0.25, sigma_albedo 0.25 */

/* Whole frame, row-major, 3 f32 per pixel in each DEVICE buffer (d_color: rtz_render_resident_linear's linear
 * colour; d_albedo / d_normal: rtz_render_guides' buffers); params NULL = the defaults above.  d_linear_out receives
 * the denoised linear colour (3 f32 per pixel), d_rgb_out its bytes (3 per pixel); either may be NULL, not both.
 * RTZ_ERR_BAD_ARG for a NULL context or input, both outputs NULL, an output that overlaps an input or the other
 * output, a zero width or height or more than 2^31 - 1 pixels, levels > 8, reserved != 0, a sigma that is <= 0 or
 * not finite, or a sigma_color so small that 4^(levels-1) / sigma_color^2 overflows f32.
 * stats: kernel_launches and total_ms (CUDA events on the context's stream); the rest 0.  Blocks like
 * rtz_render_resident. */
int32_t rtz_denoise(rtz_context* ctx, uint64_t width, uint64_t height, const float* d_color, const float* d_albedo,
                    const float* d_normal, const rtz_denoise_params* params, float* d_linear_out, uint8_t* d_rgb_out,
                    rtz_stats* stats_out);

/* rtz_render with host buffers, denoised: the linear colour of the frame (rtz_render_resident_linear), the guides of
 * its samples 0 .. guide_samples-1 (rtz_render_guides) and rtz_denoise of the three, in the cached per-device context.
 * guide_samples 0 = min(samples_per_pixel, 16).  has_seed == 0: ONE seed is drawn and keys both the render and the
 * guides (stats_out->seed_used reports it).  rgb_out (3 bytes per pixel) and linear_out (3 f32 per pixel, the
 * denoised linear colour) are HOST buffers; either may be NULL, not both.  RTZ_ERR_BAD_ARG as rtz_render and
 * rtz_denoise, and for a legacy mode or guide_samples > samples_per_pixel.  One GPU; rtz_render_multi_denoised is
 * the same frame on N.
 * stats: the render's counters as rtz_render reports them; kernel_launches counts every launch of the call and
 * total_ms runs from the first launch to the denoised bytes. */
int32_t rtz_render_denoised(const rtz_camera* camera, const rtz_sphere* spheres, uint64_t n_spheres,
                            uint64_t guide_samples, const rtz_denoise_params* params, uint8_t* rgb_out,
                            float* linear_out, rtz_stats* stats_out);

/* Rank-0 side of the tile gather: `d_gathered` holds `world` compact buffers of equal
 * size (rtz_shard_pixels of rank 0, the largest) back to back, as an all-gather /
 * gather leaves them; writes the plain row-major image to `d_rgb_out` (device). */
int32_t rtz_deinterleave(rtz_context* ctx, uint64_t width, uint64_t height, uint32_t world,
                         uint32_t tile_w, uint32_t tile_h, const uint8_t* d_gathered,
                         uint8_t* d_rgb_out);

/* The same for 3 f32 per pixel (the linear colour of rtz_render_resident_linear, the guides of
 * rtz_render_guides_sharded): `d_gathered` holds `world` compact buffers back to back, `d_out` (device) receives
 * width*height*3 f32, row-major.  Arguments and refusals as rtz_deinterleave. */
int32_t rtz_deinterleave_f32(rtz_context* ctx, uint64_t width, uint64_t height, uint32_t world,
                             uint32_t tile_w, uint32_t tile_h, const float* d_gathered, float* d_out);

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

/* rtz_render_denoised on all devices of `multi`: the same bytes and the same f32 linear colour, bit for bit, for any
 * device count, tile size and transport.  Every device traces its tiles, resolves their linear colour in f32 and runs
 * the guide kernel over them on its own stream (all enqueued before the first wait); the three f32 planes reach
 * device 0 either (P2P) stored straight into its row-major planes through peer memory, or (NCCL) as compact buffers
 * over one grouped ncclSend/ncclRecv, de-interleaved there.  Device 0 then denoises the whole frame.  One device is
 * rtz_render_denoised on it.  Arguments, defaults (guide_samples 0 = min(spp, 16); has_seed == 0: ONE seed for the
 * frame, reported in seed_used) and refusals as rtz_render_denoised; rgb_out / linear_out are HOST buffers.
 * stats: the render's counters summed over the devices (the guide rays are not samples); kernel_launches counts every
 * launch; trace_ms = slowest device's path trace; gather_ms = first launch -> the denoiser's inputs complete on
 * device 0, minus trace_ms (it holds the guide kernels and the exchange); total_ms = first launch -> denoised bytes on
 * device 0; gpus, gather and seed_used as rtz_multi_render. */
int32_t rtz_multi_render_denoised(rtz_multi* multi, const rtz_camera* camera, uint64_t guide_samples,
                                  const rtz_denoise_params* params, uint8_t* rgb_out, float* linear_out,
                                  rtz_stats* stats_out);
/* One-shot form with HOST buffers on num_gpus devices (<= 0: all), on the rtz_multi rtz_render_multi keeps. */
int32_t rtz_render_multi_denoised(const rtz_camera* camera, const rtz_sphere* spheres, uint64_t n_spheres,
                                  int32_t num_gpus, uint64_t guide_samples, const rtz_denoise_params* params,
                                  uint8_t* rgb_out, float* linear_out, rtz_stats* stats_out);

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

/* Batched probes: m records in one launch, one device thread each, through the per-ray device code of the
 * render kernels.  Inputs and outputs are f32, as the device holds them, so a CPU restatement can be compared
 * bit for bit.  The one-ray probes above are calls into these. */
typedef struct rtz_probe_ray {
    float orig[3];
    float dir[3];          /* any length: normalised as the kernels normalise a scattered direction    */
    int32_t self;          /* sphere the origin lies on (exact c = 0 for it), -1 for none              */
} rtz_probe_ray;

typedef struct rtz_ray_hit {
    int32_t best;          /* index of the sphere hit, -1 = miss                                      */
    int32_t front;         /* HitRecord.front                                                          */
    float t;               /* closest hit in DISTANCE units (t_max * len on a miss)                   */
    float len;             /* |dir|: t / len is the reference's t                                     */
    float point[3];
    float normal[3];       /* unit, against the ray                                                   */
} rtz_ray_hit;

/* HittableList.hit(ray, Interval(t_min, t_max)) for m rays (set_direction, then the sweep's gate and root).
 * Any interval is taken, a negative t_min included, as the reference's HittableList.hit takes it (its unit test
 * uses Interval(-6, 6)): this scalar sweep tests every sphere and both roots against the interval.  The render
 * calls and rtz_probe_sweeps, whose sweeps rely on t_min >= 0, refuse a negative t_min. */
int32_t rtz_probe_hits(const rtz_sphere* spheres, uint64_t n_spheres, const rtz_probe_ray* rays, uint64_t m,
                       double t_min, double t_max, rtz_ray_hit* out);

typedef struct rtz_probe_bounce {
    int32_t sphere;        /* the sphere the ray hits; t_min = 0.001, t_max = +inf, no self            */
    float orig[3];
    float dir[3];
    uint32_t pixel, sample, bounce;  /* the counter-based RNG stream of the scatter                    */
} rtz_probe_bounce;

typedef struct rtz_ray_scatter {
    int32_t term;          /* -1 scattered, 1 absorbed, -2 the ray misses the sphere                  */
    float orig[3];         /* the scattered ray (term == -1)                                           */
    float dir[3];          /* unit                                                                     */
    float len;             /* length of the direction before normalisation                             */
    float attenuation[3];
} rtz_ray_scatter;

/* Sphere.hit then Material.scatter (the kernels' shade) for m records, RNG keyed by `seed`. */
int32_t rtz_probe_scatters(const rtz_sphere* spheres, uint64_t n_spheres, const rtz_probe_bounce* recs, uint64_t m,
                           uint64_t seed, rtz_ray_scatter* out);

/* The order in which the culled constant-bank sweep visits the spheres (host only, no device needed):
 * order_out[slot] = index of the sphere in the list, for the n slots.  Sphere 0 stays in slot 0; the others are
 * regrouped by median splits of their centres into compact blocks of 32 slots. */
int32_t rtz_probe_sweep_order(const rtz_sphere* spheres, uint64_t n_spheres, int32_t* order_out);

/* The culled sweep's block bounds (host only, no device needed), on the regrouped order of rtz_probe_sweep_order:
 * for each of the ceil(n_pad / 32) blocks (n_pad = n rounded up to a multiple of 8), the padded box as the kernel
 * receives it, 6 floats {lo.x, hi.x, lo.y, hi.y, lo.z, hi.z} (block 0, always swept, has none: zeros); cull_r2, the
 * squared origin radius the padding covers; and whether a render culls this scene (1) or sweeps it plainly (0).
 * RTZ_ERR_BAD_ARG for null outputs and for the spheres rtz_scene_upload refuses. */
int32_t rtz_probe_cull_bounds(const rtz_sphere* spheres, uint64_t n_spheres, float* boxes_out, float* cull_r2_out,
                              int32_t* host_culls_out);

/* The production sweeps of the render kernels, for chosen rays: each kind runs the device function the named
 * kernel runs, with the same template arguments, and fills rtz_ray_hit as rtz_probe_hits does (best in the
 * caller's sphere indices, point and normal from the caller's rows), so one comparison against the f32 mirror
 * covers it.
 *   RTZ_SWEEP_CONST            packed sweep over the constant bank (the lockstep kernel, up to 512 spheres)
 *   RTZ_SWEEP_CULL             the culled constant-bank sweep on the regrouped rows, boxes and cull_r2 of the
 *                              upload, whether or not a render would cull the scene; split_max (0 .. 64) is the
 *                              sphere-parallel threshold a frame takes from RTZ_SPLIT
 *   RTZ_SWEEP_SKIP_SELF        the wavefront kernel's sweep, which drops the sphere a ray leaves outwards (the
 *                              flag is set from the ray's self as the shader sets it)
 *   RTZ_SWEEP_SMEM             the rows staged into shared memory (refused where they do not fit)
 *   RTZ_SWEEP_GLOBAL           the rows read from global memory
 *   RTZ_SWEEP_COOP             the drain's warp-cooperative sweep, one ray by the whole warp at a time
 *   RTZ_SWEEP_COOP_REGROUPED   the same on the regrouped rows, ties by original index
 *   RTZ_SWEEP_BVH              the RTZ_MODE_PATH_BVH traversal, one ray per thread
 *   RTZ_SWEEP_WAVE4            the four-path wavefront kernel's sweep over the constant bank (128 paths per warp,
 *                              up to 512 spheres), which drops the sphere a ray leaves outwards as SKIP_SELF does
 * The two-path kinds (CONST .. GLOBAL) take warps of 64 rays: warp w holds ray 64 w + l in lane l's first slot and
 * 64 w + 32 + l in its second, so m must be a multiple of 64.  RTZ_SWEEP_WAVE4 takes warps of 128 rays, ray
 * 128 w + l + 32 h in lane l's slot h, so m must be a multiple of 128.  RTZ_ERR_BAD_ARG (with rtz_last_error) for
 * null pointers, m > 2^31, an unknown kind, split_max outside 0 .. 64, such an m, a constant-bank kind above 512
 * spheres, t_min < 0, a ray whose self is not -1 or a sphere index, and the spheres rtz_scene_upload refuses. */
#define RTZ_SWEEP_CONST 0
#define RTZ_SWEEP_CULL 1
#define RTZ_SWEEP_SKIP_SELF 2
#define RTZ_SWEEP_SMEM 3
#define RTZ_SWEEP_GLOBAL 4
#define RTZ_SWEEP_COOP 5
#define RTZ_SWEEP_COOP_REGROUPED 6
#define RTZ_SWEEP_BVH 7
#define RTZ_SWEEP_WAVE4 8
int32_t rtz_probe_sweeps(const rtz_sphere* spheres, uint64_t n_spheres, const rtz_probe_ray* rays, uint64_t m,
                         double t_min, double t_max, int32_t kind, int32_t split_max, rtz_ray_hit* out);

/* The rows a context holds for its scene, back to back, for comparing two installs byte for byte: int32 n_spheres,
 * n_pad, cull; f32 cull_r2; then the device rows geom, pairs, aux, albedo (n_pad float4 each), wexp (n_pad f32) and the
 * f64 spheres of the legacy kernel (n_spheres x 32 B); for n_pad <= 512 also the constant-bank pair rows and block
 * boxes and, for a culled scene, the regrouped rows and slot -> index map.  *bytes_out receives the size; out NULL
 * asks for the size only, a smaller cap is RTZ_ERR_BAD_ARG. */
int32_t rtz_probe_scene_rows(rtz_context* ctx, void* out, uint64_t cap, uint64_t* bytes_out);

/* The BVH of RTZ_MODE_PATH_BVH for the context's scene, built by `builder` without installing it: the nodes (64 B
 * each, pre-order, root first) to nodes_out, the leaf ranges' sphere indices to order_out (n_spheres entries), the
 * squared origin radius the boxes cover to r2_out; *n_nodes_out receives the node count.  Any output may be NULL;
 * node_cap below the count is RTZ_ERR_BAD_ARG.  Both builders give the same nodes and r2 and the same set of spheres
 * in every leaf (order inside a leaf may differ); a render picks one by scene size.  Below 5 spheres the device
 * builder hands over to the host one. */
#define RTZ_BVH_HOST 0
#define RTZ_BVH_DEVICE 1
int32_t rtz_probe_bvh(rtz_context* ctx, int32_t builder, void* nodes_out, uint64_t node_cap, int32_t* order_out,
                      float* r2_out, uint64_t* n_nodes_out);

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
