/*
 * rtb200.h — C-ABI of the B200-native path-tracing hot path.
 *
 * This is the drop-in boundary for ONE path of patrickzbhe/ray-tracing-series-rust:
 *     render_scene(world, cam, background, config)            (src/world.rs:1181-1247)
 *     render_scene_with_time(t0, t1, path, world)             (src/world.rs:1249-1330)
 * and the operator traits that path drives
 *     Hittable::{hit, bounding_box}                           (src/hit.rs:82-85)
 *     Material::{scatter, emitted}                            (src/hit.rs:1013-1018)
 *     Texture::value                                          (src/texture.rs:7-9)
 *
 * The reference has no FFI today.  A Rust host keeps its scene-construction API
 * (Sphere::new, HittableList::add, BvhNode::from_list, Camera::new, ...) and each
 * constructor records itself through one call below (INTEGRATION.md shows the
 * `extern "C"` block and the `flatten()` shim).  Every entry point cites the
 * reference interface it replaces as  [ref: file:line].
 *
 * Conventions
 *   - plain pointers + sizes only; host arrays are copied at call time, the caller
 *     keeps ownership of its buffers;
 *   - builder calls return a non-negative id (separate id spaces for textures,
 *     materials and hittables, each counting from 0 in call order) or a negative
 *     rt_status;  everything else returns rt_status (0 = ok);
 *   - RTB_FN(last_error)() returns a thread-local, NUL-terminated description of the
 *     last failure on the calling thread;
 *   - the library owns all device memory; one scene is bound to the CUDA device that
 *     is current when RTB_FN(scene_commit) is called (one process per GPU);
 *   - there is NO CPU fallback: render/trace calls fail with RT_ERR_CUDA when no
 *     device is present.
 *
 * The same declarations, compiled with -DRTB_PREFIX_ORC, name the CPU oracle's
 * entry points (orc_*), so tests drive both sides with identical call sequences.
 */
#ifndef RTB200_H
#define RTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifdef RTB_PREFIX_ORC
#define RTB_FN(name) orc_##name
#else
#define RTB_FN(name) rt_##name
#endif

#if defined(__GNUC__)
#define RTB_EXPORT __attribute__((visibility("default")))
#else
#define RTB_EXPORT
#endif

typedef struct rt_scene rt_scene; /* opaque */

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = -1,     /* bad argument / id out of range */
    RT_ERR_STATE = -2,       /* call order (e.g. render before commit) */
    RT_ERR_UNSUPPORTED = -3, /* scene shape the flattener cannot express (documented in DESIGN.md) */
    RT_ERR_IO = -4,          /* file open / parse */
    RT_ERR_CUDA = -5,        /* no device, launch or allocation failure */
    RT_ERR_EMPTY = -6        /* empty group given to a BVH  [ref: src/bvh.rs:27-28 unwrap() panic] */
} rt_status;

/* ---------------------------------------------------------------- lifetime */
RTB_EXPORT rt_scene* RTB_FN(scene_create)(void);
RTB_EXPORT void RTB_FN(scene_destroy)(rt_scene* s);
RTB_EXPORT const char* RTB_FN(last_error)(void);
/* "rtb200 <version> sm_100a" or "oracle ..." */
RTB_EXPORT const char* RTB_FN(version)(void);

/* ---------------------------------------------------------------- textures -> tex id */
/* SolidColor::new / from_colors                    [ref: src/texture.rs:16-24, value 27-31] */
RTB_EXPORT int32_t RTB_FN(tex_solid)(rt_scene* s, const double rgb[3]);
/* Checker::new(even, odd)                          [ref: src/texture.rs:39-51, value 54-64] */
RTB_EXPORT int32_t RTB_FN(tex_checker)(rt_scene* s, int32_t even_tex, int32_t odd_tex);
/* Noise::new(scale) with the Perlin tables passed as data (the reference draws them from an
 * unseeded thread_rng, src/perlin.rs:14-26,68-83): ranvec = 256 xyz triples, perm_* = 256 ints.
 * Any table pointer NULL => the library draws all four from `seed` with the reference's
 * procedure (U[-1,1)^3 gradients; shuffle i = 254..1).        [ref: src/texture.rs:72-88] */
RTB_EXPORT int32_t RTB_FN(tex_noise)(rt_scene* s, double scale, const double* ranvec768,
                                     const int32_t* perm_x256, const int32_t* perm_y256,
                                     const int32_t* perm_z256, uint64_t seed);
/* Image texture from texels already in memory: rgb = w*h*3 doubles in file order (row 0 = top),
 * values on the 0..255 scale of a P3 file.         [ref: src/texture.rs:90-121] */
RTB_EXPORT int32_t RTB_FN(tex_image)(rt_scene* s, int32_t w, int32_t h, const double* rgb);
/* Image::from_ppm(name): P3 reader                 [ref: src/texture.rs:95-99, src/screen.rs:61-95] */
RTB_EXPORT int32_t RTB_FN(tex_image_ppm)(rt_scene* s, const char* path);

/* ---------------------------------------------------------------- materials -> mat id */
/* Lambertian::from_pointer (Lambertian::new == tex_solid + this)   [ref: src/hit.rs:1025-1051] */
RTB_EXPORT int32_t RTB_FN(mat_lambertian)(rt_scene* s, int32_t albedo_tex);
/* Metal::new(albedo, fuzz): fuzz clamped to <= 1                   [ref: src/hit.rs:1060-1083] */
RTB_EXPORT int32_t RTB_FN(mat_metal)(rt_scene* s, const double albedo[3], double fuzz);
/* Dielectric::new(ir)                                              [ref: src/hit.rs:1091-1126] */
RTB_EXPORT int32_t RTB_FN(mat_dielectric)(rt_scene* s, double ir);
/* DiffuseLight::from_pointer (new == tex_solid + this)             [ref: src/hit.rs:1134-1151] */
RTB_EXPORT int32_t RTB_FN(mat_diffuse_light)(rt_scene* s, int32_t emit_tex);
/* Isotropic::from_color via a texture id                           [ref: src/hit.rs:997-1011] */
RTB_EXPORT int32_t RTB_FN(mat_isotropic)(rt_scene* s, int32_t albedo_tex);

/* ---------------------------------------------------------------- hittables -> hittable id
 * Ids mirror Arc sharing: passing the same id twice is the same object reached twice. */
/* Sphere::new                                      [ref: src/hit.rs:187-244] */
RTB_EXPORT int32_t RTB_FN(sphere)(rt_scene* s, const double center[3], double radius, int32_t mat);
/* MovingSphere::new                                [ref: src/hit.rs:257-327] */
RTB_EXPORT int32_t RTB_FN(moving_sphere)(rt_scene* s, const double center0[3],
                                         const double center1[3], double time0, double time1,
                                         double radius, int32_t mat);
/* GravitySphere::new: the library integrates the 100 001-entry height table with the
 * reference's recurrence                           [ref: src/hit.rs:340-444] */
RTB_EXPORT int32_t RTB_FN(gravity_sphere)(rt_scene* s, const double start[3], double time0,
                                          double radius, int32_t mat);
/* XyRect::new / XzRect::new / YzRect::new          [ref: src/hit.rs:456-508, 521-573, 586-638] */
RTB_EXPORT int32_t RTB_FN(xy_rect)(rt_scene* s, double x0, double x1, double y0, double y1,
                                   double k, int32_t mat);
RTB_EXPORT int32_t RTB_FN(xz_rect)(rt_scene* s, double x0, double x1, double z0, double z1,
                                   double k, int32_t mat);
RTB_EXPORT int32_t RTB_FN(yz_rect)(rt_scene* s, double y0, double y1, double z0, double z1,
                                   double k, int32_t mat);
/* RectPrism::new(p0, p1, mat): six rect leaves in the reference's side order
 *                                                  [ref: src/hit.rs:720-785] */
RTB_EXPORT int32_t RTB_FN(box)(rt_scene* s, const double p0[3], const double p1[3], int32_t mat);
/* Triangle::new                                    [ref: src/hit.rs:96-177] */
RTB_EXPORT int32_t RTB_FN(triangle)(rt_scene* s, const double v0[3], const double v1[3],
                                    const double v2[3], int32_t mat);
/* TriangleModel::to_hittable in one call: a HittableList of nt triangles (verts = nv xyz
 * triples, idx = nt index triples), all with material `mat`
 *                                                  [ref: src/model.rs:64-76] */
RTB_EXPORT int32_t RTB_FN(triangle_mesh)(rt_scene* s, const double* verts, int64_t nv,
                                         const uint32_t* idx, int64_t nt, int32_t mat);
/* TriangleModel::load_from_file(path, scale).to_hittable(): same ASCII-PLY subset
 *                                                  [ref: src/model.rs:13-76] */
RTB_EXPORT int32_t RTB_FN(ply_load)(rt_scene* s, const char* path, double scale, int32_t mat);
/* HittableList::new + add ...                      [ref: src/hit.rs:646-710] */
RTB_EXPORT int32_t RTB_FN(list)(rt_scene* s, const int32_t* ids, int32_t n);
/* BvhNode::from_list(list, time0, time1); ids = the list's objects; n == 0 is RT_ERR_EMPTY
 *                                                  [ref: src/bvh.rs:14-116] */
RTB_EXPORT int32_t RTB_FN(bvh)(rt_scene* s, const int32_t* ids, int32_t n, double time0,
                               double time1);
/* Translate::new / RotateY::new(angle in degrees)  [ref: src/hit.rs:793-832, 843-936] */
RTB_EXPORT int32_t RTB_FN(translate)(rt_scene* s, const double offset[3], int32_t child);
RTB_EXPORT int32_t RTB_FN(rotate_y)(rt_scene* s, double angle_deg, int32_t child);
/* ConstantMedium::from_color(color, density, boundary)   [ref: src/hit.rs:945-989] */
RTB_EXPORT int32_t RTB_FN(constant_medium)(rt_scene* s, const double rgb[3], double density,
                                           int32_t boundary);

/* ---------------------------------------------------------------- scene */
RTB_EXPORT int32_t RTB_FN(scene_set_root)(rt_scene* s, int32_t hittable);
/* Camera::new — same nine arguments                [ref: src/camera.rs:20-57] */
RTB_EXPORT int32_t RTB_FN(scene_set_camera)(rt_scene* s, const double lookfrom[3],
                                            const double lookat[3], const double vup[3],
                                            double vfov_deg, double aspect_ratio, double aperture,
                                            double focus_dist, double time1, double time2);
/* the `background` argument of render_scene        [ref: src/world.rs:1184, 86-89] */
/* The same camera from the 24 f64 fields the reference's Camera stores, in declaration order: origin[3],
 * lower_left_corner[3], horizontal[3], vertical[3], u[3], v[3], w[3], lens_radius, time1, time2
 * [ref: src/camera.rs:6-17].  A Rust `Camera` keeps only these (not its constructor arguments), so this is the call
 * its flatten() makes; rt_scene_set_camera derives the same block from Camera::new's arguments. */
RTB_EXPORT int32_t RTB_FN(scene_set_camera_fields)(rt_scene* s, const double fields[24]);
RTB_EXPORT int32_t RTB_FN(scene_set_background)(rt_scene* s, const double rgb[3]);
/* Book-1 sky: a miss contributes (1 - t) * horizon + t * zenith with t = 0.5 * (unit(direction).y + 1) instead of the
 * constant background.  HEAD of the reference only has the constant (src/world.rs:86-89); the revision that rendered the
 * shipped images/book1.png (README.md:18) used this sky with horizon (1,1,1), zenith (0.5,0.7,1.0), so the option
 * exists to check renders against that reference-held image (tests/test_reference_images.py).
 * rt_scene_set_background switches back to the constant. */
RTB_EXPORT int32_t RTB_FN(scene_set_background_gradient)(rt_scene* s, const double horizon_rgb[3],
                                                         const double zenith_rgb[3]);
/* Freeze the scene: number the leaves depth-first, flatten, build the device BVH, upload to the
 * current CUDA device.  Replaces "Arc::new(world)" hand-off at src/world.rs:1181-1186. */
RTB_EXPORT int32_t RTB_FN(scene_commit)(rt_scene* s);
/* the scene library of src/world.rs:95-874 + camera presets 876-1179 restated on this API:
 * builds scene `scene_id` (ids of get_world_cam; 13 = book-1 classic static variant "C1a",
 * 14 = synthetic dragon-scale mesh room) with scene randomness drawn from `seed`, sets root,
 * camera and background, does NOT commit.  `param` = scene-specific size knob (mesh quads per
 * side for 11/14; 0 = default). */
RTB_EXPORT int32_t RTB_FN(world_build)(rt_scene* s, int32_t scene_id, uint64_t seed, int32_t param);

/* number of reporting leaves (prim ids 0..n-1) after commit */
RTB_EXPORT int32_t RTB_FN(scene_num_prims)(rt_scene* s);

/* ---------------------------------------------------------------- render */
typedef struct rt_render_config {
    int32_t image_width;       /* Config.image_width                     [ref: src/world.rs:20-50] */
    double aspect_ratio;       /* Config.aspect_ratio: H = (W / aspect) as i32   [world.rs:1192] */
    int32_t samples_per_pixel; /* Config.samples_per_pixel */
    int32_t max_depth;         /* Config.max_depth */
    int32_t compat_threads;    /* 0 = render every row; N>0 = reproduce the reference's
                                  H - N*(H/N) unrendered top rows          [world.rs:1198-1202] */
    uint64_t seed;             /* Philox key (the reference is unseeded) */
    int32_t sample_begin;      /* this call renders samples [sample_begin, sample_end) of     */
    int32_t sample_end;        /* [0, samples_per_pixel): the multi-GPU sample-range shard.    */
                               /* sample_end == 0 means samples_per_pixel.                     */
    int32_t threads;           /* oracle only: worker threads (row bands); ignored on the GPU  */
    int32_t flags;             /* RT_RENDER_* */
} rt_render_config;

#define RT_RENDER_DEFAULT 0
/* diagnostics / mode selection (GPU library; the oracle ignores them) */
#define RT_RENDER_TIMED_EXTEND 1    /* bracket every k_extend launch with CUDA events -> rt_stats.ms_extend */
#define RT_RENDER_COUNT_EVENTS 2    /* count BVH boxes tested / primitive tests on the device -> rt_stats */
#define RT_RENDER_FORCE_WAVEFRONT 4 /* wavefront mode: k_extend + k_shade_all per iteration, per-material queues */
#define RT_RENDER_FORCE_FUSED 8     /* fused mode: one persistent kernel, path state in registers */
#define RT_RENDER_FORCE_POOL 16     /* pool mode: one persistent kernel, every warp runs a small wavefront of its own in shared memory */
/* rt_render_device only: return as soon as the render is enqueued on the caller's stream instead of waiting for it, so that the
 * caller's next stream operations (the NCCL reduce, rt_resolve_device) queue up behind the kernel without a host round trip.
 * Honoured by the single-launch modes (fused, pool); the wavefront's host loop ignores it.  stats then carry only what the host
 * knows (paths, kernel_launches); segments and ms_device stay 0. */
#define RT_RENDER_NO_WAIT 32
/* Tile sharding (SURVEY.md 8(e), the GPU analogue of the reference's row bands, world.rs:1198-1227): the image is cut
 * into bands of RT_TILE_ROWS rows; a call with RT_RENDER_TILE_SHARD(rank, count) in `flags` renders only the bands
 * b with b % count == rank (all samples of their pixels); the other pixels of out_accum / out_screen stay 0.  Path ids
 * use the global pixel index, so the sum of the `count` shards is bit-identical to the unsharded render.  Both
 * libraries implement it; it composes with sample_begin / sample_end. */
#define RT_TILE_ROWS 4
#define RT_RENDER_TILE_SHARD(rank, count) ((((rank) & 0x7f) << 16) | (((count) & 0x7f) << 24))
#define RT_RENDER_TILE_RANK(flags) (((flags) >> 16) & 0x7f)
#define RT_RENDER_TILE_COUNT(flags) (((flags) >> 24) & 0x7f)
/* fixed-point scale of the radiance accumulator: sum of samples * 2^32 in an int64 per channel */
#define RT_ACCUM_SCALE_LOG2 32

typedef struct rt_stats {
    uint64_t paths;         /* camera samples traced */
    uint64_t segments;      /* world.hit queries (ray_color loop iterations) */
    uint64_t box_tests;     /* oracle: Aabb::hit calls; GPU: BVH nodes popped (0 unless counted) */
    uint64_t prim_tests[8]; /* by primitive type (rt_prim_type) */
    uint64_t scatters[5];   /* by material type (rt_mat_type) */
    uint64_t medium_queries;
    uint64_t iterations;    /* GPU: wavefront iterations */
    uint64_t kernel_launches;
    double ms_total;        /* wall ms inside the call */
    double ms_device;       /* GPU: CUDA-event ms of the render loop */
    double ms_extend;       /* GPU: CUDA-event ms summed over extend launches (when timed) */
} rt_stats;

typedef enum rt_prim_type {
    RT_PRIM_SPHERE = 0, RT_PRIM_MOVING_SPHERE = 1, RT_PRIM_GRAVITY_SPHERE = 2, RT_PRIM_RECT = 3,
    RT_PRIM_BOX = 4, RT_PRIM_TRIANGLE = 5, RT_PRIM_MEDIUM = 6
} rt_prim_type;
typedef enum rt_mat_type {
    RT_MAT_LAMBERTIAN = 0, RT_MAT_METAL = 1, RT_MAT_DIELECTRIC = 2, RT_MAT_DIFFUSE_LIGHT = 3,
    RT_MAT_ISOTROPIC = 4
} rt_mat_type;

/* render_scene: out_screen = W*H*3 doubles in Screen layout (row 0 = bottom row, integer-valued
 * 0..255 exactly as Vec3::get_normalized_color), or NULL; out_accum = W*H*3 int64 fixed-point
 * radiance sums (RT_ACCUM_SCALE_LOG2), or NULL; stats may be NULL.  Host buffers.
 *                                   [ref: src/world.rs:1181-1247, src/vec3.rs:89-107] */
RTB_EXPORT int32_t RTB_FN(render)(rt_scene* s, const rt_render_config* cfg, double* out_screen,
                                  int64_t* out_accum, rt_stats* stats);
/* The same render spread over n_gpus GPUs of this box by ONE host thread of ONE process (what a Rust render_scene_gpu calls to
 * use the whole 8 x B200 node; SURVEY.md 8(b) n_gpus / shard_mode, 8(e)).  GPU 0 is the device the scene was committed on, GPUs
 * 1..n-1 are the next visible devices; each gets the committed scene's flattened bytes (uploaded once per commit, or ahead of time
 * by rt_scene_commit_multi) and renders one shard: RT_SHARD_SAMPLES = a contiguous range of the samples of every pixel, cut evenly for any
 * sample count (whole samples plus a partial first / last one: perfect balance), RT_SHARD_TILES = every sample of the RT_TILE_ROWS-row bands b with b % n_gpus == g (the reference's row bands,
 * world.rs:1198-1227).  The shards' int64 accumulators are summed and resolved by one kernel on GPU 0 that reads the peers'
 * accumulators in place over NVLink (P2P-mapped pointers; a staged peer copy only where no P2P route exists).  Integer sums and
 * Philox streams keyed by the global pixel / sample index make the image bit-identical to rt_render for every n_gpus and either
 * mode.  cfg->sample_begin / sample_end select the range that is split; RT_RENDER_TILE_SHARD must not be set.  stats: counters
 * summed over the shards, ms_device = the slowest shard.                      [ref: src/world.rs:1181-1247, 1198-1240] */
#define RT_SHARD_SAMPLES 0
#define RT_SHARD_TILES 1
#ifndef RTB_PREFIX_ORC
RTB_EXPORT int32_t rt_render_multi(rt_scene* s, const rt_render_config* cfg, int32_t n_gpus, int32_t shard_mode,
                                   double* out_screen, int64_t* out_accum, rt_stats* stats);
/* rt_scene_commit + upload of the flattened scene to GPUs 1..n_gpus-1 (otherwise the first rt_render_multi does it). */
RTB_EXPORT int32_t rt_scene_commit_multi(rt_scene* s, int32_t n_gpus);

/* Adaptive sampling: every pixel is rendered until its noise estimate converges, at most cfg->samples_per_pixel (= max) samples.
 * Round k traces samples [k*step, min((k+1)*step, max)) of the pixels still active, alternately into two half accumulators A
 * (even k) and B (odd k).  After every odd round, at n = (k+1)*step samples with min_samples <= n < max, each active pixel's
 * error is computed in f64 from its int64 sums (h = n/2 samples in each half, S = h * 2^32):
 *     err = (((|a_r-b_r| + |a_g-b_g|) + |a_b-b_b|) / S) / sqrt(1e-4 + (((a_r+b_r) + (a_g+b_g)) + (a_b+b_b)) / (2*S))
 * A pixel stays active iff a pixel with !(err < threshold) lies within Chebyshev distance `radius` of it (on a rendered row);
 * a pixel that leaves keeps n samples, one that never leaves gets max.  Path ids are rt_render's (pixel * max + sample), so a
 * pixel's sums are exactly those of rt_render over its own samples: threshold 0 reproduces rt_render bit for bit.
 * out_accum = A + B; out_screen resolves each pixel with its own count; out_samples (W*H int32, nullable) = the counts, 0 on
 * unrendered compat_threads rows.  cfg must render the whole [0, samples_per_pixel), without a tile shard (RT_RENDER_TILE_SHARD
 * with count > 1; count 0 or 1 means no sharding, as in rt_render) and without RT_RENDER_NO_WAIT; the mode flags apply to every round.  stats: counters and ms_device summed over the rounds. */
typedef struct rt_adaptive_config {
    int32_t min_samples; /* 0 .. samples_per_pixel: no pixel stops before this many samples */
    int32_t step;        /* >= 1: samples per round; check points every 2 rounds */
    double threshold;    /* >= 0 and finite; 0 = no pixel converges (result == rt_render) */
    int32_t radius;      /* 0..8: a pixel stays active while an unconverged pixel is this close */
} rt_adaptive_config;
RTB_EXPORT int32_t rt_render_adaptive(rt_scene* s, const rt_render_config* cfg, const rt_adaptive_config* ac,
                                      double* out_screen, int64_t* out_accum, int32_t* out_samples, rt_stats* stats);
/* The same adaptive render spread over n_gpus GPUs of this box by ONE host thread of ONE process.  GPU 0 is the device the scene
 * was committed on, GPUs 1..n-1 are the next visible devices (replicas, as in rt_render_multi).  Every round's paths over the
 * active list (sample-major, the list's own path space) are cut into n_gpus even ranges, one per GPU, into that GPU's own half
 * accumulators; at each check point GPU 0 computes the error from the sums of every GPU's A and B, read in place over NVLink
 * (P2P-mapped pointers; a staged peer copy only where no P2P route exists), compacts the next list and copies it to the others.
 * Path ids (pixel * max + sample), integer sums and decisions taken from the exact int64 sums make out_accum, out_screen,
 * out_samples and the path and segment counts bit-identical to rt_render_adaptive for every n_gpus; n_gpus == 1 is
 * rt_render_adaptive.  Argument rules are rt_render_adaptive's, plus 1 <= n_gpus <= 16 and no more than the
 * visible devices.  stats: counters summed over the GPUs and the rounds; iterations, ms_device and ms_extend are the slowest
 * GPU's of each round, summed over the rounds. */
RTB_EXPORT int32_t rt_render_adaptive_multi(rt_scene* s, const rt_render_config* cfg, const rt_adaptive_config* ac, int32_t n_gpus,
                                            double* out_screen, int64_t* out_accum, int32_t* out_samples, rt_stats* stats);
#endif

/* First-hit feature buffers of the render's own paths.  For every pixel of a rendered row and every sample s of cfg's range
 * [sample_begin, sample_end): the path's camera ray (pixel jitter, lens, shutter: exactly rt_render's path id pixel*spp + s),
 * ONE world.hit(ray, 0.001, inf) with media sampled from the path's keyed stream at segment 0 (= the render's first hit), then
 *   Lambertian / Isotropic : albedo = Texture::value(u, v, p)         normal = rec.normal (Isotropic: 0)
 *   Metal                  : albedo = Metal.albedo                    normal = rec.normal
 *   Dielectric             : albedo = (1, 1, 1)                       normal = rec.normal
 *   DiffuseLight           : albedo = clamp(emitted(u, v, p), 0, 1)   normal = rec.normal
 *   miss                   : albedo = clamp(background or sky, 0, 1)  normal = 0
 * out_albedo / out_normal (W*H*3 int64, nullable): per-pixel sums of round-to-nearest-even(x * 2^32); rows >= the rendered rows
 * stay 0.  Mode flags are ignored (one kernel); a tile shard (count > 1) and RT_RENDER_NO_WAIT are RT_ERR_INVALID.
 * stats: paths = segments = rays traced.  The oracle's side is built by the tests (tests/oracle_aov). */
RTB_EXPORT int32_t RTB_FN(render_aov)(rt_scene* s, const rt_render_config* cfg, int64_t* out_albedo, int64_t* out_normal, rt_stats* stats);

#ifndef RTB_PREFIX_ORC
/* A denoised render (DESIGN.md section 11; the numpy reference is ray_tracing_series_rust_b200/denoise.py).  With n = samples_per_pixel
 * and hA = n / 2: samples [0, hA) are rendered into a half accumulator A and [hA, n) into B (out_accum = A + B = rt_render's
 * out_accum bit for bit), the feature sums of samples [0, aov_samples) as rt_render_aov, then `iterations` passes of a feature-guided
 * a-trous filter (steps 1, 2, 4, ...) in f64 over the rendered rows, starting from c = mean, v = (lum(A mean) - lum(B mean))^2 hA hB / n^2:
 *   vbar = 3x3 blur of v (1/4, 1/2, 1/4 per axis, valid taps renormalised)
 *   w(q) = h(dx) h(dy) exp(-(|lum(c_p) - lum(c_q)| / (sigma_color sqrt(vbar_p) + 1e-10) + |a_p - a_q|^2 / sigma_albedo^2 + |n_p - n_q|^2 / sigma_normal^2))
 *   over the 25 taps q = p + step (dx, dy), dx, dy in -2..2, h = (1/16, 1/4, 3/8, 1/4, 1/16);  c' = sum w c_q / sum w,  v' = sum w^2 v_q / (sum w)^2
 * lum(x) = (0.2126 r + 0.7152 g) + 0.0722 b; a, n = the feature means (the mean normal is not renormalised).  out_linear (W*H*3
 * doubles, Screen layout) = the filtered mean, out_screen = its Screen values (rt_render's quantisation); rows >= the rendered rows
 * stay 0.  Integer sums and a gather without atomics make every output identical in every render mode and on every run.
 * cfg must render the whole [0, samples_per_pixel) with samples_per_pixel >= 2, without a tile shard (count > 1) and without
 * RT_RENDER_NO_WAIT; the mode flags apply to both half renders.  stats: the half renders' counters summed; kernel_launches also
 * counts the feature pass and the filter kernels. */
typedef struct rt_denoise_config {
    int32_t aov_samples;  /* 1 .. samples_per_pixel: features from the render's samples [0, aov_samples) */
    int32_t iterations;   /* 1 .. 8: a-trous passes, steps 1, 2, 4, ... */
    double sigma_color;   /* > 0, finite: luminance edge stop, in units of the pixel's noise standard deviation */
    double sigma_albedo;  /* > 0, finite */
    double sigma_normal;  /* > 0, finite */
} rt_denoise_config;
RTB_EXPORT int32_t rt_render_denoised(rt_scene* s, const rt_render_config* cfg, const rt_denoise_config* dc,
                                      double* out_screen /* denoised Screen, nullable */, double* out_linear /* nullable */,
                                      int64_t* out_accum /* nullable: == rt_render's out_accum */, rt_stats* stats);
#endif
/* image height the config implies: (image_width as f64 / aspect_ratio) as i32 */
RTB_EXPORT int32_t RTB_FN(image_height)(const rt_render_config* cfg);

#ifndef RTB_PREFIX_ORC
/* Device-resident variants for the multi-GPU path (one process per GPU): the int64 accumulator
 * stays in device memory (caller-allocated, W*H*3 int64, zeroed by the caller or by flags) so
 * the ranks can sum it with one NCCL reduce; `cuda_stream` is a cudaStream_t (NULL = default).
 * rt_resolve_device turns a reduced accumulator into the Screen-layout image (device doubles). */
RTB_EXPORT int32_t rt_render_device(rt_scene* s, const rt_render_config* cfg,
                                    int64_t* d_accum, void* cuda_stream, rt_stats* stats);
/* A path-range shard: of the call's paths (its pixels x its samples [sample_begin, sample_end), enumerated sample-major: index =
 * sample * pixels + pixel) only [path_begin, path_end) are rendered - whole samples plus a partial first / last one.  Lets N ranks
 * split ANY sample count evenly (500 spp on 8 GPUs = 62.5 each); the sum of the shards is bit-identical to the whole render. */
RTB_EXPORT int32_t rt_render_device_paths(rt_scene* s, const rt_render_config* cfg, uint64_t path_begin, uint64_t path_end,
                                          int64_t* d_accum, void* cuda_stream, rt_stats* stats);
RTB_EXPORT int32_t rt_resolve_device(const int64_t* d_accum, double* d_screen, int32_t width,
                                     int32_t height, int32_t samples_per_pixel,
                                     int32_t rendered_rows, void* cuda_stream);
#endif

/* ---------------------------------------------------------------- peer group (product only)
 * The exchange of the one-process-per-GPU layout (torchrun) done by the library itself over NVLink peer memory instead of a
 * collective: every rank renders into an accumulator the library allocates and exports through CUDA IPC; rank 0 maps all of them
 * and ONE kernel there (the k_reduce_resolve of rt_render_multi) waits for each peer's "published" flag - written by the peer's
 * stream behind its render - reads the shards in place, sums and resolves.  No host round trip between the render and the gather.
 *   all ranks : g = rt_peer_create(rank, world, W*H*3, handle);  exchange the `world` handles (any transport);  rt_peer_connect(g, handles)
 *   per step  : rt_peer_begin(g, stream)          waits until rank 0 has consumed the previous step, clears the accumulator
 *               rt_render_device(scene, cfg | RT_RENDER_NO_WAIT, rt_peer_accum(g), stream, stats)
 *               rt_peer_publish(g, stream)
 *   rank 0    : rt_peer_gather_resolve(g, d_screen, W, H, spp, rows, stream)     Screen-layout doubles in device memory
 * Waits are bounded (~2 s): rt_peer_timed_out(g) != 0 afterwards means a peer never published.  [ref: the mpsc gather of
 * src/world.rs:1228-1240] */
#ifndef RTB_PREFIX_ORC
#define RT_PEER_HANDLE_BYTES 64
typedef struct rt_peer_group rt_peer_group;
RTB_EXPORT rt_peer_group* rt_peer_create(int32_t rank, int32_t world, int64_t n_elems, uint8_t out_handle[RT_PEER_HANDLE_BYTES]);
RTB_EXPORT int32_t rt_peer_connect(rt_peer_group* g, const uint8_t* all_handles /* world x RT_PEER_HANDLE_BYTES */);
RTB_EXPORT int64_t* rt_peer_accum(rt_peer_group* g);
RTB_EXPORT int32_t rt_peer_begin(rt_peer_group* g, void* cuda_stream);
RTB_EXPORT int32_t rt_peer_publish(rt_peer_group* g, void* cuda_stream);
RTB_EXPORT int32_t rt_peer_gather_resolve(rt_peer_group* g, double* d_screen, int32_t width, int32_t height,
                                          int32_t samples_per_pixel, int32_t rendered_rows, void* cuda_stream);
RTB_EXPORT int32_t rt_peer_timed_out(rt_peer_group* g);
RTB_EXPORT void rt_peer_destroy(rt_peer_group* g);
#endif

/* render_scene_with_time(t0, t1, path, world): the per-frame animation entry.  cfg == NULL uses the
 * reference's hard-coded frame settings: 500x500 (aspect 1.0), 500 spp, depth 50, camera
 * (13,2,3)->(0,0,0), vfov 20, aperture 0.1, focus 10, background (0.7,0.8,1), THREADS = 11 row bands
 * (so rows 495..499 stay black).  With cfg != NULL the image size / spp / depth / compat_threads / seed
 * come from cfg and the camera aspect is cfg->aspect_ratio.  The shutter [t0, t1) is set on the scene's
 * camera, the scene is re-committed (moving bounds and GravitySphere windows follow the shutter), rendered
 * and written as P3 to `path` (path NULL: no file).  out_screen may be NULL.
 *                                   [ref: src/world.rs:1249-1330] */
RTB_EXPORT int32_t RTB_FN(render_scene_with_time)(rt_scene* s, double t0, double t1, const char* path,
                                                  const rt_render_config* cfg, double* out_screen,
                                                  rt_stats* stats);

/* Screen::write_to_ppm (path NULL => stdout) / write_to_ppm_file: byte-identical P3
 *                                   [ref: src/screen.rs:40-59] */
RTB_EXPORT int32_t RTB_FN(write_ppm)(const char* path_or_null, const double* screen,
                                     int32_t width, int32_t height);

/* ---------------------------------------------------------------- parity hook */
typedef struct rt_ray {
    double o[3];
    double d[3]; /* NOT normalised; t is in units of |d| */
    double time;
} rt_ray;

typedef struct rt_hit {
    int32_t prim_id;    /* depth-first index of the leaf Hittable that produced the record; -1 = miss */
    int32_t mat_id;     /* material id (builder order) */
    double t;
    double p[3];
    double normal[3];
    double u, v;
    int32_t front_face;
    int32_t pad_;
} rt_hit;

#define RT_TRACE_SKIP_MEDIA 0   /* geometric query: ConstantMedium objects are ignored */
#define RT_TRACE_SEEDED_MEDIA 1 /* media sampled from the Philox sub-stream keyed (seed, ray index) */

/* world.hit(ray, t_min, t_max) for n caller-supplied rays   [ref: src/world.rs:68, hit.rs:82-83] */
RTB_EXPORT int32_t RTB_FN(trace_batch)(rt_scene* s, const rt_ray* rays, int64_t n, double t_min,
                                       double t_max, int32_t flags, uint64_t seed, rt_hit* out);

#ifndef RTB_PREFIX_ORC
/* ---------------------------------------------------------------- binary I/O fast paths (product only; SURVEY.md 8(f) n2)
 * The reference writes P3 text (src/screen.rs:40-59) and reads ASCII PLY / P3 (src/model.rs:13-62, screen.rs:61-95);
 * those stay byte / parse compatible above.  At 10^6 pixels and 0.87 M faces the text formats are the slowest part
 * of a run, so: rt_write_ppm_binary writes the same Screen as P6; rt_ply_load and rt_tex_image_ppm accept
 * "format binary_little_endian 1.0" PLY (vertex = three leading float/double properties, triangle faces) and P6
 * files, chosen by the file's own header; rt_write_ply_binary / rt_ply_convert_binary produce such PLY files. */
RTB_EXPORT int32_t rt_write_ppm_binary(const char* path_or_null, const double* screen, int32_t width, int32_t height);
RTB_EXPORT int32_t rt_write_ply_binary(const char* path, const double* verts, int64_t nv, const uint32_t* idx, int64_t nt);
RTB_EXPORT int32_t rt_ply_convert_binary(const char* ascii_path, const char* binary_path);

/* ---------------------------------------------------------------- diagnostics (product only)
 * rt_unit_op evaluates one device function on the GPU for unit-level parity checks (SURVEY.md
 * Appendix E3): op 0 Texture::value, 1 Perlin::noise/turbulence, 2 Philox block, 3 camera ray.
 * rt_scene_set_tuning sets the number of resident path slots of the wavefront (0 = keep). */
RTB_EXPORT int32_t rt_unit_op(rt_scene* s, int32_t op, uint32_t ia, uint32_t ib, uint32_t ic,
                              uint32_t id, const double* in8, double* out8);
RTB_EXPORT int32_t rt_scene_set_tuning(rt_scene* s, uint32_t wave_slots);
/* Which builder rt_scene_commit uses in place of BvhNode::new   [ref: src/bvh.rs:14-83; SURVEY.md 8(f) n1].
 * RT_BVH_HOST_SAH (default): binned SAH on the host, best trees.  RT_BVH_DEVICE_LBVH: instances of >= 4096
 * primitives are built on the GPU (Morton sort + Karras hierarchy, csrc/cuda/lbvh.cu): ~100x faster commit of
 * large meshes, trees that cost more boxes per ray.  Results are identical (closest hit is topology independent). */
#define RT_BVH_HOST_SAH 0
#define RT_BVH_DEVICE_LBVH 1
RTB_EXPORT int32_t rt_scene_set_bvh_builder(rt_scene* s, int32_t builder);
/* Branching factor of the tree the kernels walk   [ref: src/bvh.rs:97-112, the binary BvhNode::hit].
 * 2: sibling pairs.  4: rt_scene_commit also collapses the trees of the main world's instances into 128-byte 4-wide nodes
 * (csrc/host/bvh_wide.hpp); the kernels that have a 4-wide form walk those, the others ignore it.
 * 0 (default): 4 where it measured faster - one wrapper-free instance without media that holds only spheres of any kind
 * (Sphere, MovingSphere, GravitySphere) or a mesh of >= 4096 triangles (fused kernels), and scenes whose media all have a
 * single-sphere / single-box boundary over spheres, moving spheres, rects and boxes (wavefront kernels) - else 2.
 * Results are identical (closest hit is topology independent). */
RTB_EXPORT int32_t rt_scene_set_bvh_width(rt_scene* s, int32_t width);
/* 4 if the last rt_scene_commit built the 4-wide collapse (the fused kernels then walk it), else 2; < 0 if not committed. */
RTB_EXPORT int32_t rt_scene_bvh_width(rt_scene* s);
/* Host-only self check of the flattener and BVH builder (needs no GPU): out[0] nodes, [1] max depth,
 * [2] main instances, [3] instances, [4] media, [5..10] primitives per rt_prim_type, [11] leaves,
 * [12] invariant violations (0 = valid), [13] numbered prims, [14] bytes the last commit uploaded,
 * [15] primitives whose BVH the last commit built on the device. */
RTB_EXPORT int32_t rt_scene_host_check(rt_scene* s, int64_t out[16]);
/* Test hook (needs no GPU, computes nothing): runs the host half of rt_scene_commit and writes one DeviceScene
 * (csrc/rt_types.h; out_bytes must equal its size) whose pointers address the flattened HOST arrays, valid until the
 * next call or rt_scene_destroy.  tests/host_emul compiles csrc/cuda/rt_device.cuh for the host against it, so the
 * device functions themselves are checked against the oracle on machines without a GPU.  Never used by a render. */
RTB_EXPORT int32_t rt_debug_host_scene(rt_scene* s, void* out_scene, uint64_t out_bytes);
#endif

#ifdef __cplusplus
}
#endif
#endif /* RTB200_H */
