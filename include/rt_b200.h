/*
 * rt_b200.h -- C ABI of librt_b200.so, the B200 (sm_100a) implementation of the
 * traditional sphere ray-tracing inner loop of JoaquinRodriguezph/ray-tracer-v1.
 *
 * The reference is pure Python and has NO FFI/plugin boundary (SURVEY.md 8b): its
 * callers build Python objects and call Ray.nearestSphereIntersect /
 * Intersection.terminalRGB / TraditionalRenderer.render / RayTracerEnv.step
 * directly.  This header is the boundary a maintainer would bind underneath
 * those methods (ctypes stub shown in INTEGRATION.md); each entry cites the
 * reference interface it replaces (path:line relative to the reference root).
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++/torch types.  Every function returns an
 *     int status (RT_OK == 0); rt_last_error() gives the message of the last
 *     failure on the calling thread.
 *   - "_dev" pointers are device pointers on the handle's GPU, everything else is
 *     host memory.  `stream` is a cudaStream_t passed as void* (NULL = default
 *     stream).  Calls are asynchronous on that stream unless stated otherwise.
 *   - precision: RT_F32 = the FP32 product path; RT_F64 = the FP64 parity build
 *     (same algorithms in double, compiled without FMA contraction, following the
 *     reference's operation order; <= 1e-9 relative parity, north_star).
 *   - no hidden global state: one rt_scene handle per GPU / rank.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { RT_OK = 0, RT_ERR_INVALID = 1, RT_ERR_CUDA = 2, RT_ERR_NOMEM = 3, RT_ERR_UNSUPPORTED = 4 };
enum { RT_F32 = 0, RT_F64 = 1 };
/* RayTracerEnv info['reason'] codes (RL/ray_tracer_env.py:316-397, FB/ray_tracer_env.py:393-507) */
enum { RT_REASON_NONE = 0, RT_REASON_RAY_MISSED = 1, RT_REASON_RAY_ESCAPED = 2, RT_REASON_MAX_BOUNCES = 3,
       RT_REASON_HIT_SUN = 4, RT_REASON_ALREADY_ON_SUN = 5 };
enum { RT_ENV_RL = 0, RT_ENV_FB = 1 };
#define RT_NO_ID INT32_MIN  /* "no suppressed id" */

typedef struct rt_scene rt_scene; /* flattened scene resident in HBM (both precisions) */
typedef struct rt_env rt_env;     /* SoA state of a batch of RayTracerEnv episodes */

/* ---- scene graph, flattened (replaces list[Sphere] + light lists: object.py:4-9,
 *      material.py:4-8, light.py:12-37; TraditionalRenderer.scene/.light_sources/.small_lights,
 *      FB/fb_vs_traditional_chandelier.py:394-403).  All arrays row-major, host memory. */
typedef struct rt_scene_desc {
    int32_t n;               /* spheres */
    const double *centre;    /* [n,3] */
    const double *radius;    /* [n]   */
    const double *material;  /* [n,4] reflective, transparent, emitive, refractive_index */
    const double *colour;    /* [n,3] 0-255 scale */
    const int32_t *ids;      /* [n]   Sphere.id */
    int32_t nG;              /* GlobalLight */
    const double *g_vec;     /* [nG,3] */
    const double *g_col;     /* [nG,3] */
    const double *g_strength;
    const double *g_max_angle;
    const int32_t *g_func;
    int32_t nP;              /* PointLight */
    const int32_t *p_id;
    const double *p_pos;     /* [nP,3] */
    const double *p_col;     /* [nP,3] */
    const double *p_strength;
    const double *p_max_angle;
    const int32_t *p_func;   /* -1 no fall-off, 0 divide by distance */
    double bg[3];            /* background_colour */
    int32_t nL;              /* Algorithm B light spheres */
    const double *l_centre;  /* [nL,3] */
    const double *l_colour;  /* [nL,3] */
    const int32_t *l_index;  /* [nL] scene index of the light sphere or -1 */
    const uint8_t *small;    /* [n] member of small_lights (may be NULL) */
} rt_scene_desc;

/* ---- library / device ------------------------------------------------------------ */
const char *rt_last_error(void);
int rt_version(void);
int rt_device_count(int *count);
/* props[0..5] = SM count, cc major, cc minor, max SM clock kHz, L2 bytes, max smem/block (opt-in) */
int rt_device_props(int device, int64_t *props6, size_t *total_mem);
int rt_dev_alloc(int device, size_t bytes, void **out_dev);
int rt_dev_free(int device, void *ptr_dev);
int rt_host_alloc_pinned(size_t bytes, void **out_host);
int rt_host_free_pinned(void *ptr_host);
int rt_memcpy_h2d(int device, void *dst_dev, const void *src_host, size_t bytes, void *stream);
int rt_memcpy_d2h(int device, void *dst_host, const void *src_dev, size_t bytes, void *stream);
int rt_memset_dev(int device, void *dst_dev, int value, size_t bytes, void *stream);
int rt_stream_sync(int device, void *stream);
/* a non-blocking stream (e.g. for copies that overlap the next kernel); rt_stream_wait_stream: everything enqueued on
 * `waiter` after the call runs after everything enqueued on `waited` before it (NULL = the default stream). */
int rt_stream_create(int device, void **out_stream);
int rt_stream_destroy(int device, void *stream);
int rt_stream_wait_stream(int device, void *waiter, void *waited);
/* FP32 roofline denominator: dependent-free FFMA loop on every SM, timed with CUDA events (synchronous). */
int rt_measure_fp32_peak(int device, int repeats, double *tflops_out, double *ms_out);

/* ---- scene ------------------------------------------------------------------------ */
int rt_scene_create(int device, const rt_scene_desc *desc, rt_scene **out);
int rt_scene_update(rt_scene *scene, const rt_scene_desc *desc, void *stream); /* re-flatten a mutated scene */
int rt_scene_destroy(rt_scene *scene);
int rt_scene_info(const rt_scene *scene, int32_t *n_spheres, int32_t *device, int32_t *has_lbvh);
/* On-device LBVH (Morton codes -> radix sort -> Karras hierarchy -> AABB refit) over the spheres; spheres whose
 * radius exceeds `huge_radius` (walls) stay in a brute-force side list.  Renders use it when present. */
int rt_lbvh_build(rt_scene *scene, double huge_radius, void *stream);
int rt_lbvh_drop(rt_scene *scene);

/* ---- batched primitives (replace Ray.sphereDiscriminant ray.py:73-107, Ray.nearestSphereIntersect
 *      ray.py:160-231, Intersection.terminalRGB ray.py:37-65) ------------------------------------ */
/* m independent ray/sphere pairs.  rays [m,6] origin+raw direction, spheres [m,4] centre+radius (double, device).
 * out [m,8] = hit, t, point(3), normal(3). */
int rt_sphere_discriminant(int device, int precision, int m, const double *rays_dev, const double *spheres_dev,
                           int point, double *out_dev, void *stream);
/* m rays through nearestSphereIntersect (+ terminalRGB when rgb_dev != NULL).
 * suppress_dev [m] Sphere.id to suppress or RT_NO_ID (NULL = none); bounces0_dev [m] initial `bounces` (NULL = 0);
 * through0_dev [m] initial through_count (NULL = 0).
 * term_dev [m,11] = hit, scene index, bounces, through_count, point(3), normal(3), distance (Intersection.distance of
 * the terminal hit, signed); rgb_dev [m,3] (miss -> miss[3]). */
int rt_trace_rays(rt_scene *scene, int precision, int m, const double *rays_dev, const int32_t *suppress_dev,
                  const int32_t *bounces0_dev, const int32_t *through0_dev, int max_bounces, int shadow_max_bounces,
                  const double miss[3], double *term_dev, double *rgb_dev, void *stream);

/* Intersection.terminalRGB (ray.py:37-65) at m given hits.  hits_dev [m,7] = scene index, point(3), normal(3) (double);
 * rgb_dev [m,3] = background + illuminate(...).  shadow_max_bounces = terminalRGB's max_bounces argument. */
int rt_terminal_rgb(rt_scene *scene, int precision, int m, const double *hits_dev, int shadow_max_bounces,
                    double *rgb_dev, void *stream);

/* ---- Algorithm A frame: deterministic Whitted-style trace + terminalRGB (drivers: RL/output5.py:416-533
 *      render_true_original, :1420-1525 render_custom_scene('traditional'), notebooks' cell-0 loops) ---------- */
typedef struct rt_whitted_params {
    double cam[3];          /* ray origin */
    const double *X;        /* [W] host: x component of direction (X, Y, -1)  */
    const double *Y;        /* [H] host */
    int32_t W, H;
    int32_t y0, y1;         /* row band [y0,y1) rendered by this call (tile sharding) */
    int32_t s0, s1;         /* sample range [s0,s1) accumulated by this call (sample sharding) */
    int32_t spp;            /* total samples per pixel of the frame; jitter iff spp > 1 (output5.py:1463-1470) */
    int32_t max_bounces;
    int32_t shadow_max_bounces; /* terminalRGB(max_bounces=...) default 0 */
    double miss[3];         /* colour of a ray that terminates nowhere */
    uint64_t seed;          /* Philox key */
    int32_t prenormalise;   /* output5.py:1476-1483 normalises before Ray() normalises again */
    int32_t accumulate;     /* 0: overwrite accum rows [y0,y1); 1: add into them */
} rt_whitted_params;
/* accum_dev: [H,W,4] float (RT_F32) or double (RT_F64): sum r,g,b over the sample range + sample count.
 * hit_dev (optional) [H,W] int32 terminal scene index of the last sample (-1 miss).
 * stats_dev (optional) uint64[8]: [0] primary rays, [4] nearest-hit/occlusion queries traced, [5] sphere tests,
 * [6] AABB tests (LBVH only), [7] continuation queries NOT traced: behind a mirror / through glass with the bounce
 * limit already spent the reference still casts the ray and discards what it finds (ray.py:170-174), so
 * [4] + [7] = the reference's own query count.
 * X / Y are HOST arrays; the scene keeps their device copies resident (keyed by value), so only the first frame with
 * a given grid uploads it (asynchronously, from a pinned copy) and later frames are a pure stream-ordered kernel
 * launch: no copy, no synchronisation, graph-capturable, and safe from any number of streams.  A handle is not
 * thread-safe: serialise host calls on one rt_scene. */
int rt_render_whitted(rt_scene *scene, int precision, const rt_whitted_params *p, void *accum_dev, int32_t *hit_dev,
                      uint64_t *stats_dev, void *stream);

/* ---- Algorithm B frame: TraditionalRenderer.render / trace_ray_traditional
 *      (FB/fb_vs_traditional_chandelier.py:417-554, FB/fb_vs_traditional_complex.py:285-422) ------------------ */
typedef struct rt_path_params {
    double cam[3];
    int32_t W, H;
    double fov_deg;         /* 60 in the reference (:415) */
    int32_t y0, y1;         /* row band */
    int32_t s0, s1;         /* sample range */
    int32_t max_bounces;
    double mirror_threshold;/* material.reflective > threshold mirrors: 0.9 complex (:349), 0 chandelier (:481) */
    uint64_t seed;
    int32_t accumulate;
    int32_t schedule;       /* 0 = default.  Bit 1 (value 2): diagnostic, switch off the camera-ray candidate lists of
                               the FP32 parameter-block kernel (same image); bit 2 (value 4): diagnostic, small scenes
                               use the shared-memory sphere loop instead of the parameter-block one, which changes the
                               selection key (3 instead of 6 index bits), i.e. near-ties of the FP32 build.  Any other
                               bit (bit 0 included) is rejected with RT_ERR_INVALID */
    int32_t ksplit;         /* lanes sharing one pixel's samples: -1 = automatic (keeps >= 64 waves of CTAs in the grid),
                               0 or 1 = one thread per pixel, 2..32 = that power of two.  Same image either way. */
    int32_t reserved_;
} rt_path_params;
/* accum_dev as above.  stats_dev (optional) uint64[8]: [0] total_rays (trace calls, reference-compatible),
 * [1] total_intersections, [2] light_hits, [3] small_light_hits, [4] nearest-hit queries,
 * [5] sphere tests, [6] AABB tests (LBVH only). */
int rt_render_path(rt_scene *scene, int precision, const rt_path_params *p, void *accum_dev, uint64_t *stats_dev,
                   void *stream);
/* TraditionalRenderer.trace_ray_traditional(ray, bounce_count) (FB/fb_vs_traditional_chandelier.py:431-521) for n
 * explicit rays at once: rays_dev [n,6] doubles = origin, direction AS GIVEN (Ray() has normalised it); the path starts
 * at recursion depth bounce_count (a call with bounce_count >= max_bounces returns (2,2,5)); ray i draws its bounce
 * directions from the Philox stream of pixel ray_ids_dev[i] (NULL: i) and sample s, so a camera ray generated on the
 * host reproduces the frame's sample exactly.  accum_dev [n,4] as rt_render_path (sum over samples [s0,s1) + count).
 * p->cam / W / H / fov / y0 / y1 are ignored. */
int rt_trace_paths(rt_scene *scene, int precision, const rt_path_params *p, int32_t n, const double *rays_dev,
                   const int32_t *ray_ids_dev, int32_t bounce_count, void *accum_dev, uint64_t *stats_dev, void *stream);

/* accum [H,W,4] -> image [H,W,3] float32 = min(1, floor(sum/spp)/255) (chandelier.py:540-549; output5.py:1500-1512).
 * rows [y0,y1) only. */
int rt_resolve(int device, int precision, const void *accum_dev, int32_t W, int32_t H, int32_t y0, int32_t y1,
               int32_t spp, float *image_dev, void *stream);

/* ---- "Algorithm C" frame: SimplifiedFBRenderer.render_original_style / trace_ray_simple /
 *      calculate_lighting_exact_original in traditional mode (fb_usage_prob = 0): FB/output6.py:197-306, :434-654.
 *      Per-bounce lighting (global 0.3 cos + shadowed sun, int() truncations) accumulated with min(255, .), mirrors
 *      for a truthy `reflective`, glass 50/50 reflect / straight, cosine-weighted diffuse bounces, stop on the sun id. */
typedef struct rt_simple_params {
    double cam[3];           /* Vector(0, 0, 1), output6.py:605 */
    int32_t W, H;            /* camera grid; ignored when rays_dev != NULL */
    double fov_rad;          /* np.pi / 3, output6.py:622 */
    double sun_pos[3];       /* self.sun_position */
    double sun_col[3];       /* self.sun_color */
    int32_t sun_id;          /* 7 */
    int32_t max_bounces;     /* self.max_bounces = 5 */
    uint64_t seed;           /* Philox key; slot bounce+1 of (pixel, sample 0): glass draws word 0, diffuse words 0,1 */
    int32_t m;               /* number of explicit rays when rays_dev != NULL */
    int32_t lighting_only;   /* != 0: rays_dev holds m INTERSECTIONS [m,7] = point, normal, scene index of the sphere;
                              * rgb = calculate_lighting_exact_original(intersection) (output6.py:197-306), nothing is
                              * traced but the sun's shadow test; rgb[.,3] = 0 */
    const double *rays_dev;  /* optional [m,6] origin + raw direction (scalar trace_ray_simple = a batch of one) */
} rt_simple_params;
/* rgb_dev [n,4] int32 = accumulated r, g, b, bounce_count (n = W*H or m); image_dev (optional) [n,3] float32 =
 * min(1, c/255) (output6.py:628-632).  stats_dev (optional) uint64[8]: [0] total_rays, [1] sun_hits, [4] queries
 * (nearest-hit + shadow tests). */
int rt_render_simple(rt_scene *scene, int precision, const rt_simple_params *p, int32_t *rgb_dev, float *image_dev,
                     uint64_t *stats_dev, void *stream);
/* host buffers; rays_host ([m,6], or [m,7] with p->lighting_only) replaces p->rays_dev when not NULL.  Synchronous. */
int rt_render_simple_host(rt_scene *scene, int precision, const rt_simple_params *p, const double *rays_host,
                          int32_t *rgb_host, float *image_host, uint64_t *stats_host);

/* ---- FB training trajectories: RayTracedComplexTrainer.generate_trajectory + random_point_on_sphere /
 *      sample_cosine_weighted_direction / direction_to_action / create_observation / nearest_intersection
 *      (FB/train_complex_only.py:54-166, :254-334), n_traj random walks at once.  Trajectory j starts on a random
 *      non-emissive sphere; every step records (obs22, action2, next_obs22, reward, hit_light) until a light is hit,
 *      the ray escapes or max_steps transitions exist.  All outputs are device arrays padded to max_steps:
 *      obs/next_obs [n,max_steps,22] f32, action [n,max_steps,2] f32, reward [n,max_steps] f32, hit [n,max_steps] u8,
 *      length [n] int32 (transitions recorded), hit_light [n] u8 (obs / next_obs 8-byte aligned).  stats_dev
 *      (optional) uint64[8]: [4] queries. */
int rt_generate_trajectories(rt_scene *scene, int precision, int32_t n_traj, int32_t max_steps, int32_t max_bounces,
                             uint64_t seed, float *obs_dev, float *action_dev, float *next_obs_dev, float *reward_dev,
                             uint8_t *hit_dev, int32_t *length_dev, uint8_t *hit_light_dev, uint64_t *stats_dev,
                             void *stream);

/* ---- Algorithm B as a wavefront, for learned direction sampling: WorkingFBRenderer.trace_ray_fb / render
 *      (FB/fb_vs_traditional_complex.py:487-640).  The reference calls fb_agent.choose_direction(obs22) per hit; here
 *      the kernels stop at exactly that point, the caller's policy (a torch module) maps the observations of the paths
 *      that ask to actions on the same stream, and the next kernel consumes them.  One frame (or a row band / sample
 *      range of it, P = W * (y1-y0) * (s1-s0) <= max_paths path slots):
 *          rt_wf_begin;  repeat max_bounces times { rt_wf_trace; actions[need] = policy(obs[need]); rt_wf_bounce };
 *          rt_wf_finish (adds the folded path colours and sample counts into accum [H,W,4]).
 *      fb_usage_prob = 0 reproduces rt_render_path bit for bit (FP64) with the same Philox streams. */
typedef struct rt_wavefront rt_wavefront;
int rt_wf_create(rt_scene *scene, int precision, int32_t max_paths, int32_t max_depth, rt_wavefront **out);
int rt_wf_destroy(rt_wavefront *wf);
int rt_wf_begin(rt_wavefront *wf, const rt_path_params *p, double fb_usage_prob, uint64_t *stats_dev, void *stream);
/* obs_dev [P,22] float32 (rows of asking paths are written), need_dev [P] uint8 (1 = wants an action).
 * stats_dev (optional) uint64[8] as rt_render_path plus [7] = fb_used. */
int rt_wf_trace(rt_wavefront *wf, float *obs_dev, uint8_t *need_dev, uint64_t *stats_dev, void *stream);
/* actions_dev [P,2] float32 in [-1,1]^2, read where need_dev is 1; live_dev (int32, zeroed by the caller) receives the
 * number of paths still alive. */
int rt_wf_bounce(rt_wavefront *wf, const uint8_t *need_dev, const float *actions_dev, uint64_t *stats_dev, int32_t *live_dev,
                 void *stream);
int rt_wf_finish(rt_wavefront *wf, void *accum_dev, void *stream);

/* ---- fused multi-GPU sinks for Algorithm B frames (SURVEY.md 8e) ---------------------------------------------
 * One process per GPU; a rank's path kernel stores its result where it is needed -- its own accumulators, the
 * final image on the collecting rank, or the accumulators of the rank that owns the pixel -- through NVLink peer
 * mappings, so the tile gather / sample reduce is the render kernel's own epilogue instead of a second pass.
 *
 *   RT_SINK_ACCUM        accum_dev of rt_render_path (no sink).
 *   RT_SINK_IMAGE        tile sharding.  The launch covers the 8-row tiles tile_first, tile_first + tile_step, ...
 *                        (interleaved stripes: load balance with no contiguity constraint), all spp samples, and
 *                        stores min(1, floor(sum/spp)/255) as float32 [H,W,3] straight into `image` (local or a peer
 *                        mapping of the collecting rank's image).
 *   RT_SINK_SCATTER_ADD  sample sharding.  The launch covers every pixel for its sample range and adds
 *                        (r, g, b, samples) with one 16-byte system-scope reduction per pixel into accum[k], k = the
 *                        rank whose row band [band_y[k], band_y[k+1]) holds the pixel (reduce-scatter by direct
 *                        NVLink atomics; integer-valued FP32 sums < 2^24 are exact and order-independent).
 *                        Needs integer colours (every scene of the reference); RT_ERR_UNSUPPORTED otherwise.
 * Cross-rank ordering uses epoch flags in peer memory: rt_peer_signal after the writes, rt_peer_wait before the
 * reads (stream-ordered, system-scope release/acquire). */
enum { RT_SINK_ACCUM = 0, RT_SINK_IMAGE = 1, RT_SINK_SCATTER_ADD = 2 };
#define RT_MAX_PEERS 16
#define RT_IPC_HANDLE_BYTES 64
typedef struct rt_path_sink {
    int32_t mode;
    int32_t world;                    /* ranks (SCATTER_ADD; with sync: both modes) */
    int32_t tile_first, tile_step;    /* IMAGE: 8-row tiles rendered by this launch */
    float *image;                     /* IMAGE: [H,W,3] float32, device or peer pointer (with sync: both modes, = the
                                         collecting rank's image) */
    void *accum[RT_MAX_PEERS];        /* SCATTER_ADD: per-owner [H,W,4] float32 accumulators (zeroed by the owner) */
    int32_t band_y[RT_MAX_PEERS + 1]; /* SCATTER_ADD: owner row bands */
    /* ---- sync = 1: the WHOLE frame protocol runs inside this one launch (one kernel per rank and frame; see below) */
    int32_t sync;
    int32_t rank;                     /* this rank; rank 0 collects the image */
    uint32_t epoch;                   /* frame number, starting at 1, the same on every rank */
    uint32_t go_epoch;                /* rank 0: publish "frames <= go_epoch are consumed" to every rank at kernel start
                                         (everything queued on this stream before the launch has finished by then);
                                         0 = nothing to publish (e.g. the consumer signals from another stream) */
    uint32_t *flags[RT_MAX_PEERS];    /* flag block of every rank (own block at [rank], peer mappings elsewhere):
                                         RT_FLAG_WORDS uint32, zero-initialised: [r] added, [16 + r] done, [32] go */
    int32_t *timed_out;               /* device int32 (optional): set to 1 if a flag wait gives up */
    int32_t timeout_ms;               /* <= 0: 20 s */
    int32_t max_ctas;                 /* 0 = as many CTAs as the device keeps resident; smaller values let several
                                         "ranks" share ONE device (tests) */
    int32_t spp_total;                /* sync + SCATTER_ADD: samples per pixel of the whole frame (the band resolve
                                         divides by it; p->s0/s1 is only this rank's range) */
    int32_t col_split;                /* IMAGE, != 0: 2-D interleave instead of whole stripes -- the launch covers in EVERY
                                         8-row stripe s the column segment (tile_first + s) mod tile_step of tile_step
                                         equal segments (W a multiple of tile_step).  Every rank then holds the same
                                         number of pixels whatever H is (1080 rows are 135 stripes: 17 or 16 per rank of
                                         8), and a diagonal share of the picture.  A segment must hold whole work units
                                         (8 pixels wide for launches of >= 64 samples, up to 32 for short ones): if it
                                         does not, the launch renders whole stripes as without col_split -- every rank
                                         of a frame decides the same from the same W, H, samples and tile_step */
} rt_path_sink;
#define RT_FLAG_WORDS 64
/* sync = 1 -- one launch per rank and frame, no other kernel and no host round trip on the data path:
 *   start    every CTA waits (acquire) until go >= epoch - 2: the image / accumulator buffers of this parity are free
 *   render   as above: IMAGE stores resolved pixels into rank 0's image, SCATTER_ADD adds sums into the owners' bands
 *   publish  the last warp of the launch to finish (system fence, release store): IMAGE sets done[rank] on rank 0;
 *            SCATTER_ADD sets added[rank] on every rank
 *   resolve  SCATTER_ADD only: once added[0..world) have all reached the epoch, the CTAs of the launch resolve the own
 *            band [band_y[rank], band_y[rank+1]) of accum[rank] into rank 0's image, clear it for frame epoch + 2,
 *            and the last CTA sets done[rank] on rank 0
 *   collect  rank 0 only: the launch ends after done[0..world) have reached the epoch, i.e. kernel completion = frame
 *            complete in `image`.
 * The launches of all ranks must be able to run concurrently (one per GPU; tests: max_ctas).  When several ranks share
 * ONE device (tests), a launch that waits on a flag must be issued after the launch that sets it: streams of a process
 * share hardware queues, and a kernel issued later can be held behind a spinning one. */
/* FP32 product path only.  p->y0/y1 are ignored for RT_SINK_IMAGE (the tiles say which rows); p->s0/s1 must be the
 * full [0, spp) range there. */
int rt_render_path_sink(rt_scene *scene, const rt_path_params *p, const rt_path_sink *sink, uint64_t *stats_dev,
                        void *stream);
/* resolve rows [y0,y1) of accum into image (device or peer pointer) and, when clear != 0, zero those accum rows for
 * the next frame. */
int rt_resolve_clear(int device, void *accum_dev, int32_t W, int32_t H, int32_t y0, int32_t y1, int32_t spp,
                     float *image_dev, int32_t clear, void *stream);

/* peer memory (CUDA IPC): rt_peer_alloc = cudaMalloc + zero + export; the handle travels to the other ranks by any
 * means (torch.distributed.all_gather_object), which open it with rt_peer_open. */
int rt_peer_alloc(int device, size_t bytes, void **out_dev, unsigned char handle[RT_IPC_HANDLE_BYTES]);
int rt_peer_open(int device, const unsigned char handle[RT_IPC_HANDLE_BYTES], void **out_dev);
int rt_peer_close(int device, void *ptr_dev);
int rt_peer_free(int device, void *ptr_dev);
/* store `epoch` (system-scope release, after a system fence) into n flag words, typically one per peer */
int rt_peer_signal(int device, uint32_t *const *flag_ptrs, int32_t n, uint32_t epoch, void *stream);
/* spin (system-scope acquire) until flags_dev[i] - epoch >= 0 for all i < n; gives up after timeout_ms and sets
 * *timed_out_dev (device int32, optional) to 1 */
int rt_peer_wait(int device, const uint32_t *flags_dev, int32_t n, uint32_t epoch, int32_t timeout_ms,
                 int32_t *timed_out_dev, void *stream);

/* Host-buffer convenience entries (what a ctypes/cffi binding of the reference's render() calls): upload nothing
 * but the parameters, render, resolve, copy the float32 [H,W,3] image (and optionally the raw sums [H,W,4] in the
 * accum type, and stats) back to HOST memory.  Synchronous. */
int rt_render_whitted_host(rt_scene *scene, int precision, const rt_whitted_params *p, float *image_host,
                           void *accum_host, int32_t *hit_host, uint64_t *stats_host);
int rt_render_path_host(rt_scene *scene, int precision, const rt_path_params *p, float *image_host, void *accum_host,
                        uint64_t *stats_host);

/* ---- batched RayTracerEnv (RL/ray_tracer_env.py:21-425, FB/ray_tracer_env.py:21-538) ------------------------ */
typedef struct rt_env_desc {
    int32_t B;              /* parallel episodes */
    int32_t W, H;           /* image_width / image_height */
    double cam[3];          /* camera_position */
    double cam_angle[3];    /* camera_angle (Euler, vector.py:117-127) */
    double fov;             /* degrees */
    int32_t max_bounces;
    int32_t flavour;        /* RT_ENV_RL | RT_ENV_FB */
    int32_t sun_id;         /* FB flavour: 7 (FB/ray_tracer_env.py:256) */
    int32_t reward_mode;    /* RL flavour: 0 = RayTracerEnv._calculate_reward, 1 = AdaptiveRewardRayTracerEnv
                               (RL/train_raytracer_optimized.py:25-61: light / mirror bonuses, short-path penalty) */
    int32_t light_ids[2];   /* reward_mode 1: self.light_ids = [99, 100] (:21) */
    int32_t env_offset;     /* env-sharded rollouts: global index of this batch's first env.  Device-drawn start pixels
                               are keyed by the GLOBAL env index, so a shard equals the same rows of the unsharded batch */
    int32_t reserved_;
} rt_env_desc;
int rt_env_create(rt_scene *scene, int precision, const rt_env_desc *desc, rt_env **out);
int rt_env_destroy(rt_env *env);
/* reset(): pixels_dev [B,2] int32 (x,y) or NULL = draw uniformly with Philox(seed) on device.
 * mask_dev (optional) [B] uint8: reset only envs with mask != 0 (auto-reset of finished episodes).
 * obs_dev [B,18] float32.  pixels_out_dev (optional) [B,2] receives the pixels used. */
int rt_env_reset(rt_env *env, const int32_t *pixels_dev, const uint8_t *mask_dev, uint64_t seed, float *obs_dev,
                 int32_t *pixels_out_dev, void *stream);
/* step(): actions_dev [B,2] float32 -> obs [B,18] f32, reward [B] f64, terminated/truncated [B] u8,
 * reason [B] int32 (RT_REASON_*), info_dev (optional) [B,4] f64 = bounce_count, through_count, total_reward,
 * hit_sun.  stats_dev (optional) uint64[8]: [4] nearest-hit/occlusion queries traced, [7] discarded continuation
 * queries not traced (see rt_render_whitted).  The RL flavour shades every hit once, when it is made, and keeps the
 * colour with the episode for the next step's reward (the reference shades the same point again one step later). */
int rt_env_step(rt_env *env, const float *actions_dev, float *obs_dev, double *reward_dev, uint8_t *terminated_dev,
                uint8_t *truncated_dev, int32_t *reason_dev, double *info_dev, uint64_t *stats_dev, void *stream);
/* step() with the restart of finished episodes IN THE SAME LAUNCH (the VecEnv protocol of Stable-Baselines3, which the
 * reference trains through: RL/train_raytracer.py:128-147): an env whose episode ends in this step gets its last
 * observation written to final_obs_dev (optional, [B,18] float32, rows of finished envs only) and is reset at once --
 * start pixel = Philox(env index, episode number) under `seed`, written to pixels_out_dev (optional, [B,2]) -- so
 * obs_dev holds the FIRST observation of the new episode while reward / terminated / truncated / reason / info
 * describe the step that ended the old one.  reward_dev [B] and info_dev (optional) [B,4] are float for an RT_F32 env
 * and double for an RT_F64 env.  One launch per step, no host round trip, graph-capturable (nothing in the parameter
 * block changes from step to step). */
int rt_env_step_auto(rt_env *env, const float *actions_dev, float *obs_dev, void *reward_dev, uint8_t *terminated_dev,
                     uint8_t *truncated_dev, int32_t *reason_dev, void *info_dev, float *final_obs_dev,
                     int32_t *pixels_out_dev, uint64_t seed, uint64_t *stats_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
