// rt_launch.h -- kernel parameter blocks and launcher declarations shared by the two kernel translation units
// (rt_f32.cu: float, FMA-contracted; rt_f64.cu: double, -fmad=false) and the C-ABI layer (rt_api.cu).
#pragma once
#include <cfloat>
#include "rt_common.cuh"

namespace rt {

// Algorithm A frame (rt_whitted_params, include/rt_b200.h)
template <typename T> struct WhittedDev {
    T cam[3];
    const T *X, *Y;              // device copies of the direction grids
    int W, H, y0, y1, s0, s1, spp, max_bounces, shadow_max_bounces;
    T miss[3];
    T pitch_x, pitch_y;          // X[1]-X[0], Y[0]-Y[1] (output5.py:1465-1466)
    uint32_t k0, k1;             // Philox key
    int prenorm, accumulate;
    int gx, gy;                  // 32x8-pixel block grid of the launch (set by launch_whitted)
    unsigned *sched;             // {next warp tile, warps done, heavy tiles, -}: zero between launches (self-resetting)
    // two-pass frames (FP32, small scenes, >= 4 samples): pass 1 fills the sky tiles and LISTS the tiles whose cone of
    // camera rays can touch a sphere; pass 2 spreads (listed tile, sample) units over all warps of the device
    int split;
    unsigned *heavy;             // [gx * gy * 8] warp-tile indices listed by pass 1
    unsigned *sched2;            // pass 2: {next unit, warps done}
};

// Path-kernel work unit with 2^lk lanes per pixel: one warp traces a 2^pw x 2^ph pixel block, pw = unit_pw_log2(lk) and
// ph = (5 - lk) - pw (8x4, 8x2, 4x2, 2x2, 2x1, 1x1 for lk = 0..5), and a CTA of 4 x 2 warps a (4 << pw) x (2 << ph) one
__host__ __device__ constexpr int unit_pw_log2(int lk) { return lk == 0 ? 3 : lk == 1 ? 3 : lk == 2 ? 2 : lk <= 4 ? 1 : 0; }

// Algorithm B frame (rt_path_params).  The launch geometry -- ksplit_log2, ksplit2_log2, the tile grids, the band
// (y0, tile_step, col_*, seg_w) and fold_tab -- is set by plan_path_launch (rt_api.cu).
template <typename T> struct PathDev {
    T cam[3];
    int W, H, y0, y1, s0, s1, max_bounces;
    T aspect, half_w, half_h;    // W/H, tan(fov/2)*aspect, tan(fov/2)   (chandelier.py:412-415)
    T inv_W, inv_H;              // product build: 1/W, 1/H (the parity build divides like the reference)
    T mirror_threshold;
    int gx, gy;                          // tile grid of the launch
    // second ("fine") tile grid over the last owned stripes of the launch: same pixels-per-CTA logic with MORE lanes per
    // pixel (ksplit2_log2 > ksplit_log2), i.e. work units a quarter as long, handed out after the coarse ones so that
    // the drain at the end of the launch is a quarter as long (gx2 * gy2 = 0: none)
    int gx2, gy2, stripe2, ksplit2_log2;
    int depth0;                          // explicit rays (below); placed here because moving the fields after it by 8
                                         // bytes changes the instruction schedule ptxas picks for path_kernel
    unsigned *sched;                     // {next work unit, warps done}: zero between launches (self-resetting)
    uint32_t k0, k1;
    uint32_t rk[20];                     // Philox round keys k0 + r*W0, k1 + r*W1 (constant-bank operands of the rounds)
    int accumulate;
    int int_fold;                // every leaf colour is an integer in [0, 65535]: integer fold + uint32 accumulators
    int fold_tab;                // kMode 3, int_fold, every colour <= 255: the fold reads int(albedo * (tot / 255.0)) from a
                                 // per-CTA byte table [sphere][channel][tot] in dynamic shared memory (n * 768 bytes)
    int primary_cull;            // 1: camera rays use the warp tile's candidate list (FP32 kMode 3)
    // fused multi-GPU sinks (rt_path_sink, include/rt_b200.h); sink == 0: accum only
    int ksplit_log2;             // 2^ksplit_log2 lanes share a pixel and split its samples (integer fold only)
    int sink, tile_step, world, spp_total;
    int col_step, col_first, seg_w;      // 2-D interleave (rt_path_sink::col_split): col_step > 1: in stripe s this launch
                                         // covers columns [seg, seg + seg_w), seg = ((col_first + s) % col_step) * seg_w
    float *image;
    float4 *peer_accum[16];
    int band_y[17];
    // in-kernel frame protocol (rt_path_sink::sync): epoch flags in peer memory, see include/rt_b200.h
    int sync, rank;
    unsigned epoch, go_epoch;
    unsigned *flags[16];                 // [r] added, [16 + r] done, [32] go -- in every rank's flag block
    int *timed_out;
    long long timeout_cycles;
    int max_ctas;
    // explicit rays (rt_trace_paths: TraditionalRenderer.trace_ray_traditional(ray, bounce_count) for n rays at once):
    // ray i = (origin, direction as given -- Ray() has normalised it) starts at recursion depth depth0 and draws from
    // the Philox stream of pixel ray_ids[i] (or i).  W = n, H = 1.  Not available in the parameter-block kernel (kMode 3).
    const double *rays;
    const int *ray_ids;
};

// "Algorithm C" frame (rt_simple_params)
template <typename T> struct SimpleDev {
    T cam[3], tan_half, aspect, sun_pos[3], sun_col[3];
    int W, H, n, sun_id, max_bounces;
    uint32_t k0, k1;
    const double *rays;
    int lighting_only;                    // rays = [n,7] intersections (point, normal, scene index): lighting alone
};

// wavefront form of Algorithm B (rt_wavefront.cuh): SoA path state, one slot per (pixel, sample)
template <typename T> struct WaveDev {
    int P, max_depth;                     // path slots, stack depth
    int W, H, y0, y1, s0, s1, max_bounces;
    T cam[3], aspect, half_w, half_h, mirror_threshold, fb_prob;
    uint32_t k0, k1;
    T *O, *D, *hp, *hn;                   // [3][P] origin, direction, pending hit point / normal
    int *state, *depth;                   // [P]
    uint8_t *mirror;                      // [P] pending hit is a mirror
    uint32_t *st_idx, *st_direct;         // [max_depth][P] per-level (sphere, clamped direct light)
    double *leaf;                         // [3][P] colour at the end of the path
};

// batched RayTracerEnv state (SoA, [3][B] for vectors)
template <typename T> struct EnvDev {
    int B, W, H, max_bounces, flavour, sun_id;
    T cam[3], cam_angle[3], tan_half;
    int adaptive, light0, light1;                    // AdaptiveRewardRayTracerEnv (rt_env_desc::reward_mode)
    int b0;                                          // global index of env 0 of this batch (rt_env_desc::env_offset)
    int *has_hit, *idx, *bounce, *through, *episode, *consec, *total_hits;
    T *p, *n, *d, *acc;
    T *rgb;                                          // [3][B] RL flavour: terminalRGB of the current hit (shaded once, used twice)
    double *total;
};

template <typename T> __host__ __device__ inline size_t align32(size_t x) { return (x + 31) & ~size_t(31); }

// bytes of dynamic shared memory the staged scene needs (host + device agree on the layout)
template <typename T> __host__ __device__ inline size_t scene_smem_bytes(int n, int nG, int nP, int nL) {
    const size_t v = sizeof(typename M<T>::v4);
    size_t b = 0;
    b += (2 * (size_t)((n + 7) & ~7) + 2 * (size_t)n) * v;  // sph (padded to 8), pk (sphere pairs), mat, col
    b += 2 * (size_t)nG * v + 2 * (size_t)nP * v + 2 * (size_t)nL * v + RT_LPK_STRIDE * (size_t)((nL + 1) / 2) * v;
    b = align32<T>(b);
    b += sizeof(int) * ((size_t)n + nG + 2 * (size_t)nP + nL);
    return align32<T>(b);
}
template <typename T> static inline size_t smem_for(const SceneDev<T> &sc) {
    return scene_smem_bytes<T>(sc.n, sc.nG, sc.nP, sc.nL);
}

#define RT_SMEM_LIMIT (96 * 1024)

// kMode for a scene: shared-memory staging when it fits, hierarchy code only when a hierarchy exists
template <typename T> static inline int mode_for(const SceneDev<T> &sc, size_t extra_smem = 0) {
    const bool shared = smem_for(sc) + extra_smem <= RT_SMEM_LIMIT;
    if (!shared) return 2;
    return sc.bvh.nodes > 0 ? 1 : 0;
}

template <typename T>
cudaError_t launch_whitted(const SceneDev<T> &sc, const WhittedDev<T> &wp, void *accum, int *hit,
                           unsigned long long *stats, cudaStream_t st, unsigned *sched, unsigned *sched2 = nullptr,
                           unsigned *heavy = nullptr);
// sched2 / heavy non-NULL: the caller allows the two-pass schedule (exact only for integer-valued colours: it adds the
// samples of a pixel with FP32 reductions in no fixed order)
// kernel variant (kMode) and dynamic shared memory of a path-kernel launch (plan_path_launch, rt_api.cu)
struct PathLaunch { int mode; size_t smem; };
// where the kMoments path kernels put the second moments (sum r^2, sum g^2, sum b^2, n): the kernel's trailing parameter,
// not fields of PathDev, whose layout the plain kernels' instruction schedule depends on
struct MomentsDev {
    double4 *local;              // RT_SINK_ACCUM: [H,W,4] doubles, stored like accum
    double4 *peer[16];           // RT_SINK_SCATTER_ADD: the owners' [H,W,4] moments (own at [rank], peer mappings elsewhere)
    float *var;                  // RT_SINK_IMAGE, and RT_SINK_SCATTER_ADD under sync: rank 0's [H,W,3] variance image
};
// the trailing parameter of a list launch (kList): the moments sinks plus the pixels y * W + x to trace and their number
struct MomentsListDev : MomentsDev {
    const uint32_t *list;
    unsigned count;
};
template <typename T>
cudaError_t launch_path(const SceneDev<T> &sc, const PathDev<T> &pp, const PathLaunch &pl, void *accum,
                        unsigned long long *stats, cudaStream_t st, const PkConst *pkc, const MomentsDev *moments,
                        const MomentsListDev *listed);
// pkc: host copy of the FP32 pair arrays, read by kMode 3; pp.sched: two zeroed device counters owned by this launch;
// moments: NULL (plain kernels), or the moments sinks of the kMoments kernels; listed: NULL, or a list launch (integer
// fold, accumulate, RT_SINK_ACCUM), which takes its moments sink from there
template <typename T>
cudaError_t launch_trajectories(const SceneDev<T> &sc, int n_traj, int max_steps, int max_bounces, uint64_t seed, float *obs,
                                float *action, float *next_obs, float *reward, uint8_t *hit, int *length,
                                uint8_t *hit_light, unsigned long long *stats, cudaStream_t st);
template <typename T>
cudaError_t launch_simple(const SceneDev<T> &sc, const SimpleDev<T> &sp, int4 *rgb, float *image, unsigned long long *stats,
                          cudaStream_t st);
template <typename T>
cudaError_t launch_resolve(const void *accum, int W, int y0, int y1, int spp, float *image, cudaStream_t st);
// rt_f32.cu: resolve + clear, peer flags
cudaError_t launch_resolve_clear(float4 *accum, int W, int y0, int y1, int spp, float *image, int clear, cudaStream_t st);
// the same with the moments: also the variance of rows [y0,y1) into var (rt_resolve_variance), and clear both buffers' rows
cudaError_t launch_resolve_clear_moments(float4 *accum, double4 *moments, int W, int y0, int y1, int spp, float *image,
                                         float *var, int clear, cudaStream_t st);
struct PeerFlagTable { unsigned *p[32]; };      // flag addresses ride in the kernel's parameter block
cudaError_t launch_peer_signal(const PeerFlagTable &flags, int n, unsigned epoch, cudaStream_t st);
cudaError_t launch_peer_wait(const unsigned *flags, int n, unsigned epoch, long long timeout_cycles, int *timed_out,
                             cudaStream_t st);
template <typename T>
cudaError_t launch_sphere_disc(int m, const double *rays, const double *spheres, int point, double *out, cudaStream_t st);
template <typename T>
cudaError_t launch_trace_rays(const SceneDev<T> &sc, int m, const double *rays, const int *suppress, const int *bounces0,
                              const int *through0, int max_bounces, int shadow_max_bounces, const double miss[3],
                              double *term, double *rgb, cudaStream_t st);
template <typename T>
cudaError_t launch_shade_hits(const SceneDev<T> &sc, int m, const double *hits, int shadow_max_bounces, double *rgb,
                              cudaStream_t st);
// first-hit features of rows [pp.y0, pp.y1) over samples [pp.s0, pp.s1) (rt_render_features): pp needs the camera, W, H,
// the band, the sample range and the Philox keys; albedo / normal / fvar [H,W,3], depth [H,W] float32
template <typename T>
cudaError_t launch_features(const SceneDev<T> &sc, const PathDev<T> &pp, float *albedo, float *normal, float *depth,
                            float *fvar, cudaStream_t st);
template <typename T>
cudaError_t launch_env_reset(const SceneDev<T> &sc, const EnvDev<T> &e, const int *pixels, const uint8_t *mask,
                             uint64_t seed, float *obs, int *pixels_out, unsigned long long *stats, cudaStream_t st);
// shade the current hits again after the scene changed under running episodes (EnvDev::rgb)
template <typename T> cudaError_t launch_env_reshade(const SceneDev<T> &sc, const EnvDev<T> &e, cudaStream_t st);
template <typename T, typename R, bool kAuto>
cudaError_t launch_env_step(const SceneDev<T> &sc, const EnvDev<T> &e, const float *actions, float *obs, R *reward,
                            uint8_t *terminated, uint8_t *truncated, int *reason, R *info, float *final_obs, int *pixels_out,
                            uint64_t seed, unsigned long long *stats, cudaStream_t st);

template <typename T>
cudaError_t launch_wf_begin(const WaveDev<T> &w, const PathDev<T> &pp, unsigned long long *stats, cudaStream_t st);
template <typename T>
cudaError_t launch_wf_trace(const SceneDev<T> &sc, const WaveDev<T> &w, float *obs, uint8_t *need, unsigned long long *stats,
                            cudaStream_t st);
template <typename T>
cudaError_t launch_wf_bounce(const WaveDev<T> &w, const uint8_t *need, const float *actions, unsigned long long *stats,
                             int *live_count, cudaStream_t st);
template <typename T>
cudaError_t launch_wf_finish(const SceneDev<T> &sc, const WaveDev<T> &w, void *accum, double *moments, cudaStream_t st);
// variance of each pixel's mean from accum and moments (rt_resolve_variance): rows [y0, y1) of var [H,W,3]
template <typename T>
cudaError_t launch_resolve_variance(const void *accum, const double *moments, int W, int y0, int y1, float *var, cudaStream_t st);
// adaptive frames (rt_render_path_adaptive): the pixels of rows [y0, y1) with accum.w == c whose variance of the mean
// exceeds thr in some channel, appended to list; *count must be zero before the launch and holds their number after it
template <typename T>
cudaError_t launch_adaptive_select(const void *accum, const double *moments, int W, int y0, int y1, int c, double thr,
                                   uint32_t *list, uint32_t *count, cudaStream_t st);
// image (and optionally var and the sample counts) of rows [y0, y1), each pixel resolved by its own count accum.w
template <typename T>
cudaError_t launch_adaptive_resolve(const void *accum, const double *moments, int W, int y0, int y1, float *image,
                                    float *var, int *counts, cudaStream_t st);

// variance-guided non-local-means filter of a whole frame (rt_denoise.cu): accum [H,W,4] of T and var [H,W,3] ->
// image [H,W,3]; search radius r in [0, 15], patch radius f in [0, 5] (cudaErrorInvalidValue otherwise)
template <typename T>
cudaError_t launch_denoise(const void *accum, const float *var, int W, int H, int r, int f, float k, float *image,
                           cudaStream_t st);
// the same filter with the feature term (rt_denoise_features): albedo / normal / fvar [H,W,3] and depth [H,W] float32 as
// rt_render_features gives them; k_f > 0, tau >= 0
struct DenoiseFeatures {
    const float *albedo, *normal, *depth, *fvar;
    float kf2, tau;                      // k_f^2 and the floor of the feature denominators
};
// k^2 and k_f^2 for the filter: squared in double and clamped to FLT_MAX, so that a finite k above sqrt(FLT_MAX) keeps
// the limit k -> infinity (FLT_MAX * 0 = 0 for zero variance; an infinite product gives delta = 0) instead of inf * 0
inline float square_to_float(float k) {
    const double k2 = (double)k * k;
    return k2 < (double)FLT_MAX ? (float)k2 : FLT_MAX;
}
template <typename T>
cudaError_t launch_denoise_features(const void *accum, const float *var, const DenoiseFeatures &feat, int W, int H, int r,
                                    int f, float k, float *image, cudaStream_t st);
// halo depth of the filters (rt_denoise_halo): an output row reads rows within r + f of its own; the feature gradient
// reads y +- 1 whatever r and f are
inline int denoise_halo(int r, int f, bool features) {
    return features && r + f < 1 ? 1 : r + f;
}
// the same filters for the output rows [y0, y1) of the frame only (rt_denoise_rows, rt_denoise_features_rows): buffers
// stay [H,W,.]; the kernels read rows [max(0, y0 - h), min(H, y1 + h)) and write rows [y0, y1), 0 <= y0 < y1 <= H
template <typename T>
cudaError_t launch_denoise_rows(const void *accum, const float *var, int W, int H, int y0, int y1, int r, int f, float k,
                                float *image, cudaStream_t st);
template <typename T>
cudaError_t launch_denoise_features_rows(const void *accum, const float *var, const DenoiseFeatures &feat, int W, int H,
                                         int y0, int y1, int r, int f, float k, float *image, cudaStream_t st);

// FFMA issue-rate micro-benchmark (rt_f32.cu): `iters` trips of 16 independent FFMA per thread
cudaError_t launch_fp32_peak(int blocks, int threads, int iters, float *sink, cudaStream_t st);

}  // namespace rt
