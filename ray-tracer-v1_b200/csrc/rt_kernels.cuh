// rt_kernels.cuh -- the CUDA kernels of the hot path (templates; instantiated for float in rt_f32.cu and for
// double, without FMA contraction, in rt_f64.cu) and their launchers.
//
//   whitted_kernel   Algorithm A frame: camera ray -> nearestSphereIntersect -> terminalRGB, spp accumulation
//   path_kernel      Algorithm B frame: TraditionalRenderer.render, persistent warps whose per-pixel lanes trace one
//                    sample together, one nearest-hit query per loop trip, and fold it once the longest path has ended
//   trace_rays_kernel / sphere_disc_kernel   batched Ray.nearestSphereIntersect / sphereDiscriminant
//   env_reset_kernel / env_step_kernel       batched RayTracerEnv
//   resolve_kernel   sums -> float32 image
//
// Thread mapping for frames: 256-thread blocks cover 32 x 8 pixels; each warp owns an 8 x 4 pixel tile so primary
// rays of a warp are spatially coherent and the float4 accumulator rows it writes are full 128-byte segments.
#pragma once
#include "rt_trace.cuh"
#include "rt_launch.h"
#include <mutex>
#include <type_traits>
#include <vector>

namespace rt {

// ------------------------------------------------------------------ scene staging
template <typename T> struct Staged {
    Geo<T> g;
    LightsA<T> la;
    LightsB<T> lb;
};

template <typename T> RT_DEV void coop_copy(T *dst, const T *src, int count) {
    for (int i = threadIdx.x; i < count; i += blockDim.x) dst[i] = src[i];
}

template <typename T, bool kShared> RT_DEV void stage_scene(const SceneDev<T> &sc, unsigned char *smem, Staged<T> &S) {
    using v4 = typename M<T>::v4;
    S.g.sv.n = sc.n;
    S.g.sv.n_padded = (sc.n + 7) & ~7;      // both the staged copy and the HBM blob are padded
    S.g.sv.key_mask = sc.key_mask; S.g.sv.key_mask6 = sc.key_mask6;
    S.g.bvh = sc.bvh;
    S.la.nG = sc.nG; S.la.nP = sc.nP; S.lb.nL = sc.nL;
    S.la.bg[0] = sc.bg[0]; S.la.bg[1] = sc.bg[1]; S.la.bg[2] = sc.bg[2];
    if constexpr (kShared) {
        v4 *p = reinterpret_cast<v4 *>(smem);
        v4 *sph = p; p += (sc.n + 7) & ~7;
        v4 *pk = p; p += (sc.n + 7) & ~7;
        v4 *mat = p; p += sc.n;
        v4 *col = p; p += sc.n;
        v4 *g_vec = p; p += sc.nG;
        v4 *g_col = p; p += sc.nG;
        v4 *p_pos = p; p += sc.nP;
        v4 *p_col = p; p += sc.nP;
        v4 *l_pos = p; p += sc.nL;
        v4 *l_col = p; p += sc.nL;
        v4 *lpk = p; p += RT_LPK_STRIDE * ((sc.nL + 1) / 2);
        size_t off = align32<T>((size_t)(reinterpret_cast<unsigned char *>(p) - smem));
        int *q = reinterpret_cast<int *>(smem + off);
        int *ids = q; q += sc.n;
        int *g_func = q; q += sc.nG;
        int *p_id = q; q += sc.nP;
        int *p_func = q; q += sc.nP;
        int *l_index = q; q += sc.nL;
        coop_copy(sph, sc.sph, 2 * ((sc.n + 7) & ~7));       // sph and pk are adjacent in the blob
        coop_copy(mat, sc.mat, sc.n); coop_copy(col, sc.col, sc.n);
        coop_copy(ids, sc.ids, sc.n);
        coop_copy(g_vec, sc.g_vec, sc.nG); coop_copy(g_col, sc.g_col, sc.nG); coop_copy(g_func, sc.g_func, sc.nG);
        coop_copy(p_pos, sc.p_pos, sc.nP); coop_copy(p_col, sc.p_col, sc.nP);
        coop_copy(p_id, sc.p_id, sc.nP); coop_copy(p_func, sc.p_func, sc.nP);
        coop_copy(l_pos, sc.l_pos, sc.nL); coop_copy(l_col, sc.l_col, sc.nL); coop_copy(l_index, sc.l_index, sc.nL);
        coop_copy(lpk, sc.lpk, RT_LPK_STRIDE * ((sc.nL + 1) / 2));
        __syncthreads();
        S.g.sv.sph = sph; S.g.sv.pk = pk; S.g.sv.mat = mat; S.g.sv.col = col; S.g.sv.ids = ids;
        S.la.g_vec = g_vec; S.la.g_col = g_col; S.la.g_func = g_func;
        S.la.p_pos = p_pos; S.la.p_col = p_col; S.la.p_id = p_id; S.la.p_func = p_func;
        S.lb.l_pos = l_pos; S.lb.l_col = l_col; S.lb.l_index = l_index; S.lb.lpk = lpk;
    } else {
        S.g.sv.sph = sc.sph; S.g.sv.pk = sc.pk; S.g.sv.mat = sc.mat; S.g.sv.col = sc.col; S.g.sv.ids = sc.ids;
        S.la.g_vec = sc.g_vec; S.la.g_col = sc.g_col; S.la.g_func = sc.g_func;
        S.la.p_pos = sc.p_pos; S.la.p_col = sc.p_col; S.la.p_id = sc.p_id; S.la.p_func = sc.p_func;
        S.lb.l_pos = sc.l_pos; S.lb.l_col = sc.l_col; S.lb.l_index = sc.l_index; S.lb.lpk = sc.lpk;
    }
}

// pixel of this thread inside the launch's row band: 32x8 block tile, 8x4 warp tile
RT_DEV void tile_pixel(int &x, int &y_rel) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    x = blockIdx.x * 32 + (w & 3) * 8 + (lane & 7);
    y_rel = blockIdx.y * 8 + (w >> 2) * 4 + (lane >> 3);
}

RT_DEV void flush_stats(unsigned long long *stats, int slot, unsigned long long v) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(stats + slot, v);
}

// Kernel variants: kMode 0 = scene staged in shared memory, brute force (no hierarchy code in the kernel at all);
//                  kMode 1 = staged in shared memory + LBVH traversal; kMode 2 = scene read from global + LBVH;
//                  kMode 3 (path_kernel, FP32 only) = kMode 0 with the sphere pairs of a <= RT_PKC_MAX-sphere scene in
//                  the kernel parameter block (constant bank -> uniform registers), see brute_select_pkc.
#ifndef RT_PATH_MIN_BLOCKS
#define RT_PATH_MIN_BLOCKS 3   /* 3 x 256 threads per SM at <= 85 registers: measured 2.7 % faster than 4 at <= 64 */
#endif
#ifndef RT_WHITTED_MIN_BLOCKS
#define RT_WHITTED_MIN_BLOCKS 2   /* Algorithm A frame kernel: 120 registers unconstrained */
#endif
#ifndef RT_PATH_MIN_BLOCKS_PKC
#define RT_PATH_MIN_BLOCKS_PKC 4   /* kMode 3 needs 72 registers unconstrained: 4 CTAs/SM at 64 measured 2.2 % faster (no spills) */
#endif
#define RT_MODE_DECL constexpr bool kShared = kMode != 2; constexpr bool kBvh = kMode == 1 || kMode == 2

// ------------------------------------------------------------------ Algorithm A frame
// camera rays of a warp's 8x4 pixel tile: the spheres their cone can touch (cone_candidates, rt_trace.cuh), built once
// for all samples.  Tiles of sky get an empty list and skip the sphere loop altogether; frames are unchanged.
template <typename T> RT_DEV unsigned long long whitted_tile_candidates(const Staged<T> &S, const WhittedDev<T> &wp, int x, int y, int lane) {
    const float gx = (float)wp.X[min(x, wp.W - 1)], gy = (float)wp.Y[min(y, wp.y1 - 1)];
    float xlo = gx, xhi = gx, ylo = gy, yhi = gy;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        xlo = fminf(xlo, __shfl_xor_sync(0xffffffffu, xlo, o)); xhi = fmaxf(xhi, __shfl_xor_sync(0xffffffffu, xhi, o));
        ylo = fminf(ylo, __shfl_xor_sync(0xffffffffu, ylo, o)); yhi = fmaxf(yhi, __shfl_xor_sync(0xffffffffu, yhi, o));
    }
    const float jx = wp.spp > 1 ? 0.5f * fabsf((float)wp.pitch_x) : 0.f, jy = wp.spp > 1 ? 0.5f * fabsf((float)wp.pitch_y) : 0.f;
    const float ex = 0.5f * (xhi - xlo) + jx, ey = 0.5f * (yhi - ylo) + jy;
    const V3<float> d0 = normalise(mk<float>(0.5f * (xlo + xhi), 0.5f * (ylo + yhi), -1.f));
    const float alpha = sqrtf(ex * ex + ey * ey) * 1.001f + 1e-6f;       // angle <= distance on the z = -1 plane
    return cone_candidates(reinterpret_cast<const float4 *>(S.g.sv.sph), S.g.sv.n,
                           mk<float>((float)wp.cam[0], (float)wp.cam[1], (float)wp.cam[2]), d0, alpha, lane);
}

// one sample of one pixel: jittered camera ray (output5.py:1463-1470), nearestSphereIntersect, terminalRGB -> c[3]
template <typename T, bool kBvh>
RT_DEV int whitted_sample(const Staged<T> &S, const WhittedDev<T> &wp, V3<T> cam, T X0, T Y0, uint32_t pixel, int s,
                          unsigned long long cand, Counters &ct, T c[3]) {
    T Xj = X0, Yj = Y0;
    if (wp.spp > 1) {
        Philox4 o = philox4x32_10(pixel, (uint32_t)s, 0u, RT_PHILOX_TAG, wp.k0, wp.k1);
        Xj = X0 + (u01<T>(o.w[0]) - T(0.5)) * wp.pitch_x;
        Yj = Y0 + (u01<T>(o.w[1]) - T(0.5)) * wp.pitch_y;
    }
    V3<T> d = mk<T>(Xj, Yj, T(-1));
    if constexpr (M<T>::exact) { if (wp.prenorm) d = normalise(d); }
    d = normalise(d);                                            // Ray.__init__, ray.py:69-71
    Hit<T> h = trace_terminal<T, kBvh>(S.g, cam, d, RT_NO_ID_DEV, 0, wp.max_bounces, 0, ct, cand);
    if (h.idx >= 0) { terminal_rgb<T, kBvh>(S.g, S.la, h, wp.shadow_max_bounces, c, ct); return h.idx; }
    c[0] = wp.miss[0]; c[1] = wp.miss[1]; c[2] = wp.miss[2];
    return -1;
}

// PERSISTENT WARPS, as in path_kernel: the launch has as many CTAs as the device keeps resident, the scene is staged and
// the statistics are flushed once per CTA, and every WARP pulls its next 8x4-pixel tile from a device counter (the
// first tiles are static, the fetch for the next one is issued before the current one is traced, the last warp of the
// launch re-arms the counter).  A 1280x720 frame is 28,800 warp tiles of which typically > 95 % are sky: with one CTA
// per 32x8 block the frame cost what 3,600 CTA prologues cost (0.13 ms); now a sky tile costs a few dozen instructions.
template <typename T, int kMode>
__global__ void __launch_bounds__(256, (sizeof(T) == 4 ? RT_WHITTED_MIN_BLOCKS : 1)) whitted_kernel(SceneDev<T> sc, WhittedDev<T> wp, typename M<T>::v4 *accum,
                                                      int *hit_out, unsigned long long *stats) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int w_ = threadIdx.x >> 5, lane_ = threadIdx.x & 31;
    Counters ct = {0u, 0u, 0u, 0u};
    unsigned primaries = 0;
    const V3<T> cam = mk<T>(wp.cam[0], wp.cam[1], wp.cam[2]);
    const unsigned n_units = (unsigned)(wp.gx * wp.gy) << 3, first_dyn = (unsigned)gridDim.x << 3;
    for (unsigned unit = ((unsigned)blockIdx.x << 3) + (unsigned)w_; unit < n_units;) {
    unsigned nxt = 0;
    if (lane_ == 0) nxt = first_dyn + atomicAdd(wp.sched, 1u);
    RT_ASSERT(unit < n_units);
    const int tile = (int)(unit >> 3), wt = (int)(unit & 7u);          // 32x8-pixel block, the warp's 8x4 tile in it
    const int by = tile / wp.gx, bx = tile - by * wp.gx;
    const int x = bx * 32 + (wt & 3) * 8 + (lane_ & 7);
    const int y = wp.y0 + by * 8 + (wt >> 2) * 4 + (lane_ >> 3);
    // camera rays of this warp's 8x4 pixel tile: the spheres their cone can touch (cone_candidates, rt_trace.cuh), built
    // once for all samples.  Tiles of sky get an empty list and skip the sphere loop altogether; frames are unchanged.
    unsigned long long cand = ~0ull;
    if constexpr (!M<T>::exact && kMode == 0) {
        if (sc.n <= 64 && wp.W > 0 && wp.y1 > wp.y0) cand = whitted_tile_candidates<T>(S, wp, x, y, lane_);
    }
    bool listed = false;
    if constexpr (!M<T>::exact && kMode == 0) {
        // two-pass frame: a tile some sphere can be seen in is only LISTED here (and its pixels zeroed); pass 2 traces it,
        // one (tile, sample) unit per warp, on every warp of the device
        if (wp.split && cand != 0ull) {
            listed = true;
            if (lane_ == 0) wp.heavy[atomicAdd(wp.sched + 2, 1u)] = unit;
            if (!wp.accumulate && x < wp.W && y < wp.y1) accum[(size_t)y * wp.W + x] = M<T>::make4(T(0), T(0), T(0), T(0));
        }
    }
    if (!listed && x < wp.W && y < wp.y1) {
        const T X0 = wp.X[x], Y0 = wp.Y[y];
        const uint32_t pixel = (uint32_t)(y * wp.W + x);
        T a0 = T(0), a1 = T(0), a2 = T(0);
        int last = -1;
        if (cand == 0ull) {
            // No sphere can be touched by ANY ray of this warp tile's cone (the cone includes the jitter margin), so every
            // sample of every pixel of the tile misses: the sum is the miss colour added s1 - s0 times (the same
            // additions as the loop below would make, so the frame is unchanged) and neither the Philox jitter nor the
            // ray is needed.
            for (int s = wp.s0; s < wp.s1; ++s) { a0 += wp.miss[0]; a1 += wp.miss[1]; a2 += wp.miss[2]; }
            primaries += (unsigned)(wp.s1 - wp.s0);
            ct.queries += (unsigned)(wp.s1 - wp.s0);        // one nearestSphereIntersect per sample, over an empty candidate list
        } else
        for (int s = wp.s0; s < wp.s1; ++s) {
            T c[3];
            last = whitted_sample<T, kBvh>(S, wp, cam, X0, Y0, pixel, s, cand, ct, c);
            primaries++;
            a0 += c[0]; a1 += c[1]; a2 += c[2];
        }
        const size_t o = (size_t)y * wp.W + x;
        RT_ASSERT(o < (size_t)wp.W * wp.H);
        typename M<T>::v4 out = M<T>::make4(a0, a1, a2, T(wp.s1 - wp.s0));
        if (wp.accumulate) {
            const typename M<T>::v4 old = accum[o];
            out.x += old.x; out.y += old.y; out.z += old.z; out.w += old.w;
        }
        accum[o] = out;
        if (hit_out) hit_out[o] = last;
    }
    unit = __shfl_sync(0xffffffffu, nxt, 0);
    }   // warp tiles of this warp
    if (lane_ == 0) {
        // every warp of the launch passes here exactly once, after its last fetch: the last one re-arms the counters
        __threadfence();
        if (atomicAdd(wp.sched + 1, 1u) == (gridDim.x << 3) - 1u) { wp.sched[0] = 0u; wp.sched[1] = 0u; __threadfence(); }
    }
    if (stats) {
        flush_stats(stats, STAT_QUERIES, ct.queries); flush_stats(stats, STAT_DEAD_QUERIES, ct.dead);
        flush_stats(stats, STAT_RAYS, primaries);
        flush_stats(stats, STAT_SPHERE_TESTS, ct.tests);
        flush_stats(stats, STAT_AABB_TESTS, ct.boxes);
    }
}

// Pass 2 of a two-pass Algorithm-A frame (FP32): the listed tiles x the samples of the launch are (tile, sample) units
// pulled by every warp of the device from a counter; a unit traces ONE sample of the tile's 32 pixels and adds
// (r, g, b, 1) to the pixel with one 16-byte reduction (sums of integer-valued colours are exact in FP32, so the frame
// does not depend on the order; the API only selects this schedule when background and miss colour are integers).
// A frame whose spheres cover 1 % of the view had all its work in the few warps that own those tiles -- the frame took
// as long as ONE warp needs for 16 samples of a tile (~0.1 ms); spread over all warps it takes a fraction of that.
template <int kMode>
__global__ void __launch_bounds__(256, RT_WHITTED_MIN_BLOCKS) whitted_heavy_kernel(SceneDev<float> sc, WhittedDev<float> wp, float4 *accum,
                                                                                  int *hit_out, unsigned long long *stats) {
    using T = float;
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int w_ = threadIdx.x >> 5, lane_ = threadIdx.x & 31;
    Counters ct = {0u, 0u, 0u, 0u};
    unsigned primaries = 0;
    const V3<T> cam = mk<T>(wp.cam[0], wp.cam[1], wp.cam[2]);
    const unsigned ns = (unsigned)(wp.s1 - wp.s0);
    const unsigned n_units = __ldcg(wp.sched + 2) * ns, first_dyn = (unsigned)gridDim.x << 3;     // pass 1 has finished (stream order)
    for (unsigned unit = ((unsigned)blockIdx.x << 3) + (unsigned)w_; unit < n_units;) {
        unsigned nxt = 0;
        if (lane_ == 0) nxt = first_dyn + atomicAdd(wp.sched2, 1u);
        const unsigned tu = wp.heavy[unit / ns];
        const int s = wp.s0 + (int)(unit % ns);
        const int tile = (int)(tu >> 3), wt = (int)(tu & 7u);
        const int by = tile / wp.gx, bx = tile - by * wp.gx;
        const int x = bx * 32 + (wt & 3) * 8 + (lane_ & 7);
        const int y = wp.y0 + by * 8 + (wt >> 2) * 4 + (lane_ >> 3);
        const unsigned long long cand = whitted_tile_candidates<T>(S, wp, x, y, lane_);
        if (x < wp.W && y < wp.y1) {
            T c[3];
            const int last = whitted_sample<T, kBvh>(S, wp, cam, wp.X[x], wp.Y[y], (uint32_t)(y * wp.W + x), s, cand, ct, c);
            primaries++;
            const size_t o = (size_t)y * wp.W + x;
            RT_ASSERT(o < (size_t)wp.W * wp.H);
            asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1, %2, %3, %4};"
                         :: "l"(accum + o), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(1.f) : "memory");
            if (hit_out && s == wp.s1 - 1) hit_out[o] = last;
        }
        unit = __shfl_sync(0xffffffffu, nxt, 0);
    }
    if (lane_ == 0) {
        __threadfence();
        if (atomicAdd(wp.sched2 + 1, 1u) == (gridDim.x << 3) - 1u) {      // last warp: re-arm both passes' counters
            wp.sched2[0] = 0u; wp.sched2[1] = 0u; wp.sched[2] = 0u; __threadfence();
        }
    }
    if (stats) {
        flush_stats(stats, STAT_QUERIES, ct.queries); flush_stats(stats, STAT_DEAD_QUERIES, ct.dead);
        flush_stats(stats, STAT_RAYS, primaries);
        flush_stats(stats, STAT_SPHERE_TESTS, ct.tests);
        flush_stats(stats, STAT_AABB_TESTS, ct.boxes);
    }
}

// ------------------------------------------------------------------ epoch flags in peer memory (rt_path_sink::sync)
// wait: system-scope acquire loads until the flag has reached the epoch (wrap-safe compare); gives up after
// timeout_cycles and reports instead of hanging.  post: system-scope release store; the caller has fenced.
#ifdef RT_TRACE_WARPS
RT_DEV unsigned long long rt_globaltimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#endif
RT_DEV void flag_wait(const unsigned *flag, unsigned epoch, long long timeout_cycles, int *timed_out) {
    const long long t0 = clock64();
    for (;;) {
        unsigned v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int)(v - epoch) >= 0) return;
        if (clock64() - t0 > timeout_cycles) { if (timed_out) *timed_out = 1; return; }
        __nanosleep(64);
    }
}
RT_DEV void flag_post(unsigned *flag, unsigned epoch) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(flag), "r"(epoch) : "memory");
}
RT_DEV bool a_count_ok(int spp_total) { return spp_total > 0; }

// variance of a pixel's mean in colour levels^2, from the sum S and the sum of squares Q of its k samples:
// (Q - S^2/k) / (k (k-1)), evaluated as (k Q - S^2) / (k^2 (k-1)) -- the numerator is exact while k Q and S^2 stay below
// 2^53 (integer colours), so a pixel whose samples all agree gets exactly 0; 0 where k < 2.  Every site that resolves a
// variance (resolve_variance_kernel, the fused sinks of path_kernel, resolve_clear_moments_kernel) calls this one
// expression, so their results agree bit for bit.
RT_DEV float variance_of_mean(double S, double Q, double k) {
    double v = 0.0;
    if (k >= 2.0) {
        v = __ddiv_rn(__dsub_rn(__dmul_rn(k, Q), __dmul_rn(S, S)), __dmul_rn(__dmul_rn(k, k), k - 1.0));
        v = v > 0.0 ? v : 0.0;
    }
    return (float)v;
}
#define RT_FLAG_ADDED 0
#define RT_FLAG_DONE 16
#define RT_FLAG_GO 32

// explicit shared-memory loads off a 32-bit shared-window address (see path_kernel, kMode 3)
RT_DEV float4 lds_v4(unsigned addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
template <int kStride> RT_DEV void lds_v4x2(unsigned addr, float4 &a, float4 &b) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(addr));
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(addr), "n"(kStride));
}

// ------------------------------------------------------------------ Algorithm B frame
// TraditionalRenderer.generate_camera_ray (chandelier.py:417-429): aspect is applied twice on x.
template <typename T> RT_DEV V3<T> path_camera_ray(const PathDev<T> &pp, int x, int y, T u0, T u1) {
    T sx = T(0.5) + (u0 - T(0.5)), sy = T(0.5) + (u1 - T(0.5));         // 0.5 + jitter, chandelier.py:534-536
    T ndc_x, ndc_y;
    if constexpr (M<T>::exact) { ndc_x = (T(x) + sx) / T(pp.W); ndc_y = (T(y) + sy) / T(pp.H); }
    else { ndc_x = (T(x) + sx) * pp.inv_W; ndc_y = (T(y) + sy) * pp.inv_H; }      // two multiplies instead of two divisions
    T scx = T(2) * ndc_x - T(1), scy = T(1) - T(2) * ndc_y;
    scx *= pp.aspect; scx *= pp.half_w; scy *= pp.half_h;
    V3<T> d = normalise(mk<T>(scx, scy, T(-1)));
    if constexpr (M<T>::exact) d = normalise(d);                         // Ray() normalises again
    return d;
}

// The camera ray of a sample of pixel (x, y), rng begun at the key (pixel, sample): Philox slot 0 jitters it inside the
// pixel.  path_kernel and feature_kernel both call it, so the features see exactly the rays the frame traces.
template <typename T> RT_DEV V3<T> path_sample_ray(const PathDev<T> &pp, PathRng &rng, int x, int y) {
    uint32_t wa, wb;
    rng.pair_rk(0u, wa, wb, pp.rk);
    return path_camera_ray<T>(pp, x, y, u01<T>(wa), u01<T>(wb));
}

// One thread per pixel, looping over its samples; 8x4-pixel warps in lock-step: the warp traces sample s of all its
// 32 pixels together, one nearest-hit query per trip, until every lane's path has ended, then folds and starts sample
// s+1 together.  Everything outside the sphere loop (camera ray, Philox, fold) runs once per sample at full lane
// occupancy.
// kIntFold: integer fold through the div255 table (all leaf colours integer-valued), else the double-division fold.
// kMoments: also the second moments of the pixel's samples, (sum r^2, sum g^2, sum b^2, n), into the sink of MomentsDev
// that matches pp.sink: moments.local[o] like accum, the variance of the resolved pixel into moments.var (image sink), or
// added into the owner's moments.peer[k] (scatter-add sink).  The trailing parameter is empty otherwise, so the plain
// kernels keep their parameter offsets.  Exact: an integer-fold colour is <= 65535, so its square fits a uint32 and a
// uint64 sum of 65536 of them stays below 2^53; the double fold sums its squares in double.
// kList (with kIntFold and kMoments only): a list launch of an adaptive frame (rt_render_path_adaptive) traces only the
// pixels of moments.list, adding into their accum and moments: unit u takes entries [u (32 >> lk), (u + 1) (32 >> lk)).
template <typename T, int kMode, bool kIntFold, bool kMoments, bool kList = false>
__global__ void __launch_bounds__(256, (sizeof(T) == 4 ? (kMode == 3 ? RT_PATH_MIN_BLOCKS_PKC : RT_PATH_MIN_BLOCKS) : 1))
path_kernel(SceneDev<T> sc, PathDev<T> pp, typename M<T>::v4 *accum, unsigned long long *stats,
            const __grid_constant__ typename std::conditional<kMode == 3, PkConst, PkNone>::type pkc,
            const __grid_constant__ typename std::conditional<kMoments, typename std::conditional<kList, MomentsListDev, MomentsDev>::type,
                                                              PkNone>::type moments) {
    static_assert(!kList || (kIntFold && kMoments), "list launches fold in integers and keep the moments");
    RT_MODE_DECL;
    using PK = typename std::conditional<kMode == 3, PkConst, PkNone>::type;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    double *div255;                                                    // [256] k / 255.0, correctly rounded
    const float4 *hitrec = nullptr;                                    // kMode 3: (1/r, reflective, emissive, -) per sphere
    unsigned s_base = 0;                                               // kMode 3: shared-window address of the static block
    if constexpr (kMode == 3) {
        // <= RT_PKC_MAX spheres: STATIC shared arrays at fixed offsets, so every per-hit fetch is one LDS with an
        // immediate base (the dynamic layout costs ~8 address instructions per fetch, its offsets depend on n)
        // ONE block (sph | hit | col | cw at 1 KB strides) read with explicit ld.shared off a 32-bit base kept in a
        // register: the compiler's own addressing of static shared arrays re-derives the cluster window base (S2R
        // CgaCtaId, MOV, IADD3, LEA) at every site, 6 instructions per winner fetch
        __shared__ __align__(16) float4 s_all[4 * RT_PKC_MAX];
        __shared__ __align__(16) double s_div255[256];
        float4 *const s_sph = s_all, *const s_hit = s_all + RT_PKC_MAX, *const s_col = s_all + 2 * RT_PKC_MAX, *const s_cw = s_all + 3 * RT_PKC_MAX;
        s_base = (unsigned)__cvta_generic_to_shared(s_all);
        const int n_pad = (sc.n + 7) & ~7;
        const float *pkf = reinterpret_cast<const float *>(sc.pk);       // pair j: cx0 cx1 cy0 cy1 | cz0 cz1 w0 w1
        for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
            const float *q = pkf + 8 * (i >> 1) + (i & 1);
            s_cw[i] = make_float4(q[0], q[2], q[4], q[6]);
            s_sph[i] = reinterpret_cast<const float4 *>(sc.sph)[i];
            if (i < sc.n) {
                const float4 mt = reinterpret_cast<const float4 *>(sc.mat)[i], cl = reinterpret_cast<const float4 *>(sc.col)[i];
                s_hit[i] = make_float4(cl.w, mt.x, mt.z, 0.f);           // (1/r, reflective, emissive, -)
                s_col[i] = cl;
            }
        }
        for (int k = threadIdx.x; k < 256; k += blockDim.x) s_div255[k] = __ddiv_rn((double)k, 255.0);
        div255 = s_div255;
        S.g.sv.n = sc.n; S.g.sv.n_padded = n_pad; S.g.sv.key_mask = sc.key_mask; S.g.sv.key_mask6 = sc.key_mask6;
        S.g.bvh = sc.bvh;
        hitrec = s_hit;
        S.g.sv.sph = reinterpret_cast<const typename M<T>::v4 *>(s_sph); S.g.sv.mat = sc.mat;
        S.g.sv.col = reinterpret_cast<const typename M<T>::v4 *>(s_col); S.g.sv.pk = sc.pk; S.g.sv.ids = sc.ids; S.g.sv.cw = s_cw;
        S.lb.nL = sc.nL; S.lb.l_pos = sc.l_pos; S.lb.l_col = sc.l_col; S.lb.l_index = sc.l_index; S.lb.lpk = sc.lpk;
        S.la.nG = 0; S.la.nP = 0;
        __syncthreads();
        if constexpr (kIntFold && !M<T>::exact) {
            if (pp.fold_tab) {
                // fold table: entry [sphere][channel][tot] = int(albedo * (tot / 255.0)), the very product the fold evaluates
                // (fold_path_int), computed once per CTA -- four entries per 32-bit store
                uint32_t *tab = reinterpret_cast<uint32_t *>(smem);
                const float *colf = reinterpret_cast<const float *>(s_col);
                for (int q = threadIdx.x; q < sc.n * 192; q += blockDim.x) {
                    const int row = q >> 6, t0 = (q & 63) << 2, sph = row / 3, ch = row - 3 * sph;
                    const double a = (double)colf[4 * sph + ch];
                    uint32_t v = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) v |= ((uint32_t)__double2int_rz(__dmul_rn(a, s_div255[t0 + j])) & 255u) << (8 * j);
                    tab[q] = v;
                }
                __syncthreads();
            }
        }
    } else {
        div255 = reinterpret_cast<double *>(smem);
        for (int k = threadIdx.x; k < 256; k += blockDim.x) div255[k] = __ddiv_rn((double)k, 255.0);
        stage_scene<T, kShared>(sc, smem + 256 * sizeof(double), S);    // ends with __syncthreads() when staging
        if constexpr (!kShared) __syncthreads();
        S.g.sv.cw = nullptr;
    }
    if constexpr (!M<T>::exact && kIntFold) {
        if (pp.sync) {
            // frame protocol, start: rank 0 publishes what its stream has consumed (everything queued before this launch
            // has finished), then every CTA waits until the buffers of this frame's parity are free
            if (threadIdx.x == 0) {
                if (pp.go_epoch != 0u && blockIdx.x == 0)
                    for (int k = 0; k < pp.world; ++k) flag_post(pp.flags[k] + RT_FLAG_GO, pp.go_epoch);
                flag_wait(pp.flags[pp.rank] + RT_FLAG_GO, pp.epoch - 2u, pp.timeout_cycles, pp.timed_out);
            }
            __syncthreads();
        }
    }
    // Sample split: k = 2^ksplit_log2 lanes share one pixel, lane `sub` tracing samples s0 + sub, s0 + sub + k, ...
    // (summed with shuffles at the end).  A warp then covers 32/k pixels -- pw x ph = 8x4, 8x2, 4x2, 2x2, 2x1, 1x1 --
    // and a CTA (4 x 2 warps) 256/k pixels: finer work units for small frames, row bands and sample ranges, so the
    // grid keeps tens of waves and the drain at the end of the launch stays short.
    //
    // The work units of a launch come from TWO tile grids: the coarse one (ksplit_log2) over the first owned stripes and
    // a fine one (ksplit2_log2: four times the lanes per pixel, a quarter of the samples per lane) over the last few.
    // A coarse unit of the headline frame keeps a warp busy for ~160 us, and a launch whose last units are that long ends
    // with every warp idle for 116 us on average (tools/debug/warp_trace.py) -- nothing in a 17-ms frame, 5 % of the
    // 2.2-ms share of one of 8 GPUs; with the fine units last the drain is a quarter of that.  Sums are integers: the
    // frame does not depend on which lanes traced which samples.
    const int w_ = threadIdx.x >> 5, lane_ = threadIdx.x & 31;
    unsigned n_rays = 0, n_inter = 0, n_light = 0, n_small = 0, n_query = 0, n_tests = 0, n_boxes = 0;
    const V3<T> cam = mk<T>(pp.cam[0], pp.cam[1], pp.cam[2]);
    const int ns = pp.s1 - pp.s0;
    PathStack st;
    PathRng rng;
    // PERSISTENT WARPS: the launch has as many CTAs as the device holds at once, and every WARP pulls its next work
    // unit -- one warp tile (32 lanes: 32/k pixels x k sample lanes) of the gx x gy x 8 unit grid -- from a device
    // counter, so the scene staging, the div255 table and the statistics flush are paid once per CTA instead of once
    // per tile, the load balances at warp granularity, and the eight warps of a CTA drift apart freely (no barrier
    // inside the loop).  The first units are static (CTA c, warp w -> unit 8c + w); the counter hands out the rest.
    // A warp asks for its next unit when it has finished the current one: asking before tracing would hide the
    // counter's latency (hidden anyway by 8 warps per scheduler) but leave every warp with two units in hand when the
    // counter runs out -- twice the drain.
    // pp.sched = {next, done}: the last warp of the launch to finish resets both, so no memset precedes a launch.
    const unsigned n_coarse = (unsigned)(pp.gx * pp.gy) << 3, n_units = n_coarse + ((unsigned)(pp.gx2 * pp.gy2) << 3);
    const unsigned first_dyn = (unsigned)gridDim.x << 3;
#ifdef RT_TRACE_WARPS
    const unsigned long long rt_trace_t0 = rt_globaltimer();
    unsigned long long rt_trace_last = 0, rt_trace_unit = 0;
#endif
    for (unsigned unit = ((unsigned)blockIdx.x << 3) + (unsigned)w_; unit < n_units;) {
    RT_ASSERT(unit < n_units);
#ifdef RT_TRACE_WARPS
    rt_trace_last = rt_globaltimer(); rt_trace_unit = unit;
#endif
    const bool fine = unit >= n_coarse;                            // warp-uniform
    const unsigned u_ = fine ? unit - n_coarse : unit;
    const int lk = fine ? pp.ksplit2_log2 : pp.ksplit_log2, kk = 1 << lk;
    const int gx_ = fine ? pp.gx2 : pp.gx, stripe0 = fine ? pp.stripe2 : 0;
    const int pw_sh = unit_pw_log2(lk), ph_sh = (5 - lk) - pw_sh;
    const int sub = lane_ & (kk - 1), pl = lane_ >> lk;
    // CTA rows: cth = 2 << ph_sh of them; tile_step > 1: this launch owns every tile_step-th 8-row stripe from y0
    const int cth_sh = ph_sh + 1, cps_sh = 3 - cth_sh;                 // CTA rows per stripe = 1 << cps_sh
    const int tile = (int)(u_ >> 3), wt = (int)(u_ & 7u);          // wt: the warp's place in the 4 x 2 warp tile
    const int by = tile / gx_, bx = tile - by * gx_;
    const int ys = pp.y0 + (((by >> cps_sh) + stripe0) * pp.tile_step << 3) + ((by & ((1 << cps_sh) - 1)) << cth_sh) +
                   ((wt >> 2) << ph_sh);                           // first row of the warp's pixel block
    // 2-D interleave: in stripe s the launch owns the column segment (col_first + s) mod col_step
    const int xs = (pp.col_step > 1 ? ((pp.col_first + (by >> cps_sh) + stripe0) % pp.col_step) * pp.seg_w : 0) +
                   (((bx << 2) + (wt & 3)) << pw_sh);             // first column of the warp's pixel block
    int x = xs + (pl & ((1 << pw_sh) - 1));
    int y = ys + (pl >> pw_sh);
    bool has_pixel = x < pp.W && y < pp.y1;
    if constexpr (kList) {
        const unsigned e = u_ * (32u >> lk) + (unsigned)pl;
        has_pixel = e < moments.count;
        const unsigned q = has_pixel ? __ldg(moments.list + e) : 0u;
        y = (int)(q / (unsigned)pp.W); x = (int)(q - (unsigned)y * (unsigned)pp.W);
        RT_ASSERT(!has_pixel || (y >= pp.y0 && y < pp.y1));
    }
    const uint32_t pixel = (uint32_t)(y * pp.W + x);
    // integer-valued sums: exact in uint32 (int fold: colours <= 65535, samples per launch <= 65536) / in double
    typename std::conditional<kIntFold, unsigned, double>::type a0 = 0, a1 = 0, a2 = 0;
    typename std::conditional<kIntFold, unsigned long long, double>::type q0 = 0, q1 = 0, q2 = 0;     // kMoments: squares
    // primary rays of this warp tile: spheres its cone of camera rays can touch (cone_candidates, rt_trace.cuh)
    unsigned long long cand = ~0ull;
    bool first_trip = false;                          // warp-uniform: every live lane is about to trace its camera ray
    if constexpr (kMode == 3) if (pp.primary_cull) {
        int bw = 1 << pw_sh, bh = 1 << ph_sh;         // the warp's pixel block
        int x0 = xs;
        int y0 = ys;
        if constexpr (kList) {
            // list launch: the bounding box of the unit's pixels (a scattered unit only widens the cone)
            const unsigned xlo = __reduce_min_sync(0xffffffffu, has_pixel ? (unsigned)x : 0xffffffffu);
            const unsigned ylo = __reduce_min_sync(0xffffffffu, has_pixel ? (unsigned)y : 0xffffffffu);
            const unsigned xhi = __reduce_max_sync(0xffffffffu, has_pixel ? (unsigned)x : 0u);
            const unsigned yhi = __reduce_max_sync(0xffffffffu, has_pixel ? (unsigned)y : 0u);
            if (xlo <= xhi) { x0 = (int)xlo; y0 = (int)ylo; bw = (int)(xhi - xlo) + 1; bh = (int)(yhi - ylo) + 1; }
        }
        const V3<T> d0 = path_camera_ray<T>(pp, x0, y0, T(0.5) * T(bw), T(0.5) * T(bh));
        const float ex = 0.5f * (float)bw * (2.f / (float)pp.W) * (float)pp.aspect * (float)pp.half_w;
        const float ey = 0.5f * (float)bh * (2.f / (float)pp.H) * (float)pp.half_h;
        const float alpha = sqrtf(ex * ex + ey * ey) * 1.001f;      // angle <= distance on the z = -1 plane
        cand = cone_candidates(S.g.sv.sph, S.g.sv.n, cam, d0, alpha, lane_);
    }

    bool none = pp.max_bounces <= 0;                  // degenerate: every call returns (2,2,5) at the depth check
    if constexpr (kMode != 3) none = none || (pp.rays && pp.depth0 >= pp.max_bounces);
    if (none) {
        const int mine = has_pixel ? (ns - sub + kk - 1) >> lk : 0;      // samples of this lane
        n_rays += (unsigned)mine;
        a0 = 2 * mine; a1 = 2 * mine; a2 = 5 * mine;
        if constexpr (kMoments) { q0 = 4 * mine; q1 = 4 * mine; q2 = 25 * mine; }
    } else {
        int s = pp.s0 + sub, depth = 0;
        bool alive = has_pixel && s < pp.s1;          // lane has a path in flight
        V3<T> O = cam, D = mk<T>(T(0), T(0), T(-1));
        // colour at the end of the path: miss / depth limit give Colour(2,2,5), an emissive hit its own colour.  Lives
        // across trips (reset per sample): the fold waits for the warp's longest path.
        int leaf0 = 2, leaf1 = 2, leaf2 = 5;
        double lf0 = 2.0, lf1 = 2.0, lf2 = 5.0;
        bool pend = false;                            // lane traced a sample whose fold is still due
        auto start_sample = [&](int smp) {
            depth = 0; O = cam;
            leaf0 = 2; leaf1 = 2; leaf2 = 5; lf0 = 2.0; lf1 = 2.0; lf2 = 5.0; pend = true;
            if constexpr (kMode != 3) {
                if (pp.rays) {                        // explicit ray (rt_trace_paths): as given, from recursion depth depth0
                    const double *r = pp.rays + 6 * (size_t)pixel;
                    O = mk<T>(T(r[0]), T(r[1]), T(r[2])); D = mk<T>(T(r[3]), T(r[4]), T(r[5]));
                    depth = pp.depth0;
                    rng.begin(pp.ray_ids ? (uint32_t)pp.ray_ids[pixel] : pixel, (uint32_t)smp, pp.k0, pp.k1);
                    n_rays++;
                    return;
                }
            }
            rng.begin(pixel, (uint32_t)smp, pp.k0, pp.k1);
            if constexpr (kMode == 3) if (pp.primary_cull) n_tests += (unsigned)__popcll(cand);
            D = path_sample_ray<T>(pp, rng, x, y);
            n_rays++;                                 // trace_ray_traditional call count, chandelier.py:432
        };
        int fold_from = 0;                            // deepest-first fold stops at the level the path started on
        if constexpr (kMode != 3) fold_from = pp.rays ? pp.depth0 : 0;
        if (alive) start_sample(s);
        first_trip = true;
        for (;;) {
            const bool primary_trip = first_trip;     // this trip traces the camera rays of a sample
            first_trip = false;
            bool ended = false;
            int i = -1;
            if constexpr (kMode == 3) {
                // the selection runs on the CONVERGED warp (its pair votes take the full mask): a lane without a path in
                // flight goes through the arithmetic on its stale ray and votes "no"; its result is never read
                if (primary_trip && pp.primary_cull) i = select_candidates(S.g.sv.cw, cand, S.g.sv.key_mask6, O, D);
                else i = brute_select_pkc<true>(pkc, S.g.sv.n_padded, S.g.sv.key_mask6, O, D, alive);
            }
            if (alive) {
                // ---- one call of trace_ray_traditional below the depth limit: a nearest-hit query
                T t;
                n_query++;
                typename M<T>::v4 m;                   // material: (reflective, transparent, emissive, ior)
                T inv_r = T(0);
                V3<T> centre = mk<T>(T(0), T(0), T(0));
                if constexpr (kMode == 3) {
                    // one LDS.128 for the winner's (centre, r) -- shared by the robust distance and the normal -- and one
                    // for its (1/r, reflective, emissive) record
                    // sphere tests: the kernel counts the camera rays' candidates once per sample (start_sample) and
                    // derives the full-scene queries at the end of the launch (no counter update per trip)
                    if (i >= 0) {
                        float4 w, hr;
                        lds_v4x2<16 * RT_PKC_MAX>(s_base + 16u * (unsigned)i, w, hr);      // (centre, r) and (1/r, reflective, emissive)
                        t = winner_distance(w, O, D);
                        centre = mk<T>(w.x, w.y, w.z); inv_r = hr.x;
                        m.x = hr.y; m.y = T(0); m.z = hr.z; m.w = T(1);
                    }
                } else {
                    i = nearest<T, true, kBvh, PK>(S.g, O, D, RT_NO_ID_DEV, t, n_tests, n_boxes, pkc);
                    if (i >= 0) m = S.g.sv.mat[i];
                }
                if (i < 0) ended = true;
                else {
                    n_inter++;
                    if (m.z != T(0)) {                                               // emissive: its own colour
                        n_light++;
                        if (sc.small && sc.small[i]) n_small++;
                        typename M<T>::v4 col;
                        if constexpr (kMode == 3) col = lds_v4(s_base + 32u * RT_PKC_MAX + 16u * (unsigned)i);
                        else col = S.g.sv.col[i];
                        if constexpr (kIntFold) { leaf0 = (int)col.x; leaf1 = (int)col.y; leaf2 = (int)col.z; }
                        else { lf0 = (double)col.x; lf1 = (double)col.y; lf2 = (double)col.z; }
                        ended = true;
                    } else {
                        Hit<T> h;
                        if constexpr (kMode == 3) { h.idx = i; h.t = t; h.p = O + D * t; h.n = (h.p - centre) * inv_r; }
                        else finish_hit<T>(S.g, O, D, i, t, h);
                        RT_ASSERT(depth >= 0 && depth < RT_PATH_MAX_DEPTH && i < sc.n);
                        if constexpr (kMode != 3) st.idx[depth] = (uint32_t)i;
                        if constexpr (M<T>::exact) st.direct[depth] = direct_light<T>(S.lb, i, h.p, h.n);
                        else if constexpr (kMode == 3)       // one stack word per level: sphere index above the 24 colour bits
                            st.direct[depth] = direct_light_pkc(pkc, S.lb.nL, h.p, h.n) | ((uint32_t)i << 24);
                        else st.direct[depth] = direct_light_pk(S.lb.lpk, (S.lb.nL + 1) >> 1, h.p, h.n);
                        depth++;
                        n_rays++;                                                    // the recursive call ...
                        ended = depth >= pp.max_bounces;                             // ... returns (2,2,5) at once
                        // the bounce ray of the deepest level is never traced (counter-based RNG: skipping its
                        // draw changes nothing), so its direction is not computed either
                        if (!ended) {
                            const bool mirror = m.x > pp.mirror_threshold;
                            T r1 = T(0), r2 = T(0);
                            // (measured: letting mirror lanes fill the two-slot Philox cache at even depths, so that they
                            // need not recompute the block alone one trip later, gains 0.4 % on the complex scene and
                            // LOSES 3.5 % on the chandelier, where most surfaces mirror and the rounds would run for nobody)
                            if (!mirror) {
                                uint32_t wa, wb;
                                rng.pair_rk((uint32_t)depth, wa, wb, pp.rk);
                                r1 = u01<T>(wa); r2 = u01<T>(wb);
                            }
                            D = bounce_direction<T>(D, h.n, mirror, r1, r2);
                            O = h.p + h.n * T(0.001);
                        }
                    }
                }
            }
            // a lane whose path ends early only parks its leaf; the whole warp folds together once the sample's longest
            // path has ended (one full-occupancy fold instead of several sparse ones)
            if (ended) alive = false;                 // (ended is only ever set by a live lane)
            if (__any_sync(0xffffffffu, alive)) continue;
            if (pend) {
                pend = false;
                if constexpr (kIntFold) {
                    int c[3] = {leaf0, leaf1, leaf2};
                    fold_path_int<T, kMode == 3>(S.g, st, depth, div255, c, fold_from, s_base + 32u * RT_PKC_MAX,
                                                 (kMode == 3 && pp.fold_tab) ? (unsigned)__cvta_generic_to_shared(smem) : 0u);
                    a0 += (unsigned)c[0]; a1 += (unsigned)c[1]; a2 += (unsigned)c[2];
                    if constexpr (kMoments) {
                        q0 += (unsigned long long)((unsigned)c[0] * (unsigned)c[0]);
                        q1 += (unsigned long long)((unsigned)c[1] * (unsigned)c[1]);
                        q2 += (unsigned long long)((unsigned)c[2] * (unsigned)c[2]);
                    }
                } else {
                    double c[3] = {lf0, lf1, lf2};
                    fold_path<T, kMode == 3>(S.g, st, depth, c, fold_from);
                    a0 += c[0]; a1 += c[1]; a2 += c[2];
                    if constexpr (kMoments) { q0 += __dmul_rn(c[0], c[0]); q1 += __dmul_rn(c[1], c[1]); q2 += __dmul_rn(c[2], c[2]); }
                }
            }
            s += kk;
            if (s - sub >= pp.s1) break;              // s - sub is warp-uniform
            if (has_pixel && s < pp.s1) { alive = true; start_sample(s); }
            first_trip = true;
        }
    }
    if constexpr (kIntFold) {                        // the k lanes of a pixel are adjacent: butterfly sum
        for (int o = 1; o < kk; o <<= 1) {
            a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o);
            a2 += __shfl_xor_sync(0xffffffffu, a2, o);
            if constexpr (kMoments) {
                q0 += __shfl_xor_sync(0xffffffffu, q0, o); q1 += __shfl_xor_sync(0xffffffffu, q1, o);
                q2 += __shfl_xor_sync(0xffffffffu, q2, o);
            }
        }
    }
    if (has_pixel && ns > 0 && sub == 0) {
        const size_t o = (size_t)y * pp.W + x;
        RT_ASSERT(x >= 0 && x < pp.W && y >= pp.y0 && y < pp.y1 && y < pp.H);
        bool to_accum = true;
        if constexpr (!M<T>::exact && kIntFold) {
            if (pp.sink == 1) {
                // tile sharding: the resolved pixel goes straight to the final image (possibly a peer mapping)
                const double s = (double)pp.spp_total;
                const double r = floor((double)a0 / s) / 255.0, g = floor((double)a1 / s) / 255.0, b = floor((double)a2 / s) / 255.0;
                float *px = pp.image + 3 * o;
                px[0] = (float)(r < 1.0 ? r : 1.0); px[1] = (float)(g < 1.0 ? g : 1.0); px[2] = (float)(b < 1.0 ? b : 1.0);
                if constexpr (kMoments) {
                    // the variance rt_resolve_variance would give: S as the float accum would hold it, k = ns = spp_total
                    float *pv = moments.var + 3 * o;
                    pv[0] = variance_of_mean((double)(float)a0, (double)q0, (double)ns);
                    pv[1] = variance_of_mean((double)(float)a1, (double)q1, (double)ns);
                    pv[2] = variance_of_mean((double)(float)a2, (double)q2, (double)ns);
                }
                to_accum = false;
            } else if (pp.sink == 2) {
                // sample sharding: one 16-byte system-scope reduction into the accumulators of the pixel's owner
                int k = min(pp.world - 1, (int)(((long long)y * pp.world) / pp.H));
                while (y >= pp.band_y[k + 1]) ++k;
                while (y < pp.band_y[k]) --k;
                RT_ASSERT(k >= 0 && k < pp.world && y >= pp.band_y[k] && y < pp.band_y[k + 1]);
                float4 *dst = pp.peer_accum[k] + o;
                asm volatile("red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};"
                             :: "l"(dst), "f"((float)a0), "f"((float)a1), "f"((float)a2), "f"((float)ns) : "memory");
                if constexpr (kMoments) {
                    // the squares beside them: no vector f64 reduction exists, so four scalar ones; integer-valued
                    // doubles below 2^53 (DESIGN.md 4.8a), exact in any order
                    double *qd = reinterpret_cast<double *>(moments.peer[k] + o);
                    asm volatile("red.relaxed.sys.global.add.f64 [%0], %1;" :: "l"(qd), "d"((double)q0) : "memory");
                    asm volatile("red.relaxed.sys.global.add.f64 [%0], %1;" :: "l"(qd + 1), "d"((double)q1) : "memory");
                    asm volatile("red.relaxed.sys.global.add.f64 [%0], %1;" :: "l"(qd + 2), "d"((double)q2) : "memory");
                    asm volatile("red.relaxed.sys.global.add.f64 [%0], %1;" :: "l"(qd + 3), "d"((double)ns) : "memory");
                }
                to_accum = false;
            }
        }
        if (to_accum) {
            typename M<T>::v4 out = M<T>::make4(T(a0), T(a1), T(a2), T(ns));
            if (pp.accumulate) {
                const typename M<T>::v4 old = accum[o];
                out.x += old.x; out.y += old.y; out.z += old.z; out.w += old.w;
            }
            accum[o] = out;
            if constexpr (kMoments) {
                double4 m = make_double4((double)q0, (double)q1, (double)q2, (double)ns);
                if (pp.accumulate) {
                    const double4 old = moments.local[o];
                    m.x += old.x; m.y += old.y; m.z += old.z; m.w += old.w;
                }
                moments.local[o] = m;
            }
        }
    }
    unsigned nxt = 0;
    if (lane_ == 0) nxt = first_dyn + atomicAdd(pp.sched, 1u);
    unit = __shfl_sync(0xffffffffu, nxt, 0);
    }   // work units of this warp
#ifdef RT_TRACE_WARPS
    // development build (tools/debug/warp_trace.py): when every warp entered its unit loop and when it left it, in ns
    if (pp.timed_out && !pp.sync && lane_ == 0) {
        unsigned long long *tr = reinterpret_cast<unsigned long long *>(pp.timed_out) + 4 * ((size_t)blockIdx.x * 8 + w_);
        tr[0] = rt_trace_t0; tr[1] = rt_globaltimer(); tr[2] = rt_trace_last; tr[3] = rt_trace_unit;
    }
#endif
    bool sync = false;
    if constexpr (!M<T>::exact && kIntFold) sync = pp.sync != 0;
    if (lane_ == 0) {
        // every warp of the launch passes here exactly once, after its last fetch: the last one re-arms the counters
        // and, under the frame protocol, publishes this rank's part (its peer writes, and through the fence + counter
        // chain those of every other warp, are ordered before the release stores; the system fence orders the kMoments
        // f64 reductions into the owners' moments as it orders the f32 ones into their accumulators)
        if (sync) __threadfence_system(); else __threadfence();
        if (atomicAdd(pp.sched + 1, 1u) == (gridDim.x << 3) - 1u) {
            if (sync) {
                __threadfence_system();
                if (pp.sink == 1) flag_post(pp.flags[0] + RT_FLAG_DONE + pp.rank, pp.epoch);
                else for (int k = 0; k < pp.world; ++k) flag_post(pp.flags[k] + RT_FLAG_ADDED + pp.rank, pp.epoch);
            }
            pp.sched[0] = 0u; pp.sched[1] = 0u; __threadfence();
        }
    }
    if constexpr (!M<T>::exact && kIntFold) {
        if (sync) {
            __syncthreads();                          // the CTA's eight warps have all finished their units
            if (pp.sink == 2) {
                // resolve: once every rank's sums have arrived in this rank's band, turn it into pixels of rank 0's
                // image and clear it for the frame after next; the launch's CTAs share the band
                if ((int)threadIdx.x < pp.world) flag_wait(pp.flags[pp.rank] + RT_FLAG_ADDED + threadIdx.x, pp.epoch, pp.timeout_cycles, pp.timed_out);
                __syncthreads();
                float4 *own = pp.peer_accum[pp.rank];
                const size_t first = (size_t)pp.band_y[pp.rank] * pp.W, count = (size_t)(pp.band_y[pp.rank + 1] - pp.band_y[pp.rank]) * pp.W;
                const double spp = (double)pp.spp_total;
                for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
                    const size_t o = first + i;
                    RT_ASSERT(o < (size_t)pp.W * pp.H && a_count_ok(pp.spp_total));
                    const float4 a = __ldcg(own + o);                  // L2: where the peers' reductions landed
                    RT_ASSERT(a.w == (float)pp.spp_total);            // every rank's sums arrived before the flags said so
                    const double r = floor((double)a.x / spp) / 255.0, g = floor((double)a.y / spp) / 255.0, b = floor((double)a.z / spp) / 255.0;
                    float *px = pp.image + 3 * o;
                    px[0] = (float)(r < 1.0 ? r : 1.0); px[1] = (float)(g < 1.0 ? g : 1.0); px[2] = (float)(b < 1.0 ? b : 1.0);
                    __stcg(own + o, make_float4(0.f, 0.f, 0.f, 0.f));
                    if constexpr (kMoments) {
                        // the own band of the moments -> rank 0's variance image, as rt_resolve_variance would
                        // resolve the reduced frame; cleared for the frame after next like the sums
                        double2 *qo = reinterpret_cast<double2 *>(moments.peer[pp.rank] + o);
                        const double2 qa = __ldcg(qo), qb = __ldcg(qo + 1);
                        RT_ASSERT(qb.y == (double)pp.spp_total);
                        float *pv = moments.var + 3 * o;
                        pv[0] = variance_of_mean((double)a.x, qa.x, qb.y);
                        pv[1] = variance_of_mean((double)a.y, qa.y, qb.y);
                        pv[2] = variance_of_mean((double)a.z, qb.x, qb.y);
                        __stcg(qo, make_double2(0.0, 0.0)); __stcg(qo + 1, make_double2(0.0, 0.0));
                    }
                }
                __syncthreads();
                if (threadIdx.x == 0) {
                    __threadfence_system();
                    if (atomicAdd(pp.sched + 2, 1u) == gridDim.x - 1u) {
                        pp.sched[2] = 0u;
                        __threadfence_system();
                        flag_post(pp.flags[0] + RT_FLAG_DONE + pp.rank, pp.epoch);
                    }
                }
            }
            // collect: rank 0's launch ends when every rank's part of the image is in place
            if (pp.rank == 0 && blockIdx.x == 0 && (int)threadIdx.x < pp.world)
                flag_wait(pp.flags[0] + RT_FLAG_DONE + threadIdx.x, pp.epoch, pp.timeout_cycles, pp.timed_out);
        }
    }
    if (stats) {
        flush_stats(stats, STAT_RAYS, n_rays);
        flush_stats(stats, STAT_INTER, n_inter);
        flush_stats(stats, STAT_LIGHT, n_light);
        flush_stats(stats, STAT_SMALL, n_small);
        flush_stats(stats, STAT_QUERIES, n_query);
        unsigned long long tests = n_tests;
        if constexpr (kMode == 3) {
            // every query but the camera rays' (when those walk their candidate lists) tests the whole scene; a camera
            // ray is a trace call that no hit caused: n_rays - (n_inter - n_light)
            unsigned n_prim = 0u;
            if (pp.primary_cull) n_prim = n_rays - (n_inter - n_light);
            tests += (unsigned long long)(n_query - min(n_prim, n_query)) * (unsigned)sc.n;
        }
        flush_stats(stats, STAT_SPHERE_TESTS, tests);
        flush_stats(stats, STAT_AABB_TESTS, n_boxes);
    }
}

// ------------------------------------------------------------------ "Algorithm C" frame (FB/output6.py)
// SimplifiedFBRenderer.calculate_lighting_exact_original (output6.py:197-306).  The final int(colour * (combined /
// 255.0)) is evaluated in double in both builds: for colour 255 the product is an exact integer and a float
// reciprocal would truncate one level low.
template <typename T>
RT_DEV void simple_lighting(const Geo<T> &g, const SimpleDev<T> &sp, const Hit<T> &h, int out[3], unsigned &sun_hits,
                            unsigned &tests) {
    if (g.sv.ids[h.idx] == sp.sun_id) {                                          // :204-206
        sun_hits++;
        out[0] = (int)sp.sun_col[0]; out[1] = (int)sp.sun_col[1]; out[2] = (int)sp.sun_col[2];
        return;
    }
    const V3<T> sun = mk<T>(sp.sun_pos[0], sp.sun_pos[1], sp.sun_pos[2]);
    const V3<T> to_sun = normalise(sun - h.p);                                   // :244
    const V3<T> gdir = normalise(mk<T>(T(3), T(1), T(-0.75)));                   // :247
    T gcos = dot(h.n, gdir);
    if (!(gcos > T(0))) gcos = T(0);
    int gc[3], su[3] = {0, 0, 0};
    gc[0] = (int)(T(20) * gcos * T(0.3)); gc[1] = gc[0]; gc[2] = (int)(T(255) * gcos * T(0.3));   // :250-254
    const V3<T> so = h.p + h.n * T(0.001);                                        // :258-261
    const V3<T> sd = M<T>::exact ? normalise(to_sun) : to_sun;
    const V3<T> dv = h.p - sun;
    const T sun_distance = M<T>::sqrt(dot(dv, dv));                               // :264
    bool visible = true;
    for (int i = 0; i < g.sv.n && visible; ++i) {                                 // :266-275
        if (i == h.idx || g.sv.ids[i] == sp.sun_id) continue;
        T t;
        tests++;
        if (!sphere_test<T>(so, sd, g.sv.sph[i], 0, t)) continue;
        const V3<T> q = (so + sd * t) - h.p;
        if (M<T>::sqrt(dot(q, q)) < sun_distance) visible = false;
    }
    if (visible) {                                                                // :278-291
        T att = sun_distance > T(0) ? T(1) / (sun_distance * sun_distance) : T(1);
        att = att * T(100) < T(1) ? att * T(100) : T(1);
        T ca = dot(h.n, to_sun);
        if (!(ca > T(0))) ca = T(0);
        su[0] = (int)(sp.sun_col[0] * ca * att * T(0.9)); su[1] = (int)(sp.sun_col[1] * ca * att * T(0.9));
        su[2] = (int)(sp.sun_col[2] * ca * att * T(0.9));
    }
    const typename M<T>::v4 col = g.sv.col[h.idx];
    const double c3[3] = {(double)col.x, (double)col.y, (double)col.z};
#pragma unroll
    for (int k = 0; k < 3; ++k) {                                                 // :293-304
        const int comb = min(255, gc[k] + su[k]);
        out[k] = (int)__dmul_rn(c3[k], __ddiv_rn((double)comb, 255.0));
    }
}

// SimplifiedFBRenderer.trace_ray_simple + render_original_style (output6.py:434-577, :579-635): one thread per pixel
// (8x4 warp tiles) or per explicit ray.
template <typename T, int kMode>
__global__ void __launch_bounds__(256) simple_kernel(SceneDev<T> sc, SimpleDev<T> sp, int4 *rgb, float *image,
                                                     unsigned long long *stats) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    int x, y, i;
    bool active;
    if (sp.rays) {
        i = blockIdx.x * blockDim.x + threadIdx.x; x = y = 0;
        active = i < sp.n;
    } else {
        tile_pixel(x, y);
        active = x < sp.W && y < sp.H;
        i = y * sp.W + x;
    }
    unsigned n_rays = 0, n_sun = 0, n_query = 0, n_tests = 0, n_boxes = 0;
    if (active && sp.lighting_only) {                 // calculate_lighting_exact_original on a given intersection
        const double *r = sp.rays + 7 * (size_t)i;
        Hit<T> h;
        h.idx = (int)r[6]; h.t = T(0); h.bounces = 0; h.through = 0;
        h.p = mk<T>(T(r[0]), T(r[1]), T(r[2])); h.n = mk<T>(T(r[3]), T(r[4]), T(r[5]));
        int li[3] = {0, 0, 0};
        if (h.idx >= 0 && h.idx < S.g.sv.n) { simple_lighting<T>(S.g, sp, h, li, n_sun, n_tests); n_query++; }
        rgb[i] = make_int4(li[0], li[1], li[2], 0);
    } else if (active) {
        V3<T> O, D;
        if (sp.rays) {
            const double *r = sp.rays + 6 * (size_t)i;
            O = mk<T>(T(r[0]), T(r[1]), T(r[2]));
            D = normalise(mk<T>(T(r[3]), T(r[4]), T(r[5])));
        } else {
            T u = (T(x) / T(sp.W) - T(0.5)) * T(2), v = (T(y) / T(sp.H) - T(0.5)) * T(-2);       // :612-613
            u *= sp.aspect;                                                                      // :616-617
            D = normalise(mk<T>(u * sp.tan_half, v * sp.tan_half, T(-1)));                       // :621
            if constexpr (M<T>::exact) D = normalise(D);                                         // Ray() normalises again
            O = mk<T>(sp.cam[0], sp.cam[1], sp.cam[2]);
        }
        int acc[3] = {0, 0, 0};
        int bounce = 0;
        while (bounce < sp.max_bounces) {
            n_rays++; n_query++;
            T t;
            const int hi = nearest<T, true, kBvh>(S.g, O, D, RT_NO_ID_DEV, t, n_tests, n_boxes);
            if (hi < 0) { if (bounce == 0) { acc[0] = 2; acc[1] = 2; acc[2] = 5; } break; }      // :459-463
            Hit<T> h;
            finish_hit<T>(S.g, O, D, hi, t, h);
            int li[3];
            simple_lighting<T>(S.g, sp, h, li, n_sun, n_tests);
            n_query++;
            acc[0] = min(255, acc[0] + li[0]); acc[1] = min(255, acc[1] + li[1]); acc[2] = min(255, acc[2] + li[2]);
            if (S.g.sv.ids[hi] == sp.sun_id) break;                                              // :479-480
            const typename M<T>::v4 m = S.g.sv.mat[hi];
            V3<T> nd;
            if (m.x != T(0)) nd = reflect<T>(D, h.n);                                            // truthy reflective
            else if (m.y != T(0)) {                                                              // glass: 50/50
                const Philox4 o = philox4x32_10((uint32_t)i, 0u, ((uint32_t)bounce + 1u) >> 1, RT_PHILOX_TAG, sp.k0, sp.k1);
                const uint32_t wa = ((bounce + 1) & 1) ? o.w[2] : o.w[0];
                nd = u01<T>(wa) < T(0.5) ? reflect<T>(D, h.n) : D;
            } else {
                const Philox4 o = philox4x32_10((uint32_t)i, 0u, ((uint32_t)bounce + 1u) >> 1, RT_PHILOX_TAG, sp.k0, sp.k1);
                const bool odd = (bounce + 1) & 1;
                nd = bounce_direction<T>(D, h.n, false, u01<T>(odd ? o.w[2] : o.w[0]), u01<T>(odd ? o.w[3] : o.w[1]));
            }
            O = h.p + h.n * T(0.001);                                                            // :567-570
            D = M<T>::exact ? normalise(nd) : nd;
            bounce++;
        }
        rgb[i] = make_int4(acc[0], acc[1], acc[2], bounce);
        if (image) {
            float *px = image + 3 * (size_t)i;
            px[0] = fminf(1.f, (float)((double)acc[0] / 255.0)); px[1] = fminf(1.f, (float)((double)acc[1] / 255.0));
            px[2] = fminf(1.f, (float)((double)acc[2] / 255.0));
        }
    }
    if (stats) {
        flush_stats(stats, STAT_RAYS, n_rays);
        flush_stats(stats, STAT_INTER, n_sun);
        flush_stats(stats, STAT_QUERIES, n_query);
        flush_stats(stats, STAT_SPHERE_TESTS, n_tests);
        flush_stats(stats, STAT_AABB_TESTS, n_boxes);
    }
}

// ------------------------------------------------------------------ FB training trajectories (train_complex_only.py)
// sample_cosine_weighted_direction / direction_to_action basis (train_complex_only.py:84-89): |n.z| < 0.999 picks
// (0,0,1) x n, unlike the renderers' |n.z| > 0.9 rule.
template <typename T> RT_DEV void traj_basis(V3<T> n, V3<T> &tg, V3<T> &bt) {
    tg = M<T>::fabs(n.z) < T(0.999) ? normalise(cross(mk<T>(0, 0, 1), n)) : normalise(cross(mk<T>(1, 0, 0), n));
    bt = normalise(cross(n, tg));
}
template <typename T> RT_DEV V3<T> traj_cosine_dir(V3<T> n, T r1, T r2, V3<T> &tg, V3<T> &bt) {
    T st, ct, sp, cp;
    if constexpr (M<T>::exact) {
        const T theta = ::acos(::sqrt(r1)), phi = 2 * 3.14159265358979323846 * r2;
        st = ::sin(theta); ct = ::cos(theta); sp = ::sin(phi); cp = ::cos(phi);
    } else {
        ct = M<T>::sqrt(r1); st = M<T>::sqrt(1.f - r1);
        sincospif(2.f * r2, &sp, &cp);
    }
    traj_basis<T>(n, tg, bt);
    const T lx = st * cp, ly = st * sp, lz = ct;
    return normalise(mk<T>(lx * tg.x + ly * bt.x + lz * n.x, lx * tg.y + ly * bt.y + lz * n.y, lx * tg.z + ly * bt.z + lz * n.z));
}
// create_observation (train_complex_only.py:130-150)
template <typename T>
RT_DEV void traj_obs(const Geo<T> &g, V3<T> p, V3<T> n, V3<T> d, int bounce, T c0, T c1, T c2, int idx, int max_bounces, float *o) {
    const typename M<T>::v4 m = g.sv.mat[idx];
    o[0] = (float)p.x; o[1] = (float)p.y; o[2] = (float)p.z; o[3] = (float)d.x; o[4] = (float)d.y; o[5] = (float)d.z;
    o[6] = (float)n.x; o[7] = (float)n.y; o[8] = (float)n.z;
    o[9] = (float)m.x; o[10] = (float)m.y; o[11] = (float)m.z; o[12] = (float)m.w;
    o[13] = (float)(c0 / T(255)); o[14] = (float)(c1 / T(255)); o[15] = (float)(c2 / T(255));
    o[16] = (float)(T(bounce) / T(max_bounces)); o[17] = 0.f; o[18] = (float)(T(g.sv.ids[idx]) / T(100));
    o[19] = 0.5f; o[20] = 0.5f; o[21] = 0.5f;
}
// RayTracedComplexTrainer.generate_trajectory (train_complex_only.py:254-334): one thread per trajectory.
template <typename T, int kMode>
__global__ void __launch_bounds__(128) trajectory_kernel(SceneDev<T> sc, int n_traj, int max_steps, int max_bounces,
                                                         uint32_t k0, uint32_t k1, float *obs, float *action,
                                                         float *next_obs, float *reward, uint8_t *hit, int *length,
                                                         uint8_t *hit_light, unsigned long long *stats) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned n_query = 0, n_tests = 0, n_boxes = 0;
    if (j < n_traj) {
        int len = 0, lit_any = 0;
        int nl = 0;
        for (int i = 0; i < S.g.sv.n; ++i) nl += S.g.sv.mat[i].z == T(0);
        if (nl > 0) {
            PathRng rng;
            rng.begin((uint32_t)j, 0u, k0, k1);
            uint32_t wa, wb, wc, wd;
            rng.pair(0u, wa, wb);
            rng.pair(1u, wc, wd);
            int pick = min(nl - 1, (int)(u01<T>(wa) * T(nl)));                               // random.choice(non_light)
            int idx = 0;
            for (int i = 0; i < S.g.sv.n; ++i) if (S.g.sv.mat[i].z == T(0) && pick-- == 0) { idx = i; break; }
            const T th = T(2 * 3.14159265358979323846) * u01<T>(wb), ph = T(3.14159265358979323846) * u01<T>(wc);
            T sth, cth, sph_, cph;
            M<T>::sincos(th, &sth, &cth); M<T>::sincos(ph, &sph_, &cph);
            const typename M<T>::v4 s0 = S.g.sv.sph[idx];
            const V3<T> off = mk<T>(sph_ * cth, sph_ * sth, cph) * s0.w;                      // scaleByLength(radius)
            V3<T> p = centre_of<T>(s0) + off, n = normalise(off);
            V3<T> tg, bt;
            rng.pair(2u, wa, wb);
            const V3<T> din = traj_cosine_dir<T>(n, u01<T>(wa), u01<T>(wb), tg, bt);
            float cur[22];
            traj_obs<T>(S.g, p, n, din, 0, T(0), T(0), T(0), idx, max_bounces, cur);
            int bounce = 0;
            while (bounce < max_steps) {
                rng.pair(3u + (uint32_t)bounce, wa, wb);
                const V3<T> nd = traj_cosine_dir<T>(n, u01<T>(wa), u01<T>(wb), tg, bt);
                // direction_to_action (:99-127)
                const T lx = dot(nd, tg), ly = dot(nd, bt), lz = dot(nd, n);
                T cz = lz > T(1) ? T(1) : lz;
                if (cz < T(-1)) cz = T(-1);
                T theta, phi;
                if constexpr (M<T>::exact) { theta = ::acos(cz); phi = ::atan2(ly, lx); }
                else { theta = acosf(cz); phi = atan2f(ly, lx); }
                const T half_pi = T(3.14159265358979323846 / 2);
                if (theta > half_pi) theta = half_pi;
                const float a0 = (float)((theta / half_pi) * T(2) - T(1)), a1 = (float)(phi / T(3.14159265358979323846));
                const V3<T> ro = p + n * T(0.001);
                const V3<T> rd = M<T>::exact ? normalise(nd) : nd;                            // Ray() normalises again
                T t;
                n_query++;
                const int hi = nearest<T, true, kBvh>(S.g, ro, rd, S.g.sv.ids[idx], t, n_tests, n_boxes);
                if (hi < 0) break;                                                           // ray escaped
                Hit<T> h;
                finish_hit<T>(S.g, ro, rd, hi, t, h);
                const size_t tr = (size_t)j * max_steps + len;
                const bool lit = S.g.sv.mat[hi].z != T(0);
                float *po = obs + 22 * tr, *pn = next_obs + 22 * tr;
                // 22 floats = 88 bytes per record, 8-byte aligned for every transition index: eleven 8-byte stores
#pragma unroll
                for (int k = 0; k < 11; ++k) reinterpret_cast<float2 *>(po)[k] = make_float2(cur[2 * k], cur[2 * k + 1]);
                action[2 * tr] = a0; action[2 * tr + 1] = a1;
                const typename M<T>::v4 col = S.g.sv.col[hi];
                traj_obs<T>(S.g, h.p, h.n, rd, bounce + 1, lit ? col.x : T(0), lit ? col.y : T(0), lit ? col.z : T(0), hi,
                            max_bounces, cur);
#pragma unroll
                for (int k = 0; k < 11; ++k) reinterpret_cast<float2 *>(pn)[k] = make_float2(cur[2 * k], cur[2 * k + 1]);
                reward[tr] = lit ? 1.f : 0.f; hit[tr] = (uint8_t)lit;
                len++;
                if (lit) { lit_any = 1; break; }
                p = h.p; n = h.n; idx = hi;
                bounce++;
            }
        }
        length[j] = len; hit_light[j] = (uint8_t)lit_any;
    }
    if (stats) {
        flush_stats(stats, STAT_QUERIES, n_query);
        flush_stats(stats, STAT_SPHERE_TESTS, n_tests);
        flush_stats(stats, STAT_AABB_TESTS, n_boxes);
    }
}

// ------------------------------------------------------------------ resolve
// pixel // spp then min(1, /255) (chandelier.py:540-549; output5.py:1500-1512)
template <typename T>
__global__ void resolve_kernel(const typename M<T>::v4 *accum, int W, int y0, int y1, int spp, float *image) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t n = (size_t)(y1 - y0) * W;
    if (i >= n) return;
    const size_t o = (size_t)y0 * W + i;
    const typename M<T>::v4 a = accum[o];
    const double s = (double)spp;
    double r = floor((double)a.x / s) / 255.0, g = floor((double)a.y / s) / 255.0, b = floor((double)a.z / s) / 255.0;
    image[3 * o + 0] = (float)(r < 1.0 ? r : 1.0);
    image[3 * o + 1] = (float)(g < 1.0 ? g : 1.0);
    image[3 * o + 2] = (float)(b < 1.0 ? b : 1.0);
}

// variance of the pixel's mean in colour levels^2 (variance_of_mean) from the sums S (accum) and the sums of squares Q
// (moments) of its n samples
template <typename T>
__global__ void resolve_variance_kernel(const typename M<T>::v4 *accum, const double4 *moments, int W, int y0, int y1,
                                        float *var) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t n = (size_t)(y1 - y0) * W;
    if (i >= n) return;
    const size_t o = (size_t)y0 * W + i;
    const typename M<T>::v4 a = accum[o];
    const double4 q = moments[o];
    const double k = q.w, S[3] = {(double)a.x, (double)a.y, (double)a.z}, Q[3] = {q.x, q.y, q.z};
#pragma unroll
    for (int c = 0; c < 3; ++c) var[3 * o + c] = variance_of_mean(S[c], Q[c], k);
}

// ------------------------------------------------------------------ adaptive frames (rt_render_path_adaptive)
// After the round that took every active pixel of rows [y0, y1) to c samples: a pixel stays active when it was active
// in that round (n == c) and the variance of its mean (variance_of_mean, the float rt_resolve_variance gives, compared in
// double) exceeds thr in some channel.  Active pixels y * W + x are appended to list with one atomic per warp; a warp
// covers an 8x4 tile (tile_pixel), so neighbours stay adjacent in the list.  *count is zero on entry.
template <typename T>
__global__ void adaptive_select_kernel(const typename M<T>::v4 *accum, const double4 *moments, int W, int y0, int y1, int c,
                                       double thr, uint32_t *list, uint32_t *count) {
    int x, y_rel;
    tile_pixel(x, y_rel);
    const int y = y0 + y_rel;
    bool active = false;
    if (x < W && y < y1) {
        const size_t o = (size_t)y * W + x;
        const typename M<T>::v4 a = accum[o];
        const double4 q = moments[o];
        RT_ASSERT(q.w == (double)a.w);
        if ((double)a.w == (double)c)
            active = (double)variance_of_mean((double)a.x, q.x, q.w) > thr || (double)variance_of_mean((double)a.y, q.y, q.w) > thr ||
                     (double)variance_of_mean((double)a.z, q.z, q.w) > thr;
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, active), lane = threadIdx.x & 31;
    if (ballot == 0u) return;
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(count, (unsigned)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (active) list[base + (unsigned)__popc(ballot & ((1u << lane) - 1u))] = (uint32_t)(y * W + x);
}

// the adaptive frame's resolve: each pixel by its own sample count n = accum.w -- image min(1, floor(S/n)/255) as
// resolve_kernel, the variance as resolve_variance_kernel (var optional), n into counts (optional)
template <typename T>
__global__ void adaptive_resolve_kernel(const typename M<T>::v4 *accum, const double4 *moments, int W, int y0, int y1,
                                        float *image, float *var, int *counts) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t n = (size_t)(y1 - y0) * W;
    if (i >= n) return;
    const size_t o = (size_t)y0 * W + i;
    const typename M<T>::v4 a = accum[o];
    const double s = (double)a.w;
    double r = floor((double)a.x / s) / 255.0, g = floor((double)a.y / s) / 255.0, b = floor((double)a.z / s) / 255.0;
    image[3 * o + 0] = (float)(r < 1.0 ? r : 1.0);
    image[3 * o + 1] = (float)(g < 1.0 ? g : 1.0);
    image[3 * o + 2] = (float)(b < 1.0 ? b : 1.0);
    if (var) {
        const double4 q = moments[o];
        var[3 * o + 0] = variance_of_mean((double)a.x, q.x, q.w);
        var[3 * o + 1] = variance_of_mean((double)a.y, q.y, q.w);
        var[3 * o + 2] = variance_of_mean((double)a.z, q.z, q.w);
    }
    if (counts) counts[o] = (int)a.w;
}

// ------------------------------------------------------------------ batched primitives
template <typename T>
__global__ void sphere_disc_kernel(int m, const double *rays, const double *spheres, int point, double *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const double *r = rays + 6 * (size_t)i, *s = spheres + 4 * (size_t)i;
    V3<T> O = mk<T>(T(r[0]), T(r[1]), T(r[2]));
    V3<T> D = normalise(mk<T>(T(r[3]), T(r[4]), T(r[5])));
    typename M<T>::v4 sp = M<T>::make4(T(s[0]), T(s[1]), T(s[2]), T(s[3]));
    T t;
    double *o = out + 8 * (size_t)i;
    if (!sphere_test<T>(O, D, sp, point, t)) { for (int k = 0; k < 8; ++k) o[k] = 0.0; return; }
    V3<T> p = O + D * t, n = normalise(p - centre_of<T>(sp));
    o[0] = 1.0; o[1] = (double)t; o[2] = (double)p.x; o[3] = (double)p.y; o[4] = (double)p.z;
    o[5] = (double)n.x; o[6] = (double)n.y; o[7] = (double)n.z;
}

template <typename T, int kMode>
__global__ void __launch_bounds__(256) trace_rays_kernel(SceneDev<T> sc, int m, const double *rays, const int *suppress,
                                                         const int *bounces0, const int *through0, int max_bounces,
                                                         int shadow_max_bounces, double miss0, double miss1,
                                                         double miss2, double *term, double *rgb) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const double *r = rays + 6 * (size_t)i;
    V3<T> O = mk<T>(T(r[0]), T(r[1]), T(r[2]));
    V3<T> D = normalise(mk<T>(T(r[3]), T(r[4]), T(r[5])));
    Counters ct = {0u, 0u, 0u, 0u};
    Hit<T> h = trace_terminal<T, kBvh>(S.g, O, D, suppress ? suppress[i] : RT_NO_ID_DEV, bounces0 ? bounces0[i] : 0,
                                 max_bounces, through0 ? through0[i] : 0, ct);
    double *t = term + 11 * (size_t)i;
    t[0] = h.idx >= 0 ? 1.0 : 0.0; t[1] = (double)h.idx; t[2] = (double)h.bounces; t[3] = (double)h.through;
    t[4] = (double)h.p.x; t[5] = (double)h.p.y; t[6] = (double)h.p.z;
    t[7] = (double)h.n.x; t[8] = (double)h.n.y; t[9] = (double)h.n.z; t[10] = (double)h.t;
    if (rgb) {
        double *c = rgb + 3 * (size_t)i;
        if (h.idx >= 0) {
            T o[3];
            terminal_rgb<T, kBvh>(S.g, S.la, h, shadow_max_bounces, o, ct);
            c[0] = (double)o[0]; c[1] = (double)o[1]; c[2] = (double)o[2];
        } else { c[0] = miss0; c[1] = miss1; c[2] = miss2; }
    }
}

// First-hit features of an Algorithm B frame (rt_render_features, DESIGN §4.8d).  One thread per pixel of rows [y0, y1),
// 32 x 8 pixels per CTA.  For samples [s0, s1) it traces the camera rays path_kernel traces (path_sample_ray) to their
// nearest hit: albedo = colour / 255, normal = (p - centre) / r, depth = t; all 0 on a miss.  Per pixel: the mean of
// every channel and, per feature, the variance of the mean averaged over its channels.  The sums are doubles added in
// sample order by one thread, so the result does not depend on the launch.
template <typename T, int kMode>
__global__ void __launch_bounds__(256) feature_kernel(SceneDev<T> sc, PathDev<T> pp, float *albedo, float *normal,
                                                      float *depth, float *fvar) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = pp.y0 + blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= pp.W || y >= pp.y1) return;
    const uint32_t pixel = (uint32_t)(y * pp.W + x);
    const V3<T> cam = mk<T>(pp.cam[0], pp.cam[1], pp.cam[2]);
    PathRng rng;
    unsigned n_tests = 0, n_boxes = 0;
    double s[7] = {0, 0, 0, 0, 0, 0, 0}, q[7] = {0, 0, 0, 0, 0, 0, 0};   // albedo 0-2, normal 3-5, depth 6
    for (int smp = pp.s0; smp < pp.s1; ++smp) {
        rng.begin(pixel, (uint32_t)smp, pp.k0, pp.k1);
        const V3<T> D = path_sample_ray<T>(pp, rng, x, y);
        T t;
        const int i = nearest<T, true, kBvh>(S.g, cam, D, RT_NO_ID_DEV, t, n_tests, n_boxes);
        double f[7] = {0, 0, 0, 0, 0, 0, 0};
        if (i >= 0) {
            RT_ASSERT(i < sc.n);
            const typename M<T>::v4 col = S.g.sv.col[i];
            const V3<T> n = (cam + D * t - centre_of<T>(S.g.sv.sph[i])) * col.w;          // col.w = 1/r (finish_hit)
            f[0] = (double)col.x / 255.0; f[1] = (double)col.y / 255.0; f[2] = (double)col.z / 255.0;
            f[3] = (double)n.x; f[4] = (double)n.y; f[5] = (double)n.z; f[6] = (double)t;
        }
#pragma unroll
        for (int c = 0; c < 7; ++c) { s[c] = __dadd_rn(s[c], f[c]); q[c] = __dadd_rn(q[c], __dmul_rn(f[c], f[c])); }
    }
    const int n = pp.s1 - pp.s0;
    const double dn = (double)n;
    // variance of the mean of channel c: (sum f^2 - (sum f)^2 / n) / (n (n - 1)), 0 below two samples; rounding can take a
    // variance below zero, which is clamped
    double v[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) {
        const double num = __dsub_rn(q[c], __ddiv_rn(__dmul_rn(s[c], s[c]), dn));
        v[c] = n < 2 ? 0.0 : fmax(0.0, __ddiv_rn(num, __dmul_rn(dn, dn - 1.0)));
    }
    const size_t o = (size_t)y * pp.W + x;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        albedo[3 * o + c] = (float)__ddiv_rn(s[c], dn);
        normal[3 * o + c] = (float)__ddiv_rn(s[3 + c], dn);
    }
    depth[o] = (float)__ddiv_rn(s[6], dn);
    fvar[3 * o + 0] = (float)__ddiv_rn(__dadd_rn(__dadd_rn(v[0], v[1]), v[2]), 3.0);
    fvar[3 * o + 1] = (float)__ddiv_rn(__dadd_rn(__dadd_rn(v[3], v[4]), v[5]), 3.0);
    fvar[3 * o + 2] = (float)v[6];
}

template <typename T, int kMode>
__global__ void __launch_bounds__(256) shade_hits_kernel(SceneDev<T> sc, int m, const double *hits, int shadow_max_bounces,
                                                         double *rgb) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const double *q = hits + 7 * (size_t)i;
    Hit<T> h;
    h.idx = (int)q[0]; h.t = T(0); h.bounces = 0; h.through = 0;
    h.p = mk<T>(T(q[1]), T(q[2]), T(q[3]));
    h.n = mk<T>(T(q[4]), T(q[5]), T(q[6]));
    double *c = rgb + 3 * (size_t)i;
    if (h.idx < 0 || h.idx >= sc.n) { c[0] = c[1] = c[2] = 0.0; return; }
    Counters ct = {0u, 0u, 0u, 0u};
    T o[3];
    terminal_rgb<T, kBvh>(S.g, S.la, h, shadow_max_bounces, o, ct);
    c[0] = (double)o[0]; c[1] = (double)o[1]; c[2] = (double)o[2];
}

// ------------------------------------------------------------------ batched RayTracerEnv
// One episode's state in registers: loaded once at the top of a step (all loads in flight together), updated in place,
// stored once at the end; the observation is built from the registers, never re-read from HBM.
template <typename T> struct EnvReg {
    int idx;                      // scene index of current_intersection, -1 = None
    int bounce, through;
    V3<T> p, n, d;
    T acc[3];
    T c[3];                       // RL flavour: terminalRGB of the current hit, computed when the hit was made (see env_step_kernel)
    double total;
    RT_DEV Hit<T> hit() const {
        Hit<T> h;
        h.idx = idx; h.p = p; h.n = n; h.t = T(0); h.bounces = 0; h.through = 0;
        return h;
    }
    RT_DEV void set_hit(const Hit<T> &h, V3<T> D) { idx = h.idx; p = h.p; n = h.n; d = D; }
};

template <typename T> RT_DEV EnvReg<T> env_load(const EnvDev<T> &e, int b) {
    const size_t B = (size_t)e.B;
    EnvReg<T> s;
    const int has = e.has_hit[b], idx = e.idx[b];
    s.bounce = e.bounce[b]; s.through = e.through[b];
    s.p = mk<T>(e.p[b], e.p[B + b], e.p[2 * B + b]);
    s.n = mk<T>(e.n[b], e.n[B + b], e.n[2 * B + b]);
    s.d = mk<T>(e.d[b], e.d[B + b], e.d[2 * B + b]);
    s.acc[0] = e.acc[b]; s.acc[1] = e.acc[B + b]; s.acc[2] = e.acc[2 * B + b];
    s.total = e.total[b];
    s.idx = has ? idx : -1;
    if (e.flavour == 0) { s.c[0] = e.rgb[b]; s.c[1] = e.rgb[B + b]; s.c[2] = e.rgb[2 * B + b]; }
    else s.c[0] = s.c[1] = s.c[2] = T(0);
    return s;
}

template <typename T> RT_DEV void env_store(const EnvDev<T> &e, int b, const EnvReg<T> &s) {
    const size_t B = (size_t)e.B;
    e.has_hit[b] = s.idx >= 0; e.idx[b] = s.idx;
    e.bounce[b] = s.bounce; e.through[b] = s.through;
    e.p[b] = s.p.x; e.p[B + b] = s.p.y; e.p[2 * B + b] = s.p.z;
    e.n[b] = s.n.x; e.n[B + b] = s.n.y; e.n[2 * B + b] = s.n.z;
    e.d[b] = s.d.x; e.d[B + b] = s.d.y; e.d[2 * B + b] = s.d.z;
    e.acc[b] = s.acc[0]; e.acc[B + b] = s.acc[1]; e.acc[2 * B + b] = s.acc[2];
    e.total[b] = s.total;
    if (e.flavour == 0) { e.rgb[b] = s.c[0]; e.rgb[B + b] = s.c[1]; e.rgb[2 * B + b] = s.c[2]; }
}

// _get_observation (RL/ray_tracer_env.py:184-222): 18 x float32 into the row `o` (a shared-memory staging row: the
// CTA writes its rows out together, coalesced, see env_flush_obs)
template <typename T> RT_DEV void env_obs(const Geo<T> &g, const EnvReg<T> &s, float *o) {
    if (s.idx < 0) {
#pragma unroll
        for (int k = 0; k < 18; ++k) o[k] = 0.f;
        return;
    }
    const typename M<T>::v4 m = g.sv.mat[s.idx];
    o[0] = (float)s.p.x; o[1] = (float)s.p.y; o[2] = (float)s.p.z;
    o[3] = (float)s.d.x; o[4] = (float)s.d.y; o[5] = (float)s.d.z;
    o[6] = (float)s.n.x; o[7] = (float)s.n.y; o[8] = (float)s.n.z;
    o[9] = (float)m.x; o[10] = (float)m.y; o[11] = (float)m.z; o[12] = (float)m.w;
    o[13] = (float)(s.acc[0] / T(255)); o[14] = (float)(s.acc[1] / T(255)); o[15] = (float)(s.acc[2] / T(255));
    o[16] = (float)s.bounce; o[17] = (float)s.through;
}

// RL _calculate_reward (RL/ray_tracer_env.py:224-252); FB _calculate_reward (FB/ray_tracer_env.py:241-278)
// `c` = terminalRGB(h) (ray.py:37-65): the step kernel keeps it with the hit instead of shading the same point twice
// (once for the accumulated colour when the hit is made, once for the next step's reward)
template <typename T>
RT_DEV double env_reward_base(const Geo<T> &g, const EnvDev<T> &e, const Hit<T> &h, int bounce_count, const T *c) {
    if (h.idx < 0) return -0.1;
    if (e.flavour == 1 && g.sv.ids[h.idx] == e.sun_id) return 10.0;
    if constexpr (M<T>::exact) {
        double brightness = (c[0] + c[1] + c[2]) / (3 * 255);
        double pen = -0.01 * bounce_count;
        return brightness + pen;
    } else {
        return (double)((c[0] + c[1] + c[2]) * (1.f / 765.f) - 0.01f * (float)bounce_count);
    }
}
// + AdaptiveRewardRayTracerEnv._calculate_reward (RL/train_raytracer_optimized.py:25-61) when e.adaptive
template <typename T>
RT_DEV double env_reward(const Geo<T> &g, const EnvDev<T> &e, int b, const Hit<T> &h, int bounce_count, const T *c) {
    if (!e.adaptive) return env_reward_base<T>(g, e, h, bounce_count, c);
    if (h.idx < 0) return -0.5;
    const double base = env_reward_base<T>(g, e, h, bounce_count, c);
    double light_bonus = 0.0, reflective_bonus = 0.0, path_length_penalty = 0.0;
    const int id = g.sv.ids[h.idx];
    if (id == e.light0 || id == e.light1) {
        light_bonus = 2.0;
        const int c = e.consec[b] + 1;
        e.consec[b] = c; e.total_hits[b] += 1;
        if (c > 1) light_bonus += 0.5 * c;
    } else e.consec[b] = 0;
    if (g.sv.mat[h.idx].x > T(0.5)) reflective_bonus = 0.3;
    if (bounce_count < 2 && base > 0.0) path_length_penalty = -0.1;
    return base + light_bonus + reflective_bonus + path_length_penalty;
}

// FB _calculate_lighting_reward (FB/ray_tracer_env.py:280-336)
template <typename T> RT_DEV double env_lighting_reward(const Geo<T> &g, const EnvDev<T> &e, const Hit<T> &h) {
    if (h.idx < 0) return 0.0;
    if (g.sv.mat[h.idx].z != T(0)) return 0.0;
    int sun = -1;
    for (int i = 0; i < g.sv.n; ++i) if (g.sv.ids[i] == e.sun_id) { sun = i; break; }
    if (sun < 0) return 0.1;
    const V3<T> sc = centre_of<T>(g.sv.sph[sun]);
    V3<T> to_sun = normalise(sc - h.p);
    T ca = dot(h.n, to_sun);
    if (!(ca > T(0))) ca = T(0);
    const V3<T> so = h.p + h.n * T(0.001);
    const V3<T> sd = M<T>::exact ? normalise(to_sun) : to_sun;
    const T sun_dist = mag(sc - h.p);
    bool shadow = false;
    for (int i = 0; i < g.sv.n && !shadow; ++i) {
        if (i == h.idx || g.sv.ids[i] == e.sun_id) continue;
        T t;
        if (!sphere_test<T>(so, sd, g.sv.sph[i], 0, t)) continue;
        const V3<T> ip = so + sd * t;
        if (mag(ip - h.p) < sun_dist) shadow = true;
    }
    return shadow ? 0.3 : 0.3 + 0.7 * (double)ca;
}

// Observation rows of a CTA: every thread builds its 18 floats in shared memory (stride 18: two-way bank conflicts on
// 18 stores), then the CTA copies the block of rows to HBM as consecutive 16-byte stores -- the per-thread rows would
// be 72-byte strided 4-byte stores, 18 partial sectors per warp instruction.
#ifndef RT_ENV_BLOCK
#define RT_ENV_BLOCK 64         /* envs (one thread each) per CTA.  65,536 envs = 1,024 CTAs = 6.9 per SM: 1 % imbalance (128: 3.46 per SM, 15 %) */
#endif
// register budget of the step kernel: left to itself ptxas settles on 80 registers and spills 64 bytes; the launch
// never has more than 14 warps per SM to place (65,536 episodes / 148 SMs), so registers are free
#ifndef RT_ENV_REGS
#define RT_ENV_REGS 128
#endif
RT_DEV void env_flush_obs(const float *rows, float *obs, int B) {
    __syncthreads();
    const int base = blockIdx.x * RT_ENV_BLOCK;
    const int n = min(RT_ENV_BLOCK, B - base) * 18;                      // floats of this CTA's rows
    float *dst = obs + (size_t)base * 18;                                // 64 * 72 bytes per CTA: 16-byte aligned
    const int n4 = (((uintptr_t)obs & 15u) == 0) ? n >> 2 : 0;
    for (int j = threadIdx.x; j < n4; j += RT_ENV_BLOCK)
        reinterpret_cast<float4 *>(dst)[j] = reinterpret_cast<const float4 *>(rows)[j];
    for (int j = 4 * n4 + threadIdx.x; j < n; j += RT_ENV_BLOCK) dst[j] = rows[j];
}

// reset of one episode (RL/ray_tracer_env.py:254-293, _get_initial_ray :121-142): camera ray through pixel (px, py),
// first nearestSphereIntersect, zeroed counters.  Shared by env_reset_kernel and the auto-reset of env_step_kernel.
template <typename T, bool kBvh>
RT_DEV void env_begin_episode(const Staged<T> &S, const EnvDev<T> &e, int b, int px, int py, EnvReg<T> &st, Counters &ct,
                              bool first = false) {
    // episode number since the last reset of the whole batch: the counter the in-launch restarts key their start pixels
    // by, so reset(seed) followed by the same actions always replays the same rollout
    if (e.episode) e.episode[b] = first ? 1 : e.episode[b] + 1;
    const T aspect = T(e.W) / T(e.H);
    const T x = (T(2) * (T(px) + T(0.5)) / T(e.W) - T(1)) * aspect * e.tan_half;
    const T y = (T(1) - T(2) * (T(py) + T(0.5)) / T(e.H)) * e.tan_half;
    V3<T> d = normalise(mk<T>(x, y, T(-1)));
    if (e.cam_angle[0] != T(0) || e.cam_angle[1] != T(0) || e.cam_angle[2] != T(0))
        d = rotate<T>(d, mk<T>(e.cam_angle[0], e.cam_angle[1], e.cam_angle[2]));
    d = normalise(d);
    Hit<T> h = trace_terminal<T, kBvh>(S.g, mk<T>(e.cam[0], e.cam[1], e.cam[2]), d, RT_NO_ID_DEV, 0, e.max_bounces, 0, ct);
    st.set_hit(h, d);
    st.bounce = 0; st.through = 0;
    st.acc[0] = T(0); st.acc[1] = T(0); st.acc[2] = T(0);
    st.total = 0.0;
    if (e.adaptive) e.consec[b] = 0;
}

// reset (RL/ray_tracer_env.py:254-293, _get_initial_ray :121-142).  pixels == NULL: draw with Philox(seed) keyed by
// the env index.  mask != NULL: only envs with mask[b] != 0 are reset.
template <typename T, int kMode>
__global__ void __launch_bounds__(256) env_reset_kernel(SceneDev<T> sc, EnvDev<T> e, const int *pixels,
                                                        const uint8_t *mask, uint32_t k0, uint32_t k1, float *obs,
                                                        int *pixels_out, unsigned long long *stats) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    Counters ct = {0u, 0u, 0u, 0u};
    if (b < e.B && (!mask || mask[b])) {
        int px, py;
        if (pixels) { px = pixels[2 * b]; py = pixels[2 * b + 1]; }
        else {
            Philox4 o = philox4x32_10((uint32_t)(e.b0 + b), 0u, 0u, 0x52544556u /* "RTEV" */, k0, k1);   // key = per-reset seed
            px = (int)(((unsigned long long)o.w[0] * (unsigned)e.W) >> 32);
            py = (int)(((unsigned long long)o.w[1] * (unsigned)e.H) >> 32);
        }
        if (pixels_out) { pixels_out[2 * b] = px; pixels_out[2 * b + 1] = py; }
        EnvReg<T> st;
        env_begin_episode<T, kBvh>(S, e, b, px, py, st, ct, mask == nullptr);
        st.c[0] = st.c[1] = st.c[2] = T(0);
        if (e.flavour == 0 && st.idx >= 0) terminal_rgb<T, kBvh>(S.g, S.la, st.hit(), 0, st.c, ct);
        env_store<T>(e, b, st);
        env_obs<T>(S.g, st, obs + 18 * (size_t)b);
    }
    if (stats) { flush_stats(stats, STAT_QUERIES, ct.queries); flush_stats(stats, STAT_DEAD_QUERIES, ct.dead); }
}

// The scene changed under running episodes (rt_scene_update): shade the current hits again
template <typename T, int kMode>
__global__ void __launch_bounds__(256) env_reshade_kernel(SceneDev<T> sc, EnvDev<T> e) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    Counters ct = {0u, 0u, 0u, 0u};
    if (b < e.B && e.flavour == 0 && e.has_hit[b] && e.idx[b] >= 0 && e.idx[b] < sc.n) {
        EnvReg<T> st = env_load<T>(e, b);
        terminal_rgb<T, kBvh>(S.g, S.la, st.hit(), 0, st.c, ct);
        const size_t B = (size_t)e.B;
        e.rgb[b] = st.c[0]; e.rgb[B + b] = st.c[1]; e.rgb[2 * B + b] = st.c[2];
    }
}

// step (RL/ray_tracer_env.py:295-401, FB/ray_tracer_env.py:378-514)
// R = type of the reward / info outputs (double: rt_env_step; the env's own precision: rt_env_step_auto).
// kAuto: an episode that ends in this step is restarted IN THE SAME LAUNCH (SB3 VecEnv semantics): its last observation
// goes to final_obs (optional), the observation returned is the first one of the new episode, whose start pixel is
// Philox(env, episode number) under the key (k0, k1) -- no host round trip and no second launch per step, and the
// lanes of finished episodes go straight back to work.
// kFlav: the env flavour as a compile-time constant (0 RL) or -1 = read e.flavour: the fused launch of a small RL scene
// carries one reward model and one set of termination rules (16.2 -> 15.8 us per 65,536-env step).
template <typename T, int kMode, typename R, bool kAuto, int kFlav = -1>
__global__ void __maxnreg__(RT_ENV_REGS) env_step_kernel(SceneDev<T> sc, EnvDev<T> e_param, const float *actions, float *obs,
                                                                R *reward, uint8_t *terminated, uint8_t *truncated,
                                                                int *reason, R *info, float *final_obs, int *pixels_out,
                                                                uint32_t k0, uint32_t k1, unsigned long long *stats) {
    RT_MODE_DECL;
    EnvDev<T> e = e_param;
    if constexpr (kFlav >= 0) e.flavour = kFlav;
    extern __shared__ __align__(32) unsigned char smem[];
    __shared__ __align__(16) float s_rows[RT_ENV_BLOCK * 18];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int slot = (int)threadIdx.x;
    const int b = blockIdx.x * RT_ENV_BLOCK + slot;
    float *row = s_rows + 18 * slot;
    Counters ct = {0u, 0u, 0u, 0u};
    if (b < e.B) {
        const unsigned live = __activemask();       // the lanes of this warp that carry an episode (converged here)
        EnvReg<T> st = env_load<T>(e, b);
        RT_ASSERT(st.idx >= -1 && st.idx < sc.n && st.bounce >= 0);
        const float a0 = actions[2 * b], a1 = actions[2 * b + 1];
        const Hit<T> cur = st.hit();
        int bc = st.bounce;
        const int through = st.through;
        int rsn = 0, term = 0, trunc = 0;
        bool shade = false;                       // the step made a new hit: accumulated colour += terminalRGB(hit)
        double rw = 0.0, info_total, info_sun = -1.0;
        int info_bounce = bc;
        if (cur.idx < 0) {                                                   // ray already missed, :313-323
            rsn = 1; rw = -1.0; term = 1; info_total = st.total;
        } else if (bc >= e.max_bounces) {                                    // :325-337
            rw = e.flavour == 1 ? env_lighting_reward<T>(S.g, e, cur) : env_reward<T>(S.g, e, b, cur, bc, st.c);
            st.total += rw; info_total = st.total;
            rsn = 3; term = 1; trunc = 1;
        } else if (e.flavour == 1 && S.g.sv.ids[cur.idx] == e.sun_id) {      // FB :417-431 (total_reward not updated)
            rsn = 5; rw = 10.0; term = 1; info_total = st.total + rw; info_sun = 1.0;
        } else {
            // _action_to_direction: RL :144-182, FB :157-198
            T theta, phi;
            if (e.flavour == 1) {
                theta = (T(a0) + T(1)) * T(3.14159265358979323846) / T(4);
                phi = T(a1) * T(3.14159265358979323846);
            } else { theta = T(a0); phi = T(a1); }
            T st_, ct_, sp_, cp_;
            M<T>::sincos(theta, &st_, &ct_); M<T>::sincos(phi, &sp_, &cp_);
            const T lx = st_ * cp_, ly = st_ * sp_, lz = ct_;
            const V3<T> n = cur.n;
            V3<T> tg = M<T>::fabs(n.z) < T(0.9) ? cross(mk<T>(0, 0, 1), n) : cross(mk<T>(1, 0, 0), n);
            tg = normalise(tg);
            const V3<T> bt = normalise(cross(n, tg));
            V3<T> D = normalise(mk<T>(lx * tg.x + ly * bt.x + lz * n.x, lx * tg.y + ly * bt.y + lz * n.y,
                                      lx * tg.z + ly * bt.z + lz * n.z));
            if constexpr (M<T>::exact) D = normalise(D);                      // Ray() normalises again
            bc += 1;
            Hit<T> nx = trace_terminal<T, kBvh>(S.g, cur.p, D, S.g.sv.ids[cur.idx], bc, e.max_bounces, through, ct);
            if (e.flavour == 0) rw = env_reward<T>(S.g, e, b, cur, bc, st.c);             // reward at the PRE-update hit, :362
            else if (nx.idx >= 0) {
                if (S.g.sv.ids[nx.idx] == e.sun_id) { rw = 10.0; rsn = 4; term = 1; info_sun = 1.0; }
                else { rw = env_lighting_reward<T>(S.g, e, nx); info_sun = 0.0; }
            } else { rw = -0.1; rsn = 1; term = 1; }
            st.total += rw; info_total = st.total;
            st.set_hit(nx, D);
            st.bounce = bc; info_bounce = bc;
            shade = nx.idx >= 0;                                             // :373-381, done below
            if (e.flavour == 0) {
                if (nx.idx < 0) { term = 1; rsn = 2; }
                else if (bc >= e.max_bounces) { term = 1; trunc = 1; rsn = 3; }
            } else if (!term && bc >= e.max_bounces) { term = 1; trunc = 1; rsn = 3; }
        }
        reward[b] = (R)rw; terminated[b] = (uint8_t)term; truncated[b] = (uint8_t)trunc; reason[b] = rsn;
        if (info) {
            R *q = info + 4 * (size_t)b;
            q[0] = (R)info_bounce; q[1] = (R)through; q[2] = (R)info_total; q[3] = (R)info_sun;
        }
        // ONE shading site for the whole step.  A hit is shaded when it is made: the colour goes into the accumulated
        // colour of the observation (:373-381) and stays with the hit (EnvReg::c) as the RL flavour's reward of the NEXT
        // step (:362 shades the pre-update hit again: same point, same scene, same value).  An episode that restarts in
        // this launch shades its first hit here too, so the lanes of continuing and of restarted episodes share the
        // code; only an episode that ENDS on a hit (bounce limit) needs its colour before the restart, for final_obs.
        bool restarted = false;
        __syncwarp(live);       // the four outcomes of the step above meet again before the restarts
        if constexpr (kAuto) {
            if (term | trunc) {
                restarted = true;
                if (shade && final_obs) {
                    T c[3];
                    terminal_rgb<T, kBvh>(S.g, S.la, st.hit(), 0, c, ct);
                    st.acc[0] = st.acc[0] + c[0]; st.acc[1] = st.acc[1] + c[1]; st.acc[2] = st.acc[2] + c[2];
                }
                env_obs<T>(S.g, st, row);
                if (final_obs) {                         // 72-byte rows: nine 8-byte stores
                    float2 *fo = reinterpret_cast<float2 *>(final_obs + 18 * (size_t)b);
#pragma unroll
                    for (int k = 0; k < 9; ++k) fo[k] = make_float2(row[2 * k], row[2 * k + 1]);
                }
                const Philox4 o = philox4x32_10((uint32_t)(e.b0 + b), (uint32_t)e.episode[b], 1u, 0x52544556u /* "RTEV" */, k0, k1);
                const int px = (int)(((unsigned long long)o.w[0] * (unsigned)e.W) >> 32);
                const int py = (int)(((unsigned long long)o.w[1] * (unsigned)e.H) >> 32);
                if (pixels_out) { pixels_out[2 * b] = px; pixels_out[2 * b + 1] = py; }
                env_begin_episode<T, kBvh>(S, e, b, px, py, st, ct);
                shade = e.flavour == 0 && st.idx >= 0;
            }
        }
        __syncwarp(live);       // continuing and restarted episodes enter the shading TOGETHER (else the compiler threads
                                // the two paths into the block separately and the warp runs it twice)
        if (shade) {
            terminal_rgb<T, kBvh>(S.g, S.la, st.hit(), 0, st.c, ct);
            if (!restarted) { st.acc[0] = st.acc[0] + st.c[0]; st.acc[1] = st.acc[1] + st.c[1]; st.acc[2] = st.acc[2] + st.c[2]; }
        }
        env_obs<T>(S.g, st, row);
        env_store<T>(e, b, st);
    }
    env_flush_obs(s_rows, obs, e.B);
    if (stats) { flush_stats(stats, STAT_QUERIES, ct.queries); flush_stats(stats, STAT_DEAD_QUERIES, ct.dead); }
}

// ------------------------------------------------------------------ launchers
template <typename K> static cudaError_t allow_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return cudaSuccess;
}

#define RT_DISPATCH_MODE(mode, KERNEL, grid, block, smem_bytes, st, ...)                                       \
    do {                                                                                                        \
        cudaError_t e__ = cudaSuccess;                                                                          \
        switch (mode) {                                                                                         \
            case 0: e__ = allow_smem(KERNEL<T, 0>, smem_bytes); if (e__ != cudaSuccess) return e__;             \
                    KERNEL<T, 0><<<grid, block, smem_bytes, st>>>(__VA_ARGS__); break;                          \
            case 1: e__ = allow_smem(KERNEL<T, 1>, smem_bytes); if (e__ != cudaSuccess) return e__;             \
                    KERNEL<T, 1><<<grid, block, smem_bytes, st>>>(__VA_ARGS__); break;                          \
            default: KERNEL<T, 2><<<grid, block, 0, st>>>(__VA_ARGS__); break;                                  \
        }                                                                                                       \
    } while (0)

// CTAs of a persistent launch: what the current device keeps resident for this kernel (occupancy x SM count); the
// answer is cached per (device, kernel, shared-memory size) so that a launch costs no runtime query
template <typename K> static unsigned persistent_ctas(K kernel, size_t smem_bytes, long long tiles) {
    struct Key { int dev; const void *fn; size_t smem; long long ctas; };
    static std::mutex mu;
    static std::vector<Key> cache;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    long long g = 0;
    {
        std::lock_guard<std::mutex> lock(mu);
        for (const Key &k : cache)
            if (k.dev == dev && k.fn == (const void *)kernel && k.smem == smem_bytes) { g = k.ctas; break; }
    }
    if (g == 0) {
        int sms = 0, per_sm = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, smem_bytes) != cudaSuccess || per_sm <= 0) per_sm = 1;
        g = (long long)sms * per_sm;
        std::lock_guard<std::mutex> lock(mu);
        cache.push_back(Key{dev, (const void *)kernel, smem_bytes, g});
    }
    return (unsigned)(tiles < g ? (tiles > 0 ? tiles : 1) : g);
}

template <typename T>
cudaError_t launch_whitted(const SceneDev<T> &sc, const WhittedDev<T> &wp, void *accum, int *hit,
                           unsigned long long *stats, cudaStream_t st, unsigned *sched, unsigned *sched2, unsigned *heavy) {
    const int rows = wp.y1 - wp.y0;
    if (rows <= 0 || wp.W <= 0) return cudaSuccess;
    WhittedDev<T> wl = wp;                                        // + the 32x8 block grid the persistent warps walk
    wl.gx = (wp.W + 31) / 32; wl.gy = (rows + 7) / 8;
    wl.sched = sched; wl.sched2 = sched2; wl.heavy = heavy; wl.split = 0;
    const long long blocks = (long long)wl.gx * wl.gy;
    dim3 grid(1), block(256);
    using v4 = typename M<T>::v4;
    const int mode = mode_for(sc);
    const size_t sm = mode != 2 ? smem_for(sc) : 0;
    cudaError_t e = cudaSuccess;
    if constexpr (sizeof(T) == 4) {
        // two-pass schedule: small brute-force scenes (the candidate lists need <= 64 spheres), a few samples per pixel
        if (mode == 0 && sched2 && heavy && sc.n <= 64 && wp.s1 - wp.s0 >= 4) {
            wl.split = 1;
            e = allow_smem(whitted_kernel<T, 0>, sm); if (e != cudaSuccess) return e;
            e = allow_smem(whitted_heavy_kernel<0>, sm); if (e != cudaSuccess) return e;
            grid.x = persistent_ctas(whitted_kernel<T, 0>, sm, blocks);
            whitted_kernel<T, 0><<<grid, block, sm, st>>>(sc, wl, (v4 *)accum, hit, stats);
            e = cudaGetLastError(); if (e != cudaSuccess) return e;
            grid.x = persistent_ctas(whitted_heavy_kernel<0>, sm, blocks * 8);
            whitted_heavy_kernel<0><<<grid, block, sm, st>>>(sc, wl, (float4 *)accum, hit, stats);
            return cudaGetLastError();
        }
    }
    switch (mode) {
        case 0: e = allow_smem(whitted_kernel<T, 0>, sm); if (e != cudaSuccess) return e;
                grid.x = persistent_ctas(whitted_kernel<T, 0>, sm, blocks);
                whitted_kernel<T, 0><<<grid, block, sm, st>>>(sc, wl, (v4 *)accum, hit, stats); break;
        case 1: e = allow_smem(whitted_kernel<T, 1>, sm); if (e != cudaSuccess) return e;
                grid.x = persistent_ctas(whitted_kernel<T, 1>, sm, blocks);
                whitted_kernel<T, 1><<<grid, block, sm, st>>>(sc, wl, (v4 *)accum, hit, stats); break;
        default: grid.x = persistent_ctas(whitted_kernel<T, 2>, 0, blocks);
                 whitted_kernel<T, 2><<<grid, block, 0, st>>>(sc, wl, (v4 *)accum, hit, stats); break;
    }
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_path(const SceneDev<T> &sc, const PathDev<T> &pp, const PathLaunch &pl, void *accum,
                        unsigned long long *stats, cudaStream_t st, const PkConst *pkc, const MomentsDev *moments,
                        const MomentsListDev *listed) {
    if (pp.y1 <= pp.y0 || pp.W <= 0) return cudaSuccess;
    const long long tiles_total = (long long)pp.gx * pp.gy + (long long)pp.gx2 * pp.gy2;
    dim3 grid(1), block(256);
    using v4 = typename M<T>::v4;
    const size_t sm = pl.smem;
    cudaError_t e = cudaSuccess;
    const MomentsDev *const mom = moments;
    // one launch of path_kernel<T, M_, F_, Q_, L_>; SMOPT_: the shared memory to opt in to, PKC_: the parameter-block
    // scene (kMode 3), MOM_: the moments sinks (Q_ = true) with the pixel list (L_ = true)
#define RT_PATH_LAUNCH(M_, F_, Q_, L_, SMOPT_, PKC_, MOM_)                                                           \
    { e = allow_smem(path_kernel<T, M_, F_, Q_, L_>, SMOPT_); if (e != cudaSuccess) return e;                      \
      grid.x = persistent_ctas(path_kernel<T, M_, F_, Q_, L_>, sm, tiles_total);                                   \
      if (pp.max_ctas > 0 && grid.x > (unsigned)pp.max_ctas) grid.x = (unsigned)pp.max_ctas;                        \
      path_kernel<T, M_, F_, Q_, L_><<<grid, block, sm, st>>>(sc, pp, (v4 *)accum, stats, PKC_, MOM_); }
    if (listed) {                                     // list launches: integer fold only (rt_render_path_adaptive)
        if (!pp.int_fold) return cudaErrorInvalidValue;
        if (pl.mode == 3) { if constexpr (sizeof(T) == 4) RT_PATH_LAUNCH(3, true, true, true, sm ? sm + 8192 : 0, *pkc, *listed) }
        else if (pl.mode == 0) RT_PATH_LAUNCH(0, true, true, true, sm, PkNone(), *listed)
        else if (pl.mode == 1) RT_PATH_LAUNCH(1, true, true, true, sm, PkNone(), *listed)
        else RT_PATH_LAUNCH(2, true, true, true, sm, PkNone(), *listed)
        return cudaGetLastError();
    }
#define RT_PATH_CASE(M_, F_)                                                                                       \
    { if (mom) RT_PATH_LAUNCH(M_, F_, true, false, sm, PkNone(), *mom) else RT_PATH_LAUNCH(M_, F_, false, false, sm, PkNone(), PkNone()) }
    if (pl.mode == 3) {
        if constexpr (sizeof(T) == 4) {
            // + the static arrays: opt in above 48 KB in all
#define RT_PATH_CASE3(F_)                                                                                          \
    { if (mom) RT_PATH_LAUNCH(3, F_, true, false, sm ? sm + 8192 : 0, *pkc, *mom)                                   \
      else RT_PATH_LAUNCH(3, F_, false, false, sm ? sm + 8192 : 0, *pkc, PkNone()) }
            if (pp.int_fold) RT_PATH_CASE3(true) else RT_PATH_CASE3(false)
#undef RT_PATH_CASE3
        }
        return cudaGetLastError();
    }
    const int variant = pl.mode * 2 + (pp.int_fold ? 1 : 0);
    switch (variant) {
        case 0: RT_PATH_CASE(0, false) break;   case 1: RT_PATH_CASE(0, true) break;
        case 2: RT_PATH_CASE(1, false) break;   case 3: RT_PATH_CASE(1, true) break;
        case 4: RT_PATH_CASE(2, false) break;   default: RT_PATH_CASE(2, true) break;
    }
#undef RT_PATH_CASE
#undef RT_PATH_LAUNCH
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_trajectories(const SceneDev<T> &sc, int n_traj, int max_steps, int max_bounces, uint64_t seed, float *obs,
                                float *action, float *next_obs, float *reward, uint8_t *hit, int *length,
                                uint8_t *hit_light, unsigned long long *stats, cudaStream_t st) {
    if (n_traj <= 0) return cudaSuccess;
    const int block = 128, grid = (n_traj + block - 1) / block;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, trajectory_kernel, grid, block, smem_for(sc), st, sc, n_traj, max_steps, max_bounces, k0, k1, obs,
                     action, next_obs, reward, hit, length, hit_light, stats);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_simple(const SceneDev<T> &sc, const SimpleDev<T> &sp, int4 *rgb, float *image, unsigned long long *stats,
                          cudaStream_t st) {
    if (sp.n <= 0) return cudaSuccess;
    dim3 block(256), grid = sp.rays ? dim3((sp.n + 255) / 256) : dim3((sp.W + 31) / 32, (sp.H + 7) / 8);
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, simple_kernel, grid, block, smem_for(sc), st, sc, sp, rgb, image, stats);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_resolve(const void *accum, int W, int y0, int y1, int spp, float *image, cudaStream_t st) {
    const size_t n = (size_t)(y1 - y0) * W;
    if (n == 0) return cudaSuccess;
    resolve_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const typename M<T>::v4 *)accum, W, y0, y1, spp, image);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_resolve_variance(const void *accum, const double *moments, int W, int y0, int y1, float *var, cudaStream_t st) {
    const size_t n = (size_t)(y1 - y0) * W;
    if (n == 0) return cudaSuccess;
    resolve_variance_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const typename M<T>::v4 *)accum,
                                                                          (const double4 *)moments, W, y0, y1, var);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_adaptive_select(const void *accum, const double *moments, int W, int y0, int y1, int c, double thr,
                                   uint32_t *list, uint32_t *count, cudaStream_t st) {
    if (y1 <= y0 || W <= 0) return cudaSuccess;
    const dim3 grid((unsigned)((W + 31) / 32), (unsigned)((y1 - y0 + 7) / 8));
    adaptive_select_kernel<T><<<grid, 256, 0, st>>>((const typename M<T>::v4 *)accum, (const double4 *)moments, W, y0, y1,
                                                    c, thr, list, count);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_adaptive_resolve(const void *accum, const double *moments, int W, int y0, int y1, float *image,
                                    float *var, int *counts, cudaStream_t st) {
    const size_t n = (size_t)(y1 - y0) * W;
    if (n == 0) return cudaSuccess;
    adaptive_resolve_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const typename M<T>::v4 *)accum,
                                                                          (const double4 *)moments, W, y0, y1, image, var,
                                                                          counts);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_sphere_disc(int m, const double *rays, const double *spheres, int point, double *out, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    sphere_disc_kernel<T><<<(m + 127) / 128, 128, 0, st>>>(m, rays, spheres, point, out);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_trace_rays(const SceneDev<T> &sc, int m, const double *rays, const int *suppress, const int *bounces0,
                              const int *through0, int max_bounces, int shadow_max_bounces, const double miss[3],
                              double *term, double *rgb, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    const int block = 256, grid = (m + block - 1) / block;
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, trace_rays_kernel, grid, block, smem_for(sc), st, sc, m, rays, suppress, bounces0, through0,
                     max_bounces, shadow_max_bounces, miss[0], miss[1], miss[2], term, rgb);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_features(const SceneDev<T> &sc, const PathDev<T> &pp, float *albedo, float *normal, float *depth,
                            float *fvar, cudaStream_t st) {
    if (pp.y1 <= pp.y0 || pp.W <= 0 || pp.s1 <= pp.s0) return cudaSuccess;
    const dim3 grid((unsigned)((pp.W + 31) / 32), (unsigned)((pp.y1 - pp.y0 + 7) / 8));
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, feature_kernel, grid, 256, smem_for(sc), st, sc, pp, albedo, normal, depth, fvar);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_shade_hits(const SceneDev<T> &sc, int m, const double *hits, int shadow_max_bounces, double *rgb,
                              cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    const int block = 256, grid = (m + block - 1) / block;
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, shade_hits_kernel, grid, block, smem_for(sc), st, sc, m, hits, shadow_max_bounces, rgb);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_env_reset(const SceneDev<T> &sc, const EnvDev<T> &e, const int *pixels, const uint8_t *mask,
                             uint64_t seed, float *obs, int *pixels_out, unsigned long long *stats, cudaStream_t st) {
    if (e.B <= 0) return cudaSuccess;
    const int block = 128, grid = (e.B + block - 1) / block;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, env_reset_kernel, grid, block, smem_for(sc), st, sc, e, pixels, mask, k0, k1, obs, pixels_out,
                     stats);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_env_reshade(const SceneDev<T> &sc, const EnvDev<T> &e, cudaStream_t st) {
    if (e.B <= 0 || e.flavour != 0) return cudaSuccess;
    const int block = 128, grid = (e.B + block - 1) / block;
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, env_reshade_kernel, grid, block, smem_for(sc), st, sc, e);
    return cudaGetLastError();
}

// kAuto = false: plain step (rt_env_step); true: step + in-launch restart of finished episodes (rt_env_step_auto)
template <typename T, typename R, bool kAuto>
cudaError_t launch_env_step(const SceneDev<T> &sc, const EnvDev<T> &e, const float *actions, float *obs, R *reward,
                            uint8_t *terminated, uint8_t *truncated, int *reason, R *info, float *final_obs, int *pixels_out,
                            uint64_t seed, unsigned long long *stats, cudaStream_t st) {
    if (e.B <= 0) return cudaSuccess;
    const int block = RT_ENV_BLOCK, grid = (e.B + RT_ENV_BLOCK - 1) / RT_ENV_BLOCK;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const size_t rows = RT_ENV_BLOCK * 18 * sizeof(float);                 // static shared rows on top of the staged scene
    const int mode = mode_for(sc, rows);
    const size_t sm = mode != 2 ? smem_for(sc) : 0;
    cudaError_t e__ = cudaSuccess;
    switch (mode) {
        case 0:
            if (kAuto && e.flavour == 0) {
                e__ = allow_smem(env_step_kernel<T, 0, R, kAuto, 0>, sm); if (e__ != cudaSuccess) return e__;
                env_step_kernel<T, 0, R, kAuto, 0><<<grid, block, sm, st>>>(sc, e, actions, obs, reward, terminated, truncated, reason, info, final_obs, pixels_out, k0, k1, stats);
            } else {        // (the FB flavour specialised the same way measured SLOWER: 16.5 against 14.7 us per step)
                e__ = allow_smem(env_step_kernel<T, 0, R, kAuto>, sm); if (e__ != cudaSuccess) return e__;
                env_step_kernel<T, 0, R, kAuto><<<grid, block, sm, st>>>(sc, e, actions, obs, reward, terminated, truncated, reason, info, final_obs, pixels_out, k0, k1, stats);
            }
            break;
        case 1: e__ = allow_smem(env_step_kernel<T, 1, R, kAuto>, sm); if (e__ != cudaSuccess) return e__;
                env_step_kernel<T, 1, R, kAuto><<<grid, block, sm, st>>>(sc, e, actions, obs, reward, terminated, truncated, reason, info, final_obs, pixels_out, k0, k1, stats); break;
        default: env_step_kernel<T, 2, R, kAuto><<<grid, block, 0, st>>>(sc, e, actions, obs, reward, terminated, truncated, reason, info, final_obs, pixels_out, k0, k1, stats); break;
    }
    return cudaGetLastError();
}

#define RT_INSTANTIATE_LAUNCHERS(T)                                                                                     \
    template cudaError_t launch_whitted<T>(const SceneDev<T> &, const WhittedDev<T> &, void *, int *,                   \
                                           unsigned long long *, cudaStream_t, unsigned *, unsigned *, unsigned *);     \
    template cudaError_t launch_path<T>(const SceneDev<T> &, const PathDev<T> &, const PathLaunch &, void *,           \
                                        unsigned long long *, cudaStream_t, const PkConst *, const MomentsDev *,        \
                                        const MomentsListDev *);                                                        \
    template cudaError_t launch_resolve<T>(const void *, int, int, int, int, float *, cudaStream_t);                    \
    template cudaError_t launch_resolve_variance<T>(const void *, const double *, int, int, int, float *, cudaStream_t); \
    template cudaError_t launch_adaptive_select<T>(const void *, const double *, int, int, int, int, double, uint32_t *,  \
                                                   uint32_t *, cudaStream_t);                                           \
    template cudaError_t launch_adaptive_resolve<T>(const void *, const double *, int, int, int, float *, float *, int *, \
                                                    cudaStream_t);                                                      \
    template cudaError_t launch_trajectories<T>(const SceneDev<T> &, int, int, int, uint64_t, float *, float *, float *,  \
                                                float *, uint8_t *, int *, uint8_t *, unsigned long long *, cudaStream_t); \
    template cudaError_t launch_simple<T>(const SceneDev<T> &, const SimpleDev<T> &, int4 *, float *,                   \
                                          unsigned long long *, cudaStream_t);                                         \
    template cudaError_t launch_sphere_disc<T>(int, const double *, const double *, int, double *, cudaStream_t);       \
    template cudaError_t launch_trace_rays<T>(const SceneDev<T> &, int, const double *, const int *, const int *,       \
                                              const int *, int, int, const double[3], double *, double *,              \
                                              cudaStream_t);                                                            \
    template cudaError_t launch_shade_hits<T>(const SceneDev<T> &, int, const double *, int, double *, cudaStream_t);    \
    template cudaError_t launch_features<T>(const SceneDev<T> &, const PathDev<T> &, float *, float *, float *, float *, \
                                            cudaStream_t);                                                              \
    template cudaError_t launch_env_reset<T>(const SceneDev<T> &, const EnvDev<T> &, const int *, const uint8_t *,      \
                                             uint64_t, float *, int *, unsigned long long *, cudaStream_t);             \
    template cudaError_t launch_env_reshade<T>(const SceneDev<T> &, const EnvDev<T> &, cudaStream_t);                   \
    template cudaError_t launch_env_step<T, double, false>(const SceneDev<T> &, const EnvDev<T> &, const float *, float *, double *, \
                                            uint8_t *, uint8_t *, int *, double *, float *, int *, uint64_t, unsigned long long *, cudaStream_t); \
    template cudaError_t launch_env_step<T, T, true>(const SceneDev<T> &, const EnvDev<T> &, const float *, float *, T *,   \
                                            uint8_t *, uint8_t *, int *, T *, float *, int *, uint64_t, unsigned long long *, cudaStream_t);

}  // namespace rt
