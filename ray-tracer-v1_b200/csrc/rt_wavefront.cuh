// rt_wavefront.cuh -- Algorithm B as a wavefront, so that a learned policy can choose the diffuse directions.
//
// Reference: WorkingFBRenderer.trace_ray_fb / render (FB/fb_vs_traditional_complex.py:487-640): trace_ray_traditional,
// except that at a non-mirror hit, with probability fb_usage_prob, the bounce direction comes from
// fb_agent.choose_direction(create_observation(...)) -> (a0, a1) in [-1,1]^2, theta = (a0+1) pi/4, phi = a1 pi (:545-546).
// The policy is a torch module, so the megakernel is split at exactly that point:
//
//   wf_begin   camera rays of every (pixel, sample) of the launch's rows / sample range
//   wf_trace   one nearest-hit query + shading per live path; paths that ask the policy get their 22-float observation
//              written and need[i] = 1
//   (host)     actions[need] = policy(obs[need])                      -- torch, on the same stream
//   wf_bounce  mirror / policy / cosine-weighted direction, next ray, depth limit
//   wf_finish  fold every path (same fold as path_kernel) and add it into the pixel sums
//
// State is SoA in HBM, one slot per path: the kernels are HBM-streaming (~150 B per path and bounce) around the same
// FP32/FP64 query code as path_kernel.  Draws: jitter and (r1, r2) as in path_kernel; the use-policy decision is word
// 0 of the Philox block (pixel, sample, bounce, tag "RTFB").
#pragma once
#include "rt_kernels.cuh"

namespace rt {

#define RT_FB_TAG 0x52544642u /* "RTFB" */
enum : int { WF_DEAD = 0, WF_LIVE = 1, WF_PENDING = 2 };   // PENDING: hit shaded, waiting for its bounce direction

template <typename T> RT_DEV void wf_path_id(const WaveDev<T> &w, int i, int &x, int &y, int &s) {
    const int ns = w.s1 - w.s0;
    s = w.s0 + i % ns;
    const int px = i / ns;
    x = px % w.W;
    y = w.y0 + px / w.W;
}

template <typename T>
__global__ void __launch_bounds__(256) wf_begin_kernel(WaveDev<T> w, PathDev<T> pp, unsigned long long *stats) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned n_rays = 0;
    if (i < w.P) {
        int x, y, s;
        wf_path_id<T>(w, i, x, y, s);
        const Philox4 o = philox4x32_10((uint32_t)(y * w.W + x), (uint32_t)s, 0u, RT_PHILOX_TAG, w.k0, w.k1);
        const V3<T> d = path_camera_ray<T>(pp, x, y, u01<T>(o.w[0]), u01<T>(o.w[1]));
        const size_t P = (size_t)w.P;
        w.O[i] = w.cam[0]; w.O[P + i] = w.cam[1]; w.O[2 * P + i] = w.cam[2];
        w.D[i] = d.x; w.D[P + i] = d.y; w.D[2 * P + i] = d.z;
        w.depth[i] = 0;
        n_rays = 1;
        if (w.max_bounces <= 0) { w.state[i] = WF_DEAD; w.leaf[i] = 2.0; w.leaf[P + i] = 2.0; w.leaf[2 * P + i] = 5.0; }
        else w.state[i] = WF_LIVE;
    }
    if (stats) flush_stats(stats, STAT_RAYS, n_rays);
}

template <typename T, int kMode>
__global__ void __launch_bounds__(256) wf_trace_kernel(SceneDev<T> sc, WaveDev<T> w, float *obs, uint8_t *need,
                                                       unsigned long long *stats) {
    RT_MODE_DECL;
    extern __shared__ __align__(32) unsigned char smem[];
    Staged<T> S;
    stage_scene<T, kShared>(sc, smem, S);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned n_inter = 0, n_light = 0, n_small = 0, n_query = 0, n_tests = 0, n_boxes = 0, n_fb = 0, n_live = 0;
    if (i < w.P) {
        const size_t P = (size_t)w.P;
        uint8_t ask = 0;
        if (w.state[i] == WF_LIVE) {
            const V3<T> O = mk<T>(w.O[i], w.O[P + i], w.O[2 * P + i]), D = mk<T>(w.D[i], w.D[P + i], w.D[2 * P + i]);
            const int depth = w.depth[i];
            T t;
            n_query++;
            const int hi = nearest<T, true, kBvh>(S.g, O, D, RT_NO_ID_DEV, t, n_tests, n_boxes);
            if (hi < 0) {
                w.state[i] = WF_DEAD; w.leaf[i] = 2.0; w.leaf[P + i] = 2.0; w.leaf[2 * P + i] = 5.0;
            } else {
                n_inter++;
                const typename M<T>::v4 m = S.g.sv.mat[hi];
                if (m.z != T(0)) {
                    n_light++;
                    if (sc.small && sc.small[hi]) n_small++;
                    const typename M<T>::v4 col = S.g.sv.col[hi];
                    w.state[i] = WF_DEAD; w.leaf[i] = (double)col.x; w.leaf[P + i] = (double)col.y; w.leaf[2 * P + i] = (double)col.z;
                } else {
                    Hit<T> h;
                    finish_hit<T>(S.g, O, D, hi, t, h);
                    w.st_idx[(size_t)depth * P + i] = (uint32_t)hi;
                    if constexpr (M<T>::exact) w.st_direct[(size_t)depth * P + i] = direct_light<T>(S.lb, hi, h.p, h.n);
                    else w.st_direct[(size_t)depth * P + i] = direct_light_pk(S.lb.lpk, (S.lb.nL + 1) >> 1, h.p, h.n);
                    w.hp[i] = h.p.x; w.hp[P + i] = h.p.y; w.hp[2 * P + i] = h.p.z;
                    w.hn[i] = h.n.x; w.hn[P + i] = h.n.y; w.hn[2 * P + i] = h.n.z;
                    const bool mirror = m.x > w.mirror_threshold;
                    w.mirror[i] = (uint8_t)mirror;
                    w.state[i] = WF_PENDING;
                    n_live = 1;
                    if (!mirror && w.fb_prob > T(0)) {                    // fb_loaded and random() < fb_usage_prob, :537
                        int x, y, s;
                        wf_path_id<T>(w, i, x, y, s);
                        const Philox4 o = philox4x32_10((uint32_t)(y * w.W + x), (uint32_t)s, (uint32_t)depth, RT_FB_TAG, w.k0, w.k1);
                        if (u01<T>(o.w[0]) < w.fb_prob) {
                            ask = 1; n_fb++;
                            float *q = obs + 22 * (size_t)i;                  // create_observation, :469-485
                            q[0] = (float)h.p.x; q[1] = (float)h.p.y; q[2] = (float)h.p.z;
                            q[3] = (float)D.x; q[4] = (float)D.y; q[5] = (float)D.z;
                            q[6] = (float)h.n.x; q[7] = (float)h.n.y; q[8] = (float)h.n.z;
                            q[9] = (float)m.x; q[10] = (float)m.y; q[11] = (float)m.z; q[12] = (float)m.w;
                            q[13] = 0.f; q[14] = 0.f; q[15] = 0.f;            // accumulated_color is never updated there
                            q[16] = (float)(T(depth) / T(w.max_bounces)); q[17] = 0.f;
                            q[18] = (float)(T(S.g.sv.ids[hi]) / T(100)); q[19] = 0.5f; q[20] = 0.5f; q[21] = 0.5f;
                        }
                    }
                }
            }
        }
        need[i] = ask;
    }
    if (stats) {
        flush_stats(stats, STAT_INTER, n_inter); flush_stats(stats, STAT_LIGHT, n_light); flush_stats(stats, STAT_SMALL, n_small);
        flush_stats(stats, STAT_QUERIES, n_query); flush_stats(stats, STAT_SPHERE_TESTS, n_tests);
        flush_stats(stats, STAT_AABB_TESTS, n_boxes);
        flush_stats(stats, 7, n_fb);                      // stats[7]: fb_used
    }
    (void)n_live;
}

// direction from local spherical angles in the renderers' frame (tangent (1,0,0) when |n.z| > 0.9, :553-558)
template <typename T> RT_DEV V3<T> wf_local_to_world(V3<T> n, T st, T ct, T sp, T cp) {
    V3<T> tg = M<T>::fabs(n.z) > T(0.9) ? mk<T>(1, 0, 0) : cross(mk<T>(0, 0, 1), n);
    tg = normalise(tg);
    const V3<T> bt = normalise(cross(n, tg));
    const T lx = st * cp, ly = st * sp, lz = ct;
    V3<T> bd = normalise(mk<T>(lx * tg.x + ly * bt.x + lz * n.x, lx * tg.y + ly * bt.y + lz * n.y, lx * tg.z + ly * bt.z + lz * n.z));
    if constexpr (M<T>::exact) bd = normalise(bd);        // Ray() normalises again
    return bd;
}

template <typename T>
__global__ void __launch_bounds__(256) wf_bounce_kernel(WaveDev<T> w, const uint8_t *need, const float *actions,
                                                        unsigned long long *stats, int *live_count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned n_rays = 0, n_live = 0;
    if (i < w.P && w.state[i] == WF_PENDING) {
        const size_t P = (size_t)w.P;
        const V3<T> D = mk<T>(w.D[i], w.D[P + i], w.D[2 * P + i]);
        const V3<T> p = mk<T>(w.hp[i], w.hp[P + i], w.hp[2 * P + i]), n = mk<T>(w.hn[i], w.hn[P + i], w.hn[2 * P + i]);
        const int depth = w.depth[i];
        V3<T> nd;
        if (w.mirror[i]) nd = bounce_direction<T>(D, n, true, T(0), T(0));
        else if (need[i]) {
            const T theta = (T(actions[2 * i]) + T(1)) * T(3.14159265358979323846) / T(4);       // :545-546
            const T phi = T(actions[2 * i + 1]) * T(3.14159265358979323846);
            T st, ct, sp, cp;
            M<T>::sincos(theta, &st, &ct); M<T>::sincos(phi, &sp, &cp);
            nd = wf_local_to_world<T>(n, st, ct, sp, cp);
        } else {
            int x, y, s;
            wf_path_id<T>(w, i, x, y, s);
            PathRng rng;
            rng.begin((uint32_t)(y * w.W + x), (uint32_t)s, w.k0, w.k1);
            uint32_t wa, wb;
            rng.pair((uint32_t)depth + 1u, wa, wb);
            nd = bounce_direction<T>(D, n, false, u01<T>(wa), u01<T>(wb));
        }
        const V3<T> o2 = p + n * T(0.001);
        w.O[i] = o2.x; w.O[P + i] = o2.y; w.O[2 * P + i] = o2.z;
        w.D[i] = nd.x; w.D[P + i] = nd.y; w.D[2 * P + i] = nd.z;
        w.depth[i] = depth + 1;
        n_rays = 1;                                                   // the recursive call ...
        if (depth + 1 >= w.max_bounces) {                             // ... returns (2,2,5) at once
            w.state[i] = WF_DEAD; w.leaf[i] = 2.0; w.leaf[P + i] = 2.0; w.leaf[2 * P + i] = 5.0;
        } else { w.state[i] = WF_LIVE; n_live = 1; }
    }
    if (stats) flush_stats(stats, STAT_RAYS, n_rays);
    const unsigned long long live = warp_sum((unsigned long long)n_live);
    if ((threadIdx.x & 31) == 0 && live) atomicAdd(live_count, (int)live);
}

// fold (chandelier.py:509-521) in double with the true division (both builds), sums added to the pixel; kMoments: the
// squares and the count go into moments [H,W,4] as well (double atomics: exact for integer-valued squares)
template <typename T, bool kMoments>
__global__ void __launch_bounds__(256) wf_finish_kernel(SceneDev<T> sc, WaveDev<T> w, typename M<T>::v4 *accum,
                                                        typename std::conditional<kMoments, double *, PkNone>::type moments) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= w.P) return;
    const size_t P = (size_t)w.P;
    double c[3] = {w.leaf[i], w.leaf[P + i], w.leaf[2 * P + i]};
    const int depth = w.depth[i] < w.max_depth ? w.depth[i] : w.max_depth;
    for (int k = depth - 1; k >= 0; --k) {
        const typename M<T>::v4 col = sc.col[w.st_idx[(size_t)k * P + i]];
        const uint32_t d = w.st_direct[(size_t)k * P + i];
        double t0 = (double)(d & 255u) + c[0], t1 = (double)((d >> 8) & 255u) + c[1], t2 = (double)((d >> 16) & 255u) + c[2];
        t0 = t0 < 255.0 ? t0 : 255.0; t1 = t1 < 255.0 ? t1 : 255.0; t2 = t2 < 255.0 ? t2 : 255.0;
        c[0] = ::trunc(__dmul_rn((double)col.x, __ddiv_rn(t0, 255.0)));
        c[1] = ::trunc(__dmul_rn((double)col.y, __ddiv_rn(t1, 255.0)));
        c[2] = ::trunc(__dmul_rn((double)col.z, __ddiv_rn(t2, 255.0)));
    }
    int x, y, s;
    wf_path_id<T>(w, i, x, y, s);
    T *px = reinterpret_cast<T *>(accum + ((size_t)y * w.W + x));
    atomicAdd(px + 0, (T)c[0]); atomicAdd(px + 1, (T)c[1]); atomicAdd(px + 2, (T)c[2]); atomicAdd(px + 3, T(1));
    if constexpr (kMoments) {
        double *q = moments + 4 * ((size_t)y * w.W + x);
        atomicAdd(q + 0, __dmul_rn(c[0], c[0])); atomicAdd(q + 1, __dmul_rn(c[1], c[1])); atomicAdd(q + 2, __dmul_rn(c[2], c[2]));
        atomicAdd(q + 3, 1.0);
    }
}

// ------------------------------------------------------------------ launchers
template <typename T>
cudaError_t launch_wf_begin(const WaveDev<T> &w, const PathDev<T> &pp, unsigned long long *stats, cudaStream_t st) {
    if (w.P <= 0) return cudaSuccess;
    wf_begin_kernel<T><<<(w.P + 255) / 256, 256, 0, st>>>(w, pp, stats);
    return cudaGetLastError();
}
template <typename T>
cudaError_t launch_wf_trace(const SceneDev<T> &sc, const WaveDev<T> &w, float *obs, uint8_t *need, unsigned long long *stats,
                            cudaStream_t st) {
    if (w.P <= 0) return cudaSuccess;
    const int grid = (w.P + 255) / 256, block = 256;
    const int mode = mode_for(sc);
    RT_DISPATCH_MODE(mode, wf_trace_kernel, grid, block, smem_for(sc), st, sc, w, obs, need, stats);
    return cudaGetLastError();
}
template <typename T>
cudaError_t launch_wf_bounce(const WaveDev<T> &w, const uint8_t *need, const float *actions, unsigned long long *stats,
                             int *live_count, cudaStream_t st) {
    if (w.P <= 0) return cudaSuccess;
    wf_bounce_kernel<T><<<(w.P + 255) / 256, 256, 0, st>>>(w, need, actions, stats, live_count);
    return cudaGetLastError();
}
template <typename T>
cudaError_t launch_wf_finish(const SceneDev<T> &sc, const WaveDev<T> &w, void *accum, double *moments, cudaStream_t st) {
    if (w.P <= 0) return cudaSuccess;
    if (moments) wf_finish_kernel<T, true><<<(w.P + 255) / 256, 256, 0, st>>>(sc, w, (typename M<T>::v4 *)accum, moments);
    else wf_finish_kernel<T, false><<<(w.P + 255) / 256, 256, 0, st>>>(sc, w, (typename M<T>::v4 *)accum, PkNone());
    return cudaGetLastError();
}

#define RT_INSTANTIATE_WAVEFRONT(T)                                                                                       \
    template cudaError_t launch_wf_begin<T>(const WaveDev<T> &, const PathDev<T> &, unsigned long long *, cudaStream_t);  \
    template cudaError_t launch_wf_trace<T>(const SceneDev<T> &, const WaveDev<T> &, float *, uint8_t *,                  \
                                            unsigned long long *, cudaStream_t);                                         \
    template cudaError_t launch_wf_bounce<T>(const WaveDev<T> &, const uint8_t *, const float *, unsigned long long *,    \
                                             int *, cudaStream_t);                                                       \
    template cudaError_t launch_wf_finish<T>(const SceneDev<T> &, const WaveDev<T> &, void *, double *, cudaStream_t);

}  // namespace rt
