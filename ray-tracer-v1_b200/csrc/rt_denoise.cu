// rt_denoise.cu -- variance-guided non-local-means filter of an Algorithm B frame (rt_denoise, DESIGN §4.8c).
// Both accum precisions are instantiated here, in one translation unit with the default contraction flags: the filter's
// arithmetic is FP32 for either, so both must compile it the same way (rt_f64.cu is built with -fmad=false).
//
// For pixel p with mean u_p = S_p / n_p (levels) and variance of the mean V_p (levels^2), per offset o in [-r, r]^2:
//   delta(p, q) = 1/3 sum_c [(u_p,c - u_q,c)^2 - (V_p,c + min(V_p,c, V_q,c))] / [eps + k^2 (V_p,c + V_q,c)]
//   D(p, o)     = mean of delta(p + t, p + t + o) over t in [-f, f]^2,   w = exp(-max(0, D))
//   out_p       = u_p + sum_o w (u_{p+o} - u_p) / sum_o w   -> image = min(1, floor(out) / 255)
// The sum is taken about the centre u_p so that a window of one colour returns u_p exactly: sum_o w u_{p+o} / sum_o w
// can round just below an integer u_p for fractional weights, and the floor then takes it one level down.
// every read at (x, y) clamped into the frame, the two pixels of a pair independently.
//
// kFeatures (rt_denoise_features, DESIGN §4.8d) adds the feature term of Rousselle, Manzi and Zwicker 2013, per pixel and
// without a patch.  For feature j (albedo, normal: 3 channels; depth: 1) with mean f_j, variance of the mean Var_j and
// gradient G_j,p = mean_c [((f(x+1,y) - f(x-1,y)) / 2)^2 + ((f(x,y+1) - f(x,y-1)) / 2)^2] (reads clamped):
//   Phi_j(p, q) = [mean_c (f_j,p - f_j,q)^2 - (Var_j,p + min(Var_j,p, Var_j,q))] / [k_f^2 max(tau, Var_j,p, G_j,p)]
//   w = min(w_c, exp(-max(0, max_j Phi_j))) = exp(-max(0, D, max_j Phi_j))
// The features of p and its denominators stay in registers; the (kTile + 2r)^2 halo of the 7 feature channels and the
// 3 variances is staged beside the colour halo.
#include "rt_launch.h"

namespace rt {

namespace {
constexpr int kTile = 16;                       // output tile side: one CTA of kTile^2 threads per tile
constexpr int kThreads = kTile * kTile;
constexpr int kMaxR = 15, kMaxF = 5;            // the ABI's limits on radius and patch_radius
constexpr int kMaxRegion = kTile + 2 * kMaxF;   // side of the region whose deltas a patch sum reads
constexpr int kRegionSlots = (kMaxRegion * kMaxRegion + kThreads - 1) / kThreads;        // region positions per thread
constexpr int kRowSlots = (kMaxRegion * kTile + kThreads - 1) / kThreads;                // row sums per thread
constexpr float kEps = 255.0f * 255.0f * 1e-10f;
}  // namespace

// dynamic shared memory: the halo of u and V (6 planes of L^2 floats, L = kTile + 2(r + f)), the deltas of the
// (kTile + 2f)^2 region, and their row sums ((kTile + 2f) rows x kTile columns)
// kFeatures: + the feature halo, 10 planes of LF^2 floats, LF = kTile + 2r
static size_t denoise_smem(int r, int f, bool features) {
    const size_t L = kTile + 2 * (r + f), R = kTile + 2 * f, LF = kTile + 2 * r;
    return (6 * L * L + R * R + R * kTile + (features ? 10 * LF * LF : 0)) * sizeof(float);
}

// kBand (rt_denoise_rows, DESIGN §4.8e): the output rows [y0, y1) of the frame; every row the filter reads is clamped
// into the window [lo, hi) = [max(0, y0 - h), min(H, y1 + h)) instead of [0, H).  For an output row in [y0, y1) every
// read lies in [y0 - h, y1 + h), where both clamps give the same row, so the band equals those rows of the whole frame.
struct DenoiseRows {
    int y0, y1, lo, hi;
};
// the frame row of the tile's first row, the first and last rows a read is clamped into, the end of the rows stored;
// without kBand, exactly the whole-frame kernels' expressions, so that their code does not change
template <bool kBand>
RT_DEV unsigned tile_row(const DenoiseRows &band) { return kBand ? band.y0 + blockIdx.y * kTile : blockIdx.y * kTile; }
template <bool kBand>
RT_DEV int first_row(const DenoiseRows &band) { return kBand ? band.lo : 0; }
template <bool kBand>
RT_DEV int last_row(int H, const DenoiseRows &band) { return kBand ? band.hi - 1 : H - 1; }
template <bool kBand>
RT_DEV int end_row(int H, const DenoiseRows &band) { return kBand ? band.y1 : H; }

// The filter of one CTA; kFeatures: with the feature term; kBand: of a row band.  Four kernels below call it, so that
// the whole-frame ones keep their parameter blocks.  tid = threadIdx.x, read in the kernel, where its range
// (__launch_bounds__) is known.
template <typename T, bool kFeatures, bool kBand>
RT_DEV void denoise_nlm(const typename M<T>::v4 *__restrict__ accum, const float *__restrict__ var, int W, int H, int r,
                        int f, float k2, float *__restrict__ image, const DenoiseFeatures &feat, const DenoiseRows &band,
                        const int tid) {
    extern __shared__ float smem[];
    const int L = kTile + 2 * (r + f), LL = L * L, R = kTile + 2 * f, RR = R * R;
    float *su = smem, *sv = smem + 3 * LL;      // su[c * LL + i], sv[c * LL + i]
    float *sd = sv + 3 * LL, *sr = sd + RR;
    const int x0 = blockIdx.x * kTile - (r + f), y0 = tile_row<kBand>(band) - (r + f);
    // kFeatures: sf[j * LFF + i], planes 0-2 albedo, 3-5 normal, 6 depth, 7-9 the variances of albedo, normal, depth
    const int LF = kTile + 2 * r, LFF = LF * LF;
    float *sf = sr + R * kTile;
    if constexpr (kFeatures) {
        const int fx0 = blockIdx.x * kTile - r, fy0 = tile_row<kBand>(band) - r;
        for (int i = tid; i < LFF; i += kThreads) {
            const int x = min(max(fx0 + i % LF, 0), W - 1);
            const int y = min(max(fy0 + i / LF, first_row<kBand>(band)), last_row<kBand>(H, band));
            const size_t o = (size_t)y * W + x;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                sf[c * LFF + i] = feat.albedo[3 * o + c];
                sf[(3 + c) * LFF + i] = feat.normal[3 * o + c];
                sf[(7 + c) * LFF + i] = feat.fvar[3 * o + c];
            }
            sf[6 * LFF + i] = feat.depth[o];
        }
    }

    // halo, with clamped reads: entry (i, j) holds pixel (clamp(x0 + j), clamp(y0 + i))
    for (int i = tid; i < LL; i += kThreads) {
        const int x = min(max(x0 + i % L, 0), W - 1);
        const int y = min(max(y0 + i / L, first_row<kBand>(band)), last_row<kBand>(H, band));
        const size_t o = (size_t)y * W + x;
        const typename M<T>::v4 a = accum[o];
        RT_ASSERT(a.w >= 1);
        const double n = (double)a.w;
        su[i] = (float)((double)a.x / n);
        su[LL + i] = (float)((double)a.y / n);
        su[2 * LL + i] = (float)((double)a.z / n);
        sv[i] = var[3 * o + 0];
        sv[LL + i] = var[3 * o + 1];
        sv[2 * LL + i] = var[3 * o + 2];
    }
    __syncthreads();

    // the region positions this thread computes deltas for: their first pixel stays in registers for every offset
    int hp[kRegionSlots];
    float up[kRegionSlots][3], vp[kRegionSlots][3];
#pragma unroll
    for (int s = 0; s < kRegionSlots; ++s) {
        const int j = tid + s * kThreads;
        hp[s] = j < RR ? (j / R + r) * L + (j % R + r) : 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            up[s][c] = su[c * LL + hp[s]];
            vp[s][c] = sv[c * LL + hp[s]];
        }
    }
    // row sums: row j / kTile of the region, columns [j % kTile, j % kTile + 2f]
    int rs[kRowSlots];
#pragma unroll
    for (int s = 0; s < kRowSlots; ++s) {
        const int j = tid + s * kThreads;
        rs[s] = (j / kTile) * R + j % kTile;
    }
    const int px = tid % kTile, py = tid / kTile;
    const int hc = (py + r + f) * L + (px + r + f);           // this thread's output pixel in the halo
    const int P = 2 * f + 1;
    const float inv_area = 1.0f / (float)(P * P);
    float sw = 0.f, s0 = 0.f, s1 = 0.f, s2 = 0.f;
    const float uc0 = su[hc], uc1 = su[LL + hc], uc2 = su[2 * LL + hc];
    // kFeatures: p's features, variances and 1 / (k_f^2 max(tau, Var_j,p, G_j,p)); G from clamped global reads
    float fp[7], vfp[3], inv_den[3];
    const int hcf = (py + r) * LF + (px + r);                // this thread's output pixel in the feature halo
    if constexpr (kFeatures) {
#pragma unroll
        for (int c = 0; c < 7; ++c) fp[c] = sf[c * LFF + hcf];
#pragma unroll
        for (int j = 0; j < 3; ++j) vfp[j] = sf[(7 + j) * LFF + hcf];
        const int xc = min(blockIdx.x * kTile + px, W - 1), yc = min(tile_row<kBand>(band) + py, last_row<kBand>(H, band));
        const size_t oxm = (size_t)yc * W + max(xc - 1, 0), oxp = (size_t)yc * W + min(xc + 1, W - 1);
        const size_t oym = (size_t)max(yc - 1, first_row<kBand>(band)) * W + xc;
        const size_t oyp = (size_t)min(yc + 1, last_row<kBand>(H, band)) * W + xc;
        float g[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float gx = 0.5f * (feat.albedo[3 * oxp + c] - feat.albedo[3 * oxm + c]);
            float gy = 0.5f * (feat.albedo[3 * oyp + c] - feat.albedo[3 * oym + c]);
            g[0] += gx * gx + gy * gy;
            gx = 0.5f * (feat.normal[3 * oxp + c] - feat.normal[3 * oxm + c]);
            gy = 0.5f * (feat.normal[3 * oyp + c] - feat.normal[3 * oym + c]);
            g[1] += gx * gx + gy * gy;
        }
        const float gx = 0.5f * (feat.depth[oxp] - feat.depth[oxm]), gy = 0.5f * (feat.depth[oyp] - feat.depth[oym]);
        g[0] *= 1.0f / 3.0f; g[1] *= 1.0f / 3.0f; g[2] = gx * gx + gy * gy;
#pragma unroll
        for (int j = 0; j < 3; ++j) inv_den[j] = 1.0f / (feat.kf2 * fmaxf(feat.tau, fmaxf(vfp[j], g[j])));
    }

    for (int oy = -r; oy <= r; ++oy) {
        for (int ox = -r; ox <= r; ++ox) {
            const int d = oy * L + ox;
#pragma unroll
            for (int s = 0; s < kRegionSlots; ++s) {
                const int j = tid + s * kThreads;
                if (j < RR) {
                    const int q = hp[s] + d;
                    float acc = 0.f;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const float uq = su[c * LL + q], vq = sv[c * LL + q];
                        const float du = up[s][c] - uq, vs = vp[s][c] + vq;
                        const float num = du * du - (vp[s][c] + fminf(vp[s][c], vq));
                        acc += __fdividef(num, kEps + k2 * vs);
                    }
                    sd[j] = acc * (1.0f / 3.0f);
                }
            }
            __syncthreads();
#pragma unroll
            for (int s = 0; s < kRowSlots; ++s) {
                const int j = tid + s * kThreads;
                if (j < R * kTile) {
                    float acc = 0.f;
                    for (int t = 0; t < P; ++t) acc += sd[rs[s] + t];
                    sr[j] = acc;
                }
            }
            __syncthreads();
            float D = 0.f;
            for (int t = 0; t < P; ++t) D += sr[(py + t) * kTile + px];
            float e = D * inv_area;
            if constexpr (kFeatures) {
                // fmaxf drops a NaN (0 * inf with tau = 0 between equal features): such a feature does not lower w
                const int qf = hcf + oy * LF + ox;
                float da = 0.f, dm = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float a = fp[c] - sf[c * LFF + qf], b = fp[3 + c] - sf[(3 + c) * LFF + qf];
                    da = fmaf(a, a, da);
                    dm = fmaf(b, b, dm);
                }
                const float dz = fp[6] - sf[6 * LFF + qf];
                const float va = sf[7 * LFF + qf], vm = sf[8 * LFF + qf], vz = sf[9 * LFF + qf];
                const float pa = (da * (1.0f / 3.0f) - (vfp[0] + fminf(vfp[0], va))) * inv_den[0];
                const float pm = (dm * (1.0f / 3.0f) - (vfp[1] + fminf(vfp[1], vm))) * inv_den[1];
                const float pz = (dz * dz - (vfp[2] + fminf(vfp[2], vz))) * inv_den[2];
                e = fmaxf(e, fmaxf(fmaxf(pa, pm), pz));
            }
            const float w = __expf(-fmaxf(0.f, e));
            const int q = hc + d;
            sw += w;
            s0 = fmaf(w, su[q] - uc0, s0);
            s1 = fmaf(w, su[LL + q] - uc1, s1);
            s2 = fmaf(w, su[2 * LL + q] - uc2, s2);
        }
    }

    const int x = blockIdx.x * kTile + px, y = tile_row<kBand>(band) + py;
    if (x >= W || y >= end_row<kBand>(H, band)) return;
    // o = 0 has weight 1, so sw >= 1; the lattice is rt_resolve's: min(1, floor(value) / 255) rounded from double
    const float vals[3] = {uc0 + s0 / sw, uc1 + s1 / sw, uc2 + s2 / sw};
    const size_t o = (size_t)y * W + x;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const double v = floor((double)vals[c]) / 255.0;
        image[3 * o + c] = (float)(v < 1.0 ? v : 1.0);
    }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) denoise_nlm_kernel(const typename M<T>::v4 *__restrict__ accum,
                                                               const float *__restrict__ var, int W, int H, int r, int f,
                                                               float k2, float *__restrict__ image) {
    denoise_nlm<T, false, false>(accum, var, W, H, r, f, k2, image, DenoiseFeatures{}, DenoiseRows{}, threadIdx.x);
}

template <typename T>
__global__ void __launch_bounds__(kThreads) denoise_nlm_features_kernel(const typename M<T>::v4 *__restrict__ accum,
                                                                        const float *__restrict__ var, int W, int H, int r,
                                                                        int f, float k2, float *__restrict__ image,
                                                                        const __grid_constant__ DenoiseFeatures feat) {
    denoise_nlm<T, true, false>(accum, var, W, H, r, f, k2, image, feat, DenoiseRows{}, threadIdx.x);
}

template <typename T>
__global__ void __launch_bounds__(kThreads) denoise_nlm_rows_kernel(const typename M<T>::v4 *__restrict__ accum,
                                                                    const float *__restrict__ var, int W, int H, int r,
                                                                    int f, float k2, float *__restrict__ image,
                                                                    const DenoiseRows band) {
    denoise_nlm<T, false, true>(accum, var, W, H, r, f, k2, image, DenoiseFeatures{}, band, threadIdx.x);
}

template <typename T>
__global__ void __launch_bounds__(kThreads) denoise_nlm_features_rows_kernel(const typename M<T>::v4 *__restrict__ accum,
                                                                             const float *__restrict__ var, int W, int H,
                                                                             int r, int f, float k2,
                                                                             float *__restrict__ image,
                                                                             const __grid_constant__ DenoiseFeatures feat,
                                                                             const DenoiseRows band) {
    denoise_nlm<T, true, true>(accum, var, W, H, r, f, k2, image, feat, band, threadIdx.x);
}

template <typename K, typename... A>
static cudaError_t launch_nlm(K kernel, bool features, int W, int rows, int r, int f, cudaStream_t st, const A &...args) {
    if (r < 0 || r > kMaxR || f < 0 || f > kMaxF) return cudaErrorInvalidValue;
    const size_t smem = denoise_smem(r, f, features);
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const dim3 grid((unsigned)((W + kTile - 1) / kTile), (unsigned)((rows + kTile - 1) / kTile));
    kernel<<<grid, kThreads, smem, st>>>(args...);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_denoise(const void *accum, const float *var, int W, int H, int r, int f, float k, float *image,
                           cudaStream_t st) {
    return launch_nlm(denoise_nlm_kernel<T>, false, W, H, r, f, st, (const typename M<T>::v4 *)accum, var, W, H, r, f,
                      square_to_float(k), image);
}

template <typename T>
cudaError_t launch_denoise_features(const void *accum, const float *var, const DenoiseFeatures &feat, int W, int H, int r,
                                    int f, float k, float *image, cudaStream_t st) {
    return launch_nlm(denoise_nlm_features_kernel<T>, true, W, H, r, f, st, (const typename M<T>::v4 *)accum, var, W, H,
                      r, f, square_to_float(k), image, feat);
}

// the band [y0, y1) and its window: 0 <= y0 < y1 <= H is the caller's to check (rt_api.cu)
static DenoiseRows band_rows(int H, int y0, int y1, int r, int f, bool features) {
    const int h = denoise_halo(r, f, features);
    return DenoiseRows{y0, y1, max(0, y0 - h), min(H, y1 + h)};
}

template <typename T>
cudaError_t launch_denoise_rows(const void *accum, const float *var, int W, int H, int y0, int y1, int r, int f, float k,
                                float *image, cudaStream_t st) {
    return launch_nlm(denoise_nlm_rows_kernel<T>, false, W, y1 - y0, r, f, st, (const typename M<T>::v4 *)accum, var, W,
                      H, r, f, square_to_float(k), image, band_rows(H, y0, y1, r, f, false));
}

template <typename T>
cudaError_t launch_denoise_features_rows(const void *accum, const float *var, const DenoiseFeatures &feat, int W, int H,
                                         int y0, int y1, int r, int f, float k, float *image, cudaStream_t st) {
    return launch_nlm(denoise_nlm_features_rows_kernel<T>, true, W, y1 - y0, r, f, st, (const typename M<T>::v4 *)accum,
                      var, W, H, r, f, square_to_float(k), image, feat, band_rows(H, y0, y1, r, f, true));
}

template cudaError_t launch_denoise<float>(const void *, const float *, int, int, int, int, float, float *, cudaStream_t);
template cudaError_t launch_denoise<double>(const void *, const float *, int, int, int, int, float, float *, cudaStream_t);
template cudaError_t launch_denoise_features<float>(const void *, const float *, const DenoiseFeatures &, int, int, int, int,
                                                    float, float *, cudaStream_t);
template cudaError_t launch_denoise_features<double>(const void *, const float *, const DenoiseFeatures &, int, int, int,
                                                     int, float, float *, cudaStream_t);
template cudaError_t launch_denoise_rows<float>(const void *, const float *, int, int, int, int, int, int, float, float *,
                                                cudaStream_t);
template cudaError_t launch_denoise_rows<double>(const void *, const float *, int, int, int, int, int, int, float, float *,
                                                 cudaStream_t);
template cudaError_t launch_denoise_features_rows<float>(const void *, const float *, const DenoiseFeatures &, int, int, int,
                                                         int, int, int, float, float *, cudaStream_t);
template cudaError_t launch_denoise_features_rows<double>(const void *, const float *, const DenoiseFeatures &, int, int,
                                                          int, int, int, int, float, float *, cudaStream_t);

}  // namespace rt
