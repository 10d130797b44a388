// rt_f32.cu -- the FP32 product build of every kernel, plus the FFMA micro-benchmark that measures the FP32
// roofline denominator on the box (MEASURED_PEAKS.json has no FP32 figure).
#include "rt_kernels.cuh"
#include "rt_wavefront.cuh"
namespace rt {
RT_INSTANTIATE_LAUNCHERS(float)
RT_INSTANTIATE_WAVEFRONT(float)

// 16 independent accumulator chains per thread: enough ILP to cover the 4-cycle FFMA latency at any occupancy.
__global__ void __launch_bounds__(1024) fp32_peak_kernel(int iters, float *sink) {
    float a[16];
    const float x = 1.0f + 1e-7f * (float)threadIdx.x, y = 1e-7f * (float)blockIdx.x;
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = (float)k;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = fmaf(a[k], x, y);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += a[k];
    if (s == 123.456f) sink[0] = s;          // never true; keeps the chains alive
}

// resolve rows of an FP32 accumulator into the (possibly peer-mapped) image and clear them for the next frame
__global__ void resolve_clear_kernel(float4 *accum, int W, int y0, int y1, int spp, float *image, int clear) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t n = (size_t)(y1 - y0) * W;
    if (i >= n) return;
    const size_t o = (size_t)y0 * W + i;
    const float4 a = accum[o];
    const double s = (double)spp;
    const double r = floor((double)a.x / s) / 255.0, g = floor((double)a.y / s) / 255.0, b = floor((double)a.z / s) / 255.0;
    image[3 * o + 0] = (float)(r < 1.0 ? r : 1.0);
    image[3 * o + 1] = (float)(g < 1.0 ? g : 1.0);
    image[3 * o + 2] = (float)(b < 1.0 ? b : 1.0);
    if (clear) accum[o] = make_float4(0.f, 0.f, 0.f, 0.f);
}
cudaError_t launch_resolve_clear(float4 *accum, int W, int y0, int y1, int spp, float *image, int clear, cudaStream_t st) {
    const size_t n = (size_t)(y1 - y0) * W;
    if (n == 0) return cudaSuccess;
    resolve_clear_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(accum, W, y0, y1, spp, image, clear);
    return cudaGetLastError();
}

// resolve_clear_kernel plus the moments: the variance of the same rows into the (possibly peer-mapped) variance image
// (variance_of_mean, as rt_resolve_variance), and both buffers' rows cleared for the next frame
__global__ void resolve_clear_moments_kernel(float4 *accum, double4 *moments, int W, int y0, int y1, int spp, float *image,
                                             float *var, int clear) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t n = (size_t)(y1 - y0) * W;
    if (i >= n) return;
    const size_t o = (size_t)y0 * W + i;
    const float4 a = accum[o];
    const double4 q = moments[o];
    const double s = (double)spp;
    const double r = floor((double)a.x / s) / 255.0, g = floor((double)a.y / s) / 255.0, b = floor((double)a.z / s) / 255.0;
    image[3 * o + 0] = (float)(r < 1.0 ? r : 1.0);
    image[3 * o + 1] = (float)(g < 1.0 ? g : 1.0);
    image[3 * o + 2] = (float)(b < 1.0 ? b : 1.0);
    var[3 * o + 0] = variance_of_mean((double)a.x, q.x, q.w);
    var[3 * o + 1] = variance_of_mean((double)a.y, q.y, q.w);
    var[3 * o + 2] = variance_of_mean((double)a.z, q.z, q.w);
    if (clear) {
        accum[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        moments[o] = make_double4(0.0, 0.0, 0.0, 0.0);
    }
}
cudaError_t launch_resolve_clear_moments(float4 *accum, double4 *moments, int W, int y0, int y1, int spp, float *image,
                                         float *var, int clear, cudaStream_t st) {
    const size_t n = (size_t)(y1 - y0) * W;
    if (n == 0) return cudaSuccess;
    resolve_clear_moments_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(accum, moments, W, y0, y1, spp, image, var, clear);
    return cudaGetLastError();
}

// epoch flags in peer memory.  Signal: every write this stream issued before (kernel boundary) is ordered before the
// flag by the system fence + release store.  Wait: acquire loads until every flag has reached the epoch.
__global__ void peer_signal_kernel(PeerFlagTable flags, int n, unsigned epoch) {
    const int i = threadIdx.x;
    if (i >= n) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(flags.p[i]), "r"(epoch) : "memory");
}
__global__ void peer_wait_kernel(const unsigned *flags, int n, unsigned epoch, long long timeout_cycles, int *timed_out) {
    const int i = threadIdx.x;
    if (i >= n) return;
    const long long t0 = clock64();
    for (;;) {
        unsigned v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + i) : "memory");
        if ((int)(v - epoch) >= 0) break;
        if (clock64() - t0 > timeout_cycles) { if (timed_out) *timed_out = 1; break; }
        __nanosleep(200);
    }
    __threadfence_system();
}
cudaError_t launch_peer_signal(const PeerFlagTable &flags, int n, unsigned epoch, cudaStream_t st) {
    peer_signal_kernel<<<1, 32, 0, st>>>(flags, n, epoch);
    return cudaGetLastError();
}
cudaError_t launch_peer_wait(const unsigned *flags, int n, unsigned epoch, long long timeout_cycles, int *timed_out,
                             cudaStream_t st) {
    peer_wait_kernel<<<1, 32, 0, st>>>(flags, n, epoch, timeout_cycles, timed_out);
    return cudaGetLastError();
}

cudaError_t launch_fp32_peak(int blocks, int threads, int iters, float *sink, cudaStream_t st) {
    fp32_peak_kernel<<<blocks, threads, 0, st>>>(iters, sink);
    return cudaGetLastError();
}
}  // namespace rt
