// rt_api.cu -- the C ABI of librt_b200.so (include/rt_b200.h): scene handles resident in HBM, parameter marshalling
// and stream-ordered launches of the kernels in rt_f32.cu / rt_f64.cu / rt_lbvh.cu.  No compute happens on the host.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/rt_b200.h"
#include "rt_launch.h"
#include "rt_lbvh_build.h"

using namespace rt;

#define RT_EXPORT extern "C" __attribute__((visibility("default")))

static thread_local std::string g_err;

static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
static int cuda_fail(cudaError_t e, const char *what) {
    return fail(RT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                                              \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

// ------------------------------------------------------------------ handles
template <typename T> struct SceneBufs {
    void *blob = nullptr;
    size_t bytes = 0;
    SceneDev<T> view;
};

#define RT_SCHED_SLOTS 64
struct rt_scene {
    int device = 0;
    int n = 0, nG = 0, nP = 0, nL = 0;
    unsigned long long version = 0;            // bumped by every upload (rt_scene_create / rt_scene_update)
    SceneBufs<float> f;
    SceneBufs<double> d;
    uint8_t *small_dev = nullptr;
    // Direction grids of Algorithm-A frames, resident per scene: an entry is uploaded ONCE (from a pinned copy it owns,
    // so the copy is asynchronous and nothing synchronises) and reused by every later frame with the same X[] / Y[]
    // values and precision; launches on other streams wait for the upload event.  Entries are never overwritten while
    // a kernel may read them: a changed grid gets a new entry, the oldest of RT_GRID_SLOTS is retired after a device sync.
    struct Grid {
        std::vector<double> key;      // X[0..W) then Y[0..H), as given
        int precision = 0;
        size_t nx = 0, ny = 0;
        void *dev = nullptr, *pinned = nullptr;
        cudaEvent_t ready = nullptr;
        cudaStream_t upload_stream = nullptr;
        bool settled = false;
    };
    std::vector<Grid> grids;
    mutable unsigned *heavy_dev = nullptr;   // warp-tile list of two-pass Algorithm-A frames (launch_whitted)
    mutable size_t heavy_cap = 0;
    // pinned staging area of scene uploads (FP32 blob, FP64 blob, small-light mask): the copies are asynchronous and
    // rt_scene_update never synchronises the stream; the next update waits for `staged` before it repacks the area
    unsigned char *stage = nullptr;
    size_t stage_bytes = 0;
    cudaEvent_t staged = nullptr;
    LbvhStorage bvh;              // rt_lbvh_build.h
    bool int_colours = false;     // every colour is an integer in [0, 65535]: the path kernel may fold in integers
    bool byte_colours = false;    // ... and <= 255: the fold may come from a byte table (PathDev::fold_tab)
    mutable unsigned *sched_dev = nullptr; // RT_SCHED_SLOTS x 4 work counters of the persistent path kernel (zero at rest)
    mutable std::atomic<unsigned> sched_next{0}; // launches rotate through the slots, so launches in flight never share a pair
    PkConst pkc;                  // host copy of the FP32 sphere pairs of a small scene (path kernel parameter block)
    bool pkc_ok = false;
};

struct rt_env {
    rt_scene *scene = nullptr;
    int precision = RT_F32;
    rt_env_desc desc;
    void *blob = nullptr;
    EnvDev<float> f;
    EnvDev<double> d;
    unsigned long long shaded_version = 0;      // rt_scene::version the cached shading (EnvDev::rgb) was computed with
};

template <typename T> static size_t scene_blob_bytes(int n, int nG, int nP, int nL) {
    const size_t v = sizeof(typename M<T>::v4);
    size_t b = v * (2 * (size_t)((n + 7) & ~7) + 2 * (size_t)n + 2 * (size_t)nG + 2 * (size_t)nP + 2 * (size_t)nL +
                    RT_LPK_STRIDE * (size_t)((nL + 1) / 2));
    b += sizeof(int) * ((size_t)n + nG + 2 * (size_t)nP + nL);
    return (b + 255) & ~size_t(255);
}

// Pack the double SoA description into the vec4 arrays of one precision (layout: rt_common.cuh "scene views").
template <typename T> static void pack_scene(const rt_scene_desc *s, unsigned char *host, size_t bytes) {
    using v4 = typename M<T>::v4;
    std::memset(host, 0, bytes);
    v4 *p = reinterpret_cast<v4 *>(host);
    const int n = s->n, nG = s->nG, nP = s->nP, nL = s->nL;
    const int n_pad = (n + 7) & ~7;          // brute_select reads whole groups of 8: pad with never-hit spheres
    v4 *sph = p; p += n_pad;
    for (int i = n; i < n_pad; ++i) { sph[i].x = sph[i].y = sph[i].z = (T)0; sph[i].w = std::numeric_limits<T>::quiet_NaN(); }
    v4 *pk = p; p += n_pad;                  // sphere pairs for the packed (f32x2) selection loop, rt_trace.cuh
    v4 *mat = p; p += n;
    v4 *col = p; p += n;
    v4 *g_vec = p; p += nG;
    v4 *g_col = p; p += nG;
    v4 *p_pos = p; p += nP;
    v4 *p_col = p; p += nP;
    v4 *l_pos = p; p += nL;
    v4 *l_col = p; p += nL;
    v4 *lpk = p; p += RT_LPK_STRIDE * ((nL + 1) / 2);    // light pairs for the packed direct-light loop, rt_trace.cuh
    int *q = reinterpret_cast<int *>(p);
    int *ids = q; q += n;
    int *g_func = q; q += nG;
    int *p_id = q; q += nP;
    int *p_func = q; q += nP;
    int *l_index = q; q += nL;
    for (int i = 0; i < n; ++i) {
        sph[i].x = (T)s->centre[3 * i]; sph[i].y = (T)s->centre[3 * i + 1]; sph[i].z = (T)s->centre[3 * i + 2];
        sph[i].w = (T)s->radius[i];
        mat[i].x = (T)s->material[4 * i]; mat[i].y = (T)s->material[4 * i + 1]; mat[i].z = (T)s->material[4 * i + 2];
        mat[i].w = (T)s->material[4 * i + 3];
        col[i].x = (T)s->colour[3 * i]; col[i].y = (T)s->colour[3 * i + 1]; col[i].z = (T)s->colour[3 * i + 2];
        col[i].w = (T)(1.0 / s->radius[i]);    // normal = (p - c) * (1/r) in the product path
        ids[i] = s->ids[i];
    }
    // pair j = spheres (2j, 2j+1): pk[2j] = (cx0 cx1 cy0 cy1), pk[2j+1] = (cz0 cz1 w0 w1), w = r^2 - |c|^2 evaluated
    // in double from the T-rounded centre and radius (NaN for padding spheres: never hit)
    for (int i = 0; i < n_pad; ++i) {
        const double cx = (double)sph[i].x, cy = (double)sph[i].y, cz = (double)sph[i].z, r = (double)sph[i].w;
        // padding spheres: w = -inf, so disc = -inf on every ray (never hit, and its sign bit lets the warp vote of
        // brute_select_pkc skip the pair; a NaN would read as "maybe")
        const T w = i < n ? (T)(r * r - (cx * cx + cy * cy + cz * cz)) : -std::numeric_limits<T>::infinity();
        v4 &a = pk[i & ~1], &b = pk[(i & ~1) + 1];
        if (i & 1) { a.y = sph[i].x; a.w = sph[i].y; b.y = sph[i].z; b.w = w; }
        else { a.x = sph[i].x; a.z = sph[i].y; b.x = sph[i].z; b.z = w; }
    }
    for (int i = 0; i < nG; ++i) {
        g_vec[i].x = (T)s->g_vec[3 * i]; g_vec[i].y = (T)s->g_vec[3 * i + 1]; g_vec[i].z = (T)s->g_vec[3 * i + 2];
        g_vec[i].w = (T)s->g_max_angle[i];
        g_col[i].x = (T)s->g_col[3 * i]; g_col[i].y = (T)s->g_col[3 * i + 1]; g_col[i].z = (T)s->g_col[3 * i + 2];
        g_col[i].w = (T)s->g_strength[i];
        g_func[i] = s->g_func[i];
    }
    for (int i = 0; i < nP; ++i) {
        p_pos[i].x = (T)s->p_pos[3 * i]; p_pos[i].y = (T)s->p_pos[3 * i + 1]; p_pos[i].z = (T)s->p_pos[3 * i + 2];
        p_pos[i].w = (T)s->p_max_angle[i];
        p_col[i].x = (T)s->p_col[3 * i]; p_col[i].y = (T)s->p_col[3 * i + 1]; p_col[i].z = (T)s->p_col[3 * i + 2];
        p_col[i].w = (T)s->p_strength[i];
        p_id[i] = s->p_id[i]; p_func[i] = s->p_func[i];
    }
    for (int i = 0; i < nL; ++i) {
        l_pos[i].x = (T)s->l_centre[3 * i]; l_pos[i].y = (T)s->l_centre[3 * i + 1]; l_pos[i].z = (T)s->l_centre[3 * i + 2];
        l_pos[i].w = (T)0;
        l_col[i].x = (T)s->l_colour[3 * i]; l_col[i].y = (T)s->l_colour[3 * i + 1]; l_col[i].z = (T)s->l_colour[3 * i + 2];
        l_col[i].w = (T)0;
        l_index[i] = s->l_index[i];
    }
    // pair j = lights (2j, 2j+1): lpk[4j] = 128*(x0 x1 y0 y1), lpk[4j+1] = (128*z0 128*z1 R0 R1), lpk[4j+2] = (G0 G1 B0 B1),
    // lpk[4j+3] = (|A0|^2 |A1|^2 0 0), A = the rounded 128 * centre as stored, with (R,G,B) = colour * 0.3 * 16384
    // (direct_light_pk saturates dn/d^3 / 16384 to [0,1]); the odd slot of the last pair is a black light at (128,0,0)/128
    // -- not at the origin, so that |A - 128 p|^2 cannot vanish for a hit point at the origin
    // An odd light count: light 0 sits ALONE in pair 0 (slot 1 = the filler) and lights 1.. fill the pairs behind it, so
    // that direct_light_pkc can shade the single light with scalar instructions at a compile-time address.
    const bool odd = (nL & 1) != 0;
    for (int slot = 0; slot < 2 * ((nL + 1) / 2); ++slot) {
        const int li = !odd ? slot : slot == 0 ? 0 : slot == 1 ? -1 : slot - 1;      // light held by this slot (-1: filler)
        const bool real = li >= 0 && li < nL;
        const int i = slot;
        const double x = real ? s->l_centre[3 * li] : 1.0, y = real ? s->l_centre[3 * li + 1] : 0.0, z = real ? s->l_centre[3 * li + 2] : 0.0;
        const double k = 0.3 * 16384.0;
        const double r = real ? s->l_colour[3 * li] * k : 0.0, g = real ? s->l_colour[3 * li + 1] * k : 0.0, b = real ? s->l_colour[3 * li + 2] * k : 0.0;
        v4 *t = lpk + RT_LPK_STRIDE * (i / 2);
        const T ax = (T)(128.0 * x), ay = (T)(128.0 * y), az = (T)(128.0 * z);
        const T aa = (T)((double)ax * (double)ax + (double)ay * (double)ay + (double)az * (double)az);
        if (i & 1) { t[0].y = ax; t[0].w = ay; t[1].y = az; t[1].w = (T)r; t[2].y = (T)g; t[2].w = (T)b; t[3].y = aa; t[3].w = (T)0; }
        else { t[0].x = ax; t[0].z = ay; t[1].x = az; t[1].z = (T)r; t[2].x = (T)g; t[2].z = (T)b; t[3].x = aa; t[3].z = (T)0; }
    }
}

template <typename T> static void bind_view(SceneBufs<T> &b, const rt_scene_desc *s, const uint8_t *small_dev) {
    using v4 = typename M<T>::v4;
    SceneDev<T> &v = b.view;
    const int n = s->n, nG = s->nG, nP = s->nP, nL = s->nL;
    v.n = n; v.nG = nG; v.nP = nP; v.nL = nL;
    v4 *p = reinterpret_cast<v4 *>(b.blob);
    v.sph = p; p += (n + 7) & ~7;
    v.pk = p; p += (n + 7) & ~7;
    v.mat = p; p += n;
    v.col = p; p += n;
    v.g_vec = p; p += nG;
    v.g_col = p; p += nG;
    v.p_pos = p; p += nP;
    v.p_col = p; p += nP;
    v.l_pos = p; p += nL;
    v.l_col = p; p += nL;
    v.lpk = p; p += RT_LPK_STRIDE * ((nL + 1) / 2);
    int *q = reinterpret_cast<int *>(p);
    v.ids = q; q += n;
    v.g_func = q; q += nG;
    v.p_id = q; q += nP;
    v.p_func = q; q += nP;
    v.l_index = q; q += nL;
    v.small = small_dev;
    v.key_mask = 0x7ffffff8; v.key_mask6 = 0x7fffffc0;
    v.bg[0] = (T)s->bg[0]; v.bg[1] = (T)s->bg[1]; v.bg[2] = (T)s->bg[2];
    std::memset(&v.bvh, 0, sizeof v.bvh);
}

static int validate_desc(const rt_scene_desc *s) {
    if (!s) return fail(RT_ERR_INVALID, "scene description is NULL");
    if (s->n < 0 || s->nG < 0 || s->nP < 0 || s->nL < 0) return fail(RT_ERR_INVALID, "negative count in scene description");
    if (s->n > 0 && (!s->centre || !s->radius || !s->material || !s->colour || !s->ids))
        return fail(RT_ERR_INVALID, "sphere arrays missing");
    if (s->nG > 0 && (!s->g_vec || !s->g_col || !s->g_strength || !s->g_max_angle || !s->g_func))
        return fail(RT_ERR_INVALID, "global light arrays missing");
    if (s->nP > 0 && (!s->p_id || !s->p_pos || !s->p_col || !s->p_strength || !s->p_max_angle || !s->p_func))
        return fail(RT_ERR_INVALID, "point light arrays missing");
    if (s->nL > 0 && (!s->l_centre || !s->l_colour || !s->l_index)) return fail(RT_ERR_INVALID, "light sphere arrays missing");
    for (int i = 0; i < s->nL; ++i)
        if (s->l_index[i] >= s->n) return fail(RT_ERR_INVALID, "l_index out of range");
    return RT_OK;
}

static int upload_scene(rt_scene *sc, const rt_scene_desc *s, cudaStream_t st) {
    CU(cudaSetDevice(sc->device));
    sc->version++;
    const bool same = sc->n == s->n && sc->nG == s->nG && sc->nP == s->nP && sc->nL == s->nL && sc->f.blob;
    if (!same) {
        if (sc->f.blob) CU(cudaFree(sc->f.blob));
        if (sc->d.blob) CU(cudaFree(sc->d.blob));
        if (sc->small_dev) CU(cudaFree(sc->small_dev));
        sc->f.blob = sc->d.blob = nullptr; sc->small_dev = nullptr;
        sc->f.bytes = scene_blob_bytes<float>(s->n, s->nG, s->nP, s->nL);
        sc->d.bytes = scene_blob_bytes<double>(s->n, s->nG, s->nP, s->nL);
        CU(cudaMalloc(&sc->f.blob, sc->f.bytes));
        CU(cudaMalloc(&sc->d.blob, sc->d.bytes));
        CU(cudaMalloc((void **)&sc->small_dev, (size_t)(s->n > 0 ? s->n : 1)));
    }
    sc->n = s->n; sc->nG = s->nG; sc->nP = s->nP; sc->nL = s->nL;
    sc->int_colours = true;
    for (int i = 0; i < 3 * s->n && sc->int_colours; ++i) {
        const double c = s->colour[i];
        if (!(c >= 0.0 && c <= 65535.0 && c == std::floor(c))) sc->int_colours = false;
    }
    sc->byte_colours = sc->int_colours;
    for (int i = 0; i < 3 * s->n && sc->byte_colours; ++i)
        if (s->colour[i] > 255.0) sc->byte_colours = false;
    // pack into the pinned staging area and copy from there: nothing below waits for the stream
    const size_t n_small = (size_t)(s->n > 0 ? s->n : 1);
    const size_t need = sc->f.bytes + sc->d.bytes + ((n_small + 255) & ~size_t(255));
    if (!sc->staged) CU(cudaEventCreateWithFlags(&sc->staged, cudaEventDisableTiming));
    else CU(cudaEventSynchronize(sc->staged));          // the previous upload has left the staging area (long ago)
    if (need > sc->stage_bytes) {
        if (sc->stage) CU(cudaFreeHost(sc->stage));
        sc->stage = nullptr; sc->stage_bytes = 0;
        CU(cudaMallocHost((void **)&sc->stage, need));
        sc->stage_bytes = need;
    }
    unsigned char *hf = sc->stage, *hd = sc->stage + sc->f.bytes, *hs = hd + sc->d.bytes;
    pack_scene<float>(s, hf, sc->f.bytes);
    pack_scene<double>(s, hd, sc->d.bytes);
    std::memset(hs, 0, n_small);
    if (s->small) std::memcpy(hs, s->small, (size_t)s->n);
    CU(cudaMemcpyAsync(sc->f.blob, hf, sc->f.bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(sc->d.blob, hd, sc->d.bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(sc->small_dev, hs, n_small, cudaMemcpyHostToDevice, st));
    if (!sc->sched_dev) {                   // work counters of the persistent path kernel: zero at rest, re-armed by every launch
        CU(cudaMalloc((void **)&sc->sched_dev, 4 * RT_SCHED_SLOTS * sizeof(unsigned)));
        CU(cudaMemsetAsync(sc->sched_dev, 0, 4 * RT_SCHED_SLOTS * sizeof(unsigned), st));
    }
    CU(cudaEventRecord(sc->staged, st));
    {   // small scenes: the path kernel takes the FP32 pair array through its parameter block (kMode 3)
        const int n_pad = (s->n + 7) & ~7;
        sc->pkc_ok = n_pad > 0 && n_pad <= RT_PKC_MAX && s->nL <= RT_LPKC_MAX;
        std::memset(&sc->pkc, 0, sizeof sc->pkc);
        if (sc->pkc_ok) {
            // blob layout (pack_scene): sph[n_pad] pk[n_pad] mat[n] col[n] g_vec g_col [nG] p_pos p_col [nP] l_pos l_col [nL] lpk
            const float4 *v = reinterpret_cast<const float4 *>(hf);
            std::memcpy(sc->pkc.q, v + n_pad, (size_t)n_pad * sizeof(float4));
            const size_t lpk_at = 2 * (size_t)n_pad + 2 * (size_t)s->n + 2 * (size_t)s->nG + 2 * (size_t)s->nP + 2 * (size_t)s->nL;
            std::memcpy(sc->pkc.l, v + lpk_at, RT_LPK_STRIDE * (size_t)((s->nL + 1) / 2) * sizeof(float4));
        }
    }
    bind_view<float>(sc->f, s, sc->small_dev);
    bind_view<double>(sc->d, s, sc->small_dev);
    lbvh_drop(sc->bvh);                     // geometry changed: any hierarchy is stale
    return RT_OK;
}

#define RT_GRID_SLOTS 8
static void grid_free(rt_scene::Grid &g) {
    if (g.dev) cudaFree(g.dev);
    if (g.pinned) cudaFreeHost(g.pinned);
    if (g.ready) cudaEventDestroy(g.ready);
    g.dev = g.pinned = nullptr; g.ready = nullptr;
}

// device copy of the (X, Y) direction grid in precision T, ordered before anything launched on `st` after the call
template <typename T> static int resident_grid(rt_scene *sc, const rt_whitted_params *p, cudaStream_t st, const T **out) {
    const size_t nx = (size_t)p->W, ny = (size_t)p->H;
    const int prec = sizeof(T) == 8 ? RT_F64 : RT_F32;
    for (rt_scene::Grid &g : sc->grids) {
        if (g.precision != prec || g.nx != nx || g.ny != ny) continue;
        if (std::memcmp(g.key.data(), p->X, nx * sizeof(double)) || std::memcmp(g.key.data() + nx, p->Y, ny * sizeof(double))) continue;
        if (!g.settled) {
            if (cudaEventQuery(g.ready) == cudaSuccess) g.settled = true;
            else if (st != g.upload_stream) CU(cudaStreamWaitEvent(st, g.ready, 0));
        }
        *out = reinterpret_cast<const T *>(g.dev);
        return RT_OK;
    }
    if (sc->grids.size() >= RT_GRID_SLOTS) {          // retire the oldest entry: no kernel may still be reading it
        CU(cudaDeviceSynchronize());
        grid_free(sc->grids.front());
        sc->grids.erase(sc->grids.begin());
    }
    rt_scene::Grid g;
    g.precision = prec; g.nx = nx; g.ny = ny;
    g.key.assign(p->X, p->X + nx);
    g.key.insert(g.key.end(), p->Y, p->Y + ny);
    cudaError_t e = cudaMallocHost(&g.pinned, (nx + ny) * sizeof(T));
    if (e == cudaSuccess) e = cudaMalloc(&g.dev, (nx + ny) * sizeof(T));
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g.ready, cudaEventDisableTiming);
    if (e == cudaSuccess) {
        T *h = reinterpret_cast<T *>(g.pinned);
        for (size_t i = 0; i < nx + ny; ++i) h[i] = (T)g.key[i];
        e = cudaMemcpyAsync(g.dev, g.pinned, (nx + ny) * sizeof(T), cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess) e = cudaEventRecord(g.ready, st);
    if (e != cudaSuccess) { grid_free(g); return cuda_fail(e, "direction grid upload"); }
    g.upload_stream = st;
    *out = reinterpret_cast<const T *>(g.dev);
    sc->grids.push_back(std::move(g));
    return RT_OK;
}

static inline cudaStream_t S(void *stream) { return reinterpret_cast<cudaStream_t>(stream); }

// ------------------------------------------------------------------ library / device
RT_EXPORT const char *rt_last_error(void) { return g_err.c_str(); }
RT_EXPORT int rt_version(void) { return 100; }

RT_EXPORT int rt_device_count(int *count) {
    if (!count) return fail(RT_ERR_INVALID, "count is NULL");
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess) { *count = 0; return cuda_fail(e, "cudaGetDeviceCount"); }
    return RT_OK;
}

// cudaDeviceGetAttribute, asked once per (device, attribute): the clock rate is a slow query.  Failures are not cached.
static cudaError_t device_attr(int dev, cudaDeviceAttr attr, int *value) {
    struct Entry { int dev; cudaDeviceAttr attr; int value; };
    static std::mutex mu;
    static std::vector<Entry> cache;
    std::lock_guard<std::mutex> lock(mu);
    for (const Entry &c : cache)
        if (c.dev == dev && c.attr == attr) { *value = c.value; return cudaSuccess; }
    const cudaError_t e = cudaDeviceGetAttribute(value, attr, dev);
    if (e == cudaSuccess) cache.push_back(Entry{dev, attr, *value});
    return e;
}

RT_EXPORT int rt_device_props(int device, int64_t *props6, size_t *total_mem) {
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    int khz = 0;
    CU(device_attr(device, cudaDevAttrClockRate, &khz));
    if (props6) {
        props6[0] = p.multiProcessorCount; props6[1] = p.major; props6[2] = p.minor; props6[3] = khz;
        props6[4] = p.l2CacheSize; props6[5] = (int64_t)p.sharedMemPerBlockOptin;
    }
    if (total_mem) *total_mem = p.totalGlobalMem;
    return RT_OK;
}

RT_EXPORT int rt_dev_alloc(int device, size_t bytes, void **out_dev) {
    if (!out_dev) return fail(RT_ERR_INVALID, "out_dev is NULL");
    CU(cudaSetDevice(device));
    cudaError_t e = cudaMalloc(out_dev, bytes ? bytes : 1);
    if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); return fail(RT_ERR_NOMEM, "cudaMalloc: out of device memory"); }
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    return RT_OK;
}
RT_EXPORT int rt_dev_free(int device, void *ptr_dev) {
    CU(cudaSetDevice(device));
    CU(cudaFree(ptr_dev));
    return RT_OK;
}
RT_EXPORT int rt_host_alloc_pinned(size_t bytes, void **out_host) {
    if (!out_host) return fail(RT_ERR_INVALID, "out_host is NULL");
    CU(cudaHostAlloc(out_host, bytes ? bytes : 1, cudaHostAllocDefault));
    return RT_OK;
}
RT_EXPORT int rt_host_free_pinned(void *ptr_host) {
    CU(cudaFreeHost(ptr_host));
    return RT_OK;
}
RT_EXPORT int rt_memcpy_h2d(int device, void *dst_dev, const void *src_host, size_t bytes, void *stream) {
    CU(cudaSetDevice(device));
    CU(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, S(stream)));
    return RT_OK;
}
RT_EXPORT int rt_memcpy_d2h(int device, void *dst_host, const void *src_dev, size_t bytes, void *stream) {
    CU(cudaSetDevice(device));
    CU(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, S(stream)));
    return RT_OK;
}
RT_EXPORT int rt_memset_dev(int device, void *dst_dev, int value, size_t bytes, void *stream) {
    CU(cudaSetDevice(device));
    CU(cudaMemsetAsync(dst_dev, value, bytes, S(stream)));
    return RT_OK;
}
RT_EXPORT int rt_stream_sync(int device, void *stream) {
    CU(cudaSetDevice(device));
    CU(cudaStreamSynchronize(S(stream)));
    return RT_OK;
}

// a second stream for copies that overlap the next kernel, and "stream A waits for what stream B holds now"
RT_EXPORT int rt_stream_create(int device, void **out_stream) {
    if (!out_stream) return fail(RT_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(device));
    cudaStream_t s = nullptr;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *out_stream = s;
    return RT_OK;
}
RT_EXPORT int rt_stream_destroy(int device, void *stream) {
    if (!stream) return RT_OK;
    CU(cudaSetDevice(device));
    CU(cudaStreamDestroy(S(stream)));
    return RT_OK;
}
RT_EXPORT int rt_stream_wait_stream(int device, void *waiter, void *waited) {
    CU(cudaSetDevice(device));
    cudaEvent_t e = nullptr;
    CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    cudaError_t rc = cudaEventRecord(e, S(waited));
    if (rc == cudaSuccess) rc = cudaStreamWaitEvent(S(waiter), e, 0);
    cudaEventDestroy(e);                      // released once the recorded work has completed
    if (rc != cudaSuccess) return cuda_fail(rc, "rt_stream_wait_stream");
    return RT_OK;
}

RT_EXPORT int rt_measure_fp32_peak(int device, int repeats, double *tflops_out, double *ms_out) {
    CU(cudaSetDevice(device));
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    float *sink = nullptr;
    CU(cudaMalloc((void **)&sink, 4));
    const int blocks = p.multiProcessorCount * 2, threads = 1024, iters = 1 << 14;
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    CU(launch_fp32_peak(blocks, threads, 256, sink, nullptr));           // warm-up
    CU(cudaDeviceSynchronize());
    double best_ms = 1e30;
    for (int r = 0; r < (repeats > 0 ? repeats : 1); ++r) {
        CU(cudaEventRecord(a, nullptr));
        CU(launch_fp32_peak(blocks, threads, iters, sink, nullptr));
        CU(cudaEventRecord(b, nullptr));
        CU(cudaEventSynchronize(b));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, a, b));
        if (ms < best_ms) best_ms = ms;
    }
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(sink);
    const double flop = 2.0 * 16.0 * (double)iters * (double)threads * (double)blocks;
    if (tflops_out) *tflops_out = flop / (best_ms * 1e-3) / 1e12;
    if (ms_out) *ms_out = best_ms;
    return RT_OK;
}

// ------------------------------------------------------------------ scene
RT_EXPORT int rt_scene_create(int device, const rt_scene_desc *desc, rt_scene **out) {
    if (!out) return fail(RT_ERR_INVALID, "out is NULL");
    *out = nullptr;
    int rc = validate_desc(desc);
    if (rc) return rc;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    if (device < 0 || device >= count) return fail(RT_ERR_INVALID, "no such CUDA device");
    rt_scene *sc = new (std::nothrow) rt_scene();
    if (!sc) return fail(RT_ERR_NOMEM, "host allocation failed");
    sc->device = device;
    rc = upload_scene(sc, desc, nullptr);
    if (rc) { rt_scene_destroy(sc); return rc; }
    *out = sc;
    return RT_OK;
}

RT_EXPORT int rt_scene_update(rt_scene *scene, const rt_scene_desc *desc, void *stream) {
    if (!scene) return fail(RT_ERR_INVALID, "scene is NULL");
    int rc = validate_desc(desc);
    if (rc) return rc;
    return upload_scene(scene, desc, S(stream));
}

RT_EXPORT int rt_scene_destroy(rt_scene *scene) {
    if (!scene) return RT_OK;
    cudaSetDevice(scene->device);
    lbvh_drop(scene->bvh);
    if (scene->f.blob) cudaFree(scene->f.blob);
    if (scene->d.blob) cudaFree(scene->d.blob);
    if (scene->small_dev) cudaFree(scene->small_dev);
    if (scene->sched_dev) cudaFree(scene->sched_dev);
    if (scene->heavy_dev) cudaFree(scene->heavy_dev);
    if (scene->stage) cudaFreeHost(scene->stage);
    if (scene->staged) cudaEventDestroy(scene->staged);
    for (rt_scene::Grid &g : scene->grids) grid_free(g);
    scene->grids.clear();
    delete scene;
    return RT_OK;
}

RT_EXPORT int rt_scene_info(const rt_scene *scene, int32_t *n_spheres, int32_t *device, int32_t *has_lbvh) {
    if (!scene) return fail(RT_ERR_INVALID, "scene is NULL");
    if (n_spheres) *n_spheres = scene->n;
    if (device) *device = scene->device;
    if (has_lbvh) *has_lbvh = scene->bvh.view.nodes > 0;
    return RT_OK;
}

RT_EXPORT int rt_lbvh_build(rt_scene *scene, double huge_radius, void *stream) {
    if (!scene) return fail(RT_ERR_INVALID, "scene is NULL");
    CU(cudaSetDevice(scene->device));
    cudaError_t e = lbvh_build(scene->bvh, scene->f.view.sph, scene->n, (float)huge_radius, S(stream));
    if (e != cudaSuccess) return cuda_fail(e, "lbvh_build");
    scene->f.view.bvh = scene->bvh.view;
    scene->d.view.bvh = scene->bvh.view;
    return RT_OK;
}

RT_EXPORT int rt_lbvh_drop(rt_scene *scene) {
    if (!scene) return fail(RT_ERR_INVALID, "scene is NULL");
    CU(cudaSetDevice(scene->device));
    lbvh_drop(scene->bvh);
    std::memset(&scene->f.view.bvh, 0, sizeof(BvhView));
    std::memset(&scene->d.view.bvh, 0, sizeof(BvhView));
    return RT_OK;
}

// ------------------------------------------------------------------ batched primitives
RT_EXPORT int rt_sphere_discriminant(int device, int precision, int m, const double *rays_dev, const double *spheres_dev,
                                     int point, double *out_dev, void *stream) {
    if (m < 0 || (m > 0 && (!rays_dev || !spheres_dev || !out_dev))) return fail(RT_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(device));
    if (precision == RT_F64) CU(launch_sphere_disc<double>(m, rays_dev, spheres_dev, point, out_dev, S(stream)));
    else if (precision == RT_F32) CU(launch_sphere_disc<float>(m, rays_dev, spheres_dev, point, out_dev, S(stream)));
    else return fail(RT_ERR_INVALID, "unknown precision");
    return RT_OK;
}

RT_EXPORT int rt_trace_rays(rt_scene *scene, int precision, int m, const double *rays_dev, const int32_t *suppress_dev,
                            const int32_t *bounces0_dev, const int32_t *through0_dev, int max_bounces,
                            int shadow_max_bounces, const double miss[3], double *term_dev, double *rgb_dev,
                            void *stream) {
    if (!scene) return fail(RT_ERR_INVALID, "scene is NULL");
    if (m < 0 || (m > 0 && (!rays_dev || !term_dev))) return fail(RT_ERR_INVALID, "bad arguments");
    const double zero[3] = {0, 0, 0};
    if (!miss) miss = zero;
    CU(cudaSetDevice(scene->device));
    if (precision == RT_F64)
        CU(launch_trace_rays<double>(scene->d.view, m, rays_dev, suppress_dev, bounces0_dev, through0_dev, max_bounces,
                                     shadow_max_bounces, miss, term_dev, rgb_dev, S(stream)));
    else if (precision == RT_F32)
        CU(launch_trace_rays<float>(scene->f.view, m, rays_dev, suppress_dev, bounces0_dev, through0_dev, max_bounces,
                                    shadow_max_bounces, miss, term_dev, rgb_dev, S(stream)));
    else return fail(RT_ERR_INVALID, "unknown precision");
    return RT_OK;
}

RT_EXPORT int rt_terminal_rgb(rt_scene *scene, int precision, int m, const double *hits_dev, int shadow_max_bounces,
                              double *rgb_dev, void *stream) {
    if (!scene) return fail(RT_ERR_INVALID, "scene is NULL");
    if (m < 0 || (m > 0 && (!hits_dev || !rgb_dev))) return fail(RT_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(scene->device));
    if (precision == RT_F64) CU(launch_shade_hits<double>(scene->d.view, m, hits_dev, shadow_max_bounces, rgb_dev, S(stream)));
    else if (precision == RT_F32) CU(launch_shade_hits<float>(scene->f.view, m, hits_dev, shadow_max_bounces, rgb_dev, S(stream)));
    else return fail(RT_ERR_INVALID, "unknown precision");
    return RT_OK;
}

// ------------------------------------------------------------------ Algorithm A frame
template <typename T>
static int render_whitted_t(rt_scene *sc, const SceneDev<T> &view, const rt_whitted_params *p, void *accum, int32_t *hit,
                            uint64_t *stats, cudaStream_t st) {
    const size_t nx = (size_t)p->W;
    const T *grid = nullptr;
    int rc = resident_grid<T>(sc, p, st, &grid);      // no copy and no synchronisation once the grid is resident
    if (rc) return rc;
    WhittedDev<T> wp;
    wp.cam[0] = (T)p->cam[0]; wp.cam[1] = (T)p->cam[1]; wp.cam[2] = (T)p->cam[2];
    wp.X = grid;
    wp.Y = wp.X + nx;
    wp.W = p->W; wp.H = p->H; wp.y0 = p->y0; wp.y1 = p->y1; wp.s0 = p->s0; wp.s1 = p->s1; wp.spp = p->spp;
    wp.max_bounces = p->max_bounces; wp.shadow_max_bounces = p->shadow_max_bounces;
    wp.miss[0] = (T)p->miss[0]; wp.miss[1] = (T)p->miss[1]; wp.miss[2] = (T)p->miss[2];
    wp.pitch_x = (T)(p->W > 1 ? p->X[1] - p->X[0] : 0.0);
    wp.pitch_y = (T)(p->H > 1 ? p->Y[0] - p->Y[1] : 0.0);
    wp.k0 = (uint32_t)p->seed; wp.k1 = (uint32_t)(p->seed >> 32);
    wp.prenorm = p->prenormalise; wp.accumulate = p->accumulate;
    if (!sc->sched_dev) return fail(RT_ERR_INVALID, "scene has no scheduler counters (upload failed?)");
    const unsigned slot = sc->sched_next.fetch_add(1u) % RT_SCHED_SLOTS;
    unsigned *sched = sc->sched_dev + 4 * slot;
    // two-pass schedule (pass 1 lists the tiles a sphere can be seen in, pass 2 spreads their samples over the device):
    // FP32 reductions in no fixed order, so only for integer-valued background / miss colours (sums then exact).  Every
    // counter slot has its own tile list, so frames in flight on different streams do not share one
    unsigned *sched2 = nullptr, *heavy = nullptr;
    if (sizeof(T) == 4 && p->s1 - p->s0 >= 4 && p->s1 - p->s0 <= 4096) {
        bool ints = true;
        for (int k = 0; k < 3; ++k) {
            const double a = p->miss[k], b = (double)view.bg[k];
            ints = ints && a == std::floor(a) && b == std::floor(b) && std::fabs(a) <= 1024.0 && std::fabs(b) <= 1024.0;
        }
        const size_t tiles = (size_t)((p->W + 31) / 32) * (size_t)((p->y1 - p->y0 + 7) / 8) * 8;
        if (ints && tiles > 0) {
            if (tiles > sc->heavy_cap) {               // (cudaFree waits for the launches that may still read the old lists)
                if (sc->heavy_dev) CU(cudaFree(sc->heavy_dev));
                sc->heavy_dev = nullptr; sc->heavy_cap = 0;
                CU(cudaMalloc((void **)&sc->heavy_dev, (size_t)RT_SCHED_SLOTS * tiles * sizeof(unsigned)));
                sc->heavy_cap = tiles;
            }
            heavy = sc->heavy_dev + (size_t)slot * sc->heavy_cap;
            sched2 = sc->sched_dev + 4 * (sc->sched_next.fetch_add(1u) % RT_SCHED_SLOTS);
        }
    }
    CU(launch_whitted<T>(view, wp, accum, hit, reinterpret_cast<unsigned long long *>(stats), st, sched, sched2, heavy));
    return RT_OK;
}

static int check_band(int W, int H, int y0, int y1, int s0, int s1) {
    if (W <= 0 || H <= 0) return fail(RT_ERR_INVALID, "image size must be positive");
    if (y0 < 0 || y1 > H || y0 > y1) return fail(RT_ERR_INVALID, "row band outside the image");
    if (s0 < 0 || s0 > s1) return fail(RT_ERR_INVALID, "bad sample range");
    if ((long long)W * H > 0x7fffffffLL) return fail(RT_ERR_INVALID, "image too large");
    return RT_OK;
}

RT_EXPORT int rt_render_whitted(rt_scene *scene, int precision, const rt_whitted_params *p, void *accum_dev,
                                int32_t *hit_dev, uint64_t *stats_dev, void *stream) {
    if (!scene || !p || !accum_dev) return fail(RT_ERR_INVALID, "NULL argument");
    if (!p->X || !p->Y) return fail(RT_ERR_INVALID, "direction grids missing");
    int rc = check_band(p->W, p->H, p->y0, p->y1, p->s0, p->s1);
    if (rc) return rc;
    CU(cudaSetDevice(scene->device));
    if (precision == RT_F64) return render_whitted_t<double>(scene, scene->d.view, p, accum_dev, hit_dev, stats_dev, S(stream));
    if (precision == RT_F32) return render_whitted_t<float>(scene, scene->f.view, p, accum_dev, hit_dev, stats_dev, S(stream));
    return fail(RT_ERR_INVALID, "unknown precision");
}

// ------------------------------------------------------------------ Algorithm B frame
struct ExplicitRays { const double *rays; const int32_t *ids; int depth0; };

// chandelier.py:412-415: aspect = W/H; half_height = tan(radians(fov)/2); half_width = half_height*aspect
template <typename T> static void path_camera(PathDev<T> &pp, const rt_path_params *p) {
    for (int k = 0; k < 3; ++k) pp.cam[k] = (T)p->cam[k];
    pp.W = p->W; pp.H = p->H;
    const double aspect = (double)p->W / (double)p->H;
    const double half_h = std::tan((p->fov_deg * (M_PI / 180.0)) / 2), half_w = half_h * aspect;
    pp.aspect = (T)aspect; pp.half_w = (T)half_w; pp.half_h = (T)half_h;
    pp.inv_W = (T)(1.0 / (double)p->W); pp.inv_H = (T)(1.0 / (double)p->H);
}

// Cuts one path-kernel launch into work units: sets the band (y0, tile_step, col_*, seg_w), the sample split, both tile
// grids and fold_tab of pp (which holds W, y1 and int_fold of the request) and returns the kernel variant and its dynamic
// shared memory.  Every rank of a frame plans from the same numbers, so the launches of a frame tile it exactly.
template <typename T>
static PathLaunch plan_path_launch(PathDev<T> &pp, const SceneDev<T> &sc, const rt_path_params *p, const rt_path_sink *sink,
                                   bool xr, bool byte_colours, bool allow_pkc, int sms) {
    const int ns = p->s1 - p->s0;
    const bool image = sink && sink->mode == RT_SINK_IMAGE;
    long long pixels = 0;
    // interleave: the 2-D interleave (rt_path_sink::col_split), one column segment of every stripe; false when a segment
    // does not hold whole work units of both tile grids (32 / 16 / 8 / 4 pixels wide for 1-2 / 4 / 8-16 / 32 lanes per pixel)
    auto plan = [&](bool interleave) {
        pp.col_step = 1; pp.col_first = 0; pp.seg_w = p->W; pp.tile_step = 1; pp.y0 = p->y0;
        if (interleave) {
            pp.col_step = sink->tile_step; pp.col_first = sink->tile_first; pp.seg_w = p->W / sink->tile_step; pp.y0 = 0;
        } else if (image) {                                     // every tile_step-th 8-row stripe from tile_first
            pp.tile_step = sink->tile_step; pp.y0 = sink->tile_first * 8;
        }
        const int rows = pp.y1 - pp.y0, step = pp.tile_step;
        const int owned = ((rows + 7) / 8 + step - 1) / step;             // 8-row stripes of this launch
        pixels = (long long)pp.seg_w * ((rows + step - 1) / step);
        // sample split (automatic): k lanes per pixel so that a lane keeps about 8 samples -- measured best at 8, 16, 32
        // and 64 samples per launch (k = 1, 2, 4, 8: tighter camera-ray cones against per-unit overhead) -- and, for small
        // frames, more lanes per pixel until there are ~4 warp tiles per resident warp (every lane keeps >= 2 samples)
        int lk = 0;
        pp.ksplit2_log2 = 0;
        if (pp.int_fold && p->ksplit != 0 && !xr) {
            if (p->ksplit > 0) { while ((1 << (lk + 1)) <= p->ksplit && lk < 5) ++lk; }
            else {
                const long long want = 4LL * 32 * sms;             // warp tiles: 4 per resident warp (32 warps per SM)
                // with a hierarchy the lanes of a pixel traverse together: coherence wins, 8 lanes per pixel whenever a
                // lane keeps >= 2 samples (1e3-1e5-sphere scenes: 11.3 / 48.5 / 222 ms per 16 spp against 12.5 / 51.9 / 227)
                const int per_lane = sc.bvh.nodes > 0 ? 2 : 8;
                while (lk < 3 && (ns >> (lk + 1)) >= per_lane) ++lk;
                while (lk < 5 && (pixels << lk) / 32 < want && (ns >> (lk + 1)) >= 2) ++lk;
                // the LAST work units of the launch are finer (more lanes per pixel, every lane still keeps >= 2 samples),
                // so that the drain of the launch is a fine unit long instead of a coarse one (brute-force scenes; with a
                // hierarchy the units are short already)
                int lk2 = lk + 2 < 5 ? lk + 2 : 5;
                while (lk2 > lk && (ns >> lk2) < 2) --lk2;
                if (sc.bvh.nodes == 0 && lk2 > lk) pp.ksplit2_log2 = lk2;
            }
        }
        pp.ksplit_log2 = lk;
        const int lk2 = pp.ksplit2_log2 > lk ? pp.ksplit2_log2 : lk, pw = unit_pw_log2(lk), pw2 = unit_pw_log2(lk2);
        const int ctw = 4 << pw, cth = 2 << ((5 - lk) - pw), ctw2 = 4 << pw2, cth2 = 2 << ((5 - lk2) - pw2);
        // coarse tile grid: stripes of 8 rows (8 / cth CTA rows each); without interleaving the last stripe may be cut short
        pp.gx = (pp.seg_w + ctw - 1) / ctw;
        pp.gy = step > 1 ? owned * (8 / cth) : (rows + cth - 1) / cth;
        pp.gx2 = pp.gy2 = pp.stripe2 = 0;
        if (lk2 > lk) {
            // fine grid over the last owned stripes (see path_kernel): 1.5 coarse units' worth of pixels per resident
            // warp, whole 8-row stripes, at most half of them
            int fs = (int)((3LL * 32 * sms * (32 >> lk) / 2 + 8LL * pp.seg_w - 1) / (8LL * pp.seg_w));
            if (fs > owned / 2) fs = owned / 2;
            if (fs >= 1) {
                const int sb = owned - fs, rows_a = sb * 8;             // (tile_step == 1: rows of the coarse part)
                pp.stripe2 = sb;
                pp.gy = step > 1 ? sb * (8 / cth) : (rows_a + cth - 1) / cth;
                pp.gx2 = (pp.seg_w + ctw2 - 1) / ctw2;
                pp.gy2 = step > 1 ? fs * (8 / cth2) : (rows - rows_a + cth2 - 1) / cth2;
            }
        }
        return !interleave || (pp.seg_w % ctw == 0 && pp.seg_w % ctw2 == 0);
    };
    if (!plan(image && sink->col_split && sink->tile_step > 1)) plan(false);
    const size_t extra = 256 * sizeof(double);                  // div255 table of the integer fold
    PathLaunch pl;
    pl.mode = mode_for(sc, extra);
    if (pl.mode == 0 && allow_pkc) pl.mode = 3;   // small brute-force FP32 scenes: sphere pairs through the parameter block
    // table fold (kMode 3 only): worth its per-CTA build (n * 768 entries) from ~4 M pixel-samples up
    pp.fold_tab = pl.mode == 3 && pp.int_fold && byte_colours && pixels * ns >= (4LL << 20);
    // kMode 3 uses static shared arrays; its dynamic part is the fold table [n][3][256] bytes
    pl.smem = pl.mode == 3 ? (pp.fold_tab ? (size_t)sc.n * 768 : 0) : (pl.mode != 2 ? smem_for(sc) : 0) + extra;
    return pl;
}

template <typename T>
static int render_path_t(const rt_scene *sc, const SceneDev<T> &view, const rt_path_params *p, void *accum, uint64_t *stats,
                         cudaStream_t st, const rt_path_sink *sink = nullptr, const ExplicitRays *xr = nullptr) {
    // bit 1: no camera-ray candidate lists, bit 2: no parameter-block kernel (include/rt_b200.h)
    if (p->schedule & ~6) return fail(RT_ERR_INVALID, "unknown schedule bits");
    PathDev<T> pp;
    std::memset(&pp, 0, sizeof pp);
    if (xr) { pp.rays = xr->rays; pp.ray_ids = xr->ids; pp.depth0 = xr->depth0; }
    path_camera(pp, p);
    pp.y0 = p->y0; pp.y1 = p->y1; pp.s0 = p->s0; pp.s1 = p->s1; pp.max_bounces = p->max_bounces;
    pp.mirror_threshold = (T)p->mirror_threshold;
    pp.k0 = (uint32_t)p->seed; pp.k1 = (uint32_t)(p->seed >> 32);
    for (uint32_t r = 0; r < 10; ++r) { pp.rk[2 * r] = pp.k0 + r * 0x9E3779B9u; pp.rk[2 * r + 1] = pp.k1 + r * 0xBB67AE85u; }
    pp.accumulate = p->accumulate;
    pp.int_fold = sc->int_colours && (p->s1 - p->s0) <= 65536;
    pp.primary_cull = (p->schedule & 2) == 0;
    pp.sink = RT_SINK_ACCUM; pp.world = 1; pp.spp_total = p->s1 - p->s0;
    if (sink && sink->mode != RT_SINK_ACCUM) {
        if (!pp.int_fold) return fail(RT_ERR_UNSUPPORTED, "fused sinks need integer colours and <= 65536 samples per launch");
        pp.sink = sink->mode;
        pp.timed_out = sink->timed_out;          // read under the frame protocol only (and by the RT_TRACE_WARPS development build)
        if (sink->mode == RT_SINK_IMAGE) {
            if (!sink->image || sink->tile_step < 1 || sink->tile_first < 0) return fail(RT_ERR_INVALID, "bad image sink");
            pp.image = sink->image;
            if (sink->col_split && sink->tile_step > 1) {
                if (p->W % sink->tile_step != 0) return fail(RT_ERR_INVALID, "col_split: W must be a multiple of tile_step");
                if (sink->tile_first >= sink->tile_step) return fail(RT_ERR_INVALID, "col_split: tile_first must be < tile_step");
            }
            if (p->s0 != 0) return fail(RT_ERR_INVALID, "an image sink resolves in the kernel: the launch must cover all samples");
        } else if (sink->mode == RT_SINK_SCATTER_ADD) {
            if (sink->world < 1 || sink->world > RT_MAX_PEERS) return fail(RT_ERR_INVALID, "bad world size");
            if ((double)(p->s1 - p->s0) * 65535.0 >= 16777216.0 * 255.0)      // sums stay exact in FP32 for 8-bit colours
                return fail(RT_ERR_UNSUPPORTED, "sample range too long for exact FP32 sums");
            pp.world = sink->world;
            for (int k = 0; k < sink->world; ++k) {
                if (!sink->accum[k]) return fail(RT_ERR_INVALID, "missing peer accumulator");
                pp.peer_accum[k] = reinterpret_cast<float4 *>(sink->accum[k]);
            }
            for (int k = 0; k <= sink->world; ++k) pp.band_y[k] = sink->band_y[k];
            if (pp.band_y[0] != 0 || pp.band_y[sink->world] != p->H) return fail(RT_ERR_INVALID, "owner bands must cover the image");
        } else return fail(RT_ERR_INVALID, "unknown sink mode");
        pp.max_ctas = sink->max_ctas > 0 ? sink->max_ctas : 0;
        if (sink->sync) {
            // the whole frame protocol inside the launch (include/rt_b200.h): flags of every rank, epoch, collecting image
            if (sink->world < 1 || sink->world > RT_MAX_PEERS || sink->rank < 0 || sink->rank >= sink->world)
                return fail(RT_ERR_INVALID, "bad world / rank for a synchronised sink");
            if (sink->epoch == 0u) return fail(RT_ERR_INVALID, "epochs start at 1");
            if (!sink->image) return fail(RT_ERR_INVALID, "a synchronised sink needs the collecting rank's image");
            for (int k = 0; k < sink->world; ++k) {
                if (!sink->flags[k]) return fail(RT_ERR_INVALID, "missing flag block");
                pp.flags[k] = sink->flags[k];
            }
            pp.sync = 1; pp.rank = sink->rank; pp.world = sink->world; pp.epoch = sink->epoch; pp.go_epoch = sink->go_epoch;
            pp.image = sink->image;
            if (sink->mode == RT_SINK_SCATTER_ADD) {
                if (sink->spp_total < p->s1) return fail(RT_ERR_INVALID, "spp_total must cover the sample range");
                pp.spp_total = sink->spp_total;
            }
            pp.timed_out = sink->timed_out;
            int khz = 0;
            if (device_attr(sc->device, cudaDevAttrClockRate, &khz) != cudaSuccess || khz <= 0) khz = 2000000;
            pp.timeout_cycles = (long long)(sink->timeout_ms > 0 ? sink->timeout_ms : 20000) * (long long)khz;
        }
    }
    int sms = 0;
    if (device_attr(sc->device, cudaDevAttrMultiProcessorCount, &sms) != cudaSuccess || sms <= 0) sms = 148;
    const PathLaunch pl = plan_path_launch<T>(pp, view, p, sink, xr != nullptr, sc->byte_colours,
                                              sizeof(T) == 4 && sc->pkc_ok && !(p->schedule & 4) && !xr, sms);
    if (!sc->sched_dev) return fail(RT_ERR_INVALID, "scene has no scheduler counters (upload failed?)");
    pp.sched = sc->sched_dev + 4 * (sc->sched_next.fetch_add(1u) % RT_SCHED_SLOTS);      // {next unit, warps done, CTAs resolved, -}
    CU(launch_path<T>(view, pp, pl, accum, reinterpret_cast<unsigned long long *>(stats), st, &sc->pkc));
    return RT_OK;
}

RT_EXPORT int rt_render_path(rt_scene *scene, int precision, const rt_path_params *p, void *accum_dev, uint64_t *stats_dev,
                             void *stream) {
    if (!scene || !p || !accum_dev) return fail(RT_ERR_INVALID, "NULL argument");
    int rc = check_band(p->W, p->H, p->y0, p->y1, p->s0, p->s1);
    if (rc) return rc;
    if (p->max_bounces > RT_PATH_MAX_DEPTH) return fail(RT_ERR_UNSUPPORTED, "max_bounces above 32 is not supported by the path kernel");
    CU(cudaSetDevice(scene->device));
    if (precision == RT_F64) return render_path_t<double>(scene, scene->d.view, p, accum_dev, stats_dev, S(stream));
    if (precision == RT_F32) return render_path_t<float>(scene, scene->f.view, p, accum_dev, stats_dev, S(stream));
    return fail(RT_ERR_INVALID, "unknown precision");
}

RT_EXPORT int rt_trace_paths(rt_scene *scene, int precision, const rt_path_params *p, int32_t n, const double *rays_dev,
                             const int32_t *ray_ids_dev, int32_t bounce_count, void *accum_dev, uint64_t *stats_dev, void *stream) {
    if (!scene || !p || !accum_dev || (n > 0 && !rays_dev)) return fail(RT_ERR_INVALID, "NULL argument");
    if (n < 0 || bounce_count < 0) return fail(RT_ERR_INVALID, "negative count");
    if (n == 0) return RT_OK;
    if (p->s0 < 0 || p->s0 > p->s1) return fail(RT_ERR_INVALID, "bad sample range");
    if (p->max_bounces > RT_PATH_MAX_DEPTH) return fail(RT_ERR_UNSUPPORTED, "max_bounces above 32 is not supported by the path kernel");
    CU(cudaSetDevice(scene->device));
    rt_path_params q = *p;
    q.W = n; q.H = 1; q.y0 = 0; q.y1 = 1; q.accumulate = 0;
    const ExplicitRays xr = {rays_dev, ray_ids_dev, bounce_count};
    if (precision == RT_F64) return render_path_t<double>(scene, scene->d.view, &q, accum_dev, stats_dev, S(stream), nullptr, &xr);
    if (precision == RT_F32) return render_path_t<float>(scene, scene->f.view, &q, accum_dev, stats_dev, S(stream), nullptr, &xr);
    return fail(RT_ERR_INVALID, "unknown precision");
}

RT_EXPORT int rt_render_path_sink(rt_scene *scene, const rt_path_params *p, const rt_path_sink *sink, uint64_t *stats_dev,
                                  void *stream) {
    if (!scene || !p || !sink) return fail(RT_ERR_INVALID, "NULL argument");
    int rc = check_band(p->W, p->H, 0, p->H, p->s0, p->s1);
    if (rc) return rc;
    if (p->max_bounces > RT_PATH_MAX_DEPTH) return fail(RT_ERR_UNSUPPORTED, "max_bounces above 32 is not supported by the path kernel");
    if (sink->mode == RT_SINK_ACCUM) return fail(RT_ERR_INVALID, "use rt_render_path for the accumulator sink");
    CU(cudaSetDevice(scene->device));
    rt_path_params q = *p;
    q.y0 = 0; q.y1 = p->H;
    return render_path_t<float>(scene, scene->f.view, &q, nullptr, stats_dev, S(stream), sink);
}

RT_EXPORT int rt_resolve_clear(int device, void *accum_dev, int32_t W, int32_t H, int32_t y0, int32_t y1, int32_t spp,
                               float *image_dev, int32_t clear, void *stream) {
    if (!accum_dev || !image_dev) return fail(RT_ERR_INVALID, "NULL argument");
    if (W <= 0 || H <= 0 || y0 < 0 || y1 > H || y0 > y1 || spp <= 0) return fail(RT_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(device));
    CU(launch_resolve_clear(reinterpret_cast<float4 *>(accum_dev), W, y0, y1, spp, image_dev, clear, S(stream)));
    return RT_OK;
}

// ------------------------------------------------------------------ peer memory (CUDA IPC) and epoch flags
static_assert(sizeof(cudaIpcMemHandle_t) == RT_IPC_HANDLE_BYTES, "IPC handle size");
RT_EXPORT int rt_peer_alloc(int device, size_t bytes, void **out_dev, unsigned char handle[RT_IPC_HANDLE_BYTES]) {
    if (!out_dev || !handle || bytes == 0) return fail(RT_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(device));
    void *p = nullptr;
    CU(cudaMalloc(&p, bytes));
    cudaError_t e = cudaMemset(p, 0, bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return cuda_fail(e, "rt_peer_alloc"); }
    std::memcpy(handle, &h, sizeof h);
    *out_dev = p;
    return RT_OK;
}
RT_EXPORT int rt_peer_open(int device, const unsigned char handle[RT_IPC_HANDLE_BYTES], void **out_dev) {
    if (!out_dev || !handle) return fail(RT_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof h);
    CU(cudaIpcOpenMemHandle(out_dev, h, cudaIpcMemLazyEnablePeerAccess));
    return RT_OK;
}
RT_EXPORT int rt_peer_close(int device, void *ptr_dev) {
    if (!ptr_dev) return RT_OK;
    CU(cudaSetDevice(device));
    CU(cudaIpcCloseMemHandle(ptr_dev));
    return RT_OK;
}
RT_EXPORT int rt_peer_free(int device, void *ptr_dev) {
    if (!ptr_dev) return RT_OK;
    CU(cudaSetDevice(device));
    CU(cudaFree(ptr_dev));
    return RT_OK;
}
RT_EXPORT int rt_peer_signal(int device, uint32_t *const *flag_ptrs, int32_t n, uint32_t epoch, void *stream) {
    if (!flag_ptrs || n < 1 || n > 32) return fail(RT_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(device));
    PeerFlagTable tab;
    std::memset(&tab, 0, sizeof tab);
    for (int i = 0; i < n; ++i) {
        if (!flag_ptrs[i]) return fail(RT_ERR_INVALID, "NULL flag pointer");
        tab.p[i] = flag_ptrs[i];
    }
    cudaError_t e = launch_peer_signal(tab, n, epoch, S(stream));
    if (e != cudaSuccess) return cuda_fail(e, "rt_peer_signal");
    return RT_OK;
}
RT_EXPORT int rt_peer_wait(int device, const uint32_t *flags_dev, int32_t n, uint32_t epoch, int32_t timeout_ms,
                           int32_t *timed_out_dev, void *stream) {
    if (!flags_dev || n < 1 || n > 32) return fail(RT_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(device));
    int khz = 0;
    CU(device_attr(device, cudaDevAttrClockRate, &khz));
    const long long cycles = (long long)(timeout_ms > 0 ? timeout_ms : 2000) * (long long)(khz > 0 ? khz : 2000000);
    CU(launch_peer_wait(flags_dev, n, epoch, cycles, timed_out_dev, S(stream)));
    return RT_OK;
}

RT_EXPORT int rt_resolve(int device, int precision, const void *accum_dev, int32_t W, int32_t H, int32_t y0, int32_t y1,
                         int32_t spp, float *image_dev, void *stream) {
    if (!accum_dev || !image_dev) return fail(RT_ERR_INVALID, "NULL argument");
    if (spp <= 0) return fail(RT_ERR_INVALID, "spp must be positive");
    int rc = check_band(W, H, y0, y1, 0, spp);
    if (rc) return rc;
    CU(cudaSetDevice(device));
    if (precision == RT_F64) CU(launch_resolve<double>(accum_dev, W, y0, y1, spp, image_dev, S(stream)));
    else if (precision == RT_F32) CU(launch_resolve<float>(accum_dev, W, y0, y1, spp, image_dev, S(stream)));
    else return fail(RT_ERR_INVALID, "unknown precision");
    return RT_OK;
}

// ------------------------------------------------------------------ host-buffer convenience entries
struct DevTmp {
    void *p = nullptr;
    ~DevTmp() { if (p) cudaFree(p); }
};

static int render_host_common(rt_scene *scene, int precision, bool whitted, const void *params, float *image_host,
                              void *accum_host, int32_t *hit_host, uint64_t *stats_host) {
    if (!scene || !params) return fail(RT_ERR_INVALID, "NULL argument");
    if (precision != RT_F32 && precision != RT_F64) return fail(RT_ERR_INVALID, "unknown precision");
    const rt_whitted_params *wp = whitted ? (const rt_whitted_params *)params : nullptr;
    const rt_path_params *pp = whitted ? nullptr : (const rt_path_params *)params;
    const int W = whitted ? wp->W : pp->W, H = whitted ? wp->H : pp->H;
    const int y0 = whitted ? wp->y0 : pp->y0, y1 = whitted ? wp->y1 : pp->y1;
    const int s0 = whitted ? wp->s0 : pp->s0, s1 = whitted ? wp->s1 : pp->s1;
    int rc = check_band(W, H, y0, y1, s0, s1);
    if (rc) return rc;
    CU(cudaSetDevice(scene->device));
    const size_t px = (size_t)W * H, el = precision == RT_F64 ? sizeof(double) : sizeof(float);
    DevTmp accum, image, hit, stats;
    CU(cudaMalloc(&accum.p, px * 4 * el));
    CU(cudaMemsetAsync(accum.p, 0, px * 4 * el, nullptr));
    CU(cudaMalloc(&stats.p, 8 * sizeof(uint64_t)));
    CU(cudaMemsetAsync(stats.p, 0, 8 * sizeof(uint64_t), nullptr));
    if (whitted && hit_host) {
        CU(cudaMalloc(&hit.p, px * sizeof(int32_t)));
        CU(cudaMemsetAsync(hit.p, 0xff, px * sizeof(int32_t), nullptr));
    }
    if (whitted) rc = rt_render_whitted(scene, precision, wp, accum.p, (int32_t *)hit.p, (uint64_t *)stats.p, nullptr);
    else rc = rt_render_path(scene, precision, pp, accum.p, (uint64_t *)stats.p, nullptr);
    if (rc) return rc;
    if (image_host) {
        CU(cudaMalloc(&image.p, px * 3 * sizeof(float)));
        CU(cudaMemsetAsync(image.p, 0, px * 3 * sizeof(float), nullptr));
        const int spp = s1 - s0 > 0 ? s1 - s0 : 1;
        rc = rt_resolve(scene->device, precision, accum.p, W, H, y0, y1, spp, (float *)image.p, nullptr);
        if (rc) return rc;
        CU(cudaMemcpyAsync(image_host, image.p, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, nullptr));
    }
    if (accum_host) CU(cudaMemcpyAsync(accum_host, accum.p, px * 4 * el, cudaMemcpyDeviceToHost, nullptr));
    if (hit_host && hit.p) CU(cudaMemcpyAsync(hit_host, hit.p, px * sizeof(int32_t), cudaMemcpyDeviceToHost, nullptr));
    if (stats_host) CU(cudaMemcpyAsync(stats_host, stats.p, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, nullptr));
    CU(cudaStreamSynchronize(nullptr));
    return RT_OK;
}

RT_EXPORT int rt_render_whitted_host(rt_scene *scene, int precision, const rt_whitted_params *p, float *image_host,
                                     void *accum_host, int32_t *hit_host, uint64_t *stats_host) {
    return render_host_common(scene, precision, true, p, image_host, accum_host, hit_host, stats_host);
}

RT_EXPORT int rt_render_path_host(rt_scene *scene, int precision, const rt_path_params *p, float *image_host,
                                  void *accum_host, uint64_t *stats_host) {
    return render_host_common(scene, precision, false, p, image_host, accum_host, nullptr, stats_host);
}

// ------------------------------------------------------------------ wavefront Algorithm B (learned direction sampling)
struct rt_wavefront {
    rt_scene *scene = nullptr;
    int precision = RT_F32, max_paths = 0, max_depth = 0;
    void *blob = nullptr;
    WaveDev<float> f;
    WaveDev<double> d;
    PathDev<float> pf;
    PathDev<double> pd;
    bool begun = false;
};

template <typename T> static size_t wave_bytes(size_t P, size_t depth) {
    return 12 * P * sizeof(T) + 2 * P * sizeof(int) + P + 2 * depth * P * sizeof(uint32_t) + 3 * P * sizeof(double) + 256;
}
template <typename T> static void bind_wave(WaveDev<T> &w, void *blob, size_t P, size_t depth) {
    unsigned char *p = reinterpret_cast<unsigned char *>(blob);
    w.leaf = reinterpret_cast<double *>(p); p += 3 * P * sizeof(double);
    w.O = reinterpret_cast<T *>(p); p += 3 * P * sizeof(T);
    w.D = reinterpret_cast<T *>(p); p += 3 * P * sizeof(T);
    w.hp = reinterpret_cast<T *>(p); p += 3 * P * sizeof(T);
    w.hn = reinterpret_cast<T *>(p); p += 3 * P * sizeof(T);
    w.state = reinterpret_cast<int *>(p); p += P * sizeof(int);
    w.depth = reinterpret_cast<int *>(p); p += P * sizeof(int);
    w.st_idx = reinterpret_cast<uint32_t *>(p); p += depth * P * sizeof(uint32_t);
    w.st_direct = reinterpret_cast<uint32_t *>(p); p += depth * P * sizeof(uint32_t);
    w.mirror = p;
}

RT_EXPORT int rt_wf_create(rt_scene *scene, int precision, int32_t max_paths, int32_t max_depth, rt_wavefront **out) {
    if (!scene || !out) return fail(RT_ERR_INVALID, "NULL argument");
    *out = nullptr;
    if (precision != RT_F32 && precision != RT_F64) return fail(RT_ERR_INVALID, "unknown precision");
    if (max_paths <= 0 || max_depth <= 0 || max_depth > RT_PATH_MAX_DEPTH) return fail(RT_ERR_INVALID, "bad wavefront size");
    CU(cudaSetDevice(scene->device));
    rt_wavefront *wf = new (std::nothrow) rt_wavefront();
    if (!wf) return fail(RT_ERR_NOMEM, "host allocation failed");
    wf->scene = scene; wf->precision = precision; wf->max_paths = max_paths; wf->max_depth = max_depth;
    const size_t P = (size_t)max_paths, D = (size_t)max_depth;
    const size_t bytes = precision == RT_F64 ? wave_bytes<double>(P, D) : wave_bytes<float>(P, D);
    cudaError_t e = cudaMalloc(&wf->blob, bytes);
    if (e != cudaSuccess) { delete wf; cudaGetLastError(); return e == cudaErrorMemoryAllocation ? fail(RT_ERR_NOMEM, "out of device memory") : cuda_fail(e, "cudaMalloc"); }
    *out = wf;
    return RT_OK;
}

RT_EXPORT int rt_wf_destroy(rt_wavefront *wf) {
    if (!wf) return RT_OK;
    if (wf->blob) cudaFree(wf->blob);
    delete wf;
    return RT_OK;
}

template <typename T>
static int wf_begin_t(rt_wavefront *wf, WaveDev<T> &w, PathDev<T> &pp, const rt_path_params *p, double fb_prob, uint64_t *stats,
                      cudaStream_t st) {
    const long long P = (long long)p->W * (p->y1 - p->y0) * (p->s1 - p->s0);
    if (P > wf->max_paths) return fail(RT_ERR_INVALID, "more paths than the wavefront was created for");
    std::memset(&w, 0, sizeof w);
    std::memset(&pp, 0, sizeof pp);
    bind_wave<T>(w, wf->blob, (size_t)P, (size_t)wf->max_depth);
    w.P = (int)P; w.max_depth = wf->max_depth;
    w.W = p->W; w.H = p->H; w.y0 = p->y0; w.y1 = p->y1; w.s0 = p->s0; w.s1 = p->s1; w.max_bounces = p->max_bounces;
    path_camera(pp, p);
    for (int k = 0; k < 3; ++k) w.cam[k] = pp.cam[k];
    w.aspect = pp.aspect; w.half_w = pp.half_w; w.half_h = pp.half_h;
    w.mirror_threshold = (T)p->mirror_threshold; w.fb_prob = (T)fb_prob;
    w.k0 = (uint32_t)p->seed; w.k1 = (uint32_t)(p->seed >> 32);
    CU(launch_wf_begin<T>(w, pp, reinterpret_cast<unsigned long long *>(stats), st));
    wf->begun = true;
    return RT_OK;
}

RT_EXPORT int rt_wf_begin(rt_wavefront *wf, const rt_path_params *p, double fb_usage_prob, uint64_t *stats_dev, void *stream) {
    if (!wf || !p) return fail(RT_ERR_INVALID, "NULL argument");
    int rc = check_band(p->W, p->H, p->y0, p->y1, p->s0, p->s1);
    if (rc) return rc;
    if (p->max_bounces > wf->max_depth) return fail(RT_ERR_INVALID, "max_bounces above the wavefront's stack depth");
    if (!(fb_usage_prob >= 0.0 && fb_usage_prob <= 1.0)) return fail(RT_ERR_INVALID, "fb_usage_prob outside [0, 1]");
    CU(cudaSetDevice(wf->scene->device));
    if (wf->precision == RT_F64) return wf_begin_t<double>(wf, wf->d, wf->pd, p, fb_usage_prob, stats_dev, S(stream));
    return wf_begin_t<float>(wf, wf->f, wf->pf, p, fb_usage_prob, stats_dev, S(stream));
}

RT_EXPORT int rt_wf_trace(rt_wavefront *wf, float *obs_dev, uint8_t *need_dev, uint64_t *stats_dev, void *stream) {
    if (!wf || !obs_dev || !need_dev) return fail(RT_ERR_INVALID, "NULL argument");
    if (!wf->begun) return fail(RT_ERR_INVALID, "rt_wf_begin has not been called");
    CU(cudaSetDevice(wf->scene->device));
    unsigned long long *st = reinterpret_cast<unsigned long long *>(stats_dev);
    if (wf->precision == RT_F64) CU(launch_wf_trace<double>(wf->scene->d.view, wf->d, obs_dev, need_dev, st, S(stream)));
    else CU(launch_wf_trace<float>(wf->scene->f.view, wf->f, obs_dev, need_dev, st, S(stream)));
    return RT_OK;
}

RT_EXPORT int rt_wf_bounce(rt_wavefront *wf, const uint8_t *need_dev, const float *actions_dev, uint64_t *stats_dev,
                           int32_t *live_dev, void *stream) {
    if (!wf || !need_dev || !actions_dev || !live_dev) return fail(RT_ERR_INVALID, "NULL argument");
    if (!wf->begun) return fail(RT_ERR_INVALID, "rt_wf_begin has not been called");
    CU(cudaSetDevice(wf->scene->device));
    unsigned long long *st = reinterpret_cast<unsigned long long *>(stats_dev);
    if (wf->precision == RT_F64) CU(launch_wf_bounce<double>(wf->d, need_dev, actions_dev, st, live_dev, S(stream)));
    else CU(launch_wf_bounce<float>(wf->f, need_dev, actions_dev, st, live_dev, S(stream)));
    return RT_OK;
}

RT_EXPORT int rt_wf_finish(rt_wavefront *wf, void *accum_dev, void *stream) {
    if (!wf || !accum_dev) return fail(RT_ERR_INVALID, "NULL argument");
    if (!wf->begun) return fail(RT_ERR_INVALID, "rt_wf_begin has not been called");
    CU(cudaSetDevice(wf->scene->device));
    if (wf->precision == RT_F64) CU(launch_wf_finish<double>(wf->scene->d.view, wf->d, accum_dev, S(stream)));
    else CU(launch_wf_finish<float>(wf->scene->f.view, wf->f, accum_dev, S(stream)));
    wf->begun = false;
    return RT_OK;
}

// ------------------------------------------------------------------ FB training trajectories
RT_EXPORT int rt_generate_trajectories(rt_scene *scene, int precision, int32_t n_traj, int32_t max_steps, int32_t max_bounces,
                                       uint64_t seed, float *obs_dev, float *action_dev, float *next_obs_dev,
                                       float *reward_dev, uint8_t *hit_dev, int32_t *length_dev, uint8_t *hit_light_dev,
                                       uint64_t *stats_dev, void *stream) {
    if (!scene) return fail(RT_ERR_INVALID, "scene is NULL");
    if (n_traj < 0 || max_steps <= 0 || max_bounces <= 0) return fail(RT_ERR_INVALID, "bad trajectory counts");
    if (n_traj > 0 && (!obs_dev || !action_dev || !next_obs_dev || !reward_dev || !hit_dev || !length_dev || !hit_light_dev))
        return fail(RT_ERR_INVALID, "NULL output");
    if (((uintptr_t)obs_dev | (uintptr_t)next_obs_dev) & 7u)
        return fail(RT_ERR_INVALID, "obs / next_obs must be 8-byte aligned (88-byte records are written as 8-byte stores)");
    CU(cudaSetDevice(scene->device));
    unsigned long long *st = reinterpret_cast<unsigned long long *>(stats_dev);
    if (precision == RT_F64)
        CU(launch_trajectories<double>(scene->d.view, n_traj, max_steps, max_bounces, seed, obs_dev, action_dev, next_obs_dev,
                                       reward_dev, hit_dev, length_dev, hit_light_dev, st, S(stream)));
    else if (precision == RT_F32)
        CU(launch_trajectories<float>(scene->f.view, n_traj, max_steps, max_bounces, seed, obs_dev, action_dev, next_obs_dev,
                                      reward_dev, hit_dev, length_dev, hit_light_dev, st, S(stream)));
    else return fail(RT_ERR_INVALID, "unknown precision");
    return RT_OK;
}

// ------------------------------------------------------------------ "Algorithm C" frame (FB/output6.py)
template <typename T>
static int render_simple_t(const SceneDev<T> &view, const rt_simple_params *p, int32_t *rgb, float *image, uint64_t *stats,
                           cudaStream_t st) {
    SimpleDev<T> sp;
    std::memset(&sp, 0, sizeof sp);
    for (int k = 0; k < 3; ++k) { sp.cam[k] = (T)p->cam[k]; sp.sun_pos[k] = (T)p->sun_pos[k]; sp.sun_col[k] = (T)p->sun_col[k]; }
    sp.tan_half = (T)std::tan(p->fov_rad / 2);                 // np.tan(fov/2), output6.py:623
    sp.aspect = (T)((double)p->W / (double)(p->H > 0 ? p->H : 1));
    sp.W = p->W; sp.H = p->H; sp.sun_id = p->sun_id; sp.max_bounces = p->max_bounces;
    sp.k0 = (uint32_t)p->seed; sp.k1 = (uint32_t)(p->seed >> 32);
    sp.rays = p->rays_dev;
    sp.lighting_only = p->lighting_only != 0;
    sp.n = p->rays_dev ? p->m : p->W * p->H;
    CU(launch_simple<T>(view, sp, reinterpret_cast<int4 *>(rgb), image, reinterpret_cast<unsigned long long *>(stats), st));
    return RT_OK;
}

RT_EXPORT int rt_render_simple(rt_scene *scene, int precision, const rt_simple_params *p, int32_t *rgb_dev, float *image_dev,
                               uint64_t *stats_dev, void *stream) {
    if (!scene || !p || !rgb_dev) return fail(RT_ERR_INVALID, "NULL argument");
    if (p->rays_dev ? p->m < 0 : (p->W <= 0 || p->H <= 0 || (long long)p->W * p->H > 0x7fffffffLL))
        return fail(RT_ERR_INVALID, "bad frame size / ray count");
    if (p->lighting_only && (!p->rays_dev || image_dev)) return fail(RT_ERR_INVALID, "lighting_only needs intersections and no image");
    CU(cudaSetDevice(scene->device));
    if (precision == RT_F64) return render_simple_t<double>(scene->d.view, p, rgb_dev, image_dev, stats_dev, S(stream));
    if (precision == RT_F32) return render_simple_t<float>(scene->f.view, p, rgb_dev, image_dev, stats_dev, S(stream));
    return fail(RT_ERR_INVALID, "unknown precision");
}

RT_EXPORT int rt_render_simple_host(rt_scene *scene, int precision, const rt_simple_params *p, const double *rays_host,
                                    int32_t *rgb_host, float *image_host, uint64_t *stats_host) {
    if (!scene || !p) return fail(RT_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(scene->device));
    rt_simple_params q = *p;
    DevTmp rays, rgb, image, stats;
    if (rays_host) {
        if (q.m < 0) return fail(RT_ERR_INVALID, "negative ray count");
        const size_t row = q.lighting_only ? 7 : 6;
        CU(cudaMalloc(&rays.p, sizeof(double) * row * (size_t)(q.m > 0 ? q.m : 1)));
        CU(cudaMemcpyAsync(rays.p, rays_host, sizeof(double) * row * (size_t)q.m, cudaMemcpyHostToDevice, nullptr));
        q.rays_dev = (const double *)rays.p;
    }
    const size_t n = q.rays_dev ? (size_t)q.m : (size_t)q.W * (size_t)q.H;
    if (n == 0) return RT_OK;
    CU(cudaMalloc(&rgb.p, n * 4 * sizeof(int32_t)));
    CU(cudaMemsetAsync(rgb.p, 0, n * 4 * sizeof(int32_t), nullptr));
    CU(cudaMalloc(&stats.p, 8 * sizeof(uint64_t)));
    CU(cudaMemsetAsync(stats.p, 0, 8 * sizeof(uint64_t), nullptr));
    if (image_host) CU(cudaMalloc(&image.p, n * 3 * sizeof(float)));
    int rc = rt_render_simple(scene, precision, &q, (int32_t *)rgb.p, (float *)image.p, (uint64_t *)stats.p, nullptr);
    if (rc) return rc;
    if (rgb_host) CU(cudaMemcpyAsync(rgb_host, rgb.p, n * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, nullptr));
    if (image_host) CU(cudaMemcpyAsync(image_host, image.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, nullptr));
    if (stats_host) CU(cudaMemcpyAsync(stats_host, stats.p, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, nullptr));
    CU(cudaStreamSynchronize(nullptr));
    return RT_OK;
}

// ------------------------------------------------------------------ batched RayTracerEnv
template <typename T> static void bind_env(EnvDev<T> &e, const rt_env_desc &d, void *blob) {
    const size_t B = (size_t)d.B;
    e.B = d.B; e.W = d.W; e.H = d.H; e.max_bounces = d.max_bounces; e.flavour = d.flavour; e.sun_id = d.sun_id;
    for (int k = 0; k < 3; ++k) { e.cam[k] = (T)d.cam[k]; e.cam_angle[k] = (T)d.cam_angle[k]; }
    const double fr = d.fov * M_PI / 180;             // RL/ray_tracer_env.py:127
    e.tan_half = (T)std::tan(fr / 2);
    unsigned char *p = reinterpret_cast<unsigned char *>(blob);
    e.total = reinterpret_cast<double *>(p); p += B * sizeof(double);
    e.p = reinterpret_cast<T *>(p); p += 3 * B * sizeof(T);
    e.n = reinterpret_cast<T *>(p); p += 3 * B * sizeof(T);
    e.d = reinterpret_cast<T *>(p); p += 3 * B * sizeof(T);
    e.acc = reinterpret_cast<T *>(p); p += 3 * B * sizeof(T);
    e.rgb = reinterpret_cast<T *>(p); p += 3 * B * sizeof(T);
    e.has_hit = reinterpret_cast<int *>(p); p += B * sizeof(int);
    e.idx = reinterpret_cast<int *>(p); p += B * sizeof(int);
    e.bounce = reinterpret_cast<int *>(p); p += B * sizeof(int);
    e.through = reinterpret_cast<int *>(p); p += B * sizeof(int);
    e.episode = reinterpret_cast<int *>(p); p += B * sizeof(int);
    e.consec = reinterpret_cast<int *>(p); p += B * sizeof(int);
    e.total_hits = reinterpret_cast<int *>(p); p += B * sizeof(int);
    e.adaptive = d.reward_mode == 1; e.light0 = d.light_ids[0]; e.light1 = d.light_ids[1];
    e.b0 = d.env_offset;
}

RT_EXPORT int rt_env_create(rt_scene *scene, int precision, const rt_env_desc *desc, rt_env **out) {
    if (!scene || !desc || !out) return fail(RT_ERR_INVALID, "NULL argument");
    *out = nullptr;
    if (precision != RT_F32 && precision != RT_F64) return fail(RT_ERR_INVALID, "unknown precision");
    if (desc->B <= 0 || desc->W <= 0 || desc->H <= 0) return fail(RT_ERR_INVALID, "B, W, H must be positive");
    if (desc->flavour != RT_ENV_RL && desc->flavour != RT_ENV_FB) return fail(RT_ERR_INVALID, "unknown env flavour");
    CU(cudaSetDevice(scene->device));
    rt_env *env = new (std::nothrow) rt_env();
    if (!env) return fail(RT_ERR_NOMEM, "host allocation failed");
    env->scene = scene; env->precision = precision; env->desc = *desc;
    const size_t B = (size_t)desc->B, el = precision == RT_F64 ? sizeof(double) : sizeof(float);
    const size_t bytes = B * sizeof(double) + 15 * B * el + 7 * B * sizeof(int);
    cudaError_t e = cudaMalloc(&env->blob, bytes);
    if (e != cudaSuccess) { delete env; cudaGetLastError(); return e == cudaErrorMemoryAllocation ? fail(RT_ERR_NOMEM, "out of device memory") : cuda_fail(e, "cudaMalloc"); }
    e = cudaMemset(env->blob, 0, bytes);
    if (e != cudaSuccess) { cudaFree(env->blob); delete env; return cuda_fail(e, "cudaMemset"); }
    if (precision == RT_F64) bind_env<double>(env->d, *desc, env->blob);
    else bind_env<float>(env->f, *desc, env->blob);
    env->shaded_version = scene->version;
    *out = env;
    return RT_OK;
}

RT_EXPORT int rt_env_destroy(rt_env *env) {
    if (!env) return RT_OK;
    cudaSetDevice(env->scene->device);
    if (env->blob) cudaFree(env->blob);
    delete env;
    return RT_OK;
}

// The RL flavour keeps terminalRGB of every episode's current hit (EnvDev::rgb).  If the scene was re-uploaded since
// those were computed, shade the running episodes' hits again before the next step reads them.
static int env_reshade_if_stale(rt_env *env, cudaStream_t st) {
    if (env->shaded_version == env->scene->version) return RT_OK;
    if (env->precision == RT_F64) CU(launch_env_reshade<double>(env->scene->d.view, env->d, st));
    else CU(launch_env_reshade<float>(env->scene->f.view, env->f, st));
    env->shaded_version = env->scene->version;
    return RT_OK;
}

RT_EXPORT int rt_env_reset(rt_env *env, const int32_t *pixels_dev, const uint8_t *mask_dev, uint64_t seed, float *obs_dev,
                           int32_t *pixels_out_dev, void *stream) {
    if (!env || !obs_dev) return fail(RT_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(env->scene->device));
    if (env->precision == RT_F64)
        CU(launch_env_reset<double>(env->scene->d.view, env->d, pixels_dev, mask_dev, seed, obs_dev, pixels_out_dev, nullptr, S(stream)));
    else
        CU(launch_env_reset<float>(env->scene->f.view, env->f, pixels_dev, mask_dev, seed, obs_dev, pixels_out_dev, nullptr, S(stream)));
    return RT_OK;
}

RT_EXPORT int rt_env_step(rt_env *env, const float *actions_dev, float *obs_dev, double *reward_dev, uint8_t *terminated_dev,
                          uint8_t *truncated_dev, int32_t *reason_dev, double *info_dev, uint64_t *stats_dev, void *stream) {
    if (!env || !actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev || !reason_dev)
        return fail(RT_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(env->scene->device));
    if (int rc = env_reshade_if_stale(env, S(stream))) return rc;
    unsigned long long *st = reinterpret_cast<unsigned long long *>(stats_dev);
    if (env->precision == RT_F64)
        CU((launch_env_step<double, double, false>(env->scene->d.view, env->d, actions_dev, obs_dev, reward_dev, terminated_dev,
                                                   truncated_dev, reason_dev, info_dev, nullptr, nullptr, 0, st, S(stream))));
    else
        CU((launch_env_step<float, double, false>(env->scene->f.view, env->f, actions_dev, obs_dev, reward_dev, terminated_dev,
                                                  truncated_dev, reason_dev, info_dev, nullptr, nullptr, 0, st, S(stream))));
    return RT_OK;
}

RT_EXPORT int rt_env_step_auto(rt_env *env, const float *actions_dev, float *obs_dev, void *reward_dev, uint8_t *terminated_dev,
                               uint8_t *truncated_dev, int32_t *reason_dev, void *info_dev, float *final_obs_dev,
                               int32_t *pixels_out_dev, uint64_t seed, uint64_t *stats_dev, void *stream) {
    if (!env || !actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev || !reason_dev)
        return fail(RT_ERR_INVALID, "NULL argument");
    if (((uintptr_t)final_obs_dev) & 7u) return fail(RT_ERR_INVALID, "final_obs must be 8-byte aligned");
    CU(cudaSetDevice(env->scene->device));
    if (int rc = env_reshade_if_stale(env, S(stream))) return rc;
    unsigned long long *st = reinterpret_cast<unsigned long long *>(stats_dev);
    if (env->precision == RT_F64)
        CU((launch_env_step<double, double, true>(env->scene->d.view, env->d, actions_dev, obs_dev, (double *)reward_dev,
                                                  terminated_dev, truncated_dev, reason_dev, (double *)info_dev, final_obs_dev,
                                                  pixels_out_dev, seed, st, S(stream))));
    else
        CU((launch_env_step<float, float, true>(env->scene->f.view, env->f, actions_dev, obs_dev, (float *)reward_dev,
                                                terminated_dev, truncated_dev, reason_dev, (float *)info_dev, final_obs_dev,
                                                pixels_out_dev, seed, st, S(stream))));
    return RT_OK;
}
