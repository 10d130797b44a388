// rt_trace.cuh -- the tracing and shading functions of the hot path, as device templates.
//
//   T = float  : product path.  Robust f-vector discriminant, rsqrt normalisation, winner-only hit point.
//   T = double : parity build.  Written in the reference's operation order (compiled with -fmad=false), so it
//                tracks the IEEE-double Python arithmetic to libm precision.
//
// Reference functions restated here (path:line relative to the reference root):
//   Ray.sphereDiscriminant          RL/ray.py:73-107
//   Intersection.nearestIntersection RL/ray.py:10-20
//   Ray.sphereExitRay               RL/ray.py:109-157
//   Ray.nearestSphereIntersect      RL/ray.py:160-231
//   Intersection.terminalRGB        RL/ray.py:37-65   (+ colour.py:21-29, light.py:3-37)
//   TraditionalRenderer.trace_ray_traditional  FB/fb_vs_traditional_chandelier.py:431-521 (= complex.py:299-389)
#pragma once
#include "rt_common.cuh"
#include "rt_lbvh.cuh"

namespace rt {

// ------------------------------------------------------------------ geometry view
template <typename T> struct Geo {
    SphereView<T> sv;     // spheres (shared-memory staged or global)
    BvhView bvh;          // nodes == 0 -> brute force over sv
};

template <typename T> struct Hit {
    int idx;              // scene index, -1 = none
    T t;                  // Intersection.distance (signed)
    V3<T> p, n;
    int bounces, through;
};

template <typename T> RT_DEV V3<T> centre_of(typename M<T>::v4 s) { return mk<T>(s.x, s.y, s.z); }

// One ray/sphere test (ray.py:73-107), near root (point = 0) or far root (point = 1).  D is a unit vector.
template <typename T> RT_DEV bool sphere_test(V3<T> O, V3<T> D, typename M<T>::v4 s, int point, T &t) {
    V3<T> L = centre_of<T>(s) - O;
    T tca = dot(L, D);
    if constexpr (M<T>::exact) {
        if (tca < T(0)) return false;                     // ray.py:81-82
        T q = dot(L, L) - tca * tca;
        T d = q < T(0) ? T(0) : ::sqrt(q);                // ray.py:85-88 (math.sqrt raising -> d = 0)
        if (d > s.w) return false;                        // ray.py:89-90
        T thc = ::sqrt(s.w * s.w - d * d);
        t = point ? tca + thc : tca - thc;                // ray.py:93-96 (may be negative)
        return true;
    } else {
        // |L - tca D|^2 instead of L.L - tca^2: no catastrophic cancellation for the r = 99..1000 wall spheres
        V3<T> f = L - D * tca;
        T disc = fmaf(s.w, s.w, -dot(f, f));
        if (!(tca >= 0.f) || !(disc >= 0.f)) return false;
        T thc = M<T>::sqrt(disc);
        t = point ? tca + thc : tca - thc;
        return true;
    }
}

// key a candidate hit is ranked by
template <typename T, bool kAbs> RT_DEV T hit_key(V3<T> O, V3<T> D, T t) {
    if constexpr (!kAbs) return t;
    else if constexpr (M<T>::exact) { V3<T> p = O + D * t, d = p - O; return ::sqrt(d.x * d.x + d.y * d.y + d.z * d.z); }
    else return fabsf(t);
}

// Nearest hit over the scene.  kAbs = false: Algorithm A, smallest SIGNED distance wins (ray.py:10-20);
// kAbs = true: Algorithm B, smallest |hit - origin| wins (chandelier.py:438-444).  First in list wins ties.
// `suppress` is a Sphere.id (ray.py:165) or RT_NO_ID_DEV.  Returns the scene index or -1; t = signed distance.
template <typename T, bool kAbs> RT_DEV void consider(const Geo<T> &g, int i, V3<T> O, V3<T> D, int suppress, T &best,
                                                      T &bt, int &bi, unsigned &tests) {
    if (suppress != RT_NO_ID_DEV && g.sv.ids[i] == suppress) return;
    tests++;
    T t;
    if (!sphere_test<T>(O, D, g.sv.sph[i], 0, t)) return;
    const T key = hit_key<T, kAbs>(O, D, t);
    if (key < best || (key == best && i < bi)) { best = key; bt = t; bi = i; }
}

// FP32 brute force over a sphere array padded to a multiple of 8 (padding spheres have a NaN radius), branch-free:
// warps are incoherent after the first bounce, so a "does any lane hit" branch is almost always taken and only adds
// reconvergence overhead.  Per sphere: 11 FP32 ops for (tca, disc), one LOP3 that copies tca's sign into disc so that
// a single MUFU.SQRT turns every non-candidate (tca < 0 or disc < 0, ray.py:80-90) into NaN, one FADD, one compare
// (NaN compares false) and two predicated moves.  Selection uses the short L.L - tca^2 form; the winner's distance is
// then recomputed once with the cancellation-free form (sphere_test) by the caller.
template <bool kAbs>
RT_DEV void brute_select(const float4 *sph, int n_padded, V3<float> O, V3<float> D, float &best, int &bi) {
#pragma unroll 8
    for (int i = 0; i < n_padded; ++i) {
        const float4 s = sph[i];
        const float lx = s.x - O.x, ly = s.y - O.y, lz = s.z - O.z;
        const float tca = fmaf(lz, D.z, fmaf(ly, D.y, lx * D.x));
        const float ll = fmaf(lz, lz, fmaf(ly, ly, lx * lx));
        const float disc = fmaf(tca, tca, fmaf(s.w, s.w, -ll));
        const float dm = __int_as_float(__float_as_int(disc) | (__float_as_int(tca) & (int)0x80000000));
        const float t = tca - M<float>::sqrt(dm);
        const float key = kAbs ? fabsf(t) : t;
        if (key < best) { best = key; bi = i; }
    }
}

// The same loop for queries that exclude spheres by id (ray.py:165: secondary and shadow rays suppress the sphere they
// start on): the id test becomes one compare + one select on the key instead of a divergent early-out per sphere.
template <bool kAbs>
RT_DEV void brute_select_sup(const float4 *sph, const int *ids, int n, int suppress, V3<float> O, V3<float> D, float &best,
                             float &bt, int &bi, unsigned &tests) {
#pragma unroll 4
    for (int i = 0; i < n; ++i) {
        const float4 s = sph[i];
        const bool skip = ids[i] == suppress;
        // the discriminant of sphere_test (cancellation-free form), so hit / miss decisions are the same as there
        const V3<float> L = centre_of<float>(s) - O;
        const float tca = dot(L, D);
        const V3<float> f = L - D * tca;
        const float disc = fmaf(s.w, s.w, -dot(f, f));
        const float dm = __int_as_float(__float_as_int(disc) | (__float_as_int(tca) & (int)0x80000000));
        const float t = tca - M<float>::sqrt(dm);                // NaN unless tca >= 0 and disc >= 0
        float key = kAbs ? fabsf(t) : t;
        key = skip ? __int_as_float(0x7fc00000) : key;          // NaN compares false
        tests += skip ? 0u : 1u;
        if (key < best) { best = key; bt = t; bi = i; }
    }
}

// brute_select over the spheres of a warp-uniform candidate mask (camera rays of a warp tile, cone_candidates below):
// the same operations per sphere in the same ascending order, so the same winner.
template <bool kAbs>
RT_DEV void brute_select_mask(const float4 *sph, unsigned long long mask, V3<float> O, V3<float> D, float &best, int &bi) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        unsigned m = h ? (unsigned)(mask >> 32) : (unsigned)mask;
        while (m) {
            const int i = __ffs((int)m) - 1 + 32 * h;
            m &= m - 1u;
            const float4 s = sph[i];
            const float lx = s.x - O.x, ly = s.y - O.y, lz = s.z - O.z;
            const float tca = fmaf(lz, D.z, fmaf(ly, D.y, lx * D.x));
            const float ll = fmaf(lz, lz, fmaf(ly, ly, lx * lx));
            const float disc = fmaf(tca, tca, fmaf(s.w, s.w, -ll));
            const float dm = __int_as_float(__float_as_int(disc) | (__float_as_int(tca) & (int)0x80000000));
            const float t = tca - M<float>::sqrt(dm);
            const float key = kAbs ? fabsf(t) : t;
            if (key < best) { best = key; bi = i; }
        }
    }
}

// ---- packed FP32 (sm_100 f32x2) helpers: one issue slot for two FP32 lanes of work.  A pair lives in a 64-bit register.
typedef unsigned long long f32x2;
RT_DEV f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
RT_DEV void unpack2(f32x2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
RT_DEV f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
RT_DEV f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

#define RT_KEY_INF 0x7f800000            /* +inf as an int: the empty selection */

// Algorithm B nearest-hit selection over the sphere-pair array (SphereView::pk), branch-free, two spheres per FP32
// instruction.  With w = r^2 - |c|^2 stored per sphere and, per ray, od = O.D, oo = O.O:
//     tca  = c.D - od                                 3 FFMA2 per pair
//     disc = tca^2 + (w - oo + 2 c.O)                 1 FADD2 + 3 FFMA2 + 1 FFMA2 per pair
// i.e. 4 issue slots per sphere instead of 11 scalar ones.  Then per sphere: LOP3 (tca's sign into disc, so that ONE
// MUFU.SQRT turns both miss conditions of ray.py:80-90 into NaN), MUFU.SQRT, t = tca - sqrt (FADD2 per pair), and the
// key = bits(|t|) with the in-group index in the 3 low mantissa bits (LOP3).  Positive floats order like their bit
// patterns and NaN sorts above +inf, so the running minimum is VIMNMX3 (two keys per instruction) and the group's
// winner is folded into (best, base) with one compare + two selects per 8 spheres.  First in list wins ties
// (chandelier.py:438-444 uses a strict <).  Returns the scene index or -1; the caller recomputes the winner's
// distance with the cancellation-free form.
RT_DEV int brute_select_pk(const float4 *pk, int n_padded, int key_mask, V3<float> O, V3<float> D) {
    const float od = dot(O, D), oo = dot(O, O);
    const f32x2 Dx = pack2(D.x, D.x), Dy = pack2(D.y, D.y), Dz = pack2(D.z, D.z), nod = pack2(-od, -od);
    const f32x2 Bx = pack2(2.f * O.x, 2.f * O.x), By = pack2(2.f * O.y, 2.f * O.y), Bz = pack2(2.f * O.z, 2.f * O.z);
    const f32x2 noo = pack2(-oo, -oo), neg1 = pack2(-1.f, -1.f);
    int best = RT_KEY_INF, bbase = 0;
    const ulonglong2 *q = reinterpret_cast<const ulonglong2 *>(pk);
    for (int base = 0; base < n_padded; base += 8) {
        int key[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const ulonglong2 a = q[base + 2 * j], b = q[base + 2 * j + 1];       // (cx, cy) pairs, (cz, w) pairs
            const f32x2 tca = fma2(b.x, Dz, fma2(a.y, Dy, fma2(a.x, Dx, nod)));
            const f32x2 nm = fma2(b.x, Bz, fma2(a.y, By, fma2(a.x, Bx, add2(b.y, noo))));
            const f32x2 disc = fma2(tca, tca, nm);
            float tc0, tc1, d0, d1;
            unpack2(tca, tc0, tc1); unpack2(disc, d0, d1);
            const float s0 = M<float>::sqrt(__int_as_float(__float_as_int(d0) | (__float_as_int(tc0) & (int)0x80000000)));
            const float s1 = M<float>::sqrt(__int_as_float(__float_as_int(d1) | (__float_as_int(tc1) & (int)0x80000000)));
            float t0, t1;
            unpack2(fma2(pack2(s0, s1), neg1, tca), t0, t1);
            key[2 * j] = (__float_as_int(t0) & key_mask) | (2 * j);
            key[2 * j + 1] = (__float_as_int(t1) & key_mask) | (2 * j + 1);
        }
        int g = __vimin3_s32(key[0], key[1], key[2]);
        g = __vimin3_s32(g, key[3], key[4]);
        g = __vimin3_s32(g, key[5], key[6]);
        g = min(g, key[7]);
        if (g < best) { best = g; bbase = base; }
    }
    return best < RT_KEY_INF ? bbase + (best & 7) : -1;
}

// The same selection with the pair array in the kernel parameter block (PkConst, rt_common.cuh): the group loop is
// fully unrolled so that every LDCU.128 has an immediate constant-bank address, and the sphere operands of FFMA2 /
// FADD2 are uniform registers.  Groups at or beyond n_padded are skipped by a uniform branch.
//
// Vote skip: the second half of a pair's test -- sign merge, MUFU.SQRT, t, key, running minimum: 10 of its 27 issue
// cycles -- only matters if SOME lane can hit one of the two spheres, i.e. has tca >= 0 and disc >= 0 (the conditions
// the sign merge folds into the square root).  For the small spheres of a scene that is rare even for 32 incoherent
// bounce rays (complex scene: 2-24 % of the warp trips per pair, tools/sim/cull_sim.py), so one warp vote on the sign
// bits of (tca | disc) skips it for the whole warp; a skipped pair would have produced two NaN keys, so the winner,
// ties included, is unchanged and frames stay bit-identical.  The first RT_PKC_ALWAYS_PAIRS pairs (the wall spheres
// of every reference scene, hit by some lane in ~100 % of the trips) are finished unconditionally.
#ifndef RT_PKC_ALWAYS_PAIRS
#define RT_PKC_ALWAYS_PAIRS 3
#endif
#ifndef RT_VOTE_PAIRS
#define RT_VOTE_PAIRS 2
#endif
static_assert(RT_VOTE_PAIRS == 1 || RT_VOTE_PAIRS == 2 || RT_VOTE_PAIRS == 4, "pairs per vote");
// kWarp: ALL 32 lanes of the warp call this together (`live` = this lane carries a ray; the others only vote "no"), so
// the votes use the full mask and compile to ISETP (live folded into its predicate input) + VOTE.ANY + BRA.  Callers
// that cannot guarantee a converged warp use kWarp = false: no votes, every pair is finished.
template <bool kWarp>
RT_DEV int brute_select_pkc(const PkConst &pkc, int n_padded, int key_mask6, V3<float> O, V3<float> D, bool live = true) {
    const float od = dot(O, D), oo = dot(O, O);
    const f32x2 Dx = pack2(D.x, D.x), Dy = pack2(D.y, D.y), Dz = pack2(D.z, D.z), nod = pack2(-od, -od);
    const f32x2 Bx = pack2(2.f * O.x, 2.f * O.x), By = pack2(2.f * O.y, 2.f * O.y), Bz = pack2(2.f * O.z, 2.f * O.z);
    const f32x2 noo = pack2(-oo, -oo), neg1 = pack2(-1.f, -1.f);
    // RT_PKC_MAX = 64 spheres: the key carries the SCENE index in its 6 low mantissa bits (the unrolled loop knows it
    // at compile time), so the running minimum over all spheres is one VIMNMX3 per pair and nothing else.
    static_assert(RT_PKC_MAX == 64, "key layout: 6 index bits");
    int best = RT_KEY_INF;
#pragma unroll
    for (int base = 0; base < RT_PKC_MAX; base += 8) {
        if (base >= n_padded) break;                  // ONE exit: the groups behind it are never fetched
#pragma unroll
        for (int j0 = 0; j0 < 4; j0 += RT_VOTE_PAIRS) {
            // RT_VOTE_PAIRS pairs share one vote (1, 2 or 4: fewer votes and branches against a lower skip rate)
            f32x2 tca[RT_VOTE_PAIRS], disc[RT_VOTE_PAIRS];
            int x = -1;
#pragma unroll
            for (int v = 0; v < RT_VOTE_PAIRS; ++v) {
                const int j = j0 + v;
                const ulonglong2 a = pkc.q[base + 2 * j], b = pkc.q[base + 2 * j + 1];
                tca[v] = fma2(b.x, Dz, fma2(a.y, Dy, fma2(a.x, Dx, nod)));
                const f32x2 nm = fma2(b.x, Bz, fma2(a.y, By, fma2(a.x, Bx, add2(b.y, noo))));
                disc[v] = fma2(tca[v], tca[v], nm);
                float tc0, tc1, d0, d1;
                unpack2(tca[v], tc0, tc1); unpack2(disc[v], d0, d1);
                // sign bit of x stays set <=> no sphere so far has tca >= 0 and disc >= 0 on this lane
                x &= (__float_as_int(tc0) | __float_as_int(d0)) & (__float_as_int(tc1) | __float_as_int(d1));
            }
            const bool always = base / 2 + j0 < RT_PKC_ALWAYS_PAIRS;
            bool some = true;
            if (kWarp && !always) some = __any_sync(0xffffffffu, x >= 0 && live);
            if (__builtin_expect(some, always)) {
#pragma unroll
                for (int v = 0; v < RT_VOTE_PAIRS; ++v) {
                    const int j = j0 + v;
                    float tc0, tc1, d0, d1;
                    unpack2(tca[v], tc0, tc1); unpack2(disc[v], d0, d1);
                    const float s0 = M<float>::sqrt(__int_as_float(__float_as_int(d0) | (__float_as_int(tc0) & (int)0x80000000)));
                    const float s1 = M<float>::sqrt(__int_as_float(__float_as_int(d1) | (__float_as_int(tc1) & (int)0x80000000)));
                    float t0, t1;
                    unpack2(fma2(pack2(s0, s1), neg1, tca[v]), t0, t1);
                    best = __vimin3_s32(best, (__float_as_int(t0) & key_mask6) | (base + 2 * j),
                                        (__float_as_int(t1) & key_mask6) | (base + 2 * j + 1));
                }
            }
        }
    }
    RT_ASSERT(best >= RT_KEY_INF || (best & 63) < n_padded);
    return best < RT_KEY_INF ? (best & 63) : -1;
}

// ---- primary rays: warp-coherent candidate list.
// All rays of a warp tile start at the camera and pass through one small pixel block, i.e. they lie in a cone of
// half-angle <= alpha around the block's central direction d0.  A sphere that no ray of that cone can touch is a miss
// for every lane, so the nearest-hit query may skip it WITHOUT changing its result: keys of the remaining spheres are
// computed with the very same operations as in brute_select_pkc (scalar FFMA instead of FFMA2 lanes), so the winner,
// ties included, is identical and frames stay bit-for-bit the same.  cone_candidates builds the list once per warp
// tile (it does not depend on the sample): lane l tests spheres l and l + 32.
//   kept  <=>  camera inside the sphere, or  dist(centre, central ray) <= r + |L| alpha  and the centre is not behind
// (rotating a ray by alpha moves its closest approach to a point at distance |L| by at most |L| alpha); margins cover
// the rounding of this test itself.
RT_DEV unsigned long long cone_candidates(const float4 *sph, int n, V3<float> cam, V3<float> d0, float alpha, int lane) {
    unsigned m[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int i = lane + 32 * h;
        bool keep = false;
        if (i < n) {
            const float4 s = sph[i];
            const float lx = s.x - cam.x, ly = s.y - cam.y, lz = s.z - cam.z;
            const float ll = fmaf(lz, lz, fmaf(ly, ly, lx * lx)), tc = fmaf(lz, d0.z, fmaf(ly, d0.y, lx * d0.x));
            const float reach = fmaf(sqrtf(ll), alpha, s.w) * 1.002f + 1e-4f;        // r + |L| alpha, grown
            const float fx = fmaf(-tc, d0.x, lx), fy = fmaf(-tc, d0.y, ly), fz = fmaf(-tc, d0.z, lz);
            const float perp2 = fmaf(fz, fz, fmaf(fy, fy, fx * fx));                  // |L - tc d0|^2: no cancellation
            keep = !(ll > s.w * s.w * 1.001f) || (perp2 <= reach * reach && tc >= -reach);
            keep = keep || !(ll == ll) || !(reach == reach);                          // never cull on NaN
        }
        m[h] = __ballot_sync(0xffffffffu, keep);
    }
    return ((unsigned long long)m[1] << 32) | m[0];
}

// nearest hit among the candidates (warp-uniform mask): the keys of brute_select_pkc, one sphere at a time
RT_DEV int select_candidates(const float4 *cw, unsigned long long mask, int key_mask6, V3<float> O, V3<float> D) {
    const float od = dot(O, D), oo = dot(O, O);
    const float bx = 2.f * O.x, by = 2.f * O.y, bz = 2.f * O.z;
    int best = RT_KEY_INF;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        unsigned m = h ? (unsigned)(mask >> 32) : (unsigned)mask;
        const float4 *base = cw + 32 * h;
        while (m) {
            const int i = __ffs((int)m) - 1;
            m &= m - 1u;
            const float4 c = base[i];
            const float tca = fmaf(c.z, D.z, fmaf(c.y, D.y, fmaf(c.x, D.x, -od)));
            const float nm = fmaf(c.z, bz, fmaf(c.y, by, fmaf(c.x, bx, c.w + -oo)));
            const float disc = fmaf(tca, tca, nm);
            const float s = M<float>::sqrt(__int_as_float(__float_as_int(disc) | (__float_as_int(tca) & (int)0x80000000)));
            const float t = fmaf(s, -1.f, tca);
            best = min(best, (__float_as_int(t) & key_mask6) | (i + 32 * h));
        }
    }
    return best < RT_KEY_INF ? (best & 63) : -1;
}

// winner's distance from the cancellation-free form |L - tca D|^2; a silhouette-grazing winner whose robust
// discriminant rounds below zero gets thc = 0
RT_DEV float winner_distance(float4 w, V3<float> O, V3<float> D) {
    const V3<float> L = centre_of<float>(w) - O;
    const float tca = dot(L, D);
    const V3<float> f = L - D * tca;
    return tca - M<float>::sqrt(fmaxf(fmaf(w.w, w.w, -dot(f, f)), 0.f));
}

template <typename T, bool kAbs, bool kBvh, typename PK = PkNone>
RT_DEV int nearest(const Geo<T> &g, V3<T> O, V3<T> D, int suppress, T &t_out, unsigned &tests, unsigned &box_tests,
                   const PK &pkc = PK(), unsigned long long cand = ~0ull) {
    T best = M<T>::inf(), bt = T(0);
    int bi = -1;
    bool brute = true;
    if constexpr (kBvh) brute = g.bvh.nodes == 0;
    if (brute) {
        const int n = g.sv.n;
        if (suppress == RT_NO_ID_DEV) {
            if constexpr (!M<T>::exact) {
                if constexpr (kAbs && std::is_same<PK, PkConst>::value) bi = brute_select_pkc<false>(pkc, g.sv.n_padded, g.sv.key_mask6, O, D);
                else if constexpr (kAbs) bi = brute_select_pk(g.sv.pk, g.sv.n_padded, g.sv.key_mask, O, D);
                else if (cand != ~0ull) brute_select_mask<kAbs>(g.sv.sph, cand, O, D, best, bi);     // warp-uniform
                else brute_select<kAbs>(g.sv.sph, g.sv.n_padded, O, D, best, bi);
                if (bi >= 0) {
                    // winner's distance from the cancellation-free form |L - tca D|^2; a silhouette-grazing winner
                    // whose robust discriminant rounds below zero gets thc = 0
                    const typename M<T>::v4 w = g.sv.sph[bi];
                    const V3<T> L = centre_of<T>(w) - O;
                    const T tca = dot(L, D);
                    const V3<T> f = L - D * tca;
                    bt = tca - M<T>::sqrt(fmaxf(fmaf(w.w, w.w, -dot(f, f)), 0.f));
                }
            } else {
#pragma unroll 2
                for (int i = 0; i < n; ++i) {
                    T t;
                    if (sphere_test<T>(O, D, g.sv.sph[i], 0, t)) {
                        const T key = hit_key<T, kAbs>(O, D, t);
                        if (key < best) { best = key; bt = t; bi = i; }
                    }
                }
            }
            tests += cand != ~0ull ? (unsigned)__popcll(cand) : (unsigned)n;
        } else if constexpr (!M<T>::exact) {
            // FP32, spheres excluded by id: branch-free selection on sphere_test's own discriminant
            brute_select_sup<kAbs>(g.sv.sph, g.sv.ids, n, suppress, O, D, best, bt, bi, tests);
        } else {
#pragma unroll 2
            for (int i = 0; i < n; ++i) consider<T, kAbs>(g, i, O, D, suppress, best, bt, bi, tests);
        }
    } else if constexpr (kBvh) {
        for (int k = 0; k < g.bvh.n_huge; ++k) consider<T, kAbs>(g, g.bvh.huge[k], O, D, suppress, best, bt, bi, tests);
        // float boxes (conservatively grown at build time) cull for both precisions
        float ox = (float)O.x, oy = (float)O.y, oz = (float)O.z;
        float idx_ = 1.f / (float)D.x, idy = 1.f / (float)D.y, idz = 1.f / (float)D.z;
        int stack[RT_BVH_STACK];
        int sp = 0;
        int node = g.bvh.root;            // >= 0 internal, < 0 leaf ~prim
        for (;;) {
            if (node < 0) {
                RT_ASSERT(~node >= 0 && ~node < g.bvh.nodes && g.bvh.prims[~node] >= 0 && g.bvh.prims[~node] < g.sv.n);
                consider<T, kAbs>(g, g.bvh.prims[~node], O, D, suppress, best, bt, bi, tests);
            } else {
                RT_ASSERT(node < g.bvh.nodes - 1 || g.bvh.nodes == 1);          // n - 1 internal nodes
                const float4 a = g.bvh.node4[4 * node + 0], b = g.bvh.node4[4 * node + 1],
                             c = g.bvh.node4[4 * node + 2], ch = g.bvh.node4[4 * node + 3];
                box_tests += 2;
                float bound = (float)best * 1.00001f + 1e-6f;
                // left child
                float t0x = (a.x - ox) * idx_, t1x = (a.y - ox) * idx_, t0y = (a.z - oy) * idy, t1y = (a.w - oy) * idy;
                float t0z = (c.x - oz) * idz, t1z = (c.y - oz) * idz;
                float ln = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fminf(t0z, t1z));
                float lf = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fmaxf(t0z, t1z));
                bool hl = ln <= lf && lf >= 0.f && ln <= bound;
                t0x = (b.x - ox) * idx_; t1x = (b.y - ox) * idx_; t0y = (b.z - oy) * idy; t1y = (b.w - oy) * idy;
                t0z = (c.z - oz) * idz; t1z = (c.w - oz) * idz;
                float rn = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fminf(t0z, t1z));
                float rf = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fmaxf(t0z, t1z));
                bool hr = rn <= rf && rf >= 0.f && rn <= bound;
                int cl = __float_as_int(ch.x), cr = __float_as_int(ch.y);
                if (hl && hr) {
                    bool left_first = ln <= rn;
                    int nearc = left_first ? cl : cr, farc = left_first ? cr : cl;
                    RT_ASSERT(sp < RT_BVH_STACK);                          // a dropped subtree would lose hits
                    if (sp < RT_BVH_STACK) stack[sp++] = farc;
                    node = nearc;
                    continue;
                }
                if (hl) { node = cl; continue; }
                if (hr) { node = cr; continue; }
            }
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    t_out = bt;
    return bi;
}

template <typename T> RT_DEV void finish_hit(const Geo<T> &g, V3<T> O, V3<T> D, int i, T t, Hit<T> &h) {
    h.idx = i; h.t = t;
    h.p = O + D * t;                                          // ray.py:99
    if constexpr (M<T>::exact) h.n = normalise(h.p - centre_of<T>(g.sv.sph[i]));      // ray.py:100
    else h.n = (h.p - centre_of<T>(g.sv.sph[i])) * g.sv.col[i].w;                     // col.w = 1/r
}

// Ray.sphereExitRay (ray.py:109-157).  false = trapped (reference prints + returns None) or the reference would
// raise (entry TIR for ior < 1, degenerate chord): callers treat both as None.
template <typename T>
RT_DEV bool sphere_exit_ray(V3<T> D, typename M<T>::v4 sph, T ior, const Hit<T> &in, V3<T> &eo, V3<T> &ed) {
    V3<T> refr;
    if (!refract<T>(D, in.n, T(1), ior, refr)) return false;
    V3<T> C = centre_of<T>(sph);
    V3<T> xo = in.p, xd = M<T>::exact ? normalise(refr) : refr;
    T t;
    if (!sphere_test<T>(xo, xd, sph, 1, t)) return false;
    V3<T> xp = xo + xd * t, xn = normalise(xp - C);
    V3<T> exit_d;
    bool done = false;
    for (int k = 0; k < 10 && !done; ++k) {
        if (refract<T>(refr, -xn, ior, T(1), exit_d)) done = true;
        else {
            refr = reflect<T>(refr, xn);                      // total internal reflection, ray.py:137
            xd = M<T>::exact ? normalise(refr) : refr;
            if (!sphere_test<T>(xp, xd, sph, 1, t)) return false;
            xp = xp + xd * t;
            xn = normalise(xp - C);
        }
    }
    if (!done) return false;
    eo = xp;
    ed = M<T>::exact ? normalise(exit_d) : exit_d;
    return true;
}

struct Counters { unsigned queries, tests, boxes, dead; };      // dead: queries the reference casts and then discards (skipped)

// Ray.nearestSphereIntersect (ray.py:160-231) with the recursion unrolled: a mirror that finds nothing returns
// ITSELF (ray.py:198-201), glass that finds nothing returns None (ray.py:226-229), so a dead-ended chain yields the
// most recent mirror hit, else None.  D is a unit vector.
template <typename T, bool kBvh>
RT_DEV Hit<T> trace_terminal(const Geo<T> &g, V3<T> O, V3<T> D, int suppress, int bounces, int max_bounces, int through,
                             Counters &ct, unsigned long long cand = ~0ull) {     // cand: spheres the FIRST query may hit
    Hit<T> fallback;
    fallback.idx = -1; fallback.t = T(0); fallback.bounces = 0; fallback.through = 0;
    fallback.p = mk<T>(0, 0, 0); fallback.n = mk<T>(0, 0, 0);
    for (;;) {
        ct.queries++;
        T t;
        int i = nearest<T, false, kBvh>(g, O, D, suppress, t, ct.tests, ct.boxes, PkNone(), cand);
        cand = ~0ull;
        if (i < 0) return fallback;                           // ray.py:170-171
        if (bounces > max_bounces) return fallback;           // ray.py:173-174
        Hit<T> h;
        finish_hit<T>(g, O, D, i, t, h);
        h.bounces = bounces; h.through = through;
        const typename M<T>::v4 m = g.sv.mat[i];
        if (m.x == T(1)) {                                    // material.reflective == True, ray.py:180
            fallback = h;
            V3<T> r = reflect<T>(D, h.n);
            D = M<T>::exact ? normalise(r) : r;               // Ray() normalises again
            O = h.p;
            bounces += 1; suppress = g.sv.ids[i];
            // the reference casts the mirrored ray even when the bounce limit is spent and then discards what it finds
            // (ray.py:170-174: both exits return the mirror itself): do not trace it
            if (bounces > max_bounces) { ct.dead++; return fallback; }
            continue;
        }
        if (m.y == T(1)) {                                    // material.transparent == True, ray.py:204
            V3<T> eo, ed;
            if (!sphere_exit_ray<T>(D, g.sv.sph[i], m.w, h, eo, ed)) return fallback;
            O = eo; D = ed;
            bounces += 1; through += 1; suppress = g.sv.ids[i];
            if (bounces > max_bounces) { ct.dead++; return fallback; }      // as above: the exit ray's result is discarded
            continue;
        }
        return h;
    }
}

template <typename T> RT_DEV T incidence(T angle, T max_angle) {        // light.py:3-9
    if (angle > max_angle) return T(0);
    if (angle == T(0)) return T(1);
    return (max_angle - angle) / max_angle;
}

// lights of Algorithm A as the shading function sees them
template <typename T> struct LightsA {
    using v4 = typename M<T>::v4;
    int nG, nP;
    const v4 *g_vec, *g_col; const int *g_func;     // g_vec.w = max_angle, g_col.w = strength
    const v4 *p_pos, *p_col; const int *p_id, *p_func;
    T bg[3];
};

// Intersection.terminalRGB (ray.py:37-65) + Colour.illuminate (colour.py:21-29, round half to even, not clamped)
template <typename T, bool kBvh>
RT_DEV void terminal_rgb(const Geo<T> &g, const LightsA<T> &lt, const Hit<T> &h, int shadow_max_bounces, T out[3],
                         Counters &ct) {
    const typename M<T>::v4 m = g.sv.mat[h.idx], col = g.sv.col[h.idx];
    T il0 = col.x * m.z, il1 = col.y * m.z, il2 = col.z * m.z;            // ray.py:41
    for (int k = 0; k < lt.nG; ++k) {                                      // ray.py:43-45
        if (lt.g_func[k] != 0) continue;
        const typename M<T>::v4 gv = lt.g_vec[k], gc = lt.g_col[k];
        T ang = angle_between<T>(h.n, mk<T>(gv.x, gv.y, gv.z));
        T sc = incidence<T>(ang, gv.w) * gc.w;
        il0 = il0 + gc.x * sc; il1 = il1 + gc.y * sc; il2 = il2 + gc.z * sc;
    }
    const int own = g.sv.ids[h.idx];
    for (int k = 0; k < lt.nP; ++k) {                                      // ray.py:47-62
        const int pid = lt.p_id[k];
        if (own == pid) continue;
        const typename M<T>::v4 pp = lt.p_pos[k], pc = lt.p_col[k];
        V3<T> vl = mk<T>(pp.x, pp.y, pp.z) - h.p;
        Hit<T> s = trace_terminal<T, kBvh>(g, h.p, normalise(vl), own, 0, shadow_max_bounces, 0, ct);
        if (s.idx < 0 || g.sv.ids[s.idx] != pid) continue;
        T ang = angle_between<T>(h.n, vl);
        const int fn = lt.p_func[k];
        T sc;
        if (fn == -1) sc = incidence<T>(ang, pp.w) * pc.w;
        else if (fn == 0) sc = incidence<T>(ang, pp.w) * pc.w / mag(vl);
        else continue;
        il0 = il0 + pc.x * sc; il1 = il1 + pc.y * sc; il2 = il2 + pc.z * sc;
    }
    out[0] = lt.bg[0] + M<T>::rint(col.x * (il0 / T(255)));
    out[1] = lt.bg[1] + M<T>::rint(col.y * (il1 / T(255)));
    out[2] = lt.bg[2] + M<T>::rint(col.z * (il2 / T(255)));
}

// ------------------------------------------------------------------ Algorithm B
// light spheres of TraditionalRenderer.light_sources: l_pos.w = scene index (int bits via __T_as_int surrogate: stored
// as a separate int array), l_col = colour.
template <typename T> struct LightsB {
    using v4 = typename M<T>::v4;
    int nL;
    const v4 *l_pos, *l_col, *lpk;
    const int *l_index;
};

// Per-level record of the unrolled recursion: the hit sphere (albedo) and the direct light collected there,
// clamped to 255 per channel.  Clamping early is exact: direct is a sum of int()s and the indirect term is >= 0,
// so min(255, direct + ind) == min(255, min(255, direct) + ind).
struct PathStack {
    uint32_t idx[RT_PATH_MAX_DEPTH];
    uint32_t direct[RT_PATH_MAX_DEPTH];     // r | g << 8 | b << 16
};

// final = int(albedo * (min(255, direct + indirect) / 255.0)) per channel, folded from the leaf back to the camera
// (chandelier.py:509-521).  Always evaluated in double: the truncation must see the reference's rounding.
template <typename T, bool kPacked = false>
RT_DEV void fold_path(const Geo<T> &g, const PathStack &st, int depth, double c[3], int k0 = 0) {
    for (int k = depth - 1; k >= k0; --k) {
        const uint32_t d = st.direct[k];
        const typename M<T>::v4 col = g.sv.col[kPacked ? (d >> 24) : st.idx[k]];
        double t0 = (double)(d & 255u) + c[0], t1 = (double)((d >> 8) & 255u) + c[1], t2 = (double)((d >> 16) & 255u) + c[2];
        t0 = t0 < 255.0 ? t0 : 255.0; t1 = t1 < 255.0 ? t1 : 255.0; t2 = t2 < 255.0 ? t2 : 255.0;
        c[0] = ::trunc(__dmul_rn((double)col.x, __ddiv_rn(t0, 255.0)));
        c[1] = ::trunc(__dmul_rn((double)col.y, __ddiv_rn(t1, 255.0)));
        c[2] = ::trunc(__dmul_rn((double)col.z, __ddiv_rn(t2, 255.0)));
    }
}

// Same fold for integer-valued leaves (every scene of the reference: colours are 0-255 ints): tot is then an integer
// in [0,255] at every level, so tot/255.0 comes from a 256-entry table of correctly rounded doubles (identical to
// the division) and the running colour stays an int.  Still a double multiply: the truncation sees the same product.
// kPacked: the level's sphere index rides in bits 24-31 of `direct` (scenes of <= 256 spheres), st.idx is not used.
template <typename T, bool kPacked = false>
RT_DEV void fold_path_int(const Geo<T> &g, const PathStack &st, int depth, const double *div255, int c[3], int k0 = 0,
                          unsigned col_base = 0,              // kPacked: shared-window address of the colour array
                          unsigned tab = 0) {                 // kPacked: shared-window address of the fold table, or 0
    RT_ASSERT(depth >= 0 && depth <= RT_PATH_MAX_DEPTH);
    if constexpr (kPacked && !M<T>::exact) {
        if (tab) {
            // every colour <= 255: int(albedo * (tot / 255.0)) was tabulated per (sphere, channel, tot) when the CTA started
            // (path_kernel) with the same double product, so a level is one byte load per channel
            for (int k = depth - 1; k >= k0; --k) {
                const uint32_t d = st.direct[k];
                RT_ASSERT((int)(d >> 24) < g.sv.n);
                const unsigned row = tab + 768u * (d >> 24);
                const unsigned a0 = row + (unsigned)min(255, (int)(d & 255u) + c[0]);
                const unsigned a1 = row + (unsigned)min(255, (int)__byte_perm(d, 0u, 0x4441u) + c[1]);
                const unsigned a2 = row + (unsigned)min(255, (int)__byte_perm(d, 0u, 0x4442u) + c[2]);
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(c[0]) : "r"(a0));
                asm volatile("ld.shared.u8 %0, [%1+256];" : "=r"(c[1]) : "r"(a1));
                asm volatile("ld.shared.u8 %0, [%1+512];" : "=r"(c[2]) : "r"(a2));
            }
            return;
        }
    }
    for (int k = depth - 1; k >= k0; --k) {
        const uint32_t d = st.direct[k];
        RT_ASSERT((int)(kPacked ? (d >> 24) : st.idx[k]) < g.sv.n);
        typename M<T>::v4 col;
        if constexpr (kPacked && !M<T>::exact) {
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(col.x), "=f"(col.y), "=f"(col.z), "=f"(col.w)
                         : "r"(col_base + 16u * (d >> 24)));
        } else col = g.sv.col[kPacked ? (d >> 24) : st.idx[k]];
        const int t0 = min(255, (int)(d & 255u) + c[0]), t1 = min(255, (int)((d >> 8) & 255u) + c[1]),
                  t2 = min(255, (int)((d >> 16) & 255u) + c[2]);
        c[0] = __double2int_rz(__dmul_rn((double)col.x, div255[t0]));
        c[1] = __double2int_rz(__dmul_rn((double)col.y, div255[t1]));
        c[2] = __double2int_rz(__dmul_rn((double)col.z, div255[t2]));
    }
}

// direct light at a non-emissive hit: every light sphere, NO occlusion test (chandelier.py:463-477)
template <typename T>
RT_DEV uint32_t direct_light(const LightsB<T> &lb, int hit_idx, V3<T> p, V3<T> n) {
    T d0 = T(0), d1 = T(0), d2 = T(0);
    for (int l = 0; l < lb.nL; ++l) {
        if (lb.l_index[l] == hit_idx) continue;
        const typename M<T>::v4 lp = lb.l_pos[l], lc = lb.l_col[l];
        V3<T> tl = mk<T>(lp.x, lp.y, lp.z) - p;
        if constexpr (M<T>::exact) {
            V3<T> tln = normalise(tl);
            T ca = dot(n, tln);
            if (!(ca > T(0))) continue;
            T dist = ::sqrt(dot(tl, tl)), att = 1.0 / (dist * dist);
            d0 += ::trunc(lc.x * ca * att * 0.3); d1 += ::trunc(lc.y * ca * att * 0.3); d2 += ::trunc(lc.z * ca * att * 0.3);
        } else {
            T q = dot(tl, tl), inv = M<T>::rsqrt(q);
            T ca = dot(n, tl) * inv;
            if (!(ca > 0.f)) continue;
            T s = ca * (inv * inv) * 0.3f;
            d0 += truncf(lc.x * s); d1 += truncf(lc.y * s); d2 += truncf(lc.z * s);
        }
    }
    d0 = d0 < T(255) ? d0 : T(255); d1 = d1 < T(255) ? d1 : T(255); d2 = d2 < T(255) ? d2 : T(255);
    return (uint32_t)d0 | ((uint32_t)d1 << 8) | ((uint32_t)d2 << 16);
}

// FP32 product form of direct_light over the light-pair array (SceneDev::lpk), branch-free, two lights per FP32
// instruction.  Positions are stored times 128 (A = 128 l, with |A|^2 beside them) and colours times 0.3 * 16384, so
// with tl' = A - p', p' = 128 p:
//     tl'.tl' = |A|^2 + |p'|^2 - 2 A.p'      (1 FADD2 + 3 FFMA2 per pair: the per-hit terms are packed once)
//     n.tl'   = n.A - n.p'                    (3 FFMA2)
// -- 7 packed operations per pair instead of the 9 of (A - p') first; the cancellation costs < 1e-6 of the squared
// distance for a light a few units away (|A|^2 ~ 1e6, FP32) and 3e-4 for one 0.3 away, where the contribution saturates --
//     s' = sat(n.tl' * rsqrt(tl'.tl')^3) = sat(cos / d^2 / 16384),     x = colour' * s' = colour * cos * 0.3 / d^2
// and a contribution that saturates is >= 255 on every channel with colour >= 0.052, i.e. the final min(255, .)
// hides the clamp.  cos <= 0 saturates to 0 (chandelier.py:470: `if cos_angle > 0`); the self test of
// chandelier.py:465 is implied: for a light that is itself the (non-emissive) hit sphere, l - p = -r n, cos = -1.
// int() is FFMA2.RZ onto 2^23 (the mantissa then holds floor(x) for 0 <= x < 2^23) and the sums are integer adds.
RT_DEV f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
RT_DEV f32x2 fma2_rz(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rz.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
RT_DEV float mul_sat(float a, float b) { float d; asm("mul.rn.sat.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b)); return d; }
RT_DEV uint32_t direct_light_pk(const float4 *lpk, int n_pairs, V3<float> p, V3<float> n) {
    // array form (large scenes: hundreds of lights read through L1): tl' = A - p' first, 9 packed operations and THREE
    // vector loads per pair -- the expanded form of direct_light_pkc needs the fourth vector (|A|^2), and here the loads,
    // not the arithmetic, are what a pair costs (measured: 222 -> 242 ms per frame of the 1e5-sphere scene with it)
    const float qx = -128.f * p.x, qy = -128.f * p.y, qz = -128.f * p.z;
    const f32x2 px = pack2(qx, qx), py = pack2(qy, qy), pz = pack2(qz, qz);
    const f32x2 nx = pack2(n.x, n.x), ny = pack2(n.y, n.y), nz = pack2(n.z, n.z);
    const f32x2 magic = pack2(8388608.f, 8388608.f);
    unsigned a0 = 0u, a1 = 0u, a2 = 0u;
    const ulonglong2 *q = reinterpret_cast<const ulonglong2 *>(lpk);
#pragma unroll 2
    for (int j = 0; j < n_pairs; ++j) {
        const ulonglong2 A = q[RT_LPK_STRIDE * j], B = q[RT_LPK_STRIDE * j + 1], C = q[RT_LPK_STRIDE * j + 2];
        const f32x2 tx = add2(A.x, px), ty = add2(A.y, py), tz = add2(B.x, pz);
        const f32x2 qq = fma2(tz, tz, fma2(ty, ty, mul2(tx, tx)));
        const f32x2 dn = fma2(tz, nz, fma2(ty, ny, mul2(tx, nx)));
        float q0, q1;
        unpack2(qq, q0, q1);
        const f32x2 inv = pack2(M<float>::rsqrt(q0), M<float>::rsqrt(q1));
        float a_lo, a_hi, b_lo, b_hi;
        unpack2(mul2(dn, inv), a_lo, a_hi);
        unpack2(mul2(inv, inv), b_lo, b_hi);
        const f32x2 s = pack2(mul_sat(a_lo, b_lo), mul_sat(a_hi, b_hi));
        unsigned r_lo, r_hi, g_lo, g_hi, b0, b1;
        asm("mov.b64 {%0, %1}, %2;" : "=r"(r_lo), "=r"(r_hi) : "l"(fma2_rz(B.y, s, magic)));
        asm("mov.b64 {%0, %1}, %2;" : "=r"(g_lo), "=r"(g_hi) : "l"(fma2_rz(C.x, s, magic)));
        asm("mov.b64 {%0, %1}, %2;" : "=r"(b0), "=r"(b1) : "l"(fma2_rz(C.y, s, magic)));
        a0 += r_lo + r_hi; a1 += g_lo + g_hi; a2 += b0 + b1;
    }
    const unsigned bias = 2u * (unsigned)n_pairs * 0x4B000000u;          // bits of 2^23, once per light
    a0 = min(a0 - bias, 255u); a1 = min(a1 - bias, 255u); a2 = min(a2 - bias, 255u);
    return a0 | (a1 << 8) | (a2 << 16);
}

// direct_light_pk over the light pairs in the kernel parameter block (PkConst::l): fully unrolled, uniform operands.
// An ODD number of lights (3 in the complex scene, 21 in the chandelier) leaves one light without a partner: the host
// packs it FIRST (pair 0 = light 0 + a black filler, rt_api.cu pack_scene) and it is evaluated here with scalar
// instructions -- half the issue cycles of a packed pair whose second lane would shade the filler.
RT_DEV float fma_rz(float a, float b, float c) { float d; asm("fma.rz.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c)); return d; }
RT_DEV uint32_t direct_light_pkc(const PkConst &pkc, int n_lights, V3<float> p, V3<float> n) {
    const int n_pairs = (n_lights + 1) >> 1;
    const bool odd = (n_lights & 1) != 0;
    const float qx = 128.f * p.x, qy = 128.f * p.y, qz = 128.f * p.z;                      // p' = 128 p
    const float pp_ = fmaf(qz, qz, fmaf(qy, qy, qx * qx)), np_ = fmaf(n.z, qz, fmaf(n.y, qy, n.x * qx));
    const f32x2 px = pack2(-2.f * qx, -2.f * qx), py = pack2(-2.f * qy, -2.f * qy), pz = pack2(-2.f * qz, -2.f * qz);
    const f32x2 nx = pack2(n.x, n.x), ny = pack2(n.y, n.y), nz = pack2(n.z, n.z);
    const f32x2 pp2 = pack2(pp_, pp_), nnp = pack2(-np_, -np_);
    const f32x2 magic = pack2(8388608.f, 8388608.f);
    unsigned a0 = 0u, a1 = 0u, a2 = 0u;
#pragma unroll
    for (int j = 0; j < RT_LPKC_MAX / 2; ++j) {
        if (j >= n_pairs) break;                      // ONE exit (a guard per pair costs a taken branch per skipped pair)
        if (j == 0 && odd) {                          // (j is a compile-time constant in every unrolled copy)
            const ulonglong2 A = pkc.l[0], B = pkc.l[1], C = pkc.l[2];
            float x, y, z, R, G, Bl, AA, u_;
            unpack2(A.x, x, u_); unpack2(A.y, y, u_); unpack2(B.x, z, u_); unpack2(B.y, R, u_);
            unpack2(C.x, G, u_); unpack2(C.y, Bl, u_); unpack2(pkc.l[3].x, AA, u_);
            const float qq = fmaf(z, -2.f * qz, fmaf(y, -2.f * qy, fmaf(x, -2.f * qx, AA + pp_)));
            const float dn = fmaf(z, n.z, fmaf(y, n.y, fmaf(x, n.x, -np_)));
            const float inv = M<float>::rsqrt(qq);
            const float s = mul_sat(dn * inv, inv * inv);
            a0 += __float_as_uint(fma_rz(R, s, 8388608.f)); a1 += __float_as_uint(fma_rz(G, s, 8388608.f));
            a2 += __float_as_uint(fma_rz(Bl, s, 8388608.f));
        } else {
            const ulonglong2 A = pkc.l[RT_LPK_STRIDE * j], B = pkc.l[RT_LPK_STRIDE * j + 1], C = pkc.l[RT_LPK_STRIDE * j + 2];
            const f32x2 qq = fma2(B.x, pz, fma2(A.y, py, fma2(A.x, px, add2(pkc.l[RT_LPK_STRIDE * j + 3].x, pp2))));
            const f32x2 dn = fma2(B.x, nz, fma2(A.y, ny, fma2(A.x, nx, nnp)));
            float q0, q1;
            unpack2(qq, q0, q1);
            const f32x2 inv = pack2(M<float>::rsqrt(q0), M<float>::rsqrt(q1));
            float a_lo, a_hi, b_lo, b_hi;
            unpack2(mul2(dn, inv), a_lo, a_hi);
            unpack2(mul2(inv, inv), b_lo, b_hi);
            const f32x2 s = pack2(mul_sat(a_lo, b_lo), mul_sat(a_hi, b_hi));
            unsigned r_lo, r_hi, g_lo, g_hi, b0, b1;
            asm("mov.b64 {%0, %1}, %2;" : "=r"(r_lo), "=r"(r_hi) : "l"(fma2_rz(B.y, s, magic)));
            asm("mov.b64 {%0, %1}, %2;" : "=r"(g_lo), "=r"(g_hi) : "l"(fma2_rz(C.x, s, magic)));
            asm("mov.b64 {%0, %1}, %2;" : "=r"(b0), "=r"(b1) : "l"(fma2_rz(C.y, s, magic)));
            a0 += r_lo + r_hi; a1 += g_lo + g_hi; a2 += b0 + b1;
        }
    }
    const unsigned bias = (unsigned)n_lights * 0x4B000000u;              // bits of 2^23, once per light evaluated
    a0 = min(a0 - bias, 255u); a1 = min(a1 - bias, 255u); a2 = min(a2 - bias, 255u);
    return a0 | (a1 << 8) | (a2 << 16);
}

// next ray of a path after a non-emissive hit (chandelier.py:479-507): mirror if reflective > threshold, else a
// cosine-weighted direction around the normal from two uniforms.
template <typename T>
RT_DEV V3<T> bounce_direction(V3<T> D, V3<T> n, bool mirror, T r1, T r2) {
    if constexpr (M<T>::exact) {
        if (mirror) return normalise(reflect<T>(D, n));
        T theta = ::acos(::sqrt(r1)), phi = 2 * 3.14159265358979323846 * r2;
        T st = ::sin(theta), ct = ::cos(theta), sp = ::sin(phi), cp = ::cos(phi);
        V3<T> tg = ::fabs(n.z) > T(0.9) ? mk<T>(1, 0, 0) : cross(mk<T>(0, 0, 1), n);
        tg = normalise(tg);
        V3<T> bt = normalise(cross(n, tg));
        T lx = st * cp, ly = st * sp, lz = ct;
        V3<T> bd = normalise(mk<T>(lx * tg.x + ly * bt.x + lz * n.x, lx * tg.y + ly * bt.y + lz * n.y,
                                   lx * tg.z + ly * bt.z + lz * n.z));
        return normalise(bd);
    } else {
        // unit D and n: the mirror direction is unit already
        if (mirror) return D - n * (2.f * dot(D, n));
        // cos/sin(acos(sqrt r1)) = sqrt(r1), sqrt(1 - r1); phi - pi in [-pi, pi) for MUFU.SIN/COS (abs error 2^-20.9),
        // sin(phi) = -sin(phi - pi), cos(phi) = -cos(phi - pi)
        const float ct = M<float>::sqrt(r1), st = M<float>::sqrt(1.f - r1);
        const float x = fmaf(r2, 6.28318530717958647692f, -3.14159265358979323846f);
        float sp, cp;
        asm("sin.approx.ftz.f32 %0, %1;" : "=f"(sp) : "f"(x));
        asm("cos.approx.ftz.f32 %0, %1;" : "=f"(cp) : "f"(x));
        // tangent (1,0,0) or (0,0,1) x n = (-n.y, n.x, 0): z is 0 either way (chandelier.py:493-496)
        const bool deg = fabsf(n.z) > 0.9f;
        float tx = deg ? 1.f : -n.y, ty = deg ? 0.f : n.x;
        const float k1 = M<float>::rsqrt(fmaf(tx, tx, ty * ty));
        tx *= k1; ty *= k1;
        const float bx = -n.z * ty, by = n.z * tx, bz = fmaf(n.x, ty, -n.y * tx);            // n x tangent
        const float k2 = M<float>::rsqrt(fmaf(bx, bx, fmaf(by, by, bz * bz)));
        const float lx = -st * cp, ly = -st * sp * k2, lz = ct;
        const float dx = fmaf(lx, tx, fmaf(ly, bx, lz * n.x)), dy = fmaf(lx, ty, fmaf(ly, by, lz * n.y)),
                    dz = fmaf(ly, bz, lz * n.z);
        const float k3 = M<float>::rsqrt(fmaf(dx, dx, fmaf(dy, dy, dz * dz)));
        return mk<float>(dx * k3, dy * k3, dz * k3);
    }
}

}  // namespace rt
