// rm_fast.cuh -- the FP32 production path of the render kernel.
//
// Same predicates as rm_trace.cuh (and therefore as the reference), arranged for the B200's FP32
// pipes instead of for a literal restatement:
//
//  * Triangles (every OBJ triangle and every 3-vertex polygon) are fixed 64-byte records, four
//    128-bit shared-memory loads each, fully unrolled -- no per-edge loop, no index arithmetic.
//  * PRIMARY rays all start at the camera, so for them the whole ray/triangle test collapses to
//    four affine functions of the UN-normalised pixel direction D = (X, Y, -1):
//        dpD = n.D,   s_i = G_i.D   with  G_i = e_i(cam)*n + K*(A_i, B_i, 0),  K = (C - cam).n
//    (e_i(p) is the reference's edge term ((v_i-p) x (v_i+1-p)).z, affine in p; at the plane point
//    p = cam + t*D, t = K/dpD, one gets e_i(p)*dpD = G_i.D).  Hit <=> t >= 0, |d.n| >= 1e-6 and
//    e_i > 0 for i = 0..2 <=> (after folding sign(K) into the record) dpD > thr*|D| and s_i > 0.
//    Eight FFMAs, two FMNMX and two FSETP per triangle; the division happens only for actual hits.
//    The records are rebuilt per frame in FP64 by prepare_raster() (one thread per triangle).
//  * Secondary and shadow rays use the general form with the edge terms evaluated relative to
//    vertex 0 (see plane_intersect<float> in rm_trace.cuh for why not at the hit point itself).
//  * Spheres and n-gons (n > 3) reuse the routines of rm_trace.cuh.
#pragma once

#include <cassert>
#include <type_traits>

#include "rm_bvh.cuh"
#include "rm_trace.cuh"

namespace rm {

constexpr int kTriSrcDoubles = 16;   // n[3], dn, v0x, v0y, A0, B0, A1, B1, C1, A2, B2, thr, id, pad

#if defined(__CUDA_ARCH__)
#define RM_PIN(v) asm volatile("" : "+f"(v))
#else
#define RM_PIN(v) (void)(v)
#endif

// Camera-specialised record of one triangle (4 x R4<float>), from its FP64 source record.
//   r0 = {n'x, n'y, -n'z, |K|}   r1 = {G0x, G0y, -G0z, thr^2}   r2 = {G1x, G1y, -G1z, id}   r3 = {G2x, G2y, -G2z, 0}
// with everything multiplied by sign(K) so that a hit needs dpD > 0 and s_i > 0.
// Under a view (ViewBasis M) the world direction is M D, and n.(M D) = (M^T n).D, G_i.(M D) = (M^T G_i).D: the records
// carry M^T n and M^T G_i, the world-space K, thr and edge terms unchanged, and stage A runs on them as it is.
template <class VW = NoView>
RM_HD void prepare_raster(const double* __restrict__ src, const double cam[3], R4<float>* __restrict__ out, const VW& vw = VW()) {
    const double nx = src[0], ny = src[1], nz = src[2], dn = src[3];
    const double wx = cam[0] - src[4], wy = cam[1] - src[5];
    const double K = dn - (cam[0] * nx + cam[1] * ny + cam[2] * nz);
    const double A[3] = {src[6], src[8], src[11]}, B[3] = {src[7], src[9], src[12]}, Cc[3] = {0., src[10], 0.};
    const double s = (K < 0.) ? -1. : 1.;
    const Vec3<double> n = vw.to_camera(Vec3<double>{nx, ny, nz});
    out[0] = {(float)(s * n.x), (float)(s * n.y), (float)(-s * n.z), (float)fabs(K)};
    float last[3] = {(float)(src[13] * src[13]), 0.f, 0.f};    // thr^2: the test runs on squared quantities
    int id = (int)src[14];
#if defined(__CUDA_ARCH__)
    last[1] = __int_as_float(id);
#else
    memcpy(&last[1], &id, 4);
#endif
    for (int i = 0; i < 3; i++) {
        const double E = A[i] * wx + B[i] * wy + Cc[i];
        if constexpr (std::is_same<VW, NoView>::value) {       // (the statement as it was before views: the same code)
            out[1 + i] = {(float)(s * (E * nx + K * A[i])), (float)(s * (E * ny + K * B[i])), (float)(-s * (E * nz)), last[i]};
        } else {
            const Vec3<double> G = vw.to_camera(Vec3<double>{E * nx + K * A[i], E * ny + K * B[i], E * nz});
            out[1 + i] = {(float)(s * G.x), (float)(s * G.y), (float)(-s * G.z), last[i]};
        }
    }
}

// kBvh: scene queries walk the hierarchy of rm_bvh.cuh instead of every primitive (RmParams.accel).  The tests per
// (ray, primitive) and the rule that picks the winner are the same code either way.
template <bool kBvh, bool kCount = false> struct FastViewT {
    // spheres
    const R4<float>* sph;
    const int* sph_id;
    int n_sph;
    // triangles: tri_g = scene records {n,dn | v0x,v0y,A0,B0 | A1,B1,C1,A2 | B2,thr,id,0}, tri_r = raster records
    const R4<float>* tri_g;
    const R4<float>* tri_r;
    int n_tri;
    // n-gons: indices into the generic plane arrays
    const int* poly_slot;
    int n_poly;
    const R4<float>* pln_n;
    const R4<float>* pln_c;
    const I2* pln_v;
    const int* pln_id;
    const R4<float>* vert;
    // materials, lights
    const R4<float>* mat_a;
    const R4<float>* mat_b;
    const int* mat_f;
    const R4<float>* lgt_p;
    const R4<float>* lgt_c;
    int n_lgt;
    // hierarchy over the hittable primitives (kBvh only), and this thread's count of scene queries behind the primary
    // one (closest-hit calls of the recursion + shadow rays): the segment count of a frame too large to run through the
    // instrumented brute-force kernel (rm_scene_query_count)
    BvhView bvh;
    mutable unsigned n_queries = 0;
    mutable BvhCount cnt;          // kCount: node visits and leaf tests of this thread's walks (rm_scene_walk_stats)
    // f64 sources for the refinement of winning hits on glass paths (cast_glass below): spheres {c, r^2}, fast-path
    // triangles (the prepare kernel's source records: n at [0..2], n.C at [3]), generic planes by slot {n, n.C}
    const double* sph64 = nullptr;
    const double* tri64 = nullptr;
    const double* pln64 = nullptr;

    // Hit point and normal of the primitive an FP32 query picked, for the f64 ray (o, d): the reference's own f64 formulas
    // (sphere.rs:28-60, triangle.rs:62-69 / polygon.rs:71-78).  t32 is the FP32 ray parameter; for a sphere it selects
    // the root the FP32 test took (sphere.rs:44-51: the near one unless it lies behind the origin).
    RM_HD void refine(const int slot, const Vec3<double> o, const Vec3<double> d, const double t32, Vec3<double>& p,
                      Vec3<double>& n) const {
        if (slot < n_sph) {
            const double* q = sph64 + 4 * (size_t)slot;
            const Vec3<double> c = {q[0], q[1], q[2]};
            const Vec3<double> line = c - o;
            const double tca = dot(line, d);
            const double d2 = dot(line, line) - tca * tca;
            const double thc = Fast64::sqrt_(q[3] - d2);       // (0 for a grazing hit FP32 accepted and f64 would not: the tangent point)
            const double ta = tca - thc, tb = tca + thc;
            const double t = fabs(ta - t32) <= fabs(tb - t32) ? ta : tb;
            p = axpy(o, d, t);
            n = Fast64::normalized(p - c);
        } else {
            const double* q = slot < n_sph + n_tri ? tri64 + (size_t)kTriSrcDoubles * (slot - n_sph) : pln64 + 4 * (size_t)(slot - n_sph - n_tri);
            n = {q[0], q[1], q[2]};
            const double t = (q[3] - dot(o, n)) * Fast64::rcp_(dot(d, n));   // ((C - o).n) / (d.n)
            p = axpy(o, d, t);
        }
    }

    static RM_HD int as_int(float f) {
#if defined(__CUDA_ARCH__)
        return __float_as_int(f);
#else
        int i;
        memcpy(&i, &f, 4);
        return i;
#endif
    }

    // General ray against the triangle whose scene record starts at g, in two stages.
    // Stage 1 (tri_front): d.n and (C - o).n from the first 16 bytes of the record.  triangle.rs:65 rejects
    // t = num / dp < 0, i.e. numerator and denominator of triangle.rs:62 with strictly opposite signs -- the most
    // frequent rejection needs neither the division nor the rest of the record.
    static RM_HD bool tri_front(const R4<float> a, const Vec3<float> o, const Vec3<float> d, float& dp, float& num) {
        dp = fmaf(a.z, d.z, fmaf(a.y, d.y, a.x * d.x));
        num = fmaf(-a.z, o.z, fmaf(-a.y, o.y, fmaf(-a.x, o.x, a.w)));     // (C - o).n
        return !(num * dp < 0.f);
    }
    // Stage 2 (tri_inside): parallel test, division, the three edge terms at the hit point relative to vertex 0.
    static RM_HD bool tri_inside(const R4<float>* __restrict__ g, const Vec3<float> o, const Vec3<float> d, const float dp,
                                 const float num, float& t_out) {
        const R4<float> l = g[3];
        if (!(fabsf(dp) > l.y)) return false;                  // triangle.rs:57 (parallel)
        const float t = fast_div(num, dp);                     // triangle.rs:62
        const R4<float> b = g[1], c = g[2];
        const float qx = fmaf(t, d.x, o.x - b.x), qy = fmaf(t, d.y, o.y - b.y);
        const float e0 = fmaf(b.z, qx, b.w * qy);
        const float e1 = fmaf(c.x, qx, fmaf(c.y, qy, c.z));
        const float e2 = fmaf(c.w, qx, l.x * qy);
        if (!(fminf(fminf(e0, e1), e2) > 0.f)) return false;   // triangle.rs:72-76
        t_out = t;
        return true;
    }
    static RM_HD bool tri_hit(const R4<float>* __restrict__ g, const Vec3<float> o, const Vec3<float> d, float& t_out) {
        float dp, num;
        return tri_front(g[0], o, d, dp, num) && tri_inside(g, o, d, dp, num, t_out);
    }

    RM_HD static void keep(HitRec<float>& best, bool& hit, float t, int slot, int id) {
        if (!hit || t < best.dist || (t == best.dist && id < best.id)) {
            best.dist = t;
            best.slot = slot;
            best.id = id;
            hit = true;
        }
    }

    // (the primary query is stage A of the render kernel; this is renderer.rs:266 at level > 1)
    template <bool S> RM_HD bool closest(const Vec3<float> o, const Vec3<float> d, int /*level*/, HitRec<float>& h, Counters<S>& st) const {
        bool hit = false;
        if constexpr (kBvh) {
            h.dist = INFINITY;
            n_queries++;
            bvh_walk<kCount>(bvh, o, d,
                             [&](const int e) {
                                 float t;
                                 int slot, id;
                                 if (leaf_hit(e, o, d, t, slot, id)) keep(h, hit, t, slot, id);
                                 return false;
                             },
                             [&]() { return h.dist * 1.00001f; }, &cnt);
            return hit;
        }
        for (int i = 0; i < n_sph; i++) {
            Cand<float> c;
            if (sphere_intersect<S>(sph[i], o, d, c, st)) keep(h, hit, c.key, i, sph_id[i]);
        }
        const R4<float>* g = tri_g;
        for (int j = 0; j < n_tri; j++, g += 4) {
            float t;
            if (tri_hit(g, o, d, t)) keep(h, hit, t, n_sph + j, as_int(g[3].z));
        }
        for (int k = 0; k < n_poly; k++) {
            const int i = poly_slot[k];
            Cand<float> c;
            if (plane_intersect<S>(pln_n[i], pln_c[i], pln_v[i], vert, o, d, c, st))
                keep(h, hit, c.key, n_sph + n_tri + i, pln_id[i]);
        }
        return hit;
    }

    // One leaf entry of the hierarchy against a general ray: the routine the brute-force loops run for that kind of
    // primitive, and the slot / id they would report.
    RM_HD bool leaf_hit(const int e, const Vec3<float> o, const Vec3<float> d, float& t, int& slot, int& id) const {
        const unsigned kind = (unsigned)e >> 30;
        const int i = e & 0x3fffffff;
        Counters<false> st;
        Cand<float> c;
        if constexpr (kCount) (kind == BVH_SPHERE ? cnt.sph : cnt.pln)++;
        if (kind == BVH_TRI) {
            const R4<float>* g = tri_g + 4 * (size_t)i;
            if (!tri_hit(g, o, d, t)) return false;
            slot = n_sph + i;
            id = as_int(g[3].z);
            return true;
        }
        if (kind == BVH_SPHERE) {
            if (!sphere_intersect<false>(sph[i], o, d, c, st)) return false;
            slot = i;
            id = sph_id[i];
        } else {
            if (!plane_intersect<false>(pln_n[i], pln_c[i], pln_v[i], vert, o, d, c, st)) return false;
            slot = n_sph + n_tri + i;
            id = pln_id[i];
        }
        t = c.key;
        return true;
    }
    RM_HD bool anyhit_bvh(const Vec3<float> o, const Vec3<float> d) const {
        n_queries++;
        return bvh_walk<kCount>(bvh, o, d,
                                [&](const int e) {
                                    float t;
                                    int slot, id;
                                    return leaf_hit(e, o, d, t, slot, id);
                                },
                                []() { return INFINITY; }, &cnt);
    }

    template <bool S> RM_HD bool anyhit(const Vec3<float> o, const Vec3<float> d, Counters<S>& st) const {
        if constexpr (kBvh) return anyhit_bvh(o, d);
        Cand<float> c;
        for (int i = 0; i < n_sph; i++)
            if (sphere_intersect<S>(sph[i], o, d, c, st)) return true;
        float t;
        const R4<float>* g = tri_g;
        int j = 0;
        // four triangles per round: the four record loads and the eight independent FFMA chains of stage 1 are in
        // flight together (a single triangle per iteration leaves the warp waiting on each shared-memory load)
        for (; j + 4 <= n_tri; j += 4, g += 16) {
            float dp0, dp1, dp2, dp3, nm0, nm1, nm2, nm3;
            const R4<float> a0 = g[0], a1 = g[4], a2 = g[8], a3 = g[12];
            const bool f0 = tri_front(a0, o, d, dp0, nm0), f1 = tri_front(a1, o, d, dp1, nm1);
            const bool f2 = tri_front(a2, o, d, dp2, nm2), f3 = tri_front(a3, o, d, dp3, nm3);
            if (f0 | f1 | f2 | f3) {
                if (f0 && tri_inside(g, o, d, dp0, nm0, t)) return true;
                if (f1 && tri_inside(g + 4, o, d, dp1, nm1, t)) return true;
                if (f2 && tri_inside(g + 8, o, d, dp2, nm2, t)) return true;
                if (f3 && tri_inside(g + 12, o, d, dp3, nm3, t)) return true;
            }
        }
        for (; j < n_tri; j++, g += 4)
            if (tri_hit(g, o, d, t)) return true;
        for (int k = 0; k < n_poly; k++) {
            const int i = poly_slot[k];
            if (plane_intersect<S>(pln_n[i], pln_c[i], pln_v[i], vert, o, d, c, st)) return true;
        }
        return false;
    }

    // Branch-free tri_inside: the predicate of stage 2 as a value, for the paired shadow rays below (a garbage quotient
    // of a near-parallel ray is masked by the |d.n| test; NaNs compare false).
    static RM_HD bool tri_inside_pred(const R4<float> b, const R4<float> c, const R4<float> l, const Vec3<float> o,
                                      const Vec3<float> d, const float dp, const float num) {
        const float t = fast_div(num, dp);                     // triangle.rs:62
        const float qx = fmaf(t, d.x, o.x - b.x), qy = fmaf(t, d.y, o.y - b.y);
        const float e0 = fmaf(b.z, qx, b.w * qy);
        const float e1 = fmaf(c.x, qx, fmaf(c.y, qy, c.z));
        const float e2 = fmaf(c.w, qx, l.x * qy);
        return (fabsf(dp) > l.y) & (fminf(fminf(e0, e1), e2) > 0.f);   // triangle.rs:57, 72-76
    }

    // The shadow rays of TWO lights from one surface point together (renderer.rs:174-177, twice): every triangle record is
    // loaded once and tested against both rays, which puts two independent dependency chains per lane in flight -- the
    // shading stage is bound by instruction latency, not by issue slots.  The same arithmetic per (ray, triangle) as
    // anyhit(), so the same decisions.  `need`: bit 0 / bit 1 = ray A / B exists; returns the rays that are blocked.
    RM_HD unsigned anyhit2(const Vec3<float> oA, const Vec3<float> dA, const Vec3<float> oB, const Vec3<float> dB,
                           unsigned need) const {
        unsigned blocked = 0;
        if constexpr (kBvh) {                                   // any-hit is a boolean per ray: one walk each
            if ((need & 1u) && anyhit_bvh(oA, dA)) blocked |= 1u;
            if ((need & 2u) && anyhit_bvh(oB, dB)) blocked |= 2u;
            return blocked;
        }
        if (n_sph + n_poly > 0) {                               // spheres and n-gons: ray by ray (any-hit: the order of the
            Counters<false> st;                                 // primitives does not matter for the boolean)
            Cand<float> c;
            for (int r = 0; r < 2; r++) {
                if (!(need >> r & 1)) continue;
                const Vec3<float> o = r ? oB : oA, d = r ? dB : dA;
                bool hit = false;
                for (int i = 0; i < n_sph && !hit; i++) hit = sphere_intersect<false>(sph[i], o, d, c, st);
                for (int k = 0; k < n_poly && !hit; k++) {
                    const int i = poly_slot[k];
                    hit = plane_intersect<false>(pln_n[i], pln_c[i], pln_v[i], vert, o, d, c, st);
                }
                if (hit) blocked |= 1u << r;
            }
            need &= ~blocked;
        }
        const R4<float>* g = tri_g;
        int j = 0;
        for (; j + 2 <= n_tri && need; j += 2, g += 8) {
            const R4<float> a0 = g[0], a1 = g[4];
            float dpA0, nmA0, dpB0, nmB0, dpA1, nmA1, dpB1, nmB1;
            const bool fA0 = tri_front(a0, oA, dA, dpA0, nmA0), fB0 = tri_front(a0, oB, dB, dpB0, nmB0);
            const bool fA1 = tri_front(a1, oA, dA, dpA1, nmA1), fB1 = tri_front(a1, oB, dB, dpB1, nmB1);
            const unsigned f0 = ((unsigned)fA0 | (unsigned)fB0 << 1) & need, f1 = ((unsigned)fA1 | (unsigned)fB1 << 1) & need;
            if (f0 | f1) {
                if (f0) {
                    const R4<float> b = g[1], c = g[2], l = g[3];
                    const unsigned in = (unsigned)tri_inside_pred(b, c, l, oA, dA, dpA0, nmA0) |
                                        (unsigned)tri_inside_pred(b, c, l, oB, dB, dpB0, nmB0) << 1;
                    blocked |= in & f0;
                }
                if (f1) {
                    const R4<float> b = g[5], c = g[6], l = g[7];
                    const unsigned in = (unsigned)tri_inside_pred(b, c, l, oA, dA, dpA1, nmA1) |
                                        (unsigned)tri_inside_pred(b, c, l, oB, dB, dpB1, nmB1) << 1;
                    blocked |= in & f1;
                }
                need &= ~blocked;
            }
        }
        if (j < n_tri && need) {
            const R4<float> a0 = g[0];
            float dpA, nmA, dpB, nmB;
            const bool fA = tri_front(a0, oA, dA, dpA, nmA), fB = tri_front(a0, oB, dB, dpB, nmB);
            const unsigned f0 = ((unsigned)fA | (unsigned)fB << 1) & need;
            if (f0) {
                const R4<float> b = g[1], c = g[2], l = g[3];
                const unsigned in = (unsigned)tri_inside_pred(b, c, l, oA, dA, dpA, nmA) |
                                    (unsigned)tri_inside_pred(b, c, l, oB, dB, dpB, nmB) << 1;
                blocked |= in & f0;
            }
        }
        return blocked;
    }

    // renderer.rs:138-193 for the production path: lights taken two at a time (anyhit2), contributions added in the
    // reference's order (light l before light l + 1).
    template <bool S> RM_HD Vec3<float> direct(const Vec3<float> /*origin*/, const Vec3<float> dir, const Vec3<float> point,
                                               const Vec3<float> normal, const R4<float> ma, const R4<float> mb, Counters<S>&) const {
        Vec3<float> acc = {0.f, 0.f, 0.f};
        // renderer.rs:149 normalises origin - point; the point lies on the ray, origin - point = -t * dir with t > 0 and dir
        // a unit vector, so the view vector IS -dir -- exactly, whereas the subtraction of two far-away points in FP32 only
        // approximates it (|origin| 2^-24 against a short t)
        const Vec3<float> to_viewer = -dir;
        const Vec3<float> kd = {ma.x, ma.y, ma.z};
        auto pair = [&](const int l0) {
            const bool two = l0 + 1 < n_lgt;
            const R4<float> lpA = lgt_p[l0], lpB = lgt_p[two ? l0 + 1 : l0];
            const Vec3<float> ldA = normalized(Vec3<float>{lpA.x - point.x, lpA.y - point.y, lpA.z - point.z});   // renderer.rs:166
            const Vec3<float> ldB = normalized(Vec3<float>{lpB.x - point.x, lpB.y - point.y, lpB.z - point.z});
            const float sideA = dot(ldA, normal), sideB = dot(ldB, normal);
            const float offA = sideA < 0.f ? -1e-3f : 1e-3f, offB = sideB < 0.f ? -1e-3f : 1e-3f;    // renderer.rs:168-172
            const Vec3<float> soA = axpy(point, normal, offA), soB = axpy(point, normal, offB);
            const unsigned blocked = anyhit2(soA, ldA, soB, ldB, two ? 3u : 1u);                     // renderer.rs:174-177
#pragma unroll
            for (int r = 0; r < 2; r++) {
                if ((r && !two) || (blocked >> r & 1)) continue;
                const R4<float> lp = r ? lpB : lpA;
                const Vec3<float> ld = r ? ldB : ldA;
                const float side = r ? sideB : sideA;
                const Vec3<float> lc = xyz(lgt_c[l0 + r]);
                acc = acc + scaled(scaled(lc * kd, fmaxf(side, 0.f)), lp.w);                          // renderer.rs:138-140, 181-183
                const Vec3<float> reflected = reflect(-ld, normal);                                   // renderer.rs:144-145
                const float sf = fmaxf(dot(reflected, to_viewer), 0.f);                               // renderer.rs:150
                acc = acc + scaled(lc, pow_nonneg(sf * mb.x, mb.y));                                  // renderer.rs:186-189
            }
        };
        if constexpr (kBvh) {
            // No rolled loop around the walks (see primary_bvh for what a shared trip counter did on the B200): the lights
            // as unrolled, guarded pairs.  Scenes with more than kBvhMaxLights lights stay on the brute-force kernel.
#pragma unroll
            for (int k = 0; k < kBvhMaxLights / 2; k++)
                if (2 * k < n_lgt) pair(2 * k);
        } else {
            for (int l0 = 0; l0 < n_lgt; l0 += 2) pair(l0);
        }
        return scaled(acc, ma.w);                                                                     // renderer.rs:192
    }

    RM_HD void surface(HitRec<float>& h, const Vec3<float> o, const Vec3<float> d, Vec3<float>& normal) const {
        if (h.slot < n_sph) {
            sphere_point_normal(sph[h.slot], o, d, h.p, h.p, normal);
        } else {
            h.p = axpy(o, d, h.dist);
            normal = (h.slot < n_sph + n_tri) ? xyz(tri_g[4 * (h.slot - n_sph)]) : xyz(pln_n[h.slot - n_sph - n_tri]);
        }
    }
};
using FastView = FastViewT<false>;

// ---- primary visibility (stage A of the render kernel) ------------------------------------------
// kPx horizontally adjacent pixels of one thread (the CUDA kernel uses 4; they share Y, so each affine
// function of a triangle costs one FFMA for the row part plus one FFMA per pixel, and the four 128-bit
// record loads are amortised over kPx pixels; the independent chains give the FP32 pipe its ILP).
// best_*: ray parameter, slot and primitive id of the closest hit so far (slot < 0: none).
template <int kPx> struct PrimaryState {
    float X[kPx], Y;
    float len2[kPx];    // |D|^2 of the un-normalised pixel direction D = (X, Y, -1)
    float t[kPx];       // triangles: ray parameter in units of |D| (the same for all candidates of a pixel); primary_rest
                        // and the shading stage rescale to the unit direction
    int slot[kPx], id[kPx];
};

RM_HD float pixel_X(const FrameParams<float>& fp, int x) { return (float(x) - fp.half_w) * fp.sx; }
RM_HD float pixel_Y(const FrameParams<float>& fp, int y) { return (float(y) - fp.half_h) * fp.sy; }

template <int kPx> RM_HD void primary_begin(PrimaryState<kPx>& ps, const FrameParams<float>& fp, const int x0, const int y) {
    ps.Y = pixel_Y(fp, y);
    RM_PIN(ps.Y);   // keep the pixel coordinates in registers: ptxas otherwise rematerialises them (int->float,
                    // sub, mul per pixel) inside the triangle loop when registers are tight
#pragma unroll
    for (int k = 0; k < kPx; k++) {
        ps.X[k] = pixel_X(fp, x0 + k);
        RM_PIN(ps.X[k]);
        ps.len2[k] = fmaf(ps.X[k], ps.X[k], fmaf(ps.Y, ps.Y, 1.f));
        ps.slot[k] = -1;
        ps.id[k] = -1;
        ps.t[k] = 0.f;
    }
}

// Exact rectangle bound of a raster record.  Each of the four functions f(X, Y) = fmaf(r.x, X, fmaf(r.y, Y, r.z))
// -- evaluated with the very operations primary_tri uses per pixel -- is monotone in X and in Y because fmaf is
// correctly rounded, so its maximum over the pixels of a rectangle [Xa, Xb] x [Ya, Yb] is attained at a corner,
// bit for bit.  A triangle can only be hit inside the rectangle if all four maxima are positive; dropping the
// others changes no pixel.  (pixel_X / pixel_Y are monotone in the pixel index for the same reason.)
RM_HD float rect_max(const R4<float> r, const float Xa, const float Xb, const float Ya, const float Yb) {
    const float ba = fmaf(r.y, Ya, r.z), bb = fmaf(r.y, Yb, r.z);
    return fmaxf(fmaxf(fmaf(r.x, Xa, ba), fmaf(r.x, Xb, ba)), fmaxf(fmaf(r.x, Xa, bb), fmaf(r.x, Xb, bb)));
}
RM_HD float rect_min(const R4<float> r, const float Xa, const float Xb, const float Ya, const float Yb) {
    const float ba = fmaf(r.y, Ya, r.z), bb = fmaf(r.y, Yb, r.z);
    return fminf(fminf(fmaf(r.x, Xa, ba), fmaf(r.x, Xb, ba)), fminf(fmaf(r.x, Xa, bb), fmaf(r.x, Xb, bb)));
}
// All four functions positive at all four corners: every pixel of the rectangle lies inside the triangle (used only as
// a cost estimate by the tile schedule -- such a tile is all hits -- never for a visibility decision).
RM_HD bool tri_covers(const R4<float> r0, const R4<float> r1, const R4<float> r2, const R4<float> r3, const float Xa,
                      const float Xb, const float Ya, const float Yb) {
    return fminf(fminf(rect_min(r0, Xa, Xb, Ya, Yb), rect_min(r1, Xa, Xb, Ya, Yb)),
                 fminf(rect_min(r2, Xa, Xb, Ya, Yb), rect_min(r3, Xa, Xb, Ya, Yb))) > 0.f;
}
RM_HD bool tri_may_touch(const R4<float> r0, const R4<float> r1, const R4<float> r2, const R4<float> r3, const float Xa,
                         const float Xb, const float Ya, const float Yb) {
    return fminf(fminf(rect_max(r0, Xa, Xb, Ya, Yb), rect_max(r1, Xa, Xb, Ya, Yb)),
                 fminf(rect_max(r2, Xa, Xb, Ya, Yb), rect_max(r3, Xa, Xb, Ya, Yb))) > 0.f;
}

// One triangle (raster records r0..r3, slot) against the kPx pixels: no normalisation, no division unless a
// pixel is inside the triangle.  The pixels' predicates are folded into one branch so the common (all miss)
// case is straight-line code.
template <int kPx>
RM_HD void primary_tri(PrimaryState<kPx>& ps, const R4<float> r0, const R4<float> r1, const R4<float> r2, const R4<float> r3,
                       const int slot) {
    const float Y = ps.Y;
    const float bd = fmaf(r0.y, Y, r0.z), b0 = fmaf(r1.y, Y, r1.z), b1 = fmaf(r2.y, Y, r2.z), b2 = fmaf(r3.y, Y, r3.z);
    float mk[kPx], dpD[kPx];
    float any = 0.f;
#pragma unroll
    for (int k = 0; k < kPx; k++) {
        dpD[k] = fmaf(r0.x, ps.X[k], bd);
        const float s0 = fmaf(r1.x, ps.X[k], b0), s1 = fmaf(r2.x, ps.X[k], b1), s2 = fmaf(r3.x, ps.X[k], b2);
        mk[k] = fminf(fminf(fminf(s0, s1), s2), dpD[k]);       // > 0 <=> inside all three edges and in front
        any = fmaxf(any, mk[k]);
    }
    if (any > 0.f) {
#pragma unroll
        for (int k = 0; k < kPx; k++) {
            if (mk[k] > 0.f) {
                // |d.n| > thr (triangle.rs:57) on the unit direction d = D/|D|: dpD > thr*|D|, squared (both sides >= 0)
                if (dpD[k] * dpD[k] > r1.w * ps.len2[k]) {
                    const float t = fast_div(r0.w, dpD[k]);      // triangle.rs:62 in units of |D|: t_unit = t * |D|
                    const int id = FastView::as_int(r2.w);
                    if (ps.slot[k] < 0 || t < ps.t[k] || (t == ps.t[k] && id < ps.id[k])) {
                        ps.t[k] = t;
                        ps.slot[k] = slot;
                        ps.id[k] = id;
                    }
                }
            }
        }
    }
}

// spheres / n-gons: the general routines from the camera, one pixel of the thread after the other; the pixel state
// rotates through index 0, so every array index is a compile-time constant.  The loop over the kPx pixels is FULLY
// UNROLLED: as a rolled loop (`#pragma unroll 1`) it had the shape that went wrong in primary_bvh on the B200 -- a trip
// counter ptxas keeps in a uniform register around per-lane divergent inner loops (here: the per-edge early exits of
// plane_intersect), see the note at primary_bvh.  Unrolled there is no counter to share.
// vw: the camera's orientation (ViewBasis under a view); the rays leave along the world direction vw.apply(D / |D|).
template <int kPx, class FV, class VW = NoView>
RM_HD void primary_rest(PrimaryState<kPx>& ps, const FV& fv, const FrameParams<float>& fp, const VW& vw = VW()) {
#pragma unroll
    for (int r = 0; r < kPx; r++) {
        const float inv = fast_rsqrt(ps.len2[0]);
        const Vec3<float> d = vw.apply(Vec3<float>{ps.X[0] * inv, ps.Y * inv, -inv});
        bool hit = ps.slot[0] >= 0;
        HitRec<float> best;
        best.dist = ps.t[0] * (ps.len2[0] * inv);              // to the unit direction
        best.slot = ps.slot[0];
        best.id = ps.id[0];
        Counters<false> st;
        for (int i = 0; i < fv.n_sph; i++) {
            Cand<float> c;
            if (sphere_intersect<false>(fv.sph[i], fp.camera, d, c, st)) FastView::keep(best, hit, c.key, i, fv.sph_id[i]);
        }
        for (int q = 0; q < fv.n_poly; q++) {
            const int i = fv.poly_slot[q];
            Cand<float> c;
            if (plane_intersect<false>(fv.pln_n[i], fv.pln_c[i], fv.pln_v[i], fv.vert, fp.camera, d, c, st))
                FastView::keep(best, hit, c.key, fv.n_sph + fv.n_tri + i, fv.pln_id[i]);
        }
        const float t_new = best.dist * inv;                   // back to units of |D|, like the triangle hits
        const int slot_new = hit ? best.slot : -1, id_new = hit ? best.id : -1;
        const float X0 = ps.X[0], L0 = ps.len2[0];
#pragma unroll
        for (int k = 0; k + 1 < kPx; k++) {                     // rotate left; the finished pixel goes to the end
            ps.X[k] = ps.X[k + 1];
            ps.len2[k] = ps.len2[k + 1];
            ps.t[k] = ps.t[k + 1];
            ps.slot[k] = ps.slot[k + 1];
            ps.id[k] = ps.id[k + 1];
        }
        ps.X[kPx - 1] = X0;
        ps.len2[kPx - 1] = L0;
        ps.t[kPx - 1] = t_new;
        ps.slot[kPx - 1] = slot_new;
        ps.id[kPx - 1] = id_new;
    }
}

// Primary visibility of a thread's kPx pixels through the hierarchy (RmParams.accel), one pixel at a time.  A
// triangle leaf runs primary_tri on the triangle's raster record, a sphere / n-gon leaf the general routine from the
// camera, and the two partial winners are merged the way primary_rest merges them -- the same arithmetic per (pixel,
// primitive) and the same (distance, id) order as the brute-force stage A, hence the same t / slot / id, bit for bit.
// (Under a view the walk follows the world direction, and the triangle leaves test the rotated raster records: |M D| = |D|,
// so their distances in units of |D| stay what they are.)
template <int kPx, bool kCount, class VW = NoView>
RM_HD void primary_bvh(PrimaryState<kPx>& ps, const FastViewT<true, kCount>& fv, const FrameParams<float>& fp, const VW& vw = VW()) {
    using FastViewBvh = FastViewT<true, kCount>;
    const bool rest = fv.n_sph + fv.n_poly > 0;
    // One walk per pixel, the loop over the thread's pixels fully unrolled.  As a rolled loop (`#pragma unroll 1`, like
    // primary_rest) it went wrong on the B200 for scenes with deep hierarchies: ptxas keeps the trip counter of such a
    // loop in a uniform register behind a uniform branch, the walks inside run a different number of steps in every
    // lane, and the frames showed lanes that had skipped an iteration (results shifted by one pixel, pixels left
    // unprocessed) and, once, a kernel that never left the loop.  Unrolled there is no counter to share; the rotation
    // of the pixel state becomes a compile-time renaming.
#pragma unroll
    for (int r = 0; r < kPx; r++) {
        PrimaryState<1> p1;
        p1.X[0] = ps.X[0];
        p1.Y = ps.Y;
        p1.len2[0] = ps.len2[0];
        p1.t[0] = 0.f;
        p1.slot[0] = -1;
        p1.id[0] = -1;
        const float inv = fast_rsqrt(p1.len2[0]);
        const float len = p1.len2[0] * inv;                    // |D|: stage A's triangle distances are in units of it
        const Vec3<float> d = vw.apply(Vec3<float>{p1.X[0] * inv, p1.Y * inv, -inv});
        HitRec<float> other;                                   // closest sphere / n-gon, unit-direction distance
        other.dist = INFINITY;
        other.slot = -1;
        other.id = -1;
        bool hit_other = false;
        float tcut = INFINITY;
        bvh_walk<kCount>(fv.bvh, fp.camera, d,
                 [&](const int e) {
                     const unsigned kind = (unsigned)e >> 30;
                     const int i = e & 0x3fffffff;
                     if (kind == BVH_TRI) {
                         if constexpr (kCount) fv.cnt.pln++;
                         const R4<float>* q = fv.tri_r + 4 * (size_t)i;
                         primary_tri<1>(p1, q[0], q[1], q[2], q[3], fv.n_sph + i);
                         if (p1.slot[0] >= 0) tcut = fminf(tcut, p1.t[0] * len);
                     } else {
                         float t;
                         int slot, id;
                         if (fv.leaf_hit(e, fp.camera, d, t, slot, id)) {
                             FastViewBvh::keep(other, hit_other, t, slot, id);
                             tcut = fminf(tcut, other.dist);
                         }
                     }
                     return false;
                 },
                 [&]() { return tcut * 1.00001f; }, &fv.cnt);
        float t_new = p1.t[0];
        int slot_new = p1.slot[0], id_new = p1.id[0];
        if (rest) {                                            // primary_rest's merge and its round trip through unit distances
            bool hit = p1.slot[0] >= 0;
            HitRec<float> best;
            best.dist = p1.t[0] * len;
            best.slot = p1.slot[0];
            best.id = p1.id[0];
            if (hit_other) FastViewBvh::keep(best, hit, other.dist, other.slot, other.id);
            t_new = best.dist * inv;
            slot_new = hit ? best.slot : -1;
            id_new = hit ? best.id : -1;
        }
        const float X0 = ps.X[0], L0 = ps.len2[0];
#pragma unroll
        for (int k = 0; k + 1 < kPx; k++) {                     // rotate left; the finished pixel goes to the end
            ps.X[k] = ps.X[k + 1];
            ps.len2[k] = ps.len2[k + 1];
            ps.t[k] = ps.t[k + 1];
            ps.slot[k] = ps.slot[k + 1];
            ps.id[k] = ps.id[k + 1];
        }
        ps.X[kPx - 1] = X0;
        ps.len2[kPx - 1] = L0;
        ps.t[kPx - 1] = t_new;
        ps.slot[kPx - 1] = slot_new;
        ps.id[kPx - 1] = id_new;
#if defined(__CUDA_ARCH__) && defined(RM_BVH_SYNC_EACH_PIXEL)
        __syncwarp();
#endif
    }
}

// ---- the shading stage (stage B of the render kernel) -------------------------------------------------------------------
// An OPAQUE primary hit spawns no ray (renderer.rs:277): its colour is background + direct lighting, pure FP32.
// A GLASS-LIKE primary hit starts the reflect / refract recursion (renderer.rs:254-309), traced by cast_glass<G> with the
// ray geometry in G = float or G = double:
//   * G = float: everything FP32 (scenes whose spheres are large against the scene's coordinates, planar glass).
//   * G = double: a curved glass surface magnifies a direction error by (distance to the next hit / radius), so positions
//     rounded to FP32 at scene scale (2^-24 * 128 against radii of ~1) grow to 1e-3 relative colour errors two bounces
//     later -- measured on BASELINE.json configs[4]'s scene: only 99.5 % of the pixels within the north star's 1e-4 with
//     FP32 geometry, 99.999 % with this.  What stays FP32 is everything that is a search or a smooth function: which
//     primitive a ray hits (the O(n) / O(log n) part), the shadow rays, the lighting arithmetic.  What is f64: the ray
//     (origin, direction), the hit point and normal of the ONE primitive each query picked (FastViewT::refine) and the
//     optics (optics.rs:8-89) -- a few dozen FP64 operations per segment next to hundreds of FP32 primitive tests.
//     Opaque hits take this route as well: near a silhouette the hit point of a far sphere moves by many ulps of the
//     FP32 centre per ulp of the ray, and a specular exponent of 100 turns that into 1e-4.
// Which of the two a frame gets is decided per launch from the scene and the camera (glass_mode below).
enum GlassMode { GLASS_NONE = 0, GLASS_F32 = 1, GLASS_F64 = 2 };

#if defined(RM_CHECKED) && defined(__CUDA_ARCH__)
#define RM_FAST_CHECK(cond) assert(cond)
#else
#define RM_FAST_CHECK(cond) ((void)0)
#endif

// f64 ray geometry when some sphere is small against the coordinates rays travel through: S > 64 r_min, with S the
// largest coordinate magnitude of the scene's primitives and the camera.  (FP32 positions carry 2^-24 S; against a
// radius of S / 64 that is a normal error of 4e-6, which the recursion's magnification keeps below the tolerance; the demo
// scene of the reference -- S = 50, radii 2 to 4 -- sits at 25 and meets the north-star criteria in FP32 on 99.99 % of its
// pixels, the stress scene -- S = 170, radii from 0.3 -- at 570 and does not.)
inline int glass_mode(const bool any_glass, const int n_sph, const double coord_max, const double r_min, const double camera[3]) {
    if (!any_glass && n_sph == 0) return GLASS_NONE;
    if (n_sph == 0) return GLASS_F32;
    const double S = fmax(fmax(coord_max, fabs(camera[0])), fmax(fabs(camera[1]), fabs(camera[2])));
    return S > 64. * r_min ? GLASS_F64 : GLASS_F32;
}

// (inlined: as a function of its own -- __noinline__, so that the caller's loop state is not held in registers across the
// f64 code -- the view and the frame parameters are passed through local memory and the call costs more than the spills
// it avoids: stress_8k through the hierarchy 18.3 ms against 15.6 ms inlined, profiles/r4h_glass64_inline_ab.txt)
#if defined(__CUDACC__) && !defined(RM_GLASS64_NOINLINE)
#define RM_GLASS_FN __host__ __device__ __forceinline__
#elif defined(__CUDACC__)
#define RM_GLASS_FN __host__ __device__ __noinline__
#else
#define RM_GLASS_FN inline
#endif

RM_HD Vec3<float> to_f32(const Vec3<double> v) { return {(float)v.x, (float)v.y, (float)v.z}; }
RM_HD Vec3<float> to_f32(const Vec3<float> v) { return v; }

// renderer.rs:254-309 from the primary hit of pixel (x, y); t1 = FP32 ray parameter of that hit (unit direction).
// Under a view the primary direction is the camera-space one taken to the world by vw: in f64 from the f64 basis (the
// normative definition of include/rm_b200.h), in FP32 from its FP32 rounding.
template <typename G, class FV, class VW = NoView>
RM_HD Vec3<float> cast_glass_impl(const FV& fv, const FrameParams<float>& fp, const int x, const int y, const float t1,
                                  const int slot1, const int id1, const VW& vw = VW()) {
    struct Frame {
        Vec3<float> c;
        Vec3<G> ro, rd;
        float k;
        int state;   // bit0: a refracted ray is pending, bit1: the refracted ray is the one in flight
    };
    Frame fr[kMaxDepth];
    int sp = 0;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    Vec3<G> o, d;
    if constexpr (sizeof(G) == 8) {                             // renderer.rs:128-135 in the reference's own arithmetic
        o = {fp.cam64[0], fp.cam64[1], fp.cam64[2]};
        d = vw.apply(Fast64::normalized(Vec3<double>{2. * ((double)x * fp.inv_w64 - 0.5) * fp.hf64 * fp.ratio64,
                                                     -2. * ((double)y * fp.inv_h64 - 0.5) * fp.hf64, -1.}));
    } else {
        const float X = pixel_X(fp, x), Y = pixel_Y(fp, y);
        const float inv = fast_rsqrt(fmaf(X, X, fmaf(Y, Y, 1.f)));     // geometry.rs:104-109: scale(1/norm)
        o = fp.camera;
        d = vw.apply(Vec3<float>{X * inv, Y * inv, -inv});
    }
    Counters<false> st;
    Vec3<float> v;
    for (;;) {
        const int level = sp + 1;                               // n_recursion
        if (level > fp.max_depth) {
            v = bg;                                             // renderer.rs:262-264
        } else {
            const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
            HitRec<float> h;
            bool got = true;
            if (level == 1) {
                h.dist = t1;
                h.slot = slot1;
                h.id = id1;
            } else {
                got = fv.template closest<false>(o32, d32, level, h, st);      // renderer.rs:266: the search, FP32
            }
            if (!got) {
                v = bg;                                         // renderer.rs:300-306 (level > 1 here)
            } else {
                Vec3<G> p, n;
                Vec3<float> p32, n32;
                if constexpr (sizeof(G) == 8) {
                    fv.refine(h.slot, o, d, (double)h.dist, p, n);
                    p32 = to_f32(p);
                    n32 = to_f32(n);
                } else {
                    fv.surface(h, o32, d32, n32);
                    p32 = h.p;
                    p = p32;
                    n = n32;
                }
                const R4<float> ma = fv.mat_a[h.id];
                const R4<float> mb = fv.mat_b[h.id];
                Vec3<float> c = bg + fv.template direct<false>(o32, d32, p32, n32, ma, mb, st);   // renderer.rs:272-275
                bool pushed = false;
                if (fv.mat_f[h.id] & 1) {                       // renderer.rs:277
                    Vec3<G> ro1, rd1, ro2, rd2;
                    using N = typename std::conditional<sizeof(G) == 8, Fast64, Exact<float>>::type;
                    const bool has_refl = reflect_ray<G, N>(d, p, n, (G)mb.w, ro1, rd1);  // renderer.rs:203-207
                    const bool has_refr = refract_ray<G, N>(d, p, n, (G)mb.w, ro2, rd2);  // renderer.rs:235-239
                    if (has_refl || has_refr) {
                        RM_FAST_CHECK(sp < kMaxDepth);
                        Frame& f = fr[sp];
                        f.c = c;
                        f.k = mb.z;
                        if (has_refl) {
                            f.state = has_refr ? 1 : 0;
                            f.ro = ro2;
                            f.rd = rd2;
                            o = ro1;
                            d = rd1;
                        } else {
                            f.state = 2;
                            o = ro2;
                            d = rd2;
                        }
                        sp++;
                        pushed = true;
                    }
                }
                if (pushed) continue;
                v = c;
            }
        }
        for (;;) {                                              // return v to the callers on the stack
            if (sp == 0) return v;
            Frame& f = fr[sp - 1];
            if (f.state & 2) {
                f.c = f.c + scaled(v, 1.f - f.k);               // renderer.rs:249
                v = f.c;
                sp--;
            } else {
                f.c = f.c + scaled(v, f.k);                     // renderer.rs:219
                if (f.state & 1) {
                    o = f.ro;
                    d = f.rd;
                    f.state = 2;
                    break;
                }
                v = f.c;
                sp--;
            }
        }
    }
}
// renderer.rs:254-309 from a given ray (o, d) whose level-1 hit an FP32 query found: t1 (unit direction), slot1, id1 -- the
// thin-lens camera's sample rays (lens_shade below).  The loop is cast_glass_impl's, kept as a copy of its own: sharing it
// through one more inlined call changes the machine code of a pre-existing kernel instantiation.
template <typename G, class FV>
RM_HD Vec3<float> cast_glass_from(const FV& fv, const FrameParams<float>& fp, Vec3<G> o, Vec3<G> d, const float t1, const int slot1,
                                  const int id1) {
    struct Frame {
        Vec3<float> c;
        Vec3<G> ro, rd;
        float k;
        int state;   // bit0: a refracted ray is pending, bit1: the refracted ray is the one in flight
    };
    Frame fr[kMaxDepth];
    int sp = 0;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    Counters<false> st;
    Vec3<float> v;
    for (;;) {
        const int level = sp + 1;                               // n_recursion
        if (level > fp.max_depth) {
            v = bg;                                             // renderer.rs:262-264
        } else {
            const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
            HitRec<float> h;
            bool got = true;
            if (level == 1) {
                h.dist = t1;
                h.slot = slot1;
                h.id = id1;
            } else {
                got = fv.template closest<false>(o32, d32, level, h, st);      // renderer.rs:266: the search, FP32
            }
            if (!got) {
                v = bg;                                         // renderer.rs:300-306 (level > 1 here)
            } else {
                Vec3<G> p, n;
                Vec3<float> p32, n32;
                if constexpr (sizeof(G) == 8) {
                    fv.refine(h.slot, o, d, (double)h.dist, p, n);
                    p32 = to_f32(p);
                    n32 = to_f32(n);
                } else {
                    fv.surface(h, o32, d32, n32);
                    p32 = h.p;
                    p = p32;
                    n = n32;
                }
                const R4<float> ma = fv.mat_a[h.id];
                const R4<float> mb = fv.mat_b[h.id];
                Vec3<float> c = bg + fv.template direct<false>(o32, d32, p32, n32, ma, mb, st);   // renderer.rs:272-275
                bool pushed = false;
                if (fv.mat_f[h.id] & 1) {                       // renderer.rs:277
                    Vec3<G> ro1, rd1, ro2, rd2;
                    using N = typename std::conditional<sizeof(G) == 8, Fast64, Exact<float>>::type;
                    const bool has_refl = reflect_ray<G, N>(d, p, n, (G)mb.w, ro1, rd1);  // renderer.rs:203-207
                    const bool has_refr = refract_ray<G, N>(d, p, n, (G)mb.w, ro2, rd2);  // renderer.rs:235-239
                    if (has_refl || has_refr) {
                        RM_FAST_CHECK(sp < kMaxDepth);
                        Frame& f = fr[sp];
                        f.c = c;
                        f.k = mb.z;
                        if (has_refl) {
                            f.state = has_refr ? 1 : 0;
                            f.ro = ro2;
                            f.rd = rd2;
                            o = ro1;
                            d = rd1;
                        } else {
                            f.state = 2;
                            o = ro2;
                            d = rd2;
                        }
                        sp++;
                        pushed = true;
                    }
                }
                if (pushed) continue;
                v = c;
            }
        }
        for (;;) {                                              // return v to the callers on the stack
            if (sp == 0) return v;
            Frame& f = fr[sp - 1];
            if (f.state & 2) {
                f.c = f.c + scaled(v, 1.f - f.k);               // renderer.rs:249
                v = f.c;
                sp--;
            } else {
                f.c = f.c + scaled(v, f.k);                     // renderer.rs:219
                if (f.state & 1) {
                    o = f.ro;
                    d = f.rd;
                    f.state = 2;
                    break;
                }
                v = f.c;
                sp--;
            }
        }
    }
}
template <class FV, class VW = NoView>
RM_GLASS_FN Vec3<float> cast_glass64(const FV& fv, const FrameParams<float>& fp, const int x, const int y, const float t1,
                                     const int slot1, const int id1, const VW& vw = VW()) {
    return cast_glass_impl<double, FV, VW>(fv, fp, x, y, t1, slot1, id1, vw);
}

// One pixel whose primary ray hit (t in units of |D|, slot, id): renderer.rs:254-309 from level 1.
// kGlass = GLASS_NONE: the scene has neither glass-like materials nor spheres (every OBJ scene of the reference: obj.rs:125-138
// loads meshes opaque) -- the kernel instantiated for it carries no recursion, no f64 code and fewer registers.
template <int kGlass = GLASS_F64, class FV, class VW = NoView>
RM_HD Vec3<float> fast_shade(FV& fv, const FrameParams<float>& fp, const int x, const int y, const float t, const int slot,
                             const int id, const VW& vw = VW()) {
    const float X = pixel_X(fp, x), Y = pixel_Y(fp, y);
    const float len2 = fmaf(X, X, fmaf(Y, Y, 1.f));
    const float inv = fast_rsqrt(len2);                            // geometry.rs:104-109: scale(1/norm)
    const float dist = t * (len2 * inv);                           // stage A reports t in units of |D|
    // In the glass modes EVERY hit takes the recursion's routine (an opaque hit leaves it after its direct lighting): a
    // warp's 32 queue entries mix glass-like and opaque hits, and two routines would run the expensive part of both --
    // the shadow rays of direct() -- one after the other for the two groups of lanes (measured on the demo frame: 170
    // instead of 156 us).
    if constexpr (kGlass == GLASS_F64) return cast_glass64(fv, fp, x, y, dist, slot, id, vw);
    if constexpr (kGlass == GLASS_F32) return cast_glass_impl<float, FV, VW>(fv, fp, x, y, dist, slot, id, vw);
    const Vec3<float> d = vw.apply(Vec3<float>{X * inv, Y * inv, -inv});
    HitRec<float> h;
    h.dist = dist;
    h.slot = slot;
    h.id = id;
    Vec3<float> normal;
    fv.surface(h, fp.camera, d, normal);
    Counters<false> st;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    return bg + fv.template direct<false>(fp.camera, d, h.p, normal, fv.mat_a[id], fv.mat_b[id], st);   // renderer.rs:272-275
}

// A sample ray (o, d) of the thin-lens camera (rm_render_lens) whose level-1 closest-hit query found h (FP32, on the ray
// rounded to FP32): renderer.rs:254-309 from there.  kGlass as for fast_shade: the recursion with the f64 ray (GLASS_F64)
// or its FP32 rounding (GLASS_F32), or the direct lighting alone (GLASS_NONE).
template <int kGlass, class FV>
RM_HD Vec3<float> lens_shade(const FV& fv, const FrameParams<float>& fp, const Vec3<double> o, const Vec3<double> d, HitRec<float> h) {
    if constexpr (kGlass == GLASS_F64) return cast_glass_from<double>(fv, fp, o, d, h.dist, h.slot, h.id);
    const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
    if constexpr (kGlass == GLASS_F32) return cast_glass_from<float>(fv, fp, o32, d32, h.dist, h.slot, h.id);
    Vec3<float> normal;
    fv.surface(h, o32, d32, normal);
    Counters<false> st;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    return bg + fv.template direct<false>(o32, d32, h.p, normal, fv.mat_a[h.id], fv.mat_b[h.id], st);   // renderer.rs:272-275
}

// ---- rough glass (rm_render_rough_glass, include/rm_b200.h RmRoughGlass) --------------------------------------------------
// cast_glass_from for sample (i, j) of the thin-lens camera with the call's roughness rg: at a glass-like hit of level L
// whose primitive has g = rg.g[id] > 0, every ray the reference spawns is turned by rough_dir with the unit-disc point of
// stratum ((i + j + L) mod s, i) and leaves from the origin its producing function picks for the new direction.  Whether a
// ray exists and the weights k, 1 - k are the reference's, decided before the turn.  G = double: the turn in f64 from the f64
// ray (rough_dir<double>, the normative definition); G = float: its FP32 restatement.  Kept apart from cast_glass_from so
// that the lens kernel's machine code stays as it is.
template <typename G, class FV>
RM_HD Vec3<float> cast_glass_rough(const FV& fv, const FrameParams<float>& fp, const RoughGlass& rg, const int si, const int sj,
                                   Vec3<G> o, Vec3<G> d, const float t1, const int slot1, const int id1) {
    struct Frame {
        Vec3<float> c;
        Vec3<G> ro, rd;
        float k;
        int state;   // bit0: a refracted ray is pending, bit1: the refracted ray is the one in flight
    };
    Frame fr[kMaxDepth];
    int sp = 0;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    const int s = rg.samples;
    Counters<false> st;
    Vec3<float> v;
    for (;;) {
        const int level = sp + 1;                               // n_recursion
        if (level > fp.max_depth) {
            v = bg;                                             // renderer.rs:262-264
        } else {
            const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
            HitRec<float> h;
            bool got = true;
            if (level == 1) {
                h.dist = t1;
                h.slot = slot1;
                h.id = id1;
            } else {
                got = fv.template closest<false>(o32, d32, level, h, st);      // renderer.rs:266: the search, FP32
            }
            if (!got) {
                v = bg;                                         // renderer.rs:300-306 (level > 1 here)
            } else {
                Vec3<G> p, n;
                Vec3<float> p32, n32;
                if constexpr (sizeof(G) == 8) {
                    fv.refine(h.slot, o, d, (double)h.dist, p, n);
                    p32 = to_f32(p);
                    n32 = to_f32(n);
                } else {
                    fv.surface(h, o32, d32, n32);
                    p32 = h.p;
                    p = p32;
                    n = n32;
                }
                const R4<float> ma = fv.mat_a[h.id];
                const R4<float> mb = fv.mat_b[h.id];
                Vec3<float> c = bg + fv.template direct<false>(o32, d32, p32, n32, ma, mb, st);   // renderer.rs:272-275
                bool pushed = false;
                if (fv.mat_f[h.id] & 1) {                       // renderer.rs:277
                    Vec3<G> ro1, rd1, ro2, rd2;
                    using N = typename std::conditional<sizeof(G) == 8, Fast64, Exact<float>>::type;
                    const bool has_refl = reflect_ray<G, N>(d, p, n, (G)mb.w, ro1, rd1);  // renderer.rs:203-207
                    const bool has_refr = refract_ray<G, N>(d, p, n, (G)mb.w, ro2, rd2);  // renderer.rs:235-239
                    const float gf = rg.g[h.id];
                    if (gf > 0.f && (has_refl || has_refr)) {
                        const int k = ((sj + level) % s) * s + si;   // rough_offset(s, si, sj, level)
                        G lx, ly;
                        if constexpr (sizeof(G) == 8) {
                            lx = rg.off[2 * k];
                            ly = rg.off[2 * k + 1];
                        } else {
                            lx = rg.off32[2 * k];
                            ly = rg.off32[2 * k + 1];
                        }
                        if (lx != G(0) || ly != G(0)) {
                            if (has_refl) {
                                rd1 = rough_dir<G>(rd1, (G)gf, lx, ly);
                                ro1 = rough_reflect_origin<G>(p, n, rd1);
                            }
                            if (has_refr) {
                                rd2 = rough_dir<G>(rd2, (G)gf, lx, ly);
                                ro2 = rough_refract_origin<G>(p, n, d, rd2);
                            }
                        }
                    }
                    if (has_refl || has_refr) {
                        RM_FAST_CHECK(sp < kMaxDepth);
                        Frame& f = fr[sp];
                        f.c = c;
                        f.k = mb.z;
                        if (has_refl) {
                            f.state = has_refr ? 1 : 0;
                            f.ro = ro2;
                            f.rd = rd2;
                            o = ro1;
                            d = rd1;
                        } else {
                            f.state = 2;
                            o = ro2;
                            d = rd2;
                        }
                        sp++;
                        pushed = true;
                    }
                }
                if (pushed) continue;
                v = c;
            }
        }
        for (;;) {                                              // return v to the callers on the stack
            if (sp == 0) return v;
            Frame& f = fr[sp - 1];
            if (f.state & 2) {
                f.c = f.c + scaled(v, 1.f - f.k);               // renderer.rs:249
                v = f.c;
                sp--;
            } else {
                f.c = f.c + scaled(v, f.k);                     // renderer.rs:219
                if (f.state & 1) {
                    o = f.ro;
                    d = f.rd;
                    f.state = 2;
                    break;
                }
                v = f.c;
                sp--;
            }
        }
    }
}
// Sample (i, j) of a rough-glass frame whose level-1 query found h: lens_shade with cast_glass_rough.  Every rough scene
// has a glass-like primitive, so only the two glass modes exist.
template <int kGlass, class FV>
RM_HD Vec3<float> rough_shade(const FV& fv, const FrameParams<float>& fp, const RoughGlass& rg, const int i, const int j,
                              const Vec3<double> o, const Vec3<double> d, HitRec<float> h) {
    static_assert(kGlass == GLASS_F32 || kGlass == GLASS_F64, "rough glass is traced in a glass mode");
    if constexpr (kGlass == GLASS_F64) return cast_glass_rough<double>(fv, fp, rg, i, j, o, d, h.dist, h.slot, h.id);
    else return cast_glass_rough<float>(fv, fp, rg, i, j, to_f32(o), to_f32(d), h.dist, h.slot, h.id);
}

// ---- spherical area lights (rm_render_area_lights, include/rm_b200.h RmAreaLights) -----------------------------------------
template <class FV> struct WalksHierarchy;
template <bool kBvh, bool kCount> struct WalksHierarchy<FastViewT<kBvh, kCount>> { static constexpr bool value = kBvh; };

// The view the shading code (fast_shade, cast_glass_impl) sees on an area-light frame: closest-hit queries, surfaces and
// materials are the wrapped FastViewT's; direct() replaces every light of radius r > 0 by its s^2 sample points
// (light_frame / light_sample in FP32 from the FP32 shading point), each with the colour scaled by 1 / s^2.  FastViewT's
// own direct() is left as it is: the kernels that use it keep their machine code.
template <class FV> struct AreaView {
    const FV* fv;
    const AreaLights* al;
    const R4<float>* mat_a;
    const R4<float>* mat_b;
    const int* mat_f;

    RM_HD AreaView(const FV& v, const AreaLights& a) : fv(&v), al(&a), mat_a(v.mat_a), mat_b(v.mat_b), mat_f(v.mat_f) {}

    template <bool S> RM_HD bool closest(const Vec3<float> o, const Vec3<float> d, int level, HitRec<float>& h, Counters<S>& st) const {
        return fv->template closest<S>(o, d, level, h, st);
    }
    RM_HD unsigned anyhit2(const Vec3<float> oA, const Vec3<float> dA, const Vec3<float> oB, const Vec3<float> dB, unsigned need) const {
        return fv->anyhit2(oA, dA, oB, dB, need);
    }
    RM_HD void refine(const int slot, const Vec3<double> o, const Vec3<double> d, const double t32, Vec3<double>& p, Vec3<double>& n) const {
        fv->refine(slot, o, d, t32, p, n);
    }
    RM_HD void surface(HitRec<float>& h, const Vec3<float> o, const Vec3<float> d, Vec3<float>& normal) const { fv->surface(h, o, d, normal); }

    // renderer.rs:138-193 with area lights: lights in scene order; a light of radius 0 is the reference's point light (one
    // shadow ray), one of radius r > 0 is s^2 point lights q_ab (a outer, b inner) of colour k / s^2.  Every point light
    // contributes FastViewT::direct's term (the same arithmetic); its shadow rays go two at a time through anyhit2, and the
    // contributions are added in the normative order.
    template <bool S> RM_HD Vec3<float> direct(const Vec3<float> /*origin*/, const Vec3<float> dir, const Vec3<float> point,
                                               const Vec3<float> normal, const R4<float> ma, const R4<float> mb, Counters<S>&) const {
        Vec3<float> acc = {0.f, 0.f, 0.f};
        const Vec3<float> to_viewer = -dir;                       // (as FastViewT::direct)
        const Vec3<float> kd = {ma.x, ma.y, ma.z};
        const int ss = al->samples * al->samples;
        auto light = [&](const int l) {
            const R4<float> lp = fv->lgt_p[l];
            const Vec3<float> c = {lp.x, lp.y, lp.z};
            const float r = al->radius[l];
            const bool area = r > 0.f;
            Vec3<float> lc = xyz(fv->lgt_c[l]);
            Vec3<float> t1 = {0.f, 0.f, 0.f}, t2 = {0.f, 0.f, 0.f};
            if (area) {
                light_frame<float>(normalized(Vec3<float>{c.x - point.x, c.y - point.y, c.z - point.z}), t1, t2);
                lc = scaled(lc, al->inv_ss);
            }
            const int n = area ? ss : 1;
            auto at = [&](const int k) { return area ? light_sample<float>(c, r, t1, t2, al->off[2 * k], al->off[2 * k + 1]) : c; };
            for (int k = 0; k < n; k += 2) {
                const bool two = k + 1 < n;
                const Vec3<float> qA = at(k), qB = at(two ? k + 1 : k);
                const Vec3<float> ldA = normalized(Vec3<float>{qA.x - point.x, qA.y - point.y, qA.z - point.z});   // renderer.rs:166
                const Vec3<float> ldB = normalized(Vec3<float>{qB.x - point.x, qB.y - point.y, qB.z - point.z});
                const float sideA = dot(ldA, normal), sideB = dot(ldB, normal);
                const float offA = sideA < 0.f ? -1e-3f : 1e-3f, offB = sideB < 0.f ? -1e-3f : 1e-3f;    // renderer.rs:168-172
                const Vec3<float> soA = axpy(point, normal, offA), soB = axpy(point, normal, offB);
                const unsigned blocked = fv->anyhit2(soA, ldA, soB, ldB, two ? 3u : 1u);                 // renderer.rs:174-177
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    if ((e && !two) || (blocked >> e & 1)) continue;
                    const Vec3<float> ld = e ? ldB : ldA;
                    const float side = e ? sideB : sideA;
                    acc = acc + scaled(scaled(lc * kd, fmaxf(side, 0.f)), lp.w);                          // renderer.rs:138-140, 181-183
                    const Vec3<float> reflected = reflect(-ld, normal);                                   // renderer.rs:144-145
                    const float sf = fmaxf(dot(reflected, to_viewer), 0.f);                               // renderer.rs:150
                    acc = acc + scaled(lc, pow_nonneg(sf * mb.x, mb.y));                                  // renderer.rs:186-189
                }
            }
        };
        if constexpr (WalksHierarchy<FV>::value) {
            // as FastViewT::direct: the lights as unrolled, guarded calls (a scene with more than kBvhMaxLights lights stays
            // on brute force)
#pragma unroll
            for (int l = 0; l < kBvhMaxLights; l++)
                if (l < fv->n_lgt) light(l);
        } else {
            for (int l = 0; l < fv->n_lgt; l++) light(l);
        }
        return scaled(acc, ma.w);                                                                     // renderer.rs:192
    }
};

// ---- motion blur (rm_render_motion, include/rm_b200.h RmMotion) -------------------------------------------------------------
// Primitive k at time tau is its uploaded pose translated by tau v_k.  A ray (o, d) meets it at parameter t exactly where the
// ray (o - tau v_k, d) meets the unmoved primitive, so every per-primitive routine runs unchanged on the shifted origin.  A
// zero displacement leaves the origin's bits as they are (o - tau * 0 would turn a -0 into +0 for tau < 0).
template <typename R> RM_HD R motion_shift(const R o, const R tau, const float v) { return v != 0.f ? o - tau * (R)v : o; }
template <typename R> RM_HD Vec3<R> motion_shift(const Vec3<R> o, const R tau, const R4<float> v) {
    return {motion_shift<R>(o.x, tau, v.x), motion_shift<R>(o.y, tau, v.y), motion_shift<R>(o.z, tau, v.z)};
}
template <typename R> RM_HD Vec3<R> motion_unshift(const Vec3<R> p, const R tau, const R4<float> v) {
    return {v.x != 0.f ? p.x + tau * (R)v.x : p.x, v.y != 0.f ? p.y + tau * (R)v.y : p.y, v.z != 0.f ? p.z + tau * (R)v.z : p.z};
}

// The view the shading code (lens_shade, cast_glass_from) sees on a motion frame at one sample's time tau: the wrapped
// FastViewT's arrays, and every primitive tested with the ray origin shifted by its own displacement (FastViewT::tri_hit,
// sphere_intersect, plane_intersect and, through the swept hierarchy, FastViewT::leaf_hit, all unchanged).  Surfaces and the
// f64 refinement run FastViewT's own code on the shifted origin and shift the point back.  direct() is FastViewT::direct's
// arithmetic with the shadow rays traced at the same tau, light by light (the same decisions and the same sums as its pairs).
template <bool kBvh> struct MotionView {
    using FV = FastViewT<kBvh, false>;
    const FV* fv;
    const Motion* mo;
    float tau;
    double tau64;
    const R4<float>* mat_a;
    const R4<float>* mat_b;
    const int* mat_f;

    RM_HD MotionView(const FV& v, const Motion& m, const int q)
        : fv(&v), mo(&m), tau(m.tau32[q]), tau64(m.tau[q]), mat_a(v.mat_a), mat_b(v.mat_b), mat_f(v.mat_f) {}

    RM_HD R4<float> vel_of_slot(const int slot) const {
        if (slot < fv->n_sph) return mo->v_sph[slot];
        if (slot < fv->n_sph + fv->n_tri) return mo->v_tri[slot - fv->n_sph];
        return mo->v_pln[slot - fv->n_sph - fv->n_tri];
    }
    RM_HD R4<float> vel_of_entry(const int e) const {
        const unsigned kind = (unsigned)e >> 30;
        const int i = e & 0x3fffffff;
        return kind == BVH_SPHERE ? mo->v_sph[i] : kind == BVH_TRI ? mo->v_tri[i] : mo->v_pln[i];
    }

    template <bool S> RM_HD bool closest(const Vec3<float> o, const Vec3<float> d, int /*level*/, HitRec<float>& h, Counters<S>& st) const {
        bool hit = false;
        if constexpr (kBvh) {
            h.dist = INFINITY;
            bvh_walk<false>(fv->bvh, o, d,
                            [&](const int e) {
                                float t;
                                int slot, id;
                                if (fv->leaf_hit(e, motion_shift(o, tau, vel_of_entry(e)), d, t, slot, id)) FV::keep(h, hit, t, slot, id);
                                return false;
                            },
                            [&]() { return h.dist * 1.00001f; });
            return hit;
        }
        for (int i = 0; i < fv->n_sph; i++) {
            Cand<float> c;
            if (sphere_intersect<S>(fv->sph[i], motion_shift(o, tau, mo->v_sph[i]), d, c, st)) FV::keep(h, hit, c.key, i, fv->sph_id[i]);
        }
        const R4<float>* g = fv->tri_g;
        for (int j = 0; j < fv->n_tri; j++, g += 4) {
            float t;
            if (FV::tri_hit(g, motion_shift(o, tau, mo->v_tri[j]), d, t)) FV::keep(h, hit, t, fv->n_sph + j, FV::as_int(g[3].z));
        }
        for (int k = 0; k < fv->n_poly; k++) {
            const int i = fv->poly_slot[k];
            Cand<float> c;
            if (plane_intersect<S>(fv->pln_n[i], fv->pln_c[i], fv->pln_v[i], fv->vert, motion_shift(o, tau, mo->v_pln[i]), d, c, st))
                FV::keep(h, hit, c.key, fv->n_sph + fv->n_tri + i, fv->pln_id[i]);
        }
        return hit;
    }

    RM_HD bool anyhit(const Vec3<float> o, const Vec3<float> d) const {
        if constexpr (kBvh) {
            return bvh_walk<false>(fv->bvh, o, d,
                                   [&](const int e) {
                                       float t;
                                       int slot, id;
                                       return fv->leaf_hit(e, motion_shift(o, tau, vel_of_entry(e)), d, t, slot, id);
                                   },
                                   []() { return INFINITY; });
        }
        Counters<false> st;
        Cand<float> c;
        for (int i = 0; i < fv->n_sph; i++)
            if (sphere_intersect<false>(fv->sph[i], motion_shift(o, tau, mo->v_sph[i]), d, c, st)) return true;
        const R4<float>* g = fv->tri_g;
        for (int j = 0; j < fv->n_tri; j++, g += 4) {
            float t;
            if (FV::tri_hit(g, motion_shift(o, tau, mo->v_tri[j]), d, t)) return true;
        }
        for (int k = 0; k < fv->n_poly; k++) {
            const int i = fv->poly_slot[k];
            if (plane_intersect<false>(fv->pln_n[i], fv->pln_c[i], fv->pln_v[i], fv->vert, motion_shift(o, tau, mo->v_pln[i]), d, c, st))
                return true;
        }
        return false;
    }

    // renderer.rs:138-193: FastViewT::direct's terms, added in the same order
    template <bool S> RM_HD Vec3<float> direct(const Vec3<float> /*origin*/, const Vec3<float> dir, const Vec3<float> point,
                                               const Vec3<float> normal, const R4<float> ma, const R4<float> mb, Counters<S>&) const {
        Vec3<float> acc = {0.f, 0.f, 0.f};
        const Vec3<float> to_viewer = -dir;                       // (as FastViewT::direct)
        const Vec3<float> kd = {ma.x, ma.y, ma.z};
        auto light = [&](const int l) {
            const R4<float> lp = fv->lgt_p[l];
            const Vec3<float> ld = normalized(Vec3<float>{lp.x - point.x, lp.y - point.y, lp.z - point.z});   // renderer.rs:166
            const float side = dot(ld, normal);
            const float off = side < 0.f ? -1e-3f : 1e-3f;                                                 // renderer.rs:168-172
            if (anyhit(axpy(point, normal, off), ld)) return;                                             // renderer.rs:174-177
            const Vec3<float> lc = xyz(fv->lgt_c[l]);
            acc = acc + scaled(scaled(lc * kd, fmaxf(side, 0.f)), lp.w);                                  // renderer.rs:138-140, 181-183
            const Vec3<float> reflected = reflect(-ld, normal);                                           // renderer.rs:144-145
            const float sf = fmaxf(dot(reflected, to_viewer), 0.f);                                       // renderer.rs:150
            acc = acc + scaled(lc, pow_nonneg(sf * mb.x, mb.y));                                          // renderer.rs:186-189
        };
        if constexpr (kBvh) {
            // as FastViewT::direct: the lights as unrolled, guarded calls (a scene with more than kBvhMaxLights lights stays on
            // brute force)
#pragma unroll
            for (int l = 0; l < kBvhMaxLights; l++)
                if (l < fv->n_lgt) light(l);
        } else {
            for (int l = 0; l < fv->n_lgt; l++) light(l);
        }
        return scaled(acc, ma.w);                                                                     // renderer.rs:192
    }

    RM_HD void surface(HitRec<float>& h, const Vec3<float> o, const Vec3<float> d, Vec3<float>& normal) const {
        const R4<float> v = vel_of_slot(h.slot);
        fv->surface(h, motion_shift(o, tau, v), d, normal);
        h.p = motion_unshift(h.p, tau, v);
    }
    RM_HD void refine(const int slot, const Vec3<double> o, const Vec3<double> d, const double t32, Vec3<double>& p, Vec3<double>& n) const {
        const R4<float> v = vel_of_slot(slot);
        fv->refine(slot, motion_shift(o, tau64, v), d, t32, p, n);
        p = motion_unshift(p, tau64, v);
    }
};

// ---- distributed ray tracing (rm_render_distributed, include/rm_b200.h) ----------------------------------------------------
// The view the shading code (cast_glass_distributed, distributed_shade) sees for sample (i, j) of a distributed frame:
// closest-hit queries, surfaces and the f64 refinement are MotionView's at the sample's time when kMotion, and the wrapped
// FastViewT's otherwise (no per-primitive displacement loads).  direct() takes the recursion level L and replaces every light
// of radius r > 0 by ONE point light of its full colour, on the disc facing the shading point at the point of stratum
// area_offset(s, i, j, L); a light of radius 0 is the reference's point light.  The shadow rays go two at a time (anyhit2 of
// FastViewT, or two MotionView::anyhit at the sample's time), and the terms are FastViewT::direct's, added in its order.
template <bool kBvh, bool kMotion> struct DistributedView {
    using FV = FastViewT<kBvh, false>;
    const FV* fv;
    MotionView<kBvh> mv;
    const AreaPoints* ap;
    int si, sj;
    const R4<float>* mat_a;
    const R4<float>* mat_b;
    const int* mat_f;

    RM_HD DistributedView(const FV& v, const Motion& m, const AreaPoints& a, const int q)
        : fv(&v), mv(v, m, q), ap(&a), si(q / a.samples), sj(q % a.samples), mat_a(v.mat_a), mat_b(v.mat_b), mat_f(v.mat_f) {}

    template <bool S> RM_HD bool closest(const Vec3<float> o, const Vec3<float> d, int level, HitRec<float>& h, Counters<S>& st) const {
        if constexpr (kMotion) return mv.template closest<S>(o, d, level, h, st);
        else return fv->template closest<S>(o, d, level, h, st);
    }
    RM_HD unsigned anyhit2(const Vec3<float> oA, const Vec3<float> dA, const Vec3<float> oB, const Vec3<float> dB, unsigned need) const {
        if constexpr (kMotion) {
            unsigned blocked = 0;
            if ((need & 1u) && mv.anyhit(oA, dA)) blocked |= 1u;
            if ((need & 2u) && mv.anyhit(oB, dB)) blocked |= 2u;
            return blocked;
        } else {
            return fv->anyhit2(oA, dA, oB, dB, need);
        }
    }
    RM_HD void refine(const int slot, const Vec3<double> o, const Vec3<double> d, const double t32, Vec3<double>& p, Vec3<double>& n) const {
        if constexpr (kMotion) mv.refine(slot, o, d, t32, p, n);
        else fv->refine(slot, o, d, t32, p, n);
    }
    RM_HD void surface(HitRec<float>& h, const Vec3<float> o, const Vec3<float> d, Vec3<float>& normal) const {
        if constexpr (kMotion) mv.surface(h, o, d, normal);
        else fv->surface(h, o, d, normal);
    }

    // renderer.rs:138-193 at a shading point of level `level`, the lights in pairs as FastViewT::direct takes them
    template <bool S> RM_HD Vec3<float> direct(const int level, const Vec3<float> dir, const Vec3<float> point, const Vec3<float> normal,
                                               const R4<float> ma, const R4<float> mb, Counters<S>&) const {
        Vec3<float> acc = {0.f, 0.f, 0.f};
        const Vec3<float> to_viewer = -dir;                       // (as FastViewT::direct)
        const Vec3<float> kd = {ma.x, ma.y, ma.z};
        const int s = ap->samples;
        const int k = ((si + 2 * sj + level) % s) * s + (si + 3 * sj) % s;   // area_offset(s, i, j, level)
        const float lx = ap->off[2 * k], ly = ap->off[2 * k + 1];
        const int n_lgt = fv->n_lgt;
        auto at = [&](const int l) {                              // the light's point for this sample and level
            const R4<float> lp = fv->lgt_p[l];
            const Vec3<float> c = {lp.x, lp.y, lp.z};
            const float r = ap->radius[l];
            if (!(r > 0.f)) return c;
            Vec3<float> t1, t2;
            light_frame<float>(normalized(Vec3<float>{c.x - point.x, c.y - point.y, c.z - point.z}), t1, t2);
            return light_sample<float>(c, r, t1, t2, lx, ly);
        };
        auto pair = [&](const int l0) {
            const bool two = l0 + 1 < n_lgt;
            const Vec3<float> qA = at(l0), qB = at(two ? l0 + 1 : l0);
            const Vec3<float> ldA = normalized(Vec3<float>{qA.x - point.x, qA.y - point.y, qA.z - point.z});   // renderer.rs:166
            const Vec3<float> ldB = normalized(Vec3<float>{qB.x - point.x, qB.y - point.y, qB.z - point.z});
            const float sideA = dot(ldA, normal), sideB = dot(ldB, normal);
            const float offA = sideA < 0.f ? -1e-3f : 1e-3f, offB = sideB < 0.f ? -1e-3f : 1e-3f;    // renderer.rs:168-172
            const Vec3<float> soA = axpy(point, normal, offA), soB = axpy(point, normal, offB);
            const unsigned blocked = anyhit2(soA, ldA, soB, ldB, two ? 3u : 1u);                     // renderer.rs:174-177
#pragma unroll
            for (int r = 0; r < 2; r++) {
                if ((r && !two) || (blocked >> r & 1)) continue;
                const float w = fv->lgt_p[l0 + r].w;
                const Vec3<float> ld = r ? ldB : ldA;
                const float side = r ? sideB : sideA;
                const Vec3<float> lc = xyz(fv->lgt_c[l0 + r]);
                acc = acc + scaled(scaled(lc * kd, fmaxf(side, 0.f)), w);                             // renderer.rs:138-140, 181-183
                const Vec3<float> reflected = reflect(-ld, normal);                                   // renderer.rs:144-145
                const float sf = fmaxf(dot(reflected, to_viewer), 0.f);                               // renderer.rs:150
                acc = acc + scaled(lc, pow_nonneg(sf * mb.x, mb.y));                                  // renderer.rs:186-189
            }
        };
        if constexpr (kBvh) {
            // as FastViewT::direct: the lights as unrolled, guarded pairs (a scene with more than kBvhMaxLights lights stays on
            // brute force)
#pragma unroll
            for (int p = 0; p < kBvhMaxLights / 2; p++)
                if (2 * p < n_lgt) pair(2 * p);
        } else {
            for (int l0 = 0; l0 < n_lgt; l0 += 2) pair(l0);
        }
        return scaled(acc, ma.w);                                                                     // renderer.rs:192
    }
};

// cast_glass_rough for a DistributedView: the same recursion, the same turn of the rays a rough glass-like hit spawns (rg.g
// null: no primitive is rough), with the level passed to direct().  A copy of its own, so that the rough-glass kernel keeps its
// machine code.
template <typename G, class DV>
RM_HD Vec3<float> cast_glass_distributed(const DV& fv, const FrameParams<float>& fp, const RoughGlass& rg, Vec3<G> o, Vec3<G> d,
                                         const float t1, const int slot1, const int id1) {
    struct Frame {
        Vec3<float> c;
        Vec3<G> ro, rd;
        float k;
        int state;   // bit0: a refracted ray is pending, bit1: the refracted ray is the one in flight
    };
    Frame fr[kMaxDepth];
    int sp = 0;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    const int s = rg.samples, si = fv.si, sj = fv.sj;
    Counters<false> st;
    Vec3<float> v;
    for (;;) {
        const int level = sp + 1;                               // n_recursion
        if (level > fp.max_depth) {
            v = bg;                                             // renderer.rs:262-264
        } else {
            const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
            HitRec<float> h;
            bool got = true;
            if (level == 1) {
                h.dist = t1;
                h.slot = slot1;
                h.id = id1;
            } else {
                got = fv.template closest<false>(o32, d32, level, h, st);      // renderer.rs:266: the search, FP32
            }
            if (!got) {
                v = bg;                                         // renderer.rs:300-306 (level > 1 here)
            } else {
                Vec3<G> p, n;
                Vec3<float> p32, n32;
                if constexpr (sizeof(G) == 8) {
                    fv.refine(h.slot, o, d, (double)h.dist, p, n);
                    p32 = to_f32(p);
                    n32 = to_f32(n);
                } else {
                    fv.surface(h, o32, d32, n32);
                    p32 = h.p;
                    p = p32;
                    n = n32;
                }
                const R4<float> ma = fv.mat_a[h.id];
                const R4<float> mb = fv.mat_b[h.id];
                Vec3<float> c = bg + fv.template direct<false>(level, d32, p32, n32, ma, mb, st);   // renderer.rs:272-275
                bool pushed = false;
                if (fv.mat_f[h.id] & 1) {                       // renderer.rs:277
                    Vec3<G> ro1, rd1, ro2, rd2;
                    using N = typename std::conditional<sizeof(G) == 8, Fast64, Exact<float>>::type;
                    const bool has_refl = reflect_ray<G, N>(d, p, n, (G)mb.w, ro1, rd1);  // renderer.rs:203-207
                    const bool has_refr = refract_ray<G, N>(d, p, n, (G)mb.w, ro2, rd2);  // renderer.rs:235-239
                    const float gf = rg.g ? rg.g[h.id] : 0.f;
                    if (gf > 0.f && (has_refl || has_refr)) {
                        const int k = ((sj + level) % s) * s + si;   // rough_offset(s, si, sj, level)
                        G lx, ly;
                        if constexpr (sizeof(G) == 8) {
                            lx = rg.off[2 * k];
                            ly = rg.off[2 * k + 1];
                        } else {
                            lx = rg.off32[2 * k];
                            ly = rg.off32[2 * k + 1];
                        }
                        if (lx != G(0) || ly != G(0)) {
                            if (has_refl) {
                                rd1 = rough_dir<G>(rd1, (G)gf, lx, ly);
                                ro1 = rough_reflect_origin<G>(p, n, rd1);
                            }
                            if (has_refr) {
                                rd2 = rough_dir<G>(rd2, (G)gf, lx, ly);
                                ro2 = rough_refract_origin<G>(p, n, d, rd2);
                            }
                        }
                    }
                    if (has_refl || has_refr) {
                        RM_FAST_CHECK(sp < kMaxDepth);
                        Frame& f = fr[sp];
                        f.c = c;
                        f.k = mb.z;
                        if (has_refl) {
                            f.state = has_refr ? 1 : 0;
                            f.ro = ro2;
                            f.rd = rd2;
                            o = ro1;
                            d = rd1;
                        } else {
                            f.state = 2;
                            o = ro2;
                            d = rd2;
                        }
                        sp++;
                        pushed = true;
                    }
                }
                if (pushed) continue;
                v = c;
            }
        }
        for (;;) {                                              // return v to the callers on the stack
            if (sp == 0) return v;
            Frame& f = fr[sp - 1];
            if (f.state & 2) {
                f.c = f.c + scaled(v, 1.f - f.k);               // renderer.rs:249
                v = f.c;
                sp--;
            } else {
                f.c = f.c + scaled(v, f.k);                     // renderer.rs:219
                if (f.state & 1) {
                    o = f.ro;
                    d = f.rd;
                    f.state = 2;
                    break;
                }
                v = f.c;
                sp--;
            }
        }
    }
}
// A sample ray (o, d) of a distributed frame whose level-1 query found h: lens_shade with cast_glass_distributed, and in
// GLASS_NONE the direct lighting alone at level 1.
template <int kGlass, class DV>
RM_HD Vec3<float> distributed_shade(const DV& fv, const FrameParams<float>& fp, const RoughGlass& rg, const Vec3<double> o,
                                    const Vec3<double> d, HitRec<float> h) {
    if constexpr (kGlass == GLASS_F64) return cast_glass_distributed<double>(fv, fp, rg, o, d, h.dist, h.slot, h.id);
    const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
    if constexpr (kGlass == GLASS_F32) return cast_glass_distributed<float>(fv, fp, rg, o32, d32, h.dist, h.slot, h.id);
    Vec3<float> normal;
    fv.surface(h, o32, d32, normal);
    Counters<false> st;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    return bg + fv.template direct<false>(1, d32, h.p, normal, fv.mat_a[h.id], fv.mat_b[h.id], st);   // renderer.rs:272-275
}

// ---- diffuse interreflection (rm_render_indirect, include/rm_b200.h) -------------------------------------------------------
// cast_glass_from for sample (i, j) of the thin-lens camera with one diffuse bounce per opaque hit: at a hit of level
// L < max_depth on a primitive that is not glass-like, with diffusion > 0 and some diffuse_color component > 0, the ray
// leaves from diffuse_origin along diffuse_dir with the disc point of stratum diffuse_stratum(s, i, j, L), and its value v
// (background on a miss) is added as c + scaled(v * kd, diffusion).  Glass-like hits keep the reference's optics.  A level
// pushes at most one frame, so the stack holds at most max_depth - 1.  G = double: the bounce in f64 from the refined point
// and normal (diffuse_dir<double>, the normative definition); G = float: from the FP32 table.  kGlassOps = false (GLASS_NONE:
// the scene has no glass-like primitive) leaves out the reflect / refract branch.  Kept apart from cast_glass_from so that the
// lens kernel's machine code stays as it is.
template <typename G, bool kGlassOps, class FV>
RM_HD Vec3<float> cast_indirect(const FV& fv, const FrameParams<float>& fp, const Diffuse& df, const int si, const int sj,
                                Vec3<G> o, Vec3<G> d, const float t1, const int slot1, const int id1) {
    struct Frame {
        Vec3<float> c;
        Vec3<G> ro, rd;
        float k;
        int state;   // bit0: a refracted ray is pending, bit1: the refracted ray is the one in flight, bit2: a diffuse ray is
        int id;      // in flight from primitive id
    };
    Frame fr[kMaxDepth];
    int sp = 0;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    const int s = df.samples;
    Counters<false> st;
    Vec3<float> v;
    for (;;) {
        const int level = sp + 1;                               // n_recursion
        if (level > fp.max_depth) {
            v = bg;                                             // renderer.rs:262-264
        } else {
            const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
            HitRec<float> h;
            bool got = true;
            if (level == 1) {
                h.dist = t1;
                h.slot = slot1;
                h.id = id1;
            } else {
                got = fv.template closest<false>(o32, d32, level, h, st);      // renderer.rs:266: the search, FP32
            }
            if (!got) {
                v = bg;                                         // renderer.rs:300-306 (level > 1 here)
            } else {
                Vec3<G> p, n;
                Vec3<float> p32, n32;
                if constexpr (sizeof(G) == 8) {
                    fv.refine(h.slot, o, d, (double)h.dist, p, n);
                    p32 = to_f32(p);
                    n32 = to_f32(n);
                } else {
                    fv.surface(h, o32, d32, n32);
                    p32 = h.p;
                    p = p32;
                    n = n32;
                }
                const R4<float> ma = fv.mat_a[h.id];
                const R4<float> mb = fv.mat_b[h.id];
                Vec3<float> c = bg + fv.template direct<false>(o32, d32, p32, n32, ma, mb, st);   // renderer.rs:272-275
                bool pushed = false;
                const bool glass = kGlassOps && (fv.mat_f[h.id] & 1);
                if (glass) {                                    // renderer.rs:277
                    Vec3<G> ro1, rd1, ro2, rd2;
                    using N = typename std::conditional<sizeof(G) == 8, Fast64, Exact<float>>::type;
                    const bool has_refl = reflect_ray<G, N>(d, p, n, (G)mb.w, ro1, rd1);  // renderer.rs:203-207
                    const bool has_refr = refract_ray<G, N>(d, p, n, (G)mb.w, ro2, rd2);  // renderer.rs:235-239
                    if (has_refl || has_refr) {
                        RM_FAST_CHECK(sp < kMaxDepth);
                        Frame& f = fr[sp];
                        f.c = c;
                        f.k = mb.z;
                        if (has_refl) {
                            f.state = has_refr ? 1 : 0;
                            f.ro = ro2;
                            f.rd = rd2;
                            o = ro1;
                            d = rd1;
                        } else {
                            f.state = 2;
                            o = ro2;
                            d = rd2;
                        }
                        sp++;
                        pushed = true;
                    }
                } else if (level < fp.max_depth && ma.w > 0.f && (ma.x > 0.f || ma.y > 0.f || ma.z > 0.f)) {
                    const int k = diffuse_stratum(s, si, sj, level);
                    G lx, ly;
                    if constexpr (sizeof(G) == 8) {
                        lx = df.off[2 * k];
                        ly = df.off[2 * k + 1];
                    } else {
                        lx = df.off32[2 * k];
                        ly = df.off32[2 * k + 1];
                    }
                    const Vec3<G> nf = diffuse_normal<G>(n, d);
                    RM_FAST_CHECK(sp < kMaxDepth);
                    Frame& f = fr[sp];
                    f.c = c;
                    f.state = 4;
                    f.id = h.id;
                    o = diffuse_origin<G>(p, nf);
                    d = diffuse_dir<G>(nf, lx, ly);
                    sp++;
                    pushed = true;
                }
                if (pushed) continue;
                v = c;
            }
        }
        for (;;) {                                              // return v to the callers on the stack
            if (sp == 0) return v;
            Frame& f = fr[sp - 1];
            if (f.state & 4) {
                const R4<float> ma = fv.mat_a[f.id];
                v = f.c + scaled(v * Vec3<float>{ma.x, ma.y, ma.z}, ma.w);     // renderer.rs:181-183,192's lc * kd, diffusion
                sp--;
            } else if (f.state & 2) {
                f.c = f.c + scaled(v, 1.f - f.k);               // renderer.rs:249
                v = f.c;
                sp--;
            } else {
                f.c = f.c + scaled(v, f.k);                     // renderer.rs:219
                if (f.state & 1) {
                    o = f.ro;
                    d = f.rd;
                    f.state = 2;
                    break;
                }
                v = f.c;
                sp--;
            }
        }
    }
}
// Sample (i, j) of an indirect frame whose level-1 query found h: lens_shade with cast_indirect.  Opaque hits recurse here,
// so GLASS_NONE traces the same loop in FP32 without the glass branch.
template <int kGlass, class FV>
RM_HD Vec3<float> indirect_shade(const FV& fv, const FrameParams<float>& fp, const Diffuse& df, const int i, const int j,
                                 const Vec3<double> o, const Vec3<double> d, HitRec<float> h) {
    if constexpr (kGlass == GLASS_F64) return cast_indirect<double, true>(fv, fp, df, i, j, o, d, h.dist, h.slot, h.id);
    else return cast_indirect<float, kGlass == GLASS_F32>(fv, fp, df, i, j, to_f32(o), to_f32(d), h.dist, h.slot, h.id);
}

// ---- path-traced frames (rm_render_path, include/rm_b200.h) ---------------------------------------------------------------
// cast_glass_distributed with cast_indirect's bounce: every query, surface and shadow ray on the DistributedView of sample
// (i, j) = (fv.si, fv.sj) (the scene at the sample's time, the area lights' point of area_offset(s, i, j, L) at level L),
// rough glass-like hits turn the rays they spawn by rough_offset(s, i, j, L), and at a hit of level L < max_depth on a
// primitive that is not glass-like, with diffusion > 0 and some diffuse_color component > 0, one diffuse ray leaves from
// diffuse_origin along diffuse_dir with the disc point of stratum diffuse_stratum(s, i, j, L); its value v (background on a
// miss) is added as c + scaled(v * kd, diffusion), and its hit, a shading point of level L + 1, samples its lights at
// area_offset(s, i, j, L + 1).  A level pushes at most one frame, so the stack holds at most max_depth - 1.  G = double: the
// bounce in f64 from the refined point and normal (with motion, MotionView::refine's point at the sample's time); G = float:
// from the FP32 table.  kGlassOps = false (GLASS_NONE) leaves out the reflect / refract branch.  A copy of its own, so that
// the distributed and indirect kernels keep their machine code.
template <typename G, bool kGlassOps, class DV>
RM_HD Vec3<float> cast_path(const DV& fv, const FrameParams<float>& fp, const RoughGlass& rg, const Diffuse& df, Vec3<G> o, Vec3<G> d,
                            const float t1, const int slot1, const int id1) {
    struct Frame {
        Vec3<float> c;
        Vec3<G> ro, rd;
        float k;
        int state;   // bit0: a refracted ray is pending, bit1: the refracted ray is the one in flight, bit2: a diffuse ray is
        int id;      // in flight from primitive id
    };
    Frame fr[kMaxDepth];
    int sp = 0;
    const Vec3<float> bg = {fp.background, fp.background, fp.background};
    const int s = df.samples, si = fv.si, sj = fv.sj;
    Counters<false> st;
    Vec3<float> v;
    for (;;) {
        const int level = sp + 1;                               // n_recursion
        if (level > fp.max_depth) {
            v = bg;                                             // renderer.rs:262-264
        } else {
            const Vec3<float> o32 = to_f32(o), d32 = to_f32(d);
            HitRec<float> h;
            bool got = true;
            if (level == 1) {
                h.dist = t1;
                h.slot = slot1;
                h.id = id1;
            } else {
                got = fv.template closest<false>(o32, d32, level, h, st);      // renderer.rs:266: the search, FP32
            }
            if (!got) {
                v = bg;                                         // renderer.rs:300-306 (level > 1 here)
            } else {
                Vec3<G> p, n;
                Vec3<float> p32, n32;
                if constexpr (sizeof(G) == 8) {
                    fv.refine(h.slot, o, d, (double)h.dist, p, n);
                    p32 = to_f32(p);
                    n32 = to_f32(n);
                } else {
                    fv.surface(h, o32, d32, n32);
                    p32 = h.p;
                    p = p32;
                    n = n32;
                }
                const R4<float> ma = fv.mat_a[h.id];
                const R4<float> mb = fv.mat_b[h.id];
                Vec3<float> c = bg + fv.template direct<false>(level, d32, p32, n32, ma, mb, st);   // renderer.rs:272-275
                bool pushed = false;
                const bool glass = kGlassOps && (fv.mat_f[h.id] & 1);
                if (glass) {                                    // renderer.rs:277
                    Vec3<G> ro1, rd1, ro2, rd2;
                    using N = typename std::conditional<sizeof(G) == 8, Fast64, Exact<float>>::type;
                    const bool has_refl = reflect_ray<G, N>(d, p, n, (G)mb.w, ro1, rd1);  // renderer.rs:203-207
                    const bool has_refr = refract_ray<G, N>(d, p, n, (G)mb.w, ro2, rd2);  // renderer.rs:235-239
                    const float gf = rg.g ? rg.g[h.id] : 0.f;
                    if (gf > 0.f && (has_refl || has_refr)) {
                        const int k = ((sj + level) % s) * s + si;   // rough_offset(s, si, sj, level)
                        G lx, ly;
                        if constexpr (sizeof(G) == 8) {
                            lx = rg.off[2 * k];
                            ly = rg.off[2 * k + 1];
                        } else {
                            lx = rg.off32[2 * k];
                            ly = rg.off32[2 * k + 1];
                        }
                        if (lx != G(0) || ly != G(0)) {
                            if (has_refl) {
                                rd1 = rough_dir<G>(rd1, (G)gf, lx, ly);
                                ro1 = rough_reflect_origin<G>(p, n, rd1);
                            }
                            if (has_refr) {
                                rd2 = rough_dir<G>(rd2, (G)gf, lx, ly);
                                ro2 = rough_refract_origin<G>(p, n, d, rd2);
                            }
                        }
                    }
                    if (has_refl || has_refr) {
                        RM_FAST_CHECK(sp < kMaxDepth);
                        Frame& f = fr[sp];
                        f.c = c;
                        f.k = mb.z;
                        if (has_refl) {
                            f.state = has_refr ? 1 : 0;
                            f.ro = ro2;
                            f.rd = rd2;
                            o = ro1;
                            d = rd1;
                        } else {
                            f.state = 2;
                            o = ro2;
                            d = rd2;
                        }
                        sp++;
                        pushed = true;
                    }
                } else if (level < fp.max_depth && ma.w > 0.f && (ma.x > 0.f || ma.y > 0.f || ma.z > 0.f)) {
                    const int k = diffuse_stratum(s, si, sj, level);
                    G lx, ly;
                    if constexpr (sizeof(G) == 8) {
                        lx = df.off[2 * k];
                        ly = df.off[2 * k + 1];
                    } else {
                        lx = df.off32[2 * k];
                        ly = df.off32[2 * k + 1];
                    }
                    const Vec3<G> nf = diffuse_normal<G>(n, d);
                    RM_FAST_CHECK(sp < kMaxDepth);
                    Frame& f = fr[sp];
                    f.c = c;
                    f.state = 4;
                    f.id = h.id;
                    o = diffuse_origin<G>(p, nf);
                    d = diffuse_dir<G>(nf, lx, ly);
                    sp++;
                    pushed = true;
                }
                if (pushed) continue;
                v = c;
            }
        }
        for (;;) {                                              // return v to the callers on the stack
            if (sp == 0) return v;
            Frame& f = fr[sp - 1];
            if (f.state & 4) {
                const R4<float> ma = fv.mat_a[f.id];
                v = f.c + scaled(v * Vec3<float>{ma.x, ma.y, ma.z}, ma.w);     // renderer.rs:181-183,192's lc * kd, diffusion
                sp--;
            } else if (f.state & 2) {
                f.c = f.c + scaled(v, 1.f - f.k);               // renderer.rs:249
                v = f.c;
                sp--;
            } else {
                f.c = f.c + scaled(v, f.k);                     // renderer.rs:219
                if (f.state & 1) {
                    o = f.ro;
                    d = f.rd;
                    f.state = 2;
                    break;
                }
                v = f.c;
                sp--;
            }
        }
    }
}
// A sample ray (o, d) of a path-traced frame whose level-1 query found h: distributed_shade with cast_path.  Opaque hits
// recurse here, so GLASS_NONE traces the same loop in FP32 without the glass branch (distributed_shade's level-1 shortcut
// would drop the bounces).
template <int kGlass, class DV>
RM_HD Vec3<float> path_shade(const DV& fv, const FrameParams<float>& fp, const RoughGlass& rg, const Diffuse& df, const Vec3<double> o,
                             const Vec3<double> d, HitRec<float> h) {
    if constexpr (kGlass == GLASS_F64) return cast_path<double, true>(fv, fp, rg, df, o, d, h.dist, h.slot, h.id);
    else return cast_path<float, kGlass == GLASS_F32>(fv, fp, rg, df, to_f32(o), to_f32(d), h.dist, h.slot, h.id);
}

}  // namespace rm
