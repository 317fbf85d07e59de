// rm_trace.cuh -- per-ray work of the render hot path: closest-hit / any-hit queries over the
// flattened scene, direct lighting with shadow rays, the optics of glass-like materials and the
// depth-capped reflect/refract recursion, unrolled into an iterative per-thread stack.
//
// Each routine cites the reference lines it replaces.  The code is templated on the scalar type
// (see rm_math.cuh) and on a compile-time `S` flag that switches the event counters on (used
// once per workload outside the timed region to obtain the algorithmic work; SURVEY.md 8d).
#pragma once

#include "rm_math.cuh"

namespace rm {

constexpr int kMaxDepth = 8;   // frames of the iterative stack (reference: 3, renderer.rs:262)

// indices into Counters::c -- same order as RmStats / OrcCounters
enum CounterId {
    C_PIXELS, C_CLOSEST, C_ANYHIT, C_SPH_TEST, C_SPH_DISC, C_SPH_HIT, C_PLN_TEST, C_PLN_DIST, C_PLN_POINT,
    C_EDGE, C_CAND, C_HITS, C_LIGHT_EVAL, C_LIT, C_GLASS, C_REFL, C_REFR, C_COUNT
};

template <bool S> struct Counters {
    RM_HD void clear() {}
    RM_HD void add(int, unsigned = 1) {}
};
template <> struct Counters<true> {
    unsigned c[C_COUNT];
    RM_HD void clear() { for (int i = 0; i < C_COUNT; i++) c[i] = 0; }
    RM_HD void add(int id, unsigned n = 1) { c[id] += n; }
};

// The scene as the kernels see it (pointers into shared or global memory).
//   sph[i]    = {cx, cy, cz, r^2}                       sphere.rs:6-11
//   pln_n[i]  = {nx, ny, nz, thr}   hit needs |d.n| > thr: thr = pred(1e-6) for triangles
//                                   (triangle.rs:57), 0 for polygons (polygon.rs:66)
//   pln_c[i]  = f64: {Cx, Cy, Cz, 0} plane point (triangle.center / polygon.plane_point)
//               f32: {n.C, v0.x, v0.y, 0}
//   pln_v[i]  = {first, count} into vert[]: f64 {x, y} per vertex (only x,y are ever read:
//               triangle.rs:13-15 uses the z component of the cross product); f32 {A, B, C, 0} per edge
//   *_id[i]   = flattened primitive id (index in scene order, Obj expanded per triangle)
//   mat_a[id] = {kd.r, kd.g, kd.b, diffusion}; mat_b[id] = {specular, exponent, reflection, index}
//   mat_f[id] = bit0 is_glass_like                      shapes.rs:21-32
//   lgt_p[l]  = {px, py, pz, intensity}; lgt_c[l] = {r, g, b, 0}      lights.rs:4-8
// `order*` (instrumented variant only) lists the resident primitives in scene order so that the
// counters follow the reference's traversal: order[k] = slot (sphere i -> i, plane i -> n_sph+i),
// order_shape[k] = index of the owning shape, bit 30 set when the shape is an Obj.
template <typename R> struct VertOf { typedef R2<R> type; };
template <> struct VertOf<float> { typedef R4<float> type; };
template <typename R> using VertT = typename VertOf<R>::type;

template <typename R> struct HitRec;
template <typename R> struct SceneView;
template <typename R, bool S>
RM_HD bool find_closest_intersect(const SceneView<R>& sc, const Vec3<R> o, const Vec3<R> d, HitRec<R>& best, Counters<S>& st);
template <typename R, bool S>
RM_HD bool intersect_shape_set(const SceneView<R>& sc, const Vec3<R> o, const Vec3<R> d, Counters<S>& st);
template <typename R> RM_HD void surface_of(const SceneView<R>& sc, HitRec<R>& h, const Vec3<R> o, const Vec3<R> d, Vec3<R>& normal);
template <typename R, bool S, typename SC>
RM_HD Vec3<R> direct_lighting(const SC& sc, const Vec3<R> origin, const Vec3<R> point, const Vec3<R> normal, const R4<R> ma,
                              const R4<R> mb, Counters<S>& st);

template <typename R> struct SceneView {
    // the query interface cast_ray / direct_lighting are written against (rm_fast.cuh has a second implementation)
    template <bool S> RM_HD bool closest(const Vec3<R> o, const Vec3<R> d, int /*level*/, HitRec<R>& h, Counters<S>& st) const {
        return find_closest_intersect<R, S>(*this, o, d, h, st);
    }
    template <bool S> RM_HD bool anyhit(const Vec3<R> o, const Vec3<R> d, Counters<S>& st) const {
        return intersect_shape_set<R, S>(*this, o, d, st);
    }
    RM_HD void surface(HitRec<R>& h, const Vec3<R> o, const Vec3<R> d, Vec3<R>& normal) const { surface_of(*this, h, o, d, normal); }
    template <bool S> RM_HD Vec3<R> direct(const Vec3<R> origin, const Vec3<R> /*dir*/, const Vec3<R> point, const Vec3<R> normal,
                                           const R4<R> ma, const R4<R> mb, Counters<S>& st) const {
        return direct_lighting<R, S, SceneView<R>>(*this, origin, point, normal, ma, mb, st);
    }

    const R4<R>* sph;
    const int* sph_id;
    int n_sph;
    const R4<R>* pln_n;
    const R4<R>* pln_c;
    const I2* pln_v;
    const int* pln_id;
    int n_pln;
    const VertT<R>* vert;
    const R4<R>* mat_a;
    const R4<R>* mat_b;
    const int* mat_f;
    const R4<R>* lgt_p;
    const R4<R>* lgt_c;
    int n_lgt;
    const int* order;
    const int* order_shape;
    int n_order;
};

template <typename R> struct HitRec {
    Vec3<R> p;
    R dist;     // f64: |p - orig|^2 (shapes.rs:128); f32: the ray parameter t (same ordering, d is unit)
    int slot;   // sphere i -> i, plane i -> n_sph + i
    int id;     // flattened primitive id
};

// One candidate hit.  f64 carries the point like the reference; f32 only the ray parameter, the point
// is formed once for the winner.
template <typename R> struct Cand {
    Vec3<R> p;
    R key;
};

// ---------------------------------------------------------------- sphere.rs:27-61
template <bool S>
RM_HD bool sphere_intersect(const R4<double> s, const Vec3<double> o, const Vec3<double> d, Cand<double>& c, Counters<S>& st) {
    Vec3<double> line = {s.x - o.x, s.y - o.y, s.z - o.z};
    double tca = dot(line, d);
    double d2 = dot(line, line) - tca * tca;
    st.add(C_SPH_TEST);
    if (d2 > s.w) return false;
    st.add(C_SPH_DISC);
    double thc = sqrt(s.w - d2);
    double t0 = tca - thc;
    double t1 = tca + thc;
    if (t0 < 0.) t0 = t1;
    if (t0 < 0.) return false;
    st.add(C_SPH_HIT);
    c.p = axpy(o, d, t0);
    c.key = squared_norm(c.p - o);                             // shapes.rs:128
    return true;
}
// f32: the reference's d2 = line.line - tca^2 cancels catastrophically in single precision for a small
// far sphere (error 2^-24*|line|^2 against r^2), so the squared distance of the centre to the ray is
// taken from the perpendicular component itself: perp = line - tca*d, d2 = perp.perp.
template <bool S>
RM_HD bool sphere_intersect(const R4<float> s, const Vec3<float> o, const Vec3<float> d, Cand<float>& c, Counters<S>& st) {
    Vec3<float> line = {s.x - o.x, s.y - o.y, s.z - o.z};
    float tca = dot(line, d);
    Vec3<float> perp = axmy(line, d, tca);
    float d2 = dot(perp, perp);
    st.add(C_SPH_TEST);
    if (d2 > s.w) return false;
    st.add(C_SPH_DISC);
    float thc = sqrtf(s.w - d2);
    float t0 = tca - thc;
    if (t0 < 0.f) t0 = tca + thc;
    if (t0 < 0.f) return false;
    st.add(C_SPH_HIT);
    c.key = t0;
    return true;
}

// Hit point and unit normal of the winning sphere hit (sphere.rs:54-60).
RM_HD void sphere_point_normal(const R4<double> s, const Vec3<double>, const Vec3<double>, const Vec3<double> p_in,
                               Vec3<double>& p, Vec3<double>& n) {
    p = p_in;
    n = normalized(p_in - xyz(s));
}
// f32: p - c = (t - tca)*d - perp = -+thc*d - perp, formed from the two short vectors instead of the
// difference of two long ones (o + t*d) - c.
RM_HD void sphere_point_normal(const R4<float> s, const Vec3<float> o, const Vec3<float> d, const Vec3<float>,
                               Vec3<float>& p, Vec3<float>& n) {
    Vec3<float> line = {s.x - o.x, s.y - o.y, s.z - o.z};
    float tca = dot(line, d);
    Vec3<float> perp = axmy(line, d, tca);
    float thc = sqrtf(fmaxf(s.w - dot(perp, perp), 0.f));
    float w = (tca - thc < 0.f) ? thc : -thc;                  // same root as sphere_intersect chose
    Vec3<float> pc = {fmaf(w, d.x, -perp.x), fmaf(w, d.y, -perp.y), fmaf(w, d.z, -perp.z)};
    p = xyz(s) + pc;
    n = normalized(pc);
}

// ---------------------------------------------------------------- triangle.rs:49-83, polygon.rs:60-98
// f64: the reference's arithmetic, operation for operation.
//   pln_n = {n, thr}, pln_c = {plane point, 0}, vert[] = {x, y} of each vertex
template <bool S>
RM_HD bool plane_intersect(const R4<double> n4, const R4<double> c4, const I2 vr, const R2<double>* __restrict__ vert,
                           const Vec3<double> o, const Vec3<double> d, Cand<double>& c, Counters<S>& st) {
    Vec3<double> n = xyz(n4);
    double dp = dot(d, n);
    st.add(C_PLN_TEST);
    if (!(fabs(dp) > n4.w)) return false;                      // parallel (triangle.rs:57 / polygon.rs:66)
    Vec3<double> co = {c4.x - o.x, c4.y - o.y, c4.z - o.z};
    double dist = dot(co, n) / dp;                             // triangle.rs:62
    st.add(C_PLN_DIST);
    if (dist < 0.) return false;                               // going away
    Vec3<double> q = axpy(o, d, dist);
    st.add(C_PLN_POINT);
    // inside(): ((v_i - q) x (v_i+1 - q)).z > 0 for every edge, early out (triangle.rs:72-76)
    R2<double> v1 = vert[vr.x];
    for (int i = 0; i < vr.y; i++) {
        R2<double> v2 = vert[vr.x + ((i + 1 == vr.y) ? 0 : i + 1)];
        double ux = v1.x - q.x, uy = v1.y - q.y, vx = v2.x - q.x, vy = v2.y - q.y;
        double cz = ux * vy - uy * vx;
        st.add(C_EDGE);
        if (!(cz > 0.)) return false;
        v1 = v2;
    }
    c.p = q;
    c.key = squared_norm(q - o);                               // obj.rs:197 / shapes.rs:128
    return true;
}
// f32: same predicates in a form that is robust in single precision.  The reference evaluates the
// edge term at the hit point p = o + t*d, which loses all significance in FP32 when a grazing ray
// meets the plane far away (|p|^2 * 2^-24 exceeds the triangle's area).  The term is affine in p,
//   e_i(p) = A_i*(p.x - v0.x) + B_i*(p.y - v0.y) + C_i,   A_i = v_i.y - v_i+1.y,  B_i = v_i+1.x - v_i.x,
//   C_i = ((v_i - v0) x (v_i+1 - v0)).z,
// so it is evaluated as e_i(o) + t*(A_i*d.x + B_i*d.y): two numbers of the size of the result.
//   pln_n = {n, thr}, pln_c = {n.C, v0.x, v0.y, 0} (f64 on the host), vert[] = {A_i, B_i, C_i, 0}
template <bool S>
RM_HD bool plane_intersect(const R4<float> n4, const R4<float> k4, const I2 vr, const R4<float>* __restrict__ edge,
                           const Vec3<float> o, const Vec3<float> d, Cand<float>& c, Counters<S>& st) {
    Vec3<float> n = xyz(n4);
    float dp = dot(d, n);
    st.add(C_PLN_TEST);
    if (!(fabsf(dp) > n4.w)) return false;
    float t = (k4.x - dot(o, n)) / dp;                         // ((C - o).n) / (d.n)
    st.add(C_PLN_DIST);
    if (t < 0.f) return false;
    st.add(C_PLN_POINT);
    const float wx = o.x - k4.y, wy = o.y - k4.z;
    for (int i = 0; i < vr.y; i++) {
        const R4<float> e = edge[vr.x + i];
        float g = fmaf(e.y, d.y, e.x * d.x);
        float e0 = fmaf(e.x, wx, fmaf(e.y, wy, e.z));
        st.add(C_EDGE);
        if (!(fmaf(t, g, e0) > 0.f)) return false;
    }
    c.key = t;
    return true;
}

template <typename R>
RM_HD void consider(HitRec<R>& best, bool& hit, const Cand<R>& c, int slot, int id) {
    // strict '<' with the first primitive in scene order winning ties (shapes.rs:130, obj.rs:198);
    // the id comparison keeps that rule although spheres are traversed before planes here
    if (!hit || c.key < best.dist || (c.key == best.dist && id < best.id)) {
        best.p = c.p;
        best.dist = c.key;
        best.slot = slot;
        best.id = id;
        hit = true;
    }
}

// ---------------------------------------------------------------- shapes.rs:110-143 + obj.rs:186-216
template <typename R, bool S>
RM_HD bool find_closest_intersect(const SceneView<R>& sc, const Vec3<R> o, const Vec3<R> d, HitRec<R>& best,
                                  Counters<S>& st) {
    bool hit = false;
    st.add(C_CLOSEST);
    if constexpr (S) {
        // instrumented: scene order, so that per-event counts equal the reference traversal
        int last_shape = -1;
        for (int k = 0; k < sc.n_order; k++) {
            int slot = sc.order[k];
            int shape = sc.order_shape[k];
            Cand<R> c;
            bool got;
            int id;
            if (slot < sc.n_sph) {
                got = sphere_intersect<S>(sc.sph[slot], o, d, c, st);
                id = sc.sph_id[slot];
            } else {
                int i = slot - sc.n_sph;
                got = plane_intersect<S>(sc.pln_n[i], sc.pln_c[i], sc.pln_v[i], sc.vert, o, d, c, st);
                id = sc.pln_id[i];
            }
            if (got) {
                // one distance per hit in the shape loop (shapes.rs:128) plus, inside an Obj, one per
                // hitting triangle (obj.rs:197)
                if (shape & (1 << 30)) st.add(C_CAND, (shape != last_shape) ? 2 : 1);
                else st.add(C_CAND);
                last_shape = shape;
                consider(best, hit, c, slot, id);
            }
        }
        return hit;
    } else {
        for (int i = 0; i < sc.n_sph; i++) {
            Cand<R> c;
            if (sphere_intersect<S>(sc.sph[i], o, d, c, st)) consider(best, hit, c, i, sc.sph_id[i]);
        }
        for (int i = 0; i < sc.n_pln; i++) {
            Cand<R> c;
            if (plane_intersect<S>(sc.pln_n[i], sc.pln_c[i], sc.pln_v[i], sc.vert, o, d, c, st))
                consider(best, hit, c, sc.n_sph + i, sc.pln_id[i]);
        }
        return hit;
    }
}

// ---------------------------------------------------------------- shapes.rs:92-108
// No maximum distance: occluders behind the light still shadow.  The reference keeps scanning the
// triangles of an Obj after its first hit (obj.rs:194-210); the boolean result is the same when we
// stop at the first hitting primitive, and that is how the algorithmic work is counted.
template <typename R, bool S>
RM_HD bool intersect_shape_set(const SceneView<R>& sc, const Vec3<R> o, const Vec3<R> d, Counters<S>& st) {
    st.add(C_ANYHIT);
    Cand<R> c;
    if constexpr (S) {
        for (int k = 0; k < sc.n_order; k++) {
            int slot = sc.order[k];
            bool got;
            if (slot < sc.n_sph) got = sphere_intersect<S>(sc.sph[slot], o, d, c, st);
            else {
                int i = slot - sc.n_sph;
                got = plane_intersect<S>(sc.pln_n[i], sc.pln_c[i], sc.pln_v[i], sc.vert, o, d, c, st);
            }
            if (got) {
                if (sc.order_shape[k] & (1 << 30)) st.add(C_CAND);   // obj.rs:197
                return true;
            }
        }
        return false;
    } else {
        for (int i = 0; i < sc.n_sph; i++)
            if (sphere_intersect<S>(sc.sph[i], o, d, c, st)) return true;
        for (int i = 0; i < sc.n_pln; i++)
            if (plane_intersect<S>(sc.pln_n[i], sc.pln_c[i], sc.pln_v[i], sc.vert, o, d, c, st)) return true;
        return false;
    }
}

// ---------------------------------------------------------------- optics.rs:4-6
template <typename R> RM_HD Vec3<R> reflect(Vec3<R> incident, Vec3<R> normal) {
    return axmy(incident, normal, R(2) * dot(incident, normal));
}

// ---------------------------------------------------------------- optics.rs:8-48
template <typename R, typename N = Exact<R>>
RM_HD bool reflect_ray(Vec3<R> incident, Vec3<R> point, Vec3<R> hit_normal, R refractive_index, Vec3<R>& ro, Vec3<R>& rd) {
    Vec3<R> normal = hit_normal;
    R c = dot(normal, incident);
    R r = (c < R(0)) ? refractive_index : N::rcp_(refractive_index);
    if (c < R(0)) { c = -c; normal = -normal; }
    R cos_theta_2 = R(1) - r * r * (R(1) - c * c);
    if (cos_theta_2 > R(0)) return false;
    rd = reflect(incident, normal);
    if (dot(rd, hit_normal) < R(0)) ro = axmy(point, hit_normal, R(1e-4));
    else ro = axpy(point, hit_normal, R(1e-4));
    return true;
}

// ---------------------------------------------------------------- optics.rs:50-89
template <typename R, typename N = Exact<R>>
RM_HD bool refract_ray(Vec3<R> incident, Vec3<R> point, Vec3<R> hit_normal, R refractive_index, Vec3<R>& ro, Vec3<R>& rd) {
    Vec3<R> normal = hit_normal;
    R c = -dot(normal, incident);
    R r = (c < R(0)) ? refractive_index : N::rcp_(refractive_index);
    if (c < R(0)) { c = -c; normal = -normal; }
    R cos_theta_2 = R(1) - r * r * (R(1) - c * c);
    if (cos_theta_2 < R(0)) return false;
    rd = N::normalized(scaled(incident, r) + scaled(normal, r * c - N::sqrt_(cos_theta_2)));
    if (dot(rd, normal) > R(0)) ro = axpy(point, normal, R(1e-4));
    else ro = axmy(point, normal, R(1e-4));
    return true;
}

// point + unit normal of the winning hit (sphere.rs:54-58; planes carry their precomputed normal)
template <typename R> RM_HD void surface_of(const SceneView<R>& sc, HitRec<R>& h, const Vec3<R> o, const Vec3<R> d, Vec3<R>& normal) {
    if (h.slot < sc.n_sph) {
        sphere_point_normal(sc.sph[h.slot], o, d, h.p, h.p, normal);
    } else {
        if (sizeof(R) == 4) h.p = axpy(o, d, h.dist);          // f32: point of the winner only
        normal = xyz(sc.pln_n[h.slot - sc.n_sph]);
    }
}

// ---------------------------------------------------------------- renderer.rs:138-193
template <typename R, bool S, typename SC>
RM_HD Vec3<R> direct_lighting(const SC& sc, const Vec3<R> origin, const Vec3<R> point, const Vec3<R> normal,
                              const R4<R> ma, const R4<R> mb, Counters<S>& st) {
    Vec3<R> acc = {R(0), R(0), R(0)};
    const Vec3<R> to_viewer = normalized(origin - point);                                         // renderer.rs:149 (the same for every light)
    for (int l = 0; l < sc.n_lgt; l++) {
        R4<R> lp = sc.lgt_p[l];
        R4<R> lc4 = sc.lgt_c[l];
        Vec3<R> lc = xyz(lc4);
        Vec3<R> light_dir = normalized(Vec3<R>{lp.x - point.x, lp.y - point.y, lp.z - point.z});   // renderer.rs:166
        R side = dot(light_dir, normal);
        st.add(C_LIGHT_EVAL);
        Vec3<R> so = (side < R(0)) ? axmy(point, normal, R(1e-3)) : axpy(point, normal, R(1e-3)); // renderer.rs:168-172
        pin(so);
        pin(light_dir);
        if (sc.template anyhit<S>(so, light_dir, st)) continue;                                   // renderer.rs:174-177
        st.add(C_LIT);
        R diffusion = Num<R>::max_(side, R(0));                                                   // renderer.rs:138-140
        Vec3<R> kd = {ma.x, ma.y, ma.z};
        acc = acc + scaled(scaled(lc * kd, diffusion), lp.w);                                     // renderer.rs:181-183
        Vec3<R> reflected = reflect(-light_dir, normal);                                          // renderer.rs:144-145
        R sf = Num<R>::max_(dot(reflected, to_viewer), R(0));                                     // renderer.rs:150
        R specular = Num<R>::pow_(sf * mb.x, mb.y);                                               // renderer.rs:186-188
        acc = acc + scaled(lc, specular);                                                         // renderer.rs:189
    }
    return scaled(acc, ma.w);                                                                     // renderer.rs:192
}

// ---------------------------------------------------------------- renderer.rs:254-309
// cast_ray's recursion (branching factor 2, depth cap max_depth) as an explicit stack.  A frame is
// pushed for a glass hit that spawned at least one secondary ray; it keeps the partial sum and the
// pending refracted ray so that the additions happen in the reference's order:
//   c = bg + direct;  c += cast(reflected) * k;  c += cast(refracted) * (1 - k).
template <typename R, bool S, typename SC>
RM_HD Vec3<R> cast_ray(const SC& sc, Vec3<R> o, Vec3<R> d, R background, int max_depth, int& primary_id,
                       Counters<S>& st) {
    struct Frame {
        Vec3<R> c, ro, rd;
        R k;
        int state;   // bit0: a refracted ray is pending, bit1: the refracted ray is the one in flight
    };
    Frame fr[kMaxDepth];
    int sp = 0;
    const Vec3<R> bg = {background, background, background};
    Vec3<R> v;
    primary_id = -1;
    for (;;) {
        const int level = sp + 1;                               // n_recursion
        if (level > max_depth) {
            v = bg;                                             // renderer.rs:262-264
        } else {
            HitRec<R> h;
            bool got = sc.template closest<S>(o, d, level, h, st);      // renderer.rs:266
            if (level == 1 && got) primary_id = h.id;
            if (!got) {
                v = (level > 1) ? bg : Vec3<R>{R(0), R(0), R(0)};       // renderer.rs:300-306
            } else {
                st.add(C_HITS);
                Vec3<R> normal;
                sc.surface(h, o, d, normal);
                const R4<R> ma = sc.mat_a[h.id];
                const R4<R> mb = sc.mat_b[h.id];
                Vec3<R> c = bg + sc.template direct<S>(o, d, h.p, normal, ma, mb, st);        // renderer.rs:272-275
                bool pushed = false;
                if (sc.mat_f[h.id] & 1) {                       // renderer.rs:277
                    st.add(C_GLASS);
                    Vec3<R> ro1, rd1, ro2, rd2;
                    bool has_refl = reflect_ray<R>(d, h.p, normal, mb.w, ro1, rd1);       // renderer.rs:203-207
                    bool has_refr = refract_ray<R>(d, h.p, normal, mb.w, ro2, rd2);       // renderer.rs:235-239
                    if (has_refl) st.add(C_REFL);
                    if (has_refr) st.add(C_REFR);
                    if (has_refl || has_refr) {
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
        // return v to the callers on the stack
        for (;;) {
            if (sp == 0) return v;
            Frame& f = fr[sp - 1];
            if (f.state & 2) {
                f.c = f.c + scaled(v, R(1) - f.k);              // renderer.rs:249
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

// Per-frame constants.  backproject (renderer.rs:128-135):
//   x = 2*(j/W - 0.5)*half_fov*ratio, y = -2*(i/H - 0.5)*half_fov, z = -1, then normalised.
template <typename R> struct FrameParams {
    int width, height;
    int row_begin, row_end;       // pixel-row span of this call
    int row_step;                 // pixel rows from one rendered 32-row band to the next (32 = contiguous; 32*G when the
                                  // bands of a frame are dealt round-robin to G ranks)
    int n_bands;                  // rendered 32-row bands: rows row_begin + b*row_step + [0, 32), b < n_bands
    int buf_row0;                 // pixel row stored at offset 0 of the output buffers
    R width_r, height_r, half_fov, ratio;   // f64 path: the reference's own operands
    R half_w, half_h, sx, sy;     // f32 path: x = (j - W/2)*sx, y = (i - H/2)*sy, folded on the host in f64
    Vec3<R> camera;
    R background;
    int max_depth;
    int accel;                    // RmParams.accel: scene queries through the hierarchy (FP32 production kernel)
    // the reference's own f64 operands of backproject (renderer.rs:128-135) and the camera, whatever R is: the FP32
    // production kernel traces the paths behind a glass-like primary hit with f64 ray geometry (cast_glass, rm_fast.cuh)
    double cam64[3], w64, h64, hf64, ratio64, inv_w64, inv_h64;
};

// pixel row of the l-th rendered row of this call (l in [0, 32 * n_bands))
template <typename R> RM_HD int frame_row(const FrameParams<R>& fp, int l) { return fp.row_begin + (l >> 5) * fp.row_step + (l & 31); }

template <typename R> RM_HD Vec3<R> backproject(const FrameParams<R>& fp, int j, int i) {
    Vec3<R> v = {(R(j) - fp.half_w) * fp.sx, (R(i) - fp.half_h) * fp.sy, R(-1)};
    return normalized(v);
}
template <> RM_HD Vec3<double> backproject<double>(const FrameParams<double>& fp, int j, int i) {
    Vec3<double> v = {2. * ((double)j / fp.width_r - 0.5) * fp.half_fov * fp.ratio,
                      -2. * ((double)i / fp.height_r - 0.5) * fp.half_fov, -1.};
    return normalized(v);
}

// Camera orientation (rm_render_view, include/rm_b200.h).  The orthonormal basis u, v, w (m[0..2], m[3..5], m[6..8]) takes
// a camera-space direction d to the world direction ((u.x d.x + v.x d.y) + w.x d.z, ...); to_camera is the transpose,
// (u.g, v.g, w.g), which K0 applies to the raster records so that stage A keeps its camera-space D = (X, Y, -1).
// f: the basis rounded to FP32, for the production kernel's FP32 directions.
struct ViewBasis {
    double m[9];
    float f[9];
    RM_HD Vec3<double> apply(const Vec3<double> d) const {
        return {(m[0] * d.x + m[3] * d.y) + m[6] * d.z, (m[1] * d.x + m[4] * d.y) + m[7] * d.z,
                (m[2] * d.x + m[5] * d.y) + m[8] * d.z};
    }
    RM_HD Vec3<float> apply(const Vec3<float> d) const {
        return {fmaf(f[6], d.z, fmaf(f[3], d.y, f[0] * d.x)), fmaf(f[7], d.z, fmaf(f[4], d.y, f[1] * d.x)),
                fmaf(f[8], d.z, fmaf(f[5], d.y, f[2] * d.x))};
    }
    RM_HD Vec3<double> to_camera(const Vec3<double> g) const {
        return {(m[0] * g.x + m[1] * g.y) + m[2] * g.z, (m[3] * g.x + m[4] * g.y) + m[5] * g.z,
                (m[6] * g.x + m[7] * g.y) + m[8] * g.z};
    }
};
// The reference's camera (u, v, w = x, y, z): every pre-existing kernel instantiates its code with this, which compiles
// to exactly the code it had before the view existed.
struct NoView {
    NoView() = default;
    RM_HD explicit NoView(const ViewBasis&) {}
    template <typename R> RM_HD Vec3<R> apply(const Vec3<R> d) const { return d; }
    RM_HD Vec3<double> to_camera(const Vec3<double> g) const { return g; }
};
template <bool kView> struct ViewOf { typedef NoView type; };
template <> struct ViewOf<true> { typedef ViewBasis type; };

// Thin-lens camera (rm_render_lens, include/rm_b200.h RmLens): the normative definition in f64 without fused multiply-add.
// The kernel, the host code and the tests' host emulation all call these two functions.
// Lens point of sample (i, j) of s x s: the stratum (a, b) = ((i + j) mod s, j) -- shifted so that lens strata do not follow
// the sub-pixel strata -- taken from the square to the unit disc by the elliptical grid map.  Only sqrt, which is correctly
// rounded on host and device, so every restatement gets the same bits.
RM_HD void lens_offset(const int s, const int i, const int j, double* lx, double* ly) {
    const int a = (i + j) % s, b = j;
    const double p = (2. * a + 1.) / s - 1., q = (2. * b + 1.) / s - 1.;
    *lx = p * sqrt(1. - (q * q) * 0.5);
    *ly = q * sqrt(1. - (p * p) * 0.5);
}

struct LensCamera {
    double width, height;     // of the s x frame: backproject's operands (renderer.rs:128-135)
    double half_fov, ratio;   // tan(fov / 2) and width / height (renderer.rs:25-33)
    double cam[3];
    ViewBasis view;           // u, v, w; the identity without a view
    double aperture, focus;   // lens radius (>= 0) and distance of the plane in focus along the view axis (> 0)
    int samples;              // s
};

// The ray (o, d) of sample (i, j) of output pixel (x, y): d0 is the supersampled frame's sub-pixel (s x + j, s y + i)
// direction; through a lens of radius > 0 the ray leaves the lens point L = aperture (lx, ly, 0) towards the point
// P = d0 focus / -d0.z of the plane in focus, which every sample of the pixel shares.
RM_HD void lens_ray(const LensCamera& lc, const int x, const int y, const int i, const int j, Vec3<double>& o, Vec3<double>& d) {
    const int s = lc.samples;
    const Vec3<double> d0 = normalized(Vec3<double>{2. * ((double)(s * x + j) / lc.width - 0.5) * lc.half_fov * lc.ratio,
                                                    -2. * ((double)(s * y + i) / lc.height - 0.5) * lc.half_fov, -1.});
    if (lc.aperture == 0.) {
        o = {lc.cam[0], lc.cam[1], lc.cam[2]};
        d = lc.view.apply(d0);
        return;
    }
    double lx, ly;
    lens_offset(s, i, j, &lx, &ly);
    const double k = lc.focus / (-d0.z);
    const Vec3<double> P = {d0.x * k, d0.y * k, d0.z * k};
    const double Lx = lc.aperture * lx, Ly = lc.aperture * ly;
    const Vec3<double> e = normalized(Vec3<double>{P.x - Lx, P.y - Ly, P.z});
    const double* m = lc.view.m;
    o = {lc.cam[0] + (m[0] * Lx + m[3] * Ly), lc.cam[1] + (m[1] * Lx + m[4] * Ly), lc.cam[2] + (m[2] * Lx + m[5] * Ly)};
    d = lc.view.apply(e);
}

// Spherical area lights (rm_render_area_lights, include/rm_b200.h RmAreaLights).  R = double is the normative definition
// (no fused multiply-add: the library is compiled with -fmad=false); R = float is the production path's FP32 restatement.
// The kernel, the host emulation and the tests all call these two functions.
// light_frame: an orthonormal basis (m, t1, t2) around the unit vector m, branch-free and defined for every unit m
// (Duff et al. 2017, "Building an orthonormal basis, revisited").
template <typename R> RM_HD void light_frame(const Vec3<R> m, Vec3<R>& t1, Vec3<R>& t2) {
    const R sigma = copysign(R(1), m.z);
    const R alpha = R(-1) / (sigma + m.z);
    const R beta = (m.x * m.y) * alpha;
    t1 = {R(1) + ((sigma * m.x) * m.x) * alpha, sigma * beta, -sigma * m.x};
    t2 = {beta, sigma + (m.y * m.y) * alpha, -m.y};
}
// light_sample: the point q = c + r ((lx t1) + (ly t2)) of the disc of radius r through the light's centre c, facing the
// shading point ((lx, ly) = lens_offset(s, a, b): a point of the unit disc).
template <typename R> RM_HD Vec3<R> light_sample(const Vec3<R> c, const R r, const Vec3<R> t1, const Vec3<R> t2, const R lx, const R ly) {
    return {c.x + r * ((lx * t1.x) + (ly * t2.x)), c.y + r * ((lx * t1.y) + (ly * t2.y)), c.z + r * ((lx * t1.z) + (ly * t2.z))};
}

constexpr int kAreaMaxSamples = 8;
// The call's lights as the FP32 path reads them: radius[l] > 0 for an area light (a positive radius too small for FP32 is
// kept at 1e-30, so the light stays one of s^2 points), 0 for the reference's point light; off: the unit-disc points
// (lx, ly) = lens_offset(s, a, b) of sample a s + b, rounded to FP32; inv_ss = 1 / (s * s) in FP32.
struct AreaLights {
    const float* radius;
    float off[2 * kAreaMaxSamples * kAreaMaxSamples];
    int samples;
    float inv_ss;
};

// Rough glass (rm_render_rough_glass, include/rm_b200.h RmRoughGlass).  R = double is the normative definition (no fused
// multiply-add); R = float is the GLASS_F32 path's FP32 restatement.  The kernel, the host emulation and the tests all call
// these functions.
// rough_dir: a ray direction rd spawned at a glass-like hit of roughness g, turned by the unit-disc point (lx, ly) in the
// plane orthogonal to rd (light_frame's basis): normalized(rd + g ((lx t1) + (ly t2))).  The offset is orthogonal to rd and
// at most 1 long, so the result lies within atan(g) of rd.  g = 0 or (lx, ly) = (0, 0) leave rd as it is, bit for bit.
template <typename R> RM_HD Vec3<R> rough_dir(const Vec3<R> rd, const R g, const R lx, const R ly) {
    if (!(g > R(0)) || (lx == R(0) && ly == R(0))) return rd;
    Vec3<R> t1, t2;
    light_frame<R>(rd, t1, t2);
    return normalized(Vec3<R>{rd.x + g * ((lx * t1.x) + (ly * t2.x)), rd.y + g * ((lx * t1.y) + (ly * t2.y)),
                              rd.z + g * ((lx * t1.z) + (ly * t2.z))});
}
// The origin of a turned ray, by the rule of the function that spawned it applied to the new direction rd:
// reflect_ray's (optics.rs:41-45) against the hit normal, refract_ray's (optics.rs:82-86) against the normal turned against
// the incident ray.
template <typename R> RM_HD Vec3<R> rough_reflect_origin(const Vec3<R> point, const Vec3<R> hit_normal, const Vec3<R> rd) {
    return dot(rd, hit_normal) < R(0) ? axmy(point, hit_normal, R(1e-4)) : axpy(point, hit_normal, R(1e-4));
}
template <typename R>
RM_HD Vec3<R> rough_refract_origin(const Vec3<R> point, const Vec3<R> hit_normal, const Vec3<R> incident, const Vec3<R> rd) {
    const Vec3<R> normal = -dot(hit_normal, incident) < R(0) ? -hit_normal : hit_normal;
    return dot(rd, normal) > R(0) ? axpy(point, normal, R(1e-4)) : axmy(point, normal, R(1e-4));
}
// The unit-disc point of sample (i, j) of s x s at recursion level L (1 = the sample ray's own hit): lens_offset(s,
// (j + L) mod s, i), the stratum ((i + j + L) mod s, i) -- a bijection over the s^2 samples at every level, shifted per
// level and different from the lens's strata.
RM_HD void rough_offset(const int s, const int i, const int j, const int level, double* lx, double* ly) {
    lens_offset(s, (j + level) % s, i, lx, ly);
}
// The call's roughness as the kernel reads it: g[id] per primitive id in FP32 (a positive value too small for FP32 is kept
// at 1e-30, so that it stays positive); off: lens_offset(s, a, b) of stratum a s + b in f64, and rounded to FP32 in off32.
struct RoughGlass {
    const float* g;
    double off[2 * kAreaMaxSamples * kAreaMaxSamples];
    float off32[2 * kAreaMaxSamples * kAreaMaxSamples];
    int samples;
};

// Motion blur (rm_render_motion, include/rm_b200.h RmMotion).  The time of sample (i, j) of s x s: stratum
// m = s ((2i + j) mod s) + ((i + j) mod s) -- a bijection onto [0, s^2), since (a - b) mod s = i -- and
// tau = (m + 0.5) / s^2 - 0.5, in (-1/2, 1/2), symmetric about 0, and 0 at s = 1.  f64 without fused multiply-add; the
// kernel, the host emulation and the tests all call it.
RM_HD double motion_time(const int s, const int i, const int j) {
    const int m = s * ((2 * i + j) % s) + (i + j) % s;
    return ((double)m + 0.5) / (double)(s * s) - 0.5;
}
// The call's motion as the kernel reads it: the FP32 displacement {v, 0} of every primitive by the kernel's own indices --
// sphere i, fast-path triangle j, plane slot i of the generic arrays (the layout's full lists, so that culling changes no
// index) -- and the time of sample q = i s + j in f64 and rounded to FP32.
struct Motion {
    const R4<float>* v_sph;
    const R4<float>* v_tri;
    const R4<float>* v_pln;
    double tau[kAreaMaxSamples * kAreaMaxSamples];
    float tau32[kAreaMaxSamples * kAreaMaxSamples];
    int samples;
};

// Distributed ray tracing (rm_render_distributed, include/rm_b200.h).  The light point of sample (i, j) of s x s at a shading
// point of recursion level L: the unit-disc point (lens_offset's elliptical grid map) of the stratum
// (a, b) = ((i + 2j + L) mod s, (i + 3j) mod s).  The map (i, j) -> (a, b) has determinant 1 over Z_s, a bijection over the s^2
// samples at every level; (0, 0) at s = 1.  f64 without fused multiply-add; the kernel, the host emulation and the tests all
// call it.
RM_HD void area_offset(const int s, const int i, const int j, const int level, double* lx, double* ly) {
    const int a = (i + 2 * j + level) % s, b = (i + 3 * j) % s;
    lens_offset(s, (a - b + s) % s, b, lx, ly);                // lens_offset's stratum ((a - b) + b, b) mod s = (a, b)
}
// The call's area lights as the distributed kernel reads them: radius[l] as AreaLights has it; off[2 (a s + b)]: the unit-disc
// point of stratum (a, b) rounded to FP32.
struct AreaPoints {
    const float* radius;
    float off[2 * kAreaMaxSamples * kAreaMaxSamples];
    int samples;
};

// Diffuse interreflection (rm_render_indirect, include/rm_b200.h).  The normative definition in f64 without fused
// multiply-add; the kernel, the host emulation and the tests all call these functions.
// diffuse_point: the Shirley-Chiu concentric map (1997) of the centre of stratum (a, b) of s x s, (p, q) = ((2a + 1) / s - 1,
// (2b + 1) / s - 1), to the unit disc.  Equal-area, so Malley's lift of the points to the hemisphere is cosine-weighted.  It
// needs cos and sin, whose host and device results may differ, so it is evaluated on the host only (the kernel reads a table).
inline void diffuse_point(const int s, const int a, const int b, double* lx, double* ly) {
    const double p = (2. * a + 1.) / s - 1., q = (2. * b + 1.) / s - 1.;
    const double quarter_pi = 3.14159265358979323846 / 4.;
    if (p == 0. && q == 0.) {
        *lx = 0.;
        *ly = 0.;
        return;
    }
    double r, phi;
    if (fabs(p) > fabs(q)) {
        r = p;
        phi = quarter_pi * (q / p);
    } else {
        r = q;
        phi = 3.14159265358979323846 / 2. - quarter_pi * (p / q);
    }
    *lx = r * cos(phi);
    *ly = r * sin(phi);
}
// The stratum of sample (i, j) of s x s at recursion level L (1 = the sample ray's own hit): (a, b) = ((2i + 3j + L) mod s,
// (3i + 5j) mod s), a map of determinant 1 over Z_s, so a bijection over the s^2 samples at every level.
RM_HD int diffuse_stratum(const int s, const int i, const int j, const int level) {
    return ((2 * i + 3 * j + level) % s) * s + (3 * i + 5 * j) % s;
}
inline void diffuse_offset(const int s, const int i, const int j, const int level, double* lx, double* ly) {
    const int k = diffuse_stratum(s, i, j, level);
    diffuse_point(s, k / s, k % s, lx, ly);
}
// The hit normal turned against the incident ray d: n if dot(n, d) < 0, else -n.
template <typename R> RM_HD Vec3<R> diffuse_normal(const Vec3<R> n, const Vec3<R> d) { return dot(n, d) < R(0) ? n : -n; }
// The bounce direction around the facing normal nf: Malley's lift of the disc point (lx, ly) in light_frame's basis,
// normalized(((lx t1) + (ly t2)) + z nf) with z = sqrt(1 - ((lx lx) + (ly ly))), component by component in that order.
template <typename R> RM_HD Vec3<R> diffuse_dir(const Vec3<R> nf, const R lx, const R ly) {
    Vec3<R> t1, t2;
    light_frame<R>(nf, t1, t2);
    const R z = Num<R>::sqrt_(R(1) - ((lx * lx) + (ly * ly)));
    return normalized(Vec3<R>{((lx * t1.x) + (ly * t2.x)) + z * nf.x, ((lx * t1.y) + (ly * t2.y)) + z * nf.y,
                              ((lx * t1.z) + (ly * t2.z)) + z * nf.z});
}
// The bounce ray's origin: point + nf 1e-4, reflect_ray's offset (optics.rs:41-45).
template <typename R> RM_HD Vec3<R> diffuse_origin(const Vec3<R> point, const Vec3<R> nf) { return axpy(point, nf, R(1e-4)); }
// The call's bounce points as the kernel reads them: off[2 (a s + b)] = diffuse_point(s, a, b) in f64, and rounded to FP32
// in off32.
struct Diffuse {
    double off[2 * kAreaMaxSamples * kAreaMaxSamples];
    float off32[2 * kAreaMaxSamples * kAreaMaxSamples];
    int samples;
};

}  // namespace rm
