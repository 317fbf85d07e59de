// rm_scene.cpp -- see rm_scene.h.
#include "rm_scene.h"

#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstddef>
#include <cstring>
#include <memory>
#include <thread>

namespace rm {

RmFlatScene OwnedFlatScene::view() const {
    RmFlatScene fs{};
    fs.n_shapes = (int32_t)shapes.size();
    fs.shapes = shapes.data();
    fs.n_spheres = (int32_t)spheres.size();
    fs.spheres = spheres.data();
    fs.n_polygons = (int32_t)polygons.size();
    fs.polygons = polygons.data();
    fs.n_polygon_vertices = (int32_t)(polygon_vertices.size() / 3);
    fs.polygon_vertices = polygon_vertices.data();
    fs.n_objs = (int32_t)objs.size();
    fs.objs = objs.data();
    fs.n_triangles = (int32_t)triangles.size();
    fs.triangles = triangles.data();
    fs.triangle_reflectances = triangle_reflectances.data();
    fs.n_lights = (int32_t)lights.size();
    fs.lights = lights.data();
    return fs;
}

void OwnedFlatScene::assign(const RmFlatScene& fs, HostPool* pool) {
    auto copy_large = [&](auto& dst, const auto* src, size_t n) {
        dst.resize(n);
        const size_t bytes = n * sizeof(dst[0]), kBlock = 1 << 20;
        const int n_blocks = (int)((bytes + kBlock - 1) / kBlock);
        auto one = [&](int k) {
            const size_t at = (size_t)k * kBlock;
            std::memcpy(reinterpret_cast<char*>(dst.data()) + at, reinterpret_cast<const char*>(src) + at, std::min(kBlock, bytes - at));
        };
        if (pool && n_blocks >= 4) pool->run(n_blocks, one);
        else for (int k = 0; k < n_blocks; k++) one(k);
    };
    shapes.assign(fs.shapes, fs.shapes + fs.n_shapes);
    spheres.assign(fs.spheres, fs.spheres + fs.n_spheres);
    polygons.assign(fs.polygons, fs.polygons + fs.n_polygons);
    polygon_vertices.assign(fs.polygon_vertices, fs.polygon_vertices + 3 * (size_t)fs.n_polygon_vertices);
    objs.assign(fs.objs, fs.objs + fs.n_objs);
    copy_large(triangles, fs.triangles, (size_t)fs.n_triangles);
    copy_large(triangle_reflectances, fs.triangle_reflectances, (size_t)fs.n_triangles);
    lights.assign(fs.lights, fs.lights + fs.n_lights);
}

int validate_scene(const RmFlatScene& fs, std::string& err) {
    auto bad = [&](const char* m) { err = m; return (int)RM_ERR_SCENE; };
    if (fs.n_shapes < 0 || fs.n_spheres < 0 || fs.n_polygons < 0 || fs.n_polygon_vertices < 0 || fs.n_objs < 0 ||
        fs.n_triangles < 0 || fs.n_lights < 0)
        return bad("negative count in RmFlatScene");
    if ((fs.n_shapes && !fs.shapes) || (fs.n_spheres && !fs.spheres) || (fs.n_polygons && !fs.polygons) ||
        (fs.n_polygon_vertices && !fs.polygon_vertices) || (fs.n_objs && !fs.objs) ||
        (fs.n_triangles && (!fs.triangles || !fs.triangle_reflectances)) || (fs.n_lights && !fs.lights)) {
        err = "null array with non-zero count in RmFlatScene";
        return RM_ERR_INVALID_ARGUMENT;
    }
    for (int s = 0; s < fs.n_shapes; s++) {
        const RmShapeRef& r = fs.shapes[s];
        switch (r.kind) {
            case RM_SHAPE_SPHERE:
                if (r.index < 0 || r.index >= fs.n_spheres) return bad("shape refers to a sphere out of range");
                break;
            case RM_SHAPE_POLYGON: {
                if (r.index < 0 || r.index >= fs.n_polygons) return bad("shape refers to a polygon out of range");
                const RmPolygon& p = fs.polygons[r.index];
                if (p.n_vertices < 3) return bad("polygon with fewer than 3 vertices (polygon.rs:18)");
                if (p.first_vertex < 0 || p.first_vertex + p.n_vertices > fs.n_polygon_vertices)
                    return bad("polygon vertex range out of bounds");
                break;
            }
            case RM_SHAPE_OBJ: {
                if (r.index < 0 || r.index >= fs.n_objs) return bad("shape refers to an obj out of range");
                const RmObj& o = fs.objs[r.index];
                if (o.n_triangles < 0 || o.first_triangle < 0 || o.first_triangle + o.n_triangles > fs.n_triangles)
                    return bad("obj triangle range out of bounds");
                break;
            }
            default:
                return bad("unknown shape kind");
        }
    }
    return RM_OK;
}

namespace {

template <typename R> R pred_1e6();
template <> double pred_1e6<double>() { return std::nextafter(1e-6, 0.); }
template <> float pred_1e6<float>() { return std::nextafterf(1e-6f, 0.f); }

int align32(int x) { return (x + 31) & ~31; }

// A planar primitive while it is being packed: views of the caller's f64 arrays (nothing is copied or allocated per
// primitive -- a scene of 10^5 triangles is packed in the time its first frame takes).
struct PlaneTmp {
    const double* n;    // plane normal (triangle.rs:33-47 / polygon.rs:16-42: precomputed by the caller)
    const double* c;    // plane point
    const double* v;    // vertices, x y z each; only x and y are ever read (triangle.rs:13-15)
    int nv;
    int id, shape;
    int src;            // index of the RmPolygon / RmTriangle it views
    int cls;            // 0 hittable, 1 back-facing (projected winding clockwise), 2 degenerate projection
    bool is_triangle;   // an Obj's triangle: threshold 1e-6 on d.n (triangle.rs:61); a polygon tests == 0 (polygon.rs:67)
    double x(size_t i) const { return v[3 * i]; }
    double y(size_t i) const { return v[3 * i + 1]; }
};

// A planar primitive is hit only if every edge term ((v_i-p) x (v_i+1-p)).z is > 0
// (triangle.rs:13-15,72-76).  Their sum over the closed polygon equals 2*signed area of the
// XY-projected polygon for ANY p, so in exact arithmetic
//   class 1: clockwise projected winding (area < 0)  -> some term is < 0 -> never hit;
//   class 2: degenerate projection (normal.z == 0, area == 0) -> every term is exactly 0 for a point of
//            the plane -> `> 0` fails -> never hit.  The reference's f64 evaluation of such a primitive
//            is pure rounding noise with a common-mode error that keeps the three terms from being
//            positive together (0 hits on every test scene, checked against the oracle in tests/).
// "Degenerate" is judged at the resolution of the arithmetic that will evaluate the edge terms: for
// f64 only an (almost) exactly zero area; for f32 also slivers whose projected area is below 1e-6 of
// their squared perimeter (e.g. the dodecahedron faces whose normal.z is 5e-9 because tobj rounds
// vertices to f32): their edge terms are smaller than FP32 rounding noise, and no pixel ray of any
// test scene passes through such a sliver in the reference either.
int classify_plane(const PlaneTmp& p, bool single_precision) {
    const size_t n = (size_t)p.nv;
    double area2 = 0., scale = 0., perimeter = 0.;
    for (size_t i = 0; i < n; i++) {
        const size_t j = (i + 1) % n;
        area2 += p.x(i) * p.y(j) - p.y(i) * p.x(j);
        scale = std::fmax(scale, std::fmax(std::fabs(p.x(i)), std::fabs(p.y(i))));
        perimeter += std::hypot(p.x(j) - p.x(i), p.y(j) - p.y(i));
    }
    double tol = 1e-9 * scale * scale;
    if (single_precision) tol = std::fmax(tol, 1e-6 * perimeter * perimeter);
    if (area2 > tol) return 0;
    return (area2 < -tol) ? 1 : 2;
}

template <typename R> R4<R> mk4(double x, double y, double z, double w) { return {(R)x, (R)y, (R)z, (R)w}; }

// f64 layout: the reference's own operands -- plane point and the x,y of every vertex.
void write_plane(const PlaneTmp& p, R4<double>& c4, R2<double>* vert) {
    c4 = {p.c[0], p.c[1], p.c[2], 0.};
    for (size_t v = 0; v < (size_t)p.nv; v++) vert[v] = {p.x(v), p.y(v)};
}
// f32 layout: n.C and the affine edge functions about vertex 0, all folded in f64 and then rounded
// once (see plane_intersect<float> in rm_trace.cuh).
// edge function i of a plane about its vertex 0, in f64: e_i(q) = A*q.x + B*q.y + C, q = p - v0
void edge_about_v0(const PlaneTmp& p, size_t i, double& A, double& B, double& C) {
    const size_t nv = (size_t)p.nv, j = (i + 1) % nv;
    const double x0 = p.x(0), y0 = p.y(0);
    const double ax = p.x(i) - x0, ay = p.y(i) - y0;
    const double bx = p.x(j) - x0, by = p.y(j) - y0;
    A = ay - by;
    B = bx - ax;
    C = ax * by - ay * bx;
}
double plane_dn(const PlaneTmp& p) { return p.c[0] * p.n[0] + p.c[1] * p.n[1] + p.c[2] * p.n[2]; }

void write_plane(const PlaneTmp& p, R4<float>& k4, R4<float>* edge) {
    k4 = {(float)plane_dn(p), (float)p.x(0), (float)p.y(0), 0.f};
    for (size_t i = 0; i < (size_t)p.nv; i++) {
        double A, B, C;
        edge_about_v0(p, i, A, B, C);
        edge[i] = {(float)A, (float)B, (float)C, 0.f};
    }
}

// fast-path records of a 3-vertex plane: FP64 source for prepare_raster and the FP32 general-ray record
void write_triangle(const PlaneTmp& p, double* src, R4<float>* g) {
    double A[3], B[3], C[3];
    for (size_t i = 0; i < 3; i++) edge_about_v0(p, i, A[i], B[i], C[i]);   // C[0] == C[2] == 0: both edges touch vertex 0
    const double dn = plane_dn(p);
    const float thr = p.is_triangle ? std::nextafterf(1e-6f, 0.f) : 0.f;
    const double s[kTriSrcDoubles] = {p.n[0], p.n[1], p.n[2], dn, p.x(0), p.y(0), A[0], B[0], A[1], B[1], C[1],
                                      A[2], B[2], (double)thr, (double)p.id, 0.};
    std::memcpy(src, s, sizeof s);
    float idf;
    std::memcpy(&idf, &p.id, 4);
    g[0] = {(float)p.n[0], (float)p.n[1], (float)p.n[2], (float)dn};
    g[1] = {(float)p.x(0), (float)p.y(0), (float)A[0], (float)B[0]};
    g[2] = {(float)A[1], (float)B[1], (float)C[1], (float)A[2]};
    g[3] = {(float)B[2], thr, idf, 0.f};
}
// Bounds of the region a planar primitive can be hit in: the points of its plane whose XY projection lies inside the
// XY-projected polygon (triangle.rs:13-15,72-76 only ever look at x and y).  z is affine in (x, y) on the plane, so its
// range over the polygon is its range over the vertices; taken from the plane equation rather than from the vertices'
// own z, so that the box bounds what the intersection routine accepts even for a caller-supplied normal / plane point.
BvhPrimBox plane_bounds(const PlaneTmp& p, int code) {
    BvhPrimBox b;
    b.code = code;
    for (int a = 0; a < 3; a++) {
        b.lo[a] = INFINITY;
        b.hi[a] = -INFINITY;
    }
    for (size_t v = 0; v < (size_t)p.nv; v++) {
        const double x = p.x(v), y = p.y(v);
        const double z = p.c[2] - (p.n[0] * (x - p.c[0]) + p.n[1] * (y - p.c[1])) / p.n[2];   // non-finite for n.z == 0: unbounded box
        const double q[3] = {x, y, z};
        for (int a = 0; a < 3; a++) {
            b.lo[a] = std::fmin(b.lo[a], q[a]);      // fmin/fmax drop a NaN; build_bvh() treats lo > hi as unbounded
            b.hi[a] = std::fmax(b.hi[a], q[a]);
            if (!std::isfinite(q[a])) {
                b.lo[a] = -INFINITY;
                b.hi[a] = INFINITY;
            }
        }
    }
    return b;
}

// items [0, n) in blocks of kPackBlock on the pool's threads (in place when the pool has none)
constexpr size_t kPackBlock = 2048;
template <typename F> void for_blocks(HostPool& pool, size_t n, const F& body) {
    const int n_blocks = (int)((n + kPackBlock - 1) / kPackBlock);
    pool.run(n_blocks, [&](int b) { body((size_t)b * kPackBlock, std::min(n, (size_t)(b + 1) * kPackBlock)); });
}

template <typename R> void write_fast(const Buf<PlaneTmp>&, BlobLayout&, unsigned char*, PackedScene<R>&, HostPool&) {}
template <> void write_fast<float>(const Buf<PlaneTmp>& pln, BlobLayout& L, unsigned char* b, PackedScene<float>& out, HostPool& pool) {
    auto* g = reinterpret_cast<R4<float>*>(b + L.off_tri_g);
    auto* slot = reinterpret_cast<int*>(b + L.off_poly_slot);
    out.tri_src.resize((size_t)L.n_tri * kTriSrcDoubles + kTriSrcDoubles);      // every record is written in full below
    std::fill(out.tri_src.end() - kTriSrcDoubles, out.tri_src.end(), 0.);       // one record of padding
    // planes are sorted hittable | back-facing | degenerate: the hittable ones, in slot order, are the boxes after the spheres
    Buf<BvhPrimBox> boxes((size_t)L.n_sph + (size_t)L.n_pln_live);
    const auto* sph = reinterpret_cast<const R4<float>*>(b + L.off_sph);
    for (int i = 0; i < L.n_sph; i++) {
        // the sphere as the kernels see it: centre and r^2 already rounded to f32 (sphere.rs:6-11)
        const double r = std::sqrt((double)sph[i].w), c[3] = {sph[i].x, sph[i].y, sph[i].z};
        BvhPrimBox& bx = boxes[i];
        for (int a = 0; a < 3; a++) {
            bx.lo[a] = c[a] - r;
            bx.hi[a] = c[a] + r;
        }
        bx.code = (BVH_SPHERE << 30) | i;
    }
    // index of every non-degenerate plane in its list: triangle records / polygon slots
    Buf<int> index(pln.size());
    int t = 0, k = 0;
    for (size_t i = 0; i < pln.size(); i++) {
        if (pln[i].cls == 2) continue;
        index[i] = pln[i].nv == 3 ? t++ : k++;
    }
    for_blocks(pool, pln.size(), [&](size_t begin, size_t end) {
        for (size_t i = begin; i < end; i++) {
            if (pln[i].cls == 2) continue;
            if (pln[i].nv == 3) {
                write_triangle(pln[i], out.tri_src.data() + (size_t)index[i] * kTriSrcDoubles, g + 4 * index[i]);
                if (pln[i].cls == 0) boxes[L.n_sph + i] = plane_bounds(pln[i], (BVH_TRI << 30) | index[i]);
            } else {
                if (pln[i].cls == 0) boxes[L.n_sph + i] = plane_bounds(pln[i], (int)((unsigned)BVH_POLY << 30 | (unsigned)i));
                slot[index[i]] = (int)i;
            }
        }
    });
    const auto t0 = std::chrono::steady_clock::now();
    out.bvh_depth = build_bvh(boxes, out.bvh_nodes, out.bvh_prims, &pool);
    out.hierarchy_build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    out.bvh_boxes = std::move(boxes);
}

}  // namespace

template <typename R> int pack_scene(const RmFlatScene& fs, PackedScene<R>& out, std::string& err, HostPool* shared_pool) {
    int rc = validate_scene(fs, err);
    if (rc != RM_OK) return rc;
    out = PackedScene<R>();
    // RM_B200_PACK_TRACE=1: phase times of the packing on stderr
    static const bool trace = getenv("RM_B200_PACK_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto ms_now = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    double t_collect = 0, t_sort = 0, t_blob = 0, t_fast = 0;

    // Large scenes are packed on several threads: the caller's pool, or one of this call's own.  Every primitive's
    // records depend on that primitive alone and land at indices fixed beforehand, so the result does not depend on the
    // number of threads.
    const size_t n_planar = (size_t)fs.n_polygons + (size_t)fs.n_triangles;
    std::unique_ptr<HostPool> own_pool;
    if (!shared_pool || n_planar < 8192) {
        own_pool.reset(new HostPool(n_planar < 8192 ? 1 : host_thread_count(16)));
    }
    HostPool& pool = own_pool ? *own_pool : *shared_pool;

    struct SphTmp { const RmSphere* s; int id, shape; };
    std::vector<SphTmp> sph;
    std::vector<PlaneTmp> found;      // planar primitives in scene order
    found.reserve(n_planar);
    int id = 0;
    for (int s = 0; s < fs.n_shapes; s++) {
        const RmShapeRef& ref = fs.shapes[s];
        if (ref.kind == RM_SHAPE_SPHERE) {
            sph.push_back({&fs.spheres[ref.index], id++, s});
        } else if (ref.kind == RM_SHAPE_POLYGON) {
            const RmPolygon& p = fs.polygons[ref.index];
            found.push_back({p.plane_normal, p.plane_point, fs.polygon_vertices + 3 * (size_t)p.first_vertex, p.n_vertices, id++, s, ref.index, 0, false});
        } else {
            const RmObj& o = fs.objs[ref.index];
            for (int k = 0; k < o.n_triangles; k++) {
                const RmTriangle& tr = fs.triangles[o.first_triangle + k];
                found.push_back({tr.normal, tr.center, tr.vertices, 3, id++, s | (1 << 30), o.first_triangle + k, 0, true});
            }
        }
    }
    out.n_prims = id;
    // materials by primitive id
    out.mat_a.resize((size_t)id);
    out.mat_b.resize((size_t)id);
    out.mat_f.resize((size_t)id);
    auto put_material = [&](int at, const RmReflectance& r) {
        out.mat_a[at] = mk4<R>(r.diffuse_color[0], r.diffuse_color[1], r.diffuse_color[2], r.diffusion);
        out.mat_b[at] = mk4<R>(r.specular, r.specular_exponent, r.reflection, r.refractive_index);
        out.mat_f[at] = r.is_glass_like ? 1 : 0;
    };
    for (auto& sp : sph) put_material(sp.id, sp.s->reflectance);
    // per block: class of every plane, largest coordinate magnitude, any glass
    const size_t n_found = found.size();
    std::vector<double> block_cm((n_found + kPackBlock - 1) / kPackBlock + 1, 0.);
    for_blocks(pool, n_found, [&](size_t begin, size_t end) {
        double cm = 0.;
        for (size_t i = begin; i < end; i++) {
            PlaneTmp& t = found[i];
            t.cls = classify_plane(t, sizeof(R) == 4);
            for (int v = 0; v < t.nv; v++) cm = std::fmax(cm, std::fmax(std::fabs(t.x(v)), std::fabs(t.y(v))));
            cm = std::fmax(cm, std::fabs(t.c[2]));
            put_material(t.id, t.is_triangle ? fs.triangle_reflectances[t.src] : fs.polygons[t.src].reflectance);
        }
        block_cm[begin / kPackBlock] = cm;
    });
    t_collect = ms_now();
    for (int f : out.mat_f) out.lay.any_glass |= f & 1;
    {
        double cm = 0., rmin = INFINITY;
        for (auto& sp : sph) {
            const double r = std::sqrt(sp.s->radius_square);
            for (int a = 0; a < 3; a++) cm = std::fmax(cm, std::fabs(sp.s->center[a]) + r);
            rmin = std::fmin(rmin, r);
        }
        for (double v : block_cm) cm = std::fmax(cm, v);
        out.lay.coord_max = cm;
        out.lay.r_min = sph.empty() ? 0. : rmin;
    }

    // hittable planes first, then back-facing, then degenerate (stable: scene order inside each class)
    Buf<PlaneTmp> pln(n_found);
    {
        size_t at[3] = {0, 0, 0};
        for (const PlaneTmp& t : found) at[t.cls]++;
        at[2] = at[0] + at[1];
        at[1] = at[0];
        at[0] = 0;
        for (const PlaneTmp& t : found) pln[at[t.cls]++] = t;
    }
    found = std::vector<PlaneTmp>();

    t_sort = ms_now();
    BlobLayout& L = out.lay;
    L.n_sph = (int)sph.size();
    L.n_pln = (int)pln.size();
    L.n_pln_live = 0;
    L.n_pln_nondegenerate = 0;
    L.n_vert = 0;
    for (auto& p : pln) {
        L.n_pln_live += p.cls == 0 ? 1 : 0;
        L.n_pln_nondegenerate += p.cls != 2 ? 1 : 0;
        L.n_vert += p.nv;
    }
    L.n_lgt = fs.n_lights;
    if (sizeof(R) == 4) {
        for (auto& p : pln) {
            if (p.cls == 2) continue;
            const bool tri = p.nv == 3;
            (tri ? L.n_tri : L.n_poly)++;
            if (p.cls == 0) (tri ? L.n_tri_live : L.n_poly_live)++;
        }
    }
    int off = 0;
    L.off_sph = off;    off = align32(off + L.n_sph * (int)sizeof(R4<R>));
    L.off_pln_n = off;  off = align32(off + L.n_pln * (int)sizeof(R4<R>));
    L.off_pln_c = off;  off = align32(off + L.n_pln * (int)sizeof(R4<R>));
    L.off_vert = off;   off = align32(off + L.n_vert * (int)sizeof(VertT<R>));
    L.off_lgt_p = off;  off = align32(off + L.n_lgt * (int)sizeof(R4<R>));
    L.off_lgt_c = off;  off = align32(off + L.n_lgt * (int)sizeof(R4<R>));
    L.off_pln_v = off;  off = align32(off + L.n_pln * (int)sizeof(I2));
    L.off_sph_id = off; off = align32(off + L.n_sph * (int)sizeof(int));
    L.off_pln_id = off; off = align32(off + L.n_pln * (int)sizeof(int));
    L.off_tri_g = off;  off = align32(off + L.n_tri * 4 * (int)sizeof(R4<float>));
    L.off_poly_slot = off; off = align32(off + L.n_poly * (int)sizeof(int));
    L.bytes = std::max(off, 32);
    out.blob.resize((size_t)L.bytes / 32);
    unsigned char* b = reinterpret_cast<unsigned char*>(out.blob.data());
    for_blocks(pool, (size_t)L.bytes / 32, [&](size_t begin, size_t end) { std::memset(b + 32 * begin, 0, 32 * (end - begin)); });   // padding included
    auto* b_sph = reinterpret_cast<R4<R>*>(b + L.off_sph);
    auto* b_pn = reinterpret_cast<R4<R>*>(b + L.off_pln_n);
    auto* b_pc = reinterpret_cast<R4<R>*>(b + L.off_pln_c);
    auto* b_v = reinterpret_cast<VertT<R>*>(b + L.off_vert);
    auto* b_lp = reinterpret_cast<R4<R>*>(b + L.off_lgt_p);
    auto* b_lc = reinterpret_cast<R4<R>*>(b + L.off_lgt_c);
    auto* b_pv = reinterpret_cast<I2*>(b + L.off_pln_v);
    auto* b_sid = reinterpret_cast<int*>(b + L.off_sph_id);
    auto* b_pid = reinterpret_cast<int*>(b + L.off_pln_id);

    for (int i = 0; i < L.n_sph; i++) {
        const RmSphere& s = *sph[i].s;
        b_sph[i] = mk4<R>(s.center[0], s.center[1], s.center[2], s.radius_square);
        b_sid[i] = sph[i].id;
    }
    {
        int v0 = 0;
        for (int i = 0; i < L.n_pln; i++) {
            b_pv[i] = {v0, pln[i].nv};
            v0 += pln[i].nv;
        }
    }
    for_blocks(pool, (size_t)L.n_pln, [&](size_t begin, size_t end) {
        for (size_t i = begin; i < end; i++) {
            const PlaneTmp& p = pln[i];
            const R thr = p.is_triangle ? pred_1e6<R>() : R(0);
            b_pn[i] = {(R)p.n[0], (R)p.n[1], (R)p.n[2], thr};
            write_plane(p, b_pc[i], b_v + b_pv[i].x);
            b_pid[i] = p.id;
        }
    });
    t_blob = ms_now();
    write_fast<R>(pln, L, b, out, pool);
    t_fast = ms_now();
    if (sizeof(R) == 4) {
        // f64 sources for the refinement of winning hits on glass paths (cast_glass, rm_fast.cuh): spheres {c, r^2}
        // (sphere.rs:6-11) and planes by slot {n, n.C} (triangle.rs:33-47 / polygon.rs:16-42: precomputed normal, plane point)
        out.sph64.resize((size_t)L.n_sph * 4 + 4);
        std::fill(out.sph64.end() - 4, out.sph64.end(), 0.);
        for (int i = 0; i < L.n_sph; i++) {
            const RmSphere& sp = *sph[i].s;
            const double q[4] = {sp.center[0], sp.center[1], sp.center[2], sp.radius_square};
            std::memcpy(out.sph64.data() + 4 * (size_t)i, q, sizeof q);
        }
        out.pln64.resize((size_t)L.n_pln * 4 + 4);
        std::fill(out.pln64.end() - 4, out.pln64.end(), 0.);
        for_blocks(pool, (size_t)L.n_pln, [&](size_t begin, size_t end) {
            for (size_t i = begin; i < end; i++) {
                const double q[4] = {pln[i].n[0], pln[i].n[1], pln[i].n[2], plane_dn(pln[i])};
                std::memcpy(out.pln64.data() + 4 * i, q, sizeof q);
            }
        });
    }
    for (int l = 0; l < L.n_lgt; l++) {
        const RmLight& lg = fs.lights[l];
        b_lp[l] = mk4<R>(lg.position[0], lg.position[1], lg.position[2], lg.intensity);
        b_lc[l] = mk4<R>(lg.color[0], lg.color[1], lg.color[2], 0.);
    }

    // scene-order lists for the instrumented kernel: slots by primitive id (ids are 0 .. n_prims-1, each once)
    std::vector<int> slot_of((size_t)out.n_prims), shape_of((size_t)out.n_prims);
    for (int i = 0; i < L.n_sph; i++) {
        slot_of[sph[i].id] = i;
        shape_of[sph[i].id] = sph[i].shape;
    }
    for (int i = 0; i < L.n_pln; i++) {
        slot_of[pln[i].id] = L.n_sph + i;
        shape_of[pln[i].id] = pln[i].shape;
    }
    const int keep0 = plane_count<R>(L, false), keep1 = plane_count<R>(L, true);
    out.order[0].reserve((size_t)L.n_sph + keep0);
    out.order_shape[0].reserve((size_t)L.n_sph + keep0);
    out.order[1].reserve((size_t)L.n_sph + keep1);
    out.order_shape[1].reserve((size_t)L.n_sph + keep1);
    for (int e = 0; e < out.n_prims; e++) {
        const int slot = slot_of[e];
        if (slot < L.n_sph || (slot - L.n_sph) < keep0) {
            out.order[0].push_back(slot);
            out.order_shape[0].push_back(shape_of[e]);
        }
        if (slot < L.n_sph || (slot - L.n_sph) < keep1) {
            out.order[1].push_back(slot);
            out.order_shape[1].push_back(shape_of[e]);
        }
    }
    if (trace)
        std::fprintf(stderr, "rm pack (%s, %d primitives): collected %.1f ms, classes sorted %.1f, blob written %.1f, fast records + hierarchy %.1f (hierarchy alone %.1f), done %.1f\n",
                     sizeof(R) == 4 ? "f32" : "f64", out.n_prims, t_collect, t_sort, t_blob, t_fast, out.hierarchy_build_ms, ms_now());
    return RM_OK;
}

template int pack_scene<float>(const RmFlatScene&, PackedScene<float>&, std::string&, HostPool*);
template int pack_scene<double>(const RmFlatScene&, PackedScene<double>&, std::string&, HostPool*);

template <typename R> FrameParams<R> make_frame_params(const RmParams& p) {
    FrameParams<R> fp{};
    fp.width = p.width;
    fp.height = p.height;
    const int patch = 32;
    int n_rows = p.height / patch;                          // renderer.rs:53: rows >= floor(H/32)*32 are never rendered
    int r0 = p.patch_row_begin < 0 ? 0 : p.patch_row_begin;
    int r1 = (p.patch_row_end < 0 || p.patch_row_end > n_rows) ? n_rows : p.patch_row_end;
    if (r0 > r1) r0 = r1;
    const int stride = p.patch_row_stride < 1 ? 1 : p.patch_row_stride;
    fp.row_begin = r0 * patch;
    fp.row_end = r1 * patch;
    fp.row_step = stride * patch;
    fp.n_bands = (r1 - r0 + stride - 1) / stride;
    // renderer.rs:25-33
    const double half_fov = std::tan(p.fov / 2.);
    const double width = (double)p.width, height = (double)p.height;
    const double ratio = width / height;
    fp.width_r = (R)width;
    fp.height_r = (R)height;
    fp.half_fov = (R)half_fov;
    fp.ratio = (R)ratio;
    fp.half_w = (R)(width / 2.);
    fp.half_h = (R)(height / 2.);
    fp.sx = (R)(2. * half_fov * ratio / width);
    fp.sy = (R)(-2. * half_fov / height);
    fp.camera = {(R)p.camera[0], (R)p.camera[1], (R)p.camera[2]};
    fp.background = (R)p.background;
    fp.max_depth = p.max_depth < 0 ? 0 : (p.max_depth > kMaxDepth ? kMaxDepth : p.max_depth);
    fp.accel = p.accel == 2 ? 2 : (p.accel != 0 ? 1 : 0);     // 2: the hierarchy kernel that also counts its work
    for (int a = 0; a < 3; a++) fp.cam64[a] = p.camera[a];
    fp.w64 = width;
    fp.h64 = height;
    fp.hf64 = half_fov;
    fp.ratio64 = ratio;
    fp.inv_w64 = 1. / width;
    fp.inv_h64 = 1. / height;
    return fp;
}

template FrameParams<float> make_frame_params<float>(const RmParams&);
template FrameParams<double> make_frame_params<double>(const RmParams&);

// The normative construction of include/rm_b200.h (RmView), in f64 without contraction (-ffp-contract=off / -fmad=false):
// geometry.rs's normalized is scale(1 / norm), norm = sqrt(x*x + y*y + z*z), and cross is geometry.rs:57-63.
int view_basis(const RmView& view, double out[9], const char** err) {
    const double* f = view.forward;
    const double* up = view.up;
    for (int a = 0; a < 3; a++)
        if (!std::isfinite(f[a]) || !std::isfinite(up[a])) {
            *err = "view: forward and up must be finite";
            return RM_ERR_INVALID_ARGUMENT;
        }
    const double ff = f[0] * f[0] + f[1] * f[1] + f[2] * f[2];
    if (ff == 0.) {
        *err = "view: forward is the zero vector";
        return RM_ERR_INVALID_ARGUMENT;
    }
    auto normalized = [](const double x, const double y, const double z, double* o) {
        const double s = 1. / std::sqrt(x * x + y * y + z * z);
        o[0] = x * s; o[1] = y * s; o[2] = z * s;
    };
    double* u = out;
    double* v = out + 3;
    double* w = out + 6;
    normalized(-f[0], -f[1], -f[2], w);
    const double cx = up[1] * w[2] - up[2] * w[1], cy = up[2] * w[0] - up[0] * w[2], cz = up[0] * w[1] - up[1] * w[0];
    const double uu = up[0] * up[0] + up[1] * up[1] + up[2] * up[2];
    if (cx * cx + cy * cy + cz * cz <= 1e-20 * uu) {
        *err = "view: up is zero or parallel to forward";
        return RM_ERR_INVALID_ARGUMENT;
    }
    normalized(cx, cy, cz, u);
    v[0] = w[1] * u[2] - w[2] * u[1];
    v[1] = w[2] * u[0] - w[0] * u[2];
    v[2] = w[0] * u[1] - w[1] * u[0];
    return RM_OK;
}

LensCamera make_lens_camera(const RmParams& p, const double* basis, const RmLens& lens) {
    LensCamera lc;
    const int s = lens.samples;
    lc.width = (double)s * p.width;
    lc.height = (double)s * p.height;
    lc.half_fov = std::tan(p.fov / 2.);                         // renderer.rs:25-33, as make_frame_params
    lc.ratio = lc.width / lc.height;
    for (int a = 0; a < 3; a++) lc.cam[a] = p.camera[a];
    for (int k = 0; k < 9; k++) {
        lc.view.m[k] = basis ? basis[k] : (k % 4 == 0 ? 1. : 0.);
        lc.view.f[k] = (float)lc.view.m[k];
    }
    lc.aperture = lens.aperture;
    lc.focus = lens.focus;
    lc.samples = s;
    return lc;
}

RoughGlass make_rough_glass(const int samples, const double* roughness, const int n, std::vector<float>& g) {
    g.assign(std::max(n, 1), 0.f);
    for (int k = 0; k < n; k++) {
        const double v = roughness[k];
        g[k] = v > 0. ? std::max((float)std::min(v, (double)FLT_MAX), 1e-30f) : 0.f;
    }
    RoughGlass rg = {};
    const int s = samples;
    for (int a = 0; a < s; a++)
        for (int b = 0; b < s; b++) {
            double lx, ly;
            lens_offset(s, a, b, &lx, &ly);
            rg.off[2 * (a * s + b)] = lx;
            rg.off[2 * (a * s + b) + 1] = ly;
            rg.off32[2 * (a * s + b)] = (float)lx;
            rg.off32[2 * (a * s + b) + 1] = (float)ly;
        }
    rg.samples = s;
    return rg;
}

void motion_displacements(const PackedScene<float>& ps, const double* disp, std::vector<R4<float>>& v, double& reach) {
    const BlobLayout& L = ps.lay;
    const unsigned char* b = ps.blob_data();
    const int* sph_id = reinterpret_cast<const int*>(b + L.off_sph_id);
    const R4<float>* tri_g = reinterpret_cast<const R4<float>*>(b + L.off_tri_g);
    const int* pln_id = reinterpret_cast<const int*>(b + L.off_pln_id);
    v.assign((size_t)L.n_sph + L.n_tri + L.n_pln + 1, R4<float>{0.f, 0.f, 0.f, 0.f});
    reach = 0.;
    auto put = [&](const size_t at, const int id) {
        const double* q = disp + 3 * (size_t)id;
        v[at] = {(float)q[0], (float)q[1], (float)q[2], 0.f};
        for (int a = 0; a < 3; a++) reach = std::fmax(reach, 0.5 * std::fabs((double)(&v[at].x)[a]));
    };
    for (int i = 0; i < L.n_sph; i++) put((size_t)i, sph_id[i]);
    for (int j = 0; j < L.n_tri; j++) {
        int id;
        std::memcpy(&id, &tri_g[4 * (size_t)j + 3].z, 4);
        put((size_t)L.n_sph + j, id);
    }
    for (int i = 0; i < L.n_pln; i++) put((size_t)L.n_sph + L.n_tri + i, pln_id[i]);
}

AreaPoints make_area_points(const int samples, const double* radius, const int n, std::vector<float>& r) {
    r.assign(std::max(n, 1), 0.f);
    for (int l = 0; l < n; l++) {
        const double v = radius[l];
        r[l] = v > 0. ? std::max((float)std::min(v, (double)FLT_MAX), 1e-30f) : 0.f;
    }
    AreaPoints ap = {};
    const int s = samples;
    for (int i = 0; i < s; i++)                                 // level 0: every stratum once, the map being a bijection
        for (int j = 0; j < s; j++) {
            double lx, ly;
            area_offset(s, i, j, 0, &lx, &ly);
            const int k = ((i + 2 * j) % s) * s + (i + 3 * j) % s;
            ap.off[2 * k] = (float)lx;
            ap.off[2 * k + 1] = (float)ly;
        }
    ap.samples = s;
    return ap;
}

Motion make_motion(const int samples) {
    Motion mo = {};
    const int s = samples;
    for (int i = 0; i < s; i++)
        for (int j = 0; j < s; j++) {
            mo.tau[i * s + j] = motion_time(s, i, j);
            mo.tau32[i * s + j] = (float)mo.tau[i * s + j];
        }
    mo.samples = s;
    return mo;
}

int build_swept_bvh(const PackedScene<float>& ps, const std::vector<R4<float>>& v, std::vector<R4<float>>& nodes, std::vector<int>& prims,
                    HostPool* pool) {
    const BlobLayout& L = ps.lay;
    Buf<BvhPrimBox> boxes(ps.bvh_boxes.size());
    for (size_t k = 0; k < boxes.size(); k++) {
        BvhPrimBox bx = ps.bvh_boxes[k];
        const unsigned kind = (unsigned)bx.code >> 30;
        const size_t i = (size_t)(bx.code & 0x3fffffff);
        const R4<float>& d = v[kind == BVH_SPHERE ? i : kind == BVH_TRI ? L.n_sph + i : (size_t)L.n_sph + L.n_tri + i];
        for (int a = 0; a < 3; a++) {
            const double h = 0.5 * std::fabs((double)(&d.x)[a]);     // tau v for tau in [-1/2, 1/2]: at most |v| / 2 either way
            bx.lo[a] -= h;
            bx.hi[a] += h;
        }
        boxes[k] = bx;
    }
    return build_bvh(boxes, nodes, prims, pool);
}

Diffuse make_diffuse(const int samples) {
    Diffuse df = {};
    const int s = samples;
    for (int a = 0; a < s; a++)
        for (int b = 0; b < s; b++) {
            double lx, ly;
            diffuse_point(s, a, b, &lx, &ly);
            df.off[2 * (a * s + b)] = lx;
            df.off[2 * (a * s + b) + 1] = ly;
            df.off32[2 * (a * s + b)] = (float)lx;
            df.off32[2 * (a * s + b) + 1] = (float)ly;
        }
    df.samples = s;
    return df;
}

}  // namespace rm
