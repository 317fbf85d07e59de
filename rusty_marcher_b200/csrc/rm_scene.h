// rm_scene.h -- host-side packing of an RmFlatScene (f64 mirrors of the reference structs)
// into the layout the kernels read.  Pure C++ (no CUDA) so the same packer feeds the device
// upload and the dev-time CPU emulation of the kernel code.
//
// HBM layout.  Everything the inner loops touch is one contiguous "hot blob" of 32-byte aligned
// SoA arrays (so a CTA can stage it into shared memory with 128-bit copies):
//   [sph R4 x n_sph][pln_n R4 x n_pln][pln_c R4 x n_pln][vert R2 x n_vert][lgt_p R4 x n_lgt]
//   [lgt_c R4 x n_lgt][pln_v I2 x n_pln][sph_id int x n_sph][pln_id int x n_pln]
//   FP32 only: [tri_g 4 x R4 x n_tri][poly_slot int x n_poly]
// Planar primitives that can never pass the reference's z-only inside test are sorted to the end
// (hittable | back-facing | degenerate projection) so culling is just a shorter loop.  Materials (touched once per hit) and
// the scene-order lists of the instrumented kernel stay in plain global arrays.
#pragma once

#include <memory>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/rm_b200.h"
#include "rm_fast.cuh"
#include "rm_pool.h"

namespace rm {

struct BlobLayout {
    int n_sph = 0, n_pln = 0, n_pln_live = 0, n_pln_nondegenerate = 0, n_vert = 0, n_lgt = 0;
    int off_sph = 0, off_pln_n = 0, off_pln_c = 0, off_vert = 0, off_lgt_p = 0, off_lgt_c = 0;
    int off_pln_v = 0, off_sph_id = 0, off_pln_id = 0;
    // FP32 fast path (rm_fast.cuh): non-degenerate 3-vertex planes as fixed records, the other
    // non-degenerate planes as indices into the generic arrays; hittable ones first in both lists
    int n_tri = 0, n_tri_live = 0, n_poly = 0, n_poly_live = 0;
    int off_tri_g = 0, off_poly_slot = 0;
    int bytes = 0;
    int any_glass = 0;                // some material is glass-like (shapes.rs:29): the frame may need the reflect / refract recursion
    double coord_max = 0., r_min = 0.; // largest coordinate magnitude of the primitives, smallest sphere radius (glass_mode, rm_fast.cuh)
};

struct alignas(32) BlobChunk { unsigned char b[32]; };

// std::vector whose resize() / sized constructor leave trivially constructible elements uninitialised: the packer's large
// arrays are written once, in parallel, by the threads that first touch their pages -- not zero-filled by one thread first
// (for 10^5 primitives the arrays are ~60 MB of fresh pages; faulting and zeroing them on one thread cost as much as the
// arithmetic).
template <typename T> struct NoInit {
    using value_type = T;
    NoInit() = default;
    template <typename U> NoInit(const NoInit<U>&) {}
    T* allocate(size_t n) { return std::allocator<T>().allocate(n); }
    void deallocate(T* p, size_t n) { std::allocator<T>().deallocate(p, n); }
    template <typename U> void construct(U* p) { ::new (static_cast<void*>(p)) U; }
    template <typename U, typename... A> void construct(U* p, A&&... a) { ::new (static_cast<void*>(p)) U(std::forward<A>(a)...); }
    template <typename U> bool operator==(const NoInit<U>&) const { return true; }
    template <typename U> bool operator!=(const NoInit<U>&) const { return false; }
};
template <typename T> using Buf = std::vector<T, NoInit<T>>;

// Planar primitives traced: culling keeps the hittable class only.  Without culling the f64 kernels
// trace everything like the reference; the f32 kernels still skip the degenerate-projection class,
// whose edge terms are rounding noise that single precision cannot reproduce.
template <typename R> RM_HD int plane_count(const BlobLayout& L, bool cull) {
    return cull ? L.n_pln_live : (sizeof(R) == 4 ? L.n_pln_nondegenerate : L.n_pln);
}

RM_HD int tri_count(const BlobLayout& L, bool cull) { return cull ? L.n_tri_live : L.n_tri; }
RM_HD int poly_count(const BlobLayout& L, bool cull) { return cull ? L.n_poly_live : L.n_poly; }

// Bounds of one hittable primitive (f64, unpadded) and its entry code kind << 30 | index for the hierarchy's leaves.
struct BvhPrimBox {
    double lo[3], hi[3];
    int code;
};

template <typename R> struct PackedScene {
    BlobLayout lay;
    Buf<BlobChunk> blob;              // lay.bytes bytes, 32-byte aligned
    const unsigned char* blob_data() const { return reinterpret_cast<const unsigned char*>(blob.data()); }
    size_t blob_bytes() const { return blob.size() * sizeof(BlobChunk); }
    Buf<double> tri_src;              // FP32 pack only: kTriSrcDoubles per fast-path triangle (prepare_raster input)
    Buf<double> sph64, pln64;         // FP32 pack only: f64 {c, r^2} per sphere and {n, n.C} per plane slot (cast_glass)
    Buf<R4<R>> mat_a, mat_b;
    Buf<int> mat_f;
    // scene-order traversal lists: [0] = every primitive, [1] = after culling
    std::vector<int> order[2], order_shape[2];
    int n_prims = 0;
    // FP32 pack only: hierarchy over the hittable primitives (rm_bvh.cuh), used when RmParams.accel is set
    std::vector<R4<float>> bvh_nodes;
    std::vector<int> bvh_prims;
    Buf<BvhPrimBox> bvh_boxes;        // ... and the boxes it was built from (rm_render_motion sweeps them)
    int bvh_depth = 0;
    double hierarchy_build_ms = 0.;
};

// Builds the hierarchy of rm_bvh.cuh (nodes: 4 x R4<float> each; prims: leaf entries).  Returns its depth.
// `pool`: threads to build on (large scenes); none = threads of the call's own.
int build_bvh(const Buf<BvhPrimBox>& boxes, std::vector<R4<float>>& nodes, std::vector<int>& prims, HostPool* pool = nullptr);

// Validates `fs` and packs it.  Returns RM_OK or RM_ERR_SCENE / RM_ERR_INVALID_ARGUMENT with `err` set.
// Scenes of 8192 planar primitives and more are packed on `pool`'s threads (none = threads of the call's own); the result
// does not depend on the number of threads.
template <typename R> int pack_scene(const RmFlatScene& fs, PackedScene<R>& out, std::string& err, HostPool* pool = nullptr);

// Deep copy of a flat scene (the caller's arrays may go away after rm_scene_upload).
struct OwnedFlatScene {
    std::vector<RmShapeRef> shapes;
    std::vector<RmSphere> spheres;
    std::vector<RmPolygon> polygons;
    std::vector<double> polygon_vertices;
    std::vector<RmObj> objs;
    Buf<RmTriangle> triangles;                        // the two large arrays: copied block by block on the pool's threads
    Buf<RmReflectance> triangle_reflectances;
    std::vector<RmLight> lights;
    RmFlatScene view() const;
    void assign(const RmFlatScene& fs, HostPool* pool = nullptr);
};

int validate_scene(const RmFlatScene& fs, std::string& err);

template <typename R> FrameParams<R> make_frame_params(const RmParams& p);

// rm_view_basis (include/rm_b200.h): u, v, w of the view into out[0..8], or RM_ERR_INVALID_ARGUMENT with a reason in err.
int view_basis(const RmView& view, double out[9], const char** err);

// The thin-lens camera of rm_render_lens for the frame of p: the s x frame's backproject operands, the camera, the basis
// (u, v, w in basis[0..8], or the identity for null) and the lens.  The lens is taken as given (rm_render_lens checks it).
LensCamera make_lens_camera(const RmParams& p, const double* basis, const RmLens& lens);

// The roughness of rm_render_rough_glass as the kernel reads it: g receives the n values in FP32 (a positive value too small
// for FP32 kept at 1e-30, at least one entry), and the returned RoughGlass the unit-disc points of s x s; its g pointer is
// left for the caller to set.  The values are taken as given (rm_render_rough_glass checks them).
RoughGlass make_rough_glass(int samples, const double* roughness, int n, std::vector<float>& g);

// The disc points of rm_render_indirect's bounces as the kernel reads them: diffuse_point of every stratum of s x s.
Diffuse make_diffuse(int samples);

// The motion of rm_render_motion as the kernel reads it: v receives the FP32 displacement {v, 0} of every primitive of the
// FP32 pack ps by the kernel's indices (Motion's layout: spheres | fast-path triangles | plane slots, from the ids in the
// blob), disp holding 3 doubles per primitive id; reach receives the largest |component| of those FP32 values over 2.  The
// values are taken as given (rm_render_motion checks them).
void motion_displacements(const PackedScene<float>& ps, const double* disp, std::vector<R4<float>>& v, double& reach);
// The samples' times of s x s (motion_time in f64 and rounded to FP32); the pointers are left for the caller to set.
Motion make_motion(int samples);
// The area lights of rm_render_distributed as the kernel reads them: r receives the n radii in FP32 (as rm_render_area_lights
// keeps them: a positive radius too small for FP32 at 1e-30, at least one entry), and the returned AreaPoints the unit-disc
// point of every stratum of area_offset; its radius pointer is left for the caller to set.  The radii are taken as given.
AreaPoints make_area_points(int samples, const double* radius, int n, std::vector<float>& r);
// The swept hierarchy of a motion frame: build_bvh over the pack's boxes, each grown by |v| / 2 per axis of its primitive's
// displacement in v (make_motion's layout) -- the union of its boxes at tau = -1/2 and +1/2.  With every displacement zero
// it is the pack's own hierarchy, byte for byte.
int build_swept_bvh(const PackedScene<float>& ps, const std::vector<R4<float>>& v, std::vector<R4<float>>& nodes, std::vector<int>& prims,
                    HostPool* pool = nullptr);

}  // namespace rm
