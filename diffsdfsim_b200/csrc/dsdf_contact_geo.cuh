// Contact geometry shared by the detection kernel (dsdf_contacts.cu) and its pose-gradient kernel
// (dsdf_contacts_bwd.cu): geometry table, pose / shape loads, and _compute_contacts for one contact
// (sdf_physics/physics3d/contacts.py:161-214), templated on double | Dual.
#pragma once
#include "dsdf_dense.cuh"
#include "dsdf_sdf.cuh"

namespace dsdf {

struct BodyGeom {                 // mirrors dsdf_body_geom in include/dsdf_b200.h
    int kind, nverts, nfaces, res;
    const double* verts;          // (nverts,3) body frame; world w at verts + w*vstride
    const int* faces;             // (nfaces,3)
    const double* grid;           // res^3; world w at grid + w*gstride
    long long vstride, gstride;
    // uniform cell index over the body-frame mesh (faces binned by centroid, vertices by position); has_cells = 0 when
    // the vertices are per-world (the kernels then scan the whole mesh)
    double cell_lo[3], cell_inv;
    int cell_dims[3], has_cells;
    const int *fcell_start, *fcell_items, *vcell_start, *vcell_items;
    double max_face_rad;          // max_f max_i |centroid_f - v_i|; 0 = unknown (no fp32 pre-filter)
    // per-world topology (bodies whose mesh differs from world to world, e.g. iso-surfaces of per-world SDF grids):
    // world w uses faces + w*fstride, nfaces_w[w] faces and nverts_w[w] vertices; NULL / 0 = shared topology
    long long fstride;
    const int *nfaces_w, *nverts_w;
    double extra[2];              // further SDF parameters of the kind (rounding radius / scale)
};

// the geometry of body g as world w sees it (topology pointers / counts resolved; vertices stay strided, see load_vert)
__device__ __forceinline__ BodyGeom world_geom(const BodyGeom& g, int w) {
    BodyGeom r = g;
    r.faces = g.faces + (size_t)w * g.fstride;
    if (g.nfaces_w) r.nfaces = g.nfaces_w[w];
    if (g.nverts_w) r.nverts = g.nverts_w[w];
    return r;
}

// One out-of-line copy of the SDF evaluation for the whole contact kernel: inlining it at ~30 call sites made the
// kernel 575 KB of SASS, far beyond the instruction cache (ncu: 18 % of stall samples "no_instructions").  The shape is
// passed by reference: the contact kernel keeps it in shared memory, so a call passes one pointer, not eight registers.
#ifdef DSDF_OUTLINE_MATH
__device__ __noinline__ SdfOut<double> sdf_q(const SdfShape& sh, V3<double> p, bool want_n) {
    return sdf_query<double>(sh, p, want_n);
}
#define DSDF_GEO_FN __device__ __noinline__
#else
__device__ __forceinline__ SdfOut<double> sdf_q(const SdfShape& sh, V3<double> p, bool want_n) {
    return sdf_query<double>(sh, p, want_n);
}
#define DSDF_GEO_FN __device__ __forceinline__
#endif

__device__ __forceinline__ void load_pose(const double* p, int w, int nb, int b, Q4<double>& q, V3<double>& x) {
    const double* s = p + ((size_t)w * nb + b) * 7;
    q = q4<double>(s[0], s[1], s[2], s[3]);
    x = v3<double>(s[4], s[5], s[6]);
}
__device__ __forceinline__ SdfShape body_shape(const BodyGeom& g, const double* shape, int w, int nb, int b) {
    const double* s = shape + ((size_t)w * nb + b) * 4;
    SdfShape sh;
    sh.kind = g.kind; sh.a = s[0]; sh.b = s[1]; sh.c = s[2]; sh.scale = s[3];
    sh.grid = g.grid ? g.grid + (size_t)w * g.gstride : nullptr;
    sh.res = g.res;
    sh.e0 = g.extra[0]; sh.e1 = g.extra[1];
    return sh;
}
__device__ __forceinline__ V3<double> load_vert(const BodyGeom& g, int w, int vi) {
    const double* v = g.verts + (size_t)w * g.vstride + (size_t)vi * 3;
    return v3<double>(v[0], v[1], v[2]);
}
// vertex of b1 (body frame) -> world -> b2 frame, same operation order as contacts.py:42 / bodies.py:718
__device__ __forceinline__ V3<double> to_b2(V3<double> v, Q4<double> q1, V3<double> x1, Q4<double> q2i, V3<double> x2) {
    return qapply(q2i, (qapply(q1, v) + x1) - x2);
}

// ------------------------------------------------------------------------------------------ contact geometry
template <class S> struct ContactGeo { V3<S> n, p1, p2; S pen; };

__device__ __forceinline__ SdfOut<double> sdf_qs(const SdfShape& sh, V3<double> p, bool want_n) { return sdf_q(sh, p, want_n); }
template <class P> __device__ __forceinline__ SdfOut<Dual> sdf_qs(const SdfShapeT<P>& sh, V3<Dual> p, bool want_n) {
    return sdf_query<Dual>(sh, p, want_n);
}
template <class S> __device__ __forceinline__ V3<S> lift(V3<double> a, S proto) {
    return v3<S>(cst(proto, a.x), cst(proto, a.y), cst(proto, a.z));
}
__device__ __forceinline__ V3<Dual> lift(V3<Dual> a, Dual) { return a; }
__device__ __forceinline__ V3<double> strip(V3<double> a) { return a; }
__device__ __forceinline__ V3<Dual> strip(V3<Dual> a) { return v3<Dual>(Dual(a.x.v), Dual(a.y.v), Dual(a.z.v)); }

DSDF_GEO_FN double laplacian_fd(const SdfShape& s, V3<double> c, double d0, double h) {
    double acc = 0.0;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        V3<double> sh = v3<double>(ax == 0 ? h : 0.0, ax == 1 ? h : 0.0, ax == 2 ? h : 0.0);
        const double qp = sdf_q(s, c + sh, false).d;
        const double qm = sdf_q(s, c - sh, false).d;
        acc = acc + ((qp - 2 * d0) + qm);
    }
    return acc;
}

// contacts.py:161-214 for one contact; c_tri = sum(abc * local verts of the face) depends on the pose of neither body
// (but on b1's vertices: V3<Dual> when the derivative w.r.t. the mesh is wanted).  P: double, or Dual to differentiate
// through the shape parameters as well.
template <class S, class P, class T>
__device__ ContactGeo<S> contact_geometry(const SdfShapeT<P>& s1, const SdfShapeT<P>& s2, Q4<S> q1, V3<S> x1, Q4<S> q2,
                                          V3<S> x2, V3<T> c_tri, double fd_eps, bool detach_b2) {
    S proto = q1.w;
    V3<S> c1 = lift(c_tri, proto);
    SdfOut<S> o1 = sdf_qs(s1, c1, true);
    c1 = c1 - o1.n * o1.d;
    o1 = sdf_qs(s1, c1, true);
    V3<S> cw = qapply(q1, c1) + x1;
    V3<S> c2 = qapply(qinv(q2), cw - x2);
    if (detach_b2) c2 = strip(c2);
    SdfOut<S> o2 = sdf_qs(s2, c2, true);
    const V3<double> c1v = v3<double>(val(c1.x), val(c1.y), val(c1.z));
    const V3<double> c2v = v3<double>(val(c2.x), val(c2.y), val(c2.z));
    const double lap1 = laplacian_fd(shape_values(s1), c1v, val(o1.d), fd_eps);
    const double lap2 = laplacian_fd(shape_values(s2), c2v, val(o2.d), fd_eps);
    const bool stable = fabs(lap2) < fabs(lap1);
    ContactGeo<S> g;
    g.n = stable ? qapply(q2, o2.n) : neg(qapply(q1, o1.n));
    g.p2 = qapply(q2, c2 - o2.n * o2.d);
    g.p1 = qapply(q1, c1);
    g.pen = -o2.d;
    return g;
}


}  // namespace dsdf
