// SDF3D.query_sdfs on the device (sdf_physics/physics3d/bodies.py:721-760) for the four body kinds:
//   box / sphere / cylinder analytic value + "failsafe" direction   (bodies.py:38-125)
//   grid: trilinear value, on-the-fly central-difference direction, DiffGridSDF derivative (bodies.py:203-257)
// Scalar-generic (double or Dual) -- see dsdf_math.cuh.
#pragma once
#include "dsdf_math.cuh"
#include "../../include/dsdf_b200.h"

namespace dsdf {

// What a kernel needs to evaluate one body's SDF in that body's frame.  P = double, or Dual when the derivative with
// respect to the shape parameters themselves is wanted (radius / dimension fitting: the reference's grad-enabled
// _compute_contacts differentiates through params and scale, sdf_physics/physics3d/bodies.py:747-751).
template <class P> struct SdfShapeT {
    int kind;            // DSDF_SDF_*
    P a, b, c;           // normalised parameters: box dims/scale; sphere r/scale; cylinder r/scale, h/scale
    P scale;
    const double* grid;  // (R,R,R) row-major, this world's grid (kind == GRID)
    int res;
    double e0, e1;       // further parameters of the kind (rounded box / brick: r/scale), not differentiated
};
typedef SdfShapeT<double> SdfShape;

// a shape parameter as a scalar of the evaluation type S
template <class S> __device__ __forceinline__ S par(S proto, double c) { return cst(proto, c); }
__device__ __forceinline__ Dual par(Dual, Dual c) { return c; }
__device__ __forceinline__ const SdfShape& shape_values(const SdfShape& s) { return s; }
__device__ __forceinline__ SdfShape shape_values(const SdfShapeT<Dual>& s) {
    SdfShape r;
    r.kind = s.kind; r.a = s.a.v; r.b = s.b.v; r.c = s.c.v; r.scale = s.scale.v; r.grid = s.grid; r.res = s.res;
    r.e0 = s.e0; r.e1 = s.e1;
    return r;
}

template <class S> struct SdfOut { S d; V3<S> n; };

// ---- box (bodies.py:38-72), point u already divided by scale
template <class S, class P> __device__ __forceinline__ void box_eval(V3<S> u, P dx, P dy, P dz, bool want_n,
                                                                     S& value, V3<S>& dir) {
    const S half = cst(u.x, 0.5);
    S qx = dabs(u.x) - par(u.x, dx) * half, qy = dabs(u.y) - par(u.x, dy) * half, qz = dabs(u.z) - par(u.x, dz) * half;
    // q.max(dim=1): first maximal index carries the gradient
    S top = qx;
    if (val(qy) > val(top)) top = qy;
    if (val(qz) > val(top)) top = qz;
    value = norm3(v3<S>(clamp_min0(qx), clamp_min0(qy), clamp_min0(qz))) + clamp_max0(top);
    if (!want_n) return;
    const double sx = val(u.x) < 0.0 ? -1.0 : 1.0, sy = val(u.y) < 0.0 ? -1.0 : 1.0, sz = val(u.z) < 0.0 ? -1.0 : 1.0;
    const double tv = val(top);
    const double inside = tv <= 0.0 ? 1.0 : 0.0;
    V3<S> m = normalize3(v3<S>(maximum0(qx), maximum0(qy), maximum0(qz)));
    V3<S> g = v3<S>((m.x + cst(m.x, inside * (val(qx) == tv ? 1.0 : 0.0))) * cst(m.x, sx),
                    (m.y + cst(m.x, inside * (val(qy) == tv ? 1.0 : 0.0))) * cst(m.x, sy),
                    (m.z + cst(m.x, inside * (val(qz) == tv ? 1.0 : 0.0))) * cst(m.x, sz));
    dir = normalize3(g);
}

// ---- sphere (bodies.py:75-84)
template <class S, class P> __device__ __forceinline__ void sphere_eval(V3<S> u, P r, bool want_n, S& value, V3<S>& dir) {
    value = norm3(u) - par(u.x, r);
    if (want_n) dir = normalize3(u);
}

// ---- cylinder along local z (bodies.py:87-125)
template <class S, class P> __device__ __forceinline__ void cylinder_eval(V3<S> u, P r, P h, bool want_n, S& value,
                                                                          V3<S>& dir) {
    S rho = norm2(u.x, u.y);
    S q0 = dabs(rho) - par(rho, r), q1 = dabs(u.z) - par(rho, h) * cst(rho, 0.5);
    S top = q0;
    if (val(q1) > val(top)) top = q1;
    value = norm2(clamp_min0(q0), clamp_min0(q1)) + clamp_max0(top);
    if (!want_n) return;
    const double sz = val(u.z) < 0.0 ? -1.0 : 1.0;
    const double tv = val(top);
    const double inside = tv <= 0.0 ? 1.0 : 0.0;
    S m0 = clamp_min0(q0), m1 = clamp_min0(q1);
    normalize2(m0, m1);
    S g0 = m0 + cst(m0, inside * (val(q0) == tv ? 1.0 : 0.0));
    S g1 = m1 + cst(m0, inside * (val(q1) == tv ? 1.0 : 0.0));
    S ex = u.x, ey = u.y;
    normalize2(ex, ey);
    dir = normalize3(v3<S>(g0 * ex, g0 * ey, g1 * cst(m0, sz)));
}

// ---- brick (bodies.py:184-200): box whose first two dimensions are rounded in-plane with radius r.  Value only: the
// reference pairs it with the direction of a CUBE of side r (rounded_sdf_grad(box_sdf_grad) receives (dims, r) and passes
// r on as the box size, bodies.py:175-181,882-884) -- reproduced as it is.
template <class S, class P> __device__ __forceinline__ S brick_value(V3<S> u, P dx, P dy, P dz, double r) {
    const S half = cst(u.x, 0.5), rr = cst(u.x, r);
    S q0 = dabs(u.x) - (par(u.x, dx) * half - rr), q1 = dabs(u.y) - (par(u.x, dy) * half - rr);
    S q2 = dabs(u.z) - par(u.x, dz) * half;
    S top01 = q0;
    if (val(q1) > val(top01)) top01 = q1;
    S s01 = norm2(clamp_min0(q0), clamp_min0(q1)) + clamp_max0(top01) - rr;
    S top = s01;
    if (val(q2) > val(top)) top = q2;
    return norm2(clamp_min0(s01), clamp_min0(q2)) + clamp_max0(top);
}

// ---- bowl (bodies.py:128-163): half shell of radius r and half thickness d, opening towards +z.  The reference's
// value and direction functions shift the z coordinate IN PLACE (pts[:, 2] -= r/2) on the same tensor, so the direction is
// evaluated at z - r (shifted twice); `u` here is the point as the respective function sees it.
template <class S, class P> __device__ __forceinline__ void bowl_ps(V3<S> u, P r, P d, S& ps0, S& ps1, S& psn) {
    S rho = norm2(u.x, u.y);
    psn = norm2(rho, u.z);
    ps1 = u.z;
    S first = val(u.z) < 0.0 ? psn : rho;
    ps0 = dabs(first - par(u.x, r)) - par(u.x, d);
}
template <class S, class P> __device__ __forceinline__ S bowl_value(V3<S> u, P r, P d) {
    S ps0, ps1, psn;
    bowl_ps(u, r, d, ps0, ps1, psn);
    S top = ps0;
    if (val(ps1) > val(top)) top = ps1;
    return norm2(maximum0(ps0), maximum0(ps1)) + minimum0(top);
}
template <class S, class P> __device__ __forceinline__ V3<S> bowl_dir(V3<S> u, P r, P d) {
    S ps0, ps1, psn;
    bowl_ps(u, r, d, ps0, ps1, psn);
    const double diff = val(psn) - val(par(u.x, r));
    const double sg = diff > 0.0 ? 1.0 : (diff < 0.0 ? -1.0 : 0.0);
    V3<S> g = v3<S>(u.x * cst(u.x, sg), u.y * cst(u.x, sg), u.z * cst(u.x, sg));
    if (val(ps1) >= 0.0) {
        if (val(ps0) < 0.0) { g.x = cst(u.x, 0.0); g.y = cst(u.x, 0.0); }
        g.z = dabs(g.z);
    }
    return normalize3(g);
}

// ---- grid (bodies.py:203-257 + ev_sdf_utils.grid_interp semantics, SURVEY.md Appendix A)
// value: trilinear at idx=(u+1)/2*(R-1); direction: normalised trilinear interpolation of the central-difference
// field (zero on the two boundary planes of each axis).  No derivative flows through the interpolation indices;
// d value / d u := direction (DiffGridSDF.backward).
__device__ __forceinline__ double grid_cd(const double* g, int R, int i, int j, int k, int axis) {
    const int c = axis == 0 ? i : (axis == 1 ? j : k);
    if (c <= 0 || c >= R - 1) return 0.0;
    const size_t st = axis == 0 ? (size_t)R * R : (axis == 1 ? (size_t)R : 1);
    const size_t o = ((size_t)i * R + j) * R + k;
    return (g[o + st] - g[o - st]) * 0.5;      // exact: division by 2
}
__device__ __forceinline__ bool grid_eval_raw(const double* g, int R, double ux, double uy, double uz, bool want_n,
                                              double& value, double n[3]) {
    const double ext = (double)(R - 1);
    const double ix = (ux + 1.) * 0.5 * ext, iy = (uy + 1.) * 0.5 * ext, iz = (uz + 1.) * 0.5 * ext;
    const bool ok = ix <= ext && ix >= 0.0 && iy <= ext && iy >= 0.0 && iz <= ext && iz >= 0.0;
    value = 1.0;
    n[0] = n[1] = n[2] = 0.0;
    if (!ok) return false;
    int bx = min(max((int)floor(ix), 0), R - 2), by = min(max((int)floor(iy), 0), R - 2),
        bz = min(max((int)floor(iz), 0), R - 2);
    const double tx = ix - bx, ty = iy - by, tz = iz - bz;
    double acc = 0.0, a0 = 0.0, a1 = 0.0, a2 = 0.0;
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
        const double wx = dx ? tx : 1 - tx;
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
            const double wy = dy ? ty : 1 - ty;
#pragma unroll
            for (int dz = 0; dz < 2; ++dz) {
                const double wz = dz ? tz : 1 - tz;
                const double w = wx * wy * wz;
                const int i = bx + dx, j = by + dy, k = bz + dz;
                acc = acc + g[((size_t)i * R + j) * R + k] * w;
                if (want_n) {
                    a0 = a0 + grid_cd(g, R, i, j, k, 0) * w;
                    a1 = a1 + grid_cd(g, R, i, j, k, 1) * w;
                    a2 = a2 + grid_cd(g, R, i, j, k, 2) * w;
                }
            }
        }
    }
    value = acc;
    if (want_n) {
        V3<double> d = normalize3(v3<double>(a0, a1, a2));
        n[0] = d.x; n[1] = d.y; n[2] = d.z;
    }
    return true;
}

// ---- SDF3D.query_sdfs: p in the body frame -> sdf (scaled back) and unit direction. Outside |p|<=scale: (scale, 0).
template <class S, class P>
__device__ __forceinline__ SdfOut<S> sdf_query(const SdfShapeT<P>& sh, V3<S> p, bool want_n = true) {
    SdfOut<S> o;
    const double sc = val(sh.scale);
    S zero = cst(p.x, 0.0);
    o.n = v3<S>(zero, zero, zero);
    const bool inside = fabs(val(p.x)) <= sc && fabs(val(p.y)) <= sc && fabs(val(p.z)) <= sc;
    S scs = par(p.x, sh.scale);
    if (!inside) { o.d = cst(p.x, 1.0) * scs; return o; }
    V3<S> u = p;
    fdiv3(u.x, u.y, u.z, scs);
    S value;
    V3<S> dir = o.n;
    if (sh.kind == DSDF_SDF_BOX) box_eval(u, sh.a, sh.b, sh.c, want_n, value, dir);
    else if (sh.kind == DSDF_SDF_SPHERE) sphere_eval(u, sh.a, want_n, value, dir);
    else if (sh.kind == DSDF_SDF_CYLINDER) cylinder_eval(u, sh.a, sh.b, want_n, value, dir);
    else if (sh.kind == DSDF_SDF_BOX_ROUNDED) {                 // box(dims - 2r) - r, direction of that box
        box_eval(u, sh.a, sh.b, sh.c, want_n, value, dir);
        value = value - cst(u.x, sh.e0);
    } else if (sh.kind == DSDF_SDF_BRICK) {
        value = brick_value(u, sh.a, sh.b, sh.c, sh.e0);
        if (want_n) { S dummy; box_eval(u, sh.e0, sh.e0, sh.e0, true, dummy, dir); }
    } else if (sh.kind == DSDF_SDF_BOWL) {
        const S half = cst(u.x, 0.5);
        V3<S> u1 = v3<S>(u.x, u.y, u.z - par(u.x, sh.a) * half);
        value = bowl_value(u1, sh.a, sh.b);
        if (want_n) dir = bowl_dir(v3<S>(u1.x, u1.y, u1.z - par(u.x, sh.a) * half), sh.a, sh.b);
    } else {
        double v, n[3];
        // the custom backward (Dual pass) always needs the direction
        grid_eval_raw(sh.grid, sh.res, val(u.x), val(u.y), val(u.z), want_n || needs_tan(p.x), v, n);
        // tangent of the value := direction . du ; direction itself carries no tangent
        double dv = n[0] * tan_(u.x) + n[1] * tan_(u.y) + n[2] * tan_(u.z);
        value = cst(p.x, v);
        set_tangent(value, dv);
        dir = v3<S>(cst(p.x, n[0]), cst(p.x, n[1]), cst(p.x, n[2]));
    }
    o.d = value * scs;
    if (want_n) o.n = normalize3(dir);
    return o;
}

}  // namespace dsdf
