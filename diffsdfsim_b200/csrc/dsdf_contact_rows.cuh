// Contact-row geometry shared by the dense assembly (dsdf_dynamics.cu) and the fused solver (dsdf_dynsolve.cu).
// Scalar-generic (double | Dual), see dsdf_math.cuh.
#pragma once
#include "dsdf_math.cuh"

namespace dsdf {

// ---- contact-row geometry: tangent basis (physics3d/utils.py:247-256, physics3d/world.py:84-94), Jacobian rows
// (physics3d/world.py:56-101), world-frame inertia (bodies.py:509-511)
template <class S> __device__ __forceinline__ V3<S> tseed(V3<S> n) {
    const double ax = fabs(val(n.x)), ay = fabs(val(n.y)), az = fabs(val(n.z));
    int k = 0;
    double m = ax;
    if (ay < m) { m = ay; k = 1; }
    if (az < m) { k = 2; }
    S one = cst(n.x, 1.0), zero = cst(n.x, 0.0);
    return cross(v3<S>(k == 0 ? one : zero, k == 1 ? one : zero, k == 2 ? one : zero), n);
}
template <class S> __device__ __forceinline__ void fdirs(V3<S> n, int fd, V3<S>* dirs) {
    V3<S> d1 = normalize3(tseed(n));
    V3<S> d2 = normalize3(cross(d1, n));
    const int half = fd / 2;
    dirs[0] = d1; dirs[1] = d2;
    if (fd == 8) {
        V3<S> d3 = normalize3(d1 + d2);
        dirs[2] = d3; dirs[3] = normalize3(cross(d3, n));
    }
    for (int r = 0; r < half; ++r) dirs[half + r] = neg(dirs[r]);
}
// 12-entry row [p1 x d, d, -(p2 x d), -d]
template <class S> __device__ __forceinline__ void row12(V3<S> p1, V3<S> p2, V3<S> d, S* o) {
    V3<S> c1 = cross(p1, d), c2 = cross(p2, d);
    o[0] = c1.x; o[1] = c1.y; o[2] = c1.z; o[3] = d.x; o[4] = d.y; o[5] = d.z;
    o[6] = -c2.x; o[7] = -c2.y; o[8] = -c2.z; o[9] = -d.x; o[10] = -d.y; o[11] = -d.z;
}
template <class S> __device__ __forceinline__ M3<S> winertia(Q4<S> q, const S* I9) {
    M3<S> R = q2mat(q), I, Rt;
#pragma unroll
    for (int e = 0; e < 9; ++e) I.m[e] = I9[e];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) Rt.m[3 * i + j] = R.m[3 * j + i];
    return mat_mul(mat_mul(R, I), Rt);
}

}  // namespace dsdf
