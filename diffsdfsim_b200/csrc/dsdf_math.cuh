// Scalar-generic geometry for the stepping kernels: quaternions, exponential map, SDF evaluation.
// Every routine is templated on the scalar type S: `double` for forward passes, `Dual` (value + one
// tangent) for derivative passes.  Backward kernels obtain exact Jacobian columns by seeding one input
// at a time (forward-mode AD of the very same code path), then contract them with the incoming
// gradients.  The derivative conventions of the torch ops the reference uses are encoded here
// (abs'(0)=0, clamp sub-gradients, maximum tie = 1/2, normalize with eps clamp, arg-max routing).
//
// Third-party semantics restated (pytorch3d.transforms 0.7.5, SURVEY.md Appendix A):
//   quaternion_{raw_multiply,multiply,invert,apply,to_matrix}, matrix_to_quaternion, so3_exponential_map.
#pragma once
#include <cuda_runtime.h>
#include <math.h>

namespace dsdf {

struct Dual {
    double v, d;
    __host__ __device__ Dual() : v(0.0), d(0.0) {}
    __host__ __device__ Dual(double a) : v(a), d(0.0) {}
    __host__ __device__ Dual(double a, double b) : v(a), d(b) {}
};
#define HD __host__ __device__ __forceinline__
// IEEE-exact division / square root with the zero operand peeled off.  The hardware sequences (MUFU.RCP64H / RSQ64H +
// Newton steps) fall into a ~100-instruction slow path whenever the numerator (radicand) is zero or denormal, and the
// whole warp waits for it; exact zeros are everywhere in contact geometry (axis-aligned normals, points on coordinate
// planes, clamped box distances).  0 / b = +-0 and sqrt(+-0) = +-0 exactly, so the shortcut changes no bit.
// DSDF_OUTLINE_MATH (defined by large kernels before including this header): keep ONE out-of-line copy of the
// division / square-root / quaternion-rotation sequences instead of inlining them at every call site -- the contact
// kernel otherwise exceeds the instruction cache several times over.
#ifdef DSDF_OUTLINE_MATH
#define DSDF_MATH_FN __host__ __device__ __noinline__
#else
#define DSDF_MATH_FN HD
#endif
DSDF_MATH_FN double fdiv(double a, double b) { return (a == 0.0 && b != 0.0 && b == b) ? (b > 0.0 ? a : -a) : a / b; }
DSDF_MATH_FN double fsqrt(double a) { return a == 0.0 ? a : sqrt(a); }
// Three quotients by one divisor with ONE division: r = RN(1/b), then q = RN(a r) corrected by one exact-remainder step
// q' = fma(fma(-q, b, a), r, q).  With r the correctly rounded reciprocal and q within one ulp of a/b this is the
// correctly rounded quotient RN(a/b) (Markstein's theorem), i.e. the same bits as a / b; zero numerators stay exact
// zeros and the non-finite / tiny-divisor cases take the plain divisions.
// (The out-of-line copy takes and returns the three values by value, in registers: through references they would make
// a round trip through local memory at every call.)
struct Dbl3 { double x, y, z; };
DSDF_MATH_FN Dbl3 fdiv3_v(double x, double y, double z, double b) {
    Dbl3 o;
    if (!(b > 1e-290 && b < 1e290)) { o.x = fdiv(x, b); o.y = fdiv(y, b); o.z = fdiv(z, b); return o; }
    const double r = 1.0 / b;
    o.x = x; o.y = y; o.z = z;
    if (x != 0.0) { const double q = x * r; o.x = fma(fma(-q, b, x), r, q); }
    if (y != 0.0) { const double q = y * r; o.y = fma(fma(-q, b, y), r, q); }
    if (z != 0.0) { const double q = z * r; o.z = fma(fma(-q, b, z), r, q); }
    return o;
}
HD void fdiv3(double& x, double& y, double& z, double b) { const Dbl3 o = fdiv3_v(x, y, z, b); x = o.x; y = o.y; z = o.z; }
HD Dual operator+(Dual a, Dual b) { return Dual(a.v + b.v, a.d + b.d); }
HD Dual operator-(Dual a, Dual b) { return Dual(a.v - b.v, a.d - b.d); }
HD Dual operator-(Dual a) { return Dual(-a.v, -a.d); }
HD Dual operator*(Dual a, Dual b) { return Dual(a.v * b.v, a.d * b.v + a.v * b.d); }
HD Dual operator/(Dual a, Dual b) { double q = fdiv(a.v, b.v); return Dual(q, fdiv(a.d - q * b.d, b.v)); }
HD Dual fdiv(Dual a, Dual b) { return a / b; }
HD void fdiv3(Dual& x, Dual& y, Dual& z, Dual b) {      // values and tangents: two batches of three quotients by b.v
    double qx = x.v, qy = y.v, qz = z.v;
    fdiv3(qx, qy, qz, b.v);
    double tx = x.d - qx * b.d, ty = y.d - qy * b.d, tz = z.d - qz * b.d;
    fdiv3(tx, ty, tz, b.v);
    x = Dual(qx, tx); y = Dual(qy, ty); z = Dual(qz, tz);
}
HD Dual& operator+=(Dual& a, Dual b) { a = a + b; return a; }
HD Dual& operator-=(Dual& a, Dual b) { a = a - b; return a; }
HD Dual& operator*=(Dual& a, Dual b) { a = a * b; return a; }

HD double val(double a) { return a; }
HD double val(Dual a) { return a.v; }
HD double tan_(double) { return 0.0; }
HD double tan_(Dual a) { return a.d; }
HD void set_tangent(double&, double) {}
HD void set_tangent(Dual& a, double d) { a.d = d; }
HD bool needs_tan(double) { return false; }
HD bool needs_tan(Dual) { return true; }

HD double dsqrt(double a) { return fsqrt(a); }
HD Dual dsqrt(Dual a) { double s = fsqrt(a.v); return Dual(s, a.d / (2.0 * s)); }
HD double dsin(double a) { return sin(a); }
HD Dual dsin(Dual a) { return Dual(sin(a.v), cos(a.v) * a.d); }
HD double dcos(double a) { return cos(a); }
HD Dual dcos(Dual a) { return Dual(cos(a.v), -sin(a.v) * a.d); }
// torch.abs: derivative sign(x) with sign(0) = 0
HD double dabs(double a) { return fabs(a); }
HD Dual dabs(Dual a) { return Dual(fabs(a.v), a.v > 0.0 ? a.d : (a.v < 0.0 ? -a.d : 0.0)); }
// x.clamp(min=0): gradient passes where x >= 0
HD double clamp_min0(double a) { return a < 0.0 ? 0.0 : a; }
HD Dual clamp_min0(Dual a) { return a.v < 0.0 ? Dual(0.0, 0.0) : a; }
// x.clamp(max=0): gradient passes where x <= 0
HD double clamp_max0(double a) { return a > 0.0 ? 0.0 : a; }
HD Dual clamp_max0(Dual a) { return a.v > 0.0 ? Dual(0.0, 0.0) : a; }
// torch.max(x, 0) (binary maximum): tie splits the gradient in half
HD double maximum0(double a) { return a > 0.0 ? a : 0.0; }
HD Dual maximum0(Dual a) { return a.v > 0.0 ? a : (a.v == 0.0 ? Dual(0.0, 0.5 * a.d) : Dual(0.0, 0.0)); }
// torch.min(0, x) (binary minimum): tie splits the gradient in half
HD double minimum0(double a) { return a < 0.0 ? a : 0.0; }
HD Dual minimum0(Dual a) { return a.v < 0.0 ? a : (a.v == 0.0 ? Dual(0.0, 0.5 * a.d) : Dual(0.0, 0.0)); }
// clamp(x, lo) general lower clamp (so3_exponential_map): passes where x >= lo
HD double clamp_lo(double a, double lo) { return a < lo ? lo : a; }
HD Dual clamp_lo(Dual a, double lo) { return a.v < lo ? Dual(lo, 0.0) : a; }
HD double cst(double, double c) { return c; }
HD Dual cst(Dual, double c) { return Dual(c, 0.0); }

template <class S> struct V3 { S x, y, z; };
template <class S> struct Q4 { S w, x, y, z; };
template <class S> struct M3 { S m[9]; };

template <class S> HD V3<S> v3(S x, S y, S z) { V3<S> r; r.x = x; r.y = y; r.z = z; return r; }
template <class S> HD V3<S> operator+(V3<S> a, V3<S> b) { return v3<S>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <class S> HD V3<S> operator-(V3<S> a, V3<S> b) { return v3<S>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <class S> HD V3<S> operator*(V3<S> a, S s) { return v3<S>(a.x * s, a.y * s, a.z * s); }
template <class S> HD V3<S> neg(V3<S> a) { return v3<S>(-a.x, -a.y, -a.z); }
template <class S> HD S dot(V3<S> a, V3<S> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <class S> HD V3<S> cross(V3<S> a, V3<S> b) {
    return v3<S>(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
// torch .norm(): derivative x/|x|, 0 at the origin
HD double norm3(V3<double> a) { return fsqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
HD Dual norm3(V3<Dual> a) {
    double n = fsqrt(a.x.v * a.x.v + a.y.v * a.y.v + a.z.v * a.z.v);
    double d = n > 0.0 ? fdiv(a.x.v * a.x.d + a.y.v * a.y.d + a.z.v * a.z.d, n) : 0.0;
    return Dual(n, d);
}
HD double norm2(double a, double b) { return fsqrt(a * a + b * b); }
HD Dual norm2(Dual a, Dual b) {
    double n = fsqrt(a.v * a.v + b.v * b.v);
    return Dual(n, n > 0.0 ? fdiv(a.v * a.d + b.v * b.d, n) : 0.0);
}
// F.normalize(v, dim): v / max(|v|, 1e-12); the clamp has zero gradient when it is active
template <class S> HD V3<S> normalize3(V3<S> a) {
    S n = norm3(a);
    if (val(n) < 1e-12) n = cst(n, 1e-12);
    fdiv3(a.x, a.y, a.z, n);
    return a;
}
template <class S> HD void normalize2(S& a, S& b) {
    S n = norm2(a, b);
    if (val(n) < 1e-12) n = cst(n, 1e-12);
    a = fdiv(a, n); b = fdiv(b, n);
}

// ------------------------------------------------------------------ quaternions (w,x,y,z)
template <class S> HD Q4<S> q4(S w, S x, S y, S z) { Q4<S> r; r.w = w; r.x = x; r.y = y; r.z = z; return r; }
template <class S> HD Q4<S> qmul_raw(Q4<S> a, Q4<S> b) {
    return q4<S>(a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z,
                 a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
                 a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x,
                 a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w);
}
template <class S> HD Q4<S> qstd(Q4<S> q) { return val(q.w) < 0.0 ? q4<S>(-q.w, -q.x, -q.y, -q.z) : q; }
template <class S> HD Q4<S> qmul(Q4<S> a, Q4<S> b) { return qstd(qmul_raw(a, b)); }
template <class S> HD Q4<S> qinv(Q4<S> q) { return q4<S>(q.w, -q.x, -q.y, -q.z); }
template <class S> HD V3<S> qapply_inl(Q4<S> q, V3<S> p) {
    S zero = cst(p.x, 0.0);
    Q4<S> o = qmul_raw(qmul_raw(q, q4<S>(zero, p.x, p.y, p.z)), qinv(q));
    return v3<S>(o.x, o.y, o.z);
}
DSDF_MATH_FN V3<double> qapply(Q4<double> q, V3<double> p) { return qapply_inl<double>(q, p); }
HD V3<Dual> qapply(Q4<Dual> q, V3<Dual> p) { return qapply_inl<Dual>(q, p); }
template <class S> HD M3<S> q2mat(Q4<S> q) {
    S r = q.w, i = q.x, j = q.y, k = q.z;
    S two = cst(r, 2.0), one = cst(r, 1.0);
    S s = two / (r * r + i * i + j * j + k * k);
    M3<S> R;
    R.m[0] = one - s * (j * j + k * k); R.m[1] = s * (i * j - k * r); R.m[2] = s * (i * k + j * r);
    R.m[3] = s * (i * j + k * r); R.m[4] = one - s * (i * i + k * k); R.m[5] = s * (j * k - i * r);
    R.m[6] = s * (i * k - j * r); R.m[7] = s * (j * k + i * r); R.m[8] = one - s * (i * i + j * j);
    return R;
}
template <class S> HD V3<S> mat_apply(const M3<S>& R, V3<S> p) {
    return v3<S>(R.m[0] * p.x + R.m[1] * p.y + R.m[2] * p.z, R.m[3] * p.x + R.m[4] * p.y + R.m[5] * p.z,
                 R.m[6] * p.x + R.m[7] * p.y + R.m[8] * p.z);
}
template <class S> HD V3<S> mat_applyT(const M3<S>& R, V3<S> p) {
    return v3<S>(R.m[0] * p.x + R.m[3] * p.y + R.m[6] * p.z, R.m[1] * p.x + R.m[4] * p.y + R.m[7] * p.z,
                 R.m[2] * p.x + R.m[5] * p.y + R.m[8] * p.z);
}
template <class S> HD M3<S> mat_mul(const M3<S>& A, const M3<S>& B) {
    M3<S> C;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C.m[3 * i + j] = A.m[3 * i] * B.m[j] + A.m[3 * i + 1] * B.m[3 + j] + A.m[3 * i + 2] * B.m[6 + j];
    return C;
}
// so3_exponential_map(w, eps=1e-4): theta = sqrt(clamp(|w|^2, eps)); R = I + sin/theta K + (1-cos)/theta^2 K^2
template <class S> HD M3<S> expmap(V3<S> w) {
    S nr = w.x * w.x + w.y * w.y + w.z * w.z;
    S th = dsqrt(clamp_lo(nr, 1e-4));
    S inv = cst(th, 1.0) / th;
    S f1 = inv * dsin(th);
    S f2 = inv * inv * (cst(th, 1.0) - dcos(th));
    S zero = cst(th, 0.0);
    M3<S> K;
    K.m[0] = zero; K.m[1] = -w.z; K.m[2] = w.y;
    K.m[3] = w.z; K.m[4] = zero; K.m[5] = -w.x;
    K.m[6] = -w.y; K.m[7] = w.x; K.m[8] = zero;
    M3<S> K2 = mat_mul(K, K);
    M3<S> R;
#pragma unroll
    for (int e = 0; e < 9; ++e) R.m[e] = f1 * K.m[e] + f2 * K2.m[e];
    R.m[0] = R.m[0] + cst(th, 1.0); R.m[4] = R.m[4] + cst(th, 1.0); R.m[8] = R.m[8] + cst(th, 1.0);
    return R;
}
// _sqrt_positive_part: sqrt where x > 0 else 0 (zero sub-gradient at 0)
HD double sqrt_pos(double a) { return a > 0.0 ? sqrt(a) : 0.0; }
HD Dual sqrt_pos(Dual a) { return a.v > 0.0 ? dsqrt(a) : Dual(0.0, 0.0); }
// matrix_to_quaternion: four candidates, pick the one with the largest |component| (first on ties)
template <class S> HD Q4<S> mat2q(const M3<S>& R) {
    S one = cst(R.m[0], 1.0);
    S m00 = R.m[0], m01 = R.m[1], m02 = R.m[2], m10 = R.m[3], m11 = R.m[4], m12 = R.m[5], m20 = R.m[6], m21 = R.m[7],
      m22 = R.m[8];
    S qa[4] = {sqrt_pos(one + m00 + m11 + m22), sqrt_pos(one + m00 - m11 - m22), sqrt_pos(one - m00 + m11 - m22),
               sqrt_pos(one - m00 - m11 + m22)};
    int best = 0;
#pragma unroll
    for (int k = 1; k < 4; ++k) if (val(qa[k]) > val(qa[best])) best = k;
    S den = qa[best];
    if (val(den) < 0.1) den = cst(den, 0.1);           // q_abs.max(0.1): clamp with zero gradient when active
    den = den * cst(den, 2.0);
    S c0, c1, c2, c3;
    if (best == 0) { c0 = qa[0] * qa[0]; c1 = m21 - m12; c2 = m02 - m20; c3 = m10 - m01; }
    else if (best == 1) { c0 = m21 - m12; c1 = qa[1] * qa[1]; c2 = m10 + m01; c3 = m02 + m20; }
    else if (best == 2) { c0 = m02 - m20; c1 = m10 + m01; c2 = qa[2] * qa[2]; c3 = m12 + m21; }
    else { c0 = m10 - m01; c1 = m20 + m02; c2 = m21 + m12; c3 = qa[3] * qa[3]; }
    return q4<S>(fdiv(c0, den), fdiv(c1, den), fdiv(c2, den), fdiv(c3, den));
}

#undef HD
}  // namespace dsdf
