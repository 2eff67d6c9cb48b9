// Element-wise operators of the hot path:
//   dsdf_sdf_query[_backward]   SDF3D.query_sdfs            sdf_physics/physics3d/bodies.py:721-760 (+38-125, 203-257)
//   dsdf_integrate[_backward]   Body3D.move / set_p (pose)   sdf_physics/physics3d/bodies.py:488-511
// Backward kernels use forward-mode duals of the same device code (dsdf_math.cuh), one seed per input scalar.
#include "dsdf_sdf.cuh"
#include "dsdf_integrate.cuh"

namespace dsdf {

__device__ __forceinline__ SdfShape load_shape(int kind, const double* shape4, const double* grid, int res, double e0,
                                               double e1) {
    SdfShape s;
    s.kind = kind; s.a = shape4[0]; s.b = shape4[1]; s.c = shape4[2]; s.scale = shape4[3];
    s.grid = grid; s.res = res; s.e0 = e0; s.e1 = e1;
    return s;
}

__global__ void __launch_bounds__(256)
sdf_query_kernel(int kind, const double* __restrict__ shape, const double* __restrict__ grid, int res,
                 long long grid_stride, const double* __restrict__ pts, int N, int want_dir,
                 double* __restrict__ sdf, double* __restrict__ dir, double e0, double e1) {
    const int w = blockIdx.y;
    const SdfShape sh = load_shape(kind, shape + 4 * (size_t)w, grid ? grid + (size_t)w * grid_stride : nullptr, res, e0, e1);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const size_t o = (size_t)w * N + i;
        V3<double> p = v3<double>(pts[3 * o], pts[3 * o + 1], pts[3 * o + 2]);
        SdfOut<double> r = sdf_query<double>(sh, p, want_dir != 0);
        sdf[o] = r.d;
        if (want_dir) { dir[3 * o] = r.n.x; dir[3 * o + 1] = r.n.y; dir[3 * o + 2] = r.n.z; }
    }
}


// ---- grid bodies: the same arithmetic as grid_eval_raw / sdf_query (identical expression order, so identical bits),
// but every voxel of the 32-voxel stencil (8 corners + their axis neighbours) is loaded ONCE into registers instead
// of once per use (56 loads): the kernel is bound by L1/LSU wavefronts and FP64 issue, not by DRAM, until the
// redundant loads are gone.  One thread per point; consecutive points of a warp walk the grid's fastest axis.
// v / max(|v|, 1e-12) with ONE division: r = RN(1/n), then per component q = a r corrected by one exact-remainder
// Newton step (q' = fma(fma(-q, n, a), r, q)), which is the correctly rounded quotient whenever r is the correctly
// rounded reciprocal (Markstein); zero components stay exact zeros.  Replaces three ~35-instruction divisions.
__device__ __forceinline__ V3<double> normalize3_rcp(V3<double> a) {
    double n = norm3(a);
    if (n < 1e-12) n = 1e-12;
    const double r = 1.0 / n;
    auto q = [&](double x) {
        if (x == 0.0) return x;
        const double q0 = x * r;
        return fma(fma(-q0, n, x), r, q0);
    };
    return v3<double>(q(a.x), q(a.y), q(a.z));
}

#ifndef SDFQ_MINB_DIR
#define SDFQ_MINB_DIR 2
#endif
#ifndef SDFQ_MINB_VAL
#define SDFQ_MINB_VAL 4
#endif
#ifndef SDFQ_WAVES
#define SDFQ_WAVES 8
#endif
// Grid SDF (bodies.py:203-257): trilinear value and, with DIR, the normalised trilinear interpolation of the central
// difference field -- a 32-voxel register stencil per point.  ncu (profiles/r1_ncu_summary.md): DRAM traffic = the
// algorithmic bytes; the limits are on chip, the L1 wavefronts of the 32 gathers and ~200 FP64 instructions per point,
// which only overlap across warps.  Value-only queries get their own instantiation (8 gathers, 56 registers, 4 CTAs per
// SM: 0.84 of the measured HBM peak instead of 0.58 when it shared the direction kernel's registers).  The direction is
// accumulated in three passes over the stencil (z, x, y neighbours; each accumulator keeps the summation order of a
// single loop, so the bits are unchanged); measured: 2, 3 or 4 CTAs per SM make no difference for it (0.47-0.49, 4 CTAs
// spill) -- it sits on the L1 wavefront limit of its 32 scattered 8-byte gathers per point.
template <bool DIR>
__global__ void __launch_bounds__(256, DIR ? SDFQ_MINB_DIR : SDFQ_MINB_VAL)
sdf_query_grid_kernel(const double* __restrict__ shape, const double* __restrict__ grid, int R, long long grid_stride,
                      const double* __restrict__ pts, int N, double* __restrict__ sdf, double* __restrict__ dir) {
    const int w = blockIdx.y;
    const double sc = shape[4 * (size_t)w + 3];
    const double* __restrict__ g = grid + (size_t)w * grid_stride;
    const double ext = (double)(R - 1);
    const size_t sx = (size_t)R * R, sy = (size_t)R;
    // persistent-style loop with the NEXT point's coordinates prefetched: the DRAM latency of the point stream overlaps
    // the FP64 instructions of the current point
    const int step = gridDim.x * blockDim.x;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    double qx = 0.0, qy = 0.0, qz = 0.0;
    if (i < N) { const size_t o = (size_t)w * N + i; qx = pts[3 * o]; qy = pts[3 * o + 1]; qz = pts[3 * o + 2]; }
    for (; i < N; i += step) {
        const size_t o = (size_t)w * N + i;
        const double px = qx, py = qy, pz = qz;
        if (i + step < N) { const size_t o2 = o + step; qx = pts[3 * o2]; qy = pts[3 * o2 + 1]; qz = pts[3 * o2 + 2]; }
        double val_ = 1.0 * sc, n0 = 0.0, n1 = 0.0, n2 = 0.0;
        const bool inside = fabs(px) <= sc && fabs(py) <= sc && fabs(pz) <= sc;
        if (inside) {
            const bool unit = sc == 1.0;                       // x / 1 = x exactly
            const double ux = unit ? px : fdiv(px, sc), uy = unit ? py : fdiv(py, sc), uz = unit ? pz : fdiv(pz, sc);
            const double ix = (ux + 1.) * 0.5 * ext, iy = (uy + 1.) * 0.5 * ext, iz = (uz + 1.) * 0.5 * ext;
            const bool ok = ix <= ext && ix >= 0.0 && iy <= ext && iy >= 0.0 && iz <= ext && iz >= 0.0;
            double v = 1.0, a0 = 0.0, a1 = 0.0, a2 = 0.0;
            if (ok) {
                const int bx = min(max((int)floor(ix), 0), R - 2), by = min(max((int)floor(iy), 0), R - 2),
                          bz = min(max((int)floor(iz), 0), R - 2);
                const double tx = ix - bx, ty = iy - by, tz = iz - bz;
                const double* c = g + ((size_t)bx * R + by) * R + bz;
                // corners C[dx][dy][dz]
                double C[2][2][2];
#pragma unroll
                for (int dx = 0; dx < 2; ++dx)
#pragma unroll
                    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                        for (int dz = 0; dz < 2; ++dz) C[dx][dy][dz] = c[dx * sx + dy * sy + dz];
                double acc = 0.0;
                auto wgt = [&](int dx, int dy, int dz) { return (dx ? tx : 1 - tx) * (dy ? ty : 1 - ty) * (dz ? tz : 1 - tz); };
                if (DIR) {
                    // axis neighbours one step outside the cell.  On a boundary plane the reference's central difference
                    // is zero (bodies.py:225-234): there the neighbour is redirected to the voxel it is subtracted from,
                    // so hi - lo = 0 exactly and no per-corner select is needed.  Twice the central differences are
                    // summed; the exact factor 1/2 is applied once at the end (scaling by a power of two commutes with
                    // every rounding involved).
                    {
                        const long long ozm = bz > 0 ? -1 : 1, ozp = bz + 2 < R ? 2 : 0;
                        double ZM[2][2], ZP[2][2];
#pragma unroll
                        for (int a = 0; a < 2; ++a)
#pragma unroll
                            for (int b = 0; b < 2; ++b) { ZM[a][b] = c[a * sx + b * sy + ozm]; ZP[a][b] = c[a * sx + b * sy + ozp]; }
#pragma unroll
                        for (int dx = 0; dx < 2; ++dx)
#pragma unroll
                            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                                for (int dz = 0; dz < 2; ++dz) {
                                    const double wg = wgt(dx, dy, dz);
                                    acc = acc + C[dx][dy][dz] * wg;
                                    const double hi = dz ? ZP[dx][dy] : C[dx][dy][1], lo = dz ? C[dx][dy][0] : ZM[dx][dy];
                                    a2 = a2 + (hi - lo) * wg;
                                }
                    }
                    {
                        const long long oxm = bx > 0 ? -(long long)sx : (long long)sx, oxp = bx + 2 < R ? 2 * (long long)sx : 0;
                        double XM[2][2], XP[2][2];
#pragma unroll
                        for (int a = 0; a < 2; ++a)
#pragma unroll
                            for (int b = 0; b < 2; ++b) { XM[a][b] = c[oxm + a * sy + b]; XP[a][b] = c[oxp + a * sy + b]; }
#pragma unroll
                        for (int dx = 0; dx < 2; ++dx)
#pragma unroll
                            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                                for (int dz = 0; dz < 2; ++dz) {
                                    const double hi = dx ? XP[dy][dz] : C[1][dy][dz], lo = dx ? C[0][dy][dz] : XM[dy][dz];
                                    a0 = a0 + (hi - lo) * wgt(dx, dy, dz);
                                }
                    }
                    {
                        const long long oym = by > 0 ? -(long long)sy : (long long)sy, oyp = by + 2 < R ? 2 * (long long)sy : 0;
                        double YM[2][2], YP[2][2];
#pragma unroll
                        for (int a = 0; a < 2; ++a)
#pragma unroll
                            for (int b = 0; b < 2; ++b) { YM[a][b] = c[a * sx + oym + b]; YP[a][b] = c[a * sx + oyp + b]; }
#pragma unroll
                        for (int dx = 0; dx < 2; ++dx)
#pragma unroll
                            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                                for (int dz = 0; dz < 2; ++dz) {
                                    const double hi = dy ? YP[dx][dz] : C[dx][1][dz], lo = dy ? C[dx][0][dz] : YM[dx][dz];
                                    a1 = a1 + (hi - lo) * wgt(dx, dy, dz);
                                }
                    }
                    a0 *= 0.5; a1 *= 0.5; a2 *= 0.5;
                } else {
#pragma unroll
                    for (int dx = 0; dx < 2; ++dx)
#pragma unroll
                        for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                            for (int dz = 0; dz < 2; ++dz) acc = acc + C[dx][dy][dz] * wgt(dx, dy, dz);
                }
                v = acc;
            }
            val_ = v * sc;
            if (DIR) {
                const V3<double> d1 = ok ? normalize3_rcp(v3<double>(a0, a1, a2)) : v3<double>(0.0, 0.0, 0.0);
                const V3<double> d2 = normalize3_rcp(d1);
                n0 = d2.x; n1 = d2.y; n2 = d2.z;
            }
        }
        sdf[o] = val_;
        if (DIR) { dir[3 * o] = n0; dir[3 * o + 1] = n1; dir[3 * o + 2] = n2; }
    }
}

__global__ void __launch_bounds__(256)
sdf_query_bwd_kernel(int kind, const double* __restrict__ shape, const double* __restrict__ grid, int res,
                     long long grid_stride, const double* __restrict__ pts, int N,
                     const double* __restrict__ gsdf, const double* __restrict__ gdir, double* __restrict__ gpts,
                     double e0, double e1) {
    const int w = blockIdx.y;
    const SdfShape sh = load_shape(kind, shape + 4 * (size_t)w, grid ? grid + (size_t)w * grid_stride : nullptr, res, e0, e1);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const size_t o = (size_t)w * N + i;
        const double gs = gsdf ? gsdf[o] : 0.0;
        const double g0 = gdir ? gdir[3 * o] : 0.0, g1 = gdir ? gdir[3 * o + 1] : 0.0, g2 = gdir ? gdir[3 * o + 2] : 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            V3<Dual> p = v3<Dual>(Dual(pts[3 * o], k == 0), Dual(pts[3 * o + 1], k == 1), Dual(pts[3 * o + 2], k == 2));
            SdfOut<Dual> r = sdf_query<Dual>(sh, p, gdir != nullptr);
            gpts[3 * o + k] = gs * r.d.d + g0 * r.n.x.d + g1 * r.n.y.d + g2 * r.n.z.d;
        }
    }
}

__global__ void __launch_bounds__(128)
integrate_kernel(const double* __restrict__ p, const double* __restrict__ v, const double* __restrict__ dt,
                 const unsigned char* __restrict__ active, int W, int nb, double* __restrict__ po) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * nb) return;
    const int w = i / nb;
    double pi[7], vi[6], o[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) pi[k] = p[(size_t)i * 7 + k];
    if (active && !active[w]) {
#pragma unroll
        for (int k = 0; k < 7; ++k) po[(size_t)i * 7 + k] = pi[k];
        return;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) vi[k] = v[(size_t)i * 6 + k];
    integrate_one<double>(pi, vi, dt[w], o);
#pragma unroll
    for (int k = 0; k < 7; ++k) po[(size_t)i * 7 + k] = o[k];
}

__global__ void __launch_bounds__(128)
integrate_bwd_kernel(const double* __restrict__ p, const double* __restrict__ v, const double* __restrict__ dt,
                     const unsigned char* __restrict__ active, int W, int nb, const double* __restrict__ gpo,
                     double* __restrict__ gp, double* __restrict__ gv, double* __restrict__ gdt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * nb) return;
    const int w = i / nb;
    double g[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) g[k] = gpo[(size_t)i * 7 + k];
    if (active && !active[w]) {
#pragma unroll
        for (int k = 0; k < 7; ++k) gp[(size_t)i * 7 + k] = g[k];
#pragma unroll
        for (int k = 0; k < 6; ++k) gv[(size_t)i * 6 + k] = 0.0;
        gdt[i] = 0.0;
        return;
    }
    for (int seed = 0; seed < 14; ++seed) {
        Dual pi[7], vi[6], o[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) pi[k] = Dual(p[(size_t)i * 7 + k], seed == k ? 1.0 : 0.0);
#pragma unroll
        for (int k = 0; k < 6; ++k) vi[k] = Dual(v[(size_t)i * 6 + k], seed == 7 + k ? 1.0 : 0.0);
        Dual dti(dt[w], seed == 13 ? 1.0 : 0.0);
        integrate_one<Dual>(pi, vi, dti, o);
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < 7; ++k) acc += g[k] * o[k].d;
        if (seed < 7) gp[(size_t)i * 7 + seed] = acc;
        else if (seed < 13) gv[(size_t)i * 6 + seed - 7] = acc;
        else gdt[i] = acc;
    }
}

}  // namespace dsdf

using namespace dsdf;

extern "C" {

int dsdf_sdf_query(int kind, const double* shape, double extra0, double extra1, const double* grid, int res,
                   long long grid_world_stride, const double* pts, int W, int N, int want_dir, double* sdf, double* dir,
                   void* stream) {
    if (W <= 0 || N < 0 || kind < 0 || kind > DSDF_SDF_BOWL || (kind == DSDF_SDF_GRID && (!grid || res < 2))) return -1;
    if (N == 0) return 0;
    int bx = (N + 255) / 256;
    if (bx > 148 * 8) bx = 148 * 8;
    if (kind == DSDF_SDF_GRID) {
        // ~4 resident waves of CTAs over the whole launch (148 SMs x 3 CTAs); each thread streams several points
        int per_world = (148 * (want_dir ? SDFQ_MINB_DIR : SDFQ_MINB_VAL) * SDFQ_WAVES + W - 1) / W;
        if (per_world < 1) per_world = 1;
        if (bx > per_world) bx = per_world;
        if (want_dir)
            sdf_query_grid_kernel<true><<<dim3(bx, W), 256, 0, (cudaStream_t)stream>>>(shape, grid, res, grid_world_stride,
                                                                                       pts, N, sdf, dir);
        else
            sdf_query_grid_kernel<false><<<dim3(bx, W), 256, 0, (cudaStream_t)stream>>>(shape, grid, res, grid_world_stride,
                                                                                        pts, N, sdf, dir);
    } else
        sdf_query_kernel<<<dim3(bx, W), 256, 0, (cudaStream_t)stream>>>(kind, shape, grid, res, grid_world_stride, pts,
                                                                        N, want_dir, sdf, dir, extra0, extra1);
    return (int)cudaGetLastError();
}

int dsdf_sdf_query_backward(int kind, const double* shape, double extra0, double extra1, const double* grid, int res,
                            long long grid_world_stride, const double* pts, int W, int N, const double* gsdf,
                            const double* gdir, double* gpts, void* stream) {
    if (W <= 0 || N < 0 || kind < 0 || kind > DSDF_SDF_BOWL || (kind == DSDF_SDF_GRID && (!grid || res < 2))) return -1;
    if (N == 0) return 0;
    int bx = (N + 255) / 256;
    if (bx > 148 * 8) bx = 148 * 8;
    sdf_query_bwd_kernel<<<dim3(bx, W), 256, 0, (cudaStream_t)stream>>>(kind, shape, grid, res, grid_world_stride, pts,
                                                                        N, gsdf, gdir, gpts, extra0, extra1);
    return (int)cudaGetLastError();
}

int dsdf_integrate(const double* p, const double* v, const double* dt, const unsigned char* active, int W, int nb,
                   double* p_out, void* stream) {
    if (W <= 0 || nb <= 0) return -1;
    integrate_kernel<<<(W * nb + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p, v, dt, active, W, nb, p_out);
    return (int)cudaGetLastError();
}

int dsdf_integrate_backward(const double* p, const double* v, const double* dt, const unsigned char* active, int W,
                            int nb, const double* gp_out, double* gp, double* gv, double* gdt, void* stream) {
    if (W <= 0 || nb <= 0) return -1;
    integrate_bwd_kernel<<<(W * nb + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p, v, dt, active, W, nb, gp_out, gp,
                                                                                 gv, gdt);
    return (int)cudaGetLastError();
}

}  // extern "C"
