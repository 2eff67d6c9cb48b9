// Mixed-LCP assembly for all worlds, and its reverse-mode contraction.
//
// Replaces PdipmEngine.solve_dynamics' assembly (lcp_physics/physics/engines.py:31-79) together with
//   World3D.M / Body3D.set_p inertia update   sdf_physics/physics3d/world.py:48-50, bodies.py:509-511
//   World3D.Jc, Jf, orthogonal                 sdf_physics/physics3d/world.py:56-101, physics3d/utils.py:247-256
//   World.restitutions / mu / E                lcp_physics/physics/world.py:402-409, 480-501
// The solve itself is dsdf_lcp_forward on the matrices written here (a world without contacts gets
// nineq_w = 0 and is solved as the equality-constrained system of engines.py:40-54).
// Backward: dsdf_lcp_backward produces dQ, dp, dG, dh, dF; assemble_bwd_kernel contracts them onto the physical
// inputs (poses, velocities, masses, inertias, friction, restitution, forces, dt, contact geometry) using
// forward-mode duals of the same row-construction code.
#include "dsdf_math.cuh"
#include "dsdf_contact_rows.cuh"
#include "../../include/dsdf_b200.h"

namespace dsdf {

// Row blocks of one direction d at contact point pt: [pt x d, d]
template <class S> __device__ __forceinline__ void jac_block(V3<S> pt, V3<S> d, S* out6) {
    V3<S> c = cross(pt, d);
    out6[0] = c.x; out6[1] = c.y; out6[2] = c.z; out6[3] = d.x; out6[4] = d.y; out6[5] = d.z;
}

__global__ void __launch_bounds__(128)
assemble_kernel(const double* __restrict__ p, const double* __restrict__ v, const double* __restrict__ mass,
                const double* __restrict__ Ibody, const double* __restrict__ fric, const double* __restrict__ rest,
                const double* __restrict__ f, const double* __restrict__ dt, const unsigned char* __restrict__ active,
                const int* __restrict__ count, const int* __restrict__ cbody, const double* __restrict__ cgeo,
                int nb, int maxc, int fd,
                double* __restrict__ Q, double* __restrict__ pv, double* __restrict__ G, double* __restrict__ h,
                double* __restrict__ F, int* __restrict__ nineq_w) {
    const int w = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const int nz = 6 * nb, per = 2 + fd, niCap = maxc * per;
    if (active && !active[w]) { if (tid == 0) nineq_w[w] = -1; return; }
    const int nc = min(count[w], maxc);
    const int ni = nc * per;
    double* Qw = Q + (size_t)w * nz * nz;
    double* Gw = G + (size_t)w * niCap * nz;
    double* Fw = F + (size_t)w * niCap * niCap;
    double* hw = h + (size_t)w * niCap;
    const double* vw = v + (size_t)w * nz;
    for (int e = tid; e < nz * nz; e += nt) Qw[e] = 0.0;
    for (int e = tid; e < ni * nz; e += nt) Gw[e] = 0.0;
    for (int i = tid; i < ni; i += nt) {
        hw[i] = 0.0;
        for (int j = 0; j < ni; ++j) Fw[(size_t)i * niCap + j] = 0.0;
    }
    __syncthreads();
    // mass matrix blocks
    for (int b = tid; b < nb; b += nt) {
        const double* pb = p + ((size_t)w * nb + b) * 7;
        M3<double> Iw = winertia<double>(q4<double>(pb[0], pb[1], pb[2], pb[3]), Ibody + ((size_t)w * nb + b) * 9);
        const double m = mass[(size_t)w * nb + b];
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) Qw[(6 * b + i) * nz + 6 * b + j] = Iw.m[3 * i + j];
            Qw[(6 * b + 3 + i) * nz + 6 * b + 3 + i] = m;
        }
    }
    // contact rows
    for (int c = tid; c < nc; c += nt) {
        const size_t oo = (size_t)w * maxc + c;
        const int i1 = cbody[2 * oo], i2 = cbody[2 * oo + 1];
        const double* g = cgeo + 10 * oo;
        const V3<double> n = v3<double>(g[0], g[1], g[2]), p1 = v3<double>(g[3], g[4], g[5]), p2 = v3<double>(g[6], g[7], g[8]);
        double r1[6], r2[6];
        jac_block<double>(p1, n, r1);
        jac_block<double>(p2, n, r2);
        double jv = 0.0;
        for (int k = 0; k < 6; ++k) {
            Gw[(size_t)c * nz + 6 * i1 + k] = r1[k];
            Gw[(size_t)c * nz + 6 * i2 + k] = -r2[k];
        }
        // (Jc v) with the row as stored (sequential over the full row like a dense mat-vec)
        for (int k = 0; k < nz; ++k) jv += Gw[(size_t)c * nz + k] * vw[k];
        const double e = (rest[(size_t)w * nb + i1] + rest[(size_t)w * nb + i2]) / 2;
        hw[c] = jv * e;
        V3<double> dirs[8];
        fdirs<double>(n, fd, dirs);
        for (int r = 0; r < fd; ++r) {
            const int row = nc + fd * c + r;
            jac_block<double>(p1, dirs[r], r1);
            jac_block<double>(p2, dirs[r], r2);
            for (int k = 0; k < 6; ++k) {
                Gw[(size_t)row * nz + 6 * i1 + k] = r1[k];
                Gw[(size_t)row * nz + 6 * i2 + k] = -r2[k];
            }
            Fw[(size_t)row * niCap + nc + fd * nc + c] = 1.0;
            Fw[(size_t)(nc + fd * nc + c) * niCap + row] = -1.0;
        }
        const double mu = 0.5 * (fric[(size_t)w * nb + i1] + fric[(size_t)w * nb + i2]);
        Fw[(size_t)(nc + fd * nc + c) * niCap + c] = mu;
    }
    __syncthreads();
    // u = M v + dt f
    const double dtw = dt[w];
    for (int i = tid; i < nz; i += nt) {
        double acc = 0.0;
        for (int j = 0; j < nz; ++j) acc += Qw[(size_t)i * nz + j] * vw[j];
        pv[(size_t)w * nz + i] = acc + dtw * f[(size_t)w * nz + i];
    }
    if (tid == 0) nineq_w[w] = ni;
}

// rows of one contact (Jc row + fd friction rows), both body blocks, as a function of (n, p1, p2)
template <class S>
__device__ __forceinline__ void contact_rows(V3<S> n, V3<S> p1, V3<S> p2, int fd, bool jc_part, bool jf_part,
                                             S* jc1, S* jc2, S (*jf1)[6], S (*jf2)[6]) {
    if (jc_part) { jac_block<S>(p1, n, jc1); jac_block<S>(p2, n, jc2); }
    if (jf_part) {
        V3<S> dirs[8];
        fdirs<S>(n, fd, dirs);
        for (int r = 0; r < fd; ++r) { jac_block<S>(p1, dirs[r], jf1[r]); jac_block<S>(p2, dirs[r], jf2[r]); }
    }
}

__global__ void __launch_bounds__(128)
assemble_bwd_kernel(const double* __restrict__ p, const double* __restrict__ v, const double* __restrict__ mass,
                    const double* __restrict__ Ibody, const double* __restrict__ fric, const double* __restrict__ rest,
                    const double* __restrict__ f, const double* __restrict__ dt, const unsigned char* __restrict__ active,
                    const int* __restrict__ count, const int* __restrict__ cbody, const double* __restrict__ cgeo,
                    int nb, int maxc, int fd, int stop_contact_grad, int stop_friction_grad,
                    const double* __restrict__ Q, const double* __restrict__ G,
                    const double* __restrict__ dQ, const double* __restrict__ dp, const double* __restrict__ dG,
                    const double* __restrict__ dh, const double* __restrict__ dF,
                    double* __restrict__ gp, double* __restrict__ gv, double* __restrict__ gmass,
                    double* __restrict__ gI, double* __restrict__ gfric, double* __restrict__ grest,
                    double* __restrict__ gf, double* __restrict__ gdt, double* __restrict__ ggeo) {
    const int w = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const int nz = 6 * nb, per = 2 + fd, niCap = maxc * per;
    const bool on = !(active && !active[w]);
    const int nc = on ? min(count[w], maxc) : 0;
    const double* vw = v + (size_t)w * nz;
    const double* Qw = Q + (size_t)w * nz * nz;
    const double* Gw = G + (size_t)w * niCap * nz;
    const double* dQw = dQ + (size_t)w * nz * nz;
    const double* dpw = dp + (size_t)w * nz;
    const double* dGw = dG + (size_t)w * niCap * nz;
    const double* dhw = dh + (size_t)w * niCap;
    const double* dFw = dF + (size_t)w * niCap * niCap;
    const double dtw = dt[w];
    if (!on) {
        for (int i = tid; i < nb * 7; i += nt) gp[(size_t)w * nb * 7 + i] = 0.0;
        for (int i = tid; i < nz; i += nt) { gv[(size_t)w * nz + i] = 0.0; gf[(size_t)w * nz + i] = 0.0; }
        for (int i = tid; i < nb; i += nt) {
            gmass[(size_t)w * nb + i] = 0.0; gfric[(size_t)w * nb + i] = 0.0; grest[(size_t)w * nb + i] = 0.0;
        }
        for (int i = tid; i < nb * 9; i += nt) gI[(size_t)w * nb * 9 + i] = 0.0;
        for (int i = tid; i < maxc * 10; i += nt) ggeo[(size_t)w * maxc * 10 + i] = 0.0;
        if (tid == 0) gdt[w] = 0.0;
        return;
    }
    // gv = M' du + Jc' (e o dh) ; gf = dt du
    for (int j = tid; j < nz; j += nt) {
        double acc = 0.0;
        for (int i = 0; i < nz; ++i) acc += Qw[(size_t)i * nz + j] * dpw[i];
        for (int c = 0; c < nc; ++c) {
            const size_t oo = (size_t)w * maxc + c;
            const double e = (rest[(size_t)w * nb + cbody[2 * oo]] + rest[(size_t)w * nb + cbody[2 * oo + 1]]) / 2;
            acc += Gw[(size_t)c * nz + j] * e * dhw[c];
        }
        gv[(size_t)w * nz + j] = acc;
        gf[(size_t)w * nz + j] = dtw * dpw[j];
    }
    if (tid == 0) {
        double acc = 0.0;
        for (int i = 0; i < nz; ++i) acc += f[(size_t)w * nz + i] * dpw[i];
        gdt[w] = acc;
    }
    // per body: mass, inertia, pose (through R I R'), friction, restitution
    for (int b = tid; b < nb; b += nt) {
        // dM = dQ + du v'  (body block only: M is block diagonal)
        double dMb[36];
        for (int i = 0; i < 6; ++i)
            for (int j = 0; j < 6; ++j)
                dMb[6 * i + j] = dQw[(size_t)(6 * b + i) * nz + 6 * b + j] + dpw[6 * b + i] * vw[6 * b + j];
        gmass[(size_t)w * nb + b] = dMb[6 * 3 + 3] + dMb[6 * 4 + 4] + dMb[6 * 5 + 5];
        const double* pb = p + ((size_t)w * nb + b) * 7;
        const double* Ib = Ibody + ((size_t)w * nb + b) * 9;
        for (int seed = 0; seed < 13; ++seed) {
            Dual I9[9];
            for (int e = 0; e < 9; ++e) I9[e] = Dual(Ib[e], seed == 4 + e ? 1.0 : 0.0);
            Q4<Dual> q = q4<Dual>(Dual(pb[0], seed == 0), Dual(pb[1], seed == 1), Dual(pb[2], seed == 2), Dual(pb[3], seed == 3));
            M3<Dual> Iw = winertia<Dual>(q, I9);
            double acc = 0.0;
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) acc += dMb[6 * i + j] * Iw.m[3 * i + j].d;
            if (seed < 4) gp[((size_t)w * nb + b) * 7 + seed] = acc;
            else gI[((size_t)w * nb + b) * 9 + seed - 4] = acc;
        }
        gp[((size_t)w * nb + b) * 7 + 4] = 0.0; gp[((size_t)w * nb + b) * 7 + 5] = 0.0; gp[((size_t)w * nb + b) * 7 + 6] = 0.0;
        double gfr = 0.0, gre = 0.0;
        for (int c = 0; c < nc; ++c) {
            const size_t oo = (size_t)w * maxc + c;
            if (cbody[2 * oo] != b && cbody[2 * oo + 1] != b) continue;
            gfr += 0.5 * dFw[(size_t)(nc + fd * nc + c) * niCap + c];
            double jv = 0.0;
            for (int k = 0; k < nz; ++k) jv += Gw[(size_t)c * nz + k] * vw[k];
            gre += 0.5 * dhw[c] * jv;
        }
        gfric[(size_t)w * nb + b] = gfr;
        grest[(size_t)w * nb + b] = gre;
    }
    // contact geometry: d(n, p1, p2) from dJc (incl. the h = e Jc v path) and dJf
    for (int t = tid; t < maxc * 10; t += nt) {
        const int c = t / 10, comp = t % 10;
        double acc = 0.0;
        if (c < nc && comp < 9) {
            const size_t oo = (size_t)w * maxc + c;
            const int i1 = cbody[2 * oo], i2 = cbody[2 * oo + 1];
            const double* g = cgeo + 10 * oo;
            auto D = [&](int k) { return Dual(g[k], comp == k ? 1.0 : 0.0); };
            const V3<Dual> n = v3<Dual>(D(0), D(1), D(2)), p1 = v3<Dual>(D(3), D(4), D(5)), p2 = v3<Dual>(D(6), D(7), D(8));
            Dual jc1[6], jc2[6], jf1[8][6], jf2[8][6];
            contact_rows<Dual>(n, p1, p2, fd, !stop_contact_grad, !stop_friction_grad, jc1, jc2, jf1, jf2);
            const double e = (rest[(size_t)w * nb + i1] + rest[(size_t)w * nb + i2]) / 2;
            if (!stop_contact_grad) {
                for (int k = 0; k < 6; ++k) {
                    const double g1 = dGw[(size_t)c * nz + 6 * i1 + k] + dhw[c] * e * vw[6 * i1 + k];
                    const double g2 = dGw[(size_t)c * nz + 6 * i2 + k] + dhw[c] * e * vw[6 * i2 + k];
                    acc += g1 * jc1[k].d - g2 * jc2[k].d;
                }
            }
            if (!stop_friction_grad) {
                for (int r = 0; r < fd; ++r) {
                    const int row = nc + fd * c + r;
                    for (int k = 0; k < 6; ++k)
                        acc += dGw[(size_t)row * nz + 6 * i1 + k] * jf1[r][k].d - dGw[(size_t)row * nz + 6 * i2 + k] * jf2[r][k].d;
                }
            }
        }
        ggeo[(size_t)w * maxc * 10 + t] = acc;
    }
}

}  // namespace dsdf

using namespace dsdf;

extern "C" {

int dsdf_dynamics_assemble(const double* p, const double* v, const double* mass, const double* Ibody,
                           const double* fric, const double* rest, const double* f, const double* dt,
                           const unsigned char* active, const int32_t* count, const int32_t* cbody, const double* cgeo,
                           int W, int nb, int maxc, int fric_dirs,
                           double* Q, double* pvec, double* G, double* h, double* F, int32_t* nineq_w, void* stream) {
    if (W <= 0 || nb <= 0 || maxc <= 0 || (fric_dirs != 8 && fric_dirs != 4)) return -1;
    assemble_kernel<<<W, 128, 0, (cudaStream_t)stream>>>(p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, cgeo,
                                                         nb, maxc, fric_dirs, Q, pvec, G, h, F, nineq_w);
    return (int)cudaGetLastError();
}

int dsdf_dynamics_assemble_backward(const double* p, const double* v, const double* mass, const double* Ibody,
                                    const double* fric, const double* rest, const double* f, const double* dt,
                                    const unsigned char* active, const int32_t* count, const int32_t* cbody,
                                    const double* cgeo, int W, int nb, int maxc, int fric_dirs,
                                    int stop_contact_grad, int stop_friction_grad,
                                    const double* Q, const double* G,
                                    const double* dQ, const double* dp, const double* dG, const double* dh, const double* dF,
                                    double* gp, double* gv, double* gmass, double* gI, double* gfric, double* grest,
                                    double* gf, double* gdt, double* ggeo, void* stream) {
    if (W <= 0 || nb <= 0 || maxc <= 0 || (fric_dirs != 8 && fric_dirs != 4)) return -1;
    assemble_bwd_kernel<<<W, 128, 0, (cudaStream_t)stream>>>(p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody,
                                                             cgeo, nb, maxc, fric_dirs, stop_contact_grad,
                                                             stop_friction_grad, Q, G, dQ, dp, dG, dh, dF, gp, gv, gmass,
                                                             gI, gfric, grest, gf, gdt, ggeo);
    return (int)cudaGetLastError();
}

}  // extern "C"
