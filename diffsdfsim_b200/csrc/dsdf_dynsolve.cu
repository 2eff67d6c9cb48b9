// Fused contact dynamics: LCP assembly + primal-dual interior point + (backward) implicit differentiation,
// exploiting the contact structure of the reference's LCP instead of a dense factorisation.
//
// Replaces PdipmEngine.solve_dynamics (lcp_physics/physics/engines.py:31-83) end to end, i.e. the same mathematics
// as dsdf_dynamics_assemble + dsdf_lcp_forward/backward (which remain the dense, general LCPFunction path):
//   * PDIPM iteration, initial point, best-iterate tracking, step rules: lcp_physics/lcp/solvers/batch.py:70-237
//   * implicit backward: lcp_physics/lcp/lcp.py:156-213
// Linear algebra.  The reference eliminates x first and LU-factors the nineq x nineq matrix
// G Q^-1 G' + F + D^-1 (batch.py:413-520).  In the engine's LCP, F + D^-1 is block diagonal per contact
// (rows: normal, fric_dirs friction rows, one cone row; engines.py:72-78):
//        B_c = [[a_n, 0, 0], [0, diag(a_f), 1], [mu_c, -1', a_g]],   a = 1/d = s/z > 0
// with a closed-form inverse, so we eliminate the multipliers instead and factor the (nz+neq)^2 matrix
//        K = [[Q + sum_c G_c' B_c^-1 G_c, A'], [A, 0]]
// The equality rows of the engine are 0/1 selections of single velocity components with b = 0 (pinned bodies, axis
// locks: sdf_physics/physics3d/constraints.py:32-145), so x_P = 0 on the pinned set P throughout and K reduces once
// more: pivoted LU of the FREE block M~_FF only ((6 nb - neq)^2: 6 x 6 for the box-on-plane scene instead of
// 100 x 100), multipliers dy = r_P - M~_PF dx_F from the pinned rows.  Same Newton systems, same iterates up to
// round-off; verified against the dense kernels and the oracle in tests/test_dynsolve_gpu.py.
//
// One solver, run by a team of threads per world (SURVEY.md hard part 4: KKT beyond shared memory / body-pair block
// sparsity):
//   * WarpTeam, one warp per world: the whole world in shared memory, up to 64 contacts.  The default.
//   * CtaTeam, one CTA of 256 threads per world: many bodies (6 nb - neq free velocity components up to ~120) and / or
//     many contacts (hundreds).  Shared memory holds only what scales with the number of BODIES; what scales with the
//     number of CONTACTS lives in a caller-provided global workspace (L2 resident, ~1.5 KB per contact), so there is
//     no cap on the contact count.
// Per-body contact lists (ascending contact index, so every sum keeps a fixed order) give G'w, the assembly of M~_FF
// and the per-body gradients: cost O(nF^2 * contacts per body) instead of O(nF^2 * contacts).
#include "dsdf_math.cuh"
#include "dsdf_dense.cuh"
#include "dsdf_contact_rows.cuh"
#include "dsdf_steploop.cuh"
#include "../../include/dsdf_b200.h"

namespace dsdf {

// reference row index of contact-major row (cc, j): [normal nc | friction fd nc | cone nc]
__device__ __forceinline__ int ref_row(int cc, int j, int nc, int fd) {
    return j == 0 ? cc : (j <= fd ? nc + fd * cc + (j - 1) : nc + fd * nc + cc);
}

// ---- teams: who iterates, synchronises, reduces and factors.  Every member is called by all threads of the team.
struct WarpTeam {
    static constexpr int kThreads = 32, kFwdMinBlocks = 12, kBwdMinBlocks = 10;
    static constexpr bool kContactsInSmem = true;      // both layout regions in dynamic shared memory
    __device__ __forceinline__ static int rank() { return threadIdx.x & 31; }
    __device__ __forceinline__ static constexpr int size() { return 32; }
    __device__ __forceinline__ static void sync() { __syncwarp(); }
    __device__ __forceinline__ static double sum(double v) { return warp_sum(v); }
    __device__ __forceinline__ static double min(double v) { return warp_min(v); }
    __device__ __forceinline__ static double max(double v) { return warp_max(v); }
    __device__ __forceinline__ static int lu(double* A, int ld, int n, int* perm) { return warp_lu(A, ld, n, perm); }
    __device__ __forceinline__ static void lu_solve(const double* LU, int ld, int n, const int* perm, const double* b,
                                                    double* x) {
        warp_lu_solve(LU, ld, n, perm, b, x);
    }
};
struct CtaTeam {
    // forward: two CTAs per SM, i.e. at most 128 registers (no spills); backward: no minimum (0), one CTA per SM
    static constexpr int kThreads = 256, kFwdMinBlocks = 2, kBwdMinBlocks = 0;
    static constexpr bool kContactsInSmem = false;     // contact region in the global workspace
    __device__ __forceinline__ static int rank() { return threadIdx.x; }
    __device__ __forceinline__ static int size() { return blockDim.x; }
    __device__ __forceinline__ static void sync() { __syncthreads(); }
    __device__ __forceinline__ static double* red() { __shared__ double r[33]; return r; }
    __device__ __forceinline__ static double sum(double v) { return block_reduce<RED_SUM>(v, red()); }
    __device__ __forceinline__ static double min(double v) { return block_reduce<RED_MIN>(v, red()); }
    __device__ __forceinline__ static double max(double v) { return block_reduce<RED_MAX>(v, red()); }
    __device__ __forceinline__ static int lu(double* A, int ld, int n, int* perm) {
        __shared__ int piv[2];                         // pivot row, failure flag
        if (threadIdx.x == 0) piv[1] = 0;
        __syncthreads();
        block_lu(A, ld, n, perm, &piv[0], &piv[1]);
        __syncthreads();
        return piv[1];
    }
    __device__ __forceinline__ static void lu_solve(const double* LU, int ld, int n, const int* perm, const double* b,
                                                    double* x) {
        block_lu_solve(LU, ld, n, perm, b, x);
    }
};
// i = rank, rank + size, ... < n over the team of the enclosing template (`Team`)
#define TFOR(i, n) for (int i = Team::rank(); i < (n); i += Team::size())

// ---- per-world layout: a body region (shared memory) and a contact region (shared memory after the body region for
// the warp; the global workspace for the CTA).  Offsets in doubles.
enum { DV_S = 0, DV_Z, DV_RZ, DV_T, DV_DSA, DV_DZA, DV_DS, DV_DZ, DV_D, DV_COUNT };   // 9 row vectors per world
enum { DS_XY = 0, DS_RXY, DS_DXYA, DS_DXY, DS_BXY, DS_P, DS_RHS, DS_TF, DS_XF, DS_COUNT };   // nq-sized vectors

struct DynLayout {
    int C, per, R, nz, neq, nq, nF, ldF, nb, half, gs;   // gs = doubles of G per contact = (1 + fd/2) * 12
    size_t oK, oQ, oS, oI, body;
    size_t oG, oYG, oA, oDen, oAP, oV, oMu, oE, oH, oCb, contact;
};

__host__ __device__ inline DynLayout dyn_layout(int nb, int neq, int C, int fd) {
    DynLayout L;
    L.C = C; L.per = 2 + fd; L.R = C * L.per; L.nz = 6 * nb; L.neq = neq; L.nq = L.nz + neq; L.nb = nb;
    L.nF = L.nz - neq; L.ldF = L.nF | 1; L.half = fd / 2; L.gs = (1 + L.half) * 12;
    size_t o = 0;
    // ints first: bstart then sits at the start of dynamic shared memory, a constant address (one register fewer in the
    // one-warp backward, which spills otherwise)
    L.oI = o;   o += ((size_t)nb + 1 + 2 * C + 2 * neq + L.nF + 2 * L.nz + 1) / 2;   // ints: bstart blist eq perm fidx fpos
    L.oK = o;   o += (size_t)L.nF * L.ldF;        // M~_FF, LU in place
    L.oQ = o;   o += (size_t)nb * 36;
    L.oS = o;   o += (size_t)DS_COUNT * L.nq;
    L.body = o;
    o = 0;
    L.oG = o;   o += (size_t)C * L.gs;            // normal row + the first fd/2 friction rows (the rest are their negatives)
    L.oYG = o;  o += (size_t)C * 12;
    L.oA = o;   o += L.R;                         // a = 1/d
    L.oDen = o; o += C;
    L.oAP = o;  o += (size_t)2 * C * L.half;      // per friction pair: 1/a_q + 1/a_{q+half}, 1/a_q - 1/a_{q+half}
    L.oV = o;   o += (size_t)DV_COUNT * L.R;
    L.oMu = o;  o += C;                           // per contact: friction coefficient, restitution, h
    L.oE = o;   o += C;
    L.oH = o;   o += C;
    L.oCb = o;  o += C;                           // 2 ints per contact: its bodies
    L.contact = o;
    return L;
}

struct DynCtx {
    DynLayout L;
    int nc, ni;                                         // active contacts / rows of this world
    double *K, *Qb, *Sv;                                // body region
    int *eq, *perm, *fidx, *fpos, *bstart, *blist;     // fidx[jf] = free dof; fpos[I] = jf (free) or -(m+1) (pinned by
                                                        // row m); blist[bstart[b] .. bstart[b+1]) = 2 contact + side
    double *G, *YG, *a, *den, *AP, *V, *mu, *e, *h;     // contact region
    int* cb;
    __device__ double* vec(int k) const { return V + (size_t)k * L.R; }
    __device__ double* sv(int k) const { return Sv + (size_t)k * L.nq; }
    __device__ int gidx(int c, int k) const { return 6 * cb[2 * c + (k >= 6)] + (k % 6); }
};

__device__ inline DynCtx dyn_ctx(double* body, double* contact, const DynLayout& L) {
    DynCtx c;
    c.L = L;
    c.K = body + L.oK; c.Qb = body + L.oQ; c.Sv = body + L.oS;
    c.bstart = reinterpret_cast<int*>(body + L.oI); c.blist = c.bstart + L.nb + 1; c.eq = c.blist + 2 * L.C;
    c.perm = c.eq + 2 * L.neq; c.fidx = c.perm + L.nF; c.fpos = c.fidx + L.nz;
    c.G = contact + L.oG; c.YG = contact + L.oYG; c.a = contact + L.oA; c.den = contact + L.oDen; c.AP = contact + L.oAP;
    c.V = contact + L.oV; c.mu = contact + L.oMu; c.e = contact + L.oE; c.h = contact + L.oH;
    c.cb = reinterpret_cast<int*>(contact + L.oCb);
    c.nc = c.ni = 0;
    return c;
}

// ---- load one world's problem ------------------------------------------------------------------------------------
template <class Team>
__device__ __forceinline__ void dyn_load(DynCtx& c, int w, const double* p, const double* v, const double* mass,
                                         const double* Ibody, const double* fric, const double* rest, const double* f,
                                         double dtw, const int* count, const int* cbody, const double* cgeo,
                                         const int* eq_rows, int maxc, int fd) {
    const DynLayout& L = c.L;
    const int nb = L.nb, nz = L.nz;
    c.nc = min(min(count[w], maxc), L.C);
    c.ni = c.nc * L.per;
    TFOR(i, 2 * L.neq) c.eq[i] = eq_rows[i];
    TFOR(i, nz) c.fpos[i] = 0;
    Team::sync();
    TFOR(m, L.neq) c.fpos[6 * c.eq[2 * m] + c.eq[2 * m + 1]] = -(m + 1);
    Team::sync();
    if (Team::rank() == 0) {
        int jf = 0;
        for (int i = 0; i < nz; ++i) if (c.fpos[i] == 0) { c.fidx[jf] = i; c.fpos[i] = jf++; }
    }
    TFOR(b, nb) {
        const double* pb = p + ((size_t)w * nb + b) * 7;
        M3<double> Iw = winertia<double>(q4<double>(pb[0], pb[1], pb[2], pb[3]), Ibody + ((size_t)w * nb + b) * 9);
        const double m = mass[(size_t)w * nb + b];
        double* Q = c.Qb + 36 * b;
        for (int e = 0; e < 36; ++e) Q[e] = 0.0;
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) Q[6 * i + j] = Iw.m[3 * i + j];
            Q[6 * (3 + i) + 3 + i] = m;
        }
    }
    TFOR(cc, c.nc) {
        const size_t oo = (size_t)w * maxc + cc;
        const int i1 = cbody[2 * oo], i2 = cbody[2 * oo + 1];
        c.cb[2 * cc] = i1; c.cb[2 * cc + 1] = i2;
        const double* g = cgeo + 10 * oo;
        const V3<double> n = v3<double>(g[0], g[1], g[2]), p1 = v3<double>(g[3], g[4], g[5]), p2 = v3<double>(g[6], g[7], g[8]);
        double* Gc = c.G + (size_t)cc * L.gs;
        row12<double>(p1, p2, n, Gc);
        V3<double> dirs[8];
        fdirs<double>(n, fd, dirs);
        for (int r = 0; r < L.half; ++r) row12<double>(p1, p2, dirs[r], Gc + 12 * (1 + r));   // rows r + half = -rows r
        c.mu[cc] = 0.5 * (fric[(size_t)w * nb + i1] + fric[(size_t)w * nb + i2]);
        c.e[cc] = (rest[(size_t)w * nb + i1] + rest[(size_t)w * nb + i2]) / 2;
    }
    Team::sync();
    // per-body contact lists: entry = 2 * contact + side, ascending contact index (one thread per body).  A contact
    // joins two different bodies, so it appears at most once in a list.
    TFOR(b, nb) {
        int n = 0;
        for (int cc = 0; cc < c.nc; ++cc) n += (c.cb[2 * cc] == b) + (c.cb[2 * cc + 1] == b);
        c.bstart[b + 1] = n;
    }
    Team::sync();
    if (Team::rank() == 0) {
        c.bstart[0] = 0;
        for (int b = 0; b < nb; ++b) c.bstart[b + 1] += c.bstart[b];
    }
    Team::sync();
    TFOR(b, nb) {
        int o = c.bstart[b];
        for (int cc = 0; cc < c.nc; ++cc) {
            if (c.cb[2 * cc] == b) c.blist[o++] = 2 * cc;
            if (c.cb[2 * cc + 1] == b) c.blist[o++] = 2 * cc + 1;
        }
    }
    // u = M v + dt f
    double* pv = c.sv(DS_P);
    TFOR(i, nz) {
        const int b = i / 6, k = i % 6;
        const double* Q = c.Qb + 36 * b;
        double acc = 0.0;
        for (int j = 0; j < 6; ++j) acc += Q[6 * k + j] * v[(size_t)w * nz + 6 * b + j];
        pv[i] = acc + dtw * f[(size_t)w * nz + i];
    }
    // h = [e (Jc v); 0; 0]: one value per contact (normal row), zero on the friction and cone rows
    TFOR(cc, c.nc) {
        const double* Gc = c.G + (size_t)cc * L.gs;
        double jv = 0.0;
        for (int k = 0; k < 12; ++k) jv += Gc[k] * v[(size_t)w * nz + c.gidx(cc, k)];
        c.h[cc] = jv * c.e[cc];
    }
    Team::sync();
}

// (F z)[r] for the engine's F in contact-major rows
__device__ __forceinline__ double Fz_row(const DynCtx& c, const double* z, int r, int fd) {
    const int per = c.L.per, cc = r / per, j = r % per;
    if (j == 0) return 0.0;
    if (j <= fd) return z[cc * per + per - 1];
    double acc = c.mu[cc] * z[cc * per];
    for (int q = 1; q <= fd; ++q) acc -= z[cc * per + q];
    return acc;
}
// out = G x for all rows (contact-major): friction row q + half is the negative of row q, the cone row is zero
template <class Team> __device__ __forceinline__ void Gx_all(const DynCtx& c, const double* x, double* out) {
    const int per = c.L.per, half = c.L.half, rows = 1 + half;
    TFOR(e, c.nc * rows) {
        const int cc = e / rows, j = e % rows;
        const double* Gc = c.G + (size_t)cc * c.L.gs + 12 * j;
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < 12; ++k) acc += Gc[k] * x[c.gidx(cc, k)];
        out[cc * per + j] = acc;
        if (j >= 1) out[cc * per + j + half] = -acc;
        else out[cc * per + per - 1] = 0.0;
    }
    Team::sync();
}
// (G' w)[I] through the contact list of I's body
__device__ __forceinline__ double Gtw_row(const DynCtx& c, const double* w, int I) {
    const int per = c.L.per, half = c.L.half, b = I / 6, k6 = I % 6;
    double acc = 0.0;
    for (int t = c.bstart[b]; t < c.bstart[b + 1]; ++t) {
        const int cc = c.blist[t] >> 1, k = (c.blist[t] & 1) * 6 + k6;
        const double* Gc = c.G + (size_t)cc * c.L.gs + k;
        const double* wc = w + cc * per;
        double a2 = Gc[0] * wc[0];
        for (int q = 1; q <= half; ++q) a2 += Gc[12 * q] * (wc[q] - wc[q + half]);
        acc += a2;
    }
    return acc;
}
// solve B_c u = t for every contact in place on t (contact-major), thread per contact
template <class Team> __device__ __forceinline__ void block_solve(const DynCtx& c, double* t, int fd) {
    const int per = c.L.per;
    TFOR(cc, c.nc) {
        double* tc = t + cc * per;
        const double* ac = c.a + cc * per;
        const double un = tc[0] * ac[0];                 // ac = 1/a: reciprocals of B's diagonal (no fp64 divides here)
        double sum = 0.0;
        for (int q = 1; q <= fd; ++q) sum += tc[q] * ac[q];
        const double ug = (tc[per - 1] - c.mu[cc] * un + sum) * c.den[cc];
        tc[0] = un;
        for (int q = 1; q <= fd; ++q) tc[q] = (tc[q] - ug) * ac[q];
        tc[per - 1] = ug;
    }
    Team::sync();
}

// factor: a = 1/d, den, YG, K = [[Q + sum G' B^-1 G, A'],[A,0]] -> LU.  Returns 1 on a singular K.
template <class Team> __device__ __forceinline__ int dyn_factor(DynCtx& c, const double* d, int fd) {
    const DynLayout& L = c.L;
    const int per = L.per, nF = L.nF, ld = L.ldF, half = L.half;
    // a = 1/d is B's diagonal (batch.py:496); the kernel keeps 1/a and 1/den so the hot loops multiply
    TFOR(r, c.ni) c.a[r] = 1.0 / (1.0 / d[r]);
    Team::sync();
    TFOR(cc, c.nc) {
        const double* ac = c.a + cc * per;
        double dn = 1.0 / d[cc * per + per - 1];
        for (int q = 1; q <= fd; ++q) dn += ac[q];
        c.den[cc] = 1.0 / dn;
    }
    TFOR(e, c.nc * half) {
        const int cc = e / half, q = 1 + e % half;
        const double* ac = c.a + cc * per;
        c.AP[(size_t)2 * e] = ac[q] + ac[q + half];
        c.AP[(size_t)2 * e + 1] = ac[q] - ac[q + half];
    }
    Team::sync();
    TFOR(e, c.nc * 12) {
        const int cc = e / 12, k = e % 12;
        const double* Gc = c.G + (size_t)cc * L.gs + k;
        const double* ap = c.AP + (size_t)2 * cc * half;
        double acc = -c.mu[cc] * Gc[0] * c.a[cc * per];
        for (int q = 1; q <= half; ++q) acc += Gc[12 * q] * ap[2 * (q - 1) + 1];
        c.YG[e] = acc * c.den[cc];
    }
    Team::sync();
    // M~_FF = Q_FF + sum_c G_c' B_c^-1 G_c restricted to the free components; thread per entry.  Entry (If, jf) gathers
    // the contacts that touch BOTH bodies, walking the list of I's body.
    TFOR(e, nF * nF) {
        const int If = e / nF, jf = e % nF, I = c.fidx[If], J = c.fidx[jf], bI = I / 6, bJ = J / 6;
        double acc = bI == bJ ? c.Qb[36 * bI + 6 * (I % 6) + (J % 6)] : 0.0;
        for (int t = c.bstart[bI]; t < c.bstart[bI + 1]; ++t) {
            const int cc = c.blist[t] >> 1, sI = c.blist[t] & 1;
            int kj;
            if (bJ == bI) kj = sI * 6 + J % 6;
            else if (c.cb[2 * cc + (1 - sI)] == bJ) kj = (1 - sI) * 6 + J % 6;
            else continue;
            const int ki = sI * 6 + I % 6;
            const double* Gc = c.G + (size_t)cc * L.gs;
            const double* ap = c.AP + (size_t)2 * cc * half;
            double a2 = Gc[ki] * (Gc[kj] * c.a[cc * per]);
            const double yg = c.YG[cc * 12 + kj];
            for (int q = 1; q <= half; ++q)
                a2 += Gc[12 * q + ki] * (Gc[12 * q + kj] * ap[2 * (q - 1)] - yg * ap[2 * (q - 1) + 1]);
            acc += a2;
        }
        c.K[If * ld + jf] = acc;
    }
    Team::sync();
    return Team::lu(c.K, ld, nF, c.perm);
}

// dx of [[M~, A'], [A, 0]] [dx; dy] = rhs with A a 0/1 selection of the pinned components and rhs_y = 0 (b = 0, x_P = 0):
// dx_P = rhs_y (= 0), dx_F = (M~_FF)^-1 rhs_F.  The multipliers dy follow from the pinned rows of the un-reduced
// system once dz is known: dy = -rx_P - (G' dz)_P - (Q dx)_P   (see dyn_solve).
template <class Team> __device__ inline void kkt_solve(DynCtx& c, const double* rhs, double* dxy) {
    const DynLayout& L = c.L;
    const int nz = L.nz, nF = L.nF, ld = L.ldF;
    double *tF = c.sv(DS_TF), *xF = c.sv(DS_XF);
    TFOR(jf, nF) tF[jf] = rhs[c.fidx[jf]];
    Team::sync();
    Team::lu_solve(c.K, ld, nF, c.perm, tF, xF);
    TFOR(I, nz) { const int fp = c.fpos[I]; dxy[I] = fp >= 0 ? xF[fp] : rhs[nz + (-fp - 1)]; }
    Team::sync();
}

// KKT solve (batch.py:380-410 semantics).  rxy = [rx; ry] (NULL = 0), rs (NULL = 0), rz (NULL = 0).
// Outputs dxy = [dx; dy], ds, dz.  Scratch: vec(DV_T), sv(DS_RHS).
template <class Team>
__device__ __forceinline__ void dyn_solve(DynCtx& c, const double* d, int fd, const double* rxy, const double* rs,
                                          const double* rz, double* dxy, double* ds, double* dz) {
    const DynLayout& L = c.L;
    const int nz = L.nz, nq = L.nq;
    double* t = c.vec(DV_T);
    double* rhs = c.sv(DS_RHS);
    TFOR(r, c.ni) { const double tv = (rz ? rz[r] : 0.0) - (rs ? rs[r] / d[r] : 0.0); t[r] = tv; dz[r] = tv; }
    Team::sync();
    block_solve<Team>(c, t, fd);                                    // t <- u = B^-1 t (dz keeps a copy of t)
    TFOR(I, nq) {
        double acc = rxy ? -rxy[I] : 0.0;
        if (I < nz) acc -= Gtw_row(c, t, I);
        rhs[I] = acc;
    }
    Team::sync();
    kkt_solve<Team>(c, rhs, dxy);
    double* gx = t;                                                 // t is dead from here on
    Gx_all<Team>(c, dxy, gx);
    TFOR(r, c.ni) dz[r] = gx[r] + dz[r];                            // G dx + t
    Team::sync();
    block_solve<Team>(c, dz, fd);
    TFOR(m, L.neq) {                                                // multipliers of the pinned rows
        const int b = c.eq[2 * m], k = c.eq[2 * m + 1], I = 6 * b + k;
        double acc = (rxy ? -rxy[I] : 0.0) - Gtw_row(c, dz, I);
        for (int j = 0; j < 6; ++j) acc -= c.Qb[36 * b + 6 * k + j] * dxy[6 * b + j];
        dxy[nz + m] = acc;
    }
    TFOR(r, c.ni) ds[r] = ((rs ? -rs[r] : 0.0) - dz[r]) / d[r];
    Team::sync();
}

template <class Team> __device__ __forceinline__ double dyn_ratio_step(const DynCtx& c, const double* v, const double* dv) {
    double mx = -INFINITY;
    TFOR(r, c.ni) mx = fmax(mx, -v[r] / dv[r]);
    mx = Team::max(mx);
    const double repl = fmax(1.0, mx);
    double mn = INFINITY;
    TFOR(r, c.ni) mn = fmin(mn, dv[r] > 0.0 ? repl : -v[r] / dv[r]);
    return Team::min(mn);
}

// work: the global workspace of the CTA kernel (contact regions, one per world); unused by the warp kernel
template <class Team>
__global__ void __launch_bounds__(Team::kThreads, Team::kFwdMinBlocks)
dyn_forward_kernel(const double* __restrict__ p, const double* __restrict__ v, const double* __restrict__ mass,
                   const double* __restrict__ Ibody, const double* __restrict__ fric, const double* __restrict__ rest,
                   const double* __restrict__ f, const double* __restrict__ dt, const unsigned char* __restrict__ active,
                   const int* __restrict__ count, const int* __restrict__ cbody, const double* __restrict__ cgeo,
                   const int* __restrict__ eq_rows, int nb, int neq, int maxc, int C, int fd,
                   double eps, int not_improved_lim, int max_iter,
                   double* __restrict__ xo, double* __restrict__ nvo, double* __restrict__ nuo, double* __restrict__ lamo,
                   double* __restrict__ so, int* __restrict__ status_o, int* __restrict__ iters_o,
                   const int* __restrict__ vmap, int* __restrict__ ctrl, int cmin, int last_class,
                   double* __restrict__ work) {
    extern __shared__ double smd[];
    // loop mode (ctrl != NULL, dsdf_steploop.cu): CTA w solves virtual world w = one attempt (its own dt[w]) of the real
    // world ws = vmap[w], whose state / parameters / contacts are read in place; outputs are indexed by w
    const int w = blockIdx.x;
    if (ctrl && (loop_idle(ctrl) || w >= ctrl[CT_NVIRT])) return;
    const int ws = vmap ? vmap[w] : w;
    const DynLayout L = dyn_layout(nb, neq, C, fd);
    const int nz = L.nz, nq = L.nq, per = L.per;
    if (active && !active[w]) {               // inactive world: velocity passes through
        if (nvo) TFOR(i, nz) nvo[(size_t)w * nz + i] = v[(size_t)ws * nz + i];
        return;
    }
    // contact-count classes: one launch sized for the typical count, one for the few worlds with many contacts (a world
    // that gave up halving keeps a penetrating state with dozens of contacts; sizing every CTA for it costs occupancy)
    if (count[ws] <= cmin || (count[ws] > C && !last_class)) return;
    if (count[ws] > C) {                      // more contacts than this launch's layout holds
        TFOR(i, nz) { xo[(size_t)w * nz + i] = NAN; if (nvo) nvo[(size_t)w * nz + i] = NAN; }
        if (Team::rank() == 0) {
            status_o[w] = DSDF_LCP_TOO_LARGE; if (iters_o) iters_o[w] = 0;
            if (ctrl) atomicOr(&ctrl[CT_ABORT], DSDF_STEP_DYN_SMEM);      // the host re-launches with a larger C
        }
        return;
    }
    DynCtx c = dyn_ctx(smd, Team::kContactsInSmem ? smd + L.body : work + (size_t)w * L.contact, L);
    dyn_load<Team>(c, ws, p, v, mass, Ibody, fric, rest, f, dt[w], count, cbody, cgeo, eq_rows, maxc, fd);
    auto hrow = [&](int r) { return (r % per == 0) ? c.h[r / per] : 0.0; };
    const int niCap = maxc * per;
    TFOR(r, niCap) { lamo[(size_t)w * niCap + r] = 0.0; so[(size_t)w * niCap + r] = 0.0; }
    const int ni = c.ni;
    double *s = c.vec(DV_S), *z = c.vec(DV_Z), *rz = c.vec(DV_RZ), *dsa = c.vec(DV_DSA),
           *dza = c.vec(DV_DZA), *ds = c.vec(DV_DS), *dz = c.vec(DV_DZ),
           *d = c.vec(DV_D);
    double *xy = c.sv(DS_XY), *rxy = c.sv(DS_RXY), *dxya = c.sv(DS_DXYA), *dxy = c.sv(DS_DXY), *bxy = c.sv(DS_BXY),
           *pv = c.sv(DS_P);
    int status = 0, iters = 0;
    // One loop for the initial point (it = -1; batch.py:84-110: d = 1, solve_kkt(p, 0, -h, -b), shift s, z >= 1) and the
    // interior-point iterations (batch.py:115-231), so that the factorisation and the KKT solve are instantiated ONCE:
    // the kernel is instruction-cache bound otherwise (29 k SASS instructions with the phases written out).
    bool have_best = false;
    double best_res = INFINITY, mu_gap = 0.0, sz = 0.0;
    int stalled = 0;
    for (int it = -1; it < max_iter; ++it) {
        double res = 0.0;
        if (it < 0) {
            TFOR(r, ni) { d[r] = 1.0; rz[r] = -hrow(r); }
            TFOR(i, nq) rxy[i] = i < nz ? pv[i] : 0.0;      // ry = -b = 0
        } else {
            // residuals (batch.py:117-131)
            double nrx = 0.0, nry = 0.0, nrz = 0.0;
            sz = 0.0;
            TFOR(I, nq) {
                double acc;
                if (I < nz) {
                    const int b = I / 6, k = I % 6;
                    const int fp = c.fpos[I];
                    const double ay = fp < 0 ? xy[nz + (-fp - 1)] : 0.0;
                    double qx = 0.0;
                    for (int j = 0; j < 6; ++j) qx += xy[6 * b + j] * c.Qb[36 * b + 6 * k + j];
                    acc = ay + Gtw_row(c, z, I) + qx + pv[I];
                    nrx += acc * acc;
                } else {
                    const int m = I - nz;
                    acc = xy[6 * c.eq[2 * m] + c.eq[2 * m + 1]];          // A x - b, b = 0
                    nry += acc * acc;
                }
                rxy[I] = acc;
            }
            Gx_all<Team>(c, xy, c.vec(DV_T));
            TFOR(r, ni) {
                const double val_ = c.vec(DV_T)[r] + s[r] - hrow(r) - Fz_row(c, z, r, fd);
                rz[r] = val_;
                nrz += val_ * val_;
                sz += s[r] * z[r];
            }
            nrx = Team::sum(nrx); nry = Team::sum(nry); nrz = Team::sum(nrz); sz = Team::sum(sz);
            mu_gap = fabs(sz / ni);
            res = (L.neq > 0 ? sqrt(nry) : 0.0) + sqrt(nrz) + sqrt(nrx) + ni * mu_gap;
            TFOR(r, ni) d[r] = z[r] / s[r];
        }
        Team::sync();
        if (dyn_factor<Team>(c, d, fd)) { status |= DSDF_LCP_FACTOR_FAIL; if (it >= 0) break; }
        if (it >= 0) {
            iters = it + 1;
            if (!have_best || res < best_res) {
                have_best = true; best_res = res; stalled = 0;
                TFOR(i, nq) bxy[i] = xy[i];
                TFOR(r, ni) {        // best (lam, s) go straight to the outputs (reference row order)
                    const int rr = ref_row(r / per, r % per, c.nc, fd);
                    lamo[(size_t)w * niCap + rr] = z[r];
                    so[(size_t)w * niCap + rr] = s[r];
                }
            } else {
                ++stalled;
            }
            if (stalled == not_improved_lim || best_res < eps || mu_gap > 1e32) break;
        }
        bool init_done = false;
        for (int pass = 0; pass < 2; ++pass) {
            // pass 0: initial solve (it < 0) or affine direction (rs = z); pass 1: corrector (rs in rz)
            const double* a_rxy = pass == 0 ? rxy : nullptr;
            const double* a_rs = pass == 0 ? (it < 0 ? nullptr : z) : rz;
            const double* a_rz = pass == 0 ? rz : nullptr;
            double* o_xy = pass == 0 ? (it < 0 ? xy : dxya) : dxy;
            double* o_s = pass == 0 ? (it < 0 ? s : dsa) : ds;
            double* o_z = pass == 0 ? (it < 0 ? z : dza) : dz;
            dyn_solve<Team>(c, d, fd, a_rxy, a_rs, a_rz, o_xy, o_s, o_z);
            if (it < 0) {
                if (ni > 0) {                                   // batch.py:100-110
                    double ms = INFINITY, mz = INFINITY;
                    TFOR(r, ni) { ms = fmin(ms, s[r]); mz = fmin(mz, z[r]); }
                    ms = Team::min(ms); mz = Team::min(mz);
                    TFOR(r, ni) {
                        if (ms < 0.0) s[r] -= ms - 1.0;
                        if (mz < 0.0) z[r] -= mz - 1.0;
                    }
                    Team::sync();
                }
                init_done = true;
                break;
            }
            if (pass == 0) {
                double alpha = fmin(fmin(dyn_ratio_step<Team>(c, z, dza), dyn_ratio_step<Team>(c, s, dsa)), 1.0);
                double t3 = 0.0;
                TFOR(r, ni) t3 += (s[r] + alpha * dsa[r]) * (z[r] + alpha * dza[r]);
                t3 = Team::sum(t3);
                const double r3 = t3 / sz, sig = r3 * r3 * r3;
                // corrector: rs = (-mu sig + dsa dza) / s  (stored in rz, which is free now)
                TFOR(r, ni) rz[r] = (-mu_gap * sig + dsa[r] * dza[r]) / s[r];
                Team::sync();
            }
        }
        if (init_done) {
            if (ni == 0) {                                      // no contacts: the equality-constrained solve is the answer
                TFOR(i, nq) bxy[i] = xy[i];
                have_best = true;
                break;
            }
            continue;
        }
        TFOR(i, nq) dxy[i] += dxya[i];
        TFOR(r, ni) { ds[r] += dsa[r]; dz[r] += dza[r]; }
        Team::sync();
        const double alpha = fmin(0.999 * fmin(dyn_ratio_step<Team>(c, z, dz), dyn_ratio_step<Team>(c, s, ds)), 1.0);
        TFOR(i, nq) xy[i] += alpha * dxy[i];
        TFOR(r, ni) { s[r] += alpha * ds[r]; z[r] += alpha * dz[r]; }
        Team::sync();
    }
    if (ni > 0 && have_best && best_res > 1.0) status |= DSDF_LCP_INACCURATE;
    Team::sync();
    TFOR(i, nz) {
        xo[(size_t)w * nz + i] = have_best ? bxy[i] : NAN;
        if (nvo) nvo[(size_t)w * nz + i] = have_best ? -bxy[i] : NAN;       // engines.py:81-82
    }
    TFOR(m, L.neq) nuo[(size_t)w * L.neq + m] = have_best ? bxy[nz + m] : NAN;
    if (Team::rank() == 0) { status_o[w] = status; if (iters_o) iters_o[w] = iters; }
}

// ---- backward: implicit differentiation at the solution, contracted straight onto the physical inputs ---------
template <class Team>
__global__ void __launch_bounds__(Team::kThreads, Team::kBwdMinBlocks)
dyn_backward_kernel(const double* __restrict__ p, const double* __restrict__ v, const double* __restrict__ mass,
                    const double* __restrict__ Ibody, const double* __restrict__ fric, const double* __restrict__ rest,
                    const double* __restrict__ f, const double* __restrict__ dt, const unsigned char* __restrict__ active,
                    const int* __restrict__ count, const int* __restrict__ cbody, const double* __restrict__ cgeo,
                    const int* __restrict__ eq_rows, int nb, int neq, int maxc, int C, int fd,
                    int stop_contact_grad, int stop_friction_grad,
                    const double* __restrict__ xs, const double* __restrict__ lams, const double* __restrict__ ss,
                    const double* __restrict__ gnv,
                    double* __restrict__ gp, double* __restrict__ gv, double* __restrict__ gmass, double* __restrict__ gI,
                    double* __restrict__ gfric, double* __restrict__ grest, double* __restrict__ gf,
                    double* __restrict__ gdt, double* __restrict__ ggeo, int cmin, int last_class,
                    double* __restrict__ work) {
    extern __shared__ double smd[];
    const int w = blockIdx.x;
    const DynLayout L = dyn_layout(nb, neq, C, fd);
    const int nz = L.nz, nq = L.nq, per = L.per, niCap = maxc * per;
    const bool masked = active && !active[w];
    // contact-count classes (see dyn_forward_kernel): masked worlds are written by the first-class launch only
    if (masked ? cmin >= 0 : (count[w] <= cmin || (count[w] > C && !last_class))) return;
    const bool on = !masked && count[w] <= C;
    if (!on) {
        TFOR(i, nb * 7) gp[(size_t)w * nb * 7 + i] = 0.0;
        TFOR(i, nz) {                                       // inactive world: new_v = v
            gv[(size_t)w * nz + i] = masked ? gnv[(size_t)w * nz + i] : 0.0;
            gf[(size_t)w * nz + i] = 0.0;
        }
        TFOR(i, nb) { gmass[(size_t)w * nb + i] = 0.0; gfric[(size_t)w * nb + i] = 0.0; grest[(size_t)w * nb + i] = 0.0; }
        TFOR(i, nb * 9) gI[(size_t)w * nb * 9 + i] = 0.0;
        TFOR(i, maxc * 10) ggeo[(size_t)w * maxc * 10 + i] = 0.0;
        if (Team::rank() == 0) gdt[w] = 0.0;
        return;
    }
    DynCtx c = dyn_ctx(smd, Team::kContactsInSmem ? smd + L.body : work + (size_t)w * L.contact, L);
    const double dtw = dt[w];
    dyn_load<Team>(c, w, p, v, mass, Ibody, fric, rest, f, dtw, count, cbody, cgeo, eq_rows, maxc, fd);
    const int ni = c.ni, nc = c.nc;
    const double* vw = v + (size_t)w * nz;
    double *lam = c.vec(DV_Z), *d = c.vec(DV_D), *dl = c.vec(DV_DZ), *ds = c.vec(DV_DS);
    double *g = c.sv(DS_RXY), *dxy = c.sv(DS_DXY), *zh = c.sv(DS_XY);
    TFOR(i, nq) { g[i] = i < nz ? -gnv[(size_t)w * nz + i] : 0.0; zh[i] = i < nz ? xs[(size_t)w * nz + i] : 0.0; }
    TFOR(r, ni) {
        const int rr = ref_row(r / per, r % per, nc, fd);
        lam[r] = lams[(size_t)w * niCap + rr];
        d[r] = fmax(lam[r], 1e-8) / fmax(ss[(size_t)w * niCap + rr], 1e-8);
    }
    Team::sync();
    dyn_factor<Team>(c, d, fd);
    dyn_solve<Team>(c, d, fd, g, nullptr, nullptr, dxy, ds, dl);      // dx = dxy[:nz], dlam = dl
    // ---- dp (= du), dh, and the outer-product gradients, contracted on the fly
    // gv = M' du + Jc' (e o dh),  dh = -dlam ; gf = dt du ; gdt = f . du
    TFOR(I, nz) {
        const int b = I / 6, k = I % 6;
        double acc = 0.0;
        for (int i = 0; i < 6; ++i) acc += c.Qb[36 * b + 6 * i + k] * dxy[6 * b + i];
        for (int t = c.bstart[b]; t < c.bstart[b + 1]; ++t) {
            const int cc = c.blist[t] >> 1, kk = (c.blist[t] & 1) * 6 + k;
            acc += c.G[(size_t)cc * L.gs + kk] * c.e[cc] * (-dl[cc * per]);
        }
        gv[(size_t)w * nz + I] = acc;
        gf[(size_t)w * nz + I] = dtw * dxy[I];
    }
    {
        double acc = 0.0;
        TFOR(I, nz) acc += f[(size_t)w * nz + I] * dxy[I];
        acc = Team::sum(acc);
        if (Team::rank() == 0) gdt[w] = acc;
    }
    // per body: dM = dQ + du v' with dQ = 1/2 (dx z' + z dx')
    TFOR(b, nb) {
        double dMb[36];
        for (int i = 0; i < 6; ++i)
            for (int j = 0; j < 6; ++j)
                dMb[6 * i + j] = 0.5 * (dxy[6 * b + i] * zh[6 * b + j] + zh[6 * b + i] * dxy[6 * b + j]) +
                                 dxy[6 * b + i] * vw[6 * b + j];
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
    }
    TFOR(b, nb) {                        // a pass of its own: keeps the one-warp loop above free of spills
        double gfr = 0.0, gre = 0.0;
        for (int t = c.bstart[b]; t < c.bstart[b + 1]; ++t) {
            const int cc = c.blist[t] >> 1;
            // dF[cone row, normal col] = dlam_cone * lam_normal
            gfr += 0.5 * dl[cc * per + per - 1] * lam[cc * per];
            double jv = 0.0;
            for (int k = 0; k < 12; ++k) jv += c.G[(size_t)cc * L.gs + k] * vw[c.gidx(cc, k)];
            gre += 0.5 * (-dl[cc * per]) * jv;
        }
        gfric[(size_t)w * nb + b] = gfr;
        grest[(size_t)w * nb + b] = gre;
    }
    // contact geometry: dG row = dlam_r z' + lam_r dx'  (+ dh e v' on normal rows)
    TFOR(t, maxc * 10) {
        const int cc = t / 10, comp = t % 10;
        double acc = 0.0;
        if (cc < nc && comp < 9) {
            const double* gg = cgeo + 10 * ((size_t)w * maxc + cc);
            auto D = [&](int k) { return Dual(gg[k], comp == k ? 1.0 : 0.0); };
            const V3<Dual> n = v3<Dual>(D(0), D(1), D(2)), p1 = v3<Dual>(D(3), D(4), D(5)), p2 = v3<Dual>(D(6), D(7), D(8));
            Dual row[12];
            if (!stop_contact_grad) {
                row12<Dual>(p1, p2, n, row);
                const double dlr = dl[cc * per], lr = lam[cc * per], dh = -dlr;
                for (int k = 0; k < 12; ++k) {
                    const int I = c.gidx(cc, k);
                    acc += (dlr * zh[I] + lr * dxy[I] + dh * c.e[cc] * vw[I]) * row[k].d;
                }
            }
            if (!stop_friction_grad) {
                V3<Dual> dirs[8];
                fdirs<Dual>(n, fd, dirs);
                for (int r = 0; r < fd; ++r) {
                    row12<Dual>(p1, p2, dirs[r], row);
                    const double dlr = dl[cc * per + 1 + r], lr = lam[cc * per + 1 + r];
                    for (int k = 0; k < 12; ++k) {
                        const int I = c.gidx(cc, k);
                        acc += (dlr * zh[I] + lr * dxy[I]) * row[k].d;
                    }
                }
            }
        }
        ggeo[(size_t)w * maxc * 10 + t] = acc;
    }
}

}  // namespace dsdf

using namespace dsdf;

// ---- host dispatch ---------------------------------------------------------------------------------------------
// The one-warp kernel holds a whole world in shared memory: at most 64 contacts, and only for worlds whose layout at 16
// contacts fits in 48 KB (several CTAs per SM).  Every other world runs on the one-CTA kernel.
static constexpr int kWarpMaxContacts = 64;
static constexpr size_t kWarpSmemBytes = 48 * 1024, kMaxSmemBytes = 227 * 1024;

// dynamic shared memory of a launch sized for C contacts
static size_t dyn_smem(bool contacts_in_smem, int nb, int neq, int C, int fd) {
    const DynLayout L = dyn_layout(nb, neq, C, fd);
    return (L.body + (contacts_in_smem ? L.contact : 0)) * sizeof(double);
}

// Argument checks of both launchers: clamps *C to maxc and returns the launch's dynamic shared memory in *smem.
template <class Team> static int dyn_check(int W, int nb, int neq, int maxc, int* C, int fd, const double* work,
                                           size_t* smem) {
    if (W <= 0 || nb <= 0 || neq < 0 || maxc <= 0 || (fd != 8 && fd != 4) || (!Team::kContactsInSmem && !work))
        return -1;
    if (*C <= 0 || *C > maxc) *C = maxc;
    if (Team::kContactsInSmem && *C > kWarpMaxContacts) return -2;
    *smem = dyn_smem(Team::kContactsInSmem, nb, neq, *C, fd);
    if (*smem > kMaxSmemBytes) return -2;
    return 0;
}

// One launch of a plan: sized for C contacts, it solves the worlds with count_min < count <= C (and, if last_class,
// reports those above C as DSDF_LCP_TOO_LARGE).
struct DynLaunch { bool cta; int C, count_min, last_class; };

// The contact-count classes that cover a batch whose worlds have at most ncontacts_large contacts, most of them at most
// ncontacts_small: one-warp launches for both classes (capped at 64 contacts) and a one-CTA launch for the worlds above
// 64.  Worlds too large for the one-warp kernel, or force_cta, run on the one-CTA kernel in one class.  Returns the
// number of launches (<= 3), or -1.
static int dyn_plan(int nb, int neq, int fd, int small, int large, int force_cta, DynLaunch* out) {
    if (small <= 0 || large <= 0) return -1;
    if (force_cta || dyn_smem(true, nb, neq, 16, fd) > kWarpSmemBytes) {
        out[0] = {true, large, -1, 1};
        return 1;
    }
    const int wl = large < kWarpMaxContacts ? large : kWarpMaxContacts, ws = small < wl ? small : wl;
    const bool two = wl > ws, beyond = large > kWarpMaxContacts;
    int n = 0;
    out[n++] = {false, ws, -1, (two || beyond) ? 0 : 1};
    if (two) out[n++] = {false, wl, ws, beyond ? 0 : 1};
    if (beyond) out[n++] = {true, large, kWarpMaxContacts, 1};
    return n;
}

template <class Team>
static int dyn_launch_forward(const double* p, const double* v, const double* mass, const double* Ibody,
                              const double* fric, const double* rest, const double* f, const double* dt,
                              const unsigned char* active, const int32_t* count, const int32_t* cbody, const double* cgeo,
                              const int32_t* eq_rows, int W, int nb, int neq, int maxc, int ncontacts, int fric_dirs,
                              double eps, int not_improved_lim, int max_iter,
                              double* x, double* new_v, double* nu, double* lam, double* s, int32_t* status,
                              int32_t* iters, const int32_t* vmap, int32_t* ctrl, int count_min, int last_class,
                              double* work, void* stream) {
    static size_t granted = 0;
    size_t smem;
    int C = ncontacts;
    int rc = dyn_check<Team>(W, nb, neq, maxc, &C, fric_dirs, work, &smem);
    if (rc) return rc;
    cudaError_t e = ensure_smem(dyn_forward_kernel<Team>, smem, &granted);
    if (e != cudaSuccess) return (int)e;
    dyn_forward_kernel<Team><<<W, Team::kThreads, smem, (cudaStream_t)stream>>>(
        p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, cgeo, eq_rows, nb, neq, maxc, C, fric_dirs, eps,
        not_improved_lim, max_iter, x, new_v, nu, lam, s, status, iters, vmap, ctrl, count_min, last_class, work);
    return (int)cudaGetLastError();
}

template <class Team>
static int dyn_launch_backward(const double* p, const double* v, const double* mass, const double* Ibody,
                               const double* fric, const double* rest, const double* f, const double* dt,
                               const unsigned char* active, const int32_t* count, const int32_t* cbody,
                               const double* cgeo, const int32_t* eq_rows, int W, int nb, int neq, int maxc,
                               int ncontacts, int fric_dirs, int stop_contact_grad, int stop_friction_grad,
                               const double* x, const double* lam, const double* s, const double* g_new_v,
                               double* gp, double* gv, double* gmass, double* gI, double* gfric, double* grest,
                               double* gf, double* gdt, double* ggeo, int count_min, int last_class,
                               double* work, void* stream) {
    static size_t granted = 0;
    size_t smem;
    int C = ncontacts;
    int rc = dyn_check<Team>(W, nb, neq, maxc, &C, fric_dirs, work, &smem);
    if (rc) return rc;
    cudaError_t e = ensure_smem(dyn_backward_kernel<Team>, smem, &granted);
    if (e != cudaSuccess) return (int)e;
    dyn_backward_kernel<Team><<<W, Team::kThreads, smem, (cudaStream_t)stream>>>(
        p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, cgeo, eq_rows, nb, neq, maxc, C, fric_dirs,
        stop_contact_grad, stop_friction_grad, x, lam, s, g_new_v, gp, gv, gmass, gI, gfric, grest, gf, gdt, ggeo,
        count_min, last_class, work);
    return (int)cudaGetLastError();
}

extern "C" {

int dsdf_dynamics_plan(int W, int nb, int neq, int fric_dirs, int ncontacts_small, int ncontacts_large, int force_cta,
                       size_t* workspace_bytes) {
    if (W <= 0 || nb <= 0 || neq < 0 || (fric_dirs != 8 && fric_dirs != 4)) return -1;
    DynLaunch plan[3];
    const int n = dyn_plan(nb, neq, fric_dirs, ncontacts_small, ncontacts_large, force_cta, plan);
    if (n < 0) return n;
    size_t ws = 0;
    for (int i = 0; i < n; ++i) {
        if (dyn_smem(!plan[i].cta, nb, neq, plan[i].C, fric_dirs) > kMaxSmemBytes) return -2;
        if (plan[i].cta) ws = (size_t)W * dyn_layout(nb, neq, plan[i].C, fric_dirs).contact * sizeof(double);
    }
    if (workspace_bytes) *workspace_bytes = ws;
    return n;
}

int dsdf_dynamics_solve(const double* p, const double* v, const double* mass, const double* Ibody,
                        const double* fric, const double* rest, const double* f, const double* dt,
                        const unsigned char* active, const int32_t* count, const int32_t* cbody, const double* cgeo,
                        const int32_t* eq_rows, int W, int nb, int neq, int maxc, int ncontacts_small,
                        int ncontacts_large, int force_cta, int fric_dirs, double eps, int not_improved_lim,
                        int max_iter, double* x, double* new_v, double* nu, double* lam, double* s, int32_t* status,
                        int32_t* iters, const int32_t* vmap, int32_t* ctrl, double* workspace, void* stream) {
    DynLaunch plan[3];
    const int n = dyn_plan(nb, neq, fric_dirs, ncontacts_small, ncontacts_large, force_cta, plan);
    if (n < 0) return n;
    for (int i = 0; i < n; ++i) {
        const DynLaunch& d = plan[i];
        const int rc = (d.cta ? dyn_launch_forward<CtaTeam> : dyn_launch_forward<WarpTeam>)(
            p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, cgeo, eq_rows, W, nb, neq, maxc, d.C, fric_dirs,
            eps, not_improved_lim, max_iter, x, new_v, nu, lam, s, status, iters, vmap, ctrl, d.count_min,
            d.last_class, workspace, stream);
        if (rc) return rc;
    }
    return 0;
}

int dsdf_dynamics_solve_backward(const double* p, const double* v, const double* mass, const double* Ibody,
                                 const double* fric, const double* rest, const double* f, const double* dt,
                                 const unsigned char* active, const int32_t* count, const int32_t* cbody,
                                 const double* cgeo, const int32_t* eq_rows, int W, int nb, int neq, int maxc,
                                 int ncontacts_small, int ncontacts_large, int force_cta, int fric_dirs,
                                 int stop_contact_grad, int stop_friction_grad,
                                 const double* x, const double* lam, const double* s, const double* g_new_v,
                                 double* gp, double* gv, double* gmass, double* gI, double* gfric, double* grest,
                                 double* gf, double* gdt, double* ggeo, double* workspace, void* stream) {
    DynLaunch plan[3];
    const int n = dyn_plan(nb, neq, fric_dirs, ncontacts_small, ncontacts_large, force_cta, plan);
    if (n < 0) return n;
    for (int i = 0; i < n; ++i) {
        const DynLaunch& d = plan[i];
        const int rc = (d.cta ? dyn_launch_backward<CtaTeam> : dyn_launch_backward<WarpTeam>)(
            p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, cgeo, eq_rows, W, nb, neq, maxc, d.C, fric_dirs,
            stop_contact_grad, stop_friction_grad, x, lam, s, g_new_v, gp, gv, gmass, gI, gfric, grest, gf, gdt, ggeo,
            d.count_min, d.last_class, workspace, stream);
        if (rc) return rc;
    }
    return 0;
}

}  // extern "C"
