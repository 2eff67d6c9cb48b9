// Pose gradients of the contact geometry: VJP of the reference's grad-enabled second _compute_contacts
// (sdf_physics/physics3d/contacts.py:262-264) by forward-mode duals of the same device code.  Separate translation unit
// from the detection kernel so that the small backward kernel keeps its math inlined (the detection kernel outlines it
// to fit the instruction cache); same -fmad=false so both evaluate the identical expression tree.
#include "dsdf_contact_geo.cuh"
#include "../../include/dsdf_b200.h"

namespace dsdf {

// One CTA per world.  Work item = (contact k, seed j): j < 7 seeds component j of body i1's pose, 7 <= j < 14 component
// j - 7 of body i2's (forward-mode dual through contact_geometry); the partials of every contact go to shared memory and
// thread (body, component) then sums them over the contacts in index order (deterministic).
// With gshape != NULL the kernel also differentiates through the SHAPES (sdf_physics/physics3d/contacts.py:262-264 is
// grad-enabled w.r.t. everything the bodies carry: SDF parameters, scale and the mesh vertices): seeds 14..17 = b1's
// [a, b, c, scale], 18..21 = b2's, 22..24 = the body-frame point c_tri = sum(abc * verts of the face) on b1's mesh, whose
// gradient gctri (W,maxc,3) the caller scatters onto the vertices.
enum { GEO_POSE_SEEDS = 14, GEO_ALL_SEEDS = 25 };

__global__ void __launch_bounds__(128, 5)
contact_geometry_bwd_kernel(const BodyGeom* __restrict__ geom, const double* __restrict__ p,
                            const double* __restrict__ shape, int nb, double fd_eps, int detach_b2, int maxc,
                            const int* __restrict__ count, const int* __restrict__ cbody, const int* __restrict__ cface,
                            const double* __restrict__ cabc, const double* __restrict__ ggeo, double* __restrict__ gp,
                            const int* __restrict__ wmap, double* __restrict__ gshape, double* __restrict__ gctri) {
    extern __shared__ double part[];          // [maxc][nseeds]
    const int w = blockIdx.x;
    const int wg = wmap ? wmap[w] : w;        // row w of a compact batch belongs to world wg (shapes, per-world geometry)
    const int nc = min(count[w], maxc);
    const int nseeds = gshape ? GEO_ALL_SEEDS : GEO_POSE_SEEDS;
    for (int item = threadIdx.x; item < nc * nseeds; item += blockDim.x) {
        const int k = item / nseeds, j = item % nseeds;
        const size_t oo = (size_t)w * maxc + k;
        const int i1 = cbody[2 * oo], i2 = cbody[2 * oo + 1];
        const BodyGeom g1 = world_geom(geom[i1], wg);
        const SdfShape s1 = body_shape(g1, shape, wg, nb, i1);
        const SdfShape s2 = body_shape(geom[i2], shape, wg, nb, i2);
        const double* P1 = p + ((size_t)w * nb + i1) * 7;
        const double* P2 = p + ((size_t)w * nb + i2) * 7;
        const int s1seed = j < 7 ? j : -1, s2seed = (j >= 7 && j < 14) ? j - 7 : -1;
        auto D = [](const double* s, int k_, int seed) { return Dual(s[k_], seed == k_ ? 1.0 : 0.0); };
        Q4<Dual> q1 = q4<Dual>(D(P1, 0, s1seed), D(P1, 1, s1seed), D(P1, 2, s1seed), D(P1, 3, s1seed));
        V3<Dual> x1 = v3<Dual>(D(P1, 4, s1seed), D(P1, 5, s1seed), D(P1, 6, s1seed));
        Q4<Dual> q2 = q4<Dual>(D(P2, 0, s2seed), D(P2, 1, s2seed), D(P2, 2, s2seed), D(P2, 3, s2seed));
        V3<Dual> x2 = v3<Dual>(D(P2, 4, s2seed), D(P2, 5, s2seed), D(P2, 6, s2seed));
        const int f = cface[oo];
        const V3<double> va = load_vert(g1, wg, g1.faces[3 * f]), vb = load_vert(g1, wg, g1.faces[3 * f + 1]),
                         vc = load_vert(g1, wg, g1.faces[3 * f + 2]);
        const double a = cabc[3 * oo], b = cabc[3 * oo + 1], c = cabc[3 * oo + 2];
        const V3<double> ct = v3<double>(va.x * a + vb.x * b + vc.x * c, va.y * a + vb.y * b + vc.y * c,
                                         va.z * a + vb.z * b + vc.z * c);
        ContactGeo<Dual> g;
        if (j < GEO_POSE_SEEDS) {
            g = contact_geometry<Dual>(s1, s2, q1, x1, q2, x2, ct, fd_eps, detach_b2 != 0);
        } else {
            auto shp = [](const SdfShape& s, int seed) {
                SdfShapeT<Dual> r;
                r.kind = s.kind; r.grid = s.grid; r.res = s.res; r.e0 = s.e0; r.e1 = s.e1;
                r.a = Dual(s.a, seed == 0); r.b = Dual(s.b, seed == 1); r.c = Dual(s.c, seed == 2);
                r.scale = Dual(s.scale, seed == 3);
                return r;
            };
            const SdfShapeT<Dual> d1 = shp(s1, j - 14), d2 = shp(s2, j - 18);
            const V3<Dual> ctd = v3<Dual>(Dual(ct.x, j == 22), Dual(ct.y, j == 23), Dual(ct.z, j == 24));
            g = contact_geometry<Dual>(d1, d2, q1, x1, q2, x2, ctd, fd_eps, detach_b2 != 0);
        }
        const double* gg = ggeo + 10 * oo;
        part[item] = gg[0] * g.n.x.d + gg[1] * g.n.y.d + gg[2] * g.n.z.d + gg[3] * g.p1.x.d + gg[4] * g.p1.y.d +
                     gg[5] * g.p1.z.d + gg[6] * g.p2.x.d + gg[7] * g.p2.y.d + gg[8] * g.p2.z.d + gg[9] * g.pen.d;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nb * 7; t += blockDim.x) {
        const int body = t / 7, comp = t % 7;
        double acc = 0.0;
        for (int k = 0; k < nc; ++k) {
            const size_t oo = (size_t)w * maxc + k;
            const int i1 = cbody[2 * oo], i2 = cbody[2 * oo + 1];
            if (body == i1) acc += part[k * nseeds + comp];
            if (body == i2) acc += part[k * nseeds + 7 + comp];
        }
        gp[((size_t)w * nb + body) * 7 + comp] = acc;
    }
    if (!gshape) return;
    for (int t = threadIdx.x; t < nb * 4; t += blockDim.x) {
        const int body = t / 4, comp = t % 4;
        double acc = 0.0;
        for (int k = 0; k < nc; ++k) {
            const size_t oo = (size_t)w * maxc + k;
            const int i1 = cbody[2 * oo], i2 = cbody[2 * oo + 1];
            if (body == i1) acc += part[k * nseeds + 14 + comp];
            if (body == i2) acc += part[k * nseeds + 18 + comp];
        }
        gshape[((size_t)w * nb + body) * 4 + comp] = acc;
    }
    for (int t = threadIdx.x; t < maxc * 3; t += blockDim.x) {
        const int k = t / 3, comp = t % 3;
        gctri[(size_t)w * maxc * 3 + t] = k < nc ? part[k * nseeds + 22 + comp] : 0.0;
    }
}

}  // namespace dsdf

using namespace dsdf;

extern "C" {

int dsdf_contact_geometry_backward(const dsdf_body_geom* geom, const double* p, const double* shape, int W, int nb,
                                   double fd_eps, int detach_b2, int maxc, const int32_t* count, const int32_t* cbody,
                                   const int32_t* cface, const double* cabc, const double* ggeo, double* gp,
                                   const int32_t* wmap, double* gshape, double* gctri, void* stream) {
    if (W <= 0 || nb <= 0 || maxc <= 0 || ((gshape == nullptr) != (gctri == nullptr))) return -1;
    const size_t smem = (size_t)maxc * (gshape ? GEO_ALL_SEEDS : GEO_POSE_SEEDS) * sizeof(double);
    static size_t granted = 0;
    if (smem > 48 * 1024) {
        if (smem > 227 * 1024) return -2;
        cudaError_t e = ensure_smem(contact_geometry_bwd_kernel, smem, &granted);
        if (e != cudaSuccess) return (int)e;
    }
    contact_geometry_bwd_kernel<<<W, 128, smem, (cudaStream_t)stream>>>(reinterpret_cast<const BodyGeom*>(geom), p, shape, nb,
                                                                    fd_eps, detach_b2, maxc, count, cbody, cface, cabc,
                                                                    ggeo, gp, wmap, gshape, gctri);
    return (int)cudaGetLastError();
}

}  // extern "C"
