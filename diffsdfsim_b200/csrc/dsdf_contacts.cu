// SDF collision query for all worlds: broad phase -> cube overlap -> centroid candidate pass ->
// Frank-Wolfe refinement -> contact construction -> normal-cluster / convex-hull filter -> compaction.
//
// Replaces (paths relative to the reference):
//   World.find_contacts + py3ode broad phase   lcp_physics/physics/world.py:396-399 (AABB of the rotated cube, pairs i<j)
//   FWContactHandler.__call__/_search_contacts  sdf_physics/physics3d/contacts.py:221-272
//   _overlap                                    contacts.py:27-36
//   _frank_wolfe                                contacts.py:39-94
//   _compute_contacts                           contacts.py:161-214
//   _filter_contacts (scipy Qhull on the host)  contacts.py:97-158
// Kernels: contacts_kernel (one CTA per world, everything fused: cell-culled vertex/face scans with warp-ballot
// compaction into shared memory, FW with the reference's pair-global early exit, contact geometry, filter) and
// contact_geometry_bwd_kernel (forward-mode duals w.r.t. the two poses).
#define DSDF_OUTLINE_MATH
#include "dsdf_contact_geo.cuh"
#include "dsdf_steploop.cuh"

namespace dsdf {

// Optional per-phase cycle counters (build with -DDSDF_PHASE_PROFILE; read back with dsdf_contacts_phase_cycles).
enum { PH_OVERLAP = 0, PH_GATHER, PH_SORT_INIT, PH_FW, PH_PUSH_COMPACT, PH_GEOMETRY, PH_FILTER, PH_APPEND, PH_FW_ITERS, PH_CAND,
       PH_PREFILTER, PH_F_CLUSTER, PH_F_STATS, PH_F_AKL, PH_F_SORT, PH_F_CHAIN, PH_COUNT };
#ifdef DSDF_PHASE_PROFILE
__device__ unsigned long long g_phase[PH_COUNT];
__device__ __noinline__ void ph_mark(int k) {          // k < 0: (re)start the clock
    __shared__ long long t0;
    __syncthreads();
    if (threadIdx.x == 0) {
        const long long t = clock64();
        if (k >= 0) atomicAdd(&g_phase[k], (unsigned long long)(t - t0));
        t0 = t;
    }
}
#define PH_MARK(k) ph_mark(k)
#define PH_ADD(k, v) do { if (threadIdx.x == 0) atomicAdd(&g_phase[k], (unsigned long long)(v)); } while (0)
#else
#define PH_MARK(k) do {} while (0)
#define PH_ADD(k, v) do {} while (0)
#endif

// ------------------------------------------------------------------------------------------ conservative spatial cull
// A face can only become a candidate, and a vertex can only witness _overlap, if its position in b2's frame lies in
// the cube |x| <= scale2 (outside it query_sdfs returns (scale, 0): contacts.py:52 then fails on |grad| > 1e-12;
// contacts.py:34 tests exactly that cube).  The cube's pre-image in b1's body frame is an oriented box; its
// axis-aligned bounds (inflated by a margin far above round-off) select the cells to visit.  Everything visited still
// goes through the exact reference arithmetic, so the result sets are unchanged -- only skipped work differs.
struct CellRange { int lo[3], hi[3]; bool empty; };

__device__ __forceinline__ CellRange cube_cells(const BodyGeom& g1, Q4<double> q1, V3<double> x1, Q4<double> q2,
                                                V3<double> x2, double scale2) {
    CellRange r;
    const double n1 = q1.w * q1.w + q1.x * q1.x + q1.y * q1.y + q1.z * q1.z;      // raw quaternion products scale by |q|^2
    const double n2 = q2.w * q2.w + q2.x * q2.x + q2.y * q2.y + q2.z * q2.z;
    const M3<double> R1 = q2mat(q1), R2 = q2mat(q2);
    // x_local = R1' ((R2 x_b2) / n2 + x2 - x1) / n1
    const V3<double> ctr = mat_applyT(R1, x2 - x1);
    double c[3] = {fdiv(ctr.x, n1), fdiv(ctr.y, n1), fdiv(ctr.z, n1)};
    double h[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            // (R1' R2)_{ik}
            const double m = R1.m[i] * R2.m[k] + R1.m[3 + i] * R2.m[3 + k] + R1.m[6 + i] * R2.m[6 + k];
            acc += fabs(m);
        }
        h[i] = acc * scale2 / (n1 * n2);
    }
    const double margin = 1e-6 * (1.0 + fabs(c[0]) + fabs(c[1]) + fabs(c[2]) + 2.0 * scale2);
    r.empty = false;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double a = (c[i] - h[i] - margin - g1.cell_lo[i]) * g1.cell_inv;
        const double b = (c[i] + h[i] + margin - g1.cell_lo[i]) * g1.cell_inv;
        if (b < 0.0 || a >= (double)g1.cell_dims[i]) r.empty = true;
        r.lo[i] = a <= 0.0 ? 0 : (a >= (double)g1.cell_dims[i] ? g1.cell_dims[i] - 1 : (int)a);
        r.hi[i] = b <= 0.0 ? 0 : (b >= (double)g1.cell_dims[i] ? g1.cell_dims[i] - 1 : (int)b);
    }
    return r;
}

// _overlap half (contacts.py:31,34): any vertex of b1 inside b2's cube.  Block-cooperative, early exit.
__device__ int any_vertex_in_cube(const BodyGeom& g1, int w, Q4<double> q1, V3<double> x1, Q4<double> q2,
                                  V3<double> x2, double s2) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const Q4<double> q2i = qinv(q2);
    if (!g1.has_cells) {
        for (int base = 0; base < g1.nverts; base += blockDim.x * 4) {
            int f = 0;
            for (int u = 0; u < 4; ++u) {
                const int v = base + u * blockDim.x + tid;
                if (v < g1.nverts) {
                    const V3<double> t = to_b2(load_vert(g1, w, v), q1, x1, q2i, x2);
                    f |= (-s2 <= t.x && t.x <= s2 && -s2 <= t.y && t.y <= s2 && -s2 <= t.z && t.z <= s2);
                }
            }
            if (__syncthreads_or(f)) return 1;
        }
        return 0;
    }
    const CellRange cr = cube_cells(g1, q1, x1, q2, x2, s2);
    if (cr.empty) return 0;
    const int nx = cr.hi[0] - cr.lo[0] + 1, ny = cr.hi[1] - cr.lo[1] + 1, nzc = cr.hi[2] - cr.lo[2] + 1;
    const int ncell = nx * ny * nzc;
    for (int base = 0; base < ncell; base += nw) {
        int f = 0;
        const int ci = base + warp;
        if (ci < ncell) {
            const int ix = cr.lo[0] + ci / (ny * nzc), iy = cr.lo[1] + (ci / nzc) % ny, iz = cr.lo[2] + ci % nzc;
            const int cell = (ix * g1.cell_dims[1] + iy) * g1.cell_dims[2] + iz;
            const int s = g1.vcell_start[cell], e = g1.vcell_start[cell + 1];
            for (int k = s + lane; k < e; k += 32) {
                const V3<double> t = to_b2(load_vert(g1, w, g1.vcell_items[k]), q1, x1, q2i, x2);
                f |= (-s2 <= t.x && t.x <= s2 && -s2 <= t.y && t.y <= s2 && -s2 <= t.z && t.z <= s2);
            }
        }
        if (__syncthreads_or(f)) return 1;
    }
    return 0;
}

// contacts.py:44-52 for one face: sdf(centroid) < max_i |centroid - v_i| + eps  and  |grad| > 1e-12
__device__ __forceinline__ bool face_is_candidate(const BodyGeom& g1, int w, int f, const SdfShape& s2, Q4<double> q1,
                                                  V3<double> x1, Q4<double> q2i, V3<double> x2, double eps) {
    const int ia = g1.faces[3 * f], ib = g1.faces[3 * f + 1], ic = g1.faces[3 * f + 2];
    const V3<double> a = to_b2(load_vert(g1, w, ia), q1, x1, q2i, x2);
    const V3<double> b = to_b2(load_vert(g1, w, ib), q1, x1, q2i, x2);
    const V3<double> c = to_b2(load_vert(g1, w, ic), q1, x1, q2i, x2);
    const V3<double> ctr = v3<double>(fdiv(a.x + b.x + c.x, 3.0), fdiv(a.y + b.y + c.y, 3.0), fdiv(a.z + b.z + c.z, 3.0));
    const SdfOut<double> o = sdf_q(s2, ctr, true);
    double rad = norm3(ctr - a);
    rad = fmax(rad, norm3(ctr - b));
    rad = fmax(rad, norm3(ctr - c));
    return (o.d < rad + eps) && (norm3(o.n) > 1e-12);
}

// ---- conservative fp32 pre-filter of the candidate test ---------------------------------------------------------
// The exact test (face_is_candidate) costs ~1000 fp64-path instructions per face and rejects most faces it sees.
// A face can only pass if sdf2(centroid) < rad_f + eps <= max_face_rad + eps, and the analytic SDFs are exact distance
// fields (1-Lipschitz), so a single-precision evaluation with a margin far above its rounding error discards the
// clearly-far faces first.  Survivors -- every true candidate among them -- still take the exact fp64 test.
struct Pre32 { float R[9], t[3]; float a, b, c, scale, thresh, margin, eps; int kind; bool on; };

__device__ __forceinline__ Pre32 make_pre32(const BodyGeom& g1, const SdfShape& s2, Q4<double> q1, V3<double> x1,
                                            Q4<double> q2, V3<double> x2, double eps) {
    Pre32 P;
    P.on = g1.max_face_rad > 0.0 && s2.kind <= DSDF_SDF_CYLINDER;    // (exact distance fields with a cheap fp32 form)
    const M3<double> R1 = q2mat(q1), R2 = q2mat(q2);
    const V3<double> t = mat_applyT(R2, x1 - x2);
    double amax = fabs(t.x) + fabs(t.y) + fabs(t.z);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k)
            P.R[3 * i + k] = (float)(R2.m[i] * R1.m[k] + R2.m[3 + i] * R1.m[3 + k] + R2.m[6 + i] * R1.m[6 + k]);   // R2' R1
    P.t[0] = (float)t.x; P.t[1] = (float)t.y; P.t[2] = (float)t.z;
    P.a = (float)s2.a; P.b = (float)s2.b; P.c = (float)s2.c; P.scale = (float)s2.scale; P.kind = s2.kind;
    // margin: fp32 rounding of coordinates up to (mesh extent + offset) plus the un-normalised quaternion slack
    const double ext = 1.0 / g1.cell_inv * (g1.cell_dims[0] + g1.cell_dims[1] + g1.cell_dims[2]);
    const double margin = 1e-4 * (1.0 + amax + ext + s2.scale);
    P.thresh = (float)(g1.max_face_rad * 1.001 + eps + margin);
    P.margin = (float)margin;
    P.eps = (float)eps;
    return P;
}
// Single-precision SDF of body 2 at the centroid (cx,cy,cz) given in body 1's frame, times scale; `sure_ok` = the point
// is clearly inside body 2's cube and clearly away from the places where the reference's direction vanishes (sphere
// centre, cylinder axis), so that "small distance" alone decides the exact candidate test.
__device__ __forceinline__ float pre32_dist(const Pre32& P, float cx, float cy, float cz, bool& sure_ok) {
    const float px = P.R[0] * cx + P.R[1] * cy + P.R[2] * cz + P.t[0];
    const float py = P.R[3] * cx + P.R[4] * cy + P.R[5] * cz + P.t[1];
    const float pz = P.R[6] * cx + P.R[7] * cy + P.R[8] * cz + P.t[2];
    const float is = 1.0f / P.scale;
    const float ux = px * is, uy = py * is, uz = pz * is;
    const float lim = P.scale - P.margin;
    sure_ok = fabsf(px) < lim && fabsf(py) < lim && fabsf(pz) < lim;
    float d;
    if (P.kind == DSDF_SDF_BOX) {
        const float qx = fabsf(ux) - 0.5f * P.a, qy = fabsf(uy) - 0.5f * P.b, qz = fabsf(uz) - 0.5f * P.c;
        const float ox = fmaxf(qx, 0.f), oy = fmaxf(qy, 0.f), oz = fmaxf(qz, 0.f);
        d = sqrtf(ox * ox + oy * oy + oz * oz) + fminf(fmaxf(qx, fmaxf(qy, qz)), 0.f);
    } else if (P.kind == DSDF_SDF_SPHERE) {
        const float r = sqrtf(ux * ux + uy * uy + uz * uz);
        d = r - P.a;
        sure_ok = sure_ok && r > 1e-3f;
    } else {                                                    // cylinder along local z
        const float rho = sqrtf(ux * ux + uy * uy);
        const float q0 = rho - P.a, q1 = fabsf(uz) - 0.5f * P.b;
        const float o0 = fmaxf(q0, 0.f), o1 = fmaxf(q1, 0.f);
        d = sqrtf(o0 * o0 + o1 * o1) + fminf(fmaxf(q0, q1), 0.f);
        sure_ok = sure_ok && rho > 1e-3f;
    }
    return d * P.scale;
}

// Centroid candidate pass of one search direction into the shared list ids[0..capK) (unsorted); returns the count
// (which may exceed capK: overflow).  s_cnt: one shared int.
__device__ int gather_candidates(const BodyGeom& g1, int w, const SdfShape& s2, Q4<double> q1, V3<double> x1,
                                 Q4<double> q2, V3<double> x2, double eps, int capK, int* ids, int* s_cnt) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const Q4<double> q2i = qinv(q2);
    if (tid == 0) *s_cnt = 0;
    __syncthreads();
    auto push = [&](bool is_cand, int f) {
        const unsigned m = __ballot_sync(DSDF_FULL, is_cand);
        if (m) {
            int base = 0;
            if (lane == 0) base = atomicAdd(s_cnt, __popc(m));
            base = __shfl_sync(DSDF_FULL, base, 0);
            if (is_cand) {
                const int slot = base + __popc(m & ((1u << lane) - 1));
                if (slot < capK) ids[slot] = f;
            }
        }
    };
    if (!g1.has_cells) {
        for (int base = 0; base < g1.nfaces; base += blockDim.x) {
            const int f = base + tid;
            push(f < g1.nfaces && face_is_candidate(g1, w, f, s2, q1, x1, q2i, x2, eps), f);
        }
    } else {
        const CellRange cr = cube_cells(g1, q1, x1, q2, x2, s2.scale);
        const Pre32 P32 = make_pre32(g1, s2, q1, x1, q2, x2, eps);
        if (!cr.empty) {
            const int nx = cr.hi[0] - cr.lo[0] + 1, ny = cr.hi[1] - cr.lo[1] + 1, nzc = cr.hi[2] - cr.lo[2] + 1;
            const int ncell = nx * ny * nzc;
            for (int ci = warp; ci < ncell; ci += nw) {
                const int ix = cr.lo[0] + ci / (ny * nzc), iy = cr.lo[1] + (ci / nzc) % ny, iz = cr.lo[2] + ci % nzc;
                const int cell = (ix * g1.cell_dims[1] + iy) * g1.cell_dims[2] + iz;
                const int s = g1.fcell_start[cell], e = g1.fcell_start[cell + 1];
                for (int k0 = s; k0 < e; k0 += 32) {
                    const int k = k0 + lane;
                    const int f = k < e ? g1.fcell_items[k] : 0;
                    bool test = k < e, sure = false;
                    if (test && P32.on) {
                        // single precision decides the CLEAR cases both ways (far: not a candidate; well inside the
                        // threshold, as every face under a resting body is: a candidate); only the band of width
                        // 2 * margin around sdf = rad + eps takes the exact fp64 test, so the result set is unchanged
                        const V3<double> a = load_vert(g1, w, g1.faces[3 * f]), b = load_vert(g1, w, g1.faces[3 * f + 1]),
                                         c = load_vert(g1, w, g1.faces[3 * f + 2]);
                        const float ax = (float)a.x, ay = (float)a.y, az = (float)a.z, bx = (float)b.x, by = (float)b.y,
                                    bz = (float)b.z, cx = (float)c.x, cy = (float)c.y, cz = (float)c.z;
                        const float mx = (float)((a.x + b.x + c.x) * (1.0 / 3.0)), my = (float)((a.y + b.y + c.y) * (1.0 / 3.0)),
                                    mz = (float)((a.z + b.z + c.z) * (1.0 / 3.0));
                        bool ok;
                        const float d = pre32_dist(P32, mx, my, mz, ok);
                        if (d > P32.thresh) test = false;
                        else {
                            const float ra = (ax - mx) * (ax - mx) + (ay - my) * (ay - my) + (az - mz) * (az - mz);
                            const float rb = (bx - mx) * (bx - mx) + (by - my) * (by - my) + (bz - mz) * (bz - mz);
                            const float rc = (cx - mx) * (cx - mx) + (cy - my) * (cy - my) + (cz - mz) * (cz - mz);
                            const float rad = sqrtf(fmaxf(ra, fmaxf(rb, rc)));
                            sure = ok && (d + 2.0f * P32.margin < rad * 0.999f + P32.eps);
                        }
                    }
                    push(sure || (test && face_is_candidate(g1, w, f, s2, q1, x1, q2i, x2, eps)), f);
                }
            }
        }
    }
    __syncthreads();
    return *s_cnt;
}

// ------------------------------------------------------------------------------------------ block helpers
// Rank sorts: every element counts how many precede it (O(n^2/threads) compares on broadcast shared loads, two
// barriers) -- far cheaper here than a bitonic network's ~45 barrier-separated passes for n <= 1024.
enum { SORT_MAX_ROUNDS = 8 };                                   // n <= SORT_MAX_ROUNDS * blockDim.x
__device__ __noinline__ void rank_sort_int(int* a, int* tmp, int n) {  // ascending; DISTINCT values; a 16-byte aligned
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int x = a[i];
        int r = 0, j = 0;
        for (; j + 4 <= n; j += 4) {                           // broadcast 128-bit shared loads
            const int4 y = *reinterpret_cast<const int4*>(a + j);
            r += (y.x < x) + (y.y < x) + (y.z < x) + (y.w < x);
        }
        for (; j < n; ++j) r += a[j] < x;
        tmp[r] = x;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) a[i] = tmp[i];
    __syncthreads();
}
// (key, key2, payload) ascending lexicographically, in place
__device__ __noinline__ void rank_sort_kv(double* key, double* key2, int* pay, int n) {
    double k1[SORT_MAX_ROUNDS], k2[SORT_MAX_ROUNDS];
    int pl[SORT_MAX_ROUNDS], rk[SORT_MAX_ROUNDS];
#pragma unroll 1
    for (int rd = 0; rd < SORT_MAX_ROUNDS; ++rd) {
        const int i = rd * blockDim.x + threadIdx.x;
        rk[rd] = -1;
        if (i < n) {
            const double x = key[i], x2 = key2[i];
            const int px = pay[i];
            int r = 0;
            for (int j = 0; j < n; ++j) {
                const double y = key[j], y2 = key2[j];
                r += (y < x) || (y == x && (y2 < x2 || (y2 == x2 && (pay[j] < px || (pay[j] == px && j < i)))));
            }
            k1[rd] = x; k2[rd] = x2; pl[rd] = px; rk[rd] = r;
        }
    }
    __syncthreads();
#pragma unroll 1
    for (int rd = 0; rd < SORT_MAX_ROUNDS; ++rd)
        if (rk[rd] >= 0) { key[rk[rd]] = k1[rd]; key2[rk[rd]] = k2[rd]; pay[rk[rd]] = pl[rd]; }
    __syncthreads();
}
// order-preserving compaction offsets: returns exclusive prefix of flag over index order 0..n-1; *total = sum.
// idx loop layout: element e handled by thread e % nt in round e / nt.  scan buffer: n ints.
__device__ __noinline__ void block_exclusive_scan(int* buf, int n, int* total) {
    // simple Hillis-Steele over shared memory (n <= 1024), in place, exclusive
    __syncthreads();
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        int v = i < n ? buf[i] : 0;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(DSDF_FULL, incl, o); if (lane >= o) incl += t; }
        __shared__ int wsum[32];
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int s = lane < (int)(blockDim.x >> 5) ? wsum[lane] : 0;
            int si = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(DSDF_FULL, si, o); if (lane >= o) si += t; }
            wsum[lane] = si - s;
        }
        __syncthreads();
        const int excl = carry + wsum[warp] + incl - v;
        if (i < n) buf[i] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = excl + v;
        __syncthreads();
    }
    *total = carry;
    __syncthreads();
}

// out-of-line block reductions (the template in dsdf_dense.cuh is inlined at every call site)
__device__ __noinline__ double bred_sum(double v, double* red) { return block_reduce<RED_SUM>(v, red); }
__device__ __noinline__ double bred_min(double v, double* red) { return block_reduce<RED_MIN>(v, red); }
__device__ __noinline__ double bred_max(double v, double* red) { return block_reduce<RED_MAX>(v, red); }

// Up to 8 reductions behind ONE pair of barriers (same shuffle trees as block_reduce, so every result keeps its bits):
// the hull filter is a chain of tiny block-wide reductions over a few hundred points, dominated by barrier latency.
// ops[i] in {RED_SUM, RED_MIN, RED_MAX}; red: >= 40 doubles; blockDim.x <= 128 (4 warps x 8 values + 8 results).
__device__ __noinline__ void bred_multi(double* v, const int* ops, int n, double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    for (int i = 0; i < n; ++i) {
        double x = v[i];
        x = ops[i] == RED_SUM ? warp_sum(x) : (ops[i] == RED_MIN ? warp_min(x) : warp_max(x));
        v[i] = x;
    }
    __syncthreads();
    if (lane == 0) for (int i = 0; i < n; ++i) red[warp * 8 + i] = v[i];
    __syncthreads();
    if (warp == 0) {
        for (int i = 0; i < n; ++i) {
            const double id = ops[i] == RED_SUM ? 0.0 : (ops[i] == RED_MIN ? INFINITY : -INFINITY);
            double t = lane < nw ? red[lane * 8 + i] : id;
            t = ops[i] == RED_SUM ? warp_sum(t) : (ops[i] == RED_MIN ? warp_min(t) : warp_max(t));
            if (lane == 0) v[i] = t;
        }
    }
    __syncthreads();
    if (warp == 0 && lane == 0) for (int i = 0; i < n; ++i) red[32 + i] = v[i];
    __syncthreads();
    for (int i = 0; i < n; ++i) v[i] = red[32 + i];
}

// ------------------------------------------------------------------------------------------ 3-D convex hull
// Vertices of the convex hull of a genuinely three-dimensional cluster of contact points (contacts.py:126-133: scipy's
// Qhull on the host in the reference): gift wrapping with all threads of the CTA scanning the points of every wrap step.
// Around a directed hull edge s -> t whose known face has outward normal n0 and in-plane direction m0 (from the edge
// towards that face), the neighbouring face is spanned by the point with the smallest rotation angle phi from the
// continuation of the known plane; among points on that same plane (planar facets with more than three vertices) the next
// boundary vertex of the facet polygon wins (most clockwise about t, farthest on ties), so points inside a facet or inside
// an edge are never selected -- Qhull's merged-facet vertex set.  Faces are triangles (t, s, c); a hash set (open
// addressing, filled by thread 0) remembers which directed edges already belong to a face.
struct HullPick { int idx; double x, y, al, rho; };

// primary order: smaller rotation angle phi in [0, pi] (y is clamped at 0, so the 2x2 determinant orders the angles; phi = 0
// against phi = pi has det == 0 and is decided by x).  Strict -- a total order, exact ties by index.
__device__ __forceinline__ bool hull_phi_less(const HullPick& p, const HullPick& q) {
    if (q.idx < 0) return p.idx >= 0;
    if (p.idx < 0) return false;
    const double det = p.x * q.y - q.x * p.y;                          // > 0: phi_p < phi_q
    if (det != 0.0) return det > 0.0;
    if (p.x * q.x + p.y * q.y < 0.0) return p.x > 0.0;
    return p.idx < q.idx;
}
// secondary order among the points on the winning plane: the facet lies in the wedge at t between the direction towards s
// (angle pi) and its other neighbour of t, so the candidate with the SMALLEST angle about t is that neighbour -- a vertex
// of the facet, never an interior point; collinear with t: the farthest; exact duplicates: the lowest index.
// tol = coordinate round-off bound (Qhull's distance tolerance scale) -- both points may be off by it.
__device__ __forceinline__ bool hull_turn_less(const HullPick& p, const HullPick& q, double L, double tol) {
    if (q.idx < 0) return p.idx >= 0;
    if (p.idx < 0) return false;
    const double cr = (q.al - L) * p.rho - q.rho * (p.al - L);        // cross(q - t, p - t) > 0: angle_p > angle_q
    const double dp2 = (p.al - L) * (p.al - L) + p.rho * p.rho, dq2 = (q.al - L) * (q.al - L) + q.rho * q.rho;
    const double tol2 = tol * (sqrt(dp2) + sqrt(dq2));
    if (cr < -tol2) return true;
    if (cr > tol2) return false;
    if (dp2 != dq2) return dp2 > dq2;
    return p.idx < q.idx;
}

template <bool SECOND>
__device__ HullPick hull_reduce(HullPick best, double L, double tol, double* red) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) {
        HullPick q;
        q.idx = __shfl_xor_sync(DSDF_FULL, best.idx, o);
        q.x = __shfl_xor_sync(DSDF_FULL, best.x, o); q.y = __shfl_xor_sync(DSDF_FULL, best.y, o);
        q.al = __shfl_xor_sync(DSDF_FULL, best.al, o); q.rho = __shfl_xor_sync(DSDF_FULL, best.rho, o);
        if (SECOND ? hull_turn_less(q, best, L, tol) : hull_phi_less(q, best)) best = q;
    }
    __syncthreads();
    if (lane == 0) {
        red[warp * 5] = (double)best.idx; red[warp * 5 + 1] = best.x; red[warp * 5 + 2] = best.y;
        red[warp * 5 + 3] = best.al; red[warp * 5 + 4] = best.rho;
    }
    __syncthreads();
    HullPick b; b.idx = -1; b.x = b.y = b.al = b.rho = 0.0;
    for (int ww = 0; ww < nw; ++ww) {                                   // every thread: same order, same result
        HullPick q;
        q.idx = (int)red[ww * 5]; q.x = red[ww * 5 + 1]; q.y = red[ww * 5 + 2]; q.al = red[ww * 5 + 3]; q.rho = red[ww * 5 + 4];
        if (SECOND ? hull_turn_less(q, b, L, tol) : hull_phi_less(q, b)) b = q;
    }
    __syncthreads();
    return b;
}

// one wrap step; all threads call it; returns the chosen point (index into the cluster's member list) or -1.
// Pass 1: the point of smallest rotation angle.  Pass 2: among the points on that plane (within the round-off bound of
// the angle comparison, Qhull's coplanarity notion) the facet vertex next to t.  Defining the tie set against the single
// best point keeps the choice well defined (a pairwise tolerant comparison is not transitive).
__device__ int hull_wrap(const double* PX, const double* PY, const double* PZ, const int* HI, int m, V3<double> S,
                         V3<double> T, V3<double> n0, V3<double> m0, int skip_s, int skip_t, double tol, double* red) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const V3<double> E = T - S;
    const double L = norm3(E);
    const V3<double> e = v3<double>(E.x / L, E.y / L, E.z / L);
    auto pick = [&](int i) {
        HullPick c; c.idx = -1; c.x = c.y = c.al = c.rho = 0.0;
        if (i == skip_s || i == skip_t) return c;
        const int k = HI[i];
        const V3<double> d = v3<double>(PX[k], PY[k], PZ[k]) - S;
        c.al = dot(d, e);
        const V3<double> r = d - e * c.al;
        c.rho = norm3(r);
        if (!(c.rho > 1e-14 * (L + fabs(c.al)))) return c;              // on the edge's line: not a candidate
        c.x = -dot(r, m0);
        c.y = fmax(-dot(r, n0), 0.0);
        c.idx = i;
        return c;
    };
    HullPick best; best.idx = -1; best.x = best.y = best.al = best.rho = 0.0;
    for (int i = tid; i < m; i += nt) {
        const HullPick c = pick(i);
        if (hull_phi_less(c, best)) best = c;
    }
    HullPick star = hull_reduce<false>(best, L, tol, red);
    if (star.idx < 0) return -1;
    // the tie set is re-centred on the chosen point until it stops moving: a run of collinear / coplanar points that
    // leaves the tolerance band of the first winner is still walked to its end (its extreme point is the vertex)
#pragma unroll 1
    for (int it = 0; it < 8; ++it) {
        best.idx = -1;
        for (int i = tid; i < m; i += nt) {
            const HullPick c = pick(i);
            if (c.idx < 0) continue;
            const double det = star.x * c.y - c.x * star.y;
            if (fabs(det) > tol * (star.rho + c.rho)) continue;            // not on the winning plane
            if (star.x * c.x + star.y * c.y < 0.0) continue;                // (opposite half-plane: angle pi apart)
            if (hull_turn_less(c, best, L, tol)) best = c;
        }
        const HullPick nxt = hull_reduce<true>(best, L, tol, red);
        if (nxt.idx == star.idx) break;
        star = nxt;
    }
    return star.idx;
}

// marks KEEP[HI[i]] = 1 for the hull vertices of the cluster's m points; returns false when the work buffers are too
// small for m (the caller keeps the whole cluster and flags it).  tab: hash table of ntab ints (<= 6 m directed edges);
// stk0 / stk1: cap ints each.
__device__ bool hull3d_vertices(const double* PX, const double* PY, const double* PZ, const int* HI, int m, int* KEEP,
                                unsigned* tab, size_t ntab, int* stk0, int* stk1, int cap, double* red,
                                double maxabs) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const double tol = 2e-15 * maxabs;                                  // round-off bound of the coordinates (tuned on Qhull)
    if ((size_t)8 * m > ntab || 3 * m > 2 * cap || m > 1023) return false;          // load factor <= 0.75
    for (size_t i = tid; i < ntab; i += nt) tab[i] = 0u;
    __shared__ int s_top, s_a;
    // lexicographically smallest point (x, then y, the coordinate ties up to round-off, then z): a hull vertex -- with
    // exact ties only, round-off would pick an interior point of a hull edge parallel to the z (or y) axis
    if (tid == 0) {
        double lo = PX[HI[0]];
        for (int i = 1; i < m; ++i) lo = fmin(lo, PX[HI[i]]);
        const double xcut = lo + tol;
        lo = 1e300;
        for (int i = 0; i < m; ++i) if (PX[HI[i]] <= xcut) lo = fmin(lo, PY[HI[i]]);
        const double ycut = lo + tol;
        int a = -1;
        for (int i = 0; i < m; ++i) {
            const int k = HI[i];
            if (PX[k] <= xcut && PY[k] <= ycut && (a < 0 || PZ[k] < PZ[HI[a]])) a = i;
        }
        s_a = a; s_top = 0;
    }
    __syncthreads();
    const int a = s_a;
    auto P = [&](int i) { const int k = HI[i]; return v3<double>(PX[k], PY[k], PZ[k]); };
    auto unit = [](V3<double> v) { const double n = norm3(v); return v3<double>(v.x / n, v.y / n, v.z / n); };
    auto edge_done = [&](int u, int v) {
        const unsigned key = ((unsigned)u << 10 | (unsigned)v) + 1u;
        for (size_t h = (key * 2654435761u) % ntab;; h = h + 1 == ntab ? 0 : h + 1) {
            if (tab[h] == key) return true;
            if (tab[h] == 0u) return false;
        }
    };
    auto mark_edge = [&](int u, int v) {                               // thread 0 only
        const unsigned key = ((unsigned)u << 10 | (unsigned)v) + 1u;
        size_t h = (key * 2654435761u) % ntab;
        while (tab[h] != 0u && tab[h] != key) h = h + 1 == ntab ? 0 : h + 1;
        tab[h] = key;
    };
    auto push = [&](int s_, int t_, int w_) {
        const int top = s_top++;
        (top < cap ? stk0[top] : stk1[top - cap]) = s_ | (t_ << 10) | (w_ << 20);
    };
    // first edge: wrap around the vertical line through a (virtual end point far above every point), starting from the
    // supporting plane x = a.x: "known face" (a, virtual, a + e_y), outward normal -e_x = e_z x e_y
    const V3<double> A = P(a);
    const V3<double> Vt = A + v3<double>(0.0, 0.0, 8.0 * maxabs + 1.0);
    const int b = hull_wrap(PX, PY, PZ, HI, m, A, Vt, v3<double>(-1.0, 0.0, 0.0), v3<double>(0.0, 1.0, 0.0), a, -1, tol, red);
    if (b < 0) return true;                                             // (cannot happen for a non-degenerate cluster)
    // first face: wrap around a -> b; the known face is the vertical supporting plane (a, b, virtual) just found
    const V3<double> Bp = P(b);
    {
        const V3<double> eab = unit(Bp - A);
        V3<double> rw = (Vt - A) - eab * dot(Vt - A, eab);
        const int c = hull_wrap(PX, PY, PZ, HI, m, A, Bp, unit(cross(Bp - A, Vt - A)), unit(rw), a, b, tol, red);
        if (c < 0) return true;
        if (tid == 0) {
            KEEP[HI[a]] = 1; KEEP[HI[b]] = 1; KEEP[HI[c]] = 1;
            // face (b, a, c): counter-clockwise seen from outside
            mark_edge(b, a); mark_edge(a, c); mark_edge(c, b);
            push(b, a, c); push(a, c, b); push(c, b, a);
        }
    }
    __syncthreads();
    for (int guard = 0; guard < 8 * m + 64; ++guard) {
        __syncthreads();
        if (s_top == 0) break;
        const int top = s_top - 1;
        const int ent = top < cap ? stk0[top] : stk1[top - cap];
        const int s_ = ent & 1023, t_ = (ent >> 10) & 1023, w_ = ent >> 20;
        const bool need = !edge_done(t_, s_);                            // the face across s -> t (it contains t -> s)
        __syncthreads();
        if (tid == 0) s_top = top;
        if (!need) continue;
        const V3<double> Sp = P(s_), Tp = P(t_), Wp = P(w_);
        const V3<double> e = unit(Tp - Sp);
        const V3<double> rw = (Wp - Sp) - e * dot(Wp - Sp, e);
        const int c = hull_wrap(PX, PY, PZ, HI, m, Sp, Tp, unit(cross(Tp - Sp, Wp - Sp)), unit(rw), s_, t_, tol, red);
        if (c < 0) continue;
        if (tid == 0) {
            KEEP[HI[c]] = 1;
            // new face (t, s, c)
            mark_edge(t_, s_); mark_edge(s_, c); mark_edge(c, t_);
            if (s_top + 2 <= 2 * cap) { push(s_, c, t_); push(c, t_, s_); }
        }
    }
    __syncthreads();
    return true;
}

// ------------------------------------------------------------------------------------------ refine kernel
struct RefineSmem {
    double* P;      // [9][capK] candidate triangle in b2 frame, later GEO rows 0..8
    double* X;      // [3][capK] FW iterate, later GEO row 9 (pen) + scratch
    double* ABC;    // [3][capK]
    double* HK;     // [2][capK] hull sort keys -- aliases X rows 1,2 (free once the contact geometry is computed)
    int* ID;        // [capK] face ids
    int* SC;        // [capK] scan / flags
    int* CL;        // [capK] cluster id
    int* HI;        // [capK] hull payload
    int* KEEP;      // [capK]
    int* TMP;       // [capK] scratch flags
    double* red;    // [40]
};

__host__ __device__ inline size_t refine_smem_bytes(int capK) {
    return (size_t)capK * (15 * sizeof(double) + 6 * sizeof(int)) + 40 * sizeof(double) + 64;
}

struct DirResult { int count; int valid; };

// One search direction (mesh body i1 -> SDF body i2) for world w.  On return the first `count` slots of
// GEO (=P rows 0..8 + X row 0), ABC and ID hold the pre-filter contacts in ascending face order.
// ids: the candidate list already sitting (unsorted) in sm.ID[0..min(ncand,capK)).
__device__ DirResult search_direction(const RefineSmem& sm, int capK, const BodyGeom& g1, const SdfShape& s1,
                                      const SdfShape& s2, Q4<double> q1, V3<double> x1, Q4<double> q2, V3<double> x2,
                                      int w, int ncand, double eps, double tol, double fd_eps, bool detach_b2) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int K = min(ncand, capK);
    DirResult r; r.count = 0; r.valid = 1;
    if (K == 0) return r;
    PH_MARK(-1);
    PH_ADD(PH_CAND, K);
    rank_sort_int(sm.ID, sm.SC, K);
    const Q4<double> q2i = qinv(q2);
    // init: vertices in b2 frame, start at the vertex with the smallest SDF (contacts.py:57-61)
    for (int k = tid; k < K; k += nt) {
        const int f = sm.ID[k];
        double best = 0.0; int bi = 0;
#pragma unroll
        for (int v = 0; v < 3; ++v) {
            const V3<double> t = to_b2(load_vert(g1, w, g1.faces[3 * f + v]), q1, x1, q2i, x2);
            sm.P[(3 * v + 0) * capK + k] = t.x; sm.P[(3 * v + 1) * capK + k] = t.y; sm.P[(3 * v + 2) * capK + k] = t.z;
            const double d = sdf_q(s2, t, false).d;
            if (v == 0 || d < best) { best = d; bi = v; }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            sm.X[c * capK + k] = sm.P[(3 * bi + c) * capK + k];
            sm.ABC[c * capK + k] = c == bi ? 1.0 : 0.0;
        }
    }
    __syncthreads();
    // Frank-Wolfe, <= 32 iterations, PAIR-GLOBAL exit (contacts.py:63-82).  A candidate whose step is zero
    // (|gain| <= tol) keeps its x, so re-evaluating it would reproduce the same decision: it is skipped from then on
    // (TMP[k] = 1) -- the reference recomputes it every iteration with identical results.
    // The still-moving candidates are kept as a compact list (two ping-pong buffers in HI / CL, free until the filter),
    // so that from the second iteration on every thread evaluates at most one of the few dozen survivors instead of
    // walking all K slots: the iteration latency is one SDF evaluation, not ceil(K / threads) of them.
    __shared__ int s_nact[2];
    int* lists[2] = {sm.HI, sm.CL};
    for (int k = tid; k < K; k += nt) lists[0][k] = k;
    if (tid == 0) { s_nact[0] = K; s_nact[1] = 0; }
    __syncthreads();
    PH_MARK(PH_SORT_INIT);
    for (int it = 0; it < 32; ++it) {
        const int cur = it & 1, nxt = cur ^ 1;
        const int nact = s_nact[cur];
        const int* act_list = lists[cur];
        int any_pen = 0;
        // phase 1: evaluate (no state change until the exit test is known)
        for (int a = tid; a < nact; a += nt) {
            const int k = act_list[a];
            const V3<double> x = v3<double>(sm.X[k], sm.X[capK + k], sm.X[2 * capK + k]);
            const SdfOut<double> o = sdf_q(s2, x, true);
            double dmin = 0.0; int pick = 0;
#pragma unroll
            for (int v = 0; v < 3; ++v) {
                const double dp = sm.P[(3 * v) * capK + k] * o.n.x + sm.P[(3 * v + 1) * capK + k] * o.n.y +
                                  sm.P[(3 * v + 2) * capK + k] * o.n.z;
                if (v == 0 || dp < dmin) { dmin = dp; pick = v; }
            }
            const V3<double> s = v3<double>(sm.P[(3 * pick) * capK + k], sm.P[(3 * pick + 1) * capK + k],
                                            sm.P[(3 * pick + 2) * capK + k]);
            const double gain = (x.x - s.x) * o.n.x + (x.y - s.y) * o.n.y + (x.z - s.z) * o.n.z;
            const int act = fabs(gain) > tol;
            any_pen |= (o.d < -tol);
            sm.SC[k] = act ? pick : -1;
            // a candidate whose step is zero keeps its x, so re-evaluating it would reproduce the same decision: it leaves
            // the list for good (the reference recomputes it every iteration with identical results)
            if (act) lists[nxt][atomicAdd(&s_nact[nxt], 1)] = k;
        }
        // one barrier: the penetration flag through the barrier's predicate, "anything still moving" from the length of
        // the next list (every active candidate was appended to it before the barrier)
        const int blk_pen = __syncthreads_or(any_pen);
        const int blk_active = s_nact[nxt] > 0;
        PH_ADD(PH_FW_ITERS, 1);
        if (!blk_active || blk_pen) break;
        const double gamma = 2.0 / (it + 2.0);
        for (int a = tid; a < nact; a += nt) {
            const int k = act_list[a];
            const int pick = sm.SC[k];
            if (pick >= 0) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    sm.X[c * capK + k] = (1.0 - gamma) * sm.X[c * capK + k] + gamma * sm.P[(3 * pick + c) * capK + k];
                    sm.ABC[c * capK + k] *= (1.0 - gamma);
                }
                sm.ABC[pick * capK + k] += gamma;
            }
            // dropped candidates: gamma = 0 -> x, abc unchanged (x = 1*x + 0*s, abc *= 1, += 0)
        }
        if (tid == 0) s_nact[cur] = 0;                 // becomes the "next" counter of the following iteration
        __syncthreads();
    }
    __syncthreads();
    PH_MARK(PH_FW);
    // push onto b1's surface and final threshold (contacts.py:84-91)
    const Q4<double> rel = qmul(q2i, q1);
    for (int k = tid; k < K; k += nt) {
        const int f = sm.ID[k];
        const V3<double> va = load_vert(g1, w, g1.faces[3 * f]), vb = load_vert(g1, w, g1.faces[3 * f + 1]),
                         vc = load_vert(g1, w, g1.faces[3 * f + 2]);
        const double a = sm.ABC[k], b = sm.ABC[capK + k], c = sm.ABC[2 * capK + k];
        const V3<double> xb1 = v3<double>(va.x * a + vb.x * b + vc.x * c, va.y * a + vb.y * b + vc.y * c,
                                          va.z * a + vb.z * b + vc.z * c);
        const SdfOut<double> o1 = sdf_q(s1, xb1, true);
        const V3<double> dir = qapply(rel, o1.n);
        const V3<double> x = v3<double>(sm.X[k] - o1.d * dir.x, sm.X[capK + k] - o1.d * dir.y,
                                        sm.X[2 * capK + k] - o1.d * dir.z);
        const double d = sdf_q(s2, x, false).d;
        sm.SC[k] = d <= eps ? 1 : 0;
        // stash the body-frame triangle point for the geometry pass
        sm.X[k] = xb1.x; sm.X[capK + k] = xb1.y; sm.X[2 * capK + k] = xb1.z;
    }
    int total = 0;
    for (int k = tid; k < K; k += nt) sm.KEEP[k] = sm.SC[k];
    __syncthreads();
    block_exclusive_scan(sm.SC, K, &total);
    // order-preserving compaction into the front (read everything first, then write)
    {
        const int rounds = (K + nt - 1) / nt;
        for (int rd = 0; rd < rounds; ++rd) {
            const int k = rd * nt + tid;
            double t0 = 0, t1 = 0, t2 = 0, a0 = 0, a1 = 0, a2 = 0; int id = 0, dst = -1;
            if (k < K && sm.KEEP[k]) {
                dst = sm.SC[k];
                t0 = sm.X[k]; t1 = sm.X[capK + k]; t2 = sm.X[2 * capK + k];
                a0 = sm.ABC[k]; a1 = sm.ABC[capK + k]; a2 = sm.ABC[2 * capK + k];
                id = sm.ID[k];
            }
            __syncthreads();
            if (dst >= 0) {      // dst <= k and all smaller k already moved in earlier rounds / this round's reads done
                sm.X[dst] = t0; sm.X[capK + dst] = t1; sm.X[2 * capK + dst] = t2;
                sm.ABC[dst] = a0; sm.ABC[capK + dst] = a1; sm.ABC[2 * capK + dst] = a2;
                sm.ID[dst] = id;
            }
            __syncthreads();
        }
    }
    PH_MARK(PH_PUSH_COMPACT);
    // contact geometry for every pre-filter contact (the reference's no_grad _compute_contacts).  Faces that share a
    // vertex often end at the very same body-frame point (bit-identical coordinates: the barycentrics are a unit
    // vector); the geometry is a pure function of that point, so it is evaluated once per DISTINCT point and copied.
    int* REP = sm.TMP;                 // representative (smallest index with identical coordinates)
    int* UL = sm.HI;                   // compact list of representatives
    {
        // open-addressing hash set over the coordinates (capK slots in CL, free until the filter): a slot holds the smallest
        // index seen so far of its key.  Replaces an O(total^2) scan (9 % of the kernel's instructions, ncu round 2).
        int* TAB = sm.CL;
        for (int k = tid; k < capK; k += nt) TAB[k] = 0x7fffffff;
        __syncthreads();
        auto slot0 = [&](double a0, double a1, double a2) {
            const unsigned long long u0 = __double_as_longlong(a0 + 0.0), u1 = __double_as_longlong(a1 + 0.0),
                                     u2 = __double_as_longlong(a2 + 0.0);               // (+ 0.0: -0 and +0 compare equal)
            unsigned long long h = u0 * 0x9E3779B97F4A7C15ull;
            h = (h ^ (h >> 29)) + u1 * 0xBF58476D1CE4E5B9ull;
            h = (h ^ (h >> 31)) + u2 * 0x94D049BB133111EBull;
            h ^= h >> 32;
            return (int)((unsigned)h % (unsigned)capK);
        };
        for (int k = tid; k < total; k += nt) {
            const double a0 = sm.X[k], a1 = sm.X[capK + k], a2 = sm.X[2 * capK + k];
            int s_ = slot0(a0, a1, a2);
            for (int probes = 0; probes < capK; ++probes, s_ = s_ + 1 == capK ? 0 : s_ + 1) {
                int j = TAB[s_];
                if (j == 0x7fffffff) {
                    j = atomicCAS(&TAB[s_], 0x7fffffff, k);
                    if (j == 0x7fffffff) break;                                        // new key
                }
                // j indexes a contact with this slot's key (atomicMin only ever swaps in an equal-key index)
                if (sm.X[j] == a0 && sm.X[capK + j] == a1 && sm.X[2 * capK + j] == a2) { atomicMin(&TAB[s_], k); break; }
            }
        }
        __syncthreads();
        for (int k = tid; k < total; k += nt) {
            const double a0 = sm.X[k], a1 = sm.X[capK + k], a2 = sm.X[2 * capK + k];
            int rep = k;
            int s_ = slot0(a0, a1, a2);
            for (int probes = 0; probes < capK; ++probes, s_ = s_ + 1 == capK ? 0 : s_ + 1) {
                const int j = TAB[s_];
                if (j == 0x7fffffff) break;                                            // (NaN coordinates: own representative)
                if (sm.X[j] == a0 && sm.X[capK + j] == a1 && sm.X[2 * capK + j] == a2) { rep = j; break; }
            }
            REP[k] = rep;
            sm.SC[k] = rep == k;
        }
    }
    int nuniq = 0;
    block_exclusive_scan(sm.SC, total, &nuniq);
    for (int k = tid; k < total; k += nt) if (REP[k] == k) UL[sm.SC[k]] = k;
    __syncthreads();
    int bad = 0;
    for (int u = tid; u < nuniq; u += nt) {
        const int k = UL[u];
        const V3<double> ct = v3<double>(sm.X[k], sm.X[capK + k], sm.X[2 * capK + k]);
        const ContactGeo<double> g = contact_geometry<double>(s1, s2, q1, x1, q2, x2, ct, fd_eps, detach_b2);
        sm.P[0 * capK + k] = g.n.x; sm.P[1 * capK + k] = g.n.y; sm.P[2 * capK + k] = g.n.z;
        sm.P[3 * capK + k] = g.p1.x; sm.P[4 * capK + k] = g.p1.y; sm.P[5 * capK + k] = g.p1.z;
        sm.P[6 * capK + k] = g.p2.x; sm.P[7 * capK + k] = g.p2.y; sm.P[8 * capK + k] = g.p2.z;
        sm.X[capK + k] = g.pen;                            // park pen in X row 1 until every duplicate has read row 0
        bad |= !(g.pen <= tol);
    }
    __syncthreads();
    for (int k = tid; k < total; k += nt) {
        const int rp = REP[k];
        if (rp != k) {
#pragma unroll
            for (int c = 0; c < 9; ++c) sm.P[(size_t)c * capK + k] = sm.P[(size_t)c * capK + rp];
        }
    }
    __syncthreads();
    for (int k = tid; k < total; k += nt) sm.X[k] = sm.X[capK + REP[k]];      // X row 0 <- pen
    __syncthreads();
    r.valid = !__syncthreads_or(bad);
    r.count = total;
    PH_ADD(PH_PREFILTER, total);
    PH_MARK(PH_GEOMETRY);
    return r;
}

// Qhull-like round-off bound for coordinates of magnitude maxabs in `dim` dimensions (qh_distround)
__device__ __forceinline__ double distround(int dim, double maxabs) {
    return 2.220446049250313e-16 * (dim * sqrt((double)dim) * maxabs * 1.01 + maxabs);
}

// _filter_contacts (contacts.py:97-158): on entry n contacts in GEO (P rows) ; on exit KEEP[k] in {0,1}.
// Returns status bits (4 = 3-D hull of >4 points needed: kept all of that cluster).
__device__ int filter_contacts(const RefineSmem& sm, int capK, int n, double eps) {
    const int tid = threadIdx.x, nt = blockDim.x;
    int status = 0;
    for (int k = tid; k < n; k += nt) sm.KEEP[k] = 1;
    __syncthreads();
    if (n <= 1) return 0;
    const double* NX = sm.P; const double* NY = sm.P + capK; const double* NZ = sm.P + 2 * capK;
    const double* PX = sm.P + 3 * capK; const double* PY = sm.P + 4 * capK; const double* PZ = sm.P + 5 * capK;
    // zero normals are dropped; CL = -1 unassigned, -2 dropped
    for (int k = tid; k < n; k += nt) {
        const double nn = fsqrt(NX[k] * NX[k] + NY[k] * NY[k] + NZ[k] * NZ[k]);
        sm.CL[k] = nn > 1e-12 ? -1 : -2;
        sm.KEEP[k] = 0;
    }
    __syncthreads();
    for (int cl = 0; cl < n; ++cl) {
        // representative = first unassigned
        int first = 0x7fffffff;
        for (int k = tid; k < n; k += nt) if (sm.CL[k] == -1) { first = k; break; }
        __shared__ int s_first;
        if (tid == 0) s_first = 0x7fffffff;
        __syncthreads();
        if (first != 0x7fffffff) atomicMin(&s_first, first);
        __syncthreads();
        const int rep = s_first;
        if (rep == 0x7fffffff) break;
        const double rx = NX[rep], ry = NY[rep], rz = NZ[rep];
        for (int k = tid; k < n; k += nt) {
            if (sm.CL[k] == -1) {
                const double dp = NX[k] * rx + NY[k] * ry + NZ[k] * rz;
                if (acos(fmin(dp, 1.0)) < 1e-2) sm.CL[k] = cl;
            }
        }
        __syncthreads();
        // gather members (ascending) into HI[0..m)
        for (int k = tid; k < n; k += nt) sm.SC[k] = sm.CL[k] == cl;
        int m = 0;
        block_exclusive_scan(sm.SC, n, &m);
        for (int k = tid; k < n; k += nt) if (sm.CL[k] == cl) sm.HI[sm.SC[k]] = k;
        __syncthreads();
        if (m == 1) { if (tid == 0) sm.KEEP[sm.HI[0]] = 1; __syncthreads(); continue; }
        PH_MARK(PH_F_CLUSTER);
        // statistics: mean/variance per axis, max |coord|
        double s0 = 0, s1 = 0, s2 = 0, mx = 0;
        for (int e = tid; e < m; e += nt) {
            const int k = sm.HI[e];
            s0 += PX[k]; s1 += PY[k]; s2 += PZ[k];
            mx = fmax(mx, fmax(fabs(PX[k]), fmax(fabs(PY[k]), fabs(PZ[k]))));
        }
        {
            double rv[4] = {s0, s1, s2, mx};
            const int ro[4] = {RED_SUM, RED_SUM, RED_SUM, RED_MAX};
            bred_multi(rv, ro, 4, sm.red);
            s0 = rv[0]; s1 = rv[1]; s2 = rv[2]; mx = rv[3];
        }
        const double m0 = s0 / m, m1 = s1 / m, m2 = s2 / m;
        double v0 = 0, v1 = 0, v2 = 0;
        for (int e = tid; e < m; e += nt) {
            const int k = sm.HI[e];
            v0 += (PX[k] - m0) * (PX[k] - m0); v1 += (PY[k] - m1) * (PY[k] - m1); v2 += (PZ[k] - m2) * (PZ[k] - m2);
        }
        double var[3];
        {
            double rv[3] = {v0, v1, v2};
            const int ro[3] = {RED_SUM, RED_SUM, RED_SUM};
            bred_multi(rv, ro, 3, sm.red);
            var[0] = rv[0] / (m - 1); var[1] = rv[1] / (m - 1); var[2] = rv[2] / (m - 1);
        }
        // axis order: amin = first argmin (dropped first), then of the remaining two the first argmin is dropped next
        int amin = 0;
        if (var[1] < var[amin]) amin = 1;
        if (var[2] < var[amin]) amin = 2;
        const int r0 = amin == 0 ? 1 : 0, r1 = amin == 2 ? 1 : 2;          // remaining axes in order
        const int drop2 = var[r1] < var[r0] ? r1 : r0;                       // first argmin among remaining
        const int keep1 = drop2 == r0 ? r1 : r0;
        const double* PA[3] = {PX, PY, PZ};
        // extremes along the 1-D axis (first min / first max index, like argmin/argmax)
        double lo = INFINITY, hi = -INFINITY;
        for (int e = tid; e < m; e += nt) { const double c = PA[keep1][sm.HI[e]]; lo = fmin(lo, c); hi = fmax(hi, c); }
        {
            double rv[2] = {lo, hi};
            const int ro[2] = {RED_MIN, RED_MAX};
            bred_multi(rv, ro, 2, sm.red);
            lo = rv[0]; hi = rv[1];
        }
        __shared__ int s_lo, s_hi;
        if (tid == 0) { s_lo = 0x7fffffff; s_hi = 0x7fffffff; }
        __syncthreads();
        for (int e = tid; e < m; e += nt) {
            const double c = PA[keep1][sm.HI[e]];
            if (c == lo) atomicMin(&s_lo, e);
            if (c == hi) atomicMin(&s_hi, e);
        }
        __syncthreads();
        const int e_lo = s_lo, e_hi = s_hi;
        // --- is the set flat (3-D Qhull raises) ?  thickness w.r.t. the plane through a, b, c
        bool flat3 = m < 4;
        const int ka = sm.HI[e_lo], kb = sm.HI[e_hi];
        const V3<double> A = v3<double>(PX[ka], PY[ka], PZ[ka]), B = v3<double>(PX[kb], PY[kb], PZ[kb]);
        const V3<double> AB = B - A;
        const double lab = norm3(AB);
        // farthest point from line AB
        double far = -1.0;
        for (int e = tid; e < m; e += nt) {
            const int k = sm.HI[e];
            const V3<double> AP = v3<double>(PX[k], PY[k], PZ[k]) - A;
            const double dl = lab > 0 ? fdiv(norm3(cross(AB, AP)), lab) : norm3(AP);
            far = fmax(far, dl);
        }
        far = bred_max(far, sm.red);
        __shared__ int s_far;
        if (tid == 0) s_far = 0x7fffffff;
        __syncthreads();
        for (int e = tid; e < m; e += nt) {
            const int k = sm.HI[e];
            const V3<double> AP = v3<double>(PX[k], PY[k], PZ[k]) - A;
            const double dl = lab > 0 ? fdiv(norm3(cross(AB, AP)), lab) : norm3(AP);
            if (dl == far) atomicMin(&s_far, e);
        }
        __syncthreads();
        const bool collinear3 = !(far > 3.0 * distround(2, mx));
        if (!flat3 && !collinear3) {
            const int kc = sm.HI[s_far];
            const V3<double> C = v3<double>(PX[kc], PY[kc], PZ[kc]);
            V3<double> nrm = cross(AB, C - A);
            const double ln = norm3(nrm);
            double th = 0.0;
            for (int e = tid; e < m; e += nt) {
                const int k = sm.HI[e];
                th = fmax(th, fdiv(fabs(dot(nrm, v3<double>(PX[k], PY[k], PZ[k]) - A)), ln));
            }
            th = bred_max(th, sm.red);
            flat3 = !(th > 4.0 * distround(3, mx));
        } else {
            flat3 = true;
        }
        if (!flat3) {
            // genuine 3-D point set (contacts.py:126-133 succeeds with the 3-D Qhull): every point of a tetrahedron is a
            // hull vertex; larger sets go through the gift-wrapping hull (work buffers: HK as edge bit matrix, SC / TMP as
            // stack); a cluster too large for the buffers is kept whole and flagged
            bool done = false;
            if (m > 4) {
                done = hull3d_vertices(PX, PY, PZ, sm.HI, m, sm.KEEP, reinterpret_cast<unsigned*>(sm.HK),
                                       (size_t)4 * capK, sm.SC, sm.TMP, capK, sm.red, mx);
                if (!done) status |= 4;
            }
            if (!done) for (int e = tid; e < m; e += nt) sm.KEEP[sm.HI[e]] = 1;
            __syncthreads();
            continue;
        }
        // --- 2-D after dropping the min-variance axis: collinear (2-D Qhull raises) ?
        const int u_ax = r0, v_ax = r1;
        bool line2 = m < 3;
        if (!line2) {
            // extremes along the larger-variance remaining axis define the reference line
            const int ke_lo = sm.HI[e_lo], ke_hi = sm.HI[e_hi];
            const double ax_ = PA[u_ax][ke_lo], ay_ = PA[v_ax][ke_lo], bx_ = PA[u_ax][ke_hi], by_ = PA[v_ax][ke_hi];
            const double l2 = fsqrt((bx_ - ax_) * (bx_ - ax_) + (by_ - ay_) * (by_ - ay_));
            double fd2 = 0.0, mx2 = 0.0;
            for (int e = tid; e < m; e += nt) {
                const int k = sm.HI[e];
                const double px = PA[u_ax][k], py = PA[v_ax][k];
                const double cr = (bx_ - ax_) * (py - ay_) - (by_ - ay_) * (px - ax_);
                fd2 = fmax(fd2, l2 > 0 ? fdiv(fabs(cr), l2) : fsqrt((px - ax_) * (px - ax_) + (py - ay_) * (py - ay_)));
                mx2 = fmax(mx2, fmax(fabs(px), fabs(py)));
            }
            {
                double rv[2] = {fd2, mx2};
                const int ro[2] = {RED_MAX, RED_MAX};
                bred_multi(rv, ro, 2, sm.red);
                fd2 = rv[0]; mx2 = rv[1];
            }
            line2 = !(fd2 > 3.0 * distround(2, mx2));
        }
        if (line2) {
            // 1-D: min and max along the surviving axis, or a single point (contacts.py:143-150)
            if (tid == 0) {
                sm.KEEP[sm.HI[e_lo]] = 1;
                if (hi - lo > eps) sm.KEEP[sm.HI[e_hi]] = 1;
            }
            __syncthreads();
            continue;
        }
        PH_MARK(PH_F_STATS);
        // --- planar convex hull (strict vertices only)
        double* KU = sm.HK; double* KV = sm.HK + capK;
        for (int e = tid; e < m; e += nt) { const int k = sm.HI[e]; KU[e] = PA[u_ax][k]; KV[e] = PA[v_ax][k]; }
        __syncthreads();
        // Akl-Toussaint pre-filter: the support points of 8 directions span a polygon inscribed in the hull; points
        // STRICTLY inside it (by a margin far above the hull tolerance) cannot be hull vertices.  Dropping them in
        // parallel leaves only the boundary band for the sequential chain below.
        {
            __shared__ double s_ev[8][8];          // [warp][direction] best value
            __shared__ int s_ei[8][8];
            __shared__ double s_px[8], s_py[8];
            const double dxs[8] = {1, 1, 0, -1, -1, -1, 0, 1}, dys[8] = {0, 1, 1, 1, 0, -1, -1, -1};
            double bv[8]; int bi[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) { bv[q] = -INFINITY; bi[q] = 0x7fffffff; }
            double mxl = 0.0;
            for (int e = tid; e < m; e += nt) {
                const double x = KU[e], y = KV[e];
                mxl = fmax(mxl, fmax(fabs(x), fabs(y)));
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const double v = dxs[q] * x + dys[q] * y;
                    if (v > bv[q]) { bv[q] = v; bi[q] = e; }
                }
            }
            const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
#pragma unroll 1
            for (int q = 0; q < 8; ++q) {
#pragma unroll 1
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(DSDF_FULL, bv[q], o);
                    const int oi = __shfl_xor_sync(DSDF_FULL, bi[q], o);
                    if (ov > bv[q] || (ov == bv[q] && oi < bi[q])) { bv[q] = ov; bi[q] = oi; }
                }
                if (lane == 0) { s_ev[warp][q] = bv[q]; s_ei[warp][q] = bi[q]; }
            }
            const double mxc_all = bred_max(mxl, sm.red);     // (contains the barriers)
            if (tid < 8) {
                double v = -INFINITY; int ix = 0x7fffffff;
                for (int ww = 0; ww < nw; ++ww)
                    if (s_ev[ww][tid] > v || (s_ev[ww][tid] == v && s_ei[ww][tid] < ix)) { v = s_ev[ww][tid]; ix = s_ei[ww][tid]; }
                s_px[tid] = KU[ix]; s_py[tid] = KV[ix];
            }
            __syncthreads();
            const double margin = 1e-9 * (1.0 + mxc_all);
            for (int e = tid; e < m; e += nt) {
                const double x = KU[e], y = KV[e];
                bool inside = true;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const double ax_ = s_px[q], ay_ = s_py[q], bx_ = s_px[(q + 1) & 7], by_ = s_py[(q + 1) & 7];
                    const double ex = bx_ - ax_, ey = by_ - ay_;
                    const double len = fsqrt(ex * ex + ey * ey);
                    if (len > 0.0) inside = inside && ((ex * (y - ay_) - ey * (x - ax_)) > margin * len);
                }
                sm.SC[e] = inside ? 0 : 1;
            }
            __syncthreads();
            for (int e = tid; e < m; e += nt) sm.TMP[e] = sm.SC[e];
            int msurv = 0;
            block_exclusive_scan(sm.SC, m, &msurv);
            // order-preserving compaction of (KU, KV, HI)
            const int rounds = (m + nt - 1) / nt;
            for (int rd = 0; rd < rounds; ++rd) {
                const int e = rd * nt + tid;
                double x = 0, y = 0; int hi_ = 0, dst = -1;
                if (e < m && sm.TMP[e]) { dst = sm.SC[e]; x = KU[e]; y = KV[e]; hi_ = sm.HI[e]; }
                __syncthreads();
                if (dst >= 0) { KU[dst] = x; KV[dst] = y; sm.HI[dst] = hi_; }
                __syncthreads();
            }
            m = msurv;
            PH_MARK(PH_F_AKL);
            rank_sort_kv(KU, KV, sm.HI, m);
            // exact duplicates (faces sharing a vertex yield the same contact point): only the first of a run (lowest
            // contact index, the sort is stable in it) can be a hull vertex -- compact the others away in parallel so the
            // sequential chain below only walks distinct points
            for (int e = tid; e < m; e += nt) {
                const int keep = (e == 0) || !(KU[e] == KU[e - 1] && KV[e] == KV[e - 1]);
                sm.TMP[e] = keep; sm.SC[e] = keep;
            }
            int mu = 0;
            block_exclusive_scan(sm.SC, m, &mu);
            for (int rd = 0; rd < (m + nt - 1) / nt; ++rd) {
                const int e = rd * nt + tid;
                double x = 0, y = 0; int hi_ = 0, dst = -1;
                if (e < m && sm.TMP[e]) { dst = sm.SC[e]; x = KU[e]; y = KV[e]; hi_ = sm.HI[e]; }
                __syncthreads();
                if (dst >= 0) { KU[dst] = x; KV[dst] = y; sm.HI[dst] = hi_; }
                __syncthreads();
            }
            m = mu;
            PH_MARK(PH_F_SORT);
            if (tid == 0) sm.red[39] = mxc_all;
            __syncthreads();
        }
        if (tid == 0 || tid == 32) {
            // Monotone chain over the sorted distinct points: the lower hull (thread 0, ascending) and the upper hull
            // (thread 32, descending) are independent and run concurrently on two warps, each with its own stack.
            // b stays a vertex iff the turn a -> b -> e is left by more than the round-off bound: cr > tol |e - a|,
            // tested without the square root as cr > 0 and cr^2 > tol^2 |e - a|^2.
            const double mxc = sm.red[39];
            const double tol_d = 2.0 * distround(2, mxc), tol2 = tol_d * tol_d;
            const bool up = tid != 0;
            int* H = up ? sm.TMP : sm.SC;   // stack of sorted positions
            int top = 0;
            for (int i = 0; i < m; ++i) {
                const int e = up ? m - 1 - i : i;
                while (top >= 2) {
                    const int a = H[top - 2], b = H[top - 1];
                    const double ex = KU[e] - KU[a], ey = KV[e] - KV[a];
                    const double cr = (KU[b] - KU[a]) * ey - (KV[b] - KV[a]) * ex;   // > 0: left turn keeps b
                    if (cr > 0.0 && cr * cr > tol2 * (ex * ex + ey * ey)) break;
                    --top;
                }
                H[top++] = e;
            }
            for (int t = 0; t < top; ++t) sm.KEEP[sm.HI[H[t]]] = 1;
        }
        __syncthreads();
        PH_MARK(PH_F_CHAIN);
    }
    __syncthreads();
    return status;
}

// One CTA per world: broad phase, _overlap, and both search directions of every body pair, fused.
#ifndef DSDF_CONTACT_THREADS
#define DSDF_CONTACT_THREADS 128
#endif
enum { CONTACT_THREADS = DSDF_CONTACT_THREADS };
#ifndef DSDF_CONTACT_MINBLOCKS
#define DSDF_CONTACT_MINBLOCKS 4
#endif
__global__ void __launch_bounds__(CONTACT_THREADS, DSDF_CONTACT_MINBLOCKS)
contacts_kernel(const BodyGeom* __restrict__ geom, const int* __restrict__ pairs, int npairs,
                const double* __restrict__ p, const double* __restrict__ shape, const unsigned char* __restrict__ active,
                int nb, double eps, double tol, double fd_eps, double body_eps, int detach_b2,
                int capK, int maxc,
                int* __restrict__ count, int* __restrict__ cbody, int* __restrict__ cface, double* __restrict__ cabc,
                double* __restrict__ cgeo, int* __restrict__ wstatus, int* __restrict__ pre_ids, int* __restrict__ pre_cnt,
                const int* __restrict__ vmap, const int* __restrict__ ctrl) {
    extern __shared__ double smraw[];
    __shared__ int s_cnt;
    // loop mode (ctrl != NULL, dsdf_steploop.cu): CTA w detects the contacts of virtual world w (poses p[w], outputs [w])
    // with the shapes / per-world meshes / per-world grids of the real world wg = vmap[w]
    const int w = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    if (ctrl && (loop_idle(ctrl) || w >= ctrl[CT_NVIRT])) return;
    const int wg = vmap ? vmap[w] : w;
    if (active && !active[w]) return;
    const int ndirs = 2 * npairs;
    RefineSmem sm;
    sm.P = smraw; sm.X = sm.P + 9 * (size_t)capK; sm.ABC = sm.X + 3 * (size_t)capK; sm.HK = sm.X + (size_t)capK;
    sm.red = sm.ABC + 3 * (size_t)capK;
    sm.ID = reinterpret_cast<int*>(sm.red + 40);
    sm.SC = sm.ID + capK; sm.CL = sm.SC + capK; sm.HI = sm.CL + capK; sm.KEEP = sm.HI + capK; sm.TMP = sm.KEEP + capK;
    int nout = 0, status = 0;
    for (int pair = 0; pair < npairs; ++pair) {
        const int bi = pairs[2 * pair], bj = pairs[2 * pair + 1];
        Q4<double> qi, qj; V3<double> xi, xj;
        load_pose(p, w, nb, bi, qi, xi);
        load_pose(p, w, nb, bj, qj, xj);
        const double si = shape[((size_t)wg * nb + bi) * 4 + 3], sj = shape[((size_t)wg * nb + bj) * 4 + 3];
        // broad phase: AABB of the rotated cube of half side scale + eps (declared py3ode semantics)
        const M3<double> Ri = q2mat(qi), Rj = q2mat(qj);
        bool hit = true;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const double hi = (fabs(Ri.m[3 * a]) + fabs(Ri.m[3 * a + 1]) + fabs(Ri.m[3 * a + 2])) * (si + body_eps);
            const double hj = (fabs(Rj.m[3 * a]) + fabs(Rj.m[3 * a + 1]) + fabs(Rj.m[3 * a + 2])) * (sj + body_eps);
            const double dc = a == 0 ? xi.x - xj.x : (a == 1 ? xi.y - xj.y : xi.z - xj.z);
            hit = hit && (fabs(dc) <= hi + hj);
        }
        int ov = 0;
        PH_MARK(-1);
        if (hit) ov = any_vertex_in_cube(world_geom(geom[bi], wg), wg, qi, xi, qj, xj, sj) &&
                      any_vertex_in_cube(world_geom(geom[bj], wg), wg, qj, xj, qi, xi, si);
        PH_MARK(PH_OVERLAP);
        if (!ov) {
            if (pre_cnt && tid == 0) { pre_cnt[(size_t)w * ndirs + 2 * pair] = -1; pre_cnt[(size_t)w * ndirs + 2 * pair + 1] = -1; }
            continue;
        }
        for (int rev = 0; rev < 2; ++rev) {
            const int d = 2 * pair + rev;
            const int i1 = rev ? bj : bi, i2 = rev ? bi : bj;
            const BodyGeom g1 = world_geom(geom[i1], wg);
            const SdfShape s1 = body_shape(g1, shape, wg, nb, i1);
            const SdfShape s2 = body_shape(geom[i2], shape, wg, nb, i2);
            const Q4<double> q1 = rev ? qj : qi, q2 = rev ? qi : qj;
            const V3<double> x1 = rev ? xj : xi, x2 = rev ? xi : xj;
            PH_MARK(-1);
            const int ncand = gather_candidates(g1, wg, s2, q1, x1, q2, x2, eps, capK, sm.ID, &s_cnt);
            PH_MARK(PH_GATHER);
            if (ncand > capK) status |= 1;
            DirResult r = search_direction(sm, capK, g1, s1, s2, q1, x1, q2, x2, wg, ncand, eps, tol, fd_eps, detach_b2 != 0);
            if (pre_cnt) {
                if (tid == 0) pre_cnt[(size_t)w * ndirs + d] = r.count;
                for (int k = tid; k < r.count; k += nt) pre_ids[((size_t)w * ndirs + d) * capK + k] = sm.ID[k];
            }
            PH_MARK(-1);
            if (r.valid) status |= filter_contacts(sm, capK, r.count, eps);
            else { status |= 8; for (int k = tid; k < r.count; k += nt) sm.KEEP[k] = 1; __syncthreads(); }
            PH_MARK(PH_FILTER);
            // append kept contacts in ascending face order
            for (int k = tid; k < r.count; k += nt) sm.SC[k] = sm.KEEP[k];
            int nk = 0;
            block_exclusive_scan(sm.SC, r.count, &nk);
            for (int k = tid; k < r.count; k += nt) {
                if (!sm.KEEP[k]) continue;
                const int o = nout + sm.SC[k];
                if (o >= maxc) continue;
                const size_t oo = (size_t)w * maxc + o;
                cbody[2 * oo] = i1; cbody[2 * oo + 1] = i2;
                cface[oo] = sm.ID[k];
                cabc[3 * oo] = sm.ABC[k]; cabc[3 * oo + 1] = sm.ABC[capK + k]; cabc[3 * oo + 2] = sm.ABC[2 * capK + k];
#pragma unroll
                for (int c = 0; c < 9; ++c) cgeo[10 * oo + c] = sm.P[(size_t)c * capK + k];
                cgeo[10 * oo + 9] = sm.X[k];
            }
            if (nout + nk > maxc) status |= 2;
            nout = min(nout + nk, maxc);
            __syncthreads();
            PH_MARK(PH_APPEND);
            if (!r.valid) {                       // contacts.py:238-240: reverse direction only after a valid first one
                if (rev == 0 && pre_cnt && tid == 0) pre_cnt[(size_t)w * ndirs + d + 1] = -1;
                break;
            }
        }
    }
    if (tid == 0) { count[w] = nout; wstatus[w] = status; }
}

// _filter_contacts (contacts.py:97-158) as a stand-alone operator: one CTA per contact list.
__global__ void __launch_bounds__(CONTACT_THREADS)
filter_kernel(const double* __restrict__ normals, const double* __restrict__ p1, const int* __restrict__ n, int capK, double eps,
              int* __restrict__ keep, int* __restrict__ status) {
    extern __shared__ double smraw[];
    const int w = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    RefineSmem sm;
    sm.P = smraw; sm.X = sm.P + 9 * (size_t)capK; sm.ABC = sm.X + 3 * (size_t)capK; sm.HK = sm.X + (size_t)capK;
    sm.red = sm.ABC + 3 * (size_t)capK;
    sm.ID = reinterpret_cast<int*>(sm.red + 40);
    sm.SC = sm.ID + capK; sm.CL = sm.SC + capK; sm.HI = sm.CL + capK; sm.KEEP = sm.HI + capK; sm.TMP = sm.KEEP + capK;
    const int m = min(n[w], capK);
    for (int k = tid; k < m; k += nt) {
        const size_t o = ((size_t)w * capK + k) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) { sm.P[(size_t)c * capK + k] = normals[o + c]; sm.P[(size_t)(3 + c) * capK + k] = p1[o + c]; }
    }
    __syncthreads();
    const int st = filter_contacts(sm, capK, m, eps);
    __syncthreads();
    for (int k = tid; k < m; k += nt) keep[(size_t)w * capK + k] = sm.KEEP[k];
    if (tid == 0) status[w] = st | (n[w] > capK ? 1 : 0);
}

}  // namespace dsdf

using namespace dsdf;

extern "C" {

static size_t g_contacts_smem = 0, g_filter_smem = 0;

int dsdf_contacts_detect(const dsdf_body_geom* geom, const int32_t* pairs, int npairs, const double* p,
                         const double* shape, const unsigned char* active,
                         int W, int nb, double eps, double tol, double fd_eps, double body_eps, int detach_b2,
                         int capK, int maxc, int32_t* count, int32_t* cbody, int32_t* cface, double* cabc, double* cgeo,
                         int32_t* wstatus, int32_t* pre_ids, int32_t* pre_cnt, const int32_t* vmap, const int32_t* ctrl,
                         void* stream) {
    if (W <= 0 || nb <= 0 || npairs < 0 || capK < 32 || capK > 1024 || (capK & 3) || maxc <= 0) return -1;
    static_assert(sizeof(BodyGeom) == sizeof(dsdf_body_geom), "BodyGeom must mirror dsdf_body_geom");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = refine_smem_bytes(capK);
    if (smem > 227 * 1024) return -2;
    cudaError_t e = ensure_smem(contacts_kernel, smem, &g_contacts_smem);
    if (e != cudaSuccess) return (int)e;
    contacts_kernel<<<W, CONTACT_THREADS, smem, st>>>(reinterpret_cast<const BodyGeom*>(geom), pairs, npairs, p, shape, active, nb,
                                          eps, tol, fd_eps, body_eps, detach_b2, capK, maxc, count, cbody, cface, cabc,
                                          cgeo, wstatus, pre_ids, pre_cnt, vmap, ctrl);
    return (int)cudaGetLastError();
}

int dsdf_filter_contacts(const double* normals, const double* p1, const int32_t* n, int W, int capK, double eps,
                         int32_t* keep, int32_t* status, void* stream) {
    if (W <= 0 || capK < 32 || capK > 1024 || (capK & 3)) return -1;
    const size_t smem = refine_smem_bytes(capK);
    if (smem > 227 * 1024) return -2;
    cudaError_t e = ensure_smem(filter_kernel, smem, &g_filter_smem);
    if (e != cudaSuccess) return (int)e;
    filter_kernel<<<W, CONTACT_THREADS, smem, (cudaStream_t)stream>>>(normals, p1, n, capK, eps, keep, status);
    return (int)cudaGetLastError();
}

int dsdf_contacts_phase_cycles(unsigned long long* out8, int reset) {   /* out: PH_COUNT = 16 counters */
#ifdef DSDF_PHASE_PROFILE
    if (out8 && cudaMemcpyFromSymbol(out8, g_phase, sizeof(unsigned long long) * PH_COUNT) != cudaSuccess) return 1;
    if (reset) { unsigned long long z[PH_COUNT] = {0}; if (cudaMemcpyToSymbol(g_phase, z, sizeof(z)) != cudaSuccess) return 1; }
    return 0;
#else
    (void)out8; (void)reset;
    return -1;
#endif
}

}  // extern "C"
