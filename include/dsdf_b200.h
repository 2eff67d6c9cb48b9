/*
 * dsdf_b200 -- C ABI of the B200-native DiffSDFSim stepping hot path.
 *
 * Every entry point is extern "C", takes plain device pointers / sizes / a CUDA
 * stream (as void*), never allocates or frees caller memory, keeps no global
 * mutable state and returns an int status (0 = launched OK, <0 = argument or
 * capacity error, >0 = CUDA error code).  Per-world solver/search conditions
 * are reported through int32 status arrays on the device, never by exceptions.
 *
 * Each function names the reference interface it replaces (paths relative to
 * the upstream repository).  All floating point is IEEE binary64 ("f64"): the
 * reference computes in torch.double (lcp_physics/physics/utils.py:59).
 *
 * Batch convention: the leading dimension of every array is the world index W;
 * arrays are dense row-major with the documented trailing shape.
 */
#ifndef DSDF_B200_H
#define DSDF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSDF_VERSION 1

/* per-world LCP status bits (int32) */
#define DSDF_LCP_Q_SINGULAR   1   /* LU of Q hit a zero pivot            (batch.py:417-424) */
#define DSDF_LCP_Q_NOT_SPD    2   /* SPD check failed                    (lcp.py:109-113)   */
#define DSDF_LCP_FACTOR_FAIL  4   /* LU of R + D^-1 hit a zero pivot -> best iterate returned (batch.py:134-137) */
#define DSDF_LCP_INACCURATE   8   /* best residual > 1                   (batch.py:165,229) */
#define DSDF_LCP_TOO_LARGE   16   /* nineq_w[w] > nineq_smem: not solved (x = NaN)                  */

/* SDF kinds */
#define DSDF_SDF_BOX      0
#define DSDF_SDF_SPHERE   1
#define DSDF_SDF_CYLINDER 2
#define DSDF_SDF_GRID     3
#define DSDF_SDF_BOX_ROUNDED 4   /* bodies.py:166-181,856-870: box(dims - 2r) - r; shape = (dims-2r)/scale, extra[0] = r/scale   */
#define DSDF_SDF_BRICK    5      /* bodies.py:184-200,873-886: in-plane rounded box; shape = dims/scale, extra[0] = r/scale        */
#define DSDF_SDF_BOWL     6      /* bodies.py:128-163,1012-1026: half shell; shape = [r/scale, d/scale]                            */

int dsdf_version(void);

/* ------------------------------------------------------------------ LCP ----
 * Replaces LCPFunction(...).forward  (lcp_physics/lcp/lcp.py:48-153) with
 * pre_factor_kkt / forward / factor_kkt / solve_kkt / get_step
 * (lcp_physics/lcp/solvers/batch.py:413-479, 70-231, 485-520, 380-410, 234-237).
 *
 *   minimise 1/2 z'Qz + p'z  s.t.  G z + s = h + F lam (mixed LCP), A z = b
 *
 * Q (W,nz,nz)  p (W,nz)  G (W,nineq,nz)  h (W,nineq)  A (W,neq,nz)  b (W,neq)
 * F (W,nineq,nineq).  nineq_w (W) optional (NULL = all worlds use nineq): the
 * number of ACTIVE inequality rows of each world (rows/cols beyond it ignored).
 * Outputs: x (W,nz) nu (W,neq) lam (W,nineq) s (W,nineq) = best-residual
 * iterate; status (W) bit mask; iters (W) iterations run.
 * nineq_smem (0 = nineq): rows the launch sizes its shared memory for; lets a batch be padded to a large
 * capacity `nineq` (global strides) while the CTA only holds max_w nineq_w[w] rows.  A world with more active
 * rows gets status DSDF_LCP_TOO_LARGE.
 * ws: workspace of dsdf_lcp_workspace_bytes(...) bytes.
 * Every reduction the reference takes over the whole batch tensor is taken per
 * world here (the reference engine only ever runs nBatch = 1).
 */
size_t dsdf_lcp_workspace_bytes(int W, int nz, int neq, int nineq);
size_t dsdf_lcp_smem_bytes(int nz, int neq, int nineq);   /* > 227 KiB: problem too large for this kernel */
int dsdf_lcp_forward(const double* Q, const double* p, const double* G, const double* h,
                     const double* A, const double* b, const double* F, const int32_t* nineq_w,
                     int W, int nz, int neq, int nineq, int nineq_smem,
                     double eps, int not_improved_lim, int max_iter, int check_spd,
                     double* x, double* nu, double* lam, double* s,
                     int32_t* status, int32_t* iters, void* ws, void* stream);

/* Replaces LCPFunctionFn.backward (lcp_physics/lcp/lcp.py:156-213).
 * gz (W,nz) = dL/dzhat.  Outputs dQ (W,nz,nz) dp (W,nz) dG (W,nineq,nz) dh (W,nineq)
 * dA (W,neq,nz) db (W,neq) dF (W,nineq,nineq); any output pointer may be NULL.
 */
int dsdf_lcp_backward(const double* Q, const double* G, const double* A, const double* F,
                      const int32_t* nineq_w, const double* x, const double* nu, const double* lam,
                      const double* s, const double* gz, int W, int nz, int neq, int nineq, int nineq_smem,
                      double* dQ, double* dp, double* dG, double* dh, double* dA, double* db, double* dF,
                      int32_t* status, void* ws, void* stream);

/* ------------------------------------------------------------ SDF query ----
 * Replaces SDF3D.query_sdfs(pts_loc, return_grads)  (sdf_physics/physics3d/bodies.py:721-760) with the
 * analytic SDFs (bodies.py:38-125) and the grid SDF (bodies.py:203-257; ev_sdf_utils.grid_interp).
 * shape (W,4) = [a,b,c,scale]: box dims/scale | sphere r/scale | cylinder r/scale,h/scale | grid: unused.
 * extra0 / extra1: the further parameters of the kinds that need more than three (DSDF_SDF_BOX_ROUNDED / BRICK:
 * extra0 = r/scale); 0 for the others.
 * grid: W grids of res^3 doubles, world w at grid + w*grid_world_stride (stride 0 = shared grid).
 * pts (W,N,3) body-frame points -> sdf (W,N), dir (W,N,3) unit gradient (NULL/want_dir=0 to skip).
 * Outside the cube |p| <= scale: sdf = scale, dir = 0.
 */
int dsdf_sdf_query(int kind, const double* shape, double extra0, double extra1, const double* grid, int res,
                   long long grid_world_stride, const double* pts, int W, int N, int want_dir, double* sdf, double* dir,
                   void* stream);
/* VJP of the above w.r.t. pts with torch-autograd conventions (DiffGridSDF.backward for grids, bodies.py:253-257):
 * gpts (W,N,3) = gsdf * d sdf/d pts + gdir . d dir/d pts ; gsdf / gdir may be NULL. */
int dsdf_sdf_query_backward(int kind, const double* shape, double extra0, double extra1, const double* grid, int res,
                            long long grid_world_stride, const double* pts, int W, int N, const double* gsdf,
                            const double* gdir, double* gpts, void* stream);

/* ----------------------------------------------------------- integrator ----
 * Replaces Body3D.move (sdf_physics/physics3d/bodies.py:488-496): q <- standardize(quat(expmap(w dt)) * q),
 * x <- x + v dt.  p (W,nb,7) = [qw,qx,qy,qz,x,y,z], v (W,nb,6) = [w,v], dt (W), active (W) uint8 or NULL;
 * inactive worlds copy p through.  The world-frame inertia update of set_p (bodies.py:509-511) is fused
 * into the dynamics kernel that consumes it.
 */
int dsdf_integrate(const double* p, const double* v, const double* dt, const unsigned char* active, int W, int nb,
                   double* p_out, void* stream);
/* gp (W,nb,7), gv (W,nb,6), gdt (W,nb) [per body; caller sums over bodies] from gp_out (W,nb,7). */
int dsdf_integrate_backward(const double* p, const double* v, const double* dt, const unsigned char* active, int W,
                            int nb, const double* gp_out, double* gp, double* gv, double* gdt, void* stream);

/* ------------------------------------------------------ SDF collision query ----
 * Per-body geometry handed to the contact kernels.  Meshes and grids are INPUTS of the hot path
 * (the reference meshes bodies at construction time: bodies.py:638, 652-712).
 */
typedef struct dsdf_body_geom {
    int32_t kind, nverts, nfaces, res;
    const double* verts;          /* (nverts,3) body frame; world w at verts + w*vert_world_stride (0 = shared) */
    const int32_t* faces;         /* (nfaces,3), shared by all worlds */
    const double* grid;           /* res^3 SDF samples on [-1,1]^3 (kind == GRID); world w at grid + w*grid_world_stride */
    long long vert_world_stride, grid_world_stride;
    /* Optional uniform cell index over the body-frame mesh (has_cells = 0: scan everything).  Cell (ix,iy,iz) of
     * cell_dims covers cell_lo + [ix,ix+1) / cell_inv ...; faces are binned by centroid, vertices by position, as
     * CSR lists: items of cell c are *_items[*_start[c] .. *_start[c+1]).  Only used to SKIP work that provably
     * cannot pass the reference's tests (points outside the other body's cube); results are unchanged. */
    double cell_lo[3], cell_inv;
    int32_t cell_dims[3], has_cells;
    const int32_t *fcell_start, *fcell_items, *vcell_start, *vcell_items;
    /* max over faces of max_i |centroid - v_i| (body frame), or 0 if unknown.  Lets the candidate pass discard, with a
     * cheap conservative fp32 bound, faces whose centroid is provably farther than this radius + eps from the other
     * body; everything that survives goes through the exact fp64 test, so results are unchanged. */
    double max_face_rad;
    /* Per-world topology, for bodies whose mesh differs from world to world (iso-surfaces of per-world SDF grids):
     * world w uses faces + w*face_world_stride, nfaces_w[w] faces and nverts_w[w] vertices (nfaces / nverts above are then
     * the allocated maxima).  0 / NULL = one topology shared by all worlds. */
    long long face_world_stride;
    const int32_t *nfaces_w, *nverts_w;
    double extra[2];              /* further SDF parameters of the body kind (rounding radius / scale), shared by all worlds */
} dsdf_body_geom;

/* per-world contact status bits (int32) */
#define DSDF_CON_CAND_OVERFLOW  1   /* more centroid candidates than capK in some direction */
#define DSDF_CON_OVERFLOW       2   /* more contacts than maxc */
#define DSDF_CON_HULL3D         4   /* a non-planar cluster too large for the device 3-D hull (8 m > 4 capK) was kept whole */
#define DSDF_CON_PENETRATION    8   /* some pen > tol: the step attempt will be rejected (world.py:270) */
#define DSDF_CON_STALLED       16   /* (step loop, ctrl[14] only) a world exhausted the tape slots of one step and left it early */

/* Replaces World.find_contacts (lcp_physics/physics/world.py:396-399) with FWContactHandler
 * (sdf_physics/physics3d/contacts.py:221-272): broad phase (AABB of each body's rotated cube of half side
 * scale+body_eps, pairs (i<j) from `pairs` (npairs,2), no_contact pairs already removed), _overlap (:27-36),
 * _frank_wolfe (:39-94), _compute_contacts (:161-214), _filter_contacts (:97-158), both search directions with the
 * reference's "reverse only if the first is valid" rule (:238-240).  One CTA per world, one launch.
 * p (W,nb,7), shape (W,nb,4), active (W) uint8 or NULL (inactive worlds keep their previous outputs).
 * Outputs (capacity maxc contacts per world, ordered pair -> direction -> face id):
 *   count (W); cbody (W,maxc,2) = (mesh body, sdf body); cface (W,maxc) face id on the mesh body;
 *   cabc (W,maxc,3) barycentrics; cgeo (W,maxc,10) = [normal(3), p1(3), p2(3), pen]; wstatus (W).
 *   pre_ids (W,2*npairs,capK) / pre_cnt (W,2*npairs): PRE-filter contact face ids per direction (parity
 *   evidence; -1 = direction not searched); both may be NULL.
 * vmap / ctrl (both NULL outside the device-resident step loop below): CTA w works on VIRTUAL world w (poses p[w],
 * outputs at [w]) with the shapes and per-world geometry of the real world vmap[w]; ctrl = the loop's control block
 * (every CTA returns at once when the loop is idle).
 */
int dsdf_contacts_detect(const dsdf_body_geom* geom, const int32_t* pairs, int npairs, const double* p,
                         const double* shape, const unsigned char* active,
                         int W, int nb, double eps, double tol, double fd_eps, double body_eps, int detach_b2,
                         int capK, int maxc, int32_t* count, int32_t* cbody, int32_t* cface, double* cabc, double* cgeo,
                         int32_t* wstatus, int32_t* pre_ids, int32_t* pre_cnt, const int32_t* vmap, const int32_t* ctrl,
                         void* stream);
/* Replaces _filter_contacts (sdf_physics/physics3d/contacts.py:97-158) as a stand-alone operator: W independent contact
 * lists, list w = the first n[w] rows of normals / p1 (W,capK,3).  keep (W,capK) <- 1 for the contacts the reference keeps:
 * zero normals dropped, greedy clustering by angle < 1e-2 rad to the first remaining normal, per cluster the vertices of the
 * convex hull of p1 (3-D; min-variance axis dropped when flat -> 2-D; -> 1-D min / max, one point if the extent <= eps),
 * with Qhull's degeneracy decisions (scipy.spatial.ConvexHull in the reference).  status (W): DSDF_CON_* bits. */
int dsdf_filter_contacts(const double* normals, const double* p1, const int32_t* n, int W, int capK, double eps,
                         int32_t* keep, int32_t* status, void* stream);
/* Profiling aid: cumulative SM cycles (thread 0 of every CTA) per phase of the contact kernel
 * [overlap, gather, sort+init, frank-wolfe, push+compact, geometry, filter, append]; returns -1 unless the library
 * was built with -DDSDF_PHASE_PROFILE (DSDF_PHASE_PROFILE=1 python -m diffsdfsim_b200.build). Host pointer out8. */
int dsdf_contacts_phase_cycles(unsigned long long* out8, int reset);
/* Profiling aid: cumulative SM cycles (lane / thread 0 of every CTA) per phase of the dynamics forward kernel
 * [load, residuals, factor (a, den, AP, YG), M~_FF assembly, LU, KKT solve pass 0, ratio step + corrector,
 * KKT solve pass 1, step update, best-iterate tracking] and, last, the number of loop passes (the initial point
 * included); returns -1 unless the library was built with -DDSDF_PHASE_PROFILE. Host pointer out11. */
int dsdf_dynamics_phase_cycles(unsigned long long* out11, int reset);
/* VJP of cgeo w.r.t. the poses (the reference's grad-enabled second _compute_contacts, contacts.py:262-264):
 * gp (W,nb,7) from ggeo (W,maxc,10).  wmap (W) or NULL: row w carries the poses / contacts of world wmap[w], whose
 * shapes and per-world meshes / grids are used (a compact batch of rows; NULL: row = world).
 * With gshape / gctri the gradients w.r.t. the SHAPES as well (radius / dimension fitting: the reference's grad-enabled
 * _compute_contacts differentiates through the SDF parameters, the scale and the mesh vertices):
 * gshape (W,nb,4) = d/d[a,b,c,scale] of every body, gctri (W,maxc,3) = gradient w.r.t. the body-frame point
 * sum(abc * vertices of the face) on the mesh body of each contact (the caller scatters it onto the vertices with the
 * weights cabc).  gshape == gctri == NULL: pose gradients only. */
int dsdf_contact_geometry_backward(const dsdf_body_geom* geom, const double* p, const double* shape, int W, int nb,
                                   double fd_eps, int detach_b2, int maxc, const int32_t* count, const int32_t* cbody,
                                   const int32_t* cface, const double* cabc, const double* ggeo, double* gp,
                                   const int32_t* wmap, double* gshape, double* gctri, void* stream);

/* ------------------------------------------------------------- dynamics ----
 * Replaces the matrix assembly of PdipmEngine.solve_dynamics (lcp_physics/physics/engines.py:31-79) with
 * World3D.M/Jc/Jf (sdf_physics/physics3d/world.py:48-101), orthogonal (physics3d/utils.py:247-256) and
 * World.restitutions/mu/E (lcp_physics/physics/world.py:402-409, 480-501), for all worlds:
 *   Q = blockdiag_b(R(q_b) I_b R(q_b)', m_b 1)      (W,nz,nz),  nz = 6 nb
 *   pvec = Q v + dt f                                (W,nz)
 *   G = [Jc; Jf; 0]   h = [e (Jc v); 0; 0]           (W,niCap,nz), (W,niCap),  niCap = maxc (2 + fric_dirs)
 *   F  (E, mu, -E' blocks)                            (W,niCap,niCap)
 *   nineq_w = nc (2 + fric_dirs), or -1 for inactive worlds (dsdf_lcp_* then skip them)
 * Inputs: p (W,nb,7) v (W,nb,6) mass (W,nb) Ibody (W,nb,3,3) fric (W,nb) rest (W,nb) f (W,nb,6) dt (W)
 * active (W) uint8|NULL, contacts count (W) cbody (W,maxc,2) cgeo (W,maxc,10).  fric_dirs in {4, 8}.
 * The equality rows A (pinned bodies / axis locks) are constant and supplied by the caller to dsdf_lcp_*.
 * new_v = -x of dsdf_lcp_forward (engines.py:81-82).
 */
int dsdf_dynamics_assemble(const double* p, const double* v, const double* mass, const double* Ibody,
                           const double* fric, const double* rest, const double* f, const double* dt,
                           const unsigned char* active, const int32_t* count, const int32_t* cbody, const double* cgeo,
                           int W, int nb, int maxc, int fric_dirs,
                           double* Q, double* pvec, double* G, double* h, double* F, int32_t* nineq_w, void* stream);
/* Reverse mode of the assembly: contracts the LCP gradients (dQ, dp, dG, dh, dF of dsdf_lcp_backward) onto the
 * physical inputs.  stop_contact_grad / stop_friction_grad detach the contact tuple in Jc / Jf
 * (physics3d/world.py:59-62, 77-80).  Outputs: gp (W,nb,7) gv (W,nb,6) gmass (W,nb) gI (W,nb,3,3) gfric (W,nb)
 * grest (W,nb) gf (W,nb,6) gdt (W) ggeo (W,maxc,10). */
int dsdf_dynamics_assemble_backward(const double* p, const double* v, const double* mass, const double* Ibody,
                                    const double* fric, const double* rest, const double* f, const double* dt,
                                    const unsigned char* active, const int32_t* count, const int32_t* cbody,
                                    const double* cgeo, int W, int nb, int maxc, int fric_dirs,
                                    int stop_contact_grad, int stop_friction_grad,
                                    const double* Q, const double* G,
                                    const double* dQ, const double* dp, const double* dG, const double* dh, const double* dF,
                                    double* gp, double* gv, double* gmass, double* gI, double* gfric, double* grest,
                                    double* gf, double* gdt, double* ggeo, void* stream);

/* ------------------------------------------------- fused contact dynamics ----
 * Replaces PdipmEngine.solve_dynamics (lcp_physics/physics/engines.py:31-83) end to end:
 * assembly (as dsdf_dynamics_assemble) + the PDIPM of lcp_physics/lcp/solvers/batch.py:70-237 with the Newton
 * systems reduced through the per-contact block structure of F + D^-1 (closed-form block inverse, pivoted LU of
 * the free block of the (6 nb + neq)^2 reduced KKT matrix) instead of the dense nineq^2 factorisation.
 * Same iterates as dsdf_lcp_forward on the assembled matrices up to round-off.
 * eq_rows (neq,2) int32 = [body, velocity component] of each equality row (rows of Je are 0/1 selections:
 * sdf_physics/physics3d/constraints.py:32-145).
 * Outputs x (W,6nb), new_v (W,6nb) = -x (engines.py:81-82; inactive worlds: v passed through; may be NULL),
 * nu (W,neq), lam / s (W, maxc (2+fric_dirs)) in the reference's row order [normal | friction | cone], status (W),
 * iters (W).
 *
 * One call runs one to three kernel launches, one per contact-count class: a launch sized for C contacts solves the
 * worlds with count_min < count <= C, and the last class reports the worlds above its C as DSDF_LCP_TOO_LARGE.
 * ncontacts_small (> 0): contacts of the bulk of the worlds; ncontacts_large: of the few worlds with many more
 * (ncontacts_large <= ncontacts_small: one class); both are clamped to maxc.  Two kernels run the classes:
 *   one warp per world, the whole world in shared memory: up to 64 contacts, small worlds (the default);
 *   one CTA of 256 threads per world for many bodies (up to ~120 free velocity components) and / or more than 64
 *   contacts: shared memory holds what scales with the bodies, a global workspace holds what scales with the contacts
 *   (no cap on their number).
 * force_cta = 1 runs every world on the one-CTA kernel.  dsdf_dynamics_plan returns the number of launches of a call
 * (or -2: the world does not fit the one-CTA kernel's shared memory) and the bytes of the workspace it needs, 0 when no
 * world goes to the one-CTA kernel (workspace may then be NULL).
 * vmap / ctrl (both NULL outside the device-resident step loop below): CTA w solves VIRTUAL world w (its own dt[w],
 * outputs at [w]) with the state, parameters and current contacts of the real world vmap[w]; ctrl = the loop's
 * control block (every CTA returns at once when the loop is idle).
 */
int dsdf_dynamics_plan(int W, int nb, int neq, int fric_dirs, int ncontacts_small, int ncontacts_large, int force_cta,
                       size_t* workspace_bytes);
int dsdf_dynamics_solve(const double* p, const double* v, const double* mass, const double* Ibody,
                        const double* fric, const double* rest, const double* f, const double* dt,
                        const unsigned char* active, const int32_t* count, const int32_t* cbody, const double* cgeo,
                        const int32_t* eq_rows, int W, int nb, int neq, int maxc, int ncontacts_small,
                        int ncontacts_large, int force_cta, int fric_dirs, double eps, int not_improved_lim,
                        int max_iter, double* x, double* new_v, double* nu, double* lam, double* s, int32_t* status,
                        int32_t* iters, const int32_t* vmap, int32_t* ctrl, double* workspace, void* stream);
/* Replaces LCPFunctionFn.backward (lcp_physics/lcp/lcp.py:156-213) + the autograd of the assembly, fused: from
 * g_new_v = dL/dnew_v (W,6nb) straight to the gradients of the physical inputs (no dense dG / dF is materialised).
 * Inactive worlds pass g_new_v through to gv.  Contact-count classes, kernels and workspace as in the forward. */
int dsdf_dynamics_solve_backward(const double* p, const double* v, const double* mass, const double* Ibody,
                                 const double* fric, const double* rest, const double* f, const double* dt,
                                 const unsigned char* active, const int32_t* count, const int32_t* cbody,
                                 const double* cgeo, const int32_t* eq_rows, int W, int nb, int neq, int maxc,
                                 int ncontacts_small, int ncontacts_large, int force_cta, int fric_dirs,
                                 int stop_contact_grad, int stop_friction_grad,
                                 const double* x, const double* lam, const double* s, const double* g_new_v,
                                 double* gp, double* gv, double* gmass, double* gI, double* gfric, double* grest,
                                 double* gf, double* gdt, double* ggeo, double* workspace, void* stream);

/* ------------------------------------------------------ step bookkeeping ----
 * Replaces the accept / reject / halve-dt / remaining-time / time-of-contact control flow of World.step_dt and
 * World.step (lcp_physics/physics/world.py:119-139, 241-356) for all worlds after one attempt
 * (solve -> move -> find_contacts).  One thread per world, no host round trip except the 4 flags.
 * In:  active (W) uint8, dt_try (W), t (W), end_t (W) or NULL (fixed_dt = False), world_dt, strict (0/1),
 *      toc_enabled (0/1); the previous contact set (*_o) and the freshly detected one (*_n, capacity maxc).
 * Out: accept (W) uint8; t_out = t (+ dt_try if accepted); dt_next (halved on reject, remaining time after a short
 *      accepted sub-step); active_next (W); toc_now (W) / toc_mask (W,maxc): contacts whose body pair had no contact
 *      before (world.py:273-274); toc_flag (W) updated in place; *_n: worlds that did not accept get the previous set
 *      back; flags[4] (device int32) = [capacity overflow (bit 0: capK, bit 1: maxc), number of worlds still active, any time-of-contact, max contact
 *      count after the merge].
 */
int dsdf_attempt_commit(int W, int nb, int maxc, const unsigned char* active, const double* dt_try,
                        const double* t, const double* end_t, double world_dt, int strict, int toc_enabled,
                        const int32_t* count_o, const int32_t* status_o, const int32_t* body_o,
                        const int32_t* face_o, const double* abc_o, const double* geo_o,
                        int32_t* count_n, int32_t* status_n, int32_t* body_n, int32_t* face_n, double* abc_n,
                        double* geo_n, unsigned char* toc_flag, unsigned char* accept, double* t_out,
                        double* dt_next, unsigned char* active_next, unsigned char* toc_now,
                        unsigned char* toc_mask, int32_t* flags, void* stream);

/* ---------------------------------------------------- time-of-contact ----
 * Replaces World.H.backward (lcp_physics/physics/world.py:141-237) together with the gather that feeds it
 * (world.py:275-327), for all worlds.  H.forward is the identity on dt, so there is no forward entry point.
 * In:  dt (W) the sub-step length that entered the attempt; toc_mask (W,maxc) uint8 = contacts whose body pair had
 *      no contact before; cbody (W,maxc,2); p (W,nb,7) / v (W,nb,6) the end-of-attempt poses and velocities;
 *      geo (W,maxc,10) contact tuples; f (W,nb,6) generalized forces; mass (W,nb); g_dt_h (W) = dL/d(dt after H).
 * Out: g_dt (W) = g_dt_h + the dependence of the reconstructed start-of-step frame on dt; gp (W,nb,7), gv (W,nb,6),
 *      ggeo (W,maxc,10), gf (W,nb,6), gmass (W,nb) = -(dD/dh)^+ dD/dtheta g_dt_h  (zero for worlds without new
 *      contacts).  base_tol = 1e-6 (lcp_physics/physics/utils.py:43).
 */
int dsdf_toc_backward(int W, int nb, int maxc, const double* dt, const unsigned char* toc_mask,
                      const int32_t* cbody, const double* p, const double* v, const double* geo,
                      const double* f, const double* mass, const double* g_dt_h, double base_tol,
                      double* g_dt, double* gp, double* gv, double* ggeo, double* gf, double* gmass, void* stream);

/* ------------------------------------------------- device-resident step ----
 * World.step / World.step_dt (lcp_physics/physics/world.py:119-139, 241-379) as a state machine that lives on the
 * device: the host launches ROUNDS (one attempt of every world still inside its step: prep -> solve -> move ->
 * find_contacts -> commit) in bursts and reads one small control block per burst; accept / reject / halve dt /
 * give up below dt/2^10 / remaining time / time-of-contact flags are decided per world by the commit kernel, which also
 * writes the TAPE of accepted sub-steps that the reverse sweep consumes.  See csrc/dsdf_steploop.cu.
 *
 * All fields are 8 bytes wide (no padding).  Arrays are device memory; (W..) = per real world, (V..) = per virtual world
 * (V = vcap rows; attempt d of the i-th active world is row d * n_active + i).
 */
#define DSDF_STEP_MAX_SLOTS 64
/* bits of ctrl[0] (abort word): what the host must do before launching further rounds */
#define DSDF_STEP_CAPK        1   /* a paused world overflowed the candidate list: enlarge capK          */
#define DSDF_STEP_MAXC        2   /* a paused world found more than maxc contacts: enlarge maxc           */
#define DSDF_STEP_DYN_SMEM    4   /* a world has more contacts than ncontacts_large: round voided          */
#define DSDF_STEP_TAPE        8   /* a paused world found its tape slot missing or full: add / enlarge slots (the host
                                     clamps the slot's row counter to its capacity before resuming)           */
#define DSDF_STEP_MAX_ROUNDS 16   /* max_rounds reached with worlds still active                           */
/* words of the control block (int32[16 + DSDF_STEP_MAX_SLOTS]) the host reads back; word 16 + k = rows used in tape slot k */
#define DSDF_CTRL_ABORT 0
#define DSDF_CTRL_NACTIVE 1
#define DSDF_CTRL_MAXCOUNT 3
#define DSDF_CTRL_ROUNDS 4
#define DSDF_CTRL_MAXNSUB 5
#define DSDF_CTRL_ANYTOC 8
#define DSDF_CTRL_LCPSTATUS 9
#define DSDF_CTRL_MAXCLEAN 13
#define DSDF_CTRL_CONSTATUS 14

typedef struct dsdf_step_slot {      /* tape of the k-th accepted sub-step of this step: one self-contained ROW per world  */
    int64_t cap;                     /* rows allocated.  Slot 0: row = world (cap = W); slot k > 0: rows are handed out  */
    int32_t* world;                  /* (cap) world of each row          in commit order, ctrl[16 + k] counts them      */
    double *p_in, *v_in;             /* (cap,nb,7), (cap,nb,6) state the sub-step started from                           */
    double *x, *new_v, *p_try;       /* (cap,6nb) LCP solution, (cap,nb,6) = -x, (cap,nb,7) pose after the move          */
    double *dt_raw, *dt_used;        /* (cap) sub-step length; value that entered solve / move (world.py:253-257)        */
    double* t_in;                    /* (cap) simulated time at the start of the sub-step (the reference's trajectory stamp) */
    double *lam, *s;                 /* (cap, maxc (2+fd)) multipliers / slacks, reference row order                     */
    unsigned char *toc_flag_in, *toc_now, *toc_mask;   /* (cap), (cap), (cap,maxc)                                        */
    int32_t *count_in, *body_in; double* geo_in;       /* contacts the solve used: (cap), (cap,maxc,2), (cap,maxc,10)     */
    int32_t *count, *body, *face;    /* contact set found at the END of the sub-step: (cap), (cap,maxc,2), (cap,maxc)    */
    double *abc, *geo;               /* (cap,maxc,3), (cap,maxc,10)                                                      */
} dsdf_step_slot;

typedef struct dsdf_step_args {
    int64_t W, nb, neq, maxc, fric_dirs, capK, npairs;
    int64_t depth;                   /* attempts (dt, dt/2, ..) evaluated at once when <= spec_threshold worlds are active */
    int64_t spec_threshold;
    int64_t depth2, spec_threshold2; /* a second, deeper level for the nearly empty rounds (depth2 >= depth, threshold2 <= threshold) */
    int64_t vcap, n_slots;
    int64_t slots_final;             /* 1: n_slots cannot grow any more -- a world that needs a further slot is STALLED: it
                                        leaves the step early (its time stays behind) and DSDF_CON_STALLED is reported */
    int64_t max_iter, max_rounds;
    int64_t strict, toc_enabled, fixed_dt, detach_b2;
    int64_t force_cta;               /* 1: every world on the one-CTA dynamics kernel; 0: dsdf_dynamics_solve chooses */
    double world_dt, eps, tol, fd_eps, body_eps;
    const dsdf_body_geom* geom; const int32_t* pairs; const int32_t* eq_rows;
    const double *mass, *Ibody, *fric, *rest, *f, *shape;              /* (W,nb..) constant during the step */
    double *p, *v, *t, *dt_try, *end_t, *last_dt;                      /* state, updated in place */
    unsigned char *active, *toc_flag, *had;
    int32_t* nsub; int64_t* attempts;
    int32_t *count, *status, *body, *face; double *abc, *geo;          /* current contact set, updated in place */
    int32_t *vmap, *vidx; double *dt_raw_v, *dt_used_v;                /* (V), (W), (V), (V) */
    double *x_v, *new_v_v, *nu_v, *lam_v, *s_v, *p_try_v; int32_t *lcp_status_v, *iters_v;
    int32_t *count_v, *status_v, *body_v, *face_v; double *abc_v, *geo_v;
    double* dyn_ws;                                                    /* workspace of the one-CTA dynamics kernel (V worlds) */
    int32_t* ctrl;                                                     /* int32[16 + DSDF_STEP_MAX_SLOTS] */
    const dsdf_step_slot* slots;                                       /* DEVICE array of n_slots tape slots */
} dsdf_step_args;

/* Start a step: every world active with dt_try = world_dt, end_t = t + world_dt, control block reset. */
int dsdf_step_begin(const dsdf_step_args* a, void* stream);
/* Clear the abort word after the host enlarged a buffer (a may carry new pointers / sizes from here on). */
int dsdf_step_resume(const dsdf_step_args* a, void* stream);
/* Launch n_rounds rounds (4 kernels + the 1-3 of dsdf_dynamics_solve each) without any host synchronisation.
 * ncontacts_small / ncontacts_large: the contact-count classes of dsdf_dynamics_solve (large <= small: one class).
 * a is a HOST pointer; it is passed to the kernels by value. */
int dsdf_step_rounds(const dsdf_step_args* a, int n_rounds, int ncontacts_small, int ncontacts_large, void* stream);
/* Diagnostics: per-kernel device time of the rounds.  dsdf_step_profile(1) makes dsdf_step_rounds bracket every launch
 * with CUDA events on its stream; dsdf_step_profile_read synchronises, writes the summed milliseconds and launch counts
 * of the five phases [prep, dynamics, move, contacts, commit] (host arrays of 5) and clears the events. */
int dsdf_step_profile(int enable);
int dsdf_step_profile_read(double* ms_out, int32_t* launches_out);

/* Measured FMA peaks of this device (dependent-chain microbenchmark, 8 chains per thread): the roofline denominators
 * for the FP64-bound stepping kernels.  scratch: >= 2.5 MB of device memory.  Outputs are host pointers (TFLOP/s). */
int dsdf_fma_peaks(int iters, void* scratch, double* fp64_tflops, double* fp32_tflops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DSDF_B200_H */
