// Device-resident World.step: the per-world state machine of lcp_physics/physics/world.py:119-139, 241-379
// (solve -> move -> find_contacts -> accept | halve dt and retry | give up below dt / 2^10 | take the remaining time |
// time-of-contact bookkeeping) runs ON THE DEVICE, round after round, with no host decision in between.
//
// One ROUND = one attempt of every world that is still inside its step = these launches on one stream:
//   step_prep_kernel      compacts the active worlds into "virtual worlds" (attempt d of world i uses dt / 2^d: a
//                         rejected sub-step is retried from the SAME start state with half the step, world.py:344-356,
//                         so when few worlds are left the halved retries are evaluated speculatively in one round)
//   dyn_forward_kernel    (dsdf_dynsolve.cu, loop mode)   PdipmEngine.solve_dynamics         engines.py:31-83
//                         one to three launches, one per contact-count class (dsdf_dynamics_plan)
//   step_integrate_kernel                                 Body3D.move                       bodies.py:488-496
//   contacts_kernel       (dsdf_contacts.cu, loop mode)   World.find_contacts                world.py:396-399
//   step_commit_kernel    accept / reject bookkeeping, first accepted attempt in the reference's order wins; an accepted
//                         sub-step is written to the TAPE (what the hand-written reverse sweep needs) and committed to
//                         the in-place state; its last CTA publishes the number of worlds still active.
// The host launches rounds in bursts (dsdf_step_rounds) without looking at the results: every kernel returns at once
// when no world is active or when a kernel asked for help (CT_ABORT), so surplus rounds cost a few empty launches.
// ONE small device-to-host copy of the control block per burst tells the host whether the step is complete.
//
// Capacity problems never void work that is already committed: a world whose attempt cannot be committed (candidate
// list / contact list / tape full) is PAUSED -- left untouched and active -- and retried after the host enlarged the
// buffers; worlds are independent, so the others simply go on.  Only "dynamics shared memory too small" voids a round
// (it is detected by the first kernel of the round, before anything changed).
#include "dsdf_math.cuh"
#include "dsdf_integrate.cuh"
#include "dsdf_steploop.cuh"
#include "../../include/dsdf_b200.h"
#include <vector>

namespace dsdf {

typedef dsdf_step_args Args;

// Optional per-kernel device timing of the rounds (dsdf_step_profile): CUDA events on the launching stream around every
// launch of a round, summed per phase when read.  Off by default; the timed benchmark pass runs without it.
enum { PHASE_PREP = 0, PHASE_DYN, PHASE_MOVE, PHASE_CONTACTS, PHASE_COMMIT, PHASE_COUNT };
static bool g_profile = false;
static std::vector<cudaEvent_t> g_events[PHASE_COUNT];      // start, end, start, end, ...
struct PhaseTimer {
    int phase; cudaStream_t st;
    PhaseTimer(int ph, cudaStream_t s) : phase(ph), st(s) { mark(); }
    ~PhaseTimer() { mark(); }
    void mark() {
        if (!g_profile) return;
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        cudaEventRecord(e, st);
        g_events[phase].push_back(e);
    }
};

__global__ void __launch_bounds__(256)
step_begin_kernel(const __grid_constant__ Args a) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0) {
        int* c = a.ctrl;
        c[CT_ABORT] = 0; c[CT_NACT] = (int)a.W; c[CT_CURSOR] = 0; c[CT_ROUNDS] = 0; c[CT_MAXNSUB] = 0; c[CT_DEFF] = 1;
        c[CT_NNEXT] = 0; c[CT_ANYTOC] = 0; c[CT_LCPSTAT] = 0; c[CT_NVIRT] = 0; c[CT_PENDING] = 0; c[CT_TICKET] = 0;
        c[CT_CONSTAT] = 0;
        for (int k = 0; k < DSDF_STEP_MAX_SLOTS; ++k) c[CT_SLOTROWS + k] = 0;
        c[CT_SLOTROWS] = (int)a.W;
    }
    if (w >= a.W) return;
    a.active[w] = 1;
    a.had[w] = 0;
    a.nsub[w] = 0;
    a.dt_try[w] = a.world_dt;
    if (a.fixed_dt) a.end_t[w] = a.t[w] + a.world_dt;                     // world.py:122
}

__global__ void __launch_bounds__(256)
step_prep_kernel(const __grid_constant__ Args a) {
    const int* c = a.ctrl;
    if (loop_idle(c)) return;
    const int n = c[CT_NACT];
    int deff = (a.depth > 1 && n <= a.spec_threshold) ? (int)a.depth : 1;
    if (a.depth2 > deff && n <= a.spec_threshold2) deff = (int)a.depth2;
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0) { a.ctrl[CT_DEFF] = deff; a.ctrl[CT_NVIRT] = n * deff; }
    if (w >= a.W || !a.active[w]) return;
    const int i = atomicAdd(&a.ctrl[CT_CURSOR], 1);
    a.vidx[w] = i;
    const double dt0 = a.dt_try[w];
    const bool carry = a.toc_enabled && a.toc_flag[w];
    const double last = a.last_dt[w];
    double scale = 1.0;
    for (int d = 0; d < deff; ++d, scale *= 0.5) {
        const int vv = d * n + i;
        const double dr = dt0 * scale;                                     // exact: powers of two
        a.vmap[vv] = w;
        a.dt_raw_v[vv] = dr;
        // world.py:253-257: dt_ = -last_dt + (last_dt.detach() + dt): the value the solve and the move see
        a.dt_used_v[vv] = carry ? (-last) + (last + dr) : dr;
    }
}

__global__ void __launch_bounds__(128)
step_integrate_kernel(const __grid_constant__ Args a) {
    const int* c = a.ctrl;
    if (loop_idle(c)) return;
    const int nb = (int)a.nb;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c[CT_NVIRT] * nb) return;
    const int vv = i / nb, b = i % nb;
    const int ws = a.vmap[vv];
    double pi[7], vi[6], o[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) pi[k] = a.p[((size_t)ws * nb + b) * 7 + k];
#pragma unroll
    for (int k = 0; k < 6; ++k) vi[k] = a.new_v_v[((size_t)vv * nb + b) * 6 + k];
    integrate_one<double>(pi, vi, a.dt_used_v[vv], o);
#pragma unroll
    for (int k = 0; k < 7; ++k) a.p_try_v[((size_t)vv * nb + b) * 7 + k] = o[k];
}

// One warp per real world.
__global__ void __launch_bounds__(128)
step_commit_kernel(const __grid_constant__ Args a) {
    int* c = a.ctrl;
    if (loop_idle(c)) return;                                  // uniform over the grid: written by earlier launches only
    const int n = c[CT_NACT], deff = c[CT_DEFF];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w = blockIdx.x * (blockDim.x >> 5) + warp;
    const int nb = (int)a.nb, maxc = (int)a.maxc, per = 2 + (int)a.fric_dirs, nz = 6 * nb, niCap = maxc * per;
    if (w < a.W && a.active[w]) {
        const int i = a.vidx[w];
        int win = -1, pause = 0;
        for (int d = 0; d < deff; ++d) {
            const int vv = d * n + i;
            const int st = a.status_v[vv];
            const bool acc = attempt_accepted(!(st & DSDF_CON_PENETRATION), a.strict, a.dt_raw_v[vv], a.world_dt);
            if (st & DSDF_CON_CAND_OVERFLOW) pause |= DSDF_STEP_CAPK;
            if (acc && (st & DSDF_CON_OVERFLOW)) pause |= DSDF_STEP_MAXC;
            if (acc && win < 0) win = d;
        }
        const int k = a.nsub[w];
        // tape row of this sub-step: slot 0 is indexed by world, later slots hand out rows in commit order
        int row = w;
        if (!pause && win >= 0 && k >= a.n_slots && a.slots_final) {
            // no tape left for this world (it keeps giving up at dt / 2^10 and would need hundreds of sub-steps): it leaves
            // the step here, with its time behind the others, and is reported
            if (lane == 0) { a.active[w] = 0; atomicOr(&c[CT_CONSTAT], DSDF_CON_STALLED); }
            win = -2;
        }
        if (!pause && win >= 0) {
            if (k >= a.n_slots) pause |= DSDF_STEP_TAPE;
            else if (k > 0) {
                if (lane == 0) row = atomicAdd(&c[CT_SLOTROWS + k], 1);
                row = __shfl_sync(0xffffffffu, row, 0);
                if (row >= a.slots[k].cap) pause |= DSDF_STEP_TAPE;      // the host clamps the counter before resuming
            }
        }
        if (pause) {
            if (lane == 0) { atomicOr(&c[CT_PENDING], pause); atomicAdd(&c[CT_NNEXT], 1); }
        } else if (win == -2) {                                 // stalled (above)
        } else if (win < 0) {                                   // every attempt of this round rejected: go on halving
            if (lane == 0) {
                double dn = a.dt_try[w];
                for (int d = 0; d < deff; ++d) dn = dn / 2;                                    // world.py:348
                a.dt_try[w] = dn;
                a.attempts[w] += deff;
                atomicAdd(&c[CT_NNEXT], 1);
            }
        } else {
            const int vv = win * n + i;
            const dsdf_step_slot& S = a.slots[k];
            const size_t r = (size_t)row;
            const int st = a.status_v[vv];
            const bool clean = !(st & DSDF_CON_PENETRATION);
            const int cn = min(a.count_v[vv], maxc), co = min(a.count[w], maxc);
            // time-of-contact set (world.py:273-274): contacts whose body pair had no contact at the start of the sub-step
            int any_toc = 0;
            for (int kk = lane; kk < maxc; kk += 32) {
                const unsigned char m = a.toc_enabled && clean && kk < cn &&
                                        new_body_pair(a.body_v + ((size_t)vv * maxc + kk) * 2, a.body + (size_t)w * maxc * 2,
                                                      co, nb);
                S.toc_mask[r * maxc + kk] = m;
                any_toc |= m;
            }
            any_toc = __any_sync(0xffffffffu, any_toc);
            // the contacts the solve used (the current set, about to be replaced)
            for (int e = lane; e < co * 2; e += 32) S.body_in[r * maxc * 2 + e] = a.body[(size_t)w * maxc * 2 + e];
            for (int e = lane; e < co * 10; e += 32) S.geo_in[r * maxc * 10 + e] = a.geo[(size_t)w * maxc * 10 + e];
            __syncwarp();
            // tape + state
            for (int e = lane; e < nb * 7; e += 32) {
                const size_t o = (size_t)w * nb * 7 + e;
                const double pt = a.p_try_v[(size_t)vv * nb * 7 + e];
                S.p_in[r * nb * 7 + e] = a.p[o];
                S.p_try[r * nb * 7 + e] = pt;
                a.p[o] = pt;          // H.forward is the identity on dt (world.py:147), so the redone move gives p_try again
            }
            for (int e = lane; e < nz; e += 32) {
                const size_t o = (size_t)w * nz + e;
                const double nv = a.new_v_v[(size_t)vv * nz + e];
                S.v_in[r * nz + e] = a.v[o];
                S.x[r * nz + e] = a.x_v[(size_t)vv * nz + e];
                S.new_v[r * nz + e] = nv;
                a.v[o] = nv;
            }
            for (int e = lane; e < co * per; e += 32) {          // multipliers of the contacts the solve used
                S.lam[r * niCap + e] = a.lam_v[(size_t)vv * niCap + e];
                S.s[r * niCap + e] = a.s_v[(size_t)vv * niCap + e];
            }
            // the contact set found at the end of this sub-step: tape row and current set
            for (int e = lane; e < cn * 2; e += 32) {
                const int bv = a.body_v[(size_t)vv * maxc * 2 + e];
                S.body[r * maxc * 2 + e] = bv; a.body[(size_t)w * maxc * 2 + e] = bv;
            }
            for (int e = lane; e < cn; e += 32) {
                const int fv = a.face_v[(size_t)vv * maxc + e];
                S.face[r * maxc + e] = fv; a.face[(size_t)w * maxc + e] = fv;
            }
            for (int e = lane; e < cn * 3; e += 32) {
                const double av = a.abc_v[(size_t)vv * maxc * 3 + e];
                S.abc[r * maxc * 3 + e] = av; a.abc[(size_t)w * maxc * 3 + e] = av;
            }
            for (int e = lane; e < cn * 10; e += 32) {
                const double gv = a.geo_v[(size_t)vv * maxc * 10 + e];
                S.geo[r * maxc * 10 + e] = gv; a.geo[(size_t)w * maxc * 10 + e] = gv;
            }
            if (lane == 0) {
                const double dtr = a.dt_raw_v[vv], dtu = a.dt_used_v[vv];
                S.world[r] = w;
                S.count_in[r] = a.count[w];
                S.count[r] = a.count_v[vv]; a.count[w] = a.count_v[vv]; a.status[w] = st;
                S.dt_raw[r] = dtr; S.dt_used[r] = dtu;
                S.t_in[r] = a.t[w];                                                   // world.py:378 stamps the start
                S.toc_flag_in[r] = a.toc_flag[w];
                S.toc_now[r] = (unsigned char)any_toc;
                if (a.toc_enabled && clean) a.toc_flag[w] = (unsigned char)any_toc;   // a give-up accept leaves the flag untouched
                if (any_toc) { a.last_dt[w] = dtu; c[CT_ANYTOC] = 1; }               // world.py:341 (value of H(dt_) = dt_)
                const double tn = a.t[w] + dtr;
                a.t[w] = tn;
                a.nsub[w] = k + 1;
                a.attempts[w] += win + 1;
                if (cn > 0) a.had[w] = 1;
                bool more = false;
                if (a.fixed_dt) more = tn < a.end_t[w];                             // world.py:128-132
                if (more) { a.dt_try[w] = a.end_t[w] - tn; atomicAdd(&c[CT_NNEXT], 1); }
                else a.active[w] = 0;
                atomicMax(&c[CT_MAXNSUB], k + 1);
                atomicMax(&c[CT_MAXCOUNT], cn);
                if (clean) atomicMax(&c[CT_MAXCLEAN], cn);
                const int ls = a.lcp_status_v[vv];
                if (ls) atomicOr(&c[CT_LCPSTAT], ls);
                if (st & DSDF_CON_HULL3D) atomicOr(&c[CT_CONSTAT], DSDF_CON_HULL3D);
            }
        }
    }
    // last CTA done: publish the round
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&c[CT_TICKET], 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        const int nn = atomicExch(&c[CT_NNEXT], 0);
        const int pend = atomicExch(&c[CT_PENDING], 0);
        const int rounds = c[CT_ROUNDS] + 1;
        c[CT_ROUNDS] = rounds;
        c[CT_CURSOR] = 0;
        c[CT_TICKET] = 0;
        int ab = pend;
        if (nn > 0 && rounds >= a.max_rounds) ab |= DSDF_STEP_MAX_ROUNDS;
        c[CT_NACT] = nn;
        if (ab) c[CT_ABORT] = ab;
        __threadfence();
    }
}

}  // namespace dsdf

using namespace dsdf;

extern "C" {

static int step_check(const dsdf_step_args* a) {
    if (!a || a->W <= 0 || a->nb <= 0 || a->maxc <= 0 || a->vcap < a->W || a->depth < 1 || a->depth > 16 || !a->ctrl) return -1;
    if (a->n_slots < 1 || a->n_slots > DSDF_STEP_MAX_SLOTS) return -1;
    if (a->depth * a->spec_threshold > a->vcap || a->depth2 > 16 || a->depth2 * a->spec_threshold2 > a->vcap) return -1;
    return 0;
}

int dsdf_step_begin(const dsdf_step_args* a, void* stream) {
    if (step_check(a)) return -1;
    step_begin_kernel<<<(unsigned)((a->W + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*a);
    return (int)cudaGetLastError();
}

__global__ void step_resume_kernel(int* c) {
    c[CT_ABORT] = 0; c[CT_CURSOR] = 0; c[CT_PENDING] = 0; c[CT_TICKET] = 0; c[CT_NNEXT] = 0;
}

int dsdf_step_resume(const dsdf_step_args* a, void* stream) {
    if (step_check(a)) return -1;
    step_resume_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(a->ctrl);
    return (int)cudaGetLastError();
}

int dsdf_step_rounds(const dsdf_step_args* a, int n_rounds, int ncontacts_small, int ncontacts_large, void* stream) {
    if (step_check(a) || n_rounds < 0 || ncontacts_small <= 0) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    const int W = (int)a->W, nb = (int)a->nb, V = (int)a->vcap;
    for (int r = 0; r < n_rounds; ++r) {
        { PhaseTimer t(PHASE_PREP, st); step_prep_kernel<<<(W + 255) / 256, 256, 0, st>>>(*a); }
        PhaseTimer* td = new PhaseTimer(PHASE_DYN, st);
        // dsdf_dynamics_solve picks the contact-count classes of the round and the kernel of each (dsdf_dynsolve.cu)
        int rc = dsdf_dynamics_solve(a->p, a->v, a->mass, a->Ibody, a->fric, a->rest, a->f, a->dt_used_v, nullptr, a->count,
                                     a->body, a->geo, a->eq_rows, V, nb, (int)a->neq, (int)a->maxc, ncontacts_small,
                                     ncontacts_large, (int)a->force_cta, (int)a->fric_dirs, 1e-12, 3, (int)a->max_iter,
                                     a->x_v, a->new_v_v, a->nu_v, a->lam_v, a->s_v, a->lcp_status_v, a->iters_v, a->vmap,
                                     a->ctrl, a->dyn_ws, stream);
        delete td;
        if (rc) return rc;
        { PhaseTimer t(PHASE_MOVE, st); step_integrate_kernel<<<(V * nb + 127) / 128, 128, 0, st>>>(*a); }
        PhaseTimer* tc = new PhaseTimer(PHASE_CONTACTS, st);
        rc = dsdf_contacts_detect(a->geom, a->pairs, (int)a->npairs, a->p_try_v, a->shape, nullptr, V, nb, a->eps, a->tol,
                                  a->fd_eps, a->body_eps, (int)a->detach_b2, (int)a->capK, (int)a->maxc, a->count_v,
                                  a->body_v, a->face_v, a->abc_v, a->geo_v, a->status_v, nullptr, nullptr, a->vmap,
                                  a->ctrl, stream);
        delete tc;
        if (rc) return rc;
        { PhaseTimer t(PHASE_COMMIT, st); step_commit_kernel<<<(W + 3) / 4, 128, 0, st>>>(*a); }
    }
    return (int)cudaGetLastError();
}

int dsdf_step_profile(int enable) {
    g_profile = enable != 0;
    return 0;
}

int dsdf_step_profile_read(double* ms_out, int32_t* launches_out) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return (int)e;
    for (int ph = 0; ph < PHASE_COUNT; ++ph) {
        double tot = 0.0;
        std::vector<cudaEvent_t>& v = g_events[ph];
        for (size_t i = 0; i + 1 < v.size(); i += 2) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, v[i], v[i + 1]) == cudaSuccess) tot += ms;
        }
        if (ms_out) ms_out[ph] = tot;
        if (launches_out) launches_out[ph] = (int32_t)(v.size() / 2);
        for (cudaEvent_t ev : v) cudaEventDestroy(ev);
        v.clear();
    }
    return 0;
}

}  // extern "C"
