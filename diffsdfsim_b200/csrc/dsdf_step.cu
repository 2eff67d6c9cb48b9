// Per-world bookkeeping of one step attempt: accept / reject / halve dt / remaining time / time-of-contact flags,
// and the merge of the freshly detected contact set with the previous one for worlds that did not accept.
//
// Replaces the control flow around the three physics calls in World.step_dt (lcp_physics/physics/world.py:241-356):
//   :270      accept iff every penetration <= tol            -> status bit DSDF_CON_PENETRATION of the detection
//   :344-348  reject: restore state, dt /= 2 ; not strict: give up (accept) once dt < world.dt / 2^10
//   :128-132  fixed_dt: after an accepted short sub-step take the remaining time next
//   :273-274  "new" contacts = body pairs without a contact at the start of the sub-step (time-of-contact set)
// One thread per world; everything a host loop needs afterwards comes back in four int32 flags (one D2H copy).
#include <cuda_runtime.h>
#include <stdint.h>
#include "dsdf_steploop.cuh"
#include "../../include/dsdf_b200.h"

namespace dsdf {

__global__ void __launch_bounds__(128)
attempt_commit_kernel(int W, int nb, int maxc, const unsigned char* __restrict__ active,
                      const double* __restrict__ dt_try, const double* __restrict__ t, const double* __restrict__ end_t,
                      double world_dt, int strict, int toc_enabled,
                      const int* __restrict__ count_o, const int* __restrict__ status_o, const int* __restrict__ body_o,
                      const int* __restrict__ face_o, const double* __restrict__ abc_o, const double* __restrict__ geo_o,
                      int* __restrict__ count_n, int* __restrict__ status_n, int* __restrict__ body_n,
                      int* __restrict__ face_n, double* __restrict__ abc_n, double* __restrict__ geo_n,
                      unsigned char* __restrict__ toc_flag, unsigned char* __restrict__ accept_o,
                      double* __restrict__ t_out, double* __restrict__ dt_next, unsigned char* __restrict__ active_next,
                      unsigned char* __restrict__ toc_now_o, unsigned char* __restrict__ toc_mask,
                      int* __restrict__ flags) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    const bool act = active[w] != 0;
    const int st = status_n[w];
    const bool clean = act && !(st & DSDF_CON_PENETRATION);
    const double dtw = dt_try[w];
    const bool accept = act && attempt_accepted(clean, strict, dtw, world_dt);
    int bad = 0;                                   // bit 0: candidate list overflow (capK), bit 1: contact overflow (maxc)
    if (act && (st & DSDF_CON_CAND_OVERFLOW)) bad |= 1;
    if (accept && (st & DSDF_CON_OVERFLOW)) bad |= 2;
    const double tn = accept ? t[w] + dtw : t[w];
    double dn = (act && !accept) ? dtw / 2 : dtw;                                     // world.py:348
    bool nact = act && !accept;
    if (end_t) {
        const bool more = accept && (tn < end_t[w]);                                  // world.py:128-132
        if (more) dn = end_t[w] - tn;
        nact = nact || more;
    }
    // time-of-contact set (world.py:273-274): pairs of the new set that the old set does not have
    int any_toc = 0;
    const int cn = min(count_n[w], maxc), co = min(count_o[w], maxc);
    if (toc_enabled) {
        for (int k = 0; k < maxc; ++k) {
            const unsigned char m = clean && k < cn &&
                                    new_body_pair(body_n + ((size_t)w * maxc + k) * 2, body_o + (size_t)w * maxc * 2, co, nb);
            toc_mask[(size_t)w * maxc + k] = m;
            any_toc |= m;
        }
        toc_now_o[w] = (unsigned char)any_toc;
        if (clean) toc_flag[w] = (unsigned char)any_toc;      // a give-up accept leaves the flag untouched
    }
    // worlds that did not accept keep their previous contact set
    if (!accept) {
        count_n[w] = count_o[w];
        status_n[w] = status_o[w];
        for (int k = 0; k < co; ++k) {
            const size_t o = (size_t)w * maxc + k;
            body_n[2 * o] = body_o[2 * o]; body_n[2 * o + 1] = body_o[2 * o + 1];
            face_n[o] = face_o[o];
            for (int c = 0; c < 3; ++c) abc_n[3 * o + c] = abc_o[3 * o + c];
            for (int c = 0; c < 10; ++c) geo_n[10 * o + c] = geo_o[10 * o + c];
        }
    }
    accept_o[w] = accept;
    t_out[w] = tn;
    dt_next[w] = dn;
    active_next[w] = nact;
    const int cnt_after = accept ? cn : co;
    if (bad) atomicOr(&flags[0], bad);
    if (nact) atomicAdd(&flags[1], 1);             // number of worlds still active
    if (any_toc) atomicOr(&flags[2], 1);
    atomicMax(&flags[3], cnt_after);
}

}  // namespace dsdf

extern "C" int dsdf_attempt_commit(int W, int nb, int maxc, const unsigned char* active, const double* dt_try,
                                   const double* t, const double* end_t, double world_dt, int strict, int toc_enabled,
                                   const int32_t* count_o, const int32_t* status_o, const int32_t* body_o,
                                   const int32_t* face_o, const double* abc_o, const double* geo_o,
                                   int32_t* count_n, int32_t* status_n, int32_t* body_n, int32_t* face_n, double* abc_n,
                                   double* geo_n, unsigned char* toc_flag, unsigned char* accept, double* t_out,
                                   double* dt_next, unsigned char* active_next, unsigned char* toc_now,
                                   unsigned char* toc_mask, int32_t* flags, void* stream) {
    if (W <= 0 || nb <= 0 || maxc <= 0 || !active || !flags) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(flags, 0, 4 * sizeof(int32_t), st);
    if (e != cudaSuccess) return (int)e;
    dsdf::attempt_commit_kernel<<<(W + 127) / 128, 128, 0, st>>>(
        W, nb, maxc, active, dt_try, t, end_t, world_dt, strict, toc_enabled, count_o, status_o, body_o, face_o, abc_o,
        geo_o, count_n, status_n, body_n, face_n, abc_n, geo_n, toc_flag, accept, t_out, dt_next, active_next, toc_now,
        toc_mask, flags);
    return (int)cudaGetLastError();
}
