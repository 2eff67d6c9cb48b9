// Device-resident step loop: control block shared by the kernels of one round (dsdf_steploop.cu) and the
// loop-mode variants of the dynamics / contact kernels.  See dsdf_steploop.cu for the protocol.
#pragma once
namespace dsdf {
// int32 control words (device memory, one block per world batch)
enum {
    CT_ABORT = 0,     // != 0: every kernel of the following rounds returns at once; bits DSDF_STEP_*
    CT_NACT,          // worlds still inside their step (set by the last CTA of the commit kernel)
    CT_CURSOR,        // compaction cursor of the prep kernel
    CT_MAXCOUNT,      // running max of the accepted contact counts
    CT_ROUNDS,        // rounds executed in this step
    CT_MAXNSUB,       // max accepted sub-steps of one world in this step
    CT_DEFF,          // attempts (dt, dt/2, ...) evaluated per world in the current round
    CT_NNEXT,         // accumulator of CT_NACT for the next round
    CT_ANYTOC,        // some accepted sub-step of this step had a new (time-of-contact) contact
    CT_LCPSTAT,       // OR of the LCP status words of the accepted solves
    CT_NVIRT,         // virtual worlds of the current round = CT_NACT * CT_DEFF
    CT_PENDING,       // pause bits collected by the commit kernel, promoted to CT_ABORT by its last CTA
    CT_TICKET,        // "last CTA done" ticket of the commit kernel
    CT_MAXCLEAN,      // running max of the accepted contact counts of NON-penetrating states
    CT_CONSTAT,       // OR of the contact status words of the accepted sub-steps of this step (DSDF_CON_HULL3D ...)
    CT_SLOTROWS = 16, // + k: rows handed out in tape slot k (k >= 1; slot 0 is indexed by world)
    CT_WORDS = 16 + 64
};
// true when this launch has nothing to do (a previous kernel asked the host for help, or every world is done)
__device__ __forceinline__ bool loop_idle(const int* ctrl) { return ctrl[CT_ABORT] != 0 || ctrl[CT_NACT] == 0; }

// The two rules of the reference that both commit kernels (step_commit_kernel here, attempt_commit_kernel of the
// host-driven loop in dsdf_step.cu) apply to an attempt.
//
// world.py:345-347: a sub-step is accepted when its state does not penetrate (clean), or, when not strict, once its dt
// fell below world_dt / 2^10 (give up halving).
__device__ __forceinline__ bool attempt_accepted(bool clean, bool strict, double dt, double world_dt) {
    return clean || (!strict && dt < world_dt / 1024.0);
}
// world.py:273-274: the contact with body pair `pair` (2 ints) is new when none of the n_old contacts of the set at
// the start of the sub-step (old_pairs, 2 ints each) joins the same two bodies.
__device__ __forceinline__ bool new_body_pair(const int* pair, const int* old_pairs, int n_old, int nb) {
    const int pid = min(pair[0], pair[1]) * nb + max(pair[0], pair[1]);
    bool seen = false;
    for (int j = 0; j < n_old; ++j) {
        const int a = old_pairs[2 * j], b = old_pairs[2 * j + 1];
        seen = seen || (min(a, b) * nb + max(a, b) == pid);
    }
    return !seen;
}
}  // namespace dsdf
