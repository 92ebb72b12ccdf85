// Kernels, iteration control and the C ABI of the batched HS-DDP solver (sm_100a).
//
//   MultiPhaseDDP::solve            HSDDPSolver/source/MultiPhaseDDP.cpp:232-428  -> solve_block / k_solve
//   MultiPhaseDDP::line_search      :98-138                                       -> line_search_block
//   step-level public methods       HSDDPSolver/header/MultiPhaseDDP.h:42-69      -> k_step<OP>
// One thread block per problem; k_solve is persistent (blocks pull problem indices
// from a device-side queue so problems with few iterations retire early).
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <map>
#include <algorithm>
#include "hsddp_device.cuh"
#include "hsddp_sweep.cuh"
#include "hsddp_sweep_w1.cuh"
#include "hsddp_lr_w1.cuh"

// resident blocks per SM the kernels are compiled for (register budget = 65536 / (128 * HSDDP_MIN_BLOCKS))
#ifndef HSDDP_MIN_BLOCKS
#define HSDDP_MIN_BLOCKS 6
#endif

namespace hsddp {

// ---------------------------------------------------------------------------
// iteration control
// ---------------------------------------------------------------------------
__device__ inline void prepare_merit_block(Smem& sm) {  // MultiPhaseDDP.cpp:331-337 (Q5)
    if (threadIdx.x == 0) {
        SolverState& st = sm.st;
        const double dV_abs = fabs(st.dV_1 + 0.5 * st.dV_2);
        st.merit_rho = (st.feas > sm.opt.dynamics_feas_thresh) ? dV_abs / ((1 - sm.opt.merit_scale) * st.feas) + sm.opt.merit_offset : 0;
        st.merit = st.actual_cost + st.merit_rho * st.feas;
    }
    __syncthreads();
}

// MultiPhaseDDP::line_search.  Returns success; eps_out = accepted step (0 if none).
template <bool LINEARISED>
__device__ inline bool line_search_block(Smem& sm, double& eps_out, int& n_trials) {
    double eps = 1;
    const double merit_prev = sm.st.merit;
    const double feas_prev = sm.st.feas;
    const double merit_rho = sm.st.merit_rho;
    const double dV_1 = sm.st.dV_1, dV_2 = sm.st.dV_2;
    bool success = false;
    n_trials = 0;
    __syncthreads();
    while (eps > 1e-3) {  // 1, .1, .010000000000000002, .0010000000000000002 (Q6)
        const bool rollout_success = hybrid_rollout_block<LINEARISED>(sm, eps);
        compute_cost_block(sm);
        if (threadIdx.x == 0) { sm.ctl.trial_cost = sm.st.actual_cost; sm.ctl.trial_feas = sm.st.feas; sm.ctl.have_trial = 1; }
        const double merit = sm.st.actual_cost + merit_rho * sm.st.feas;
        ++n_trials;
        const double exp_cost_change = eps * dV_1 + 0.5 * eps * eps * dV_2;
        const double exp_merit_change = exp_cost_change - eps * merit_rho * feas_prev;
        __syncthreads();
        if (threadIdx.x == 0) sm.st.merit = merit;
        __syncthreads();
        if ((merit <= merit_prev + sm.opt.gamma * exp_merit_change) && rollout_success) { success = true; break; }
        eps *= sm.opt.alpha;
    }
    eps_out = success ? eps : 0.0;
    return success;
}

// ---------------------------------------------------------------------------
// Concurrent line search (north_star (3): "all line-search step sizes concurrently").  The latency kernel k_solve_lat4 gives
// every problem a CLUSTER of four blocks: block 0 runs the solve; at a line search the four blocks evaluate the reference's
// first four step sizes (1, alpha, alpha^2, alpha^3) at the same time, each into its own trial arrays, and block 0 then
// accepts the first one that passes IN THE REFERENCE'S ORDER and commits its arrays -- exactly the state the sequential
// search leaves (MultiPhaseDDP.cpp:98-138; Q2: if none passes, the state of the last trial).  A diverged rollout leaves a
// partially updated state that depends on the trial before it (Q16), so in that (rare) case the concurrent results are
// discarded and the sequential search runs instead.  For throughput the sequential search with early exit is the better
// schedule (1.63 trials per iteration on the benchmark workload); this one is for the latency of a single solve.
// ---------------------------------------------------------------------------
struct TrialPtrs { double *X, *U, *U_t, *Xsim_t, *Defect, *gcon, *hcon; };

// The trial arrays, results and mailbox of a cluster belong to its position in the launch, not to its problem: a solve of listed
// problems (hsddp_batch_solve_problems) in a batch of more than kClusterLsMax problems has them for kClusterLsMax positions only.
__device__ __forceinline__ int ls_pos() { return (int)blockIdx.x >> 2; }

__device__ inline TrialPtrs swap_trial_arrays(Smem& sm, const TrialPtrs& t) {
    TrialPtrs old = {sm.X, sm.U, sm.U_t, sm.Xsim_t, sm.Defect, sm.gcon, sm.hcon};
    __syncthreads();
    if (threadIdx.x == 0) { sm.X = t.X; sm.U = t.U; sm.U_t = t.U_t; sm.Xsim_t = t.Xsim_t; sm.Defect = t.Defect; sm.gcon = t.gcon; sm.hcon = t.hcon; }
    __syncthreads();
    return old;
}
__device__ inline TrialPtrs trial_arrays(const BatchPtrs& bp, int pos, int r) {
    const size_t q = (size_t)pos * 4 + r, sn = (size_t)bp.max_nodes * 24, ss = (size_t)bp.max_stages * 24;
    return TrialPtrs{bp.ls_X + q * sn, bp.ls_U + q * ss, bp.ls_Ut + q * ss, bp.ls_Xsim + q * sn, bp.ls_Defect + q * sn,
                     bp.ls_gcon + q * bp.max_stages * 20, bp.ls_hcon + q * MAXPH * 4};
}
// one trial into the trial arrays of step r; the block's own arrays are untouched
__device__ inline void run_trial(Smem& sm, const BatchPtrs& bp, int r, double eps) {
    const TrialPtrs keep = swap_trial_arrays(sm, trial_arrays(bp, ls_pos(), r));
    // (touchdown values of legs without a constraint are never written by a rollout: start from the current ones)
    for (int e = threadIdx.x; e < MAXPH * 4; e += kThreads) sm.hcon[e] = keep.hcon[e];
    for (int e = threadIdx.x; e < sm.sc.n_stages * 20; e += kThreads) sm.gcon[e] = keep.gcon[e];  // (likewise the rows of swing legs)
    __syncthreads();
    const bool ok = hybrid_rollout_block<true>(sm, eps);
    compute_cost_block(sm);
    if (threadIdx.x == 0) {
        double* res = bp.ls_res + ((size_t)ls_pos() * 4 + r) * 8;
        res[0] = sm.st.actual_cost; res[1] = sm.st.feas; res[2] = sm.st.max_pconstr; res[3] = sm.st.max_tconstr; res[4] = ok ? 1.0 : 0.0;
    }
    swap_trial_arrays(sm, keep);
}
__device__ inline void commit_trial(Smem& sm, const BatchPtrs& bp, int r) {
    const TrialPtrs t = trial_arrays(bp, ls_pos(), r);
    const DevSchedule& sc = sm.sc;
    for (int e = threadIdx.x; e < sc.n_nodes * 24; e += kThreads) { sm.X[e] = t.X[e]; sm.Defect[e] = t.Defect[e]; }
    for (int e = threadIdx.x; e < sc.n_stages * 24; e += kThreads) sm.U[e] = t.U[e];
    for (int e = threadIdx.x; e < sc.n_stages * 20; e += kThreads) sm.gcon[e] = t.gcon[e];
    for (int e = threadIdx.x; e < MAXPH * 4; e += kThreads) sm.hcon[e] = t.hcon[e];
    if (threadIdx.x == 0) {
        const double* res = bp.ls_res + ((size_t)ls_pos() * 4 + r) * 8;
        sm.st.actual_cost = res[0]; sm.st.feas = res[1]; sm.st.max_pconstr = res[2]; sm.st.max_tconstr = res[3]; sm.st.rollout_ok = 1;
        sm.ctl.trial_cost = res[0]; sm.ctl.trial_feas = res[1]; sm.ctl.have_trial = 1;
    }
    __syncthreads();
}

// block 0 of the cluster: the line search of one DDP iteration
__device__ inline bool line_search_cluster(Smem& sm, const BatchPtrs& bp, double& eps_out, int& n_trials) {
    namespace cg = cooperative_groups;
    const double merit_prev = sm.st.merit, feas_prev = sm.st.feas, merit_rho = sm.st.merit_rho;
    const double dV_1 = sm.st.dV_1, dV_2 = sm.st.dV_2;
    double epsv[4];
    int nv = 0;
    for (double e = 1; e > 1e-3 && nv < 4; e *= sm.opt.alpha) epsv[nv++] = e;  // 1, .1, .010000000000000002, .0010000000000000002 (Q6)
    __syncthreads();
    if (threadIdx.x == 0) { bp.ls_mail[ls_pos()] = 1; __threadfence(); }
    cg::this_cluster().sync();  // [A] the helpers start their trials
    if (nv > 0) run_trial(sm, bp, 0, epsv[0]);
    __threadfence();
    cg::this_cluster().sync();  // [B] every trial is in its arrays
    bool diverged = false;
    int accepted = -1;
    for (int r = 0; r < nv; ++r) {
        const double* res = bp.ls_res + ((size_t)ls_pos() * 4 + r) * 8;
        const double cost = __ldcg(res), feas = __ldcg(res + 1);
        const bool ok = __ldcg(res + 4) != 0.0;
        if (!ok) { diverged = true; break; }
        const double merit = cost + merit_rho * feas;
        const double exp_merit_change = (epsv[r] * dV_1 + 0.5 * epsv[r] * epsv[r] * dV_2) - epsv[r] * merit_rho * feas_prev;
        if (merit <= merit_prev + sm.opt.gamma * exp_merit_change) { accepted = r; break; }
    }
    if (diverged) return line_search_block<true>(sm, eps_out, n_trials);  // (nothing has been committed: the sequential search starts afresh)
    const int last = accepted >= 0 ? accepted : nv - 1;
    if (last >= 0) {
        commit_trial(sm, bp, last);
        if (threadIdx.x == 0) sm.st.merit = sm.st.actual_cost + merit_rho * sm.st.feas;
        __syncthreads();
    }
    n_trials = last + 1;
    if (accepted >= 0) { eps_out = epsv[accepted]; return true; }
    // more than four step sizes (alpha > 0.1...): the search goes on sequentially from the state of the fourth trial
    double eps = (nv > 0 ? epsv[nv - 1] : 1.0) * sm.opt.alpha;
    bool success = false;
    while (nv == 4 && eps > 1e-3) {
        const bool rollout_success = hybrid_rollout_block<true>(sm, eps);
        compute_cost_block(sm);
        if (threadIdx.x == 0) { sm.ctl.trial_cost = sm.st.actual_cost; sm.ctl.trial_feas = sm.st.feas; sm.ctl.have_trial = 1; }
        const double merit = sm.st.actual_cost + merit_rho * sm.st.feas;
        ++n_trials;
        const double exp_merit_change = (eps * dV_1 + 0.5 * eps * eps * dV_2) - eps * merit_rho * feas_prev;
        __syncthreads();
        if (threadIdx.x == 0) sm.st.merit = merit;
        __syncthreads();
        if ((merit <= merit_prev + sm.opt.gamma * exp_merit_change) && rollout_success) { success = true; break; }
        eps *= sm.opt.alpha;
    }
    eps_out = success ? eps : 0.0;
    return success;
}

// blocks 1..3 of the cluster
__device__ inline void line_search_helper_loop(Smem& sm, const BatchPtrs& bp, int r) {
    namespace cg = cooperative_groups;
    for (;;) {
        cg::this_cluster().sync();  // [A]
        const int op = *((volatile int*)(bp.ls_mail + ls_pos()));
        if (op != 1) break;
        double eps = 1;
        for (int q = 0; q < r; ++q) eps *= sm.opt.alpha;
        // the solver scalars and the state the trial starts from live in HBM and in block 0: Xbar, Ubar, dX, dU, K dX and the
        // ReB / AL parameters are read from HBM (written by block 0 before [A])
        if (eps > 1e-3) run_trial(sm, bp, r, eps);
        __threadfence();
        cg::this_cluster().sync();  // [B]
    }
}

// ---------------------------------------------------------------------------
// MultiPhaseDDP::solve (MultiPhaseDDP.cpp:232-428) as a resumable state machine.
//   solve_begin_block      :257-260 + the head of the first outer iteration (:282-302)
//   iter_prep_block        :306-319  compute_cost, LQ_approximation
//   iter_sweep_block       :320-324  backward_sweep_regularized
//   iter_forward_block     :326-409  linear rollout, merit, line search, termination tests, AL / ReB updates
// k_solve runs them back to back for one problem (persistent blocks, small batches / latency);
// k_phase runs ONE of them for every running problem (large batches: all co-resident blocks execute
// the same code, which keeps the instruction cache hot, see DESIGN.md §4).
// ---------------------------------------------------------------------------
__device__ inline void outer_start_block(Smem& sm) {  // :283-302
    __syncthreads();
    if (threadIdx.x == 0) {
        sm.ctl.iter_ou++;
        sm.ctl.iter_in = 0;
        sm.ctl.have_trial = 0;  // the AL / ReB parameters have changed: the next iteration evaluates the cost afresh
        sm.st.max_tconstr_prev = sm.st.max_tconstr; sm.st.max_pconstr_prev = sm.st.max_pconstr; sm.st.reg = 0;
    }
    __syncthreads();
}

// end of an outer iteration (:383-413).  Leaves ctl.active = 0 when the solve is over.
__device__ inline void outer_end_block(Smem& sm) {
    const hsddp_options& opt = sm.opt;
    for (;;) {
        if (opt.AL_active) update_al_block(sm);
        if (opt.ReB_active) update_reb_block(sm);
        __syncthreads();
        const SolverState& st = sm.st;
        int status = -1;
        if (st.max_tconstr < opt.tconstr_thresh && fabs(st.max_pconstr) < opt.pconstr_thresh && st.feas <= opt.dynamics_feas_thresh) status = HSDDP_STATUS_CONVERGED;
        else if (fabs(st.max_tconstr - st.max_tconstr_prev) < 0.0001 && fabs(st.max_pconstr - st.max_pconstr_prev) < 0.0001 && st.feas <= opt.dynamics_feas_thresh) status = HSDDP_STATUS_STALLED;
        else if (sm.ctl.iter_ou >= sm.ctl.max_al) status = HSDDP_STATUS_MAX_ITER;
        __syncthreads();
        if (status >= 0) {
            if (threadIdx.x == 0) { sm.ctl.status = status; sm.ctl.active = 0; }
            __syncthreads();
            return;
        }
        outer_start_block(sm);
        if (sm.ctl.max_ddp > 0) return;  // (an empty inner loop falls straight through to the next outer end)
    }
}

__device__ inline void solve_begin_block(Smem& sm, const BatchPtrs& bp) {
    const int tid = threadIdx.x;
    __syncthreads();
    if (tid == 0) {
        SolveCtl c = {};
        c.status = HSDDP_STATUS_MAX_ITER; c.active = 1;
        c.max_al = sm.opt.max_AL_iter; c.max_ddp = sm.opt.max_DDP_iter;
        if (bp.budget && bp.budget[2 * sm.pid] >= 0) { c.max_al = bp.budget[2 * sm.pid]; c.max_ddp = bp.budget[2 * sm.pid + 1]; }
        sm.ctl = c;
        sm.st.actual_cost = 0; sm.st.max_pconstr = 0; sm.st.max_pconstr_prev = 0; sm.st.max_tconstr = 0; sm.st.max_tconstr_prev = 0;
    }
    __syncthreads();
    hybrid_rollout_block<true>(sm, 0.0);  // (eps = 0: both forms give U = Ubar)
    update_nominal_block(sm);
    compute_cost_block(sm);
    if (tid == 0) { sm.ctl.cost0 = sm.st.actual_cost; sm.ctl.feas0 = sm.st.feas; }
    __syncthreads();
    if (sm.ctl.max_al <= 0) {
        if (tid == 0) sm.ctl.active = 0;
        __syncthreads();
        return;
    }
    outer_start_block(sm);
    if (sm.ctl.max_ddp <= 0) outer_end_block(sm);
}

__device__ inline void iter_prep_block(Smem& sm, const BatchPtrs& bp) {
    // compute_cost + measure_dynamics_feasibility at the top of the inner loop (:306-308).  After the first iteration
    // of an outer iteration the trajectories and parameters are exactly those of the last line-search trial (accepted or
    // not, Q2), whose cost and feasibility were just evaluated: reuse them instead of a second identical pass.
    if (sm.ctl.have_trial) {
        if (threadIdx.x == 0) { sm.st.actual_cost = sm.ctl.trial_cost; sm.st.feas = sm.ctl.trial_feas; }
        __syncthreads();
    } else {
        compute_cost_block(sm);
    }
    if (threadIdx.x == 0) {
        sm.ctl.iter_in++; sm.ctl.iter++;
        if (sm.ctl.iter <= HSDDP_TRACE_CAP) {
            hsddp_iter_record rec;
            rec.outer = sm.ctl.iter_ou; rec.inner = sm.ctl.iter_in; rec.cost_before = sm.st.actual_cost; rec.feas_before = sm.st.feas;
            rec.reg_after = rec.n_sweeps = 0;
            rec.dV_1 = rec.dV_2 = rec.merit_rho = rec.eps_accepted = rec.n_trials = 0; rec._pad = 0;
            rec.cost_after = rec.feas_after = rec.max_tconstr = rec.max_pconstr = 0;
            bp.trace[(size_t)sm.pid * HSDDP_TRACE_CAP + sm.ctl.iter - 1] = rec;
        }
    }
    __syncthreads();
    lq_approximation_block(sm);
}

__device__ inline void finish_sweep_block(Smem& sm, const BatchPtrs& bp, bool success, int nsw) {
    if (threadIdx.x == 0) {
        sm.ctl.n_sweeps += nsw;
        if (sm.ctl.iter <= HSDDP_TRACE_CAP) {
            hsddp_iter_record& rec = bp.trace[(size_t)sm.pid * HSDDP_TRACE_CAP + sm.ctl.iter - 1];
            rec.n_sweeps = nsw; rec.reg_after = sm.st.reg;
        }
        if (!success) { sm.ctl.status = HSDDP_STATUS_REG_OVERFLOW; sm.ctl.active = 0; }  // bad_solve (:321-324,421-427)
    }
    __syncthreads();
}

__device__ inline void iter_sweep_block(Smem& sm, const BatchPtrs& bp) {
    int nsw = 0;
    const bool success = backward_sweep_regularized_block(sm, nsw);
    finish_sweep_block(sm, bp, success, nsw);
}

// ---------------------------------------------------------------------------
// Regularisation retries side by side (phased driver, rounds of the four-warp sweep; DESIGN.md §4.3).
// backward_sweep_regularized tries r_0 = st.reg, r_1, ... (r_{j+1} = max(r_j update_regularization, 1e-3), until one is PD or
// r_j > 1e2) one after another, and every attempt reads the same inputs.  Candidate j of a listed problem runs attempt j on a
// block of its own; the last of the spec_S blocks to arrive leaves what the loop would have left: the first PD attempt, or the
// state after every candidate failed, from which it runs the rest of the loop itself.
// ---------------------------------------------------------------------------
// r := r_j of the retry sequence that starts at r; false: r_j is past the limit (the loop never runs attempt j)
__device__ __forceinline__ bool retry_reg(double& r, int j, double up) {
    for (int i = 0; i < j; ++i) {
        r = fmax(r * up, 1e-03);
        if (r > 1e2) return false;
    }
    return true;
}

// the prep of a round the four-warp sweep takes: list the problem if it regularises (its last sweep of this solve needed a
// retry, or it starts from reg > 0).  Scheduling only: an unlisted problem runs the loop on its own block.
__device__ inline void spec_flag_block(Smem& sm, const BatchPtrs& bp) {
    if (threadIdx.x == 0) {
        const int row = sm.ctl.iter - 1;  // this iteration's trace row; row - 1 is the last sweep's
        bool flag = sm.st.reg > 0;
        if (row >= 1 && row <= HSDDP_TRACE_CAP) flag = flag || bp.trace[(size_t)sm.pid * HSDDP_TRACE_CAP + row - 1].n_sweeps > 1;
        int e = -1;
        if (flag) {
            e = atomicAdd(bp.spec_count, 1);
            if (e < bp.spec_cap) bp.spec_list[e] = sm.pid;
            else e = -1;
        }
        bp.spec_entry[sm.pid] = e;
    }
}

// A candidate j > 0 marks the first dU word of every stage of its slice with this signalling-NaN pattern before it sweeps.  No
// arithmetic result has it, so a failed candidate's slice shows which stages the sweep wrote (the sweep runs from the last stage down).
constexpr unsigned long long kSpecUnwritten = 0x7ff0dead5eed0001ull;

// Candidate j of list entry e has run its attempt (ran: its regularisation is within the limit; ok: PD).  The last of the spec_S
// blocks to arrive takes over the state the sequential loop has after its last attempt among the candidates -- the first PD one,
// w, or the m that ran all failed -- and returns true with success, reg = that attempt's regularisation and nsw = the attempts
// so far.  The other blocks return false.
__device__ inline bool spec_commit_block(Smem& sm, const BatchPtrs& bp, int e, int j, bool ran, bool ok, double& reg, int& nsw, bool& success) {
    const int tid = threadIdx.x, S = bp.spec_S, N = sm.sc.n_stages;
    const size_t ms = (size_t)bp.max_stages, slice = ms * 312 + 600;
    SpecRec* rec = bp.spec_rec + (size_t)e * S;
    const double* out = bp.spec_out + (size_t)e * (S - 1) * slice;  // + (c - 1) * slice: candidate c >= 1
    if (tid == 0) rec[j] = SpecRec{ran ? (ok ? 1 : 0) : -1, 0, sm.st.dV_1, sm.st.dV_2};
    __threadfence();
    __syncthreads();
    if (tid == 0) sm.ibuf[2] = atomicAdd(bp.spec_arrive + e, 1) == S - 1;
    __syncthreads();
    if (!sm.ibuf[2]) return false;
    __threadfence();
    if (tid == 0) {
        bp.spec_arrive[e] = 0;  // (for the next round)
        int w = -1, m = 0;
        while (m < S) {
            const int c = __ldcg(&rec[m].ok);
            if (c < 0) break;
            ++m;
            if (c) { w = m - 1; break; }
        }
        const int c = w >= 0 ? w : m - 1;
        sm.ibuf[2] = w; sm.ibuf[3] = m;
        const size_t pid = (size_t)sm.pid;
        sm.K = bp.K + pid * ms * 288; sm.dU = bp.dU + pid * ms * 24; sm.g0h0 = bp.g0h0 + pid * 600;
        sm.st.dV_1 = __ldcg(&rec[c].dV_1); sm.st.dV_2 = __ldcg(&rec[c].dV_2); sm.st.sweep_ok = w >= 0 ? 1 : 0;
        atomicAdd(bp.counters + 1, 1ull);
        if (w != 0) atomicAdd(bp.counters + (w > 0 ? 2 : 3), 1ull);
    }
    __syncthreads();
    const int w = sm.ibuf[2], m = sm.ibuf[3];
    // the problem's arrays as the loop leaves them: candidate w's outputs, or, every candidate failed, per stage those of the last
    // candidate that wrote the stage (candidate 0 wrote in place)
    for (int c = (w >= 0 ? w : 1); c <= (w >= 0 ? w : m - 1); ++c) {
        if (c == 0) continue;
        const double* o = out + (c - 1) * slice;
        const unsigned long long* mark = reinterpret_cast<const unsigned long long*>(o + ms * 288);
        for (int x = tid; x < 288 * N; x += kThreads)
            if (w >= 0 || __ldcg(mark + 24 * (x / 288)) != kSpecUnwritten) sm.K[x] = __ldcg(o + x);
        for (int x = tid; x < 24 * N; x += kThreads)
            if (w >= 0 || __ldcg(mark + 24 * (x / 24)) != kSpecUnwritten) sm.dU[x] = __ldcg(o + ms * 288 + x);
        if (w >= 0)
            for (int x = tid; x < 600; x += kThreads) sm.g0h0[x] = __ldcg(o + ms * 312 + x);
        __syncthreads();
    }
    success = w >= 0;
    nsw = success ? w + 1 : m;
    reg = sm.st.reg;
    retry_reg(reg, success ? w : m - 1, sm.opt.update_regularization);
    return true;
}

// The backward sweep of a phased round (k_phase<PH_SWEEP>): the loop of backward_sweep_regularized_block for an unlisted problem
// (e < 0), candidate j of list entry e for a listed one.  Returns false in the candidate blocks that did not commit: they must
// not store the problem's state.
__device__ inline bool sweep_round_block(Smem& sm, const BatchPtrs& bp, int e, int j) {
    const int tid = threadIdx.x;
    const double up = sm.opt.update_regularization;
    double reg = sm.st.reg;
    int nsw = 0;
    bool success = false, run = e < 0 || retry_reg(reg, j, up);
    if (e >= 0 && j > 0 && run) {  // outputs to the candidate's slice, with the first dU word of every stage marked unwritten
        const size_t ms = (size_t)bp.max_stages;
        double* o = bp.spec_out + ((size_t)e * (bp.spec_S - 1) + j - 1) * (ms * 312 + 600);
        for (int s = tid; s < sm.sc.n_stages; s += kThreads) reinterpret_cast<unsigned long long*>(o + ms * 288)[24 * s] = kSpecUnwritten;
        if (tid == 0) { sm.K = o; sm.dU = o + ms * 288; sm.g0h0 = o + ms * 312; }
    }
    __syncthreads();
    for (;;) {  // (the kernel's only call of the sweep: its code stays one sweep long)
        if (run) { ++nsw; success = backward_sweep_block(sm, reg); }
        if (e >= 0) {
            if (!spec_commit_block(sm, bp, e, j, run, success, reg, nsw, success)) return false;
            e = -1;
        }
        if (success) break;
        reg = fmax(reg * up, 1e-03);
        if (reg > 1e2) break;
        run = true;
    }
    reg = reg / 20;
    if (reg < 1e-06) reg = 0;
    if (tid == 0) sm.st.reg = reg;
    __syncthreads();
    finish_sweep_block(sm, bp, success, nsw);
    return true;
}

template <bool CLUSTER_LS = false>
__device__ inline void iter_forward_block(Smem& sm, const BatchPtrs& bp) {
    const int tid = threadIdx.x;
    const hsddp_options& opt = sm.opt;
    hsddp_iter_record* rec = (sm.ctl.iter <= HSDDP_TRACE_CAP) ? bp.trace + (size_t)sm.pid * HSDDP_TRACE_CAP + sm.ctl.iter - 1 : nullptr;
    if (opt.MS && !bp.lr_external) linear_rollout_block(sm, 1.0);  // (phased driver: k_lr_w1 has left dX, K dX, dV_1, dV_2)
    prepare_merit_block(sm);
    const double cost_prev = sm.st.actual_cost, merit_prev = sm.st.merit;
    const double dV_abs = fabs(sm.st.dV_1 + 0.5 * sm.st.dV_2);
    bool leave_inner = false;
    if (tid == 0 && rec) { rec->dV_1 = sm.st.dV_1; rec->dV_2 = sm.st.dV_2; rec->merit_rho = sm.st.merit_rho; }
    if ((dV_abs < opt.cost_thresh) && (sm.st.feas <= opt.dynamics_feas_thresh)) {  // :340-343
        if (tid == 0 && rec) {
            rec->eps_accepted = -1; rec->n_trials = 0;
            rec->cost_after = sm.st.actual_cost; rec->feas_after = sm.st.feas; rec->max_tconstr = sm.st.max_tconstr; rec->max_pconstr = sm.st.max_pconstr;
        }
        leave_inner = true;
    } else {
        double eps_acc = 0;
        int ntr = 0;
        if (CLUSTER_LS ? line_search_cluster(sm, bp, eps_acc, ntr) : line_search_block<true>(sm, eps_acc, ntr)) {
            update_nominal_block(sm);
        } else {  // Q2: only the scalars are restored
            __syncthreads();
            if (tid == 0) { sm.st.actual_cost = cost_prev; sm.st.merit = merit_prev; }
            __syncthreads();
        }
        if (tid == 0) {
            sm.ctl.n_trials += ntr;
            if (rec) {
                rec->eps_accepted = eps_acc; rec->n_trials = ntr;
                rec->cost_after = sm.st.actual_cost; rec->feas_after = sm.st.feas; rec->max_tconstr = sm.st.max_tconstr; rec->max_pconstr = sm.st.max_pconstr;
            }
        }
        if ((fabs((cost_prev - sm.st.actual_cost) / cost_prev) < opt.cost_thresh) && (sm.st.feas <= opt.dynamics_feas_thresh)) leave_inner = true;  // :358-359
    }
    __syncthreads();
    if (leave_inner || sm.ctl.iter_in >= sm.ctl.max_ddp) outer_end_block(sm);
}

__device__ inline void solve_finish_block(Smem& sm, const BatchPtrs& bp) {
    __syncthreads();
    if (threadIdx.x == 0) {
        hsddp_info& info = bp.info[sm.pid];
        const SolveCtl& c = sm.ctl;
        info.status = c.status; info.n_iter = c.iter; info.n_outer = c.iter_ou; info.n_sweeps = c.n_sweeps; info.n_trials = c.n_trials; info._pad = 0;
        info.cost = sm.st.actual_cost; info.feas = sm.st.feas; info.max_tconstr = sm.st.max_tconstr; info.max_pconstr = sm.st.max_pconstr;
        info.cost0 = c.cost0; info.feas0 = c.feas0;
        atomicAdd(bp.counters, (unsigned long long)c.n_sweeps * (unsigned long long)sm.sc.n_stages);
    }
    __syncthreads();
}

template <bool CLUSTER_LS = false>
__device__ inline void solve_block(Smem& sm, const BatchPtrs& bp) {
    solve_begin_block(sm, bp);
    while (sm.ctl.active) {
        iter_prep_block(sm, bp);
        iter_sweep_block(sm, bp);
        if (!sm.ctl.active) break;
        iter_forward_block<CLUSTER_LS>(sm, bp);
    }
    solve_finish_block(sm, bp);
}

__device__ __forceinline__ void solve_persistent(Smem& sm, const BatchPtrs& bp, const hsddp_options& opt);

// throughput build: HSDDP_MIN_BLOCKS resident blocks per SM (80 registers / thread)
__global__ void __launch_bounds__(kThreads, HSDDP_MIN_BLOCKS) k_solve(BatchPtrs bp, hsddp_options opt) {
    __shared__ Smem sm;
    solve_persistent(sm, bp, opt);
}
// latency build: the same code compiled for two resident blocks (255 registers / thread: nothing spills, nothing is
// rematerialised); used when the batch does not fill the GPU anyway (single-solve latency, MPC tick of one robot)
__global__ void __launch_bounds__(kThreads, 2) k_solve_lat(BatchPtrs bp, hsddp_options opt) {
    __shared__ Smem sm;
    solve_persistent(sm, bp, opt);
}

// latency build with the concurrent line search: one cluster of four blocks per problem (block rank 0 solves, ranks 1..3 evaluate
// the other step sizes of every line search).  Cluster q solves problem bp.order[q] (nullptr: problem q).
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(kThreads, 2) k_solve_lat4(BatchPtrs bp, hsddp_options opt) {
    namespace cg = cooperative_groups;
    __shared__ Smem sm;
    const int pid = bp.order ? bp.order[ls_pos()] : ls_pos(), r = (int)cg::this_cluster().block_rank();
    if (threadIdx.x == 0) assign_rotation(bp.sm_slots, sm.rot);
    bind_problem(sm, bp, pid);
    if (threadIdx.x == 0) sm.opt = opt;
    __syncthreads();
    if (r == 0) {
        solve_block<true>(sm, bp);
        if (threadIdx.x == 0) { bp.state[pid] = sm.st; bp.ctl[pid] = sm.ctl; bp.ls_mail[ls_pos()] = 2; __threadfence(); }
        cg::this_cluster().sync();  // [A] of the helpers' last round: exit
    } else {
        line_search_helper_loop(sm, bp, r);
    }
}

__device__ __forceinline__ void solve_persistent(Smem& sm, const BatchPtrs& bp, const hsddp_options& opt) {
    if (threadIdx.x == 0) assign_rotation(bp.sm_slots, sm.rot);
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) {
            const int q = atomicAdd(bp.work_counter, 1);
            sm.ibuf[3] = (q < bp.n_problems && bp.order) ? bp.order[q] : q;
        }
        __syncthreads();
        const int pid = sm.ibuf[3];
        if (pid >= bp.n_problems) break;
        bind_problem(sm, bp, pid);
        if (threadIdx.x == 0) sm.opt = opt;
        __syncthreads();
#ifdef HSDDP_PROFILE
        if (threadIdx.x == 0) for (int i = 0; i < 16; ++i) sm.profacc[i] = 0;
        __syncthreads();
#endif
        solve_block(sm, bp);
        if (threadIdx.x == 0) { bp.state[pid] = sm.st; bp.ctl[pid] = sm.ctl; }
#ifdef HSDDP_PROFILE
        if (threadIdx.x == 0) for (int i = 0; i < 16; ++i) atomicAdd(&sm.prof[i], sm.profacc[i]);
#endif
    }
}

// One phase of solve() for every running problem: block b works on problem bp.active[b] (or b).
enum SolvePhase { PH_BEGIN = 0, PH_PREP, PH_SWEEP, PH_FORWARD };
// Register budgets of the per-phase kernels (resident blocks per SM they are compiled for).  Measured on 16,384
// config-3 problems: the backward-sweep kernel, bound by shared-memory wavefronts, is best at 5 blocks (102
// registers, nothing spills in the stage loop): 418 ms against 427 (6 blocks) and 438 (4); the prep and forward
// kernels are best at 6.
#ifndef HSDDP_MINB_SWEEP
#define HSDDP_MINB_SWEEP 5
#endif
#ifndef HSDDP_MINB_OTHER
#define HSDDP_MINB_OTHER 6
#endif
template <int PH>
__global__ void __launch_bounds__(kThreads, PH == 2 ? HSDDP_MINB_SWEEP : HSDDP_MINB_OTHER) k_phase(BatchPtrs bp, hsddp_options opt) {
    __shared__ Smem sm;
    // (the counter of the list this round appends to is cleared even when no problem is left: the next round reads it)
    if (PH == PH_PREP && bp.zero_count && blockIdx.x == 0 && threadIdx.x == 0) {
        *bp.zero_count = 0;
        if (bp.spec_zero) *bp.spec_zero = 0;
    }
    // sweep with speculation: the first spec_cap x (spec_S - 1) blocks are candidates 1 .. spec_S - 1 of the listed problems
    // (the lowest block indices, so that the long retry chains start first), the problems' own blocks follow
    int blk = (int)blockIdx.x, cand = 0, entry = -1;
    if (PH == PH_SWEEP && bp.spec_list) {
        const int ns = bp.spec_cap * (bp.spec_S - 1);
        if (blk < ns) { entry = blk / (bp.spec_S - 1); cand = 1 + blk % (bp.spec_S - 1); }
        blk -= ns;
    }
    if (bp.n_active && blk >= *bp.n_active) return;  // (the grid is the group's full size: see BatchPtrs::active)
    if (PH == PH_SWEEP && bp.n_active && bp.sweep_w1_min > 0 && *bp.n_active >= bp.sweep_w1_min) return;  // (k_sweep_w1 takes this round)
    if (PH == PH_SWEEP && cand > 0 && entry >= min(*bp.spec_count, bp.spec_cap)) return;
    const int pid = cand > 0 ? bp.spec_list[entry] : bp.active ? bp.active[blk] : blk;
    if (threadIdx.x == 0) assign_rotation(bp.sm_slots, sm.rot);
    bind_problem(sm, bp, pid);
    if (threadIdx.x == 0) sm.opt = opt;
    __syncthreads();
#ifdef HSDDP_PROFILE
    if (threadIdx.x == 0) for (int i = 0; i < 16; ++i) sm.profacc[i] = 0;
    __syncthreads();
#endif
    bool store = true;
    if (PH == PH_BEGIN) solve_begin_block(sm, bp);
    if (PH == PH_PREP) {
        iter_prep_block(sm, bp);
        if (bp.spec_list && (bp.sweep_w1_min == 0 || *bp.n_active < bp.sweep_w1_min)) spec_flag_block(sm, bp);
    }
    if (PH == PH_SWEEP) {
        if (bp.spec_list && cand == 0) entry = bp.spec_entry[pid];
        store = sweep_round_block(sm, bp, entry, cand);
    }
    if (PH == PH_FORWARD) {
        if (sm.ctl.active) iter_forward_block(sm, bp);  // (a failed sweep already ended the solve)
    }
    __syncthreads();
    if (PH == PH_BEGIN || PH == PH_FORWARD) {
        if (sm.ctl.active) {
            if (threadIdx.x == 0) bp.next_active[atomicAdd(bp.next_count, 1)] = pid;
        } else {
            solve_finish_block(sm, bp);
        }
    }
    if (store && threadIdx.x == 0) { bp.state[pid] = sm.st; bp.ctl[pid] = sm.ctl; }
#ifdef HSDDP_PROFILE
    if (threadIdx.x == 0) for (int i = 0; i < 16; ++i) atomicAdd(&sm.prof[i], sm.profacc[i]);
#endif
}

enum StepOp { OP_RESET = 0, OP_ROLLOUT, OP_COST, OP_LQ, OP_SWEEP, OP_SWEEP_REG, OP_LINEAR, OP_MERIT, OP_FORWARD, OP_NOMINAL, OP_AL, OP_REB };

// step-level kernel: one block per problem, state round-trips through HBM
__global__ void __launch_bounds__(kThreads, HSDDP_MIN_BLOCKS) k_step(BatchPtrs bp, hsddp_options opt, int op, double arg, double* darg, int* ok) {
    __shared__ Smem sm;
    const int pid = blockIdx.x;
    if (threadIdx.x == 0) assign_rotation(bp.sm_slots, sm.rot);
    bind_problem(sm, bp, pid);
    if (threadIdx.x == 0) sm.opt = opt;
    __syncthreads();
    int okv = 1;
    switch (op) {
        case OP_RESET: cold_start_block(sm); break;
        case OP_ROLLOUT: okv = hybrid_rollout_block<false>(sm, arg) ? 1 : 0; break;
        case OP_COST: compute_cost_block(sm); break;
        case OP_LQ: lq_approximation_block(sm); break;
        case OP_SWEEP: okv = backward_sweep_block(sm, arg) ? 1 : 0; break;
        case OP_SWEEP_REG: {
            if (threadIdx.x == 0) sm.st.reg = darg[pid];
            __syncthreads();
            int nsw;
            okv = backward_sweep_regularized_block(sm, nsw) ? 1 : 0;
            if (threadIdx.x == 0) darg[pid] = sm.st.reg;
        } break;
        case OP_LINEAR: linear_rollout_block(sm, arg); break;
        case OP_MERIT: prepare_merit_block(sm); break;
        case OP_FORWARD: {
            const double cost_prev = sm.st.actual_cost, merit_prev = sm.st.merit;
            double eps_acc; int ntr;
            okv = line_search_block<false>(sm, eps_acc, ntr) ? 1 : 0;
            if (!okv) { __syncthreads(); if (threadIdx.x == 0) { sm.st.actual_cost = cost_prev; sm.st.merit = merit_prev; } }
            if (threadIdx.x == 0 && darg) darg[pid] = eps_acc;
        } break;
        case OP_NOMINAL: update_nominal_block(sm); break;
        case OP_AL: update_al_block(sm); break;
        case OP_REB: update_reb_block(sm); break;
        default: break;
    }
    __syncthreads();
    if (threadIdx.x == 0) { bp.state[pid] = sm.st; if (ok) ok[pid] = okv; }
}

// HKDMPCSolver::publish_mpc_cmd + update_foot_placement (HKDMPC/HKDMPC.cpp:207-298): one block per problem packs the
// command record.  Stage k of the command = stage s of phase i, walked with the reference's (k, s, i) loop.  Block j packs
// problem list[j] (nullptr: problem j) into out[j].
__global__ void k_command(BatchPtrs bp, int n_steps, hsddp_mpc_command* out, const int* list) {
    const int pid = list ? list[blockIdx.x] : (int)blockIdx.x;
    const DevSchedule& sc = bp.sched[bp.sched_id[pid]];
    hsddp_mpc_command& cmd = out[blockIdx.x];
    __shared__ int s_stage[HSDDP_CMD_MAX_STEPS], s_node[HSDDP_CMD_MAX_STEPS], s_phase[HSDDP_CMD_MAX_STEPS];
    if (threadIdx.x == 0) {
        int s = 0, i = 0;
        for (int k = 0; k < n_steps; ++k) {
            if (s >= sc.horizon[i]) { s = 0; i++; }
            if (i >= sc.n_phases) { i = sc.n_phases - 1; s = sc.horizon[i] - 1; }  // (horizon shorter than the command: repeat the last stage)
            s_stage[k] = sc.stage_off[i] + s; s_node[k] = sc.node_off[i] + s; s_phase[k] = i;
            s++;
        }
        cmd.N_mpcsteps = n_steps; cmd._pad = 0;
    }
    __syncthreads();
    const double* Xbar = bp.Xbar + (size_t)pid * bp.max_nodes * 24;
    const double* Ubar = bp.Ubar + (size_t)pid * bp.max_stages * 24;
    const double* K = bp.K + (size_t)pid * bp.max_stages * 288;
    for (int e = threadIdx.x; e < HSDDP_CMD_MAX_STEPS * 24; e += blockDim.x) {
        const int k = e / 24, j = e % 24;
        cmd.hkd_controls[k][j] = (k < n_steps) ? (float)Ubar[24 * s_stage[k] + j] : 0.f;
        if (j < 12) cmd.des_body_state[k][j] = (k < n_steps) ? (float)Xbar[24 * s_node[k] + j] : 0.f;
        if (j < 4) cmd.contacts[k][j] = (k < n_steps) ? (int)((sc.cmask[s_phase[k]] >> j) & 1u) : 0;
    }
    for (int e = threadIdx.x; e < HSDDP_CMD_MAX_STEPS * 144; e += blockDim.x) {
        const int k = e / 144, m = (e % 144) / 12, n = e % 12;
        float v = 0.f;
        // K(m, n), m < 12: GRF component m; non-zero only for a stance leg, where it is the coupled control m
        if (k < n_steps && ((sc.cmask[s_phase[k]] >> (m / 3)) & 1u)) v = (float)K[288 * (size_t)s_stage[k] + 12 * n + m];
        cmd.feedback[k][m][n] = v;
    }
    if (threadIdx.x < 4) {
        const int l = threadIdx.x;
        int found = 0;
        float pf[3] = {0.f, 0.f, 0.f};
        for (int i = 0; i < sc.n_phases - 1 && !found; ++i) {
            if (!((sc.cmask[i] >> l) & 1u) && ((sc.cmask[i + 1] >> l) & 1u)) {
                const double* q = Xbar + 24 * sc.node_off[i + 1] + 12 + 3 * l;
                pf[0] = (float)q[0]; pf[1] = (float)q[1]; pf[2] = (float)q[2];
                found = 1;
            }
            if (i >= 4) break;
        }
        cmd.foot_found[l] = found;
        cmd.foot_placement[3 * l] = pf[0]; cmd.foot_placement[3 * l + 1] = pf[1]; cmd.foot_placement[3 * l + 2] = pf[2];
    }
}


// ---------------------------------------------------------------------------
// N2: reference ingestion on the device.  The gait library (QuadReference::tp_data of every gait, already parsed
// through stof) is resident in HBM; one kernel builds, for every (gait, window start), what QuadReference::initialize
// + HKDProblem::initialization produce: the phase table (HKDProblem.cpp:26-68), the contact after each phase
// (:268-299, Q17) and the per-node reference rows the cost callbacks and the initial guess see (HKDReference.cpp:8-57,
// HKDProblem.cpp:84-90).  The host builder (host/hkd_problem.cpp: hkd_schedule_build) is restated here with the
// SAME float arithmetic — every float / double product-sum that the host rounds twice is written with
// __fmul_rn / __fadd_rn / __dmul_rn / __dadd_rn so that the compiler cannot contract it — and the two are compared
// bit for bit in tests/test_gpu_parity.py::test_device_schedule_builder_bit_exact.
// ---------------------------------------------------------------------------
struct GaitLib {
    const double *body_state, *qJ, *foot, *grf;  // concatenated over gaits, [row][12]
    const int* contact;                          // [row][4]
    const int* row_off;                          // first row of gait g
    const int* n_rows;                           // rows of gait g
    const float* dt;                             // sample period of gait g
    float plan;                                  // plan duration of every schedule of the batch
    int node_stride;                             // reference rows per schedule slot
};

// dt_sim (one MPC tick) and dt_mpc (the stage length) of the reference's MPC loop: both 0.01 s
constexpr float kTickDt = 0.01f;

// Per-schedule state of the receding-horizon update (HKDProblemData of HKDProblem.h:28-66 + QuadReference::k_cur / t_cur):
// everything HKDProblem::update needs beyond the phase table itself.
struct MpcSched {
    float start[MAXPH], end[MAXPH];        // pdata->phase_start_times / phase_end_times (absolute, float)
    unsigned char reach_end[MAXPH];        // pdata->is_phase_reach_end
    unsigned char has_tconstr[MAXPH];      // add_tconstr_one_phase has bound a reset map to the phase
    int k_cur;                             // samples the reference window has moved since initialisation
    float t_cur;                           // QuadReference::t_cur (accumulated in float)
    // what the last update did, for the per-problem shift kernel
    int front_nodes;                       // nodes dropped at the front: 1 (pop_front) or horizon+1 of a popped phase
    int front_phase_popped;                // 1: the first phase was removed
    int back_new_phase;                    // 1: a new last phase was created (horizon 1), 0: the last phase grew by one stage
    int old_n_nodes;                       // node count before the update
    int new_td_phase, new_td_object;       // touchdown-constraint object added by this update (-1: none)
    int status;                            // 0 ok, 1 reference exhausted, 2 table limits exceeded
};

__device__ __forceinline__ bool approx_eq_f(float a, float b) { return fabsf(__fsub_rn(a, b)) <= 1e-6f; }
__device__ __forceinline__ bool approx_leq_f(float a, float b) { return a < b || approx_eq_f(a, b); }
__device__ __forceinline__ bool approx_geq_f(float a, float b) { return a > b || approx_eq_f(a, b); }
// QuadReference::get_a_reference_ptr_at_t index rule (QuadReference.cpp:65-80), float arithmetic
__device__ __forceinline__ int ref_index_at(float t, float dt, int sz) {
    int k = (int)floorf(__fdiv_rn(t, dt));
    const float rem = __fsub_rn(t, __fmul_rn((float)k, dt));
    if ((double)rem > __dmul_rn(0.5, (double)dt)) k++;
    if (k > sz) k = sz;
    return k;
}

// samples in the reference window of a schedule: plan duration over the gait's sample period, plus one
__device__ __forceinline__ int ref_window_size(const GaitLib& lib, float dtg) { return (int)roundf(__fdiv_rn(lib.plan, dtg)) + 1; }

__device__ __forceinline__ unsigned contact_mask_at(const GaitLib& lib, size_t row) {
    const int* c = lib.contact + 4 * row;
    return (c[0] ? 1u : 0u) | (c[1] ? 2u : 0u) | (c[2] ? 4u : 0u) | (c[3] ? 8u : 0u);
}

// pass 1: phase tables and update state, one thread per schedule.  status[i] != 0 marks an unusable window.  Schedule i
// goes to slot slot[i] (nullptr: slot i) and may have at most stage_cap stages.
__global__ void k_build_phase_tables(GaitLib lib, int n_sched, const int* sched_gait, const int* sched_window, const int* slot, int stage_cap,
                                     DevSchedule* out, MpcSched* mpc, int* status) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_sched) return;
    const int si = slot ? slot[i] : i;
    const int gi = sched_gait[i], k0 = sched_window[i];
    const float dtg = lib.dt[gi];
    const int sz = ref_window_size(lib, dtg);
    DevSchedule d;
    memset(&d, 0, sizeof d);
    MpcSched m;
    memset(&m, 0, sizeof m);
    m.new_td_phase = -1; m.new_td_object = -1;
    int st = 0;
    if (k0 < 0 || k0 + sz >= lib.n_rows[gi]) st = 1;
    const size_t row0 = (size_t)(lib.row_off[gi] + k0);
    if (!st) {
        int n_phases = 0;
        float phase_start = 0.f, t = 0.f;
        size_t rprev = row0 + ref_index_at(t, dtg, sz);  // sample whose contact flags the current phase has
        while (approx_leq_f(t, lib.plan)) {
            const size_t r = row0 + ref_index_at(t, dtg, sz);
            bool change = false;
            for (int l = 0; l < 4; ++l) change = change || (lib.contact[4 * r + l] != lib.contact[4 * rprev + l]);
            if (change || approx_geq_f(t, lib.plan)) {
                if (n_phases >= MAXPH) { st = 2; break; }
                const int hz = (int)roundf(__fdiv_rn(__fsub_rn(t, phase_start), kTickDt));
                d.horizon[n_phases] = hz;
                d.cmask[n_phases] = contact_mask_at(lib, rprev);
                d.ss_size[n_phases] = (unsigned char)(hz + 1);  // update_SS_config(horizon + 1), HKDProblem.cpp:104
                m.start[n_phases] = phase_start; m.end[n_phases] = t; m.reach_end[n_phases] = 0; m.has_tconstr[n_phases] = 1;
                ++n_phases;
                rprev = r;
                phase_start = t;
            }
            t = __fadd_rn(t, kTickDt);
        }
        if (!st && (n_phases < 1 || !layout_phases(d, n_phases, stage_cap, lib.node_stride))) st = 2;
    }
    d.dt = (double)kTickDt;
    d.ref_off = (long long)si * lib.node_stride;
    out[si] = d;
    status[i] = st;
    m.status = st;
    mpc[si] = m;
}

// pass 2: reference rows, one block per entry i: schedule slot slot[i] (nullptr: slot i) of gait gait[i] and initial window
// window[i], whose phase table and update state are in place.  Entries of a free slot (gait -1) or of a failed build or
// update are skipped.  xinit != nullptr: the call completes a build (pass 1): it also writes the initial-guess rows and the
// contact after each phase with its touchdown legs.
__global__ void k_reference_rows(GaitLib lib, int n, const int* gait, const int* window, const int* slot,
                                 DevSchedule* scheds, const MpcSched* mpc, double* xr, double* ur, double* prel, double* xinit) {
    const int i = blockIdx.x;
    if (i >= n) return;
    const int si = slot ? slot[i] : i, gi = gait[i];
    if (gi < 0 || mpc[si].status) return;
    DevSchedule& d = scheds[si];
    const MpcSched& m = mpc[si];
    const float dtg = lib.dt[gi];
    const int sz = ref_window_size(lib, dtg);
    const size_t row0 = (size_t)(lib.row_off[gi] + window[i] + m.k_cur);
    // HKDReference.cpp:33-56 (Q12): foot placement if the SAMPLE's contact flag is set, else joint angle
    auto state_row = [&](size_t r, double* x) {
        for (int j = 0; j < 12; ++j) x[j] = lib.body_state[12 * r + j];
        for (int l = 0; l < 4; ++l)
            for (int j = 0; j < 3; ++j)
                x[12 + 3 * l + j] = (lib.contact[4 * r + l] > 0) ? lib.foot[12 * r + 3 * l + j] : lib.qJ[12 * r + 3 * l + j];
    };
    for (int nd = threadIdx.x; nd < d.n_nodes; nd += blockDim.x) {
        const int ph = d.ph_of_node[nd], k = nd - d.node_off[ph];
        const size_t node = (size_t)d.ref_off + nd;
        // time seen by the cost callbacks: float(t_offset + k*dt), t_offset = start - start[0] in float (set_time_offset),
        // dt widened to double (SinglePhase.cpp:243,254)
        const float t_offset = __fsub_rn(m.start[ph], m.start[0]);
        const float tc = (float)__dadd_rn((double)t_offset, __dmul_rn((double)k, d.dt));
        const size_t r = row0 + ref_index_at(tc, dtg, sz);
        state_row(r, xr + 24 * node);
        for (int j = 0; j < 12; ++j) { ur[24 * node + j] = lib.grf[12 * r + j]; ur[24 * node + 12 + j] = 0.0; }  // qJd is never loaded: zeros
        for (int l = 0; l < 4; ++l)
            for (int j = 0; j < 3; ++j) prel[12 * node + 3 * l + j] = lib.foot[12 * r + 3 * l + j] - lib.body_state[12 * r + 3 + j];
        // time used for the initial guess: float(phase_start + k*dt_sim), all float (HKDProblem.cpp:86-90)
        if (xinit) state_row(row0 + ref_index_at(__fadd_rn(m.start[ph], __fmul_rn((float)k, kTickDt)), dtg, sz), xinit + 24 * node);
    }
    if (xinit && threadIdx.x < d.n_phases) {  // contact after each phase (reset map / touchdown wiring), HKDProblem.cpp:268-299, Q17
        const int p = threadIdx.x;
        const unsigned nm = p < d.n_phases - 1 ? d.cmask[p + 1] : contact_mask_at(lib, row0 + ref_index_at(__fadd_rn(lib.plan, kTickDt), dtg, sz));
        d.nmask[p] = nm;
        d.tdmask[0][p] = (unsigned char)touchdown_legs(d.cmask[p], nm);
        d.tdmask[1][p] = 0;
    }
}

// ---------------------------------------------------------------------------
// N1: receding-horizon update on the device (HKDProblem::update, HKDMPC/HKD-TrajOpt/HKDProblem.cpp:117-222, as
// HKDMPCSolver::update drives it every MPC step, HKDMPC.cpp:97-166).  All problems of a batch tick together, so a
// schedule (gait, initial window) stays shared by the problems that use it:
//   k_mpc_update_schedules  one thread per schedule (entry i: slot slot[i], nullptr: slot i): QuadReference::step (QuadReference.cpp:33-47), front end (drop the first
//                           node or the whole first phase), back end (grow the last phase or open a new one; add_tconstr_one_phase
//                           when the last phase has reached its end), shooting sets -- with the reference's float time arithmetic
//   k_reference_rows        the per-node reference rows of the shifted window (HKDReference.cpp:8-57)
//   k_mpc_shift             one block per problem: Trajectory::pop_front / push_back_state (TrajectoryManagement.cpp:118-207),
//                           PathConstraintBase::pop_front / push_back (ConstraintsBase.h:271-280) on the problem-major arrays
// ---------------------------------------------------------------------------
__global__ void k_mpc_update_schedules(GaitLib lib, int n_sched, const int* sched_gait, const int* sched_window, const int* slot,
                                       DevSchedule* scheds, MpcSched* mpc, int* err) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_sched) return;
    const int gi = sched_gait[i], si = slot ? slot[i] : i;
    if (gi < 0) return;  // a free slot (hsddp_batch_restart_problems)
    DevSchedule d = scheds[si];
    MpcSched m = mpc[si];
    const float dtg = lib.dt[gi];
    const int sz = ref_window_size(lib, dtg);
    m.old_n_nodes = d.n_nodes;
    m.new_td_phase = -1; m.new_td_object = -1;
    // QuadReference::step(dt_sim)
    for (int q = 1; approx_leq_f(__fmul_rn((float)q, dtg), kTickDt); ++q) { m.k_cur++; m.t_cur = __fadd_rn(m.t_cur, dtg); }
    const float new_start = m.t_cur, new_end = __fadd_rn(m.t_cur, lib.plan);
    const size_t row0 = (size_t)(lib.row_off[gi] + sched_window[i] + m.k_cur);
    if (sched_window[i] + m.k_cur + sz >= lib.n_rows[gi]) { m.status = 1; mpc[si] = m; atomicMax(err, 1); return; }
    int n = d.n_phases;
    // ---- front end ----
    m.start[0] = __fadd_rn(m.start[0], kTickDt);
    if (approx_leq_f(m.end[0], new_start)) {  // the first phase has shrunk to a point: pop_front_phase
        m.front_nodes = d.horizon[0] + 1; m.front_phase_popped = 1;
        for (int p = 0; p + 1 < n; ++p) {
            d.horizon[p] = d.horizon[p + 1]; d.cmask[p] = d.cmask[p + 1]; d.nmask[p] = d.nmask[p + 1]; d.ss_size[p] = d.ss_size[p + 1];
            d.tdmask[0][p] = d.tdmask[0][p + 1]; d.tdmask[1][p] = d.tdmask[1][p + 1];
            m.start[p] = m.start[p + 1]; m.end[p] = m.end[p + 1]; m.reach_end[p] = m.reach_end[p + 1]; m.has_tconstr[p] = m.has_tconstr[p + 1];
        }
        --n;
    } else {
        m.front_nodes = 1; m.front_phase_popped = 0;
        d.horizon[0]--;
        m.start[0] = new_start;
    }
    // ---- back end ----
    const unsigned newc = contact_mask_at(lib, row0 + ref_index_at(__fsub_rn(new_end, new_start), dtg, sz));
    const bool change = newc != d.cmask[n - 1];
    if (change && m.reach_end[n - 1]) {
        if (n >= MAXPH) { m.status = 2; mpc[si] = m; atomicMax(err, 2); return; }
        m.start[n] = m.end[n - 1]; m.end[n] = new_end; m.reach_end[n] = 0; m.has_tconstr[n] = 0;
        d.horizon[n] = (int)roundf(__fdiv_rn(__fsub_rn(m.end[n], m.start[n]), kTickDt));
        d.cmask[n] = newc; d.nmask[n] = 0; d.tdmask[0][n] = 0; d.tdmask[1][n] = 0; d.ss_size[n] = 0;  // (SinglePhase::initialization clears SS_set)
        m.back_new_phase = 1;
        ++n;
    } else {
        m.end[n - 1] = new_end;
        if (change) m.reach_end[n - 1] = 1;
        d.horizon[n - 1]++;
        m.back_new_phase = 0;
    }
    if (m.reach_end[n - 1]) {  // add_tconstr_one_phase(last phase): the contact after it is the reference's at plan_duration + dt_mpc
        const unsigned nm = contact_mask_at(lib, row0 + ref_index_at(__fadd_rn(lib.plan, kTickDt), dtg, sz));
        d.nmask[n - 1] = nm; m.has_tconstr[n - 1] = 1;
        const unsigned td = touchdown_legs(d.cmask[n - 1], nm);
        if (td) {
            const int ob = d.tdmask[0][n - 1] ? (d.tdmask[1][n - 1] ? 2 : 1) : 0;
            if (ob >= 2) { m.status = 2; mpc[si] = m; atomicMax(err, 2); return; }  // (needs a one-sample contact blip in the reference)
            d.tdmask[ob][n - 1] = (unsigned char)td;
            m.new_td_phase = n - 1; m.new_td_object = ob;
        }
    }
    // ---- shooting configuration (HKDProblem.cpp:205-221) and the derived tables ----
    for (int p = 0; p < n; ++p)
        if ((p == n - 1 && d.horizon[p] > 2) || p < n - 1) d.ss_size[p] = (unsigned char)(d.horizon[p] + 1);
    if (!layout_phases(d, n, HSDDP_MAX_STAGES, lib.node_stride)) { m.status = 2; mpc[si] = m; atomicMax(err, 2); return; }
    scheds[si] = d;
    mpc[si] = m;
}

// rows [shift, total) of a row-major array move down to [0, total - shift); the last `shift` rows are then filled by the caller.
// In place: a chunk is read by every thread before any thread writes it (the destination of a chunk overlaps only chunks
// that have been read already).
__device__ inline void shift_rows_down(double* a, int total_rows, int row_len, int shift_rows) {
    const int n = (total_rows - shift_rows) * row_len, off = shift_rows * row_len;
    for (int c = 0; c < n; c += 4 * kThreads) {
        double v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { const int e = c + q * kThreads + threadIdx.x; v[q] = (e < n) ? a[e + off] : 0.0; }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) { const int e = c + q * kThreads + threadIdx.x; if (e < n) a[e] = v[q]; }
        __syncthreads();
    }
}

// The device commit of a call that moves listed problems to new schedule slots (plan_slot_moves), once they have been built: block j
// binds problem[j] to slot[j], block 0 writes gait / window of the m target slots and gait -1 of the f freed ones (a free slot
// carries gait -1 on the device, which the receding-horizon update skips; the targets carry it until here).
struct SlotMoves {
    int *problem, *slot;          // [launch blocks] (problem nullptr: no move)
    int *target, *gait, *window;  // [m]
    int* freed;                   // [f]
    int m, f;
    int *sched_gait, *sched_window;  // per slot
};

__device__ inline void write_slot_moves(const SlotMoves& mv, const int* sched_id) {
    if (threadIdx.x == 0) const_cast<int*>(sched_id)[mv.problem[blockIdx.x]] = mv.slot[blockIdx.x];
    if (blockIdx.x != 0) return;
    for (int e = threadIdx.x; e < mv.m; e += blockDim.x) { mv.sched_gait[mv.target[e]] = mv.gait[e]; mv.sched_window[mv.target[e]] = mv.window[e]; }
    for (int e = threadIdx.x; e < mv.f; e += blockDim.x) mv.sched_gait[mv.freed[e]] = -1;
}

// block j shifts problem j, or with moves (hsddp_batch_mpc_update_problems) moves problem mv.problem[j] to its stepped copy
// mv.slot[j] and shifts it there (a block reads its slot from the list, not the sched_id that another block writes)
__global__ void __launch_bounds__(kThreads) k_mpc_shift(BatchPtrs bp, const MpcSched* mpc, SlotMoves mv) {
    if (mv.problem) write_slot_moves(mv, bp.sched_id);
    const int pid = mv.problem ? mv.problem[blockIdx.x] : (int)blockIdx.x, tid = threadIdx.x;
    const int sid = mv.problem ? mv.slot[blockIdx.x] : bp.sched_id[pid];
    const MpcSched& m = mpc[sid];
    if (m.status) return;
    const DevSchedule& sc = bp.sched[sid];  // the schedule AFTER the update
    __shared__ double xback[24];
    const size_t sn = (size_t)bp.max_nodes * 24, ss = (size_t)bp.max_stages * 24;
    double *Xbar = bp.Xbar + pid * sn, *X = bp.X + pid * sn, *Ubar = bp.Ubar + pid * ss, *U = bp.U + pid * ss;
    double* K = bp.K + (size_t)pid * bp.max_stages * 288;
    double* reb = bp.reb + (size_t)pid * bp.max_stages * 40;
    double* al = bp.al + (size_t)pid * MAXPH * 16;
    double* hcon = bp.hcon + (size_t)pid * MAXPH * 4;
    const int N = sc.n_stages;              // unchanged by an update: one stage leaves at the front, one arrives at the back
    const int old_nodes = m.old_n_nodes, new_nodes = sc.n_nodes, kept = old_nodes - m.front_nodes;
    if (tid < 24) xback[tid] = X[24 * (old_nodes - 1) + tid];  // X.back() of the last phase, before anything moves
    __syncthreads();
    shift_rows_down(Xbar, old_nodes, 24, m.front_nodes);
    shift_rows_down(X, old_nodes, 24, m.front_nodes);
    shift_rows_down(Ubar, N, 24, 1);
    shift_rows_down(U, N, 24, 1);
    shift_rows_down(K, N, 288, 1);
    shift_rows_down(reb, N, 40, 1);
    // back end
    for (int e = tid; e < (new_nodes - kept) * 24; e += kThreads) {
        const double v = m.back_new_phase ? 0.0 : xback[e % 24];  // push_back_state(X.back()) / a zero-initialised Trajectory
        Xbar[24 * kept + e] = v; X[24 * kept + e] = v;
    }
    for (int e = tid; e < 24; e += kThreads) { Ubar[24 * (N - 1) + e] = 0.0; U[24 * (N - 1) + e] = 0.0; }
    for (int e = tid; e < 288; e += kThreads) K[288 * (size_t)(N - 1) + e] = 0.0;
    for (int e = tid; e < 20; e += kThreads) {
        // the new stage's ReB parameters: a copy of the phase's last stage (params.push_back(params.back())), the initial
        // values for a new phase
        const bool copy = !m.back_new_phase && N >= 2;
        reb[40 * (N - 1) + 2 * e] = copy ? reb[40 * (N - 2) + 2 * e] : bp.cp.grf_eps;
        reb[40 * (N - 1) + 2 * e + 1] = copy ? reb[40 * (N - 2) + 2 * e + 1] : bp.cp.grf_delta;
    }
    __syncthreads();
    // per-phase touchdown data: phases move down by one when the first phase was removed
    if (m.front_phase_popped) {
        double v[2];
        for (int q = 0; q < 2; ++q) { const int e = tid + q * kThreads; v[q] = (e < (MAXPH - 1) * 16) ? al[e + 16] : 0.0; }
        const double hv = (tid < (MAXPH - 1) * 4) ? hcon[tid + 4] : 0.0;
        __syncthreads();
        for (int q = 0; q < 2; ++q) { const int e = tid + q * kThreads; if (e < (MAXPH - 1) * 16) al[e] = v[q]; }
        if (tid < (MAXPH - 1) * 4) hcon[tid] = hv;
        __syncthreads();
    }
    if (tid < 8) {
        const int L = sc.n_phases - 1;
        if (m.back_new_phase) {  // a new phase starts with fresh constraint objects
            al[16 * L + 2 * tid] = bp.cp.td_sigma; al[16 * L + 2 * tid + 1] = bp.cp.td_lambda;
            if (tid < 4) hcon[4 * L + tid] = 0.0;
        }
        if (m.new_td_phase >= 0 && tid < 4) {  // a touchdown-constraint object added by this update: initial AL parameters
            al[16 * m.new_td_phase + 8 * m.new_td_object + 2 * tid] = bp.cp.td_sigma;
            al[16 * m.new_td_phase + 8 * m.new_td_object + 2 * tid + 1] = bp.cp.td_lambda;
        }
    }
    if (tid < 24) Ubar[tid] = 0.0;  // trajectory_ptrs.front()->Ubar[0].setZero(), HKDProblem.cpp:220
}

// ---------------------------------------------------------------------------
// HKDMPCSolver::initialize (HKDMPC.cpp:44-69) for a subset of the batch (hsddp_batch_restart_problems).  Launched only after
// the new schedules have been built and checked, so nothing here can fail.  One block per restarted problem j:
//   - the slot moves of the call (write_slot_moves: problem j is mv.problem[j]);
//   - the workspace arrays marked WS_RESTART are zeroed over the batch's full row count (what a fresh batch starts from: rows
//     the new schedule does not have stay zero, and no lq / tq record of the old schedule survives), info / ctl are reset,
//     then the cold start of a new problem;
//   - the initial state x0[j] and the iteration budget of the next solve (-1: the solve's options).
// ---------------------------------------------------------------------------
constexpr int kRestartClearMax = 32;
struct RestartArgs {
    const double* x0;  // [n][24]
    int max_al, max_ddp;
    int n_clear;
    struct { unsigned* base; size_t words; } clear[kRestartClearMax];  // arrays to zero: base, 4-byte words per problem
};

__global__ void __launch_bounds__(kThreads) k_restart(BatchPtrs bp, SlotMoves mv, RestartArgs ra) {
    __shared__ Smem sm;
    const int j = blockIdx.x, pid = mv.problem[j];
    write_slot_moves(mv, bp.sched_id);
    const size_t P = pid;
    for (int a = 0; a < ra.n_clear; ++a) {
        unsigned* p = ra.clear[a].base + P * ra.clear[a].words;
        for (size_t e = threadIdx.x; e < ra.clear[a].words; e += kThreads) p[e] = 0u;
    }
    if (threadIdx.x == 0) {
        bp.info[pid] = hsddp_info{};
        bp.ctl[pid] = SolveCtl{};
        if (bp.budget) { int* q = const_cast<int*>(bp.budget) + 2 * pid; q[0] = ra.max_al; q[1] = ra.max_ddp; }
    }
    if (threadIdx.x < 24) bp.x0[P * 24 + threadIdx.x] = ra.x0[24 * (size_t)j + threadIdx.x];
    __syncthreads();
    bind_problem(sm, bp, pid);
    cold_start_block(sm);
    if (threadIdx.x == 0) bp.state[pid] = sm.st;
}

// ---------------------------------------------------------------------------
// Receding-horizon update of listed problems (hsddp_batch_mpc_update_problems).  Problems share a schedule slot, so a slot that
// listed problems use is first copied, one block per slot: slot src[j] goes to the free slot dst[j] in every slot array but gait /
// window (the copy stays free until the commit), the copy gets its own reference rows (ref_off = dst[j] x node_stride), and gait /
// window of entry j are listed for the update kernels, which then step the copies only, and for the commit.
// ---------------------------------------------------------------------------
constexpr int kSlotArraysMax = 8;
struct SlotCopyArgs {
    const int *src, *dst;                    // [n]
    const int *sched_gait, *sched_window;    // per slot
    int *gait, *window;                      // [n] out
    DevSchedule* sched;
    int node_stride, n_arrays;
    struct { unsigned* base; size_t words; } arr[kSlotArraysMax];  // slot arrays: base, 4-byte words per slot
};

__global__ void k_copy_slots(SlotCopyArgs a) {
    const int j = blockIdx.x;
    const size_t s = (size_t)a.src[j], t = (size_t)a.dst[j];
    for (int k = 0; k < a.n_arrays; ++k)
        for (size_t e = threadIdx.x; e < a.arr[k].words; e += blockDim.x) a.arr[k].base[t * a.arr[k].words + e] = a.arr[k].base[s * a.arr[k].words + e];
    __syncthreads();
    if (threadIdx.x == 0) {
        a.sched[t].ref_off = (long long)t * a.node_stride;
        a.gait[j] = a.sched_gait[s]; a.window[j] = a.sched_window[s];
    }
}

// row idx[j] of dst := row j of src (src_stride 0: the same row for every j), rows of `words` 4-byte words.  Writes the per-problem
// rows of the list-driven entry points: initial states and cleared budgets.
__global__ void k_scatter_rows(unsigned* dst, int words, const int* idx, const unsigned* src, int src_stride, int n) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)n * words) return;
    const int j = (int)(e / words), w = (int)(e % words);
    dst[(size_t)idx[j] * words + w] = src[(size_t)j * src_stride + w];
}

// HKDMPCSolver::update's initial condition from the robot's measurement (hsddp_batch_set_measured_state_dev), one thread per
// listed problem: x0 row list[j] (nullptr: row j) := [meas[0:12], compute_hkd_state(eul, pos, qJ, contact)] (HKDModel.h:65-96)
// with meas row j = eul pos omega_body v_world qJ[12].  contact: the caller's flags row j (nonzero = stance) or, without them,
// the first phase of the problem's schedule as it stands when the kernel runs.
__global__ void k_measured_state(BatchPtrs bp, const double* meas, const int* contact, const int* list, int n) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int p = list ? list[j] : j;
    const double* m = meas + (size_t)j * 24;
    unsigned cm = 0;
    if (contact) for (int l = 0; l < 4; ++l) cm |= contact[4 * j + l] ? 1u << l : 0u;
    else cm = bp.sched[bp.sched_id[p]].cmask[0];
    double x[24];
    for (int i = 0; i < 12; ++i) x[i] = m[i];
    hkd::hkd_state(m, m + 3, m + 12, cm, x + 12);
    double* x0 = bp.x0 + (size_t)p * 24;
    for (int i = 0; i < 24; ++i) x0[i] = x[i];
}

// FP64 throughput probes (roofline denominators measured on the box)
__global__ void k_dfma_probe(double* out, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
__global__ void k_dmma_probe(double* out, int iters) {
    double c0[2] = {0, 0}, c1[2] = {0, 0}, c2[2] = {0, 0}, c3[2] = {0, 0};
    const double a = 1.0 + threadIdx.x * 1e-6, b = 1.0 - threadIdx.x * 1e-6;
    for (int i = 0; i < iters; ++i) {
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0[0]), "+d"(c0[1]) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c1[0]), "+d"(c1[1]) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c2[0]), "+d"(c2[1]) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c3[0]), "+d"(c3[1]) : "d"(a), "d"(b));
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = c0[0] + c0[1] + c1[0] + c1[1] + c2[0] + c2[1] + c3[0] + c3[1];
}

}  // namespace hsddp

// ===========================================================================
// host side: the C ABI
// ===========================================================================
using namespace hsddp;

static thread_local std::string g_last_error;
const char* hsddp_last_error(void) { return g_last_error.c_str(); }
namespace hsddp { void set_last_error(const std::string& s) { g_last_error = s; } }  // for the other translation units

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            g_last_error = std::string(#call) + ": " + cudaGetErrorString(e_);                     \
            return HSDDP_ERR_CUDA;                                                                 \
        }                                                                                          \
    } while (0)

struct hsddp_batch {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t slots[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    unsigned long long n_solve_launches = 0, n_step_launches = 0;
    int n_sm = 0, blocks_per_sm = 1;
    BatchPtrs bp{};
    std::vector<void*> allocs;
    std::vector<DevSchedule> h_sched;
    std::vector<int> h_sched_id;
    bool has_problems = false;
    int* d_ok = nullptr;
    double* d_darg = nullptr;
    // phased driver (one kernel per solve phase over the running problems)
    int solve_mode = 0;            // 0 auto, 1 persistent k_solve, 2 phased k_phase<...>
    int* d_active[2] = {nullptr, nullptr};
    int* d_count = nullptr;
    // phased driver's backward-sweep kernel, chosen per round on the device: one warp per problem (k_sweep_w1) for rounds of at
    // least kSweepW1Min running problems (full waves: fewer instructions and shared-memory wavefronts per stage), four warps
    // (k_phase<PH_SWEEP>) below (shorter dependent chain per problem when the GPU is not full)
    static constexpr int kSweepW1Min = 1036;  // (about one wave of k_sweep_w1, 148 SMs x 7 when it was set; measured flat between 800 and 2,072, 2 % worse at 3,000)
    // phased driver, rounds of the four-warp sweep: regularisation retries of a problem that regularises run as candidates on
    // sweep_spec blocks side by side (BatchPtrs::spec_list; 0 or 1: one after another on the problem's block).  Scratch per group:
    // kSpecCap x (sweep_spec - 1) slices of max_stages x 312 + 600 doubles (0.55 GB for the benchmark: 4 groups, 60 stages, S = 8).
    // 8 against 4 and off on 16,384 config-3 problems: 58.9-59.0 k, 57.5-57.7 k and 57.0-57.2 k solves/s (profiles/r03b_*)
    int sweep_spec = 8;
    static constexpr int kSpecCap = 128;
    int* d_spec_int = nullptr;     // per group: list [kSpecCap] | arrival counters [kSpecCap] | list counters [2]; then spec_entry [P]
    SpecRec* d_spec_rec = nullptr;
    double* d_spec_out = nullptr;
    size_t d_spec_int_cap = 0, d_spec_rec_cap = 0, d_spec_out_cap = 0;
    bool lr_w1 = true;             // phased driver: linear rollout as its own one-warp-per-problem kernel (k_lr_w1) between sweep and forward
    int* d_order = nullptr;        // persistent kernel: queue order by the previous solve's iteration counts (k_order_by_iterations)
    bool have_order = false;
    // latency kernel with the concurrent line search (k_solve_lat4) for batches of at most kClusterLsMax problems
    static constexpr int kClusterLsMax = 32;  // 4 blocks per problem: every block of every cluster still gets an SM of its own (148 SMs); beyond that the helpers compete with the solving blocks (64 problems: 13.0 ms without, 13.8 ms with)
    static constexpr int kMaxGroups = 4;  // index ranges the phased driver drives concurrently on their own streams (config 3, 16,384 problems, round 2: 1: 381 ms, 2: 354, 4: 336, 8: 341, 16: 354)
    static constexpr int kPhasedMinGroup = 1024;  // smallest index range the phased driver drives on its own stream
    cudaStream_t gstream[kMaxGroups] = {};
    cudaEvent_t gevent[kMaxGroups] = {};
    cudaEvent_t ev_fork = nullptr;
    hsddp_mpc_command* d_cmd = nullptr;  // lives in `allocs` (freed with the problem set)
    // receding-horizon update (problems set through hsddp_batch_set_problems_from_gaits: the gait library is resident in HBM)
    bool mpc_ready = false;
    GaitLib lib{};
    int *d_sched_gait = nullptr, *d_sched_window = nullptr, *d_mpc_err = nullptr;
    MpcSched* d_mpc = nullptr;
    int n_sched = 0;
    bool h_sched_stale = false;
    cudaEvent_t ev_u0 = nullptr, ev_u1 = nullptr;
    int n_gaits = 0;
    // problem restarts (hsddp_batch_restart_problems).  Nothing below is allocated before the first restart.  n_sched counts
    // the schedule SLOTS; a slot is free when no problem uses it (gait -1 on the device, listed in slot_free).
    std::vector<int> slot_refs;    // problems per slot (empty until the first restart)
    std::vector<int> slot_free;    // free slots, marked on the device
    int* d_args = nullptr;         // per-call argument lists of the calls that take problem lists (ints), d_args_cap of them
    double* d_args_x0 = nullptr;
    size_t d_args_cap = 0, d_args_x0_cap = 0;
    int* d_budget = nullptr;       // BatchPtrs::budget
    long long budget_rounds = -1;  // largest max_AL_iter x max_DDP_iter among the pending overrides (-1: none pending)
    std::vector<char> budget_pending;  // [P] the problem's override is still pending (allocated with d_budget)
    int n_budget_pending = 0;
    bool slots_marked = false;     // the slots no problem used are on the free list (done by the first restart)
    // the _dev entry points (buffers in device memory, ordered on the caller's stream): ev_in joins the caller's stream into the
    // handle's at the start of a call, ev_out the handle's stream into the caller's after its last launch
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    // their problem lists go up from pinned host buffers: a pageable source lets cudaMemcpyAsync wait for the handle's stream,
    // which waits for the caller's work.  A buffer is reused once the copy that read it has run (`read`).
    struct PinnedList { int* h = nullptr; size_t cap = 0; cudaEvent_t read = nullptr; };
    std::vector<PinnedList> pinned_lists;
};

namespace {

// No C++ exception may cross the C ABI (std::vector staging buffers can throw bad_alloc: 4.5 GB of dense gains at 16k problems)
template <class F>
int guarded(F&& body) {
    try {
        return body();
    } catch (const std::bad_alloc&) {
        g_last_error = "out of host memory";
        return HSDDP_ERR_ARG;
    } catch (const std::exception& e) {
        g_last_error = std::string("unexpected exception: ") + e.what();
        return HSDDP_ERR_STATE;
    } catch (...) {
        g_last_error = "unexpected exception";
        return HSDDP_ERR_STATE;
    }
}

int dalloc_bytes(hsddp_batch* b, void** p, size_t bytes) {
    void* q = nullptr;
    CK(cudaMalloc(&q, bytes));
    b->allocs.push_back(q);
    *p = q;
    return HSDDP_OK;
}

template <class T>
int dalloc(hsddp_batch* b, T** p, size_t n) { return dalloc_bytes(b, (void**)p, n * sizeof(T)); }

// *d := a new device copy of the n elements at h, kept in `allocs`
template <class T>
int upload(hsddp_batch* b, const T** d, const T* h, size_t n) {
    if (int rc = dalloc(b, d, n)) return rc;
    CK(cudaMemcpy((void*)*d, h, n * sizeof(T), cudaMemcpyHostToDevice));
    return HSDDP_OK;
}

// *p := q in `allocs`; the old allocation (if any) is freed, so nothing may still use it on the device
void replace_alloc(hsddp_batch* b, void** p, void* q) {
    if (*p) {
        for (void*& a : b->allocs)
            if (a == *p) a = q;
        cudaFree(*p);
    } else {
        b->allocs.push_back(q);
    }
    *p = q;
}

// device scratch of at least `n` elements, kept in `allocs` (freed with the problem set)
template <class T>
int scratch(hsddp_batch* b, T** p, size_t* cap, size_t n) {
    if (*cap >= n) return HSDDP_OK;
    void* q = nullptr;
    CK(cudaMalloc(&q, n * sizeof(T)));
    if (*p) CK(cudaStreamSynchronize(b->stream));
    replace_alloc(b, (void**)p, q);
    *cap = n;
    return HSDDP_OK;
}

// Every array of the batch's workspace (DESIGN.md §3.1), from the batch dimensions in b->bp.  alloc_workspace allocates and
// zero-fills each one, k_restart zeroes a restarted problem's part of those marked WS_RESTART, and the C ABI's stored views
// (hsddp_batch_get_array / _rows / set_array) are the entries with an HSDDP_ARR_* id.  Budget and command buffers are
// allocated lazily elsewhere, so batches that never restart or read commands do not pay for them.
enum : unsigned {
    WS_SET = 1,      // hsddp_batch_set_array may overwrite it
    WS_RESTART = 2,  // k_restart zeroes it (every array a solve reads that the restart does not write itself)
    WS_SMALL = 4,    // only for n_problems <= kClusterLsMax: trial arrays of the concurrent line search, four per problem
    WS_BATCH = 8,    // one per batch, not per problem
};
struct WsArray {
    void** field;      // the BatchPtrs / handle member it fills
    size_t rows, row_bytes;  // per problem (per batch: WS_BATCH); a C ABI row is row_bytes / 8 doubles
    int abi;           // HSDDP_ARR_* id of the stored view, -1: none
    unsigned flags;
    size_t bytes() const { return rows * row_bytes; }
};

std::vector<WsArray> workspace_arrays(hsddp_batch* b) {
    BatchPtrs& bp = b->bp;
    const size_t S = bp.max_nodes, N = bp.max_stages, D = sizeof(double), I = sizeof(int);
    return {
        {(void**)&bp.x0, 1, 24 * D, -1, 0},
        {(void**)&bp.Xbar, S, 24 * D, HSDDP_ARR_XBAR, WS_SET | WS_RESTART},
        {(void**)&bp.X, S, 24 * D, HSDDP_ARR_X, WS_SET | WS_RESTART},
        {(void**)&bp.Xsim_t, S, 24 * D, -1, WS_RESTART},
        {(void**)&bp.Defect, S, 24 * D, HSDDP_ARR_DEFECT, WS_RESTART},
        {(void**)&bp.dX, S, 24 * D, HSDDP_ARR_DX, WS_SET | WS_RESTART},
        {(void**)&bp.Ubar, N, 24 * D, HSDDP_ARR_UBAR, WS_SET | WS_RESTART},
        {(void**)&bp.U, N, 24 * D, HSDDP_ARR_U, WS_SET | WS_RESTART},
        {(void**)&bp.U_t, N, 24 * D, -1, WS_RESTART},
        {(void**)&bp.dU, N, 24 * D, HSDDP_ARR_DU, WS_SET | WS_RESTART},
        {(void**)&bp.KdX, N, 12 * D, -1, WS_RESTART},
        {(void**)&bp.K, N, 288 * D, -1, WS_RESTART},  // (HSDDP_ARR_K is the dense view, get_gains)
        {(void**)&bp.lq, N, CR_STRIDE * D, -1, WS_RESTART},
        {(void**)&bp.tq, MAXPH, TQ_STRIDE * D, -1, WS_RESTART},
        {(void**)&bp.gcon, N, 20 * D, HSDDP_ARR_GCON, WS_RESTART},
        {(void**)&bp.reb, N, 40 * D, HSDDP_ARR_REB, WS_RESTART},
        {(void**)&bp.hcon, MAXPH, 4 * D, HSDDP_ARR_HCON, WS_RESTART},
        {(void**)&bp.al, MAXPH, 16 * D, HSDDP_ARR_AL, WS_RESTART},
        {(void**)&bp.g0h0, 1, 600 * D, -1, WS_RESTART},  // (HSDDP_ARR_G0 / H0 are strided views of it)
        {(void**)&bp.state, 1, sizeof(SolverState), -1, 0},
        {(void**)&bp.ctl, 1, sizeof(SolveCtl), -1, 0},
        {(void**)&b->d_active[0], 1, I, -1, 0},
        {(void**)&b->d_active[1], 1, I, -1, 0},
        {(void**)&b->d_order, 1, I, -1, 0},
        {(void**)&bp.ls_X, 4 * S, 24 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_Defect, 4 * S, 24 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_Xsim, 4 * S, 24 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_U, 4 * N, 24 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_Ut, 4 * N, 24 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_gcon, 4 * N, 20 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_hcon, 4 * MAXPH, 4 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_res, 4, 8 * D, -1, WS_SMALL | WS_RESTART},
        {(void**)&bp.ls_mail, 1, I, -1, WS_SMALL | WS_RESTART},
        {(void**)&b->d_count, 2 * hsddp_batch::kMaxGroups, I, -1, WS_BATCH},
        {(void**)&bp.info, 1, sizeof(hsddp_info), -1, 0},
        {(void**)&bp.trace, HSDDP_TRACE_CAP, sizeof(hsddp_iter_record), -1, WS_RESTART},
        {(void**)&bp.counters, 32, sizeof(unsigned long long), -1, WS_BATCH},
        {(void**)&bp.work_counter, 4, I, -1, WS_BATCH},
        {(void**)&bp.sm_slots, 256, I, -1, WS_BATCH},
        {(void**)&b->d_ok, 1, I, -1, 0},
        {(void**)&b->d_darg, 1, D, -1, 0},
    };
}

// the table entry of stored view `which` of the C ABI
bool stored_array(hsddp_batch* b, int which, WsArray* out) {
    if (which < 0) return false;
    for (const WsArray& a : workspace_arrays(b))
        if (a.abi == which) { *out = a; return true; }
    return false;
}

// The schedule-slot storage of a batch built from gaits: per slot its phase table, update state, gait / window and
// node_stride reference rows (slot s owns rows [s * node_stride, (s + 1) * node_stride), so ref_off survives a growth).
struct SlotArray { void** field; size_t bytes; };

std::vector<SlotArray> slot_arrays(hsddp_batch* b) {
    BatchPtrs& bp = b->bp;
    const size_t rows = (size_t)b->lib.node_stride, D = sizeof(double);
    return {
        {(void**)&bp.sched, sizeof(DevSchedule)}, {(void**)&b->d_mpc, sizeof(MpcSched)},
        {(void**)&b->d_sched_gait, sizeof(int)}, {(void**)&b->d_sched_window, sizeof(int)},
        {(void**)&bp.xr, 24 * rows * D}, {(void**)&bp.ur, 24 * rows * D}, {(void**)&bp.prel, 12 * rows * D}, {(void**)&bp.xinit, 24 * rows * D},
    };
}

void free_problem_allocs(hsddp_batch* b) {
    for (void* p : b->allocs) cudaFree(p);
    b->allocs.clear();
    b->d_cmd = nullptr;
    b->has_problems = false;
    b->mpc_ready = false;
    b->h_sched_stale = false;
    b->slot_refs.clear(); b->slot_free.clear();
    b->d_args = nullptr; b->d_args_x0 = nullptr; b->d_args_cap = b->d_args_x0_cap = 0;
    b->d_budget = nullptr; b->budget_rounds = -1; b->budget_pending.clear(); b->n_budget_pending = 0;
    b->d_spec_int = nullptr; b->d_spec_rec = nullptr; b->d_spec_out = nullptr; b->d_spec_int_cap = b->d_spec_rec_cap = b->d_spec_out_cap = 0;
    b->slots_marked = false;
}

hsddp_options default_options() {
    hsddp_options o;
    std::memset(&o, 0, sizeof o);
    o.alpha = 0.1; o.gamma = 0.01; o.update_penalty = 5; o.update_relax = 1; o.update_regularization = 2; o.update_ReB = 1;
    o.max_DDP_iter = 10; o.max_AL_iter = 5; o.cost_thresh = 1e-3; o.tconstr_thresh = 1e-3; o.pconstr_thresh = 1e-3;
    o.dynamics_feas_thresh = 1e-3; o.merit_scale = 0.2; o.merit_offset = 1e2; o.AL_active = 1; o.ReB_active = 1; o.MS = 1;
    return o;
}

hsddp_constraint_params default_constraint_params() {
    hsddp_constraint_params cp;
    std::memset(&cp, 0, sizeof cp);
    cp.grf_delta = 0.1; cp.grf_delta_min = 0.1; cp.grf_eps = 0.1; cp.td_sigma = 50; cp.td_sigma_max = 1e4; cp.td_lambda = 0; cp.mu = 0.7;
    return cp;
}

// the iteration budget rules of check_opt
const char* check_budget(int max_AL_iter, int max_DDP_iter) {
    if (max_DDP_iter < 0 || max_AL_iter < 0) return "max_DDP_iter / max_AL_iter must be >= 0";
    if ((long long)max_DDP_iter * (long long)max_AL_iter > 1000000LL) return "max_DDP_iter x max_AL_iter exceeds 1e6";
    return nullptr;
}

int check_opt(const hsddp_options* opt) {
    if (!opt) return HSDDP_OK;
    // The reference's loops `while (eps > 1e-3) eps *= alpha` (MultiPhaseDDP.cpp:113,132) and `reg = max(reg * update_regularization,
    // 1e-3)` until PD or reg > 1e2 (:159-167) terminate only for 0 < alpha < 1 and update_regularization > 1.  On the host a
    // bad value spins one thread; on the device it would hang the stream, so such options are refused here.
    auto fin = [](double v) { return v == v && v - v == 0.0; };
    const char* bad = nullptr;
    if (!(opt->alpha > 0.0 && opt->alpha < 1.0)) bad = "alpha must be in (0, 1)";
    else if (!(opt->update_regularization > 1.0) || !fin(opt->update_regularization)) bad = "update_regularization must be finite and > 1";
    else if (!fin(opt->gamma) || !fin(opt->update_penalty) || !fin(opt->update_relax) || !fin(opt->update_ReB)) bad = "gamma / update_penalty / update_relax / update_ReB must be finite";
    else if (!fin(opt->cost_thresh) || !fin(opt->tconstr_thresh) || !fin(opt->pconstr_thresh) || !fin(opt->dynamics_feas_thresh)) bad = "thresholds must be finite";
    else if (!fin(opt->merit_scale) || opt->merit_scale == 1.0 || !fin(opt->merit_offset)) bad = "merit_scale must be finite and != 1, merit_offset finite";
    else bad = check_budget(opt->max_AL_iter, opt->max_DDP_iter);
    if (bad) { g_last_error = std::string("invalid hsddp_options: ") + bad; return HSDDP_ERR_ARG; }
    return HSDDP_OK;
}

int launch_step(hsddp_batch* b, const hsddp_options* opt, int op, double arg, double* darg_dev, int32_t* ok_host, bool sync = true) {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_STATE; }
    int rc = check_opt(opt);
    if (rc) return rc;
    CK(cudaSetDevice(b->device));
    const hsddp_options o = opt ? *opt : default_options();
    k_step<<<b->bp.n_problems, kThreads, 0, b->stream>>>(b->bp, o, op, arg, darg_dev, b->d_ok);
    CK(cudaGetLastError());
    b->n_step_launches++;
    if (ok_host) CK(cudaMemcpyAsync(ok_host, b->d_ok, sizeof(int) * b->bp.n_problems, cudaMemcpyDeviceToHost, b->stream));
    if (sync || ok_host) CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
}

}  // namespace

extern "C" {

static int batch_init(hsddp_batch* b, int device) {
    CK(cudaSetDevice(device));
    b->device = device;
    CK(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&b->ev0));
    CK(cudaEventCreate(&b->ev1));
    CK(cudaEventCreate(&b->ev_u0));
    CK(cudaEventCreate(&b->ev_u1));
    for (int i = 0; i < 8; ++i) CK(cudaEventCreate(&b->slots[i]));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    b->n_sm = prop.multiProcessorCount;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b->blocks_per_sm, k_solve, kThreads, 0));
    if (b->blocks_per_sm < 1) b->blocks_per_sm = 1;
    CK(cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&b->ev_in, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&b->ev_out, cudaEventDisableTiming));
    CK(cudaFuncSetAttribute(k_sweep_w1, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    CK(cudaFuncSetAttribute(k_lr_w1, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    if (const char* e = getenv("HSDDP_SWEEP_SPEC")) { const int v = atoi(e); b->sweep_spec = (v >= 2 && v <= 32) ? v : 0; }
    if (const char* e = getenv("HSDDP_LR_W1")) b->lr_w1 = atoi(e) != 0;              // tuning / experiments only
    return HSDDP_OK;
}

int hsddp_batch_create(int device, hsddp_batch** out) {
    if (!out) return HSDDP_ERR_ARG;
    *out = nullptr;
    int n = 0;
    CK(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) { g_last_error = "no such CUDA device (this library has no CPU fallback)"; return HSDDP_ERR_CUDA; }
    return guarded([&]() -> int {
        hsddp_batch* b = new hsddp_batch();
        const int rc = batch_init(b, device);
        if (rc != HSDDP_OK) { hsddp_batch_destroy(b); return rc; }  // (streams / events created so far are released)
        *out = b;
        return HSDDP_OK;
    });
}

int hsddp_batch_destroy(hsddp_batch* b) {
    if (!b) return HSDDP_OK;
    cudaSetDevice(b->device);
    free_problem_allocs(b);
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    if (b->ev_u0) cudaEventDestroy(b->ev_u0);
    if (b->ev_u1) cudaEventDestroy(b->ev_u1);
    for (int i = 0; i < 8; ++i) if (b->slots[i]) cudaEventDestroy(b->slots[i]);
    if (b->stream) cudaStreamDestroy(b->stream);
    if (b->ev_fork) cudaEventDestroy(b->ev_fork);
    if (b->ev_in) cudaEventDestroy(b->ev_in);
    if (b->ev_out) cudaEventDestroy(b->ev_out);
    for (auto& s : b->pinned_lists) {
        if (s.read) cudaEventDestroy(s.read);
        if (s.h) cudaFreeHost(s.h);
    }
    for (int g = 0; g < hsddp_batch::kMaxGroups; ++g) {
        if (b->gevent[g]) cudaEventDestroy(b->gevent[g]);
        if (b->gstream[g]) cudaStreamDestroy(b->gstream[g]);
    }
    delete b;
    return HSDDP_OK;
}

// the workspace (workspace_arrays), zero-filled; bp.n_problems / max_stages / max_nodes are set by the caller
static int alloc_workspace(hsddp_batch* b) {
    const size_t P = (size_t)b->bp.n_problems;
    for (const WsArray& a : workspace_arrays(b)) {
        if ((a.flags & WS_SMALL) && P > (size_t)hsddp_batch::kClusterLsMax) continue;
        const size_t bytes = a.bytes() * ((a.flags & WS_BATCH) ? 1 : P);
        if (int rc = dalloc_bytes(b, a.field, bytes)) return rc;
        CK(cudaMemsetAsync(*a.field, 0, bytes, b->stream));
    }
    b->have_order = false;
    return HSDDP_OK;
}

// first step of both ways to set the problems: schedule_id checked and kept (host and device), bp cleared and given the
// constraint parameters
static int begin_problem_set(hsddp_batch* b, int n_schedules, int n_problems, const int32_t* schedule_id, const hsddp_constraint_params* cparams) {
    for (int i = 0; i < n_problems; ++i)
        if (schedule_id[i] < 0 || schedule_id[i] >= n_schedules) { g_last_error = "schedule_id out of range"; return HSDDP_ERR_ARG; }
    b->h_sched_id.assign(schedule_id, schedule_id + n_problems);
    BatchPtrs& bp = b->bp;
    std::memset(&bp, 0, sizeof bp);
    bp.n_problems = n_problems;
    bp.cp = cparams ? *cparams : default_constraint_params();
    return upload(b, &bp.sched_id, schedule_id, (size_t)n_problems);
}

// last step of both: the workspace for these row counts, then the batch reset
static int finish_problem_set(hsddp_batch* b, int max_stages, int max_nodes) {
    b->bp.max_stages = max_stages; b->bp.max_nodes = max_nodes;
    if (int rc = alloc_workspace(b)) return rc;
    b->has_problems = true;
    return hsddp_batch_reset(b);
}

int hsddp_batch_set_problems(hsddp_batch* b, int n_schedules, const hsddp_schedule* schedules, int n_problems,
                             const int32_t* schedule_id, const hsddp_constraint_params* cparams) {
    return guarded([&]() -> int {
    if (!b || n_schedules <= 0 || !schedules || n_problems <= 0 || !schedule_id) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    free_problem_allocs(b);
    // flatten schedules
    b->h_sched.assign(n_schedules, DevSchedule{});
    size_t total_nodes = 0;
    int max_stages = 0, max_nodes = 0;
    for (int i = 0; i < n_schedules; ++i) {
        const hsddp_schedule& s = schedules[i];
        if (s.n_phases < 1 || s.n_phases > MAXPH || s.n_stages > HSDDP_MAX_STAGES || !s.xr || !s.ur || !s.prel_r || !s.xinit) {
            g_last_error = "invalid schedule";
            return HSDDP_ERR_ARG;
        }
        DevSchedule& d = b->h_sched[i];
        d.dt = s.dt; d.ref_off = (long long)total_nodes;
        for (int p = 0; p < s.n_phases; ++p) {
            if (s.horizon[p] < 1) { g_last_error = "phase with empty horizon"; return HSDDP_ERR_ARG; }
            d.horizon[p] = s.horizon[p];
            unsigned cm = 0, nm = 0;
            for (int l = 0; l < 4; ++l) { cm |= (s.contact[p][l] ? 1u : 0u) << l; nm |= (s.next_contact[p][l] ? 1u : 0u) << l; }
            d.cmask[p] = cm; d.nmask[p] = nm;
            d.ss_size[p] = (unsigned char)(s.horizon[p] + 1);
            d.tdmask[0][p] = (unsigned char)touchdown_legs(cm, nm); d.tdmask[1][p] = 0;
        }
        if (!layout_phases(d, s.n_phases, HSDDP_MAX_STAGES, HSDDP_MAX_STAGES + MAXPH) || d.n_nodes != s.n_nodes || d.n_stages != s.n_stages) {
            g_last_error = "schedule node/stage counts inconsistent";
            return HSDDP_ERR_ARG;
        }
        total_nodes += (size_t)s.n_nodes;
        max_stages = std::max(max_stages, s.n_stages);
        max_nodes = std::max(max_nodes, s.n_nodes);
    }
    int rc;
    if ((rc = begin_problem_set(b, n_schedules, n_problems, schedule_id, cparams))) return rc;

    std::vector<double> xr(total_nodes * 24), ur(total_nodes * 24), prel(total_nodes * 12), xinit(total_nodes * 24);
    for (int i = 0; i < n_schedules; ++i) {
        const hsddp_schedule& s = schedules[i];
        const size_t o = (size_t)b->h_sched[i].ref_off, nn = (size_t)s.n_nodes;
        std::memcpy(&xr[o * 24], s.xr, nn * 24 * sizeof(double));
        std::memcpy(&ur[o * 24], s.ur, nn * 24 * sizeof(double));
        std::memcpy(&prel[o * 12], s.prel_r, nn * 12 * sizeof(double));
        std::memcpy(&xinit[o * 24], s.xinit, nn * 24 * sizeof(double));
    }
    BatchPtrs& bp = b->bp;
    if ((rc = upload(b, &bp.sched, (const DevSchedule*)b->h_sched.data(), (size_t)n_schedules)) || (rc = upload(b, &bp.xr, xr.data(), xr.size())) ||
        (rc = upload(b, &bp.ur, ur.data(), ur.size())) || (rc = upload(b, &bp.prel, prel.data(), prel.size())) ||
        (rc = upload(b, &bp.xinit, xinit.data(), xinit.size())))
        return rc;
    return finish_problem_set(b, max_stages, max_nodes);
    });
}

// builds schedule slot slot[i] (nullptr: slot i) from gait[i] and window[i] for i < n: phase table, update state, reference
// rows.  status[i] != 0: the window does not fit the gait table (1) or the schedule exceeds the table limits (2).
static void launch_schedule_build(hsddp_batch* b, int n, const int* gait, const int* window, const int* slot, int stage_cap, int* status) {
    DevSchedule* sched = const_cast<DevSchedule*>(b->bp.sched);
    k_build_phase_tables<<<(n + 127) / 128, 128, 0, b->stream>>>(b->lib, n, gait, window, slot, stage_cap, sched, b->d_mpc, status);
    k_reference_rows<<<n, 128, 0, b->stream>>>(b->lib, n, gait, window, slot, sched, b->d_mpc, const_cast<double*>(b->bp.xr),
                                               const_cast<double*>(b->bp.ur), const_cast<double*>(b->bp.prel), const_cast<double*>(b->bp.xinit));
    b->n_step_launches += 2;
}

int hsddp_batch_set_problems_from_gaits(hsddp_batch* b, int n_gaits, const int32_t* gait_rows, const float* gait_dt,
                                        const double* body_state, const double* qJ, const double* foot_placements, const double* grf,
                                        const int32_t* contact, int n_schedules, const int32_t* sched_gait, const int32_t* sched_window,
                                        float plan_duration, int n_problems, const int32_t* schedule_id, const hsddp_constraint_params* cparams) {
    return guarded([&]() -> int {
    if (!b || n_gaits <= 0 || !gait_rows || !gait_dt || !body_state || !qJ || !foot_placements || !grf || !contact || n_schedules <= 0 ||
        !sched_gait || !sched_window || n_problems <= 0 || !schedule_id || !(plan_duration > 0.f))
        return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    free_problem_allocs(b);
    for (int i = 0; i < n_schedules; ++i)
        if (sched_gait[i] < 0 || sched_gait[i] >= n_gaits) { g_last_error = "sched_gait out of range"; return HSDDP_ERR_ARG; }
    int rc;
    if ((rc = begin_problem_set(b, n_schedules, n_problems, schedule_id, cparams))) return rc;
    // gait library -> HBM
    std::vector<int> row_off(n_gaits);
    size_t rows = 0;
    for (int g = 0; g < n_gaits; ++g) { row_off[g] = (int)rows; rows += (size_t)gait_rows[g]; }
    GaitLib& lib = b->lib;
    if ((rc = upload(b, &lib.body_state, body_state, rows * 12)) || (rc = upload(b, &lib.qJ, qJ, rows * 12)) ||
        (rc = upload(b, &lib.foot, foot_placements, rows * 12)) || (rc = upload(b, &lib.grf, grf, rows * 12)) ||
        (rc = upload(b, &lib.contact, contact, rows * 4)) || (rc = upload(b, &lib.row_off, row_off.data(), (size_t)n_gaits)) ||
        (rc = upload(b, &lib.n_rows, gait_rows, (size_t)n_gaits)) || (rc = upload(b, &lib.dt, gait_dt, (size_t)n_gaits)))
        return rc;
    lib.plan = plan_duration;
    lib.node_stride = std::min(HSDDP_MAX_STAGES, (int)std::lround(plan_duration / kTickDt) + 1) + MAXPH;
    for (const SlotArray& a : slot_arrays(b)) {  // one schedule slot per schedule
        if ((rc = dalloc_bytes(b, a.field, (size_t)n_schedules * a.bytes))) return rc;
        // zero-filled as grow_slots fills new slots: an update adds node rows it does not write (xinit), and those must read
        // back the same in every handle whatever the allocation held before (gait and window are copied in below)
        if (a.field != (void**)&b->d_sched_gait && a.field != (void**)&b->d_sched_window)
            CK(cudaMemsetAsync(*a.field, 0, (size_t)n_schedules * a.bytes, b->stream));
    }
    int *d_status, *d_err;
    if ((rc = dalloc(b, &d_status, (size_t)n_schedules)) || (rc = dalloc(b, &d_err, (size_t)4))) return rc;
    CK(cudaMemcpy(b->d_sched_gait, sched_gait, n_schedules * sizeof(int), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_sched_window, sched_window, n_schedules * sizeof(int), cudaMemcpyHostToDevice));
    CK(cudaMemsetAsync(d_err, 0, 4 * sizeof(int), b->stream));
    launch_schedule_build(b, n_schedules, b->d_sched_gait, b->d_sched_window, nullptr, HSDDP_MAX_STAGES, d_status);
    CK(cudaGetLastError());
    // the host keeps the phase tables too (dense gain / Jacobian getters, workspace sizing)
    b->h_sched.assign(n_schedules, DevSchedule{});
    std::vector<int> status(n_schedules);
    CK(cudaMemcpyAsync(b->h_sched.data(), b->bp.sched, sizeof(DevSchedule) * n_schedules, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(status.data(), d_status, sizeof(int) * n_schedules, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    int max_stages = 0;
    for (int i = 0; i < n_schedules; ++i) {
        if (status[i]) { g_last_error = status[i] == 1 ? "window does not fit the gait table" : "schedule exceeds HSDDP_MAX_PHASES / HSDDP_MAX_STAGES"; free_problem_allocs(b); return status[i] == 1 ? HSDDP_ERR_ARG : HSDDP_ERR_UNSUPPORTED; }
        max_stages = std::max(max_stages, b->h_sched[i].n_stages);
    }
    b->d_mpc_err = d_err; b->n_sched = n_schedules; b->n_gaits = n_gaits; b->mpc_ready = true;
    // (node rows with headroom: a receding-horizon update can add phases, i.e. nodes, while the stage count stays the same)
    return finish_problem_set(b, max_stages, std::min(lib.node_stride, max_stages + MAXPH));
    });
}

/* HKDProblem::update for every problem of the batch (see the kernels above).  The solver state that the reference keeps
 * across MPC steps stays in the handle: nominal trajectories, gains, ReB / AL parameters. */
int hsddp_batch_mpc_update(hsddp_batch* b) {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_STATE; }
    if (!b->mpc_ready) { g_last_error = "hsddp_batch_mpc_update needs the gait library on the device: set the problems with hsddp_batch_set_problems_from_gaits"; return HSDDP_ERR_STATE; }
    CK(cudaSetDevice(b->device));
    CK(cudaEventRecord(b->ev_u0, b->stream));
    DevSchedule* d_sched = const_cast<DevSchedule*>(b->bp.sched);
    k_mpc_update_schedules<<<(b->n_sched + 127) / 128, 128, 0, b->stream>>>(b->lib, b->n_sched, b->d_sched_gait, b->d_sched_window, nullptr, d_sched,
                                                                              b->d_mpc, b->d_mpc_err);
    k_reference_rows<<<b->n_sched, 128, 0, b->stream>>>(b->lib, b->n_sched, b->d_sched_gait, b->d_sched_window, nullptr, d_sched, b->d_mpc,
                                                        const_cast<double*>(b->bp.xr), const_cast<double*>(b->bp.ur), const_cast<double*>(b->bp.prel), nullptr);
    k_mpc_shift<<<b->bp.n_problems, kThreads, 0, b->stream>>>(b->bp, b->d_mpc, SlotMoves{});
    CK(cudaGetLastError());
    b->n_step_launches += 3;
    CK(cudaEventRecord(b->ev_u1, b->stream));
    int err = 0;
    CK(cudaMemcpyAsync(&err, b->d_mpc_err, sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    b->h_sched_stale = true;
    b->have_order = false;  // (the queue order of the previous problem layout is still a good hint, but the solve after a tick is 2 iterations long)
    if (err) {
        g_last_error = err == 1 ? "receding-horizon update: the reference table is exhausted" : "receding-horizon update: schedule exceeds HSDDP_MAX_PHASES / node capacity";
        return err == 1 ? HSDDP_ERR_ARG : HSDDP_ERR_UNSUPPORTED;
    }
    return HSDDP_OK;
}

int hsddp_batch_last_update_ms(hsddp_batch* b, float* ms) {
    if (!b || !ms) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaEventSynchronize(b->ev_u1));
    CK(cudaEventElapsedTime(ms, b->ev_u0, b->ev_u1));
    return HSDDP_OK;
}

// the host copy of the phase tables (dense gain / Jacobian getters) after a receding-horizon update
static int refresh_host_schedules(hsddp_batch* b) {
    if (!b->h_sched_stale) return HSDDP_OK;
    CK(cudaMemcpy(b->h_sched.data(), b->bp.sched, sizeof(DevSchedule) * b->h_sched.size(), cudaMemcpyDeviceToHost));
    b->h_sched_stale = false;
    return HSDDP_OK;
}

/* device-built schedule i back on the host (tests): phase table + reference rows, row counts as in hsddp_schedule */
int hsddp_batch_get_schedule(hsddp_batch* b, int i, int32_t* n_phases, int32_t* horizon, int32_t* contact, int32_t* next_contact,
                             double* xr, double* ur, double* prel_r, double* xinit) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems || i < 0 || i >= (int)b->h_sched.size()) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    DevSchedule d;
    CK(cudaMemcpy(&d, b->bp.sched + i, sizeof d, cudaMemcpyDeviceToHost));
    if (n_phases) *n_phases = d.n_phases;
    for (int p = 0; p < d.n_phases; ++p) {
        if (horizon) horizon[p] = d.horizon[p];
        for (int l = 0; l < 4; ++l) {
            if (contact) contact[4 * p + l] = (d.cmask[p] >> l) & 1u;
            if (next_contact) next_contact[4 * p + l] = (d.nmask[p] >> l) & 1u;
        }
    }
    const size_t o = (size_t)d.ref_off, nn = (size_t)d.n_nodes;
    if (xr) CK(cudaMemcpy(xr, b->bp.xr + o * 24, nn * 24 * sizeof(double), cudaMemcpyDeviceToHost));
    if (ur) CK(cudaMemcpy(ur, b->bp.ur + o * 24, nn * 24 * sizeof(double), cudaMemcpyDeviceToHost));
    if (prel_r) CK(cudaMemcpy(prel_r, b->bp.prel + o * 12, nn * 12 * sizeof(double), cudaMemcpyDeviceToHost));
    if (xinit) CK(cudaMemcpy(xinit, b->bp.xinit + o * 24, nn * 24 * sizeof(double), cudaMemcpyDeviceToHost));
    return HSDDP_OK;
    });
}

// `add` more schedule slots: the slot arrays are reallocated and the existing slots copied device to device (ref_off stays
// valid: slot s keeps reference rows [s * node_stride, (s + 1) * node_stride)).  The new slots are free.
static int grow_slots(hsddp_batch* b, int add) {
    const size_t cap = (size_t)b->n_sched, ncap = cap + (size_t)add;
    const std::vector<SlotArray> arrays = slot_arrays(b);
    std::vector<void*> nw(arrays.size(), nullptr);
    for (size_t a = 0; a < arrays.size(); ++a) {
        const cudaError_t e = cudaMalloc(&nw[a], ncap * arrays[a].bytes);
        if (e != cudaSuccess) {
            for (void* q : nw) cudaFree(q);
            g_last_error = std::string("growing the schedule slots: ") + cudaGetErrorString(e);
            return HSDDP_ERR_CUDA;
        }
    }
    for (size_t a = 0; a < arrays.size(); ++a) {
        const size_t bytes = arrays[a].bytes;
        const int fill = arrays[a].field == (void**)&b->d_sched_gait ? 0xff : 0;  // (gait -1: free)
        CK(cudaMemcpyAsync(nw[a], *arrays[a].field, cap * bytes, cudaMemcpyDeviceToDevice, b->stream));
        CK(cudaMemsetAsync((char*)nw[a] + cap * bytes, fill, (ncap - cap) * bytes, b->stream));
    }
    CK(cudaStreamSynchronize(b->stream));
    for (size_t a = 0; a < arrays.size(); ++a) replace_alloc(b, arrays[a].field, nw[a]);
    b->n_sched = (int)ncap;
    b->slot_refs.resize(ncap, 0);
    b->h_sched.resize(ncap);
    b->h_sched_stale = true;
    for (size_t s = ncap; s-- > cap;) b->slot_free.push_back((int)s);  // (taken from the back: lowest index first)
    return HSDDP_OK;
}

// a host list of n distinct problem indices, 1 <= n <= n_problems
static int check_problem_list(hsddp_batch* b, int n, const int32_t* problem, const char* what) {
    const int P = b->bp.n_problems;
    if (n <= 0 || n > P || !problem) { g_last_error = std::string(what) + ": n must be in [1, n_problems] and the list given"; return HSDDP_ERR_ARG; }
    std::vector<char> seen(P, 0);
    for (int k = 0; k < n; ++k) {
        if (problem[k] < 0 || problem[k] >= P) { g_last_error = std::string(what) + ": problem index out of range"; return HSDDP_ERR_ARG; }
        if (seen[problem[k]]) { g_last_error = std::string(what) + ": repeated problem index"; return HSDDP_ERR_ARG; }
        seen[problem[k]] = 1;
    }
    return HSDDP_OK;
}

// *d := the host ints h in the call's device argument list (queued on the handle's stream)
static int stage_ints(hsddp_batch* b, const std::vector<int>& h, int** d) {
    if (int rc = scratch(b, &b->d_args, &b->d_args_cap, h.size())) return rc;
    CK(cudaMemcpyAsync(b->d_args, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, b->stream));
    *d = b->d_args;
    return HSDDP_OK;
}

// A call that moves the n listed problems to m new schedule slots (restart, per-problem update) plans the move before it builds
// anything and commits it only once the build has succeeded (commit_slot_moves here, write_slot_moves on the device), so a
// refused call leaves the slots as they were.  Listed problem k goes to the call's new slot entry[k] < m.
struct SlotPlan {
    std::vector<int> slot;              // [n] new slot of listed problem k
    std::vector<int> target;            // [m] the new slots, taken from the free list
    std::vector<int> freed;             // slots the call leaves without a problem
    std::vector<int> refs, free_after;  // slot_refs and slot_free (without the freed slots) after the call
};

static int plan_slot_moves(hsddp_batch* b, int n, const int32_t* problem, const std::vector<int>& entry, int m, SlotPlan* p) {
    if (b->slot_refs.empty()) {  // problems per slot, counted by the first such call
        b->slot_refs.assign(b->n_sched, 0);
        for (int s : b->h_sched_id) b->slot_refs[s]++;
    }
    // at least m free slots: grow by half the capacity at least (a growth copies every slot), but never beyond the n_problems + n
    // slots a call can need (at most n_problems are referenced, plus the m <= n being built)
    const int need = m - (int)b->slot_free.size();
    if (need > 0)
        if (int rc = grow_slots(b, std::max(need, std::min(b->n_sched / 2, b->bp.n_problems + n - b->n_sched)))) return rc;
    p->refs = b->slot_refs; p->free_after = b->slot_free;
    p->target.resize(m); p->slot.resize(n);
    for (int j = 0; j < m; ++j) { p->target[j] = p->free_after.back(); p->free_after.pop_back(); }
    for (int k = 0; k < n; ++k) { p->slot[k] = p->target[entry[k]]; p->refs[b->h_sched_id[problem[k]]]--; p->refs[p->slot[k]]++; }
    // freed: old slots of the listed problems that no problem uses any more (at the first such call: every unused slot)
    std::vector<char> on_free(b->n_sched, 0);
    for (int s : p->free_after) on_free[s] = 1;
    auto release = [&](int s) { if (p->refs[s] == 0 && !on_free[s]) { on_free[s] = 1; p->freed.push_back(s); } };
    if (!b->slots_marked) for (int s = 0; s < b->n_sched; ++s) release(s);
    else for (int k = 0; k < n; ++k) release(b->h_sched_id[problem[k]]);
    return HSDDP_OK;
}

static void commit_slot_moves(hsddp_batch* b, SlotPlan& p, int n, const int32_t* problem) {
    b->slot_refs.swap(p.refs);
    for (int s : p.freed) p.free_after.push_back(s);
    b->slot_free.swap(p.free_after);
    for (int k = 0; k < n; ++k) b->h_sched_id[problem[k]] = p.slot[k];
    b->h_sched_stale = true;
    b->slots_marked = true;
}

// the device list of a slot move, problem[n] slot[n] | target[m] gait[m] window[m] | freed[f], then the caller's `tail` (*d_tail)
static int stage_slot_moves(hsddp_batch* b, const SlotPlan& p, int n, const int32_t* problem, const std::vector<int>& gait,
                            const std::vector<int>& window, const std::vector<int>& tail, SlotMoves* mv, int** d_tail) {
    std::vector<int> h(problem, problem + n);
    for (const std::vector<int>* v : {&p.slot, &p.target, &gait, &window, &p.freed, &tail}) h.insert(h.end(), v->begin(), v->end());
    int* d;
    if (int rc = stage_ints(b, h, &d)) return rc;
    const int m = (int)p.target.size(), f = (int)p.freed.size();
    *mv = SlotMoves{d, d + n, d + 2 * n, d + 2 * n + m, d + 2 * n + 2 * m, d + 2 * n + 3 * m, m, f, b->d_sched_gait, b->d_sched_window};
    *d_tail = d + 2 * n + 3 * m + f;
    return HSDDP_OK;
}

// k_scatter_rows on the handle's stream: row idx[j] of dst := row j of src (src_stride 0: one row for all), for j < n
static int scatter_rows(hsddp_batch* b, void* dst, int words, const int* idx, const void* src, int src_stride, int n) {
    const long long total = (long long)n * words;
    k_scatter_rows<<<(unsigned)((total + 255) / 256), 256, 0, b->stream>>>((unsigned*)dst, words, idx, (const unsigned*)src, src_stride, n);
    CK(cudaGetLastError());
    b->n_step_launches++;
    return HSDDP_OK;
}

int hsddp_batch_restart_problems(hsddp_batch* b, int n, const int32_t* problem, const int32_t* gait, const int32_t* window,
                                 const double* x0, const hsddp_options* first_solve) {
    return guarded([&]() -> int {
    if (!b) return HSDDP_ERR_ARG;
    if (!b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_STATE; }
    if (!b->mpc_ready) { g_last_error = "hsddp_batch_restart_problems needs the gait library on the device: set the problems with hsddp_batch_set_problems_from_gaits"; return HSDDP_ERR_STATE; }
    const int P = b->bp.n_problems;
    int rc;
    if ((rc = check_problem_list(b, n, problem, "restart"))) return rc;
    if (!gait || !window || !x0) { g_last_error = "restart: gait, window and x0 must be given"; return HSDDP_ERR_ARG; }
    if (first_solve)
        if (const char* bad = check_budget(first_solve->max_AL_iter, first_solve->max_DDP_iter)) { g_last_error = std::string("invalid first_solve: ") + bad; return HSDDP_ERR_ARG; }
    for (int k = 0; k < n; ++k) {
        if (gait[k] < 0 || gait[k] >= b->n_gaits) { g_last_error = "restart: unknown gait"; return HSDDP_ERR_ARG; }
        if (window[k] < 0) { g_last_error = "restart: window does not fit the gait table"; return HSDDP_ERR_ARG; }
    }
    CK(cudaSetDevice(b->device));
    if (first_solve && !b->d_budget) {
        if ((rc = dalloc(b, &b->d_budget, (size_t)2 * P))) return rc;
        CK(cudaMemsetAsync(b->d_budget, 0xff, sizeof(int) * 2 * P, b->stream));
        b->bp.budget = b->d_budget;
        b->budget_pending.assign(P, 0);
    }
    // the call's distinct (gait, window) pairs, one new slot each
    std::map<std::pair<int, int>, int> pair_index;
    std::vector<int> bgait, bwin, pair_of(n);
    for (int k = 0; k < n; ++k) {
        auto it = pair_index.emplace(std::make_pair((int)gait[k], (int)window[k]), (int)bgait.size());
        if (it.second) { bgait.push_back(gait[k]); bwin.push_back(window[k]); }
        pair_of[k] = it.first->second;
    }
    const int m = (int)bgait.size();
    SlotPlan plan;
    SlotMoves mv;
    std::vector<int> status(m, 0);
    int* d_st;
    if ((rc = plan_slot_moves(b, n, problem, pair_of, m, &plan)) || (rc = stage_slot_moves(b, plan, n, problem, bgait, bwin, status, &mv, &d_st)) ||
        (rc = scratch(b, &b->d_args_x0, &b->d_args_x0_cap, (size_t)n * 24))) return rc;
    CK(cudaMemcpyAsync(b->d_args_x0, x0, (size_t)n * 24 * sizeof(double), cudaMemcpyHostToDevice, b->stream));
    // build into the free slots, then one host synchronise for the build status
    launch_schedule_build(b, m, mv.gait, mv.window, mv.target, b->bp.max_stages, d_st);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(status.data(), d_st, sizeof(int) * m, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    for (int j = 0; j < m; ++j) {
        if (status[j] == 1) { g_last_error = "restart: window does not fit the gait table"; return HSDDP_ERR_ARG; }
        if (status[j]) { g_last_error = "restart: schedule exceeds HSDDP_MAX_PHASES / the batch's node capacity"; return HSDDP_ERR_UNSUPPORTED; }
    }
    RestartArgs ra{b->d_args_x0, first_solve ? first_solve->max_AL_iter : -1, first_solve ? first_solve->max_DDP_iter : -1, 0, {}};
    // (the trial arrays of a batch larger than kClusterLsMax belong to launch positions, not to problems: hsddp_batch_solve_problems)
    for (const WsArray& a : workspace_arrays(b))
        if ((a.flags & WS_RESTART) && *a.field && !((a.flags & WS_SMALL) && P > hsddp_batch::kClusterLsMax)) {
            if (ra.n_clear == kRestartClearMax) { g_last_error = "restart: more workspace arrays than kRestartClearMax"; return HSDDP_ERR_STATE; }
            ra.clear[ra.n_clear++] = {(unsigned*)*a.field, a.bytes() / sizeof(unsigned)};
        }
    commit_slot_moves(b, plan, n, problem);
    k_restart<<<n, kThreads, 0, b->stream>>>(b->bp, mv, ra);
    CK(cudaGetLastError());
    b->n_step_launches++;
    if (first_solve) b->budget_rounds = std::max(b->budget_rounds, (long long)first_solve->max_AL_iter * first_solve->max_DDP_iter);
    if (b->d_budget)
        for (int k = 0; k < n; ++k) {
            char& q = b->budget_pending[problem[k]];
            b->n_budget_pending += (first_solve ? 1 : 0) - q;
            q = first_solve ? 1 : 0;
        }
    if (b->d_budget && b->n_budget_pending == 0) b->budget_rounds = -1;
    return HSDDP_OK;
    });
}

/* HKDProblem::update of the listed problems (see hsddp_batch_mpc_update and k_copy_slots).  Built before it is committed: the
 * slots of the listed problems are copied to free slots and the copies stepped; only when every copy has succeeded do the listed
 * problems move to them and get shifted, so a refusal leaves the batch as it was. */
int hsddp_batch_mpc_update_problems(hsddp_batch* b, int n, const int32_t* problem) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_STATE; }
    if (!b->mpc_ready) { g_last_error = "hsddp_batch_mpc_update_problems needs the gait library on the device: set the problems with hsddp_batch_set_problems_from_gaits"; return HSDDP_ERR_STATE; }
    int rc;
    if ((rc = check_problem_list(b, n, problem, "mpc_update_problems"))) return rc;
    CK(cudaSetDevice(b->device));
    // the distinct slots of the listed problems, one copy each (problems that share a slot share its copy)
    std::map<int, int> copy_of;
    std::vector<int> src, entry(n);
    for (int k = 0; k < n; ++k) {
        auto it = copy_of.emplace(b->h_sched_id[problem[k]], (int)src.size());
        if (it.second) src.push_back(b->h_sched_id[problem[k]]);
        entry[k] = it.first->second;
    }
    const int m = (int)src.size();
    SlotPlan plan;
    SlotMoves mv;
    int* d_src;  // src[m] | error flag
    std::vector<int> tail = src, gw(m, 0);  // (gait / window of the copies: written by k_copy_slots)
    tail.push_back(0);
    if ((rc = plan_slot_moves(b, n, problem, entry, m, &plan)) || (rc = stage_slot_moves(b, plan, n, problem, gw, gw, tail, &mv, &d_src))) return rc;
    int* d_err = d_src + m;
    DevSchedule* sched = const_cast<DevSchedule*>(b->bp.sched);
    SlotCopyArgs ca{d_src, mv.target, b->d_sched_gait, b->d_sched_window, mv.gait, mv.window, sched, b->lib.node_stride, 0, {}};
    for (const SlotArray& a : slot_arrays(b)) {
        if (a.field == (void**)&b->d_sched_gait || a.field == (void**)&b->d_sched_window) continue;  // (written by the commit)
        if (ca.n_arrays == kSlotArraysMax) { g_last_error = "mpc_update_problems: more slot arrays than kSlotArraysMax"; return HSDDP_ERR_STATE; }
        ca.arr[ca.n_arrays++] = {(unsigned*)*a.field, a.bytes / sizeof(unsigned)};
    }
    CK(cudaEventRecord(b->ev_u0, b->stream));
    k_copy_slots<<<m, 128, 0, b->stream>>>(ca);
    k_mpc_update_schedules<<<(m + 127) / 128, 128, 0, b->stream>>>(b->lib, m, mv.gait, mv.window, mv.target, sched, b->d_mpc, d_err);
    k_reference_rows<<<m, 128, 0, b->stream>>>(b->lib, m, mv.gait, mv.window, mv.target, sched, b->d_mpc, const_cast<double*>(b->bp.xr),
                                              const_cast<double*>(b->bp.ur), const_cast<double*>(b->bp.prel), nullptr);
    CK(cudaGetLastError());
    b->n_step_launches += 3;
    int err = 0;
    CK(cudaMemcpyAsync(&err, d_err, sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    if (err) {  // the copies are dropped: their slots stay on the free list and were never marked in use on the device
        CK(cudaEventRecord(b->ev_u1, b->stream));
        g_last_error = err == 1 ? "receding-horizon update: the reference table is exhausted" : "receding-horizon update: schedule exceeds HSDDP_MAX_PHASES / node capacity";
        return err == 1 ? HSDDP_ERR_ARG : HSDDP_ERR_UNSUPPORTED;
    }
    // commit: the listed problems move to the stepped copies and slots nobody uses any more are freed, in the shift's launch
    k_mpc_shift<<<n, kThreads, 0, b->stream>>>(b->bp, b->d_mpc, mv);
    CK(cudaGetLastError());
    b->n_step_launches++;
    CK(cudaEventRecord(b->ev_u1, b->stream));
    commit_slot_moves(b, plan, n, problem);
    return HSDDP_OK;
    });
}

int hsddp_batch_get_schedule_ids(hsddp_batch* b, int32_t* out) {
    if (!b || !out) return HSDDP_ERR_ARG;
    if (!b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_STATE; }
    std::copy(b->h_sched_id.begin(), b->h_sched_id.end(), out);
    return HSDDP_OK;
}

int hsddp_batch_set_initial_condition(hsddp_batch* b, const double* x0) {
    if (!b || !b->has_problems || !x0) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaMemcpyAsync(b->bp.x0, x0, sizeof(double) * 24 * b->bp.n_problems, cudaMemcpyHostToDevice, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
}

int hsddp_batch_set_initial_condition_problems(hsddp_batch* b, int n, const int32_t* problem, const double* x0) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems || !x0) return HSDDP_ERR_ARG;
    int rc, *d;
    if ((rc = check_problem_list(b, n, problem, "set_initial_condition_problems"))) return rc;
    CK(cudaSetDevice(b->device));
    if ((rc = stage_ints(b, std::vector<int>(problem, problem + n), &d)) || (rc = scratch(b, &b->d_args_x0, &b->d_args_x0_cap, (size_t)n * 24))) return rc;
    CK(cudaMemcpyAsync(b->d_args_x0, x0, (size_t)n * 24 * sizeof(double), cudaMemcpyHostToDevice, b->stream));
    return scatter_rows(b, b->bp.x0, 48, d, b->d_args_x0, 48, n);
    });
}

int hsddp_batch_reset(hsddp_batch* b) {
    // queued on the handle's stream without a host synchronise, so reset + solve run back to back
    return launch_step(b, nullptr, OP_RESET, 0.0, nullptr, nullptr, false);
}

// Phased driver: every round advances all running problems by one DDP iteration with one launch per phase
// (prep, backward sweep, forward).  Blocks that are co-resident on an SM execute the same phase, so the instruction
// cache holds one phase's code instead of six different ones.  The batch is split into `groups` index ranges, each
// driven round by round on its own stream: the launch tail of one group's kernel (its last, partially filled wave of
// blocks) overlaps with the other groups' kernels.
// The whole solve is queued WITHOUT a host round trip: the list of running problems and its length live in HBM
// (BatchPtrs::active / n_active), every round is launched with the group's full grid, and blocks beyond the current
// length leave at once.  max_AL_iter x max_DDP_iter rounds are queued (no problem can run more DDP iterations); the
// rounds after a group's last running problem has finished cost a few microseconds each.
__global__ void k_iota(int* a, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = i;
}

// Work-queue order of the persistent kernel for the NEXT solve: problems sorted by the number of DDP iterations their last
// solve took, longest first (counting sort, one block).  Iteration counts differ a lot inside a batch (6 .. 50 on the
// benchmark workload) and change little between consecutive solves of the same problems (MPC ticks, repeated cold solves),
// so starting the long ones first keeps the tail of the launch short (longest-processing-time-first list scheduling).
// It only permutes the order in which blocks pick problems up: results do not depend on it.
// The key is the previous solve's WORK, not its iteration count alone: an iteration costs one prep + one linear rollout
// (~ 1/3 of a nominal iteration), every backward sweep ~ 1/2 (regularisation retries repeat it) and every line-search trial
// ~ 1/8; problems that regularise or reject steps run several times longer per iteration than the others, and with the
// count alone they were started late (the eight 2,048-problem shards of config 3 ranged from 50 to 69 ms).
__device__ __forceinline__ int order_bin(const hsddp_info& q) {
    const int work = 33 * q.n_iter + 48 * q.n_sweeps + 12 * q.n_trials;  // in 1/93 of a nominal iteration
    return 255 - min(max(work >> 6, 0), 255);
}
__global__ void k_order_by_iterations(const hsddp_info* info, int n, int* order) {
    __shared__ int bins[256], start[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) bins[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) atomicAdd(&bins[order_bin(info[i])], 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int i = 0; i < 256; ++i) { start[i] = acc; acc += bins[i]; }
    }
    __syncthreads();
    // (stable inside a bin: every bin is filled by one thread in index order, so the order is reproducible)
    for (int bi = threadIdx.x; bi < 256; bi += blockDim.x) {
        if (!bins[bi]) continue;
        int pos = start[bi];
        for (int i = 0; i < n; ++i)
            if (order_bin(info[i]) == bi) order[pos++] = i;
    }
}

// problem[0 .. P) run (nullptr: every problem of the batch, P = n_problems)
static int solve_phased(hsddp_batch* b, const hsddp_options& o, int P, const int32_t* problem) {
    const int G = std::min(hsddp_batch::kMaxGroups, std::max(1, P / hsddp_batch::kPhasedMinGroup));  // problems per group at least kPhasedMinGroup
    for (int g = 0; g < G; ++g) {
        if (!b->gstream[g]) {
            CK(cudaStreamCreateWithFlags(&b->gstream[g], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&b->gevent[g], cudaEventDisableTiming));
        }
    }
    const int S = b->sweep_spec, cap = hsddp_batch::kSpecCap;
    const size_t slice = (size_t)b->bp.max_stages * 312 + 600, spec_ints = (size_t)G * (2 * cap + 2) + b->bp.n_problems;
    if (S) {
        int rs = scratch(b, &b->d_spec_int, &b->d_spec_int_cap, spec_ints);
        if (!rs) rs = scratch(b, &b->d_spec_rec, &b->d_spec_rec_cap, (size_t)G * cap * S);
        if (!rs) rs = scratch(b, &b->d_spec_out, &b->d_spec_out_cap, (size_t)G * cap * (S - 1) * slice);
        if (rs) return rs;
    }
    CK(cudaEventRecord(b->ev0, b->stream));
    CK(cudaMemsetAsync(b->d_count, 0, 2 * hsddp_batch::kMaxGroups * sizeof(int), b->stream));
    if (S) CK(cudaMemsetAsync(b->d_spec_int, 0, spec_ints * sizeof(int), b->stream));
    if (problem) CK(cudaMemcpyAsync(b->d_active[0], problem, sizeof(int) * P, cudaMemcpyHostToDevice, b->stream));
    else k_iota<<<(P + 255) / 256, 256, 0, b->stream>>>(b->d_active[0], P);
    CK(cudaEventRecord(b->ev_fork, b->stream));
    // (restarted problems may have a larger budget for this solve: BatchPtrs::budget)
    const int rounds = (int)std::min<long long>(std::max((long long)std::max(0, o.max_AL_iter) * (long long)std::max(0, o.max_DDP_iter), b->budget_rounds), 1000000LL);
    int rc = HSDDP_OK;
    for (int g = 0; g < G && rc == HSDDP_OK; ++g) {
        const int lo = (int)((long long)P * g / G), n = (int)((long long)P * (g + 1) / G) - lo;
        if (n <= 0) continue;
        cudaStream_t st = b->gstream[g];
        int* cnt[2] = {b->d_count + 2 * g, b->d_count + 2 * g + 1};
        int* list[2] = {b->d_active[0] + lo, b->d_active[1] + lo};
        if (cudaStreamWaitEvent(st, b->ev_fork, 0) != cudaSuccess) { rc = HSDDP_ERR_CUDA; break; }
        BatchPtrs bp = b->bp;
        bp.sweep_w1_min = hsddp_batch::kSweepW1Min;
        bp.lr_external = (b->lr_w1 && o.MS) ? 1 : 0;
        // round 0: begin (initial rollout, first outer iteration set-up) over every problem of the group
        bp.active = list[0]; bp.n_active = nullptr; bp.next_active = list[1]; bp.next_count = cnt[1]; bp.zero_count = nullptr;
        k_phase<PH_BEGIN><<<n, kThreads, 0, st>>>(bp, o);
        b->n_solve_launches++;
        int* spec = b->d_spec_int + (size_t)g * (2 * cap + 2);
        if (S) {
            bp.spec_list = spec; bp.spec_arrive = spec + cap; bp.spec_entry = b->d_spec_int + (size_t)G * (2 * cap + 2);
            bp.spec_rec = b->d_spec_rec + (size_t)g * cap * S; bp.spec_out = b->d_spec_out + (size_t)g * cap * (S - 1) * slice;
            bp.spec_S = S; bp.spec_cap = cap;
        }
        for (int r = 1; r <= rounds; ++r) {
            const int cur = r & 1;
            bp.active = list[cur]; bp.n_active = cnt[cur]; bp.next_active = list[cur ^ 1]; bp.next_count = cnt[cur ^ 1]; bp.zero_count = cnt[cur ^ 1];
            if (S) { bp.spec_count = spec + 2 * cap + cur; bp.spec_zero = spec + 2 * cap + (cur ^ 1); }
            k_phase<PH_PREP><<<n, kThreads, 0, st>>>(bp, o);
            k_phase<PH_SWEEP><<<n + (S ? cap * (S - 1) : 0), kThreads, 0, st>>>(bp, o);
            k_sweep_w1<<<n, 32, 0, st>>>(bp, o);
            if (bp.lr_external) k_lr_w1<<<n, 32, 0, st>>>(bp, o);
            k_phase<PH_FORWARD><<<n, kThreads, 0, st>>>(bp, o);
            b->n_solve_launches += 4 + (bp.lr_external ? 1 : 0);
        }
        if (cudaGetLastError() != cudaSuccess) { rc = HSDDP_ERR_CUDA; g_last_error = "kernel launch failed in the phased driver"; }
    }
    // join (also on an error exit: the handle's stream continues after every group, so later calls never see half-finished state)
    for (int g = 0; g < G; ++g) {
        if (!b->gstream[g]) continue;
        if (cudaEventRecord(b->gevent[g], b->gstream[g]) == cudaSuccess) cudaStreamWaitEvent(b->stream, b->gevent[g], 0);
    }
    CK(cudaEventRecord(b->ev1, b->stream));
    return rc;
}

int hsddp_batch_set_solve_mode(hsddp_batch* b, int mode) {
    if (!b || mode < 0 || mode > 2) return HSDDP_ERR_ARG;
    b->solve_mode = mode;
    return HSDDP_OK;
}

// the per-problem budgets of restarted problems apply to one solve: those of the problems it ran (problem[0 .. n), nullptr:
// every problem) are cleared on the stream once it is queued
static int consume_budget(hsddp_batch* b, int n, const int32_t* problem) {
    if (b->budget_rounds < 0) return HSDDP_OK;
    if (!problem) {
        CK(cudaMemsetAsync(b->d_budget, 0xff, sizeof(int) * 2 * b->bp.n_problems, b->stream));
        std::fill(b->budget_pending.begin(), b->budget_pending.end(), 0);
        b->n_budget_pending = 0;
    } else {
        std::vector<int> h;
        for (int k = 0; k < n; ++k)
            if (b->budget_pending[problem[k]]) { h.push_back(problem[k]); b->budget_pending[problem[k]] = 0; }
        const int c = (int)h.size();
        if (c) {
            b->n_budget_pending -= c;
            h.push_back(-1); h.push_back(-1);
            int rc, *d;
            if ((rc = stage_ints(b, h, &d)) || (rc = scatter_rows(b, b->d_budget, 2, d, d + c, 0, c))) return rc;
        }
    }
    if (b->n_budget_pending == 0) b->budget_rounds = -1;
    return HSDDP_OK;
}

// trial arrays of k_solve_lat4 for kClusterLsMax launch positions, allocated by the first solve of at most kClusterLsMax listed
// problems in a batch too large to have them per problem
static int alloc_cluster_ls(hsddp_batch* b) {
    for (const WsArray& a : workspace_arrays(b)) {
        if (!(a.flags & WS_SMALL)) continue;
        const size_t bytes = a.bytes() * hsddp_batch::kClusterLsMax;
        if (int rc = dalloc_bytes(b, a.field, bytes)) return rc;
        CK(cudaMemsetAsync(*a.field, 0, bytes, b->stream));
    }
    return HSDDP_OK;
}

// the solve of problem[0 .. n) (nullptr: every problem, n = n_problems), in the driver a batch of n problems takes
static int solve_list(hsddp_batch* b, const hsddp_options* opt, int n, const int32_t* problem) {
    int rc = check_opt(opt);
    if (rc) return rc;
    CK(cudaSetDevice(b->device));
    const hsddp_options o = opt ? *opt : default_options();
    const int P = b->bp.n_problems;
    // auto: the persistent kernel up to ~7 waves of blocks (its work queue visits the problems longest-first from the second
    // solve on, which keeps the tail short); beyond that the phased driver, whose phase-homogeneous kernels keep the
    // instruction cache hot and whose launch tails are hidden by driving four index ranges on their own streams
    // (measured on config 3, persistent vs phased, ms, final code of round 2: 2,048 problems 57 vs 69, 4,096: 98 vs 100,
    // 5,120: ~121 vs 117, 6,144: 145 vs 135, 8,192: 199 vs 163 -- profiles/r02an_*: the switch is at 5.5 waves of blocks, 4,884 problems)
    const bool phased = b->solve_mode == 2 || (b->solve_mode == 0 && 2 * n >= 11 * b->n_sm * b->blocks_per_sm);
    if (phased) {
        rc = solve_phased(b, o, n, problem);
        if (rc == HSDDP_OK) rc = consume_budget(b, n, problem);
        return rc;
    }
    const bool cluster = n <= hsddp_batch::kClusterLsMax && o.MS;
    if (cluster && problem && !b->bp.ls_mail && (rc = alloc_cluster_ls(b))) return rc;
    const int grid = (n <= 2 * b->n_sm) ? n : std::min(n, b->n_sm * b->blocks_per_sm);
    BatchPtrs bp = b->bp;
    if (problem) {
        // the work queue (the cluster index of k_solve_lat4): the list, then n_problems, which ends a block, up to the last
        // entry a block can draw.  It replaces the queue-order hint of the whole batch.
        std::vector<int> q(std::min(P, n + grid), P);
        std::copy(problem, problem + n, q.begin());
        CK(cudaMemcpyAsync(b->d_order, q.data(), q.size() * sizeof(int), cudaMemcpyHostToDevice, b->stream));
        bp.order = b->d_order;
        b->have_order = false;
    }
    CK(cudaMemsetAsync(b->bp.work_counter, 0, sizeof(int), b->stream));
    CK(cudaEventRecord(b->ev0, b->stream));
    if (b->bp.ls_mail && cluster) {
        k_solve_lat4<<<4 * n, kThreads, 0, b->stream>>>(bp, o);
    } else if (n <= 2 * b->n_sm) {
        k_solve_lat<<<n, kThreads, 0, b->stream>>>(bp, o);
    } else {
        if (!problem) bp.order = b->have_order ? b->d_order : nullptr;
        k_solve<<<grid, kThreads, 0, b->stream>>>(bp, o);
    }
    CK(cudaGetLastError());
    b->n_solve_launches++;
    CK(cudaEventRecord(b->ev1, b->stream));
    if ((rc = consume_budget(b, n, problem))) return rc;
    if (!problem && P > 2 * b->n_sm) {  // (after the timed region of last_solve_ms: ~10 us, part of every bench step)
        k_order_by_iterations<<<1, 256, 0, b->stream>>>(b->bp.info, b->bp.n_problems, b->d_order);
        CK(cudaGetLastError());
        b->n_solve_launches++;
        b->have_order = true;
    }
    return HSDDP_OK;
}

int hsddp_batch_solve_async(hsddp_batch* b, const hsddp_options* opt) {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_STATE; }
    return solve_list(b, opt, b->bp.n_problems, nullptr);
}

int hsddp_batch_solve_problems_async(hsddp_batch* b, int n, const int32_t* problem, const hsddp_options* opt) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_STATE; }
    if (int rc = check_problem_list(b, n, problem, "solve_problems")) return rc;
    return solve_list(b, opt, n, problem);
    });
}

int hsddp_batch_sync(hsddp_batch* b) {
    if (!b) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
}

int hsddp_batch_solve(hsddp_batch* b, const hsddp_options* opt) {
    int rc = hsddp_batch_solve_async(b, opt);
    if (rc) return rc;
    return hsddp_batch_sync(b);
}

int hsddp_batch_solve_problems(hsddp_batch* b, int n, const int32_t* problem, const hsddp_options* opt) {
    int rc = hsddp_batch_solve_problems_async(b, n, problem, opt);
    if (rc) return rc;
    return hsddp_batch_sync(b);
}

int hsddp_batch_last_solve_ms(hsddp_batch* b, float* ms) {
    if (!b || !ms) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaEventSynchronize(b->ev1));
    CK(cudaEventElapsedTime(ms, b->ev0, b->ev1));
    return HSDDP_OK;
}

int hsddp_batch_hybrid_rollout(hsddp_batch* b, double eps, const hsddp_options* opt, int32_t* ok) { return launch_step(b, opt, OP_ROLLOUT, eps, nullptr, ok); }
int hsddp_batch_compute_cost(hsddp_batch* b, const hsddp_options* opt) { return launch_step(b, opt, OP_COST, 0, nullptr, nullptr); }
int hsddp_batch_lq_approximation(hsddp_batch* b, const hsddp_options* opt) { return launch_step(b, opt, OP_LQ, 0, nullptr, nullptr); }
int hsddp_batch_backward_sweep(hsddp_batch* b, double regularization, int32_t* ok) { return launch_step(b, nullptr, OP_SWEEP, regularization, nullptr, ok); }
int hsddp_batch_backward_sweep_regularized(hsddp_batch* b, double* regularization, const hsddp_options* opt, int32_t* ok) {
    if (!b || !b->has_problems || !regularization) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaMemcpy(b->d_darg, regularization, sizeof(double) * b->bp.n_problems, cudaMemcpyHostToDevice));
    int rc = launch_step(b, opt, OP_SWEEP_REG, 0, b->d_darg, ok);
    if (rc) return rc;
    CK(cudaMemcpy(regularization, b->d_darg, sizeof(double) * b->bp.n_problems, cudaMemcpyDeviceToHost));
    return HSDDP_OK;
}
int hsddp_batch_linear_rollout(hsddp_batch* b, double eps, const hsddp_options* opt) { return launch_step(b, opt, OP_LINEAR, eps, nullptr, nullptr); }
int hsddp_batch_prepare_merit(hsddp_batch* b, const hsddp_options* opt) { return launch_step(b, opt, OP_MERIT, 0, nullptr, nullptr); }
int hsddp_batch_forward_sweep(hsddp_batch* b, const hsddp_options* opt, int32_t* ok, double* eps_accepted) {
    int rc = launch_step(b, opt, OP_FORWARD, 0, b ? b->d_darg : nullptr, ok);
    if (rc) return rc;
    if (eps_accepted) CK(cudaMemcpy(eps_accepted, b->d_darg, sizeof(double) * b->bp.n_problems, cudaMemcpyDeviceToHost));
    return HSDDP_OK;
}
int hsddp_batch_update_nominal(hsddp_batch* b) { return launch_step(b, nullptr, OP_NOMINAL, 0, nullptr, nullptr); }
int hsddp_batch_update_al_params(hsddp_batch* b, const hsddp_options* opt) { return launch_step(b, opt, OP_AL, 0, nullptr, nullptr); }
int hsddp_batch_update_reb_params(hsddp_batch* b, const hsddp_options* opt) { return launch_step(b, opt, OP_REB, 0, nullptr, nullptr); }

int hsddp_batch_dims(hsddp_batch* b, int32_t* n_problems, int32_t* max_stages, int32_t* max_nodes) {
    if (!b || !b->has_problems) return HSDDP_ERR_STATE;
    if (n_problems) *n_problems = b->bp.n_problems;
    if (max_stages) *max_stages = b->bp.max_stages;
    if (max_nodes) *max_nodes = b->bp.max_nodes;
    return HSDDP_OK;
}

int hsddp_batch_get_info(hsddp_batch* b, hsddp_info* out) {
    if (!b || !b->has_problems || !out) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaMemcpyAsync(out, b->bp.info, sizeof(hsddp_info) * b->bp.n_problems, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
}

int hsddp_batch_get_trace(hsddp_batch* b, hsddp_iter_record* out) {
    if (!b || !b->has_problems || !out) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaMemcpyAsync(out, b->bp.trace, sizeof(hsddp_iter_record) * HSDDP_TRACE_CAP * b->bp.n_problems, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
}

int hsddp_batch_get_scalars(hsddp_batch* b, double* out) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems || !out) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    std::vector<SolverState> st(b->bp.n_problems);
    CK(cudaMemcpy(st.data(), b->bp.state, sizeof(SolverState) * st.size(), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < st.size(); ++i) {
        double* o = out + 8 * i;
        o[0] = st[i].actual_cost; o[1] = st[i].merit; o[2] = st[i].feas; o[3] = st[i].dV_1; o[4] = st[i].dV_2;
        o[5] = st[i].max_tconstr; o[6] = st[i].max_pconstr; o[7] = st[i].merit_rho;
    }
    return HSDDP_OK;
    });
}

// Dense column-major 24x24 feedback gains for stages [row0, row0+nrows) from the compact K_r store.
static int refresh_host_schedules(hsddp_batch* b);
static int get_gains(hsddp_batch* b, int row0, int nrows, double* out) {
    if (int rc = refresh_host_schedules(b)) return rc;
    const BatchPtrs& bp = b->bp;
    const size_t P = (size_t)bp.n_problems;
    if (row0 < 0 || nrows <= 0 || row0 + nrows > bp.max_stages) return HSDDP_ERR_ARG;
    std::vector<double> kr(P * nrows * 288);
    CK(cudaMemcpy2DAsync(kr.data(), (size_t)nrows * 288 * sizeof(double), bp.K + (size_t)row0 * 288, (size_t)bp.max_stages * 288 * sizeof(double),
                         (size_t)nrows * 288 * sizeof(double), P, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    std::memset(out, 0, P * nrows * 576 * sizeof(double));
    for (size_t p = 0; p < P; ++p) {
        const DevSchedule& sc = b->h_sched[b->h_sched_id[p]];
        for (int ph = 0; ph < sc.n_phases; ++ph)
            for (int k = 0; k < sc.horizon[ph]; ++k) {
                const int s = sc.stage_off[ph] + k;
                if (s < row0 || s >= row0 + nrows) continue;
                const double* src = &kr[(p * nrows + (s - row0)) * 288];
                double* o = out + (p * nrows + (s - row0)) * 576;
                for (int c = 0; c < 12; ++c) {
                    const int i = ((sc.cmask[ph] >> (c / 3)) & 1u) ? c : 12 + c;
                    for (int j = 0; j < 24; ++j) o[i + 24 * j] = src[j * 12 + c];
                }
            }
    }
    return HSDDP_OK;
}

int hsddp_batch_get_array(hsddp_batch* b, int which, double* out) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems || !out) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    const BatchPtrs& bp = b->bp;
    const size_t P = (size_t)bp.n_problems;
    if (which == HSDDP_ARR_A || which == HSDDP_ARR_B || which == HSDDP_ARR_LX || which == HSDDP_ARR_LU ||
        which == HSDDP_ARR_LUU || which == HSDDP_ARR_LXX) {
        // dense views reconstructed on the host from the compact LQ records
        if (int rc = refresh_host_schedules(b)) return rc;
        std::vector<double> lq(P * bp.max_stages * CR_STRIDE);
        CK(cudaMemcpy(lq.data(), bp.lq, lq.size() * sizeof(double), cudaMemcpyDeviceToHost));
        const bool vec = (which == HSDDP_ARR_LX || which == HSDDP_ARR_LU);
        const size_t per = (size_t)bp.max_stages * (vec ? 24 : 576);
        std::memset(out, 0, P * per * sizeof(double));
        for (size_t p = 0; p < P; ++p) {
            const DevSchedule& sc = b->h_sched[b->h_sched_id[p]];
            for (int ph = 0; ph < sc.n_phases; ++ph)
                for (int k = 0; k < sc.horizon[ph]; ++k) {
                    const int s = sc.stage_off[ph] + k;
                    const double* rec = &lq[(p * bp.max_stages + s) * CR_STRIDE];
                    double* o = out + p * per + (size_t)s * (vec ? 24 : 576);
                    const unsigned cm = sc.cmask[ph];
                    if (which == HSDDP_ARR_LX) std::memcpy(o, rec + CR_LX, 24 * sizeof(double));
                    else if (which == HSDDP_ARR_LU) std::memcpy(o, rec + CR_LU, 24 * sizeof(double));
                    else if (which == HSDDP_ARR_A || which == HSDDP_ARR_B) {
                        double A[576], B[576];
                        hkd::expand_AB(rec + CR_R, sc.dt, cm, A, B);
                        std::memcpy(o, which == HSDDP_ARR_A ? A : B, 576 * sizeof(double));
                    } else if (which == HSDDP_ARR_LUU) {
                        for (int i = 0; i < 24; ++i) o[i * 25] = sc.dt * (i < 12 ? .2 : .1);
                        for (int l = 0; l < 4; ++l)
                            for (int a = 0; a < 3; ++a)
                                for (int c = 0; c < 3; ++c) o[(3 * l + a) + 24 * (3 * l + c)] += rec[CR_LUU + 9 * l + 3 * a + c];
                    } else {  // LXX: dt*Q + foot regulariser block (HKDCost.cpp:36-37)
                        const double q[12] = {1, 4, 5, 1, 1, 30, .2, .2, .2, 4, 1, .5};
                        for (int i = 0; i < 24; ++i) {
                            const double Q = i < 12 ? q[i] : .2 * (1 - (int)((cm >> ((i - 12) / 3)) & 1u));
                            o[i * 25] = sc.dt * Q;
                        }
                        for (int l = 0; l < 4; ++l) {
                            const double c = (double)((cm >> l) & 1u);
                            const double wf[3] = {3 * c * 20, c * 20, 0.0};
                            for (int j = 0; j < 3; ++j) {
                                const double wc = (sc.dt * c * wf[j]) * c;
                                o[(3 + j) * 25] += wc; o[(12 + 3 * l + j) * 25] += wc;
                                o[(3 + j) + 24 * (12 + 3 * l + j)] += -wc; o[(12 + 3 * l + j) + 24 * (3 + j)] += -wc;
                            }
                        }
                    }
                }
        }
        return HSDDP_OK;
    }
    if (which == HSDDP_ARR_K) return get_gains(b, 0, bp.max_stages, out);
    if (which == HSDDP_ARR_G0 || which == HSDDP_ARR_H0) {  // strided views of g0h0
        const size_t off = (which == HSDDP_ARR_G0) ? 0 : 24, cnt = (which == HSDDP_ARR_G0) ? 24 : 576;
        CK(cudaMemcpy2DAsync(out, cnt * sizeof(double), bp.g0h0 + off, 600 * sizeof(double), cnt * sizeof(double), P, cudaMemcpyDeviceToHost, b->stream));
        CK(cudaStreamSynchronize(b->stream));
        return HSDDP_OK;
    }
    WsArray a;
    if (!stored_array(b, which, &a)) return HSDDP_ERR_ARG;
    CK(cudaMemcpyAsync(out, *a.field, P * a.bytes(), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
    });
}

int hsddp_batch_set_array(hsddp_batch* b, int which, const double* in) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems || !in) return HSDDP_ERR_ARG;
    WsArray a;
    if (!stored_array(b, which, &a) || !(a.flags & WS_SET)) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaMemcpyAsync(*a.field, in, (size_t)b->bp.n_problems * a.bytes(), cudaMemcpyHostToDevice, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
    });
}

int hsddp_batch_get_array_rows(hsddp_batch* b, int which, int row0, int nrows, double* out) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems || !out || row0 < 0 || nrows <= 0) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    if (which == HSDDP_ARR_K) return get_gains(b, row0, nrows, out);
    WsArray a;
    if (!stored_array(b, which, &a) || (size_t)row0 + (size_t)nrows > a.rows) return HSDDP_ERR_ARG;
    CK(cudaMemcpy2DAsync(out, nrows * a.row_bytes, (const char*)*a.field + row0 * a.row_bytes, a.bytes(), nrows * a.row_bytes,
                         (size_t)b->bp.n_problems, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
    });
}

int hsddp_batch_get_gains_compact(hsddp_batch* b, int row0, int nrows, double* out) {
    if (!b || !b->has_problems || !out || row0 < 0 || nrows <= 0 || row0 + nrows > b->bp.max_stages) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaMemcpy2DAsync(out, (size_t)nrows * 288 * sizeof(double), b->bp.K + (size_t)row0 * 288, (size_t)b->bp.max_stages * 288 * sizeof(double),
                         (size_t)nrows * 288 * sizeof(double), (size_t)b->bp.n_problems, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
}

// the command records of problem[0 .. n) (nullptr: every problem, n = n_problems) into out[0 .. n), one transfer
static int get_commands(hsddp_batch* b, int n_steps, int n, const int32_t* problem, hsddp_mpc_command* out) {
    CK(cudaSetDevice(b->device));
    if (!b->d_cmd) {
        void* q = nullptr;
        CK(cudaMalloc(&q, sizeof(hsddp_mpc_command) * (size_t)b->bp.n_problems));
        b->allocs.push_back(q);
        b->d_cmd = (hsddp_mpc_command*)q;
    }
    int* d = nullptr;
    if (problem)
        if (int rc = stage_ints(b, std::vector<int>(problem, problem + n), &d)) return rc;
    k_command<<<n, 128, 0, b->stream>>>(b->bp, n_steps, b->d_cmd, d);
    CK(cudaGetLastError());
    b->n_step_launches++;
    CK(cudaMemcpyAsync(out, b->d_cmd, sizeof(hsddp_mpc_command) * (size_t)n, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return HSDDP_OK;
}

int hsddp_batch_get_mpc_command(hsddp_batch* b, int n_steps, hsddp_mpc_command* out) {
    if (!b || !b->has_problems || !out || n_steps < 1 || n_steps > HSDDP_CMD_MAX_STEPS) return HSDDP_ERR_ARG;
    return get_commands(b, n_steps, b->bp.n_problems, nullptr, out);
}

int hsddp_batch_get_mpc_command_problems(hsddp_batch* b, int n_steps, int n, const int32_t* problem, hsddp_mpc_command* out) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems || !out || n_steps < 1 || n_steps > HSDDP_CMD_MAX_STEPS) return HSDDP_ERR_ARG;
    if (int rc = check_problem_list(b, n, problem, "get_mpc_command_problems")) return rc;
    return get_commands(b, n_steps, n, problem, out);
    });
}

// --- the _dev entry points: buffers in device memory of the handle's GPU, ordered on the caller's stream ---

// a list the _dev calls take: n distinct indices, or nullptr for every problem in index order (then n == n_problems)
static int check_dev_list(hsddp_batch* b, int n, const int32_t* problem, const char* what) {
    if (problem) return check_problem_list(b, n, problem, what);
    if (n != b->bp.n_problems) { g_last_error = std::string(what) + ": without a list n must be n_problems"; return HSDDP_ERR_ARG; }
    return HSDDP_OK;
}

// p must be device or managed memory of the handle's GPU, aligned to `align` bytes
static int check_dev_buffer(hsddp_batch* b, const void* p, size_t align, const char* what) {
    if (!p) { g_last_error = std::string(what) + ": NULL buffer"; return HSDDP_ERR_ARG; }
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();  // (not a sticky error: clear it so that it is not reported by a later call)
        g_last_error = std::string(what) + ": not a CUDA pointer";
        return HSDDP_ERR_ARG;
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != b->device) {
        g_last_error = std::string(what) + ": the buffer is not device memory of the handle's GPU";
        return HSDDP_ERR_ARG;
    }
    if ((uintptr_t)p % align) { g_last_error = std::string(what) + ": misaligned buffer"; return HSDDP_ERR_ARG; }
    return HSDDP_OK;
}

// *d := the listed indices in the call's device argument list, copied from a pinned host buffer on the handle's stream
static int stage_list_pinned(hsddp_batch* b, int n, const int32_t* problem, int** d) {
    hsddp_batch::PinnedList* s = nullptr;
    for (auto& q : b->pinned_lists) {
        if (q.cap < (size_t)n) continue;
        const cudaError_t e = cudaEventQuery(q.read);
        if (e == cudaSuccess) { s = &q; break; }
        if (e != cudaErrorNotReady) CK(e);
        cudaGetLastError();  // (clear the not-ready status)
    }
    if (!s) {
        hsddp_batch::PinnedList q;
        q.cap = std::max((size_t)n, (size_t)1024);
        CK(cudaHostAlloc((void**)&q.h, q.cap * sizeof(int), cudaHostAllocDefault));
        if (cudaEventCreateWithFlags(&q.read, cudaEventDisableTiming) != cudaSuccess) {
            cudaFreeHost(q.h);
            g_last_error = "cudaEventCreateWithFlags failed";
            return HSDDP_ERR_CUDA;
        }
        b->pinned_lists.push_back(q);
        s = &b->pinned_lists.back();
    }
    std::memcpy(s->h, problem, (size_t)n * sizeof(int));
    if (int rc = scratch(b, &b->d_args, &b->d_args_cap, (size_t)n)) return rc;
    CK(cudaMemcpyAsync(b->d_args, s->h, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, b->stream));
    CK(cudaEventRecord(s->read, b->stream));
    *d = b->d_args;
    return HSDDP_OK;
}

// The stream contract: the handle's stream waits for what the caller queued on `stream` before the call (join_caller), and
// the caller's stream for the call's last launch (release_caller).  Neither synchronises the host.
static int join_caller(hsddp_batch* b, void* stream) {
    CK(cudaEventRecord(b->ev_in, (cudaStream_t)stream));
    CK(cudaStreamWaitEvent(b->stream, b->ev_in, 0));
    return HSDDP_OK;
}

static int release_caller(hsddp_batch* b, void* stream) {
    CK(cudaEventRecord(b->ev_out, b->stream));
    CK(cudaStreamWaitEvent((cudaStream_t)stream, b->ev_out, 0));
    return HSDDP_OK;
}

int hsddp_batch_set_initial_condition_dev(hsddp_batch* b, int n, const int32_t* problem, const double* x0_dev, void* stream) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_ARG; }
    int rc, *d = nullptr;
    if ((rc = check_dev_list(b, n, problem, "set_initial_condition_dev")) || (rc = check_dev_buffer(b, x0_dev, sizeof(double), "set_initial_condition_dev")))
        return rc;
    CK(cudaSetDevice(b->device));
    if (problem && (rc = stage_list_pinned(b, n, problem, &d))) return rc;
    if ((rc = join_caller(b, stream))) return rc;
    if (problem) {
        if ((rc = scatter_rows(b, b->bp.x0, 48, d, x0_dev, 48, n))) return rc;
    } else {
        CK(cudaMemcpyAsync(b->bp.x0, x0_dev, sizeof(double) * 24 * (size_t)n, cudaMemcpyDeviceToDevice, b->stream));
    }
    return release_caller(b, stream);
    });
}

int hsddp_batch_set_measured_state_dev(hsddp_batch* b, int n, const int32_t* problem, const double* meas_dev,
                                       const int32_t* contact_dev, void* stream) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_ARG; }
    int rc, *d = nullptr;
    if ((rc = check_dev_list(b, n, problem, "set_measured_state_dev")) || (rc = check_dev_buffer(b, meas_dev, sizeof(double), "set_measured_state_dev")))
        return rc;
    if (contact_dev && (rc = check_dev_buffer(b, contact_dev, sizeof(int32_t), "set_measured_state_dev (contact)"))) return rc;
    CK(cudaSetDevice(b->device));
    if (problem && (rc = stage_list_pinned(b, n, problem, &d))) return rc;
    if ((rc = join_caller(b, stream))) return rc;
    k_measured_state<<<(n + 127) / 128, 128, 0, b->stream>>>(b->bp, meas_dev, contact_dev, d, n);
    CK(cudaGetLastError());
    b->n_step_launches++;
    return release_caller(b, stream);
    });
}

int hsddp_batch_get_mpc_command_dev(hsddp_batch* b, int n_steps, int n, const int32_t* problem, hsddp_mpc_command* out_dev, void* stream) {
    return guarded([&]() -> int {
    if (!b || !b->has_problems) { g_last_error = "no problems set"; return HSDDP_ERR_ARG; }
    if (n_steps < 1 || n_steps > HSDDP_CMD_MAX_STEPS) { g_last_error = "get_mpc_command_dev: n_steps must be in [1, HSDDP_CMD_MAX_STEPS]"; return HSDDP_ERR_ARG; }
    int rc, *d = nullptr;
    if ((rc = check_dev_list(b, n, problem, "get_mpc_command_dev")) || (rc = check_dev_buffer(b, out_dev, alignof(hsddp_mpc_command), "get_mpc_command_dev")))
        return rc;
    CK(cudaSetDevice(b->device));
    if (problem && (rc = stage_list_pinned(b, n, problem, &d))) return rc;
    if ((rc = join_caller(b, stream))) return rc;
    k_command<<<n, 128, 0, b->stream>>>(b->bp, n_steps, out_dev, d);
    CK(cudaGetLastError());
    b->n_step_launches++;
    return release_caller(b, stream);
    });
}

int hsddp_batch_event_record(hsddp_batch* b, int slot) {
    if (!b || slot < 0 || slot >= 8) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaEventRecord(b->slots[slot], b->stream));
    return HSDDP_OK;
}

int hsddp_batch_event_elapsed_ms(hsddp_batch* b, int slot0, int slot1, float* ms) {
    if (!b || !ms || slot0 < 0 || slot0 >= 8 || slot1 < 0 || slot1 >= 8) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaEventSynchronize(b->slots[slot1]));
    CK(cudaEventElapsedTime(ms, b->slots[slot0], b->slots[slot1]));
    return HSDDP_OK;
}

int hsddp_batch_get_counters(hsddp_batch* b, unsigned long long out[4]) {
    if (!b || !b->has_problems || !out) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaStreamSynchronize(b->stream));
    CK(cudaMemcpy(out, b->bp.counters, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    out[1] = b->n_solve_launches; out[2] = b->n_step_launches; out[3] = 0;
    return HSDDP_OK;
}

int hsddp_batch_get_speculation(hsddp_batch* b, unsigned long long out[3]) {
    if (!b || !b->has_problems || !out) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaStreamSynchronize(b->stream));
    CK(cudaMemcpy(out, b->bp.counters + 1, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return HSDDP_OK;
}

int hsddp_batch_get_profile(hsddp_batch* b, unsigned long long out[16]) {
    if (!b || !b->has_problems || !out) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaStreamSynchronize(b->stream));
    CK(cudaMemcpy(out, b->bp.counters + 8, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return HSDDP_OK;
}

int hsddp_batch_reset_counters(hsddp_batch* b) {
    if (!b || !b->has_problems) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(b->device));
    CK(cudaMemsetAsync(b->bp.counters, 0, 32 * sizeof(unsigned long long), b->stream));
    b->n_solve_launches = 0; b->n_step_launches = 0;
    return HSDDP_OK;
}

int hsddp_fp64_peak_tflops(int device, int kind, double* tflops) {
    if (!tflops) return HSDDP_ERR_ARG;
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 20000;
    double* d = nullptr;
    CK(cudaMalloc(&d, sizeof(double) * blocks * threads));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(e0));
        if (kind == 0) k_dfma_probe<<<blocks, threads>>>(d, iters);
        else k_dmma_probe<<<blocks, threads>>>(d, iters);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        const double flop = (kind == 0) ? (double)blocks * threads * iters * 8.0 * 2.0
                                        : (double)blocks * (threads / 32) * iters * 4.0 * (8.0 * 8.0 * 4.0 * 2.0);
        if (rep > 0) best = std::max(best, flop / (ms * 1e-3) / 1e12);
    }
    CK(cudaEventDestroy(e0));
    CK(cudaEventDestroy(e1));
    CK(cudaFree(d));
    *tflops = best;
    return HSDDP_OK;
}

}  // extern "C"
