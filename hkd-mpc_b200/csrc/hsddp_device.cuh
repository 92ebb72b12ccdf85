// Device-side data layout and per-problem building blocks of the batched HS-DDP
// solver.  One thread block owns one problem; every *_block function below is
// executed by the whole block (kThreads threads) and contains block barriers, so
// it must be called under block-uniform control flow.
//
// Reference functions restated here (all FP64, <double,24,24,0> instantiation):
//   SinglePhase::hybrid_rollout      HSDDPSolver/source/SinglePhase.cpp:182-233
//   SinglePhase::compute_cost        :236-262   (+ ReB/AL folding :370-378,402-411)
//   SinglePhase::LQ_approximation    :265-296   (+ :381-394,414-426)
//   SinglePhase::linear_rollout      :145-178
//   MultiPhaseDDP::{hybrid_rollout,linear_rollout,compute_cost,LQ_approximation,
//     update_nominal_trajectory,measure_dynamics_feasibility,update_AL_params,update_REB_params}
//                                     HSDDPSolver/source/MultiPhaseDDP.cpp:20-95,431-448,487-529
//   costs / constraints / reset map  HKDMPC/HKD-TrajOpt/{HKDCost.h,HKDCost.cpp,HKDConstraints.cpp,HKDReset.h}
//   ReB / AL formulas and updates    HSDDPSolver/header/ConstraintsBase.h:168-263,349-399
// The Riccati recursion lives in hsddp_sweep.cuh, the iteration control in hsddp_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstddef>
#include "../../include/hsddp_b200.h"
#include "hkd_model.cuh"

// Optional per-phase cycle accounting (build with -DHSDDP_PROFILE): thread 0 of every block adds the
// clock64() deltas between PROF_MARK points into BatchPtrs::counters[8 + slot].
#ifdef HSDDP_PROFILE
#define PROF_DECL long long prof_t0_ = clock64();
#define PROF_MARK(sm, slot)                                                         \
    do {                                                                            \
        if (threadIdx.x == 0) {                                                     \
            const long long t1_ = clock64();                                        \
            (sm).profacc[slot] += (unsigned long long)(t1_ - prof_t0_);             \
            prof_t0_ = t1_;                                                         \
        }                                                                           \
    } while (0)
#else
#define PROF_DECL
#define PROF_MARK(sm, slot) do { } while (0)
#endif

namespace hsddp {

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr int MAXPH = HSDDP_MAX_PHASES;

// per-stage LQ record.  In HBM (BatchPtrs::lq) it is compact, CR_STRIDE doubles: the 111 structural entries of
// [A - I | B_r] (hkd_model.cuh), then lx, lu and the ReB Hessian blocks.  In shared memory (Smem::rec) the sweep
// works on the dense tile R[12][44] followed by the same three vectors (LQ_* offsets); cp.async scatters the compact
// entries into the dense tile (8-byte copies) and copies the vectors (16-byte copies).
constexpr int CR_R = 0;                           // [112] compact [A - I | B_r] entries (hkd::kCrSize)
constexpr int CR_LX = CR_R + hkd::kCrSize;        // [24]
constexpr int CR_LU = CR_LX + 24;                 // [24]
constexpr int CR_LUU = CR_LU + 24;                // [4][3][3] ReB Hessian blocks per leg (dt folded in)
constexpr int CR_STRIDE = 200;                    // 196 used; 1600 bytes, 16-byte aligned
constexpr int LQ_R = 0;                           // [12][44] rows 0..11 of [A - I | B_r] (hkd::kRld = 44)
constexpr int LQ_LX = LQ_R + hkd::kRSize;         // [24]
constexpr int LQ_LU = LQ_LX + 24;                 // [24]
constexpr int LQ_LUU = LQ_LU + 24;                // [4][3][3]
constexpr int LQ_STRIDE = 616;                    // 612 used
// Row offsets of the shared-memory tiles of the sweep.  Rows are laid out in PAIRS: row r of a 24-wide tile starts at
// ro(r) = 24 r + 4 (r / 2) doubles, i.e. the start residues mod 16 doubles cycle through 0, 8, 4, 12.  That makes both
// fragment access patterns of the FP64 m8n8k4 MMA free of bank conflicts (no uniform row stride can: the 8-byte operand
// loads need stride = 4 or 12 mod 16, the 16-byte accumulator loads/stores need 8 mod 16):
//   * operand loads: rows t, t+4, t+8.. x eight consecutive columns, one half-warp = 4 rows with residues {0, 8, 4, 12}
//   * accumulator tiles: rows g x column pairs, one quarter-warp = rows 2q, 2q+1, whose starts differ by 24 = 8 mod 16
// ro() is additive over multiples of two rows: ro(r + 2m) = ro(r) + 52 m.  zo() is the same idea for the 16-wide Z.
__host__ __device__ constexpr int ro(int r) { return 26 * r - 2 * (r & 1); }
__host__ __device__ constexpr int zo(int r) { return 22 * r + 2 * (r & 1); }
constexpr int RO4 = ro(4), RO8 = ro(8), ZO4 = zo(4), ZO8 = zo(8);
constexpr int kQuuPad = 4;                        // Quu starts 4 mod 16 doubles after Qux: the Gauss-Jordan column loads
                                                  // (12 Quu columns + Qux columns in one half-warp) then hit distinct banks
constexpr int kSweepDoubles = 2 * ro(24) + zo(24) + ro(16) + kQuuPad + ro(12) + 2 * 616;  // H, Y, Z, Qux, Quu, rec: contiguous, free outside the sweep
// per-phase terminal record
constexpr int TQ_PHIX = 0;   // [24]
constexpr int TQ_HX = 24;    // [4][24] touchdown-constraint gradients, by leg
constexpr int TQ_WH = 120;   // [4] AL Hessian weights sigma(1+h)+lambda (0: no constraint on that leg)
constexpr int TQ_JC = 124;   // [4][3][6] foot Jacobians (d/d eul, d/d qleg) at the phase's terminal state (reset-map Jacobian)
constexpr int TQ_STRIDE = 200;

struct DevSchedule {
    int n_phases, n_stages, n_nodes, _pad;
    int horizon[MAXPH];
    int node_off[MAXPH];    // first state node of the phase
    int stage_off[MAXPH];   // first control stage of the phase
    unsigned cmask[MAXPH];  // contact bit mask of the phase
    unsigned nmask[MAXPH];  // contact after the phase
    long long ref_off;      // node offset of this schedule inside the concatenated reference arrays
    double dt;
    unsigned char ph_of_stage[HSDDP_MAX_STAGES];           // filled by layout_phases
    unsigned char ph_of_node[HSDDP_MAX_STAGES + MAXPH];
    // shooting set of the phase: nodes 0 .. ss_size-1 (SinglePhase::update_SS_config).  horizon + 1 = every node (what
    // HKDProblem::initialization sets); after a receding-horizon update the LAST phase can have fewer: 0 for a phase created
    // by HKDProblem::update until its horizon exceeds 2 (HKDProblem.cpp:212-218)
    unsigned char ss_size[MAXPH];
    // leg masks of the touchdown-constraint OBJECTS of the phase (add_tconstr_one_phase runs again when a phase reaches
    // its end during an update, so a phase can carry two objects, each with its own AL parameters)
    unsigned char tdmask[2][MAXPH];
};
static_assert(sizeof(DevSchedule) % 4 == 0, "bind_problem copies the schedule word by word");

// The phase layout of a schedule from horizon[0 .. n_phases): phase p has horizon[p] stages and horizon[p] + 1 nodes, laid
// out one phase after the other (node_off, stage_off, ph_of_stage, ph_of_node and the counts).  False, with the table partly
// written, when a phase is empty or the schedule has more than stage_cap stages or node_cap nodes.  The caps must not exceed
// the table sizes, HSDDP_MAX_STAGES and HSDDP_MAX_STAGES + MAXPH.
__host__ __device__ inline bool layout_phases(DevSchedule& d, int n_phases, int stage_cap, int node_cap) {
    int so = 0, no = 0;
    for (int p = 0; p < n_phases; ++p) {
        const int h = d.horizon[p];
        if (h < 1 || so + h > stage_cap || no + h + 1 > node_cap) return false;
        d.node_off[p] = no; d.stage_off[p] = so;
        for (int k = 0; k < h; ++k) d.ph_of_stage[so + k] = (unsigned char)p;
        for (int k = 0; k <= h; ++k) d.ph_of_node[no + k] = (unsigned char)p;
        no += h + 1; so += h;
    }
    d.n_phases = n_phases; d.n_stages = so; d.n_nodes = no;
    return true;
}

// legs that go from swing (not in the phase's contact mask) to stance (in the contact after it): one touchdown-constraint object
__host__ __device__ inline unsigned touchdown_legs(unsigned cmask, unsigned nmask) { return ~cmask & nmask & 15u; }

// solver scalars of one problem (MultiPhaseDDP.h:92-104) + bookkeeping
struct SolverState {
    double actual_cost, merit, feas, dV_1, dV_2;
    double max_tconstr_prev, max_pconstr_prev, max_tconstr, max_pconstr, merit_rho;
    double reg;
    int rollout_ok, sweep_ok;
};

// iteration-control state of one problem: the locals of MultiPhaseDDP::solve (MultiPhaseDDP.cpp:232-428),
// kept in a struct so that solve() can be resumed phase by phase (one kernel per phase) or run in one go
struct SolveCtl {
    int iter, iter_ou, iter_in, n_sweeps, n_trials, status;
    int active;  // 1 while the solve is running
    int have_trial;  // 1: trial_cost / trial_feas hold the last compute_cost of this outer iteration's line search
    int max_al, max_ddp;  // iteration budget of this solve: the options' max_AL_iter / max_DDP_iter or the problem's override
    double cost0, feas0;
    double trial_cost, trial_feas;
};

// one candidate of a speculated backward sweep: ok = 1 PD, 0 failed, -1 not run (its regularisation is past the limit);
// dV_1 / dV_2 as the sweep left them
struct SpecRec {
    int ok, _pad;
    double dV_1, dV_2;
};

struct BatchPtrs {
    int n_problems, max_stages, max_nodes, _pad;
    const DevSchedule* sched;
    const int* sched_id;
    const double *xr, *ur, *prel, *xinit;  // concatenated over schedules, per node
    double* x0;                            // [P][24]
    // problem-major workspace
    double *Xbar, *X, *Xsim_t, *Defect, *dX;  // [P][max_nodes][24]
    double *Ubar, *U, *U_t, *dU;              // [P][max_stages][24]
    double* KdX;                              // [P][max_stages][12] K_r dX of the last linear rollout (reduced control index)
    double* K;                                // [P][max_stages][24][12] compact gains, transposed: KT[j][c] = K_r[c][j] (c <-> coupled control of leg c/3)
    double* lq;                               // [P][max_stages][CR_STRIDE] compact stage records
    double* tq;                               // [P][MAXPH][TQ_STRIDE]
    double* gcon;                             // [P][max_stages][20]
    double* reb;                              // [P][max_stages][20][2]  (eps, delta)
    double* hcon;                             // [P][MAXPH][4]
    double* al;                               // [P][MAXPH][2][4][2]     (sigma, lambda) per touchdown-constraint object and leg
    double* g0h0;                             // [P][600] value gradient / Hessian at the first node
    SolverState* state;                       // [P]
    SolveCtl* ctl;                            // [P]
    // phased driver: the problems of this round are active[0 .. *n_active), survivors are appended to next_active /
    // next_count.  All four live in HBM, so a whole solve is queued without a host round trip: every round is launched
    // with the group's full grid and blocks beyond *n_active leave at once.  active == nullptr: problem = blockIdx.x.
    const int* active;
    const int* n_active;
    int* next_active;
    int* next_count;
    int* zero_count;                          // counter the first kernel of a round clears for the round after next (nullptr: none)
    int sweep_w1_min;                         // phased driver: rounds with at least this many problems run k_sweep_w1 instead of k_phase<PH_SWEEP> (0: never)
    int lr_external;                          // phased driver: the linear rollout of the iteration was done by k_lr_w1 (the forward phase skips it)
    int _pad2;
    // concurrent line search of the latency kernel (k_solve_lat4): per problem and step size, the arrays a trial writes
    // (X, Defect, Xsim: [P][4][max_nodes][24]; U, U scratch: [P][4][max_stages][24]; gcon [P][4][max_stages][20];
    // hcon [P][4][MAXPH][4]); results [P][4][8] = cost, feas, max_pconstr, max_tconstr, rollout ok; mail [P] = 1 trial, 2 exit
    double *ls_X, *ls_Defect, *ls_Xsim, *ls_U, *ls_Ut, *ls_gcon, *ls_hcon, *ls_res;
    int* ls_mail;
    const int* order;                         // persistent kernel: the work queue visits problems in this order (nullptr: by index)
    const int* budget;                        // [P][2] max_AL_iter, max_DDP_iter of the next solve of a restarted problem, -1: the
                                              // solve's options (nullptr until a restart sets one, hsddp_batch_restart_problems)
    hsddp_info* info;                         // [P]
    hsddp_iter_record* trace;                 // [P][HSDDP_TRACE_CAP]
    unsigned long long* counters;             // [0] = sum over problems of (backward sweeps x stages)
    int* work_counter;                        // dynamic problem queue of the persistent kernel
    int* sm_slots;                            // [256] per-SM arrival counter: gives co-resident blocks distinct warp-role rotations
    hsddp_constraint_params cp;
    // phased driver, regularisation retries run side by side (DESIGN.md §4.3): in rounds the four-warp sweep takes, the prep lists
    // the problems that regularise (spec_list / spec_count, at most spec_cap, spec_entry[pid] = list entry or -1) and the sweep
    // runs candidates 1 .. spec_S - 1 of each on extra blocks (candidate 0 is the problem's own block).  Candidate j > 0 writes
    // its gains, feed-forward and g0h0 to its slice of spec_out; the last of the spec_S blocks to arrive (spec_arrive[entry])
    // commits.  spec_list == nullptr: off.
    int* spec_list;
    int* spec_count;
    int* spec_zero;                           // spec counter the prep clears for the next round (the zero_count scheme)
    int* spec_arrive;
    int* spec_entry;                          // [P]
    SpecRec* spec_rec;                        // [spec_cap][spec_S]
    double* spec_out;                         // [spec_cap][spec_S - 1] slices: K [max_stages][288] | dU [max_stages][24] | g0h0 [600]
    int spec_S, spec_cap;
};

// Shared-memory working set of one block.
struct Smem;
struct __align__(16) Smem {
    // --- sweep tiles; contiguous, reused as streaming buffers by the linear rollout ---
    double H[ro(24)], Y[ro(24)];  // [24][24], row r at ro(r)
    double Z[zo(24)];             // H B_r [24][16], row r at zo(r); after P2 the same storage holds K_r^T [24][12]
    double Qux[ro(16) + kQuuPad]; // Qux_r [16][24], row r at ro(r)
    double Quu[ro(12)];           // Quu_r [12][24], row r at ro(r)
    double rec[2][LQ_STRIDE];  // stage records, cp.async double buffer
    // --- vectors ---
    double dfc2[2][24];
    double G[24], Gn[24], Qx[24], Qu[24], wu[24], vtmp[24], vtmp2[24];
    double lxxd[24], lxxTd[24], lxxw[12], lxxTw[12];
    double swdt[4];            // per-phase constants (1-c_l) dt
    double swc[16];            // (1-c_l) dt per reduced control column c = 3l+j, zero for c >= 12
    double red[kThreads];
    DevSchedule sc;
    SolverState st;
    SolveCtl ctl;
    hsddp_constraint_params cp;
    hsddp_options opt;
    // per-problem base pointers
    double *Xbar, *X, *Xsim_t, *Defect, *dX, *Ubar, *U, *U_t, *dU, *KdX, *K, *lqg, *tq, *gcon, *reb, *hcon, *al, *g0h0;
    const double *xr, *ur, *prel, *xinit, *x0;
    unsigned long long* prof;
    unsigned long long profacc[16];
    int pid;
    int rot;   // warp-role rotation of this block (0..3), see virtual_tid()
    int flag;
    int ibuf[4];
    double dbuf[8];
};

static_assert(offsetof(Smem, dfc2) - offsetof(Smem, H) == sizeof(double) * kSweepDoubles, "kSweepDoubles must cover H..rec");
static_assert(32 * 113 <= kSweepDoubles, "LQ staging buffer does not fit");

// ---------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------
// Warp w of every block is scheduled on SM sub-partition w % 4.  The solver has serial roles
// (Gauss-Jordan pivot columns, the linear-rollout recursion, thread-per-stage passes that fill only
// the first two warps), so co-resident blocks would pile them onto the same scheduler.  Each block
// therefore works with a ROTATED thread index: role r is played by hardware warp (r - rot) & 3.
__device__ __forceinline__ int virtual_tid(const Smem& sm);
__device__ inline void assign_rotation(int* sm_slots, int& rot_out) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    rot_out = atomicAdd(&sm_slots[smid & 255], 1) & 3;
}
__device__ __forceinline__ int virtual_tid(const Smem& sm) { return (int)((threadIdx.x + 32u * (unsigned)sm.rot) & (kThreads - 1)); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// block-wide reductions; result valid in every thread.  Contains barriers.
// Flat pass over n elements, element e = tid, tid + kThreads, ...: `load(e)` gathers what the element needs from memory,
// `use(e, v)` computes and stores.  Measured with the loads of 2 and of 4 consecutive elements of a thread issued together
// (more loads in flight per thread): 316 and 332 ms per 16,384-problem solve against 300, single solve 6.2 and 5.7 ms
// against 4.2 (profiles/r02ab_*) -- the larger loop bodies cost more than the memory-level parallelism returns.
template <class LoadF, class UseF>
__device__ __forceinline__ void flat_pass(int n, int tid, LoadF&& load, UseF&& use) {
    for (int e = tid; e < n; e += kThreads) use(e, load(e));
}

template <int OP>  // 0 sum, 1 min, 2 max
__device__ __noinline__ double block_reduce(Smem& sm, double v) {
    v = (OP == 0) ? warp_sum(v) : (OP == 1) ? warp_min(v) : warp_max(v);
    __syncthreads();
    // partials are indexed by the ROLE of the warp, not by the hardware warp: the warp-role rotation of a block depends
    // on arrival order, and the result must not (bitwise run-to-run determinism)
    if ((threadIdx.x & 31) == 0) sm.red[virtual_tid(sm) >> 5] = v;
    __syncthreads();
    double r = sm.red[0];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) r = (OP == 0) ? r + sm.red[w] : (OP == 1) ? fmin(r, sm.red[w]) : fmax(r, sm.red[w]);
    return r;
}

// phase of a stage / node: byte tables built once per problem by bind_problem (sc lives in the block's Smem)
__device__ __forceinline__ void phase_of_stage(const DevSchedule& sc, int s, int& ph, int& k) {
    ph = sc.ph_of_stage[s];
    k = s - sc.stage_off[ph];
}
__device__ __forceinline__ void phase_of_node(const DevSchedule& sc, int n, int& ph, int& k) {
    ph = sc.ph_of_node[n];
    k = n - sc.node_off[ph];
}

// tracking weights (HKDCost.h:11-37), table driven so that the cost / LQ passes can stay rolled
// (the solver kernel is instruction-fetch bound; see tools/code_size.py)
__constant__ double c_wQ[12] = {1, 4, 5, 1, 1, 30, .2, .2, .2, 4, 1, .5};
__constant__ double c_wQfScale[24] = {1, 1, 2, 1, 1, 20, .3, .3, .3, 1, 3, 1, .01, .01, .01, .01, .01, .01, .01, .01, .01, .01, .01, .01};
__device__ __forceinline__ double weight_Q(int j, unsigned cmask) {
    return (j < 12) ? c_wQ[j] : .2 * (double)(1 - (int)((cmask >> ((j - 12) / 3)) & 1u));
}
__device__ __forceinline__ double weight_Qf(int j, unsigned cmask) { return (20 * c_wQfScale[j]) * weight_Q(j, cmask); }
__device__ __forceinline__ double weight_R(int j) { return j < 12 ? .2 : .1; }
// foot-placement regulariser weight 20*diag(3c, c, 0) (HKDCost.h:56-69)
__device__ __forceinline__ double weight_foot(int l, int j, unsigned cmask) {
    const double c = (double)((cmask >> l) & 1u);
    return ((j == 0) ? 3 * c : (j == 1) ? c : 0.0) * 20;
}
// single out-of-line copies of the leg kinematics (code size, see tools/code_size.py)
__device__ __noinline__ void foot_position_nl(const double* x, int l, double* pf) { hkd::foot_position(x + 3, x, x + 12 + 3 * l, l, pf); }
__device__ __noinline__ void foot_jacobian_nl(const double* x, int l, double* Jc) { hkd::foot_jacobian_compact(x, x + 12 + 3 * l, l, Jc); }

__device__ inline void bind_problem(Smem& sm, const BatchPtrs& bp, int pid) {
    if (threadIdx.x == 0) {
        sm.pid = pid;
        const size_t sn = (size_t)bp.max_nodes * 24, ss = (size_t)bp.max_stages * 24;
        sm.Xbar = bp.Xbar + pid * sn; sm.X = bp.X + pid * sn; sm.Xsim_t = bp.Xsim_t + pid * sn;
        sm.Defect = bp.Defect + pid * sn; sm.dX = bp.dX + pid * sn;
        sm.Ubar = bp.Ubar + pid * ss; sm.U = bp.U + pid * ss; sm.U_t = bp.U_t + pid * ss; sm.dU = bp.dU + pid * ss;
        sm.K = bp.K + (size_t)pid * bp.max_stages * 288;
        sm.KdX = bp.KdX + (size_t)pid * bp.max_stages * 12;
        sm.lqg = bp.lq + (size_t)pid * bp.max_stages * CR_STRIDE;
        sm.tq = bp.tq + (size_t)pid * MAXPH * TQ_STRIDE;
        sm.gcon = bp.gcon + (size_t)pid * bp.max_stages * 20;
        sm.reb = bp.reb + (size_t)pid * bp.max_stages * 40;
        sm.hcon = bp.hcon + (size_t)pid * MAXPH * 4;
        sm.al = bp.al + (size_t)pid * MAXPH * 16;
        sm.g0h0 = bp.g0h0 + (size_t)pid * 600;
        sm.x0 = bp.x0 + (size_t)pid * 24;
        sm.prof = bp.counters + 8;
        sm.cp = bp.cp;
        sm.st = bp.state[pid];
        sm.ctl = bp.ctl[pid];
    }
    const DevSchedule* src = bp.sched + bp.sched_id[pid];
    const int nw = (int)(sizeof(DevSchedule) / sizeof(int));
    for (int i = threadIdx.x; i < nw; i += kThreads) ((int*)&sm.sc)[i] = ((const int*)src)[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        const size_t roff = (size_t)sm.sc.ref_off;
        sm.xr = bp.xr + roff * 24; sm.ur = bp.ur + roff * 24; sm.prel = bp.prel + roff * 12; sm.xinit = bp.xinit + roff * 24;
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------
// reset map (HKDReset.h:41-75) — single thread
// ---------------------------------------------------------------------------
__device__ inline void resetmap_thread(const double* x, unsigned c, unsigned cn, double* xn) {
    for (int i = 0; i < 24; ++i) xn[i] = x[i];
    for (int l = 0; l < 4; ++l) {
        const bool cl = (c >> l) & 1u, nl = (cn >> l) & 1u;
        if (cl && !nl) { xn[12 + 3 * l] = 0.0; xn[13 + 3 * l] = -0.8; xn[14 + 3 * l] = 1.7; }
        if (!cl && nl) {
            double pf[3];
            foot_position_nl(x, l, pf);
            xn[12 + 3 * l] = 1.0 * pf[0]; xn[13 + 3 * l] = 1.0 * pf[1]; xn[14 + 3 * l] = 0.0 * pf[2];
        }
    }
}

// dense Px (HKDReset.h:78-136), ROW-major into P[r * S + c] (S = row stride in doubles).  Jc: the foot Jacobians cached
// by the LQ approximation in the phase's terminal record ([4][3][6]: d/d eul, d/d qleg per leg).
__device__ inline void resetmap_partial_block(const double* Jc_all, unsigned c, unsigned cn, double* P) {
    for (int e = threadIdx.x; e < 576; e += kThreads) P[ro(e / 24) + e % 24] = ((e % 24) == (e / 24)) ? 1.0 : 0.0;
    __syncthreads();
    if (threadIdx.x < 12) {
        const int l = threadIdx.x / 3, r = threadIdx.x % 3;
        const bool cl = (c >> l) & 1u, nl = (cn >> l) & 1u;
        const int row = 12 + 3 * l + r;
        double* Prow = P + ro(row);
        if (cl && !nl) Prow[row] = 0.0;
        if (!cl && nl) {
            const double* Jc = Jc_all + 18 * l + 6 * r;
            const double cmap = (r == 2) ? 0.0 : 1.0;
            Prow[row] = 0.0;
            for (int cc = 0; cc < 3; ++cc) {
                Prow[cc] = cmap * Jc[cc];                          // d/d eul
                Prow[3 + cc] = cmap * ((r == cc) ? 1.0 : 0.0);     // d/d pos
                Prow[12 + 3 * l + cc] = cmap * Jc[3 + cc];         // d/d qleg
            }
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------
// hybrid rollout (MultiPhaseDDP::hybrid_rollout + SinglePhase::hybrid_rollout).
// With multiple shooting every node is a shooting node (update_SS_config(horizon+1),
// HKDProblem.cpp:104), so all stages are rolled out concurrently.  Pass 1 writes
// trial controls / simulated states; the commit pass reproduces the reference's
// partial-update semantics when a stage diverges (SURVEY.md Q16).
// ---------------------------------------------------------------------------
// LINEARISED = true (inside solve(), where the linear rollout of the same iteration precedes every trial): with
// multiple shooting the trial states are X = Xbar + eps dX, so the feedback term K (X - Xbar) equals eps (K dX), and
// K_r dX was already formed by the linear rollout (sm.KdX).  The trial then needs no gain at all: one fused
// multiply-add per control instead of re-reading 2.3 KB of gains per stage and trial.  Differs from the literal form
// by the rounding of (Xbar + eps dX) - Xbar only.  LINEARISED = false evaluates the literal form (step-level API,
// where the caller decides what precedes a rollout).
// Nodes OUTSIDE the shooting set are propagated: X[k] = Xsim[k] (X[0] = x_init when the set is empty), and their controls see
// the true feedback K (X - Xbar) (SinglePhase.cpp:185-220).  HKDProblem::initialization makes every node a shooting node, so
// with multiple shooting this path is empty; it is taken
//   * after a receding-horizon update, by the LAST phase while its shooting set is short (DevSchedule::ss_size): <= 3 stages;
//   * with single shooting (option.MS = false): every phase is propagated from its first node (which stays a shooting node:
//     SS_set is non-empty and starts at 0, SinglePhase.cpp:187-193).
// One thread walks phase `ph` from node `kf` on, after the parallel pass of hybrid_rollout_block; out of line so that its
// local arrays cost the common path nothing.  Returns the first diverged stage (0x7fffffff: none).
__device__ __noinline__ int rollout_sequential_phase(Smem& sm, double eps, double* xs, double* xd, bool dev_in_smem, int ph, int kf, int ss_eff) {
    const DevSchedule& sc = sm.sc;
    const int hz = sc.horizon[ph];
    const unsigned cm = sc.cmask[ph];
    for (int k = kf; k <= hz; ++k) {
        const int n = sc.node_off[ph] + k, s = sc.stage_off[ph] + k;
        double* x = xs + 24 * n;
        if (k >= ss_eff) {
            const double* xsim = (k == 0) ? sm.Xsim_t + 24 * n : (dev_in_smem ? xd + 24 * (n - 1) : sm.Xsim_t + 24 * n);
            for (int j = 0; j < 24; ++j) x[j] = xsim[j];
        }
        if (k == hz) break;
        double dxl[24], ul[24];
        for (int j = 0; j < 24; ++j) { dxl[j] = x[j] - sm.Xbar[24 * n + j]; ul[j] = sm.Ubar[24 * s + j] + eps * sm.dU[24 * s + j]; }
        const double* KT = sm.K + 288 * (size_t)s;
        for (int c = 0; c < 12; ++c) {
            double acc = 0.0;
            for (int j = 0; j < 24; ++j) acc = fma(KT[12 * j + c], dxl[j], acc);
            ul[((cm >> (c / 3)) & 1u) ? c : 12 + c] += acc;  // the coupled control of the leg
        }
        double* slot = dev_in_smem ? xd + 24 * n : sm.Xsim_t + 24 * (n + 1);
        for (int j = 0; j < 24; ++j) sm.U_t[24 * s + j] = ul[j];
        hkd::dynamics(x, ul, sc.dt, cm, slot);
        double nrm2 = 0.0;
        for (int j = 0; j < 24; ++j) nrm2 = fma(slot[j], slot[j], nrm2);
        if (sqrt(nrm2) > 1e6) return s;
    }
    return 0x7fffffff;
}

template <bool LINEARISED>
__device__ inline bool hybrid_rollout_block(Smem& sm, double eps) {
    const DevSchedule& sc = sm.sc;
    const int tid = virtual_tid(sm), lane = tid & 31, warp = tid >> 5;
    const int N = sc.n_stages;
    const bool ms = sm.opt.MS != 0;
    PROF_DECL
    double* xs = sm.H;  // trial states of all nodes [n_nodes][24] (the sweep's tile storage is free here)
    // (a0) trial states X = Xbar + eps dX for every node, and the deviations X - Xbar the feedback acts on
    //      (kept in shared memory next to the states when both fit, else re-read from HBM)
    const bool dev_in_smem = sc.n_nodes * 48 <= kSweepDoubles;
    double* xd = xs + sc.n_nodes * 24;
    flat_pass(sc.n_nodes * 24, tid, [&](int e) { return make_double2(sm.Xbar[e], sm.dX[e]); },
                 [&](int e, const double2& v) {
                     const double x = v.x + eps * v.y;
                     xs[e] = x;
                     if (dev_in_smem && !LINEARISED) xd[e] = x - v.x;
                 });
    __syncthreads();
    // (a) controls: U = (Ubar + eps dU) + K (X - Xbar), one warp per stage.  K is stored compactly as
    //     K_r^T [24][12] (only the coupled control of each leg has a non-zero gain row, see hsddp_sweep.cuh).
    //     Lane (p, q) = (lane & 7, lane >> 3) accumulates the control pair (2p, 2p+1) over the state
    //     components j = q, q+4, ..: every load is a 16-byte piece of a 384-byte contiguous run of K.
    if (LINEARISED) {
        flat_pass(N * 24, tid,
                     [&](int e) {
                         const int s = e / 24, i = e % 24, c = i % 12;
                         const bool stance = (sc.cmask[sc.ph_of_stage[s]] >> (c / 3)) & 1u;
                         double3 v;
                         v.x = sm.Ubar[e]; v.y = sm.dU[e];
                         v.z = ((i < 12) == stance) ? sm.KdX[12 * s + c] : 0.0;  // the coupled control of the leg
                         return v;
                     },
                     [&](int e, const double3& v) {
                         const int s = e / 24, i = e % 24, c = i % 12;
                         int ph, k;
                         phase_of_stage(sc, s, ph, k);
                         const bool stance = (sc.cmask[ph] >> (c / 3)) & 1u;
                         double u = v.x + eps * v.y;
                         if ((i < 12) == stance) u += eps * v.z;
                         sm.U_t[e] = u;
                         if (dev_in_smem) xd[24 * (sc.node_off[ph] + k) + i] = u;
                     });
    } else {
        const int p = lane & 7, q = lane >> 3;
        const bool kact = p < 6;
        for (int s = warp; s < N; s += kWarps) {
            int ph, k;
            phase_of_stage(sc, s, ph, k);
            const int n = sc.node_off[ph] + k;
            const unsigned cm = sc.cmask[ph];
            const double2* K2 = reinterpret_cast<const double2*>(sm.K + 288 * (size_t)s) + p;
            double2 kv[6];
            double dv[6];
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                const int j = q + 4 * i;
                kv[i] = kact ? K2[6 * j] : make_double2(0.0, 0.0);
                dv[i] = dev_in_smem ? xd[24 * n + j] : xs[24 * n + j] - sm.Xbar[24 * n + j];
            }
            double ub = 0.0;
            if (lane < 24) ub = sm.Ubar[24 * s + lane] + eps * sm.dU[24 * s + lane];
            double ax = 0.0, ay = 0.0;
#pragma unroll
            for (int i = 0; i < 6; ++i) { ax = fma(kv[i].x, dv[i], ax); ay = fma(kv[i].y, dv[i], ay); }
            ax += __shfl_xor_sync(0xffffffffu, ax, 8);  ay += __shfl_xor_sync(0xffffffffu, ay, 8);
            ax += __shfl_xor_sync(0xffffffffu, ax, 16); ay += __shfl_xor_sync(0xffffffffu, ay, 16);
            // control i = lane: coupled iff (i < 12) == stance(leg); its gain row is reduced index c = i % 12
            const int c = lane % 12;
            const double vx = __shfl_sync(0xffffffffu, ax, c >> 1), vy = __shfl_sync(0xffffffffu, ay, c >> 1);
            __syncwarp();  // (every lane has read its state deviations: the slot is reused for the trial control)
            if (lane < 24) {
                const bool stance = (cm >> (c / 3)) & 1u;
                const double acc = ((lane < 12) == stance) ? ((c & 1) ? vy : vx) : 0.0;
                sm.U_t[24 * s + lane] = ub + acc;
                if (dev_in_smem) xd[24 * n + lane] = ub + acc;
            }
        }
    }
    __syncthreads();
    PROF_MARK(sm, 0);
    // (b) dynamics, one thread per stage; phase-initial simulated states.  With the shared-memory staging the stage's
    //     slot of `xd` holds its trial control on entry and its simulated successor state on exit (the strided
    //     per-thread accesses stay on chip); otherwise both go through HBM.
    int first_bad = 0x7fffffff;
    for (int s = tid; s < N; s += kThreads) {
        int ph, k;
        phase_of_stage(sc, s, ph, k);
        const int n = sc.node_off[ph] + k;
        double* slot = dev_in_smem ? xd + 24 * n : sm.Xsim_t + 24 * (n + 1);
        const double* usrc = dev_in_smem ? slot : sm.U_t + 24 * s;
        double ul[24];
#pragma unroll
        for (int j = 0; j < 24; ++j) ul[j] = usrc[j];
        hkd::dynamics(xs + 24 * n, ul, sc.dt, sc.cmask[ph], slot);
        double nrm2 = 0.0;
#pragma unroll
        for (int j = 0; j < 24; ++j) nrm2 = fma(slot[j], slot[j], nrm2);
        if (sqrt(nrm2) > 1e6 && k < (ms ? (int)sc.ss_size[ph] : 0)) first_bad = min(first_bad, s);  // (the other stages are redone in (b2))
    }
    if (tid >= 64 && tid < 64 + sc.n_phases) {
        const int ph = tid - 64;
        double* xi = sm.Xsim_t + 24 * sc.node_off[ph];
        if (ph == 0) {
            for (int j = 0; j < 24; ++j) xi[j] = sm.x0[j];
        } else {
            const int ne = sc.node_off[ph - 1] + sc.horizon[ph - 1];
            resetmap_thread(xs + 24 * ne, sc.cmask[ph - 1], sc.nmask[ph - 1], xi);
        }
    }
    // (b2) nodes outside the shooting set (rollout_sequential_phase): the last phase after a receding-horizon update, every
    //      phase with single shooting
    if (!ms || sc.ss_size[sc.n_phases - 1] < sc.horizon[sc.n_phases - 1] + 1) {
        __syncthreads();
        if (tid < sc.n_phases && sc.ss_size[tid] >= 1) {  // phases whose first node is a shooting node are independent of each other
            const int ss_eff = ms ? (int)sc.ss_size[tid] : 1;
            if (ss_eff <= sc.horizon[tid]) first_bad = min(first_bad, rollout_sequential_phase(sm, eps, xs, xd, dev_in_smem, tid, ms ? ss_eff : 0, ss_eff));
        }
        __syncthreads();
        if (tid >= 64 && tid < 64 + sc.n_phases && tid > 64) {  // phase-initial simulated states again: the previous phase's end state may have moved
            const int ph = tid - 64;
            const int ne = sc.node_off[ph - 1] + sc.horizon[ph - 1];
            resetmap_thread(xs + 24 * ne, sc.cmask[ph - 1], sc.nmask[ph - 1], sm.Xsim_t + 24 * sc.node_off[ph]);
        }
        __syncthreads();
        if (tid == 0 && sc.ss_size[sc.n_phases - 1] == 0)  // a last phase with an EMPTY shooting set starts from x_init
            first_bad = min(first_bad, rollout_sequential_phase(sm, eps, xs, xd, dev_in_smem, sc.n_phases - 1, 0, 0));
    }
    // first diverged stage in the reference's sequential order
    const int bad = (int)block_reduce<1>(sm, (double)first_bad);
    PROF_MARK(sm, 1);
    int bad_ph = sc.n_phases, bad_k = 0;
    if (bad != 0x7fffffff) phase_of_stage(sc, bad, bad_ph, bad_k);
    // (c) commit exactly what the sequential reference would have written
    for (int e = tid; e < sc.n_nodes * 24; e += kThreads) {
        const int n = e / 24;
        int ph, k;
        phase_of_node(sc, n, ph, k);
        if (ph < bad_ph || (ph == bad_ph && k <= bad_k)) {
            const double x = xs[e];
            sm.X[e] = x;
            if (ph < bad_ph) {  // compute_defect only after a complete phase
                const double xsim = (dev_in_smem && k > 0) ? xd[e - 24] : sm.Xsim_t[e];
                sm.Defect[e] = xsim - x;
            }
        }
    }
    double gmin = 0.0;
    const double mu = sm.cp.mu;
    flat_pass(N * 24, tid, [&](int e) { return sm.U_t[e]; },
                 [&](int e, double u) {
                     int ph, k;
                     phase_of_stage(sc, e / 24, ph, k);
                     if (ph < bad_ph || (ph == bad_ph && k <= bad_k)) sm.U[e] = u;
                 });
    for (int e = tid; e < N * 4; e += kThreads) {  // GRFConstraint::compute_violation, one (stage, leg) per thread
        const int s = e >> 2, l = e & 3;
        int ph, k;
        phase_of_stage(sc, s, ph, k);
        if (((sc.cmask[ph] >> l) & 1u) && (ph < bad_ph || (ph == bad_ph && k < bad_k))) {
            const double fx = sm.U_t[24 * s + 3 * l], fy = sm.U_t[24 * s + 3 * l + 1], fz = sm.U_t[24 * s + 3 * l + 2];
            double* g = sm.gcon + 20 * s + 5 * l;
            g[0] = fz; g[1] = -fx + mu * fz; g[2] = fx + mu * fz; g[3] = -fy + mu * fz; g[4] = fy + mu * fz;
            if (ph < bad_ph) gmin = fmin(gmin, fmin(fmin(fmin(g[0], g[1]), fmin(g[2], g[3])), g[4]));
        }
    }
    double hmax = 0.0;
    if (tid < sc.n_phases * 4) {  // TouchDownConstraint::compute_violation
        const int ph = tid >> 2, l = tid & 3;
        const bool td = ((sc.tdmask[0][ph] | sc.tdmask[1][ph]) >> l) & 1u;
        if (td && ph < bad_ph) {
            const int ne = sc.node_off[ph] + sc.horizon[ph];
            const double* xe = xs + 24 * ne;
            double pf[3];
            foot_position_nl(xe, l, pf);
            sm.hcon[4 * ph + l] = pf[2] - 0.0;
            hmax = fabs(pf[2]);
        }
    }
    const double gm = block_reduce<1>(sm, gmin);
    const double hm = block_reduce<2>(sm, hmax);
    if (tid == 0) {
        sm.st.actual_cost = 0.0;
        sm.st.max_pconstr = gm;
        sm.st.max_tconstr = hm;
        sm.st.rollout_ok = (bad_ph == sc.n_phases);
    }
    __syncthreads();
    PROF_MARK(sm, 2);
    return bad_ph == sc.n_phases;
}

// ---------------------------------------------------------------------------
// compute_cost + measure_dynamics_feasibility (MultiPhaseDDP.cpp:431-439,514-529)
// ---------------------------------------------------------------------------
__device__ inline void foot_rel_error(const double* x, const double* prel_r, double d[12]) {
#pragma unroll
    for (int l = 0; l < 4; ++l)
#pragma unroll
        for (int j = 0; j < 3; ++j) d[3 * l + j] = (x[12 + 3 * l + j] - x[3 + j]) - prel_r[3 * l + j];
}

__device__ inline void compute_cost_block(Smem& sm) {
    const DevSchedule& sc = sm.sc;
    const int tid = virtual_tid(sm);
    PROF_DECL
    const int N = sc.n_stages;
    const double dt = sc.dt;
    double csum = 0.0;
    // Every term of the running / terminal costs is a sum over (node or stage, component): the passes below walk
    // those index spaces flat, so all 128 threads work and every global access is coalesced.
    // (1) state tracking, (node, j): running 1/2 dt Q dx^2, terminal 1/2 Qf dx^2
    flat_pass(sc.n_nodes * 24, tid, [&](int e) { return make_double2(sm.X[e], sm.xr[e]); },
                 [&](int e, const double2& v) {
                     const int n = e / 24, j = e % 24;
                     const int ph = sc.ph_of_node[n];
                     const unsigned cm = sc.cmask[ph];
                     const bool terminal = (n - sc.node_off[ph]) == sc.horizon[ph];
                     const double dx = v.x - v.y;
                     csum += terminal ? 0.5 * ((dx * weight_Qf(j, cm)) * dx) : ((0.5 * dx * weight_Q(j, cm)) * dx) * dt;
                 });
    // (2) control effort, (stage, j)
    flat_pass(N * 24, tid,
                 [&](int e) {
                     const int s = e / 24, j = e % 24;
                     int ph, k;
                     phase_of_stage(sc, s, ph, k);
                     return make_double2(sm.U[e], sm.ur[24 * (sc.node_off[ph] + k) + j]);
                 },
                 [&](int e, const double2& v) {
                     const double du = v.x - v.y;
                     csum += ((0.5 * du * weight_R(e % 24)) * du) * dt;
                 });
    // (3) foot-placement regulariser, (node, leg component)
    flat_pass(sc.n_nodes * 12, tid,
                 [&](int e) {
                     const int n = e / 12, q = e % 12;
                     const double* x = sm.X + 24 * n;
                     double3 v;
                     v.x = x[12 + q]; v.y = x[3 + q % 3]; v.z = sm.prel[e];
                     return v;
                 },
                 [&](int e, const double3& v) {
                     const int n = e / 12, q = e % 12;
                     const int ph = sc.ph_of_node[n];
                     const unsigned cm = sc.cmask[ph];
                     const bool terminal = (n - sc.node_off[ph]) == sc.horizon[ph];
                     const double d = (v.x - v.y) - v.z;
                     const double w = weight_foot(q / 3, q % 3, cm);
                     csum += terminal ? (10 * d * w) * d : ((.5 * d * w) * d) * dt;
                 });
    // (4) relaxed-barrier terms of the GRF constraints, (stage, row)  (compute_ReB_cost, ConstraintsBase.h:204-222)
    if (sm.opt.ReB_active) {
        const double2* reb2 = reinterpret_cast<const double2*>(sm.reb);
        flat_pass(N * 20, tid,
                     [&](int i) {
                         double3 v;
                         v.x = 0.0; v.y = 0.0; v.z = 0.0;
                         if ((sc.cmask[sc.ph_of_stage[i / 20]] >> ((i % 20) / 5)) & 1u) {
                             const double2 p = reb2[i];  // (eps, delta)
                             v.x = sm.gcon[i]; v.y = p.x; v.z = p.y;
                         }
                         return v;
                     },
                     [&](int i, const double3& v) {
                         if (!((sc.cmask[sc.ph_of_stage[i / 20]] >> ((i % 20) / 5)) & 1u)) return;
                         const double g = v.x;
                         double barr;
                         if (g > v.z) barr = -hkd::log_nl(g);
                         else { const double z = (g - 2 * v.z) / v.z; barr = .5 * (z * z - 1); barr -= hkd::log_nl(v.z); }
                         csum += dt * (v.y * barr);
                     });
    }
    // (5) augmented-Lagrangian terms of the touchdown constraints, (phase, leg)  (compute_AL_cost, ConstraintsBase.h:374-385)
    if (sm.opt.AL_active && tid < sc.n_phases * 4) {
        const int ph = tid >> 2, l = tid & 3;
        const double h = sm.hcon[4 * ph + l];
#pragma unroll
        for (int ob = 0; ob < 2; ++ob)
            if ((sc.tdmask[ob][ph] >> l) & 1u) {
                const double sigma = sm.al[16 * ph + 8 * ob + 2 * l], lambda = sm.al[16 * ph + 8 * ob + 2 * l + 1];
                csum += 0.5 * sigma * h * h + lambda * h;
            }
    }
    double dsum = 0.0;
    flat_pass(sc.n_nodes * 24, tid, [&](int e) { return sm.Defect[e]; }, [&](int, double d) { dsum += d * d; });
    const double cost = block_reduce<0>(sm, csum);
    const double f2 = block_reduce<0>(sm, dsum);
    if (tid == 0) { sm.st.actual_cost = cost; sm.st.feas = sqrt(f2); }
    __syncthreads();
    PROF_MARK(sm, 3);
}

// ---------------------------------------------------------------------------
// LQ_approximation: two threads per stage write the compact record; one thread per
// phase the terminal record.
// ---------------------------------------------------------------------------
__device__ inline void lq_approximation_block(Smem& sm) {
    const DevSchedule& sc = sm.sc;
    const int tid = virtual_tid(sm);
    PROF_DECL
    const int N = sc.n_stages;
    const double dt = sc.dt;
    // (0) terminal records, one thread per phase ON THE FOURTH WARP, before anything else: the thread's work is a long
    //     dependent chain (foot Jacobians, AL weights), so it runs while warps 0 and 1 compute the dynamics Jacobians of
    //     (1) instead of after them with the whole block waiting at the last barrier (that wait was 23 % of the prep
    //     kernel's stall samples, profiles/r02x_*).  Jacobians and the touchdown gradients stay in registers; only the
    //     non-zero entries of hx (columns 0..2, 5 and the leg's three foot columns) feed Phix.
    if (tid >= 96 && tid - 96 < sc.n_phases) {
        const int ph = tid - 96;
        const unsigned cm = sc.cmask[ph];
        const int n = sc.node_off[ph] + sc.horizon[ph];
        const double* x = sm.X + 24 * n;
        const double* xr = sm.xr + 24 * n;
        double* rec = sm.tq + ph * TQ_STRIDE;
        double phix[24];
        for (int j = 0; j < 24; ++j) phix[j] = weight_Qf(j, cm) * (x[j] - xr[j]);
        double d[12];
        foot_rel_error(x, sm.prel + 12 * n, d);
        for (int l = 0; l < 4; ++l) {
            const double c = (double)((cm >> l) & 1u);
            for (int j = 0; j < 3; ++j) {
                const double w = 20 * c * weight_foot(l, j, cm);
                phix[3 + j] += -(w * d[3 * l + j]);
                phix[12 + 3 * l + j] += w * d[3 * l + j];
            }
        }
        for (int l = 0; l < 4; ++l) {
            double* hx = rec + TQ_HX + 24 * l;
            const bool rm = !((cm >> l) & 1u) && ((sc.nmask[ph] >> l) & 1u);  // reset map moves this leg's foot (touchdown)
            const unsigned tdo = ((sc.tdmask[0][ph] >> l) & 1u) | (((sc.tdmask[1][ph] >> l) & 1u) << 1);  // constraint objects on this leg
            const bool al = tdo && sm.opt.AL_active;
            double h = 0.0, sg[2] = {0.0, 0.0}, lm[2] = {0.0, 0.0};
            if (al) {  // (loads issued before the Jacobian's long chain)
                h = sm.hcon[4 * ph + l];
                for (int ob = 0; ob < 2; ++ob)
                    if ((tdo >> ob) & 1u) { sg[ob] = sm.al[16 * ph + 8 * ob + 2 * l]; lm[ob] = sm.al[16 * ph + 8 * ob + 2 * l + 1]; }
            }
            double Jc[18];
            if (rm || tdo) {  // foot Jacobian, cached for the sweep and the linear rollout (reset-map Jacobian) and used by the AL terms
                foot_jacobian_nl(x, l, Jc);
                for (int c = 0; c < 18; ++c) rec[TQ_JC + 18 * l + c] = Jc[c];
            }
            double wh = 0.0;
            for (int j = 0; j < 24; ++j) hx[j] = 0.0;
            if (al) {
                double wg = 0.0;
                for (int ob = 0; ob < 2; ++ob)
                    if ((tdo >> ob) & 1u) {
                        wg += sg[ob] * h + lm[ob];
                        wh += sg[ob] * (1 + h) + lm[ob];  // Q3
                    }
                for (int c = 0; c < 3; ++c) {
                    hx[c] = Jc[2 * 6 + c]; hx[12 + 3 * l + c] = Jc[2 * 6 + 3 + c];
                    phix[c] += wg * Jc[2 * 6 + c];
                    phix[12 + 3 * l + c] += wg * Jc[2 * 6 + 3 + c];
                }
                hx[5] = 1.0;
                phix[5] += wg * 1.0;
            }
            rec[TQ_WH + l] = wh;
        }
        for (int j = 0; j < 24; ++j) rec[TQ_PHIX + j] = phix[j];
    }
    // (1) dynamics Jacobians.  Two threads share a stage (disjoint halves of the record, hkd_model.cuh) and write its
    //     compact record into shared memory (row stride 113 doubles: the per-thread rows do not collide on banks);
    //     after each pass of 32 stages all threads copy the rows out with coalesced stores.
    {
        double* stg = sm.H;  // the sweep's tile storage is free here (kSweepDoubles >= 32 * 113)
        for (int s0 = 0; s0 < N; s0 += 32) {
            const int s = s0 + (tid & 31);
            if (tid < 64 && s < N) {
                int ph, k;
                phase_of_stage(sc, s, ph, k);
                const int n = sc.node_off[ph] + k;
                double* row = stg + 113 * (tid & 31);
                if (tid < 32) hkd::dynamics_partial_parts<1>(sm.X + 24 * n, sm.U + 24 * s, dt, sc.cmask[ph], row);
                else hkd::dynamics_partial_parts<2>(sm.X + 24 * n, sm.U + 24 * s, dt, sc.cmask[ph], row);
            }
            __syncthreads();
            const int ns = min(32, N - s0);
            for (int e = tid; e < ns * hkd::kCrNnz; e += kThreads) {
                const int r = e / hkd::kCrNnz, i = e % hkd::kCrNnz;
                sm.lqg[(size_t)(s0 + r) * CR_STRIDE + CR_R + i] = stg[113 * r + i];
            }
            __syncthreads();
        }
    }
    // (2) cost gradients, flat over (stage, component), loads batched (flat_pass): the lu of the joint-velocity commands
    //     (12 per stage); lx of every component but the position (21); lx of the position rows (3), which accumulate the
    //     foot-placement regulariser over the legs in order.
    flat_pass(N * 12, tid,
                 [&](int e) {
                     const int s = e / 12, i = 12 + e % 12;
                     int ph, k;
                     phase_of_stage(sc, s, ph, k);
                     return make_double2(sm.U[24 * s + i], sm.ur[24 * (sc.node_off[ph] + k) + i]);
                 },
                 [&](int e, const double2& v) {
                     const int s = e / 12, i = 12 + e % 12;
                     sm.lqg[(size_t)s * CR_STRIDE + CR_LU + i] = (dt * weight_R(i)) * (v.x - v.y);
                 });
    flat_pass(N * 21, tid,
                 [&](int e) {
                     const int s = e / 21, jr = e % 21, j = jr < 3 ? jr : jr + 3;
                     int ph, k;
                     phase_of_stage(sc, s, ph, k);
                     const int n = sc.node_off[ph] + k;
                     const double* x = sm.X + 24 * n;
                     double4 v;
                     v.x = x[j]; v.y = sm.xr[24 * n + j]; v.z = 0.0; v.w = 0.0;
                     if (j >= 12) { v.z = x[3 + (j - 12) % 3]; v.w = sm.prel[12 * n + j - 12]; }
                     return v;
                 },
                 [&](int e, const double4& q) {
                     const int s = e / 21, jr = e % 21, j = jr < 3 ? jr : jr + 3;
                     const unsigned cm = sc.cmask[sc.ph_of_stage[s]];
                     double v = (dt * weight_Q(j, cm)) * (q.x - q.y);
                     if (j >= 12) {
                         const int l = (j - 12) / 3, jj = (j - 12) % 3;
                         const double c = (double)((cm >> l) & 1u);
                         const double d = (q.x - q.z) - q.w;
                         const double w = dt * c * weight_foot(l, jj, cm);
                         v += w * d;
                     }
                     sm.lqg[(size_t)s * CR_STRIDE + CR_LX + j] = v;
                 });
    {
        struct PosRow { double xj, xrj, xf[4], pr[4]; };
        flat_pass(N * 3, tid,
                     [&](int e) {
                         const int s = e / 3, j = 3 + e % 3;
                         int ph, k;
                         phase_of_stage(sc, s, ph, k);
                         const int n = sc.node_off[ph] + k;
                         const double* x = sm.X + 24 * n;
                         PosRow r;
                         r.xj = x[j]; r.xrj = sm.xr[24 * n + j];
#pragma unroll
                         for (int l = 0; l < 4; ++l) { r.xf[l] = x[12 + 3 * l + j - 3]; r.pr[l] = sm.prel[12 * n + 3 * l + j - 3]; }
                         return r;
                     },
                     [&](int e, const PosRow& r) {
                         const int s = e / 3, j = 3 + e % 3;
                         const unsigned cm = sc.cmask[sc.ph_of_stage[s]];
                         double v = (dt * weight_Q(j, cm)) * (r.xj - r.xrj);
#pragma unroll
                         for (int l = 0; l < 4; ++l) {
                             const double c = (double)((cm >> l) & 1u);
                             const double d = (r.xf[l] - r.xj) - r.pr[l];
                             const double w = dt * c * weight_foot(l, j - 3, cm);
                             v += -(w * d);
                         }
                         sm.lqg[(size_t)s * CR_STRIDE + CR_LX + j] = v;
                     });
    }
    // (3) GRF controls and the ReB folding, flat over (stage, leg)  (compute_ReB_partials, ConstraintsBase.h:224-263;
    //     only gu is non-zero)
    {
        const double mu = sm.cp.mu;
        for (int e = tid; e < N * 4; e += kThreads) {
            const int s = e >> 2, l = e & 3;
            int ph, k;
            phase_of_stage(sc, s, ph, k);
            const int n = sc.node_off[ph] + k;
            const unsigned cm = sc.cmask[ph];
            double* rec = sm.lqg + (size_t)s * CR_STRIDE;
            double hess[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, grad[3] = {0, 0, 0};
            if (sm.opt.ReB_active && ((cm >> l) & 1u)) {
#pragma unroll
                for (int r = 0; r < 5; ++r) {
                    // friction-pyramid row r: (0,0,1), (-1,0,mu), (1,0,mu), (0,-1,mu), (0,1,mu)
                    const double row[3] = {(r == 1) ? -1.0 : (r == 2) ? 1.0 : 0.0, (r == 3) ? -1.0 : (r == 4) ? 1.0 : 0.0, (r == 0) ? 1.0 : mu};
                    const double g = sm.gcon[20 * s + 5 * l + r];
                    const double eps_b = sm.reb[40 * s + 2 * (5 * l + r)], delta = sm.reb[40 * s + 2 * (5 * l + r) + 1];
                    double bd, bdd;
                    if (g > delta) { bd = -1.0 / g; bdd = 1.0 / (g * g); }
                    else { bd = (g - 2 * delta) / delta / delta; bdd = 1.0 / (delta * delta); }
#pragma unroll
                    for (int a = 0; a < 3; ++a) grad[a] += eps_b * bd * row[a];
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int b = 0; b < 3; ++b) hess[3 * a + b] += eps_b * (bdd * row[a] * row[b]);
                }
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const int i = 3 * l + a;
                rec[CR_LU + i] = (dt * weight_R(i)) * (sm.U[24 * s + i] - sm.ur[24 * n + i]) + dt * grad[a];
            }
#pragma unroll
            for (int a = 0; a < 9; ++a) rec[CR_LUU + 9 * l + a] = dt * hess[a];
        }
    }
    __syncthreads();
    PROF_MARK(sm, 4);
}

// ---------------------------------------------------------------------------
// update_nominal_trajectory (TrajectoryManagement.cpp:110-115)
// ---------------------------------------------------------------------------
__device__ inline void update_nominal_block(Smem& sm) {
    flat_pass(sm.sc.n_nodes * 24, (int)threadIdx.x, [&](int e) { return sm.X[e]; }, [&](int e, double v) { sm.Xbar[e] = v; });
    flat_pass(sm.sc.n_stages * 24, (int)threadIdx.x, [&](int e) { return sm.U[e]; }, [&](int e, double v) { sm.Ubar[e] = v; });
    __syncthreads();
}

// update_AL_params / update_REB_params (ConstraintsBase.h:168-183,349-365)
__device__ inline void update_al_block(Smem& sm) {
    const DevSchedule& sc = sm.sc;
    if (threadIdx.x < sc.n_phases * 4) {
        const int ph = threadIdx.x >> 2, l = threadIdx.x & 3;
        const double h = sm.hcon[4 * ph + l];
        for (int ob = 0; ob < 2; ++ob) {
            if (!((sc.tdmask[ob][ph] >> l) & 1u)) continue;
            double& sigma = sm.al[16 * ph + 8 * ob + 2 * l];
            double& lambda = sm.al[16 * ph + 8 * ob + 2 * l + 1];
            if (!(fabs(h) < sm.opt.tconstr_thresh)) {
                if (fabs(h) > 0.005) { sigma *= sm.opt.update_penalty; sigma = fmin(sigma, sm.cp.td_sigma_max); }
                else lambda += h * sigma;
            }
        }
    }
    __syncthreads();
}
__device__ inline void update_reb_block(Smem& sm) {
    const DevSchedule& sc = sm.sc;
    for (int e = threadIdx.x; e < sc.n_stages * 20; e += kThreads) {
        const int s = e / 20, l = (e % 20) / 5;
        int ph, k;
        phase_of_stage(sc, s, ph, k);
        if (!((sc.cmask[ph] >> l) & 1u)) continue;
        if (sm.gcon[e] > -sm.opt.pconstr_thresh) continue;
        sm.reb[2 * e] *= sm.opt.update_ReB;
        double delta = sm.reb[2 * e + 1] * sm.opt.update_relax;
        sm.reb[2 * e + 1] = fmax(delta, sm.cp.grf_delta_min);
    }
    __syncthreads();
}

// cold start (HKDProblem.cpp:84-90, TrajectoryManagement.cpp:11-32, constraint initialize_params)
__device__ inline void cold_start_block(Smem& sm) {
    const DevSchedule& sc = sm.sc;
    for (int e = threadIdx.x; e < sc.n_nodes * 24; e += kThreads) {
        const double v = sm.xinit[e];
        sm.Xbar[e] = v; sm.X[e] = v; sm.dX[e] = 0.0; sm.Defect[e] = 0.0; sm.Xsim_t[e] = 0.0;
    }
    for (int e = threadIdx.x; e < sc.n_stages * 24; e += kThreads) { sm.Ubar[e] = 0.0; sm.U[e] = 0.0; sm.dU[e] = 0.0; sm.U_t[e] = 0.0; }
    for (size_t e = threadIdx.x; e < (size_t)sc.n_stages * 288; e += kThreads) sm.K[e] = 0.0;
    for (int e = threadIdx.x; e < sc.n_stages * 12; e += kThreads) sm.KdX[e] = 0.0;
    for (int e = threadIdx.x; e < sc.n_stages * 20; e += kThreads) {
        sm.gcon[e] = 0.0; sm.reb[2 * e] = sm.cp.grf_eps; sm.reb[2 * e + 1] = sm.cp.grf_delta;
    }
    for (int e = threadIdx.x; e < MAXPH * 4; e += kThreads) sm.hcon[e] = 0.0;
    for (int e = threadIdx.x; e < MAXPH * 8; e += kThreads) { sm.al[2 * e] = sm.cp.td_sigma; sm.al[2 * e + 1] = sm.cp.td_lambda; }
    if (threadIdx.x == 0) {
        SolverState z = {};
        z.rollout_ok = 1; z.sweep_ok = 1;
        sm.st = z;
    }
    __syncthreads();
}

}  // namespace hsddp
