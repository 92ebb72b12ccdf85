/*
 * hsddp_b200.h — C ABI of the B200-native batched Hybrid-Systems DDP solver.
 *
 * Drop-in boundary for ONE path of heli-sudoo/HKD-MPC: MultiPhaseDDP<double>::solve()
 * and the SinglePhase<double,24,24,0> sweeps under it, for the Mini Cheetah HKD
 * problem.  The reference has no C ABI (it exports C++ template instantiations
 * from libhsddp.so, HSDDPSolver/CMakeLists.txt:1-3); every entry point below cites
 * the reference interface it replaces.  Plain pointers and sizes only; all
 * `double*`/`int*` arguments are HOST pointers unless a name ends in `_dev`.
 *
 * Conventions
 *   - state x[24]  = [eul(yaw,pitch,roll) pos omega_body v_world qdummy(12)]
 *     control u[24] = [GRF(12) qJd(12)]                       (HKDModel.h:12-14)
 *   - matrices are column-major 24x24 (Eigen default), K is (u-row, x-col)
 *   - "node" layout: phases concatenated; phase i contributes horizon_i+1 state
 *     nodes (the last one is the phase's terminal state) and horizon_i control stages
 *   - a *schedule* is what HKDProblem::initialization derives from a reference
 *     window: the phase table plus per-node reference rows.  Many problems of a
 *     batch may share one schedule (e.g. perturbed initial states).
 *   - every function returns HSDDP_OK (0) or a negative HSDDP_ERR_* code; there
 *     is no CPU fallback: without a CUDA device the batch functions fail.
 */
#ifndef HSDDP_B200_H
#define HSDDP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HSDDP_NX 24
#define HSDDP_NU 24
#define HSDDP_MAX_PHASES 16
#define HSDDP_MAX_STAGES 128

#define HSDDP_OK 0
#define HSDDP_ERR_ARG (-1)
#define HSDDP_ERR_CUDA (-2)
#define HSDDP_ERR_UNSUPPORTED (-3)
#define HSDDP_ERR_STATE (-4)
#define HSDDP_ERR_IO (-5)

/* per-problem termination status (hsddp_info.status) — replaces the printf-only
 * outcomes of MultiPhaseDDP::solve, HSDDPSolver/source/MultiPhaseDDP.cpp:397-427 */
#define HSDDP_STATUS_CONVERGED 0     /* "all constraints satisfied"            :397-402 */
#define HSDDP_STATUS_STALLED 1       /* "constraints stop decreasing"          :403-408 */
#define HSDDP_STATUS_MAX_ITER 2      /* "maximum iteration reached"            :410-413 */
#define HSDDP_STATUS_REG_OVERFLOW 3  /* "too large regularization" (bad_solve) :162-167,421-427 */

/* HSDDP_OPTION, HSDDPSolver/common/HSDDP_CompoundTypes.h:18-60 (fields solve() reads). */
typedef struct hsddp_options {
    double alpha, gamma, update_penalty, update_relax, update_regularization, update_ReB;
    int32_t max_DDP_iter, max_AL_iter;
    double cost_thresh, tconstr_thresh, pconstr_thresh, dynamics_feas_thresh;
    double merit_scale, merit_offset;
    int32_t AL_active, ReB_active, MS, _pad;
} hsddp_options;

/* REB_Param_Struct / AL_Param_Struct initial values (ConstraintsBase.h:58-86,
 * HKDMPC/settings/constraint_params.info) and the friction coefficient (HKDConstraints.h:17). */
typedef struct hsddp_constraint_params {
    double grf_delta, grf_delta_min, grf_eps;
    double td_sigma, td_sigma_max, td_lambda;
    double mu;
} hsddp_constraint_params;

/* One reference window flattened: what HKDProblem::initialization
 * (HKDMPC/HKD-TrajOpt/HKDProblem.cpp:15-111,225-310) builds into phase objects. */
typedef struct hsddp_schedule {
    int32_t n_phases;
    int32_t n_stages;                         /* sum of horizons            */
    int32_t n_nodes;                          /* n_stages + n_phases        */
    int32_t horizon[HSDDP_MAX_PHASES];
    int32_t contact[HSDDP_MAX_PHASES][4];      /* phase contact flags        */
    int32_t next_contact[HSDDP_MAX_PHASES][4]; /* contact after the phase    */
    float start_time[HSDDP_MAX_PHASES];        /* pdata->phase_start_times   */
    double dt;                                 /* (double)(float)0.01        */
    /* per node (n_nodes rows): reference rows exactly as the cost callbacks see them */
    double* xr;     /* [n_nodes][24]  HKDSinglePhaseReference::get_reference_at_t     */
    double* ur;     /* [n_nodes][24]  (terminal nodes: unused)                        */
    double* prel_r; /* [n_nodes][12]  foot_placements - rep4(pos_ref), HKDCost.cpp:15 */
    double* xinit;  /* [n_nodes][24]  initial guess Xbar = X, HKDProblem.cpp:84-90    */
} hsddp_schedule;

/* per-problem result record (replaces reading MultiPhaseDDP privates / stdout) */
typedef struct hsddp_info {
    int32_t status, n_iter, n_outer, n_sweeps, n_trials, _pad;
    double cost, feas, max_tconstr, max_pconstr; /* final actual_cost, feas, violations */
    double cost0, feas0;                         /* after the initial rollout           */
} hsddp_info;

/* one row per DDP iteration (the natural per-iteration parity record; superset of
 * the four get_solver_info buffers, MultiPhaseDDP.cpp:277-280,368-371,532-541) */
typedef struct hsddp_iter_record {
    double outer, inner, cost_before, feas_before, reg_after, n_sweeps, dV_1, dV_2, merit_rho,
        eps_accepted, n_trials, cost_after, feas_after, max_tconstr, max_pconstr, _pad;
} hsddp_iter_record;
#define HSDDP_TRACE_CAP 64

/* ------------------------------------------------------------------------
 * Host-side problem assembly (CPU; no GPU needed)
 * ---------------------------------------------------------------------- */
typedef struct hkd_gait hkd_gait; /* QuadReference::tp_data, Reference/QuadReference.h:144-153 */

/* QuadReference::load_top_level_data(fname), Reference/QuadReference.cpp:129-285 */
int hkd_gait_load(const char* path, hkd_gait** out);
/* same table from arrays already parsed to float (n rows) */
int hkd_gait_create(int n, float dt, const float* body_state, const float* qJ, const float* foot_placements,
                    const float* grf, const int32_t* contact, hkd_gait** out);
int hkd_gait_size(const hkd_gait* g);
void hkd_gait_destroy(hkd_gait* g);

/* QuadReference::initialize + HKDProblem::initialization for the window that
 * starts at sample `window_start`; allocates the schedule's arrays. */
int hkd_schedule_build(const hkd_gait* g, int window_start, float plan_duration, hsddp_schedule* out);
void hkd_schedule_free(hsddp_schedule* s);

/* compute_hkd_state, HKDMPC/HKD-TrajOpt/HKDModel.h:65-96 */
void hkd_compute_state(const double eul[3], const double pos[3], const double qJ[12], const int32_t contact[4], double qdummy[12]);
/* initial condition of HKDMPCSolver::initialize, HKDMPC/HKDMPC.cpp:44-54 */
void hkd_default_x0(const hsddp_schedule* s, double x0[24]);

/* model functions on the host (same code the kernels run; unit-test hooks)
 * HKD::Model::dynamics / dynamics_partial (HKDModel.h:33-61), foot position /
 * Jacobian as used by HKDReset.h:41-136 and HKDConstraints.cpp:69-171.
 * A,B: 24x24 column-major; J: 3x18 column-major, columns [pos eul qJ(12)]. */
void hkd_model_dynamics(const double x[24], const double u[24], double dt, const int32_t contact[4], double xnext[24]);
void hkd_model_dynamics_partial(const double x[24], const double u[24], double dt, const int32_t contact[4], double A[576], double B[576]);
void hkd_model_foot_position(const double pos[3], const double eul[3], const double qleg[3], int leg, double p[3]);
void hkd_model_foot_jacobian(const double pos[3], const double eul[3], const double qleg[3], int leg, double J[54]);

/* ------------------------------------------------------------------------
 * Batched solver (one handle = one GPU + one stream; MultiPhaseDDP x n_problems)
 * ---------------------------------------------------------------------- */
typedef struct hsddp_batch hsddp_batch;

int hsddp_batch_create(int device, hsddp_batch** out);
int hsddp_batch_destroy(hsddp_batch* b);
const char* hsddp_last_error(void);

/* MultiPhaseDDP::set_multiPhaseProblem (MultiPhaseDDP.h:27-35): uploads the
 * schedules, allocates the problem-major workspace and resets every problem to
 * the cold-start guess (Xbar = X = reference states, Ubar = K = dU = 0,
 * HKDProblem.cpp:84-90, TrajectoryManagement.cpp:11-32). */
int hsddp_batch_set_problems(hsddp_batch* b, int n_schedules, const hsddp_schedule* schedules, int n_problems,
                             const int32_t* schedule_id, const hsddp_constraint_params* cparams);
/* MultiPhaseDDP::set_initial_condition (MultiPhaseDDP.h:37): x0 is [n_problems][24] on the host */
/* Reference ingestion on the device (SURVEY.md §8f N2).  The gait library — QuadReference::tp_data of n_gaits
 * reference files, every value already passed through stof (Reference/QuadReference.cpp:129-285), rows of all gaits
 * concatenated — is copied to HBM once; a kernel then does, for every schedule i = (sched_gait[i], sched_window[i]),
 * what QuadReference::initialize (QuadReference.cpp:6-26) and HKDProblem::initialization (HKDProblem.cpp:15-111,
 * 225-310) do on the host: phase split with the reference's float time arithmetic, contact after each phase, and the
 * per-node reference rows.  Bit-identical to hkd_schedule_build + hsddp_batch_set_problems. */
int hsddp_batch_set_problems_from_gaits(hsddp_batch* b, int n_gaits, const int32_t* gait_rows, const float* gait_dt,
                                        const double* body_state, const double* qJ, const double* foot_placements, const double* grf,
                                        const int32_t* contact, int n_schedules, const int32_t* sched_gait, const int32_t* sched_window,
                                        float plan_duration, int n_problems, const int32_t* schedule_id, const hsddp_constraint_params* cparams);
/* schedule i as the device holds it (n_phases; horizon [phases]; contact, next_contact [phases][4]; reference rows) */
int hsddp_batch_get_schedule(hsddp_batch* b, int i, int32_t* n_phases, int32_t* horizon, int32_t* contact, int32_t* next_contact,
                             double* xr, double* ur, double* prel_r, double* xinit);
int hsddp_batch_set_initial_condition(hsddp_batch* b, const double* x0);
/* re-arm the cold-start guess and the ReB/AL parameters without re-uploading schedules */
int hsddp_batch_reset(hsddp_batch* b);

/* HKDProblem::update (HKDMPC/HKD-TrajOpt/HKDProblem.cpp:117-222) for every problem of the batch: the receding-horizon shift
 * by one MPC step that HKDMPCSolver::update runs before each re-solve (HKDMPC/HKDMPC.cpp:97-166), on the device.
 *   - the reference window moves by one sample (QuadReference::step, Reference/QuadReference.cpp:33-47);
 *   - front end: the first node of the first phase is dropped (Trajectory::pop_front, TrajectoryManagement.cpp:118-146;
 *     PathConstraintBase::pop_front, ConstraintsBase.h:271-275), or the whole phase once it has shrunk to a point;
 *   - back end: the last phase grows by one stage whose state is a copy of the last trial state
 *     (Trajectory::push_back_state, TrajectoryManagement.cpp:178-207) or, one step after a contact change of the reference,
 *     a new phase of horizon 1 is opened with a zero-initialised trajectory, an EMPTY shooting set and no reset map;
 *     a phase that reaches its end gets its reset map and touchdown constraint then (add_tconstr_one_phase, a second
 *     constraint object if it already had one);
 *   - shooting sets, time offsets and the first control (zeroed) as HKDProblem.cpp:205-221; ReB / AL parameters persist
 *     (reset_params is a no-op in the reference).
 * Needs the gait library on the device (hsddp_batch_set_problems_from_gaits).  Follow with
 * hsddp_batch_set_initial_condition (the measured state) and hsddp_batch_solve with max_AL_iter = 2, max_DDP_iter = 1. */
int hsddp_batch_mpc_update(hsddp_batch* b);
/* milliseconds of the last update's kernels (CUDA events) */
int hsddp_batch_last_update_ms(hsddp_batch* b, float* ms);

/* HKDMPCSolver::initialize (HKDMPC/HKDMPC.cpp:44-69) for a SUBSET of the batch: problem[k] is re-targeted to the reference
 * window that starts at sample window[k] of gait gait[k] (index into the gait library of hsddp_batch_set_problems_from_gaits),
 * gets the cold-start guess, fresh ReB / AL parameters and initial state x0[k] ([n][24], host), as a new problem would.
 * The other problems are untouched.  first_solve (nullable): max_AL_iter / max_DDP_iter of the NEXT solve for these
 * problems only (e.g. 5 x 10 while the batch ticks at 2 x 1); its other fields are ignored.
 * Needs the gait library on the device (HSDDP_ERR_STATE otherwise).  HSDDP_ERR_ARG for out-of-range or repeated problem
 * indices, an unknown gait, a window that does not fit its table, or an invalid budget; HSDDP_ERR_UNSUPPORTED for a
 * schedule beyond HSDDP_MAX_PHASES / the batch's node capacity.  On any error nothing has changed.
 * A restarted problem gets a schedule slot of its own (problems restarted to the same gait and window in one call share
 * one); slots no problem uses any more are reused, so a handle never holds more than n_problems + n slots
 * (or the schedule count it was set with, if larger).
 * In an MPC tick: hsddp_batch_mpc_update, hsddp_batch_set_initial_condition, then this (the restarted problems start at their
 * new window after this tick's shift; x0 here overrides the state just set), then hsddp_batch_solve. */
int hsddp_batch_restart_problems(hsddp_batch* b, int n, const int32_t* problem, const int32_t* gait, const int32_t* window,
                                 const double* x0, const hsddp_options* first_solve);
/* schedule index of every problem ([n_problems]); pass it to hsddp_batch_get_schedule */
int hsddp_batch_get_schedule_ids(hsddp_batch* b, int32_t* out);

/* Per-problem MPC ticks.  In the reference every robot runs HKDMPCSolver::update (HKDMPC/HKDMPC.cpp:169-200) when its own
 * mpc_data LCM message arrives, so the robots of a fleet tick at their own times, not in lockstep.  These entry points tick
 * the LISTED problems of a batch: `problem` is a host list of n distinct indices in [0, n_problems), 1 <= n <= n_problems
 * (HSDDP_ERR_ARG otherwise, nothing changed).  Each listed problem gets exactly what the whole-batch call computes for it;
 * every other problem keeps its trajectories, gains, ReB / AL parameters, info, trace, pending first_solve budget and schedule
 * slot bit for bit.  A tick of some robots: update, initial states, solve, commands of the same list (restart a problem, if
 * needed, after the update of its tick, as for the whole batch).
 *
 * HKDProblem::update (HKDProblem.cpp:117-222, as hsddp_batch_mpc_update) of the listed problems.  Schedules are shared by slot,
 * so each slot a listed problem uses is copied to a free slot and the copy is stepped; once every copy has succeeded the listed
 * problems move to their copies (problems of the call that shared a slot share its copy) and are shifted.  HSDDP_ERR_ARG (the
 * reference table is exhausted) and HSDDP_ERR_UNSUPPORTED (table limits) leave the batch as it was.  A handle never holds more
 * than n_problems + n slots (or the schedule count it was set with, if larger).  Needs the gait library on the device. */
int hsddp_batch_mpc_update_problems(hsddp_batch* b, int n, const int32_t* problem);
/* MultiPhaseDDP::set_initial_condition (MultiPhaseDDP.h:37) of the listed problems: x0 is [n][24] on the host, row k for
 * problem[k] */
int hsddp_batch_set_initial_condition_problems(hsddp_batch* b, int n, const int32_t* problem, const double* x0);
/* MultiPhaseDDP::solve (MultiPhaseDDP.cpp:232-428) of the listed problems, in the kernel a batch of n problems would run
 * (same thresholds and hsddp_batch_set_solve_mode rules).  Pending first_solve budgets of the listed problems are used and
 * cleared; those of the other problems stay pending.  The _async form returns once the work is queued (pair with
 * hsddp_batch_sync); one solve at a time per handle. */
int hsddp_batch_solve_problems(hsddp_batch* b, int n, const int32_t* problem, const hsddp_options* opt);
int hsddp_batch_solve_problems_async(hsddp_batch* b, int n, const int32_t* problem, const hsddp_options* opt);

/* MultiPhaseDDP::solve(HSDDP_OPTION) (MultiPhaseDDP.cpp:232-428) for every problem:
 * one persistent kernel, one thread block per problem, iteration control on the device. */
int hsddp_batch_solve(hsddp_batch* b, const hsddp_options* opt);
/* same, without the trailing stream synchronise (pair with hsddp_batch_sync) */
int hsddp_batch_solve_async(hsddp_batch* b, const hsddp_options* opt);
int hsddp_batch_sync(hsddp_batch* b);
/* How solve() is scheduled on the GPU (results agree to rounding; each mode is bitwise reproducible):
 *   1 persistent — one kernel, every block runs whole solves pulled from a queue (small batches, latency).  From the
 *                  second solve of a problem set on, the queue visits the problems in the order of their previous
 *                  work (iterations, backward sweeps, trials), longest first (a scheduling hint only: results do not depend on it)
 *   2 phased     — per DDP iteration one kernel per phase (prep / backward sweep / linear rollout / forward sweep) over the problems
 *                  still running, up to four index ranges driven concurrently on their own streams.  The list of
 *                  running problems and its length stay in HBM, so the whole solve is queued without a host round trip
 *                  and hsddp_batch_solve_async returns as soon as the launches are queued
 *   0 auto       — phased when the batch fills the GPU five and a half times over (>= 4,884 problems on a B200).
 * Any other mode is refused with HSDDP_ERR_ARG. */
int hsddp_batch_set_solve_mode(hsddp_batch* b, int mode);
/* milliseconds of the last solve kernel, CUDA events on the handle's stream */
int hsddp_batch_last_solve_ms(hsddp_batch* b, float* ms);

/* Step-level API: the public methods of MultiPhaseDDP (MultiPhaseDDP.h:42-69),
 * each applied to all problems.  `ok` (optional, [n_problems]) receives the bool
 * the reference method returns. */
int hsddp_batch_hybrid_rollout(hsddp_batch* b, double eps, const hsddp_options* opt, int32_t* ok); /* :57-95  */
int hsddp_batch_compute_cost(hsddp_batch* b, const hsddp_options* opt);  /* :431-439 + measure_dynamics_feasibility :514-529 */
int hsddp_batch_lq_approximation(hsddp_batch* b, const hsddp_options* opt);                         /* :442-448 */
int hsddp_batch_backward_sweep(hsddp_batch* b, double regularization, int32_t* ok);                 /* :190-229 */
int hsddp_batch_backward_sweep_regularized(hsddp_batch* b, double* regularization /*[n] in/out*/, const hsddp_options* opt, int32_t* ok); /* :141-181 */
int hsddp_batch_linear_rollout(hsddp_batch* b, double eps, const hsddp_options* opt);               /* :20-50   */
/* forward sweep = line_search (:98-138): backtracking over the reference's step sizes,
 * hybrid rollout + cost + feasibility + Armijo test on the merit; needs merit/merit_rho
 * set by hsddp_batch_prepare_merit. `eps_accepted` gets the accepted step (0 = none). */
int hsddp_batch_prepare_merit(hsddp_batch* b, const hsddp_options* opt);                            /* :331-337 */
int hsddp_batch_forward_sweep(hsddp_batch* b, const hsddp_options* opt, int32_t* ok, double* eps_accepted);
int hsddp_batch_update_nominal(hsddp_batch* b);                                                      /* :505-511 */
int hsddp_batch_update_al_params(hsddp_batch* b, const hsddp_options* opt);                          /* :496-502 */
int hsddp_batch_update_reb_params(hsddp_batch* b, const hsddp_options* opt);                         /* :487-493 */

/* Results.  Trajectory getters copy [n_problems][rows][cols] with the batch-wide
 * row stride returned by hsddp_batch_dims (rows beyond a problem's own count are zero). */
int hsddp_batch_dims(hsddp_batch* b, int32_t* n_problems, int32_t* max_stages, int32_t* max_nodes);
int hsddp_batch_get_info(hsddp_batch* b, hsddp_info* out /*[n_problems]*/);
int hsddp_batch_get_trace(hsddp_batch* b, hsddp_iter_record* out /*[n_problems][HSDDP_TRACE_CAP]*/);
/* solver scalars per problem: [actual_cost, merit, feas, dV_1, dV_2, max_tconstr, max_pconstr, merit_rho] */
int hsddp_batch_get_scalars(hsddp_batch* b, double* out /*[n_problems][8]*/);

#define HSDDP_ARR_XBAR 0   /* [nodes][24]  Trajectory::Xbar (TrajectoryManagement.h:57) */
#define HSDDP_ARR_X 1      /* [nodes][24]  */
#define HSDDP_ARR_DEFECT 3 /* [nodes][24]  */
#define HSDDP_ARR_DX 4     /* [nodes][24]  */
#define HSDDP_ARR_UBAR 10  /* [stages][24] */
#define HSDDP_ARR_U 11     /* [stages][24] */
#define HSDDP_ARR_DU 12    /* [stages][24]  feed-forward dU */
#define HSDDP_ARR_K 20     /* [stages][576] feedback gains, column-major */
#define HSDDP_ARR_A 21     /* [stages][576] dense A reconstructed from the compact LQ record */
#define HSDDP_ARR_B 22     /* [stages][576] */
#define HSDDP_ARR_LX 30    /* [stages][24]  */
#define HSDDP_ARR_LU 31    /* [stages][24]  */
#define HSDDP_ARR_LUU 25   /* [stages][576] */
#define HSDDP_ARR_LXX 24   /* [stages][576] */
#define HSDDP_ARR_G0 5     /* [1][24]   value gradient at the first node after the last sweep */
#define HSDDP_ARR_H0 27    /* [1][576]  value Hessian at the first node after the last sweep  */
#define HSDDP_ARR_GCON 52  /* [stages][20] GRF constraint values, 5 per leg (swing legs zero) */
#define HSDDP_ARR_HCON 50  /* [HSDDP_MAX_PHASES][4] touchdown constraint values per phase/leg */
#define HSDDP_ARR_AL 51    /* [HSDDP_MAX_PHASES][2][4][2] (sigma, lambda) per touchdown-constraint object (0, 1) and leg */
#define HSDDP_ARR_REB 53   /* [stages][20][2] ReB parameters (eps, delta) of the GRF rows, 5 per leg (REB_Param_Struct, ConstraintsBase.h:58-70) */
int hsddp_batch_get_array(hsddp_batch* b, int which, double* out);
/* overwrite Xbar/X/Ubar/U (warm start); same layout as the getter */
int hsddp_batch_set_array(hsddp_batch* b, int which, const double* in);
/* first `n_ctrl` controls and the 12x12 body-feedback block is NOT extracted here
 * (that is HKDMPCSolver::publish_mpc_cmd, SURVEY.md §8f N3). */

/* copy rows [row0, row0+nrows) of a per-problem array (same `which` codes; K rows are
 * 576-double stages): out is [n_problems][nrows][cols].  This is the per-tick copy-out the
 * MPC caller needs (first controls, states and feedback gains, HKDMPC/HKDMPC.cpp:245-275). */
int hsddp_batch_get_array_rows(hsddp_batch* b, int which, int row0, int nrows, double* out);

/* feedback gains in the solver's own compact layout, no host-side expansion: out is
 * [n_problems][nrows][24][12] with out[..][j][c] = K(coupled control c of the stage, state j);
 * coupled control c = 3*leg + i is GRF component i of a stance leg or joint-velocity command i of
 * a swing leg; the 12 other controls of the stage have identically zero gain rows. */
int hsddp_batch_get_gains_compact(hsddp_batch* b, int row0, int nrows, double* out);

/* What leaves the GPU after an MPC solve: the payload of the hkd_command LCM message, lcmtypes/hkd_command_lcmt.lcm, as
 * HKDMPCSolver::publish_mpc_cmd (HKDMPC/HKDMPC.cpp:243-298) and update_foot_placement (:207-240) fill it, packed on
 * the device into one record per problem (single-precision like the LCM message) and copied out in one transfer.
 *   hkd_controls[k], des_body_state[k], feedback[k] : Ubar, Xbar[0:12] and K(0:12, 0:12) of the k-th stage of the
 *       horizon, walking the phases exactly as publish_mpc_cmd does; contacts[k] = contact flags of that phase
 *   foot_placement[3l..3l+2] : qdummy of leg l at the first node of the first phase (among the first five phase
 *       boundaries) where the leg goes swing -> stance; foot_found[l] = 0 if there is none (the reference then keeps
 *       its previous value).
 * mpc_times / statusTimes / solve_time of the LCM message are host-side bookkeeping, not solver outputs. */
#define HSDDP_CMD_MAX_STEPS 10
typedef struct hsddp_mpc_command {
    int32_t N_mpcsteps;
    int32_t foot_found[4];
    int32_t contacts[HSDDP_CMD_MAX_STEPS][4];
    float hkd_controls[HSDDP_CMD_MAX_STEPS][24];
    float des_body_state[HSDDP_CMD_MAX_STEPS][12];
    float feedback[HSDDP_CMD_MAX_STEPS][12][12];
    float foot_placement[12];
    int32_t _pad;
} hsddp_mpc_command;
/* n_steps = nsteps_between_mpc + 7 (8 in the reference), at most HSDDP_CMD_MAX_STEPS; out: [n_problems] on the host */
int hsddp_batch_get_mpc_command(hsddp_batch* b, int n_steps, hsddp_mpc_command* out);
/* HKDMPCSolver::publish_mpc_cmd + update_foot_placement (HKDMPC.cpp:207-298) of the listed problems (see
 * hsddp_batch_mpc_update_problems): out is [n] on the host, record k for problem[k] */
int hsddp_batch_get_mpc_command_problems(hsddp_batch* b, int n_steps, int n, const int32_t* problem, hsddp_mpc_command* out);

/* Ticks from GPU memory: the robots' states come in and the command records go out through the CALLER's device buffers,
 * ordered on the caller's CUDA stream, for fleets whose states are produced on the same GPU (e.g. a simulator's tensors).
 *   - problem: a HOST list of n distinct indices (as the _problems entry points), or NULL for every problem in index order
 *     (then n == n_problems); row / record k belongs to problem[k].
 *   - stream: the caller's cudaStream_t passed as void* (NULL = the default stream, as in CUDA).
 * Stream contract.  Each call records an event on `stream` and makes the handle's stream wait on it, so the inputs are read
 * only after all work queued on `stream` before the call.  After its last launch it records an event on the handle's stream
 * and makes `stream` wait on it, so work queued on `stream` afterwards sees the outputs and may reuse the input buffers.  None of
 * the three synchronises the host: they return once the work is queued.  hsddp_batch_solve[_problems]_async queues on the
 * handle's stream, so set_*_dev -> solve_async -> get_mpc_command_dev needs no further synchronisation.
 * Refusals return before anything is queued and leave the batch unchanged: HSDDP_ERR_ARG for a handle without problems, a NULL
 * buffer, a buffer that is not device or managed memory of the handle's GPU (pageable or pinned host memory, another GPU), a
 * buffer not aligned to its element type (double, int32_t, hsddp_mpc_command), a bad problem list, or n_steps outside
 * [1, HSDDP_CMD_MAX_STEPS]. */
/* MultiPhaseDDP::set_initial_condition (MultiPhaseDDP.h:37): x0_dev is [n][24] doubles in device memory, row k for problem[k] */
int hsddp_batch_set_initial_condition_dev(hsddp_batch* b, int n, const int32_t* problem, const double* x0_dev, void* stream);
/* HKDMPCSolver::update's initial condition from the robot's measurement, on the device.
 * meas_dev: [n][24] doubles = eul(yaw,pitch,roll) pos omega_body v_world (x0's first 12 entries) followed by qJ[12].
 * x0 = [meas[0:12], compute_hkd_state(eul, pos, qJ, contact)] (hkd_compute_state) with contact = contact_dev[k][4] (nonzero =
 * stance) if given, else the contact flags of the problem's FIRST PHASE as the device holds it when the kernel runs (after
 * this tick's hsddp_batch_mpc_update).  That NULL rule is the one hkd_default_x0 and the workloads apply at the window start;
 * the reference's own update-time source of the contact (HKDMPC.cpp:119-129) is not restated in this library, so a caller
 * with contact sensing passes its own flags. */
int hsddp_batch_set_measured_state_dev(hsddp_batch* b, int n, const int32_t* problem, const double* meas_dev,
                                       const int32_t* contact_dev, void* stream);
/* hsddp_batch_get_mpc_command[_problems] straight into out_dev ([n] records in device memory), record k for problem[k] */
int hsddp_batch_get_mpc_command_dev(hsddp_batch* b, int n_steps, int n, const int32_t* problem, hsddp_mpc_command* out_dev, void* stream);

/* CUDA-event timing on the handle's stream (slots 0..7): record, then elapsed ms between two slots */
int hsddp_batch_event_record(hsddp_batch* b, int slot);
int hsddp_batch_event_elapsed_ms(hsddp_batch* b, int slot0, int slot1, float* ms);
/* work counters of all solves since set_problems/reset_counters:
 * out[0] = sum over problems of (backward sweeps x stages), out[1] = k_solve launches, out[2] = k_step launches */
int hsddp_batch_get_counters(hsddp_batch* b, unsigned long long out[4]);
int hsddp_batch_reset_counters(hsddp_batch* b);
/* regularisation retries run side by side (phased driver, HSDDP_SWEEP_SPEC), since set_problems/reset_counters:
 * out[0] = problem-rounds speculated, out[1] = of those, rounds whose first PD attempt was not the first one,
 * out[2] = rounds in which every candidate failed (the problem's block went on retrying alone) */
int hsddp_batch_get_speculation(hsddp_batch* b, unsigned long long out[3]);
/* per-phase cycle counters (all zero unless the library was built with -DHSDDP_PROFILE) */
int hsddp_batch_get_profile(hsddp_batch* b, unsigned long long out[16]);

/* ------------------------------------------------------------------------
 * The reference's OTHER instantiations (SURVEY.md 8f N4): SinglePhase<double,12,12,0> and <36,12,12>
 * (HSDDPSolver/source/SinglePhase.cpp:538-540; <24,24,0> is accepted too, in its dense form).
 * The reference ships no model, cost or problem for them and host plug-ins cannot run on the device, so the boundary
 * is the phase's storage after LQ_approximation (SinglePhase.cpp:265-296): the plug-in outputs go in, the
 * model-independent sweeps run on the device for a batch of independent phases of equal horizon.
 * All matrices column-major (Eigen default); arrays are problem-major, then stage-major:
 *   A [n][N][xs*xs]  B [n][N][xs*us]  C [n][N][ys*xs]  D [n][N][ys*us]                (dynamics_partial, SinglePhase.h:45-50)
 *   lx [n][N][xs] lu [n][N][us] ly [n][N][ys] lxx [n][N][xs*xs] luu [n][N][us*us] lux [n][N][us*xs] lyy [n][N][ys*ys]
 *                                                                                      (RCostData, HSDDP_CompoundTypes.h:90-127)
 *   Phix [n][xs]  Phixx [n][xs*xs]                                                     (TCostData, :129-150)
 *   Defect [n][N+1][xs]                                                                (Trajectory::Defect)
 * Inputs never set are zero.
 * ---------------------------------------------------------------------- */
typedef struct hsddp_phase_batch hsddp_phase_batch;
#define HSDDP_PH_A 0
#define HSDDP_PH_B 1
#define HSDDP_PH_C 2
#define HSDDP_PH_D 3
#define HSDDP_PH_LX 4
#define HSDDP_PH_LU 5
#define HSDDP_PH_LY 6
#define HSDDP_PH_LXX 7
#define HSDDP_PH_LUU 8
#define HSDDP_PH_LUX 9
#define HSDDP_PH_LYY 10
#define HSDDP_PH_PHIX 11
#define HSDDP_PH_PHIXX 12
#define HSDDP_PH_DEFECT 13
#define HSDDP_PH_N_INPUTS 14
#define HSDDP_PH_OUT_DU 0 /* [n][N][us]      feed-forward                         */
#define HSDDP_PH_OUT_K 1  /* [n][N][us*xs]   feedback gains                       */
#define HSDDP_PH_OUT_G 2  /* [n][N+1][xs]    value gradient                       */
#define HSDDP_PH_OUT_H 3  /* [n][N+1][xs*xs] value Hessian                        */
#define HSDDP_PH_OUT_DX 4 /* [n][N+1][xs]    linear-rollout direction             */
#define HSDDP_PH_OUT_DV 5 /* [n][2]          dV_1, dV_2 of the LAST sweep / rollout */
#define HSDDP_PH_N_OUTPUTS 6
/* HSDDP_ERR_UNSUPPORTED for any (xs, us, ys) the reference does not instantiate */
int hsddp_phase_batch_create(int device, int xs, int us, int ys, int horizon, int n_problems, hsddp_phase_batch** out);
int hsddp_phase_batch_destroy(hsddp_phase_batch* b);
int hsddp_phase_batch_set(hsddp_phase_batch* b, int which, const double* host);
/* SinglePhase::backward_sweep(regularization, Gprime, Hprime) (SinglePhase.cpp:299-367): Gprime [n][xs], Hprime [n][xs*xs]
 * (null = zero: a last phase); ok [n] (optional) receives the bool the reference returns.  After a failed stage the
 * stages below it keep what the storage held, and G[0] += H[0] Defect[0] still runs (:365), as in the reference. */
int hsddp_phase_batch_backward_sweep(hsddp_phase_batch* b, double regularization, const double* Gprime, const double* Hprime, int32_t* ok);
/* SinglePhase::linear_rollout(eps) (SinglePhase.cpp:145-178) with the gains of the last sweep (or set_gains);
 * dx_init [n][xs] (null = zero: a first phase) */
int hsddp_phase_batch_linear_rollout(hsddp_phase_batch* b, double eps, const double* dx_init);
int hsddp_phase_batch_set_gains(hsddp_phase_batch* b, const double* dU, const double* K);
int hsddp_phase_batch_get(hsddp_phase_batch* b, int which, double* host);
/* milliseconds of the last sweep / rollout kernel (CUDA events on the handle's stream) */
int hsddp_phase_batch_last_ms(hsddp_phase_batch* b, float* ms);

/* device-side FP64 FMA throughput probe (TFLOP/s) used as the measured roofline
 * denominator by bench.py; kind 0 = DFMA on CUDA cores, 1 = DMMA m8n8k4 tensor tiles */
int hsddp_fp64_peak_tflops(int device, int kind, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* HSDDP_B200_H */
