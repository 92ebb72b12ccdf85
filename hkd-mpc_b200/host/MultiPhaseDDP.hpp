// Header-only C++ shim over the C ABI (include/hsddp_b200.h) that keeps the reference's
// solver surface for the one path this repository replaces:
//
//   MultiPhaseDDP<T>      HSDDPSolver/header/MultiPhaseDDP.h:18-122   (T = double only)
//   HSDDP_OPTION          HSDDPSolver/common/HSDDP_CompoundTypes.h:18-60
//   QuadReference         Reference/QuadReference.h:144-191           (load_top_level_data, initialize)
//
// Differences a maintainer must know about (see INTEGRATION.md):
//   * one solver object owns a BATCH of independent problems; every method acts on all of them and
//     the bool-returning methods return one flag per problem;
//   * phases are not SinglePhase objects with std::function callbacks (host callables cannot run on
//     the device): a problem is (schedule, x0), where a schedule is the flattened result of
//     HKDProblem::initialization for one reference window, and the HKD model / costs / reset map /
//     constraints are the device-compiled ones;
//   * results are copied out explicitly (get_Xbar, get_Ubar, get_K, ...), not read from Trajectory objects;
//   * there is no CPU fallback: construction throws when no CUDA device is present.
#pragma once
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>
#include "../../include/hsddp_b200.h"

namespace hsddp_b200 {

inline void check(int rc, const char* what) {
    if (rc != HSDDP_OK) throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) + "): " + hsddp_last_error());
}

// HSDDP_OPTION with the values solve() actually consumes from HKDMPC/settings/ddp_setting.info
struct HSDDP_OPTION : hsddp_options {
    HSDDP_OPTION() {
        alpha = 0.1; gamma = 0.01; update_penalty = 5; update_relax = 1; update_regularization = 2; update_ReB = 1;
        max_DDP_iter = 10; max_AL_iter = 5; cost_thresh = 1e-3; tconstr_thresh = 1e-3; pconstr_thresh = 1e-3;
        dynamics_feas_thresh = 1e-3; merit_scale = 0.2; merit_offset = 1e2; AL_active = 1; ReB_active = 1; MS = 1; _pad = 0;
    }
};

// Top-level reference table + per-window schedules (QuadReference + HKDProblem::initialization).
class QuadReference {
public:
    QuadReference() = default;
    ~QuadReference() { if (gait_) hkd_gait_destroy(gait_); }
    QuadReference(const QuadReference&) = delete;
    QuadReference& operator=(const QuadReference&) = delete;
    void load_top_level_data(const std::string& fname) {
        if (gait_) { hkd_gait_destroy(gait_); gait_ = nullptr; }
        check(hkd_gait_load(fname.c_str(), &gait_), "hkd_gait_load");
    }
    int size() const { return hkd_gait_size(gait_); }
    const hkd_gait* handle() const { return gait_; }
private:
    hkd_gait* gait_ = nullptr;
};

// RAII owner of one hsddp_schedule
class Schedule {
public:
    Schedule(const QuadReference& ref, int window_start, float plan_duration) {
        check(hkd_schedule_build(ref.handle(), window_start, plan_duration, &s_), "hkd_schedule_build");
    }
    ~Schedule() { hkd_schedule_free(&s_); }
    Schedule(const Schedule&) = delete;
    Schedule& operator=(const Schedule&) = delete;
    const hsddp_schedule& get() const { return s_; }
    std::vector<double> default_x0() const { std::vector<double> x(24); hkd_default_x0(&s_, x.data()); return x; }
private:
    hsddp_schedule s_{};
};

// SinglePhase<T,24,24,0> (HSDDPSolver/header/SinglePhase.h:28-170) as the reference's problem-assembly code sees it.
// Host callables cannot run on the device: the HKD model, costs, reset map and constraints are the device-compiled ones,
// selected by the schedule, so every plug-in setter ACCEPTS its argument and ignores it.  Code written against the
// reference's phase interface (HKDProblem::create_problem_one_phase / add_tconstr_one_phase, HKDProblem.cpp:225-310)
// therefore compiles unchanged; what it configures comes from the schedule instead.
template <typename T, size_t xs, size_t us, size_t ys>
class SinglePhase {
    static_assert(xs == 24 && us == 24 && ys == 0, "only the <double,24,24,0> HKD instantiation is built for the device");
public:
    template <class F> void set_dynamics(F&&) {}                    // SinglePhase.h:41-44
    template <class F> void set_dynamics_partial(F&&) {}            // :45-50
    template <class F> void set_resetmap(F&&) {}                    // :66-72
    template <class F> void set_resetmap_partial(F&&) {}            // :73-80
    template <class P> void add_cost(P&&) {}                        // :84-86
    template <class P> void add_pathConstraint(P&&) {}              // :88-90
    template <class P> void add_terminalConstraint(P&&) {}          // :92-94
    template <class P> void set_trajectory(P&&) {}                  // SinglePhase.cpp:130-135
    void set_time_offset(float) {}                                  // :82
    void initialization() {}                                        // SinglePhase.cpp:22-35
    void update_SS_config(int) {}                                   // :161-164
    void reset_params() {}                                          // :155 (a no-op in the reference as well)
};

template <typename T>
class MultiPhaseDDP;

template <>
class MultiPhaseDDP<double> {
public:
    explicit MultiPhaseDDP(int device = 0) { check(hsddp_batch_create(device, &b_), "hsddp_batch_create"); }
    ~MultiPhaseDDP() { hsddp_batch_destroy(b_); }
    MultiPhaseDDP(const MultiPhaseDDP&) = delete;
    MultiPhaseDDP& operator=(const MultiPhaseDDP&) = delete;

    // set_multiPhaseProblem: `schedule_id[i]` selects the schedule of problem i
    void set_multiPhaseProblem(const std::vector<const Schedule*>& schedules, const std::vector<int32_t>& schedule_id,
                               const hsddp_constraint_params* cparams = nullptr) {
        std::vector<hsddp_schedule> flat;
        for (const Schedule* s : schedules) flat.push_back(s->get());
        check(hsddp_batch_set_problems(b_, (int)flat.size(), flat.data(), (int)schedule_id.size(), schedule_id.data(), cparams), "hsddp_batch_set_problems");
        n_ = (int)schedule_id.size();
        check(hsddp_batch_dims(b_, nullptr, &max_stages_, &max_nodes_), "hsddp_batch_dims");
    }
    // the same from the gait library resident on the device (schedules built by a kernel): the form that supports update()
    void set_multiPhaseProblem_from_gaits(const std::vector<int32_t>& gait_rows, const std::vector<float>& gait_dt, const std::vector<double>& body_state,
                                          const std::vector<double>& qJ, const std::vector<double>& foot_placements, const std::vector<double>& grf,
                                          const std::vector<int32_t>& contact, const std::vector<int32_t>& sched_gait, const std::vector<int32_t>& sched_window,
                                          float plan_duration, const std::vector<int32_t>& schedule_id, const hsddp_constraint_params* cparams = nullptr) {
        check(hsddp_batch_set_problems_from_gaits(b_, (int)gait_rows.size(), gait_rows.data(), gait_dt.data(), body_state.data(), qJ.data(), foot_placements.data(),
                                                  grf.data(), contact.data(), (int)sched_gait.size(), sched_gait.data(), sched_window.data(), plan_duration,
                                                  (int)schedule_id.size(), schedule_id.data(), cparams), "hsddp_batch_set_problems_from_gaits");
        n_ = (int)schedule_id.size();
        check(hsddp_batch_dims(b_, nullptr, &max_stages_, &max_nodes_), "hsddp_batch_dims");
    }
    // HKDProblem::update (HKDProblem.cpp:117-222) for every problem: the receding-horizon shift before an MPC re-solve
    void update() { check(hsddp_batch_mpc_update(b_), "hsddp_batch_mpc_update"); }
    // HKDMPCSolver::initialize (HKDMPC.cpp:44-69) for the listed problems only: new reference window (gait, window start),
    // cold-start guess, fresh ReB / AL parameters, x0 (24 doubles per listed problem); first_solve (nullable) sets
    // max_AL_iter / max_DDP_iter of their next solve.  The other problems keep their warm state.
    void restart_problems(const std::vector<int32_t>& problem, const std::vector<int32_t>& gait, const std::vector<int32_t>& window,
                          const std::vector<double>& x0, const HSDDP_OPTION* first_solve = nullptr) {
        if (gait.size() != problem.size() || window.size() != problem.size() || x0.size() != 24 * problem.size())
            throw std::invalid_argument("restart_problems: one gait, one window and 24 doubles of x0 per problem");
        check(hsddp_batch_restart_problems(b_, (int)problem.size(), problem.data(), gait.data(), window.data(), x0.data(), first_solve),
              "hsddp_batch_restart_problems");
    }
    std::vector<int32_t> get_schedule_ids() {
        std::vector<int32_t> v(n_);
        check(hsddp_batch_get_schedule_ids(b_, v.data()), "hsddp_batch_get_schedule_ids");
        return v;
    }
    void set_initial_condition(const std::vector<double>& x0) {
        if ((int)x0.size() != 24 * n_) throw std::invalid_argument("x0 must hold 24 doubles per problem");
        check(hsddp_batch_set_initial_condition(b_, x0.data()), "hsddp_batch_set_initial_condition");
    }
    void reset() { check(hsddp_batch_reset(b_), "hsddp_batch_reset"); }
    void solve(HSDDP_OPTION option) { check(hsddp_batch_solve(b_, &option), "hsddp_batch_solve"); }
    void solve_async(HSDDP_OPTION option) { check(hsddp_batch_solve_async(b_, &option), "hsddp_batch_solve_async"); }
    void sync() { check(hsddp_batch_sync(b_), "hsddp_batch_sync"); }
    // measure_dynamics_feasibility(norm_id) (MultiPhaseDDP.cpp:514-529; the reference's solve() uses the default norm_id = 2):
    // sqrt(sum ||Defect||^2) of every problem, as evaluated by the last compute_cost / solve
    std::vector<double> measure_dynamics_feasibility(int norm_id = 2) {
        if (norm_id != 2) throw std::invalid_argument("only the 2-norm (the one solve() uses) is evaluated on the device");
        std::vector<double> sc((size_t)n_ * 8), f(n_);
        check(hsddp_batch_get_scalars(b_, sc.data()), "hsddp_batch_get_scalars");
        for (int i = 0; i < n_; ++i) f[i] = sc[(size_t)8 * i + 2];
        return f;
    }

    // step-level API (same names as the reference's public methods)
    void linear_rollout(double eps, HSDDP_OPTION& o) { check(hsddp_batch_linear_rollout(b_, eps, &o), "linear_rollout"); }
    std::vector<int32_t> hybrid_rollout(double eps, HSDDP_OPTION& o) { std::vector<int32_t> ok(n_); check(hsddp_batch_hybrid_rollout(b_, eps, &o, ok.data()), "hybrid_rollout"); return ok; }
    std::vector<int32_t> line_search(HSDDP_OPTION& o) { std::vector<int32_t> ok(n_); check(hsddp_batch_forward_sweep(b_, &o, ok.data(), nullptr), "forward_sweep"); return ok; }
    void compute_cost(const HSDDP_OPTION& o) { check(hsddp_batch_compute_cost(b_, &o), "compute_cost"); }
    void LQ_approximation(HSDDP_OPTION& o) { check(hsddp_batch_lq_approximation(b_, &o), "lq_approximation"); }
    std::vector<int32_t> backward_sweep(double regularization) { std::vector<int32_t> ok(n_); check(hsddp_batch_backward_sweep(b_, regularization, ok.data()), "backward_sweep"); return ok; }
    std::vector<int32_t> backward_sweep_regularized(std::vector<double>& regularization, HSDDP_OPTION& o) {
        std::vector<int32_t> ok(n_);
        check(hsddp_batch_backward_sweep_regularized(b_, regularization.data(), &o, ok.data()), "backward_sweep_regularized");
        return ok;
    }
    void update_nominal_trajectory() { check(hsddp_batch_update_nominal(b_), "update_nominal"); }
    void update_AL_params(HSDDP_OPTION& o) { check(hsddp_batch_update_al_params(b_, &o), "update_al_params"); }
    void update_REB_params(HSDDP_OPTION& o) { check(hsddp_batch_update_reb_params(b_, &o), "update_reb_params"); }

    // results
    std::vector<hsddp_info> get_info() { std::vector<hsddp_info> v(n_); check(hsddp_batch_get_info(b_, v.data()), "get_info"); return v; }
    std::vector<double> get_actual_cost() { auto v = get_info(); std::vector<double> c(n_); for (int i = 0; i < n_; ++i) c[i] = v[i].cost; return c; }
    std::vector<double> get_array(int which, size_t per_problem) { std::vector<double> v((size_t)n_ * per_problem); check(hsddp_batch_get_array(b_, which, v.data()), "get_array"); return v; }
    std::vector<double> get_Xbar() { return get_array(HSDDP_ARR_XBAR, (size_t)max_nodes_ * 24); }
    std::vector<double> get_Ubar() { return get_array(HSDDP_ARR_UBAR, (size_t)max_stages_ * 24); }
    std::vector<double> get_K() { return get_array(HSDDP_ARR_K, (size_t)max_stages_ * 576); }
    // get_solver_info: the four float history buffers of problem i (MultiPhaseDDP.cpp:532-541)
    void get_solver_info(int i, std::vector<float>& cost, std::vector<float>& dyn_feas, std::vector<float>& eqn_feas, std::vector<float>& ineq_feas) {
        std::vector<hsddp_iter_record> tr((size_t)n_ * HSDDP_TRACE_CAP);
        check(hsddp_batch_get_trace(b_, tr.data()), "get_trace");
        auto info = get_info();
        cost.assign(1, (float)info[i].cost0); dyn_feas.assign(1, (float)info[i].feas0); eqn_feas.clear(); ineq_feas.clear();
        for (int k = 0; k < info[i].n_iter && k < HSDDP_TRACE_CAP; ++k) {
            const hsddp_iter_record& r = tr[(size_t)i * HSDDP_TRACE_CAP + k];
            if (r.eps_accepted < 0) break;  // early exits do not append to the history (MultiPhaseDDP.cpp:340-343)
            cost.push_back((float)r.cost_after); dyn_feas.push_back((float)r.feas_after);
            eqn_feas.push_back((float)r.max_tconstr); ineq_feas.push_back((float)r.max_pconstr);
        }
    }
    // what HKDMPCSolver::publish_mpc_cmd + update_foot_placement ship to the robot (HKDMPC/HKDMPC.cpp:207-298):
    // packed on the device, one record per problem
    std::vector<hsddp_mpc_command> get_mpc_command(int n_steps = 8) {
        std::vector<hsddp_mpc_command> v(n_);
        check(hsddp_batch_get_mpc_command(b_, n_steps, v.data()), "get_mpc_command");
        return v;
    }
    // 0 auto, 1 persistent kernel, 2 one kernel per solve phase (include/hsddp_b200.h)
    void set_solve_mode(int mode) { check(hsddp_batch_set_solve_mode(b_, mode), "set_solve_mode"); }
    int n_problems() const { return n_; }
    int max_stages() const { return max_stages_; }
    int max_nodes() const { return max_nodes_; }
    hsddp_batch* handle() { return b_; }

private:
    hsddp_batch* b_ = nullptr;
    int n_ = 0;
    int32_t max_stages_ = 0, max_nodes_ = 0;
};

// One solver object over SEVERAL GPUs of a box: problems are independent, so problem i goes to device i * n_dev / n (contiguous
// index ranges, no data-path traffic between the GPUs).  solve() queues the work on every device before it waits for any
// (hsddp_batch_solve_async returns as soon as the launches are queued), so one host thread keeps all GPUs busy.
class MultiGpuDDP {
public:
    explicit MultiGpuDDP(const std::vector<int>& devices) {
        for (int d : devices) parts_.emplace_back(new MultiPhaseDDP<double>(d));
    }
    int n_devices() const { return (int)parts_.size(); }
    // contiguous shard [lo, hi) of device g (sizes differ by at most one)
    static void shard_range(int n_total, int g, int n_dev, int& lo, int& hi) {
        const int base = n_total / n_dev, rem = n_total % n_dev;
        lo = g * base + (g < rem ? g : rem);
        hi = lo + base + (g < rem ? 1 : 0);
    }
    void set_multiPhaseProblem(const std::vector<const Schedule*>& schedules, const std::vector<int32_t>& schedule_id, const hsddp_constraint_params* cparams = nullptr) {
        n_ = (int)schedule_id.size();
        for (int g = 0; g < n_devices(); ++g) {
            int lo, hi;
            shard_range(n_, g, n_devices(), lo, hi);
            // every device gets only the schedules its problems use
            std::vector<int32_t> remap(schedules.size(), -1), sid;
            std::vector<const Schedule*> used;
            for (int i = lo; i < hi; ++i) {
                int32_t& r = remap[schedule_id[i]];
                if (r < 0) { r = (int32_t)used.size(); used.push_back(schedules[schedule_id[i]]); }
                sid.push_back(r);
            }
            parts_[g]->set_multiPhaseProblem(used, sid, cparams);
        }
    }
    void set_initial_condition(const std::vector<double>& x0) {
        for (int g = 0; g < n_devices(); ++g) {
            int lo, hi;
            shard_range(n_, g, n_devices(), lo, hi);
            parts_[g]->set_initial_condition(std::vector<double>(x0.begin() + (size_t)24 * lo, x0.begin() + (size_t)24 * hi));
        }
    }
    void reset() { for (auto& p : parts_) p->reset(); }
    // restart_problems with GLOBAL problem indices: each listed problem goes to the device whose shard holds it.  The indices
    // are checked for all devices first; a device that refuses its part throws after the devices before it have restarted theirs.
    void restart_problems(const std::vector<int32_t>& problem, const std::vector<int32_t>& gait, const std::vector<int32_t>& window,
                          const std::vector<double>& x0, const HSDDP_OPTION* first_solve = nullptr) {
        if (gait.size() != problem.size() || window.size() != problem.size() || x0.size() != 24 * problem.size())
            throw std::invalid_argument("restart_problems: one gait, one window and 24 doubles of x0 per problem");
        std::vector<char> seen(n_, 0);
        for (int32_t p : problem) {
            if (p < 0 || p >= n_ || seen[p]) throw std::invalid_argument("restart_problems: problem index out of range or repeated");
            seen[p] = 1;
        }
        for (int g = 0; g < n_devices(); ++g) {
            int lo, hi;
            shard_range(n_, g, n_devices(), lo, hi);
            std::vector<int32_t> lp, lg, lw;
            std::vector<double> lx;
            for (size_t k = 0; k < problem.size(); ++k) {
                if (problem[k] < lo || problem[k] >= hi) continue;
                lp.push_back(problem[k] - lo); lg.push_back(gait[k]); lw.push_back(window[k]);
                lx.insert(lx.end(), x0.begin() + 24 * k, x0.begin() + 24 * (k + 1));
            }
            if (!lp.empty()) parts_[g]->restart_problems(lp, lg, lw, lx, first_solve);
        }
    }
    void solve(HSDDP_OPTION option) {
        for (auto& p : parts_) p->solve_async(option);
        for (auto& p : parts_) p->sync();
    }
    std::vector<hsddp_info> get_info() {
        std::vector<hsddp_info> all;
        for (auto& p : parts_) { auto v = p->get_info(); all.insert(all.end(), v.begin(), v.end()); }
        return all;
    }
    std::vector<hsddp_mpc_command> get_mpc_command(int n_steps = 8) {
        std::vector<hsddp_mpc_command> all;
        for (auto& p : parts_) { auto v = p->get_mpc_command(n_steps); all.insert(all.end(), v.begin(), v.end()); }
        return all;
    }
    MultiPhaseDDP<double>& part(int g) { return *parts_[g]; }
private:
    std::vector<std::unique_ptr<MultiPhaseDDP<double>>> parts_;
    int n_ = 0;
};

// The reference's other instantiations, SinglePhase<T,12,12,0> and SinglePhase<T,36,12,12> (SinglePhase.cpp:538-540; SURVEY.md 8f
// N4), and <24,24,0> in its dense form: the model-independent sweeps on a batch of independent phases of equal horizon.
// The reference ships no model, cost or problem for them and host plug-ins cannot run on the device, so the phase's storage
// after LQ_approximation goes in (column-major matrices, layouts in include/hsddp_b200.h) and dU, K, G, H, dX, dV come out.
template <typename T, size_t xs, size_t us, size_t ys>
class SinglePhaseSweeps {
    static_assert((xs == 24 && us == 24 && ys == 0) || (xs == 12 && us == 12 && ys == 0) || (xs == 36 && us == 12 && ys == 12),
                  "the reference instantiates <24,24,0>, <12,12,0> and <36,12,12> only");
public:
    SinglePhaseSweeps(int horizon, int n_problems, int device = 0) : n_(n_problems) {
        check(hsddp_phase_batch_create(device, (int)xs, (int)us, (int)ys, horizon, n_problems, &b_), "hsddp_phase_batch_create");
    }
    ~SinglePhaseSweeps() { hsddp_phase_batch_destroy(b_); }
    SinglePhaseSweeps(const SinglePhaseSweeps&) = delete;
    SinglePhaseSweeps& operator=(const SinglePhaseSweeps&) = delete;
    void set(int which, const std::vector<T>& v) { check(hsddp_phase_batch_set(b_, which, v.data()), "hsddp_phase_batch_set"); }
    // SinglePhase::backward_sweep(regularization, Gprime, Hprime), SinglePhase.cpp:299-367; one bool per problem
    std::vector<int32_t> backward_sweep(T regularization, const T* Gprime = nullptr, const T* Hprime = nullptr) {
        std::vector<int32_t> ok(n_problems());
        check(hsddp_phase_batch_backward_sweep(b_, regularization, Gprime, Hprime, ok.data()), "hsddp_phase_batch_backward_sweep");
        return ok;
    }
    // SinglePhase::linear_rollout(eps, option), SinglePhase.cpp:145-178
    void linear_rollout(T eps, const T* dx_init = nullptr) { check(hsddp_phase_batch_linear_rollout(b_, eps, dx_init), "hsddp_phase_batch_linear_rollout"); }
    void get(int which, std::vector<T>& out) { check(hsddp_phase_batch_get(b_, which, out.data()), "hsddp_phase_batch_get"); }
    int n_problems() const { return n_; }
private:
    hsddp_phase_batch* b_ = nullptr;
    int n_ = 0;
};

}  // namespace hsddp_b200
