"""hkd-mpc_b200 — B200-native batched Hybrid-Systems DDP (host-side Python binding).

Thin ctypes layer over the C ABI of include/hsddp_b200.h (libhsddp_b200.so, built
in-tree by `make -C hkd-mpc_b200`).  It mirrors the reference's solver surface for
the one hot path this repository replaces:

    MultiPhaseDDP<double>            HSDDPSolver/header/MultiPhaseDDP.h:18-122
    HKDProblem<double>::initialization  HKDMPC/HKD-TrajOpt/HKDProblem.cpp:15-111
    QuadReference                    Reference/QuadReference.h:144-191

There is NO CPU fallback: every Batch method runs CUDA kernels and raises
HsddpError when the library or a device is missing.  The directory name has a
hyphen (the repository's contract), so import it with
`importlib.import_module("hkd-mpc_b200")` or via `tests/conftest.py::load_pkg`.
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# HSDDP_LIB selects a development variant of the library (profiling builds); the default is the in-tree product build
LIB_PATH = os.environ.get("HSDDP_LIB") or os.path.join(_HERE, "libhsddp_b200.so")

MAX_PHASES = 16
MAX_STAGES = 128
TRACE_CAP = 64

STATUS_NAMES = {0: "converged", 1: "stalled", 2: "max_iter", 3: "reg_overflow"}

ARR = dict(Xbar=0, X=1, Defect=3, dX=4, G0=5, Ubar=10, U=11, dU=12, K=20, A=21, B=22, lxx=24, luu=25, H0=27,
           lx=30, lu=31, h=50, al=51, g=52, reb=53)


class HsddpError(RuntimeError):
    """A C-ABI call failed; `code` is its HSDDP_ERR_* return value."""

    def __init__(self, msg, code=None):
        super().__init__(msg)
        self.code = code


ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED, ERR_STATE = -1, -2, -3, -4


class Options(C.Structure):
    """HSDDP_OPTION (HSDDPSolver/common/HSDDP_CompoundTypes.h:18-60) as consumed by solve():
    the values of HKDMPC/settings/ddp_setting.info, update_regularization = 2 (never loaded)."""
    _fields_ = [("alpha", C.c_double), ("gamma", C.c_double), ("update_penalty", C.c_double), ("update_relax", C.c_double),
                ("update_regularization", C.c_double), ("update_ReB", C.c_double), ("max_DDP_iter", C.c_int32),
                ("max_AL_iter", C.c_int32), ("cost_thresh", C.c_double), ("tconstr_thresh", C.c_double),
                ("pconstr_thresh", C.c_double), ("dynamics_feas_thresh", C.c_double), ("merit_scale", C.c_double),
                ("merit_offset", C.c_double), ("AL_active", C.c_int32), ("ReB_active", C.c_int32), ("MS", C.c_int32),
                ("_pad", C.c_int32)]

    def __init__(self, **over):
        super().__init__()
        d = dict(alpha=0.1, gamma=0.01, update_penalty=5, update_relax=1, update_regularization=2, update_ReB=1,
                 max_DDP_iter=10, max_AL_iter=5, cost_thresh=1e-3, tconstr_thresh=1e-3, pconstr_thresh=1e-3,
                 dynamics_feas_thresh=1e-3, merit_scale=0.2, merit_offset=1e2, AL_active=1, ReB_active=1, MS=1)
        d.update(over)
        for k, v in d.items():
            setattr(self, k, v)


class ConstraintParams(C.Structure):
    """HKDMPC/settings/constraint_params.info + mu (HKDConstraints.h:17)."""
    _fields_ = [("grf_delta", C.c_double), ("grf_delta_min", C.c_double), ("grf_eps", C.c_double), ("td_sigma", C.c_double),
                ("td_sigma_max", C.c_double), ("td_lambda", C.c_double), ("mu", C.c_double)]

    def __init__(self, **over):
        super().__init__()
        d = dict(grf_delta=0.1, grf_delta_min=0.1, grf_eps=0.1, td_sigma=50.0, td_sigma_max=1e4, td_lambda=0.0, mu=0.7)
        d.update(over)
        for k, v in d.items():
            setattr(self, k, v)


class ScheduleStruct(C.Structure):
    _fields_ = [("n_phases", C.c_int32), ("n_stages", C.c_int32), ("n_nodes", C.c_int32),
                ("horizon", C.c_int32 * MAX_PHASES), ("contact", (C.c_int32 * 4) * MAX_PHASES),
                ("next_contact", (C.c_int32 * 4) * MAX_PHASES), ("start_time", C.c_float * MAX_PHASES), ("dt", C.c_double),
                ("xr", C.POINTER(C.c_double)), ("ur", C.POINTER(C.c_double)), ("prel_r", C.POINTER(C.c_double)),
                ("xinit", C.POINTER(C.c_double))]


class Info(C.Structure):
    _fields_ = [("status", C.c_int32), ("n_iter", C.c_int32), ("n_outer", C.c_int32), ("n_sweeps", C.c_int32),
                ("n_trials", C.c_int32), ("_pad", C.c_int32), ("cost", C.c_double), ("feas", C.c_double),
                ("max_tconstr", C.c_double), ("max_pconstr", C.c_double), ("cost0", C.c_double), ("feas0", C.c_double)]


INFO_DTYPE = np.dtype([("status", "i4"), ("n_iter", "i4"), ("n_outer", "i4"), ("n_sweeps", "i4"), ("n_trials", "i4"),
                       ("_pad", "i4"), ("cost", "f8"), ("feas", "f8"), ("max_tconstr", "f8"), ("max_pconstr", "f8"),
                       ("cost0", "f8"), ("feas0", "f8")])
TRACE_COLS = ["outer", "inner", "cost_before", "feas_before", "reg_after", "n_sweeps", "dV_1", "dV_2", "merit_rho",
              "eps_accepted", "n_trials", "cost_after", "feas_after", "max_tconstr", "max_pconstr", "pad"]

CMD_MAX_STEPS = 10
CMD_DTYPE = np.dtype([("N_mpcsteps", "i4"), ("foot_found", "i4", (4,)), ("contacts", "i4", (CMD_MAX_STEPS, 4)),
                      ("hkd_controls", "f4", (CMD_MAX_STEPS, 24)), ("des_body_state", "f4", (CMD_MAX_STEPS, 12)),
                      ("feedback", "f4", (CMD_MAX_STEPS, 12, 12)), ("foot_placement", "f4", (12,)), ("_pad", "i4")])

_lib = None


def build(force=False):
    """Compile libhsddp_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))]
    srcs += [os.path.join(_HERE, "host", f) for f in os.listdir(os.path.join(_HERE, "host"))]
    srcs.append(os.path.join(_HERE, "..", "include", "hsddp_b200.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        if not os.path.exists("/usr/local/cuda/bin/nvcc"):
            raise HsddpError("libhsddp_b200.so is missing or stale and nvcc is not available to build it")
        subprocess.check_call(["make", "-C", _HERE, "libhsddp_b200.so"], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        L = C.CDLL(LIB_PATH)
        dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_void_p
        L.hsddp_last_error.restype = C.c_char_p
        L.hkd_gait_create.argtypes = [C.c_int, C.c_float] + [C.POINTER(C.c_float)] * 4 + [ip, C.POINTER(vp)]
        L.hkd_gait_load.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.hkd_gait_size.argtypes = [vp]
        L.hkd_gait_destroy.argtypes = [vp]
        L.hkd_schedule_build.argtypes = [vp, C.c_int, C.c_float, C.POINTER(ScheduleStruct)]
        L.hkd_schedule_free.argtypes = [C.POINTER(ScheduleStruct)]
        L.hkd_compute_state.argtypes = [dp, dp, dp, ip, dp]
        L.hkd_default_x0.argtypes = [C.POINTER(ScheduleStruct), dp]
        L.hkd_model_dynamics.argtypes = [dp, dp, C.c_double, ip, dp]
        L.hkd_model_dynamics_partial.argtypes = [dp, dp, C.c_double, ip, dp, dp]
        L.hkd_model_foot_position.argtypes = [dp, dp, dp, C.c_int, dp]
        L.hkd_model_foot_jacobian.argtypes = [dp, dp, dp, C.c_int, dp]
        L.hsddp_batch_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.hsddp_batch_destroy.argtypes = [vp]
        L.hsddp_batch_set_problems.argtypes = [vp, C.c_int, C.POINTER(ScheduleStruct), C.c_int, ip, C.POINTER(ConstraintParams)]
        L.hsddp_batch_set_initial_condition.argtypes = [vp, dp]
        L.hsddp_batch_reset.argtypes = [vp]
        L.hsddp_batch_mpc_update.argtypes = [vp]
        L.hsddp_batch_last_update_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.hsddp_batch_restart_problems.argtypes = [vp, C.c_int, ip, ip, ip, dp, C.POINTER(Options)]
        L.hsddp_batch_get_schedule_ids.argtypes = [vp, ip]
        for f in ("hsddp_batch_solve", "hsddp_batch_solve_async", "hsddp_batch_compute_cost", "hsddp_batch_lq_approximation",
                  "hsddp_batch_prepare_merit", "hsddp_batch_update_al_params", "hsddp_batch_update_reb_params"):
            getattr(L, f).argtypes = [vp, C.POINTER(Options)]
        L.hsddp_batch_sync.argtypes = [vp]
        L.hsddp_batch_update_nominal.argtypes = [vp]
        L.hsddp_batch_last_solve_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.hsddp_batch_hybrid_rollout.argtypes = [vp, C.c_double, C.POINTER(Options), ip]
        L.hsddp_batch_backward_sweep.argtypes = [vp, C.c_double, ip]
        L.hsddp_batch_backward_sweep_regularized.argtypes = [vp, dp, C.POINTER(Options), ip]
        L.hsddp_batch_linear_rollout.argtypes = [vp, C.c_double, C.POINTER(Options)]
        L.hsddp_batch_forward_sweep.argtypes = [vp, C.POINTER(Options), ip, dp]
        L.hsddp_batch_dims.argtypes = [vp, ip, ip, ip]
        L.hsddp_batch_get_info.argtypes = [vp, vp]
        L.hsddp_batch_get_trace.argtypes = [vp, dp]
        L.hsddp_batch_get_scalars.argtypes = [vp, dp]
        L.hsddp_batch_get_array.argtypes = [vp, C.c_int, dp]
        L.hsddp_batch_set_array.argtypes = [vp, C.c_int, dp]
        L.hsddp_fp64_peak_tflops.argtypes = [C.c_int, C.c_int, dp]
        L.hsddp_batch_get_array_rows.argtypes = [vp, C.c_int, C.c_int, C.c_int, dp]
        L.hsddp_batch_get_gains_compact.argtypes = [vp, C.c_int, C.c_int, dp]
        L.hsddp_batch_get_mpc_command.argtypes = [vp, C.c_int, vp]
        L.hsddp_batch_set_problems_from_gaits.argtypes = [vp, C.c_int, ip, C.POINTER(C.c_float), dp, dp, dp, dp, ip, C.c_int, ip, ip, C.c_float, C.c_int, ip,
                                                          C.POINTER(ConstraintParams)]
        L.hsddp_batch_get_schedule.argtypes = [vp, C.c_int, ip, ip, ip, ip, dp, dp, dp, dp]
        L.hsddp_batch_set_solve_mode.argtypes = [vp, C.c_int]
        L.hsddp_batch_event_record.argtypes = [vp, C.c_int]
        L.hsddp_batch_event_elapsed_ms.argtypes = [vp, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.hsddp_batch_get_counters.argtypes = [vp, C.POINTER(C.c_ulonglong)]
        L.hsddp_batch_reset_counters.argtypes = [vp]
        L.hsddp_batch_get_speculation.argtypes = [vp, C.POINTER(C.c_ulonglong)]
        L.hsddp_batch_get_profile.argtypes = [vp, C.POINTER(C.c_ulonglong)]
        L.hsddp_phase_batch_create.argtypes = [C.c_int] * 6 + [C.POINTER(vp)]
        L.hsddp_phase_batch_destroy.argtypes = [vp]
        L.hsddp_phase_batch_set.argtypes = [vp, C.c_int, dp]
        L.hsddp_phase_batch_backward_sweep.argtypes = [vp, C.c_double, dp, dp, ip]
        L.hsddp_phase_batch_linear_rollout.argtypes = [vp, C.c_double, dp]
        L.hsddp_phase_batch_set_gains.argtypes = [vp, dp, dp]
        L.hsddp_phase_batch_get.argtypes = [vp, C.c_int, dp]
        L.hsddp_phase_batch_last_ms.argtypes = [vp, C.POINTER(C.c_float)]
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _check(rc, what):
    if rc != 0:
        raise HsddpError(f"{what} failed with code {rc}: {lib().hsddp_last_error().decode()}", rc)


# --------------------------------------------------------------------------
# host-side model functions (same code the kernels run)
# --------------------------------------------------------------------------
def model_dynamics(x, u, dt, contact):
    x = np.ascontiguousarray(x, np.float64); u = np.ascontiguousarray(u, np.float64)
    c = np.ascontiguousarray(contact, np.int32); xn = np.zeros(24)
    lib().hkd_model_dynamics(_dp(x), _dp(u), float(dt), _ip(c), _dp(xn))
    return xn


def model_dynamics_partial(x, u, dt, contact):
    x = np.ascontiguousarray(x, np.float64); u = np.ascontiguousarray(u, np.float64)
    c = np.ascontiguousarray(contact, np.int32); A = np.zeros(576); B = np.zeros(576)
    lib().hkd_model_dynamics_partial(_dp(x), _dp(u), float(dt), _ip(c), _dp(A), _dp(B))
    return A.reshape(24, 24).T.copy(), B.reshape(24, 24).T.copy()


def model_foot_position(pos, eul, q, leg):
    pos = np.ascontiguousarray(pos, np.float64); eul = np.ascontiguousarray(eul, np.float64); q = np.ascontiguousarray(q, np.float64)
    p = np.zeros(3)
    lib().hkd_model_foot_position(_dp(pos), _dp(eul), _dp(q), int(leg), _dp(p))
    return p


def model_foot_jacobian(pos, eul, q, leg):
    pos = np.ascontiguousarray(pos, np.float64); eul = np.ascontiguousarray(eul, np.float64); q = np.ascontiguousarray(q, np.float64)
    J = np.zeros(54)
    lib().hkd_model_foot_jacobian(_dp(pos), _dp(eul), _dp(q), int(leg), _dp(J))
    return J.reshape(18, 3).T.copy()


def compute_hkd_state(eul, pos, qJ, contact):
    """compute_hkd_state, HKDModel.h:65-96."""
    eul = np.ascontiguousarray(eul, np.float64); pos = np.ascontiguousarray(pos, np.float64); qJ = np.ascontiguousarray(qJ, np.float64)
    c = np.ascontiguousarray(contact, np.int32); qd = np.zeros(12)
    lib().hkd_compute_state(_dp(eul), _dp(pos), _dp(qJ), _ip(c), _dp(qd))
    return qd


# --------------------------------------------------------------------------
# problem assembly
# --------------------------------------------------------------------------
class QuadReference:
    """Top-level reference table (QuadReference::tp_data)."""

    def __init__(self, source):
        h = C.c_void_p()
        if isinstance(source, (str, bytes)) and not str(source).endswith(".npz"):
            _check(lib().hkd_gait_load(str(source).encode(), C.byref(h)), "hkd_gait_load")
        else:
            d = np.load(source) if isinstance(source, (str, bytes)) else source
            self._keep = [np.ascontiguousarray(d[k], np.float32) for k in ("body_state", "qJ", "foot_placements", "grf")]
            contact = np.ascontiguousarray(d["contact"], np.int32)
            self._keep.append(contact)
            self.dt = float(d["dt"])
            _check(lib().hkd_gait_create(contact.shape[0], C.c_float(float(d["dt"])), *[_fp(a) for a in self._keep[:4]],
                                         _ip(contact), C.byref(h)), "hkd_gait_create")
        self.handle = h
        self.n = lib().hkd_gait_size(h)

    def __del__(self):
        try:
            lib().hkd_gait_destroy(self.handle)
        except Exception:
            pass


class Schedule:
    """HKDProblem::initialization for one reference window."""

    def __init__(self, ref: QuadReference, window_start=0, plan_duration=0.6):
        self.s = ScheduleStruct()
        _check(lib().hkd_schedule_build(ref.handle, int(window_start), C.c_float(plan_duration), C.byref(self.s)), "hkd_schedule_build")
        self.ref = ref
        self.n_phases, self.n_stages, self.n_nodes = self.s.n_phases, self.s.n_stages, self.s.n_nodes
        self.horizon = [self.s.horizon[i] for i in range(self.n_phases)]
        self.contact = [list(self.s.contact[i]) for i in range(self.n_phases)]
        self.next_contact = [list(self.s.next_contact[i]) for i in range(self.n_phases)]
        self.start_time = [self.s.start_time[i] for i in range(self.n_phases)]
        self.dt = self.s.dt

    def array(self, name):
        cols = 12 if name == "prel_r" else 24
        return np.ctypeslib.as_array(getattr(self.s, name), shape=(self.n_nodes, cols)).copy()

    def default_x0(self):
        x0 = np.zeros(24)
        lib().hkd_default_x0(C.byref(self.s), _dp(x0))
        return x0

    def __del__(self):
        try:
            lib().hkd_schedule_free(C.byref(self.s))
        except Exception:
            pass


class MultiPhaseDDPBatch:
    """MultiPhaseDDP<double> over a batch of independent HKD problems on one GPU."""

    def __init__(self, device=0):
        h = C.c_void_p()
        _check(lib().hsddp_batch_create(int(device), C.byref(h)), "hsddp_batch_create")
        self.h = h
        self.n = 0

    def __del__(self):
        try:
            lib().hsddp_batch_destroy(self.h)
        except Exception:
            pass

    # set_multiPhaseProblem
    def set_problems(self, schedules, schedule_id, cparams=None):
        arr = (ScheduleStruct * len(schedules))(*[s.s for s in schedules])
        sid = np.ascontiguousarray(schedule_id, np.int32)
        cp = cparams or ConstraintParams()
        _check(lib().hsddp_batch_set_problems(self.h, len(schedules), arr, len(sid), _ip(sid), C.byref(cp)), "hsddp_batch_set_problems")
        self.n = len(sid)
        self.schedules = list(schedules)
        self.schedule_id = sid
        ms, mn, n = C.c_int32(), C.c_int32(), C.c_int32()
        lib().hsddp_batch_dims(self.h, C.byref(n), C.byref(ms), C.byref(mn))
        self.max_stages, self.max_nodes = ms.value, mn.value

    def set_problems_from_gaits(self, refs, sched_gait, sched_window, plan_duration, schedule_id, cparams=None):
        """Reference ingestion on the device (SURVEY.md §8f N2): the gait tables `refs` (QuadReference objects created
        from arrays) go to HBM once, and a kernel builds the schedule of every (gait, window start) pair."""
        rows = np.array([r.n for r in refs], np.int32)
        dts = np.array([r.dt for r in refs], np.float32)
        cat = [np.ascontiguousarray(np.concatenate([np.asarray(r._keep[k], np.float64).reshape(-1, 12) for r in refs])) for k in range(4)]
        contact = np.ascontiguousarray(np.concatenate([r._keep[4].reshape(-1, 4) for r in refs]), np.int32)
        sg = np.ascontiguousarray(sched_gait, np.int32); sw = np.ascontiguousarray(sched_window, np.int32)
        sid = np.ascontiguousarray(schedule_id, np.int32)
        cp = cparams or ConstraintParams()
        _check(lib().hsddp_batch_set_problems_from_gaits(self.h, len(refs), _ip(rows), dts.ctypes.data_as(C.POINTER(C.c_float)), *[_dp(a) for a in cat],
                                                        _ip(contact), len(sg), _ip(sg), _ip(sw), C.c_float(plan_duration), len(sid), _ip(sid),
                                                        C.byref(cp)), "hsddp_batch_set_problems_from_gaits")
        n, ms, mn = C.c_int32(), C.c_int32(), C.c_int32()
        lib().hsddp_batch_dims(self.h, C.byref(n), C.byref(ms), C.byref(mn))
        self.n, self.max_stages, self.max_nodes = n.value, ms.value, mn.value

    def device_schedule(self, i):
        """Schedule i as the device holds it (phase table + reference rows)."""
        nph = C.c_int32()
        hz = np.zeros(MAX_PHASES, np.int32); c = np.zeros((MAX_PHASES, 4), np.int32); cn = np.zeros((MAX_PHASES, 4), np.int32)
        mn = self.max_nodes
        xr, ur, pr, xi = np.zeros((mn, 24)), np.zeros((mn, 24)), np.zeros((mn, 12)), np.zeros((mn, 24))
        _check(lib().hsddp_batch_get_schedule(self.h, int(i), C.byref(nph), _ip(hz), _ip(c), _ip(cn), _dp(xr), _dp(ur), _dp(pr), _dp(xi)), "get_schedule")
        P = nph.value
        nn = int(hz[:P].sum()) + P
        return dict(n_phases=P, horizon=hz[:P].tolist(), contact=c[:P].tolist(), next_contact=cn[:P].tolist(), xr=xr[:nn], ur=ur[:nn], prel_r=pr[:nn], xinit=xi[:nn])

    def set_initial_condition(self, x0):
        x0 = np.ascontiguousarray(x0, np.float64).reshape(self.n, 24)
        _check(lib().hsddp_batch_set_initial_condition(self.h, _dp(x0)), "hsddp_batch_set_initial_condition")

    def reset(self):
        _check(lib().hsddp_batch_reset(self.h), "hsddp_batch_reset")

    def mpc_update(self):
        """HKDProblem::update for every problem (receding-horizon shift by one MPC step, on the device)."""
        _check(lib().hsddp_batch_mpc_update(self.h), "hsddp_batch_mpc_update")

    def restart(self, problems, gait, window, x0, first_solve=None):
        """HKDMPCSolver::initialize for some problems of the batch: problem problems[k] restarts on the reference window that
        starts at sample window[k] of gait gait[k] (index into the gait list of set_problems_from_gaits) from state x0[k], with
        the cold-start guess and fresh ReB / AL parameters; the other problems keep everything.  first_solve (Options or None):
        max_AL_iter / max_DDP_iter of the next solve of these problems only.  Call it after mpc_update and
        set_initial_condition of the tick, before solve."""
        p = np.ascontiguousarray(problems, np.int32).ravel()
        g = np.ascontiguousarray(np.broadcast_to(np.asarray(gait, np.int32), p.shape))
        w = np.ascontiguousarray(np.broadcast_to(np.asarray(window, np.int32), p.shape))
        x = np.ascontiguousarray(x0, np.float64).reshape(len(p), 24)
        _check(lib().hsddp_batch_restart_problems(self.h, len(p), _ip(p), _ip(g), _ip(w), _dp(x), None if first_solve is None else C.byref(first_solve)),
               "hsddp_batch_restart_problems")

    def schedule_ids(self):
        """Schedule slot of every problem (the index device_schedule takes)."""
        out = np.zeros(self.n, np.int32)
        _check(lib().hsddp_batch_get_schedule_ids(self.h, _ip(out)), "hsddp_batch_get_schedule_ids")
        return out

    def last_update_ms(self):
        ms = C.c_float()
        _check(lib().hsddp_batch_last_update_ms(self.h, C.byref(ms)), "hsddp_batch_last_update_ms")
        return ms.value

    def solve(self, opt=None):
        opt = opt or Options()
        _check(lib().hsddp_batch_solve(self.h, C.byref(opt)), "hsddp_batch_solve")

    def solve_async(self, opt=None):
        opt = opt or Options()
        _check(lib().hsddp_batch_solve_async(self.h, C.byref(opt)), "hsddp_batch_solve_async")

    def set_solve_mode(self, mode):
        """0 auto, 1 persistent kernel, 2 phased kernels (see include/hsddp_b200.h)."""
        _check(lib().hsddp_batch_set_solve_mode(self.h, int(mode)), "hsddp_batch_set_solve_mode")

    def sync(self):
        _check(lib().hsddp_batch_sync(self.h), "hsddp_batch_sync")

    def last_solve_ms(self):
        ms = C.c_float()
        _check(lib().hsddp_batch_last_solve_ms(self.h, C.byref(ms)), "hsddp_batch_last_solve_ms")
        return ms.value

    # step-level API
    def hybrid_rollout(self, eps, opt=None):
        opt = opt or Options(); ok = np.zeros(self.n, np.int32)
        _check(lib().hsddp_batch_hybrid_rollout(self.h, float(eps), C.byref(opt), _ip(ok)), "hybrid_rollout")
        return ok.astype(bool)

    def compute_cost(self, opt=None):
        opt = opt or Options(); _check(lib().hsddp_batch_compute_cost(self.h, C.byref(opt)), "compute_cost")

    def lq_approximation(self, opt=None):
        opt = opt or Options(); _check(lib().hsddp_batch_lq_approximation(self.h, C.byref(opt)), "lq_approximation")

    def backward_sweep(self, reg):
        ok = np.zeros(self.n, np.int32)
        _check(lib().hsddp_batch_backward_sweep(self.h, float(reg), _ip(ok)), "backward_sweep")
        return ok.astype(bool)

    def backward_sweep_regularized(self, reg, opt=None):
        opt = opt or Options(); ok = np.zeros(self.n, np.int32)
        reg = np.ascontiguousarray(np.broadcast_to(np.asarray(reg, np.float64), (self.n,))).copy()
        _check(lib().hsddp_batch_backward_sweep_regularized(self.h, _dp(reg), C.byref(opt), _ip(ok)), "backward_sweep_regularized")
        return ok.astype(bool), reg

    def linear_rollout(self, eps, opt=None):
        opt = opt or Options(); _check(lib().hsddp_batch_linear_rollout(self.h, float(eps), C.byref(opt)), "linear_rollout")

    def prepare_merit(self, opt=None):
        opt = opt or Options(); _check(lib().hsddp_batch_prepare_merit(self.h, C.byref(opt)), "prepare_merit")

    def forward_sweep(self, opt=None):
        opt = opt or Options(); ok = np.zeros(self.n, np.int32); eps = np.zeros(self.n)
        _check(lib().hsddp_batch_forward_sweep(self.h, C.byref(opt), _ip(ok), _dp(eps)), "forward_sweep")
        return ok.astype(bool), eps

    def update_nominal(self):
        _check(lib().hsddp_batch_update_nominal(self.h), "update_nominal")

    def update_al_params(self, opt=None):
        opt = opt or Options(); _check(lib().hsddp_batch_update_al_params(self.h, C.byref(opt)), "update_al_params")

    def update_reb_params(self, opt=None):
        opt = opt or Options(); _check(lib().hsddp_batch_update_reb_params(self.h, C.byref(opt)), "update_reb_params")

    # results
    def info(self):
        out = np.zeros(self.n, INFO_DTYPE)
        _check(lib().hsddp_batch_get_info(self.h, out.ctypes.data_as(C.c_void_p)), "get_info")
        return out

    def trace(self):
        out = np.zeros((self.n, TRACE_CAP, 16))
        _check(lib().hsddp_batch_get_trace(self.h, _dp(out)), "get_trace")
        return out

    def scalars(self):
        out = np.zeros((self.n, 8))
        _check(lib().hsddp_batch_get_scalars(self.h, _dp(out)), "get_scalars")
        return out  # actual_cost, merit, feas, dV_1, dV_2, max_tconstr, max_pconstr, merit_rho

    def get(self, name):
        which = ARR[name]
        S, N = self.max_nodes, self.max_stages
        shape = {"Xbar": (S, 24), "X": (S, 24), "Defect": (S, 24), "dX": (S, 24), "Ubar": (N, 24), "U": (N, 24), "dU": (N, 24),
                 "K": (N, 24, 24), "A": (N, 24, 24), "B": (N, 24, 24), "lxx": (N, 24, 24), "luu": (N, 24, 24), "lx": (N, 24),
                 "lu": (N, 24), "G0": (24,), "H0": (24, 24), "g": (N, 20), "h": (MAX_PHASES, 4), "al": (MAX_PHASES, 2, 4, 2), "reb": (N, 20, 2)}[name]
        out = np.zeros((self.n,) + shape)
        _check(lib().hsddp_batch_get_array(self.h, which, _dp(out)), "get_array")
        if name in ("K", "A", "B", "lxx", "luu", "H0"):
            out = np.ascontiguousarray(np.swapaxes(out, -1, -2))  # column-major blocks -> [row, col]
        return out

    def get_rows(self, name, row0, nrows, out=None):
        cols = {"K": 576, "g": 20, "h": 4, "al": 16, "reb": 40}.get(name, 24)
        if out is None:
            out = np.zeros((self.n, nrows, cols))
        _check(lib().hsddp_batch_get_array_rows(self.h, ARR[name], int(row0), int(nrows), _dp(out)), "get_array_rows")
        return out

    def get_gains_compact(self, row0, nrows, out=None):
        if out is None:
            out = np.zeros((self.n, nrows, 24, 12))
        _check(lib().hsddp_batch_get_gains_compact(self.h, int(row0), int(nrows), _dp(out)), "get_gains_compact")
        return out

    def mpc_command(self, n_steps=8, out=None):
        """hkd_command_lcmt payload of every problem (HKDMPC.cpp:207-298), packed on the device."""
        if out is None:
            out = np.zeros(self.n, dtype=CMD_DTYPE)
        _check(lib().hsddp_batch_get_mpc_command(self.h, int(n_steps), out.ctypes.data_as(C.c_void_p)), "get_mpc_command")
        return out

    def event_record(self, slot):
        _check(lib().hsddp_batch_event_record(self.h, int(slot)), "event_record")

    def event_elapsed_ms(self, slot0, slot1):
        ms = C.c_float()
        _check(lib().hsddp_batch_event_elapsed_ms(self.h, int(slot0), int(slot1), C.byref(ms)), "event_elapsed_ms")
        return ms.value

    def counters(self):
        out = (C.c_ulonglong * 4)()
        _check(lib().hsddp_batch_get_counters(self.h, out), "get_counters")
        return dict(sweep_stages=int(out[0]), solve_launches=int(out[1]), step_launches=int(out[2]))

    def speculation(self):
        """Regularisation retries run side by side since set_problems / reset_counters (HSDDP_SWEEP_SPEC): problem-rounds
        speculated, rounds that kept a later candidate than the first, rounds in which every candidate failed."""
        out = (C.c_ulonglong * 3)()
        _check(lib().hsddp_batch_get_speculation(self.h, out), "get_speculation")
        return dict(rounds=int(out[0]), later=int(out[1]), exceeded=int(out[2]))

    def profile(self):
        out = (C.c_ulonglong * 16)()
        _check(lib().hsddp_batch_get_profile(self.h, out), "get_profile")
        return [int(v) for v in out]

    def reset_counters(self):
        _check(lib().hsddp_batch_reset_counters(self.h), "reset_counters")

    def set(self, name, arr):
        arr = np.ascontiguousarray(arr, np.float64)
        if name == "K":
            arr = np.ascontiguousarray(np.swapaxes(arr, -1, -2))
        _check(lib().hsddp_batch_set_array(self.h, ARR[name], _dp(arr)), "set_array")



class SinglePhaseBatch:
    """The model-independent sweeps of SinglePhase<double, xs, us, ys> (HSDDPSolver/source/SinglePhase.cpp:145-178,
    299-367) for the reference's other instantiations <12,12,0> and <36,12,12> (and <24,24,0>, dense), on a batch of
    independent phases of equal horizon.  Inputs are what LQ_approximation leaves in the phase's storage; matrices are
    given and returned as [..., row, col] arrays (the C ABI is column-major)."""
    INPUTS = ["A", "B", "C", "D", "lx", "lu", "ly", "lxx", "luu", "lux", "lyy", "Phix", "Phixx", "Defect"]
    OUTPUTS = ["dU", "K", "G", "H", "dX", "dV"]
    _MATS = {"A", "B", "C", "D", "lxx", "luu", "lux", "lyy", "Phixx", "K", "H"}

    def __init__(self, xs, us, ys, horizon, n_problems, device=0):
        self.xs, self.us, self.ys, self.N, self.n = int(xs), int(us), int(ys), int(horizon), int(n_problems)
        self.h = C.c_void_p()
        _check(lib().hsddp_phase_batch_create(int(device), self.xs, self.us, self.ys, self.N, self.n, C.byref(self.h)), "hsddp_phase_batch_create")

    def __del__(self):
        try:
            if self.h:
                lib().hsddp_phase_batch_destroy(self.h)
        except Exception:
            pass

    def shape(self, name):
        xs, us, ys, N, n = self.xs, self.us, self.ys, self.N, self.n
        return dict(A=(n, N, xs, xs), B=(n, N, xs, us), C=(n, N, ys, xs), D=(n, N, ys, us), lx=(n, N, xs), lu=(n, N, us), ly=(n, N, ys),
                    lxx=(n, N, xs, xs), luu=(n, N, us, us), lux=(n, N, us, xs), lyy=(n, N, ys, ys), Phix=(n, xs), Phixx=(n, xs, xs),
                    Defect=(n, N + 1, xs), dU=(n, N, us), K=(n, N, us, xs), G=(n, N + 1, xs), H=(n, N + 1, xs, xs), dX=(n, N + 1, xs),
                    dV=(n, 2), Gprime=(n, xs), Hprime=(n, xs, xs), dx_init=(n, xs))[name]

    def _to_c(self, name, arr):
        a = np.asarray(arr, np.float64)
        if a.shape != self.shape(name):
            raise ValueError(f"{name}: shape {a.shape}, expected {self.shape(name)}")
        if name in self._MATS | {"Hprime"}:
            a = np.swapaxes(a, -1, -2)
        return np.ascontiguousarray(a)

    def set(self, name, arr):
        a = self._to_c(name, arr)
        if a.size:
            _check(lib().hsddp_phase_batch_set(self.h, self.INPUTS.index(name), _dp(a)), "hsddp_phase_batch_set")

    def backward_sweep(self, reg, Gprime=None, Hprime=None):
        ok = np.zeros(self.n, np.int32)
        g = None if Gprime is None else self._to_c("Gprime", Gprime)
        h = None if Hprime is None else self._to_c("Hprime", Hprime)
        _check(lib().hsddp_phase_batch_backward_sweep(self.h, float(reg), None if g is None else _dp(g), None if h is None else _dp(h), _ip(ok)),
               "hsddp_phase_batch_backward_sweep")
        return ok.astype(bool)

    def linear_rollout(self, eps, dx_init=None):
        d = None if dx_init is None else self._to_c("dx_init", dx_init)
        _check(lib().hsddp_phase_batch_linear_rollout(self.h, float(eps), None if d is None else _dp(d)), "hsddp_phase_batch_linear_rollout")

    def set_gains(self, dU, K):
        _check(lib().hsddp_phase_batch_set_gains(self.h, _dp(self._to_c("dU", dU)), _dp(self._to_c("K", K))), "hsddp_phase_batch_set_gains")

    def get(self, name):
        shp = self.shape(name)
        cshape = shp[:-2] + (shp[-1], shp[-2]) if name in self._MATS else shp
        out = np.zeros(cshape)
        _check(lib().hsddp_phase_batch_get(self.h, self.OUTPUTS.index(name), _dp(out)), "hsddp_phase_batch_get")
        return np.ascontiguousarray(np.swapaxes(out, -1, -2)) if name in self._MATS else out

    def last_ms(self):
        ms = C.c_float()
        _check(lib().hsddp_phase_batch_last_ms(self.h, C.byref(ms)), "hsddp_phase_batch_last_ms")
        return ms.value


def fp64_peak_tflops(device=0, kind=0):
    out = C.c_double()
    _check(lib().hsddp_fp64_peak_tflops(int(device), int(kind), C.byref(out)), "hsddp_fp64_peak_tflops")
    return out.value
