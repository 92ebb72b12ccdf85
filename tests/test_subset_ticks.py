"""Per-problem MPC ticks (hsddp_batch_mpc_update_problems, _set_initial_condition_problems, _solve_problems,
_get_mpc_command_problems): staggered cohorts against batches of each cohort alone, isolation of the unlisted problems, the
latency kernel inside a large batch, the oracle, per-problem budgets, refusals, bounded schedule slots and the C++ shim."""
import os
import subprocess

import numpy as np
import pytest
from conftest import GAIT_PATH, ROOT

pytestmark = pytest.mark.gpu
RTOL = 1e-9
TICK = dict(max_AL_iter=2, max_DDP_iter=1)
COLD = dict(max_AL_iter=5, max_DDP_iter=10)
PLAN = 0.6


# --- helpers after the pattern of test_restart.py ---
def _refs(pkg, workloads):
    return [pkg.QuadReference(workloads.gait_path(g)) for g in workloads.GAITS]


def _x0(pkg, workloads, cases, first_perturbation=0):
    """Reference body state at the window start (+ a perturbation) and the matching foot state."""
    entries = [(g, k0, "reference", first_perturbation + i) for i, (g, k0) in enumerate(cases)]
    return workloads.initial_states(entries, pkg.compute_hkd_state)


def _batch(pkg, workloads, refs, cases, mode=0):
    order = list(workloads.GAITS)
    keys, sid = [], []
    for c in cases:
        if c not in keys:
            keys.append(c)
        sid.append(keys.index(c))
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems_from_gaits(refs, [order.index(g) for g, _ in keys], [k for _, k in keys], PLAN, sid)
    B.set_solve_mode(mode)
    return B


# every array get() returns as stored (the dense views A, B, lx, lu, lxx, luu are rebuilt from the stage records)
STORED = ("Xbar", "X", "Defect", "dX", "Ubar", "U", "dU", "K", "g", "h", "al", "reb", "G0", "H0")


def _state(B):
    """Everything a problem keeps, including the device schedule of its slot (read now: slots change under later calls)."""
    sid = B.schedule_ids()
    return dict(info=B.info(), trace=B.trace(), sid=sid, sched=[B.device_schedule(s) for s in sid], **{k: B.get(k) for k in STORED})


def _same_schedule(a, b):
    return (a["n_phases"] == b["n_phases"] and a["horizon"] == b["horizon"] and a["contact"] == b["contact"]
            and a["next_contact"] == b["next_contact"] and all(a[k].tobytes() == b[k].tobytes() for k in ("xr", "ur", "prel_r", "xinit")))


def _assert_problem_equal(A, i, B, j, what):
    """Problem i of state A and problem j of state B: bitwise equal results (rows up to the smaller row stride; the rest zero)."""
    assert A["info"][i].tobytes() == B["info"][j].tobytes(), (what, A["info"][i], B["info"][j])
    assert A["trace"][i].tobytes() == B["trace"][j].tobytes(), what
    for k in STORED:
        a, b = A[k][i], B[k][j]
        r = min(len(a), len(b))
        assert a[:r].tobytes() == b[:r].tobytes(), (what, k)
        assert not np.any(a[r:]) and not np.any(b[r:]), (what, k)
    assert _same_schedule(A["sched"][i], B["sched"][j]), what


def _assert_untouched(S0, S1, idx, what):
    for i in idx:
        assert S0["sid"][i] == S1["sid"][i], (what, i)
        _assert_problem_equal(S0, i, S1, i, (what, i))


# 24 problems, three gaits: shared schedules (trot 0 x4, bound 5 x4, ...) and schedules of one problem (trot 100, bound 200, pronk 300)
CASES = ([("trot", 0)] * 4 + [("trot", 30)] * 3 + [("trot", 100)] + [("bound", 5)] * 4 + [("bound", 60)] * 2 + [("bound", 200)]
         + [("pronk", 0)] * 3 + [("pronk", 40)] * 3 + [("pronk", 300)] + [("pronk", 120)] * 2)


def _subset_tick(pkg, M, idx, C=None, x=None, opt=None, snapshots=False):
    """One tick of the listed problems of M (update, states, solve, commands); C: a batch of just those problems, ticked with
    the whole-batch calls and the same states.  snapshots: every unlisted problem is checked unchanged around every call."""
    opt = opt or pkg.Options(**TICK)
    x = M.get_rows("Xbar", 1, 1)[idx, 0, :].copy() if x is None else x
    others = [i for i in range(M.n) if i not in idx]
    calls = [lambda: M.mpc_update(problems=idx), lambda: M.set_initial_condition(x, problems=idx), lambda: M.solve(opt, problems=idx),
             lambda: M.mpc_command(8, problems=idx)]
    S0 = _state(M) if snapshots else None
    out = None
    for k, call in enumerate(calls):
        out = call()
        if snapshots:
            S1 = _state(M)
            _assert_untouched(S0, S1, others, ("isolation", k))
            S0 = S1
    if C is not None:
        C.mpc_update()
        C.set_initial_condition(x)
        C.solve(opt)
        assert out.tobytes() == C.mpc_command(8).tobytes()
    return out


@pytest.mark.parametrize("mode", [0, 2], ids=["auto", "phased"])
def test_staggered_cohorts_match_batches_of_each_cohort(pkg, workloads, mode):
    """Cohort A (even problems) ticks every tick, cohort B (odd) every second tick, in one batch whose cohorts share most
    schedule slots.  Every problem is bitwise what a batch of its cohort alone computes with the whole-batch calls, and no subset
    call changes a problem it does not list."""
    refs = _refs(pkg, workloads)
    x0 = _x0(pkg, workloads, CASES)
    A, Bc = list(range(0, len(CASES), 2)), list(range(1, len(CASES), 2))
    M = _batch(pkg, workloads, refs, CASES, mode)
    CA, CB = _batch(pkg, workloads, refs, [CASES[i] for i in A], mode), _batch(pkg, workloads, refs, [CASES[i] for i in Bc], mode)
    for B, x in ((M, x0), (CA, x0[A]), (CB, x0[Bc])):
        B.set_initial_condition(x)
        B.solve(pkg.Options())
    for t in range(1, 9):
        for idx, C in [(A, CA)] + ([(Bc, CB)] if t % 2 == 0 else []):
            _subset_tick(pkg, M, idx, C, snapshots=True)
        SM, SA, SB = _state(M), _state(CA), _state(CB)
        for j, i in enumerate(A):
            _assert_problem_equal(SM, i, SA, j, ("A", t, i))
        for j, i in enumerate(Bc):
            _assert_problem_equal(SM, i, SB, j, ("B", t, i))


def test_one_problem_of_a_large_batch_runs_the_latency_kernel(pkg, workloads):
    """One problem of a 64-problem batch (beyond the concurrent line search's 32) solved and ticked alone five times is
    bitwise a one-problem batch with the same history: the cluster kernel with trial arrays per launch position."""
    refs = _refs(pkg, workloads)
    cases = (CASES * 3)[:64]
    x0 = _x0(pkg, workloads, cases)
    p = 37
    M, F = _batch(pkg, workloads, refs, cases), _batch(pkg, workloads, refs, [cases[p]])
    M.set_initial_condition(x0)
    F.set_initial_condition(x0[[p]])
    M.solve(pkg.Options(), problems=[p])
    F.solve(pkg.Options())
    for t in range(5):
        _subset_tick(pkg, M, [p], F)
        SM, SF = _state(M), _state(F)
        _assert_problem_equal(SM, p, SF, 0, ("latency", t))
    # a second listed problem takes launch position 0 on its own and 1 next to p; p keeps matching its control
    q = 5
    G = _batch(pkg, workloads, refs, [cases[q]])
    G.set_initial_condition(x0[[q]])
    M.solve(pkg.Options(), problems=[q])
    G.solve(pkg.Options())
    x = M.get_rows("Xbar", 1, 1)[[q, p], 0, :].copy()
    _subset_tick(pkg, M, [q, p], x=x)
    for C, i, xi in ((G, q, x[:1]), (F, p, x[1:])):
        C.mpc_update()
        C.set_initial_condition(xi)
        C.solve(pkg.Options(**TICK))
        _assert_problem_equal(_state(M), i, _state(C), 0, ("pair", i))


def test_staggered_ticks_match_oracle(pkg, orc, workloads):
    """Six problems in two cohorts (one ticks every tick, the other every third) for 20 ticks, against the oracle's
    Problem.mpc_update + 2 x 1 solves: the same phase tables, the same decisions and 1e-9 per row for well-posed problems."""
    import parity_check as pc
    refs = _refs(pkg, workloads)
    cases = [("trot", 0), ("trot", 0), ("bound", 5), ("pronk", 40), ("trot", 30), ("bound", 60)]
    x0 = _x0(pkg, workloads, cases)
    M = _batch(pkg, workloads, refs, cases)
    M.set_initial_condition(x0)
    M.solve(pkg.Options())
    tables = {g: orc.GaitTable(GAIT_PATH(g)) for g in workloads.GAITS}
    models = [orc.default_model()] + ([orc.MODEL_PORT] if orc.ref_available() else [])
    Q = [[orc.Problem(tables[g], w, PLAN, model=m) for m in models] for g, w in cases]
    for i, qs in enumerate(Q):
        for q in qs:
            q.x0 = x0[i]
            q.solve(COLD)
    alive = np.ones(len(cases), bool)
    for tick in range(1, 21):
        idx = [0, 2, 4] + ([1, 3, 5] if tick % 3 == 0 else [])
        x = np.array([Q[i][0].get("Xbar")[1] for i in idx])  # "measured" state: the oracle plan's next node
        _subset_tick(pkg, M, idx, x=x)
        info, Xb, Ub, K, sid = M.info(), M.get("Xbar"), M.get("Ubar"), M.get("K"), M.schedule_ids()
        for j, i in enumerate(idx):
            res = []
            for q in Q[i]:
                q.mpc_update()
                q.x0 = x[j]
                res.append(q.solve(TICK)[0])
            if len(res) > 1 and not (res[0]["n_iter"] == res[1]["n_iter"] and res[0]["status"] == res[1]["status"]
                                     and abs(res[0]["cost"] - res[1]["cost"]) <= 1e-10 * abs(res[0]["cost"])):
                alive[i] = False
            q, s = Q[i][0], res[0]
            d = M.device_schedule(sid[i])
            assert d["n_phases"] == q.n_phases and d["horizon"] == [ph["horizon"] for ph in q.phases], (tick, i)
            assert d["contact"] == [ph["contact"] for ph in q.phases], (tick, i)
            if not alive[i]:
                continue
            assert info["n_iter"][i] == int(s["n_iter"]) and info["status"][i] == int(s["status"]), (tick, i, s, info[i])
            S, N = q.n_states, q.n_stages
            assert float(pc.rel_err_rows(Xb[i, :S][None], q.get("Xbar")[None], 1e-6)[0]) < RTOL, (tick, i)
            assert float(pc.rel_err_rows(Ub[i, :N][None], q.get("Ubar")[None], 1e-6)[0]) < RTOL, (tick, i)
            assert float(pc.rel_err_rows(K[i, :N][None], q.get("K")[None], 1e-6)[0]) < RTOL, (tick, i)
            assert abs(info["cost"][i] - s["cost"]) <= RTOL * abs(s["cost"]), (tick, i)
    assert alive.sum() >= len(cases) - 1, alive


def test_subset_solves_use_only_the_listed_budgets(pkg, workloads):
    """Two problems restarted with a 5 x 10 first solve; a solve of one of them uses its cold budget and leaves the other's
    pending: each is bitwise a fresh batch solved cold, and the first is back to the tick budget at its next solve."""
    refs = _refs(pkg, workloads)
    order = list(workloads.GAITS)
    M = _batch(pkg, workloads, refs, CASES)
    M.set_initial_condition(_x0(pkg, workloads, CASES))
    M.solve(pkg.Options())
    M.mpc_update()
    M.set_initial_condition(M.get_rows("Xbar", 1, 1)[:, 0, :].copy())
    probs, new_cases = [3, 10], [("bound", 10), ("pronk", 200)]
    xr = _x0(pkg, workloads, new_cases, first_perturbation=100)
    M.restart(probs, [order.index(g) for g, _ in new_cases], [w for _, w in new_cases], xr, pkg.Options(**COLD))
    for j, p in enumerate(probs):
        M.solve(pkg.Options(**TICK), problems=[p])
        F = _batch(pkg, workloads, refs, [new_cases[j]])
        F.set_initial_condition(xr[[j]])
        F.solve(pkg.Options(**COLD))
        _assert_problem_equal(_state(M), p, _state(F), 0, ("cold budget", p))
        assert M.info()["n_iter"][p] > 2
    M.solve(pkg.Options(**TICK), problems=[3])
    assert M.info()["n_iter"][3] <= 2


def test_refused_subset_calls_change_nothing(pkg, workloads):
    """Every refusal returns the documented code and leaves the batch as it was: the next tick is bitwise that of a batch
    that was never asked.  A listed problem whose table runs out fails the whole update, the other listed problems included."""
    refs = _refs(pkg, workloads)
    ahead = 2
    last = refs[0].n - int(round(PLAN / 0.01)) - 2  # the last window of the trot table that fits
    cases = [("trot", last - ahead), ("trot", 0), ("trot", 0), ("bound", 5), ("pronk", 40), ("bound", 60)]
    x0 = _x0(pkg, workloads, cases)
    R, C = _batch(pkg, workloads, refs, cases), _batch(pkg, workloads, refs, cases)
    for B in (R, C):
        B.set_initial_condition(x0)
        B.solve(pkg.Options())
    lib, ip = pkg.lib(), pkg._ip
    one, z1 = np.array([1], np.int32), np.zeros((1, 24))
    for bad in ([1, 1], [6], [-1], []):
        for call in (lambda p: R.mpc_update(problems=p), lambda p: R.set_initial_condition(np.zeros((len(p), 24)), problems=p),
                     lambda p: R.solve(pkg.Options(**TICK), problems=p), lambda p: R.mpc_command(8, problems=p)):
            with pytest.raises(pkg.HsddpError) as e:
                call(bad)
            assert e.value.code == pkg.ERR_ARG, (bad, e.value)
    assert lib.hsddp_batch_set_initial_condition_problems(R.h, 1, ip(one), None) == pkg.ERR_ARG
    assert lib.hsddp_batch_get_mpc_command_problems(R.h, 8, 1, ip(one), None) == pkg.ERR_ARG
    assert lib.hsddp_batch_get_mpc_command_problems(R.h, 0, 1, ip(one), np.zeros(1, pkg.CMD_DTYPE).ctypes.data_as(pkg.C.c_void_p)) == pkg.ERR_ARG
    with pytest.raises(pkg.HsddpError) as e:
        R.solve(pkg.Options(alpha=2.0), problems=[1])
    assert e.value.code == pkg.ERR_ARG
    for tick in range(ahead):  # whole-batch ticks; the second leaves problem 0 at the end of its table
        x = R.get_rows("Xbar", 1, 1)[:, 0, :].copy()
        for B in (R, C):
            B.mpc_update()
            B.set_initial_condition(x)
            B.solve(pkg.Options(**TICK))
        SR, SC = _state(R), _state(C)
        for i in range(len(cases)):
            _assert_problem_equal(SR, i, SC, i, ("refused", tick, i))
    with pytest.raises(pkg.HsddpError) as e:
        R.mpc_update(problems=[2, 0, 3])
    assert e.value.code == pkg.ERR_ARG and "exhausted" in str(e.value)
    idx = [1, 2, 3, 4, 5]
    x = R.get_rows("Xbar", 1, 1)[idx, 0, :].copy()
    for B in (R, C):
        _subset_tick(pkg, B, idx, x=x)
    SR, SC = _state(R), _state(C)
    for i in range(len(cases)):
        _assert_problem_equal(SR, i, SC, i, ("after the exhausted table", i))
    # a batch of host-built schedules has no gait library on the device
    w = workloads.config3(pkg, 6)
    H = pkg.MultiPhaseDDPBatch(0)
    H.set_problems(w.schedules, w.schedule_id)
    with pytest.raises(pkg.HsddpError) as e:
        H.mpc_update(problems=[0])
    assert e.value.code == pkg.ERR_STATE


def test_schedule_slots_stay_bounded(pkg, workloads):
    """30 staggered ticks of three cohorts (every tick, every second, every third): schedule slots stay below
    n_problems + the 24 a call may list, and a whole-batch tick afterwards succeeds."""
    refs = _refs(pkg, workloads)
    M = _batch(pkg, workloads, refs, CASES)
    M.set_initial_condition(_x0(pkg, workloads, CASES))
    M.solve(pkg.Options())
    cohorts = [list(range(0, 24, 3)), list(range(1, 24, 3)), list(range(2, 24, 3))]
    for t in range(1, 31):
        for c, every in zip(cohorts, (1, 2, 3)):
            if t % every == 0:
                _subset_tick(pkg, M, c)
                assert M.schedule_ids().max() < len(CASES) + 24, (t, M.schedule_ids())
    M.mpc_update()
    M.set_initial_condition(M.get_rows("Xbar", 1, 1)[:, 0, :].copy())
    M.solve(pkg.Options(**TICK))
    assert np.all(np.isfinite(M.get("Xbar")))


def test_cpp_shim_subset_ticks_match_python(pkg, workloads, tmp_path):
    """examples/subset_tick.cpp drives MultiPhaseDDP<double>::{update,set_initial_condition,solve,get_mpc_command}_problems and
    MultiGpuDDP's global-index split (one part); its command records equal the Python path's bit for bit."""
    t = workloads.gait_table("trot")
    rows = len(t["contact"])
    refs = [pkg.QuadReference(workloads.gait_path("trot"))]
    cases = [("trot", 0), ("trot", 0), ("trot", 20), ("trot", 20), ("trot", 0), ("trot", 20)]
    x0 = _x0(pkg, workloads, cases)
    inp, cmd = str(tmp_path / "input.bin"), str(tmp_path / "commands.bin")
    with open(inp, "wb") as f:
        f.write(np.int32(rows).tobytes() + np.float32(t["dt"]).tobytes())
        for k in ("body_state", "qJ", "foot_placements", "grf"):
            f.write(np.ascontiguousarray(np.asarray(t[k], np.float32).astype(np.float64).reshape(rows, 12)).tobytes())
        f.write(np.ascontiguousarray(t["contact"], np.int32).tobytes())
        f.write(np.ascontiguousarray(x0, np.float64).tobytes())
    exe = str(tmp_path / "subset_tick")
    libdir = os.path.dirname(pkg.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-Wall", os.path.join(ROOT, "examples", "subset_tick.cpp"), "-L" + libdir, "-lhsddp_b200",
                           "-Wl,-rpath," + libdir, "-o", exe])
    r = subprocess.run([exe, inp, cmd], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = np.fromfile(cmd, dtype=pkg.CMD_DTYPE)
    M = pkg.MultiPhaseDDPBatch(0)
    M.set_problems_from_gaits(refs, [0, 0], [0, 20], PLAN, [0, 0, 1, 1, 0, 1])
    M.set_initial_condition(x0)
    M.solve(pkg.Options())
    want = []
    for tick in range(1, 5):
        idx = [0, 2, 5, 1, 3] if tick % 2 == 0 else [0, 2, 5]
        x = x0[idx].copy()
        x[:, 3] += 0.0005 * tick
        want.append(_subset_tick(pkg, M, idx, x=x))
    want = np.concatenate(want)
    assert len(got) == len(want) and got.tobytes() == want.tobytes()
