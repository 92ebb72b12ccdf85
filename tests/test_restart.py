"""Restarting individual problems of a running batch (hsddp_batch_restart_problems): isolation from the other problems,
equivalence with a fresh batch, receding-horizon ticks after a restart against the oracle, recycling a problem whose gait
table runs out, bounded schedule slots, and refusals that leave the batch untouched."""
import numpy as np
import pytest
from conftest import GAIT_PATH, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-9
TICK = dict(max_AL_iter=2, max_DDP_iter=1)
COLD = dict(max_AL_iter=5, max_DDP_iter=10)
PLAN = 0.6


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


def _tick(B, x=None):
    x = B.get_rows("Xbar", 1, 1)[:, 0, :].copy() if x is None else x
    B.mpc_update()
    B.set_initial_condition(x)
    return x


# every array get() returns as stored (the dense views A, B, lx, lu, lxx, luu are rebuilt from the stage records)
STORED = ("Xbar", "X", "Defect", "dX", "Ubar", "U", "dU", "K", "g", "h", "al", "reb", "G0", "H0")


def _state(B):
    return dict(info=B.info(), trace=B.trace(), sid=B.schedule_ids(), **{k: B.get(k) for k in STORED})


def _same_schedule(a, b):
    return (a["n_phases"] == b["n_phases"] and a["horizon"] == b["horizon"] and a["contact"] == b["contact"]
            and a["next_contact"] == b["next_contact"] and all(a[k].tobytes() == b[k].tobytes() for k in ("xr", "ur", "prel_r", "xinit")))


def _assert_problem_equal(A, i, B, j, dA, dB, what):
    """Problem i of batch A and problem j of batch B: bitwise equal results (rows up to the smaller row stride; the rest zero)."""
    assert A["info"][i].tobytes() == B["info"][j].tobytes(), (what, A["info"][i], B["info"][j])
    assert A["trace"][i].tobytes() == B["trace"][j].tobytes(), what
    for k in STORED:
        a, b = A[k][i], B[k][j]
        r = min(len(a), len(b))
        assert a[:r].tobytes() == b[:r].tobytes(), (what, k)
        assert not np.any(a[r:]) and not np.any(b[r:]), (what, k)
    assert _same_schedule(dA.device_schedule(A["sid"][i]), dB.device_schedule(B["sid"][j])), what


# 24 problems, three gaits: shared schedules (trot 0 x4, bound 5 x4, ...) and schedules of one problem (trot 100, bound 200, pronk 300)
CASES = ([("trot", 0)] * 4 + [("trot", 30)] * 3 + [("trot", 100)] + [("bound", 5)] * 4 + [("bound", 60)] * 2 + [("bound", 200)]
         + [("pronk", 0)] * 3 + [("pronk", 40)] * 3 + [("pronk", 300)] + [("pronk", 120)] * 2)
# (problem, gait, window): two problems of the shared trot-0 schedule to the same new (gait, window) (one slot for both), the only
# user of trot 100, a problem of a shared bound schedule back to trot window 0, a pronk problem to another pronk window, one of the
# pronk-120 pair to a bound window
RESTARTS = [(0, "bound", 10), (1, "bound", 10), (7, "pronk", 200), (9, "trot", 0), (20, "pronk", 41), (22, "bound", 33)]


def _restart_setup(pkg, workloads, mode):
    refs = _refs(pkg, workloads)
    order = list(workloads.GAITS)
    x0 = _x0(pkg, workloads, CASES)
    R, C = _batch(pkg, workloads, refs, CASES, mode), _batch(pkg, workloads, refs, CASES, mode)
    for B in (R, C):
        B.set_initial_condition(x0)
        B.solve(pkg.Options())
    for _ in range(5):
        x = _tick(R)
        _tick(C, x)
        R.solve(pkg.Options(**TICK)); C.solve(pkg.Options(**TICK))
    x = _tick(R)
    _tick(C, x)
    probs = [p for p, _, _ in RESTARTS]
    new_cases = [(g, w) for _, g, w in RESTARTS]
    xr = _x0(pkg, workloads, new_cases, first_perturbation=100)
    R.restart(probs, [order.index(g) for g in [c[0] for c in new_cases]], [w for _, w in new_cases], xr, pkg.Options(**COLD))
    return refs, R, C, probs, new_cases, xr


@pytest.mark.parametrize("mode", [0, 2], ids=["auto", "phased"])
def test_restart_isolation_and_fresh_equivalence(pkg, workloads, mode):
    """Untouched problems are bitwise what a batch without the restart computes; restarted problems are bitwise what a fresh
    batch of just those (gait, window, x0) computes with a cold 5 x 10 solve, in the same driver."""
    refs, R, C, probs, new_cases, xr = _restart_setup(pkg, workloads, mode)
    sid = R.schedule_ids()
    assert sid[0] == sid[1] and len(set(sid[probs])) == len(probs) - 1  # (one slot for the pair restarted to the same window)
    R.solve(pkg.Options(**TICK)); C.solve(pkg.Options(**TICK))
    F = _batch(pkg, workloads, refs, new_cases, mode)
    F.set_initial_condition(xr)
    F.solve(pkg.Options(**COLD))
    SR, SC, SF = _state(R), _state(C), _state(F)
    for i in range(len(CASES)):
        if i not in probs:
            _assert_problem_equal(SR, i, SC, i, R, C, ("untouched", i))
    for j, p in enumerate(probs):
        _assert_problem_equal(SR, p, SF, j, R, F, ("restarted", p))
    assert SR["info"]["n_iter"][probs].max() > 2  # (the cold budget was used, not the tick's)
    # the override is consumed by that solve: the next tick runs every problem on the tick budget
    _tick(R)
    R.solve(pkg.Options(**TICK))
    assert R.info()["n_iter"].max() <= 2


def test_ticks_after_restart_match_oracle(pkg, orc, workloads):
    """The restarted problems, then 20 receding-horizon ticks with the MPC budget, against the oracle's Problem(table, window):
    cold solve, then mpc_update + 2 x 1 solves.  Phase tables equal the oracle's; well-posed problems take the oracle's decisions
    and agree to 1e-9 per row."""
    refs, R, C, probs, new_cases, xr = _restart_setup(pkg, workloads, 0)
    tables = {g: orc.GaitTable(GAIT_PATH(g)) for g in workloads.GAITS}
    models = [orc.default_model()] + ([orc.MODEL_PORT] if orc.ref_available() else [])
    Q = [[orc.Problem(tables[g], w, PLAN, model=m) for m in models] for g, w in new_cases]
    alive = np.ones(len(probs), bool)
    import parity_check as pc
    for tick in range(21):
        if tick > 0:
            x = R.get_rows("Xbar", 1, 1)[:, 0, :].copy()
            for j, p in enumerate(probs):
                x[p] = Q[j][0].get("Xbar")[1]  # "measured" state: the oracle plan's next node
            _tick(R, x)
        R.solve(pkg.Options(**TICK))
        info, Xb, Ub, K, sid = R.info(), R.get("Xbar"), R.get("Ubar"), R.get("K"), R.schedule_ids()
        for j, p in enumerate(probs):
            res = []
            for q in Q[j]:
                if tick > 0:
                    q.mpc_update()
                    q.x0 = x[p]
                else:
                    q.x0 = xr[j]
                res.append(q.solve(TICK if tick > 0 else COLD)[0])
            if len(res) > 1 and not (res[0]["n_iter"] == res[1]["n_iter"] and res[0]["status"] == res[1]["status"]
                                     and abs(res[0]["cost"] - res[1]["cost"]) <= 1e-10 * abs(res[0]["cost"])):
                alive[j] = False
            q, s = Q[j][0], res[0]
            d = R.device_schedule(sid[p])
            assert d["n_phases"] == q.n_phases and d["horizon"] == [ph["horizon"] for ph in q.phases], (tick, p)
            assert d["contact"] == [ph["contact"] for ph in q.phases], (tick, p)
            if not alive[j]:
                continue
            assert info["n_iter"][p] == int(s["n_iter"]) and info["status"][p] == int(s["status"]), (tick, p, s, info[p])
            S, N = q.n_states, q.n_stages
            assert float(pc.rel_err_rows(Xb[p, :S][None], q.get("Xbar")[None], 1e-6)[0]) < RTOL, (tick, p)
            assert float(pc.rel_err_rows(Ub[p, :N][None], q.get("Ubar")[None], 1e-6)[0]) < RTOL, (tick, p)
            assert float(pc.rel_err_rows(K[p, :N][None], q.get("K")[None], 1e-6)[0]) < RTOL, (tick, p)
            assert abs(info["cost"][p] - s["cost"]) <= RTOL * abs(s["cost"]), (tick, p)
    assert alive.sum() >= len(probs) - 1, alive


def test_restart_recycles_a_problem_past_the_end_of_its_table(pkg, workloads):
    """A problem a few ticks before the end of its gait table: without a restart the batch's update fails when the table runs
    out; restarted to window 0 one tick earlier, the batch keeps ticking (the old schedule's slot is free and skipped)."""
    refs = _refs(pkg, workloads)
    n_trot = refs[0].n
    # the last window that fits: a restart one sample later is refused
    probe = _batch(pkg, workloads, refs, [("trot", 0)])
    probe.set_initial_condition(_x0(pkg, workloads, [("trot", 0)]))
    last = n_trot - int(round(PLAN / 0.01)) - 2
    with pytest.raises(pkg.HsddpError) as e:
        probe.restart([0], [0], [last + 1], np.zeros((1, 24)))
    assert e.value.code == pkg.ERR_ARG
    probe.restart([0], [0], [last], np.zeros((1, 24)))
    ahead = 3
    cases = [("trot", last - ahead), ("bound", 0), ("pronk", 0)]
    x0 = _x0(pkg, workloads, cases)
    R, C = _batch(pkg, workloads, refs, cases), _batch(pkg, workloads, refs, cases)
    for B in (R, C):
        B.set_initial_condition(x0)
        B.solve(pkg.Options())
    for tick in range(1, ahead + 1):
        _tick(C)
        C.solve(pkg.Options(**TICK))
    with pytest.raises(pkg.HsddpError) as e:
        C.mpc_update()
    assert e.value.code == pkg.ERR_ARG and "exhausted" in str(e.value)
    for tick in range(1, ahead + 1):
        _tick(R)
        if tick == ahead:
            R.restart([0], [0], [0], _x0(pkg, workloads, [("trot", 0)]), pkg.Options(**COLD))
        R.solve(pkg.Options(**TICK))
    for tick in range(20):
        _tick(R)
        R.solve(pkg.Options(**TICK))
    assert np.all(np.isfinite(R.get("Xbar"))) and np.all(R.info()["status"] >= 0)


def test_schedule_slots_are_recycled(pkg, workloads):
    """200 single-problem restarts of a 9-problem batch: schedule slots stay bounded by the problem count (n_problems + the one
    being built), however many restarts there have been; the batch keeps ticking on the recycled slots."""
    refs = _refs(pkg, workloads)
    cases = [("trot", 0), ("trot", 0), ("trot", 23), ("bound", 0), ("bound", 5), ("bound", 240), ("pronk", 0), ("pronk", 100), ("pronk", 40)]
    B = _batch(pkg, workloads, refs, cases)
    B.set_initial_condition(_x0(pkg, workloads, cases))
    B.solve(pkg.Options())
    rng = np.random.default_rng(7)
    for call in range(200):
        p, g = call % 9, int(rng.integers(0, 3))
        B.restart([p], [g], [int(rng.integers(0, 200))], _x0(pkg, workloads, [(workloads.GAITS[g], 0)]))
        ids = B.schedule_ids()
        assert ids.max() < len(cases) + 1, (call, ids)
        if call % 20 == 19:
            _tick(B)
            B.solve(pkg.Options(**TICK))
    assert np.all(np.isfinite(B.get("Xbar")))


def test_refused_restarts_change_nothing(pkg, workloads):
    """Every refusal returns the documented code, and the next tick of the batch is bitwise that of a batch never asked."""
    refs = _refs(pkg, workloads)
    cases = [("trot", 0), ("trot", 0), ("bound", 5), ("pronk", 40), ("pronk", 100), ("bound", 60)]
    x0 = _x0(pkg, workloads, cases)
    R, C = _batch(pkg, workloads, refs, cases), _batch(pkg, workloads, refs, cases)
    for B in (R, C):
        B.set_initial_condition(x0)
        B.solve(pkg.Options())
    z1, z2 = np.zeros((1, 24)), np.zeros((2, 24))
    n_trot = refs[0].n
    refusals = [
        (dict(problems=[1, 1], gait=[0, 0], window=[0, 0], x0=z2), pkg.ERR_ARG),             # repeated index
        (dict(problems=[6], gait=[0], window=[0], x0=z1), pkg.ERR_ARG),                     # out of range
        (dict(problems=[-1], gait=[0], window=[0], x0=z1), pkg.ERR_ARG),
        (dict(problems=[2], gait=[3], window=[0], x0=z1), pkg.ERR_ARG),                     # unknown gait
        (dict(problems=[2], gait=[-1], window=[0], x0=z1), pkg.ERR_ARG),
        (dict(problems=[0, 2], gait=[0, 0], window=[3, n_trot - 10], x0=z2), pkg.ERR_ARG),  # a window past its table (the other fits)
        (dict(problems=[2], gait=[0], window=[-1], x0=z1), pkg.ERR_ARG),
        (dict(problems=[2], gait=[0], window=[0], x0=z1, first_solve=pkg.Options(max_AL_iter=-1)), pkg.ERR_ARG),
        (dict(problems=[2], gait=[0], window=[0], x0=z1, first_solve=pkg.Options(max_AL_iter=2000, max_DDP_iter=1000)), pkg.ERR_ARG),
    ]
    for kw, code in refusals:
        with pytest.raises(pkg.HsddpError) as e:
            R.restart(**kw)
        assert e.value.code == code, (kw, e.value)
    x = _tick(R)
    _tick(C, x)
    R.solve(pkg.Options(**TICK)); C.solve(pkg.Options(**TICK))
    SR, SC = _state(R), _state(C)
    for i in range(len(cases)):
        _assert_problem_equal(SR, i, SC, i, R, C, ("refused", i))
    # a batch of host-built schedules has no gait library on the device
    w = workloads.config3(pkg, 6)
    H, H2 = pkg.MultiPhaseDDPBatch(0), pkg.MultiPhaseDDPBatch(0)
    for B in (H, H2):
        B.set_problems(w.schedules, w.schedule_id)
        B.set_initial_condition(w.x0)
    with pytest.raises(pkg.HsddpError) as e:
        H.restart([0], [0], [0], z1)
    assert e.value.code == pkg.ERR_STATE
    H.solve(); H2.solve()
    assert H.info().tobytes() == H2.info().tobytes() and H.trace().tobytes() == H2.trace().tobytes()
    assert H.get("Xbar").tobytes() == H2.get("Xbar").tobytes() and H.get("K").tobytes() == H2.get("K").tobytes()
