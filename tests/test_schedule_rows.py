"""Reference rows of the schedules the device builds from the gait library: after the build and after every receding-horizon
update, every node row of xr / ur / prel_r equals the oracle's reference for that stage bit for bit; and a restarted
problem's new schedule slot holds exactly what a fresh batch builds for the same (gait, window)."""
import numpy as np
import pytest
from conftest import GAIT_PATH

pytestmark = pytest.mark.gpu
PLAN = 0.6
# the windows of test_receding_horizon_ticks_match_oracle: first phases removed, last phases grown and opened, a phase
# reaching its end, two problems sharing a schedule
CASES = [("trot", 0), ("trot", 0), ("trot", 23), ("bound", 0), ("bound", 5), ("bound", 240), ("pronk", 0), ("pronk", 100), ("pronk", 40)]
# (problem, new gait, new window) of the restart: a pair used twice, and a window another schedule started from
RESTARTS = [(0, "bound", 30), (3, "pronk", 7), (5, "bound", 30), (8, "trot", 23)]
TICKS, RESTART_TICK = 30, 12


def _assert_rows_match_oracle(d, Q, what):
    """Schedule d (device_schedule) against oracle problem Q: phase table and, per node, xr / ur and prel_r = foot_r - body_r[3:6]."""
    assert d["n_phases"] == Q.n_phases and d["horizon"] == [p["horizon"] for p in Q.phases], (what, d["horizon"])
    assert d["contact"] == [p["contact"] for p in Q.phases], what
    n = 0
    for ph, p in enumerate(Q.phases):
        for k in range(p["horizon"] + 1):
            xr, ur, body_r, foot_r, _ = Q.stage_reference(ph, k)
            prel = (foot_r.reshape(4, 3) - body_r[3:6]).reshape(12)
            assert d["xr"][n].tobytes() == xr.tobytes(), (what, ph, k, "xr")
            assert d["ur"][n].tobytes() == ur.tobytes(), (what, ph, k, "ur")
            assert d["prel_r"][n].tobytes() == prel.tobytes(), (what, ph, k, "prel_r")
            n += 1
    assert n == len(d["xr"]), what


def _assert_same_schedule(a, b, what):
    for key in ("n_phases", "horizon", "contact", "next_contact"):
        assert a[key] == b[key], (what, key)
    for key in ("xr", "ur", "prel_r", "xinit"):
        assert a[key].tobytes() == b[key].tobytes(), (what, key)


def test_receding_horizon_and_restart_rows_are_bit_exact(pkg, orc, workloads):
    order = list(workloads.GAITS)
    refs = [pkg.QuadReference(workloads.gait_path(g)) for g in order]
    tables = {g: orc.GaitTable(GAIT_PATH(g)) for g in order}
    keys, sid = [], []
    for c in CASES:
        if c not in keys:
            keys.append(c)
        sid.append(keys.index(c))
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems_from_gaits(refs, [order.index(g) for g, _ in keys], [k for _, k in keys], PLAN, sid)
    P = [orc.Problem(tables[g], k0, PLAN) for g, k0 in CASES]
    for tick in range(-1, TICKS):
        if tick >= 0:
            B.mpc_update()
            for Q in P:
                Q.mpc_update()
        if tick == RESTART_TICK:
            probs = [i for i, _, _ in RESTARTS]
            x0 = np.stack([B.get("Xbar")[i, 0] for i in probs])
            B.restart(probs, [order.index(g) for _, g, _ in RESTARTS], [k0 for _, _, k0 in RESTARTS], x0)
            for i, g, k0 in RESTARTS:
                P[i] = orc.Problem(tables[g], k0, PLAN)
            # the new slots hold what a fresh batch builds for the same pairs
            pairs = sorted({(g, k0) for _, g, k0 in RESTARTS})
            F = pkg.MultiPhaseDDPBatch(0)
            F.set_problems_from_gaits(refs, [order.index(g) for g, _ in pairs], [k0 for _, k0 in pairs], PLAN, np.arange(len(pairs)))
            slots = B.schedule_ids()
            for i, g, k0 in RESTARTS:
                _assert_same_schedule(B.device_schedule(slots[i]), F.device_schedule(pairs.index((g, k0))), (tick, i, g, k0))
        slots = B.schedule_ids()
        for i, Q in enumerate(P):
            _assert_rows_match_oracle(B.device_schedule(slots[i]), Q, (tick, i))
