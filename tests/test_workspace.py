"""The batch workspace of a reused handle: set_problems on a handle that held a batch with longer horizons leaves nothing of
it behind (rows past each problem's schedule are zero, and every array is bitwise what a fresh handle computes), and
get_rows reads each array with the row width get() uses."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
NODE = ("Xbar", "X", "Defect", "dX")              # [max_nodes][...]
STAGE = ("Ubar", "U", "dU", "K", "g", "reb")      # [max_stages][...]
PHASE = ("h", "al")                               # [MAX_PHASES][...]
STORED = NODE + STAGE + PHASE + ("G0", "H0")


def _solve(B, w):
    B.set_problems(w.schedules, w.schedule_id)
    B.set_initial_condition(w.x0)
    B.reset()
    B.solve()
    return dict(info=B.info(), trace=B.trace(), **{k: B.get(k) for k in STORED})


def _mixed(workloads, parts):
    """One batch of the problems of several workloads (schedules of different lengths side by side)."""
    off = np.cumsum([0] + [len(w.schedules) for w in parts[:-1]])
    return workloads.Workload("mixed", sum((w.schedules for w in parts), []), np.concatenate([w.schedule_id + o for w, o in zip(parts, off)]),
                              np.concatenate([w.x0 for w in parts]), sum((w.keys for w in parts), []), None)


def test_reused_handle_starts_from_zeros(pkg, workloads):
    # (both batches at most 32 problems, so they also have the trial arrays of the concurrent line search)
    longer = workloads.config3(pkg, 30, plan=0.9)
    shorter = _mixed(workloads, [workloads.config3(pkg, 12, plan=0.5), workloads.config3(pkg, 12, plan=0.3)])
    B = pkg.MultiPhaseDDPBatch(0)
    _solve(B, longer)
    reused = _solve(B, shorter)
    fresh = _solve(pkg.MultiPhaseDDPBatch(0), shorter)
    for k, v in fresh.items():
        assert reused[k].shape == v.shape and reused[k].tobytes() == v.tobytes(), k
    for i, s in enumerate(shorter.schedule_id):
        sc = shorter.schedules[s]
        for k in NODE:
            assert not np.any(reused[k][i, sc.n_nodes:]), (k, i)
        for k in STAGE:
            assert not np.any(reused[k][i, sc.n_stages:]), (k, i)

    # get_rows against get: every row-readable array, in get_rows' layout (K column-major), and the row counts
    rows = dict(**{k: B.max_nodes for k in NODE}, **{k: B.max_stages for k in STAGE}, **{k: pkg.MAX_PHASES for k in PHASE})
    for k, n in rows.items():
        full = reused[k]
        if k == "K":
            full = np.swapaxes(full, -1, -2)
        full = full.reshape(B.n, n, -1)
        for r0, nr in ((0, n), (3, 5), (n - 2, 2)):
            assert B.get_rows(k, r0, nr).tobytes() == np.ascontiguousarray(full[:, r0:r0 + nr]).tobytes(), (k, r0, nr)
        with pytest.raises(pkg.HsddpError) as e:
            B.get_rows(k, n - 2, 3)
        assert e.value.code == pkg.ERR_ARG, k
