"""Regularisation retries run side by side in the phased driver (HSDDP_SWEEP_SPEC): a batch of problems that regularise, solved
with the four-warp sweep in every round, gives bitwise the results of the sequential retry loop for 2, 4 and 8 candidates -- when
a candidate succeeds, when every candidate fails and the problem's block goes on alone, and when the retries end in
REG_OVERFLOW."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
STORED = ("Xbar", "X", "Defect", "dX", "Ubar", "U", "dU", "K", "g", "h", "al", "reb", "G0", "H0")
SCAN = 8192


def _handle(pkg, monkeypatch, spec):
    # HSDDP_SWEEP_SPEC is read at handle creation.  The batch (at most 32 problems) never reaches the one-warp sweep's
    # threshold, so every round of the phased driver takes the four-warp sweep and is eligible
    monkeypatch.setenv("HSDDP_SWEEP_SPEC", str(spec))
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_solve_mode(2)
    return B


def _solve(pkg, monkeypatch, w, spec, opt):
    B = _handle(pkg, monkeypatch, spec)
    B.set_problems(w.schedules, w.schedule_id)
    B.set_initial_condition(w.x0)
    B.reset()
    B.reset_counters()
    B.solve(opt)
    return dict(info=B.info(), trace=B.trace(), **{k: B.get(k) for k in STORED}), B.speculation()


@pytest.fixture(scope="module")
def regularising(pkg, workloads):
    """Config-3 entries whose solve retries the backward sweep (most retries per iteration first), and a few that never do."""
    import os
    name, e = workloads.define("config3", SCAN)
    w = workloads.from_entries(pkg, name, e)
    old = os.environ.get("HSDDP_SWEEP_SPEC")
    os.environ["HSDDP_SWEEP_SPEC"] = "0"
    try:
        B = pkg.MultiPhaseDDPBatch(0)
    finally:
        if old is None:
            del os.environ["HSDDP_SWEEP_SPEC"]
        else:
            os.environ["HSDDP_SWEEP_SPEC"] = old
    B.set_problems(w.schedules, w.schedule_id)
    B.set_initial_condition(w.x0)
    B.solve()
    most = B.trace()[:, :, 5].max(axis=1)  # sweeps of the iteration that needed the most
    reg = np.argsort(-most, kind="stable")[:24]
    reg = reg[most[reg] >= 2]
    calm = np.flatnonzero(most == 1)[:8]
    assert len(reg) >= 4 and (most[reg] >= 3).any(), "config 3 has regularising problems with retry chains"
    return [e[i] for i in np.concatenate([reg, calm])], most[reg]


@pytest.mark.parametrize("case", ["window", "overflow"])
def test_speculated_retries_match_sequential_in_the_phased_driver(pkg, workloads, monkeypatch, regularising, case):
    entries, _ = regularising
    w = workloads.from_entries(pkg, "regularising", entries)
    # overflow: r_2 = 1e3 > 1e2, so every problem whose sweep fails at reg 1e-3 ends in REG_OVERFLOW (candidates 2.. never run)
    opt = pkg.Options(update_regularization=1e6) if case == "overflow" else pkg.Options()
    ref, off = _solve(pkg, monkeypatch, w, 0, opt)
    assert off == dict(rounds=0, later=0, exceeded=0)
    if case == "overflow":
        assert (ref["info"]["status"] == 3).any(), "some problem ends in REG_OVERFLOW"
    for spec in (2, 4, 8):
        got, cnt = _solve(pkg, monkeypatch, w, spec, opt)
        for k, v in ref.items():
            assert got[k].shape == v.shape and got[k].tobytes() == v.tobytes(), (case, spec, k)
        assert cnt["rounds"] > 0, (case, spec, cnt)
        if case == "window" and spec == 8:
            assert cnt["later"] > 0, cnt     # a candidate past the first was kept
        if case == "window" and spec == 2:
            assert cnt["exceeded"] > 0, cnt  # both candidates failed: the problem's block retried on its own
