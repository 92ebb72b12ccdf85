"""Both calls that move problems between schedule slots in one batch: whole-batch ticks, restarts (hsddp_batch_restart_problems)
and per-problem ticks (hsddp_batch_mpc_update_problems and the other list calls) interleaved, every problem checked after every
call against fresh batches of the problems that share its history, a refused per-problem update followed by a restart and a
whole-batch update, and the bound on the schedule slots."""
import numpy as np
import pytest
from test_subset_ticks import CASES, COLD, PLAN, TICK, _assert_problem_equal, _batch, _refs, _state, _x0

pytestmark = pytest.mark.gpu
# the per-problem cohort: problem 0 shares trot 0 with the unlisted 1..3, problem 8 shares bound 5 with the unlisted 9..11, and
# problem 5 is restarted together with the unlisted 12 onto one (gait, window)
COHORT = [0, 5, 8, 15, 21]
PAIR, PAIR_CASE = [5, 12], ("bound", 10)
LONGEST_LIST = len(COHORT)


class Mirror:
    """The batch M and its controls: problem i of M is problem ctl[i][1] of the fresh batch ctl[i][0], which takes every call that
    M's problem i takes as a whole-batch call.  A control's problems that no longer stand for a problem of M (restarted in M)
    follow along and are not compared."""

    def __init__(self, pkg, workloads):
        self.pkg, self.workloads, self.refs = pkg, workloads, _refs(pkg, workloads)
        x0 = _x0(pkg, workloads, CASES)
        self.M = _batch(pkg, workloads, self.refs, CASES)
        self.M.set_initial_condition(x0)
        self.ctl, self.cold = {}, set()
        rest = [i for i in range(len(CASES)) if i not in COHORT]
        for idx in (COHORT, rest):
            C = _batch(pkg, workloads, self.refs, [CASES[i] for i in idx])
            C.set_initial_condition(x0[idx])
            for j, i in enumerate(idx):
                self.ctl[i] = (C, j)
        self.solve(None, pkg.Options())

    def controls(self, idx):
        out = []
        for i in idx:
            if self.ctl[i][0] not in out:
                out.append(self.ctl[i][0])
        return out

    def check(self, what):
        SM = _state(self.M)
        assert SM["sid"].max() < len(CASES) + LONGEST_LIST, (what, SM["sid"])
        states = {id(C): _state(C) for C in self.controls(range(len(CASES)))}
        for i, (C, j) in self.ctl.items():
            _assert_problem_equal(SM, i, states[id(C)], j, (what, i))

    def update(self, idx):
        self.M.mpc_update(problems=idx)
        for C in self.controls(idx or range(len(CASES))):
            C.mpc_update()
        self.check(("update", idx))

    def states(self, idx):
        rows = idx or list(range(len(CASES)))
        x = self.M.get_rows("Xbar", 1, 1)[rows, 0, :].copy()
        self.M.set_initial_condition(x, problems=idx)
        for C in self.controls(rows):
            xc = C.get_rows("Xbar", 1, 1)[:, 0, :].copy()
            for k, i in enumerate(rows):
                if self.ctl[i][0] is C:
                    xc[self.ctl[i][1]] = x[k]
            C.set_initial_condition(xc)
        self.check(("states", idx))

    def solve(self, idx, opt):
        self.M.solve(opt, problems=idx)
        for C in self.controls(idx or range(len(CASES))):
            C.solve(self.pkg.Options(**COLD) if C in self.cold else opt)
            self.cold.discard(C)
        self.check(("solve", idx))

    def command(self, idx):
        got = self.M.mpc_command(8, problems=idx)
        want = {id(C): C.mpc_command(8) for C in self.controls(idx)}
        for k, i in enumerate(idx):
            C, j = self.ctl[i]
            assert got[k].tobytes() == want[id(C)][j].tobytes(), ("command", i)

    def tick(self, idx=None):
        """update, states, solve and (listed problems) commands of the listed problems, None: of the whole batch"""
        self.update(idx)
        self.states(idx)
        self.solve(idx, self.pkg.Options(**TICK))
        if idx:
            self.command(idx)

    def restart(self, probs, case, seed):
        order = list(self.workloads.GAITS)
        xr = _x0(self.pkg, self.workloads, [case] * len(probs), first_perturbation=seed)
        self.M.restart(probs, order.index(case[0]), case[1], xr, self.pkg.Options(**COLD))
        for k, i in enumerate(probs):  # one fresh batch per restarted problem: they tick with different cohorts afterwards
            F = _batch(self.pkg, self.workloads, self.refs, [case])
            F.set_initial_condition(xr[[k]])
            self.ctl[i] = (F, 0)
            self.cold.add(F)
        self.check(("restart", probs, case))


def test_restarts_and_per_problem_ticks_in_one_batch(pkg, workloads):
    """Whole-batch ticks, a restart of two problems onto one shared (gait, window) and per-problem ticks of a cohort that holds
    one of them and problems whose slots unlisted problems share: after every call every problem is bitwise its control.  Then a
    per-problem update that the end of a gait table refuses, a restart of that problem back to window 0, and a whole-batch
    update that must succeed: a copy dropped by the refusal that still counted as in use would be stepped off its table."""
    X = Mirror(pkg, workloads)
    X.tick()
    X.tick(COHORT)
    X.restart(PAIR, PAIR_CASE, 100)
    sid = X.M.schedule_ids()
    assert sid[PAIR[0]] == sid[PAIR[1]]
    X.tick(COHORT)
    X.tick()
    X.tick(COHORT)
    assert len(set(X.M.schedule_ids()[PAIR])) == 2
    # problem 14 at the last window of the trot table that builds: its next update runs out of reference rows.  It is listed
    # after problem 1, so that its dropped copy is not the free slot that the restart to trot window 0 takes next.  That slot
    # is the dropped copy of problem 1's trot-0 slot: its initial-guess rows past the ones the restart builds are those of a
    # fresh trot-0 schedule too, and an update that adds a node reads one of them.
    last = X.refs[0].n - int(round(PLAN / 0.01)) - 2
    X.restart([14], ("trot", last), 200)
    with pytest.raises(pkg.HsddpError) as e:
        X.M.mpc_update(problems=[1, 14])
    assert e.value.code == pkg.ERR_ARG and "exhausted" in str(e.value)
    X.check("refused")
    X.restart([14], ("trot", 0), 300)
    X.tick()
    X.tick(COHORT)
    X.tick()
