"""Ticks from GPU memory (hsddp_batch_set_initial_condition_dev, _set_measured_state_dev, _get_mpc_command_dev): the same
results as the host path bit for bit, the measured-state ingest against compute_hkd_state on the host, the stream contract on
the caller's stream (inputs read after the caller's work, outputs visible to it, no host synchronise) and refusals that change
nothing."""
import os
import subprocess
import sys

import numpy as np
import pytest
from conftest import ROOT

TICK = dict(max_AL_iter=2, max_DDP_iter=1)
PLAN = 0.6
SLEEP_CYCLES = 500_000_000  # torch.cuda._sleep: a few hundred milliseconds at the B200's clocks


# --- helpers after the pattern of test_subset_ticks.py ---
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
    """Everything a problem keeps, including the device schedule of its slot."""
    sid = B.schedule_ids()
    return dict(info=B.info(), trace=B.trace(), sid=sid, sched=[B.device_schedule(s) for s in sid], **{k: B.get(k) for k in STORED})


def _same_schedule(a, b):
    return (a["n_phases"] == b["n_phases"] and a["horizon"] == b["horizon"] and a["contact"] == b["contact"]
            and a["next_contact"] == b["next_contact"] and all(a[k].tobytes() == b[k].tobytes() for k in ("xr", "ur", "prel_r", "xinit")))


def _assert_same_state(A, B, what):
    assert A["info"].tobytes() == B["info"].tobytes(), what
    assert A["trace"].tobytes() == B["trace"].tobytes(), what
    assert np.array_equal(A["sid"], B["sid"]), what
    for k in STORED:
        assert A[k].tobytes() == B[k].tobytes(), (what, k)
    assert all(_same_schedule(a, b) for a, b in zip(A["sched"], B["sched"])), what


# 24 problems, three gaits: shared schedules (trot 0 x4, bound 5 x4, ...) and schedules of one problem (trot 100, bound 200, pronk 300)
CASES = ([("trot", 0)] * 4 + [("trot", 30)] * 3 + [("trot", 100)] + [("bound", 5)] * 4 + [("bound", 60)] * 2 + [("bound", 200)]
         + [("pronk", 0)] * 3 + [("pronk", 40)] * 3 + [("pronk", 300)] + [("pronk", 120)] * 2)
SUBSET = [0, 2, 5, 7, 8, 13, 14, 16, 20, 23]


def _cmd_tensor(torch, pkg, n):
    return torch.full((n, pkg.CMD_DTYPE.itemsize), 0xAB, dtype=torch.uint8, device="cuda:0")


@pytest.fixture(scope="module")
def torch():
    t = pytest.importorskip("torch")
    if not t.cuda.is_available():
        pytest.skip("no CUDA device")
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 2], ids=["auto", "phased"])
@pytest.mark.parametrize("listed", [False, True], ids=["batch", "subset"])
def test_device_ticks_match_host_ticks(pkg, workloads, torch, mode, listed):
    """Two handles of one mixed-gait batch: one ticks with NumPy states and host commands, the other with the same states as
    CUDA tensors, solve_async and commands into a CUDA tensor.  Command records, info, trace and every stored array agree bit
    for bit after every tick."""
    refs = _refs(pkg, workloads)
    x0 = _x0(pkg, workloads, CASES)
    H, D = _batch(pkg, workloads, refs, CASES, mode), _batch(pkg, workloads, refs, CASES, mode)
    H.set_initial_condition(x0)
    D.set_initial_condition(torch.from_numpy(x0).cuda())
    for B in (H, D):
        B.solve(pkg.Options())
    _assert_same_state(_state(H), _state(D), "cold solve")
    p = SUBSET if listed else None
    opt = pkg.Options(**TICK)
    for t in range(1, 5):
        x = H.get_rows("Xbar", 1, 1)[:, 0, :]
        x = x[SUBSET].copy() if listed else x.copy()
        H.mpc_update(problems=p)
        H.set_initial_condition(x, problems=p)
        H.solve(opt, problems=p)
        want = H.mpc_command(8, problems=p)
        D.mpc_update(problems=p)
        D.set_initial_condition(torch.from_numpy(x).cuda(), problems=p)
        D.solve_async(opt, problems=p)
        out = D.mpc_command(8, out=_cmd_tensor(torch, pkg, len(x)), problems=p)
        got = out.cpu().numpy()
        assert got.tobytes() == want.tobytes(), ("commands", t)
        _assert_same_state(_state(H), _state(D), ("tick", t))


def _tick_until_contact_changes(pkg, workloads, B):
    """Whole-batch ticks until some problems' first phase has a contact other than the one at their window start."""
    tables = {g: workloads.gait_table(g) for g in workloads.GAITS}
    for t in range(1, 41):
        x = B.get_rows("Xbar", 1, 1)[:, 0, :].copy()
        B.mpc_update()
        B.set_initial_condition(x)
        B.solve(pkg.Options(**TICK))
        first = [B.device_schedule(s)["contact"][0] for s in B.schedule_ids()]
        start = [list(np.asarray(tables[g]["contact"][k0], np.int32)) for g, k0 in CASES]
        changed = [i for i in range(len(CASES)) if list(first[i]) != start[i]]
        if len(changed) >= 3:
            return changed
    pytest.fail("no first phase changed its contact in 40 ticks")


def _defect0(B):
    """Defect of node 0 after a rollout at step 0: x0 minus the (unchanged) trial state of node 0, so it carries x0."""
    B.hybrid_rollout(0.0)
    return B.get("Defect")[:, 0, :]


def _host_x0(pkg, meas, contact):
    """[meas[:12], compute_hkd_state(eul, pos, qJ, contact)] on the host."""
    x = meas.copy()
    for i in range(len(meas)):
        x[i, 12:] = pkg.compute_hkd_state(meas[i, 0:3], meas[i, 3:6], meas[i, 12:24], (np.asarray(contact[i]) != 0).astype(np.int32))
    return x


def _assert_ingested(Dd, Dh, contact, what):
    """Node-0 defects after the device ingest (Dd) and after the host-computed x0 (Dh): body rows and swing legs bitwise,
    stance-leg foot positions to 1e-12 (the device contracts the foot kinematics into FMAs)."""
    for i in range(len(Dd)):
        assert Dd[i, :12].tobytes() == Dh[i, :12].tobytes(), (what, i)
        for l in range(4):
            a, b = Dd[i, 12 + 3 * l:15 + 3 * l], Dh[i, 12 + 3 * l:15 + 3 * l]
            if contact[i][l]:
                assert np.abs(a - b).max() <= 1e-12, (what, i, l, a, b)
            else:
                assert a.tobytes() == b.tobytes(), (what, i, l)


@pytest.mark.gpu
def test_measured_state_ingest(pkg, workloads, torch):
    """set_measured_state after ticks across contact changes: x0 is the measured body state and compute_hkd_state of the
    measured joint angles with the contact of the problem's first phase as the device holds it (or the caller's flags), as
    the host computes it; a subset call leaves the other problems' x0 alone."""
    refs = _refs(pkg, workloads)
    B = _batch(pkg, workloads, refs, CASES)
    B.set_initial_condition(_x0(pkg, workloads, CASES))
    B.solve(pkg.Options())
    _tick_until_contact_changes(pkg, workloads, B)
    # the rollout at step 0 carries x0 into the defect of node 0, and depends on nothing else that changes here
    x = B.get_rows("Xbar", 1, 1)[:, 0, :].copy()
    B.set_initial_condition(x)
    D = _defect0(B)
    assert np.abs(D + B.get("X")[:, 0, :] - x).max() <= 1e-12 * max(1.0, np.abs(x).max())
    assert _defect0(B).tobytes() == D.tobytes()
    rng = np.random.default_rng(7)
    n = len(CASES)
    meas = np.concatenate([x[:, :12], np.tile(workloads.DEFAULT_QJ, (n, 1)) + rng.uniform(-0.2, 0.2, (n, 12))], axis=1)
    first = [B.device_schedule(s)["contact"][0] for s in B.schedule_ids()]
    B.set_initial_condition(_host_x0(pkg, meas, first))
    Dh = _defect0(B)
    B.set_measured_state(torch.from_numpy(meas).cuda())
    _assert_ingested(_defect0(B), Dh, first, "first phase")
    # the caller's contact flags (any nonzero value is stance)
    contact = rng.integers(0, 2, (n, 4)).astype(np.int32) * rng.integers(1, 4, (n, 4)).astype(np.int32)
    B.set_initial_condition(_host_x0(pkg, meas, contact))
    Dh = _defect0(B)
    B.set_measured_state(torch.from_numpy(meas).cuda(), contact=torch.from_numpy(contact).cuda())
    _assert_ingested(_defect0(B), Dh, contact, "caller's contact")
    # listed problems only: the others keep the x0 set before
    others = [i for i in range(n) if i not in SUBSET]
    meas2 = meas[SUBSET] + rng.uniform(-0.01, 0.01, (len(SUBSET), 24))
    for c in (None, contact[SUBSET]):
        fc = [first[i] for i in SUBSET] if c is None else c
        xe = x.copy()
        xe[SUBSET] = _host_x0(pkg, meas2, fc)
        B.set_initial_condition(xe)
        Dh = _defect0(B)
        B.set_initial_condition(x)
        Dx = _defect0(B)
        B.set_measured_state(torch.from_numpy(meas2).cuda(), problems=SUBSET, contact=None if c is None else torch.from_numpy(c).cuda())
        Dd = _defect0(B)
        _assert_ingested(Dd[SUBSET], Dh[SUBSET], fc, ("subset", c is None))
        assert Dd[others].tobytes() == Dx[others].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("listed", [False, True], ids=["batch", "subset"])
def test_stream_contract(pkg, workloads, torch, listed):
    """Inputs written on a side stream behind a long sleep are read after it; the command tensor read on that stream right
    after get_mpc_command_dev is complete; and no _dev call waits on the host for the sleeping stream."""
    refs = _refs(pkg, workloads)
    x0 = _x0(pkg, workloads, CASES)
    H, D = _batch(pkg, workloads, refs, CASES), _batch(pkg, workloads, refs, CASES)
    for B in (H, D):
        B.set_initial_condition(x0)
        B.solve(pkg.Options())
    p = SUBSET if listed else None
    n = len(SUBSET) if listed else len(CASES)
    opt = pkg.Options(**TICK)
    side = torch.cuda.Stream()
    # warm-up of the list staging and its device scratch (their first use may allocate)
    with torch.cuda.stream(side):
        D.mpc_command(8, out=_cmd_tensor(torch, pkg, n), problems=p)
    side.synchronize()
    for t in range(1, 3):
        x = H.get_rows("Xbar", 1, 1)[:, 0, :]
        x = x[SUBSET].copy() if listed else x.copy()
        H.mpc_update(problems=p)
        H.set_initial_condition(x, problems=p)
        H.solve(opt, problems=p)
        want = H.mpc_command(8, problems=p)
        src = torch.from_numpy(x).cuda()
        xt = torch.zeros_like(src)
        out = _cmd_tensor(torch, pkg, n)
        torch.cuda.synchronize()
        D.mpc_update(problems=p)
        with torch.cuda.stream(side):
            torch.cuda._sleep(SLEEP_CYCLES)
            xt.copy_(src)                                  # the states exist only after the sleep
            D.set_initial_condition(xt, problems=p)
            assert not side.query(), "set_initial_condition_dev waited on the host"
            D.solve_async(opt, problems=p)
            D.mpc_command(8, out=out, problems=p)
            snap = out.clone()                             # read on the caller's stream right after the call
            xt.zero_()                                     # the input buffer may be reused
        side.synchronize()
        assert snap.cpu().numpy().tobytes() == want.tobytes(), ("commands", t)
        _assert_same_state(_state(H), _state(D), ("tick", t))
    # the command read-out behind a sleep
    out = _cmd_tensor(torch, pkg, n)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        D.mpc_command(8, out=out, problems=p)
        assert not side.query(), "get_mpc_command_dev waited on the host"
        snap = out.clone()
    side.synchronize()
    assert snap.cpu().numpy().tobytes() == H.mpc_command(8, problems=p).tobytes()
    # the measured-state ingest behind a sleep: no host wait either, and it reads the states written after the sleep
    meas = np.concatenate([x[:, :12], np.tile(workloads.DEFAULT_QJ, (n, 1))], axis=1)
    src = torch.from_numpy(meas).cuda()
    mt = torch.zeros_like(src)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        mt.copy_(src)
        D.set_measured_state(mt, problems=p)
        assert not side.query(), "set_measured_state_dev waited on the host"
        mt.zero_()
    side.synchronize()
    Dd = _defect0(D)
    D.set_initial_condition(meas, problems=p)   # (the body rows are what the ingest must have read; the legs do not matter here)
    Dh = _defect0(D)
    rows = SUBSET if listed else list(range(len(CASES)))
    assert Dd[rows, :12].tobytes() == Dh[rows, :12].tobytes()


@pytest.mark.gpu
def test_refused_device_calls_change_nothing(pkg, workloads, torch):
    """Host buffers (pinned or pageable), NULL, misaligned buffers, bad lists, n_steps 0 and 11 and wrong dtypes are refused
    with HSDDP_ERR_ARG before anything is queued: every stored array, info, trace, schedule and x0 stay as they were, and the
    next call works."""
    refs = _refs(pkg, workloads)
    x0 = _x0(pkg, workloads, CASES)
    B, C = _batch(pkg, workloads, refs, CASES), _batch(pkg, workloads, refs, CASES)  # C: a batch that is never asked
    for A in (B, C):
        A.set_initial_condition(x0)
        A.solve(pkg.Options())
    n = len(CASES)
    S0 = _state(B)
    L, ip, vp = pkg.lib(), pkg._ip, pkg.C.c_void_p
    one = np.array([1], np.int32)
    itemsize = pkg.CMD_DTYPE.itemsize
    pinned = torch.zeros((n, itemsize), dtype=torch.uint8).pin_memory()
    pageable = np.zeros((n, itemsize), np.uint8)
    good_x, good_c = torch.zeros((n, 24), dtype=torch.float64, device="cuda:0"), torch.zeros((n, 4), dtype=torch.int32, device="cuda:0")
    good_out = _cmd_tensor(torch, pkg, n)
    raw = torch.zeros(n * itemsize + 8, dtype=torch.uint8, device="cuda:0")
    for ptr in (pinned.data_ptr(), pageable.ctypes.data, None, raw.data_ptr() + 1):
        assert L.hsddp_batch_set_initial_condition_dev(B.h, n, None, ptr, None) == pkg.ERR_ARG
        assert L.hsddp_batch_set_initial_condition_dev(B.h, 1, ip(one), ptr, None) == pkg.ERR_ARG
        assert L.hsddp_batch_set_measured_state_dev(B.h, n, None, ptr, None, None) == pkg.ERR_ARG
        if ptr is not None:  # (NULL contact flags are valid: the first phase's)
            assert L.hsddp_batch_set_measured_state_dev(B.h, n, None, good_x.data_ptr(), ptr, None) == pkg.ERR_ARG
        assert L.hsddp_batch_get_mpc_command_dev(B.h, 8, n, None, ptr, None) == pkg.ERR_ARG
    # without a list n must be n_problems
    assert L.hsddp_batch_set_initial_condition_dev(B.h, n - 1, None, good_x.data_ptr(), None) == pkg.ERR_ARG
    for bad in ([1, 1], [n], [-1]):
        m = len(bad)
        for call in (lambda: B.set_initial_condition(good_x[:m].contiguous(), problems=bad),
                     lambda: B.set_measured_state(good_x[:m].contiguous(), problems=bad),
                     lambda: B.set_measured_state(good_x[:m].contiguous(), problems=bad, contact=good_c[:m].contiguous()),
                     lambda: B.mpc_command(8, out=good_out[:m].contiguous(), problems=bad)):
            with pytest.raises(pkg.HsddpError) as e:
                call()
            assert e.value.code == pkg.ERR_ARG, (bad, e.value)
    for steps in (0, 11):
        with pytest.raises(pkg.HsddpError) as e:
            B.mpc_command(steps, out=good_out)
        assert e.value.code == pkg.ERR_ARG
    for call in (lambda: B.set_initial_condition(good_x.float()), lambda: B.set_measured_state(good_x.float()),
                 lambda: B.set_measured_state(good_x, contact=good_c.long()), lambda: B.mpc_command(8, out=good_out.view(torch.int32)),
                 lambda: B.set_initial_condition(good_x[:, :12]), lambda: B.set_measured_state(good_x.t().contiguous().t()),
                 lambda: B.set_measured_state(good_x.cpu())):
        with pytest.raises(pkg.HsddpError) as e:
            call()
        assert e.value.code == pkg.ERR_ARG
    assert (good_out == 0xAB).all()
    _assert_same_state(S0, _state(B), "refusals")
    for A in (B, C):  # x0 untouched: the next solve from it is the never-asked batch's, bit for bit
        A.solve(pkg.Options(**TICK))
    _assert_same_state(_state(B), _state(C), "solve after the refusals")
    # a handle without problems
    E = pkg.MultiPhaseDDPBatch(0)
    assert L.hsddp_batch_set_initial_condition_dev(E.h, 1, None, good_x.data_ptr(), None) == pkg.ERR_ARG
    assert L.hsddp_batch_get_mpc_command_dev(E.h, 8, 1, None, good_out.data_ptr(), None) == pkg.ERR_ARG
    # the next call works
    B.mpc_command(8, out=good_out)
    torch.cuda.synchronize()
    assert good_out.cpu().numpy().tobytes() == B.mpc_command(8).tobytes()


@pytest.mark.gpu
def test_wrong_device_is_refused(pkg, workloads, torch):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    refs = _refs(pkg, workloads)
    B = _batch(pkg, workloads, refs, CASES)
    B.set_initial_condition(_x0(pkg, workloads, CASES))
    S0 = _state(B)
    n = len(CASES)
    other = torch.zeros((n, 24), dtype=torch.float64, device="cuda:1")
    with pytest.raises(pkg.HsddpError) as e:
        B.set_initial_condition(other)
    assert e.value.code == pkg.ERR_ARG
    L = pkg.lib()
    assert L.hsddp_batch_set_initial_condition_dev(B.h, n, None, other.data_ptr(), None) == pkg.ERR_ARG
    assert L.hsddp_batch_set_measured_state_dev(B.h, n, None, other.data_ptr(), None, None) == pkg.ERR_ARG
    out = torch.zeros((n, pkg.CMD_DTYPE.itemsize), dtype=torch.uint8, device="cuda:1")
    assert L.hsddp_batch_get_mpc_command_dev(B.h, 8, n, None, out.data_ptr(), None) == pkg.ERR_ARG
    _assert_same_state(S0, _state(B), "wrong device")


def test_package_imports_and_takes_numpy_without_torch():
    """The NumPy paths never import torch: importing the package and telling a NumPy array from a tensor leave it unloaded."""
    code = ("import importlib, sys, numpy as np; pkg = importlib.import_module('hkd-mpc_b200'); "
            "assert pkg._torch_tensor(np.zeros(3)) is None and pkg._torch_tensor([1.0]) is None; "
            "assert 'torch' not in sys.modules")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT))
