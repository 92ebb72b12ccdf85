"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle.

Tolerance (BASELINE.json north_star): 1e-9 relative on per-iteration cost, gains and
state/control trajectories; identical accepted-step sequence, iteration count and
termination status.  "Relative" is max-norm over the compared array.
"""
import os
import numpy as np
import pytest
from conftest import GOLDEN, GAIT_PATH, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-9


def rel_err_rows(a, b, floor=1e-6):
    """max over rows of (max-norm error of the row) / max(max-norm of the row, floor * max-norm of the array): a whole-array
    max-norm would say nothing about the small rows of K (gains of weakly coupled controls)."""
    import parity_check as pc
    return float(pc.rel_err_rows(np.asarray(a)[None], np.asarray(b)[None], floor)[0])


def _scale_check(pkg, orc, w, B, idx, k_rows=8, opts=None, gpu_opt=None):
    """Parity of many problems at once (oracle/parity_check.py): classify with the oracle's arithmetic variants, compare the
    CUDA results of the well-posed ones.  Returns (report, well_posed mask, per-problem match mask)."""
    import parity_check as pc
    tables = {}
    tabs, k0 = [], []
    for i in idx:
        gait, k = w.keys[w.schedule_id[i]]
        if gait not in tables:
            tables[gait] = _table(orc, gait)
        tabs.append(tables[gait]); k0.append(k)
    idx = np.asarray(list(idx))
    base, others = pc.oracle_runs(orc, tabs, k0, w.x0[idx], B.max_nodes, B.max_stages, w.plan, k_rows=k_rows, opts=opts)
    well, sens = pc.classify(base, others)
    K = B.get_rows("K", 0, k_rows)[idx].reshape(len(idx), k_rows, 24, 24)
    gpu = dict(info=B.info()[idx], Xbar=B.get_rows("Xbar", 0, B.max_nodes)[idx], Ubar=B.get_rows("Ubar", 0, B.max_stages)[idx],
               K=np.ascontiguousarray(np.swapaxes(K, -1, -2)))
    rep, detail = pc.compare_gpu(base, well, gpu)
    return rep, well, detail


def _table(orc, gait):
    return orc.GaitTable(GAIT_PATH(gait))


def _batch_for(pkg, w):
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems(w.schedules, w.schedule_id)
    B.set_initial_condition(w.x0)
    return B


def _oracle_problem(orc, w, i, tables):
    gait, k0 = w.keys[w.schedule_id[i]]
    if gait not in tables:
        tables[gait] = _table(orc, gait)
    P = orc.Problem(tables[gait], k0, w.plan)
    P.x0 = w.x0[i]
    return P


def _g_by_leg(P):
    """oracle GRF constraint values are packed by stance leg; the GPU layout is 5 per leg."""
    g = P.get("g")
    out = np.zeros_like(g)
    s = 0
    for ph in P.phases:
        legs = [l for l in range(4) if ph["contact"][l]]
        for k in range(ph["horizon"]):
            for j, l in enumerate(legs):
                out[s, 5 * l:5 * l + 5] = g[s, 5 * j:5 * j + 5]
            s += 1
    return out


def _oracle_pair(orc, w, i, tables):
    """Solve problem i with the oracle twice: on the reference's compiled CasADi model and on the
    independent model port.  The two differ by ~1e-16 per model call, so their disagreement after a
    whole solve measures how strongly THIS problem amplifies rounding noise.  A problem is
    well-posed for parity when both give the same step sequence and agree to 1e-11; the
    non-converging long-flight problems of config 4 are not (SURVEY.md §7.2: report such
    problems as ill-posed for parity rather than failures).  Without the compiled reference model
    the oracle runs on the port, and the FMA-contracted build of the same restatement is the
    second arithmetic (oracle/parity_check.py)."""
    P = _oracle_problem(orc, w, i, tables)
    s, otr = P.solve()
    gait, k0 = w.keys[w.schedule_id[i]]
    if not orc.ref_available():
        import parity_check as pc
        base, others = pc.oracle_runs(orc, [tables[gait]], [k0], w.x0[i:i + 1], P.n_states, P.n_stages, w.plan,
                                      k_rows=P.n_stages, variants=("fma",))
        assert others, "no second arithmetic variant of the oracle to classify problems with"
        well, sens = pc.classify(base, others)
        return P, s, otr, bool(well[0]), float(sens[0])
    Q = orc.Problem(tables[gait], k0, w.plan, model=orc.MODEL_PORT)
    Q.x0 = w.x0[i]
    s2, otr2 = Q.solve()
    same = (s["n_iter"] == s2["n_iter"] and s["status"] == s2["status"] and np.array_equal(otr[:, 9], otr2[:, 9])
            and np.array_equal(otr[:, 10], otr2[:, 10]) and np.array_equal(otr[:, 4], otr2[:, 4]))
    if not same:
        return P, s, otr, False, np.inf
    sens = max(rel_err(otr2[:, 11], otr[:, 11]), rel_err(Q.get("Xbar"), P.get("Xbar")), rel_err(Q.get("Ubar"), P.get("Ubar")),
               rel_err(Q.get("K"), P.get("K")), rel_err(Q.get("dU"), P.get("dU")))
    return P, s, otr, sens < 1e-11, sens


def _compare_solution(pkg, orc, w, B, idx, tables, max_ill_posed=0):
    info, tr = B.info(), B.trace()
    Xb, Ub, K, dU = B.get("Xbar"), B.get("Ubar"), B.get("K"), B.get("dU")
    ill = []
    for i in idx:
        P, s, otr, well_posed, sens = _oracle_pair(orc, w, i, tables)
        n = int(s["n_iter"])
        S, N = P.n_states, P.n_stages
        assert info["status"][i] in (0, 1, 2, 3) and np.isfinite(Xb[i]).all() and np.isfinite(K[i]).all()
        assert not np.any(Xb[i, S:]) and not np.any(K[i, N:])  # padding rows stay zero
        if not well_posed:
            ill.append((int(i), sens))
            continue
        assert info["n_iter"][i] == n and info["status"][i] == int(s["status"]) and info["n_outer"][i] == int(s["n_outer"]), (i, s, info[i])
        assert info["n_sweeps"][i] == int(s["n_sweeps"])
        assert np.array_equal(tr[i, :n, 9], otr[:, 9]), (i, "accepted step sizes differ")
        assert np.array_equal(tr[i, :n, 10], otr[:, 10]), (i, "line-search trial counts differ")
        assert np.array_equal(tr[i, :n, 4], otr[:, 4]), (i, "regularisation schedule differs")
        for col in (2, 3, 11, 12, 6, 7):  # cost/feas before and after, dV_1, dV_2
            assert rel_err(tr[i, :n, col], otr[:, col]) < RTOL, (i, col)
        assert rel_err(Xb[i, :S], P.get("Xbar")) < RTOL and rel_err(Ub[i, :N], P.get("Ubar")) < RTOL, i
        assert rel_err(K[i, :N], P.get("K")) < RTOL and rel_err(dU[i, :N], P.get("dU")) < RTOL, i
        # per-stage relative error of the gains and of the trajectories (rows = stages / nodes)
        assert rel_err_rows(K[i, :N], P.get("K")) < RTOL and rel_err_rows(Xb[i, :S], P.get("Xbar")) < RTOL, i
        assert rel_err_rows(Ub[i, :N], P.get("Ubar")) < RTOL, i
        assert abs(info["cost"][i] - s["cost"]) <= RTOL * abs(s["cost"])
    assert len(ill) <= max_ill_posed, f"ill-posed-for-parity problems: {ill}"
    return ill


def test_device_peaks_probe(pkg):
    assert pkg.fp64_peak_tflops(0, 0) > 5.0 and pkg.fp64_peak_tflops(0, 1) > 5.0


def test_step_level_parity(pkg, orc, workloads):
    """hybrid_rollout / compute_cost / LQ_approximation / backward_sweep / linear_rollout one by one."""
    w = workloads.config1(pkg)
    B = _batch_for(pkg, w)
    P = _oracle_problem(orc, w, 0, {})
    N, S = P.n_stages, P.n_states
    assert P.hybrid_rollout(0.0) and B.hybrid_rollout(0.0)[0]
    assert np.array_equal(B.get("X")[0, :S], P.get("X"))
    P.update_nominal(); B.update_nominal()
    for it, eps in enumerate((1.0, 0.1, 0.1)):
        P.compute_cost(); B.compute_cost()
        so, sg = P.scalars(), B.scalars()[0]
        assert abs(so["actual_cost"] - sg[0]) < RTOL * abs(so["actual_cost"]) and abs(so["feas"] - sg[2]) <= RTOL * so["feas"]
        P.lq_approximation(); B.lq_approximation()
        for nm in ("A", "B", "lx", "lu", "lxx", "luu"):
            assert rel_err(B.get(nm)[0, :N], P.get(nm)) < 1e-13, nm
        assert P.backward_sweep(0.0) and B.backward_sweep(0.0)[0]
        assert rel_err(B.get("K")[0, :N], P.get("K")) < RTOL and rel_err(B.get("dU")[0, :N], P.get("dU")) < RTOL
        assert rel_err(B.get("G0")[0], P.get("G")[0]) < RTOL and rel_err(B.get("H0")[0], P.get("H")[0]) < RTOL
        so, sg = P.scalars(), B.scalars()[0]
        assert abs(so["dV_1"] - sg[3]) < RTOL * abs(so["dV_1"]) and abs(so["dV_2"] - sg[4]) < RTOL * abs(so["dV_2"])
        P.linear_rollout(1.0); B.linear_rollout(1.0)
        so, sg = P.scalars(), B.scalars()[0]
        assert rel_err(B.get("dX")[0, :S], P.get("dX")) < RTOL
        assert abs(so["dV_1"] - sg[3]) < RTOL * abs(so["dV_1"]) and abs(so["dV_2"] - sg[4]) < RTOL * abs(so["dV_2"])
        assert P.hybrid_rollout(eps) and B.hybrid_rollout(eps)[0]
        for nm in ("X", "Defect"):
            assert rel_err(B.get(nm)[0, :S], P.get(nm)) < RTOL, nm
        assert rel_err(B.get("U")[0, :N], P.get("U")) < RTOL
        assert rel_err(B.get("g")[0, :N], _g_by_leg(P)) < RTOL
        so, sg = P.scalars(), B.scalars()[0]
        assert abs(so["max_tconstr"] - sg[5]) <= RTOL and abs(so["max_pconstr"] - sg[6]) <= RTOL
        P.update_nominal(); B.update_nominal()


def test_config1_single_solve_and_golden_record(pkg, orc, workloads):
    w = workloads.config1(pkg)
    B = _batch_for(pkg, w)
    B.solve()
    _compare_solution(pkg, orc, w, B, [0], {})
    g = np.load(os.path.join(GOLDEN, "oracle_solves.npz"))
    info, tr = B.info(), B.trace()
    gs = g["trot_0.6/summary"]
    assert info["n_iter"][0] == gs[1] == 13 and info["status"][0] == gs[0]
    assert rel_err(B.get("Xbar")[0, :65], g["trot_0.6/Xbar"]) < RTOL and rel_err(B.get("Ubar")[0, :60], g["trot_0.6/Ubar"]) < RTOL
    assert rel_err(B.get("K")[0, :8], g["trot_0.6/K_first8"]) < RTOL
    assert rel_err(tr[0, :13, 11], g["trot_0.6/trace"][:, 11]) < RTOL


@pytest.mark.parametrize("plan", [0.25, 0.5, 1.0])
def test_horizon_sweep(pkg, orc, workloads, plan):
    w = workloads.config1(pkg, plan)
    B = _batch_for(pkg, w)
    B.solve()
    _compare_solution(pkg, orc, w, B, [0], {})


def test_config2_perturbed_trot_batch(pkg, orc, workloads):
    w = workloads.config2(pkg, 24)
    B = _batch_for(pkg, w)
    B.solve()
    _compare_solution(pkg, orc, w, B, range(w.n), {})


def test_config3_mixed_gaits_ragged_schedules(pkg, orc, workloads):
    w = workloads.config3(pkg, 30)
    assert len({s.n_stages for s in w.schedules}) >= 1 and len({s.n_phases for s in w.schedules}) > 1
    B = _batch_for(pkg, w)
    B.solve()
    ill = _compare_solution(pkg, orc, w, B, range(w.n), {}, max_ill_posed=3)
    print("config3 ill-posed-for-parity:", ill)


def test_solve_modes_agree_and_unknown_modes_are_refused(pkg, orc, workloads):
    """The kernel-per-phase driver (solve mode 2), the persistent kernel (mode 1, throughput build: the batch is
    larger than 2 x 148) and the latency build of the persistent kernel (batch of 3) run the same device
    functions.  They are separate compilations (the compiler contracts and schedules FMAs differently), so their
    results agree to rounding, not bitwise: each mode meets the oracle bar, and the modes agree with each other
    to 1e-9 on every problem whose iteration count coincides (all but the rounding-chaotic ones)."""
    w = workloads.config3(pkg, 330)
    out = {}
    for mode in (1, 2):
        B = _batch_for(pkg, w)
        B.set_solve_mode(mode)
        B.solve()
        out[mode] = (B.info().copy(), B.get("Xbar").copy(), B.get("Ubar").copy(), B.get("K").copy())
        _compare_solution(pkg, orc, w, B, range(0, 12), {}, max_ill_posed=2)
    i1, i2 = out[1][0], out[2][0]
    same = (i1["n_iter"] == i2["n_iter"]) & (i1["status"] == i2["status"])
    assert same.mean() > 0.95, same.mean()
    for a, b in zip(out[1][1:], out[2][1:]):
        for i in np.nonzero(same)[0]:
            assert rel_err(a[i], b[i]) < RTOL, i
    w3 = workloads.config3(pkg, 3)
    B3 = _batch_for(pkg, w3)
    B3.solve()
    _compare_solution(pkg, orc, w3, B3, range(3), {}, max_ill_posed=1)
    for mode in (-1, 3):  # the modes are 0 auto, 1 persistent, 2 phased
        with pytest.raises(pkg.HsddpError):
            B3.set_solve_mode(mode)


def test_linear_rollout_kernel_of_the_phased_driver_matches_the_block_version(pkg, orc, workloads, monkeypatch):
    """The phased driver runs the linear rollout as its own one-warp-per-problem kernel (k_lr_w1); HSDDP_LR_W1=0 leaves it
    inside the forward kernel (linear_rollout_block).  Same recursion, dV_1 / dV_2 summed in a different order: after ONE
    DDP iteration the expected cost change, the search direction and the accepted trajectories agree to rounding, and
    whole solves take the same decisions."""
    w = workloads.config3(pkg, 96)
    res = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("HSDDP_LR_W1", flag)
        B = _batch_for(pkg, w)
        B.set_solve_mode(2)
        B.solve(pkg.Options(max_AL_iter=1, max_DDP_iter=1))
        one = (B.trace()[:, 0, :].copy(), B.get("dX").copy(), B.get("Xbar").copy())
        B.reset()
        B.solve()
        res[flag] = one + (B.info().copy(), B.get("Xbar").copy())
    monkeypatch.delenv("HSDDP_LR_W1")
    (t1, dx1, x1, i1, xf1), (t0, dx0, x0, i0, xf0) = res["1"], res["0"]
    cols = [pkg.TRACE_COLS.index(c) for c in ("dV_1", "dV_2", "eps_accepted", "n_trials", "cost_after")]
    assert np.array_equal(t1[:, cols[2:4]], t0[:, cols[2:4]])  # accepted step and trial count of the first iteration
    for c in (cols[0], cols[1], cols[4]):
        assert np.allclose(t1[:, c], t0[:, c], rtol=1e-9, atol=1e-9 * np.abs(t0[:, c]).max()), pkg.TRACE_COLS[c]
    assert np.array_equal(dx1, dx0)  # the recursion itself is bit-identical
    assert rel_err(x1, x0) < 1e-12
    same = (i1["n_iter"] == i0["n_iter"]) & (i1["status"] == i0["status"])
    assert same.mean() > 0.95, same.mean()
    for i in np.nonzero(same)[0]:
        assert rel_err(xf1[i], xf0[i]) < RTOL, i
    _compare_solution(pkg, orc, w, B, range(0, 6), {}, max_ill_posed=1)


def test_mpc_command_extraction(pkg, orc, workloads):
    """What leaves the GPU after a solve (hkd_command_lcmt payload, HKDMPC.cpp:207-298): packed on the device,
    compared with the restated publish_mpc_cmd / update_foot_placement applied to the oracle's trajectories."""
    w = workloads.config3(pkg, 9)
    B = _batch_for(pkg, w)
    B.solve()
    cmd = B.mpc_command(8)
    tables = {}
    checked = 0
    for i in range(w.n):
        P, s, otr, well_posed, sens = _oracle_pair(orc, w, i, tables)
        if not well_posed:
            continue
        ref = orc.mpc_command(P, 8)
        assert cmd["N_mpcsteps"][i] == 8
        assert np.array_equal(cmd["contacts"][i, :8], ref["contacts"]) and np.array_equal(cmd["foot_found"][i], ref["foot_found"])
        for name in ("hkd_controls", "des_body_state", "feedback"):
            a, b = cmd[name][i, :8].astype(np.float64), ref[name].astype(np.float64)
            assert np.abs(a - b).max() <= 2e-7 * max(1.0, np.abs(b).max()), (i, name)   # float32 payload
            assert not np.any(cmd[name][i, 8:])
        assert np.abs(cmd["foot_placement"][i] - ref["foot_placement"]).max() <= 2e-7
        checked += 1
    assert checked >= 6


def test_device_schedule_builder_bit_exact(pkg, orc, workloads):
    """Reference ingestion on the device (N2): schedules built by the kernel from the HBM-resident gait library are
    bit-identical to the host builder's (phase tables and every reference row), for all three gaits, several windows
    and horizons; and a solve on them gives bit-identical results to a solve on host-built schedules."""
    refs = {g: pkg.QuadReference(workloads.gait_path(g)) for g in workloads.GAITS}
    order = list(workloads.GAITS)
    for plan in (0.25, 0.5, 0.6, 1.0):
        sg, sw, host = [], [], []
        for gi, g in enumerate(order):
            for k0 in (0, 1, 7, 50, 101, 233, 250, refs[g].n - int(round(plan / 0.01)) - 3):
                sg.append(gi); sw.append(k0); host.append(pkg.Schedule(refs[g], k0, plan))
        B = pkg.MultiPhaseDDPBatch(0)
        B.set_problems_from_gaits([refs[g] for g in order], sg, sw, plan, np.arange(len(sg)))
        for i, S in enumerate(host):
            d = B.device_schedule(i)
            assert d["n_phases"] == S.n_phases and d["horizon"] == S.horizon, (plan, i)
            assert d["contact"] == S.contact and d["next_contact"] == S.next_contact, (plan, i)
            for name in ("xr", "ur", "prel_r", "xinit"):
                assert d[name].tobytes() == S.array(name).tobytes(), (plan, i, name)
    # same solve either way
    w = workloads.config3(pkg, 24)
    Bh = _batch_for(pkg, w)
    Bh.solve()
    Bd = pkg.MultiPhaseDDPBatch(0)
    Bd.set_problems_from_gaits([refs[g] for g in order], [order.index(g) for g, _ in w.keys], [k for _, k in w.keys], w.plan, w.schedule_id)
    Bd.set_initial_condition(w.x0)
    Bd.solve()
    assert Bd.info().tobytes() == Bh.info().tobytes()
    S = min(Bd.get("Xbar").shape[1], Bh.get("Xbar").shape[1])
    assert np.array_equal(Bd.get("Xbar")[:, :S], Bh.get("Xbar")[:, :S]) and np.array_equal(Bd.get("K"), Bh.get("K"))


def test_config4_long_flight_phase(pkg, orc, workloads):
    w = workloads.config4(pkg, 12)
    assert any(max(s.horizon) >= 30 for s in w.schedules)
    B = _batch_for(pkg, w)
    B.solve()
    # the non-converging long-flight windows amplify rounding noise chaotically (the oracle's own two
    # model back ends disagree on them); they are reported, the rest must meet the 1e-9 bar
    # the non-converging long-flight windows amplify rounding noise chaotically; measured rate of ill-posed problems in
    # this configuration: 35 % (33 of 93 over all 31 windows, test_parity_at_scale_config4_all_schedules), none of them converged
    ill = _compare_solution(pkg, orc, w, B, range(w.n), {}, max_ill_posed=5)
    assert all(B.info()["status"][i] >= 2 for i, _ in ill), ill


def test_parity_at_scale_config3(pkg, orc, workloads):
    """The bench workload at a size the oracle finishes in seconds: the first 768 config-3 problems (256 windows of each gait),
    all compared.  Measured on the oracle alone: 762 of 768 are well-posed (0.8 % ill-posed, every one of them a problem that
    does not converge).  Every well-posed problem must take the oracle's decisions and agree to 1e-9."""
    n = 768
    w = workloads.config3(pkg, n)
    B = _batch_for(pkg, w)
    B.solve()
    rep, well, det = _scale_check(pkg, orc, w, B, range(n))
    print("parity config3:", rep)
    assert rep["checked"] == n and rep["ill_posed"] <= 0.02 * n, rep
    bad = np.nonzero(well & ~det["match"])[0]
    assert len(bad) == 0, (rep, bad[:10], det["err"][bad[:10]])
    assert rep["within_1e-9"] == rep["well_posed"] == rep["iter_status_match"]
    # ill-posed problems are exactly of the kind SURVEY.md §7.2 describes: none of them converges
    assert np.all(B.info()["status"][:n][~well] >= 2)
    # the same problems inside the phased multi-stream driver (what `auto` selects for the 16,384-problem benchmark)
    B2 = _batch_for(pkg, w)
    B2.set_solve_mode(2)
    B2.solve()
    rep2, well2, det2 = _scale_check(pkg, orc, w, B2, range(n))
    bad2 = np.nonzero(well2 & ~det2["match"])[0]
    assert len(bad2) == 0, (rep2, bad2[:10])


def test_parity_at_scale_config4_all_schedules(pkg, orc, workloads):
    """All 31 distinct reference windows of config 4 (window starts 236..266: the 30-step flight phase moves through the
    horizon), three perturbed initial states each.  Measured on the oracle alone: 60 of 93 well-posed; the ill-posed ones all
    fail to converge (max iterations or regularisation overflow)."""
    w = workloads.config4(pkg, 4096)
    seen, idx = {}, []
    for i, sid in enumerate(w.schedule_id):
        if seen.get(int(sid), 0) < 3:
            seen[int(sid)] = seen.get(int(sid), 0) + 1
            idx.append(i)
    assert len(seen) == 31 and len(idx) == 93
    B = _batch_for(pkg, w)
    B.solve()
    rep, well, det = _scale_check(pkg, orc, w, B, idx)
    print("parity config4:", rep)
    assert rep["ill_posed"] <= 0.45 * len(idx), rep
    bad = np.nonzero(well & ~det["match"])[0]
    assert len(bad) == 0, (rep, [idx[b] for b in bad[:10]], det["err"][bad[:10]])
    assert np.all(B.info()["status"][np.asarray(idx)][~well] >= 2)
    # every problem that converges is well-posed and compared
    conv = B.info()["status"][np.asarray(idx)] <= 1
    assert np.all(well[conv]) and conv.sum() >= 30


@pytest.mark.parametrize("mode", [0, 2], ids=["auto", "phased"])
def test_receding_horizon_ticks_match_oracle(pkg, orc, workloads, mode):
    """N1: HKDProblem::update on the device + warm re-solve with the reference's MPC budget (2 AL x 1 DDP, HKDMPC.cpp:97-166),
    30 consecutive ticks of nine problems (three gaits, several windows, two problems sharing a schedule), against the oracle's
    restated update.  The windows are chosen so that the ticks exercise: a first phase shrinking to a point and being removed, a
    last phase growing, a phase reaching its end (second touchdown-constraint object: trot window 0 at tick 0), a new last
    phase with an empty shooting set (horizon 1 and 2), and the shooting set being restored at horizon 3.  `phased`: the same
    ticks through the kernel-per-phase driver (one-warp linear-rollout kernel on the updated schedules)."""
    order = list(workloads.GAITS)
    refs = {g: pkg.QuadReference(workloads.gait_path(g)) for g in order}
    cases = [("trot", 0), ("trot", 0), ("trot", 23), ("bound", 0), ("bound", 5), ("bound", 240), ("pronk", 0), ("pronk", 100), ("pronk", 40)]
    keys, sid = [], []
    for c in cases:
        if c not in keys:
            keys.append(c)
        sid.append(keys.index(c))
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems_from_gaits([refs[g] for g in order], [order.index(g) for g, _ in keys], [k for _, k in keys], 0.6, sid)
    B.set_solve_mode(mode)
    tables = {g: _table(orc, g) for g in order}
    models = [orc.default_model()] + ([orc.MODEL_PORT] if orc.ref_available() else [])
    P = [[orc.Problem(tables[g], k0, 0.6, model=m) for m in models] for g, k0 in cases]
    x0 = np.zeros((len(cases), 24))
    for i, (g, k0) in enumerate(cases):
        body = np.load(workloads.gait_path(g))["body_state"][k0].astype(np.float64)
        if i == 1:
            body = body + workloads.perturbation(1)
        x0[i, :12] = body
        x0[i, 12:] = pkg.compute_hkd_state(body[0:3], body[3:6], workloads.DEFAULT_QJ, P[i][0].phases[0]["contact"])
    tick_opt = dict(max_AL_iter=2, max_DDP_iter=1)
    alive = np.ones(len(cases), bool)  # problems still well-posed (the oracle's two model back ends take the same decisions)
    seen = dict(pop_phase=False, new_phase=False, two_objects=False, empty_ss=False)
    for tick in range(-1, 30):
        if tick >= 0:
            x0 = np.stack([P[i][0].get("Xbar")[1] for i in range(len(cases))])  # "measured" state: the plan's next node
            B.mpc_update()
        B.set_initial_condition(x0)
        B.solve(pkg.Options(**tick_opt) if tick >= 0 else None)
        info, Xb, Ub, K = B.info(), B.get("Xbar"), B.get("Ubar"), B.get("K")
        for i in range(len(cases)):
            res = []
            for Q in P[i]:
                if tick >= 0:
                    seen["pop_phase"] |= Q.phases[0]["horizon"] == 1  # (a first phase of one stage shrinks to a point: removed)
                    Q.mpc_update()
                Q.x0 = x0[i]
                res.append(Q.solve(tick_opt if tick >= 0 else None)[0])
            Q = P[i][0]
            seen["new_phase"] |= tick >= 0 and Q.phases[-1]["horizon"] == 1
            seen["two_objects"] |= any(p["n_td_objects"] > 1 for p in Q.phases)
            seen["empty_ss"] |= Q.phases[-1]["ss_size"] == 0
            if len(res) > 1 and not (res[0]["n_iter"] == res[1]["n_iter"] and res[0]["status"] == res[1]["status"]
                                     and abs(res[0]["cost"] - res[1]["cost"]) <= 1e-10 * abs(res[0]["cost"])):
                alive[i] = False
            if not alive[i]:
                continue
            s = res[0]
            d = B.device_schedule(sid[i])
            assert d["n_phases"] == Q.n_phases and d["horizon"] == [p["horizon"] for p in Q.phases], (tick, i, d["horizon"], Q.phases)
            assert d["contact"] == [p["contact"] for p in Q.phases], (tick, i)
            assert info["n_iter"][i] == int(s["n_iter"]) and info["status"][i] == int(s["status"]), (tick, i, s, info[i])
            assert abs(info["cost"][i] - s["cost"]) <= RTOL * abs(s["cost"]), (tick, i, info["cost"][i], s["cost"])
            S, N = Q.n_states, Q.n_stages
            assert N == 60
            assert rel_err_rows(Xb[i, :S], Q.get("Xbar")) < RTOL and rel_err_rows(Ub[i, :N], Q.get("Ubar")) < RTOL, (tick, i)
            assert rel_err_rows(K[i, :N], Q.get("K")) < RTOL, (tick, i)
    assert alive.sum() >= 7, alive
    assert all(seen.values()), seen


def test_reb_update_rule_off_the_noop(pkg, orc, workloads):
    """update_REB_params with update_relax, update_ReB != 1 (the shipped settings make it a no-op, ConstraintsBase.h:168-183):
    a weak barrier (small eps) lets the GRF constraints be violated, so the rule fires: eps *= update_ReB and
    delta = max(delta * update_relax, delta_min) on the violated rows only."""
    w = workloads.config3(pkg, 18)
    cp = dict(grf_eps=1e-6, grf_delta=0.5, grf_delta_min=0.01)
    o = dict(update_relax=0.5, update_ReB=3.0, max_AL_iter=4, max_DDP_iter=4)
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems(w.schedules, w.schedule_id, pkg.ConstraintParams(**cp))
    B.set_initial_condition(w.x0)
    B.solve(pkg.Options(**o))
    info, tr = B.info(), B.trace()
    tables = {}
    fired = 0
    for i in range(w.n):
        gait, k0 = w.keys[w.schedule_id[i]]
        if gait not in tables:
            tables[gait] = _table(orc, gait)
        P = orc.Problem(tables[gait], k0, w.plan, cparams=cp)
        P.x0 = w.x0[i]
        s, otr = P.solve(o)
        n = int(s["n_iter"])
        reb = P.get("reb")  # [stages, 20, 2] (eps, delta), by leg like the GPU layout
        fired += int(np.any(reb[..., 0] != cp["grf_eps"]))
        assert info["n_iter"][i] == n and info["status"][i] == int(s["status"]) and info["n_outer"][i] == int(s["n_outer"]), (i, s, info[i])
        assert np.array_equal(tr[i, :n, 9], otr[:, 9])
        assert rel_err(tr[i, :n, 11], otr[:, 11]) < RTOL
        assert rel_err(B.get("Xbar")[i, :P.n_states], P.get("Xbar")) < RTOL
        assert np.array_equal(B.get("reb")[i, :P.n_stages], reb), i
    assert fired >= 3, "the case did not exercise the ReB update"


def test_warm_start_resolve_matches_oracle(pkg, orc, workloads):
    """MPC-style re-solve (2 AL x 1 DDP, HKDMPC.cpp:102-103) continuing from the previous solution."""
    w = workloads.config2(pkg, 4)
    B = _batch_for(pkg, w)
    B.solve()
    opt = pkg.Options(max_AL_iter=2, max_DDP_iter=1)
    B.solve(opt)
    info, tr = B.info(), B.trace()
    tables = {}
    for i in range(w.n):
        P = _oracle_problem(orc, w, i, tables)
        P.solve()
        s, otr = P.solve(dict(max_AL_iter=2, max_DDP_iter=1))
        n = int(s["n_iter"])
        assert info["n_iter"][i] == n and info["status"][i] == int(s["status"])
        assert np.array_equal(tr[i, :n, 9], otr[:, 9])
        assert rel_err(B.get("Xbar")[i, :P.n_states], P.get("Xbar")) < RTOL
        assert rel_err(B.get("K")[i, :P.n_stages], P.get("K")) < RTOL


@pytest.mark.parametrize("grf_eps,expect_overflow", [(-5.0, False), (-40.0, True)])
def test_regularisation_retry_path(pkg, orc, workloads, grf_eps, expect_overflow):
    """A negative barrier weight makes Quu indefinite: the PD test must fail on the same stages and the
    regularisation schedule 1e-3, 2e-3, ... (MultiPhaseDDP.cpp:141-181) must match the oracle's."""
    w = workloads.config2(pkg, 3)
    cp = dict(grf_eps=grf_eps)
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems(w.schedules, w.schedule_id, pkg.ConstraintParams(**cp))
    B.set_initial_condition(w.x0)
    opt = pkg.Options(max_AL_iter=1, max_DDP_iter=3)
    B.solve(opt)
    info, tr = B.info(), B.trace()
    T = _table(orc, "trot")
    saw_retry = False
    for i in range(w.n):
        P = orc.Problem(T, 0, w.plan, cparams=cp)
        P.x0 = w.x0[i]
        s, otr = P.solve(dict(max_AL_iter=1, max_DDP_iter=3))
        n = int(s["n_iter"])
        saw_retry = saw_retry or s["n_sweeps"] > n
        assert info["n_iter"][i] == n and info["status"][i] == int(s["status"]) and info["n_sweeps"][i] == int(s["n_sweeps"])
        assert np.array_equal(tr[i, :n, 5], otr[:, 5]) and np.array_equal(tr[i, :n, 4], otr[:, 4])
        assert np.array_equal(tr[i, :n, 9], otr[:, 9])
        assert (int(s["status"]) == 3) == expect_overflow
        if not expect_overflow:
            assert rel_err(B.get("Xbar")[i, :P.n_states], P.get("Xbar")) < RTOL
    assert saw_retry, "the case did not exercise the retry loop"


def test_rollout_divergence_partial_update(pkg, orc, workloads):
    """||Xsim|| > 1e6 at one stage: the reference stops mid-phase and leaves later stages stale (Q16)."""
    w = workloads.config1(pkg)
    B = _batch_for(pkg, w)
    P = _oracle_problem(orc, w, 0, {})
    assert P.hybrid_rollout(0.0) and B.hybrid_rollout(0.0)[0]
    P.update_nominal(); B.update_nominal()
    Ub = P.get("Ubar").copy()
    Ub[25, 2] = 1e12  # a huge vertical force in the second phase
    P.set("Ubar", Ub)
    Ug = B.get("Ubar"); Ug[0, 25, 2] = 1e12; B.set("Ubar", Ug)
    okc, okg = P.hybrid_rollout(0.0), B.hybrid_rollout(0.0)[0]
    assert (not okc) and (not okg)
    N, S = P.n_stages, P.n_states
    for nm in ("X", "Defect"):
        assert np.array_equal(B.get(nm)[0, :S], P.get(nm)), nm
    assert np.array_equal(B.get("U")[0, :N], P.get("U"))
    assert np.array_equal(B.get("g")[0, :N], _g_by_leg(P))
    so, sg = P.scalars(), B.scalars()[0]
    assert so["max_tconstr"] == sg[5] and so["max_pconstr"] == sg[6]
    P.compute_cost(); B.compute_cost()
    so, sg = P.scalars(), B.scalars()[0]
    assert abs(so["actual_cost"] - sg[0]) <= RTOL * abs(so["actual_cost"])


def test_single_shooting_matches_oracle(pkg, orc, workloads):
    """option.MS = false (SinglePhase.cpp:211-220): every phase is propagated from its first node (which stays a shooting node,
    :187-193), no linear rollout, the expected cost change comes from the backward sweep (MultiPhaseDDP.cpp:326-329)."""
    w = workloads.config3(pkg, 9)
    B = _batch_for(pkg, w)
    o = dict(MS=0)
    B.solve(pkg.Options(**o))
    info, tr = B.info(), B.trace()
    Xb, Ub, K = B.get("Xbar"), B.get("Ubar"), B.get("K")
    tables, checked = {}, 0
    for i in range(w.n):
        P = _oracle_problem(orc, w, i, tables)
        s, otr = P.solve(o)
        Q = _oracle_problem(orc, w, i, tables)  # sensitivity: the same solve on the other model back end
        if orc.ref_available():
            gait, k0 = w.keys[w.schedule_id[i]]
            Q = orc.Problem(tables[gait], k0, w.plan, model=orc.MODEL_PORT)
            Q.x0 = w.x0[i]
        s2, otr2 = Q.solve(o)
        if not (s["n_iter"] == s2["n_iter"] and s["status"] == s2["status"] and np.array_equal(otr[:, 9], otr2[:, 9])
                and abs(s["cost"] - s2["cost"]) <= 1e-11 * abs(s["cost"])):
            continue  # ill-posed for parity
        n = int(s["n_iter"])
        assert info["n_iter"][i] == n and info["status"][i] == int(s["status"]) and info["n_sweeps"][i] == int(s["n_sweeps"]), (i, s, info[i])
        assert np.array_equal(tr[i, :n, 9], otr[:, 9]) and np.array_equal(tr[i, :n, 10], otr[:, 10]), i
        for col in (2, 3, 11, 12, 6, 7):
            assert rel_err(tr[i, :n, col], otr[:, col]) < RTOL, (i, col)
        assert rel_err_rows(Xb[i, :P.n_states], P.get("Xbar")) < RTOL and rel_err_rows(Ub[i, :P.n_stages], P.get("Ubar")) < RTOL, i
        assert rel_err_rows(K[i, :P.n_stages], P.get("K")) < RTOL, i
        checked += 1
    assert checked >= 6, checked


def test_invalid_options_are_refused(pkg, workloads):
    """Options for which the reference's own loops do not terminate would hang the stream: refused with an error."""
    w = workloads.config1(pkg)
    B = _batch_for(pkg, w)
    for bad in (dict(alpha=1.0), dict(alpha=0.0), dict(update_regularization=1.0), dict(cost_thresh=float("nan")), dict(max_DDP_iter=-1)):
        with pytest.raises(pkg.HsddpError):
            B.solve(pkg.Options(**bad))
    B.solve()
    assert B.info()["n_iter"][0] == 13


def test_full_size_config2_properties(pkg, orc, workloads):
    """1,024 problems (BASELINE configs[1]): size-independent properties + oracle spot checks."""
    w = workloads.config2(pkg, 1024)
    B = _batch_for(pkg, w)
    B.solve()
    info = B.info()
    assert np.all(np.isin(info["status"], (0, 1, 2))) and np.all(info["n_iter"] >= 1)
    assert np.all(info["cost"] < info["cost0"]) and np.all(info["feas"] <= 1e-3)
    assert np.isfinite(B.get("Xbar")).all() and np.isfinite(B.get("K")).all()
    Xb, K = B.get("Xbar").copy(), B.get("K").copy()
    # idempotence / determinism: reset + solve again gives bit-identical results
    B.reset(); B.solve()
    assert np.array_equal(B.get("Xbar"), Xb) and np.array_equal(B.get("K"), K)
    assert np.array_equal(B.info()["n_iter"], info["n_iter"])
    # problems are independent: a permuted batch gives the same per-problem answers
    perm = np.random.default_rng(0).permutation(w.n)
    B2 = pkg.MultiPhaseDDPBatch(0)
    B2.set_problems(w.schedules, w.schedule_id[perm])
    B2.set_initial_condition(w.x0[perm])
    B2.solve()
    assert np.array_equal(B2.get("Xbar"), Xb[perm]) and np.array_equal(B2.info()["n_iter"], info["n_iter"][perm])
    # oracle spot checks across the batch
    B.reset(); B.solve()
    _compare_solution(pkg, orc, w, B, [0, 1, 511, 1023], {})


@pytest.mark.parametrize("mode", [1, 2])
def test_full_size_config3_properties(pkg, orc, workloads, mode):
    """16,384 mixed-gait problems (BASELINE configs[2], the bench workload): size-independent properties, for the
    persistent kernel (mode 1) and the phased multi-stream driver (mode 2, what `auto` picks at this size).
    Determinism, independence of the shard a problem is solved in (the multi-GPU claim: index sharding with no
    data-path collective changes nothing), sane termination records, and a command record that is a view of the
    trajectories."""
    n = 16384
    w = workloads.config3(pkg, n)
    B = _batch_for(pkg, w)
    B.set_solve_mode(mode)
    B.solve()
    info = B.info().copy()
    assert np.all(np.isin(info["status"], (0, 1, 2, 3))) and np.all(info["n_iter"] >= 1) and np.all(info["n_iter"] <= 50)
    assert np.all(info["n_sweeps"] >= info["n_iter"]) and np.all(info["n_trials"] <= 4 * info["n_iter"])
    done = info["status"] <= 1
    assert done.mean() > 0.8 and np.all(info["feas"][done] <= 1e-3) and np.all(np.isfinite(info["cost"]))
    Ub = B.get_rows("Ubar", 0, 8)
    Xb = B.get_rows("Xbar", 0, 8)
    assert np.isfinite(Ub).all() and np.isfinite(Xb).all()
    B.reset(); B.solve()
    assert B.info().tobytes() == info.tobytes() and np.array_equal(B.get_rows("Ubar", 0, 8), Ub)
    # rank r of an 8-way index sharding solves problems [2048 r, 2048 (r+1)) alone: same bits as inside the big batch
    for r in (0, 5):
        ws = workloads.config3(pkg, 2048, first=2048 * r)
        Bs = _batch_for(pkg, ws)
        Bs.set_solve_mode(mode)
        Bs.solve()
        assert Bs.info().tobytes() == info[2048 * r:2048 * (r + 1)].tobytes()
        assert np.array_equal(Bs.get_rows("Ubar", 0, 8), Ub[2048 * r:2048 * (r + 1)])
    # the command record of a problem is (float32 of) its first stages: phase 0 is at least 8 stages long for most windows
    cmd = B.mpc_command(8)
    first_len = np.array([w.schedules[s].horizon[0] for s in w.schedule_id])
    sel = np.nonzero(first_len >= 8)[0][:2000]
    assert len(sel) > 100
    assert np.array_equal(cmd["hkd_controls"][sel, :8], Ub[sel].astype(np.float32))
    assert np.array_equal(cmd["des_body_state"][sel, :8], Xb[sel][:, :, :12].astype(np.float32))
    if mode == 2:  # the two drivers agree to rounding on the well-conditioned problems (separate compilations)
        B1 = _batch_for(pkg, w)
        B1.set_solve_mode(1)
        B1.solve()
        i1 = B1.info()
        same = (i1["n_iter"] == info["n_iter"]) & (i1["status"] == info["status"])
        assert same.mean() > 0.97, same.mean()
        U1 = B1.get_rows("Ubar", 0, 8)
        err = np.abs(U1[same] - Ub[same]).reshape(same.sum(), -1).max(axis=1) / np.maximum(1.0, np.abs(Ub[same]).reshape(same.sum(), -1).max(axis=1))
        assert np.quantile(err, 0.99) < 1e-9, np.quantile(err, [0.5, 0.99, 1.0])


def _write_quad_reference_csv(npz_path, out_path, n_rows=120):
    """Text form of a gait fixture in the reference's quad_reference.csv format (3 decimals, as
    scripts/ReferenceGen/generate_reference.m writes it)."""
    d = np.load(npz_path)
    with open(out_path, "w") as f:
        f.write("dt\n%4.3f\n" % float(d["dt"]))
        for i in range(n_rows):
            for key, name in (("body_state", "body_state "), ("qJ", "qJ"), ("foot_placements", "foot_placements"), ("grf", "grf")):
                f.write(name + "\n" + "".join("%6.3f " % v for v in d[key][i]) + "\n")
            f.write("torque\n" + "".join("%6.3f " % 0.0 for _ in range(12)) + "\n")
            f.write("contact\n" + "".join("%d " % v for v in d["contact"][i]) + "\n")
            f.write("status_dur\n" + "".join("%6.3f " % v for v in d["status_dur"][i]) + "\n")


def test_cpp_shim_example_matches_oracle(pkg, orc, tmp_path):
    """The C++ drop-in surface (MultiPhaseDDP<double>::solve via hkd-mpc_b200/host/MultiPhaseDDP.hpp),
    fed through the text loader (QuadReference::load_top_level_data)."""
    import subprocess
    from conftest import ROOT
    csv = str(tmp_path / "quad_reference.csv")
    _write_quad_reference_csv(GAIT_PATH("trot"), csv)
    exe = str(tmp_path / "solve_trot")
    libdir = os.path.dirname(pkg.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", os.path.join(ROOT, "examples", "solve_trot.cpp"), "-L" + libdir, "-lhsddp_b200",
                           "-Wl,-rpath," + libdir, "-o", exe])
    out = subprocess.run([exe, csv, "3"], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    assert len(out) == 4 and out[3].startswith("command of problem 0: 8 steps")
    T = _table(orc, "trot")
    for i, line in enumerate(out[:3]):
        tok = line.replace("=", " ").split()
        status, iters, cost = int(tok[1]), int(tok[3]), float(tok[6])
        P = orc.Problem(T, 0, 0.6)
        x0 = P.x0
        x0[3] += 0.001 * i
        P.x0 = x0
        s, _ = P.solve()
        assert status == int(s["status"]) and iters == int(s["n_iter"]) and abs(cost - s["cost"]) < 1e-7 * abs(s["cost"])
        if i == 0:  # the command line of the example: first GRF z of leg 0 and one feedback entry
            ref = orc.mpc_command(P, 8)
            tok = out[3].replace("=", " ").replace(",", " ").split()
            fz, fb = float(tok[tok.index("N") - 1]), float(tok[-1])
            assert abs(fz - ref["hkd_controls"][0, 2]) < 1e-3 and abs(fb - ref["feedback"][0, 2, 5]) < 1e-3
