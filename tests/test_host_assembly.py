"""Host-side logic and the C-ABI boundary (CPU; no GPU compute calls)."""
import ctypes as C
import os
import re
import numpy as np
import pytest
from conftest import GOLDEN, GAIT_PATH, ROOT


def test_library_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, "include", "hsddp_b200.h")).read()
    names = set(re.findall(r"\b((?:hsddp|hkd)_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) > 40
    L = C.CDLL(pkg.LIB_PATH)
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert not missing, missing


def test_struct_layouts_match_the_header(pkg):
    assert C.sizeof(pkg.Options) == 6 * 8 + 2 * 4 + 6 * 8 + 4 * 4
    assert C.sizeof(pkg.ConstraintParams) == 7 * 8
    assert C.sizeof(pkg.Info) == 6 * 4 + 6 * 8
    assert pkg.INFO_DTYPE.itemsize == C.sizeof(pkg.Info)
    assert C.sizeof(pkg.ScheduleStruct) == 656 + 8 + 4 * 8
    # hsddp_mpc_command: 1 + 4 + 40 ints, 240 + 120 + 1440 + 12 floats, 1 pad int
    assert pkg.CMD_DTYPE.itemsize == 4 * (1 + 4 + 40 + 240 + 120 + 1440 + 12 + 1)


def test_no_gpu_means_loud_failure(pkg):
    """There is no CPU fallback: without a device the solver handle cannot be created."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.HsddpError):
        pkg.MultiPhaseDDPBatch(0)


@pytest.mark.parametrize("gait,starts", [("trot", [0, 7, 100, 333, 680]), ("bound", [0, 250, 266, 500]), ("pronk", [0, 50, 300, 687])])
def test_schedule_builder_equals_oracle_assembly(pkg, orc, gait, starts):
    T = orc.GaitTable(GAIT_PATH(gait))
    R = pkg.QuadReference(GAIT_PATH(gait))
    for k0 in starts:
        for plan in (0.25, 0.5, 0.6, 1.0):
            if k0 + round(plan / 0.01) + 2 > T.n:
                continue
            P = orc.Problem(T, k0, plan)
            S = pkg.Schedule(R, k0, plan)
            assert S.horizon == [p["horizon"] for p in P.phases]
            assert S.contact == [p["contact"] for p in P.phases] and S.next_contact == [p["next_contact"] for p in P.phases]
            xr, ur, pr, xi = S.array("xr"), S.array("ur"), S.array("prel_r"), S.array("xinit")
            n = 0
            for i, p in enumerate(P.phases):
                for k in range(p["horizon"] + 1):
                    a, b, br, fr, _ = P.stage_reference(i, k)
                    assert np.array_equal(a, xr[n]) and np.array_equal(b, ur[n])
                    assert np.array_equal(fr - np.tile(br[3:6], 4), pr[n])
                    n += 1
            assert np.array_equal(xi, P.get("Xbar"))          # initial guess = reference states (bit exact)
            assert np.array_equal(S.default_x0(), P.x0)


def test_window_past_the_table_is_rejected(pkg):
    R = pkg.QuadReference(GAIT_PATH("trot"))
    with pytest.raises(pkg.HsddpError):
        pkg.Schedule(R, R.n - 10, 0.6)


def test_text_loader_reproduces_the_fixture(pkg):
    """tests/golden/quad_reference_trot.csv: the first 120 rows of the trot table in the reference's quad_reference.csv
    format (3 decimals, which every value of the fixture round-trips through exactly)."""
    path = os.path.join(GOLDEN, "quad_reference_trot.csv")
    S1 = pkg.Schedule(pkg.QuadReference(path), 0, 0.6)
    S2 = pkg.Schedule(pkg.QuadReference(GAIT_PATH("trot")), 0, 0.6)
    for name in ("xr", "ur", "prel_r", "xinit"):
        assert np.array_equal(S1.array(name), S2.array(name))


def test_workload_generators(pkg, workloads):
    w1 = workloads.config1(pkg)
    assert w1.n == 1 and np.array_equal(w1.x0[0], w1.schedules[0].default_x0())
    w2 = workloads.config2(pkg, 16)
    assert len(w2.schedules) == 1 and np.array_equal(w2.x0[0], w1.x0[0])
    d = w2.x0[1:, :12] - w1.x0[0, :12]
    amp = np.array([0.05] * 3 + [0.02] * 3 + [0.2] * 3 + [0.1] * 3)
    assert np.all(np.abs(d) <= amp + 1e-15) and np.abs(d).max() > 0
    w3 = workloads.config3(pkg, 12)
    assert [k[0] for k in w3.keys[:3]] == ["trot", "bound", "pronk"] and w3.keys[3] == ("trot", 7)
    # sharding by index reproduces the same problems
    w3b = workloads.config3(pkg, 6, first=6)
    assert np.array_equal(w3b.x0, w3.x0[6:])
    # splitmix64 known answer (seed 0 -> 0xE220A8397B1DCDAF)
    assert workloads.splitmix64_uniform(0, 1)[0] == (0xE220A8397B1DCDAF >> 11) / 2.0 ** 53


def test_cpp_shim_compiles_and_fails_loudly_without_gpu(pkg, tmp_path):
    """The header-only C++ mirror of MultiPhaseDDP (hkd-mpc_b200/host/MultiPhaseDDP.hpp) builds against
    the C ABI; on a box without a GPU the example must exit non-zero (no CPU fallback)."""
    import subprocess
    exe = str(tmp_path / "solve_trot")
    libdir = os.path.dirname(pkg.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-Wall", os.path.join(ROOT, "examples", "solve_trot.cpp"), "-L" + libdir,
                           "-lhsddp_b200", "-Wl,-rpath," + libdir, "-o", exe])
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the GPU run of the example is in test_gpu_parity.py")
    r = subprocess.run([exe, os.path.join(GOLDEN, "quad_reference_trot.csv")], capture_output=True, text=True)
    assert r.returncode != 0 and "error" in r.stderr


def test_config3_shards_by_index_contiguous_and_interleaved(workloads):
    """Problem j of a shard is problem first + j * stride of the configuration: contiguous ranges (bench.py's strong block)
    and interleaved shards (tools/strong_shards.py) cover the same 48 problems exactly once."""
    full = workloads.entries_config3(48)
    cont = [e for r in range(4) for e in workloads.entries_config3(12, first=12 * r)]
    inter = [workloads.entries_config3(12, first=r, stride=4) for r in range(4)]
    assert cont == full
    assert [inter[j % 4][j // 4] for j in range(48)] == full
