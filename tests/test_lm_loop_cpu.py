"""Host logic without a GPU: the Python mirror of optimize_lm_ours (rootba_b200.bundle_adjust_manual, after
solver/bal_bundle_adjustment.cpp:249-544) driven by an ORACLE-backed Linearizor must reproduce the oracle's own C++
restatement of the same loop step for step -- same costs, same accept / reject decisions, same lambda schedule, same PCG
iteration counts -- because both then run identical arithmetic.  This isolates the loop logic (lambda / vee updates in
Scalar precision, step quality, function-tolerance stop, backup / restore protocol) from the CUDA path, which
tests/test_gpu_parity.py::test_lm_trajectory covers on the GPU."""
import numpy as np
import pytest

import rootba_b200 as rb
from oracle import oracle_py as orc


class OracleLinearizor:
    """rootba::Linearizor interface (solver/linearizor.hpp:56-82) on top of the CPU oracle"""

    def __init__(self, oracle):
        self.o = oracle
        self.it_summary = None

    def start_iteration(self, it_summary=None):
        self.it_summary = it_summary

    def finish_iteration(self):
        pass

    def compute_error(self):
        return self.o.compute_error()

    def linearize(self):
        assert self.o.linearize()

    def solve(self, lam):
        inc, iters = self.o.solve(lam)
        self.it_summary["linear_solver_iterations"] = iters
        return inc

    def apply(self, inc):
        return self.o.apply(inc)

    # BalProblem.backup / restore / sync_from_device forward to these when a linearizor is attached
    def _backup(self):
        self.o.backup()

    def _restore(self):
        self.o.restore()

    def download_state(self):
        pass


CASES = [
    (np.float64, {}),
    (np.float32, {}),
    (np.float64, {"preconditioner_type": "JACOBI"}),
    (np.float32, {"robust_norm": "HUBER", "huber_parameter": 2.0}),
    (np.float64, {"optimized_cost": "ERROR_VALID"}),
    (np.float32, {"optimized_cost": "ERROR_VALID_AVG"}),
    (np.float64, {"hard": True}),                                   # strongly perturbed start: rejected steps, vee growth, recovery
    (np.float32, {"hard": True}),
    (np.float64, {"hard": True, "min_relative_decrease": 0.5}),     # mediocre steps are rejected too
    (np.float64, {"hard": True, "initial_trust_region_radius": 1e12, "min_trust_region_radius": 1e-3}),  # runs into max lambda
]


@pytest.fixture(scope="module")
def hard_problem():
    from rootba_b200.synthetic import synth_bal
    return synth_bal(20, 500, 4.1, seed=7, perturb_rot=0.3, perturb_trans=3.0, perturb_lm=2.0)


@pytest.mark.parametrize("dtype,kw", CASES)
def test_python_lm_loop_equals_oracle_lm_loop(small_problem, hard_problem, dtype, kw):
    kw = dict(kw)
    hard = kw.pop("hard", False)
    small_problem = hard_problem if hard else small_problem
    n_it = 12 if hard else 8
    so = rb.SolverOptions(max_num_iterations=n_it)
    okw = {"max_num_iterations": n_it, "num_threads": 1}
    for k, v in kw.items():
        if k == "preconditioner_type":
            so.preconditioner_type = v; okw[k] = {"JACOBI": 0, "SCHUR_JACOBI": 1}[v]
        elif k == "robust_norm":
            so.residual.robust_norm = v; okw[k] = 1
        elif k == "huber_parameter":
            so.residual.huber_parameter = v; okw[k] = v
        elif k == "optimized_cost":
            so.optimized_cost = v; okw[k] = {"ERROR": 0, "ERROR_VALID": 1, "ERROR_VALID_AVG": 2}[v]
            okw["use_valid_projections_only"] = int(so.use_projection_validity_check())
        else:
            setattr(so, k, v); okw[k] = v
    ref = orc.Oracle(small_problem, dtype, orc.default_options(**okw))
    rows, term = ref.optimize()
    drv = orc.Oracle(small_problem, dtype, orc.default_options(**okw))
    bp = rb.BalProblem.from_arrays(small_problem, dtype)
    lin = OracleLinearizor(drv)
    bp._linearizor = lin
    summ = rb.bundle_adjust_manual(bp, so, linearizor=lin)
    its = summ["iterations"]
    assert len(its) == len(rows)
    for a, b in zip(its, rows):
        assert a["iteration"] == int(b["iteration"])
        assert bool(a["step_is_successful"]) == bool(b["step_is_successful"]), a["iteration"]
        if "cost" in a:  # (absent only in the non-finite-increment branch)
            assert a["cost"]["all"]["error"] == b["cost"], a["iteration"]        # identical arithmetic: bit-equal
            assert a["cost"]["valid"]["error"] == b["cost_valid"]
        assert a["trust_region_radius"] == pytest.approx(b["trust_region_radius"], rel=1e-15)
        if a["iteration"] > 0:
            assert a["linear_solver_iterations"] == int(b["cg_iterations"])
            assert a["l_diff"] == pytest.approx(b["l_diff"], rel=1e-15)
            assert a["relative_decrease"] == pytest.approx(b["relative_decrease"], rel=1e-15)
    if hard:
        assert not all(bool(r["step_is_successful"]) for r in rows[1:])  # the case really exercises the reject branch
    # final state identical on both sides
    c1, l1 = ref.get_state()
    c2, l2 = drv.get_state()
    assert np.array_equal(c1, c2) and np.array_equal(l1, l2)


# ---- the C++ host's LM loop (rootba_b200/host/solver.hpp::optimize_lm), same idea ------------------------------------

CPP_CASES = [
    ([], {}, False),
    (["--float"], {}, False),
    (["--jacobi"], {"preconditioner_type": 0}, False),
    (["--float", "--huber", "2.0"], {"robust_norm": 1, "huber_parameter": 2.0}, False),
    (["--optimized-cost", "ERROR_VALID"], {"optimized_cost": 1, "use_valid_projections_only": 1}, False),
    (["--optimized-cost", "ERROR_VALID_AVG", "--float"], {"optimized_cost": 2, "use_valid_projections_only": 1}, False),
    (["--givens"], {"use_householder": 0}, True),
    ([], {}, True),
    (["--float"], {}, True),
    (["--min-relative-decrease", "0.5"], {"min_relative_decrease": 0.5}, True),
    (["--initial-trust-region-radius", "1e12", "--min-trust-region-radius", "1e-3"],
     {"initial_trust_region_radius": 1e12, "min_trust_region_radius": 1e-3}, True),
]


@pytest.mark.parametrize("flags,okw,hard", CPP_CASES)
def test_cpp_lm_loop_equals_oracle_lm_loop(tmp_path, small_problem, hard_problem, flags, okw, hard):
    """tests/cpp/lm_loop_cpu.cpp runs rootba_b200::optimize_lm (the loop `bal_qr` uses on the GPU) with an oracle-backed
    Linearizor; the oracle's own loop on the arrays that driver loaded must give the same trajectory."""
    import os
    import subprocess
    from conftest import ROOT
    from rootba_b200 import _lib
    from rootba_b200.synthetic import BalArrays, write_bal
    from test_host_cpp import _read_dump
    _lib.build()
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "cpp"), "-s"])
    prob = hard_problem if hard else small_problem
    n_it = 12 if hard else 8
    path, dump = str(tmp_path / "p.txt"), str(tmp_path / "arrays.bin")
    write_bal(prob, path)
    out = subprocess.check_output([os.path.join(ROOT, "tests", "cpp", "_build", "lm_loop_cpu"), "--input", path, "--dump", dump,
                                   "--max-num-iterations", str(n_it)] + flags, text=True)
    got = []
    for line in out.splitlines():
        t = line.split()
        if t[0] == "it":
            got.append({"iteration": int(t[1]), "cost": float(t[3]), "cost_valid": float(t[5]), "ok": int(t[7]), "valid": int(t[9]),
                        "trr": float(t[11]), "rho": float(t[13]), "cg": int(t[15])})
    cams, lms, off, oc, xy = _read_dump(dump)
    dtype = np.float32 if "--float" in flags else np.float64
    ref = orc.Oracle(BalArrays(cams, lms, off, oc, xy), dtype, orc.default_options(max_num_iterations=n_it, num_threads=1, **okw))
    rows, _ = ref.optimize()
    assert len(got) == len(rows)
    for a, b in zip(got, rows):
        assert a["iteration"] == int(b["iteration"]) and a["ok"] == int(bool(b["step_is_successful"])), a
        # same source, same compiler flags: the arithmetic is identical.  A rejected step logs the rejected cost on both sides.
        assert a["cost"] == pytest.approx(b["cost"], rel=1e-13) and a["cost_valid"] == pytest.approx(b["cost_valid"], rel=1e-13)
        assert a["trr"] == pytest.approx(b["trust_region_radius"], rel=1e-13)
        if a["iteration"] > 0:
            assert a["cg"] == int(b["cg_iterations"]) and a["rho"] == pytest.approx(b["relative_decrease"], rel=1e-9, abs=1e-12)
    if hard:
        assert not all(a["ok"] for a in got[1:])


def test_function_tolerance_compares_with_the_previous_logged_cost():
    """The stop after a successful step compares its cost with the previous log entry's (bal_bundle_adjustment.cpp:69-72,
    :174-201), which after rejected steps is the last rejected cost.  Here iterations 1-6 are rejected and 7 is accepted
    with a cost within 10% of the linearisation point's but 62% away from iteration 6's, so the loop goes on and stops at
    iteration 10.  Pinned for the oracle and the Python mirror; tests/test_gpu_pcg_paths.py holds rba_lm_run to it."""
    from rootba_b200.synthetic import synth_bal
    prob = synth_bal(49, 1800, 4.1, seed=38401, perturb_rot=0.2, perturb_trans=1.0, perturb_lm=2.0)
    kw = dict(max_num_iterations=20, min_relative_decrease=0.99, function_tolerance=0.1)
    rows, term = orc.Oracle(prob, np.float64, orc.default_options(num_threads=1, **kw)).optimize()
    assert [bool(r["step_is_successful"]) for r in rows] == [True] + [False] * 6 + [True, False, False, True]
    assert term == 1  # CONVERGENCE
    c = [r["cost"] for r in rows]
    assert abs(c[0] - c[7]) <= 0.1 * c[7] < abs(c[6] - c[7])  # the linearisation point's cost would have stopped at 7
    assert abs(c[9] - c[10]) <= 0.1 * c[10]  # the rejected iteration 9's cost stops at 10
    drv = orc.Oracle(prob, np.float64, orc.default_options(num_threads=1, **kw))
    bp = rb.BalProblem.from_arrays(prob, np.float64)
    lin = OracleLinearizor(drv)
    bp._linearizor = lin
    summ = rb.bundle_adjust_manual(bp, rb.SolverOptions(**kw), linearizor=lin)
    its = summ["iterations"]
    assert summ["termination_type"] == "CONVERGENCE" and len(its) == len(rows)
    for a, b in zip(its, rows):
        assert bool(a["step_is_successful"]) == bool(b["step_is_successful"]) and a["cost"]["all"]["error"] == b["cost"]
        if a["iteration"] > 0:
            assert a["linear_solver_iterations"] == int(b["cg_iterations"])
