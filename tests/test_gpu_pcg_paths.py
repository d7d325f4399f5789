"""GPU tests of the PCG paths and settings the parity tests leave out, and of the native LM loop's stopping rule.

Which PCG path a single-GPU solve takes: k_pcg_vec runs on one cluster of up to 16 CTAs, and a CTA keeps its share of the
cameras in registers when 9 * ceil(nc / cluster) <= VEC_THREADS * VEC_EPT = 1024 scalars.  Then the operator's
per-camera sums reach it as per-segment partial sums (k_cam_reduce).  Otherwise -- more than 1808 cameras with the 16-CTA
cluster, as on Final-13682 -- k_cam_reduce_final sums every camera into D.y (arrival counters) and k_pcg_vec round-trips
q, r and z through global memory.  Three environment variables, read when a handle is created, select the other paths:
  RBA_PCG_CLUSTER=c   caps the cluster at c CTAs.  The device may grant fewer, which only makes a CTA's share larger, so a
                      camera count above 113 * c is on the global-memory path whatever is granted;
  RBA_PCG_PARTIALS=0  register-resident path, but with the per-camera sums in D.y (documented as bit-identical);
  RBA_PDL=0           no programmatic dependent launch (scheduling only: bit-identical).
pcg_check_period (how far the host enqueues ahead, and so how many no-op kernels run after the end) must not change
results either.  The bars are those of test_gpu_parity.py."""
import numpy as np
import pytest

from conftest import rel_err
from test_gpu_parity import TOL1, TOLB, TOLS, make_pair, mixed_problem  # noqa: F401  (mixed_problem is a fixture)

pytestmark = pytest.mark.gpu

VEC_SCALARS = 1024  # VEC_THREADS * VEC_EPT of k_pcg_vec
NO_CONVERGENCE, SUCCESS = 0, 1
STRIPPED = [5, 97]  # cameras without observations in stripped_problem


def register_resident(nc, cluster):
    return 9 * -(-nc // cluster) <= VEC_SCALARS


def create(monkeypatch, env, arrays, dtype, **kw):
    """make_pair with exactly the RBA_* variables of `env` set while the handle is created"""
    with monkeypatch.context() as m:
        for k in ("RBA_PCG_CLUSTER", "RBA_PCG_PARTIALS", "RBA_PDL"):
            m.delenv(k, raising=False)
        for k, v in env.items():
            m.setenv(k, str(v))
        return make_pair(arrays, dtype, **kw)


def strip_cameras(a, cams):
    """`a` without any observation of `cams`, then without the landmarks left with fewer than 2 observations"""
    from rootba_b200.synthetic import BalArrays
    lm_of = np.repeat(np.arange(a.nl), np.diff(a.lm_off))
    keep = ~np.isin(a.obs_cam, cams)
    lm_ok = np.bincount(lm_of[keep], minlength=a.nl) >= 2
    keep &= lm_ok[lm_of]
    new_lm = (np.cumsum(lm_ok) - 1)[lm_of[keep]]
    off = np.concatenate([[0], np.cumsum(np.bincount(new_lm, minlength=int(lm_ok.sum())))]).astype(np.int64)
    return BalArrays(a.cams.copy(), a.lms[lm_ok].copy(), off, a.obs_cam[keep].copy(), a.obs_xy[keep].copy())


@pytest.fixture(scope="module")
def large_problem():
    """Final-13682's track statistics with just enough cameras for the global-memory path at any cluster size"""
    from rootba_b200.synthetic import synth_bal
    a = synth_bal(1850, 20000, 6.5, seed=5, locality=6.0)
    assert a.nc == 1850 and not register_resident(a.nc, 16)  # 116 cameras per CTA (110 in the last): 1044 > 1024
    return a


@pytest.fixture(scope="module")
def ragged_problem():
    """915 cameras: global-memory path with a cluster of 2, 4 or 8 CTAs, and the last CTA short in each (457, 228, 110
    cameras); register-resident with the default 16-CTA cluster (58 per CTA)"""
    from rootba_b200.synthetic import synth_bal
    return synth_bal(915, 8000, 6.5, seed=5, locality=6.0)


@pytest.fixture(scope="module")
def stripped_problem(mixed_problem):
    a = strip_cameras(mixed_problem, STRIPPED)
    assert a.nc == mixed_problem.nc and not np.isin(a.obs_cam, STRIPPED).any()
    assert np.diff(a.lm_off).min() >= 2 and a.nl > 0.99 * mixed_problem.nl
    return a


# ---- A. the global-memory PCG path against the oracle ----------------------------------------------------------------

@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("which,cluster", [("large", None), ("mixed", 1), ("ragged", 2), ("ragged", 4), ("ragged", 8)])
def test_global_memory_pcg_path_against_oracle(request, monkeypatch, dtype, which, cluster):
    """k_cam_reduce_final<false> + the global-memory branch of k_pcg_vec: `large` reaches it by its camera count, the others
    through RBA_PCG_CLUSTER.  Then the same solve on the default path: within the single-stage bar of it (same operator,
    the dot products summed over other CTA shares), and bit-identical between the two register-resident hand-overs."""
    arrays = request.getfixturevalue(f"{which}_problem")
    if cluster is None:
        env = {}
        assert not register_resident(arrays.nc, 16)
    else:
        env = {"RBA_PCG_CLUSTER": cluster}
        assert not register_resident(arrays.nc, cluster) and register_resident(arrays.nc, 16)
        if cluster > 1:
            assert arrays.nc % cluster != 0  # the last CTA's share is short
    tol = TOL1[dtype]
    lam = 1e-2
    bp, lin, o, _ = create(monkeypatch, env, arrays, dtype)
    lin.linearize(); assert o.linearize()
    inc_g = lin.solve(lam)
    inc_c, dbg = o.solve(lam, want_debug=True)
    assert rel_err(lin.get_rhs(), dbg["b"]) < tol * 4
    inv_g, _ = lin.get_preconditioner()
    assert max(rel_err(inv_g[c], dbg["inv_blocks"][c]) for c in range(lin.nc)) < TOLB[dtype]
    x = np.random.default_rng(6).uniform(-1, 1, 9 * lin.nc).astype(dtype)
    assert rel_err(lin.right_multiply(x), o.right_multiply(x)) < tol * 4
    assert abs(lin.last_cg.num_iterations - dbg["cg_iterations"]) <= 2
    assert lin.last_cg.termination_type == dbg["cg_termination"]
    assert rel_err(inc_g, inc_c) < TOLS[dtype]
    it_g = lin.last_cg.num_iterations
    lin.close()
    if cluster is None:
        return
    res = {}
    for name, env2 in (("default", {}), ("no_partials", {"RBA_PCG_PARTIALS": 0})):
        _, l2, _, _ = create(monkeypatch, env2, arrays, dtype)
        l2.linearize()
        res[name] = (l2.solve(lam), l2.last_cg.num_iterations, l2.last_cg.termination_type)
        l2.close()
    assert rel_err(inc_g, res["default"][0]) < tol
    if dtype == np.float64:
        assert it_g == res["default"][1]
    assert np.array_equal(res["no_partials"][0], res["default"][0]) and res["no_partials"][1:] == res["default"][1:]


# ---- B. PCG stop branches on both paths -------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("path", ["register", "global"])
@pytest.mark.parametrize("kw,term", [
    ({"max_linear_solver_iterations": 3, "eta": 1e-4}, NO_CONVERGENCE),   # ends on the is_last write of inc (9 iterations unbounded)
    ({"min_linear_solver_iterations": 25, "eta": 0.1}, SUCCESS),           # residual refreshes at i = 10 and 20 (2 unbounded)
])
def test_pcg_stop_branches(monkeypatch, mixed_problem, dtype, path, kw, term):
    env = {"RBA_PCG_CLUSTER": 1} if path == "global" else {}
    assert register_resident(mixed_problem.nc, 16) and not register_resident(mixed_problem.nc, 1)
    bp, lin, o, _ = create(monkeypatch, env, mixed_problem, dtype, **kw)
    lin.linearize(); assert o.linearize()
    lam = 1e-2
    inc_g = lin.solve(lam)
    inc_c, dbg = o.solve(lam, want_debug=True)
    assert dbg["cg_termination"] == term and lin.last_cg.termination_type == term
    if term == NO_CONVERGENCE:
        assert lin.last_cg.num_iterations == dbg["cg_iterations"] == 3
    else:
        assert dbg["cg_iterations"] >= 25 and abs(lin.last_cg.num_iterations - dbg["cg_iterations"]) <= 2
    assert np.all(np.isfinite(inc_g)) and rel_err(inc_g, inc_c) < TOLS[dtype]
    lin.close()


# ---- C. cameras without observations ----------------------------------------------------------------------------------

def _solve_twice_around_right_multiply(lin, solve_oracle, dtype, check):
    """solve, right_multiply (which leaves H x + lambda x in the operator's output vector), solve at another lambda"""
    x = np.random.default_rng(12).uniform(-1, 1, 9 * lin.nc).astype(dtype)
    idx = np.concatenate([np.arange(9 * c, 9 * c + 9) for c in STRIPPED])
    for k, lam in enumerate((1e-2, 1e-3)):
        inc_g = lin.solve(lam)
        inc_c = solve_oracle(lam)
        assert np.all(inc_c[idx] == 0), k
        assert np.all(inc_g[idx] == 0), (k, np.abs(inc_g[idx]).max())
        check(inc_g, inc_c)
        if k == 0:
            y = lin.right_multiply(x)
            assert np.array_equal(y[idx], (dtype(lam) * x[idx]).astype(dtype))  # H has no entries for these cameras


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("path", ["register", "global", "no_partials"])
def test_cameras_without_observations(monkeypatch, stripped_problem, dtype, path):
    env = {"register": {}, "global": {"RBA_PCG_CLUSTER": 1}, "no_partials": {"RBA_PCG_PARTIALS": 0}}[path]
    bp, lin, o, _ = create(monkeypatch, env, stripped_problem, dtype)
    lin.linearize(); assert o.linearize()

    def solve_oracle(lam):
        inc, dbg = o.solve(lam, want_debug=True)
        solve_oracle.dbg = dbg
        return inc

    def check(inc_g, inc_c):
        assert abs(lin.last_cg.num_iterations - solve_oracle.dbg["cg_iterations"]) <= 2
        assert lin.last_cg.termination_type == solve_oracle.dbg["cg_termination"]
        assert rel_err(inc_g, inc_c) < TOLS[dtype]

    _solve_twice_around_right_multiply(lin, solve_oracle, dtype, check)
    lin.close()


@pytest.mark.parametrize("solver_type,cluster", [("SCHUR_COMPLEMENT", None), ("SCHUR_COMPLEMENT", 1), ("POWER_SCHUR_COMPLEMENT", None)])
def test_cameras_without_observations_schur(monkeypatch, stripped_problem, solver_type, cluster):
    """the Schur-complement solvers against the oracle's restatements, at test_gpu_sc.py's float64 bar; Power-SC always
    sums the operator into D.y"""
    import rootba_b200 as rb
    from oracle import oracle_py as orc
    dtype, order = np.float64, 20
    with monkeypatch.context() as m:
        for k in ("RBA_PCG_CLUSTER", "RBA_PCG_PARTIALS", "RBA_PDL"):
            m.delenv(k, raising=False)
        if cluster is not None:
            m.setenv("RBA_PCG_CLUSTER", str(cluster))
        lin = rb.LinearizorQR.create(rb.BalProblem.from_arrays(stripped_problem, dtype),
                                     rb.SolverOptions(solver_type=solver_type, power_order=order))
    o = orc.Oracle(stripped_problem, dtype, orc.default_options(num_threads=0))
    lin.linearize(); o.scl_linearize()
    power = solver_type == "POWER_SCHUR_COMPLEMENT"

    def solve_oracle(lam):
        inc, dbg = o.scl_power_solve(lam, order, 0.1) if power else o.scl_solve(lam)
        solve_oracle.dbg = dbg
        return inc

    def check(inc_g, inc_c):
        d = solve_oracle.dbg
        if power:
            assert abs(lin.last_cg.num_iterations - d["power_order"]) <= 1 and lin.last_cg.termination_type == d["termination"]
            if lin.last_cg.num_iterations != d["power_order"]:
                return
        else:
            assert abs(lin.last_cg.num_iterations - d["cg_iterations"]) <= 2 and lin.last_cg.termination_type == d["cg_termination"]
        assert rel_err(inc_g, inc_c) < 1e-8

    _solve_twice_around_right_multiply(lin, solve_oracle, dtype, check)
    lin.close()


# ---- D. scheduling settings do not change results ---------------------------------------------------------------------

def _three_lm_steps(monkeypatch, arrays, env, **kw):
    bp, lin, _, _ = create(monkeypatch, env, arrays, np.float32, **kw)
    lam, out = 1e-4, []
    for _ in range(3):
        r = lin.lm_step(lam, True)
        assert not r["solve_failed"]
        out.append((r["l_diff"], r["cost"], lin.last_cg.num_iterations, lin.last_cg.termination_type))
        out.append(lin.solve(lam))  # the step's increment again: same linearisation and lambda
        lam /= 3
    lin.download_state()
    lin.close()
    return out, bp.cams.copy(), bp.lms.copy()


@pytest.mark.parametrize("env,kw", [({}, {"pcg_check_period": 1}), ({}, {"pcg_check_period": 64}), ({"RBA_PDL": 0}, {})])
def test_scheduling_settings_are_bit_identical(monkeypatch, mixed_problem, env, kw):
    ref, cams0, lms0 = _three_lm_steps(monkeypatch, mixed_problem, {}, pcg_check_period=4)
    got, cams1, lms1 = _three_lm_steps(monkeypatch, mixed_problem, env, **kw)
    assert ref[0][2] > 1  # PCG iterations: the settings have something to reorder
    for a, b in zip(ref, got):
        if isinstance(a, np.ndarray):
            assert np.array_equal(a, b)
        else:
            assert a == b
    assert np.array_equal(cams0, cams1) and np.array_equal(lms0, lms1)


# ---- E. the native LM loop's stopping rule ----------------------------------------------------------------------------

@pytest.fixture(scope="module")
def reject_problem():
    from rootba_b200.synthetic import synth_bal
    return synth_bal(49, 1800, 4.1, seed=38401, perturb_rot=0.2, perturb_trans=1.0, perturb_lm=2.0)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_native_lm_loop_stops_against_the_previous_logged_cost(reject_problem, dtype):
    """The function tolerance compares a step's cost with the previous LOG ENTRY's (bal_bundle_adjustment.cpp:69-72,
    :174-201): after rejected steps that is the last rejected cost, not the cost at the linearisation point.  In float64
    iterations 1-6 are rejected and 7 is accepted within 10% of the linearisation point's cost but not of iteration 6's,
    so the loop goes on to iteration 10 (tests/test_lm_loop_cpu.py pins that trajectory on the oracle).  rba_lm_run must
    equal the Python mirror bit for bit, and the oracle's loop in decisions."""
    import rootba_b200 as rb
    from oracle import oracle_py as orc
    okw = dict(max_num_iterations=20, min_relative_decrease=0.99, function_tolerance=0.1)
    so = rb.SolverOptions(**okw)
    bpa, bpb = rb.BalProblem.from_arrays(reject_problem, dtype), rb.BalProblem.from_arrays(reject_problem, dtype)
    summ = rb.bundle_adjust_manual(bpa, so)
    lin = rb.LinearizorQR.create(bpb, so)
    its, term, _ = lin.lm_run(64)
    py = summ["iterations"][1:]
    assert [bool(a["step_is_successful"]) for a in py] == [b["accepted"] for b in its]
    for a, b in zip(py, its):
        assert a["linear_solver_iterations"] == b["cg_iterations"] and a["linear_solver_termination"] == b["cg_termination"]
        assert a["cost"]["all"]["error"] == b["cost"] and a["lam"] == b["lambda"], a["iteration"]
    assert summ["termination_type"] == "CONVERGENCE" and term and its[-1]["terminated"]
    assert not any(b["terminated"] for b in its[:-1])
    lin.download_state()
    assert np.array_equal(bpa.cams, bpb.cams) and np.array_equal(bpa.lms, bpb.lms)
    lin.close()
    if dtype == np.float64:
        rows, _ = orc.Oracle(reject_problem, dtype, orc.default_options(num_threads=0, **okw)).optimize()
        assert [bool(r["step_is_successful"]) for r in rows[1:]] == [b["accepted"] for b in its]
        assert [b["accepted"] for b in its] == [False] * 6 + [True, False, False, True]
