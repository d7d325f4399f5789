"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle on identical seeded inputs.

Tolerances (relative norm ||a-b||/(||a||+||b||), reference testing/eigen_utils.hpp:104-108):
  single stage, identical inputs:   f32 1e-5 (the reference's default_test_precision, testing/float_utils.hpp:62-69), f64 1e-11
  SCHUR_JACOBI inverse blocks:      f32 1e-4 (explicit inverse of a 9x9 block: round-off x its condition number), f64 1e-8
  after a PCG solve (inc, l_diff):  f32 1e-4, f64 1e-8   (error growth through PCG; CG iteration count +-2)
  indices / counts:                 bit-exact
Measured on B200 (profiles/r2_f32_trajectory_diag.txt): GPU-f32 vs oracle-f32 inc 3e-6 .. 1e-5, while BOTH are 2e-5 .. 4e-5 from the
float64 oracle (b 4e-5, H x 2e-4, inverse blocks 1e-4 .. 3e-4): the float32 linearisation itself is the noise floor.

Order: the cheap single-solve checks of every option branch come first, the LM-trajectory tests last, so that one
trajectory failure cannot hide the rest under `pytest -x`.
"""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

TOL1 = {np.float32: 1e-5, np.float64: 1e-11}
TOLS = {np.float32: 1e-4, np.float64: 1e-8}
TOLB = {np.float32: 1e-4, np.float64: 1e-8}  # explicit inverse of the preconditioner blocks


def make_pair(arrays, dtype, **opt_kw):
    import rootba_b200 as rb
    from oracle import oracle_py as orc
    okw = {}
    so = rb.SolverOptions()
    if "preconditioner_type" in opt_kw:
        so.preconditioner_type = opt_kw["preconditioner_type"]
        okw["preconditioner_type"] = {"JACOBI": 0, "SCHUR_JACOBI": 1}[so.preconditioner_type]
    if "robust_norm" in opt_kw:
        so.residual.robust_norm = opt_kw["robust_norm"]
        so.residual.huber_parameter = opt_kw.get("huber_parameter", 1.0)
        okw["robust_norm"] = 1 if so.residual.robust_norm == "HUBER" else 0
        okw["huber_parameter"] = so.residual.huber_parameter
    if "optimized_cost" in opt_kw:
        so.optimized_cost = opt_kw["optimized_cost"]
        okw["optimized_cost"] = {"ERROR": 0, "ERROR_VALID": 1, "ERROR_VALID_AVG": 2}[so.optimized_cost]
        okw["use_valid_projections_only"] = int(so.use_projection_validity_check())
    if "use_householder_marginalization" in opt_kw:
        so.use_householder_marginalization = bool(opt_kw["use_householder_marginalization"])
        okw["use_householder"] = int(so.use_householder_marginalization)
    if "operator_form" in opt_kw:
        so.operator_form = opt_kw["operator_form"]  # device-side choice only: the oracle always does the dense product
    if "stage2_form" in opt_kw:
        so.stage2_form = opt_kw["stage2_form"]      # device-side choice only: the oracle always reads the Q2 panel
    if "max_num_iterations" in opt_kw:
        so.max_num_iterations = okw["max_num_iterations"] = opt_kw["max_num_iterations"]
    for k in ("min_linear_solver_iterations", "max_linear_solver_iterations", "eta"):  # PCG stopping rule, both sides
        if k in opt_kw:
            setattr(so, k, opt_kw[k])
            okw[k] = opt_kw[k]
    if "pcg_check_period" in opt_kw:
        so.pcg_check_period = opt_kw["pcg_check_period"]  # device-side scheduling only
    bp = rb.BalProblem.from_arrays(arrays, dtype)
    lin = rb.LinearizorQR.create(bp, so)
    o = orc.Oracle(arrays, dtype, orc.default_options(num_threads=0, **okw))
    return bp, lin, o, so


@pytest.fixture(scope="module")
def mixed_problem():
    """small problem with a wide range of track lengths (covers every group-size class incl. row chunks)"""
    from rootba_b200.synthetic import synth_bal
    return synth_bal(150, 1500, 9.0, seed=11, max_track=150)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_compute_error(small_problem, dtype):
    bp, lin, o, _ = make_pair(small_problem, dtype)
    g, c = lin.compute_error(), o.compute_error()
    assert g["all"]["num_obs"] == c["all"]["num_obs"] == small_problem.nobs
    assert g["valid"]["num_obs"] == c["valid"]["num_obs"]
    assert g["is_numerically_valid"] and c["is_numerically_valid"]
    # float32: a handful of near-camera observations dominate the synthetic cost and make it sensitive to
    # round-off (oracle-f32 vs oracle-f64 differ by ~1e-4), so the f32 bar is "as close to the f64 value as
    # the reference-arithmetic f32 restatement is" (x3) + 1e-5; f64 is held to 1e-12.
    from oracle import oracle_py as orc
    ref = orc.Oracle(small_problem, np.float64).compute_error() if dtype == np.float32 else c
    for key in ("error", "residual_sum"):
        floor = abs(c["all"][key] - ref["all"][key])
        tol = 3 * floor + (1e-5 if dtype == np.float32 else 1e-12) * ref["all"][key]
        assert abs(g["all"][key] - ref["all"][key]) <= tol, (key, g["all"][key], c["all"][key], ref["all"][key])
    lin.close()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("which", ["small", "mixed"])
@pytest.mark.parametrize("qr", ["householder", "givens"])  # ref: ipp:717-743 (default) / ipp:700-715
def test_stage_parity(small_problem, mixed_problem, dtype, which, qr):
    arrays = small_problem if which == "small" else mixed_problem
    bp, lin, o, _ = make_pair(arrays, dtype, use_householder_marginalization=(qr == "householder"))
    tol = TOL1[dtype]
    lam = 0.1
    lin.linearize()
    assert o.linearize()
    s_g, d_g = lin.get_jacobian_scaling()
    assert rel_err(s_g, o.get_scaling()) < tol
    # solve on both (stage 2 + preconditioner + PCG)
    inc_g = lin.solve(lam)
    inc_c, dbg = o.solve(lam, want_debug=True)
    assert rel_err(lin.get_rhs(), dbg["b"]) < tol * 4
    inv_g, blk_g = lin.get_preconditioner()
    worst = max(rel_err(inv_g[c], dbg["inv_blocks"][c]) for c in range(lin.nc))
    assert worst < TOLB[dtype], worst
    # blocks in the reference storage layout: Q1 rows, R, Q1^T r, Q2 panel incl. damping rows
    n_all = arrays.track_lengths()
    picks = sorted(set([int(np.argmax(n_all)), int(np.argmin(n_all)), 0, arrays.nl - 1] +
                       [int(np.nonzero(n_all == k)[0][0]) for k in np.unique(n_all)[:12]]))
    for lm in picks:
        bg, lm_idx, res_idx, jls_g = lin.debug_get_block(lm)
        bc, li, ri, jls_c = o.get_block(lm)
        assert (li, ri) == (lm_idx, res_idx) and bg.shape == bc.shape
        n = n_all[lm]
        assert rel_err(jls_g, jls_c) < tol
        assert rel_err(bg[:3, :9 * n], bc[:3, :9 * n]) < tol * 4, lm
        assert rel_err(np.triu(bg[:3, lm_idx:lm_idx + 3]), np.triu(bc[:3, lm_idx:lm_idx + 3])) < tol * 4, lm
        assert rel_err(bg[:3, res_idx], bc[:3, res_idx]) < tol * 4, lm
        assert rel_err(bg[3:, :9 * n], bc[3:, :9 * n]) < tol * 4, (lm, n)
    # operator
    rng = np.random.default_rng(3)
    x = rng.uniform(-1, 1, 9 * lin.nc).astype(dtype)
    assert rel_err(lin.right_multiply(x), o.right_multiply(x)) < tol * 4
    # PCG result
    assert abs(lin.last_cg.num_iterations - dbg["cg_iterations"]) <= 2
    assert lin.last_cg.termination_type == dbg["cg_termination"]
    assert rel_err(inc_g, inc_c) < TOLS[dtype]
    # back substitution with the SAME increment on both sides
    pose_inc = (rng.uniform(-1, 1, 9 * lin.nc) * 0.01).astype(dtype)
    l_g = lin.back_substitute(pose_inc)
    l_c, ok = o.back_substitute(pose_inc)
    assert ok and abs(l_g - l_c) <= tol * 20 * abs(l_c)
    lin.download_state()
    _, lms_c = o.get_state()
    assert rel_err(bp.lms, lms_c) < tol
    lin.close()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_apply_camera_update(small_problem, dtype):
    bp, lin, o, _ = make_pair(small_problem, dtype)
    lin.linearize(); assert o.linearize()
    lin.solve(1e-4); o.solve(1e-4)
    rng = np.random.default_rng(5)
    inc = (rng.uniform(-1, 1, 9 * lin.nc) * 0.05).astype(dtype)
    l_g = lin.apply(inc.copy())
    l_c = o.apply(inc.copy())
    assert abs(l_g - l_c) <= TOL1[dtype] * 20 * abs(l_c)
    lin.download_state()
    cams_c, lms_c = o.get_state()
    assert rel_err(bp.cams, cams_c) < (1e-6 if dtype == np.float32 else 1e-13)
    assert rel_err(bp.lms, lms_c) < TOL1[dtype]
    lin.close()


def test_backup_restore(small_problem):
    bp, lin, o, _ = make_pair(small_problem, np.float64)
    cams0, lms0 = bp.cams.copy(), bp.lms.copy()
    lin.linearize()
    inc = lin.solve(1e-4)
    bp.backup()
    lin.apply(inc)
    lin.download_state()
    assert not np.array_equal(bp.lms, lms0)
    bp.restore()
    lin.download_state()
    assert np.array_equal(bp.lms, lms0) and np.array_equal(bp.cams, cams0)
    lin.close()


@pytest.mark.parametrize("dtype,kw", [
    (np.float32, {"preconditioner_type": "JACOBI"}),                    # linearizor_qr.cpp:94-112, 196-237; ipp:554-569
    (np.float64, {"preconditioner_type": "JACOBI"}),
    (np.float32, {"robust_norm": "HUBER", "huber_parameter": 2.0}),     # bal_bundle_adjustment_helper.cpp:43-66
    (np.float64, {"robust_norm": "HUBER", "huber_parameter": 0.5}),
    (np.float32, {"optimized_cost": "ERROR_VALID"}),                    # use_valid_projections_only, ipp:113
    (np.float64, {"optimized_cost": "ERROR_VALID"}),
    (np.float32, {"stage2_form": "IDENTITY"}),                          # gradient / blocks through the orthogonality identities
    (np.float64, {"stage2_form": "IDENTITY"}),
])
def test_option_branches_single_solve(small_problem, dtype, kw):
    """one linearize + solve + apply per option branch the reference ships, against the oracle with the same option"""
    bp, lin, o, _ = make_pair(small_problem, dtype, **kw)
    tol = TOL1[dtype]
    eg, ec = lin.compute_error(), o.compute_error()
    assert eg["valid"]["num_obs"] == ec["valid"]["num_obs"] and eg["all"]["num_obs"] == ec["all"]["num_obs"]
    assert abs(eg["all"]["error"] - ec["all"]["error"]) <= (20 * tol) * ec["all"]["error"]
    lin.linearize(); assert o.linearize()
    assert rel_err(lin.get_jacobian_scaling()[0], o.get_scaling()) < tol
    lam = 1e-2
    inc_g = lin.solve(lam)
    inc_c, dbg = o.solve(lam, want_debug=True)
    assert rel_err(lin.get_rhs(), dbg["b"]) < tol * 4
    inv_g, _ = lin.get_preconditioner()
    # the identity form cancels (Jp^T Jp - Q1d^T Q1d): one decade more in float32, see DESIGN.md section 2
    tb = TOLB[dtype] * (10 if kw.get("stage2_form") == "IDENTITY" and dtype == np.float32 else 1)
    assert max(rel_err(inv_g[c], dbg["inv_blocks"][c]) for c in range(lin.nc)) < tb
    x = np.random.default_rng(5).uniform(-1, 1, 9 * lin.nc).astype(dtype)
    assert rel_err(lin.right_multiply(x), o.right_multiply(x)) < tol * 4
    assert abs(lin.last_cg.num_iterations - dbg["cg_iterations"]) <= 2
    assert lin.last_cg.termination_type == dbg["cg_termination"]
    assert rel_err(inc_g, inc_c) < TOLS[dtype]
    l_g, l_c = lin.apply(inc_g), o.apply(inc_c)
    assert abs(l_g - l_c) <= 20 * TOLS[dtype] * abs(l_c)
    lin.download_state()
    cams_c, lms_c = o.get_state()
    assert rel_err(bp.lms, lms_c) < 10 * TOLS[dtype] and rel_err(bp.cams, cams_c) < TOLS[dtype]
    lin.close()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("which", ["small", "mixed"])
def test_implicit_operator_form(small_problem, mixed_problem, dtype, which):
    """operator_form=IMPLICIT (Jp^T Jp x - Q1d^T Q1d x from the per-observation records) against the oracle's dense
    Q2-panel product (ipp:400-441).  f64 at the single-stage tolerance; f32 one decade looser: the implicit form
    subtracts two nearly equal positive terms (DESIGN.md section 9)."""
    arrays = small_problem if which == "small" else mixed_problem
    bp, lin, o, _ = make_pair(arrays, dtype, operator_form="IMPLICIT")
    tol = TOL1[dtype] * (10 if dtype == np.float32 else 1)
    lin.linearize(); assert o.linearize()
    for lam in (0.1, 1e-4):
        inc_g = lin.solve(lam)
        inc_c, dbg = o.solve(lam, want_debug=True)
        x = np.random.default_rng(7).uniform(-1, 1, 9 * lin.nc).astype(dtype)
        assert rel_err(lin.right_multiply(x), o.right_multiply(x)) < tol * 4
        assert lin.last_cg.termination_type == dbg["cg_termination"]
        assert abs(lin.last_cg.num_iterations - dbg["cg_iterations"]) <= (2 if dtype == np.float64 else max(2, int(0.3 * dbg["cg_iterations"])))
        assert rel_err(inc_g, inc_c) < TOLS[dtype] * (5 if dtype == np.float32 else 1)
    l_g, l_c = lin.apply(inc_g), o.apply(inc_c)
    assert abs(l_g - l_c) <= 50 * TOLS[dtype] * abs(l_c)
    import rootba_b200 as rb
    with pytest.raises(rb.RbaError):  # no Q2 panels are stored in this mode
        lin.debug_get_block(0)
    dense = rb.LinearizorQR.create(rb.BalProblem.from_arrays(arrays, dtype), rb.SolverOptions())
    assert lin.stats()["device_bytes"] < dense.stats()["device_bytes"]
    dense.close()
    lin.close()


def test_long_tracks_generic_path():
    """track lengths beyond the register-resident classes (KP > 16) take the shared-memory matvec variant"""
    from rootba_b200.synthetic import synth_bal
    arrays = synth_bal(300, 120, 60.0, seed=4, max_track=300)
    assert arrays.track_lengths().max() > 113
    for dtype, hh in ((np.float32, True), (np.float64, True), (np.float64, False)):
        bp, lin, o, _ = make_pair(arrays, dtype, use_householder_marginalization=hh)
        lin.linearize(); assert o.linearize()
        inc_g = lin.solve(0.01)
        inc_c, _ = o.solve(0.01)
        x = np.random.default_rng(0).uniform(-1, 1, 9 * lin.nc).astype(dtype)
        assert rel_err(lin.right_multiply(x), o.right_multiply(x)) < TOL1[dtype] * 4
        assert rel_err(inc_g, inc_c) < TOLS[dtype]
        lin.close()


def test_minimal_tracks_and_ragged_tiles():
    """n = 2 only, landmark count not a multiple of the tile width"""
    from rootba_b200.synthetic import synth_bal
    arrays = synth_bal(9, 77, 2.0001, seed=2)
    assert arrays.track_lengths().max() <= 3
    bp, lin, o, _ = make_pair(arrays, np.float64)
    lin.linearize(); assert o.linearize()
    inc_g = lin.solve(1e-3); inc_c, _ = o.solve(1e-3)
    assert rel_err(inc_g, inc_c) < 1e-8
    lin.close()


def test_rejects_bad_input(small_problem):
    import rootba_b200 as rb
    a = small_problem
    # a landmark with a single observation: the reference LOG(FATAL)s (ipp:73-76); we return an error
    off = a.lm_off.copy()
    off[1] = off[0] + 1
    bp = rb.BalProblem(a.cams, a.lms, off, a.obs_cam, a.obs_xy)
    with pytest.raises(rb.RbaError):
        rb.LinearizorQR.create(bp, rb.SolverOptions())
    # solve before linearize is a protocol violation
    bp2 = rb.BalProblem.from_arrays(a)
    lin = rb.LinearizorQR.create(bp2, rb.SolverOptions())
    with pytest.raises(rb.RbaError):
        lin.solve(1e-4)
    lin.close()


def test_full_size_properties():
    """BASELINE configs[1] shape (ladybug-1723-156502, float32): size-independent properties"""
    import rootba_b200 as rb
    from rootba_b200.synthetic import synth_config
    arrays = synth_config("ladybug-1723")
    bp = rb.BalProblem.from_arrays(arrays, np.float32)
    so = rb.SolverOptions(use_double=False, max_num_iterations=3)
    lin = rb.LinearizorQR.create(bp, so)
    st = lin.stats()
    n = arrays.track_lengths()
    assert st["sum_n2"] == int((n * n).sum()) and st["num_observations_local"] == arrays.nobs  # bit-exact indexing
    e0 = lin.compute_error()
    assert e0["all"]["num_obs"] == arrays.nobs and e0["is_numerically_valid"]
    lin.linearize()
    lin.solve(1e-4)
    rng = np.random.default_rng(1)
    x = rng.uniform(-1, 1, 9 * lin.nc).astype(np.float32)
    y = rng.uniform(-1, 1, 9 * lin.nc).astype(np.float32)
    Hx, Hy = lin.right_multiply(x).astype(np.float64), lin.right_multiply(y).astype(np.float64)
    # symmetry, positive definiteness, linearity of the RCS operator
    assert abs(y @ Hx - x @ Hy) <= 1e-4 * (abs(y @ Hx) + abs(x @ Hy))
    assert x @ Hx > 0
    Hxy = lin.right_multiply((x + 2 * y).astype(np.float32)).astype(np.float64)
    assert rel_err(Hxy, Hx + 2 * Hy) < 1e-4
    # two runs of the deterministic scatter give bit-identical results
    assert np.array_equal(lin.right_multiply(x), lin.right_multiply(x))
    summ = rb.bundle_adjust_manual(bp, so, linearizor=lin)
    costs = [it["cost"]["all"]["error"] for it in summ["iterations"] if it.get("step_is_successful")]
    assert costs[-1] < 0.5 * costs[0]
    lin.close()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_lm_step_fused_equals_separate_calls(small_problem, dtype):
    """rba_lm_step ([linearize] + solve + backup + apply + compute_error, ONE host synchronisation; SURVEY 8f row 2) gives
    bit-identical results to the separate entry points, over accepted and rejected (restored) steps"""
    import rootba_b200 as rb
    so = rb.SolverOptions()
    bpa, bpb = rb.BalProblem.from_arrays(small_problem, dtype), rb.BalProblem.from_arrays(small_problem, dtype)
    a, b = rb.LinearizorQR.create(bpa, so), rb.LinearizorQR.create(bpb, so)
    lam = 1e-4
    new_point = True
    for it in range(5):
        reject = it == 2  # exercise restore in the middle
        if new_point:
            ea, eb = a.compute_error(), b.compute_error()
            assert ea == eb
            a.linearize()
        a.solve(lam, to_host=False)
        bpa.backup()
        l_a = a.apply(None)
        e_a = a.compute_error()
        r = b.lm_step(lam, new_point)
        assert not r["solve_failed"]
        assert (l_a == r["l_diff"]) or (np.isnan(l_a) and np.isnan(r["l_diff"]))
        assert e_a == r["cost"]
        assert a.last_cg.num_iterations == b.last_cg.num_iterations and a.last_cg.termination_type == b.last_cg.termination_type
        if reject:
            bpa.restore(); bpb.restore()
            lam *= 4
            new_point = False
        else:
            lam /= 3
            new_point = True
    a.download_state(); b.download_state()
    assert np.array_equal(bpa.cams, bpb.cams) and np.array_equal(bpa.lms, bpb.lms)
    # the cost before a new linearisation point is answered from the cache (no kernel launch), bit-identical
    l0 = b.timings()["kernel_launches"]
    assert b.compute_error() == r["cost"] and b.timings()["kernel_launches"] == l0
    a.close(); b.close()


@pytest.mark.parametrize("dtype,kw", [(np.float64, {}), (np.float32, {}), (np.float64, {"optimized_cost": "ERROR_VALID"}),
                                      (np.float32, {"robust_norm": "HUBER", "huber_parameter": 2.0})])
def test_native_lm_loop_equals_the_python_loop(small_problem, dtype, kw):
    """rba_lm_run (optimize_lm_ours inside the library, one host synchronisation per iteration) reproduces the Python mirror
    of the same loop (bundle_adjust_manual, separate entry points) bit for bit: cost, decisions, PCG iterations, final state"""
    import rootba_b200 as rb
    so = rb.SolverOptions(max_num_iterations=8)
    if "optimized_cost" in kw:
        so.optimized_cost = kw["optimized_cost"]
    if "robust_norm" in kw:
        so.residual.robust_norm, so.residual.huber_parameter = kw["robust_norm"], kw["huber_parameter"]
    bpa, bpb = rb.BalProblem.from_arrays(small_problem, dtype), rb.BalProblem.from_arrays(small_problem, dtype)
    summ = rb.bundle_adjust_manual(bpa, so)
    lin = rb.LinearizorQR.create(bpb, so)
    its, term, tot = lin.lm_run(64)
    py = summ["iterations"][1:]
    assert len(its) == len(py) and term == (summ["termination_type"] == "CONVERGENCE" or len(py) >= so.max_num_iterations)
    key = "all" if so.optimized_cost == "ERROR" else "valid"
    for a, b in zip(py, its):
        assert bool(a["step_is_successful"]) == b["accepted"], a["iteration"]
        assert a["linear_solver_iterations"] == b["cg_iterations"]
        assert a["cost"][key]["error"] == b["cost"], (a["iteration"], a["cost"][key]["error"], b["cost"])
        assert a["lam"] == b["lambda"]
    lin.download_state()
    assert np.array_equal(bpa.cams, bpb.cams) and np.array_equal(bpa.lms, bpb.lms)
    assert tot["solve_reduced_system_time"] > 0 and all(i["device_seconds"] > 0 for i in its)
    lin.close()


@pytest.mark.parametrize("config,dtype,kw", [
    ("ladybug-1723", np.float32, {}),                                      # BASELINE configs[1]
    ("trafalgar-257", np.float64, {"preconditioner_type": "JACOBI"}),      # BASELINE configs[2]
])
def test_full_size_against_oracle(config, dtype, kw):
    """GPU vs oracle on the BASELINE-size stand-ins: one linearize + solve + back-substitution (the oracle needs seconds)"""
    from rootba_b200.synthetic import synth_config
    arrays = synth_config(config)
    bp, lin, o, _ = make_pair(arrays, dtype, **kw)
    tol = TOL1[dtype]
    eg, ec = lin.compute_error(), o.compute_error()
    assert eg["all"]["num_obs"] == ec["all"]["num_obs"] == arrays.nobs
    assert abs(eg["all"]["error"] - ec["all"]["error"]) <= 20 * tol * ec["all"]["error"]
    lin.linearize(); assert o.linearize()
    assert rel_err(lin.get_jacobian_scaling()[0], o.get_scaling()) < tol
    lam = 1e-4
    inc_g = lin.solve(lam)
    inc_c, dbg = o.solve(lam, want_debug=True)
    assert rel_err(lin.get_rhs(), dbg["b"]) < tol * 4
    inv_g, _ = lin.get_preconditioner()
    assert max(rel_err(inv_g[c], dbg["inv_blocks"][c]) for c in range(lin.nc)) < TOLB[dtype]
    x = np.random.default_rng(9).uniform(-1, 1, 9 * lin.nc).astype(dtype)
    assert rel_err(lin.right_multiply(x), o.right_multiply(x)) < tol * 4
    assert abs(lin.last_cg.num_iterations - dbg["cg_iterations"]) <= 2
    assert rel_err(inc_g, inc_c) < TOLS[dtype]
    pose_inc = (np.random.default_rng(2).uniform(-1, 1, 9 * lin.nc) * 0.01).astype(dtype)
    l_g = lin.back_substitute(pose_inc)
    l_c, ok = o.back_substitute(pose_inc)
    assert ok and abs(l_g - l_c) <= tol * 20 * abs(l_c)
    lin.download_state()
    assert rel_err(bp.lms, o.get_state()[1]) < tol
    lin.close()


@pytest.mark.parametrize("dtype,kw", [
    (np.float64, {}),
    (np.float32, {}),
    (np.float64, {"preconditioner_type": "JACOBI"}),
    (np.float32, {"robust_norm": "HUBER", "huber_parameter": 2.0}),
    (np.float64, {"optimized_cost": "ERROR_VALID"}),
    (np.float64, {"use_householder_marginalization": False}),
    (np.float64, {"operator_form": "IMPLICIT"}),
])
def test_lm_trajectory(small_problem, dtype, kw):
    """The whole LM loop (host loop of the Python mirror driving the CUDA path) against the oracle's loop.

    float64 pins the trajectory: same number of logged iterations, every accept/reject decision, cost at 1e-9, PCG
    iterations +-2.  In float32 the function-tolerance stop (|dcost| <= 1e-6 cost, bal_bundle_adjustment.cpp:174-201) sits
    at the round-off level of the cost itself -- the float32 ORACLE needs 5, 6 or 9 logged iterations on these problems where
    the float64 oracle needs 6 (profiles/r2_f32_trajectory_diag.txt), and GPU-f32 / oracle-f32 / oracle-f64 costs agree to
    1e-6 .. 3e-6 on every iteration they share.  So float32 compares what is above that noise: the cost of every shared
    iteration at 1e-5 (SURVEY 8c allows 1e-4), decisions and PCG counts while the step still lowers the cost by more than
    1e-5 relative, and the final cost at 1e-5; the number of noise-level iterations at the end is not compared."""
    import rootba_b200 as rb
    bp, lin, o, so = make_pair(small_problem, dtype, max_num_iterations=8, **kw)
    summ = rb.bundle_adjust_manual(bp, so, linearizor=lin)
    rows, term = o.optimize()
    g_it = summ["iterations"]
    f32 = dtype == np.float32
    if not f32:
        assert len(g_it) == len(rows)
    tol = 1e-5 if f32 else 1e-9
    noise = 1e-5 if f32 else 0.0
    cost0 = rows[0]["cost"]
    prev = cost0
    compared = 0
    for a, b in zip(g_it, rows):
        assert a["iteration"] == int(b["iteration"])
        ca = a["cost"]["all"]["error"]
        assert abs(ca - b["cost"]) <= tol * b["cost"] + (1e-7 if f32 else 1e-12) * cost0, (a["iteration"], ca, b["cost"])
        significant = abs(prev - b["cost"]) > noise * prev
        if significant:
            compared += 1
            assert bool(a["step_is_successful"]) == bool(b["step_is_successful"]), a["iteration"]
            if a["iteration"] > 0:
                assert abs(a["linear_solver_iterations"] - int(b["cg_iterations"])) <= 2, a["iteration"]
        prev = b["cost"]
    assert compared >= 3
    assert g_it[-1]["cost"]["all"]["error"] < 0.2 * g_it[0]["cost"]["all"]["error"]
    best_g = min(it["cost"]["all"]["error"] for it in g_it if it.get("step_is_successful"))
    best_c = min(r["cost"] for r in rows if r["step_is_successful"])
    assert abs(best_g - best_c) <= max(tol, 1e-9) * best_c
    lin.close()
