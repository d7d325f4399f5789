"""CPU-side checks of the C-ABI library: it loads without a GPU, exports every symbol the public header
declares, refuses to run without a device (no CPU fallback), and its host-only helpers work."""
import ctypes as C
import os

import numpy as np
import pytest

import rootba_b200 as rb
from rootba_b200 import _lib


def test_library_exports_every_declared_symbol():
    _lib.build()
    L = _lib.lib()
    syms = _lib.declared_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/rootba_b200.h but not exported"
    assert L.rba_abi_version() == 1


def test_no_cpu_fallback():
    """run in a child process with every device hidden, so that the check holds on a machine with a GPU too"""
    import subprocess
    import sys
    from conftest import ROOT
    code = ("import rootba_b200 as rb\n"
            "from rootba_b200.synthetic import synth_bal\n"
            "bp = rb.BalProblem.from_arrays(synth_bal(12, 300, 4.1, seed=1))\n"
            "try:\n"
            "    rb.LinearizorQR.create(bp, rb.SolverOptions())\n"
            "except rb.RbaError as e:\n"
            "    print('code', e.code)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split() == ["code", "-2"]  # RBA_ERR_NO_DEVICE


def test_partition_landmarks(small_problem):
    off = small_problem.lm_off
    n = np.diff(off).astype(np.float64)
    w = n * n + 4 * n
    for nranks in (1, 2, 3, 8):
        b = rb.partition_landmarks(off, nranks)
        assert b[0] == 0 and b[-1] == small_problem.nl and np.all(np.diff(b) >= 0)
        loads = np.array([w[b[r]:b[r + 1]].sum() for r in range(nranks)])
        assert loads.max() <= loads.mean() * 1.05 + w.max()


def test_default_opts_match_reference_defaults():
    o = _lib.SolverOpts()
    _lib.lib().rba_default_solver_opts(C.byref(o))
    # bal/solver_options.hpp: SCHUR_JACOBI, max 500 its, eta 0.1, Householder
    assert (o.preconditioner_type, o.max_linear_solver_iterations, o.eta, o.use_householder_marginalization) == (1, 500, 0.1, 1)
    assert o.residual_reset_period == 10 and o.nranks == 1


def test_default_lm_opts_match_reference_defaults():
    """rba_lm_run's schedule parameters default to SolverOptions' (bal/solver_options.hpp: trust region 1e4 in [1e-32, 1e16],
    vee 2 x 2, function tolerance 1e-6, 20 iterations, optimized_cost ERROR)"""
    o = _lib.LmOpts()
    _lib.lib().rba_default_lm_opts(C.byref(o))
    assert (o.initial_trust_region_radius, o.min_trust_region_radius, o.max_trust_region_radius) == (1e4, 1e-32, 1e16)
    assert (o.min_relative_decrease, o.initial_vee, o.vee_factor, o.function_tolerance) == (0.0, 2.0, 2.0, 1e-6)
    assert (o.max_num_iterations, o.optimized_cost) == (20, 0)
    # the Python mirror of the options carries the same defaults
    import rootba_b200 as rb
    so = rb.SolverOptions()
    assert (so.initial_trust_region_radius, so.min_trust_region_radius, so.max_trust_region_radius) == (1e4, 1e-32, 1e16)
    assert (so.initial_vee, so.vee_factor, so.function_tolerance, so.max_num_iterations) == (2.0, 2.0, 1e-6, 20)


@pytest.mark.parametrize("shape", [(12, 300, 4.1, 400), (150, 1500, 9.0, 150), (300, 120, 60.0, 300), (9, 77, 2.0001, 400)])
def test_layout_selftest(shape):
    """indexing is bit-exact: every observation lands in exactly one slot with its camera, row chunks tile every panel
    once, the camera-major CSRs cover every slot once, for 1, 2, 3 and 8 shards and both scalar classes"""
    from rootba_b200.synthetic import synth_bal
    nc, nl, mean_n, max_track = shape
    a = synth_bal(nc, nl, mean_n, seed=3, max_track=max_track)
    L = _lib.lib()
    off = np.ascontiguousarray(a.lm_off, np.int64)
    oc = np.ascontiguousarray(a.obs_cam, np.int32)
    xy = np.ascontiguousarray(a.obs_xy, np.float64)
    pv = _lib.ProblemView(a.nc, a.nl, a.nobs, off.ctypes.data, oc.ctypes.data, xy.ctypes.data)
    for nranks in (1, 2, 3, 8):
        for rank in range(nranks):
            for ssz in (4, 8):
                rc = L.rba_layout_selftest(C.byref(pv), rank, nranks, ssz)
                assert rc == 0, (nranks, rank, ssz, L.rba_last_error())


def test_layout_rejects_unsorted_and_short_tracks(tiny_problem):
    a = tiny_problem
    L = _lib.lib()
    off = np.ascontiguousarray(a.lm_off, np.int64)
    xy = np.ascontiguousarray(a.obs_xy, np.float64)
    oc = np.ascontiguousarray(a.obs_cam, np.int32).copy()
    oc[[0, 1]] = oc[[1, 0]]  # first landmark no longer ascending
    pv = _lib.ProblemView(a.nc, a.nl, a.nobs, off.ctypes.data, oc.ctypes.data, xy.ctypes.data)
    assert L.rba_layout_selftest(C.byref(pv), 0, 1, 8) != 0
    off2 = off.copy(); off2[1] = off2[0] + 1  # a landmark with one observation (reference: LOG(FATAL), ipp:73-76)
    oc2 = np.ascontiguousarray(a.obs_cam, np.int32)
    pv2 = _lib.ProblemView(a.nc, a.nl, a.nobs, off2.ctypes.data, oc2.ctypes.data, xy.ctypes.data)
    assert L.rba_layout_selftest(C.byref(pv2), 0, 1, 8) != 0


def test_header_is_plain_c_and_links(tmp_path):
    """the drop-in boundary is a C ABI: the header must compile as C99 (no C++ types), a C program must link and run
    against the library without a GPU, and the ctypes mirrors of the structs must have the C sizes"""
    import subprocess
    from conftest import ROOT
    structs = {"rba_problem_view": _lib.ProblemView, "rba_solver_opts": _lib.SolverOpts, "rba_residual_info": _lib.ResidualInfo,
               "rba_cg_summary": _lib.CgSummary, "rba_stage_timings": _lib.StageTimings, "rba_workload_stats": _lib.WorkloadStats,
               "rba_lm_step_result": _lib.LmStepResult, "rba_lm_opts": _lib.LmOpts, "rba_lm_iteration": _lib.LmIteration}
    src = tmp_path / "abi.c"
    src.write_text(
        '#include "rootba_b200.h"\n#include <stdio.h>\n'
        "int main(void) {\n  rba_solver_opts o;\n  rba_default_solver_opts(&o);\n"
        '  printf("%d %d", (int)rba_abi_version(), (int)o.max_linear_solver_iterations);\n'
        + "".join(f'  printf(" %d", (int)sizeof({n}));\n' for n in structs)
        + '  printf("\\n");\n  return 0;\n}\n')
    exe = str(tmp_path / "abi")
    libdir = os.path.join(ROOT, "rootba_b200")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                           "-L", libdir, "-lrootba_b200", "-Wl,-rpath," + libdir, "-o", exe])
    out = subprocess.check_output([exe], text=True).split()
    assert out[:2] == ["1", "500"]
    assert [int(v) for v in out[2:]] == [C.sizeof(t) for t in structs.values()], dict(zip(structs, out[2:]))
