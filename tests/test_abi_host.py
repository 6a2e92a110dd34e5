"""CPU-side checks of the C-ABI library: it loads, exports every symbol include/b200kkt.h declares, refuses to
compute without a GPU (no fallback), and its host-side (symbolic) entry points agree with the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import madnlp_oracle as o
import madnlp_jl_b200 as pkg

capi = pkg.capi
lib = capi.lib
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "b200kkt.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(b2d?_[a-z0-9_]+)\s*\(", txt)))


def test_every_declared_symbol_is_exported_and_bound():
    syms = _header_symbols()
    assert len(syms) >= 50
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/b200kkt.h but not exported by libb200kkt.so"
        assert s in capi.PROTOTYPES, f"{s} has no ctypes prototype in capi.py"
    for s in capi.PROTOTYPES:
        assert s in syms, f"{s} bound in capi.py but not declared in the header"


def test_no_cpu_fallback_without_device():
    if capi.device_count() > 0:
        pytest.skip("a GPU is visible")
    colptr = np.array([0, 2, 3], dtype=np.int32); rowval = np.array([0, 1, 1], dtype=np.int32)
    h = C.c_void_p()
    opt = capi.default_options()
    rc = lib.b2_create(2, 3, colptr.ctypes.data, rowval.ctypes.data, None, C.byref(opt), None, C.byref(h))
    assert rc == capi.B2_ERR_NO_DEVICE and "no CPU fallback" in capi.last_error()
    with pytest.raises(capi.B2Error):
        capi.require_device()
    # a symbolic-only handle refuses every numeric call
    capi.check(lib.b2_create_symbolic_only(2, 3, colptr.ctypes.data, rowval.ctypes.data, C.byref(opt), None, C.byref(h)))
    assert lib.b2_factorize(h, None) == capi.B2_ERR_INVALID
    assert lib.b2_solve(h, None, 1, None) == capi.B2_ERR_INVALID
    lib.b2_destroy(h)


def test_options_default_and_errors():
    opt = capi.default_options()
    assert opt.ordering == capi.ORDER_METIS_ND and opt.use_cuda_graph == 1 and opt.n_parts == 1
    h = C.c_void_p()
    colptr = np.array([0, 1, 5], dtype=np.int32); rowval = np.array([0, 1], dtype=np.int32)
    assert lib.b2_create_symbolic_only(2, 2, colptr.ctypes.data, rowval.ctypes.data, C.byref(opt), None, C.byref(h)) == capi.B2_ERR_INVALID
    with pytest.raises(TypeError):
        capi.default_options(no_such_option=1)


@pytest.mark.parametrize("seed", [0, 1])
def test_coo_to_csc_matches_oracle(seed):
    """b2_coo_to_csc vs the restated src/matrixtools.jl:55-95 incl. duplicates, empty columns, unsorted input."""
    rng = np.random.default_rng(seed)
    m, n, nnz = 17, 13, 90
    I = rng.integers(0, m, nnz); J = rng.integers(0, n - 2, nnz)      # last two columns empty
    I[:5] = I[5:10]; J[:5] = J[5:10]                                   # guaranteed duplicates
    cp0, rv0, mp0 = o.coo_to_csc(I, J, m, n)
    I32, J32 = I.astype(np.int32), J.astype(np.int32)
    cp = np.zeros(n + 1, dtype=np.int32); rv = np.zeros(nnz, dtype=np.int32); mp = np.zeros(nnz, dtype=np.int64)
    k = C.c_int64(0)
    capi.check(lib.b2_coo_to_csc(m, n, nnz, I32.ctypes.data, J32.ctypes.data, cp.ctypes.data, rv.ctypes.data, mp.ctypes.data, C.byref(k)))
    assert k.value == len(rv0)
    assert (cp == cp0).all() and (rv[:k.value] == rv0).all() and (mp == mp0).all()
    # empty input
    capi.check(lib.b2_coo_to_csc(3, 3, 0, None, None, cp.ctypes.data, rv.ctypes.data, mp.ctypes.data, C.byref(k)))
    assert k.value == 0 and (cp[:4] == 0).all()
    # out-of-range index is rejected
    bad = np.array([99], dtype=np.int32)
    assert lib.b2_coo_to_csc(3, 3, 1, bad.ctypes.data, bad.ctypes.data, cp.ctypes.data, rv.ctypes.data, mp.ctypes.data, C.byref(k)) == capi.B2_ERR_INVALID


@pytest.mark.parametrize("case", ["hs15", "case30_synth", "case300_synth"])
def test_condensed_symbolic_matches_oracle(case):
    """b2_condensed_symbolic (pattern + map sizes) vs the restated build_condensed_aug_symbolic (condensed.jl:201-301)."""
    if case == "hs15":
        cb = o.HS15Model.callback()
    else:
        model, st = pkg.workloads.acopf_case(case)
        cb = o.Callback(st.nvar, st.ncon, st.jac_I, st.jac_J, st.hess_I, st.hess_J, st.ind_ineq, st.ind_lb, st.ind_ub)
    k = o.SparseCondensedKKTSystem(cb)
    h = C.c_void_p(); nnz = C.c_int64(0)
    capi.check(lib.b2_condensed_symbolic(k.n, k.m, k.hess_colptr.ctypes.data, k.hess_rowval.ctypes.data,
                                         k.jt_colptr.ctypes.data, k.jt_rowval.ctypes.data, C.byref(h), C.byref(nnz)))
    assert nnz.value == len(k.aug_rowval)
    cp = np.zeros(k.n + 1, dtype=np.int32); rv = np.zeros(nnz.value, dtype=np.int32)
    capi.check(lib.b2_condensed_pattern(h, cp.ctypes.data, rv.ctypes.data))
    assert (cp == k.aug_colptr).all() and (rv == k.aug_rowval).all()
    a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
    capi.check(lib.b2_condensed_plan_sizes(h, C.byref(a), C.byref(b), C.byref(c)))
    assert (a.value, b.value, c.value) == (len(k.dptr), len(k.hptr), len(k.jptr))
    lib.b2_condensed_plan_destroy(h)


def test_argument_validation_never_touches_the_device():
    """Invalid arguments are rejected on the host (B2_ERR_INVALID + message) before any CUDA call -- also on a box
    without a GPU; numeric calls on handles that were never created fail loudly instead of falling back."""
    E = capi.B2_ERR_INVALID
    assert lib.b2_copy_many(17, None, None, None, None) == E and b"16" in lib.b2_last_error()
    assert lib.b2_copy_many(1, None, None, None, None) == E
    assert lib.b2_copy_many(0, None, None, None, None) == capi.B2_OK
    assert lib.b2_richardson_update(-1, None, None, None, None, None) == E
    assert lib.b2_richardson_update(4, None, None, None, None, None) == E
    assert lib.b2_richardson_begin(4, None, None, None, None, None) == E
    assert lib.b2d_gemv_n(4, 4, 2, None, None, None, 1.0, 0.0, None) == E          # lda < rows
    assert lib.b2d_gemv_t(-1, 4, 4, None, None, None, 1.0, 0.0, None) == E
    assert lib.b2d_symv_lower(4, 4, None, None, None, 1.0, 0.0, None) == E
    assert lib.b2d_symv_lower(0, 0, None, None, None, 1.0, 0.0, None) == capi.B2_OK
    assert lib.b2_norm_inf(3, None, None, None) == E
    assert lib.b2_inertia_enqueue(None, None) != capi.B2_OK and lib.b2_inertia_fetch(None, None, None, None) != capi.B2_OK
    assert lib.b2d_inertia_enqueue(None, None) != capi.B2_OK and lib.b2d_inertia_fetch(None, None, None, None) != capi.B2_OK


from hypothesis import given, settings, strategies as st_  # noqa: E402


@settings(max_examples=100, deadline=None)
@given(n=st_.integers(min_value=1, max_value=40), m=st_.integers(min_value=0, max_value=50),
       dh=st_.floats(min_value=0.0, max_value=0.5), dj=st_.floats(min_value=0.0, max_value=0.4), seed=st_.integers(0, 10**6))
def test_condensed_symbolic_random_patterns(n, m, dh, dj, seed):
    """b2_condensed_symbolic on arbitrary H (lower) / Jt (n x m) patterns -- empty constraint columns, empty Hessian, dense
    columns -- gives the same lower-CSC pattern and map sizes as the restated build_condensed_aug_symbolic (condensed.jl:201-301)."""
    rng = np.random.default_rng(seed)

    def csc_of(mask):                                           # mask[row, col] -> (colptr, rowval) with sorted rows
        nrow, ncol = mask.shape
        cols, rows = np.nonzero(mask.T)
        colptr = np.zeros(ncol + 1, dtype=np.int32)
        np.add.at(colptr, cols + 1, 1)
        return np.cumsum(colptr).astype(np.int32), rows.astype(np.int32)

    hcp, hrv = csc_of(np.tril(rng.random((n, n)) < dh))
    jcp, jrv = csc_of(rng.random((n, m)) < dj)
    cp0, rv0, dptr, hptr, jptr = o.build_condensed_aug_symbolic(hcp, hrv, n, jcp, jrv, m)
    h = C.c_void_p(); nnz = C.c_int64(0)
    capi.check(lib.b2_condensed_symbolic(n, m, hcp.ctypes.data, hrv.ctypes.data if len(hrv) else None,
                                         jcp.ctypes.data, jrv.ctypes.data if len(jrv) else None, C.byref(h), C.byref(nnz)))
    assert nnz.value == len(rv0)
    cp = np.zeros(n + 1, dtype=np.int32); rv = np.zeros(max(nnz.value, 1), dtype=np.int32)
    capi.check(lib.b2_condensed_pattern(h, cp.ctypes.data, rv.ctypes.data))
    assert (cp == cp0).all() and (rv[:nnz.value] == rv0).all()
    a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
    capi.check(lib.b2_condensed_plan_sizes(h, C.byref(a), C.byref(b), C.byref(c)))
    assert (a.value, b.value, c.value) == (len(dptr), len(hptr), len(jptr))
    lib.b2_condensed_plan_destroy(h)


@settings(max_examples=100, deadline=None)
@given(m=st_.integers(1, 30), n=st_.integers(1, 30), nnz=st_.integers(0, 200), seed=st_.integers(0, 10**6))
def test_coo_to_csc_random(m, n, nnz, seed):
    """b2_coo_to_csc on arbitrary COO lists (duplicates, empty columns, any order) == src/matrixtools.jl:55-95 restated."""
    rng = np.random.default_rng(seed)
    I = rng.integers(0, m, nnz); J = rng.integers(0, n, nnz)
    cp0, rv0, mp0 = o.coo_to_csc(I, J, m, n)
    I32, J32 = I.astype(np.int32), J.astype(np.int32)
    cp = np.zeros(n + 1, dtype=np.int32); rv = np.zeros(max(nnz, 1), dtype=np.int32); mp = np.zeros(max(nnz, 1), dtype=np.int64)
    k = C.c_int64(0)
    capi.check(lib.b2_coo_to_csc(m, n, nnz, I32.ctypes.data if nnz else None, J32.ctypes.data if nnz else None,
                                 cp.ctypes.data, rv.ctypes.data, mp.ctypes.data, C.byref(k)))
    assert k.value == len(rv0) and (cp == cp0).all() and (rv[:k.value] == rv0).all() and (mp[:nnz] == mp0).all()


def test_reference_arm_runs_without_the_product_library():
    """bench.py --impl reference: one JSON line with the contract's keys, the requested --steps/--warmup, the same `config` dict the
    B200 arm prints, and NO import of the product package (whose __init__ loads libb200kkt.so) -- VERDICT r1 'fix the import so
    the record is clean'."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, json; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '3', '--warmup', '1', '--workload', 'case300_synth'];"
            "import bench; bench.main();"
            "bad = [m for m in sys.modules if m.startswith('madnlp_jl_b200') or m.startswith('madnlp.jl_b200')];"
            "print(json.dumps({'loaded_product_modules': bad}))")
    out = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    line, probe = json.loads(lines[0]), json.loads(lines[-1])
    assert probe["loaded_product_modules"] == []
    assert line["impl"] == "reference" and line["steps"] == 3 and line["warmup"] == 1 and line["metric"] == "ipm_iters_per_sec"
    for key in ("value", "unit", "n_gpus", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    import bench
    class A: workload = "case300_synth"; no_flush = False
    class S: nvar = line["config"]["n"]; ncon = line["config"]["m"]
    assert line["config"] == bench.config_of(A, S, 1)


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs DIR (reference arm): float64 .npy files of what the last of the --steps timed steps returned -- the same
    on every run (seeded inputs) and equal to a replay of exactly --warmup + --steps steps; --steps 0 is refused."""
    import subprocess, sys
    import bench
    cmd = [sys.executable, "bench.py", "--impl", "reference", "--steps", "3", "--warmup", "1", "--workload", "case300_synth"]
    got = []
    for name in ("a", "b"):
        out = subprocess.run(cmd + ["--dump-outputs", str(tmp_path / name)], cwd=ROOT, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-2000:]
        assert len([l for l in out.stdout.splitlines() if l.startswith("{")]) == 1
        assert sorted(os.listdir(tmp_path / name)) == ["direction.npy", "inertia.npy"]
        got.append({k: np.load(tmp_path / name / f"{k}.npy") for k in ("direction", "inertia")})
    for k in ("direction", "inertia"):
        assert got[0][k].dtype == np.float64 and np.array_equal(got[0][k], got[1][k]), k
    model, st, its = bench.make_workload("case300_synth")
    la = bench._cpu_replay(st)
    bench._cpu_run(la, its, 1, 3)
    assert np.array_equal(got[0]["direction"], la.d.full()) and tuple(got[0]["inertia"]) == tuple(la.last_inertia)
    out = subprocess.run([sys.executable, "bench.py", "--steps", "0"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode == 2 and "--steps" in out.stderr
