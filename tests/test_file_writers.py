"""`user_problem_file` / `solution_file` (constants.h parameter names; the reference's solve_lp writes them around the
solve, cpp/src/linear_programming/solve.cu:586-601).  The MPS writer restates cpp/src/mip/problem/write_mps.cu; what it
writes is read back by this repo's reader AND, as recorded in tests/golden/writer_golden.json, by the reference's own
libmps_parser."""
import hashlib
import os

import numpy as np
import pytest

from conftest import load_golden, mps_path, problem_arrays
from cuopt_b200 import capi, lpgen


def write_via_solve(problem, path):
    """cuOptSolve writes the problem before it touches the GPU, so this works (and is tested) without one."""
    s = capi.Settings(method=capi.CUOPT_METHOD_PDLP, log_to_console=False, iteration_limit=1)
    s.set("user_problem_file", path)
    sol = capi.solve(problem, s)
    assert os.path.exists(path)
    return sol


def same_problem(a, b):
    assert np.array_equal(a["offsets"], b["offsets"]) and np.array_equal(a["indices"], b["indices"])
    assert np.array_equal(a["values"], b["values"])          # max_digits10: bit-exact round trip
    for k in ("c", "var_lb", "var_ub", "con_lb", "con_ub"):
        assert np.array_equal(a[k], b[k]), k
    assert a["maximize"] == b["maximize"]


@pytest.mark.parametrize("rel", ["linear_programming/afiro_original.mps", "linear_programming/good-max.mps",
                                 "linear_programming/good-mps-some-var-bounds.mps", "mip/sudoku.mps"])
def test_written_mps_reads_back_identically(tmp_path, rel):
    p = capi.Problem.read(mps_path(rel))
    out = str(tmp_path / "written.mps")
    write_via_solve(p, out)
    q = capi.Problem.read(out)
    a, b = problem_arrays(p), problem_arrays(q)
    # the writer walks A column by column: rows come back with their entries in column order, the set is the same
    import scipy.sparse as sp
    A = sp.csr_matrix((a["values"], a["indices"], a["offsets"]), shape=(len(a["con_lb"]), len(a["c"])))
    B = sp.csr_matrix((b["values"], b["indices"], b["offsets"]), shape=(len(b["con_lb"]), len(b["c"])))
    assert (A != B).nnz == 0
    for k in ("c", "var_lb", "var_ub", "con_lb", "con_ub"):
        assert np.array_equal(a[k], b[k]), k
    assert a["maximize"] == b["maximize"] and p.is_mip == q.is_mip


WRITER_LP = dict(m=300, n=250, nnz_per_row=5, seed=3)   # lpgen.sparse_lp: E / L / G rows, x >= 0


def lp_digests(m, n, offsets, indices, values, c, con_lb, con_ub, var_lb, var_ub):
    """Digests of an LP with its matrix in canonical CSR (a reader may order the entries of a row differently)."""
    import scipy.sparse as sp
    A = sp.csr_matrix((np.asarray(values, np.float64), indices, offsets), shape=(m, n))
    A.sort_indices()
    arrays = dict(offsets=A.indptr.astype(np.int64), indices=A.indices.astype(np.int64), values=A.data, c=c,
                  con_lb=con_lb, con_ub=con_ub, var_lb=var_lb, var_ub=var_ub)
    return {k: hashlib.sha256(np.ascontiguousarray(a, dtype=np.int64 if k in ("offsets", "indices") else np.float64)
                              .tobytes()).hexdigest()[:16] for k, a in arrays.items()}


def test_reference_parser_reads_what_we_write(tmp_path):
    # the reference's own libmps_parser read the file this writer writes for WRITER_LP back as exactly that LP
    # (tests/golden/writer_golden.json, scripts/gen_golden.py); the verdict holds for a byte-identical file
    gold = load_golden("writer_golden.json")
    lp = lpgen.sparse_lp(WRITER_LP["m"], WRITER_LP["n"], WRITER_LP["nnz_per_row"], seed=WRITER_LP["seed"])
    p = capi.Problem.create_ranged(lp.offsets, lp.indices, lp.values, lp.con_lb, lp.con_ub, lp.c, lp.var_lb, lp.var_ub)
    out = tmp_path / "written.mps"
    write_via_solve(p, str(out))
    assert hashlib.sha256(out.read_bytes()).hexdigest() == gold["file_sha256"]
    ref = gold["reference_parse"]
    assert (ref["m"], ref["n"]) == (lp.m, lp.n)
    assert ref["digests"] == lp_digests(lp.m, lp.n, lp.offsets, lp.indices, lp.values, lp.c, lp.con_lb, lp.con_ub,
                                        lp.var_lb, lp.var_ub)


def test_ranged_rows_are_written_like_the_reference_writes_them(tmp_path):
    # write_mps.cu:60-70, 109-140: a row with two finite, different bounds becomes 'L' with RHS = lower bound and
    # RANGES = upper - lower (flagged in file_writers.cpp: not the MPS convention for 'L' rows, kept for output parity)
    from test_capi_host import RANGED_LP as d
    p = capi.Problem.create_ranged(d["offsets"], d["indices"], d["values"], d["con_lb"], d["con_ub"], d["c"],
                                   d["var_lb"], d["var_ub"], maximize=True)
    out = str(tmp_path / "ranged.mps")
    write_via_solve(p, out)
    text = open(out).read()
    assert "OBJSENSE\n MAXIMIZE\n" in text
    assert " L  R2\n" in text and "    RHS1      R2 2\n" in text and "RANGES\n    RNG1      R2 6\n" in text
    assert " UP BOUND1    C0 10\n" in text and "ENDATA\n" in text


@pytest.mark.gpu
def test_solution_file(tmp_path):
    p = capi.Problem.read(mps_path("linear_programming/afiro_original.mps"))
    out = str(tmp_path / "afiro.sol")
    s = capi.Settings(method=capi.CUOPT_METHOD_PDLP, log_to_console=False)
    s.set("solution_file", out)
    sol = capi.solve(p, s)
    assert sol.termination_status == 1
    lines = open(out).read().splitlines()
    assert lines[0] == "# Status: Optimal"                      # solution_writer.cu:42
    assert lines[1].startswith("# Objective value: ")
    assert float(lines[1].split(": ")[1]) == sol.stats().primal_objective
    x = sol.primal()
    assert len(lines) == 2 + len(x)
    name, value = lines[2].split(" ")
    assert name == "X01" and float(value) == x[0]
