"""The C-API TESTs of the reference (cpp/tests/linear_programming/c_api_tests/c_api_tests.cpp), run against this repo's
libcuopt.so through the raw C ABI: the same sequence of cuOpt* calls per TEST, the same problems and the same expected
return codes, termination statuses and objectives.  The problems and outcomes are stored in
tests/golden/c_api_problems.json, so the tests need nothing outside this repository.
Not reproduced: the time-limit fixture (its instances square41 / enlight_hard are not in the tree)."""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden, mps_path
from cuopt_b200 import capi

INF = float("inf")
SUCCESS, INVALID_ARGUMENT, MPS_FILE_ERROR, VALIDATION_ERROR = 0, 1, 2, 4
OPTIMAL, INFEASIBLE, ITERATION_LIMIT = 1, 2, 4
CUOPT_METHOD, CUOPT_TIME_LIMIT, CUOPT_ITERATION_LIMIT = b"method", b"time_limit", b"iteration_limit"


def problem_data(name):
    """One problem of c_api_problems.json with its arrays as numpy ('inf' / '-inf' as floats)."""
    d = dict(load_golden("c_api_problems.json")[name])
    for k in ("c", "values", "rhs", "con_lb", "con_ub", "var_lb", "var_ub"):
        if k in d:
            d[k] = np.array([float(v) for v in d[k]])
    for k in ("offsets", "indices"):
        d[k] = np.array(d[k], np.int32)
    return d


def create_problem(d):
    """cuOptCreateProblem (sense form) of a problem of c_api_problems.json, and the getter round trip that the
    reference's check_problem does right after it."""
    p = capi.Problem.create(d["offsets"], d["indices"], d["values"], d["sense"].encode(), d["rhs"], d["c"], d["var_lb"],
                            d["var_ub"], maximize=d["maximize"], objective_offset=d["objective_offset"],
                            variable_types=d["variable_types"].encode())
    m, n = len(d["rhs"]), len(d["c"])
    assert (p.num_constraints, p.num_variables, p.num_nonzeros) == (m, n, len(d["values"]))
    assert p.objective_sense == (capi.CUOPT_MAXIMIZE if d["maximize"] else capi.CUOPT_MINIMIZE)
    assert p.objective_offset == d["objective_offset"]
    np.testing.assert_array_equal(p.objective_coefficients(), d["c"])
    off, idx, val = p.constraint_matrix()
    np.testing.assert_array_equal(off, d["offsets"])
    np.testing.assert_array_equal(idx, d["indices"])
    np.testing.assert_array_equal(val, d["values"])
    assert p.constraint_sense() == d["sense"].encode()
    np.testing.assert_array_equal(p.rhs(), d["rhs"])
    np.testing.assert_array_equal(p.variable_lower_bounds(), d["var_lb"])
    np.testing.assert_array_equal(p.variable_upper_bounds(), d["var_ub"])
    assert p.variable_types() == d["variable_types"].encode()
    return p


def solve_mps_file(path, time_limit, iteration_limit, method):
    """Read an MPS file, set method and time limit (and the iteration limit when finite), solve.
    Returns (return code of the first call that failed or of cuOptSolve, termination status or -1)."""
    L = capi.lib()
    p = capi.Problem.read(path)
    p.is_mip  # noqa: B018  (capi raises when cuOptIsMIP fails)
    s = capi.Settings()
    assert L.cuOptSetIntegerParameter(s.h, CUOPT_METHOD, method) == SUCCESS
    assert L.cuOptSetFloatParameter(s.h, CUOPT_TIME_LIMIT, time_limit) == SUCCESS
    if iteration_limit < INF:
        assert L.cuOptSetIntegerParameter(s.h, CUOPT_ITERATION_LIMIT, int(iteration_limit)) == SUCCESS
    sol = capi.solve(p, s)
    if sol.return_code != SUCCESS:
        return sol.return_code, -1
    assert sol.solve_time >= 0.0
    status = sol.termination_status
    sol.objective_value  # noqa: B018  (capi raises when cuOptGetObjectiveValue fails)
    return SUCCESS, status


# ---- no GPU needed -------------------------------------------------------------------------------------------
def test_int_and_float_size():               # TEST(c_api, int_size) / TEST(c_api, float_size)
    assert capi.lib().cuOptGetIntSize() == 4 and capi.lib().cuOptGetFloatSize() == 8


def test_missing_file(tmp_path):             # TEST(c_api, test_missing_file)
    L = capi.lib()
    h = C.c_void_p()
    assert L.cuOptReadProblem(str(tmp_path / "missing_file.mps").encode(), C.byref(h)) == MPS_FILE_ERROR
    L.cuOptDestroyProblem(C.byref(h))        # destroying the handle a failed read left is allowed


def test_bad_parameter_name():               # TEST(c_api, bad_parameter_name): every setter and getter refuses it
    L = capi.lib()
    s = capi.Settings()
    name, buf, i, f = b"bad_parameter_name", C.create_string_buffer(64), C.c_int32(), C.c_double()
    assert L.cuOptSetParameter(s.h, name, b"1") == INVALID_ARGUMENT
    assert L.cuOptGetParameter(s.h, name, 64, buf) == INVALID_ARGUMENT
    assert L.cuOptSetIntegerParameter(s.h, name, 1) == INVALID_ARGUMENT
    assert L.cuOptSetFloatParameter(s.h, name, 1.0) == INVALID_ARGUMENT
    assert L.cuOptGetIntegerParameter(s.h, name, C.byref(i)) == INVALID_ARGUMENT
    assert L.cuOptGetFloatParameter(s.h, name, C.byref(f)) == INVALID_ARGUMENT


def test_burglar_is_a_mip_and_is_refused():  # TEST(c_api, burglar) expects SUCCESS from the reference's MIP solver;
    p = create_problem(problem_data("burglar"))
    assert p.is_mip
    s = capi.Settings()
    s.get_str("time_limit")
    assert capi.solve(p, s).return_code == VALIDATION_ERROR  # this LP-only build refuses before touching the GPU


# ---- on the GPU ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_afiro():                            # TEST(c_api, afiro): method DUAL_SIMPLEX, 60 s, no iteration limit
    rc, status = solve_mps_file(mps_path("linear_programming/afiro_original.mps"), 60.0, INF,
                                capi.CUOPT_METHOD_DUAL_SIMPLEX)
    assert rc == SUCCESS and status == OPTIMAL


@pytest.mark.gpu
def test_iteration_limit():                  # TEST(c_api, iteration_limit)
    rc, status = solve_mps_file(mps_path("linear_programming/afiro_original.mps"), 60.0, 1.0,
                                capi.CUOPT_METHOD_DUAL_SIMPLEX)
    assert rc == SUCCESS and status == ITERATION_LIMIT


@pytest.mark.gpu
def test_infeasible_problem():               # TEST(c_api, test_infeasible_problem): checks the status itself
    d = problem_data("infeasible")
    p = create_problem(d)
    s = capi.Settings()
    assert capi.lib().cuOptSetIntegerParameter(s.h, CUOPT_METHOD, capi.CUOPT_METHOD_DUAL_SIMPLEX) == SUCCESS
    sol = capi.solve(p, s)
    assert sol.return_code == SUCCESS
    assert sol.solve_time >= 0.0
    assert sol.termination_status == d["expected_termination_status"] == INFEASIBLE
    sol.objective_value  # noqa: B018  (capi raises when cuOptGetObjectiveValue fails)


@pytest.mark.gpu
def test_ranged_problem():                   # TEST(c_api, test_ranged_problem)
    d = problem_data("ranged")
    p = capi.Problem.create_ranged(d["offsets"], d["indices"], d["values"], d["con_lb"], d["con_ub"], d["c"],
                                   d["var_lb"], d["var_ub"], maximize=d["maximize"],
                                   variable_types=d["variable_types"].encode())
    np.testing.assert_array_equal(p.constraint_lower_bounds(), d["con_lb"])
    np.testing.assert_array_equal(p.constraint_upper_bounds(), d["con_ub"])
    s = capi.Settings()
    assert capi.lib().cuOptSetIntegerParameter(s.h, CUOPT_METHOD, capi.CUOPT_METHOD_DUAL_SIMPLEX) == SUCCESS
    sol = capi.solve(p, s)
    assert sol.return_code == SUCCESS
    assert sol.termination_status == d["expected_termination_status"] == OPTIMAL
    assert sol.objective_value == pytest.approx(d["expected_objective"], abs=d["objective_abs"])
