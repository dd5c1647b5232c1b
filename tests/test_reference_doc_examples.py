"""The two complete C programs of the reference's C-API documentation
(docs/cuopt/source/cuopt-c/lp-milp/lp-example.rst: `lp_example.c`, `lp_example_mps.c`), run against this repo's
library through the same cuOpt* calls: the problem built from arrays, and the documentation's sample MPS file
(tests/golden/mps/docs/lp_example_sample.mps).  Problem data and expected values are in tests/golden/c_api_problems.json;
the values are the documentation's own "You should see the following output" blocks: Termination status: Optimal (1),
Objective value: -0.360000, x1 = 1.800000, x2 = 0.000000."""
import pytest

from conftest import mps_path
from cuopt_b200 import capi
from test_reference_c_api_tests import SUCCESS, problem_data

pytestmark = pytest.mark.gpu


def solve_like_the_example(p, d):
    """cuOptCreateSolverSettings, absolute primal tolerance 1e-4, cuOptSolve, then what the example prints."""
    s = capi.Settings()
    assert capi.lib().cuOptSetFloatParameter(s.h, b"absolute_primal_tolerance", d["absolute_primal_tolerance"]) == SUCCESS
    sol = capi.solve(p, s)
    assert sol.return_code == SUCCESS, sol.error_string
    assert sol.solve_time >= 0.0
    assert sol.termination_status == d["expected_termination_status"]
    assert sol.objective_value == pytest.approx(d["expected_objective"], abs=d["objective_abs"])
    assert sol.primal() == pytest.approx(d["expected_primal"], abs=d["primal_abs"])


def test_lp_example_with_data():
    d = problem_data("doc_lp_example")
    p = capi.Problem.create_ranged(d["offsets"], d["indices"], d["values"], d["con_lb"], d["con_ub"], d["c"],
                                   d["var_lb"], d["var_ub"], maximize=d["maximize"],
                                   variable_types=d["variable_types"].encode())
    solve_like_the_example(p, d)


def test_lp_example_with_mps_file():
    p = capi.Problem.read(mps_path("docs/lp_example_sample.mps"))
    assert p.num_variables == 2
    solve_like_the_example(p, problem_data("doc_lp_example"))
