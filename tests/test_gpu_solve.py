"""GPU parity of the one-call Broyden solves against the float64 oracle: the native conv runtime (both modes, every
evaluation path, every run-ahead depth), the persistent MLP kernels, every way a solve can end, and back-to-back
solves on one workspace.  The cases live in tests/solve_cases.py."""
import pytest

from tests import solve_cases as cases

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _on_gpu():
    cases.DEV['device'] = 'cuda'
    yield


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('name', list(cases.CONV))
def test_conv_solve_vs_oracle(name, mode):
    cases.case_conv_vs_oracle(name, mode)


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('name', list(cases.CONV) + list(cases.CONV_BENCH))
def test_conv_solve_runahead_bitwise(name, mode):
    cases.case_conv_runahead(name, mode)


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('name', cases.CONV_STOP)
@pytest.mark.parametrize('rule', cases.STOP_RULES)
def test_conv_solve_stopping_rules(rule, name, mode):
    cases.case_conv_stop(rule, name, mode)


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('rule', cases.STOP_RULES)
def test_mlp_solve_stopping_rules(rule, mode):
    if rule == 'zero_rows' and mode == 0:
        pytest.skip('the MLP kernel sums f in another order than prog.forward: no exactly-zero mode-0 row')
    cases.case_mlp_stop(rule, mode)


@pytest.mark.parametrize('name', cases.MLP_VJP)
def test_mlp_vjp_solve_vs_oracle(name):
    cases.case_mlp_vjp(name)


@pytest.mark.parametrize('name', cases.MLP_BEYOND)
def test_mlp_solve_beyond_kernel_limits(name):
    cases.case_mlp_beyond_limits(name)


@pytest.mark.parametrize('solver', cases.B2B_SOLVERS)
def test_back_to_back_solves_on_one_workspace(solver):
    cases.case_back_to_back(solver)
