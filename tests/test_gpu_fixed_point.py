"""GPU parity of the one-call fixed-point solves (iResBlock / ResidualFlow inverse, the Banach fallback of RootFind):
the native conv runtime bit for bit against the host loop at every evaluation path and run-ahead depth, both solvers
against the float64 oracle, every way a solve ends, back-to-back and side-stream solves, and whole flows.  The cases
live in tests/fixed_point_cases.py."""
import pytest

from tests import fixed_point_cases as cases
from tests import solve_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _on_gpu():
    solve_cases.DEV['device'] = 'cuda'
    yield


@pytest.mark.parametrize('name', cases.CONV)
def test_conv_fixed_point_bitwise_vs_host_loop(name):
    cases.case_conv_bitwise(name)


@pytest.mark.parametrize('name', cases.CONV_ORACLE)
def test_conv_fixed_point_vs_oracle(name):
    cases.case_conv_oracle(name)


@pytest.mark.parametrize('name', cases.MLP)
def test_mlp_fixed_point_vs_oracle(name):
    cases.case_mlp_oracle(name)


@pytest.mark.parametrize('name', cases.MLP_BEYOND)
def test_mlp_fixed_point_beyond_kernel_limits(name):
    cases.case_mlp_beyond_limits(name)


@pytest.mark.parametrize('rule', cases.STOP_RULES)
def test_conv_fixed_point_stopping_rules(rule):
    cases.case_conv_stop(rule)


@pytest.mark.parametrize('rule', cases.STOP_RULES)
def test_mlp_fixed_point_stopping_rules(rule):
    cases.case_mlp_stop(rule)


@pytest.mark.parametrize('kind', ['conv', 'mlp'])
def test_fixed_point_back_to_back_and_side_stream(kind):
    cases.case_back_to_back(kind)


@pytest.mark.parametrize('kind,batch', [('conv', 8), ('mlp', 1000)])
def test_residual_flow_inverse_round_trip(kind, batch):
    cases.case_module_round_trip(kind, batch)


@pytest.mark.parametrize('kind,batch', [('conv', 8), ('mlp', 1000)])
def test_iresblock_inverse_makes_no_synchronising_torch_call(kind, batch):
    cases.case_no_sync(kind, batch)


@pytest.mark.parametrize('kind', ['conv', 'mlp'])
def test_banach_find_root_on_compiled_branches(kind):
    cases.case_banach_find_root(kind)
