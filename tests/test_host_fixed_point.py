"""The fixed-point cases of test_gpu_fixed_point.py at small shapes on the C-ABI emulator with its fixed-point entry
points (tests/cabi_emulator_fixed_point.py): host logic of BranchProgram.fixed_point, the fixed-point workspace and the
routing of iResBlock.inverse / RootFind.banach_find_root."""
import pytest

from tests import cabi_emulator_fixed_point
from tests import fixed_point_cases as cases
from tests import imblock_cases


@pytest.fixture(autouse=True)
def _emulated(monkeypatch):
    imblock_cases.DEV['device'] = 'cpu'
    lib = cabi_emulator_fixed_point.install(monkeypatch)
    yield lib
    imblock_cases.DEV['device'] = 'cuda'


@pytest.mark.parametrize('name', ['tile', 'gemm3_3'])
def test_conv_fixed_point_bitwise_vs_host_loop(name):
    cases.case_conv_bitwise(name)


@pytest.mark.parametrize('name', ['tile', 'gemm3_3'])
def test_conv_fixed_point_vs_oracle(name):
    cases.case_conv_oracle(name)


@pytest.mark.parametrize('name', ['b1', 'relu43'])
def test_mlp_fixed_point_vs_oracle(name):
    cases.case_mlp_oracle(name)


def test_mlp_fixed_point_beyond_kernel_limits():
    cases.case_mlp_beyond_limits('d129')


@pytest.mark.parametrize('rule', cases.STOP_RULES)
def test_conv_fixed_point_stopping_rules(rule):
    cases.case_conv_stop(rule)


@pytest.mark.parametrize('rule', cases.STOP_RULES)
def test_mlp_fixed_point_stopping_rules(rule):
    cases.case_mlp_stop(rule)


@pytest.mark.parametrize('kind', ['conv', 'mlp'])
def test_fixed_point_back_to_back(kind):
    cases.case_back_to_back(kind)


def test_mlp_residual_flow_inverse_round_trip():
    cases.case_module_round_trip('mlp', 64)


@pytest.mark.parametrize('kind', ['conv', 'mlp'])
def test_banach_find_root_on_compiled_branches(kind):
    cases.case_banach_find_root(kind)
