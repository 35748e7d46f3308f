"""Lop layers (LopLinear / LopConv2d, vnorms '122f') on the branch-program path, host logic on the C-ABI emulator
(tests/cabi_emulator_lop.py): the reference's 30 layer cases through the norm / prep / gradient-chain entry points,
the reference's 122f training step, 122f branches against the module path and the route of their solves.  The same cases at full widths on the GPU: tests/test_gpu_lop_program.py."""
import pytest

from tests import cabi_emulator_lop
from tests import imblock_cases as cases
from tests import lop_cases


@pytest.fixture(autouse=True)
def _emulated(monkeypatch):
    cases.DEV['device'] = 'cpu'
    lib = cabi_emulator_lop.install(monkeypatch)
    yield lib
    cases.DEV['device'] = 'cuda'


def test_lop_golden_layers(golden):
    lop_cases.case_golden_layers(golden, 'cpu')


def test_imblock_lop_train_on_program(golden, monkeypatch):
    """The reference's 122f block training step (golden tolerances) with its Lop layers prepared by the program path."""
    from impflow_b200 import ops
    calls = []
    norms = ops.lop_norms
    monkeypatch.setattr(ops, 'lop_norms', lambda *a, **k: calls.append(1) or norms(*a, **k))
    cases.case_imblock_lop_train(golden)
    assert calls


@pytest.mark.parametrize('ties', [False, True])
def test_lop_layer_widths(ties):
    lop_cases.case_real_widths('cpu', ('c3', 8, 24), ties)
    lop_cases.case_real_widths('cpu', ('c3', 24, 8), ties)
    lop_cases.case_real_widths('cpu', ('c1', 16, 16), ties)


@pytest.mark.parametrize('kind,c,idim,B', [('conv', 3, 32, 2), ('fc', 6, 32, 9), ('mlp', 6, 32, 9)])
def test_lop_program_matches_module(kind, c, idim, B):
    lop_cases.case_program_matches_module(kind, c, idim, B, 'cpu')


@pytest.mark.parametrize('kind', ['conv', 'mlp'])
def test_lop_block_solves_take_native_route(kind, monkeypatch):
    lop_cases.case_solves_take_native_route(kind, 'cpu', monkeypatch)
