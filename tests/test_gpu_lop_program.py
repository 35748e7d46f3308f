"""Lop layers (LopLinear / LopConv2d, vnorms '122f') on the branch-program path with the real kernels: the reference's
30 layer cases, the image flows' widths against float64 autograd of compute_weight(), 122f branches against the module
/ autograd path, the route of their solves, and full-size 122f flows.  Host-logic twins on the C-ABI emulator:
tests/test_host_lop_program.py."""
import pytest

from tests import imblock_cases as cases
from tests import lop_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _on_gpu():
    cases.DEV['device'] = 'cuda'
    yield


def test_lop_golden_layers(golden):
    lop_cases.case_golden_layers(golden, 'cuda')


@pytest.mark.parametrize('shape', lop_cases.REAL_SHAPES)
@pytest.mark.parametrize('ties', [False, True])
def test_lop_layer_widths(shape, ties):
    lop_cases.case_real_widths('cuda', shape, ties)


@pytest.mark.parametrize('kind,c,hw', [('conv', 3, 32), ('conv', 12, 16), ('conv', 48, 8)])
def test_lop_conv_program_matches_module(kind, c, hw):
    lop_cases.case_program_matches_module(kind, c, 512, 8, 'cuda', hw=hw)


@pytest.mark.parametrize('d', [6, 63])
def test_lop_fc_program_matches_module(d):
    lop_cases.case_program_matches_module('fc', d, 128, 1000, 'cuda')


@pytest.mark.parametrize('kind', ['conv', 'mlp'])
def test_lop_block_solves_take_native_route(kind, monkeypatch):
    lop_cases.case_solves_take_native_route(kind, 'cuda', monkeypatch)


# the thresholds of tests/test_gpu_fullsize.py
@pytest.mark.parametrize('workload', ['cifar', 'tabular-power'])
def test_lop_full_size_round_trip(workload, monkeypatch):
    import bench
    from scripts import lop_bench
    vnorms = '122f'
    if workload == 'cifar':
        monkeypatch.setattr(bench, 'build_model', lambda pkg, wl, batch: lop_bench.cifar_flow(pkg, vnorms, batch))
    else:
        monkeypatch.setattr(bench, 'build_model', lambda pkg, wl, batch: lop_bench.power_flow(pkg, vnorms, scale_last=False))
    # (workload_round_trip scales the last layers as bench.py does)
    r = cases.workload_round_trip(workload)
    print(workload, vnorms, r)
    assert r['round_trip'] < 1e-4, r
    assert r['residual'] < 1e-5, r
    assert r['deterministic'], r
    assert len(r['fwd_nstep']) == r['blocks'] and len(r['inv_nstep']) == r['blocks'], r
