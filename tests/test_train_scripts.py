"""The drop-in claim, executed: the reference's OWN train_toy.py and train_tabular.py run unmodified with
`impflow_b200.compat.install()` in front — model code (`lib.layers*`) resolves to this package, everything else
(`lib.utils`, `lib.optimizers`, `lib.toy_data`, ...) to the reference checkout the scripts live in.

CPU only: the C ABI is replaced by the numpy emulator (tests/cabi_emulator.py), plotting (matplotlib,
lib.visualize_flow) and the on-disk tabular datasets (lib.tabular needs h5py + downloaded data) are stubbed with
synthetic stand-ins.  The tests that run the reference's own scripts need its checkout (directory named by
IMPFLOW_REFERENCE_ROOT) and are skipped without one; the model-only test runs everywhere."""
import os
import runpy
import sys
import types
from unittest import mock

import numpy as np
import pytest
import torch

from tests import cabi_emulator

REF = os.environ.get('IMPFLOW_REFERENCE_ROOT', '')
needs_reference = pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, 'train_toy.py'))),
                                     reason='no reference checkout (set IMPFLOW_REFERENCE_ROOT)')


@pytest.fixture
def dropin(monkeypatch, tmp_path):
    cabi_emulator.install(monkeypatch)
    import impflow_b200
    saved = {k: v for k, v in sys.modules.items() if k == 'lib' or k.startswith('lib.')}
    impflow_b200.compat.install(REF or None)
    # plotting is not part of the path: matplotlib is absent from this image, lib.visualize_flow draws on it
    for name in ('matplotlib', 'matplotlib.pyplot'):
        monkeypatch.setitem(sys.modules, name, mock.MagicMock(name=name))
    viz = types.ModuleType('lib.visualize_flow')
    viz.visualize_transform = lambda *a, **k: None
    monkeypatch.setitem(sys.modules, 'lib.visualize_flow', viz)
    monkeypatch.setattr(sys, 'path', ([REF] if REF else []) + sys.path)
    monkeypatch.chdir(tmp_path)
    yield tmp_path
    impflow_b200.compat.uninstall()
    sys.modules.update(saved)


def _run(script, argv, monkeypatch):
    monkeypatch.setattr(sys, 'argv', [script] + argv)
    return runpy.run_path(os.path.join(REF, script), run_name='__main__')


@needs_reference
def test_train_toy_runs_on_the_package(dropin, monkeypatch):
    import impflow_b200
    ns = _run('train_toy.py', ['--arch', 'implicit', '--data', 'checkerboard', '--niters', '2', '--batch_size', '64',
                               '--test_batch_size', '64', '--dims', '16-16', '--nblocks', '2', '--act', 'sin',
                               '--brute-force', 'True', '--coeff', '0.99', '--n-lipschitz-iters', '20', '--vnorms',
                               '2222', '--save', str(dropin / 'toy')], monkeypatch)
    model = ns['model'].module
    blocks = [m for m in model.modules() if isinstance(m, impflow_b200.layers.imBlock)]
    assert len(blocks) == 2 and type(model) is impflow_b200.layers.SequentialFlow
    assert all('fwd' in b.solver_stats for b in blocks)                  # the package's solver ran
    assert ns['optim'].__name__ == 'lib.optimizers' and ns['optim'].__file__.startswith(REF)   # the rest: reference
    assert np.isfinite(ns['loss'].item()) and np.isfinite(ns['best_loss'])
    assert os.path.isfile(dropin / 'toy' / 'checkpt.pth')


def test_iresnet_arch_model_of_train_toy(dropin):
    """`--arch iresnet` (train_toy.py:205-223) cannot run in the reference itself: SequentialFlow passes restore=
    to iResBlock.forward (quirk #20) and the script's plotting hook dereferences `model.module` on an unwrapped
    model.  The same model built through the drop-in names trains and inverts here."""
    import lib.layers as layers
    blocks = [layers.iResBlock(torch.nn.Sequential(layers.base.get_linear(2, 16, coeff=0.9, n_iterations=5, domain=2,
                                                                         codomain=2),
                                                   layers.base.Swish(),
                                                   layers.base.get_linear(16, 2, coeff=0.9, n_iterations=5, domain=2,
                                                                          codomain=2)),
                               n_dist='geometric', brute_force=True, neumann_grad=False, grad_in_forward=False)
              for _ in range(2)]
    model = layers.SequentialFlow(blocks)
    x = torch.randn(32, 2)
    with torch.no_grad():
        model(x, restore=True)
    z, dlogp = model(x.requires_grad_(True), torch.zeros(32, 1))
    (-(dlogp.mean()) + z.pow(2).mean()).backward()
    assert all(p.grad is not None for n, p in model.named_parameters() if 'weight' in n)
    with torch.no_grad():
        assert float((model.inverse(z.detach()) - x).abs().max()) < 1e-3


def _fake_tabular():
    mod = types.ModuleType('lib.tabular')

    def get_tabular_datasets(name, root):
        d = {'power': 6, 'gas': 8, 'hepmass': 21, 'miniboone': 43, 'bsds300': 63}[name]
        g = torch.Generator().manual_seed(0)
        mk = lambda n: torch.utils.data.TensorDataset(torch.randn(n, d, generator=g), torch.zeros(n))
        return mk(128), mk(64), mk(64)
    mod.get_tabular_datasets = get_tabular_datasets
    return mod


@needs_reference
def test_train_tabular_runs_on_the_package(dropin, monkeypatch):
    import impflow_b200
    monkeypatch.setitem(sys.modules, 'lib.tabular', _fake_tabular())
    ns = _run('train_tabular.py', ['--data', 'power', '--nblocks', '2', '--dims', '16-16', '--act', 'sin', '--coeff',
                                   '0.99', '--vnorms', '2222', '--epsf', '1e-5', '--nepochs', '1', '--batchsize', '64',
                                   '--val-batchsize', '64', '--nworkers', '0', '--seed', '0', '--save',
                                   str(dropin / 'tab')], monkeypatch)
    model = ns['model']
    assert type(model) is impflow_b200.layers.SequentialFlow
    blocks = [m for m in model.modules() if isinstance(m, impflow_b200.layers.imBlock)]
    assert len(blocks) == 2 and all('fwd' in b.solver_stats for b in blocks)
    assert np.isfinite(ns['best_test_bpd'])
    assert type(ns['optimizer']).__module__ == 'lib.optimizers'           # the reference's vendored Adam drove it
    assert len(ns['ema'].shadow_params) > 0
    assert os.path.isfile(dropin / 'tab' / 'models' / 'most_recent.pth')


@needs_reference
def test_train_tabular_with_closed_form_norms(dropin, monkeypatch):
    """--vnorms 122f: the script's build_nnet (train_tabular.py:292-318) asks the factories for 1 -> 2 and 2 -> inf layers,
    i.e. LopLinear first and last, an induced 2 -> 2 layer in between; the blocks run through the module / autograd
    path, and the script's Lipschitz-constant logging reads the Lop layers' `scale` (train_tabular.py:565-571)."""
    import impflow_b200
    monkeypatch.setitem(sys.modules, 'lib.tabular', _fake_tabular())
    ns = _run('train_tabular.py', ['--data', 'power', '--nblocks', '1', '--dims', '16-16', '--act', 'swish', '--coeff',
                                   '0.9', '--vnorms', '122f', '--epsf', '1e-5', '--nepochs', '1', '--batchsize', '64',
                                   '--val-batchsize', '64', '--nworkers', '0', '--seed', '0', '--save',
                                   str(dropin / 'tab_lop')], monkeypatch)
    model = ns['model']
    kinds = [type(m).__name__ for m in model.modules() if hasattr(m, 'compute_weight') and '_copy' not in type(m).__name__]
    assert kinds.count('LopLinear') >= 2 and 'InducedNormLinear' in kinds, kinds
    blk = [m for m in model.modules() if isinstance(m, impflow_b200.layers.imBlock)][0]
    assert 'fwd' in blk.solver_stats and np.isfinite(ns['best_test_bpd'])
    lop = [m for m in model.modules() if isinstance(m, impflow_b200.layers.base.LopLinear)]
    assert all(float(m.scale) > 0 for m in lop)


@needs_reference
def test_all_four_script_preambles_import(dropin, monkeypatch):
    """Everything the four train scripts touch on `lib.layers` / `lib.layers.base` / `lib.implicit_flow` at
    import or model-construction time exists (train_toy.py:21-32, train_tabular.py:23-35, train_img.py:15-20,230,
    train_classification.py:84)."""
    import lib.layers as layers
    import lib.layers.base as base_layers
    from lib.implicit_flow import ACT_FNS, ImplicitFlow
    from lib.resflow import ResidualFlow
    import lib.optimizers as optim
    import lib.utils as utils
    from lib.lr_scheduler import CosineAnnealingWarmRestarts
    for name in ('Identity', 'FullSort', 'MaxMin', 'Swish', 'LipschitzCube', 'Sin', 'Zero', 'InducedNormConv2d',
                 'InducedNormLinear', 'SpectralNormConv2d', 'SpectralNormLinear', 'LopConv2d', 'LopLinear',
                 'get_linear', 'get_conv2d'):
        assert hasattr(base_layers, name), name
    for name in ('imBlock', 'iResBlock', 'SequentialFlow', 'ActNorm1d', 'ActNorm2d', 'MovingBatchNorm1d',
                 'MovingBatchNorm2d', 'CouplingBlock', 'Normalize', 'ZeroMeanTransform', 'LogitTransform',
                 'SqueezeLayer', 'InvertibleLinear', 'InvertibleConv2d'):
        assert hasattr(layers, name), name
    x = torch.randn(3, 4)
    np.testing.assert_allclose(base_layers.MaxMin()(x).numpy(),
                               torch.cat([x.view(3, 2, 2).max(2)[0], x.view(3, 2, 2).min(2)[0]], 1).numpy())
    assert torch.equal(base_layers.FullSort()(x), torch.sort(x, 1)[0])
    t = torch.tensor([-2., -0.5, 0.5, 2.])
    np.testing.assert_allclose(base_layers.LipschitzCube()(t).numpy(), [-2 + 2 / 3, -0.125 / 3, 0.125 / 3, 2 - 2 / 3],
                               rtol=1e-6)
    norm = layers.Normalize((0.4914, 0.4822, 0.4465), (0.2023, 0.1994, 0.2010))      # train_img.py:230
    img = torch.rand(2, 3, 4, 4)
    y, lp = norm(img, torch.zeros(2, 1))
    np.testing.assert_allclose(norm.inverse(y).numpy(), img.numpy(), atol=1e-6)
    np.testing.assert_allclose(lp.numpy(), np.full((2, 1), 16 * np.log([0.2023, 0.1994, 0.2010]).sum()), rtol=1e-5)
    assert callable(optim.Adam) and callable(utils.ExponentialMovingAverage) and callable(CosineAnnealingWarmRestarts)
    assert ImplicitFlow.__module__.startswith('impflow_b200') and issubclass(ResidualFlow, ImplicitFlow)
    assert set(ACT_FNS) >= {'softplus', 'elu', 'swish', 'identity', 'relu', 'sin', 'zero'}
