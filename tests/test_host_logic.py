"""CPU tests of the product's HOST logic (autograd wiring of the kernel primitives, conv-as-GEMM
weight layouts, Broyden host loop, RNG / roulette handling, state-dict compatibility) with the
C ABI replaced by the numpy emulator in tests/cabi_emulator.py.  The same cases run against the
real kernels in test_gpu_imblock.py."""
import numpy as np
import pytest
import torch

from tests import branch_cases, cabi_emulator
from tests import imblock_cases as cases
from tests.helpers import rel_err


@pytest.fixture(autouse=True)
def _emulated(monkeypatch):
    cases.DEV['device'] = 'cpu'
    lib = cabi_emulator.install(monkeypatch)
    yield lib
    cases.DEV['device'] = 'cuda'


@pytest.mark.parametrize('tag', list(cases.MLP))
def test_imblock_mlp_train(golden, tag):
    cases.case_imblock_mlp_train(golden, tag)


@pytest.mark.parametrize('tag', ['tab6'])
def test_imblock_mlp_train_reference_rng(golden, tag):
    cases.case_imblock_mlp_train_reference_rng(golden, tag)


@pytest.mark.parametrize('tag', ['tab6', 'tab43'])
def test_imblock_mlp_eval_and_inverse(golden, tag):
    cases.case_imblock_mlp_eval_and_inverse(golden, tag)


@pytest.mark.parametrize('tag', list(cases.CONV))
@pytest.mark.parametrize('backend', ['simt', 'tc'])
def test_imblock_conv_train(golden, tag, backend):
    cases.case_imblock_conv_train(golden, tag, backend)


def test_imblock_classifier_block(golden):
    cases.case_imblock_classifier_block(golden)


def test_imblock_conv_train_unfused(golden):
    """Same parity through the module / autograd path (graph-free branch programs switched off)."""
    from impflow_b200.layers import implicit_block
    implicit_block.FUSED['on'] = False
    try:
        cases.case_imblock_conv_train(golden, 'cifar', 'simt')
        cases.case_imblock_classifier_block(golden)
    finally:
        implicit_block.FUSED['on'] = True


def test_implicit_flow_density_step(golden):
    cases.case_implicit_flow_density_step(golden)


def test_mlp_solver_per_layer_beta():
    cases.case_mlp_solver_per_layer_beta()


def test_direct_grad_sink_matches_autograd(golden):
    cases.case_direct_grad_sink_matches_autograd(golden)


@pytest.mark.parametrize('tag', list(cases.IRES))
def test_iresblock(golden, tag):
    cases.case_iresblock(golden, tag)


def test_imblock_banach_fallback(golden):
    cases.case_imblock_banach_fallback(golden)


@pytest.mark.parametrize('tag', list(cases.EDGE))
def test_imblock_edge_train(golden, tag):
    cases.case_imblock_edge_train(golden, tag)


def test_imblock_fc_tail(golden):
    cases.case_imblock_fc_tail(golden)


def test_fused_adam_matches_reference_golden(golden):
    cases.case_fused_adam_matches_reference_golden(golden)


@pytest.mark.parametrize('tag', ['small', 'wide', 'capped', 'protbreak'])
def test_broyden_host_loop(golden, tag):
    import impflow_b200
    fx = golden('broyden_analytic')
    B, d, T, eps, scale, gain = fx[tag + '_meta']
    W, c = torch.from_numpy(fx[tag + '_W']), torch.from_numpy(fx[tag + '_c'])
    g = (lambda x: c - float(scale) * torch.tanh(x @ W) - x) if gain < 0 else (lambda x: c + float(gain) * x)
    res = impflow_b200.layers.broyden.broyden(g, torch.zeros(int(B), int(d)), int(T), float(eps))
    nstep, lowest_step, prot = fx[tag + '_ints']
    assert (res['nstep'], res['lowest_step'], int(res['prot_break'])) == (nstep, lowest_step, prot)
    assert rel_err(res['result'], fx[tag + '_result']) < 1e-5
    assert len(res['trace']) == nstep + 1


def test_state_dict_keys_match_reference(golden):
    """Key-for-key state-dict compatibility with the reference modules (SURVEY.md §5 checkpoint row)."""
    import impflow_b200
    layers = impflow_b200.layers
    fx = golden('imblock_mlp')
    blk = cases.make_mlp_block('tab6')
    ref_keys = sorted(k[len('tab6_sd_'):] for k in fx if k.startswith('tab6_sd_'))
    assert sorted(blk.state_dict().keys()) == ref_keys
    fx = golden('imblock_conv')
    blk = layers.imBlock(cases.build_conv_branch(layers, 4, 32, 0.9, 1e-3, True),
                         cases.build_conv_branch(layers, 4, 32, 0.9, 1e-3, True))
    ref_keys = sorted(k[len('cifar_sd_'):] for k in fx if k.startswith('cifar_sd_'))
    assert sorted(blk.state_dict().keys()) == ref_keys
    assert 'geom_p' not in blk.state_dict() and 'lamb' in blk.state_dict()       # quirk #12


def test_compat_install_registers_reference_import_names():
    import impflow_b200
    impflow_b200.compat.install()
    import lib.layers as L
    import lib.layers.base as BL
    from lib.implicit_flow import ImplicitFlow
    from lib.layers.broyden import broyden
    assert L.imBlock is impflow_b200.layers.imBlock and BL.get_conv2d is impflow_b200.layers.base.get_conv2d
    assert ImplicitFlow is impflow_b200.ImplicitFlow and callable(broyden)
    import sys
    for k in [k for k in sys.modules if k == 'lib' or k.startswith('lib.')]:
        del sys.modules[k]


def test_induced_norm_layers_vs_golden(golden):
    import impflow_b200
    BL = impflow_b200.layers.base
    fx = golden('induced_norm')
    lin = BL.InducedNormLinear(6, 16, coeff=0.5, domain=2, codomain=2, atol=1e-3, rtol=1e-3)
    lin.load_state_dict({k[len('lin_init_'):]: torch.from_numpy(v) for k, v in fx.items() if k.startswith('lin_init_')})
    with torch.no_grad():
        lin.weight.copy_(torch.from_numpy(fx['lin_weight2']))
    W = lin.compute_weight(update=True)
    np.testing.assert_allclose(W.detach().numpy(), fx['lin_W_tol'], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(lin.scale.numpy(), fx['lin_scale_tol'], rtol=1e-5)
    W = lin.compute_weight(update=True, n_iterations=5)
    np.testing.assert_allclose(W.detach().numpy(), fx['lin_W_it5'], rtol=1e-5, atol=1e-6)
    y = lin(torch.from_numpy(fx['lin_x']))
    np.testing.assert_allclose(y.detach().numpy(), fx['lin_y'], rtol=1e-4, atol=1e-5)
    lin.zero_grad()
    lin(torch.from_numpy(fx['lin_x'])).pow(2).sum().backward()
    np.testing.assert_allclose(lin.weight.grad.numpy(), fx['lin_grad_weight'], rtol=1e-3, atol=1e-5)

    conv = BL.InducedNormConv2d(5, 8, 3, 1, 1, coeff=0.4, domain=2, codomain=2, atol=1e-3, rtol=1e-3)
    x = torch.from_numpy(fx['conv_x'])
    with torch.no_grad():
        conv(x)
    conv.load_state_dict({k[len('conv_init_'):]: torch.from_numpy(v) for k, v in fx.items() if k.startswith('conv_init_')})
    np.testing.assert_allclose(conv(x).detach().numpy(), fx['conv_y'], rtol=1e-4, atol=1e-5)
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(fx['conv_weight2']))
    W = conv.compute_weight(update=True)
    np.testing.assert_allclose(conv.u.numpy(), fx['conv_u_tol'], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(W.detach().numpy(), fx['conv_W_tol'], rtol=1e-5, atol=1e-6)
    conv.zero_grad()
    conv(x).pow(2).sum().backward()
    np.testing.assert_allclose(conv.weight.grad.numpy(), fx['conv_grad_weight'], rtol=2e-3, atol=1e-4)

    c1 = BL.InducedNormConv2d(8, 8, 1, 1, 0, coeff=0.3, domain=2, codomain=2, atol=1e-3, rtol=1e-3)
    x = torch.from_numpy(fx['c1_x'])
    with torch.no_grad():
        c1(x)
    c1.load_state_dict({k[len('c1_init_'):]: torch.from_numpy(v) for k, v in fx.items() if k.startswith('c1_init_')})
    np.testing.assert_allclose(c1(x).detach().numpy(), fx['c1_y'], rtol=1e-4, atol=1e-5)
    with torch.no_grad():
        c1.weight.copy_(torch.from_numpy(fx['c1_weight2']))
    W = c1.compute_weight(update=True)
    np.testing.assert_allclose(W.detach().numpy(), fx['c1_W_tol'], rtol=1e-5, atol=1e-6)


def test_mixed_norm_layers_vs_golden(golden):
    cases.case_mixed_norm_layers(golden)


def test_learn_p_flow_state_dict(golden):
    cases.case_learn_p_flow_state_dict(golden)


@pytest.mark.parametrize('name', branch_cases.NAMES)
@pytest.mark.parametrize('backend', ['simt', 'tc'])
def test_branch_program_matches_module_autograd(name, backend):
    branch_cases.case_matches_module_autograd(name, backend)


def test_branch_program_rejects_unknown_modules():
    from impflow_b200.branch_program import compile_branch
    assert compile_branch(torch.nn.Sequential(torch.nn.Linear(3, 3))) is None
    assert compile_branch(torch.nn.Tanh()) is None


@pytest.mark.parametrize('name', branch_cases.NAMES)
@pytest.mark.parametrize('backend', ['simt', 'tc'])
def test_branch_program_gradients_match_autograd(name, backend):
    branch_cases.case_gradients_match_autograd(name, backend)


def test_fused3_tile_kernel_is_taken():
    assert branch_cases.case_fused3_is_taken('fused3_lead') == 2       # forward + vjp
    assert branch_cases.case_fused3_is_taken('fused3_512') == 2
    assert branch_cases.case_fused3_is_taken('cifar_lead') == 0        # width 32: three GEMMs


def test_fused_paths_are_taken(golden, monkeypatch, _emulated):
    """Guards against silently falling back to the module/autograd path: one CIFAR-style training
    forward+backward must run the Neumann gradient, the attach backward and all vjps on the
    graph-free branch programs and never build an autograd graph through the branch."""
    import impflow_b200
    from impflow_b200 import branch_program as bp
    from impflow_b200.layers import implicit_block as ib
    counts = {'neumann': 0, 'backward_full': 0, 'vjp': 0, 'autograd_estimator': 0, 'module_calls': 0, 'chain': 0,
              'solve': 0}

    def wrap(cls, name, key):
        orig = getattr(cls, name)

        def f(*a, **k):
            counts[key] += 1
            return orig(*a, **k)
        monkeypatch.setattr(cls, name, f)
    wrap(bp.BranchProgram, 'neumann', 'neumann')
    wrap(bp.BranchProgram, 'backward_full', 'backward_full')
    wrap(bp.BranchProgram, 'vjp', 'vjp')
    wrap(_emulated, 'impflow_conv3_power_series', 'chain')
    wrap(_emulated, 'impflow_conv3_broyden', 'solve')
    orig_est = ib.neumann_logdet_estimator
    monkeypatch.setattr(ib, 'neumann_logdet_estimator',
                        lambda *a, **k: (counts.__setitem__('autograd_estimator', counts['autograd_estimator'] + 1),
                                         orig_est(*a, **k))[1])
    fx = golden('imblock_conv')
    layers = impflow_b200.layers
    blk = layers.imBlock(cases.build_conv_branch(layers, 4, 32, 0.9, 1e-3, True),
                         cases.build_conv_branch(layers, 4, 32, 0.9, 1e-3, True), **cases.CONV['cifar']['kw'])
    blk = cases.load_block(blk, fx, 'cifar', torch.from_numpy(fx['cifar_x']))
    hook = lambda m, i: counts.__setitem__('module_calls', counts['module_calls'] + 1)
    hs = [blk.nnet_x.register_forward_pre_hook(hook), blk.nnet_z.register_forward_pre_hook(hook)]
    cases.run_train(blk, fx, 'cifar')
    for h in hs:
        h.remove()
    assert counts['neumann'] == 2 and counts['backward_full'] == 2
    assert counts['autograd_estimator'] == 0 and counts['module_calls'] == 0
    # the vjp chains and both solves run inside the native runtime (one C call each): csrc/conv3_plan.cu
    assert counts['chain'] == 2 and counts['solve'] >= 2 and counts['vjp'] == 1      # 1: dl_dx = v^T (I + J_x)


def test_update_lipschitz_batched_dense():
    cases.case_update_lipschitz_batched_dense()


def test_workload_round_trip_reduced():
    """The full-size GPU property test (tests/test_gpu_fullsize.py) at a reduced size on the emulator."""
    r = cases.workload_round_trip('cifar-small', batch=2)
    print(r)
    assert r['round_trip'] < 1e-3 and r['residual'] < 1e-4 and r['deterministic'], r
    r = cases.workload_round_trip('tabular-power', batch=16)
    print(r)
    assert r['round_trip'] < 1e-3 and r['residual'] < 1e-4 and r['deterministic'], r


def test_lop_layers(golden):
    cases.case_lop_layers(golden)


def test_imblock_lop_train(golden):
    cases.case_imblock_lop_train(golden)


def test_flow_options(golden):
    cases.case_flow_options(golden)


def test_sigma_cache_follows_power_iteration():
    cases.case_sigma_cache_follows_power_iteration()


def test_training_trajectory_matches_oracle(golden):
    cases.case_training_trajectory_matches_oracle(golden)


def test_fused_adam_matches_reference_step():
    cases.case_fused_adam_matches_reference_step()


def test_imblock_without_saved_forward_memo(golden):
    """Same goldens with the saved-forward memo switched off (every use re-evaluates the branch)."""
    from impflow_b200 import branch_program
    branch_program.MEMO['on'] = False
    try:
        cases.case_imblock_conv_train(golden, 'cifar', 'tc')
    finally:
        branch_program.MEMO['on'] = True


def test_saved_forward_memo_is_hit(golden, monkeypatch):
    """One training forward+backward of a conv imBlock evaluates each branch's saved forward once per distinct
    point: nnet_x at x (x_embed, re-attach, estimate share it), nnet_z at z* and at z (estimate and implicit
    backward share it)."""
    from impflow_b200 import branch_program as bp
    calls = []
    orig = bp.BranchProgram._forward_saved_impl

    def counted(self, rows, meta, M, ws, save):
        calls.append(save)
        return orig(self, rows, meta, M, ws, save)
    monkeypatch.setattr(bp.BranchProgram, '_forward_saved_impl', counted)
    cases.case_imblock_conv_train(golden, 'cifar', 'tc')
    n_saved = sum(1 for s in calls if s)
    bp.MEMO['on'] = False
    try:
        del calls[:]
        cases.case_imblock_conv_train(golden, 'cifar', 'tc')
    finally:
        bp.MEMO['on'] = True
    assert n_saved < sum(1 for s in calls if s)


def test_wide_conv_block_vs_oracle():
    cases.case_wide_conv_block_vs_oracle(verbose=True)


def test_actnorm_fused_matches_expression():
    from tests import imblock_cases
    imblock_cases.case_actnorm_fused_matches_expression()


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('name', ['tile', 'chain23_8', 'gemm3_3'])
def test_solve_conv_vs_oracle(name, mode):
    """The solver-level cases of test_gpu_solve.py at small shapes: one-call conv solve against the float64 oracle."""
    from tests import solve_cases
    solve_cases.case_conv_vs_oracle(name, mode)


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('rule', ['cap', 'cap_roundoff', 'prot_break', 'zero_rows'])
def test_solve_conv_stopping_rules(rule, mode):
    from tests import solve_cases
    solve_cases.case_conv_stop(rule, 'tile_small', mode)


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('rule', ['cap', 'cap_roundoff', 'prot_break'])
def test_solve_mlp_stopping_rules(rule, mode):
    from tests import solve_cases
    solve_cases.case_mlp_stop(rule, mode)


def test_solve_mlp_vjp_and_limits():
    from tests import solve_cases
    solve_cases.case_mlp_stop('zero_rows', 1)
    solve_cases.case_mlp_vjp('b1')
    solve_cases.case_mlp_vjp('relu43')
    solve_cases.case_mlp_beyond_limits('d129')


@pytest.mark.parametrize('solver', ['conv', 'mlp', 'rows'])
def test_solve_back_to_back_on_one_workspace(solver):
    from tests import solve_cases
    solve_cases.case_back_to_back(solver)


def test_mlp_backward_solve_runs_in_the_persistent_kernel(golden, monkeypatch):
    """The implicit backward of a small MLP imBlock is ONE solver launch (impflow_mlp_broyden_solve_vjp), with the
    golden iteration counts and gradients; switched off, the host-driven loop gives the same answer."""
    from impflow_b200 import branch_program
    from impflow_b200.layers import broyden
    from tests import imblock_cases
    calls = []
    orig = broyden.broyden_mlp_vjp

    def counted(*a, **k):
        calls.append(1)
        return orig(*a, **k)
    monkeypatch.setattr(broyden, 'broyden_mlp_vjp', counted)
    imblock_cases.case_imblock_mlp_train(golden, 'tab6')
    assert len(calls) >= 1
    n = len(calls)
    branch_program.MLP_SOLVER['on'] = False
    try:
        imblock_cases.case_imblock_mlp_train(golden, 'tab6')
    finally:
        branch_program.MLP_SOLVER['on'] = True
    assert len(calls) == n
