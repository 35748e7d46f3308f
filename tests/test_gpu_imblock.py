"""GPU parity of the imBlock / ImplicitFlow module API against the reference's golden fixtures
(real kernels, through the C ABI).  The cases live in tests/imblock_cases.py."""
import pytest

from tests import imblock_cases as cases

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _on_gpu():
    cases.DEV['device'] = 'cuda'
    yield


@pytest.mark.parametrize('tag', list(cases.MLP))
def test_imblock_mlp_train(golden, tag):
    cases.case_imblock_mlp_train(golden, tag)


@pytest.mark.parametrize('tag', ['tab6', 'tab43'])
def test_imblock_mlp_train_reference_rng(golden, tag):
    cases.case_imblock_mlp_train_reference_rng(golden, tag)


@pytest.mark.parametrize('tag', ['tab6', 'tab43'])
def test_imblock_mlp_eval_and_inverse(golden, tag):
    cases.case_imblock_mlp_eval_and_inverse(golden, tag)


@pytest.mark.parametrize('tag', list(cases.CONV))
@pytest.mark.parametrize('backend', ['simt', 'auto'])
def test_imblock_conv_train(golden, tag, backend):
    cases.case_imblock_conv_train(golden, tag, backend)


def test_imblock_classifier_block(golden):
    cases.case_imblock_classifier_block(golden)


def test_imblock_unfused_path(golden):
    from impflow_b200.layers import implicit_block
    implicit_block.FUSED['on'] = False
    try:
        cases.case_imblock_conv_train(golden, 'cifar', 'auto')
        cases.case_imblock_mlp_train(golden, 'tab6')
    finally:
        implicit_block.FUSED['on'] = True


def test_implicit_flow_density_step(golden):
    cases.case_implicit_flow_density_step(golden)


def test_mlp_solver_per_layer_beta():
    cases.case_mlp_solver_per_layer_beta()


def test_direct_grad_sink_matches_autograd(golden):
    cases.case_direct_grad_sink_matches_autograd(golden)


@pytest.mark.parametrize('c,hw', [(3, 32), (12, 16), (48, 8)])
def test_block_at_cifar_scale_real_width(c, hw):
    """One training step of a conv imBlock at each CIFAR scale with the REAL hidden width (C = 512; c = 3 @ 32x32,
    12 @ 16x16, 48 @ 8x8; B = 8) against the CPU oracle on the same weights, roulette draw and probes: forward
    iteration count exact, z <= 1e-5, log-det <= 1e-4, gradients.  Scale 0 runs on k_branch3, scales 1 / 2 on the
    layer-1 GEMM + k_chain23."""
    res = cases.case_wide_conv_block_vs_oracle(width=512, c=c, hw=hw, batch=8, verbose=True)
    assert res['fwd_nstep'][0] == res['fwd_nstep'][1]


def test_sweep_graphs_match_eager():
    cases.case_sweep_graphs_match_eager()


def test_mixed_norm_layers_vs_golden(golden):
    cases.case_mixed_norm_layers(golden)


def test_sweep_graphs_mlp_match_eager():
    cases.case_sweep_graphs_mlp_match_eager()


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


def test_smoke_entry():
    import __graft_entry__
    __graft_entry__.smoke()


def test_update_lipschitz_batched_dense():
    cases.case_update_lipschitz_batched_dense()


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
        cases.case_imblock_conv_train(golden, 'cifar', 'auto')
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
    cases.case_imblock_conv_train(golden, 'cifar', 'auto')
    n_saved = sum(1 for s in calls if s)
    bp.MEMO['on'] = False
    try:
        del calls[:]
        cases.case_imblock_conv_train(golden, 'cifar', 'auto')
    finally:
        bp.MEMO['on'] = True
    assert n_saved < sum(1 for s in calls if s)


def test_wide_conv_block_vs_oracle():
    cases.case_wide_conv_block_vs_oracle(verbose=True)


def test_actnorm_fused_matches_expression():
    cases.case_actnorm_fused_matches_expression()


def test_mlp_backward_solve_runs_in_the_persistent_kernel(golden, monkeypatch):
    """The implicit backward of a small MLP imBlock is ONE solver launch (impflow_mlp_broyden_solve_vjp), with the
    golden iteration counts and gradients; switched off, the host-driven loop gives the same answer."""
    from impflow_b200 import branch_program
    from impflow_b200.layers import broyden
    calls = []
    orig = broyden.broyden_mlp_vjp

    def counted(*a, **k):
        calls.append(1)
        return orig(*a, **k)
    monkeypatch.setattr(broyden, 'broyden_mlp_vjp', counted)
    cases.case_imblock_mlp_train(golden, 'tab6')
    assert len(calls) >= 1
    n = len(calls)
    branch_program.MLP_SOLVER['on'] = False
    try:
        cases.case_imblock_mlp_train(golden, 'tab6')
    finally:
        branch_program.MLP_SOLVER['on'] = True
    assert len(calls) == n
