"""Shared parity cases (device-parameterised; collected by test_gpu_imblock.py on the GPU and by
test_host_logic.py on the CPU through the C-ABI emulator).

Parity of the imBlock / ImplicitFlow module API against fixtures produced by the
unmodified reference (tests/golden).  State dicts are loaded with the reference's own keys.

Tolerances (BASELINE.json north_star): forward Broyden iteration counts exact; z within 1e-5
rel; log-det within 1e-4 rel.  Backward-solve counts are asserted only where the reference's
own trace clears eps with margin — several fixtures sit at fp32 round-off (eps_backward=1e-10,
SURVEY.md §7 hard part 2) and end on the 30-step cap or a NaN objective."""
import numpy as np
import pytest
import torch

from tests.helpers import rel_err, sub_sd

DEV = {"device": "cuda"}


def dev(t):
    return t.to(DEV["device"])


def _pkg():
    import impflow_b200
    return impflow_b200


def build_mlp(layers, dims, coeff, n_iterations, tol, data_dim):
    mods = []
    for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
        if i > 0:
            mods.append(layers.base.Sin())
        mods.append(layers.base.get_linear(a, b, coeff=coeff, n_iterations=n_iterations, atol=tol, rtol=tol,
                                           domain=2, codomain=2, zero_init=(b == data_dim)))
    return torch.nn.Sequential(*mods)


def build_conv_branch(layers, c, idim, coeff, tol, leading_act):
    mods = []
    if leading_act:
        mods.append(layers.base.Swish())
    mk = lambda a, b, k: layers.base.get_conv2d(a, b, k, 1, k // 2, coeff=coeff, n_iterations=None, domain=2,
                                                codomain=2, atol=tol, rtol=tol)
    mods += [mk(c, idim, 3), layers.base.Swish(), mk(idim, idim, 1), layers.base.Swish(), mk(idim, c, 3)]
    return torch.nn.Sequential(*mods)


def std_normal_logprob(z):
    return -0.5 * np.log(2 * np.pi) - z.pow(2) / 2


def load_block(blk, fx, tag, x):
    blk = blk.to(DEV["device"])
    with torch.no_grad():
        blk(x, restore=True)         # lazy u/v shaping before loading (train_img.py:481-500)
    sd = {k: v.to(DEV["device"]) for k, v in sub_sd(fx, tag + '_sd_').items()}
    missing, unexpected = blk.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    return blk


_BAND = {}


def _bwd_band(tag):
    """Backward iteration counts of the unmodified reference over equivalent re-orderings of its own arithmetic
    (tests/golden/make_golden.py: gen_bwd_band), or None for cases without a measurement."""
    import os
    if not _BAND:
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'bwd_band.npz')
        _BAND.update(dict(np.load(path)))
    key = tag + '_fwd_bwd_nstep'
    return [int(v) for v in _BAND[key][:, 1]] if key in _BAND else None


def run_train(blk, fx, tag, inject=True):
    blk.train()
    x = torch.from_numpy(fx[tag + '_x']).to(DEV["device"]).requires_grad_(True)
    if inject:
        blk._inject_n = fx[tag + '_n_draws'].astype(np.int64)
        blk._inject_probes = (torch.from_numpy(fx[tag + '_vareps_x']), torch.from_numpy(fx[tag + '_vareps_z']))
    else:
        np.random.seed(int(fx[tag + '_seed']))
        torch.manual_seed(int(fx[tag + '_seed']))
    z, dlogp = blk(x, torch.zeros(x.shape[0], 1, device=DEV["device"]))
    logpz = std_normal_logprob(z).reshape(z.size(0), -1).sum(1, keepdim=True)
    loss = -(logpz - dlogp).mean()
    loss.backward()
    return x, z, dlogp, loss


def check_train(blk, fx, tag, x, z, dlogp, loss, bwd_exact=False, grad_tol=1e-3):
    pkg = _pkg()
    assert blk.solver_stats['fwd']['nstep'] == int(fx[tag + '_fwd_nstep'][0])
    bwd = pkg.layers.imBlock.Backward.last_info['nstep']
    print('%s: fwd nstep %d  bwd nstep %d (reference %d)' % (tag, blk.solver_stats['fwd']['nstep'], bwd,
                                                            int(fx[tag + '_bwd_nstep'][0])))
    if bwd_exact:
        assert bwd == int(fx[tag + '_bwd_nstep'][0])
    else:
        # The implicit-backward solve runs with eps_backward = 1e-10 * sqrt(B d), below fp32 round-off: it ends on
        # the 30-step cap, on a NaN objective or on a lucky cancellation.  tests/golden/bwd_band.npz holds the
        # REFERENCE's own counts when its arithmetic is merely re-ordered (intra-op threads, batch order, hidden
        # units re-numbered: toy 6..30, tab6 13..30, cap cases 30): the forward count is invariant, the backward
        # count is not a reproducible quantity of the reference.  Assert the measured band.
        band = _bwd_band(tag)
        lo, hi = (min(band), max(band)) if band is not None else (1, 30)     # no band measured: cap only
        assert lo <= bwd <= hi, (tag, bwd, lo, hi)
    assert rel_err(z.detach().cpu(), fx[tag + '_z']) < 1e-5
    assert rel_err(dlogp.detach().cpu(), fx[tag + '_dlogp']) < 1e-4
    np.testing.assert_allclose(loss.item(), fx[tag + '_loss'], rtol=1e-5)
    assert rel_err(x.grad.cpu(), fx[tag + '_grad_x']) < grad_tol
    worst = 0.0
    for n, p in blk.named_parameters():
        key = tag + '_grad_' + n
        if key in fx:
            assert p.grad is not None, n
            worst = max(worst, rel_err(p.grad.cpu(), fx[key]))
    assert worst < grad_tol, worst


MLP = {
    'toy': dict(dims=[2, 32, 32, 2], n_it=20, tol=None, kw=dict(n_dist='geometric', brute_force=True, n_samples=1,
                                                                neumann_grad=False, grad_in_forward=False)),
    'tab6': dict(dims=[6, 64, 64, 6], n_it=None, tol=1e-3, kw=dict(n_dist='geometric', n_samples=1, n_exact_terms=2,
                                                                   neumann_grad=False, grad_in_forward=False,
                                                                   eps_forward=1e-5)),
    'tab43': dict(dims=[43, 64, 64, 43], n_it=None, tol=1e-3, kw=dict(n_dist='geometric', n_samples=1,
                                                                      n_exact_terms=2, neumann_grad=False,
                                                                      grad_in_forward=False, eps_forward=1e-5)),
}


def make_mlp_block(tag):
    layers = _pkg().layers
    c = MLP[tag]
    d = c['dims'][0]
    return layers.imBlock(build_mlp(layers, c['dims'], 0.99, c['n_it'], c['tol'], d),
                          build_mlp(layers, c['dims'], 0.99, c['n_it'], c['tol'], d), **c['kw'])


# @parametrize('tag', list(MLP))
def case_imblock_mlp_train(golden, tag):
    fx = golden('imblock_mlp')
    blk = load_block(make_mlp_block(tag), fx, tag, torch.from_numpy(fx[tag + '_x']).to(DEV["device"]))
    x, z, dlogp, loss = run_train(blk, fx, tag)
    check_train(blk, fx, tag, x, z, dlogp, loss)


# @parametrize('tag', ['tab6', 'tab43'])
def case_imblock_mlp_train_reference_rng(golden, tag):
    """No injection: the product draws n and the probes with the reference's own RNG calls."""
    fx = golden('imblock_mlp')
    blk = load_block(make_mlp_block(tag), fx, tag, torch.from_numpy(fx[tag + '_x']).to(DEV["device"]))
    x, z, dlogp, loss = run_train(blk, fx, tag, inject=False)
    np.testing.assert_array_equal(blk.last_n_samples.cpu().numpy(), fx[tag + '_n_draws'])   # term counts exact
    assert rel_err(dlogp.detach().cpu(), fx[tag + '_dlogp']) < 1e-4


# @parametrize('tag', ['tab6', 'tab43'])
def case_imblock_mlp_eval_and_inverse(golden, tag):
    fx = golden('imblock_mlp')
    blk = load_block(make_mlp_block(tag), fx, tag, torch.from_numpy(fx[tag + '_x']).to(DEV["device"]))
    blk.eval()
    if tag + 'eval_n_draws' in fx:
        blk._inject_n = fx[tag + 'eval_n_draws'].astype(np.int64)
    if tag + 'eval_vareps_x' in fx:
        blk._inject_probes = (torch.from_numpy(fx[tag + 'eval_vareps_x']), torch.from_numpy(fx[tag + 'eval_vareps_z']))
    x = torch.from_numpy(fx[tag + '_x']).to(DEV["device"])
    z, dlogp = blk(x, torch.zeros(x.shape[0], 1, device=DEV["device"]))
    assert blk.solver_stats['fwd']['nstep'] == int(fx[tag + 'eval_fwd_nstep'][0])
    assert rel_err(z.detach().cpu(), fx[tag + 'eval_z']) < 1e-5
    assert rel_err(dlogp.detach().cpu(), fx[tag + 'eval_dlogp']) < 1e-4
    with torch.no_grad():
        x_rec = blk.inverse(torch.from_numpy(fx[tag + '_z']).to(DEV["device"]))
    assert blk.solver_stats['inv']['nstep'] == int(fx[tag + '_inv_nstep'][0])
    assert rel_err(x_rec.cpu(), fx[tag + '_x_rec']) < 1e-5
    assert rel_err(x_rec.cpu(), fx[tag + '_x']) < 1e-3           # round trip


CONV = {
    'cifar': dict(lead=True, kw=dict(n_dist='poisson', n_samples=1, n_exact_terms=3, neumann_grad=True,
                                     grad_in_forward=True)),
    'cifar_basic': dict(lead=False, kw=dict(n_dist='poisson', n_samples=1, n_exact_terms=3, neumann_grad=False,
                                            grad_in_forward=False)),
}


# @parametrize('tag', list(CONV))
# @parametrize('backend', ['simt', 'auto'])
def case_imblock_conv_train(golden, tag, backend):
    pkg = _pkg()
    pkg.ops.set_gemm_backend(backend)
    try:
        fx = golden('imblock_conv')
        layers = pkg.layers
        c = CONV[tag]
        blk = layers.imBlock(build_conv_branch(layers, 4, 32, 0.9, 1e-3, c['lead']),
                             build_conv_branch(layers, 4, 32, 0.9, 1e-3, c['lead']), **c['kw'])
        blk = load_block(blk, fx, tag, torch.from_numpy(fx[tag + '_x']).to(DEV["device"]))
        x, z, dlogp, loss = run_train(blk, fx, tag)
        check_train(blk, fx, tag, x, z, dlogp, loss, grad_tol=2e-3)
    finally:
        pkg.ops.set_gemm_backend('auto')


def case_imblock_classifier_block(golden):
    pkg = _pkg()
    layers = pkg.layers
    fx = golden('imblock_conv')
    mk = lambda a, b: layers.base.get_conv2d(a, b, kernel_size=3, stride=1, padding=1, bias=False, coeff=0.9,
                                             n_iterations=None, domain=2, codomain=2, atol=1e-3, rtol=1e-3)
    net = lambda: torch.nn.Sequential(mk(8, 16), torch.nn.ReLU(), mk(16, 8), torch.nn.ReLU())
    blk = load_block(layers.imBlock(net(), net()), fx, 'cls', torch.from_numpy(fx['cls_x']).to(DEV["device"]))
    blk.train()
    x = torch.from_numpy(fx['cls_x']).to(DEV["device"]).requires_grad_(True)
    z = blk(x)
    loss = (z ** 2).mean()
    loss.backward()
    assert blk.solver_stats['fwd']['nstep'] == int(fx['cls_fwd_nstep'][0])
    print('cls bwd nstep %d (reference %d)' % (layers.imBlock.Backward.last_info['nstep'], int(fx['cls_bwd_nstep'][0])))
    assert rel_err(z.detach().cpu(), fx['cls_z']) < 1e-5
    np.testing.assert_allclose(loss.item(), fx['cls_loss'], rtol=1e-5)
    assert rel_err(x.grad.cpu(), fx['cls_grad_x']) < 1e-3
    for n, p in blk.named_parameters():
        if 'cls_grad_' + n in fx:
            assert rel_err(p.grad.cpu(), fx['cls_grad_' + n]) < 2e-3, n


def case_implicit_flow_density_step(golden):
    """Whole multiscale model (LogitTransform, ActNorm2d, imBlock, Squeeze) at the reference's
    CIFAR recipe, scaled down: bits/dim, solver counts, reconstruction (train_img.py:517-549)."""
    pkg = _pkg()
    layers = pkg.layers
    fx = golden('flow_small')
    B, c, hw = 4, 3, 8
    model = pkg.ImplicitFlow(
        (B, c, hw, hw), n_blocks=[1, 1], intermediate_dim=16, factor_out=False, quadratic=False,
        init_layer=layers.LogitTransform(0.05), actnorm=True, fc_actnorm=False, batchnorm=False, dropout=0.,
        fc=False, coeff=0.9, vnorms='2222', n_lipschitz_iters=None, sn_atol=1e-3, sn_rtol=1e-3,
        n_power_series=None, n_dist='poisson', n_samples=1, kernels='3-1-3', activation_fn='swish', fc_end=False,
        fc_idim=128, n_exact_terms=3, preact=True, neumann_grad=True, grad_in_forward=True, first_resblock=True,
        learn_p=False, classification=False, classification_hdim=64, n_classes=10).to(DEV["device"])
    x = torch.from_numpy(fx['x']).to(DEV["device"])
    with torch.no_grad():
        model(x, restore=True)
    sd = {k: v.to(DEV["device"]) for k, v in sub_sd(fx, 'sd_').items()}
    model.load_state_dict(sd, strict=True)
    model.train()
    np.random.seed(int(fx['seed']))
    torch.manual_seed(int(fx['seed']))
    z, dlogp = model(x, 0)
    ndim = c * hw * hw
    logpz = std_normal_logprob(z).view(z.size(0), -1).sum(1, keepdim=True)
    bpd = -torch.mean(logpz - dlogp - np.log(256) * ndim) / ndim / np.log(2)
    bpd.backward()
    blocks = [m for m in model.modules() if isinstance(m, layers.imBlock)]
    assert [b.solver_stats['fwd']['nstep'] for b in blocks] == fx['fwd_nstep'].tolist()
    np.testing.assert_array_equal(np.stack([b.last_n_samples.cpu().numpy() for b in blocks]), fx['n_draws'])
    assert rel_err(z.detach().cpu(), fx['z']) < 1e-5
    assert rel_err(dlogp.detach().cpu(), fx['dlogp']) < 1e-4
    np.testing.assert_allclose(bpd.item(), fx['bpd'], rtol=1e-5)
    worst = 0.0
    for n, p in model.named_parameters():
        if 'grad_' + n in fx and p.grad is not None:
            ref = fx['grad_' + n]
            if np.linalg.norm(ref) < 1e-6:      # gradients that are pure round-off in the reference
                assert float(p.grad.norm()) < 1e-5, n
                continue
            worst = max(worst, rel_err(p.grad.cpu(), ref))
    assert worst < 5e-3, worst
    model.eval()
    with torch.no_grad():
        x_rec = model(z.detach(), inverse=True)
    assert rel_err(x_rec.cpu(), fx['x_rec']) < 1e-4
    assert rel_err(x_rec.cpu(), fx['x']) < 1e-3


def case_update_lipschitz_batched_dense():
    """update_lipschitz refreshes every dense (Linear / 1x1) 2-norm layer of a model in ONE launch
    (impflow_sn_power_iter_batch, one CTA per layer): u, v and sigma equal the per-layer launches' bit for bit, for
    fixed iteration counts and for the tolerance mode, with mixed shapes in one batch (train_img.py:786-792)."""
    import copy
    import impflow_b200
    from impflow_b200.layers.base import mixed_lipschitz as ML
    L = impflow_b200.layers
    dev = DEV['device']
    for kw in (dict(n_iterations=None, atol=1e-3, rtol=1e-3), dict(n_iterations=5, atol=None, rtol=None)):
        torch.manual_seed(11)
        lin = lambda a, b: L.base.get_linear(a, b, coeff=0.9, domain=2, codomain=2, **kw)
        conv = lambda a, b, k: L.base.get_conv2d(a, b, k, 1, k // 2, coeff=0.9, domain=2, codomain=2, **kw)
        mlp = torch.nn.Sequential(lin(6, 128), L.base.Swish(), lin(128, 128), L.base.Swish(), lin(128, 40),
                                  L.base.Swish(), lin(40, 6))
        cnn = torch.nn.Sequential(conv(3, 32, 3), L.base.Swish(), conv(32, 48, 1), L.base.Swish(), conv(48, 3, 3))
        model = torch.nn.ModuleList([mlp, cnn]).to(dev)
        with torch.no_grad():
            cnn(torch.randn(2, 3, 8, 8, device=dev))          # shapes the conv layers' u / v
            for p in model.parameters():
                if p.dim() > 1:
                    p.copy_(torch.randn_like(p))
        twin = copy.deepcopy(model)
        launches = getattr(impflow_b200._cabi.load(), 'launches', None)
        ML.BATCH_DENSE['on'] = True
        try:
            L.base.update_lipschitz(model, kw['n_iterations'])
            if launches is not None:        # the emulator counts launches: 1 for the 5 dense layers + 2 conv 3x3
                assert impflow_b200._cabi.load().launches - launches == 3
            ML.BATCH_DENSE['on'] = False
            L.base.update_lipschitz(twin, kw['n_iterations'])
        finally:
            ML.BATCH_DENSE['on'] = True
        n = 0
        for a, b in zip(model.modules(), twin.modules()):
            if hasattr(a, 'sigma_gradient'):
                n += 1
                assert torch.equal(a.u, b.u) and torch.equal(a.v, b.v) and torch.equal(a.scale, b.scale), type(a)
                assert ML.sigma_of(a) is not None
                assert float(a.scale) > 0
        assert n == 7
        # a second refresh reuses the cached descriptor table and still writes the live buffers
        with torch.no_grad():
            for m, t in zip(model.modules(), twin.modules()):
                if hasattr(m, 'sigma_gradient'):
                    m.weight.mul_(1.5)
                    t.weight.mul_(1.5)
        L.base.update_lipschitz(model, kw['n_iterations'])
        ML.BATCH_DENSE['on'] = False
        try:
            L.base.update_lipschitz(twin, kw['n_iterations'])
        finally:
            ML.BATCH_DENSE['on'] = True
        for a, b in zip(model.modules(), twin.modules()):
            if hasattr(a, 'sigma_gradient'):
                assert torch.equal(a.scale, b.scale) and torch.equal(a.u, b.u)


def case_sigma_cache_follows_power_iteration():
    """u / v are updated in place by the power-iteration kernels: every host cache keyed on them (d sigma/d W,
    the effective weights of the branch programs) must see the change (regression: stale sigma after
    update_lipschitz)."""
    import impflow_b200
    from impflow_b200.branch_program import compile_branch
    L = impflow_b200.layers
    dev = DEV['device']
    torch.manual_seed(3)
    mk = lambda a, b, k: L.base.get_conv2d(a, b, k, 1, k // 2, coeff=0.9, n_iterations=None, domain=2, codomain=2,
                                           atol=1e-3, rtol=1e-3)
    net = torch.nn.Sequential(mk(3, 32, 3), L.base.Swish(), mk(32, 32, 1), L.base.Swish(), mk(32, 3, 3)).to(dev)
    lin = L.base.get_linear(8, 16, coeff=0.9, n_iterations=None, atol=1e-3, rtol=1e-3, domain=2, codomain=2).to(dev)
    x = torch.randn(2, 3, 8, 8, device=dev)
    with torch.no_grad():
        net(x)
        prog = compile_branch(net)
        prog.forward(x)
        for m in list(net) + [lin]:
            if hasattr(m, 'sigma_gradient'):
                m.sigma_gradient()                    # fill the caches
        for p in list(net.parameters()) + list(lin.parameters()):
            if p.dim() > 1:
                p.copy_(torch.randn_like(p))          # a big "optimiser step": the singular vectors move
        L.base.update_lipschitz(net)
        lin.compute_weight(update=True)
        for m in list(net) + [lin]:
            if not hasattr(m, 'sigma_gradient'):
                continue
            D = m.sigma_gradient()
            sigma_cached = float((m.weight * D).sum())
            assert abs(sigma_cached - float(m.scale)) < 1e-4 * max(1.0, abs(float(m.scale))), type(m).__name__
        y_prog = prog.forward(x)
        y_mod = net(x)
    assert float((y_prog - y_mod).abs().max()) < 1e-5 * max(1.0, float(y_mod.abs().max()))


def case_training_trajectory_matches_oracle(golden, n_steps=3):
    """Several full training steps (forward, bits/dim, backward, clip, Adam, update_lipschitz:
    train_img.py:591-660, 786-792) of the small multiscale flow, product vs the oracle port, same seeds and
    therefore the same roulette draws and probes: loss per step and forward solver iteration counts."""
    from oracle import flow_oracle
    pkg = _pkg()
    layers = pkg.layers
    fx = golden('flow_small')
    B, c, hw = 4, 3, 8
    model = pkg.ImplicitFlow(
        (B, c, hw, hw), n_blocks=[1, 1], intermediate_dim=16, factor_out=False, quadratic=False,
        init_layer=layers.LogitTransform(0.05), actnorm=True, fc_actnorm=False, batchnorm=False, dropout=0.,
        fc=False, coeff=0.9, vnorms='2222', n_lipschitz_iters=None, sn_atol=1e-3, sn_rtol=1e-3,
        n_power_series=None, n_dist='poisson', n_samples=1, kernels='3-1-3', activation_fn='swish', fc_end=False,
        fc_idim=128, n_exact_terms=3, preact=True, neumann_grad=True, grad_in_forward=True, first_resblock=True,
        learn_p=False, classification=False, classification_hdim=64, n_classes=10).to(DEV["device"])
    x = torch.from_numpy(fx['x']).to(DEV["device"])
    with torch.no_grad():
        model(x, restore=True)
    sd = {k: v.to(DEV["device"]) for k, v in sub_sd(fx, 'sd_').items()}
    model.load_state_dict(sd, strict=True)
    model.train()
    seed = int(fx['seed'])
    ndim = c * hw * hw
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=1e-3, betas=(0.9, 0.99))
    blocks = [m for m in model.modules() if isinstance(m, layers.imBlock)]
    np.random.seed(seed)
    torch.manual_seed(seed)
    got, got_steps = [], []
    for _ in range(n_steps):
        opt.zero_grad()
        z, dlogp = model(x, 0)
        logpz = std_normal_logprob(z).view(z.size(0), -1).sum(1, keepdim=True)
        bpd = -torch.mean(logpz - dlogp - np.log(256) * ndim) / ndim / np.log(2)
        bpd.backward()
        torch.nn.utils.clip_grad_norm_(params, 1.)
        opt.step()
        layers.base.update_lipschitz(model)
        got.append(float(bpd))
        got_steps.append([b.solver_stats['fwd']['nstep'] for b in blocks])
    # oracle trajectory from the same state dict
    cfg = dict(flow_oracle.CIFAR_CFG, n_exact_terms=3)
    flow = flow_oracle.OracleFlow({k: v.clone() for k, v in sub_sd(fx, 'sd_').items()}, [1, 1], cfg, coeff=0.9)
    oopt = torch.optim.Adam(flow.params, lr=1e-3, betas=(0.9, 0.99))
    np.random.seed(seed)
    torch.manual_seed(seed)
    stats = {}
    want = [flow.train_step(torch.from_numpy(fx['x']), oopt, stats) for _ in range(n_steps)]
    np.testing.assert_allclose(got[0], want[0], rtol=1e-5)
    np.testing.assert_allclose(got, want, rtol=2e-3)          # later steps inherit the 5e-3 gradient tolerance
    assert sum(got_steps, []) == [int(v) for v in stats['fwd_nstep']]


def case_fused_adam_matches_reference_step():
    """optim.FusedAdam.step() == clip_grad_norm_ + the vendored Adam + EMA (train_img.py:652-658), several steps."""
    from oracle import impflow_oracle as orc
    pkg = _pkg()
    dev = DEV['device']
    torch.manual_seed(11)
    shapes = [(32, 3, 3, 3), (32,), (7, 5), (1,), (64, 32, 1, 1)]
    params = [torch.nn.Parameter(torch.randn(*s, device=dev)) for s in shapes]
    ref_p = [p.detach().cpu().clone() for p in params]
    ref_m = [torch.zeros_like(p) for p in ref_p]
    ref_v = [torch.zeros_like(p) for p in ref_p]
    ref_e = [p.clone() for p in ref_p]
    bucket = pkg.parallel.FlatGradBucket(params)
    opt = pkg.optim.FusedAdam(params, lr=1e-2, betas=(0.9, 0.99), bucket=bucket, max_grad_norm=1.0, ema_decay=0.9)
    versions = [p._version for p in params]
    for t in range(1, 5):
        grads = [torch.randn(*s) * (3.0 if t % 2 else 0.01) for s in shapes]     # clipped and unclipped steps
        bucket.zero()
        for p, g in zip(params, grads):
            p.grad = g.to(dev)       # outside the bucket, as autograd leaves them: step() gathers
        opt.step()
        orc.clip_adam_ema_step(ref_p, [g.clone() for g in grads], ref_m, ref_v, t, 1e-2, (0.9, 0.99), 1e-8, 1.0, ref_e,
                               0.9)
        total = float(torch.sqrt(sum((g.double() ** 2).sum() for g in grads)))
        assert abs(float(opt.grad_norm()) - total) < 1e-4 * total
        for p, r in zip(params, ref_p):
            assert rel_err(p.detach().cpu(), r) < 2e-6
    for r, off in zip(ref_e, bucket.offsets):
        assert rel_err(opt.ema[off:off + r.numel()].cpu().view_as(r), r) < 2e-6
    assert all(p._version > v for p, v in zip(params, versions))      # host caches are keyed on versions


def case_wide_conv_block_vs_oracle(width=256, c=3, hw=8, batch=2, verbose=False):
    """A CIFAR-recipe conv imBlock at a width the one-launch tile kernel and the native runtime take
    (9c <= 32, width % 256 == 0): one training step (Broyden solve, re-attach, Neumann estimator with the
    memory-efficient backward, implicit backward) against the CPU oracle on the same weights, roulette draw and
    probes.  Returns the error summary (used by __graft_entry__.smoke)."""
    from oracle import impflow_oracle as orc
    from tests.helpers import oracle_branch
    pkg = _pkg()
    layers = pkg.layers
    dev = DEV['device']
    torch.manual_seed(5)
    np.random.seed(5)
    kw = dict(n_dist='poisson', n_samples=1, n_exact_terms=3, neumann_grad=True, grad_in_forward=True)
    blk = layers.imBlock(build_conv_branch(layers, c, width, 0.9, 1e-3, True),
                         build_conv_branch(layers, c, width, 0.9, 1e-3, True), **kw).to(dev)
    x0 = torch.randn(batch, c, hw, hw)
    with torch.no_grad():
        blk(x0.to(dev), restore=True)                 # lazy u / v shaping
        for n, p in blk.named_parameters():           # make the branches (and the spectral rescale) do real work
            if n.endswith('weight') and p.requires_grad:
                p.mul_(3.0)
        layers.base.update_lipschitz(blk)
    sd = {k: v.detach().cpu().clone() for k, v in blk.state_dict().items()}
    blk.train()
    n_draws = np.array([2])
    vx = (torch.randint(0, 2, x0.shape) * 2 - 1).float()
    vz = (torch.randint(0, 2, x0.shape) * 2 - 1).float()
    blk._inject_n, blk._inject_probes = n_draws, (vx, vz)
    pkg.ops.GEMM_PROFILE['on'], pkg.ops.GEMM_PROFILE['shapes'] = True, {}
    try:
        xg = x0.clone().to(dev).requires_grad_(True)
        z, dlogp = blk(xg, torch.zeros(batch, 1, device=dev))
        loss = -(std_normal_logprob(z).reshape(batch, -1).sum(1, keepdim=True) - dlogp).mean()
        loss.backward()
        fused = sum(v for k, v in pkg.ops.GEMM_PROFILE['shapes'].items() if k[0] in ('branch3', 'chain23'))
    finally:
        pkg.ops.GEMM_PROFILE['on'], pkg.ops.GEMM_PROFILE['shapes'] = False, {}
    sub = lambda pre: {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}
    bx = oracle_branch(sub('nnet_x.'), 'swish', 0.9, 1e-3)
    bz = oracle_branch(sub('nnet_z.'), 'swish', 0.9, 1e-3)
    cfg = dict(orc.DEFAULT_CFG, n_dist='poisson', n_exact_terms=3, neumann_grad=True, grad_in_forward=True)
    xo = x0.detach().clone().requires_grad_(True)
    stats = {}
    zo, dlo = orc.imblock_forward(bx, bz, xo, torch.zeros(batch, 1), cfg, True, n_draws=n_draws, probes=(vx, vz),
                                  stats=stats)
    lo = -(std_normal_logprob(zo).reshape(batch, -1).sum(1, keepdim=True) - dlo).mean()
    lo.backward()
    res = {'z': rel_err(z.detach().cpu(), zo.detach()), 'logdet': rel_err(dlogp.detach().cpu(), dlo.detach()),
           'loss': abs(float(loss) - float(lo)) / abs(float(lo)), 'grad_x': rel_err(xg.grad.cpu(), xo.grad),
           'fwd_nstep': (blk.solver_stats['fwd']['nstep'], stats['fwd_nstep'][0]), 'fused_launches': fused}
    worst = 0.0
    names = [n for n, _ in blk.named_parameters() if n.startswith('nnet_x.') or n.startswith('nnet_z.')]
    oparams = dict(zip([n for n in names if n.startswith('nnet_x.')], bx.parameters()))
    oparams.update(zip([n for n in names if n.startswith('nnet_z.')], bz.parameters()))
    for n, p in blk.named_parameters():
        if n in oparams and p.grad is not None and oparams[n].grad is not None and float(oparams[n].grad.norm()) > 1e-6:
            worst = max(worst, rel_err(p.grad.cpu(), oparams[n].grad))
    res['grad_params'] = worst
    if verbose:
        print('wide conv imBlock vs oracle:', res)
    assert res['fwd_nstep'][0] == res['fwd_nstep'][1]
    assert res['z'] < 1e-5 and res['logdet'] < 1e-4 and res['loss'] < 1e-5
    assert res['grad_x'] < 2e-3 and res['grad_params'] < 5e-3
    assert fused > 0, 'the fused tile kernels (k_branch3 / k_chain23) were not used'
    return res


def case_actnorm_fused_matches_expression():
    """ops.actnorm (fused kernels through the C ABI) == the tensor expression of act_norm.py:39-62: y, the log-density
    update and all four gradients, 2d and 1d, with and without logpx."""
    pkg = _pkg()
    from impflow_b200.layers import glue
    dev = DEV['device']
    torch.manual_seed(3)
    for shape, cls, cl in [((5, 12, 16, 16), glue.ActNorm2d, False), ((64, 3, 32, 32), glue.ActNorm2d, False),
                           ((6, 48, 8, 8), glue.ActNorm2d, True), ((37, 6), glue.ActNorm1d, False)]:
        layer = cls(shape[1]).to(dev)
        x0 = torch.randn(*shape, device=dev) * 2 + 0.3
        if cl:      # channels-last memory order, as the branch kernels leave their outputs
            x0 = x0.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
        with torch.no_grad():
            layer(x0)                                  # data-dependent init
            layer.weight.add_(0.1 * torch.randn_like(layer.weight))
        lp0 = torch.randn(shape[0], 1, device=dev)
        r = torch.randn(*shape, device=dev)
        wts = torch.arange(1, shape[0] + 1, device=dev, dtype=torch.float32).view(-1, 1)
        for with_lp in (True, False):
            outs = []
            for fused in (True, False):
                glue.FUSED_ACTNORM['on'] = fused
                try:
                    x = x0.clone().requires_grad_(True)
                    lp = lp0.clone().requires_grad_(True) if with_lp else None
                    for p in layer.parameters():
                        p.grad = None
                    res = layer(x, lp) if with_lp else layer(x)
                    y, lp_out = res if with_lp else (res, None)
                    loss = (y * r).sum()
                    if with_lp:
                        loss = loss + (lp_out * wts).sum()
                    loss.backward()
                    outs.append([y.detach(), lp_out.detach() if with_lp else None, x.grad, lp.grad if with_lp else None,
                                 layer.bias.grad.clone(), layer.weight.grad.clone()])
                finally:
                    glue.FUSED_ACTNORM['on'] = True
            a, b = outs
            for u, v in zip(a, b):
                if u is None:
                    assert v is None
                    continue
                scale = max(float(v.abs().max()), 1e-30)
                assert float((u - v).abs().max()) / scale < 5e-6


def case_mlp_solver_per_layer_beta():
    """Every Swish module owns its learnable beta (activations.py:64-71): the persistent small-d solver must
    evaluate layer l's activation with layer l's beta (regression: it used the first one for all).  Forward and
    inverse solves of an MLP imBlock with diverged betas, persistent kernel vs the host-driven loop."""
    pkg = _pkg()
    layers = pkg.layers
    from impflow_b200 import branch_program
    dev = DEV['device']
    torch.manual_seed(21)
    d, dims = 6, [6, 32, 32, 32, 6]

    def net():
        mods = []
        for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
            if i > 0:
                mods.append(layers.base.Swish())
            mods.append(layers.base.get_linear(a, b, coeff=0.9, n_iterations=None, atol=1e-3, rtol=1e-3, domain=2,
                                               codomain=2))
        return torch.nn.Sequential(*mods)
    blk = layers.imBlock(net(), net(), n_dist='geometric', neumann_grad=False, grad_in_forward=False,
                         eps_forward=1e-6).to(dev)
    with torch.no_grad():
        betas = [m.beta for m in blk.modules() if isinstance(m, layers.base.Swish)]
        for i, b in enumerate(betas):
            b.fill_(-1.5 + 1.1 * i)                   # softplus(beta) from 0.2 to > 4
        for n, p in blk.named_parameters():
            if n.endswith('weight') and p.requires_grad:
                p.mul_(4.0)
        layers.base.update_lipschitz(blk)
    blk.eval()
    x = torch.randn(64, d, device=dev)
    outs = {}
    for persistent in (True, False):
        branch_program.MLP_SOLVER['on'] = persistent
        try:
            with torch.no_grad():
                z = blk(x)
                xr = blk.inverse(z)
            outs[persistent] = (z.cpu(), xr.cpu(), blk.solver_stats['fwd']['nstep'], blk.solver_stats['inv']['nstep'])
        finally:
            branch_program.MLP_SOLVER['on'] = True
    a, b = outs[True], outs[False]
    assert a[2] == b[2] and a[3] == b[3], (a[2:], b[2:])
    assert rel_err(a[0], b[0]) < 1e-5 and rel_err(a[1], b[1]) < 1e-5
    assert rel_err(a[1], x.cpu()) < 1e-3
    # and the solved point really satisfies the block equation of the *module* networks
    with torch.no_grad():
        res = a[0].to(dev) + blk.nnet_z(a[0].to(dev)) - x - blk.nnet_x(x)
    assert float(res.norm()) < 1e-4 * float(x.norm())


# ---- round 2: iResBlock, the imBlock branches no shipped config reaches, the step tail against the reference ----

IRES = {
    'mlp2': dict(dims=[2, 32, 32, 2], n_it=20, tol=None, kw=dict(n_dist='geometric', brute_force=True, n_samples=1,
                                                                 neumann_grad=False, grad_in_forward=False)),
    'mlp6': dict(dims=[6, 64, 64, 6], n_it=None, tol=1e-3, kw=dict(n_dist='geometric', n_samples=1, n_exact_terms=2,
                                                                   neumann_grad=False, grad_in_forward=False)),
    'mlp6n': dict(dims=[6, 64, 64, 6], n_it=None, tol=1e-3, kw=dict(n_dist='poisson', n_samples=2, n_exact_terms=3,
                                                                    neumann_grad=True, grad_in_forward=True)),
    'conv': dict(dims=None, kw=dict(n_dist='poisson', n_samples=1, n_exact_terms=3, neumann_grad=True,
                                    grad_in_forward=True)),
}


# @parametrize('tag', list(IRES))
def case_iresblock(golden, tag):
    """iResBlock (lib/layers/iresblock.py:54-164,186-235) against fixtures of the reference: training step with the
    roulette draw and the Gaussian probe injected (y, log-det, loss, all gradients), the eval-mode estimate
    (20 exact terms / 2x2 closed form) and the fixed-point inverse."""
    pkg = _pkg()
    layers = pkg.layers
    fx = golden('iresblock')
    c = IRES[tag]
    dvc = DEV['device']
    if c['dims'] is None:
        net = build_conv_branch(layers, 4, 32, 0.9, 1e-3, True)
    else:
        net = build_mlp(layers, c['dims'], 0.9, c['n_it'], c['tol'], c['dims'][0])
    blk = layers.iResBlock(net, **c['kw']).to(dvc)
    x0 = torch.from_numpy(fx[tag + '_x']).to(dvc)
    with torch.no_grad():
        blk(x0)                      # lazy u / v shaping
    sd = {k: v.to(dvc) for k, v in sub_sd(fx, tag + '_sd_').items()}
    missing, unexpected = blk.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    blk.train()
    blk._inject_n = fx[tag + '_n_draws'].astype(np.int64)
    blk._inject_probes = torch.from_numpy(fx[tag + '_vareps'])
    x = x0.clone().requires_grad_(True)
    y, dlogp = blk(x, torch.zeros(x.shape[0], 1, device=dvc))
    loss = -(std_normal_logprob(y).reshape(y.size(0), -1).sum(1, keepdim=True) - dlogp).mean()
    loss.backward()
    assert rel_err(y.detach().cpu(), fx[tag + '_y']) < 1e-5
    assert rel_err(dlogp.detach().cpu(), fx[tag + '_dlogp']) < 1e-4
    np.testing.assert_allclose(loss.item(), fx[tag + '_loss'], rtol=1e-5)
    assert rel_err(x.grad.cpu(), fx[tag + '_grad_x']) < 2e-3
    worst = 0.0
    for n, p in blk.named_parameters():
        key = tag + '_grad_' + n
        if key in fx and np.linalg.norm(fx[key]) > 1e-7:
            assert p.grad is not None, n
            worst = max(worst, rel_err(p.grad.cpu(), fx[key]))
    assert worst < 5e-3, worst
    if c['kw'].get('brute_force') is not True:
        np.testing.assert_array_equal(blk.last_n_samples.cpu().numpy(), fx[tag + '_n_draws'])
    blk.eval()
    blk._inject_n = fx[tag + 'eval_n_draws'].astype(np.int64)
    blk._inject_probes = torch.from_numpy(fx[tag + 'eval_vareps'])
    ye, dle = blk(x0.clone(), torch.zeros(x.shape[0], 1, device=dvc))
    assert rel_err(ye.detach().cpu(), fx[tag + 'eval_y']) < 1e-5
    assert rel_err(dle.detach().cpu(), fx[tag + 'eval_dlogp']) < 1e-4
    with torch.no_grad():
        x_rec = blk.inverse(torch.from_numpy(fx[tag + '_y']).to(dvc))
    assert rel_err(x_rec.cpu(), fx[tag + '_x_rec']) < 1e-5
    assert rel_err(x_rec.cpu(), fx[tag + '_x']) < 1e-3
    assert blk.inverse_iterations is not None and blk.inverse_iterations < 1000


class Affine(torch.nn.Module):
    """y = a x: stand-in x-branch of the Banach fixture (tests/golden/make_golden.py)."""

    def __init__(self, a):
        super(Affine, self).__init__()
        self.a = a

    def forward(self, x):
        return self.a * x


class Cliff(torch.nn.Module):
    """-0.5 z on z > -1, a 1e8-steep wall below: Broyden's first step from zeros (z1 = -x_embed) lands behind the
    wall and trips the 1e6 protective break; the Banach iteration from z0 = x stays on the contractive side."""

    def forward(self, z):
        return torch.where(z > -1, -0.5 * z, -0.5 * z + 1e8 * (z + 1))


def case_imblock_banach_fallback(golden):
    """prot_break -> find_fixed_point (implicit_block.py:17-28,74-75) through the block API."""
    pkg = _pkg()
    fx = golden('imblock_edge')
    blk = pkg.layers.imBlock(Affine(0.1), Cliff()).to(DEV['device'])
    x = torch.from_numpy(fx['banach_x']).to(DEV['device'])
    with torch.no_grad():
        z = blk(x)
    info = blk.solver_stats['fwd']
    assert [info['nstep'], int(info['prot_break'])] == fx['banach_ints'].tolist()
    assert rel_err(z.cpu(), fx['banach_z']) < 1e-6


EDGE = {
    'exact': dict(dims=[6, 32, 32, 6], kw=dict(n_dist='geometric', exact_trace=True, n_samples=1, n_exact_terms=2,
                                               neumann_grad=False, grad_in_forward=False, eps_forward=1e-5)),
    'ns3': dict(dims=[12, 32, 32, 12], kw=dict(n_dist='geometric', n_samples=3, n_exact_terms=2, neumann_grad=False,
                                               grad_in_forward=False, eps_forward=1e-5)),
    'nps': dict(dims=[12, 32, 32, 12], kw=dict(n_dist='poisson', n_power_series=4, neumann_grad=True,
                                               grad_in_forward=True, eps_forward=1e-5)),
}


# @parametrize('tag', list(EDGE))
def case_imblock_edge_train(golden, tag):
    """exact_trace (implicit_block.py:327-343), n_samples = 3 (:270-289) and a fixed n_power_series (:275-277)."""
    layers = _pkg().layers
    fx = golden('imblock_edge')
    c = EDGE[tag]
    d = c['dims'][0]
    blk = layers.imBlock(build_mlp(layers, c['dims'], 0.9, None, 1e-3, d), build_mlp(layers, c['dims'], 0.9, None, 1e-3, d),
                         **c['kw'])
    blk = load_block(blk, fx, tag, torch.from_numpy(fx[tag + '_x']).to(DEV["device"]))
    blk.train()
    x = torch.from_numpy(fx[tag + '_x']).to(DEV["device"]).requires_grad_(True)
    if tag != 'nps':
        blk._inject_n = fx[tag + '_n_draws'].astype(np.int64)
    if tag != 'exact':
        blk._inject_probes = (torch.from_numpy(fx[tag + '_vareps_x']), torch.from_numpy(fx[tag + '_vareps_z']))
    z, dlogp = blk(x, torch.zeros(x.shape[0], 1, device=DEV["device"]))
    loss = -(std_normal_logprob(z).reshape(z.size(0), -1).sum(1, keepdim=True) - dlogp).mean()
    loss.backward()
    check_train(blk, fx, tag, x, z, dlogp, loss, grad_tol=2e-3)
    if tag == 'ns3':
        np.testing.assert_array_equal(blk.last_n_samples.cpu().numpy(), fx[tag + '_n_draws'])


def case_imblock_fc_tail(golden):
    """imBlock over FCNet branches (implicit_flow.py:321-356,437-474: the `fc_end` tail of the image flows)."""
    pkg = _pkg()
    layers = pkg.layers
    from impflow_b200.implicit_flow import FCNet
    fx = golden('imblock_edge')
    shape = (2, 4, 4)
    fc = lambda: FCNet(input_shape=shape, idim=24, lipschitz_layer=layers.base.get_linear, nhidden=2, coeff=0.9,
                       domains=[2., 2., 2.], codomains=[2., 2., 2.], n_iterations=None, activation_fn='swish',
                       preact=True, dropout=0, sn_atol=1e-3, sn_rtol=1e-3, learn_p=False)
    blk = layers.imBlock(fc(), fc(), n_dist='poisson', n_samples=1, n_exact_terms=3, neumann_grad=True,
                         grad_in_forward=True)
    blk = load_block(blk, fx, 'fc', torch.from_numpy(fx['fc_x']).to(DEV["device"]))
    x, z, dlogp, loss = run_train(blk, fx, 'fc')
    check_train(blk, fx, 'fc', x, z, dlogp, loss, grad_tol=2e-3)


def case_fused_adam_matches_reference_golden(golden):
    """optim.FusedAdam against the reference's own clip_grad_norm_ + lib/optimizers.Adam + ExponentialMovingAverage
    (tests/golden/step_tail.npz): parameters and EMA shadow after each of four steps, incl. the copy-only first
    EMA apply (lib/utils.py:140-142); then a state_dict round trip into a fresh optimiser."""
    pkg = _pkg()
    dev = DEV['device']
    fx = golden('step_tail')
    n_steps, n_p, lr, b1, b2, eps, max_norm, decay = fx['meta']
    n_steps, n_p = int(n_steps), int(n_p)

    def fresh(values):
        ps = [torch.nn.Parameter(torch.from_numpy(v).clone().to(dev)) for v in values]
        bucket = pkg.parallel.FlatGradBucket(ps)
        return ps, bucket, pkg.optim.FusedAdam(ps, lr=lr, betas=(b1, b2), eps=eps, weight_decay=1e-3, bucket=bucket,
                                               max_grad_norm=max_norm, ema_decay=decay)
    params, bucket, opt = fresh([fx['p0_%d' % i] for i in range(n_p)])

    def do_step(ps, bucket, opt, t):
        bucket.zero()
        for i, p in enumerate(ps):
            p.grad = torch.from_numpy(fx['g%d_%d' % (t, i)]).to(dev)
        opt.step()

    for t in range(n_steps):
        if t == 2:        # checkpoint / resume in the middle of the trajectory
            state = opt.state_dict()
            params, bucket, opt2 = fresh([p.detach().cpu().numpy() for p in params])
            opt2.load_state_dict(state)
            opt = opt2
        do_step(params, bucket, opt, t)
        np.testing.assert_allclose(float(opt.grad_norm()), float(fx['gnorm%d' % t]), rtol=1e-5)
        shadow = opt.ema_params()
        for i, p in enumerate(params):
            np.testing.assert_allclose(p.detach().cpu().numpy(), fx['p%d_%d' % (t + 1, i)], rtol=3e-6, atol=1e-7)
            np.testing.assert_allclose(shadow[i].cpu().numpy(), fx['ema%d_%d' % (t + 1, i)], rtol=3e-6, atol=1e-7)


def case_sweep_graphs_match_eager():
    """BranchProgram.neumann / backward_full replayed from their CUDA graphs (branch_program.SWEEP_GRAPHS) against
    the eager launch sequences, over several "steps" in which the inputs, the saved forward, the weights, the betas
    and the singular vectors all change: a graph must read every one of them through its static inputs."""
    pkg = _pkg()
    from impflow_b200 import branch_program as bp
    from impflow_b200.branch_program import compile_branch
    L = pkg.layers
    dev = DEV['device']
    if dev == 'cpu':
        pytest.skip('CUDA graphs need the GPU')
    torch.manual_seed(17)
    for kind in ('conv', 'conv_noact0'):
        net = build_conv_branch(L, 4, 64, 0.9, 1e-3, kind == 'conv').to(dev)
        shape = (4, 4, 8, 8)
        with torch.no_grad():
            net(torch.randn(*shape, device=dev))
        prog = compile_branch(net)
        calls_before = len(prog._sweep_graphs)
        for step in range(6):
            with torch.no_grad():
                for p in net.parameters():                    # an "optimiser step": weights, biases and betas move
                    p.add_(0.05 * torch.randn_like(p))
                torch.autograd.graph.increment_version(list(net.parameters()))
                L.base.update_lipschitz(net)
                x = torch.randn(*shape, device=dev)
                w, v = torch.randn(*shape, device=dev), torch.randn(*shape, device=dev)
                seed = torch.rand(shape[0], device=dev) + 0.5
                got, want = [], []
                for on, sink in ((True, got), (False, want)):
                    bp.SWEEP_GRAPHS['on'] = on
                    try:
                        _, saved = prog.forward_saved(x)
                        S, gx, gp, tang = prog.neumann(saved, w, v, seed_scale=seed, want_tangent=True)
                        gx2, gp2 = prog.backward_full(saved, w)
                        sink.extend([S, gx, tang, gx2] + [g for g in gp if g is not None] +
                                    [g for g in gp2 if g is not None])
                    finally:
                        bp.SWEEP_GRAPHS['on'] = True
                assert len(got) == len(want)
                for a, b in zip(got, want):
                    scale = max(float(b.abs().max()), 1e-30)
                    assert float((a - b).abs().max()) / scale < 1e-5, (kind, step)
        graphs = [g for g in prog._sweep_graphs.values() if g['graph'] is not None]
        assert len(graphs) == 2, 'both sweeps must have been captured and replayed'


def case_sweep_graphs_mlp_match_eager():
    """The same for an MLP branch (tabular flows): the batched two-adjoint sweep runs over an n-fold batch whose n
    follows the roulette draw, so the program collects one graph per row count, all in one private pool; every graph
    must reproduce the eager sweep while weights and inputs move, in any order of the row counts."""
    pkg = _pkg()
    from impflow_b200 import branch_program as bp
    from impflow_b200.branch_program import compile_branch
    L = pkg.layers
    dev = DEV['device']
    if dev == 'cpu':
        pytest.skip('CUDA graphs need the GPU')
    torch.manual_seed(23)
    d, B = 6, 50
    dims = [d, 64, 64, d]
    mods = []
    for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
        if i > 0:
            mods.append(L.base.Swish())
        mods.append(L.base.get_linear(a, b, coeff=0.9, n_iterations=None, atol=1e-3, rtol=1e-3, domain=2, codomain=2))
    net = torch.nn.Sequential(*mods).to(dev)
    prog = compile_branch(net)
    for step, n in enumerate([3, 3, 4, 3, 5, 4, 3, 5, 4, 3]):
        with torch.no_grad():
            for p in net.parameters():
                p.add_(0.05 * torch.randn_like(p))
            torch.autograd.graph.increment_version(list(net.parameters()))
            L.base.update_lipschitz(net)
            x = torch.randn(B, d, device=dev)
            w, v = torch.randn(n * B, d, device=dev), torch.randn(n * B, d, device=dev)
            seed = torch.rand(n * B, device=dev) + 0.5
            got, want = [], []
            for on, sink in ((True, got), (False, want)):
                bp.SWEEP_GRAPHS['on'], bp.SWEEP_GRAPHS['mlp'] = on, True
                try:
                    _, saved = prog.forward_saved(x)
                    saved_n = prog.tile_saved(saved, n)
                    S, gx, gp = prog.neumann(saved_n, w, v, seed_scale=seed)
                    gx2, gp2 = prog.backward_full(saved, w[:B].contiguous())
                    sink.extend([S, gx, gx2] + [g for g in gp if g is not None] + [g for g in gp2 if g is not None])
                finally:
                    bp.SWEEP_GRAPHS['on'], bp.SWEEP_GRAPHS['mlp'] = True, True
            assert len(got) == len(want)
            for a, b in zip(got, want):
                scale = max(float(b.abs().max()), 1e-30)
                assert float((a - b).abs().max()) / scale < 1e-5, (step, n)
    graphs = [g for g in prog._sweep_graphs.values() if g['graph'] is not None]
    assert len(graphs) == 4, 'three row counts of the batched sweep + the first-order backward: %d' % len(graphs)


def case_mixed_norm_layers(golden):
    """Induced p -> q norms other than 2 -> 2 and learnable orders against the reference (golden mixed_norm.npz):
    constructor incl. the random restarts (same seed: u, v, scale), one-iteration estimate, tolerance-mode update
    after a weight change (u, v as stored — including the orders whose buffer the reference does not write back —,
    sigma, rescaled weight), forward and the weight gradient through sigma."""
    pkg = _pkg()
    BL = pkg.layers.base
    dev = DEV['device']
    fx = golden('mixed_norm')
    tn = lambda a: torch.from_numpy(np.asarray(a)).to(dev)
    close = lambda got, want, rtol=2e-4, atol=2e-5: np.testing.assert_allclose(got.detach().cpu().numpy(), want,
                                                                               rtol=rtol, atol=atol)
    for i, tag in enumerate(['l23', 'l33', 'l13', 'l3i', 'l15_25']):
        dom, cod = [float(t) for t in fx[tag + '_norms']]
        torch.manual_seed(40 + i)
        lin = BL.InducedNormLinear(6, 7, coeff=0.6, domain=dom, codomain=cod, atol=1e-3, rtol=1e-3)
        for k in ('weight', 'bias', 'u', 'v', 'scale'):      # the constructor ran on the host: same draws, same restarts
            close(getattr(lin, k), fx[tag + '_init_' + k], rtol=1e-4, atol=1e-5)
        lin = lin.to(dev)
        with torch.no_grad():
            lin.weight.copy_(tn(fx[tag + '_weight2']))
        close(lin.compute_one_iter(), fx[tag + '_one_iter'])
        W = lin.compute_weight(update=True)
        close(lin.u, fx[tag + '_u_tol'])
        close(lin.v, fx[tag + '_v_tol'])
        close(lin.scale, fx[tag + '_scale_tol'])
        close(W, fx[tag + '_W_tol'])
        x = tn(fx[tag + '_x'])
        close(lin(x), fx[tag + '_y'])
        lin.zero_grad()
        lin(x).pow(2).sum().backward()
        close(lin.weight.grad, fx[tag + '_grad_weight'], rtol=2e-3, atol=1e-4)
    for tag in ['c1_3i', 'c1_13', 'c1_33', 'c3_23', 'c3_33', 'c3_32']:
        dom, cod, k = [float(t) for t in fx[tag + '_norms']]
        k = int(k)
        conv = BL.InducedNormConv2d(3, 4, k, 1, k // 2, coeff=0.5, domain=dom, codomain=cod, atol=1e-3, rtol=1e-3)
        conv = conv.to(dev)
        x = tn(fx[tag + '_x'])
        with torch.no_grad():
            conv(x)                                        # lazy shaping (device generator: values replaced below)
        conv.load_state_dict({kk[len(tag + '_init_'):]: tn(v) for kk, v in fx.items() if kk.startswith(tag + '_init_')})
        close(conv(x), fx[tag + '_y'])
        with torch.no_grad():
            conv.weight.copy_(tn(fx[tag + '_weight2']))
        close(conv.compute_one_iter(), fx[tag + '_one_iter'])
        W = conv.compute_weight(update=True)
        close(conv.u, fx[tag + '_u_tol'])
        close(conv.v, fx[tag + '_v_tol'])
        close(conv.scale, fx[tag + '_scale_tol'])
        close(W, fx[tag + '_W_tol'])
        close(conv(x), fx[tag + '_y2'])
        conv.zero_grad()
        conv(x).pow(2).sum().backward()
        close(conv.weight.grad, fx[tag + '_grad_weight'], rtol=2e-3, atol=1e-4)
    # learnable orders
    torch.manual_seed(80)
    pd, pc = torch.nn.Parameter(torch.tensor(0.)), torch.nn.Parameter(torch.tensor(0.4))
    lin = BL.InducedNormLinear(5, 6, coeff=0.6, domain=pd, codomain=pc, atol=1e-3, rtol=1e-3)
    assert sorted(lin.state_dict().keys()) == sorted(k[len('lp_init_'):] for k in fx if k.startswith('lp_init_'))
    for k in ('weight', 'u', 'v', 'scale', 'domain', 'codomain'):
        close(getattr(lin, k), fx['lp_init_' + k], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose([float(o) for o in lin.compute_domain_codomain()], fx['lp_orders'], rtol=1e-6)
    lin = lin.to(dev)
    with torch.no_grad():
        lin.weight.copy_(tn(fx['lp_weight2']))
    W = lin.compute_weight(update=True)
    close(lin.u, fx['lp_u_tol'])
    close(lin.v, fx['lp_v_tol'])
    close(W, fx['lp_W_tol'])


def case_learn_p_flow_state_dict(golden):
    """ImplicitFlow(learn_p=True): the shared order parameters appear under the same state-dict keys as in the
    reference, with the same parameter count."""
    pkg = _pkg()
    fx = golden('mixed_norm')
    torch.manual_seed(81)
    flow = pkg.ImplicitFlow((2, 3, 8, 8), n_blocks=[1, 1], intermediate_dim=8, factor_out=False, quadratic=False,
                            init_layer=None, actnorm=False, fc_actnorm=False, batchnorm=False, dropout=0., fc=False,
                            coeff=0.9, vnorms='2222', n_lipschitz_iters=None, sn_atol=1e-3, sn_rtol=1e-3,
                            n_power_series=None, n_dist='poisson', n_samples=1, kernels='3-1-3',
                            activation_fn='swish', fc_end=False, fc_idim=16, n_exact_terms=2, preact=True,
                            neumann_grad=True, grad_in_forward=True, first_resblock=True, learn_p=True,
                            classification=False, classification_hdim=64, n_classes=10)
    assert sorted(flow.state_dict().keys()) == [str(k) for k in fx['lp_flow_keys']]
    assert sum(p.numel() for p in flow.parameters()) == int(fx['lp_flow_nparams'][0])


def case_direct_grad_sink_matches_autograd(golden):
    """FlatGradBucket(direct=True): the graph-free backward sweeps add their finished parameter gradients straight
    into the bucket (parallel.sink_grads) instead of returning them to autograd; the flat gradient after one step of
    the small multiscale flow must equal the one autograd's AccumulateGrad nodes build (direct=False)."""
    pkg = _pkg()
    layers = pkg.layers
    fx = golden('flow_small')
    B, c, hw = 4, 3, 8
    flats = []
    for direct in (True, False):
        torch.manual_seed(0)
        model = pkg.ImplicitFlow(
            (B, c, hw, hw), n_blocks=[1, 1], intermediate_dim=16, factor_out=False, quadratic=False,
            init_layer=layers.LogitTransform(0.05), actnorm=True, fc_actnorm=False, batchnorm=False, dropout=0.,
            fc=False, coeff=0.9, vnorms='2222', n_lipschitz_iters=None, sn_atol=1e-3, sn_rtol=1e-3,
            n_power_series=None, n_dist='poisson', n_samples=1, kernels='3-1-3', activation_fn='swish', fc_end=False,
            fc_idim=128, n_exact_terms=3, preact=True, neumann_grad=True, grad_in_forward=True, first_resblock=True,
            learn_p=False, classification=False, classification_hdim=64, n_classes=10).to(DEV["device"])
        x = torch.from_numpy(fx['x']).to(DEV["device"])
        with torch.no_grad():
            model(x, restore=True)
        model.load_state_dict({k: v.to(DEV["device"]) for k, v in sub_sd(fx, 'sd_').items()}, strict=True)
        model.train()
        params = [p for p in model.parameters() if p.requires_grad]
        bucket = pkg.parallel.FlatGradBucket(params, direct=direct)
        np.random.seed(int(fx['seed']))
        torch.manual_seed(int(fx['seed']))
        bucket.zero()
        z, dlogp = model(x, 0)
        ndim = c * hw * hw
        logpz = std_normal_logprob(z).view(z.size(0), -1).sum(1, keepdim=True)
        bpd = -torch.mean(logpz - dlogp - np.log(256) * ndim) / ndim / np.log(2)
        bpd.backward()
        if direct:
            assert any(bucket._touched), 'no gradient took the direct path'
        bucket.gather_strays()
        assert all(p.grad is v for p, v in zip(bucket.params, bucket.views))
        flats.append((bucket.flat.detach().cpu().clone(), list(bucket.had_grad)))
    (a, ha), (b, hb) = flats
    assert ha == hb
    assert rel_err(a, b) < 1e-6
    # and against the reference's gradients
    worst = 0.0
    for (n, p), v in zip([(n, p) for n, p in model.named_parameters() if p.requires_grad], bucket.views):
        ref = fx.get('grad_' + n)
        if ref is not None and np.linalg.norm(ref) > 1e-6:
            worst = max(worst, rel_err(v.detach().cpu(), ref))
    assert worst < 5e-3, worst


def workload_round_trip(workload, batch=None):
    """Size-independent properties of a whole bench workload (bench.WORKLOADS, the BASELINE.json configurations at
    their FULL sizes on the GPU; a reduced one on the emulator): data -> latent -> data round trip through every
    imBlock's forward and inverse Broyden solve (implicit_flow.py:221-251, train_img.py:756-761), the fixed-point
    residual  z + f(z) - x - g(x)  of every block (implicit_block.py:51-100), and run-to-run determinism of the
    forward (fixed-order reductions, no atomics).  Returns the measured figures; the tests hold the thresholds."""
    import bench
    pkg = _pkg()
    dev = DEV['device']
    wl = bench.WORKLOADS[workload]
    batch = batch or wl['batch']
    is_mlp = wl.get('kind') == 'mlp'
    is_cls = wl.get('kind') == 'cls'      # a classifier is not invertible as a whole: residuals and determinism only
    torch.manual_seed(0)
    np.random.seed(0)
    model = bench.build_model(pkg, wl, batch).to(dev)
    if is_mlp:
        bench.scale_mlp_last_layers(model, wl)
    x, _ = bench.synthetic_batch(wl, batch, torch.Generator().manual_seed(1234))
    x = x.to(dev)
    with torch.no_grad():
        if is_mlp:
            model(x)
        else:
            model(x, restore=True)           # ActNorm data init + lazy u / v shaping
        if is_cls:
            for b_ in model.modules():         # BasicImplicitBlock: the first call was the restore pass
                if type(b_).__name__ == 'BasicImplicitBlock':
                    b_.initialized = True
    model.eval()
    blocks = [m for m in model.modules() if isinstance(m, pkg.layers.imBlock)]
    seen = {}
    hooks = [b.register_forward_hook(lambda m, inp, out, i=i: seen.__setitem__(i, (inp[0].detach(), (
        out[0] if isinstance(out, tuple) else out).detach()))) for i, b in enumerate(blocks)]
    with torch.no_grad():
        z = model(x)
        for h in hooks:
            h.remove()
        z2 = model(x)
        x_rec = None if is_cls else model.inverse(z) if is_mlp else model(z, inverse=True)
        residual = 0.0
        for i, b in enumerate(blocks):
            xb, zb = seen[i]
            r = zb + b.nnet_z(zb) - xb - b.nnet_x(xb)
            residual = max(residual, float(r.norm() / xb.norm()))
    assert len(seen) == len(blocks) and bool(torch.isfinite(z).all())
    assert is_cls or bool(torch.isfinite(x_rec).all())
    return {'round_trip': None if is_cls else rel_err(x_rec.cpu(), x.cpu()), 'residual': residual, 'deterministic': bool(torch.equal(z, z2)),
            'blocks': len(blocks), 'batch': batch,
            'fwd_nstep': [b.solver_stats['fwd']['nstep'] for b in blocks if 'fwd' in b.solver_stats],
            'inv_nstep': [b.solver_stats['inv']['nstep'] for b in blocks if 'inv' in b.solver_stats]}


def case_lop_layers(golden):
    """LopLinear / LopConv2d (lipschitz.py:274-366) against the reference: effective weight, `scale` buffer, forward
    and all three gradients for the five closed-form (domain, codomain) pairs, local and global constraint."""
    pkg = _pkg()
    L = pkg.layers.base
    fx = golden('lop')
    dev = DEV['device']
    tags = [str(t) for t in fx['lop_tags']]
    assert len(tags) == 30
    for tag in tags:
        kind = tag.split('_')[1]
        dom, cod, local = [float(v) for v in fx[tag + '_norms']]
        dom = int(dom) if dom != float('inf') else dom
        cod = int(cod) if cod != float('inf') else cod
        if kind == 'lin':
            m = L.get_linear(6, 7, coeff=0.3, domain=dom, codomain=cod, local_constraint=bool(local))
        else:
            k = 1 if kind == 'c1' else 3
            m = L.get_conv2d(3, 4, k, 1, k // 2, coeff=0.3, domain=dom, codomain=cod, local_constraint=bool(local))
        assert type(m).__name__ == ('LopLinear' if kind == 'lin' else 'LopConv2d')
        m = m.to(dev)
        sd = {k_: v.to(dev) for k_, v in sub_sd(fx, tag + '_sd_').items()}
        sd['scale'] = torch.zeros_like(sd['scale'])            # recomputed by the forward
        missing, unexpected = m.load_state_dict(sd, strict=True)
        assert not missing and not unexpected
        x = torch.from_numpy(fx[tag + '_x']).to(dev).requires_grad_(True)
        y = m(x)
        y.pow(2).sum().backward()
        assert rel_err(m.compute_weight().detach().cpu(), fx[tag + '_W']) < 5e-6, tag
        assert abs(float(m.scale) - float(fx[tag + '_sd_scale'])) < 5e-6 * max(1.0, abs(float(m.scale))), tag
        assert rel_err(y.detach().cpu(), fx[tag + '_y']) < 1e-5, tag
        assert rel_err(x.grad.cpu(), fx[tag + '_grad_x']) < 1e-5, tag
        assert rel_err(m.weight.grad.cpu(), fx[tag + '_grad_weight']) < 1e-5, tag
        assert rel_err(m.bias.grad.cpu(), fx[tag + '_grad_bias']) < 1e-5, tag


def case_imblock_lop_train(golden):
    """A training step of an imBlock whose conv branches the factories build under vnorms '122f'
    (implicit_flow.py:359-398: first layer 1 -> 2 and last layer 2 -> inf are Lop layers, the 1x1 in the middle an
    induced 2 -> 2 layer): forward count, z, log-det, loss and every gradient against the reference."""
    pkg = _pkg()
    layers = pkg.layers
    fx = golden('lop')
    INF = float('inf')

    def branch(c, idim, coeff, tol):
        doms, cods = [1, 2, 2], [2, 2, INF]
        mk = lambda a, b, k, j: layers.base.get_conv2d(a, b, k, 1, k // 2, coeff=coeff, n_iterations=None,
                                                       domain=doms[j], codomain=cods[j], atol=tol, rtol=tol)
        return torch.nn.Sequential(layers.base.Swish(), mk(c, idim, 3, 0), layers.base.Swish(), mk(idim, idim, 1, 1),
                                   layers.base.Swish(), mk(idim, c, 3, 2))
    blk = layers.imBlock(branch(4, 16, 0.9, 1e-3), branch(4, 16, 0.9, 1e-3), n_dist='poisson', n_samples=1,
                         n_exact_terms=3, neumann_grad=True, grad_in_forward=True)
    assert type(blk.nnet_x[1]).__name__ == 'LopConv2d' and type(blk.nnet_x[5]).__name__ == 'LopConv2d'
    blk = load_block(blk, fx, 'lopblk', torch.from_numpy(fx['lopblk_x']).to(DEV["device"]))
    x, z, dlogp, loss = run_train(blk, fx, 'lopblk')
    check_train(blk, fx, 'lopblk', x, z, dlogp, loss, grad_tol=2e-3)
    blk.eval()
    with torch.no_grad():
        x_rec = blk.inverse(z.detach())
    assert rel_err(x_rec.cpu(), fx['lopblk_x_rec']) < 1e-4


def case_flow_options(golden):
    """The stack builders' optional layers (implicit_flow.py:374-396, 463): batchnorm=True, dropout > 0, vnorms '122f',
    FC tail.  Same module sequence and state-dict keys as the reference (strict load), the eval-mode latent of the
    reference's state, and a training step that runs (its values depend on dropout draws and on how often the running
    means were touched, which the reference does not pin)."""
    pkg = _pkg()
    fx = golden('lop')
    dev = DEV['device']
    torch.manual_seed(14)
    flow = pkg.ImplicitFlow((2, 3, 8, 8), n_blocks=[1, 1], intermediate_dim=8, factor_out=False, quadratic=False,
                            init_layer=pkg.layers.LogitTransform(0.05), actnorm=True, fc_actnorm=False, batchnorm=True,
                            dropout=0.2, fc=False, coeff=0.9, vnorms='122f', n_lipschitz_iters=None, sn_atol=1e-3,
                            sn_rtol=1e-3, n_power_series=None, n_dist='poisson', n_samples=1, kernels='3-1-3',
                            activation_fn='swish', fc_end=True, fc_idim=16, n_exact_terms=2, preact=True,
                            neumann_grad=True, grad_in_forward=True, first_resblock=True, learn_p=False,
                            classification=False, classification_hdim=64, n_classes=10).to(dev)
    assert [type(m).__name__ for m in flow.modules()] == [str(t) for t in fx['fopt_modules']]
    x = torch.from_numpy(fx['fopt_x']).to(dev)
    with torch.no_grad():
        flow(x, restore=True)
    sd = {k: v.to(dev) for k, v in sub_sd(fx, 'fopt_sd_').items()}
    missing, unexpected = flow.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    flow.eval()
    with torch.no_grad():
        z = flow(x)
        x_rec = flow(z, inverse=True)
    assert rel_err(z.cpu(), fx['fopt_z']) < 1e-5
    assert rel_err(x_rec.cpu(), fx['fopt_x']) < 1e-3
    flow.train()
    np.random.seed(5)
    zt, dlogp = flow(x, 0)
    (zt.pow(2).sum() - dlogp.sum()).backward()
    grads = [p.grad for p in flow.parameters() if p.grad is not None]
    assert grads and all(bool(torch.isfinite(g).all()) for g in grads)
    with pytest.raises(NotImplementedError):
        pkg.ImplicitFlow((2, 3, 8, 8), n_blocks=[1], quadratic=True)
