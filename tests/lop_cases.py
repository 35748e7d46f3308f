"""Device-parameterised checks of the Lop layers (LopLinear / LopConv2d) on the branch-program path: the norm kernel,
the factor-mode weight preparation and the gradient chain against the reference's goldens and float64 autograd of
compute_weight(), and whole 122f branches against the module / autograd path.  Run on CPU under the C-ABI emulator
(tests/test_host_lop_program.py) and on the GPU with the real kernels (tests/test_gpu_lop_program.py)."""
import copy

import torch

from tests.helpers import rel_err

INF = float('inf')
PAIRS = [(1, 1), (1, 2), (1, INF), (2, INF), (INF, INF)]


def _pkg():
    import impflow_b200
    return impflow_b200


def _kind(m):
    """(kind, forward GEMM shape, transposed GEMM shape) of impflow_prep_weights for the layer."""
    cout, cin = m.weight.shape[:2]
    if m.weight.dim() == 2 or m.weight.shape[2:] == (1, 1):
        return 0, (cout, cin), (cin, cout)
    if cin <= cout:
        return 1, (cout, 9 * cin), (9 * cin, cout)
    return 2, (9 * cout, cin), (cin, 9 * cout)


def to_gemm_layout(G, kind):
    """Module-layout [cout][cin](kh kw) tensor -> the forward GEMM layout of kind 0 / 1 / 2."""
    cout, cin = G.shape[:2]
    if kind == 0:
        return G.reshape(cout, cin)
    if kind == 1:
        return G.permute(0, 2, 3, 1).reshape(cout, 9 * cin)
    return G.flip(2, 3).permute(2, 3, 0, 1).reshape(9 * cout, cin)


def _pad(shape, by=32):
    return shape[0], (shape[1] + by - 1) // by * by


def run_layer(m, Gbar):
    """Norms, prep (padded K, planes) and the chain of `m` through the ops wrappers: (fwd, fwd planes, bwd, bwd
    planes, dL/dW) with Gbar = dL/dW_eff in the module layout (fed to the chain in a padded GEMM layout)."""
    ops = _pkg().ops
    W = m.weight.detach()
    axis, nt = m.max_across_dim, ops.lop_norm_type(m.norm_type)
    norms = ops.lop_norms(W, axis, nt, scale_out=m.scale)
    group = (ops.LOP_ROW if axis == 0 else ops.LOP_COL) if m.local_constraint else ops.LOP_ONE
    kind, fs, bs = _kind(m)
    fwd, fsp, bwd, bsp = ops.prep_weights_lop(W, norms if m.local_constraint else norms[-1:], group, m.coeff, kind,
                                              _pad(fs), True, _pad(bs), True)
    Gl = to_gemm_layout(Gbar.float(), kind)
    Gp = Gl.new_zeros(Gl.shape[0], Gl.shape[1] + 5)          # row stride longer than the payload
    Gp[:, :Gl.shape[1]] = Gl
    gW = ops.lop_scale_grad_layout(Gp, kind, W.shape[0], W.shape[1], W.contiguous(), norms, m.coeff, axis, nt,
                                   m.local_constraint)
    return (fwd, fsp, bwd, bsp, gW), (kind, fs, bs)


def check_prep(m, W_eff, out, layout, tol):
    fwd, fsp, bwd, bsp, _ = out
    kind, fs, bs = layout
    f_ref = to_gemm_layout(W_eff, kind)
    b_ref = f_ref.t() if kind == 0 else (
        W_eff.permute(2, 3, 1, 0).reshape(bs) if kind == 1 else W_eff.flip(2, 3).permute(1, 2, 3, 0).reshape(bs))
    for got, planes, ref, shp in ((fwd, fsp, f_ref, fs), (bwd, bsp, b_ref, bs)):
        assert rel_err(got[:, :shp[1]].cpu(), ref.float().cpu()) < tol
        assert float(got[:, shp[1]:].abs().max()) == 0 if got.shape[1] > shp[1] else True
        assert torch.equal(planes[0] + planes[1], got)


def case_golden_layers(golden, device):
    """The 30 reference layer cases (lin / 1x1 / 3x3 x five norm pairs x local / global): prep against the effective
    weight, the `scale` buffer, and the chain against the reference's weight gradient of sum(y^2)."""
    L = _pkg().layers.base
    fx = golden('lop')
    for tag in [str(t) for t in fx['lop_tags']]:
        kind = tag.split('_')[1]
        dom, cod, local = [float(v) for v in fx[tag + '_norms']]
        dom = int(dom) if dom != INF else dom
        cod = int(cod) if cod != INF else cod
        if kind == 'lin':
            m = L.get_linear(6, 7, coeff=0.3, domain=dom, codomain=cod, local_constraint=bool(local))
        else:
            k = 1 if kind == 'c1' else 3
            m = L.get_conv2d(3, 4, k, 1, k // 2, coeff=0.3, domain=dom, codomain=cod, local_constraint=bool(local))
        sd = {k_: torch.from_numpy(fx[tag + '_sd_' + k_]) for k_ in ('weight', 'bias')}
        sd['scale'] = torch.zeros(())
        m.load_state_dict(sd, strict=True)
        m = m.to(device)
        # dL/dW_eff of L = sum(y^2) in float64 from the golden input and output
        x = torch.from_numpy(fx[tag + '_x']).double()
        gy = 2 * torch.from_numpy(fx[tag + '_y']).double()
        if kind == 'lin':
            Gbar = gy.reshape(-1, gy.shape[-1]).t() @ x.reshape(-1, x.shape[-1])
        else:
            Gbar = torch.nn.grad.conv2d_weight(x, m.weight.shape, gy, padding=m.padding)
        out, layout = run_layer(m, Gbar.to(device))
        W_eff = torch.from_numpy(fx[tag + '_W']).to(device).reshape(m.weight.shape)
        check_prep(m, W_eff, out, layout, 5e-6)
        assert abs(float(m.scale) - float(fx[tag + '_sd_scale'])) < 5e-6 * max(1.0, abs(float(m.scale))), tag
        assert rel_err(out[4].cpu(), fx[tag + '_grad_weight']) < 1e-5, tag


def _reference(m, Gbar):
    """(effective weight, dL/dW) by float64 autograd of the module's own compute_weight()."""
    m64 = copy.deepcopy(m).double()
    We = m64.compute_weight()
    (g,) = torch.autograd.grad((We * Gbar.double()).sum(), m64.weight)
    return We.detach(), g, float(m64.scale)


REAL_SHAPES = [('c1', 512, 512), ('c3', 3, 512), ('c3', 512, 3), ('c3', 48, 512), ('c3', 512, 48)]


def case_real_widths(device, shape, ties):
    """Every norm pair, local and global, at the widths of the image flows, against float64 autograd of
    compute_weight().  ties: integer-valued weights, so that the signed maxima and the largest group norms tie."""
    L = _pkg().layers.base
    kind, cin, cout = shape
    for dom, cod in PAIRS:
        for local in (True, False):
            torch.manual_seed(3)
            k = 1 if kind == 'c1' else 3
            m = L.get_conv2d(cin, cout, k, 1, k // 2, coeff=0.97, domain=dom, codomain=cod, local_constraint=local)
            with torch.no_grad():
                if ties:
                    m.weight.copy_(torch.randint(-2, 3, m.weight.shape).float())
                else:
                    m.weight.mul_(5.0)
            m = m.to(device)
            Gbar = torch.randn(m.weight.shape, dtype=torch.float64, device=device)
            out, layout = run_layer(m, Gbar)
            We, g_ref, scale = _reference(m, Gbar)
            check_prep(m, We, out, layout, 2e-6)
            assert abs(float(m.scale) - scale) <= 1e-6 * abs(scale)
            assert rel_err(out[4].double().cpu(), g_ref.cpu()) < 1e-5, (shape, dom, cod, local, ties)


def branch_122f(kind, c, idim, device):
    """A 122f residual branch: 'conv', the image flows' Swish 3x3 (1 -> 2) Swish 1x1 (2 -> 2) Swish 3x3 (2 -> inf)
    (implicit_flow.py:359-398); 'fc', FCNet's d -> idim -> idim -> d Swish MLP with the same norms; 'mlp', the tabular
    flows' Sin MLP d -> idim -> idim -> d (train_tabular.py build_nnet)."""
    L = _pkg().layers
    doms, cods = [1, 2, 2], [2, 2, INF]
    torch.manual_seed(0)
    if kind == 'conv':
        mk = lambda a, b, k, j: L.base.get_conv2d(a, b, k, 1, k // 2, coeff=0.9, n_iterations=None, domain=doms[j],
                                                  codomain=cods[j], atol=1e-3, rtol=1e-3)
        net = torch.nn.Sequential(L.base.Swish(), mk(c, idim, 3, 0), L.base.Swish(), mk(idim, idim, 1, 1),
                                  L.base.Swish(), mk(idim, c, 3, 2))
    elif kind == 'mlp':
        mk = lambda a, b, j: L.base.get_linear(a, b, coeff=0.9, n_iterations=None, domain=doms[j], codomain=cods[j],
                                               atol=1e-3, rtol=1e-3)
        net = torch.nn.Sequential(mk(c, idim, 0), L.base.Sin(), mk(idim, idim, 1), L.base.Sin(), mk(idim, c, 2))
    else:
        from impflow_b200.implicit_flow import FCNet
        net = FCNet((c, 1, 1), idim, L.base.get_linear, 2, 0.9, doms, cods, None, 'swish', False, 0., 1e-3, 1e-3,
                    False)
    return net.to(device)


def case_program_matches_module(kind, c, idim, B, device, hw=8):
    """forward, vjp, backward_full (every parameter gradient) and neumann of the compiled 122f branch against the
    module / autograd path, with the tolerances of tests/branch_cases.py."""
    from impflow_b200.branch_program import compile_branch
    net = branch_122f(kind, c, idim, device)
    shape = (B, c, hw, hw) if kind == 'conv' else ((B, c, 1, 1) if kind == 'fc' else (B, c))
    x = torch.randn(*shape, device=device)
    with torch.no_grad():
        net(x)                                    # lazy u / v shaping of the induced-norm layer
        for p in net.parameters():
            if p.dim() > 1:
                p.mul_(3.0)                       # every rescale active
    prog = compile_branch(net)
    assert prog is not None and prog.is_linear == (kind != 'conv')
    params = list(net.parameters())
    xr = x.clone().requires_grad_(True)
    y_ref = net(xr)
    v = torch.randn_like(y_ref)
    ref = torch.autograd.grad(y_ref, [xr] + params, v)
    with torch.no_grad():
        y, saved = prog.forward_saved(x)
        vjp = prog.vjp(v, saved)
        gx, pg = prog.backward_full(saved, v)
    assert rel_err(y.cpu(), y_ref.detach().cpu()) < 1e-5
    assert rel_err(vjp.cpu(), ref[0].cpu()) < 1e-5
    assert rel_err(gx.cpu(), ref[0].cpu()) < 1e-5
    for p, g, r in zip(params, pg, ref[1:]):
        assert rel_err(g.cpu(), r.cpu()) < 2e-5, tuple(p.shape)
    w, vv = torch.randn_like(y_ref), torch.randn_like(x)
    xr = x.clone().requires_grad_(True)
    (wJ,) = torch.autograd.grad(net(xr), xr, w, create_graph=True)
    S_ref = (wJ.reshape(B, -1) * vv.reshape(B, -1)).sum(1)
    ref = torch.autograd.grad(S_ref.sum(), [xr] + params, allow_unused=True)
    with torch.no_grad():
        _, saved = prog.forward_saved(x)
        S, gx, pg = prog.neumann(saved, w, vv)
    assert rel_err(S.cpu(), S_ref.detach().cpu()) < 1e-5
    assert rel_err(gx.cpu(), ref[0].cpu()) < 2e-5
    for p, g, r in zip(params, pg, ref[1:]):
        if r is None or float(r.norm()) == 0:
            assert g is None or float(g.norm()) < 1e-6
        else:
            assert rel_err(g.cpu(), r.cpu()) < 5e-5, tuple(p.shape)
    # state dicts stay those of the module path: the program wrote the `scale` buffers the forward writes
    lop = [m for m in net.modules() if type(m).__name__.startswith('Lop')]
    assert len(lop) == 2
    for m in lop:
        with torch.no_grad():
            expect = m.scale.clone()
            m.compute_weight()
        assert abs(float(expect) - float(m.scale)) <= 1e-6 * abs(float(m.scale))
    return prog


def case_solves_take_native_route(kind, device, monkeypatch, c=3, idim=32, B=4, hw=8):
    """A 122f imBlock builds branch programs and its Broyden solves run on the native conv runtime (conv branch) or
    the persistent MLP solver kernel (MLP branch), not the generic loop."""
    from impflow_b200 import branch_program as bp
    from impflow_b200.layers import broyden
    L = _pkg().layers
    blk = L.imBlock(branch_122f(kind, c, idim, device), branch_122f(kind, c, idim, device), n_dist='poisson',
                    n_samples=1, n_exact_terms=2, neumann_grad=True, grad_in_forward=True).to(device)
    calls = {'native': 0, 'mlp': 0, 'generic': 0}
    lib = _pkg()._cabi.load()
    native = lib.impflow_conv3_broyden

    def count(key, fn):
        def wrapped(*a, **k):
            calls[key] += 1
            return fn(*a, **k)
        return wrapped
    monkeypatch.setattr(lib, 'impflow_conv3_broyden', count('native', native))
    monkeypatch.setattr(broyden, 'broyden_mlp', count('mlp', broyden.broyden_mlp))
    monkeypatch.setattr(broyden, 'broyden_mlp_vjp', count('mlp', broyden.broyden_mlp_vjp))
    monkeypatch.setattr(broyden, 'broyden', count('generic', broyden.broyden))
    shape = (B, c, hw, hw) if kind == 'conv' else (B, c)
    x = torch.randn(*shape, device=device) * 0.5
    blk.train()
    z, dlogp = blk(x, torch.zeros(B, 1, device=device))
    (z.pow(2).sum() - dlogp.sum()).backward()
    progs = [getattr(n, '_impflow_program', None) for n in (blk.nnet_x, blk.nnet_z)]
    assert all(isinstance(p, bp.BranchProgram) for p in progs)
    assert all(p.grad is not None for p in blk.nnet_x.parameters())
    route = 'native' if kind == 'conv' else 'mlp'
    assert calls[route] >= 2 and calls['generic'] == 0, calls
    return calls
