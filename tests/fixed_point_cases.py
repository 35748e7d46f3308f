"""Cases of the one-call fixed-point solves (device-parameterised like tests/solve_cases.py: collected by
test_gpu_fixed_point.py on the GPU and, for the small cases, by test_host_fixed_point.py on the C-ABI emulator).

BranchProgram.fixed_point(rhs, start, atol, rtol, threshold) runs the Banach iteration x_k = rhs - f(x_{k-1}) from
x_0 = start (iResBlock.inverse: rhs = start = y; the Banach fallback of RootFind: rhs = x_embed, start = z0) in one of
three ways: the native conv runtime (impflow_conv3_fixed_point, csrc/conv3_plan.cu: up to `runahead` gated speculative
evaluations behind the last decision the host has seen), the persistent MLP kernel (impflow_mlp_fixed_point,
csrc/mlp_solver.cu) or the host loop find_fixed_point over prog.forward.  The native conv solve evaluates f with the
kernels prog.forward uses and rounds x and the stopping test as the torch expression does, so it must equal the host
loop bit for bit; the MLP kernel sums f in another order, so it is held to the float64 oracle and to the host loop's
iteration count.  Oracle comparisons skip no step: every case is checked to keep each oracle step's worst element
ratio (x_k - x_{k-1})^2 / tol clear of 1 (see _guard), where fp32 round-off could move the count."""
import contextlib

import torch

from oracle import impflow_oracle as orc
from tests import solve_cases as sc
from tests.helpers import rel_err
from tests.imblock_cases import DEV, build_conv_branch

TOL = 1e-5               # atol = rtol of both reference loops
T_FP = 1000              # their threshold
TIE_MARGIN = 0.03
TOL_RESULT = 1e-5        # against the float64 oracle
TOL_MLP_HOST = 1e-6      # MLP kernel against the host loop (same count, f summed in another order)
T_NAN = 30               # cap of the NaN cases (they run to it)

# every evaluation path of the native conv runtime (solve_cases.CONV at the image flows' coefficient 0.9: the two
# coeff-3 shapes there are not contractions); 'chain23_m112' has M = 112, below one tile
CONV = ['tile_lead', 'tile', 'chain23_16', 'chain23_48', 'chain23_m112', 'chain23_a32', 'gemm3_12', 'gemm3_3', 'b1']
CONV_ORACLE = ['tile', 'chain23_48', 'chain23_m112', 'gemm3_3', 'b1']        # the float64 oracle is run on the CPU
MLP = ['sin2', 'swish6', 'relu43', 'b1', 'limits']
MLP_BEYOND = ['d129', 'l9']
CAPS = (0, 1, 5)
STOP_RULES = ['cap', 'converged_start', 'nan_rhs', 'banach_form']


# The solver cases' branches contract ~10-fold per evaluation (1 - 4 iterations to 1e-5): too few for run-ahead and
# cap tests.  The fixed-point cases build the same branches with a larger per-layer bound, chosen per case for 5 - 30
# iterations (above these bounds some of the branches stop contracting).
CONV_COEFF = {'b1': 3.0}                      # default 3.5
MLP_COEFF = {'b1': 1.2, 'relu43': 2.2}        # default 2.0
_BUILT = {}


def _pkg():
    import impflow_b200
    return impflow_b200


def conv_case(name):
    """solve_cases.conv_case(name) with the per-layer bound CONV_COEFF (same seeds, weights x10, pinned u / v)."""
    key = ('conv', name, DEV['device'])
    if key not in _BUILT:
        spec = sc.CONV[name]
        layers = _pkg().layers
        seed = spec.get('seed', 11)
        coeff = CONV_COEFF.get(name, 3.5)
        torch.manual_seed(seed)
        net = build_conv_branch(layers, spec['c'], spec['C'], coeff, 1e-3, spec['lead']).to(DEV['device'])
        shape = (spec['B'], spec['c'], spec['hw'], spec['hw'])
        with torch.no_grad():
            net(torch.randn(*shape).to(DEV['device']))            # lazy u / v shaping
            for n, p in net.named_parameters():
                if n.endswith('weight'):
                    p.mul_(10.0)
            layers.base.update_lipschitz(net)
            sc._pin_power_iteration(net, seed)
        _BUILT[key] = sc._finish(key, net, 'swish', coeff, shape, seed, spec)
    return _BUILT[key]


def mlp_case(name):
    """solve_cases.mlp_case(name) with the per-layer bound MLP_COEFF (same seeds, weights x4, pinned u / v)."""
    key = ('mlp', name, DEV['device'])
    if key not in _BUILT:
        B, d, hidden, n_lin, act = sc.MLP[name]
        L = _pkg().layers
        seed = sc.MLP_SEED.get(name, B + d)
        coeff = MLP_COEFF.get(name, 2.0)
        torch.manual_seed(seed)
        acts = {'sin': L.base.Sin, 'swish': L.base.Swish, 'relu': L.base.ReLU}
        dims = [d] + [hidden] * (n_lin - 1) + [d]
        mods = []
        for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
            if i > 0:
                mods.append(acts[act]())
            mods.append(L.base.get_linear(a, b, coeff=coeff, n_iterations=None, atol=1e-3, rtol=1e-3, domain=2,
                                          codomain=2))
        net = torch.nn.Sequential(*mods)
        with torch.no_grad():
            for i, m in enumerate(m for m in net if isinstance(m, L.base.Swish)):
                m.beta.fill_(-1.5 + 0.7 * i)
            for n, p in net.named_parameters():
                if n.endswith('weight'):
                    p.mul_(4.0)
        net = net.to(DEV['device'])
        with torch.no_grad():
            L.base.update_lipschitz(net)
            sc._pin_power_iteration(net, seed)
        _BUILT[key] = sc._finish(key, net, act, coeff, (B, d), seed)
    return _BUILT[key]


@contextlib.contextmanager
def counting():
    """Counts the calls of the two one-call solvers: {'conv': n, 'mlp': n}."""
    bp = _pkg().branch_program
    bmod = _pkg().layers.broyden
    calls = {'conv': 0, 'mlp': 0}
    orig_conv, orig_mlp = bp.BranchProgram._native_fixed_point, bmod.fixed_point_mlp

    def conv(*a, **k):
        calls['conv'] += 1
        return orig_conv(*a, **k)

    def mlp(*a, **k):
        calls['mlp'] += 1
        return orig_mlp(*a, **k)
    bp.BranchProgram._native_fixed_point, bmod.fixed_point_mlp = conv, mlp
    try:
        yield calls
    finally:
        bp.BranchProgram._native_fixed_point, bmod.fixed_point_mlp = orig_conv, orig_mlp


def solve(cs, rhs, start, threshold=T_FP, runahead=None):
    """prog.fixed_point at the given native run-ahead depth (None: leave it); returns (x, iterations, calls)."""
    lib = _pkg()._cabi.load()
    prev = lib.impflow_conv3_set_runahead(runahead) if runahead is not None else None
    try:
        with torch.no_grad(), counting() as calls:
            x, n = cs.prog.fixed_point(rhs, start, TOL, TOL, threshold)
    finally:
        if prev is not None:
            lib.impflow_conv3_set_runahead(prev)
    return x.clone(), n, dict(calls)


def host_loop(prog, rhs, start, threshold=T_FP):
    """The reference loop over the branch program's module-layout forward."""
    from impflow_b200.layers.implicit_block import find_fixed_point
    ops = _pkg().ops
    with torch.no_grad():
        return find_fixed_point(lambda x: ops.lincomb3(rhs, 1.0, prog.forward(x), -1.0), start, threshold, TOL, TOL)


def oracle(cs, rhs, start, threshold=T_FP):
    """orc.banach_iterate on the float64 branch: (x, iterations, worst element ratio of every step)."""
    r, s = rhs.detach().cpu().double(), start.detach().cpu().double()
    tol = TOL + TOL * s.abs()
    ratios = []

    def g(z):
        out = r - cs.br(z)
        ratios.append(float(((out - z) ** 2 / tol).max()))
        return out
    with torch.no_grad():
        x = orc.banach_iterate(g, s, threshold, TOL)
    return x, len(ratios) - 1, ratios


def _guard(ratios, what):
    near = [r for r in ratios if abs(r - 1.0) <= TIE_MARGIN]
    assert not near, '%s: an oracle step ends within 3%% of the stopping boundary (%s): choose another seed' % (
        what, near)


def _bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def assert_same(a, b, what):
    """Bit-for-bit equal, except that any NaN equals any NaN (the host loop and the kernels may carry different NaN
    payloads)."""
    na, nb = torch.isnan(a).cpu(), torch.isnan(b).cpu()
    assert torch.equal(na, nb), (what, 'NaN positions')
    assert torch.equal(_bits(a)[~na], _bits(b)[~nb]), (what, 'bits')


def _report(what, **kv):
    print('fixed-point %s %s' % (what, ' '.join('%s=%s' % item for item in sorted(kv.items()))))


# ---------------------------------------------------------------- native conv solve: bitwise against the host loop
def case_conv_bitwise(name):
    """Every run-ahead depth: the iteration count of the host loop and its result, bit for bit."""
    cs = conv_case(name)
    with sc.conv_path(cs):
        assert cs.prog.native_plan(cs.rhs) is not None, name
        ref, n_ref = host_loop(cs.prog, cs.rhs, cs.rhs)
        for ra in sc.RUNAHEADS:
            x, n, calls = solve(cs, cs.rhs, cs.rhs, runahead=ra)
            assert calls == {'conv': 1, 'mlp': 0}, (name, calls)
            assert n == n_ref, (name, ra, n, n_ref)
            assert x.shape == cs.rhs.shape and x.is_contiguous()
            assert_same(x, ref, '%s run-ahead %d' % (name, ra))
    _report('conv bitwise %s' % name, iterations=n_ref)


# ---------------------------------------------------------------- against the float64 oracle
def case_conv_oracle(name):
    cs = conv_case(name)
    with sc.conv_path(cs):
        x, n, calls = solve(cs, cs.rhs, cs.rhs)
    assert calls['conv'] == 1
    ref, n_ref, ratios = oracle(cs, cs.rhs, cs.rhs)
    _guard(ratios, 'conv ' + name)
    err = rel_err(x.cpu(), ref)
    assert n == n_ref and err <= TOL_RESULT, (name, n, n_ref, err)
    _report('conv oracle %s' % name, iterations=n, result=err)


def case_mlp_oracle(name):
    """The persistent kernel: the oracle's count and result, and the host loop's count."""
    cs = mlp_case(name)
    x, n, calls = solve(cs, cs.rhs, cs.rhs)
    assert calls == {'conv': 0, 'mlp': 1}, (name, calls)
    ref, n_ref, ratios = oracle(cs, cs.rhs, cs.rhs)
    _guard(ratios, 'mlp ' + name)
    err = rel_err(x.cpu(), ref)
    assert n == n_ref and err <= TOL_RESULT, (name, n, n_ref, err)
    host, n_host = host_loop(cs.prog, cs.rhs, cs.rhs)
    assert n_host == n and rel_err(x.cpu(), host.cpu()) <= TOL_MLP_HOST, (name, n_host, n)
    _report('mlp oracle %s' % name, iterations=n, result=err)


def case_mlp_beyond_limits(name):
    """One past a persistent-kernel limit: the host loop runs (no one-call solver), with the oracle's answer."""
    cs = mlp_case(name)
    assert cs.prog.mlp_solver_spec(cs.rhs) is None, name
    x, n, calls = solve(cs, cs.rhs, cs.rhs)
    assert calls == {'conv': 0, 'mlp': 0}, (name, calls)
    host, n_host = host_loop(cs.prog, cs.rhs, cs.rhs)
    assert n == n_host
    assert_same(x, host, name)
    ref, n_ref, ratios = oracle(cs, cs.rhs, cs.rhs)
    _guard(ratios, 'mlp ' + name)
    assert n == n_ref and rel_err(x.cpu(), ref) <= TOL_RESULT, (name, n, n_ref)


# ---------------------------------------------------------------- stopping rules
def _stop_inputs(cs, rule):
    """(rhs, start, threshold) of one stopping rule."""
    if rule == 'converged_start':
        with torch.no_grad():
            xs, _ = host_loop(cs.prog, cs.rhs, cs.rhs)
        return cs.rhs, xs, T_FP
    if rule == 'nan_rhs':
        rhs = cs.rhs.clone()
        rhs.view(rhs.shape[0], -1)[0, 0] = float('nan')
        return rhs, rhs, T_NAN
    assert rule == 'banach_form'
    return cs.rhs, cs.xpt, T_FP


def _check_stop(cs, rule, run, exact, what):
    """run(rhs, start, threshold) -> (x, n) of the solver under test; exact: bitwise against the host loop (conv),
    else the same count and TOL_MLP_HOST."""
    def compare(x, n, host, n_host, tag):
        assert n == n_host, (tag, n, n_host)
        if exact:
            assert_same(x, host, tag)
        else:
            assert torch.equal(torch.isnan(x), torch.isnan(host)), tag
            keep = ~torch.isnan(host)
            assert rel_err(x[keep].cpu(), host[keep].cpu()) <= TOL_MLP_HOST, tag

    if rule == 'cap':
        for T in CAPS:
            host, n_host = host_loop(cs.prog, cs.rhs, cs.rhs, T)
            assert n_host == T + 1, '%s: the case converges within %d evaluations' % (what, T + 2)
            x, n = run(cs.rhs, cs.rhs, T)
            compare(x, n, host, n_host, '%s T %d' % (what, T))
            # the result is evaluation T + 2
            y = cs.rhs
            with torch.no_grad():
                for _ in range(T + 2):
                    y = _pkg().ops.lincomb3(cs.rhs, 1.0, cs.prog.forward(y), -1.0)
            if exact:
                assert_same(x, y, '%s T %d: evaluation T + 2' % (what, T))
        return
    rhs, start, T = _stop_inputs(cs, rule)
    host, n_host = host_loop(cs.prog, rhs, start, T)
    if rule == 'converged_start':
        assert n_host == 0, (what, n_host)
    if rule == 'nan_rhs':
        assert n_host == T + 1 and bool(torch.isnan(host).any()), (what, n_host)
    x, n = run(rhs, start, T)
    compare(x, n, host, n_host, what)


def case_conv_stop(rule, name='tile'):
    cs = conv_case(name)
    what = 'conv %s %s' % (rule, name)

    def run(rhs, start, T):
        out = None
        for ra in (0, 2):
            x, n, calls = solve(cs, rhs, start, T, runahead=ra)
            assert calls['conv'] == 1, (what, calls)
            if out is not None:
                assert n == out[1], (what, n, out[1])
                assert_same(x, out[0], '%s run-ahead 2 vs 0' % what)
            out = (x, n)
        return out
    with sc.conv_path(cs):
        _check_stop(cs, rule, run, True, what)
    _report(what)


def case_mlp_stop(rule, name='relu43'):
    cs = mlp_case(name)
    what = 'mlp %s %s' % (rule, name)

    def run(rhs, start, T):
        x, n, calls = solve(cs, rhs, start, T)
        assert calls['mlp'] == 1, (what, calls)
        return x, n
    _check_stop(cs, rule, run, False, what)
    _report(what)


# ---------------------------------------------------------------- back-to-back solves and a side stream
def case_back_to_back(kind):
    """Two solves on one cached workspace, and one on a side stream, equal the same solves in isolation."""
    bmod = _pkg().layers.broyden
    cs = conv_case('tile') if kind == 'conv' else mlp_case('relu43')
    ctx = sc.conv_path(cs) if kind == 'conv' else contextlib.nullcontext()
    with ctx:
        bmod._fp_workspaces.clear()
        a = solve(cs, cs.rhs, cs.rhs)
        bmod._fp_workspaces.clear()
        b = solve(cs, cs.rhs, cs.xpt)
        seq = [solve(cs, cs.rhs, cs.rhs), solve(cs, cs.rhs, cs.xpt)]
        for (x, n, _), (y, m, _) in zip([a, b], seq):
            assert n == m
            assert_same(x, y, '%s back to back' % kind)
        if cs.rhs.is_cuda:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                x, n, _ = solve(cs, cs.rhs, cs.xpt)
            torch.cuda.current_stream().wait_stream(side)
            assert n == b[1]
            assert_same(x, b[0], '%s side stream' % kind)


# ---------------------------------------------------------------- module level
def _conv_resflow(batch):
    """A ResidualFlow at CIFAR shape with the benchmark's recipe and one block per scale less than it (idim 512,
    3-1-3 LipSwish branches at c = 3 / 12 / 48)."""
    pkg = _pkg()
    layers = pkg.layers
    torch.manual_seed(0)
    model = pkg.ResidualFlow(
        (batch, 3, 32, 32), n_blocks=[1, 1, 1], intermediate_dim=512, factor_out=False, quadratic=False,
        init_layer=layers.LogitTransform(0.05), actnorm=True, fc_actnorm=False, batchnorm=False, dropout=0., fc=False,
        coeff=0.9, vnorms='2222', n_lipschitz_iters=None, sn_atol=1e-3, sn_rtol=1e-3, n_power_series=None,
        n_dist='poisson', n_samples=1, kernels='3-1-3', activation_fn='swish', fc_end=False, fc_idim=128,
        n_exact_terms=2, preact=True, neumann_grad=True, grad_in_forward=True, first_resblock=True)
    return model.to(DEV['device'])


def _mlp_resflow(d, n_blocks):
    """A tabular flow of iResBlocks over Sin MLP branches (train_tabular.py's recipe, weights x4 under coeff 0.9)."""
    layers = _pkg().layers
    torch.manual_seed(1)
    dims = [d, 128, 128, d]

    def net():
        mods = []
        for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
            if i > 0:
                mods.append(layers.base.Sin())
            mods.append(layers.base.get_linear(a, b, coeff=0.9, n_iterations=None, atol=1e-3, rtol=1e-3, domain=2,
                                               codomain=2))
        return torch.nn.Sequential(*mods)
    model = layers.SequentialFlow([layers.iResBlock(net(), n_dist='geometric', n_samples=1, n_exact_terms=2,
                                                    neumann_grad=False, grad_in_forward=False)
                                   for _ in range(n_blocks)])
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith('weight'):
                p.mul_(4.0)
    model = model.to(DEV['device'])
    with torch.no_grad():
        layers.base.update_lipschitz(model)
    return model


@contextlib.contextmanager
def host_fixed_point():
    """Every BranchProgram.fixed_point replaced by the host loop over the program's forward (the reference)."""
    bp = _pkg().branch_program
    orig = bp.BranchProgram.fixed_point

    def host(self, rhs, start, atol, rtol, threshold):
        assert (atol, rtol, threshold) == (TOL, TOL, T_FP)
        return host_loop(self, rhs, start, threshold)
    bp.BranchProgram.fixed_point = host
    try:
        yield
    finally:
        bp.BranchProgram.fixed_point = orig


def case_module_round_trip(kind, batch):
    """inverse(forward(x)) through the one-call solves: the round trip the reference loop gives, every block's
    inverse_iterations equal to the host loop's, results bit-identical (conv) or within TOL_MLP_HOST (MLP)."""
    pkg = _pkg()
    dev = DEV['device']
    g = torch.Generator().manual_seed(7)
    if kind == 'conv':
        model = _conv_resflow(batch)
        x = torch.rand(batch, 3, 32, 32, generator=g).to(dev)
        with torch.no_grad():
            model(x, restore=True)
        fwd, inv = (lambda t: model(t)), (lambda t: model(t, inverse=True))
    else:
        model = _mlp_resflow(6, 3)
        x = torch.randn(batch, 6, generator=g).to(dev)
        fwd, inv = model, model.inverse
    model.eval()
    blocks = [m for m in model.modules() if isinstance(m, pkg.layers.iResBlock)]
    assert blocks
    with torch.no_grad(), counting() as calls:
        z = fwd(x)
        x_rec = inv(z)
    counts = [b.inverse_iterations for b in blocks]
    with torch.no_grad(), host_fixed_point():
        x_host = inv(z)
    host_counts = [b.inverse_iterations for b in blocks]
    assert counts == host_counts, (counts, host_counts)
    assert calls[kind] == len(blocks), (calls, len(blocks))
    if kind == 'conv':
        assert_same(x_rec, x_host, 'conv ResidualFlow inverse')
    else:
        assert rel_err(x_rec.cpu(), x_host.cpu()) <= TOL_MLP_HOST
    rt, rt_host = rel_err(x_rec.cpu(), x.cpu()), rel_err(x_host.cpu(), x.cpu())
    assert rt <= max(2 * rt_host, 1e-6), (rt, rt_host)
    _report('module %s' % kind, iterations=counts, round_trip=rt, round_trip_host=rt_host)
    return model, z


def case_no_sync(kind, batch):
    """iResBlock.inverse on the native path makes no synchronising torch call (the solves drain the stream inside the
    library, once per solve)."""
    pkg = _pkg()
    dev = DEV['device']
    g = torch.Generator().manual_seed(7)
    if kind == 'conv':
        model = _conv_resflow(batch)
        x = torch.rand(batch, 3, 32, 32, generator=g).to(dev)
        with torch.no_grad():
            model(x, restore=True)
    else:
        model = _mlp_resflow(6, 3)
        x = torch.randn(batch, 6, generator=g).to(dev)
    model.eval()
    blk = [m for m in model.modules() if isinstance(m, pkg.layers.iResBlock)][0]
    seen = []
    h = blk.register_forward_hook(lambda m, inp, out: seen.append(out[0] if isinstance(out, tuple) else out))
    with torch.no_grad():
        model(x)
    h.remove()
    y = seen[0].detach().clone()
    with torch.no_grad():
        blk.inverse(y)           # warm: effective weights, plans, workspaces
        prev = torch.cuda.get_sync_debug_mode()
        torch.cuda.set_sync_debug_mode('error')
        try:
            with counting() as calls:
                blk.inverse(y)
        finally:
            torch.cuda.set_sync_debug_mode(prev)
    assert calls[kind] == 1, calls


def case_banach_find_root(kind):
    """RootFind.banach_find_root on compiled branches = the reference's find_fixed_point over the module's branches
    (bitwise on the conv runtime)."""
    pkg = _pkg()
    ib = pkg.layers.implicit_block
    cs = conv_case('tile') if kind == 'conv' else mlp_case('relu43')
    ctx = sc.conv_path(cs) if kind == 'conv' else contextlib.nullcontext()
    with ctx, torch.no_grad():
        with counting() as calls:
            z = ib.RootFind.banach_find_root(cs.net, cs.net, cs.xpt, cs.rhs, TOL, T_FP)
        assert calls[kind] == 1, calls
        x_embed = ib.branch_eval(cs.net, cs.rhs) + cs.rhs
        ref, _ = ib.find_fixed_point(lambda t: x_embed - ib.branch_eval(cs.net, t), cs.xpt, T_FP, TOL, TOL)
    if kind == 'conv':
        assert_same(z, ref, 'banach_find_root conv')
    else:
        assert rel_err(z.cpu(), ref.cpu()) <= TOL_MLP_HOST
