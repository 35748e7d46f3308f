"""Solver-level cases of the one-call Broyden solves (device-parameterised like tests/imblock_cases.py: collected by
test_gpu_solve.py on the GPU and, for the small cases, by test_host_logic.py on the C-ABI emulator).

BranchProgram.solve(mode, rhs, saved, threshold, eps) runs one of three solvers: the native conv runtime
(impflow_conv3_broyden, csrc/conv3_plan.cu: sync-free, up to `runahead` gated speculative iterations behind the last
decision the host has seen), the persistent MLP kernels (impflow_mlp_broyden_solve / _vjp, csrc/mlp_solver.cu) and
the generic kernel loop of layers/broyden.py in rows layout.  Every case here compares one of them with the reference
solver run in float64 on the CPU (oracle.impflow_oracle.broyden_solve) on the same branch:

  mode 0   g(z) = rhs - f(z) - z   from z = 0     (forward / inverse solve)
  mode 1   g(v) = v^T J + v - rhs  from v = 0     (implicit backward; J at the point the saved forward came from)

eps = 1e-6 is above fp32 round-off, so iteration counts are determinate and asserted exactly; every oracle trace is
checked to stay clear of the stopping tolerance (see _guard).  The measured errors are printed as `solve-err` lines."""
import contextlib

import numpy as np
import torch

from oracle import impflow_oracle as orc
from tests.helpers import oracle_branch, rel_err
from tests.imblock_cases import DEV, build_conv_branch

EPS = 1e-6              # convergent cases
EPS_ROUNDOFF = 1e-10    # the implicit backward's eps_backward: the solve ends at fp32 round-off
T_SOLVE = 40            # threshold of the convergent cases (every one converges well before it)
T_MAX = 63              # the solvers' ABI maximum
RUNAHEADS = (0, 1, 2, 8)
TOL_RESULT = 1e-5       # result against the oracle / between solvers
TOL_TRACE = 5e-3        # trace entries above 1e-3 * trace[0] (below that the residual is fp32 round-off)
TIE_MARGIN = 0.03       # no oracle trace entry within 3 % of the scaled eps or of the protective-break factor
# A step that grows the oracle residual more than GROWTH-fold comes from a rank-1 update with a near-zero denominator:
# it amplifies fp32 round-off, so the trace entry it ends is compared at TOL_TRACE_GROWTH (measured on the GPU and in
# the fp32 numpy emulation alike: 7-fold growth, 1.3 % trace difference; the count and result stay exact / within
# TOL_RESULT).  The implicit-backward solves of the narrow MLP branches (d = 2, 6) are linear systems that Broyden
# finishes through such a step.
GROWTH = 5.0
TOL_TRACE_GROWTH = 5e-2
ZERO_ROWS_SEED = 5      # rhs of the zero-row cases

# (c, hw, B, C): the native conv runtime's evaluation paths.  'path' is the one the case must take.  coeff: the
# per-layer spectral bound (default 0.9, the image flows' recipe); the two shapes the stopping-rule cases use take 3.0,
# so that their solves need more steps (8 - 33) than the threshold caps those cases set.  seed: torch seed of the
# branch and its inputs (default 11), chosen where the default puts an oracle trace entry within 10 % of eps.
CONV = {
    'tile_lead': dict(c=3, hw=32, B=8, C=512, lead=True, path='branch3'),
    'tile': dict(c=3, hw=8, B=2, C=256, lead=False, path='branch3'),
    # d = 108: the solver's rank-1 update runs in k_update_small; M = 180 rows: a ragged last tile
    'tile_small': dict(c=3, hw=6, B=5, C=256, lead=True, path='branch3', coeff=3.0),
    'chain23_16': dict(c=12, hw=16, B=8, C=512, lead=True, path='chain23', seed=18),
    'chain23_8': dict(c=12, hw=8, B=3, C=256, lead=True, path='chain23', coeff=3.0),
    'chain23_48': dict(c=48, hw=8, B=8, C=512, lead=True, path='chain23'),
    'chain23_m112': dict(c=48, hw=4, B=7, C=512, lead=True, path='chain23'),      # M = 112: below one tile
    'chain23_a32': dict(c=12, hw=16, B=4, C=512, lead=True, path='chain23_a32', seed=20),  # single fp32 A plane
    'gemm3_12': dict(c=12, hw=8, B=3, C=256, lead=True, path='gemm3'),
    'gemm3_3': dict(c=3, hw=8, B=2, C=256, lead=False, path='gemm3'),
    # B = 1: the batch norm of the stopping rule is the sample norm.  M = 16 is below the 'auto' backend's tensor-core
    # threshold, so the case selects the tcgen05 backend explicitly (the native plan needs every layer on it)
    'b1': dict(c=48, hw=4, B=1, C=256, lead=True, path='chain23', backend='tc'),
}
# the benchmark's scale-0 branch: run-ahead only (no oracle at this size)
CONV_BENCH = {'bench': dict(c=3, hw=32, B=64, C=512, lead=True, path='branch3')}
CONV_STOP = ['tile_small', 'chain23_8']          # one tile-kernel shape (k_update_small), one k_chain23 shape (cluster)

# (B, d, hidden, Linear layers, act)
MLP = {
    'sin2': (5000, 2, 128, 3, 'sin'),
    'swish6': (1000, 6, 128, 5, 'swish'),         # one beta per Swish, all different
    'relu43': (37, 43, 64, 3, 'relu'),
    'b1': (1, 5, 16, 2, 'sin'),
    'limits': (3, 128, 256, 8, 'swish'),          # d = 128, width 256, 8 layers: the persistent kernels' limits
    'd129': (4, 129, 64, 3, 'sin'),               # one past the d limit
    'l9': (3, 8, 32, 9, 'sin'),                   # one past the layer limit
}
MLP_SEED = {'relu43': 13}                                  # torch seed per case (default B + d)
MLP_VJP = ['sin2', 'swish6', 'relu43', 'b1', 'limits']
# d = 2 with 5000 samples: the implicit-backward solve is a 2 x 2 linear system per sample, which Broyden finishes in
# four steps through a near-singular rank-1 update (the oracle's residual grows 50- to 5000-fold at step 3 for every
# seed tried, then drops to ~1e-6 of eps).  fp32 cannot follow that step, on the GPU or in fp32 numpy: the count is
# not determinate.  The case asserts the solve contract and the oracle's trace up to that step.
MLP_VJP_UNSTABLE = {'sin2'}
MLP_BEYOND = ['d129', 'l9']
MLP_STOP = 'relu43'
STOP_RULES = ['cap', 'cap_roundoff', 'prot_break', 'zero_rows']

_BUILT = {}
_ORACLE = {}


def _pkg():
    import impflow_b200
    return impflow_b200


def _lib():
    return _pkg()._cabi.load()


class _Case(object):
    """A branch, its program, the float64 oracle of it and the seeded solve inputs."""

    def __init__(self, key, net, br, rhs, xpt, conv_spec=None):
        from impflow_b200.branch_program import compile_branch
        self.key, self.net, self.br, self.rhs, self.xpt, self.spec = key, net, br, rhs, xpt, conv_spec
        self.prog = compile_branch(net)
        assert self.prog is not None

    def saved(self):
        with torch.no_grad():
            return self.prog.forward_saved(self.xpt)[1]


def _finish(key, net, act, coeff, shape, seed, conv_spec=None):
    dev = DEV['device']
    sd = {k: v.detach().cpu().double() for k, v in net.state_dict().items()}
    br = oracle_branch(sd, act, coeff, 1e-3, requires_grad=False)
    # a generator of their own: the lazy u / v initialisation draws from the device's generator, so the global CPU
    # stream would leave the inputs differing between the GPU and the emulator
    g = torch.Generator().manual_seed(seed)
    rhs, xpt = torch.randn(*shape, generator=g).to(dev), torch.randn(*shape, generator=g).to(dev)
    return _Case(key, net, br, rhs, xpt, conv_spec)


def _pin_power_iteration(net, seed):
    """Overwrite every layer's u / v with a float64 power iteration on the CPU from a seeded start (fixed length, no
    tolerance exit).  update_lipschitz starts from the lazily initialised u / v, which come from the device's
    generator, and stops at a 1e-3 tolerance: left at that, the effective weights, and with them every oracle trace,
    would differ between the GPU and the emulator by far more than fp32 round-off."""
    L = _pkg().layers.base
    g = torch.Generator().manual_seed(seed)
    for m in net.modules():
        if not isinstance(m, (L.InducedNormConv2d, L.InducedNormLinear)):
            continue
        W = m.weight.detach().cpu().double()
        u0 = torch.randn(m.u.shape, generator=g, dtype=torch.float64)
        v0 = torch.randn(m.v.shape, generator=g, dtype=torch.float64)
        if W.dim() == 2 or W.shape[-1] == 1:
            u, v, _ = orc.power_iterate_matrix(W.reshape(W.shape[0], W.shape[1]), u0, v0, n_iterations=100)
        else:
            h, w = [int(t) for t in m.spatial_dims.tolist()]
            u, v, _ = orc.power_iterate_conv(W, u0, v0, (W.shape[1], h, w), 1, W.shape[-1] // 2, n_iterations=100)
        m.u.copy_(u.reshape(m.u.shape).float())
        m.v.copy_(v.reshape(m.v.shape).float())


def conv_case(name, prot_break=False):
    """The conv branch of CONV / CONV_BENCH[name] (product constructors; weights x10 so the spectral rescale is
    active).  prot_break: coeff 1e9 (no rescale), weights x1000 and zero biases, so the first Broyden step grows the
    residual ~1e9-fold while every value stays far below the fp32 range."""
    key = ('conv', name, prot_break, DEV['device'])
    if key not in _BUILT:
        spec = dict(CONV, **CONV_BENCH)[name]
        layers = _pkg().layers
        torch.manual_seed(spec.get('seed', 11))
        coeff = 1e9 if prot_break else spec.get('coeff', 0.9)
        net = build_conv_branch(layers, spec['c'], spec['C'], coeff, 1e-3, spec['lead']).to(DEV['device'])
        shape = (spec['B'], spec['c'], spec['hw'], spec['hw'])
        with torch.no_grad():
            net(torch.randn(*shape).to(DEV['device']))            # lazy u / v shaping
            for n, p in net.named_parameters():
                if n.endswith('weight'):
                    p.mul_(1000.0 if prot_break else 10.0)
                elif n.endswith('bias') and prot_break:
                    p.zero_()
            layers.base.update_lipschitz(net)
            _pin_power_iteration(net, spec.get('seed', 11))
        _BUILT[key] = _finish(key, net, 'swish', coeff, shape, spec.get('seed', 11), spec)
    return _BUILT[key]


def mlp_case(name, prot_break=False):
    """The MLP branch of MLP[name] (get_linear + Sin / Swish / ReLU; weights x4 so the spectral rescale is active).
    prot_break: a single get_linear(d, d) with weight -1e8 I and coeff 1e9 (no rescale): the first step grows the
    residual ~1e8-fold, in both modes (J is constant)."""
    key = ('mlp', name, prot_break, DEV['device'])
    if key not in _BUILT:
        B, d, hidden, n_lin, act = MLP[name]
        L = _pkg().layers
        seed = MLP_SEED.get(name, B + d)
        torch.manual_seed(seed)
        acts = {'sin': L.base.Sin, 'swish': L.base.Swish, 'relu': L.base.ReLU}
        mk = lambda a, b, coeff: L.base.get_linear(a, b, coeff=coeff, n_iterations=None, atol=1e-3, rtol=1e-3,
                                                   domain=2, codomain=2)
        if prot_break:
            coeff = 1e9
            net = torch.nn.Sequential(mk(d, d, coeff))
            with torch.no_grad():
                net[0].weight.copy_(-1e8 * torch.eye(d))
        else:
            coeff = 0.9
            dims = [d] + [hidden] * (n_lin - 1) + [d]
            mods = []
            for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
                if i > 0:
                    mods.append(acts[act]())
                mods.append(mk(a, b, coeff))
            net = torch.nn.Sequential(*mods)
            with torch.no_grad():
                for i, m in enumerate(m for m in net if isinstance(m, L.base.Swish)):
                    m.beta.fill_(-1.5 + 0.7 * i)                  # softplus(beta) from 0.2 up: one beta per layer
                for n, p in net.named_parameters():
                    if n.endswith('weight'):
                        p.mul_(4.0)
        net = net.to(DEV['device'])
        with torch.no_grad():
            L.base.update_lipschitz(net)
            _pin_power_iteration(net, seed)
        _BUILT[key] = _finish(key, net, act, coeff, (B, d), seed)
    return _BUILT[key]


@contextlib.contextmanager
def conv_path(cs):
    """Select the evaluation path the case names; every switch is restored on exit."""
    from impflow_b200 import branch_program as bp, ops
    lib = _lib()
    path = cs.spec['path']
    restore = []
    try:
        if cs.spec.get('backend'):
            prev_backend = ops.get_gemm_backend()
            ops.set_gemm_backend(cs.spec['backend'])
            restore.append(lambda: ops.set_gemm_backend(prev_backend))
        if path == 'chain23_a32':
            prev_a32 = lib.impflow_conv3_set_chain23_a32(1)
            restore.append(lambda: lib.impflow_conv3_set_chain23_a32(prev_a32))
        if path == 'gemm3':
            prev_c23 = lib.impflow_conv3_set_chain23(0)
            restore.append(lambda: lib.impflow_conv3_set_chain23(prev_c23))
            ops.CHAIN23['on'] = False
            restore.append(lambda: ops.CHAIN23.__setitem__('on', True))
            if cs.spec['c'] == 3:
                bp.FUSED3['on'] = False
                restore.append(lambda: bp.FUSED3.__setitem__('on', True))
        yield
    finally:
        for f in reversed(restore):
            f()


@contextlib.contextmanager
def _switch(table, on):
    prev = table['on']
    table['on'] = on
    try:
        yield
    finally:
        table['on'] = prev


def solve(cs, mode, T, eps, rhs=None, runahead=None, profile=False):
    """cs.prog.solve(...) at the given native run-ahead depth (None: leave it).  profile=True also returns the set of
    fused-kernel kinds ('branch3' / 'chain23') the solve recorded in ops.GEMM_PROFILE."""
    ops = _pkg().ops
    lib = _lib()
    rhs = cs.rhs if rhs is None else rhs
    saved = cs.saved() if mode == 1 else None
    prev_ra = lib.impflow_conv3_set_runahead(runahead) if runahead is not None else None
    prev_prof = (ops.GEMM_PROFILE['on'], ops.GEMM_PROFILE['shapes'])
    if profile:
        ops.GEMM_PROFILE['on'], ops.GEMM_PROFILE['shapes'] = True, {}
    try:
        with torch.no_grad():
            res = cs.prog.solve(mode, rhs, saved, T, eps)
        kinds = {k[0] for k in ops.GEMM_PROFILE['shapes']} & {'branch3', 'chain23'} if profile else None
    finally:
        if profile:
            ops.GEMM_PROFILE['on'], ops.GEMM_PROFILE['shapes'] = prev_prof
        if prev_ra is not None:
            lib.impflow_conv3_set_runahead(prev_ra)
    return (res, kinds) if profile else res


def oracle(cs, mode, T, eps, rhs=None, tag=''):
    """The reference solver in float64 on the CPU (cached per case, mode, threshold, eps and rhs tag)."""
    key = (cs.key, mode, T, eps, tag)
    if key not in _ORACLE:
        r = (cs.rhs if rhs is None else rhs).detach().cpu().double()
        z0 = torch.zeros_like(r)
        if mode == 0:
            with torch.no_grad():
                ref = orc.broyden_solve(lambda z: r - cs.br(z) - z, z0, T, eps)
        else:
            with torch.enable_grad():
                xp = cs.xpt.detach().cpu().double().requires_grad_(True)
                y = cs.br(xp)
                ref = orc.broyden_solve(lambda v: torch.autograd.grad(y, xp, v, retain_graph=True)[0] + v - r, z0, T,
                                        eps)
        ref['result'] = ref['result'].detach()
        _ORACLE[key] = ref
    return _ORACLE[key]


def _guard(ref, what):
    """Fixture check: an oracle trace entry within TIE_MARGIN of the scaled eps (or of the protective-break factor)
    would make the fp32 iteration count a coin toss.  Returns the smallest distance to the scaled eps."""
    tr = np.asarray(ref['trace'], dtype=np.float64)
    margin = float(np.min(np.abs(tr / ref['eps'] - 1.0)))
    near_prot = np.abs(tr / (tr[0] * 1e6) - 1.0) <= TIE_MARGIN
    assert margin > TIE_MARGIN and not near_prot.any(), \
        '%s: an oracle trace entry lies within 3%% of a stopping boundary (%s, eps %g): choose another seed' % (
            what, tr.tolist(), ref['eps'])
    return margin


def _report(what, **errs):
    print('solve-err %s %s' % (what, ' '.join('%s=%.3g' % kv for kv in sorted(errs.items()))))


def match_oracle(res, ref, what, rows=None):
    """nstep / lowest_step / prot_break exact, result within TOL_RESULT, trace within TOL_TRACE above round-off.
    rows: compare only these result rows.  Returns the measured errors."""
    margin = _guard(ref, what)
    assert (res['nstep'], res['lowest_step'], res['prot_break']) == \
        (ref['nstep'], ref['lowest_step'], ref['prot_break']), (what, res['trace'], ref['trace'])
    a, b = res['result'].detach().cpu(), ref['result']
    if rows is not None:
        a, b = a[rows], b[rows]
    err = rel_err(a, b)
    assert err <= TOL_RESULT, (what, err)
    tp, tr = np.asarray(res['trace']), np.asarray(ref['trace'])
    assert len(tp) == len(tr) == res['nstep'] + 1
    big = tr > 1e-3 * tr[0]
    grown = np.zeros_like(big)
    if not ref['prot_break']:
        grown[1:] = tr[1:] > GROWTH * tr[:-1]
    dev = np.abs(tp / tr - 1.0)
    terr = float(np.max(dev[big & ~grown])) if (big & ~grown).any() else 0.0
    np.testing.assert_allclose(tp[big & ~grown], tr[big & ~grown], rtol=TOL_TRACE, err_msg=what)
    np.testing.assert_allclose(tp[big & grown], tr[big & grown], rtol=TOL_TRACE_GROWTH, err_msg=what)
    errs = {'result': err, 'trace': terr, 'tie_margin': margin}
    if (big & grown).any():
        errs['trace_after_growth'] = float(np.max(dev[big & grown]))
    return errs


def _bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def snapshot(res):
    return dict(res, result=res['result'].detach().clone(), diff_detail=res['diff_detail'].detach().clone(),
                trace=list(res['trace']))


def assert_identical(a, b, what):
    """Bit-for-bit equal result dicts (NaN included)."""
    for k in ('nstep', 'lowest_step', 'prot_break', 'threshold'):
        assert a[k] == b[k], (what, k, a[k], b[k])
    assert np.array_equal(np.asarray(a['trace']), np.asarray(b['trace']), equal_nan=True), (what, a['trace'], b['trace'])
    assert np.array_equal(np.float64(a['diff']), np.float64(b['diff']), equal_nan=True), (what, a['diff'], b['diff'])
    assert torch.equal(_bits(a['result']), _bits(b['result'])), (what, 'result')
    assert torch.equal(_bits(a['diff_detail']), _bits(b['diff_detail'])), (what, 'diff_detail')


def _native_solve_all(cs, mode, T, eps, rhs=None, runaheads=RUNAHEADS):
    """The same native solve at each run-ahead depth; all must agree bit for bit.  Returns the depth-0 result."""
    base = None
    for k in runaheads:
        res = snapshot(solve(cs, mode, T, eps, rhs=rhs, runahead=k))
        if base is None:
            base = res
        else:
            assert_identical(base, res, '%s mode %d T %d eps %g: run-ahead %d vs %d' % (cs.key[1], mode, T, eps, k,
                                                                                        runaheads[0]))
    return base


# ---------------------------------------------------------------- native conv solve against the oracle
def case_conv_vs_oracle(name, mode):
    """prog.solve on the native conv runtime == the float64 oracle, on the evaluation path the case names; the generic
    rows loop (CONV3_NATIVE off) gives the same counts and result."""
    from impflow_b200 import branch_program as bp
    cs = conv_case(name)
    what = 'conv %s mode %d' % (name, mode)
    with conv_path(cs):
        assert cs.prog.native_plan(cs.rhs) is not None, '%s: no native plan' % what
        res, kinds = solve(cs, mode, T_SOLVE, EPS, profile=True)
        want = {'branch3': {'branch3'}, 'chain23': {'chain23'}, 'chain23_a32': {'chain23'}, 'gemm3': set()}
        assert kinds == want[cs.spec['path']], (what, kinds)
        res = snapshot(res)
        with _switch(bp.CONV3_NATIVE, False):
            assert cs.prog.native_plan(cs.rhs) is None
            rows = solve(cs, mode, T_SOLVE, EPS)
    errs = match_oracle(res, oracle(cs, mode, T_SOLVE, EPS), what)
    assert (rows['nstep'], rows['lowest_step']) == (res['nstep'], res['lowest_step']), (what, rows['trace'],
                                                                                         res['trace'])
    errs['rows_loop'] = rel_err(rows['result'].cpu(), res['result'].cpu())
    assert errs['rows_loop'] <= TOL_RESULT, (what, errs)
    _report(what, nstep=res['nstep'], **errs)


def case_conv_runahead(name, mode):
    """Run-ahead 0 (one synchronisation per iteration) and 1 / 2 / 8 differ only by gated speculative launches: the
    result dicts must be identical bit for bit."""
    cs = conv_case(name)
    with conv_path(cs):
        assert cs.prog.native_plan(cs.rhs) is not None
        _native_solve_all(cs, mode, T_SOLVE, EPS)


# ---------------------------------------------------------------- every way a solve can end
def _check_cap(res, ref, T, what):
    assert res['nstep'] == T and len(res['trace']) == T + 1, (what, res['trace'])
    return match_oracle(res, ref, what)


def _check_contract(res, T, what):
    """The solve contract where iteration counts are not determinate."""
    n, tr = res['nstep'], np.asarray(res['trace'], dtype=np.float64)
    assert 1 <= n <= T and len(tr) == n + 1, (what, tr)
    assert not res['prot_break'], (what, tr)
    finite = np.where(np.isnan(tr), np.inf, tr)
    assert res['lowest_step'] == int(np.argmin(finite)), (what, res['lowest_step'], tr)
    assert res['diff'] == tr[res['lowest_step']]
    dd = float(res['diff_detail'].double().norm())
    assert abs(dd - res['diff']) <= 1e-5 * res['diff'], (what, dd, res['diff'])
    assert bool(torch.isfinite(res['result']).all())
    if n < T:        # the reference's only early exits: converged, or a NaN objective
        assert np.isnan(tr[-1]) or tr[-1] < res['eps'], (what, tr)


def _check_roundoff(res, ref_conv, T, what):
    """The solve contract at fp32 round-off, and the result against the oracle's converged solution."""
    _check_contract(res, T, what)
    err = rel_err(res['result'].cpu(), ref_conv['result'])
    assert err <= TOL_RESULT, (what, err)
    return {'result': err}


def _zero_rows_rhs(cs, mode):
    rhs = torch.randn(cs.rhs.shape, generator=torch.Generator().manual_seed(ZERO_ROWS_SEED)).to(cs.rhs.device)
    if mode == 1:
        rhs[0] = 0
        rhs[-1] = 0
        return rhs, [0, rhs.shape[0] - 1]
    with torch.no_grad():
        f0 = cs.prog.forward(torch.zeros_like(rhs))
    rhs[0] = f0[0]           # g(0) of that row is exactly 0: the solve evaluates f with the same kernels
    return rhs, [0]


def _stop_rule(cs, rule, mode, run, what):
    """One stopping rule through `run(T, eps, rhs) -> result dict` (already checked for run-ahead invariance)."""
    if rule == 'cap':
        errs = {}
        for T in (1, 2, 5):
            ref = oracle(cs, mode, T, EPS)
            assert ref['nstep'] == T, '%s: the case converges within %d steps' % (what, T)
            e = _check_cap(run(T, EPS, None), ref, T, '%s T %d' % (what, T))
            errs['result_T%d' % T] = e['result']
        return errs
    if rule == 'cap_roundoff':
        ref = oracle(cs, mode, T_MAX, EPS_ROUNDOFF)
        errs = {}
        for T in (30, T_MAX):
            res = run(T, EPS_ROUNDOFF, None)
            errs['result_T%d' % T] = _check_roundoff(res, ref, T, '%s T %d' % (what, T))['result']
            errs['nstep_T%d' % T] = res['nstep']
        return errs
    if rule == 'prot_break':
        ref = oracle(cs, mode, T_SOLVE, EPS)
        tr = ref['trace']
        assert ref['prot_break'] and tr[1] / tr[0] > 1e7, \
            '%s: the first step must grow the residual > 1e7-fold (%s): scale the weights up' % (what, tr)
        res = run(T_SOLVE, EPS, None)
        assert res['prot_break'] and res['nstep'] == 1 and res['lowest_step'] == 0, (what, res['trace'])
        assert torch.equal(_bits(res['result']), _bits(torch.zeros_like(res['result']))), what
        match_oracle(res, ref, what)
        return {'growth': res['trace'][1] / res['trace'][0]}
    assert rule == 'zero_rows'
    rhs, zero = _zero_rows_rhs(cs, mode)
    res = run(T_SOLVE, EPS, rhs)
    for t in (res['result'], res['diff_detail']):
        assert not bool(torch.isnan(t).any()), what
    assert not np.isnan(res['trace']).any(), (what, res['trace'])
    for j in zero:
        assert bool((res['result'][j] == 0).all()), '%s: row %d is not exactly zero' % (what, j)
    keep = [j for j in range(rhs.shape[0]) if j not in zero]
    return match_oracle(res, oracle(cs, mode, T_SOLVE, EPS, rhs=rhs, tag='zero_rows'), what, rows=keep)


def case_conv_stop(rule, name, mode):
    """A stopping rule of the native conv solve against the oracle, identical at run-ahead 0 and 2."""
    cs = conv_case(name, prot_break=(rule == 'prot_break'))
    what = 'conv %s %s mode %d' % (rule, name, mode)
    with conv_path(cs):
        assert cs.prog.native_plan(cs.rhs) is not None, what
        errs = _stop_rule(cs, rule, mode, lambda T, eps, rhs: _native_solve_all(cs, mode, T, eps, rhs, (0, 2)), what)
    _report(what, **errs)


def _mlp_solve(cs, mode, T, eps, rhs=None):
    """prog.solve through the persistent MLP kernel (asserted taken)."""
    from impflow_b200.layers import broyden as bmod
    name = 'broyden_mlp_vjp' if mode == 1 else 'broyden_mlp'
    orig, calls = getattr(bmod, name), []

    def counted(*a, **k):
        calls.append(1)
        return orig(*a, **k)
    setattr(bmod, name, counted)
    try:
        res = snapshot(solve(cs, mode, T, eps, rhs=rhs))
    finally:
        setattr(bmod, name, orig)
    assert calls == [1], '%s was not called' % name
    return res


def case_mlp_stop(rule, mode):
    """A stopping rule of the persistent MLP kernel against the oracle."""
    cs = mlp_case(MLP_STOP, prot_break=(rule == 'prot_break'))
    what = 'mlp %s mode %d' % (rule, mode)
    errs = _stop_rule(cs, rule, mode, lambda T, eps, rhs: _mlp_solve(cs, mode, T, eps, rhs), what)
    _report(what, **errs)


# ---------------------------------------------------------------- persistent MLP kernel, implicit-backward mode
def case_mlp_vjp(name):
    """prog.solve(1, ...) runs in impflow_mlp_broyden_solve_vjp and matches the oracle and the generic loop."""
    from impflow_b200 import branch_program as bp
    cs = mlp_case(name)
    what = 'mlp vjp %s' % name
    assert cs.prog.mlp_vjp_spec(cs.saved()) is not None, what
    res = _mlp_solve(cs, 1, T_SOLVE, EPS)
    with _switch(bp.MLP_SOLVER, False):
        assert cs.prog.mlp_vjp_spec(cs.saved()) is None
        rows = solve(cs, 1, T_SOLVE, EPS)
    ref = oracle(cs, 1, T_SOLVE, EPS)
    if name in MLP_VJP_UNSTABLE:
        tr = np.asarray(ref['trace'])
        jumps = np.nonzero(tr[1:] > GROWTH * tr[:-1])[0]
        assert len(jumps), '%s: no near-singular step any more: assert it exactly (drop it from MLP_VJP_UNSTABLE)' % what
        g = int(jumps[0]) + 1
        for r in (res, rows):
            _check_contract(r, T_SOLVE, what)
            assert len(r['trace']) > g, (what, r['trace'])
            np.testing.assert_allclose(r['trace'][:g], tr[:g], rtol=TOL_TRACE, err_msg=what)
        _report(what, nstep=res['nstep'], nstep_rows=rows['nstep'], nstep_oracle=ref['nstep'])
        return
    errs = match_oracle(res, ref, what)
    assert (rows['nstep'], rows['lowest_step']) == (res['nstep'], res['lowest_step']), (what, rows['trace'],
                                                                                         res['trace'])
    errs['rows_loop'] = rel_err(rows['result'].cpu(), res['result'].cpu())
    assert errs['rows_loop'] <= TOL_RESULT, (what, errs)
    _report(what, nstep=res['nstep'], **errs)


def case_mlp_beyond_limits(name):
    """A branch one past a persistent-kernel limit gets no spec and still solves correctly through the rows loop."""
    cs = mlp_case(name)
    assert cs.prog.mlp_vjp_spec(cs.saved()) is None and cs.prog.mlp_solver_spec(cs.rhs) is None, name
    for mode in (0, 1):
        what = 'mlp rows %s mode %d' % (name, mode)
        errs = match_oracle(solve(cs, mode, T_SOLVE, EPS), oracle(cs, mode, T_SOLVE, EPS), what)
        _report(what, **errs)


# ---------------------------------------------------------------- back-to-back solves on one workspace
B2B_SOLVERS = ['conv', 'mlp', 'rows']
_B2B_STEPS = [(0, EPS_ROUNDOFF), (0, EPS), (1, EPS), (0, EPS)]      # capped round-off, convergent, mode 1, mode 0


def case_back_to_back(solver):
    """Solves that share one cached _Workspace leave nothing behind: each result dict of a sequence equals the same
    solve on a fresh workspace bit for bit, and no returned result changes under later solves (no aliasing)."""
    from impflow_b200 import branch_program as bp
    from impflow_b200.layers import broyden as bmod
    T = 30
    if solver == 'mlp':
        cs, ctx = mlp_case(MLP_STOP), contextlib.nullcontext()
    else:
        cs = conv_case('tile_small')
        ctx = conv_path(cs) if solver == 'conv' else _switch(bp.CONV3_NATIVE, False)
    with ctx:
        assert (cs.prog.native_plan(cs.rhs) is not None) == (solver == 'conv')
        assert (cs.prog.mlp_solver_spec(cs.rhs) is not None) == (solver == 'mlp')
        bmod._workspaces.clear()
        seq = [solve(cs, mode, T, eps) for mode, eps in _B2B_STEPS]
        copies = [snapshot(r) for r in seq]
        for i, (mode, eps) in enumerate(_B2B_STEPS):
            bmod._workspaces.clear()
            assert_identical(copies[i], solve(cs, mode, T, eps), '%s step %d vs a fresh workspace' % (solver, i))
        for i, (r, c) in enumerate(zip(seq, copies)):
            assert_identical(r, c, '%s step %d changed after later solves' % (solver, i))
