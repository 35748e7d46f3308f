"""imBlock: the implicit invertible block  z + f(z) = x + g(x)  — API / state-dict mirror of
lib/layers/implicit_block.py (imBlock :103-355, RootFind :51-100, Backward :165-217, estimators
:373-450, roulette helpers :457-483).

What runs where:
  * forward / inverse root solves and the implicit-differentiation solve in backward: the CUDA
    Broyden kernels (layers/broyden.py) with the residual g assembled by a fused elementwise
    kernel; g's branch evaluations run on the impflow GEMM / conv / activation kernels;
  * log-det estimators: vjp chains through the differentiable kernel primitives (ops.py), the
    Neumann accumulation and Hutchinson dots on fused kernels;
  * host: the Russian-roulette draw and coefficient table (a handful of Python floats) and, in the
    default parity mode, the probe draw on the CPU generator exactly as the reference does.
"""
import copy
import math

import numpy as np
import torch
import torch.nn as nn
from torch.autograd import Function

from .. import ops
from ..parallel import sink_grads
from .broyden import broyden

__all__ = ['imBlock']

# 'reference': n and probes are drawn with the very calls the reference makes (global NumPy RNG,
# CPU torch generator, implicit_block.py:274,297-298) -> identical draws under identical seeds.
# 'device': probes come from the CUDA generator (no host->device copy on the hot path).
PROBE_MODE = {'mode': 'reference'}

# Graph-free fused evaluation (branch_program.py) of the no-grad hot loops: Broyden g evaluations,
# the vjps of the implicit backward solve and of the Neumann / eval-mode power series.  Off = every
# branch evaluation goes through the module and autograd (same kernels, many more launches).
FUSED = {'on': True}


def _program(nnet):
    if not FUSED['on']:
        return None
    prog = getattr(nnet, '_impflow_program', False)
    if prog is False:
        from ..branch_program import compile_branch
        prog = compile_branch(nnet) if isinstance(nnet, nn.Module) else None
        try:
            nnet._impflow_program = prog
        except Exception:
            pass
    return prog


def branch_eval(nnet, x, keep=False):
    """nnet(x) under no_grad, through the fused program when the branch is compilable.  keep=True also keeps
    the pre-activations: the program hands the same saved forward to the re-attach and to the log-det
    estimate, which evaluate the branch at the same point (branch_program.MEMO)."""
    prog = _program(nnet)
    if prog is None:
        return nnet(x)
    return prog.forward_saved(x)[0] if keep else prog.forward(x)


class _BranchApply(Function):
    """y = nnet(x) evaluated and differentiated (first order) by the graph-free branch program:
    one fused forward, one fused backward sweep with the weight gradients (implicit_block.py:227)."""

    @staticmethod
    def forward(ctx, x, prog, *params):
        y, saved = prog.forward_saved(x.detach())
        ctx.prog, ctx.saved_state = prog, saved
        ctx.need_x = x.requires_grad
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        gx, pgrads = ctx.prog.backward_full(ctx.saved_state, gout, need_input_grad=ctx.need_x)
        ctx.saved_state = None
        # finished gradients go straight into the flat bucket when there is one (no AccumulateGrad launches)
        return (gx, None) + tuple(sink_grads(ctx.prog.params, pgrads))


def branch_apply(nnet, x):
    """nnet(x) with gradients to the branch parameters; fused when the branch is compilable."""
    prog = _program(nnet)
    if prog is None or not torch.is_grad_enabled():
        return nnet(x) if prog is None else prog.forward(x)
    return _BranchApply.apply(x, prog, *prog.params)


# Solver-phase timing for bench.py (SURVEY.md section 8d: Broyden solves/s = solves / time spent in solver phases): when
# on, every forward / inverse / implicit-backward solve is bracketed by CUDA events on the current stream.
SOLVER_TIMING = {'on': False, 'events': []}


def _timed(kind, like, fn):
    if not (SOLVER_TIMING['on'] and like.is_cuda):
        return fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    SOLVER_TIMING['events'].append((kind, e0, e1))
    return out


# Independent halves of a block's work (the log-det estimates of the x- and z-branch) on two streams.
OVERLAP = {'on': True}
HOST_AHEAD = {'on': True}     # imBlock.forward: twin refresh and random draws in front of the forward solve
_side = {}


class _overlap(object):
    """`with _overlap(t) as side: with side: <work A>; <work B>` runs A on a side stream that forks from and
    joins back into the current stream of t's device; a no-op (A then B in order) off the GPU."""

    def __init__(self, like):
        self.dev = like.device if (like.is_cuda and OVERLAP['on']) else None

    def __enter__(self):
        if self.dev is None:
            import contextlib
            return contextlib.nullcontext()
        self.main = torch.cuda.current_stream(self.dev)
        self.side = _side.get(self.dev.index)
        if self.side is None:
            self.side = _side[self.dev.index] = torch.cuda.Stream(device=self.dev)
        fork = torch.cuda.Event()
        fork.record(self.main)
        self.side.wait_event(fork)
        return torch.cuda.stream(self.side)

    def __exit__(self, *exc):
        if self.dev is not None:
            join = torch.cuda.Event()
            join.record(self.side)
            self.main.wait_event(join)
        return False


def _twin_slots(net):
    """(dict, name) of every parameter / buffer slot of `net` in module order.  The tensors are looked up through the
    slots on every call (a buffer may have been re-registered, a parameter's storage re-pointed); only the walk
    over the module tree is cached (it cost 0.3 ms of host time per call, right after a solve has drained the
    stream, i.e. while the GPU idles)."""
    slots = net.__dict__.get('_impflow_twin_slots')
    n_mod = sum(1 for _ in net.children())
    if slots is None or slots[0] != n_mod:
        lst = []
        for m in net.modules():
            lst += [(m._parameters, k) for k, v in m._parameters.items() if v is not None]
        for m in net.modules():
            lst += [(m._buffers, k) for k, v in m._buffers.items() if v is not None]
        mirrors = [m for m in net.modules() if hasattr(m, '_hw')]
        slots = net.__dict__['_impflow_twin_slots'] = (n_mod, lst, mirrors)
    return slots


def _twin_versions(net):
    _, slots, _ = _twin_slots(net)
    return [dct[k]._version for dct, k in slots]


def _sync_twin(dst, src, fallback=True):
    """dst.load_state_dict(src.state_dict()) for two structurally identical nets, as one multi-tensor copy
    (the reference refreshes the frozen twins after every forward, implicit_block.py:228-229).  Falls back
    to load_state_dict whenever a shape differs (lazily shaped u / v before their first use) — or, with
    fallback=False, does nothing then and returns False (the caller retries later)."""
    with torch.no_grad():
        _, dslots, mirrors = _twin_slots(dst)
        _, sslots, _ = _twin_slots(src)
        d = [dct[k] for dct, k in dslots]
        s = [dct[k] for dct, k in sslots]
        if len(d) == len(s):
            key = tuple([(t.data_ptr(), t.numel()) for t in d] + [(t.data_ptr(), t.numel()) for t in s])
            cache = dst.__dict__.get('_impflow_twin_cache')
            if cache is None or cache[0] != key:
                cache = None
                if all(a.shape == b.shape and a.dtype == b.dtype for a, b in zip(d, s)):
                    # the multi-tensor fast path needs one dtype per call and equal strides: group by dtype and copy
                    # flat views (a mixed list silently degrades to one cudaMemcpy per tensor)
                    groups, singles = {}, []
                    for a, b in zip(d, s):
                        if a.is_contiguous() and b.is_contiguous():
                            groups.setdefault(a.dtype, ([], []))
                            groups[a.dtype][0].append(a.view(-1))
                            groups[a.dtype][1].append(b.detach().view(-1))
                        else:
                            singles.append((a, b))
                    cache = dst.__dict__['_impflow_twin_cache'] = (key, list(groups.values()), singles)
            if cache is not None:
                for a, b in cache[2]:
                    a.copy_(b)
                for da, sa in cache[1]:
                    torch._foreach_copy_(da, sa)
                for m in mirrors:                 # python mirrors of buffers that load_state_dict would reset
                    m._hw = None
                    m._init_known = None
                return True
    if not fallback:
        return False
    dst.load_state_dict(src.state_dict())
    return True


_pinned = {}


def _upload(host_t, like):
    """Host tensor -> device of `like` through a reusable pinned staging buffer (async H2D)."""
    if not like.is_cuda:
        return host_t.to(like)
    slots = _pinned.setdefault(host_t.numel(), [])
    # two alternating buffers per size: the previous upload of the same size may still be in flight
    if len(slots) < 4:
        slots.append(torch.empty(host_t.numel(), dtype=torch.float32).pin_memory())
    buf = slots.pop(0)
    slots.append(buf)
    buf.copy_(host_t.reshape(-1))
    return buf.to(like.device, non_blocking=True).view(host_t.shape)


def find_fixed_point(g, y, threshold=1000, atol=1e-5, rtol=1e-5):
    """Banach iteration x <- g(x) from y on the host (implicit_block.py:17-28, iresblock.py:69-79): until every
    (x - x_prev)^2 / (atol + |y| rtol) < 1, at most threshold + 2 evaluations of g.  Returns (x, i), i the reference's
    iteration count.  Builds a graph through g when grad mode is on."""
    x, x_prev = g(y), y
    i = 0
    tol = atol + y.abs() * rtol
    while not torch.all((x - x_prev) ** 2 / tol < 1.):
        x, x_prev = g(x), x
        i += 1
        if i > threshold:
            break
    return x, i


def solve_fixed_point(nnet, rhs, start, atol, rtol, threshold=1000):
    """x = rhs - nnet(x) by Banach iteration from x = start, the tolerance scaled by |start|: (x, iterations).
    iResBlock's inverse has rhs = start = y (iresblock.py:69-79); the Banach fallback of RootFind has rhs = x_embed,
    start = z0 (implicit_block.py:17-28, 74-75).  Without a graph, a compiled branch runs BranchProgram.fixed_point
    (one call per solve where the branch allows it); otherwise the host loop goes through the module, building the
    graph when one is needed."""
    graph_free = not (torch.is_grad_enabled() and (rhs.requires_grad or start.requires_grad
                                                   or any(p.requires_grad for p in nnet.parameters())))
    prog = _program(nnet) if graph_free else None
    if prog is not None:
        with torch.no_grad():
            return prog.fixed_point(rhs, start, atol, rtol, threshold)
    with torch.set_grad_enabled(not graph_free):
        return find_fixed_point(lambda x: rhs - nnet(x), start, threshold, atol, rtol)


class RootFind(Function):
    """Solve z + nnet_z(z) = x + nnet_x(x) for z without building a graph (implicit_block.py:51-100)."""
    last_info = None   # result dict of the most recent Broyden solve (read by tests / bench)

    @staticmethod
    def f(nnet_z, nnet_x, z, x):
        return nnet_x(x) - nnet_z(z)

    @staticmethod
    def banach_find_root(nnet_z, nnet_x, z0, x, *args):
        eps, threshold = args[-2], args[-1]
        x_embed = branch_eval(nnet_x, x) + x
        z_est, _ = solve_fixed_point(nnet_z, x_embed, z0, eps, eps, threshold)
        return z_est.clone().detach()

    @staticmethod
    def broyden_find_root(nnet_z, nnet_x, z0, x, *args):
        eps, threshold = args[-2], args[-1]
        x_embed = ops.lincomb3(branch_eval(nnet_x, x, keep=getattr(nnet_x, 'training', False)), 1.0, x, 1.0)
        prog_z = _program(nnet_z)
        if prog_z is not None:
            info = prog_z.solve(0, x_embed, None, threshold, eps)
        else:
            def g(z):     # x_embed - nnet_z(z) - z in one kernel (implicit_block.py:72)
                return ops.lincomb3(x_embed, 1.0, branch_eval(nnet_z, z), -1.0, z, -1.0)

            info = broyden(g, torch.zeros_like(z0), threshold=threshold, eps=eps, name='forward')
        RootFind.last_info = info
        if info['prot_break']:
            return RootFind.banach_find_root(nnet_z, nnet_x, z0, x, eps, 1000)
        return info['result'].detach()          # already a private copy of the solver's best iterate

    @staticmethod
    def forward(ctx, nnet_z, nnet_x, z0, x, method, *args):
        root_find = RootFind.broyden_find_root if method == 'broyden' else RootFind.banach_find_root
        ctx.args_len = len(args)
        with torch.no_grad():
            return _timed('fwd', x, lambda: root_find(nnet_z, nnet_x, z0, x, *args))

    @staticmethod
    def backward(ctx, grad_z):
        assert 0, 'Cannot backward to this function.'


class imBlock(nn.Module):

    def __init__(self, nnet_x, nnet_z, geom_p=0.5, lamb=2., n_power_series=None, exact_trace=False,
                 brute_force=False, n_samples=1, n_exact_terms=2, n_exact_terms_test=20, n_dist='geometric',
                 neumann_grad=True, grad_in_forward=True, eps_forward=1e-6, eps_backward=1e-10, eps_sample=1e-5,
                 threshold=30):
        super(imBlock, self).__init__()
        self.nnet_x = nnet_x
        self.nnet_z = nnet_z
        # frozen twins used by the implicit backward; kept for state-dict compatibility (:136-141)
        self.nnet_x_copy = copy.deepcopy(self.nnet_x)
        self.nnet_z_copy = copy.deepcopy(self.nnet_z)
        for p in self.nnet_x_copy.parameters():
            p.requires_grad_(False)
        for p in self.nnet_z_copy.parameters():
            p.requires_grad_(False)
        self.n_dist = n_dist
        # quirk #12: geom_p ends up a plain fp32 tensor (not in the state dict), lamb a Parameter
        self.geom_p = nn.Parameter(torch.tensor(np.log(geom_p) - np.log(1. - geom_p))).float()
        self.lamb = nn.Parameter(torch.tensor(lamb)).float()
        self.n_samples = n_samples
        self.n_power_series = n_power_series
        self.exact_trace = exact_trace
        self.brute_force = brute_force
        self.n_exact_terms = n_exact_terms
        self.n_exact_terms_test = n_exact_terms_test
        self.grad_in_forward = grad_in_forward
        self.neumann_grad = neumann_grad
        self.eps_forward = eps_forward
        self.eps_backward = eps_backward
        self.eps_sample = eps_sample
        self.threshold = threshold
        self.register_buffer('last_n_samples', torch.zeros(self.n_samples))
        self.register_buffer('last_firmom', torch.zeros(1))
        self.register_buffer('last_secmom', torch.zeros(1))
        # hooks for tests / multi-GPU parity: inject the roulette draw and the probes
        self._inject_n = None
        self._inject_probes = None
        self.solver_stats = {}

    class Backward(Function):
        """Identity in forward; implicit differentiation in backward (implicit_block.py:165-217):
        solve v^T (I + J_z) = grad with Broyden, then dl_dx = v^T (I + J_x)."""
        last_info = None
        x_alias = None
        stats_sink = None        # the calling block's solver_stats dict: receives the backward solve's info as 'bwd'

        @staticmethod
        def forward(ctx, nnet_z, nnet_x, z, x, *args):
            ctx.save_for_backward(z, x)
            ctx.nnet_z = nnet_z
            ctx.nnet_x = nnet_x
            ctx.args = args
            ctx.stats, imBlock.Backward.stats_sink = imBlock.Backward.stats_sink, None
            # a detached tensor with x's values whose saved forward the x-branch program may still hold
            ctx.x_alias, imBlock.Backward.x_alias = imBlock.Backward.x_alias, None
            return z

        @staticmethod
        def backward(ctx, grad):
            grad = grad.clone()
            z, x = ctx.saved_tensors
            args = ctx.args
            eps, threshold = args[-2:]
            nnet_z, nnet_x = ctx.nnet_z, ctx.nnet_x
            prog_z, prog_x = _program(nnet_z), _program(nnet_x)
            if prog_z is not None and prog_x is not None:
                # graph-free: v^T (I + J_z) from the fused vjp kernels
                with torch.no_grad():
                    z, x = z.detach(), x.detach()
                    _, saved_z = prog_z.forward_saved(z)
                    # everything the x-branch vjp behind the solve needs is set up in front of it (the solve drains
                    # the stream: host work after it runs while the GPU idles)
                    xa = ctx.x_alias if (ctx.x_alias is not None and ctx.x_alias.shape == x.shape) else x
                    _, saved_x = prog_x.forward_saved(xa)
                    prog_x.prepare_vjp(saved_x)

                    info = _timed('bwd', grad, lambda: prog_z.solve(1, grad, saved_z, threshold, eps))
                    imBlock.Backward.last_info = info
                    if ctx.stats is not None:
                        ctx.stats['bwd'] = info
                    dl_dh = info['result']
                    dl_dx = ops.lincomb3(prog_x.vjp(dl_dh, saved_x), 1.0, dl_dh, 1.0)
                return (None, None, dl_dh, dl_dx) + (None,) * len(args)
            z = z.clone().detach().requires_grad_()
            x = x.clone().detach().requires_grad_()
            with torch.enable_grad():
                Fz = nnet_z(z) + z

            def g(v):     # v^T dFz/dz - grad: one vjp through the branch per call (:199-203)
                with ops.activations_only():
                    (vJ,) = torch.autograd.grad(Fz, z, v, retain_graph=True)
                return ops.lincomb3(vJ, 1.0, grad, -1.0)

            info = _timed('bwd', grad, lambda: broyden(g, torch.zeros_like(grad), threshold=threshold, eps=eps,
                                                       name='backward'))
            imBlock.Backward.last_info = info
            if ctx.stats is not None:
                ctx.stats['bwd'] = info
            dl_dh = info['result']
            del Fz
            with torch.enable_grad():
                Fx = nnet_x(x) + x
            with ops.activations_only():
                (dl_dx,) = torch.autograd.grad(Fx, x, dl_dh)
            return (None, None, dl_dh, dl_dx) + (None,) * len(args)

    def forward(self, x, logpx=None, restore=False):
        z0 = x.clone().detach()
        self._z0 = z0          # same values as x: lets the x-branch estimate reuse the saved forward at z0
        if restore:
            with torch.no_grad():
                _ = self.nnet_x_copy(z0)
                _ = self.nnet_z_copy(z0)
        # Host-side work that does not depend on the solve goes IN FRONT of it: the solve drains the stream, so
        # whatever the host still has to do afterwards runs while the GPU idles.  The twin refresh copies weights the
        # solve does not change; the roulette draw and the probes come from generators the solve does not touch, in
        # the reference's order (n, then vareps_x, vareps_z; :270-298), so every stream position is unchanged.
        early = HOST_AHEAD['on'] and x.is_cuda
        synced = False
        if early:
            # == load_state_dict(state_dict()) (:228-229); before the first use of a net its u / v are not shaped yet
            # (the solve does that): then the refresh stays behind the solve
            synced = _sync_twin(self.nnet_x_copy, self.nnet_x, fallback=False) and \
                _sync_twin(self.nnet_z_copy, self.nnet_z, fallback=False)
            versions = _twin_versions(self.nnet_x) + _twin_versions(self.nnet_z) if synced else None
            self._pre = self._predraw(z0) if logpx is not None else None
        z = RootFind.apply(self.nnet_z, self.nnet_x, z0, z0, 'broyden', self.eps_forward, self.threshold)
        self.solver_stats['fwd'] = RootFind.last_info
        # re-attach: gradients reach the branch parameters through this expression (:227).  The z-branch evaluation is
        # issued first: it launches kernels on an empty stream, the x-branch value is a memo hit (host work only)
        fz = branch_apply(self.nnet_z, z.detach())
        z = branch_apply(self.nnet_x, z0) - fz + z0
        if synced and versions != _twin_versions(self.nnet_x) + _twin_versions(self.nnet_z):
            synced = False          # the forward wrote a buffer of the live nets (scale, lazily shaped u / v)
        if not synced:
            _sync_twin(self.nnet_x_copy, self.nnet_x)
            _sync_twin(self.nnet_z_copy, self.nnet_z)
        if FUSED['on']:      # the frozen twins hold the same weights: share the live nets' programs
            self.nnet_z_copy._impflow_program = _program(self.nnet_z)
            self.nnet_x_copy._impflow_program = _program(self.nnet_x)
        imBlock.Backward.x_alias = z0
        imBlock.Backward.stats_sink = self.solver_stats
        z = self.Backward.apply(self.nnet_z_copy, self.nnet_x_copy, z, x, 'broyden', self.eps_backward,
                                self.threshold)
        if logpx is None:
            return z
        out = z, logpx - self._logdetgrad(z, x)
        self._z0 = None
        self._pre = None
        return out

    def inverse(self, z, logpy=None):
        x0 = z.clone().detach()
        x = RootFind.apply(self.nnet_x, self.nnet_z, x0, z, 'broyden', self.eps_sample, self.threshold)
        self.solver_stats['inv'] = RootFind.last_info
        if logpy is None:
            return x
        return x, logpy + self._logdetgrad(z, x)

    # --------------------------------------------------------------------------------------
    def _rate(self):
        """geom p / poisson lambda as a python float: one device read per change of the tensor
        (the reference reads it with .item() once per _logdetgrad call, :264-269)."""
        t = self.geom_p if self.n_dist == 'geometric' else self.lamb
        key = (self.n_dist, t._version, t.data_ptr())
        cached = getattr(self, '_rate_cache', None)
        if cached is None or cached[0] != key:
            val = torch.sigmoid(t).item() if self.n_dist == 'geometric' else t.item()
            cached = self._rate_cache = (key, val)
        return cached[1]

    def _draw_n(self):
        if self._inject_n is not None:
            return np.asarray(self._inject_n)
        if self.n_dist == 'geometric':
            return geometric_sample(self._rate(), self.n_samples)
        return poisson_sample(self._rate(), self.n_samples)

    def _rcdf(self, k, offset):
        if self.n_dist == 'geometric':
            return geometric_1mcdf(self._rate(), k, offset)
        return poisson_1mcdf(self._rate(), k, offset)

    def _draw_probes(self, x, z):
        if self._inject_probes is not None:
            vx, vz = self._inject_probes
            return vx.to(x), vz.to(z)
        if PROBE_MODE['mode'] == 'device':
            if x.shape == z.shape and x.dtype == z.dtype and x.device == z.device:
                v = torch.randint(0, 2, (2,) + tuple(x.shape), device=x.device, dtype=x.dtype).mul_(2).sub_(1)
                return v[0], v[1]
            vx = torch.randint(0, 2, x.shape, device=x.device, dtype=x.dtype).mul_(2).sub_(1)
            vz = torch.randint(0, 2, z.shape, device=z.device, dtype=z.dtype).mul_(2).sub_(1)
            return vx, vz
        # same draws as the reference (CPU generator, vareps_x before vareps_z, :297-298); the
        # +-1 values are staged in pinned memory so the upload does not synchronise the stream
        bern = torch.distributions.bernoulli.Bernoulli(torch.Tensor([0.5]))
        vx = _upload(bern.sample(x.shape).reshape(x.shape) * 2 - 1, x)
        vz = _upload(bern.sample(z.shape).reshape(z.shape) * 2 - 1, z)
        return vx, vz

    def _predraw(self, x):
        """The random inputs of the coming _logdetgrad(z, x) call (z has x's shape), drawn before the solve: the
        roulette sample count and the two probe tensors, or None where _logdetgrad draws nothing / something else
        (brute force, exact trace, evaluation mode)."""
        if not self.training or self.exact_trace:
            return None
        if self.brute_force and x.ndimension() == 2 and x.shape[1] <= 10:
            return None
        n_samples = self._draw_n() if self.n_power_series is None else None
        return n_samples, self._draw_probes(x, x)

    def _logdetgrad(self, z, x):
        """logdet |dz/dx| = logdet(I + J_x) - logdet(I + J_z)  (implicit_block.py:245-350)."""
        pre, self._pre = getattr(self, '_pre', None), None
        with torch.enable_grad():
            if (self.brute_force or not self.training) and (x.ndimension() == 2 and x.shape[1] <= 10):
                px, pz = _program(self.nnet_x), _program(self.nnet_z)
                if GRAPH_FREE_BRUTE['on'] and px is not None and pz is not None:
                    # graph-free: Jacobian columns from d tangent sweeps, the gradient from d bilinear-form sweeps
                    return (_GraphFreeBruteForce.apply(x, px, *px.params) -
                            _GraphFreeBruteForce.apply(z, pz, *pz.params)).view(-1, 1)
                x = x.requires_grad_(True)
                z = z.requires_grad_(True)
                Jx = batch_jacobian(x + self.nnet_x(x), x)
                Jz = batch_jacobian(z + self.nnet_z(z), z)
                return (torch.logdet(Jx) - torch.logdet(Jz)).view(-1, 1)

            n_samples = None
            if self.training and self.n_power_series is not None:
                n_power_series = self.n_power_series          # truncated (biased) estimation
                coeff_fn = lambda k: 1.
            else:
                n_exact = self.n_exact_terms if self.training else self.n_exact_terms_test
                n_samples = pre[0] if pre is not None else self._draw_n()
                n_power_series = int(max(n_samples) + n_exact)
                coeff_fn = lambda k: 1 / self._rcdf(k, n_exact) * sum(n_samples >= k - n_exact) / len(n_samples)

            if not self.exact_trace:
                vareps_x, vareps_z = pre[1] if pre is not None else self._draw_probes(x, z)
                if self.training and self.neumann_grad:
                    estimator_fn = neumann_logdet_estimator
                else:
                    estimator_fn = basic_logdet_estimator
                if self.training and self.grad_in_forward:
                    # the two estimates are independent: the z-branch runs on a side stream so that kernels
                    # that cannot fill the GPU on their own (the deeper, smaller scales) overlap
                    # (only the graph-free evaluations: the autograd nodes are created on the current stream)
                    est = MemoryEfficientLogDetEstimator
                    with _overlap(x) as side:
                        with side:
                            pz = est.payload(estimator_fn, self.nnet_z, z, n_power_series, vareps_z, coeff_fn, True)
                        z0 = getattr(self, '_z0', None)
                        x_at = z0 if (z0 is not None and z0.shape == x.shape and z0.device == x.device) else x
                        px = est.payload(estimator_fn, self.nnet_x, x_at, n_power_series, vareps_x, coeff_fn, True)
                    logdet_x = mem_eff_wrapper(estimator_fn, self.nnet_x, x, n_power_series, vareps_x, coeff_fn,
                                               self.training, px)
                    logdet_z = mem_eff_wrapper(estimator_fn, self.nnet_z, z, n_power_series, vareps_z, coeff_fn,
                                               self.training, pz)
                else:
                    x = x.requires_grad_(True)
                    z = z.requires_grad_(True)
                    logdet_x = estimator_fn(self.nnet_x(x), x, n_power_series, vareps_x, coeff_fn, self.training,
                                            _program(self.nnet_x))
                    logdet_z = estimator_fn(self.nnet_z(z), z, n_power_series, vareps_z, coeff_fn, self.training,
                                            _program(self.nnet_z))
                logdetgrad = logdet_x - logdet_z
            else:
                x = x.requires_grad_(True)
                z = z.requires_grad_(True)
                logdetgrad = _exact_trace_series(self.nnet_x(x), x, n_power_series, coeff_fn) - \
                    _exact_trace_series(self.nnet_z(z), z, n_power_series, coeff_fn)

            if self.training and self.n_power_series is None:
                # pinned staging: a pageable H2D copy would wait for every kernel queued so far (a device sync
                # per imBlock and step)
                self.last_n_samples.copy_(_upload(torch.as_tensor(np.asarray(n_samples), dtype=torch.float32),
                                                  self.last_n_samples))
                estimator = logdetgrad.detach()
                self.last_firmom.copy_(torch.mean(estimator).to(self.last_firmom))
                self.last_secmom.copy_(torch.mean(estimator ** 2).to(self.last_secmom))
            return logdetgrad.view(-1, 1)

    def extra_repr(self):
        return ('dist={}, n_samples={}, n_power_series={}, neumann_grad={}, exact_trace={}, brute_force={}, '
                'grad_in_forward={}'.format(self.n_dist, self.n_samples, self.n_power_series, self.neumann_grad,
                                            self.exact_trace, self.brute_force, self.grad_in_forward))


def batch_jacobian(g, x, create_graph=True):
    """(B,d,d) Jacobian from d vjps (implicit_block.py:358-362)."""
    rows = []
    for j in range(g.shape[1]):
        with ops.activations_only():
            (r,) = torch.autograd.grad(torch.sum(g[:, j]), x, create_graph=create_graph)
        rows.append(r.view(x.shape[0], 1, x.shape[1]))
    return torch.cat(rows, 1)


def batch_trace(M):
    return M.view(M.shape[0], -1)[:, ::M.shape[1] + 1].sum(1)


def _exact_trace_series(g, x, n_power_series, coeff_fn):
    J = batch_jacobian(g, x)
    out = batch_trace(J)
    Jk = J
    for k in range(2, n_power_series + 1):
        Jk = torch.bmm(J, Jk)
        out = out + (-1) ** (k + 1) / k * coeff_fn(k) * batch_trace(Jk)
    return out


# ------------------------------------------------------------------------------------------
# log-det estimators
# ------------------------------------------------------------------------------------------

class MemoryEfficientLogDetEstimator(torch.autograd.Function):
    """Back-prop in forward: the gradients of the estimate w.r.t. x and the branch parameters
    are taken immediately and only scaled in backward (implicit_block.py:373-415)."""

    @staticmethod
    def payload(estimator_fn, gnet, x, n_power_series, vareps, coeff_fn, training):
        """The graph-free evaluation (estimate, d/dx, d/dtheta) of the Neumann estimator: fused forward, the
        n-term vjp chain, then the hand-derived tangent / reverse sweeps.  Plain tensors in and out, so it can
        run on a side stream; None when this branch / estimator has no graph-free form."""
        prog = _program(gnet)
        if not (training and prog is not None and estimator_fn is neumann_logdet_estimator):
            return None
        with torch.no_grad():
            xd = x.detach()
            _, saved = prog.forward_saved(xd)
            coeffs = [float((-1) ** k * coeff_fn(k)) for k in range(1, n_power_series + 1)]
            return prog.neumann(saved, prog.neumann_chain(saved, vareps, coeffs), vareps)

    @staticmethod
    def forward(ctx, estimator_fn, gnet, x, n_power_series, vareps, coeff_fn, training, payload, *g_params):
        ctx.training = training
        ctx.g_params = g_params
        if payload is None:
            payload = MemoryEfficientLogDetEstimator.payload(estimator_fn, gnet, x, n_power_series, vareps, coeff_fn,
                                                             training)
        if payload is not None:
            logdetgrad, grad_x, grad_params = payload
            ctx.none_mask = [gp is None for gp in grad_params]
            ctx.save_for_backward(grad_x, *[gp if gp is not None else grad_x.new_zeros(()) for gp in grad_params])
            return logdetgrad
        prog = _program(gnet)
        with torch.enable_grad():
            x = x.detach().requires_grad_(True)
            g = gnet(x)
            logdetgrad = estimator_fn(g, x, n_power_series, vareps, coeff_fn, training, prog)
            if training:
                grad_x, *grad_params = torch.autograd.grad(logdetgrad.sum(), (x,) + g_params, retain_graph=False,
                                                           allow_unused=True)
                if grad_x is None:
                    grad_x = torch.zeros_like(x)
                ctx.none_mask = [gp is None for gp in grad_params]
                ctx.save_for_backward(grad_x, *[gp if gp is not None else x.new_zeros(()) for gp in grad_params])
        return safe_detach(logdetgrad)

    @staticmethod
    def backward(ctx, grad_logdetgrad):
        if not ctx.training:
            raise ValueError('Provide training=True if using backward.')
        grad_x, *grad_params = ctx.saved_tensors
        dL = grad_logdetgrad[0].detach()      # quirk #13: assumes a uniform upstream gradient
        with torch.no_grad():
            # one multi-tensor launch for the whole list instead of one small kernel per parameter
            live = [grad_x] + [gp for gp, m in zip(grad_params, ctx.none_mask) if not m]
            scaled = iter(torch._foreach_mul(live, dL.reshape(())))
            grad_x = next(scaled)
            grad_params = tuple(sink_grads(ctx.g_params, [None if m else next(scaled) for m in ctx.none_mask]))
        return (None, None, grad_x, None, None, None, None, None) + grad_params


GRAPH_FREE_BRUTE = {'on': True}     # brute-force log-det (d <= 10) without the autograd double backward


class _GraphFreeBruteForce(Function):
    """logdet(I + J(x)) of a small-d branch (implicit_block.py:249-260) WITH its gradient, graph-free.  The reference
    assembles J from d autograd passes with create_graph=True and differentiates torch.logdet through them.  Here:
        forward : column j of J = J e_j from one tangent sweep (d sweeps), logdet(I + J) by the library LU on (B, d, d)
        backward: d logdet = tr((I + J)^-1 dJ) = sum_j a_j^T (dJ) e_j with a_j = row j of (I + J)^-1: d bilinear-form
                  gradients at the saved point (BranchProgram.neumann), seeded with the upstream gradient."""

    @staticmethod
    def forward(ctx, x, prog, *params):
        xd = x.detach()
        B, d = xd.shape
        _, saved = prog.forward_saved(xd)
        eye = torch.eye(d, device=xd.device, dtype=xd.dtype)
        cols = [prog.tangent(saved, eye[j].expand(B, d).contiguous()) for j in range(d)]
        M = torch.stack(cols, 2) + eye                    # M[b, i, j] = delta_ij + d g_i / d x_j
        ctx.prog, ctx.saved_fwd, ctx.M = prog, saved, M
        return torch.logdet(M)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        prog, saved, M = ctx.prog, ctx.saved_fwd, ctx.M
        B, d = M.shape[0], M.shape[1]
        Minv = torch.linalg.inv(M)                        # (B, d, d), d <= 10
        eye = torch.eye(d, device=M.device, dtype=M.dtype)
        seed = gout.reshape(-1).contiguous()
        gx, gparams = None, None
        for j in range(d):
            w_j = Minv[:, j, :].contiguous()              # row j of the inverse
            _, gx_j, gp_j = prog.neumann(saved, w_j, eye[j].expand(B, d).contiguous(), seed_scale=seed)
            if gx is None:
                gx, gparams = gx_j, list(gp_j)
            else:
                gx = gx + gx_j
                live = [(a, b) for a, b in zip(gparams, gp_j) if a is not None and b is not None]
                if live:
                    torch._foreach_add_([a for a, _ in live], [b for _, b in live])
        ctx.saved_fwd = ctx.M = None
        return (gx, None) + tuple(sink_grads(prog.params, gparams))


GRAPH_FREE_BASIC = {'on': True}     # hand-derived training gradient of the basic estimator (off = autograd double backward)


class _GraphFreeBasic(Function):
    """The basic power-series estimator S = sum_k c_k v^T J^k v (implicit_block.py:418-426) WITH its training
    gradient, graph-free.  The reference builds the n-term vjp chain with create_graph=True and lets autograd
    differentiate through it (double backward).  Here:
        forward : l_0 = v, l_k = J^T l_{k-1} (fused vjp kernels), S = sum_k c_k <l_k, v>
        backward: dS = sum_k c_k sum_{i=1..k} l_{i-1}^T (dJ) r_{k-i},  r_m = J^m v,  which regroups to
                  dS = sum_{m=0..n-1} w_m^T (dJ) r_m,   w_m = sum_{a=0..n-1-m} c_{a+m+1} l_a
                  i.e. n bilinear-form gradients d(w^T J r): each is one tangent sweep (which also yields
                  r_{m+1} = J r_m) and one two-adjoint reverse sweep (BranchProgram.neumann), seeded with the
                  per-sample upstream gradient."""

    @staticmethod
    def forward(ctx, x, prog, vareps, coeffs, *params):
        xd = x.detach()
        _, saved = prog.forward_saved(xd)
        ctx.series = None
        spec = prog.mlp_series_spec(saved) if 1 <= len(coeffs) <= 32 else None
        if spec is not None:
            # small-d MLP branch: both chains, the combinations and the estimate in ONE launch (k_mlp_series)
            out, _, Rs, Wm = ops.mlp_series(spec, vareps, coeffs)
            ctx.series = (Rs, Wm)
            ctx.prog, ctx.saved_fwd, ctx.ls, ctx.coeffs = prog, saved, None, coeffs
            return out
        ls = [vareps]
        out = torch.zeros(xd.shape[0], device=xd.device, dtype=torch.float32)
        for c in coeffs:
            ls.append(prog.vjp(ls[-1], saved))
            ops.rowdot(ls[-1], vareps, out=out, alpha=float(c), beta=1.0)
        ctx.prog, ctx.saved_fwd, ctx.ls, ctx.coeffs = prog, saved, ls, coeffs
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        prog, saved, ls, coeffs = ctx.prog, ctx.saved_fwd, ctx.ls, ctx.coeffs
        n = len(coeffs)
        seed = gout.reshape(-1).contiguous()
        if ctx.series is not None:
            Rs, Wm = ctx.series             # (n, B, d) each: r_m and w_m from the forward's launch
            B, d = Rs.shape[1], Rs.shape[2]
            if n > 1 and prog.sweep_graphable(saved, Rs):
                # CUDA-graph mode of the MLP flows: the n bilinear-form gradients as n replays of ONE graph over B rows
                # (an n-fold batch would need a graph per distinct n, i.e. per roulette draw)
                gx, gparams = None, None
                for m in range(n):
                    _, gx_m, gp_m = prog.neumann(saved, Wm[m], Rs[m], seed_scale=seed)
                    if gx is None:
                        gx, gparams = gx_m, list(gp_m)
                    else:
                        gx = gx + gx_m
                        live = [(a, b) for a, b in zip(gparams, gp_m) if a is not None and b is not None]
                        if live:
                            torch._foreach_add_([a for a, _ in live], [b for _, b in live])
            elif n > 1:
                saved_n = prog.tile_saved(saved, n)
                _, gx_n, gparams = prog.neumann(saved_n, Wm.view(n * B, d), Rs.view(n * B, d), seed_scale=seed.repeat(n))
                gx = gx_n.reshape(n, B, d).sum(0)
            else:
                _, gx, gparams = prog.neumann(saved, Wm[0], Rs[0], seed_scale=seed)
            ctx.series = ctx.saved_fwd = None
            return (gx, None, None, None) + tuple(sink_grads(prog.params, gparams))
        B = ls[0].shape[0]
        # right vectors r_m = J^m v (n - 1 tangent sweeps) and left combinations w_m = sum_a c_{a+m+1} l_a
        rs = [ls[0]]
        for _ in range(n - 1):
            rs.append(prog.tangent(saved, rs[-1]))
        wsum = []
        for m in range(n):
            w = None
            for a in range(n - m):
                c = float(coeffs[a + m])
                w = ops.lincomb3(ls[a], c) if w is None else ops.lincomb3(w, 1.0, ls[a], c)
            wsum.append(w)
        # all n bilinear-form gradients in ONE two-adjoint sweep over an n-fold batch (same point, same weights:
        # the parameter gradients are sums over rows anyway; the input gradient is summed over the n copies)
        if n > 1:
            saved_n = prog.tile_saved(saved, n)
            _, gx_n, gparams = prog.neumann(saved_n, torch.cat(wsum, 0), torch.cat(rs, 0), seed_scale=seed.repeat(n))
            gx = gx_n.reshape((n, B) + tuple(gx_n.shape[1:])).sum(0)
        else:
            _, gx, gparams = prog.neumann(saved, wsum[0], rs[0], seed_scale=seed)
        ctx.ls = ctx.saved_fwd = None
        return (gx, None, None, None) + tuple(sink_grads(prog.params, gparams))


def basic_logdet_estimator(g, x, n_power_series, vareps, coeff_fn, training, program=None):
    """sum_k (-1)^(k+1)/k coeff(k) <v^T J^k, v>  (implicit_block.py:418-426)."""
    if not training and program is not None:
        # eval mode builds no graph: the whole chain runs on the fused vjp kernels
        with torch.no_grad():
            _, saved = program.forward_saved(x.detach())
            return program.hutchinson_series(saved, vareps, [(-1) ** (k + 1) / k * coeff_fn(k)
                                                             for k in range(1, n_power_series + 1)])
    if training and program is not None and GRAPH_FREE_BASIC['on'] and n_power_series >= 1:
        coeffs = [(-1) ** (k + 1) / k * coeff_fn(k) for k in range(1, n_power_series + 1)]
        return _GraphFreeBasic.apply(x, program, vareps, coeffs, *program.params)
    vjp = vareps
    logdetgrad = torch.zeros((), device=x.device, dtype=x.dtype)
    for k in range(1, n_power_series + 1):
        with ops.activations_only():
            vjp = torch.autograd.grad(g, x, vjp, create_graph=training, retain_graph=True)[0]
        tr = ops.rowdot_fn(vjp, vareps)
        logdetgrad = logdetgrad + (-1) ** (k + 1) / k * coeff_fn(k) * tr
    return logdetgrad


def neumann_logdet_estimator(g, x, n_power_series, vareps, coeff_fn, training, program=None):
    """Neumann-series gradient estimator: a surrogate whose gradient is unbiased for the log-det
    gradient (implicit_block.py:429-438)."""
    vjp = vareps
    neumann_vjp = vareps
    with torch.no_grad():
        if program is not None:
            program.forward(x.detach(), save=True)
        for k in range(1, n_power_series + 1):
            if program is not None:
                vjp = program.vjp(vjp)
            else:
                with ops.activations_only():
                    vjp = torch.autograd.grad(g, x, vjp, retain_graph=True)[0]
            neumann_vjp = ops.lincomb3(neumann_vjp, 1.0, vjp, float((-1) ** k * coeff_fn(k)))
    with ops.activations_only():
        vjp_jac = torch.autograd.grad(g, x, neumann_vjp, create_graph=training)[0]
    return ops.rowdot_fn(vjp_jac, vareps)


def mem_eff_wrapper(estimator_fn, gnet, x, n_power_series, vareps, coeff_fn, training, payload=None):
    if not isinstance(gnet, nn.Module):
        raise ValueError('g is required to be an instance of nn.Module.')
    return MemoryEfficientLogDetEstimator.apply(estimator_fn, gnet, x, n_power_series, vareps, coeff_fn, training,
                                                payload, *list(gnet.parameters()))


# ---- roulette helpers: python floats, global NumPy RNG (implicit_block.py:457-483) -----------

def geometric_sample(p, n_samples):
    return np.random.geometric(p, n_samples)


def geometric_1mcdf(p, k, offset):
    """P(n >= k - offset)"""
    if k <= offset:
        return 1.
    k = k - offset
    return (1 - p) ** max(k - 1, 0)


def poisson_sample(lamb, n_samples):
    return np.random.poisson(lamb, n_samples)


def poisson_1mcdf(lamb, k, offset):
    """P(n >= k - offset)"""
    if k <= offset:
        return 1.
    k = k - offset
    s = 1.
    for i in range(1, k):
        s += lamb ** i / math.factorial(i)
    return 1 - np.exp(-lamb) * s


def safe_detach(tensor):
    return tensor.detach().requires_grad_(tensor.requires_grad)
