"""iResBlock: the explicit residual block y = x + g(x) with the same Russian-roulette power-series log-det
estimators as imBlock — API / state-dict mirror of lib/layers/iresblock.py (block :13-170, fixed-point inverse
:69-79, estimators :186-270).

What runs where (shared with imBlock, see implicit_block.py):
  * g(x) and its first-order backward: the graph-free branch program (one fused forward, one fused backward
    sweep with the weight gradients) whenever the branch is compilable;
  * training log-det with neumann_grad + grad_in_forward (the configuration the image flows use): the no-grad
    vjp chain and the hand-derived gradient of the Neumann surrogate (branch_program.neumann), saved and scaled
    in backward exactly like the reference's MemoryEfficientLogDetEstimator (:186-235) — the reference's variant
    also returns g and back-propagates grad_g through the kept graph; here g is the output of the branch
    program's own autograd node, so autograd adds the two contributions;
  * eval-mode log-det (20 exact terms): the vjp chain on the fused kernels with in-place Hutchinson dots;
  * inverse: Banach iteration x <- y - g(x) (:69-79), convergence test as in the reference: one call per solve on
    the native conv runtime or the persistent MLP kernel where the branch allows it (BranchProgram.fixed_point).
Gaussian probes are drawn with randn_like on the device like the reference does (:129); tests inject them.

`forward` additionally accepts (and ignores) `restore=`: SequentialFlow passes it to every layer, which makes
the reference's own iResBlock unusable inside a flow (SURVEY.md quirk #20)."""
import numpy as np
import torch
import torch.nn as nn

from . import implicit_block as ib

__all__ = ['iResBlock']


class iResBlock(nn.Module):

    def __init__(self, nnet, geom_p=0.5, lamb=2., n_power_series=None, exact_trace=False, brute_force=False,
                 n_samples=1, n_exact_terms=2, n_dist='geometric', neumann_grad=True, grad_in_forward=False):
        nn.Module.__init__(self)
        self.nnet = nnet
        self.n_dist = n_dist
        self.geom_p = nn.Parameter(torch.tensor(np.log(geom_p) - np.log(1. - geom_p)))   # float64 Parameter (quirk #12)
        self.lamb = nn.Parameter(torch.tensor(lamb))
        self.n_samples = n_samples
        self.n_power_series = n_power_series
        self.exact_trace = exact_trace
        self.brute_force = brute_force
        self.n_exact_terms = n_exact_terms
        self.grad_in_forward = grad_in_forward
        self.neumann_grad = neumann_grad
        self.register_buffer('last_n_samples', torch.zeros(self.n_samples))
        self.register_buffer('last_firmom', torch.zeros(1))
        self.register_buffer('last_secmom', torch.zeros(1))
        # hooks for tests / multi-GPU parity: inject the roulette draw and the probe
        self._inject_n = None
        self._inject_probes = None
        self.inverse_iterations = None      # Banach iterations of the latest inverse()

    def forward(self, x, logpx=None, restore=False):
        if logpx is None:
            return x + ib.branch_apply(self.nnet, x)
        g, logdetgrad = self._logdetgrad(x)
        return x + g, logpx - logdetgrad

    def inverse(self, y, logpy=None):
        x = self._inverse_fixed_point(y)
        if logpy is None:
            return x
        return x, logpy + self._logdetgrad(x)[1]

    def _inverse_fixed_point(self, y, atol=1e-5, rtol=1e-5):
        """x <- y - g(x) until every (x - x_prev)^2 / (atol + rtol |y|) < 1, cap 1000 (iresblock.py:69-79)."""
        x, self.inverse_iterations = ib.solve_fixed_point(self.nnet, y, y, atol, rtol, 1000)
        return x

    # --------------------------------------------------------------------------------------
    def _rate(self):
        t = self.geom_p if self.n_dist == 'geometric' else self.lamb
        key = (self.n_dist, t._version, t.data_ptr())
        cached = getattr(self, '_rate_cache', None)
        if cached is None or cached[0] != key:
            val = torch.sigmoid(t).item() if self.n_dist == 'geometric' else t.item()
            cached = self._rate_cache = (key, val)
        return cached[1]

    def _roulette(self):
        """(n_power_series, coeff_fn, n_samples or None) of this call (iresblock.py:96-123)."""
        if self.training and self.n_power_series is not None:
            return self.n_power_series, (lambda k: 1.), None          # truncated (biased) estimation
        rate = self._rate()
        if self.n_dist == 'geometric':
            sample_fn, rcdf = ib.geometric_sample, (lambda k, off: ib.geometric_1mcdf(rate, k, off))
        else:
            sample_fn, rcdf = ib.poisson_sample, (lambda k, off: ib.poisson_1mcdf(rate, k, off))
        n_exact = self.n_exact_terms if self.training else 20       # hard-coded 20 in eval (quirk #17)
        n_samples = np.asarray(self._inject_n) if self._inject_n is not None else sample_fn(rate, self.n_samples)
        coeff_fn = lambda k: 1 / rcdf(k, n_exact) * sum(n_samples >= k - n_exact) / len(n_samples)
        return int(max(n_samples) + n_exact), coeff_fn, n_samples

    def _logdetgrad(self, x):
        """Returns g(x) and logdet|d(x+g(x))/dx|  (iresblock.py:81-164)."""
        with torch.enable_grad():
            if (self.brute_force or not self.training) and (x.ndimension() == 2 and x.shape[1] == 2):
                # closed-form 2x2 determinant of I + J (:85-94)
                x = x.requires_grad_(True)
                g = self.nnet(x)
                jac = ib.batch_jacobian(g, x)
                dets = (jac[:, 0, 0] + 1) * (jac[:, 1, 1] + 1) - jac[:, 0, 1] * jac[:, 1, 0]
                return g, torch.log(torch.abs(dets)).view(-1, 1)

            n_power_series, coeff_fn, n_samples = self._roulette()
            if not self.exact_trace:
                vareps = self._inject_probes.to(x) if self._inject_probes is not None else torch.randn_like(x)
                if self.training and self.neumann_grad:
                    estimator_fn = ib.neumann_logdet_estimator
                else:
                    estimator_fn = ib.basic_logdet_estimator
                if self.training and self.grad_in_forward:
                    g = ib.branch_apply(self.nnet, x)
                    logdetgrad = ib.mem_eff_wrapper(estimator_fn, self.nnet, x, n_power_series, vareps, coeff_fn,
                                                    self.training)
                else:
                    x = x.requires_grad_(True)
                    g = self.nnet(x)
                    logdetgrad = estimator_fn(g, x, n_power_series, vareps, coeff_fn, self.training,
                                              ib._program(self.nnet))
            else:
                x = x.requires_grad_(True)
                g = self.nnet(x)
                logdetgrad = ib._exact_trace_series(g, x, n_power_series, coeff_fn)

            if self.training and self.n_power_series is None:
                self.last_n_samples.copy_(ib._upload(torch.as_tensor(np.asarray(n_samples), dtype=torch.float32),
                                                     self.last_n_samples))
                estimator = logdetgrad.detach()
                self.last_firmom.copy_(torch.mean(estimator).to(self.last_firmom))
                self.last_secmom.copy_(torch.mean(estimator ** 2).to(self.last_secmom))
            return g, logdetgrad.view(-1, 1)

    def extra_repr(self):
        return 'dist={}, n_samples={}, n_power_series={}, neumann_grad={}, exact_trace={}, brute_force={}'.format(
            self.n_dist, self.n_samples, self.n_power_series, self.neumann_grad, self.exact_trace, self.brute_force)
