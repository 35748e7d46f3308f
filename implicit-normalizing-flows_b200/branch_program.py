"""Graph-free evaluation of a residual branch: forward, vjp, first-order backward and the
hand-derived gradient of the Neumann log-det estimator — all as short sequences of impflow
kernel launches, with no autograd graph.

Why: an ImpFlow step evaluates each branch ~60 times (Broyden g evaluations, implicit-backward
vjps, the n-term vjp chain of the power series, the estimator's double backward).  Driving every
one of them through nn.Module.__call__ + autograd costs thousands of tiny launches; the arithmetic
is a handful of GEMMs.  A BranchProgram compiles an nn.Sequential of
    [act] layer act layer ... layer [act]
(InducedNormLinear / InducedNormConv2d and LopLinear / LopConv2d, 1x1 / 3x3, + Sin / Swish / ReLU: every branch the
shipped configs build — train_toy.py:146-171, train_tabular.py:292-311, implicit_flow.py:359-398,
train_classification.py:152-167) into:

  forward(x)            nnet(x)                                      (implicit_block.py:68-80)
  vjp(v)                v^T J                                        (:199-203, :432-435)
  backward_full(g)      (g^T J, dL/dtheta)  for z = f_x(z0) - f_z(z*) + z0   (:227)
  neumann(w, v)         S = <w^T J, v>, dS/dx, dS/dtheta             (:386-388, :429-438)

Layer forms (rows = pixels or samples, channels contiguous):
  mm   : linear / 1x1 conv          y = A W^T
  c3 A : 3x3, cin <= cout           y = im2col(A) Wr^T        transpose: col2im(G W2t^T)
  c3 B : 3x3, cin >  cout           y = col2im(A W2^T)        transpose: im2col(G) Wrt^T
The rescaled weights (compute_weight(update=False) of an induced-norm layer, compute_weight() of a Lop layer), their GEMM
re-layouts and tf32 hi/lo planes are cached until a parameter / u / v / beta changes version.

neumann() differentiates S = sum_b <w_b, J_b v_b> by hand: S is the forward-mode tangent of the
branch in direction v contracted with w, so one tangent sweep (t_{l} = W phi'(p) t_{l-1}) plus one
reverse sweep carrying two adjoints per layer (of the tangent and of the primal) replaces
autograd's double backward:
    tbar_a = W^T tbar_y                abar = W^T ybar
    Wbar  += tbar_y (x) t_a + ybar (x) a          bbar += sum ybar
    tbar_p = phi'(p) tbar_a            pbar = phi''(p) t_p tbar_a + phi'(p) abar
"""
import ctypes
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi, ops
from .layers import broyden as _broyden
from .layers.base.activations import ReLU, Sin, Swish
from .layers.base.lipschitz import LopConv2d, LopLinear
from .layers.base.mixed_lipschitz import InducedNormConv2d, InducedNormLinear, sigma_of

__all__ = ['BranchProgram', 'compile_branch', 'FUSED3', 'CONV3_NATIVE', 'MEMO', 'SWEEP_GRAPHS', 'MLP_SERIES']

# One-launch tile kernel for the 3-layer conv branch (csrc/branch_fused.cu); off = three GEMM launches.
FUSED3 = {'on': True}
# Native host runtime for the 3-layer conv branch (csrc/conv3_plan.cu): one C call per evaluation / power
# series / Broyden solve; off = the Python-driven launch sequences below.
CONV3_NATIVE = {'on': True}

# Every Broyden solve of a small MLP branch (forward / inverse and implicit backward) in one launch of the persistent
# solver kernel (csrc/mlp_solver.cu); off = the generic kernel loop of layers/broyden.py.
MLP_SOLVER = {'on': True}
FUSED_SN_GRAD = {'on': True}     # weight-layout gradient + spectral chain in one C call
# One-pass activation step of the Neumann reverse sweep (csrc/elementwise.cu: k_neumann_act_bwd); off = act_second +
# two act_beta_grad + colsum + split.
NEUMANN_FUSED = {'on': True}

# The same branch is evaluated at the same point several times per step (nnet_x(x) for x_embed, for the
# re-attach and for the log-det estimate; nnet_z(z) for the estimate and again in the implicit backward).  The
# last saved forward of a program is kept and handed out again while input storage, version and weights match.
MEMO = {'on': True}
# CUDA graphs of the Python-driven gradient sweeps (BranchProgram.backward_full / neumann) where they are host-bound:
# conv branches with at most max_rows pixel rows (B=64: the deepest CIFAR scale; smaller per-GPU batches, i.e. strong
# scaling: more of them), captured after `warmup` eager calls.  Measured (bench.py, e2e ms/step, B200): B=64 71.6 ->
# 69.6 (max_rows 8192; 20000: 70.9), B=16 46.8 -> 38.0.
# 'mlp': graphs of the MLP flows' sweeps too.  The basic estimator's n bilinear-form gradients then run as n replays of
# ONE graph over B rows (layers/implicit_block.py _GraphFreeBasic.backward) instead of one sweep over an n-fold batch,
# whose row count follows the roulette draw and would need a graph per distinct n (~200 captures of ~28 ms for a
# 20-block flow); with one graph per program and sweep kind the 80 captures fall into the first two steps.
TC_MIN_FLOPS = {'program': 2.5e8}      # smallest GEMM a branch program sends to the tcgen05 kernel in 'auto' mode
MLP_SERIES = {'on': True}      # one-launch vjp / tangent chains of the basic estimator's training path (MLP branches)
SWEEP_GRAPHS = {'on': True, 'max_rows': 16384, 'warmup': 1, 'mlp': True}

_LINEAR = (InducedNormLinear, LopLinear)          # layers of the linear kind; the others are convolutions
_LOP = (LopLinear, LopConv2d)                       # closed-form operator-norm layers (rescaled by group norms)
_conv3_ws = {}      # (device index, stream) -> workspace tensor shared by every plan used on that stream


def _conv3_workspace(n_floats, device):
    key = (device.index, torch._C._cuda_getCurrentRawStream(device.index) if device.type == 'cuda' else 0)
    t = _conv3_ws.get(key)
    if t is None or t.numel() < n_floats:
        t = _conv3_ws[key] = torch.empty(int(n_floats), device=device, dtype=torch.float32)
    return t


def _device_solve(t):
    """Whether the one-call fixed-point solves take `t`: they drive a CUDA stream (evaluations enqueued ahead of the
    device's decisions, progress records in mapped pinned memory, one drain per solve), so CUDA tensors only.  A CPU
    tensor takes the host loop, whose kernel launches refuse it (there is no CPU execution path), as before these
    solves existed; the numpy C-ABI emulator of the CPU test suite runs that loop."""
    return t.is_cuda


def _device_lop(w):
    """Whether a branch with Lop layers whose weight is `w` compiles to a program: the Lop weight preparation and
    gradient chain are CUDA kernels, so CUDA weights only.  A branch on the CPU keeps the module path, as before these
    kernels existed (the product has no CPU execution path; the numpy C-ABI emulator of the CPU test suite runs it)."""
    return w.is_cuda


def _round_up(n, m):
    return (n + m - 1) // m * m


class _Act(object):
    def __init__(self, kind, module=None):
        self.kind = kind
        self.module = module       # Swish module (for beta) or None
        self._beta = None          # softplus(beta) device scalar, refreshed by BranchProgram._prep

    def refresh(self):
        if self.kind == ops.ACT_LIPSWISH:
            self._beta = F.softplus(self.module.beta.detach())

    def beta_sp(self):
        if self.kind != ops.ACT_LIPSWISH:
            return None
        if self._beta is None:
            self.refresh()
        return self._beta


# epilogue stub: the dmul operand already holds act'(pre) (see BranchProgram._deriv)
_MULT = _Act(ops.ACT_MULTIPLIER)


class _Weights(object):
    """Effective weights of one layer in the layouts the fused path needs (fp32 + optional planes)."""
    __slots__ = ('fwd', 'fwd_split', 'bwd', 'bwd_split', 'bias', 'kind', 'cin', 'cout', 'fwd_k', 'bwd_k', 'a_type',
                 'sigma', 'src', 'norms')     # sigma: induced-norm layers; src (raw W) and norms: Lop layers


class _T(object):
    """A rows-space activation: fp32 tensor and/or its tf32 hi/lo planes."""
    __slots__ = ('f', 's', 'colsum')

    def __init__(self, f=None, s=None):
        self.f, self.s, self.colsum = f, s, None

    def f32(self):
        if self.f is None:
            self.f = ops.lincomb3(self.s[0], 1.0, self.s[1], 1.0)
        return self.f

    def planes(self):
        """tf32 hi/lo planes, split at most once per tensor (they feed both the next GEMM as its K-major A
        operand and the weight-gradient contraction as an MN-major operand)."""
        if self.s is None:
            self.s = ops.split_tf32(self.f)
        return self.s


class _Saved(object):
    __slots__ = ('rows', 'meta', 'M', 'pres', 'ains', 'derivs')


def _act_of(m):
    if isinstance(m, Sin):
        return _Act(ops.ACT_SIN)
    if isinstance(m, Swish):
        return _Act(ops.ACT_LIPSWISH, m)
    if isinstance(m, (ReLU, nn.ReLU)):
        return _Act(ops.ACT_RELU)
    return None


def compile_branch(nnet):
    """BranchProgram for `nnet`, or None if it contains a module this path does not know."""
    flatten = False
    seq = nnet
    if hasattr(nnet, 'nnet') and isinstance(getattr(nnet, 'nnet'), nn.Sequential) and hasattr(nnet, 'input_shape'):
        seq, flatten = nnet.nnet, True            # FCNet wrapper (implicit_flow.py:437-474)
    if not isinstance(seq, nn.Sequential):
        return None
    stages, pending = [], None
    for m in seq:
        a = _act_of(m)
        if a is not None:
            if pending is not None:
                return None
            pending = a
        elif isinstance(m, (InducedNormLinear, InducedNormConv2d) + _LOP):
            stages.append((pending, m))
            pending = None
        else:
            return None
    if not stages:
        return None
    if any(isinstance(m, _LOP) for _, m in stages) and not _device_lop(stages[0][1].weight):
        return None
    kinds = {isinstance(m, _LINEAR) for _, m in stages}
    if len(kinds) != 1:
        return None
    return BranchProgram(stages, pending, flatten, list(nnet.parameters()))


class BranchProgram(object):

    def __init__(self, stages, post_act, flatten, params):
        self.stages = stages            # [(pre_act or None, layer module)]
        self.post_act = post_act
        self.flatten = flatten
        self.params = params            # nnet.parameters() order: the order gradients are returned in
        self.is_linear = isinstance(stages[0][1], _LINEAR)
        self._key = None
        self._weights = None
        self._saved = None
        self._D_static = None           # d sigma / d W twins while a sweep graph is captured (see _graphed)
        self._sweep_graphs = {}
        self._sweep_eager = {}      # MLP programs: eager calls per sweep kind before the first capture
        self._sweep_pool = None

    # ---------------------------------------------------------------- weights
    def _acts(self):
        return [a for a, _ in self.stages] + [self.post_act]

    def _version_key(self):
        key = []
        for act, m in self.stages:
            key += [m.weight._version, m.weight.data_ptr(), (m.bias._version if m.bias is not None else -1)]
            if not isinstance(m, _LOP):
                key += [m.u._version, m.v._version]
        for act in self._acts():
            if act is not None and act.module is not None:
                key += [act.module.beta._version, act.module.beta.data_ptr()]
        return tuple(key)

    def _use_tc(self, M, N, K):
        mode = ops.get_gemm_backend()
        if mode == 'simt':
            return False
        if mode == 'tc':
            return True
        # below ~0.25 GFLOP a tcgen05 launch is all fill / drain (21 us for the 33 MFLOP MLP layers of the tabular flows
        # against 6 us on the CUDA cores, which are exact fp32 as well)
        # (MLP programs only: a conv branch takes the native tile-kernel plan, which needs every layer on tensor-core planes)
        if self.is_linear and 2.0 * M * N * K < TC_MIN_FLOPS['program']:
            return False
        return M >= 64 and N >= 8 and K >= 32

    def _prep(self, M, meta=None):
        """(Re)build the cached effective weights; M = rows of the activation matrices."""
        key = (self._version_key(), M, ops.get_gemm_backend())
        if key == self._key:
            return self._weights
        ws = []
        with torch.no_grad():
            # softplus(beta) of every LipSwish of the branch in one launch (views of one small tensor)
            swish = [a for a in self._acts() if a is not None and a.kind == ops.ACT_LIPSWISH]
            if len(swish) > 1:
                sp = F.softplus(torch.cat([a.module.beta.detach().reshape(1) for a in swish]))
                for i, a in enumerate(swish):
                    a._beta = sp[i:i + 1]
            elif swish:
                swish[0].refresh()
            for act, m in self.stages:
                w = _Weights()
                if isinstance(m, InducedNormConv2d) and not m.is_initialized() and meta is not None:
                    # first use: record the spatial dims like InducedNormConv2d.forward does
                    m.spatial_dims.copy_(torch.tensor([float(meta[1][1]), float(meta[1][2])]).to(m.spatial_dims))
                    m._hw = None
                if isinstance(m, InducedNormConv2d) and not m.is_initialized():
                    m.compute_weight(update=False)                      # lazy u/v init (first use only)
                Wt = m.weight.detach()
                w.bias = m.bias.detach() if m.bias is not None else None
                w.sigma = w.src = w.norms = None
                if isinstance(m, _LOP):
                    # group norms (and the `scale` buffer, as compute_weight() writes it), then W / max(1, n_k/coeff)
                    w.src = Wt
                    w.norms = ops.lop_norms(Wt, m.max_across_dim, ops.lop_norm_type(m.norm_type), scale_out=m.scale)
                else:
                    w.sigma = sigma_of(m)
                cout, cin = Wt.shape[0], Wt.shape[1]
                if isinstance(m, _LINEAR) or m.kernel_size == (1, 1):
                    w.kind, w.cin, w.cout, w.a_type, kind = 'mm', cin, cout, True, 0
                    fshape, bshape = (cout, cin), (cin, cout)
                else:
                    w.kind, w.cin, w.cout = 'c3', cin, cout
                    w.a_type = cin <= cout
                    if w.a_type:     # forward: im2col + GEMM(K=9cin); transpose: GEMM(N=9cin) + col2im
                        kind, fshape, bshape = 1, (cout, 9 * cin), (9 * cin, cout)
                    else:            # forward: GEMM(N=9cout) + col2im; transpose: im2col + GEMM(K=9cout)
                        kind, fshape, bshape = 2, (9 * cout, cin), (cin, 9 * cout)
                tc_f = self._use_tc(M, fshape[0], _round_up(fshape[1], 32))
                tc_b = self._use_tc(M, bshape[0], _round_up(bshape[1], 32))
                fshape = (fshape[0], _round_up(fshape[1], 32) if tc_f else fshape[1])
                bshape = (bshape[0], _round_up(bshape[1], 32) if tc_b else bshape[1])
                # effective weight in every layout the kernels consume: one launch
                if w.norms is not None:
                    group = (ops.LOP_ROW if m.max_across_dim == 0 else ops.LOP_COL) if m.local_constraint \
                        else ops.LOP_ONE
                    w.fwd, w.fwd_split, w.bwd, w.bwd_split = ops.prep_weights_lop(
                        Wt, w.norms if m.local_constraint else w.norms[-1:], group, m.coeff, kind, fshape, tc_f,
                        bshape, tc_b)
                else:
                    w.fwd, w.fwd_split, w.bwd, w.bwd_split = ops.prep_weights(Wt, w.sigma, m.coeff, kind, fshape,
                                                                              tc_f, bshape, tc_b)
                w.fwd_k, w.bwd_k = fshape[1], bshape[1]
                ws.append(w)
        self._key, self._weights = key, ws
        return ws

    def _mlp_weights(self, M):
        """(effective weights, widths [d, h_1, ..., d]) of a branch the persistent small-d kernels (csrc/mlp_solver.cu)
        take at M rows: Linear act Linear ... act Linear with no leading or trailing activation, d <= 128, widths <=
        256, at most 8 layers.  None for any other branch."""
        if not self.is_linear or self.post_act is not None or self.stages[0][0] is not None \
                or any(a is None for a, _ in self.stages[1:]):
            return None
        ws = self._prep(M)
        dims = [ws[0].cin] + [w.cout for w in ws]
        if dims[0] != dims[-1] or dims[0] > 128 or max(dims) > 256 or len(ws) > 8:
            return None
        return ws, dims

    def _mlp_wt(self):
        """The effective weights transposed to (in, out), as the kernels' forward evaluation reads them; cached until
        the weights change."""
        cached = getattr(self, '_mlp_spec', None)
        if cached is None or cached[0] != self._key:
            cached = self._mlp_spec = (self._key, [w.fwd[:, :w.cin].t().contiguous() for w in self._weights])
        return cached[1]

    def mlp_solver_spec(self, x):
        """Arguments of the persistent solver's forward / inverse mode (impflow_mlp_broyden_solve) for inputs shaped
        like x, or None if the branch does not qualify (_mlp_weights, and one activation kind throughout)."""
        if not MLP_SOLVER['on'] or not self.is_linear or len({a.kind for a, _ in self.stages[1:] if a is not None}) > 1:
            return None
        fit = self._mlp_weights(self._to_rows(x)[0].shape[0])
        if fit is None:
            return None
        ws, dims = fit
        acts = [a for a, _ in self.stages[1:]]          # acts[l] sits behind layer l; each Swish owns its beta
        kind = acts[0].kind if acts else ops.ACT_NONE
        betas = [a.beta_sp() for a in acts] if kind == ops.ACT_LIPSWISH else None
        return (self._mlp_wt(), [w.bias for w in ws], dims, kind, betas)

    def _mlp_vjp_operands(self, saved):
        """(effective weights [out][ld], their row strides, act' multipliers (None for layer 0), dims) of the
        persistent kernels' vjp mode at the point of `saved`, or None if the branch does not qualify."""
        fit = self._mlp_weights(saved.M)
        if fit is None:
            return None
        ws, dims = fit
        if any(w.fwd is None or w.fwd.stride(1) != 1 for w in ws):
            return None
        dmul = [None] + [self._deriv(saved, i).contiguous() for i in range(1, len(ws))]
        if any(t.shape != (saved.M, dims[i]) for i, t in enumerate(dmul) if t is not None):
            return None
        return [w.fwd for w in ws], [w.fwd.stride(0) for w in ws], dmul, dims

    def mlp_vjp_spec(self, saved):
        """Arguments of the persistent solver's implicit-backward mode (impflow_mlp_broyden_solve_vjp) at the point
        of `saved`, or None if the branch does not qualify."""
        return self._mlp_vjp_operands(saved) if MLP_SOLVER['on'] else None

    def mlp_series_spec(self, saved):
        """Arguments of the one-launch MLP power series (impflow_mlp_series) at the point of `saved`, or None if the
        branch does not qualify: the kernel takes (samples, d) inputs.  Its 1..32 terms are the caller's to check."""
        if not MLP_SERIES['on'] or saved.meta[0] != 'lin' or len(saved.meta[1]) != 2:
            return None
        vs = self._mlp_vjp_operands(saved)
        if vs is None:
            return None
        W, ldw, dmul, dims = vs
        return W, ldw, self._mlp_wt(), dmul, dims

    # ---------------------------------------------------------------- plumbing
    def _to_rows(self, x):
        """Module-level tensor -> (rows matrix, meta)."""
        if self.is_linear:
            x2 = x.reshape(x.shape[0], -1) if self.flatten else x.reshape(-1, x.shape[-1])
            return x2.contiguous(), ('lin', tuple(x.shape))
        B, C, H, W = x.shape
        rows = x.permute(0, 2, 3, 1).contiguous().view(B * H * W, C)
        return rows, ('conv', (B, H, W))

    def _from_rows(self, y, meta):
        if meta[0] == 'lin':
            shape = meta[1]
            return y.view(*shape[:-1], y.shape[-1]) if not self.flatten else y.view(*shape)
        B, H, W = meta[1]
        return y.view(B, H, W, y.shape[-1]).permute(0, 3, 1, 2)

    def _gemm(self, A, A_split, Wm, Wk, W_split, bias, act, want_pre, want_act, dmul_pre, want_split):
        """One fused GEMM launch; A is (M, Wk) fp32 and/or its planes.  Epilogue as in the header:
        normal: pre = acc+bias, act = act(pre); dmul: pre = acc*act'(dmul_pre), act = acc (raw)."""
        lib = _cabi.load()
        M = (A if A is not None else A_split[0]).shape[0]
        N = Wm.shape[0]
        dev = Wm.device
        kind = act.kind if act is not None else ops.ACT_NONE
        beta = act.beta_sp() if act is not None else None
        if W_split is None:
            want_split = False
            if not want_act and not want_pre:
                want_pre = True
        pre = torch.empty(M, N, device=dev, dtype=torch.float32) if want_pre else None
        out_act = torch.empty(M, N, device=dev, dtype=torch.float32) if want_act else None
        if W_split is not None:
            if A_split is None:
                A_split = ops.split_tf32(A)
            sh = torch.empty(M, N, device=dev, dtype=torch.float32) if want_split else None
            sl = torch.empty(M, N, device=dev, dtype=torch.float32) if want_split else None
            _cabi.check(lib.impflow_gemm_nt_tc(
                _cabi.ptr(A_split[0]), _cabi.ptr(A_split[1]), Wk, _cabi.ptr(W_split[0]), _cabi.ptr(W_split[1]), Wk,
                _cabi.ptr(bias, 'bias', True), _cabi.ptr(pre, 'pre', True), _cabi.ptr(out_act, 'act', True),
                _cabi.ptr(dmul_pre, 'dmul', True), _cabi.ptr(sh, 'sh', True), _cabi.ptr(sl, 'sl', True), N, M, N, Wk,
                kind, _cabi.ptr(beta, 'beta', True), None, _cabi.stream()), 'gemm_nt_tc')
            if ops.GEMM_PROFILE['on']:
                ops.record_gemm(M, N, Wk, pre is not None, out_act is not None, dmul_pre is not None, want_split,
                                False)
            return pre, out_act, ((sh, sl) if want_split else None)
        if A is None:
            A = ops.lincomb3(A_split[0], 1.0, A_split[1], 1.0)
        _cabi.check(lib.impflow_gemm_nt(
            _cabi.ptr(A), Wk, _cabi.ptr(Wm), Wk, _cabi.ptr(bias, 'bias', True), _cabi.ptr(pre, 'pre', True),
            _cabi.ptr(out_act, 'act', True), _cabi.ptr(dmul_pre, 'dmul', True), N, M, N, Wk, kind,
            _cabi.ptr(beta, 'beta', True), _cabi.stream()), 'gemm_nt')
        return pre, out_act, None

    @staticmethod
    def _pad_cols(A, Kp):
        if A.shape[1] == Kp:
            return A
        out = A.new_zeros(A.shape[0], Kp)
        out[:, :A.shape[1]] = A
        return out

    @staticmethod
    def _im2col_first(w, transpose):
        """True when (this direction of) the layer is im2col + GEMM; False for GEMM (+ col2im)."""
        return w.kind == 'c3' and (w.a_type != transpose)

    def _wants_planes(self, w, transpose, channels):
        """Can the layer (in this direction) consume hi/lo planes of a `channels`-wide input directly?"""
        if w.kind == 'c3' and self._im2col_first(w, transpose):
            return False
        Wk, Wsp = (w.bwd_k, w.bwd_split) if transpose else (w.fwd_k, w.fwd_split)
        return Wsp is not None and Wk == channels

    def _apply(self, w, X, meta, transpose, bias=None, act=None, want_pre=True, want_act=False, dmul_pre=None,
               want_split=False):
        """Apply layer `w` (or its transpose) to the rows-space handle X with the fused epilogue.
        Returns (pre, act_out, split)."""
        Wm, Wk, Wsp = (w.bwd, w.bwd_k, w.bwd_split) if transpose else (w.fwd, w.fwd_k, w.fwd_split)
        cin = w.cout if transpose else w.cin
        cout = w.cin if transpose else w.cout
        M = (X.f if X.f is not None else X.s[0]).shape[0]
        next_is_pre = dmul_pre is not None or act is None      # which output feeds the next layer
        if w.kind == 'mm' or self._im2col_first(w, transpose):
            if w.kind == 'c3':
                B, H, Wd = meta[1]
                if Wsp is not None:      # patches written directly as the GEMM's tf32 planes
                    A, A_split = None, ops.im2col3x3_split(X.f32().view(B, H, Wd, cin), ld=Wk)
                else:
                    A, A_split = ops.im2col3x3(X.f32().view(B, H, Wd, cin), ld=Wk), None
            else:
                A_split = X.planes() if (Wsp is not None and cin == Wk) else None
                A = self._pad_cols(X.f32(), Wk) if A_split is None else None
            if want_split and Wsp is None:          # CUDA-core GEMM: planes come from the split kernel below
                want_pre, want_act = (True, want_act) if next_is_pre else (want_pre, True)
            pre, a_out, split = self._gemm(A, A_split, Wm, Wk, Wsp, bias, act, want_pre, want_act, dmul_pre,
                                           want_split)
        else:
            B, H, Wd = meta[1]
            A_split = X.planes() if (Wsp is not None and cin == Wk) else None
            A = self._pad_cols(X.f32(), Wk) if A_split is None else None
            Y, _, _ = self._gemm(A, A_split, Wm, Wk, Wsp, None, None, True, False, None, False)
            if want_split:
                want_pre, want_act = (True, want_act) if next_is_pre else (want_pre, True)
            pre, a_out = ops.col2im3x3(Y, B, H, Wd, cout, bias, act.kind if act is not None else ops.ACT_NONE,
                                       act.beta_sp() if act is not None else None, want_pre=want_pre,
                                       want_act=want_act,
                                       dmul_pre=dmul_pre.view(B, H, Wd, cout) if dmul_pre is not None else None)
            pre = pre.view(M, cout) if pre is not None else None
            a_out = a_out.view(M, cout) if a_out is not None else None
            split = None
        if want_split and split is None:
            split = ops.split_tf32(pre if next_is_pre else a_out)
        return pre, a_out, split


    # ---------------------------------------------------------------- native 3-layer conv runtime
    def _conv3(self, ws, meta):
        """impflow_conv3_plan (ctypes) for this branch, or None when it is not the
        [act] 3x3(c->C) act 1x1(C->C) act 3x3(C->c) stack of the image flows (implicit_flow.py:359-398)
        with every layer on the tcgen05 path."""
        if not CONV3_NATIVE['on'] or self.is_linear or len(ws) != 3 or self.post_act is not None or meta[0] != 'conv':
            return None
        w0, w1, w2 = ws
        a1, a2 = self.stages[1][0], self.stages[2][0]
        if a1 is None or a2 is None or a1.kind != a2.kind:
            return None
        C, c = w1.cout, w0.cin
        ok = (w0.kind == 'c3' and w0.a_type and w0.cout == C and w1.kind == 'mm' and w1.cin == C
              and w2.kind == 'c3' and not w2.a_type and w2.cin == C and w2.cout == c
              and w0.fwd_k == w2.bwd_k and w0.fwd_k % 32 == 0 and C % 32 == 0
              and w1.fwd_k == C and w1.bwd_k == C and w2.fwd_k == C and w0.bwd_k == C
              and all(w.fwd_split is not None and w.bwd_split is not None for w in ws))
        if not ok:
            return None
        B, H, Wd = meta[1]
        k0 = w0.fwd_k
        lib = _cabi.load()
        wsp = _conv3_workspace(lib.impflow_conv3_workspace_floats(B, H, Wd, c, C, k0), w0.fwd.device)
        key = (self._key, meta[1], FUSED3['on'], wsp.data_ptr())
        cache = getattr(self, '_conv3_cache', None)
        if cache is None or cache.get('weights') != self._key:
            cache = self._conv3_cache = {'weights': self._key}       # plans of older weights are dropped
        if key in cache:
            return cache[key][0]
        act0 = self.stages[0][0]
        P = _cabi.Conv3Plan()
        P.B, P.H, P.W, P.c, P.C, P.k0 = B, H, Wd, c, C, k0
        P.act_kind = a1.kind
        P.act0_kind = act0.kind if act0 is not None else ops.ACT_NONE
        P.allow_fused = 1 if FUSED3['on'] else 0
        dp = lambda t: (t.data_ptr() if t is not None else None)
        P.beta0 = dp(act0.beta_sp()) if act0 is not None else None
        P.beta1, P.beta2 = dp(a1.beta_sp()), dp(a2.beta_sp())
        P.W1f_hi, P.W1f_lo = dp(w0.fwd_split[0]), dp(w0.fwd_split[1])
        P.W2f_hi, P.W2f_lo = dp(w1.fwd_split[0]), dp(w1.fwd_split[1])
        P.W3f_hi, P.W3f_lo = dp(w2.fwd_split[0]), dp(w2.fwd_split[1])
        P.b1, P.b2, P.b3 = dp(w0.bias), dp(w1.bias), dp(w2.bias)
        P.W3b_hi, P.W3b_lo = dp(w2.bwd_split[0]), dp(w2.bwd_split[1])
        P.W2b_hi, P.W2b_lo = dp(w1.bwd_split[0]), dp(w1.bwd_split[1])
        P.W1b_hi, P.W1b_lo = dp(w0.bwd_split[0]), dp(w0.bwd_split[1])
        P.ws = wsp.data_ptr()
        # the weights / betas stay alive in self._weights and the _Act objects; the plan only borrows them
        cache[key] = (P, (ws, wsp, [a.beta_sp() for a in self._acts() if a is not None]))
        return P

    @staticmethod
    def _plan_ptr(P):
        return ctypes.c_void_p(ctypes.addressof(P))

    def _record_conv3(self, P, is_vjp, save, count=1):
        """bench.py roofline bookkeeping: which tensor-core launches one native evaluation makes."""
        M = P.B * P.H * P.W
        tile = P.allow_fused and P.k0 == 32 and P.C % 256 == 0 and 9 * P.c <= 32
        for _ in range(count):
            if tile:
                ops.record_branch3(M, P.C, 9 * P.c, is_vjp, save)
            elif P.allow_fused and P.C % 128 == 0 and ops.CHAIN23['on']:
                ops.record_gemm(M, P.C, P.k0, save, False, is_vjp, True, False)
                ops.record_chain23(M, P.C, 9 * P.c, is_vjp, save)
            else:
                ops.record_gemm(M, P.C, P.k0, save, False, is_vjp, True, False)
                ops.record_gemm(M, P.C, P.C, save, False, is_vjp, True, False)
                ops.record_gemm(M, 9 * P.c, P.C, True, False, False, False, False)

    def _native_forward(self, P, rows, meta, save):
        M = rows.shape[0]
        dev = rows.device
        y = torch.empty(M, P.c, device=dev, dtype=torch.float32)
        pre1 = torch.empty(M, P.C, device=dev, dtype=torch.float32) if save else None
        pre2 = torch.empty(M, P.C, device=dev, dtype=torch.float32) if save else None
        _cabi.check(_cabi.load().impflow_conv3_forward(self._plan_ptr(P), _cabi.ptr(rows), _cabi.ptr(y),
                                                       _cabi.ptr(pre1, 'pre1', True), _cabi.ptr(pre2, 'pre2', True),
                                                       _cabi.stream()), 'conv3_forward')
        if ops.GEMM_PROFILE['on']:
            self._record_conv3(P, False, save)
        saved = None
        if save:
            saved = _Saved()
            saved.rows, saved.meta, saved.M, saved.derivs = rows, meta, M, {}
            saved.pres = [rows if self.stages[0][0] is not None else None, pre1, pre2, None]
            saved.ains = None       # backward_full / neumann re-evaluate the layer inputs from the pre-activations
        return self._from_rows(y, meta), saved

    def _vjp_operands(self, saved, P=None):
        if P is not None and 1 not in saved.derivs and 2 not in saved.derivs:
            # both act' multipliers of this saved forward in one call of the native runtime
            d1, d2 = torch.empty_like(saved.pres[1]), torch.empty_like(saved.pres[2])
            _cabi.check(_cabi.load().impflow_conv3_prepare_vjp(self._plan_ptr(P), _cabi.ptr(saved.pres[1]),
                                                               _cabi.ptr(saved.pres[2]), _cabi.ptr(d1), _cabi.ptr(d2),
                                                               _cabi.stream()), 'conv3_prepare_vjp')
            saved.derivs[1], saved.derivs[2] = d1, d2
        return (_cabi.ptr(saved.pres[0], 'pre0', True), _cabi.ptr(self._deriv(saved, 1)),
                _cabi.ptr(self._deriv(saved, 2)))

    def prepare_vjp(self, saved):
        """Evaluate what vjp(., saved) needs beyond the vector (the act' multipliers of a native plan) now, so that a
        later vjp call is a single launch sequence with no set-up in front of it."""
        P = self._conv3(self._prep(saved.M), saved.meta)
        if P is not None:
            self._vjp_operands(saved, P)

    def _native_vjp(self, P, v, saved):
        t, _ = self._to_rows(v)
        out = torch.empty_like(t)
        pre0, d1, d2 = self._vjp_operands(saved, P)
        _cabi.check(_cabi.load().impflow_conv3_vjp(self._plan_ptr(P), pre0, d1, d2, _cabi.ptr(t), _cabi.ptr(out),
                                                   _cabi.stream()), 'conv3_vjp')
        if ops.GEMM_PROFILE['on']:
            self._record_conv3(P, True, False)
        return self._from_rows(out, saved.meta)

    def native_plan(self, x):
        """The native plan for inputs shaped like x (module layout), or None."""
        if self.is_linear or x.dim() != 4:
            return None
        meta = ('conv', (x.shape[0], x.shape[2], x.shape[3]))
        return self._conv3(self._prep(x.shape[0] * x.shape[2] * x.shape[3], meta), meta)

    def neumann_chain(self, saved, vareps, coeffs):
        """w = v + sum_k coeffs[k-1] v^T J^k (implicit_block.py:431-435): one C call with a native plan, else a chain
        of vjp evaluations."""
        P = self._conv3(self._prep(saved.M), saved.meta)
        if P is None:
            vjp = w = vareps
            for c in coeffs:
                vjp = self.vjp(vjp, saved)
                w = ops.lincomb3(w, 1.0, vjp, c)
            return w
        t, _ = self._to_rows(vareps)
        w_rows = torch.empty_like(t)
        n = len(coeffs)
        arr = (ctypes.c_double * max(n, 1))(*[float(c) for c in coeffs])
        pre0, d1, d2 = self._vjp_operands(saved, P)
        _cabi.check(_cabi.load().impflow_conv3_power_series(self._plan_ptr(P), pre0, d1, d2, _cabi.ptr(t), arr, n,
                                                            _cabi.ptr(w_rows), None, None, _cabi.stream()),
                    'conv3_power_series')
        if ops.GEMM_PROFILE['on']:
            self._record_conv3(P, True, False, n)
        return self._from_rows(w_rows, saved.meta)

    def hutchinson_series(self, saved, vareps, dot_coeffs):
        """sum_k dot_coeffs[k-1] <v^T J^k, v> per sample — the basic estimator's no-graph form (eval mode,
        implicit_block.py:418-426): one C call with a native plan, else a chain of vjp evaluations and row dots
        accumulated in place."""
        P = self._conv3(self._prep(saved.M), saved.meta)
        if P is None:
            out = torch.zeros(vareps.shape[0], device=vareps.device, dtype=torch.float32)
            vjp = vareps
            for c in dot_coeffs:
                vjp = self.vjp(vjp, saved)
                ops.rowdot(vjp, vareps, out=out, alpha=float(c), beta=1.0)
            return out
        t, _ = self._to_rows(vareps)
        n = len(dot_coeffs)
        out = torch.empty(vareps.shape[0], device=t.device, dtype=torch.float32)
        arr = (ctypes.c_double * max(n, 1))(*[float(c) for c in dot_coeffs])
        pre0, d1, d2 = self._vjp_operands(saved, P)
        _cabi.check(_cabi.load().impflow_conv3_power_series(self._plan_ptr(P), pre0, d1, d2, _cabi.ptr(t), None, n,
                                                            None, arr, _cabi.ptr(out), _cabi.stream()),
                    'conv3_power_series')
        if ops.GEMM_PROFILE['on']:
            self._record_conv3(P, True, False, n)
        return out

    def solve(self, mode, rhs, saved, threshold, eps):
        """Broyden solve of this branch's implicit equation, with rhs and result in module layout.
        Mode 0: rhs - nnet(z) - z = 0 from z = 0 (forward / inverse, implicit_block.py:68-80); mode 1: v^T J + v - rhs
        = 0 at the point of `saved` from v = 0 (implicit backward, :199-207).  Returns the reference's result dict
        (broyden.py:184-193).

        The whole solve is one call where the branch allows it: the persistent kernel of a small MLP branch
        (csrc/mlp_solver.cu), or the native runtime of a 3-layer conv branch (csrc/conv3_plan.cu).  Otherwise the
        generic kernel loop of layers/broyden.py iterates in rows layout, which for a conv branch saves the NCHW <->
        NHWC copies of every evaluation: a sample is a contiguous block either way, and the solver's per-sample dots
        and norms do not depend on the order inside it.  For an MLP branch rows layout is module layout."""
        if mode == 0:
            spec = self.mlp_solver_spec(rhs)
            if spec is not None:
                return _broyden.broyden_mlp(spec, rhs, torch.zeros_like(rhs), threshold, eps)
        else:
            spec = self.mlp_vjp_spec(saved)
            if spec is not None:
                return _broyden.broyden_mlp_vjp(spec, rhs, threshold, eps)
        P = self.native_plan(rhs)
        rows, meta = self._to_rows(rhs)
        B, M = rhs.shape[0], rows.shape[0]
        d = rows.numel() // B
        if P is not None:
            eps_scaled = _broyden.scaled_eps(eps, B, d)
            wk = _broyden._workspace(B, d, threshold, rows.device)
            wk.one_call_buffers()
            wk.xa.zero_()
            pre0, d1, d2 = self._vjp_operands(saved, P) if mode == 1 else (None, None, None)
            vp = lambda t: ctypes.c_void_p(t.data_ptr())
            _cabi.check(_cabi.load().impflow_conv3_broyden(
                self._plan_ptr(P), mode, _cabi.ptr(rows), pre0, d1, d2, vp(wk.xa), vp(wk.xb), vp(wk.ga), vp(wk.gb),
                vp(wk.low_x), vp(wk.low_g), vp(wk.Ut), vp(wk.Vt), vp(wk.sample_sq), vp(wk.low_sq), vp(wk.partial),
                vp(wk.state), vp(wk.state_host), threshold, float(eps_scaled), _cabi.stream()), 'conv3_broyden')
            best = wk.low_x.clone()     # first: the stream is empty after the solve, host work comes after the launch
            info = _broyden._result_dict(wk, wk.host_state(), (B, d), eps_scaled, threshold, result=best)
            if ops.GEMM_PROFILE['on']:
                self._record_conv3(P, mode == 1, False, info['nstep'] + 1)
        else:
            if mode == 0:
                def g(z2d):
                    zr = z2d.view(M, -1)
                    return ops.lincomb3(rows, 1.0, self.forward_rows(zr, meta), -1.0, zr, -1.0).view(B, -1)
            else:
                def g(v2d):
                    vr = v2d.view(M, -1)
                    return ops.lincomb3(self.vjp_rows(vr, saved), 1.0, vr, 1.0, rows, -1.0).view(B, -1)
            info = _broyden.broyden(g, torch.zeros(B, d, device=rows.device), threshold, eps)
        info['result'] = self._from_rows(info['result'].view(M, -1), meta)
        return info

    def fixed_point(self, rhs, start, atol, rtol, threshold):
        """Banach iteration x_k = rhs - nnet(x_{k-1}) from x_0 = start until every (x_k - x_{k-1})^2 /
        (atol + |start| rtol) < 1, at most threshold + 2 evaluations (iresblock.py:69-79, implicit_block.py:17-28).
        Returns (x, the reference's iteration count), x in module layout.

        The whole iteration is one call where the branch allows it: the persistent kernel of a small MLP branch
        (csrc/mlp_solver.cu), or the native runtime of a 3-layer conv branch (csrc/conv3_plan.cu), which computes what
        the host loop over forward() computes, bit for bit.  Otherwise (another branch, a CPU tensor, a threshold above
        the calls' limit of 1000) it is the host loop (find_fixed_point)."""
        if _device_solve(rhs) and 0 <= threshold <= _broyden.FIXED_POINT_MAX_THRESHOLD:
            spec = self.mlp_solver_spec(rhs)
            if spec is not None:
                return _broyden.fixed_point_mlp(spec, rhs, start, atol, rtol, threshold)
            P = self.native_plan(rhs)
            if P is not None:
                return self._native_fixed_point(P, rhs, start, atol, rtol, threshold)
        from .layers.implicit_block import find_fixed_point
        return find_fixed_point(lambda x: ops.lincomb3(rhs, 1.0, self.forward(x), -1.0), start, threshold, atol, rtol)

    def _native_fixed_point(self, P, rhs, start, atol, rtol, threshold):
        rows, meta = self._to_rows(rhs)
        srows = rows if start is rhs else self._to_rows(start)[0]
        ws = _broyden.fixed_point_workspace(rhs.shape[0], rows.numel() // rhs.shape[0], rows.device)
        out = torch.empty_like(rows)
        vp = lambda t: ctypes.c_void_p(t.data_ptr())
        _cabi.check(_cabi.load().impflow_conv3_fixed_point(
            self._plan_ptr(P), _cabi.ptr(rows), _cabi.ptr(srows), _cabi.ptr(out), _cabi.ptr(ws.xa), _cabi.ptr(ws.xb),
            vp(ws.state), vp(ws.state_host), float(atol), float(rtol), int(threshold), _cabi.stream()),
            'conv3_fixed_point')
        iterations = ws.iterations()
        if ops.GEMM_PROFILE['on']:
            self._record_conv3(P, False, False, iterations + 1)
        return self._from_rows(out, meta).contiguous(), iterations

    def _ains(self, saved):
        """Layer-input handles of a saved forward (the fused forward keeps only the pre-activations)."""
        if saved.ains is None:
            acts = self._acts()
            ws = self._weights
            ains = []
            for i in range(len(self.stages)):
                src = saved.rows if i == 0 else saved.pres[i]
                a = acts[i]
                w = ws[i] if ws is not None and i < len(ws) else None
                # a wide input that the weight gradient reads as planes is produced as planes straight away
                as_planes = (a is not None and w is not None and w.fwd_split is not None and ops.WGRAD_MN_MAJOR['on']
                             and w.cin == w.fwd_k and (w.kind == 'mm' or not w.a_type))
                if as_planes:
                    ains.append(_T(s=ops.act_split(src, a.kind, 0, a.beta_sp())))
                else:
                    ains.append(_T(f=src if a is None else ops.act_mul(src, None, a.kind, 0, a.beta_sp())))
            saved.ains = ains
        return saved.ains

    def _deriv(self, saved, i):
        """act'(pres[i]) of the activation in front of layer i, evaluated once per saved forward."""
        d = saved.derivs.get(i)
        if d is None:
            a = self._acts()[i]
            d = saved.derivs[i] = ops.act_mul(saved.pres[i], None, a.kind, 1, a.beta_sp())
        return d

    # ---------------------------------------------------------------- forward
    def forward_saved(self, x, save=True):
        """(nnet(x), saved) without a graph; saved feeds vjp / backward_full / neumann."""
        if not self.is_linear and x.dim() == 4:
            # shape bookkeeping first: a memo hit must not pay for the NCHW -> rows copy of _to_rows
            meta = ('conv', (x.shape[0], x.shape[2], x.shape[3]))
            M, rows = x.shape[0] * x.shape[2] * x.shape[3], None
        else:
            rows, meta = self._to_rows(x)
            M = rows.shape[0]
        ws = self._prep(M, meta)
        memo_key = None
        if save and MEMO['on']:
            # the memo keeps `x` alive, so an equal (data_ptr, shape, strides) can only be the same storage, and
            # an unchanged version counter means unchanged contents
            memo_key = (x.data_ptr(), tuple(x.shape), tuple(x.stride()), x._version, self._key)
            m = getattr(self, '_memo', None)
            if m is not None and m[0] == memo_key:
                return m[2], m[3]
        if rows is None:
            rows, meta = self._to_rows(x)
        out = self._forward_saved_impl(rows, meta, M, ws, save)
        if memo_key is not None:
            self._memo = (memo_key, x, out[0], out[1])
        return out

    def _forward_saved_impl(self, rows, meta, M, ws, save):
        P = self._conv3(ws, meta)
        if P is not None:
            return self._native_forward(P, rows, meta, save)
        n = len(self.stages)
        pres = [None] * (n + 1)       # pres[i] = input of the activation in front of layer i (pres[n]: post act)
        ains = [None] * n             # ains[i] = input handle of layer i (after its activation)
        X = _T(f=rows)
        act0 = self.stages[0][0]
        if act0 is not None:
            pres[0] = rows
            X = _T(f=ops.act_mul(rows, None, act0.kind, 0, act0.beta_sp()))
        for i in range(n):
            w = ws[i]
            last = i == n - 1
            nxt = self.post_act if last else self.stages[i + 1][0]
            ains[i] = X
            want_split = (not last) and self._wants_planes(ws[i + 1], False, w.cout)
            need_pre = (nxt is None) or save
            want_act = nxt is not None and (last or not want_split)
            pre, a_out, split = self._apply(w, X, meta, False, bias=w.bias, act=nxt, want_pre=need_pre,
                                            want_act=want_act, want_split=want_split)
            if nxt is not None:
                pres[i + 1] = pre
            X = _T(f=(a_out if nxt is not None else pre), s=split)
        out = X.f32()
        saved = None
        if save:
            saved = _Saved()
            saved.rows, saved.meta, saved.M, saved.pres, saved.ains, saved.derivs = rows, meta, M, pres, ains, {}
        return self._from_rows(out, meta), saved

    def forward_rows(self, rows, meta):
        """nnet applied to activations already in rows (NHWC) layout, result in rows layout: no layout copies.  The
        generic Broyden loop of a conv branch without a native plan iterates in this layout (a sample is a contiguous
        block either way; the solver algebra does not care about the order inside it)."""
        M = rows.shape[0]
        y, _ = self._forward_saved_impl(rows, meta, M, self._prep(M, meta), False)
        return y.permute(0, 2, 3, 1).reshape(M, -1) if meta[0] == 'conv' else y.reshape(M, -1)

    def forward(self, x, save=False):
        y, saved = self.forward_saved(x, save)
        if save:
            self._saved = saved
        return y

    # ---------------------------------------------------------------- vjp
    def vjp(self, v, saved=None):
        """v^T J at the point of `saved` (default: the last forward(save=True))."""
        saved = saved if saved is not None else self._saved
        if saved is None:
            raise RuntimeError('BranchProgram.vjp: call forward(save=True) first')
        meta, M, pres = saved.meta, saved.M, saved.pres
        ws = self._prep(M)
        P = self._conv3(ws, meta)
        if P is not None:
            return self._native_vjp(P, v, saved)
        t, _ = self._to_rows(v)
        return self._from_rows(self.vjp_rows(t, saved), meta)

    def vjp_rows(self, t, saved):
        """v^T J with v and the result in rows (NHWC) layout (generic launch sequence; see forward_rows)."""
        meta, M, pres = saved.meta, saved.M, saved.pres
        ws = self._prep(M)
        n = len(self.stages)
        T = _T(f=t)
        if self.post_act is not None:
            T = _T(f=ops.act_mul(pres[n], t, self.post_act.kind, 1, self.post_act.beta_sp()))
        for i in range(n - 1, -1, -1):
            w = ws[i]
            act = self.stages[i][0]            # activation in front of layer i: multiply by act'(pres[i])
            dm = self._deriv(saved, i) if act is not None else None      # evaluated once per saved forward
            want_split = i > 0 and self._wants_planes(ws[i - 1], True, w.cin)
            pre, _, split = self._apply(w, T, meta, True, act=(_MULT if act is not None else None),
                                        want_pre=not want_split, dmul_pre=dm, want_split=want_split)
            T = _T(f=pre, s=split)
        return T.f32()

    # ---------------------------------------------------------------- parameter gradients
    def _wgrad_gemm_layout(self, w, meta, G, Xin):
        """dL/d(w.fwd) (N, Kpad) from the output adjoint G (M, cout) (tensor or handle) and the layer input
        handle.  Wide operands go in as their cached hi/lo planes."""
        Gh = G if isinstance(G, _T) else _T(f=G)
        tc = w.fwd_split is not None and ops.WGRAD_MN_MAJOR['on']
        if w.kind == 'c3':
            B, H, Wd = meta[1]
            if w.a_type:
                Am = ops.im2col3x3(Xin.f32().view(B, H, Wd, w.cin), ld=w.fwd_k)
                if tc and w.cout % 4 == 0:
                    return ops.wgrad_gemm(None, Am, G_split=Gh.planes())
                Gm = Gh.f32()
            else:
                # patch rows padded to a multiple of 4 floats (16-byte rows for TMA); the extra output rows are cut
                Gm = ops.im2col3x3(Gh.f32().view(B, H, Wd, w.cout), ld=_round_up(9 * w.cout, 4))
                if tc and w.cin == w.fwd_k:
                    return ops.wgrad_gemm(Gm, None, A_split=Xin.planes())[:9 * w.cout]
                Am = self._pad_cols(Xin.f32(), w.fwd_k)
                return ops.wgrad_gemm(Gm, Am)[:9 * w.cout]
        else:
            if tc and w.cin == w.fwd_k and w.cout % 4 == 0:
                return ops.wgrad_gemm(None, None, G_split=Gh.planes(), A_split=Xin.planes())
            Gm, Am = Gh.f32(), self._pad_cols(Xin.f32(), w.fwd_k)
        return ops.wgrad_gemm(Gm, Am)

    @staticmethod
    def _to_weight_layout(w, Wbar):
        """GEMM-layout gradient -> gradient of the effective weight in the module's weight layout."""
        if w.kind == 'mm':
            return Wbar[:, :w.cin]
        if w.a_type:
            return Wbar[:, :9 * w.cin].reshape(w.cout, 3, 3, w.cin).permute(0, 3, 1, 2)
        return Wbar[:, :w.cin].reshape(3, 3, w.cout, w.cin).flip(0, 1).permute(2, 3, 0, 1)

    def _finish_param_grads(self, ws, wbars, bbars, betabars):
        """Chain the effective-weight gradients through the spectral rescale W / max(1, sigma/coeff)
        (mixed_lipschitz.py:125-131: differentiable through sigma with u, v constant) or a Lop layer's rescale by its
        group norms (lipschitz.py:72-79), and order everything like nnet.parameters()."""
        by_id = {}
        for i, (act, m) in enumerate(self.stages):
            if wbars[i] is not None and ws[i].norms is not None:
                w, Wbar = ws[i], wbars[i]
                Wbar = Wbar if Wbar.stride(-1) == 1 else Wbar.contiguous()
                kind = 0 if w.kind == 'mm' else (1 if w.a_type else 2)
                by_id[id(m.weight)] = ops.lop_scale_grad_layout(
                    Wbar, kind, w.cout, w.cin, w.src, w.norms, m.coeff, m.max_across_dim,
                    ops.lop_norm_type(m.norm_type), m.local_constraint).view(m.weight.shape)
            elif wbars[i] is not None:
                w, Wbar = ws[i], wbars[i]
                W = m.weight.detach()
                D = self._D_static[id(m)] if self._D_static is not None else m.sigma_gradient()
                if FUSED_SN_GRAD['on'] and Wbar.dim() == 2 and Wbar.stride(1) == 1 and W.is_contiguous() \
                        and D.is_contiguous() and D.shape == W.shape:
                    kind = 0 if w.kind == 'mm' else (1 if w.a_type else 2)
                    by_id[id(m.weight)] = ops.sn_scale_grad_layout(Wbar, kind, w.cout, w.cin, W, D, w.sigma, m.coeff)
                else:
                    g_eff = self._to_weight_layout(w, Wbar).reshape(m.weight.shape).contiguous()
                    by_id[id(m.weight)] = ops.sn_scale_grad(g_eff, W, D, w.sigma, m.coeff)
            if m.bias is not None and bbars[i] is not None:
                by_id[id(m.bias)] = bbars[i]
        # d/d(raw beta) = d/d softplus(beta) * sigmoid(beta): two multi-tensor launches for all activations
        live = [(act.module.beta, gb) for act, gb in zip(self._acts(), betabars)
                if act is not None and act.module is not None and gb is not None]
        if live:
            sig = torch._foreach_sigmoid([b.detach() for b, _ in live])
            for (b, _), g in zip(live, torch._foreach_mul([gb for _, gb in live], sig)):
                by_id[id(b)] = g
        return [by_id.get(id(p)) for p in self.params]

    @staticmethod
    def _add(a, b):
        if a is None:
            return b
        if b is None:
            return a
        return ops.lincomb3(a, 1.0, b, 1.0)

    def backward_full(self, saved, gout, need_input_grad=True):
        """First-order backward of y = nnet(x): returns (g^T J or None, [dL/dp for p in parameters()])."""
        if self._graphable(saved, gout):
            out = self._graphed('backward_full', saved, (gout,), (bool(need_input_grad),))
            return out[0], list(out[1:])
        return self._backward_full_eager(saved, gout, need_input_grad)

    def _backward_full_eager(self, saved, gout, need_input_grad=True):
        meta, M, pres, ains = saved.meta, saved.M, saved.pres, self._ains(saved)
        ws = self._prep(M)
        n = len(self.stages)
        acts = self._acts()
        wbars, bbars, betabars = [None] * n, [None] * n, [None] * (n + 1)
        g, _ = self._to_rows(gout)
        if self.post_act is not None:
            pa = self.post_act
            if pa.module is not None:
                betabars[n] = ops.act_beta_grad(pres[n], g, 0, pa.beta_sp())
            g = ops.act_mul(pres[n], g, pa.kind, 1, pa.beta_sp())
        G = _T(f=g)
        for i in range(n - 1, -1, -1):
            w = ws[i]
            act = acts[i]
            Gf = G.f32()
            wbars[i] = self._wgrad_gemm_layout(w, meta, G, ains[i])
            if w.bias is not None:
                bbars[i] = ops.colsum(Gf)
            if i == 0 and not need_input_grad and (act is None or act.module is None):
                break
            # the adjoint handed to layer i-1 also leaves the GEMM as hi/lo planes when that layer consumes planes
            # (its transposed GEMM and its weight gradient): no separate split pass
            planes = i > 0 and self._wants_planes(ws[i - 1], True, w.cin)
            if act is not None:
                want_raw = act.module is not None
                pbar, abar, split = self._apply(w, G, meta, True, act=_MULT, want_pre=True, want_act=want_raw,
                                                dmul_pre=self._deriv(saved, i), want_split=planes)
                if want_raw:
                    betabars[i] = ops.act_beta_grad(pres[i], abar, 0, act.beta_sp())
            else:
                pbar, _, split = self._apply(w, G, meta, True, want_pre=True, want_split=planes)
            G = _T(f=pbar, s=split)
        gx = self._from_rows(G.f32(), meta) if need_input_grad else None
        return gx, self._finish_param_grads(ws, wbars, bbars, betabars)

    # ---------------------------------------------------------------- CUDA graphs of the gradient sweeps
    # backward_full() and neumann() are fixed sequences of 35 / 50 launches with no data-dependent control flow.  At
    # the deeper scales (and for the MLP flows) the GPU finishes them faster than Python can issue them, so after
    # SWEEP_GRAPHS['warmup'] eager calls a sweep is captured once into a CUDA graph over STATIC copies of everything
    # it reads that changes between steps (saved pre-activations, the incoming vectors, the prepared weight planes,
    # softplus(beta), sigma and d sigma / d W, a Lop layer's raw weight and group norms), and every later call is: one
    # multi-tensor copy into the static inputs, one graph launch, one multi-tensor copy of the results out of the
    # graph's private pool.
    def _graphable(self, saved, like):
        # MLP flows: the row count of the batched sweep follows the roulette draw of every step (n-fold batch), so a
        # program collects one graph per distinct n (a handful: n = exact terms + a geometric draw); they share one
        # private memory pool per program (never replayed concurrently) and are captured at their first occurrence
        # once the program has run eagerly SWEEP_GRAPHS['warmup'] times
        if self.is_linear and not SWEEP_GRAPHS['mlp']:
            return False
        return (SWEEP_GRAPHS['on'] and like.is_cuda and saved.M <= SWEEP_GRAPHS['max_rows']
                and not torch.cuda.is_current_stream_capturing())

    def sweep_graphable(self, saved, like):
        """Would neumann() / backward_full() at this saved forward replay a CUDA graph?"""
        return self._graphable(saved, like)

    def _dynamic_inputs(self, saved, vecs):
        ws = self._prep(saved.M)
        dyn = [saved.rows] + [p for p in saved.pres if p is not None and p is not saved.rows]
        dyn += [v for v in vecs if v is not None]
        for w in ws:
            # what the gradient chain reads: sigma (and d sigma / d W below), or the raw weight and its group norms
            dyn += [w.fwd, w.bwd] + ([w.sigma] if w.norms is None else [w.src, w.norms])
            dyn += list(w.fwd_split) if w.fwd_split is not None else []
            dyn += list(w.bwd_split) if w.bwd_split is not None else []
        dyn += [a._beta for a in self._acts() if a is not None and a.beta_sp() is not None]
        dyn += [m.sigma_gradient() for _, m in self.stages if not isinstance(m, _LOP)]
        return dyn, ws

    def _graphed(self, kind, saved, vecs, flags):
        dyn, ws = self._dynamic_inputs(saved, vecs)
        key = (kind, flags, saved.M, saved.meta, tuple(v is None for v in vecs),
               tuple((tuple(t.shape), t.dtype) for t in dyn), tuple(p.data_ptr() for p in self.params),
               ops.get_gemm_backend(), dyn[0].device.index)
        G = self._sweep_graphs.get(key)
        if G is None:
            if len(self._sweep_graphs) > (32 if self.is_linear else 8):
                self._sweep_graphs.clear()
                self._sweep_pool = None
            G = self._sweep_graphs[key] = {'calls': 0, 'graph': None}
        eager = self._backward_full_eager if kind == 'backward_full' else self._neumann_eager
        if G['graph'] is None:
            G['calls'] += 1
            # conv programs: warm-up per key; MLP programs: per program and kind (every n-fold batch size is a new
            # key, but the lazy set-up the warm-up calls are there for does not depend on the row count)
            warm = self._sweep_eager.get(kind, 0) if self.is_linear else G['calls'] - 1
            if warm < SWEEP_GRAPHS['warmup']:
                self._sweep_eager[kind] = self._sweep_eager.get(kind, 0) + 1
                out = eager(saved, *vecs, *flags)
                return self._flatten_sweep(kind, out, flags)
            self._capture_sweep(G, kind, eager, saved, vecs, flags, dyn, ws)
        else:
            torch._foreach_copy_(G['static_in'], dyn)
        G['graph'].replay()
        if ops.GEMM_PROFILE['on']:
            for k, c in G['gemm_profile'].items():
                ops.GEMM_PROFILE['shapes'][k] = ops.GEMM_PROFILE['shapes'].get(k, 0) + c
        _cabi.load().impflow_add_launch_count(G['launches'])
        live = [o for o in G['outputs'] if o is not None]
        fresh = [torch.empty_like(o) for o in live]
        torch._foreach_copy_(fresh, live)
        it = iter(fresh)
        return [None if o is None else next(it) for o in G['outputs']]

    @staticmethod
    def _flatten_sweep(kind, out, flags):
        if kind == 'backward_full':
            return [out[0]] + list(out[1])
        if flags[0]:
            return [out[0], out[1]] + list(out[2]) + [out[3]]
        return [out[0], out[1]] + list(out[2])

    def _capture_sweep(self, G, kind, eager, saved, vecs, flags, dyn, ws):
        if os.environ.get('IMPFLOW_TRACE_CAPTURE', '') == '1':       # diagnostic: when do captures happen
            import sys
            import time
            sys.stderr.write('[capture] t=%.3f %s rows=%d flags=%s\n' % (time.perf_counter(), kind, saved.M, flags))
        static_in = [t.clone() for t in dyn]
        twin = {id(t): s_ for t, s_ in zip(dyn, static_in)}
        T = lambda t: None if t is None else twin[id(t)]
        saved_s = _Saved()
        saved_s.rows, saved_s.meta, saved_s.M = T(saved.rows), saved.meta, saved.M
        saved_s.pres = [T(p) for p in saved.pres]
        saved_s.ains, saved_s.derivs = None, {}
        ws_s = []
        for w in ws:
            w2 = _Weights()
            for name in _Weights.__slots__:
                setattr(w2, name, getattr(w, name, None))
            w2.fwd, w2.bwd, w2.sigma, w2.src, w2.norms = T(w.fwd), T(w.bwd), T(w.sigma), T(w.src), T(w.norms)
            w2.fwd_split = tuple(T(t) for t in w.fwd_split) if w.fwd_split is not None else None
            w2.bwd_split = tuple(T(t) for t in w.bwd_split) if w.bwd_split is not None else None
            ws_s.append(w2)
        acts = [a for a in self._acts() if a is not None and a._beta is not None]
        old_betas = [a._beta for a in acts]
        old_weights = self._weights
        launches0 = _cabi.launch_count()
        prof_on, prof_old = ops.GEMM_PROFILE['on'], ops.GEMM_PROFILE['shapes']
        graph = torch.cuda.CUDAGraph()
        try:
            for a in acts:
                a._beta = T(a._beta)
            self._weights = ws_s
            self._D_static = {id(m): T(m.sigma_gradient()) for _, m in self.stages if not isinstance(m, _LOP)}
            ops.GEMM_PROFILE['on'], ops.GEMM_PROFILE['shapes'] = True, {}
            # capture_begin / capture_end directly: the torch.cuda.graph context manager also synchronises the device
            # and EMPTIES the caching allocator, after which the following steps re-allocate everything
            cur = torch.cuda.current_stream()
            side = SWEEP_GRAPHS.get('stream')
            if side is None or side.device != cur.device:
                side = SWEEP_GRAPHS['stream'] = torch.cuda.Stream(device=cur.device)
            side.wait_stream(cur)
            pool = None
            if self.is_linear:        # one pool for all graphs of this program (sequential replays only)
                if getattr(self, '_sweep_pool', None) is None:
                    self._sweep_pool = torch.cuda.graph_pool_handle()
                pool = self._sweep_pool
            with torch.cuda.stream(side):
                if pool is not None:
                    graph.capture_begin(pool=pool)
                else:
                    graph.capture_begin()
                try:
                    out = eager(saved_s, *[T(v) for v in vecs], *flags)
                finally:
                    graph.capture_end()
            cur.wait_stream(side)
            G['gemm_profile'] = dict(ops.GEMM_PROFILE['shapes'])
        finally:
            ops.GEMM_PROFILE['on'], ops.GEMM_PROFILE['shapes'] = prof_on, prof_old
            self._weights = old_weights
            self._D_static = None
            for a, b in zip(acts, old_betas):
                a._beta = b
        G['launches'] = _cabi.launch_count() - launches0
        G['static_in'], G['outputs'], G['graph'] = static_in, self._flatten_sweep(kind, out, flags), graph

    # ---------------------------------------------------------------- tangent sweep / batched bilinear gradients
    def tangent(self, saved, v_vec):
        """J v at the point of `saved` (forward-mode sweep t_l = W phi'(p) t_{l-1}), module layout."""
        meta, M, pres = saved.meta, saved.M, saved.pres
        ws = self._prep(M)
        n = len(self.stages)
        acts = self._acts()
        tp0, _ = self._to_rows(v_vec)
        TA = _T(f=tp0)
        if acts[0] is not None:
            TA = _T(f=ops.act_mul(pres[0], tp0, acts[0].kind, 1, acts[0].beta_sp()))
        for i in range(n):
            w = ws[i]
            last = i == n - 1
            nxt = acts[i + 1]
            want_split = (not last) and self._wants_planes(ws[i + 1], False, w.cout)
            if nxt is not None:
                prod, _, split = self._apply(w, TA, meta, False, act=_MULT, want_pre=(last or not want_split),
                                             dmul_pre=self._deriv(saved, i + 1), want_split=want_split)
                TA = _T(f=prod, s=split)
            else:
                pre, _, split = self._apply(w, TA, meta, False, want_pre=True, want_split=want_split)
                TA = _T(f=pre, s=split)
        return self._from_rows(TA.f32(), meta)

    def tile_saved(self, saved, n):
        """The saved forward of the batch repeated n times along the batch dimension: lets n bilinear-form gradients
        d(w_m^T J r_m), m = 1..n, at the SAME point run as one sweep over an n-fold batch (rows are sample-major)."""
        t = _Saved()
        rep = lambda a: a.repeat(n, 1) if a is not None else None
        t.rows, t.M = rep(saved.rows), saved.M * n
        t.pres = [rep(p) for p in saved.pres]
        t.ains = None
        t.derivs = {k: rep(v) for k, v in saved.derivs.items()}
        if saved.meta[0] == 'lin':
            shape = tuple(saved.meta[1])
            t.meta = ('lin', (shape[0] * n,) + shape[1:])
        else:
            B, H, W = saved.meta[1]
            t.meta = ('conv', (B * n, H, W))
        return t

    # ---------------------------------------------------------------- Neumann estimator gradient
    def neumann(self, saved, w_vec, v_vec, seed_scale=None, want_tangent=False):
        """S_b = <w_b^T J_b, v_b> together with dS/dx and dS/dtheta of S = sum_b c_b S_b
        (c = seed_scale or 1), by one tangent sweep and one two-adjoint reverse sweep.
        want_tangent: also return J v (module layout), the by-product of the tangent sweep."""
        if self._graphable(saved, w_vec):
            out = self._graphed('neumann', saved, (w_vec, v_vec, seed_scale), (bool(want_tangent),))
            if want_tangent:
                return out[0], out[1], list(out[2:-1]), out[-1]
            return out[0], out[1], list(out[2:])
        return self._neumann_eager(saved, w_vec, v_vec, seed_scale, want_tangent)

    def _neumann_eager(self, saved, w_vec, v_vec, seed_scale=None, want_tangent=False):
        meta, M, pres, ains = saved.meta, saved.M, saved.pres, self._ains(saved)
        ws = self._prep(M)
        n = len(self.stages)
        acts = self._acts()
        Bsz = v_vec.shape[0]
        # ---- tangent sweep: t_p (tangent of every activation input), t_a (tangent of every layer input)
        tps = [None] * (n + 1)
        tas = [None] * n
        tp0, _ = self._to_rows(v_vec)
        TA = _T(f=tp0)
        if acts[0] is not None:
            tps[0] = tp0
            TA = _T(f=ops.act_mul(pres[0], tp0, acts[0].kind, 1, acts[0].beta_sp()))
        for i in range(n):
            w = ws[i]
            last = i == n - 1
            nxt = acts[i + 1]
            tas[i] = TA
            want_split = (not last) and self._wants_planes(ws[i + 1], False, w.cout)
            if nxt is not None:
                prod, raw, split = self._apply(w, TA, meta, False, act=_MULT, want_pre=(last or not want_split),
                                               want_act=True, dmul_pre=self._deriv(saved, i + 1),
                                               want_split=want_split)
                tps[i + 1] = raw
                TA = _T(f=prod, s=split)
            else:
                pre, _, split = self._apply(w, TA, meta, False, want_pre=True, want_split=want_split)
                TA = _T(f=pre, s=split)
        tout = TA.f32()
        wrows, _ = self._to_rows(w_vec)
        S = ops.rowdot(tout.view(Bsz, -1), wrows.view(Bsz, -1))
        if seed_scale is not None:
            wrows = (wrows.view(Bsz, -1) * seed_scale.view(Bsz, 1)).view_as(wrows)
        # ---- reverse sweep with two adjoints: Tbar (of the tangent) and Ybar (of the primal)
        wbars, bbars, betabars = [None] * n, [None] * n, [None] * (n + 1)
        Tbar, Ybar = _T(f=wrows), None
        if self.post_act is not None:
            pa = self.post_act
            if pa.module is not None:
                betabars[n] = ops.act_beta_grad(pres[n], wrows, 1, pa.beta_sp(), g2=tps[n])
            Ybar = _T(f=ops.act_second(pres[n], tps[n], wrows, None, pa.kind, pa.beta_sp()))
            Tbar = _T(f=ops.act_mul(pres[n], wrows, pa.kind, 1, pa.beta_sp()))
        for i in range(n - 1, -1, -1):
            w = ws[i]
            act = acts[i]
            wb = self._wgrad_gemm_layout(w, meta, Tbar, tas[i])
            if Ybar is not None:
                wb = self._add(wb, self._wgrad_gemm_layout(w, meta, Ybar, ains[i]))
                if w.bias is not None:
                    bbars[i] = Ybar.colsum if Ybar.colsum is not None else ops.colsum(Ybar.f32())
            wbars[i] = wb
            abar = None
            if Ybar is not None:
                abar, _, _ = self._apply(w, Ybar, meta, True, want_pre=True)
            if act is not None:
                # one launch: tbar_p = phi'(p) * (W^T Tbar) in `prod`, the raw W^T Tbar in `raw`
                planes = i > 0 and self._wants_planes(ws[i - 1], True, w.cin)
                prod, tabar, tsplit = self._apply(w, Tbar, meta, True, act=_MULT, want_pre=(i > 0 and not planes),
                                                  want_act=True, dmul_pre=self._deriv(saved, i), want_split=planes)
                fuse = (NEUMANN_FUSED['on'] and act.module is not None and act.kind == ops.ACT_LIPSWISH and i > 0
                        and tabar.dim() == 2 and tabar.shape[1] >= 64 and ws[i - 1].fwd_split is not None)
                if fuse:
                    # one pass: ybar planes, their column sums (bias gradient of layer i-1) and d/dbeta
                    planes, ybar_colsum, betabars[i] = ops.neumann_act_bwd(pres[i], tps[i], tabar, abar,
                                                                          act.beta_sp())
                    Ybar = _T(s=planes)
                    Ybar.colsum = ybar_colsum
                else:
                    if act.module is not None:
                        gb = ops.act_beta_grad(pres[i], tabar, 1, act.beta_sp(), g2=tps[i])
                        if abar is not None:
                            gb = gb + ops.act_beta_grad(pres[i], abar, 0, act.beta_sp())
                        betabars[i] = gb
                    Ybar = _T(f=ops.act_second(pres[i], tps[i], tabar, abar, act.kind, act.beta_sp()))
                Tbar = _T(f=prod, s=tsplit)
            else:
                if i > 0:
                    tabar, _, _ = self._apply(w, Tbar, meta, True, want_pre=True)
                    Tbar = _T(f=tabar)
                Ybar = _T(f=abar) if abar is not None else None
        if Ybar is not None:
            gx = self._from_rows(Ybar.f32(), meta)
        else:
            gx = torch.zeros_like(v_vec)
        if want_tangent:
            return S, gx, self._finish_param_grads(ws, wbars, bbars, betabars), self._from_rows(tout, meta)
        return S, gx, self._finish_param_grads(ws, wbars, bbars, betabars)
