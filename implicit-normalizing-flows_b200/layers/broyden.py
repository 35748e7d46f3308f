"""Batched limited-memory Broyden root solver — API mirror of lib/layers/broyden.py:123-193.

`g_` is any callable on CUDA tensors (one branch evaluation / one vjp per call); all of the
solver algebra (rank-1 updates, low-rank mat-vecs, norms, best-iterate tracking, break rules)
runs in the impflow CUDA kernels with the bookkeeping kept on the device.  The host reads a
600-byte state record per iteration to learn whether the loop continues."""
import ctypes
import math

import numpy as np
import torch

from .. import _cabi

__all__ = ['broyden_mlp_vjp', 'broyden', 'broyden_mlp', 'fixed_point_mlp']

_STATE_DTYPE = np.dtype([('nstep', '<i4'), ('lowest_step', '<i4'), ('active', '<i4'), ('prot_break', '<i4'),
                         ('converged', '<i4'), ('stagnated', '<i4'), ('do_update', '<i4'), ('new_lowest', '<i4'),
                         ('threshold', '<i4'), ('counter', '<i4'), ('eps', '<f8'), ('init_objective', '<f8'),
                         ('lowest', '<f8'), ('objective', '<f8'), ('trace', '<f8', (64,))])

_workspaces = {}


class _Workspace(object):
    """Device buffers of one (B, d, T) problem size, reused across solves."""

    def __init__(self, B, d, T, device):
        lib = _cabi.load()
        f32 = dict(device=device, dtype=torch.float32)
        self.xa = torch.empty(B, d, **f32)
        self.xb = torch.empty(B, d, **f32)
        self.low_x = torch.empty(B, d, **f32)
        self.low_g = torch.empty(B, d, **f32)
        self.Ut = torch.empty(B, T, d, **f32)
        self.Vt = torch.empty(B, T, d, **f32)
        self.sample_sq = torch.empty(B, **f32)
        self.low_sq = torch.empty(B, **f32)
        self.partial = torch.empty(max(int(lib.impflow_broyden_workspace_floats(B, d, T)), 1), **f32)
        nbytes = int(lib.impflow_broyden_state_bytes())
        assert nbytes == _STATE_DTYPE.itemsize, 'state layout mismatch between header and host'
        self.state = torch.zeros(nbytes, device=device, dtype=torch.uint8)
        # pinned (and therefore device-mapped) host memory: the final state record, followed by the per-iteration
        # progress records the sync-free conv solver polls (impflow_conv3_broyden_host_bytes)
        self.state_nbytes = nbytes
        self.state_host = _cabi.pinned_bytes(max(nbytes, int(lib.impflow_conv3_broyden_host_bytes(T))))
        self.ga = self.gb = self.partial_d = None

    def one_call_buffers(self, mlp=False):
        """Allocate on first use what the one-call solvers need beyond the generic loop's buffers: the residual pair
        ga / gb and, for the persistent MLP kernel (mlp=True), its fp64 partial sums."""
        if self.ga is None:
            self.ga, self.gb = torch.empty_like(self.xa), torch.empty_like(self.xa)
        if mlp and self.partial_d is None:
            self.partial_d = torch.empty(int(_cabi.load().impflow_mlp_solver_partial_doubles()), device=self.xa.device,
                                         dtype=torch.float64)

    def read_state(self):
        self.state_host[:self.state_nbytes].copy_(self.state, non_blocking=True)
        _cabi.sync_stream()
        return self.host_state()

    def host_state(self):
        return self.state_host[:self.state_nbytes].numpy().view(_STATE_DTYPE)[0]


def _workspace(B, d, T, device):
    key = (B, d, T, device.index)
    ws = _workspaces.get(key)
    if ws is None:
        if len(_workspaces) > 16:
            _workspaces.clear()
        ws = _workspaces[key] = _Workspace(B, d, T, device)
    return ws


_FP_STATE_DTYPE = np.dtype([('iterations', '<i4'), ('active', '<i4'), ('fails', '<i4'), ('ticket', '<i4')])
FIXED_POINT_MAX_THRESHOLD = 1000        # the one-call fixed-point solves' ABI limit
_fp_workspaces = {}


class _FixedPointWorkspace(object):
    """Buffers of the one-call fixed-point solves (impflow_conv3_fixed_point / impflow_mlp_fixed_point) of one (B, d)
    size: the two iterates, the device state record, its pinned host copy followed by the conv solve's progress
    records, and the MLP kernel's per-CTA counts (on first use)."""

    def __init__(self, B, d, device):
        lib = _cabi.load()
        f32 = dict(device=device, dtype=torch.float32)
        self.xa = torch.empty(B, d, **f32)
        self.xb = torch.empty(B, d, **f32)
        self.state = torch.zeros(_FP_STATE_DTYPE.itemsize, device=device, dtype=torch.uint8)
        self.state_host = _cabi.pinned_bytes(int(lib.impflow_conv3_fixed_point_host_bytes(FIXED_POINT_MAX_THRESHOLD)))
        self.counts = None

    def mlp_counts(self):
        if self.counts is None:
            n = 2 * int(_cabi.load().impflow_mlp_solver_partial_doubles())
            self.counts = torch.empty(n, device=self.xa.device, dtype=torch.int32)
        return self.counts

    def iterations(self):
        return int(self.state_host[:_FP_STATE_DTYPE.itemsize].numpy().view(_FP_STATE_DTYPE)[0]['iterations'])


def fixed_point_workspace(B, d, device):
    """The fixed-point workspace of (B, d) on the current stream, cached like _workspace.  A solve drains its stream
    before it returns, so back-to-back solves may share one; solves on different streams get their own."""
    key = (B, d, device.index, getattr(_cabi.stream(), 'value', None))
    ws = _fp_workspaces.get(key)
    if ws is None:
        if len(_fp_workspaces) > 16:
            _fp_workspaces.clear()
        ws = _fp_workspaces[key] = _FixedPointWorkspace(B, d, device)
    return ws


def scaled_eps(eps, B, d):
    """The stopping tolerance of a solve on the norm of the whole (B, d) residual (broyden.py:131)."""
    return eps * math.sqrt(B * d)


def _result_dict(ws, state, shape, eps_scaled, threshold, result=None):
    """The reference's return dict (broyden.py:184-193).  `result`: a copy of ws.low_x the caller already took (the
    copy is the first thing enqueued after a solve: the stream is empty at that point)."""
    nstep = int(state['nstep'])
    return {'result': (result if result is not None else ws.low_x.clone()).view(shape),
            'nstep': nstep,
            'tnstep': nstep,
            'lowest_step': int(state['lowest_step']),
            'diff': float(state['lowest']),
            'diff_detail': torch.sqrt(ws.low_sq),
            'prot_break': bool(state['prot_break']),
            'trace': [float(t) for t in state['trace'][:nstep + 1]],
            'eps': eps_scaled,
            'threshold': threshold}


def broyden_mlp(spec, x_embed, z0, threshold, eps):
    """Whole forward/inverse solve of x_embed - f(z) - z = 0 in ONE persistent cooperative kernel
    (csrc/mlp_solver.cu) for small-d MLP branches.  `spec` comes from BranchProgram.mlp_solver_spec():
    (Wt list, bias list, dims, act_kind, per-layer softplus(beta) list or None).  Same return dict as broyden()."""
    _cabi.require_device(z0, 'broyden_mlp z0')
    lib = _cabi.load()
    Wt, bias, dims, act_kind, beta_sp = spec
    shape = z0.shape
    B = shape[0]
    d = z0.numel() // B
    assert d == dims[0] == dims[-1]
    eps_scaled = scaled_eps(eps, B, d)
    ws = _workspace(B, d, threshold, z0.device)
    ws.one_call_buffers(mlp=True)
    ws.xa.copy_(z0.reshape(B, d))
    L = len(Wt)
    wt_arr, b_arr, dims_arr, beta_arr = _mlp_arrays(Wt, bias, dims, beta_sp)
    xe = x_embed.reshape(B, d).contiguous()
    _cabi.check(lib.impflow_mlp_broyden_solve(
        _cabi.ptr(xe), wt_arr, b_arr, dims_arr, L, act_kind, beta_arr, _cabi.ptr(ws.xa),
        _cabi.ptr(ws.ga), _cabi.ptr(ws.xb), _cabi.ptr(ws.gb), _cabi.ptr(ws.low_x), _cabi.ptr(ws.low_g),
        _cabi.ptr(ws.Ut), _cabi.ptr(ws.Vt), _cabi.ptr(ws.sample_sq), _cabi.ptr(ws.low_sq),
        ctypes.c_void_p(ws.partial_d.data_ptr()), ctypes.c_void_p(ws.state.data_ptr()), B, threshold,
        float(eps_scaled), _cabi.stream()), 'mlp_broyden_solve')
    state = ws.read_state()
    return _result_dict(ws, state, shape, eps_scaled, threshold)


def broyden_mlp_vjp(spec, rhs, threshold, eps):
    """Whole implicit-backward solve v^T (I + J) = rhs (implicit_block.py:199-207) from zeros in ONE persistent
    cooperative kernel for small-d MLP branches.  `spec` comes from BranchProgram.mlp_vjp_spec(saved):
    (effective weights [out][ld], row strides, act' multipliers (None for layer 0), dims).  Same return dict as
    broyden()."""
    _cabi.require_device(rhs, 'broyden_mlp_vjp rhs')
    lib = _cabi.load()
    W, ldw, dmul, dims = spec
    shape = rhs.shape
    B = shape[0]
    d = rhs.numel() // B
    assert d == dims[0] == dims[-1]
    eps_scaled = scaled_eps(eps, B, d)
    ws = _workspace(B, d, threshold, rhs.device)
    ws.one_call_buffers(mlp=True)
    ws.xa.zero_()
    L = len(W)
    w_arr = (ctypes.c_void_p * L)(*[w.data_ptr() for w in W])
    ld_arr = (ctypes.c_int * L)(*[int(v) for v in ldw])
    dm_arr = (ctypes.c_void_p * L)(*[(t.data_ptr() if t is not None else None) for t in dmul])
    dims_arr = (ctypes.c_int * (L + 1))(*dims)
    r = rhs.reshape(B, d).contiguous()
    _cabi.check(lib.impflow_mlp_broyden_solve_vjp(
        _cabi.ptr(r), w_arr, ld_arr, dm_arr, dims_arr, L, _cabi.ptr(ws.xa), _cabi.ptr(ws.ga), _cabi.ptr(ws.xb),
        _cabi.ptr(ws.gb), _cabi.ptr(ws.low_x), _cabi.ptr(ws.low_g), _cabi.ptr(ws.Ut), _cabi.ptr(ws.Vt),
        _cabi.ptr(ws.sample_sq), _cabi.ptr(ws.low_sq), ctypes.c_void_p(ws.partial_d.data_ptr()),
        ctypes.c_void_p(ws.state.data_ptr()), B, threshold, float(eps_scaled), _cabi.stream()), 'mlp_broyden_solve_vjp')
    state = ws.read_state()
    return _result_dict(ws, state, shape, eps_scaled, threshold)


def _mlp_arrays(Wt, bias, dims, beta_sp):
    """ctypes arrays of the persistent kernels' forward-mode weight description (BranchProgram.mlp_solver_spec)."""
    L = len(Wt)
    wt_arr = (ctypes.c_void_p * L)(*[w.data_ptr() for w in Wt])
    b_arr = (ctypes.c_void_p * L)(*[(b.data_ptr() if b is not None else None) for b in bias])
    dims_arr = (ctypes.c_int * (L + 1))(*dims)
    # one device scalar per activation: every Swish module owns its own learnable beta (activations.py:64-71)
    beta_arr = None
    if beta_sp is not None:
        beta_arr = (ctypes.c_void_p * L)(*([_cabi.ptr(b, 'beta') for b in beta_sp] + [None] * (L - len(beta_sp))))
    return wt_arr, b_arr, dims_arr, beta_arr


def fixed_point_mlp(spec, rhs, start, atol, rtol, threshold):
    """Banach iteration x <- rhs - f(x) from `start` (iresblock.py:69-79, implicit_block.py:17-28) in ONE persistent
    cooperative kernel (csrc/mlp_solver.cu: k_mlp_fixed_point) for the MLP branches `spec` describes
    (BranchProgram.mlp_solver_spec).  Returns (x shaped like rhs, the reference's iteration count)."""
    _cabi.require_device(rhs, 'fixed_point_mlp rhs')
    lib = _cabi.load()
    Wt, bias, dims, act_kind, beta_sp = spec
    d = dims[0]
    r = rhs.reshape(-1, d).contiguous()
    s = start.reshape(-1, d).contiguous()
    B = r.shape[0]
    ws = fixed_point_workspace(B, d, r.device)
    out = torch.empty_like(r)
    wt_arr, b_arr, dims_arr, beta_arr = _mlp_arrays(Wt, bias, dims, beta_sp)
    _cabi.check(lib.impflow_mlp_fixed_point(
        _cabi.ptr(r), _cabi.ptr(s), _cabi.ptr(out), wt_arr, b_arr, dims_arr, len(Wt), act_kind, beta_arr,
        _cabi.ptr(ws.xa), _cabi.ptr(ws.xb), ctypes.c_void_p(ws.mlp_counts().data_ptr()),
        ctypes.c_void_p(ws.state.data_ptr()), ctypes.c_void_p(ws.state_host.data_ptr()), B, float(atol), float(rtol),
        int(threshold), _cabi.stream()), 'mlp_fixed_point')
    return out.view(rhs.shape), ws.iterations()


def broyden(g_, x0, threshold, eps, ls=False, name='unknown'):
    """Find x with g_(x) = 0, starting at x0.  Same return dict as the reference
    (broyden.py:184-193)."""
    if ls:
        raise NotImplementedError('impflow_b200: the Armijo line search is dead code in the reference '
                                  '(both call sites use ls=False) and is not implemented')
    _cabi.require_device(x0, 'broyden x0')
    lib = _cabi.load()
    shape = x0.shape
    B = shape[0]
    d = x0.numel() // B
    eps_scaled = scaled_eps(eps, B, d)
    ws = _workspace(B, d, threshold, x0.device)
    st = _cabi.stream

    def g(x2d):
        out = g_(x2d.view(shape))
        out = out.reshape(B, d)
        if out.dtype != torch.float32 or not out.is_contiguous():
            out = out.contiguous().float()
        return out

    x_old, xn = ws.xa, ws.xb
    x_old.copy_(x0.reshape(B, d))
    gx = g(x_old)
    sp = ctypes.c_void_p(ws.state.data_ptr())
    _cabi.check(lib.impflow_broyden_begin(_cabi.ptr(x_old), _cabi.ptr(gx), _cabi.ptr(xn), _cabi.ptr(ws.low_x),
                                          _cabi.ptr(ws.low_g), _cabi.ptr(ws.sample_sq), _cabi.ptr(ws.low_sq),
                                          _cabi.ptr(ws.partial), sp, B, d, threshold, float(eps_scaled), st()),
                'broyden_begin')
    state = ws.read_state()
    while state['active']:
        gn = g(xn)
        _cabi.check(lib.impflow_broyden_step(_cabi.ptr(x_old), _cabi.ptr(gx), _cabi.ptr(xn), _cabi.ptr(gn),
                                             _cabi.ptr(ws.Ut), _cabi.ptr(ws.Vt), _cabi.ptr(ws.low_x),
                                             _cabi.ptr(ws.low_g), _cabi.ptr(ws.sample_sq), _cabi.ptr(ws.low_sq),
                                             _cabi.ptr(ws.partial), sp, B, d, threshold, st()), 'broyden_step')
        x_old, xn = xn, x_old        # the kernel wrote the next iterate into the old buffer
        gx = gn
        state = ws.read_state()
    return _result_dict(ws, state, shape, eps_scaled, threshold)
