"""Python-side operator layer over the C ABI.

Two kinds of entry points:
  * raw launchers (``act_mul``, ``gemm_nt`` ...): allocate outputs with torch, call the kernel
    on the current CUDA stream; used directly on the no-grad hot loops (Broyden g evaluations,
    Neumann vjp chain);
  * ``torch.autograd.Function`` primitives built from those launchers whose backward passes are
    expressed with the same primitives, so the graph can be differentiated repeatedly (the
    log-det estimators differentiate through vjps: implicit_block.py:386-388, 418-438).
"""
import ctypes

import torch

from . import _cabi

ACT_NONE, ACT_SIN, ACT_LIPSWISH, ACT_RELU = 0, 1, 2, 3
ACT_MULTIPLIER = 4      # dmul epilogues only: the dmul operand already holds act'(pre)

# GEMM backend policy: 'auto' uses the tcgen05 3xTF32 kernel whenever its layout constraints hold
# and the problem is big enough to fill tiles; 'simt' forces the exact-fp32 CUDA-core kernel.
# min_flops_tc_autograd: below this the autograd primitive stays on the CUDA cores (one launch instead of two plane
# splits + the tensor-core launch; the MLP layers of the toy / tabular flows are 33 MFLOP)
_BACKEND = {'mode': 'auto', 'min_flops_tc': 2 * 128 * 128 * 64, 'min_flops_tc_autograd': 1.0e9}


# bench.py switches this on inside its timed region to collect (start, end, flop) CUDA events of
# every tcgen05 GEMM launch for the roofline line.
GEMM_PROFILE = {'on': False, 'shapes': {}}


CHAIN23 = {'on': True}      # mirrors impflow_conv3_set_chain23 (bookkeeping of the launches a native call makes)


def record_gemm(M, N, K, has_pre, has_act, has_dmul, has_split, split_k):
    key = (int(M), int(N), int(K), bool(has_pre), bool(has_act), bool(has_dmul), bool(has_split), bool(split_k))
    GEMM_PROFILE['shapes'][key] = GEMM_PROFILE['shapes'].get(key, 0) + 1


def time_gemm_shape(key, reps=5, flush=None):
    """Median CUDA-event duration (ms) of one tcgen05 GEMM launch of the recorded shape `key`, with the
    L2 flushed by a 256 MB memset that also keeps the stream busy while the launch is enqueued (so the
    event pair brackets the kernel alone, not host latency)."""
    M, N, K, has_pre, has_act, has_dmul, has_split, split_k = key
    dev = torch.device('cuda', torch.cuda.current_device())
    A = torch.randn(M, K, device=dev)
    Bm = torch.randn(N, K, device=dev) / max(K, 1) ** 0.5
    As, Bs = split_tf32(A), split_tf32(Bm)
    dm = torch.randn(M, N, device=dev) if has_dmul else None
    beta = torch.full((1,), 0.97, device=dev)
    if flush is None:
        flush = torch.empty(64 * 1024 * 1024, device=dev)
    times = []
    was = GEMM_PROFILE['on']
    GEMM_PROFILE['on'] = False
    for i in range(reps + 1):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gemm_nt(A, Bm, None, act_kind=ACT_MULTIPLIER if has_dmul else (ACT_LIPSWISH if has_act or has_split else ACT_NONE),
                beta_sp=beta,
                want_pre=has_pre and not has_dmul, want_act=has_act, dmul_pre=dm, A_split=As, B_split=Bs,
                want_split=has_split)
        e1.record()
        torch.cuda.synchronize()
        if i > 0:
            times.append(e0.elapsed_time(e1))
    GEMM_PROFILE['on'] = was
    return sorted(times)[len(times) // 2]


def time_branch3_shape(key, reps=5, flush=None):
    """Median CUDA-event duration (ms) of one fused branch tile-kernel launch of the recorded shape."""
    _, M, C, N3, is_vjp, save_pre = key
    dev = torch.device('cuda', torch.cuda.current_device())
    x0 = torch.zeros(M, 32, device=dev)
    x0[:, :N3] = torch.randn(M, N3, device=dev)
    W1 = split_tf32(torch.randn(C, 32, device=dev) / 5)
    W2 = split_tf32(torch.randn(C, C, device=dev) / C ** 0.5)
    W3 = split_tf32(torch.randn(N3, C, device=dev) / C ** 0.5)
    b1, b2 = torch.randn(C, device=dev), torch.randn(C, device=dev)
    beta = torch.full((1,), 0.97, device=dev)
    m1 = torch.randn(M, C, device=dev) if is_vjp else None
    m2 = torch.randn(M, C, device=dev) if is_vjp else None
    if flush is None:
        flush = torch.empty(64 * 1024 * 1024, device=dev)
    was = GEMM_PROFILE['on']
    GEMM_PROFILE['on'] = False
    times = []
    for i in range(reps + 1):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if is_vjp:
            branch3_tc(x0, W1, W2, W3, N3, mul1=m1, mul2=m2)
        else:
            branch3_tc(x0, W1, W2, W3, N3, bias1=b1, bias2=b2, act_kind=ACT_LIPSWISH, beta1=beta, beta2=beta,
                       save_pre=save_pre)
        e1.record()
        torch.cuda.synchronize()
        if i > 0:
            times.append(e0.elapsed_time(e1))
    GEMM_PROFILE['on'] = was
    return sorted(times)[len(times) // 2]


def time_wgrad_shape(key, reps=5, flush=None):
    """Median CUDA-event duration (ms) of one MN-major weight-gradient launch (kernel + fixed-order reduce)."""
    _, M, N1, N2 = key
    dev = torch.device('cuda', torch.cuda.current_device())
    Gs = split_tf32(torch.randn(M, N1, device=dev))
    As = split_tf32(torch.randn(M, N2, device=dev))
    if flush is None:
        flush = torch.empty(64 * 1024 * 1024, device=dev)
    was = GEMM_PROFILE['on']
    GEMM_PROFILE['on'] = False
    times = []
    for i in range(reps + 1):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        wgrad_gemm(None, None, G_split=Gs, A_split=As)
        e1.record()
        torch.cuda.synchronize()
        if i > 0:
            times.append(e0.elapsed_time(e1))
    GEMM_PROFILE['on'] = was
    return sorted(times)[len(times) // 2]


# While a caller differentiates w.r.t. ACTIVATIONS only (the vjp chains of the log-det estimators,
# implicit_block.py:422,434,436), the parameter-gradient branches of the primitives' backward
# passes (weight-gradient GEMMs with their transposes, bias column sums, LipSwish beta reductions)
# are dead work: ctx.needs_input_grad is fixed at forward time and cannot tell.  The estimators
# switch this flag on around those torch.autograd.grad calls.
_ACT_ONLY = {'on': False}


class activations_only(object):
    """Context manager: backward passes of the kernel primitives skip parameter gradients."""

    def __enter__(self):
        self._prev = _ACT_ONLY['on']
        _ACT_ONLY['on'] = True

    def __exit__(self, *exc):
        _ACT_ONLY['on'] = self._prev


def set_gemm_backend(mode):
    assert mode in ('auto', 'simt', 'tc')
    _BACKEND['mode'] = mode


def get_gemm_backend():
    return _BACKEND['mode']


def _lib():
    return _cabi.load()


def _dense(t):
    """A tensor whose memory is one dense block (contiguous in *some* permutation)."""
    if t.is_contiguous() or (t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last)):
        return t
    return t.contiguous()


def _match_layout(t, ref):
    """t laid out in memory exactly like ref (same strides)."""
    if t.stride() == ref.stride() and t.shape == ref.shape:
        return t
    out = torch.empty_like(ref)
    out.copy_(t)
    return out


# ------------------------------------------------------------------------------------------
# raw launchers
# ------------------------------------------------------------------------------------------

def act_mul(x, g, kind, order, beta_sp=None, out=None):
    """out = g * act^(order)(x); x dense in any memory order, g (optional) in the same order."""
    x = _dense(x)
    if g is not None:
        g = _match_layout(g, x)
    if out is None:
        out = torch.empty_like(x)
    _cabi.check(_lib().impflow_act_mul(_cabi.ptr(x, 'x'), _cabi.ptr(g, 'g', True), _cabi.ptr(out, 'out'),
                                       x.numel(), kind, order, _cabi.ptr(beta_sp, 'beta_sp', True),
                                       _cabi.stream()), 'act_mul')
    return out


def act_split(x, kind, order, beta_sp=None):
    """(hi, lo) tf32 planes of act^(order)(x) in one pass."""
    x = x.contiguous()
    hi, lo = torch.empty_like(x), torch.empty_like(x)
    _cabi.check(_lib().impflow_act_split(_cabi.ptr(x), _cabi.ptr(hi), _cabi.ptr(lo), x.numel(), kind, order,
                                         _cabi.ptr(beta_sp, 'beta_sp', True), _cabi.stream()), 'act_split')
    return hi, lo


def act_beta_grad(x, g, order, beta_sp, g2=None):
    """sum(g * g2 * d/dbeta act^(order)(x)) as a 1-element tensor."""
    x = _dense(x)
    g = _match_layout(g, x)
    if g2 is not None:
        g2 = _match_layout(g2, x)
    out = torch.empty(1, device=x.device, dtype=torch.float32)
    ws = torch.empty(int(_lib().impflow_reduce_workspace_floats(x.numel())), device=x.device, dtype=torch.float32)
    _cabi.check(_lib().impflow_act_beta_grad(_cabi.ptr(x), _cabi.ptr(g), _cabi.ptr(g2, 'g2', True), _cabi.ptr(out),
                                             _cabi.ptr(ws), x.numel(), order, _cabi.ptr(beta_sp), _cabi.stream()),
                'act_beta_grad')
    return out


def act_second(p, t, ga, gb, kind, beta_sp=None):
    """act''(p) * t * ga + act'(p) * gb  (gb optional)."""
    p = _dense(p)
    t, ga = _match_layout(t, p), _match_layout(ga, p)
    if gb is not None:
        gb = _match_layout(gb, p)
    out = torch.empty_like(p)
    _cabi.check(_lib().impflow_act_second(_cabi.ptr(p), _cabi.ptr(t), _cabi.ptr(ga), _cabi.ptr(gb, 'gb', True),
                                          _cabi.ptr(out), p.numel(), kind, _cabi.ptr(beta_sp, 'beta', True),
                                          _cabi.stream()), 'act_second')
    return out


def neumann_act_bwd(p, t, ta, ab, beta_sp):
    """Fused activation step of the Neumann reverse sweep (LipSwish): returns ((ybar_hi, ybar_lo), colsum (N,),
    beta_grad (1,)) for ybar = act''(p) t ta + act'(p) ab; see impflow_neumann_act_bwd."""
    p = p.contiguous()
    M, N = p.shape
    t, ta = _match_layout(t, p), _match_layout(ta, p)
    if ab is not None:
        ab = _match_layout(ab, p)
    dev = p.device
    hi, lo = torch.empty_like(p), torch.empty_like(p)
    colsum_out = torch.empty(N, device=dev, dtype=torch.float32)
    bg = torch.empty(1, device=dev, dtype=torch.float32)
    lib = _lib()
    ws = torch.empty(int(lib.impflow_neumann_act_bwd_workspace_floats(M, N)), device=dev, dtype=torch.float32)
    _cabi.check(lib.impflow_neumann_act_bwd(_cabi.ptr(p), _cabi.ptr(t), _cabi.ptr(ta), _cabi.ptr(ab, 'ab', True),
                                            _cabi.ptr(hi), _cabi.ptr(lo), _cabi.ptr(colsum_out), _cabi.ptr(bg),
                                            _cabi.ptr(ws), M, N, _cabi.ptr(beta_sp), _cabi.stream()),
                'neumann_act_bwd')
    return (hi, lo), colsum_out, bg


def lincomb3(a, ca, b=None, cb=0.0, c=None, cc=0.0, out=None):
    """out = ca*a + cb*b + cc*c (same shapes; laid out like a)."""
    a = _dense(a)
    if b is not None:
        b = _match_layout(b, a)
    if c is not None:
        c = _match_layout(c, a)
    if out is None:
        out = torch.empty_like(a)
    _cabi.check(_lib().impflow_lincomb3(_cabi.ptr(a), ca, _cabi.ptr(b, 'b', True), cb, _cabi.ptr(c, 'c', True), cc,
                                        _cabi.ptr(out), a.numel(), _cabi.stream()), 'lincomb3')
    return out


def rowdot(a, c, out=None, alpha=1.0, beta=0.0):
    """out[b] = beta*out[b] + alpha*<a[b], c[b]> over everything but dim 0."""
    a = _dense(a)
    c = _match_layout(c, a)
    B = a.shape[0]
    if out is None:
        out = torch.empty(B, device=a.device, dtype=torch.float32)
        beta = 0.0
    _cabi.check(_lib().impflow_rowdot(_cabi.ptr(a), _cabi.ptr(c), _cabi.ptr(out), B, a.numel() // max(B, 1), alpha,
                                      beta, _cabi.stream()), 'rowdot')
    return out


def colsum(a2d):
    a2d = a2d.contiguous()
    M, N = a2d.shape
    out = torch.empty(N, device=a2d.device, dtype=torch.float32)
    chunks = int(_lib().impflow_colsum_chunks(M, N))
    partial = torch.empty(chunks * N, device=a2d.device, dtype=torch.float32) if chunks > 1 else None
    _cabi.check(_lib().impflow_colsum(_cabi.ptr(a2d), _cabi.ptr(out), _cabi.ptr(partial, 'partial', True), M, N,
                                      _cabi.stream()), 'colsum')
    return out


def transpose2d(a2d):
    a2d = a2d.contiguous()
    out = torch.empty(a2d.shape[1], a2d.shape[0], device=a2d.device, dtype=torch.float32)
    _cabi.check(_lib().impflow_transpose(_cabi.ptr(a2d), _cabi.ptr(out), a2d.shape[0], a2d.shape[1], _cabi.stream()),
                'transpose')
    return out


def im2col3x3(x_nhwc, ld=None):
    """(B,H,W,C) -> (B*H*W, ld) patch matrix, ld >= 9*C (tail zero-filled)."""
    x_nhwc = x_nhwc.contiguous()
    B, H, W, C = x_nhwc.shape
    ld = 9 * C if ld is None else ld
    col = torch.empty(B * H * W, ld, device=x_nhwc.device, dtype=torch.float32)
    _cabi.check(_lib().impflow_im2col3x3(_cabi.ptr(x_nhwc), _cabi.ptr(col), B, H, W, C, ld, _cabi.stream()),
                'im2col3x3')
    return col


def im2col3x3_split(x_nhwc, ld=None):
    """im2col3x3 written directly as the tf32 (hi, lo) planes the tcgen05 GEMM consumes."""
    x_nhwc = x_nhwc.contiguous()
    B, H, W, C = x_nhwc.shape
    ld = 9 * C if ld is None else ld
    hi = torch.empty(B * H * W, ld, device=x_nhwc.device, dtype=torch.float32)
    lo = torch.empty_like(hi)
    _cabi.check(_lib().impflow_im2col3x3_split(_cabi.ptr(x_nhwc), _cabi.ptr(hi), _cabi.ptr(lo), B, H, W, C, ld,
                                               _cabi.stream()), 'im2col3x3_split')
    return hi, lo


def transpose_split(a2d):
    """tf32 (hi, lo) planes of a2d^T in one pass."""
    a2d = a2d.contiguous()
    M, N = a2d.shape
    hi = torch.empty(N, M, device=a2d.device, dtype=torch.float32)
    lo = torch.empty_like(hi)
    _cabi.check(_lib().impflow_transpose_split(_cabi.ptr(a2d), _cabi.ptr(hi), _cabi.ptr(lo), M, N, _cabi.stream()),
                'transpose_split')
    return hi, lo


WGRAD_MN_MAJOR = {'on': True}      # A/B switch: False = transposed copies + the K-major GEMM


def wgrad_gemm(G, A, G_split=None, A_split=None):
    """dW (N1, N2) = G^T A for G (M, N1), A (M, N2): the weight-gradient contraction over all rows (pixels).
    tcgen05 path: the row-major hi/lo planes of both operands go to the tensor core as MN-major tiles
    (csrc/wgrad_tcgen05.cu); planes that already exist (they also feed the neighbouring GEMMs) are reused."""
    M, N1 = G.shape if G is not None else G_split[0].shape
    N2 = A.shape[1] if A is not None else A_split[0].shape[1]
    dev = (G if G is not None else G_split[0]).device
    if _tc_ok(N1, N2, M, M, M) and WGRAD_MN_MAJOR['on'] and N1 % 4 == 0 and N2 % 4 == 0:
        lib = _lib()
        Gs = G_split if G_split is not None else split_tf32(G)
        As = A_split if A_split is not None else split_tf32(A)
        assert Gs[0].is_contiguous() and As[0].is_contiguous()
        out = torch.empty(N1, N2, device=dev, dtype=torch.float32)
        # the wider operand becomes the 128-row (M) side of the MMA tiles
        swap = N1 < N2 and N1 < 128
        (Xs, n_x), (Ys, n_y) = ((As, N2), (Gs, N1)) if swap else ((Gs, N1), (As, N2))
        ws = torch.empty(int(lib.impflow_wgrad_tc_workspace_floats(M, n_x, n_y)), device=dev, dtype=torch.float32)
        _cabi.check(lib.impflow_wgrad_tc(_cabi.ptr(Xs[0]), _cabi.ptr(Xs[1]), n_x, _cabi.ptr(Ys[0]), _cabi.ptr(Ys[1]),
                                         n_y, _cabi.ptr(out), N2, 1 if swap else 0, M, n_x, n_y, _cabi.ptr(ws),
                                         _cabi.stream()), 'wgrad_tc')
        if GEMM_PROFILE['on']:
            key = ('wgrad', int(M), int(n_x), int(n_y))
            GEMM_PROFILE['shapes'][key] = GEMM_PROFILE['shapes'].get(key, 0) + 1
        return out
    if G is None:
        G = lincomb3(G_split[0], 1.0, G_split[1], 1.0)
    if A is None:
        A = lincomb3(A_split[0], 1.0, A_split[1], 1.0)
    if _tc_ok(N1, N2, M, M, M):
        return gemm_nt(None, None, A_split=transpose_split(G), B_split=transpose_split(A))[0]
    # small / ragged shapes (MLP flows): exact fp32, split along the rows, no transposed copies
    lib = _lib()
    G, A = G.contiguous(), A.contiguous()
    out = torch.empty(N1, N2, device=dev, dtype=torch.float32)
    ws = torch.empty(max(int(lib.impflow_wgrad_simt_workspace_floats(M, N1, N2)), 1), device=dev, dtype=torch.float32)
    _cabi.check(lib.impflow_wgrad_simt(_cabi.ptr(G), G.stride(0), _cabi.ptr(A), A.stride(0), _cabi.ptr(out), N2, M,
                                       N1, N2, _cabi.ptr(ws), _cabi.stream()), 'wgrad_simt')
    return out


def mlp_series(spec, v, coeffs):
    """Left / right vectors, their combinations and the estimate of the basic power series of a small-d MLP branch in
    one launch (csrc/mlp_solver.cu k_mlp_series).  spec: BranchProgram.mlp_series_spec(saved).  Returns
    (S (B,), Ls (n+1, B, d), Rs (n, B, d), Wm (n, B, d))."""
    W, ldw, Wt, dmul, dims = spec
    lib = _lib()
    v2 = v.reshape(v.shape[0], -1).contiguous()
    B, d = v2.shape
    n, L = len(coeffs), len(W)
    dev = v2.device
    Ls = torch.empty(n + 1, B, d, device=dev, dtype=torch.float32)
    Rs = torch.empty(n, B, d, device=dev, dtype=torch.float32)
    Wm = torch.empty(n, B, d, device=dev, dtype=torch.float32)
    S = torch.empty(B, device=dev, dtype=torch.float32)
    w_arr = (ctypes.c_void_p * L)(*[w.data_ptr() for w in W])
    ld_arr = (ctypes.c_int * L)(*[int(t) for t in ldw])
    wt_arr = (ctypes.c_void_p * L)(*[w.data_ptr() for w in Wt])
    dm_arr = (ctypes.c_void_p * L)(*[(t.data_ptr() if t is not None else None) for t in dmul])
    dims_arr = (ctypes.c_int * (L + 1))(*dims)
    c_arr = (ctypes.c_double * n)(*[float(c) for c in coeffs])
    _cabi.check(lib.impflow_mlp_series(_cabi.ptr(v2), w_arr, ld_arr, wt_arr, dm_arr, dims_arr, L, B, n, c_arr,
                                       _cabi.ptr(Ls), _cabi.ptr(Rs), _cabi.ptr(Wm), _cabi.ptr(S), _cabi.stream()),
                'mlp_series')
    return S, Ls, Rs, Wm


def col2im3x3(col, B, H, W, C, bias=None, act_kind=ACT_NONE, beta_sp=None, want_pre=True, want_act=False,
              dmul_pre=None):
    col = col.contiguous()
    dev = col.device
    pre = torch.empty(B, H, W, C, device=dev, dtype=torch.float32) if (want_pre or dmul_pre is not None) else None
    act = torch.empty(B, H, W, C, device=dev, dtype=torch.float32) if want_act else None
    _cabi.check(_lib().impflow_col2im3x3(_cabi.ptr(col), B, H, W, C, _cabi.ptr(bias, 'bias', True),
                                         _cabi.ptr(pre, 'pre', True), _cabi.ptr(act, 'act', True),
                                         _cabi.ptr(dmul_pre, 'dmul', True), act_kind,
                                         _cabi.ptr(beta_sp, 'beta', True), _cabi.stream()), 'col2im3x3')
    return pre, act


def split_tf32(a):
    a = a.contiguous()
    hi = torch.empty_like(a)
    lo = torch.empty_like(a)
    _cabi.check(_lib().impflow_split_tf32(_cabi.ptr(a), _cabi.ptr(hi), _cabi.ptr(lo), a.numel(), _cabi.stream()),
                'split_tf32')
    return hi, lo


def _tc_ok(M, N, K, lda, ldb):
    mode = _BACKEND['mode']
    if mode == 'simt':
        return False
    ok = (K % 32 == 0) and (lda % 4 == 0) and (ldb % 4 == 0)
    if mode == 'tc':
        return ok
    return ok and (2 * M * N * K >= _BACKEND['min_flops_tc']) and N >= 8


def gemm_nt(A, Bm, bias=None, act_kind=ACT_NONE, beta_sp=None, want_pre=True, want_act=False, dmul_pre=None,
            A_split=None, B_split=None, want_split=False):
    """C = A @ Bm^T (+bias) with the fused epilogue.  A (M,K), Bm (N,K) row-major.

    Returns (pre, act, split) where split is None or the (hi, lo) tf32 planes of the value that
    feeds the next GEMM (only produced by the tcgen05 backend)."""
    if A is None or Bm is None:      # operands given as planes only
        assert A_split is not None and B_split is not None, 'gemm_nt: planes missing'
        M, K = A_split[0].shape
        N = B_split[0].shape[0]
        assert B_split[0].shape[1] == K, 'gemm_nt: inner dimensions differ'
    else:
        A = A.contiguous()
        Bm = Bm.contiguous()
        M, K = A.shape
        N = Bm.shape[0]
        assert Bm.shape[1] == K, 'gemm_nt: inner dimensions differ'
    if K % 32 != 0 and _BACKEND['mode'] != 'simt' and N >= 8 and 2 * M * N * K >= 64 * _BACKEND['min_flops_tc'] \
            and A_split is None and B_split is None:
        # a large GEMM with an odd inner dimension (e.g. K = 9*3 = 27): zero-pad K so that it runs on
        # the tcgen05 kernel instead of CUDA cores
        pad = (K + 31) // 32 * 32 - K
        A = torch.nn.functional.pad(A, (0, pad))
        Bm = torch.nn.functional.pad(Bm, (0, pad))
        K += pad
    dev = (A if A is not None else A_split[0]).device
    need_pre = want_pre or dmul_pre is not None
    pre = torch.empty(M, N, device=dev, dtype=torch.float32) if need_pre else None
    act = torch.empty(M, N, device=dev, dtype=torch.float32) if want_act else None
    if dmul_pre is not None:
        dmul_pre = dmul_pre.contiguous()
    lib = _lib()
    if _tc_ok(M, N, K, K, K):
        Ah, Al = A_split if A_split is not None else split_tf32(A)
        Bh, Bl = B_split if B_split is not None else split_tf32(Bm)
        sh = torch.empty(M, N, device=dev, dtype=torch.float32) if want_split else None
        sl = torch.empty(M, N, device=dev, dtype=torch.float32) if want_split else None
        ws = None
        if act is None and dmul_pre is None and not want_split:
            splits = int(lib.impflow_gemm_tc_splits(M, N, K))
            if splits > 1:
                ws = torch.empty(splits * M * N, device=dev, dtype=torch.float32)
        _cabi.check(lib.impflow_gemm_nt_tc(_cabi.ptr(Ah), _cabi.ptr(Al), K, _cabi.ptr(Bh), _cabi.ptr(Bl), K,
                                           _cabi.ptr(bias, 'bias', True), _cabi.ptr(pre, 'pre', True),
                                           _cabi.ptr(act, 'act', True), _cabi.ptr(dmul_pre, 'dmul', True),
                                           _cabi.ptr(sh, 'sh', True), _cabi.ptr(sl, 'sl', True), N, M, N, K,
                                           act_kind, _cabi.ptr(beta_sp, 'beta', True),
                                           _cabi.ptr(ws, 'ws', True), _cabi.stream()),
                    'gemm_nt_tc')
        if GEMM_PROFILE['on']:
            record_gemm(M, N, K, pre is not None, act is not None, dmul_pre is not None, want_split, ws is not None)
        return pre, act, ((sh, sl) if want_split else None)
    _cabi.check(lib.impflow_gemm_nt(_cabi.ptr(A), K, _cabi.ptr(Bm), K, _cabi.ptr(bias, 'bias', True),
                                    _cabi.ptr(pre, 'pre', True), _cabi.ptr(act, 'act', True),
                                    _cabi.ptr(dmul_pre, 'dmul', True), N, M, N, K, act_kind,
                                    _cabi.ptr(beta_sp, 'beta', True), _cabi.stream()), 'gemm_nt')
    return pre, act, None


def branch3_tc(x0, W1s, W2s, W3s, N3, bias1=None, bias2=None, mul1=None, mul2=None, act_kind=ACT_NONE, beta1=None,
               beta2=None, save_pre=False):
    """Fused narrow -> C -> C -> narrow chain (csrc/branch_fused.cu): returns (Y (M,N3), pre1, pre2).

    x0 (M, >=32) fp32; W1s/W2s/W3s = (hi, lo) tf32 planes of (C,32), (C,C), (N3,C) K-major weights.
    mul_l given: psi_l(t) = t * mul_l (vjp through the activation); else psi_l(t) = act(t + bias_l)."""
    x0 = x0.contiguous()
    M, ldx = x0.shape
    C = W2s[0].shape[0]
    dev = x0.device
    pre1 = torch.empty(M, C, device=dev, dtype=torch.float32) if save_pre else None
    pre2 = torch.empty(M, C, device=dev, dtype=torch.float32) if save_pre else None
    out = torch.zeros(M, N3, device=dev, dtype=torch.float32) if C > 256 else \
        torch.empty(M, N3, device=dev, dtype=torch.float32)
    _cabi.check(_lib().impflow_branch3_tc(
        _cabi.ptr(x0), ldx, _cabi.ptr(W1s[0]), _cabi.ptr(W1s[1]), _cabi.ptr(W2s[0]), _cabi.ptr(W2s[1]),
        _cabi.ptr(W3s[0]), _cabi.ptr(W3s[1]), _cabi.ptr(bias1, 'bias1', True), _cabi.ptr(bias2, 'bias2', True),
        _cabi.ptr(mul1, 'mul1', True), _cabi.ptr(mul2, 'mul2', True), _cabi.ptr(pre1, 'pre1', True),
        _cabi.ptr(pre2, 'pre2', True), _cabi.ptr(out), N3, M, C, N3, act_kind, _cabi.ptr(beta1, 'beta1', True),
        _cabi.ptr(beta2, 'beta2', True), _cabi.stream()), 'branch3_tc')
    if GEMM_PROFILE['on']:
        record_branch3(M, C, N3, mul1 is not None, save_pre)
    return out, pre1, pre2


def chain23_tc(A_split, W2s, W3s, N3, bias2=None, mul2=None, act_kind=ACT_NONE, beta2=None, save_pre=False):
    """Fused layers 2 + 3 (csrc/chain23_fused.cu): returns (partials (Q, M, N3) with Q = C/128, pre2 or None);
    the layer output is partials.sum(0) (summed in fixed order by the col2im kernel on the product path).

    A_split = (hi, lo) tf32 planes of the (M, C) layer-2 input, or ONE fp32 tensor (the kernel then derives the planes
    on chip: same roundings, same result); W2s / W3s = planes of the (C, C) and (N3, C)
    K-major weights; mul2 given: psi2(t) = t * mul2, else psi2(t) = act(t + bias2)."""
    if torch.is_tensor(A_split):
        A_split = (A_split, None)
    M, C = A_split[0].shape
    dev = A_split[0].device
    Q = int(_lib().impflow_chain23_parts(C))
    pre2 = torch.empty(M, C, device=dev, dtype=torch.float32) if save_pre else None
    out = torch.empty(Q, M, N3, device=dev, dtype=torch.float32)
    _cabi.check(_lib().impflow_chain23_tc(
        _cabi.ptr(A_split[0]), _cabi.ptr(A_split[1], 'A_lo', True), C, _cabi.ptr(W2s[0]), _cabi.ptr(W2s[1]), _cabi.ptr(W3s[0]),
        _cabi.ptr(W3s[1]), _cabi.ptr(bias2, 'bias2', True), _cabi.ptr(mul2, 'mul2', True), _cabi.ptr(pre2, 'pre2', True),
        _cabi.ptr(out), N3, M * N3, M, C, N3, act_kind, _cabi.ptr(beta2, 'beta2', True), _cabi.stream()), 'chain23_tc')
    if GEMM_PROFILE['on']:
        record_chain23(M, C, N3, mul2 is not None, save_pre)
    return out, pre2


def record_chain23(M, C, N3, is_vjp, save_pre):
    key = ('chain23', int(M), int(C), int(N3), bool(is_vjp), bool(save_pre))
    GEMM_PROFILE['shapes'][key] = GEMM_PROFILE['shapes'].get(key, 0) + 1


def time_chain23_shape(key, reps=5, flush=None):
    """Median CUDA-event duration (ms) of one fused layer-2+3 launch of the recorded shape."""
    _, M, C, N3, is_vjp, save_pre = key
    dev = torch.device('cuda', torch.cuda.current_device())
    A = split_tf32(torch.randn(M, C, device=dev))
    W2 = split_tf32(torch.randn(C, C, device=dev) / C ** 0.5)
    W3 = split_tf32(torch.randn(N3, C, device=dev) / C ** 0.5)
    b2 = torch.randn(C, device=dev)
    beta = torch.full((1,), 0.97, device=dev)
    m2 = torch.randn(M, C, device=dev) if is_vjp else None
    if flush is None:
        flush = torch.empty(64 * 1024 * 1024, device=dev)
    was = GEMM_PROFILE['on']
    GEMM_PROFILE['on'] = False
    times = []
    for i in range(reps + 1):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if is_vjp:
            chain23_tc(A, W2, W3, N3, mul2=m2)
        else:
            chain23_tc(A, W2, W3, N3, bias2=b2, act_kind=ACT_LIPSWISH, beta2=beta, save_pre=save_pre)
        e1.record()
        torch.cuda.synchronize()
        if i > 0:
            times.append(e0.elapsed_time(e1))
    GEMM_PROFILE['on'] = was
    return sorted(times)[len(times) // 2]


def record_branch3(M, C, N3, is_vjp, save_pre):
    key = ('branch3', int(M), int(C), int(N3), bool(is_vjp), bool(save_pre))
    GEMM_PROFILE['shapes'][key] = GEMM_PROFILE['shapes'].get(key, 0) + 1


def _mark_written(*tensors):
    """Kernels that update a caller's tensor in place through its raw pointer must bump its autograd version:
    the host caches (effective weights, d sigma / d W) are keyed on `_version`."""
    torch.autograd.graph.increment_version(tensors)


def sn_power_iter(W2d, u, v, n_iterations, atol, rtol, sigma_out=None):
    """In-place power iteration on (u, v); returns (sigma (1,), iters (1,) int32) device tensors.  sigma_out: a
    1-element fp32 tensor (e.g. the layer's `scale` buffer) that receives sigma directly."""
    W2d = W2d.contiguous()
    sigma = torch.empty(1, device=W2d.device, dtype=torch.float32) if sigma_out is None else sigma_out.view(1)
    iters = torch.empty(1, device=W2d.device, dtype=torch.int32)       # always written by the kernel
    n_it = -1 if n_iterations is None else int(n_iterations)
    _cabi.check(_lib().impflow_sn_power_iter(_cabi.ptr(W2d), _cabi.ptr(u), _cabi.ptr(v), _cabi.ptr(sigma),
                                             _cabi.iptr(iters), W2d.shape[0], W2d.shape[1], n_it,
                                             float(atol if atol is not None else 0.0),
                                             float(rtol if rtol is not None else 0.0), _cabi.stream()),
                'sn_power_iter')
    if n_it != 0:
        _mark_written(u, v)
    if sigma_out is not None:
        _mark_written(sigma_out)
    return sigma, iters


def sn_power_iter_conv(W, u, v, h, w, n_iterations, atol, rtol, want_D=False, sigma_out=None):
    """In-place power iteration of the 3x3 conv W (Cout,Cin,3,3) on one h x w image: one cooperative launch.
    Returns (sigma (1,), iters (1,) int32[, D = d sigma / d W]) device tensors, or None when the shape is not
    supported by the kernel (narrow side too large for shared memory) and the caller has to iterate itself."""
    W = W.contiguous()
    co, ci = W.shape[0], W.shape[1]
    n_ws = int(_lib().impflow_sn_conv_workspace_floats(co, ci, h, w))
    if n_ws == 0:
        return None
    ws = torch.empty(n_ws, device=W.device, dtype=torch.float32)
    sigma = torch.empty(1, device=W.device, dtype=torch.float32) if sigma_out is None else sigma_out.view(1)
    iters = torch.empty(1, device=W.device, dtype=torch.int32)         # always written by the kernel
    n_it = -1 if n_iterations is None else int(n_iterations)
    D = torch.empty_like(W) if want_D else None
    _cabi.check(_lib().impflow_sn_power_iter_conv3x3(
        _cabi.ptr(W), _cabi.ptr(u), _cabi.ptr(v), _cabi.ptr(sigma), _cabi.iptr(iters), co, ci, h, w, n_it,
        float(atol if atol is not None else 0.0), float(rtol if rtol is not None else 0.0), _cabi.ptr(ws),
        _cabi.ptr(D, 'D', True), _cabi.stream()), 'sn_power_iter_conv3x3')
    if n_it != 0:
        _mark_written(u, v)
    if sigma_out is not None:
        _mark_written(sigma_out)
    return (sigma, iters, D) if want_D else (sigma, iters)


def sn_rescale(W, sigma, coeff, scale_out=None):
    """W / max(1, sigma/coeff) with sigma a device scalar (no graph)."""
    W = W.contiguous()
    out = torch.empty_like(W)
    _cabi.check(_lib().impflow_sn_scale(_cabi.ptr(W), _cabi.ptr(sigma), float(coeff), _cabi.ptr(out),
                                        _cabi.ptr(scale_out, 'scale', True), W.numel(), _cabi.stream()), 'sn_scale')
    return out


def _prep_layouts(W, fwd_shape, fwd_planes, bwd_shape, bwd_planes):
    """Output tensors of the weight-preparation launch and the layout arguments after the scale operands."""
    dev = W.device
    mk = lambda shp: torch.empty(shp[0], shp[1], device=dev, dtype=torch.float32)
    f, b = mk(fwd_shape), mk(bwd_shape)
    fs = (mk(fwd_shape), mk(fwd_shape)) if fwd_planes else None
    bs = (mk(bwd_shape), mk(bwd_shape)) if bwd_planes else None
    args = (W.shape[0], W.shape[1], _cabi.ptr(f), _cabi.ptr(fs[0] if fs else None, 'fh', True),
            _cabi.ptr(fs[1] if fs else None, 'fl', True), fwd_shape[0], fwd_shape[1], _cabi.ptr(b),
            _cabi.ptr(bs[0] if bs else None, 'bh', True), _cabi.ptr(bs[1] if bs else None, 'bl', True), bwd_shape[0],
            bwd_shape[1], _cabi.stream())
    return (f, fs, b, bs), args


def prep_weights(W, sigma, coeff, kind, fwd_shape, fwd_planes, bwd_shape, bwd_planes):
    """Rescaled weight in the forward / transposed GEMM layouts (+ hi/lo planes) in one launch; see
    impflow_prep_weights.  *_shape = (rows, padded K)."""
    W = W.contiguous()
    out, args = _prep_layouts(W, fwd_shape, fwd_planes, bwd_shape, bwd_planes)
    _cabi.check(_lib().impflow_prep_weights(_cabi.ptr(W), _cabi.ptr(sigma), float(coeff), kind, *args),
                'prep_weights')
    return out


# Lop layers (LopLinear / LopConv2d): norm types of impflow_lop_norms and group modes of impflow_prep_weights_lop
LOP_L1, LOP_L2, LOP_MAX = 1, 2, 3
LOP_ONE, LOP_ROW, LOP_COL = 0, 1, 2


def lop_norm_type(norm_type):
    return {1: LOP_L1, 2: LOP_L2, float('inf'): LOP_MAX}[norm_type]


def lop_norms(W, axis, norm_type, scale_out=None):
    """Group norms of a Lop layer's weight (module layout), followed by their maximum: (groups + 1,) device tensor;
    scale_out (the layer's `scale` buffer) receives the maximum too.  See impflow_lop_norms."""
    W = W.contiguous()
    taps = W[0, 0].numel()
    norms = torch.empty((W.shape[0] if axis == 0 else W.shape[1]) + 1, device=W.device, dtype=torch.float32)
    _cabi.check(_lib().impflow_lop_norms(_cabi.ptr(W), W.shape[0], W.shape[1], taps, axis, norm_type,
                                         _cabi.ptr(norms), _cabi.ptr(scale_out, 'scale', True), _cabi.stream()),
                'lop_norms')
    return norms


def prep_weights_lop(W, norms, group, coeff, kind, fwd_shape, fwd_planes, bwd_shape, bwd_planes):
    """prep_weights for a Lop layer: W / max(1, n/coeff) with n one norm (group LOP_ONE: norms[0]) or the norm of
    each output row / input channel (LOP_ROW / LOP_COL); see impflow_prep_weights_lop."""
    W = W.contiguous()
    out, args = _prep_layouts(W, fwd_shape, fwd_planes, bwd_shape, bwd_planes)
    _cabi.check(_lib().impflow_prep_weights_lop(_cabi.ptr(W), _cabi.ptr(norms), group, float(coeff), kind, *args),
                'prep_weights_lop')
    return out


def _flat_dot(a, b):
    """<a, b> over all elements as a 1-element device tensor.  Large operands are viewed as 256 rows so
    that the row-dot kernel spreads over the SMs (one CTA per row), then the 256 partials are summed."""
    n = a.numel()
    if n >= 65536 and n % 256 == 0:
        return rowdot(a.view(256, -1), b.view(256, -1)).sum().view(1)
    return rowdot(a.view(1, -1), b.view(1, -1))


def sn_scale(W, D, coeff, scale_out=None):
    """(W / max(1, sigma/coeff), sigma) with sigma = <W, D> computed and consumed on the device."""
    W = W.contiguous()
    sigma = _flat_dot(W, D)
    out = torch.empty_like(W)
    _cabi.check(_lib().impflow_sn_scale(_cabi.ptr(W), _cabi.ptr(sigma), float(coeff), _cabi.ptr(out),
                                        _cabi.ptr(scale_out, 'scale', True), W.numel(), _cabi.stream()), 'sn_scale')
    return out, sigma


def sn_scale_grad(G, W, D, sigma, coeff):
    """Gradient of <G, W / max(1, sigma(W)/coeff)> w.r.t. W (sigma linear in W with gradient D)."""
    G = G.contiguous()
    W = W.contiguous()
    t = _flat_dot(G, W)
    out = torch.empty_like(W)
    _cabi.check(_lib().impflow_sn_scale_grad(_cabi.ptr(G), _cabi.ptr(D), _cabi.ptr(sigma), _cabi.ptr(t),
                                             float(coeff), _cabi.ptr(out), W.numel(), _cabi.stream()),
                'sn_scale_grad')
    return out


def sn_scale_grad_layout(Wbar, kind, cout, cin, W, D, sigma, coeff):
    """sn_scale_grad reading dL/dW_eff from the GEMM layout of the weight-gradient kernels (kind 0 / 1 / 2 as in
    prep_weights, rows may be longer than the payload) and returning the module's weight layout; two launches
    from one C call instead of flip / permute / contiguous / dot / scale."""
    assert Wbar.stride(-1) == 1 and W.is_contiguous() and D.is_contiguous()
    out = torch.empty_like(W)
    ws = torch.empty(1024, device=W.device, dtype=torch.float32)
    _cabi.check(_lib().impflow_sn_scale_grad_layout(_cabi.ptr(Wbar), Wbar.stride(0), _cabi.ptr(W), _cabi.ptr(D),
                                                    _cabi.ptr(sigma), float(coeff), kind, cout, cin, _cabi.ptr(out),
                                                    _cabi.ptr(ws), _cabi.stream()), 'sn_scale_grad_layout')
    return out


def lop_scale_grad_layout(Wbar, kind, cout, cin, W, norms, coeff, axis, norm_type, local):
    """dL/dW of a Lop layer from dL/dW_eff in the GEMM layout (kind 0 / 1 / 2 as in sn_scale_grad_layout), in the
    module's weight layout; norms as lop_norms returned them.  See impflow_lop_scale_grad_layout."""
    assert Wbar.stride(-1) == 1 and W.is_contiguous()
    out = torch.empty_like(W)
    ws = torch.empty(2 * (cout if axis == 0 else cin), device=W.device, dtype=torch.float32)
    _cabi.check(_lib().impflow_lop_scale_grad_layout(_cabi.ptr(Wbar), Wbar.stride(0), _cabi.ptr(W), _cabi.ptr(norms),
                                                     float(coeff), kind, cout, cin, axis, norm_type, int(bool(local)),
                                                     _cabi.ptr(out), _cabi.ptr(ws), _cabi.stream()),
                'lop_scale_grad_layout')
    return out


def _dense_layout(x):
    """0 = (B, C, ...) contiguous, 1 = channels-last dense (the memory order of the rows-space kernels), None = other."""
    if x.is_contiguous():
        return 0
    if x.dim() == 4 and x.permute(0, 2, 3, 1).is_contiguous():
        return 1
    return None


class _ActNorm(torch.autograd.Function):
    """y = (x + bias_c) exp(weight_c), logpx' = logpx - HW sum(weight): one launch forward, one C call backward
    (act_norm.py:39-62).  Keeps the input's memory order (NCHW or channels-last)."""

    @staticmethod
    def forward(ctx, x, bias, weight, logpx):
        cl = _dense_layout(x)
        if cl is None:
            x, cl = x.contiguous(), 0
        B, C = x.shape[0], x.shape[1]
        HW = x.numel() // (B * C)
        y = torch.empty_like(x)          # same strides
        out_lp = None
        if logpx is not None:
            logpx = logpx.contiguous()
            assert logpx.numel() == B and logpx.dtype == torch.float32, 'actnorm: logpx must hold one float per sample'
            out_lp = torch.empty_like(logpx)
        _cabi.check(_lib().impflow_actnorm_forward(_cabi.ptr(x), _cabi.ptr(bias), _cabi.ptr(weight), _cabi.ptr(y),
                                                   _cabi.ptr(logpx, 'logpx', True), _cabi.ptr(out_lp, 'logpx_out', True),
                                                   B, C, HW, cl, _cabi.stream()), 'actnorm_forward')
        ctx.save_for_backward(y, weight)
        ctx.dims = (B, C, HW, cl)
        if logpx is None:
            return y
        return y, out_lp

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy, g_lp=None):
        y, weight = ctx.saved_tensors
        B, C, HW, cl = ctx.dims
        if gy is None:
            gy = torch.zeros_like(y)
        elif gy.stride() != y.stride():
            gy = torch.empty_like(y).copy_(gy)
        g_lp = g_lp.contiguous() if g_lp is not None else None
        gx = torch.empty_like(y)
        gb, gw = torch.empty_like(weight), torch.empty_like(weight)
        lib = _lib()
        ws = torch.empty(int(lib.impflow_actnorm_workspace_floats(C)), device=y.device, dtype=torch.float32)
        _cabi.check(lib.impflow_actnorm_backward(_cabi.ptr(gy), _cabi.ptr(y), _cabi.ptr(weight),
                                                 _cabi.ptr(g_lp, 'g_logpx', True), _cabi.ptr(gx), _cabi.ptr(gb),
                                                 _cabi.ptr(gw), _cabi.ptr(ws), B, C, HW, cl, _cabi.stream()),
                    'actnorm_backward')
        return gx, gb, gw, g_lp


def actnorm(x, bias, weight, logpx=None):
    """Fused ActNorm forward (+ log-density update) with its hand-written backward."""
    return _ActNorm.apply(x, bias, weight, logpx)


# ------------------------------------------------------------------------------------------
# differentiable primitives (closed under differentiation)
# ------------------------------------------------------------------------------------------

class _ActMul(torch.autograd.Function):
    """out = g * f^(order)(x; beta).  d/dg = f^(order), d/dx = g f^(order+1), d/dbeta via reduction."""

    @staticmethod
    def forward(ctx, x, g, beta_sp, kind, order):
        ctx.kind, ctx.order = kind, order
        ctx.has_g = g is not None
        ctx.save_for_backward(x, g if g is not None else x.new_empty(0), beta_sp if beta_sp is not None else x.new_empty(0))
        return act_mul(x, g, kind, order, beta_sp)

    @staticmethod
    def backward(ctx, gout):
        x, g, beta_sp = ctx.saved_tensors
        g = g if ctx.has_g else None
        beta_sp = beta_sp if beta_sp.numel() else None
        kind, order = ctx.kind, ctx.order
        gx = gg = gbeta = None
        inner = gout if g is None else gout * g
        if ctx.needs_input_grad[0]:
            if kind == ACT_RELU and order >= 1:
                gx = torch.zeros_like(x)
            elif order + 1 > 3:
                raise RuntimeError('impflow_b200: activation derivatives above order 3 are not implemented')
            else:
                gx = _ActMul.apply(x, inner, beta_sp, kind, order + 1)
        if g is not None and ctx.needs_input_grad[1]:
            gg = _ActMul.apply(x, gout, beta_sp, kind, order)
        if beta_sp is not None and ctx.needs_input_grad[2] and not _ACT_ONLY['on']:
            if order > 2:
                raise RuntimeError('impflow_b200: beta gradient above order 2 is not implemented')
            gbeta = act_beta_grad(x, inner.detach(), order, beta_sp.detach()).view_as(beta_sp)
        return gx, gg, gbeta, None, None


def activation(x, kind, beta_sp=None):
    return _ActMul.apply(x, None, beta_sp, kind, 0)


class _Transpose(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a):
        return transpose2d(a)

    @staticmethod
    def backward(ctx, g):
        return _Transpose.apply(g)


class _ColSum(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a):
        ctx.M = a.shape[0]
        return colsum(a)

    @staticmethod
    def backward(ctx, g):
        return g.unsqueeze(0).expand(ctx.M, -1)


def gemm_strided(A, ta, Bm, tb, bias=None):
    """op(A) op(B) (+ bias) on the CUDA cores without transposed copies: op(X) = X^T if its flag is set.
    A is (M,K) or (K,M) when ta; Bm is (K,N) or (N,K) when tb."""
    A, Bm = A.contiguous(), Bm.contiguous()
    M, K = (A.shape[1], A.shape[0]) if ta else (A.shape[0], A.shape[1])
    N = Bm.shape[0] if tb else Bm.shape[1]
    assert (Bm.shape[1] if tb else Bm.shape[0]) == K, 'gemm_strided: inner dimensions differ'
    lda, ldb = A.shape[1], Bm.shape[1]
    out = torch.empty(M, N, device=A.device, dtype=torch.float32)
    sA = (1, lda) if ta else (lda, 1)
    sB = (ldb, 1) if tb else (1, ldb)
    _cabi.check(_lib().impflow_gemm_strided(_cabi.ptr(A), sA[0], sA[1], _cabi.ptr(Bm), sB[0], sB[1],
                                            _cabi.ptr(bias, 'bias', True), _cabi.ptr(out), N, M, N, K, _cabi.stream()),
                'gemm_strided')
    return out


class _MM(torch.autograd.Function):
    """C = op(A) op(B) with transpose flags; closed under differentiation (the derivative of a GEMM is a GEMM with
    other flags), so the small-shape autograd paths (toy / tabular / classifier, incl. the double backward of the
    log-det estimators) never materialise a transpose."""

    @staticmethod
    def forward(ctx, A, Bm, ta, tb):
        ctx.save_for_backward(A, Bm)
        ctx.ta, ctx.tb = ta, tb
        return gemm_strided(A, ta, Bm, tb)

    @staticmethod
    def backward(ctx, G):
        A, Bm = ctx.saved_tensors
        ta, tb = ctx.ta, ctx.tb
        gA = gB = None
        if ctx.needs_input_grad[0]:
            gA = _MM.apply(Bm, G, tb, True) if ta else _MM.apply(G, Bm, False, not tb)
        if ctx.needs_input_grad[1]:
            gB = _MM.apply(G, A, True, ta) if tb else _MM.apply(A, G, not ta, False)
        return gA, gB, None, None


class _GemmNT(torch.autograd.Function):
    """C = A B^T + bias;  dA = G B,  dB = G^T A,  dbias = colsum(G).  Large shapes run on the tcgen05 kernel
    (transposed copies + planes); small ones on the CUDA-core strided kernel via _MM."""

    @staticmethod
    def forward(ctx, A, Bm, bias):
        ctx.save_for_backward(A, Bm)
        ctx.has_bias = bias is not None
        M, K = A.shape
        N = Bm.shape[0]
        ctx.small = not _tc_ok(M, N, (K + 31) // 32 * 32, 4, 4) or (
            _BACKEND['mode'] == 'auto' and 2.0 * M * N * K < _BACKEND['min_flops_tc_autograd'])
        if ctx.small:
            return gemm_strided(A, False, Bm, True, bias)
        pre, _, _ = gemm_nt(A, Bm, bias)
        return pre

    @staticmethod
    def backward(ctx, G):
        A, Bm = ctx.saved_tensors
        gA = gB = gbias = None
        G = G.contiguous()
        if ctx.small:
            if ctx.needs_input_grad[0]:
                gA = _MM.apply(G, Bm, False, False)
            if ctx.needs_input_grad[1] and not _ACT_ONLY['on']:
                gB = _MM.apply(G, A, True, False)
        else:
            if ctx.needs_input_grad[0]:
                gA = _GemmNT.apply(G, _Transpose.apply(Bm), None)
            if ctx.needs_input_grad[1] and not _ACT_ONLY['on']:
                gB = _GemmNT.apply(_Transpose.apply(G), _Transpose.apply(A), None)
        if ctx.has_bias and ctx.needs_input_grad[2] and not _ACT_ONLY['on']:
            gbias = _ColSum.apply(G)
        return gA, gB, gbias


def linear(x2d, W, bias=None):
    return _GemmNT.apply(x2d, W, bias)


class _Im2col(torch.autograd.Function):
    """(B,H,W,C) -> (B*H*W, ld) patches, ld >= 9C zero padded; adjoint = _Col2im on the first 9C columns."""

    @staticmethod
    def forward(ctx, x_nhwc, ld):
        ctx.shape = tuple(x_nhwc.shape)
        ctx.ld = ld
        return im2col3x3(x_nhwc, ld)

    @staticmethod
    def backward(ctx, g):
        B, H, W, C = ctx.shape
        if ctx.ld != 9 * C:
            g = g[:, :9 * C]           # the zero-padded tail carries no gradient
        return _Col2im.apply(g, B, H, W, C), None


class _Col2im(torch.autograd.Function):
    @staticmethod
    def forward(ctx, col, B, H, W, C):
        ctx.C = C
        pre, _ = col2im3x3(col, B, H, W, C)
        return pre

    @staticmethod
    def backward(ctx, g):
        return _Im2col.apply(g, 9 * ctx.C), None, None, None, None


def conv3x3_nhwc(x_nhwc, W_oihw, bias=None):
    """3x3 / stride 1 / pad 1 cross-correlation on an NHWC tensor (F.conv2d semantics,
    mixed_lipschitz.py:391) as im2col+GEMM (narrow input) or GEMM+col2im (narrow output)."""
    B, H, Wd, Cin = x_nhwc.shape
    Cout = W_oihw.shape[0]
    if Cin <= Cout:
        K = 9 * Cin
        Kp = (K + 31) // 32 * 32 if _BACKEND['mode'] != 'simt' else K    # K % 32 == 0 -> tcgen05 kernel
        Wr = W_oihw.permute(0, 2, 3, 1).reshape(Cout, K)                 # (co, ky, kx, ci)
        if Kp != K:
            Wr = torch.nn.functional.pad(Wr, (0, Kp - K))
        y = _GemmNT.apply(_Im2col.apply(x_nhwc, Kp), Wr, bias)
        return y.view(B, H, Wd, Cout)
    W2 = W_oihw.flip(2, 3).permute(2, 3, 0, 1).reshape(9 * Cout, Cin)    # (ky, kx, co) <- flipped taps
    Y = _GemmNT.apply(x_nhwc.reshape(B * H * Wd, Cin), W2, None)
    y = _Col2im.apply(Y, B, H, Wd, Cout)
    if bias is not None:
        y = y + bias
    return y


def conv1x1_nhwc(x_nhwc, W_oihw, bias=None):
    B, H, Wd, Cin = x_nhwc.shape
    Cout = W_oihw.shape[0]
    y = _GemmNT.apply(x_nhwc.reshape(B * H * Wd, Cin), W_oihw.reshape(Cout, Cin), bias)
    return y.view(B, H, Wd, Cout)


class _RowDot(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, c):
        ctx.save_for_backward(a, c)
        return rowdot(a, c)

    @staticmethod
    def backward(ctx, g):
        a, c = ctx.saved_tensors
        shape = [-1] + [1] * (a.dim() - 1)
        gv = g.view(*shape)
        return (gv * c if ctx.needs_input_grad[0] else None), (gv * a if ctx.needs_input_grad[1] else None)


def rowdot_fn(a, c):
    return _RowDot.apply(a, c)
