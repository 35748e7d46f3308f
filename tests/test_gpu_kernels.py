"""GPU parity tests of the individual CUDA kernels, called through the C ABI (ctypes)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import impflow_oracle as orc
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops():
    import impflow_b200
    return impflow_b200.ops


def _dev():
    return torch.device('cuda:0')


@pytest.mark.parametrize('M,N,K', [(1, 1, 1), (7, 5, 3), (100, 128, 2), (1000, 128, 128), (257, 6, 128),
                                   (64, 43, 64), (300, 200, 77), (4096, 512, 512)])
def test_gemm_simt(ops, M, N, K):
    ops.set_gemm_backend('simt')
    g = torch.Generator().manual_seed(M * 7 + N)
    A = torch.randn(M, K, generator=g)
    B = torch.randn(N, K, generator=g)
    bias = torch.randn(N, generator=g)
    ref = (A.double() @ B.double().t() + bias.double())
    pre, act, _ = ops.gemm_nt(A.cuda(), B.cuda(), bias.cuda(), act_kind=ops.ACT_SIN, want_pre=True, want_act=True)
    assert rel_err(pre.cpu(), ref) < 2e-6          # fp32 accumulate
    assert rel_err(act.cpu(), orc.sin_act(pre.cpu())) < 2e-6   # epilogue activation of the kernel's own pre-activation
    ops.set_gemm_backend('auto')


@pytest.mark.parametrize('M,N,K', [(1000, 128, 6), (1000, 128, 128), (64, 43, 77), (5, 3, 2), (300, 200, 129)])
def test_gemm_strided_all_transposes(ops, M, N, K):
    """CUDA-core GEMM with element strides: op(A) op(B) for all four transpose combinations, and the autograd
    primitive built on it (first and second derivatives against torch.matmul)."""
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).cuda()
    B = torch.randn(K, N, generator=g).cuda()
    bias = torch.randn(N, generator=g).cuda()
    ref = A.double() @ B.double()
    for ta in (False, True):
        for tb in (False, True):
            Ax = A.t().contiguous() if ta else A
            Bx = B.t().contiguous() if tb else B
            out = ops.gemm_strided(Ax, ta, Bx, tb)
            assert rel_err(out.cpu(), ref.cpu()) < 2e-6, (ta, tb)
    out = ops.gemm_strided(A, False, B.t().contiguous(), True, bias)
    assert rel_err(out.cpu(), (ref + bias.double()).cpu()) < 2e-6
    # autograd: d/dA and d/dB of <C, R>, and a second derivative through them
    Ar, Br = A.clone().requires_grad_(True), B.t().contiguous().clone().requires_grad_(True)
    R = torch.randn(M, N, generator=g).cuda()
    C = ops.linear(Ar, Br, bias)
    gA, gB = torch.autograd.grad((C * R).sum(), [Ar, Br], create_graph=True)
    At, Bt = A.clone().double().requires_grad_(True), B.t().contiguous().clone().double().requires_grad_(True)
    Ct = At @ Bt.t() + bias.double()
    gAt, gBt = torch.autograd.grad((Ct * R.double()).sum(), [At, Bt], create_graph=True)
    assert rel_err(gA.detach().cpu(), gAt.detach().cpu()) < 2e-6 and rel_err(gB.detach().cpu(), gBt.detach().cpu()) < 2e-6
    (hA,) = torch.autograd.grad((gB * gB).sum(), Ar)
    (hAt,) = torch.autograd.grad((gBt * gBt).sum(), At)
    assert rel_err(hA.cpu(), hAt.cpu()) < 5e-6


@pytest.mark.parametrize('M,N,K', [(128, 128, 32), (256, 512, 512), (1000, 128, 128), (4096, 512, 512),
                                   (130, 27, 64), (777, 108, 512), (2048, 432, 96), (128, 16, 32), (65536, 512, 32)])
def test_gemm_tcgen05_3xtf32(ops, M, N, K):
    """tolerance: 3xTF32 keeps ~22 mantissa bits per operand -> 1e-5 rel stated by north_star."""
    ops.set_gemm_backend('tc')
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g)
    B = torch.randn(N, K, generator=g) / np.sqrt(K)
    bias = torch.randn(N, generator=g)
    ref = (A.double() @ B.double().t() + bias.double())
    pre, act, split = ops.gemm_nt(A.cuda(), B.cuda(), bias.cuda(), act_kind=ops.ACT_RELU, want_pre=True,
                                  want_act=True, want_split=True)
    torch.cuda.synchronize()
    assert rel_err(pre.cpu(), ref) < 3e-6
    assert rel_err(act.cpu(), torch.relu(ref)) < 3e-6
    hi, lo = split
    assert rel_err((hi + lo).cpu(), act.cpu()) < 1e-7
    # exact-fp32 CUDA-core kernel agrees as well
    ops.set_gemm_backend('simt')
    pre2, _, _ = ops.gemm_nt(A.cuda(), B.cuda(), bias.cuda())
    assert rel_err(pre.cpu(), pre2.cpu()) < 3e-6
    ops.set_gemm_backend('auto')


@pytest.mark.parametrize('M,N,K', [(27, 512, 65536), (512, 512, 16384), (512, 27, 4096), (130, 70, 8192)])
def test_gemm_tcgen05_split_k(ops, M, N, K):
    """Weight-gradient shapes: small M x N, long K -> split-K partials + fixed-order reduce."""
    import impflow_b200
    ops.set_gemm_backend('tc')
    g = torch.Generator().manual_seed(M + N)
    A = torch.randn(M, K, generator=g)
    B = torch.randn(N, K, generator=g) / np.sqrt(K)
    bias = torch.randn(N, generator=g)
    assert impflow_b200._cabi.load().impflow_gemm_tc_splits(M, N, K) > 1
    pre, _, _ = ops.gemm_nt(A.cuda(), B.cuda(), bias.cuda())
    pre_again, _, _ = ops.gemm_nt(A.cuda(), B.cuda(), bias.cuda())
    ref = A.double() @ B.double().t() + bias.double()
    assert rel_err(pre.cpu(), ref) < 1e-5         # fp32 accumulation over up to 65 536 terms
    assert torch.equal(pre, pre_again)            # deterministic reduce order
    ops.set_gemm_backend('auto')


@pytest.mark.parametrize('M,N,K', [(16384, 512, 512), (16384 + 77, 432, 128), (65536, 256, 64), (20000, 512, 96),
                                   (256 * 74 * 3 + 130, 300, 32)])
def test_gemm_tcgen05_cta_pair(ops, M, N, K):
    """CTA-pair tiles (tcgen05.mma.cta_group::2, 256x256 per cluster): every epilogue mode against fp64 and against
    the single-CTA kernel, incl. ragged M (second CTA of the last pair partly / fully out of range) and ragged N."""
    import impflow_b200
    lib = impflow_b200._cabi.load()
    ops.set_gemm_backend('tc')
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).cuda()
    B = (torch.randn(N, K, generator=g) / np.sqrt(K)).cuda()
    bias = torch.randn(N, generator=g).cuda()
    P = torch.randn(M, N, generator=g).cuda()
    beta = F.softplus(torch.tensor([0.9])).cuda()
    ref = (A.double() @ B.double().t()).cpu()
    bias_c = bias.double().cpu()

    def run():
        pre, act, split = ops.gemm_nt(A, B, bias, act_kind=ops.ACT_RELU, want_pre=True, want_act=True, want_split=True)
        dm, raw, dsplit = ops.gemm_nt(A, B, None, act_kind=ops.ACT_LIPSWISH, beta_sp=beta, dmul_pre=P, want_act=True,
                                      want_split=True)
        torch.cuda.synchronize()
        return [None if t is None else t.cpu() for t in (pre, act, split[0], split[1], dm, raw, dsplit[0], dsplit[1])]
    assert lib.impflow_gemm_tc_set_pair(1) == 1
    outs = run()
    lib.impflow_gemm_tc_set_pair(0)
    try:
        outs1 = run()
    finally:
        lib.impflow_gemm_tc_set_pair(1)
    pre, act, s_hi, s_lo, dm, raw = outs[:6]
    assert rel_err(pre, ref + bias_c) < 3e-6
    assert rel_err(act, torch.relu(ref + bias_c)) < 3e-6
    assert rel_err(s_hi + s_lo, act) < 1e-7
    assert rel_err(raw, ref) < 5e-6
    for a, b in zip(outs, outs1):
        if a is None:
            assert b is None
            continue
        assert rel_err(a, b) < 1e-6
    ops.set_gemm_backend('auto')


@pytest.mark.parametrize('kind,cout,cin,ld', [(0, 512, 512, 512), (0, 128, 6, 32), (1, 512, 3, 32), (1, 512, 12, 128),
                                              (2, 12, 512, 512), (2, 48, 512, 512)])
def test_sn_scale_grad_layout(ops, kind, cout, cin, ld):
    """GEMM-layout weight gradient -> module layout + spectral chain in one call == permute / flip / dot / scale."""
    g = torch.Generator().manual_seed(kind * 1000 + cout + cin)
    rows = 9 * cout if kind == 2 else cout
    Wbar = torch.randn(rows + (3 if kind == 2 else 0), ld, generator=g).cuda()[:rows]
    shape = (cout, cin) if kind == 0 else (cout, cin, 3, 3)
    W, D = torch.randn(*shape, generator=g).cuda(), torch.randn(*shape, generator=g).cuda()
    for sg in (0.5, 2.0):          # below and above the coeff: rescale inactive / active
        sigma = torch.tensor([sg]).cuda()
        if kind == 0:
            G = Wbar[:, :cin]
        elif kind == 1:
            G = Wbar[:, :9 * cin].reshape(cout, 3, 3, cin).permute(0, 3, 1, 2)
        else:
            G = Wbar[:, :cin].reshape(3, 3, cout, cin).flip(0, 1).permute(2, 3, 0, 1)
        Gc = G.reshape(shape).contiguous()
        old = ops.sn_scale_grad(Gc, W, D, sigma, 0.9)
        got = ops.sn_scale_grad_layout(Wbar, kind, cout, cin, W, D, sigma, 0.9)
        assert got.shape == W.shape
        # fp64 statement of the chain; the two kernels differ only in the summation order of <G, W>
        ratio = sg / 0.9
        sc, ds = (1.0 / ratio, -0.9 / (sg * sg)) if ratio > 1 else (1.0, 0.0)
        ref = sc * Gc.double() + ds * (Gc.double() * W.double()).sum() * D.double()
        assert rel_err(got.cpu(), ref.cpu()) < 1e-5
        assert rel_err(old.cpu(), ref.cpu()) < 1e-5


def test_colsum_large(ops):
    g = torch.Generator().manual_seed(9)
    a = torch.randn(65536, 512, generator=g)
    out = ops.colsum(a.cuda()).cpu()
    torch.testing.assert_close(out, a.double().sum(0).float(), rtol=1e-4, atol=1e-2)
    a = torch.randn(70, 5, generator=g)
    torch.testing.assert_close(ops.colsum(a.cuda()).cpu(), a.double().sum(0).float(), rtol=1e-5, atol=1e-5)


def test_gemm_tcgen05_dmul(ops):
    ops.set_gemm_backend('tc')
    g = torch.Generator().manual_seed(5)
    M, N, K = 512, 256, 128
    A, B, P = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / 11, torch.randn(M, N, generator=g)
    beta = torch.tensor([0.9])
    Pd = P.clone().requires_grad_(True)
    (d1,) = torch.autograd.grad(orc.lipswish(Pd, beta).sum(), Pd)
    ref = (A.double() @ B.double().t()) * d1.double()
    pre, _, _ = ops.gemm_nt(A.cuda(), B.cuda(), None, act_kind=ops.ACT_LIPSWISH,
                            beta_sp=F.softplus(beta).cuda(), dmul_pre=P.cuda())
    assert rel_err(pre.cpu(), ref) < 5e-6
    ops.set_gemm_backend('auto')


@pytest.mark.parametrize('M,C,N3,mode', [(128, 256, 27, 'fwd'), (300, 512, 27, 'fwd'), (1024, 512, 27, 'vjp'),
                                         (128 * 160, 512, 32, 'fwd'), (128 * 301, 512, 27, 'vjp'),
                                         (640, 256, 9, 'vjp')])
def test_branch3_fused_chain(ops, M, C, N3, mode):
    """Fused narrow->C->C->narrow tile kernel against the same chain in fp64 (forward with saved
    pre-activations, and the vjp form with act' multipliers), incl. ragged M and multi-item CTAs."""
    g = torch.Generator().manual_seed(M + C + N3)
    x0 = torch.zeros(M, 32)
    x0[:, :27] = torch.randn(M, 27, generator=g)
    W1 = torch.randn(C, 32, generator=g) / 27 ** 0.5
    W1[:, 27:] = 0
    W2 = torch.randn(C, C, generator=g) / C ** 0.5
    W3 = torch.randn(N3, C, generator=g) / C ** 0.5
    b1, b2 = torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    beta1, beta2 = torch.tensor([0.9]), torch.tensor([1.3])
    dev = _dev()
    sp = lambda t: ops.split_tf32(t.to(dev))
    if mode == 'fwd':
        y, p1, p2 = ops.branch3_tc(x0.to(dev), sp(W1), sp(W2), sp(W3), N3, bias1=b1.to(dev), bias2=b2.to(dev),
                                   act_kind=ops.ACT_LIPSWISH, beta1=beta1.to(dev), beta2=beta2.to(dev), save_pre=True)
        sw = lambda t, b: t * torch.sigmoid(t * b.double()) / 1.1
        r1 = x0.double() @ W1.double().t() + b1.double()
        r2 = sw(r1, beta1) @ W2.double().t() + b2.double()
        ry = sw(r2, beta2) @ W3.double().t()
        assert rel_err(p1.cpu(), r1) < 3e-6       # one 3xTF32 GEMM (same bound as test_gemm_tcgen05_3xtf32)
        assert rel_err(p2.cpu(), r2) < 6e-6       # two chained
    else:
        m1 = torch.randn(M, C, generator=g)
        m2 = torch.randn(M, C, generator=g)
        y, _, _ = ops.branch3_tc(x0.to(dev), sp(W1), sp(W2), sp(W3), N3, mul1=m1.to(dev), mul2=m2.to(dev))
        ry = (((x0.double() @ W1.double().t()) * m1.double()) @ W2.double().t() * m2.double()) @ W3.double().t()
    assert y.shape == (M, N3)
    assert rel_err(y.cpu(), ry) < 1e-5            # three chained: the north_star bound


@pytest.mark.parametrize('M,C,N3,mode', [(128, 128, 108, 'fwd'), (300, 512, 108, 'fwd'), (4096, 512, 432, 'fwd'),
                                         (4096, 512, 432, 'vjp'), (16384, 512, 108, 'vjp'), (128 * 41 + 5, 256, 200, 'fwd'),
                                         (640, 512, 27, 'vjp'), (128 * 149, 384, 130, 'fwd')])
def test_chain23_fused_layers(ops, M, C, N3, mode):
    """Fused layer 2 + 3 kernel of the wider scales (csrc/chain23_fused.cu) against the same chain in fp64:
    forward with bias + LipSwish and the saved pre-activation, and the vjp form with an act' multiplier; one and
    several 128-column passes, ragged M, several items per CTA, C/128 = 1..4 partial sums."""
    g = torch.Generator().manual_seed(M + C + N3)
    A = torch.randn(M, C, generator=g)
    W2 = torch.randn(C, C, generator=g) / C ** 0.5
    W3 = torch.randn(N3, C, generator=g) / C ** 0.5
    b2 = torch.randn(C, generator=g) * 0.1
    beta2 = torch.tensor([1.3])
    dev = _dev()
    sp = lambda t: ops.split_tf32(t.to(dev))
    if mode == 'fwd':
        parts, p2 = ops.chain23_tc(sp(A), sp(W2), sp(W3), N3, bias2=b2.to(dev), act_kind=ops.ACT_LIPSWISH,
                                   beta2=beta2.to(dev), save_pre=True)
        r2 = A.double() @ W2.double().t() + b2.double()
        ry = (r2 * torch.sigmoid(r2 * beta2.double()) / 1.1) @ W3.double().t()
        assert rel_err(p2.cpu(), r2) < 6e-6       # one 3xTF32 GEMM over K = C
    else:
        m2 = torch.randn(M, C, generator=g)
        parts, _ = ops.chain23_tc(sp(A), sp(W2), sp(W3), N3, mul2=m2.to(dev))
        ry = ((A.double() @ W2.double().t()) * m2.double()) @ W3.double().t()
    assert parts.shape == (C // 128, M, N3)
    assert rel_err(parts.sum(0).cpu(), ry) < 1e-5        # two chained: the north_star bound
    # each partial is the contribution of one 128-channel quarter
    if mode == 'vjp':
        q = C // 128 - 1
        h = ((A.double() @ W2.double().t()) * m2.double())[:, q * 128:(q + 1) * 128]
        assert rel_err(parts[q].cpu(), h @ W3.double()[:, q * 128:(q + 1) * 128].t()) < 1e-5


@pytest.mark.parametrize('M,C,N3,mode', [(300, 512, 108, 'fwd'), (4096, 512, 432, 'vjp'), (128 * 149 + 7, 384, 130, 'fwd')])
def test_chain23_single_plane_input(ops, M, C, N3, mode):
    """Layer-2 input as ONE fp32 plane (A_lo = NULL: the kernel derives the tf32 hi / lo planes in shared memory)
    gives bit-identical results to the route through hi / lo planes in HBM."""
    g = torch.Generator().manual_seed(M + C + N3 + 1)
    dev = _dev()
    A = torch.randn(M, C, generator=g).to(dev)
    W2 = ops.split_tf32((torch.randn(C, C, generator=g) / C ** 0.5).to(dev))
    W3 = ops.split_tf32((torch.randn(N3, C, generator=g) / C ** 0.5).to(dev))
    if mode == 'fwd':
        kw = dict(bias2=(torch.randn(C, generator=g) * 0.1).to(dev), act_kind=ops.ACT_LIPSWISH,
                  beta2=torch.tensor([1.3]).to(dev), save_pre=True)
    else:
        kw = dict(mul2=torch.randn(M, C, generator=g).to(dev))
    for rep in range(3):          # several launches: the split ring's phases line up across items
        pa, p2a = ops.chain23_tc(ops.split_tf32(A), W2, W3, N3, **kw)
        pb, p2b = ops.chain23_tc(A, W2, W3, N3, **kw)
        assert torch.equal(pa, pb)
        if p2a is not None:
            assert torch.equal(p2a, p2b)


def test_activation_orders_vs_golden(ops, golden):
    fx = golden('activations')
    x = torch.from_numpy(fx['x']).cuda()
    bsp = F.softplus(torch.tensor([0.5])).cuda()
    for name, kind, b in (('sin', ops.ACT_SIN, None), ('swish', ops.ACT_LIPSWISH, bsp)):
        for order, key in enumerate(['y', 'd1', 'd2', 'd3']):
            out = ops.act_mul(x, None, kind, order, b).cpu().numpy()
            np.testing.assert_allclose(out, fx[name + '_' + key], rtol=2e-5, atol=2e-5)
    # beta gradient of sum(w * swish(x))
    beta = torch.tensor([0.5], requires_grad=True, device='cuda')
    import impflow_b200
    y = impflow_b200.ops.activation(x, ops.ACT_LIPSWISH, F.softplus(beta))
    (gb,) = torch.autograd.grad((y * torch.from_numpy(fx['swish_w']).cuda()).sum(), beta)
    np.testing.assert_allclose(gb.cpu().numpy(), fx['swish_grad_beta'], rtol=1e-4)


def test_elementwise_helpers(ops):
    g = torch.Generator().manual_seed(3)
    for shape in [(5, 7), (64, 3072), (3, 1001)]:
        a, b, c = (torch.randn(*shape, generator=g) for _ in range(3))
        out = ops.lincomb3(a.cuda(), 1.0, b.cuda(), -1.0, c.cuda(), -0.5).cpu()
        torch.testing.assert_close(out, a - b - 0.5 * c, rtol=1e-6, atol=1e-6)
        d = ops.rowdot(a.cuda(), b.cuda()).cpu()
        torch.testing.assert_close(d, (a.double() * b.double()).sum(1).float(), rtol=1e-5, atol=1e-4)
        torch.testing.assert_close(ops.colsum(a.cuda()).cpu(), a.double().sum(0).float(), rtol=1e-5, atol=1e-4)
        torch.testing.assert_close(ops.transpose2d(a.cuda()).cpu(), a.t().contiguous())
        hi, lo = ops.split_tf32(a.cuda())
        torch.testing.assert_close((hi + lo).cpu(), a, rtol=0, atol=0)
        assert int((hi.cpu().view(torch.int32) & 0x1FFF).abs().max()) == 0     # tf32-representable


def test_im2col_col2im(ops):
    g = torch.Generator().manual_seed(4)
    B, H, W, C = 3, 6, 5, 4
    x = torch.randn(B, C, H, W, generator=g)
    col = ops.im2col3x3(x.permute(0, 2, 3, 1).contiguous().cuda()).cpu()
    ref = F.unfold(x, 3, padding=1).view(B, C, 9, H * W).permute(0, 3, 2, 1).reshape(B * H * W, 9 * C)
    torch.testing.assert_close(col, ref)
    # adjoint: <im2col(x), y> == <x, col2im(y)>
    y = torch.randn(B * H * W, 9 * C, generator=g)
    back, _ = ops.col2im3x3(y.cuda(), B, H, W, C)
    lhs = (col.double() * y.double()).sum()
    rhs = (x.permute(0, 2, 3, 1).double() * back.cpu().double()).sum()
    assert abs(lhs - rhs) / abs(lhs) < 1e-5


@pytest.mark.parametrize('M,N1,N2', [(4096, 512, 512), (65536, 512, 32), (16384, 28, 512), (2048, 128, 128),
                                     (1024, 512, 448), (8192, 108, 512), (640, 256, 64)])
def test_wgrad_mn_major(ops, M, N1, N2):
    """dW = G^T A straight from the row-major planes (MN-major tcgen05 operands, csrc/wgrad_tcgen05.cu) against
    fp64, the transposed-copy path, and with planes supplied by the caller."""
    g = torch.Generator().manual_seed(M + N1 + N2)
    G = torch.randn(M, N1, generator=g).cuda()
    A = torch.randn(M, N2, generator=g).cuda()
    ref = G.double().t() @ A.double()
    out = ops.wgrad_gemm(G, A)
    assert out.shape == (N1, N2)
    assert rel_err(out.cpu(), ref.cpu()) < 1e-5      # fp32 accumulation over up to 65536 terms per split
    out2 = ops.wgrad_gemm(None, None, G_split=ops.split_tf32(G), A_split=ops.split_tf32(A))
    assert torch.equal(out, out2)
    ops.WGRAD_MN_MAJOR['on'] = False
    try:
        old = ops.wgrad_gemm(G, A)
    finally:
        ops.WGRAD_MN_MAJOR['on'] = True
    assert rel_err(out.cpu(), old.cpu()) < 1e-5


@pytest.mark.parametrize('M,N1,N2', [(1000, 128, 128), (3000, 128, 6), (5000, 6, 128), (37, 5, 3), (6000, 63, 128),
                                     (1, 2, 2), (4001, 130, 70)])
def test_wgrad_simt_ragged_rows(ops, M, N1, N2):
    """dW = G^T A of the small / ragged shapes (MLP flows: rows = n x batch, not a multiple of 32): exact-fp32 CUDA-core
    kernel split along the rows (csrc/gemm_simt.cu k_wgrad_simt) against fp64; planes as inputs; strided views."""
    g = torch.Generator().manual_seed(M + N1 + N2)
    G = torch.randn(M, N1, generator=g).cuda()
    A = torch.randn(M, N2, generator=g).cuda()
    ref = G.double().t() @ A.double()
    out = ops.wgrad_gemm(G, A)
    assert out.shape == (N1, N2)
    assert rel_err(out.cpu(), ref.cpu()) < 2e-6
    out2 = ops.wgrad_gemm(G, A)
    assert torch.equal(out, out2)                     # fixed-order reduction: deterministic
    if N1 % 4 == 0 and N2 % 4 == 0:
        out3 = ops.wgrad_gemm(None, None, G_split=ops.split_tf32(G), A_split=ops.split_tf32(A))
        assert rel_err(out3.cpu(), ref.cpu()) < 2e-6


@pytest.mark.parametrize('M,N,with_ab', [(4096, 512, True), (1000, 256, True), (65536, 512, False), (77, 64, True)])
def test_neumann_act_bwd_fused(ops, M, N, with_ab):
    """One-pass activation step of the Neumann reverse sweep against the separate kernels / fp64."""
    g = torch.Generator().manual_seed(M + N)
    p, t, ta, ab = [torch.randn(M, N, generator=g).cuda() for _ in range(4)]
    beta = torch.tensor([0.83], device='cuda')
    planes, colsum, bg = ops.neumann_act_bwd(p, t, ta, ab if with_ab else None, beta)
    y_ref = ops.act_second(p, t, ta, ab if with_ab else None, ops.ACT_LIPSWISH, beta)
    y = planes[0] + planes[1]
    assert rel_err(y.cpu(), y_ref.cpu()) < 1e-6
    assert torch.equal(planes[0], ops.split_tf32(y)[0])
    assert rel_err(colsum.cpu(), y_ref.double().sum(0).cpu()) < 1e-5
    bg_ref = ops.act_beta_grad(p, ta, 1, beta, g2=t)
    if with_ab:
        bg_ref = bg_ref + ops.act_beta_grad(p, ab, 0, beta)
    assert abs(float(bg) - float(bg_ref)) < 1e-4 * max(1.0, abs(float(bg_ref)))


@pytest.mark.parametrize('M,N', [(64, 32), (65536, 27), (1000, 77), (4096, 512), (130, 513)])
def test_transpose_split(ops, M, N):
    a = torch.randn(M, N, generator=torch.Generator().manual_seed(M + N)).cuda()
    hi, lo = ops.transpose_split(a)
    assert hi.shape == (N, M)
    assert torch.equal(hi + lo, a.t())                               # exact: lo is the rounding residual
    assert torch.equal(hi, ops.split_tf32(a.t().contiguous())[0])    # same rounding as the plain split kernel


@pytest.mark.parametrize('B,H,W,C,ld', [(2, 8, 8, 3, 32), (3, 5, 7, 12, 128), (1, 4, 4, 48, 448), (2, 6, 6, 3, 27)])
def test_im2col_split_planes(ops, B, H, W, C, ld):
    x = torch.randn(B, H, W, C, generator=torch.Generator().manual_seed(C)).cuda()
    col = ops.im2col3x3(x, ld=ld)
    ref = F.unfold(x.permute(0, 3, 1, 2), 3, padding=1).view(B, C, 9, H * W).permute(0, 3, 2, 1).reshape(B * H * W, 9 * C)
    assert torch.equal(col[:, :9 * C], ref) and float(col[:, 9 * C:].abs().sum()) == 0.0
    hi, lo = ops.im2col3x3_split(x, ld=ld)
    assert torch.equal(hi + lo, col)
    assert torch.equal(hi, ops.split_tf32(col)[0])


def test_split_tf32_vectorised_and_tail(ops):
    for n in (4096, 4099, 3):
        a = torch.randn(n).cuda()
        hi, lo = ops.split_tf32(a)
        assert torch.equal(hi + lo, a)
        assert int((hi.view(torch.int32) & 0x1FFF).abs().sum()) == 0       # tf32: low 13 mantissa bits clear


@pytest.mark.parametrize('cin,cout', [(3, 16), (16, 3), (8, 8)])
def test_conv3x3_matches_conv2d(ops, cin, cout):
    g = torch.Generator().manual_seed(cin * 31 + cout)
    x = torch.randn(2, cin, 8, 8, generator=g)
    w = torch.randn(cout, cin, 3, 3, generator=g) / 5
    b = torch.randn(cout, generator=g)
    ref = F.conv2d(x.double(), w.double(), b.double(), 1, 1)
    y = ops.conv3x3_nhwc(x.permute(0, 2, 3, 1).contiguous().cuda(), w.cuda(), b.cuda()).permute(0, 3, 1, 2)
    assert rel_err(y.cpu(), ref) < 3e-6
    # gradients through the kernel primitives
    xg = x.clone().cuda().requires_grad_(True)
    wg = w.clone().cuda().requires_grad_(True)
    y = ops.conv3x3_nhwc(xg.permute(0, 2, 3, 1).contiguous(), wg, b.cuda()).permute(0, 3, 1, 2)
    t = torch.randn(ref.shape, generator=g)
    gx, gw = torch.autograd.grad((y * t.cuda()).sum(), (xg, wg))
    xr, wr = x.clone().double().requires_grad_(True), w.clone().double().requires_grad_(True)
    gxr, gwr = torch.autograd.grad((F.conv2d(xr, wr, b.double(), 1, 1) * t.double()).sum(), (xr, wr))
    assert rel_err(gx.cpu(), gxr) < 5e-6
    assert rel_err(gw.cpu(), gwr) < 5e-6


def test_sn_power_iter_vs_golden(ops, golden):
    fx = golden('induced_norm')
    W = torch.from_numpy(fx['lin_weight2']).cuda()
    u, v = torch.from_numpy(fx['lin_init_u']).cuda(), torch.from_numpy(fx['lin_init_v']).cuda()
    sigma, iters = ops.sn_power_iter(W, u, v, None, 1e-3, 1e-3)
    np.testing.assert_allclose(u.cpu().numpy(), fx['lin_u_tol'], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(v.cpu().numpy(), fx['lin_v_tol'], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(sigma.cpu().numpy()[0], fx['lin_scale_tol'], rtol=1e-5)
    sigma, iters = ops.sn_power_iter(W, u, v, 5, 0.0, 0.0)
    assert int(iters.item()) == 5
    np.testing.assert_allclose(u.cpu().numpy(), fx['lin_u_it5'], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(sigma.cpu().numpy()[0], fx['lin_scale_it5'], rtol=1e-5)
    # iteration count of the tolerance rule equals the oracle's
    W0 = torch.from_numpy(fx['lin_weight2'])
    _, _, used = orc.power_iterate_matrix(W0, torch.from_numpy(fx['lin_init_u']), torch.from_numpy(fx['lin_init_v']),
                                          None, 1e-3, 1e-3)
    u, v = torch.from_numpy(fx['lin_init_u']).cuda(), torch.from_numpy(fx['lin_init_v']).cuda()
    _, iters = ops.sn_power_iter(W, u, v, None, 1e-3, 1e-3)
    assert int(iters.item()) == used


@pytest.mark.parametrize('kind,cout,cin', [(0, 512, 512), (0, 6, 128), (1, 512, 3), (1, 32, 4), (2, 3, 512), (2, 12, 512),
                                           (2, 4, 32)])
def test_prep_weights_layouts(ops, kind, cout, cin):
    """One-launch weight preparation (rescale + GEMM layouts of both directions + hi/lo planes) against the
    permute / flip / pad expressions it replaces."""
    g = torch.Generator().manual_seed(kind * 100 + cout + cin)
    shape = (cout, cin) + ((1, 1) if kind == 0 else (3, 3))
    W = torch.randn(*shape, generator=g).cuda()
    sigma = torch.tensor([1.7], device='cuda')
    coeff = 0.9
    Ws = W / max(1.0, 1.7 / coeff)
    if kind == 0:
        f, b = Ws.reshape(cout, cin), Ws.reshape(cout, cin).t()
    elif kind == 1:
        f, b = Ws.permute(0, 2, 3, 1).reshape(cout, 9 * cin), Ws.permute(2, 3, 1, 0).reshape(9 * cin, cout)
    else:
        f = Ws.flip(2, 3).permute(2, 3, 0, 1).reshape(9 * cout, cin)
        b = Ws.flip(2, 3).permute(1, 2, 3, 0).reshape(cin, 9 * cout)
    pad = lambda k: (k + 31) // 32 * 32
    for planes in (True, False):
        fs = (f.shape[0], pad(f.shape[1]) if planes else f.shape[1])
        bs = (b.shape[0], pad(b.shape[1]) if planes else b.shape[1])
        of, ofs, ob, obs = ops.prep_weights(W, sigma, coeff, kind, fs, planes, bs, planes)
        for ref, out, sp in ((f, of, ofs), (b, ob, obs)):
            assert torch.allclose(out[:, :ref.shape[1]], ref, rtol=1e-6, atol=0)
            assert float(out[:, ref.shape[1]:].abs().sum()) == 0.0
            assert (sp is not None) == planes
            if planes:
                assert torch.equal(sp[0] + sp[1], out) and torch.equal(sp[0], ops.split_tf32(out)[0])


@pytest.mark.parametrize('co,ci,h,w,n_it', [(512, 3, 32, 32, None), (3, 512, 32, 32, None), (512, 12, 16, 16, 3),
                                            (48, 512, 8, 8, None), (32, 4, 8, 8, 5), (5, 40, 6, 7, None),
                                            (16, 16, 8, 8, None), (512, 3, 32, 32, 0)])
def test_sn_power_iter_conv_vs_oracle(ops, co, ci, h, w, n_it):
    """One-launch cooperative conv power iteration against the oracle's loop (mixed_lipschitz.py:328-386):
    both layer orientations (wide output / wide input), tolerance and fixed-count modes, odd image shapes."""
    g = torch.Generator().manual_seed(co * 7 + ci)
    W = torch.randn(co, ci, 3, 3, generator=g) / (3.0 * ci ** 0.5)
    u0 = F.normalize(torch.randn(co * h * w, generator=g), dim=0)
    v0 = F.normalize(torch.randn(ci * h * w, generator=g), dim=0)
    tol = 1e-3 if n_it is None else None
    if n_it == 0:
        u_ref, v_ref, used = u0, v0, 0
    else:
        u_ref, v_ref, used = orc.power_iterate_conv(W, u0.clone(), v0.clone(), (ci, h, w), 1, 1, n_it, tol, tol)
    s_ref = orc.sigma_conv(W, u_ref, v_ref, (ci, h, w), 1, 1)
    u, v = u0.clone().cuda(), v0.clone().cuda()
    res = ops.sn_power_iter_conv(W.cuda(), u, v, h, w, n_it, tol, tol, want_D=True)
    assert res is not None
    sigma, iters, D = res
    Wg = W.clone().requires_grad_(True)       # d <u, conv(v; W)> / dW at the final (u, v)
    (D_ref,) = torch.autograd.grad(torch.dot(u.cpu(), F.conv2d(v.cpu().view(1, ci, h, w), Wg, padding=1).reshape(-1)),
                                   Wg)
    assert rel_err(D.cpu(), D_ref) < 1e-5
    assert int(iters.item()) == used
    assert rel_err(u.cpu(), u_ref) < 1e-5
    assert rel_err(v.cpu(), v_ref) < 1e-5
    assert abs(float(sigma.item()) - float(s_ref)) < 1e-5 * max(1.0, abs(float(s_ref)))


def test_sn_power_iter_conv_unsupported_shape(ops):
    assert ops.sn_power_iter_conv(torch.randn(64, 64, 3, 3).cuda(), torch.randn(64 * 1024).cuda(),
                                  torch.randn(64 * 1024).cuda(), 32, 32, None, 1e-3, 1e-3) is None


@pytest.mark.parametrize('tag', ['small', 'wide', 'capped', 'long', 'protbreak'])
def test_broyden_vs_golden(golden, tag):
    import impflow_b200
    fx = golden('broyden_analytic')
    B, d, T, eps, scale, gain = fx[tag + '_meta']
    W, c = torch.from_numpy(fx[tag + '_W']).cuda(), torch.from_numpy(fx[tag + '_c']).cuda()
    if gain < 0:
        g = lambda x: c - float(scale) * torch.tanh(x @ W) - x
    else:
        g = lambda x: c + float(gain) * x
    res = impflow_b200.layers.broyden.broyden(g, torch.zeros(int(B), int(d), device='cuda'), int(T), float(eps))
    nstep, lowest_step, prot = fx[tag + '_ints']
    trace_ref = fx[tag + '_trace']
    assert int(res['prot_break']) == prot
    if tag == 'long':
        # 30 non-converging steps of a chaotic map: fp32 round-off decorrelates the late iterates;
        # the iteration COUNT is still exact and the early trace agrees.
        assert res['nstep'] == nstep
        np.testing.assert_allclose(res['trace'][:6], trace_ref[:6], rtol=1e-3)
        return
    assert res['nstep'] == nstep
    assert res['lowest_step'] == lowest_step
    np.testing.assert_allclose(res['trace'][:3], trace_ref[:3], rtol=1e-5)
    assert rel_err(res['result'].cpu(), fx[tag + '_result']) < 1e-5
    np.testing.assert_allclose(res['diff'], fx[tag + '_diff'], rtol=0.5, atol=1e-6)
    assert res['diff_detail'].shape == (int(B),)


@pytest.mark.parametrize('B,d', [(3, 2), (5, 130), (4, 3072), (2, 16384), (2, 65536), (3, 1026), (3, 1028), (2, 5000),
                                 (1, 40004)])
def test_broyden_shapes_against_oracle(B, d):
    """Same seeded contraction solved by the CUDA solver and by the CPU oracle at several sizes
    (warp-per-sample, single-CTA, multi-CTA cluster and non-float4 paths; ragged last slices of a cluster)."""
    import impflow_b200
    g = torch.Generator().manual_seed(d)
    c = torch.randn(B, d, generator=g)
    a = torch.rand(d, generator=g) * 0.8 + 0.1
    shift = 7 if d > 7 else 1
    f_cpu = lambda x: c - 0.6 * torch.sin(x * a + torch.roll(x, shift, 1)) - x
    cg, ag = c.cuda(), a.cuda()
    f_gpu = lambda x: cg - 0.6 * torch.sin(x * ag + torch.roll(x, shift, 1)) - x
    ref = orc.broyden_solve(f_cpu, torch.zeros(B, d), 30, 1e-6)
    res = impflow_b200.layers.broyden.broyden(f_gpu, torch.zeros(B, d, device='cuda'), 30, 1e-6)
    assert res['nstep'] == ref['nstep'], (res['trace'], ref['trace'])
    assert res['lowest_step'] == ref['lowest_step']
    assert rel_err(res['result'].cpu(), ref['result']) < 1e-5
    np.testing.assert_allclose(res['trace'][:-1], ref['trace'][:-1], rtol=2e-3)


@pytest.mark.parametrize('B,d,hidden,nh,act', [(5000, 2, 128, 2, 'sin'), (1000, 6, 128, 4, 'sin'), (1000, 63, 128, 4, 'sin'),
                                              (37, 43, 64, 2, 'swish'), (1, 5, 16, 1, 'relu')])
def test_persistent_mlp_solver(B, d, hidden, nh, act):
    """One-launch persistent solver (csrc/mlp_solver.cu) == host-driven kernel loop == CPU oracle."""
    import impflow_b200
    from impflow_b200.branch_program import compile_branch
    from impflow_b200.layers import broyden as bmod
    L = impflow_b200.layers
    torch.manual_seed(B + d)
    acts = {'sin': L.base.Sin, 'swish': L.base.Swish, 'relu': L.base.ReLU}
    dims = [d] + [hidden] * nh + [d]
    mods = []
    for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
        if i > 0:
            mods.append(acts[act]())
        mods.append(L.base.get_linear(a, b, coeff=0.9, n_iterations=None, atol=1e-3, rtol=1e-3, domain=2, codomain=2))
    net = torch.nn.Sequential(*mods)
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() > 1:
                p.mul_(4.0)
    net = net.cuda()
    prog = compile_branch(net)
    x_embed = torch.randn(B, d, device='cuda')
    z0 = torch.zeros(B, d, device='cuda')
    with torch.no_grad():
        spec = prog.mlp_solver_spec(z0)
        assert spec is not None
        res_p = bmod.broyden_mlp(spec, x_embed, z0, 30, 1e-6)
        low_p = res_p['result'].clone()
        g = lambda z: impflow_b200.ops.lincomb3(x_embed, 1.0, prog.forward(z), -1.0, z, -1.0)
        res_h = bmod.broyden(g, z0, 30, 1e-6)
        # CPU oracle on the same effective weights
        ws = prog._prep(B)
        Ws = [w.fwd[:, :w.cin].cpu() for w in ws]
        bs = [w.bias.cpu() for w in ws]
        beta = torch.nn.functional.softplus(torch.tensor([0.5]))

        def f_cpu(z):
            h = z
            for i, (W, b) in enumerate(zip(Ws, bs)):
                h = h @ W.t() + b
                if i + 1 < len(Ws):
                    h = orc.sin_act(h) if act == 'sin' else (orc.lipswish(h, torch.tensor([0.5])) if act == 'swish'
                                                             else torch.relu(h))
            return h
        xe = x_embed.cpu()
        ref = orc.broyden_solve(lambda z: xe - f_cpu(z) - z, torch.zeros(B, d), 30, 1e-6)
    assert res_p['nstep'] == res_h['nstep'] == ref['nstep'], (res_p['trace'], res_h['trace'], ref['trace'])
    assert res_p['lowest_step'] == ref['lowest_step']
    assert rel_err(low_p.cpu(), ref['result']) < 1e-5
    assert rel_err(low_p.cpu(), res_h['result'].cpu()) < 1e-5
    tp, tr = np.array(res_p['trace']), np.array(ref['trace'])
    big = tr > 1e-3 * tr[0]                  # below that the residual is fp32 round-off of the branch
    np.testing.assert_allclose(tp[big], tr[big], rtol=5e-3)
    assert res_p['diff_detail'].shape == (B,)
