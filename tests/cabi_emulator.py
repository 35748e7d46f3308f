"""TEST INFRASTRUCTURE ONLY — a numpy emulation of the C ABI in include/impflow_b200.h.

The CPU test-suite (`-m "not gpu"`) uses it to exercise the *host* logic of the product package
(autograd wiring of the kernel primitives, weight re-layouts for the conv-as-GEMM paths, the
Broyden host loop, RNG / coefficient handling, state-dict compatibility) without a GPU.  It
restates what each kernel computes, with the same formulas as the .cu sources, on host memory
addressed by the raw pointers the product passes.  It is never importable from the product and
nothing here is timed or shipped; the GPU tests (`-m gpu`) run the real kernels.
"""
import ctypes
import math

import numpy as np
import torch

ACT_NONE, ACT_SIN, ACT_LIPSWISH, ACT_RELU, ACT_MULTIPLIER = 0, 1, 2, 3, 4


def _addr(p):
    if p is None:
        return None
    if isinstance(p, ctypes.c_void_p):
        return p.value
    return int(p)


def _f32(p, n):
    a = _addr(p)
    if a is None:
        return None
    return np.ctypeslib.as_array((ctypes.c_float * int(n)).from_address(a))


def _act(kind, x, order, beta):
    x = x.astype(np.float32)
    if kind == ACT_NONE:
        return x if order == 0 else (np.ones_like(x) if order == 1 else np.zeros_like(x))
    if kind == ACT_SIN:
        two_pi = np.float32(2 * math.pi)
        s, c = np.sin(two_pi * x), np.cos(two_pi * x)
        return [s / np.float32(math.pi) * np.float32(0.5), c, -two_pi * s, -two_pi * two_pi * c][order]
    if kind == ACT_MULTIPLIER:
        assert order == 1
        return x
    if kind == ACT_RELU:
        return [np.maximum(x, 0), (x > 0).astype(np.float32), np.zeros_like(x), np.zeros_like(x)][order]
    bx = beta * x
    s = 1 / (1 + np.exp(-bx))
    q = s * (1 - s)
    inv = np.float32(1 / 1.1)
    if order == 0:
        return x * s * inv
    if order == 1:
        return (s + bx * q) * inv
    if order == 2:
        return (2 * beta * q + beta * bx * q * (1 - 2 * s)) * inv
    return (3 * beta * beta * q * (1 - 2 * s) + beta * beta * bx * q * (1 - 6 * s + 6 * s * s)) * inv


def _dbeta(x, order, beta):
    bx = beta * x
    s = 1 / (1 + np.exp(-bx))
    q = s * (1 - s)
    r1, r2 = 1 - 2 * s, 1 - 6 * s + 6 * s * s
    inv = 1 / 1.1
    if order == 0:
        return x * x * q * inv
    if order == 1:
        return (2 * x * q + bx * x * q * r1) * inv
    return (2 * q + 4 * bx * q * r1 + bx * bx * q * r2) * inv


def _beta(p):
    return None if _addr(p) is None else np.float32(_f32(p, 1)[0])


def _epilogue(acc, bias, pre_out, act_out, dmul_pre, act_kind, beta, split_hi=None, split_lo=None):
    """acc: (M,N) float32; outputs are flat views written in place."""
    if dmul_pre is not None:
        nxt = (acc * _act(act_kind, dmul_pre.reshape(acc.shape), 1, beta)).astype(np.float32)
        if pre_out is not None:
            pre_out[:] = nxt.ravel()
        if act_out is not None:
            act_out[:] = acc.astype(np.float32).ravel()
    else:
        v = acc + (bias[None, :] if bias is not None else 0)
        v = v.astype(np.float32)
        if pre_out is not None:
            pre_out[:] = v.ravel()
        nxt = _act(act_kind, v, 0, beta).astype(np.float32)
        if act_out is not None:
            act_out[:] = nxt.ravel()
    if split_hi is not None:
        hi = _tf32(nxt)
        split_hi[:] = hi.ravel()
        split_lo[:] = (nxt - hi).ravel()


def _tf32(a):
    b = a.astype(np.float32).view(np.uint32).astype(np.uint64)
    b = (b + 0x1000) & 0xFFFFE000          # round to nearest (ties away), keep 10 mantissa bits
    return b.astype(np.uint32).view(np.float32)


STATE_DTYPE = np.dtype([('nstep', '<i4'), ('lowest_step', '<i4'), ('active', '<i4'), ('prot_break', '<i4'),
                        ('converged', '<i4'), ('stagnated', '<i4'), ('do_update', '<i4'), ('new_lowest', '<i4'),
                        ('threshold', '<i4'), ('counter', '<i4'), ('eps', '<f8'), ('init_objective', '<f8'),
                        ('lowest', '<f8'), ('objective', '<f8'), ('trace', '<f8', (64,))])


def _state(p):
    buf = (ctypes.c_uint8 * STATE_DTYPE.itemsize).from_address(_addr(p))
    return np.ctypeslib.as_array(buf).view(STATE_DTYPE)


class EmulatedLib(object):
    """Attribute-compatible stand-in for the ctypes CDLL of libimpflow_b200.so."""

    def __init__(self):
        self.launches = 0
        self._err = b''

    # ---- misc ----
    def impflow_version(self):
        return 1

    def impflow_last_error(self):
        return self._err

    def impflow_launch_count(self):
        return self.launches

    def impflow_broyden_state_bytes(self):
        return STATE_DTYPE.itemsize

    def impflow_broyden_workspace_floats(self, B, d, T):
        return B * 64

    def impflow_reduce_workspace_floats(self, n):
        return 148 * 16

    # ---- broyden (csrc/broyden.cu) ----
    def _decide(self, st, total, init):
        s = st[0]
        obj = float(np.float32(np.sqrt(total)))
        s['objective'] = obj
        if init:
            s['nstep'] = 0
            s['lowest_step'] = 0
            s['init_objective'] = obj
            s['lowest'] = obj
            s['trace'][0] = obj
            for k in ('prot_break', 'converged', 'stagnated', 'do_update', 'new_lowest'):
                s[k] = 0
            s['active'] = int(obj >= s['eps'] and 0 < s['threshold'])
            return
        T = int(s['threshold'])
        nstep = int(s['nstep']) + 1
        s['nstep'] = nstep
        s['trace'][nstep] = obj
        new_low = 0
        if obj < s['lowest']:
            s['lowest'] = obj
            s['lowest_step'] = nstep
            new_low = 1
        s['new_lowest'] = new_low
        conv = int(obj < s['eps'])
        stag = 0
        if not conv and obj < 3 * s['eps'] and nstep == T:
            tr = s['trace'][nstep - T + 1:nstep + 1]
            stag = int(np.max(tr) / np.min(tr) < 1.3)
        prot = int((not conv) and (not stag) and obj > s['init_objective'] * 1e6)
        s['converged'], s['stagnated'], s['prot_break'] = conv, stag, prot
        upd = 0 if (conv or stag or prot) else 1
        s['do_update'] = upd
        s['active'] = int(bool(upd) and obj >= s['eps'] and nstep < T)

    def impflow_broyden_begin(self, x0, g0, xn, low_x, low_g, sample_sq, low_sq, partial, state, B, d, T, eps, stream):
        n = B * d
        x0, g0, xn, low_x, low_g = (_f32(p, n) for p in (x0, g0, xn, low_x, low_g))
        ssq, lsq = _f32(sample_sq, B), _f32(low_sq, B)
        st = _state(state)
        st[0]['threshold'] = T
        st[0]['eps'] = eps
        st[0]['counter'] = 0
        low_x[:] = x0
        low_g[:] = g0
        xn[:] = x0 + (-g0)
        ssq[:] = (g0.reshape(B, d) ** 2).sum(1)
        lsq[:] = ssq
        self._decide(st, float(ssq.astype(np.float64).sum()), True)
        self.launches += 2
        return 0

    def impflow_broyden_step(self, x_old, g_old, xn, gn, Ut, Vt, low_x, low_g, sample_sq, low_sq, partial, state,
                             B, d, T, stream):
        n = B * d
        x_old, g_old, xn, gn, low_x, low_g = (_f32(p, n) for p in (x_old, g_old, xn, gn, low_x, low_g))
        U, V = _f32(Ut, B * T * d).reshape(B, T, d), _f32(Vt, B * T * d).reshape(B, T, d)
        ssq, lsq = _f32(sample_sq, B), _f32(low_sq, B)
        st = _state(state)
        with np.errstate(all='ignore'):
            ssq[:] = (gn.reshape(B, d) ** 2).sum(1)
            self._decide(st, float(ssq.astype(np.float64).sum()), False)
            s = st[0]
            if s['new_lowest']:
                lsq[:] = ssq
                low_x[:] = xn
                low_g[:] = gn
            self.launches += 2
            if not s['do_update']:
                return 0
            k = int(s['nstep']) - 1
            X, G = xn.reshape(B, d), gn.reshape(B, d)
            dx, dg = X - x_old.reshape(B, d), G - g_old.reshape(B, d)
            Uk, Vk = U[:, :k], V[:, :k]
            a = np.einsum('bi,bji->bj', dx, Uk)
            bb = np.einsum('bji,bi->bj', Vk, dg)
            c = np.einsum('bji,bi->bj', Vk, G)
            vT = -dx + np.einsum('bj,bji->bi', a, Vk)
            w = -dg + np.einsum('bj,bji->bi', bb, Uk)
            S = np.einsum('bj,bji->bi', c, Uk)
            den = (vT * dg).sum(1, keepdims=True)
            vs = np.where(np.isnan(vT), 0, vT).astype(np.float32)
            ck = (vs * G).sum(1, keepdims=True)
            u = (dx - w) / den
            u = np.where(np.isnan(u), 0, u).astype(np.float32)
            V[:, k] = vs
            U[:, k] = u
            upd = -((-G) + (S + u * ck))
            x_old.reshape(B, d)[:] = X + upd
        return 0

    # ---- persistent MLP solver (csrc/mlp_solver.cu) ----
    def impflow_mlp_solver_limits(self, a, b, c):
        return 0

    def impflow_mlp_solver_partial_doubles(self):
        return 2 * 148 * 8

    def impflow_mlp_broyden_solve(self, x_embed, Wt, bias, dims, L, act_kind, beta_sp, za, ga, zb, gb, low_z, low_g,
                                  Ut, Vt, sample_sq, low_sq, partial, state, B, T, eps, stream):
        dims = [int(v) for v in dims]
        d = dims[0]
        betas = [(_beta(beta_sp[l]) if (beta_sp and l + 1 < L and beta_sp[l]) else None) for l in range(L)]
        Ws = [_f32(Wt[l], dims[l] * dims[l + 1]).reshape(dims[l], dims[l + 1]) for l in range(L)]
        bs = [(_f32(bias[l], dims[l + 1]) if bias[l] else None) for l in range(L)]
        xe = _f32(x_embed, B * d).reshape(B, d)

        def f(z):
            h = z
            for l in range(L):
                h = (h @ Ws[l]).astype(np.float32)
                if bs[l] is not None:
                    h = h + bs[l]
                if l + 1 < L:
                    h = _act(act_kind, h, 0, betas[l]).astype(np.float32)
            return h

        bufs = {'x': za, 'g': ga, 'xn': zb, 'gn': gb}
        x0 = _f32(za, B * d).reshape(B, d)
        _f32(ga, B * d)[:] = (xe - f(x0) - x0).ravel()
        self.impflow_broyden_begin(za, ga, zb, low_z, low_g, sample_sq, low_sq, None, state, B, d, T, eps, None)
        st = _state(state)
        while st[0]['active']:
            xn = _f32(bufs['xn'], B * d).reshape(B, d)
            _f32(bufs['gn'], B * d)[:] = (xe - f(xn) - xn).ravel()
            self.impflow_broyden_step(bufs['x'], bufs['g'], bufs['xn'], bufs['gn'], Ut, Vt, low_z, low_g, sample_sq,
                                      low_sq, None, state, B, d, T, None)
            bufs['x'], bufs['xn'] = bufs['xn'], bufs['x']
            bufs['g'], bufs['gn'] = bufs['gn'], bufs['g']
        self.launches += 1
        return 0

    def impflow_mlp_broyden_solve_vjp(self, rhs, W, ldw, dmul, dims, L, za, ga, zb, gb, low_z, low_g, Ut, Vt,
                                      sample_sq, low_sq, partial, state, B, T, eps, stream):
        dims = [int(v) for v in dims]
        d = dims[0]
        Ws = []
        for l in range(L):
            ld = int(ldw[l])
            Ws.append(_f32(W[l], (dims[l + 1] - 1) * ld + dims[l]).copy() if ld == dims[l] else None)
            full = np.lib.stride_tricks.as_strided(_f32(W[l], (dims[l + 1] - 1) * ld + dims[l]),
                                                   shape=(dims[l + 1], dims[l]), strides=(4 * ld, 4))
            Ws[-1] = np.array(full)
        Ds = [(_f32(dmul[l], B * dims[l]).reshape(B, dims[l]) if dmul[l] else None) for l in range(L)]
        r = _f32(rhs, B * d).reshape(B, d)

        def f(v):
            h = v
            for l in range(L - 1, -1, -1):
                h = (h @ Ws[l]).astype(np.float32)
                if Ds[l] is not None:
                    h = h * Ds[l]
            return h

        bufs = {'x': za, 'g': ga, 'xn': zb, 'gn': gb}
        x0 = _f32(za, B * d).reshape(B, d)
        _f32(ga, B * d)[:] = (f(x0) + x0 - r).ravel()
        self.impflow_broyden_begin(za, ga, zb, low_z, low_g, sample_sq, low_sq, None, state, B, d, T, eps, None)
        st = _state(state)
        while st[0]['active']:
            xn = _f32(bufs['xn'], B * d).reshape(B, d)
            _f32(bufs['gn'], B * d)[:] = (f(xn) + xn - r).ravel()
            self.impflow_broyden_step(bufs['x'], bufs['g'], bufs['xn'], bufs['gn'], Ut, Vt, low_z, low_g, sample_sq,
                                      low_sq, None, state, B, d, T, None)
            bufs['x'], bufs['xn'] = bufs['xn'], bufs['x']
            bufs['g'], bufs['gn'] = bufs['gn'], bufs['g']
        self.launches += 1
        return 0

    def impflow_mlp_series(self, v, W, ldw, Wt, dmul, dims, L, B, n, coeffs, Ls, Rs, Wm, S, stream):
        dims = [int(t) for t in dims]
        d = dims[0]
        Ws = []
        for l in range(L):
            ld = int(ldw[l])
            full = np.lib.stride_tricks.as_strided(_f32(W[l], (dims[l + 1] - 1) * ld + dims[l]),
                                                   shape=(dims[l + 1], dims[l]), strides=(4 * ld, 4))
            Ws.append(np.array(full))
        Ds = [(_f32(dmul[l], B * dims[l]).reshape(B, dims[l]) if dmul[l] else None) for l in range(L)]
        c = [float(coeffs[k]) for k in range(n)]
        v0 = _f32(v, B * d).reshape(B, d)

        def vjp(h):
            for l in range(L - 1, -1, -1):
                h = (h @ Ws[l]).astype(np.float32)
                if Ds[l] is not None:
                    h = h * Ds[l]
            return h

        def tan(h):
            for l in range(L):
                h = (h @ Ws[l].T).astype(np.float32)
                if l + 1 < L:
                    h = h * Ds[l + 1]
            return h

        ls, rs = [v0.copy()], [v0.copy()]
        for _ in range(n):
            ls.append(vjp(ls[-1]))
        for _ in range(n - 1):
            rs.append(tan(rs[-1]))
        _f32(Ls, (n + 1) * B * d)[:] = np.stack(ls).ravel()
        _f32(Rs, n * B * d)[:] = np.stack(rs).ravel()
        s_out = np.zeros(B, np.float32)
        for k in range(1, n + 1):
            s_out += np.float32(c[k - 1]) * (ls[k] * v0).sum(1).astype(np.float32)
        _f32(S, B)[:] = s_out
        wm = []
        for m in range(n):
            w = np.float32(c[m]) * ls[0]
            for a in range(1, n - m):
                w = w + np.float32(c[a + m]) * ls[a]
            wm.append(w.astype(np.float32))
        _f32(Wm, n * B * d)[:] = np.stack(wm).ravel()
        self.launches += 1
        return 0

    # ---- elementwise (csrc/elementwise.cu) ----
    def impflow_act_mul(self, x, g, out, n, kind, order, beta_sp, stream):
        xv, gv, ov = _f32(x, n), _f32(g, n), _f32(out, n)
        with np.errstate(all='ignore'):
            r = _act(kind, xv, order, _beta(beta_sp))
        ov[:] = r if gv is None else r * gv
        self.launches += 1
        return 0

    def impflow_act_split(self, x, hi, lo, n, kind, order, beta_sp, stream):
        v = _act(kind, _f32(x, n), order, _beta(beta_sp)).astype(np.float32)
        h = _tf32(v)
        _f32(hi, n)[:] = h
        _f32(lo, n)[:] = v - h
        self.launches += 1
        return 0

    def impflow_act_beta_grad(self, x, g, g2, out, partial, n, order, beta_sp, stream):
        xv, gv = _f32(x, n).astype(np.float64), _f32(g, n).astype(np.float64)
        if _addr(g2) is not None:
            gv = gv * _f32(g2, n).astype(np.float64)
        _f32(out, 1)[0] = np.float32((gv * _dbeta(xv, order, float(_beta(beta_sp)))).sum())
        self.launches += 2
        return 0

    def impflow_act_second(self, p, t, ga, gb, out, n, kind, beta_sp, stream):
        pv = _f32(p, n)
        beta = _beta(beta_sp)
        with np.errstate(all='ignore'):
            r = _act(kind, pv, 2, beta) * _f32(t, n) * _f32(ga, n)
            if _addr(gb) is not None:
                r = r + _act(kind, pv, 1, beta) * _f32(gb, n)
        _f32(out, n)[:] = r
        self.launches += 1
        return 0

    def impflow_clip_adam_ema(self, p, g, m, v, ema, n, gnorm_sq, max_norm, step_size, beta1, beta2, eps, ema_decay,
                              stream):
        f = np.float32
        P, G, M, V = _f32(p, n), _f32(g, n), _f32(m, n), _f32(v, n)
        coef = f(1)
        if _addr(gnorm_sq) is not None and max_norm > 0:
            coef = min(f(1), f(max_norm) / (np.sqrt(_f32(gnorm_sq, 1)[0]) + f(1e-6)))
        G[:] = G * coef
        M[:] = f(beta1) * M + f(1 - beta1) * G
        V[:] = f(beta2) * V + f(1 - beta2) * G * G
        P[:] = P - f(step_size) * M / (np.sqrt(V) + f(eps))
        if _addr(ema) is not None:
            E = _f32(ema, n)
            E[:] = E - f(1 - ema_decay) * (E - P)
        self.launches += 1
        return 0

    def impflow_neumann_act_bwd_workspace_floats(self, M, N):
        return 8

    def impflow_neumann_act_bwd(self, p, t, ta, ab, y_hi, y_lo, colsum, beta_grad, ws, M, N, beta_sp, stream):
        n = M * N
        beta = _beta(beta_sp)
        P, T, TA = _f32(p, n), _f32(t, n), _f32(ta, n)
        AB = _f32(ab, n) if _addr(ab) is not None else np.zeros(n, dtype=np.float32)
        y = (_act(ACT_LIPSWISH, P, 2, beta) * T * TA + _act(ACT_LIPSWISH, P, 1, beta) * AB).astype(np.float32)
        h = _tf32(y)
        _f32(y_hi, n)[:] = h
        _f32(y_lo, n)[:] = y - h
        _f32(colsum, N)[:] = y.reshape(M, N).astype(np.float64).sum(0).astype(np.float32)
        bg = (TA * T * _dbeta(P, 1, beta)).astype(np.float64).sum()
        if _addr(ab) is not None:
            bg += (AB * _dbeta(P, 0, beta)).astype(np.float64).sum()
        _f32(beta_grad, 1)[0] = np.float32(bg)
        self.launches += 3
        return 0

    def impflow_lincomb3(self, a, ca, b, cb, c, cc, out, n, stream):
        r = _f32(a, n) * np.float32(ca)
        if _addr(b) is not None:
            r = r + _f32(b, n) * np.float32(cb)
        if _addr(c) is not None:
            r = r + _f32(c, n) * np.float32(cc)
        _f32(out, n)[:] = r
        self.launches += 1
        return 0

    def impflow_rowdot(self, a, c, out, B, d, alpha, beta, stream):
        av, cv, ov = _f32(a, B * d).reshape(B, d), _f32(c, B * d).reshape(B, d), _f32(out, B)
        dot = (av * cv).sum(1)
        ov[:] = (0 if beta == 0 else beta * ov) + alpha * dot
        self.launches += 1
        return 0

    def impflow_colsum_chunks(self, M, N):
        return 1

    def impflow_gemm_tc_splits(self, M, N, K):
        return 1

    def impflow_gemm_tc_set_tma_store(self, on):
        return 1

    def impflow_gemm_tc_set_pair(self, on):
        return 1

    def impflow_set_pdl(self, on):
        return 1

    def impflow_colsum(self, a, out, partial, M, N, stream):
        _f32(out, N)[:] = _f32(a, M * N).reshape(M, N).sum(0)
        self.launches += 1
        return 0

    def impflow_transpose(self, a, out, M, N, stream):
        _f32(out, M * N)[:] = _f32(a, M * N).reshape(M, N).T.ravel()
        self.launches += 1
        return 0

    def impflow_im2col3x3(self, x, col, B, H, W, C, ld, stream):
        xv = _f32(x, B * H * W * C).reshape(B, H, W, C)
        xp = np.zeros((B, H + 2, W + 2, C), np.float32)
        xp[:, 1:-1, 1:-1] = xv
        full = _f32(col, B * H * W * ld).reshape(B, H, W, ld)
        full[...] = 0
        for tap in range(9):
            ky, kx = tap // 3, tap % 3
            full[:, :, :, tap * C:(tap + 1) * C] = xp[:, ky:ky + H, kx:kx + W]
        self.launches += 1
        return 0

    def impflow_im2col3x3_split(self, x, col_hi, col_lo, B, H, W, C, ld, stream):
        full = np.zeros((B * H * W, ld), dtype=np.float32)
        self.impflow_im2col3x3(x, ctypes.c_void_p(full.ctypes.data), B, H, W, C, ld, stream)
        h = _tf32(full.reshape(-1))
        _f32(col_hi, full.size)[:] = h
        _f32(col_lo, full.size)[:] = full.reshape(-1) - h
        return 0

    def impflow_transpose_split(self, a, out_hi, out_lo, M, N, stream):
        t = np.ascontiguousarray(_f32(a, M * N).reshape(M, N).T).reshape(-1)
        h = _tf32(t)
        _f32(out_hi, M * N)[:] = h
        _f32(out_lo, M * N)[:] = t - h
        self.launches += 1
        return 0

    def impflow_col2im3x3(self, col, B, H, W, C, bias, pre_out, act_out, dmul_pre, act_kind, beta_sp, stream):
        cv = _f32(col, B * H * W * 9 * C).reshape(B, H, W, 9, C)
        acc = np.zeros((B, H + 2, W + 2, C), np.float32)
        for tap in range(9):
            ky, kx = tap // 3, tap % 3
            acc[:, ky:ky + H, kx:kx + W] += cv[:, :, :, tap]
        acc = acc[:, 1:-1, 1:-1].reshape(B * H * W, C)
        n = B * H * W * C
        _epilogue(acc, _f32(bias, C), _f32(pre_out, n), _f32(act_out, n), _f32(dmul_pre, n), act_kind,
                  _beta(beta_sp))
        self.launches += 1
        return 0

    def impflow_split_tf32(self, a, hi, lo, n, stream):
        av = _f32(a, n)
        h = _tf32(av)
        _f32(hi, n)[:] = h
        _f32(lo, n)[:] = av - h
        self.launches += 1
        return 0

    # ---- GEMMs (csrc/gemm_simt.cu, csrc/gemm_tcgen05.cu) ----
    def impflow_gemm_nt(self, A, lda, Bm, ldb, bias, pre_out, act_out, dmul_pre, ldc, M, N, K, act_kind, beta_sp,
                        stream):
        assert lda == K and ldb == K and ldc == N
        acc = (_f32(A, M * K).reshape(M, K) @ _f32(Bm, N * K).reshape(N, K).T).astype(np.float32)
        _epilogue(acc, _f32(bias, N), _f32(pre_out, M * N), _f32(act_out, M * N), _f32(dmul_pre, M * N), act_kind,
                  _beta(beta_sp))
        self.launches += 1
        return 0

    def impflow_gemm_strided(self, A, sAm, sAk, Bm, sBn, sBk, bias, out, ldc, M, N, K, stream):
        na = (M - 1) * sAm + (K - 1) * sAk + 1
        nb = (N - 1) * sBn + (K - 1) * sBk + 1
        a = np.lib.stride_tricks.as_strided(_f32(A, na), shape=(M, K), strides=(4 * sAm, 4 * sAk))
        b = np.lib.stride_tricks.as_strided(_f32(Bm, nb), shape=(N, K), strides=(4 * sBn, 4 * sBk))
        c = (a @ b.T).astype(np.float32)
        if _addr(bias) is not None:
            c = c + _f32(bias, N)
        _f32(out, M * ldc).reshape(M, ldc)[:, :N] = c
        self.launches += 1
        return 0

    def impflow_wgrad_simt_workspace_floats(self, M, N1, N2):
        return N1 * N2

    def impflow_wgrad_simt(self, G, ldg, A, lda, out, ldo, M, N1, N2, ws, stream):
        g = _f32(G, M * ldg).reshape(M, ldg)[:, :N1]
        a = _f32(A, M * lda).reshape(M, lda)[:, :N2]
        _f32(out, N1 * ldo).reshape(N1, ldo)[:, :N2] = (g.T.astype(np.float64) @ a.astype(np.float64)).astype(np.float32)
        self.launches += 2
        return 0

    def impflow_gemm_nt_tc(self, A_hi, A_lo, lda, B_hi, B_lo, ldb, bias, pre_out, act_out, dmul_pre, split_hi,
                           split_lo, ldc, M, N, K, act_kind, beta_sp, splitk_ws, stream):
        if K % 32 or lda % 4 or ldb % 4:
            self._err = b'gemm_nt_tc: layout'
            return -2
        ah, al = _f32(A_hi, M * K).reshape(M, K).astype(np.float64), _f32(A_lo, M * K).reshape(M, K).astype(np.float64)
        bh, bl = _f32(B_hi, N * K).reshape(N, K).astype(np.float64), _f32(B_lo, N * K).reshape(N, K).astype(np.float64)
        acc = (al @ bh.T + ah @ bl.T + ah @ bh.T).astype(np.float32)
        _epilogue(acc, _f32(bias, N), _f32(pre_out, M * N), _f32(act_out, M * N), _f32(dmul_pre, M * N), act_kind,
                  _beta(beta_sp), _f32(split_hi, M * N), _f32(split_lo, M * N))
        self.launches += 1
        return 0

    def impflow_branch3_tc(self, x0, ldx, W1_hi, W1_lo, W2_hi, W2_lo, W3_hi, W3_lo, bias1, bias2, mul1, mul2, pre1_out,
                           pre2_out, out, ldo, M, C, N3, act_kind, beta1, beta2, stream):
        if C % 256 or N3 > 32 or ldx < 32 or ldx % 4 or ldo < N3:
            self._err = b'branch3_tc: layout'
            return -2
        pl = lambda p, r, c: _f32(p, r * c).reshape(r, c).astype(np.float64)
        x = _f32(x0, M * ldx).reshape(M, ldx)[:, :32]
        xh = _tf32(x)
        xl = (x - xh).astype(np.float32)

        def mm(ah, al, bh, bl):
            return (al.astype(np.float64) @ bh.T + ah.astype(np.float64) @ bl.T + ah.astype(np.float64) @ bh.T
                    ).astype(np.float32)

        def psi(acc, bias, mul, pre_out, beta):
            if mul is not None:
                return acc * _f32(mul, M * C).reshape(M, C)
            v = acc + (_f32(bias, C) if _addr(bias) is not None else np.float32(0))
            if _addr(pre_out) is not None:
                _f32(pre_out, M * C).reshape(M, C)[:] = v
            return _act(act_kind, v, 0, beta)

        a1 = psi(mm(xh, xl, pl(W1_hi, C, 32), pl(W1_lo, C, 32)), bias1, mul1 if _addr(mul1) else None, pre1_out,
                 _beta(beta1)).astype(np.float32)
        a1h = _tf32(a1)
        a2 = psi(mm(a1h, a1 - a1h, pl(W2_hi, C, C), pl(W2_lo, C, C)), bias2, mul2 if _addr(mul2) else None, pre2_out,
                 _beta(beta2)).astype(np.float32)
        a2h = _tf32(a2)
        y = mm(a2h, a2 - a2h, pl(W3_hi, N3, C), pl(W3_lo, N3, C))
        _f32(out, M * ldo).reshape(M, ldo)[:, :N3] = y
        self.launches += 1
        return 0

    def impflow_wgrad_tc_workspace_floats(self, Mpix, N1, N2):
        return 16

    def impflow_wgrad_tc(self, G_hi, G_lo, ldg, A_hi, A_lo, lda, out, ldo, transpose_out, Mpix, N1, N2, ws, stream):
        if Mpix % 32 or ldg % 4 or lda % 4:
            self._err = b'wgrad_tc: layout'
            return -2
        gh = _f32(G_hi, Mpix * ldg).reshape(Mpix, ldg)[:, :N1].astype(np.float64)
        gl = _f32(G_lo, Mpix * ldg).reshape(Mpix, ldg)[:, :N1].astype(np.float64)
        ah = _f32(A_hi, Mpix * lda).reshape(Mpix, lda)[:, :N2].astype(np.float64)
        al = _f32(A_lo, Mpix * lda).reshape(Mpix, lda)[:, :N2].astype(np.float64)
        c = (gl.T @ ah + gh.T @ al + gh.T @ ah).astype(np.float32)
        if transpose_out:
            _f32(out, N2 * ldo).reshape(N2, ldo)[:, :N1] = c.T
        else:
            _f32(out, N1 * ldo).reshape(N1, ldo)[:, :N2] = c
        self.launches += 1
        return 0

    # ---- native conv3 runtime (csrc/conv3_plan.cu): the same orchestration over the emulated kernels ----
    @staticmethod
    def _plan(p):
        from impflow_b200._cabi import Conv3Plan
        return Conv3Plan.from_address(_addr(p))

    @staticmethod
    def _tmp(*shape):
        a = np.zeros(shape, dtype=np.float32)
        return a, ctypes.c_void_p(a.ctypes.data)

    def impflow_chain23_parts(self, C):
        return C // 128

    def impflow_conv3_set_chain23_a32(self, on):
        return 1

    def impflow_conv3_set_chain23(self, on):
        return 1

    def impflow_wgrad_set_slice_major(self, on):
        return 1

    def impflow_add_launch_count(self, n):
        self.launches += int(n)

    def impflow_sn_conv_set_ctas(self, ctas):
        return 32

    def impflow_chain23_tc(self, A_hi, A_lo, lda, W2_hi, W2_lo, W3_hi, W3_lo, bias2, mul2, pre2_out, out, ldo,
                           part_stride, M, C, N3, act_kind, beta2, stream):
        A = _f32(A_hi, M * lda) + (_f32(A_lo, M * lda) if _addr(A_lo) is not None else 0)
        A = A.reshape(M, lda)[:, :C]
        W2 = (_f32(W2_hi, C * C) + _f32(W2_lo, C * C)).reshape(C, C)
        W3 = (_f32(W3_hi, N3 * C) + _f32(W3_lo, N3 * C)).reshape(N3, C)
        H = (A @ W2.T).astype(np.float32)
        if _addr(mul2) is not None:
            A2 = H * _f32(mul2, M * C).reshape(M, C)
        else:
            if _addr(bias2) is not None:
                H = H + _f32(bias2, C)
            if _addr(pre2_out) is not None:
                _f32(pre2_out, M * C)[:] = H.ravel()
            A2 = _act(act_kind, H, 0, _beta(beta2)).astype(np.float32)
        for q in range(C // 128):
            part = (A2[:, q * 128:(q + 1) * 128] @ W3[:, q * 128:(q + 1) * 128].T).astype(np.float32)
            dst = _f32(out, (C // 128 - 1) * part_stride + M * ldo)[q * part_stride:q * part_stride + M * ldo]
            dst.reshape(M, ldo)[:, :N3] = part
        self.launches += 1
        return 0

    def impflow_conv3_workspace_floats(self, B, H, W, c, C, k0):
        return 64

    def _conv3_chain(self, P, xin_ptr, W1, W2, W3, b1, b2, mul1, mul2, pre1, pre2, act_kind, beta1, beta2):
        M, N3 = P.B * P.H * P.W, 9 * P.c
        Y, Yp = self._tmp(M, N3)
        if P.allow_fused and P.k0 == 32 and P.C % 256 == 0 and N3 <= 32:
            x0, x0p = self._tmp(M, 32)
            assert self.impflow_im2col3x3(xin_ptr, x0p, P.B, P.H, P.W, P.c, 32, None) == 0
            assert self.impflow_branch3_tc(x0p, 32, W1[0], W1[1], W2[0], W2[1], W3[0], W3[1], b1, b2, mul1, mul2, pre1,
                                           pre2, Yp, N3, M, P.C, N3, act_kind, beta1, beta2, None) == 0
            return Y, Yp
        xh, xhp = self._tmp(M, P.k0)
        xl, xlp = self._tmp(M, P.k0)
        h1h, h1hp = self._tmp(M, P.C)
        h1l, h1lp = self._tmp(M, P.C)
        h2h, h2hp = self._tmp(M, P.C)
        h2l, h2lp = self._tmp(M, P.C)
        assert self.impflow_im2col3x3_split(xin_ptr, xhp, xlp, P.B, P.H, P.W, P.c, P.k0, None) == 0
        k1 = ACT_MULTIPLIER if mul1 is not None else act_kind
        assert self.impflow_gemm_nt_tc(xhp, xlp, P.k0, W1[0], W1[1], P.k0, b1, pre1, None, mul1, h1hp, h1lp, P.C, M, P.C,
                                       P.k0, k1, beta1, None, None) == 0
        assert self.impflow_gemm_nt_tc(h1hp, h1lp, P.C, W2[0], W2[1], P.C, b2, pre2, None, mul2, h2hp, h2lp, P.C, M, P.C,
                                       P.C, k1, beta2, None, None) == 0
        assert self.impflow_gemm_nt_tc(h2hp, h2lp, P.C, W3[0], W3[1], P.C, None, Yp, None, None, None, None, N3, M, N3,
                                       P.C, ACT_NONE, None, None, None) == 0
        return Y, Yp

    def impflow_conv3_forward(self, plan, x_rows, y_rows, pre1, pre2, stream):
        P = self._plan(plan)
        M = P.B * P.H * P.W
        xin = x_rows
        if P.act0_kind != ACT_NONE:
            t, tp = self._tmp(M, P.c)
            self.impflow_act_mul(x_rows, None, tp, M * P.c, P.act0_kind, 0, P.beta0, None)
            xin = tp
        none = lambda v: v if _addr(v) is not None else None
        Y, Yp = self._conv3_chain(P, xin, (P.W1f_hi, P.W1f_lo), (P.W2f_hi, P.W2f_lo), (P.W3f_hi, P.W3f_lo), none(P.b1),
                                  none(P.b2), None, None, none(pre1), none(pre2), P.act_kind, none(P.beta1),
                                  none(P.beta2))
        return self.impflow_col2im3x3(Yp, P.B, P.H, P.W, P.c, none(P.b3), y_rows, None, None, ACT_NONE, None, None)

    def impflow_conv3_prepare_vjp(self, plan, pre1, pre2, d1, d2, stream):
        P = self._plan(plan)
        n = P.B * P.H * P.W * P.C
        self.impflow_act_mul(pre1, None, d1, n, P.act_kind, 1, P.beta1, None)
        return self.impflow_act_mul(pre2, None, d2, n, P.act_kind, 1, P.beta2, None)

    def impflow_conv3_vjp(self, plan, pre0, d1, d2, v_rows, out_rows, stream):
        P = self._plan(plan)
        Y, Yp = self._conv3_chain(P, v_rows, (P.W3b_hi, P.W3b_lo), (P.W2b_hi, P.W2b_lo), (P.W1b_hi, P.W1b_lo), None, None,
                                  d2, d1, None, None, ACT_NONE, None, None)
        if P.act0_kind != ACT_NONE:
            return self.impflow_col2im3x3(Yp, P.B, P.H, P.W, P.c, None, out_rows, None, pre0, P.act0_kind, P.beta0, None)
        return self.impflow_col2im3x3(Yp, P.B, P.H, P.W, P.c, None, out_rows, None, None, ACT_NONE, None, None)

    def impflow_conv3_power_series(self, plan, pre0, d1, d2, v_rows, coeffs, n, w_rows, dot_coeffs, dot_out, stream):
        P = self._plan(plan)
        nel = P.B * P.H * P.W * P.c
        v = _f32(v_rows, nel)
        w = None
        if _addr(w_rows) is not None:
            w = _f32(w_rows, nel)
            w[:] = v
        dots = None
        if _addr(dot_out) is not None:
            dots = _f32(dot_out, P.B)
            dots[:] = 0
        cur, curp = self._tmp(nel)
        cur[:] = v
        for k in range(n):
            nxt, nxtp = self._tmp(nel)
            assert self.impflow_conv3_vjp(plan, pre0, d1, d2, curp, nxtp, None) == 0
            if w is not None:
                w += np.float32(coeffs[k]) * nxt
            if dots is not None:
                dots += np.float32(dot_coeffs[k]) * (nxt.reshape(P.B, -1) * v.reshape(P.B, -1)).sum(1, dtype=np.float32)
            cur, curp = nxt, nxtp
        return 0

    def impflow_conv3_broyden_host_bytes(self, threshold):
        return STATE_DTYPE.itemsize + 8 * (threshold + 2)

    def impflow_conv3_set_runahead(self, iterations):
        return 2

    def impflow_conv3_set_chain_fuse(self, on):
        return 1

    def impflow_conv3_broyden(self, plan, mode, rhs_rows, pre0, d1, d2, xa, xb, ga, gb, low_x, low_g, Ut, Vt, sample_sq,
                              low_sq, partial, state_dev, state_host, threshold, eps_scaled, stream):
        P = self._plan(plan)
        nel = P.B * P.H * P.W * P.c
        d = P.H * P.W * P.c
        rhs = _f32(rhs_rows, nel)

        def eval_g(xp, gp):
            t, tp = self._tmp(nel)
            if mode == 0:
                assert self.impflow_conv3_forward(plan, xp, tp, None, None, None) == 0
                _f32(gp, nel)[:] = rhs - t - _f32(xp, nel)
            else:
                assert self.impflow_conv3_vjp(plan, pre0, d1, d2, xp, tp, None) == 0
                _f32(gp, nel)[:] = t + _f32(xp, nel) - rhs

        x_old, xn, g_old, gn = xa, xb, ga, gb
        eval_g(x_old, g_old)
        self.impflow_broyden_begin(x_old, g_old, xn, low_x, low_g, sample_sq, low_sq, partial, state_dev, P.B, d,
                                   threshold, eps_scaled, None)
        while _state(state_dev)[0]['active']:
            eval_g(xn, gn)
            self.impflow_broyden_step(x_old, g_old, xn, gn, Ut, Vt, low_x, low_g, sample_sq, low_sq, partial, state_dev,
                                      P.B, d, threshold, None)
            x_old, xn = xn, x_old
            g_old, gn = gn, g_old
        ctypes.memmove(_addr(state_host), _addr(state_dev), STATE_DTYPE.itemsize)
        return 0

    # ---- spectral (csrc/spectral.cu) ----
    def impflow_prep_weights(self, W, sigma, coeff, kind, cout, cin, fwd, fwd_hi, fwd_lo, fwd_rows, fwd_k, bwd, bwd_hi,
                             bwd_lo, bwd_rows, bwd_k, stream):
        taps = 1 if kind == 0 else 9
        Wt = torch.from_numpy(_f32(W, cout * cin * taps).copy()).view(cout, cin, *((1, 1) if kind == 0 else (3, 3)))
        Wt = Wt / max(np.float32(1), _f32(sigma, 1)[0] / np.float32(coeff))
        if kind == 0:
            f, b = Wt.reshape(cout, cin), Wt.reshape(cout, cin).t()
        elif kind == 1:
            f = Wt.permute(0, 2, 3, 1).reshape(cout, 9 * cin)
            b = Wt.permute(2, 3, 1, 0).reshape(9 * cin, cout)
        else:
            f = Wt.flip(2, 3).permute(2, 3, 0, 1).reshape(9 * cout, cin)
            b = Wt.flip(2, 3).permute(1, 2, 3, 0).reshape(cin, 9 * cout)
        for m, out, hi, lo, rows, kp in ((f, fwd, fwd_hi, fwd_lo, fwd_rows, fwd_k), (b, bwd, bwd_hi, bwd_lo, bwd_rows, bwd_k)):
            assert m.shape[0] == rows and m.shape[1] <= kp
            full = np.zeros((rows, kp), dtype=np.float32)
            full[:, :m.shape[1]] = m.numpy()
            _f32(out, rows * kp)[:] = full.reshape(-1)
            if _addr(hi) is not None:
                h = _tf32(full.reshape(-1))
                _f32(hi, rows * kp)[:] = h
                _f32(lo, rows * kp)[:] = full.reshape(-1) - h
        self.launches += 1
        return 0

    def impflow_sn_scale(self, W, sigma, coeff, out, scale_out, n, stream):
        sg = _f32(sigma, 1)[0]
        _f32(out, n)[:] = _f32(W, n) / max(np.float32(1), sg / np.float32(coeff))
        if _addr(scale_out) is not None:
            _f32(scale_out, 1)[0] = sg
        self.launches += 1
        return 0

    def impflow_sn_scale_grad(self, G, D, sigma, gw_dot, coeff, out, n, stream):
        sg = float(_f32(sigma, 1)[0])
        ratio = sg / coeff
        s_ = 1.0 / ratio if ratio > 1 else 1.0
        ds = -coeff / (sg * sg) if ratio > 1 else 0.0
        _f32(out, n)[:] = np.float32(s_) * _f32(G, n) + np.float32(ds * float(_f32(gw_dot, 1)[0])) * _f32(D, n)
        self.launches += 1
        return 0

    def impflow_sn_scale_grad_layout(self, Wbar, ldw, W, D, sigma, coeff, kind, cout, cin, out, ws, stream):
        taps = 1 if kind == 0 else 9
        n = cout * cin * taps
        rows = 9 * cout if kind == 2 else cout
        Wb = _f32(Wbar, (rows - 1) * ldw + (cin if kind != 1 else 9 * cin))
        i = np.arange(n)
        if kind == 0:
            idx = (i // cin) * ldw + (i % cin)
        else:
            co, r = i // (cin * 9), i % (cin * 9)
            ci, t = r // 9, r % 9
            idx = co * ldw + t * cin + ci if kind == 1 else ((8 - t) * cout + co) * ldw + ci
        G = Wb[idx]
        Wv, Dv = _f32(W, n), _f32(D, n)
        sg = float(_f32(sigma, 1)[0])
        ratio = sg / coeff
        s_ = 1.0 / ratio if ratio > 1 else 1.0
        ds = -coeff / (sg * sg) if ratio > 1 else 0.0
        t_ = float((G.astype(np.float64) * Wv).sum())
        _f32(out, n)[:] = np.float32(s_) * G + np.float32(ds * t_) * Dv
        self.launches += 2
        return 0

    @staticmethod
    def _actnorm_view(ptr, B, C, HW, channels_last):
        """(B, C, HW)-indexed numpy view of either memory order."""
        if channels_last:
            return _f32(ptr, B * C * HW).reshape(B, HW, C).transpose(0, 2, 1)
        return _f32(ptr, B * C * HW).reshape(B, C, HW)

    def impflow_actnorm_forward(self, x, bias, weight, y, logpx, logpx_out, B, C, HW, channels_last, stream):
        xv = self._actnorm_view(x, B, C, HW, channels_last)
        b, w = _f32(bias, C), _f32(weight, C)
        self._actnorm_view(y, B, C, HW, channels_last)[:] = (xv + b[None, :, None]) * np.exp(w)[None, :, None]
        if _addr(logpx_out) is not None:
            _f32(logpx_out, B)[:] = _f32(logpx, B) - np.float32(w.sum() * HW)
        self.launches += 1
        return 0

    def impflow_actnorm_workspace_floats(self, C):
        return 64 * C

    def impflow_actnorm_backward(self, gy, y, weight, g_logpx, gx, gbias, gweight, ws, B, C, HW, channels_last,
                                 stream):
        g = self._actnorm_view(gy, B, C, HW, channels_last)
        yv = self._actnorm_view(y, B, C, HW, channels_last)
        w = _f32(weight, C)
        e = np.exp(w)
        self._actnorm_view(gx, B, C, HW, channels_last)[:] = g * e[None, :, None]
        _f32(gbias, C)[:] = (g.astype(np.float64) * e[None, :, None]).sum((0, 2))
        gl = float(_f32(g_logpx, B).astype(np.float64).sum()) if _addr(g_logpx) is not None else 0.0
        _f32(gweight, C)[:] = (g.astype(np.float64) * yv).sum((0, 2)) - HW * gl
        self.launches += 2
        return 0

    def impflow_sn_power_iter(self, W, u, v, sigma, iters, out_f, in_f, n_iterations, atol, rtol, stream):
        Wm = _f32(W, out_f * in_f).reshape(out_f, in_f)
        uv, vv = _f32(u, out_f), _f32(v, in_f)
        nrm = lambda t: t / max(np.float32(np.sqrt((t * t).sum())), np.float32(1e-12))
        tol_mode = n_iterations < 0
        used = 0
        un, vn = uv.copy(), vv.copy()
        for _ in range(200 if tol_mode else n_iterations):
            ou, ov = un, vn
            un = nrm(Wm @ vn).astype(np.float32)
            vn = nrm(Wm.T @ un).astype(np.float32)
            used += 1
            if tol_mode:
                err_u = np.sqrt(((un - ou) ** 2).sum()) / np.sqrt(out_f)
                err_v = np.sqrt(((vn - ov) ** 2).sum()) / np.sqrt(in_f)
                if err_u < atol + rtol * un.max() and err_v < atol + rtol * vn.max():
                    break
        _f32(sigma, 1)[0] = np.float32(un @ (Wm @ vn))
        if _addr(iters) is not None:
            np.ctypeslib.as_array((ctypes.c_int32 * 1).from_address(_addr(iters)))[0] = used
        if used > 0:
            uv[:] = un
            vv[:] = vn
        self.launches += 1
        return 0

    def impflow_sn_power_iter_batch(self, descs, n, max_out, max_in, n_iterations, atol, rtol, stream):
        from impflow_b200._cabi import SnDesc
        arr = (SnDesc * n).from_address(_addr(descs))
        for d in arr:
            self.impflow_sn_power_iter(ctypes.c_void_p(d.W), ctypes.c_void_p(d.u), ctypes.c_void_p(d.v),
                                       ctypes.c_void_p(d.sigma), ctypes.c_void_p(d.iters) if d.iters else None,
                                       d.out_f, d.in_f, n_iterations, atol, rtol, stream)
            self.launches -= 1
        self.launches += 1
        return 0

    def impflow_sn_conv_workspace_floats(self, Cout, Cin, H, W):
        narrow = min(Cout, Cin) * H * W
        return 0 if 2 * narrow * 4 > 160 * 1024 else 128 * narrow + narrow + 5 * 128

    def impflow_sn_power_iter_conv3x3(self, W, u, v, sigma, iters, Cout, Cin, H, Wd, n_iterations, atol, rtol, ws, D,
                                      stream):
        import torch.nn.functional as F
        Wt = torch.from_numpy(_f32(W, Cout * Cin * 9).reshape(Cout, Cin, 3, 3).copy())
        uv, vv = _f32(u, Cout * H * Wd), _f32(v, Cin * H * Wd)
        un, vn = torch.from_numpy(uv.copy()), torch.from_numpy(vv.copy())
        nrm = lambda t: t / max(float(t.norm()), 1e-12)
        conv = lambda t: F.conv2d(t.view(1, Cin, H, Wd), Wt, padding=1).reshape(-1)
        convT = lambda t: F.conv_transpose2d(t.view(1, Cout, H, Wd), Wt, padding=1).reshape(-1)
        tol_mode = n_iterations < 0
        used = 0
        for _ in range(200 if tol_mode else n_iterations):
            ou, ov = un, vn
            un = nrm(conv(vn))
            vn = nrm(convT(un))
            used += 1
            if tol_mode:
                err_u = float((un - ou).norm()) / un.numel() ** 0.5
                err_v = float((vn - ov).norm()) / vn.numel() ** 0.5
                if err_u < atol + rtol * float(un.max()) and err_v < atol + rtol * float(vn.max()):
                    break
        _f32(sigma, 1)[0] = np.float32(float(torch.dot(un, conv(vn))))
        if _addr(D) is not None:      # d <u, conv(v; W)> / dW
            with torch.enable_grad():
                Wg = Wt.clone().requires_grad_(True)
                s_ = torch.dot(un, F.conv2d(vn.view(1, Cin, H, Wd), Wg, padding=1).reshape(-1))
                _f32(D, Cout * Cin * 9)[:] = torch.autograd.grad(s_, Wg)[0].reshape(-1).numpy()
        if _addr(iters) is not None:
            np.ctypeslib.as_array((ctypes.c_int32 * 1).from_address(_addr(iters)))[0] = used
        if used > 0:
            uv[:] = un.numpy()
            vv[:] = vn.numpy()
        self.launches += 1
        return 0


def install(monkeypatch):
    """Route the product's C-ABI calls to the numpy emulation for the duration of one test."""
    import impflow_b200
    cabi = impflow_b200._cabi
    lib = EmulatedLib()
    monkeypatch.setattr(cabi, '_lib', lib)
    monkeypatch.setattr(cabi, 'load', lambda: lib)
    monkeypatch.setattr(cabi, 'require_device', lambda t, what='tensor': None)
    monkeypatch.setattr(cabi, '_CHECK_DEVICE', [False])
    monkeypatch.setattr(cabi, 'pinned_bytes', lambda n: torch.zeros(n, dtype=torch.uint8))
    monkeypatch.setattr(cabi, 'sync_stream', lambda: None)
    monkeypatch.setattr(cabi, 'stream', lambda: None)
    return lib
