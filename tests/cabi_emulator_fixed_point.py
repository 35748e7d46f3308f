"""TEST INFRASTRUCTURE ONLY — numpy emulation of the one-call fixed-point entry points of include/impflow_b200.h
(impflow_conv3_fixed_point, impflow_conv3_fixed_point_host_bytes, impflow_mlp_fixed_point) on top of the C-ABI
emulator in tests/cabi_emulator.py, for the CPU cases of tests/test_host_fixed_point.py.

The one-call solves take CUDA tensors only (branch_program._device_solve); install() also lets them take the CPU
tensors of the emulated suite, so that the host logic around the calls (routing, workspaces, state read-back, layouts)
runs without a GPU.  Like the base emulator it restates what the kernels compute, with the same roundings."""
import ctypes

import numpy as np

from tests import cabi_emulator
from tests.cabi_emulator import _act, _addr, _beta, _f32


class FixedPointEmulatedLib(cabi_emulator.EmulatedLib):

    @staticmethod
    def _fixed_point(f, rhs, start, out, state_host, nel, atol, rtol, threshold):
        """The Banach loop of impflow_conv3_fixed_point / impflow_mlp_fixed_point over the evaluation f (numpy float32
        operations round once each, as the kernels' __f*_rn do)."""
        r, s = _f32(rhs, nel), _f32(start, nel)
        tol = np.float32(atol) + np.abs(s) * np.float32(rtol)
        prev, k = s, 1
        with np.errstate(all='ignore'):
            while True:
                x = (r - f(prev)).astype(np.float32)
                d = x - prev
                if k - 1 > threshold or bool((d * d / tol < 1).all()):
                    break
                prev, k = x, k + 1
        _f32(out, nel)[:] = x
        st = np.ctypeslib.as_array((ctypes.c_int32 * 4).from_address(_addr(state_host)))
        st[:] = (k - 1, 0, 0, 0)
        return 0

    def impflow_mlp_fixed_point(self, rhs, start, out, Wt, bias, dims, L, act_kind, beta_sp, xa, xb, counts, state_dev,
                                state_host, B, atol, rtol, threshold, stream):
        dims = [int(v) for v in dims]
        d = dims[0]
        betas = [(_beta(beta_sp[l]) if (beta_sp and l + 1 < L and beta_sp[l]) else None) for l in range(L)]
        Ws = [_f32(Wt[l], dims[l] * dims[l + 1]).reshape(dims[l], dims[l + 1]) for l in range(L)]
        bs = [(_f32(bias[l], dims[l + 1]) if bias[l] else None) for l in range(L)]

        def f(z):
            h = z.reshape(B, d)
            for l in range(L):
                h = (h @ Ws[l]).astype(np.float32)
                if bs[l] is not None:
                    h = h + bs[l]
                if l + 1 < L:
                    h = _act(act_kind, h, 0, betas[l]).astype(np.float32)
            return h.ravel()

        self.launches += 1
        return self._fixed_point(f, rhs, start, out, state_host, B * d, atol, rtol, threshold)

    def impflow_conv3_fixed_point_host_bytes(self, threshold):
        return 16 + 8 * (threshold + 2)

    def impflow_conv3_fixed_point(self, plan, rhs_rows, start_rows, out_rows, xa, xb, state_dev, state_host, atol, rtol,
                                  threshold, stream):
        P = self._plan(plan)
        nel = P.B * P.H * P.W * P.c

        def f(x):
            t, tp = self._tmp(nel)
            xx, xp = self._tmp(nel)
            xx[:] = x
            assert self.impflow_conv3_forward(plan, xp, tp, None, None, None) == 0
            return t

        return self._fixed_point(f, rhs_rows, start_rows, out_rows, state_host, nel, atol, rtol, threshold)


def install(monkeypatch):
    """cabi_emulator.install with the fixed-point entry points, and the one-call solves open to CPU tensors."""
    import impflow_b200
    cabi_emulator.install(monkeypatch)
    lib = FixedPointEmulatedLib()
    monkeypatch.setattr(impflow_b200._cabi, '_lib', lib)
    monkeypatch.setattr(impflow_b200._cabi, 'load', lambda: lib)
    monkeypatch.setattr(impflow_b200.branch_program, '_device_solve', lambda t: True)
    return lib
