"""TEST INFRASTRUCTURE ONLY — numpy emulation of the Lop-layer entry points of include/impflow_b200.h
(impflow_lop_norms, impflow_prep_weights_lop, impflow_lop_scale_grad_layout) on top of the C-ABI emulator in
tests/cabi_emulator.py, for the CPU cases of tests/test_host_lop_program.py.

Branches with Lop layers compile to a BranchProgram for CUDA weights only (branch_program._device_lop); install() also
lets CPU weights compile, so that the host logic of the program path (preparation, gradient chain, routing) runs
without a GPU.  Like the base emulator it restates what the kernels compute."""
import numpy as np

from tests import cabi_emulator
from tests.cabi_emulator import _addr, _f32


class LopEmulatedLib(cabi_emulator.EmulatedLib):

    @staticmethod
    def _lop_groups(a, cout, cin, taps, axis):
        """(groups, rest) view of a module-layout [cout][cin][taps] array: rows are output rows or input channels."""
        a = a.reshape(cout, cin, taps)
        return (a if axis == 0 else a.transpose(1, 0, 2)).reshape(cout if axis == 0 else cin, -1)

    def impflow_lop_norms(self, W, cout, cin, taps, axis, norm_type, norms, scale_out, stream):
        g = self._lop_groups(_f32(W, cout * cin * taps), cout, cin, taps, axis)
        nv = (np.abs(g).sum(1) if norm_type == 1 else np.sqrt((g * g).sum(1)) if norm_type == 2
              else g.max(1)).astype(np.float32)
        out = _f32(norms, len(nv) + 1)
        out[:-1], out[-1] = nv, nv.max()
        if _addr(scale_out) is not None:
            _f32(scale_out, 1)[0] = nv.max()
        self.launches += 2
        return 0

    def impflow_prep_weights_lop(self, W, norms, group, coeff, kind, cout, cin, fwd, fwd_hi, fwd_lo, fwd_rows, fwd_k,
                                 bwd, bwd_hi, bwd_lo, bwd_rows, bwd_k, stream):
        taps = 1 if kind == 0 else 9
        w = _f32(W, cout * cin * taps).reshape(cout, cin, taps)
        nv = _f32(norms, [1, cout, cin][group])
        f = np.maximum(np.float32(1), nv * (np.float32(1) / np.float32(coeff)))
        f = f[0] if group == 0 else (f[:, None, None] if group == 1 else f[None, :, None])
        scaled = np.ascontiguousarray((w / f).astype(np.float32))
        unit = np.zeros(1, dtype=np.float32)          # sigma 0: the layouts of impflow_prep_weights, unscaled
        return self.impflow_prep_weights(scaled.ctypes.data, unit.ctypes.data, coeff, kind, cout, cin, fwd, fwd_hi,
                                         fwd_lo, fwd_rows, fwd_k, bwd, bwd_hi, bwd_lo, bwd_rows, bwd_k, stream)

    def impflow_lop_scale_grad_layout(self, Wbar, ldw, W, norms, coeff, kind, cout, cin, axis, norm_type, local, out,
                                      ws, stream):
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
        G = self._lop_groups(Wb[idx], cout, cin, taps, axis)
        w = self._lop_groups(_f32(W, n), cout, cin, taps, axis)
        groups = G.shape[0]
        nall = _f32(norms, groups + 1)
        nv, N = nall[:groups, None], nall[groups]
        ratio = (nv if local else N) * (np.float32(1) / np.float32(coeff))
        f = np.maximum(np.float32(1), ratio)
        c = np.where(ratio > 1, 1.0, np.where(ratio == 1, 0.5, 0.0))
        tk = (G.astype(np.float64) * w).sum(1, keepdims=True)
        if norm_type == 1:
            dn = np.sign(w)
        elif norm_type == 2:
            dn = w / nv
        else:
            dn = (w == nv) / (w == nv).sum(1, keepdims=True)
        if not local:
            tied = nv == N
            dn, tk = dn * tied / tied.sum(), tk.sum()
        g = G / f - (c * tk / (coeff * f.astype(np.float64) ** 2)) * dn
        res = g.astype(np.float32).reshape(cout, -1, taps) if axis == 0 else \
            g.astype(np.float32).reshape(cin, cout, taps).transpose(1, 0, 2)
        _f32(out, n)[:] = np.ascontiguousarray(res).reshape(-1)
        self.launches += 2
        return 0


def install(monkeypatch):
    """cabi_emulator.install with the Lop entry points, and Lop branches compiled for CPU weights."""
    import impflow_b200
    cabi_emulator.install(monkeypatch)
    lib = LopEmulatedLib()
    monkeypatch.setattr(impflow_b200._cabi, '_lib', lib)
    monkeypatch.setattr(impflow_b200._cabi, 'load', lambda: lib)
    monkeypatch.setattr(impflow_b200.branch_program, '_device_lop', lambda t: True)
    return lib
