"""ctypes binding of libimpflow_b200.so (C ABI declared in include/impflow_b200.h).

There is no CPU fallback: if the library is missing, or a tensor is not a dense fp32 CUDA
tensor, the call raises."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libimpflow_b200.so')

_c_fp = ctypes.c_void_p
_ll = ctypes.c_longlong
_i = ctypes.c_int
_f = ctypes.c_float
_d = ctypes.c_double

# name -> (restype, argtypes); mirrors include/impflow_b200.h one to one
SIGNATURES = {
    'impflow_version': (_i, []),
    'impflow_last_error': (ctypes.c_char_p, []),
    'impflow_launch_count': (_ll, []),
    'impflow_add_launch_count': (None, [_ll]),
    'impflow_broyden_state_bytes': (ctypes.c_size_t, []),
    'impflow_broyden_workspace_floats': (ctypes.c_size_t, [_i, _ll, _i]),
    'impflow_broyden_begin': (_i, [_c_fp] * 9 + [_i, _ll, _i, _d, _c_fp]),
    'impflow_broyden_step': (_i, [_c_fp] * 12 + [_i, _ll, _i, _c_fp]),
    'impflow_mlp_solver_limits': (_i, [_c_fp, _c_fp, _c_fp]),
    'impflow_mlp_solver_partial_doubles': (ctypes.c_size_t, []),
    'impflow_mlp_broyden_solve': (_i, [_c_fp, _c_fp, _c_fp, _c_fp, _i, _i, _c_fp] + [_c_fp] * 12 + [_i, _i, _d, _c_fp]),
    'impflow_mlp_broyden_solve_vjp': (_i, [_c_fp, _c_fp, _c_fp, _c_fp, _c_fp, _i] + [_c_fp] * 12 + [_i, _i, _d, _c_fp]),
    'impflow_mlp_fixed_point': (_i, [_c_fp] * 6 + [_i, _i] + [_c_fp] * 6 + [_i, _f, _f, _i, _c_fp]),
    'impflow_mlp_series': (_i, [_c_fp] * 6 + [_i, _i, _i, _c_fp, _c_fp, _c_fp, _c_fp, _c_fp, _c_fp]),
    'impflow_act_mul': (_i, [_c_fp, _c_fp, _c_fp, _ll, _i, _i, _c_fp, _c_fp]),
    'impflow_act_split': (_i, [_c_fp, _c_fp, _c_fp, _ll, _i, _i, _c_fp, _c_fp]),
    'impflow_reduce_workspace_floats': (ctypes.c_size_t, [_ll]),
    'impflow_act_beta_grad': (_i, [_c_fp, _c_fp, _c_fp, _c_fp, _c_fp, _ll, _i, _c_fp, _c_fp]),
    'impflow_act_second': (_i, [_c_fp, _c_fp, _c_fp, _c_fp, _c_fp, _ll, _i, _c_fp, _c_fp]),
    'impflow_neumann_act_bwd_workspace_floats': (ctypes.c_size_t, [_ll, _i]),
    'impflow_neumann_act_bwd': (_i, [_c_fp] * 9 + [_ll, _i, _c_fp, _c_fp]),
    'impflow_lincomb3': (_i, [_c_fp, _f, _c_fp, _f, _c_fp, _f, _c_fp, _ll, _c_fp]),
    'impflow_clip_adam_ema': (_i, [_c_fp] * 5 + [_ll, _c_fp, _f, _f, _f, _f, _f, _f, _c_fp]),
    'impflow_actnorm_forward': (_i, [_c_fp] * 6 + [_ll, _i, _ll, _i, _c_fp]),
    'impflow_actnorm_workspace_floats': (ctypes.c_size_t, [_i]),
    'impflow_actnorm_backward': (_i, [_c_fp] * 8 + [_ll, _i, _ll, _i, _c_fp]),
    'impflow_rowdot': (_i, [_c_fp, _c_fp, _c_fp, _i, _ll, _f, _f, _c_fp]),
    'impflow_colsum_chunks': (_i, [_ll, _i]),
    'impflow_colsum': (_i, [_c_fp, _c_fp, _c_fp, _ll, _i, _c_fp]),
    'impflow_transpose': (_i, [_c_fp, _c_fp, _ll, _ll, _c_fp]),
    'impflow_im2col3x3': (_i, [_c_fp, _c_fp, _i, _i, _i, _i, _i, _c_fp]),
    'impflow_im2col3x3_split': (_i, [_c_fp, _c_fp, _c_fp, _i, _i, _i, _i, _i, _c_fp]),
    'impflow_transpose_split': (_i, [_c_fp, _c_fp, _c_fp, _ll, _ll, _c_fp]),
    'impflow_col2im3x3': (_i, [_c_fp, _i, _i, _i, _i, _c_fp, _c_fp, _c_fp, _c_fp, _i, _c_fp, _c_fp]),
    'impflow_gemm_nt': (_i, [_c_fp, _ll, _c_fp, _ll, _c_fp, _c_fp, _c_fp, _c_fp, _ll, _ll, _i, _i, _i, _c_fp, _c_fp]),
    'impflow_gemm_strided': (_i, [_c_fp, _ll, _ll, _c_fp, _ll, _ll, _c_fp, _c_fp, _ll, _ll, _i, _i, _c_fp]),
    'impflow_wgrad_simt_workspace_floats': (ctypes.c_size_t, [_ll, _i, _i]),
    'impflow_wgrad_simt': (_i, [_c_fp, _ll, _c_fp, _ll, _c_fp, _ll, _ll, _i, _i, _c_fp, _c_fp]),
    'impflow_gemm_nt_tc': (_i, [_c_fp, _c_fp, _ll, _c_fp, _c_fp, _ll, _c_fp, _c_fp, _c_fp, _c_fp, _c_fp, _c_fp,
                                _ll, _ll, _i, _i, _i, _c_fp, _c_fp, _c_fp]),
    'impflow_branch3_tc': (_i, [_c_fp, _ll] + [_c_fp] * 13 + [_ll, _ll, _i, _i, _i, _c_fp, _c_fp, _c_fp]),
    'impflow_chain23_parts': (_i, [_i]),
    'impflow_chain23_tc': (_i, [_c_fp, _c_fp, _ll] + [_c_fp] * 8 + [_ll, _ll, _ll, _i, _i, _i, _c_fp, _c_fp]),
    'impflow_conv3_set_chain23': (_i, [_i]),
    'impflow_conv3_set_chain23_a32': (_i, [_i]),
    'impflow_conv3_workspace_floats': (ctypes.c_size_t, [_i] * 6),
    'impflow_conv3_forward': (_i, [_c_fp] * 6),
    'impflow_conv3_prepare_vjp': (_i, [_c_fp] * 6),
    'impflow_conv3_vjp': (_i, [_c_fp] * 7),
    'impflow_conv3_power_series': (_i, [_c_fp] * 6 + [_i, _c_fp, _c_fp, _c_fp, _c_fp]),
    'impflow_conv3_broyden_host_bytes': (ctypes.c_size_t, [_i]),
    'impflow_conv3_set_runahead': (_i, [_i]),
    'impflow_conv3_set_chain_fuse': (_i, [_i]),
    'impflow_conv3_broyden': (_i, [_c_fp, _i] + [_c_fp] * 17 + [_i, _d, _c_fp]),
    'impflow_conv3_fixed_point_host_bytes': (ctypes.c_size_t, [_i]),
    'impflow_conv3_fixed_point': (_i, [_c_fp] * 8 + [_f, _f, _i, _c_fp]),
    'impflow_wgrad_set_slice_major': (_i, [_i]),
    'impflow_wgrad_tc_workspace_floats': (ctypes.c_size_t, [_ll, _i, _i]),
    'impflow_wgrad_tc': (_i, [_c_fp, _c_fp, _ll, _c_fp, _c_fp, _ll, _c_fp, _ll, _i, _ll, _i, _i, _c_fp, _c_fp]),
    'impflow_gemm_tc_splits': (_i, [_ll, _i, _i]),
    'impflow_gemm_tc_set_tma_store': (_i, [_i]),
    'impflow_gemm_tc_set_pair': (_i, [_i]),
    'impflow_set_pdl': (_i, [_i]),
    'impflow_split_tf32': (_i, [_c_fp, _c_fp, _c_fp, _ll, _c_fp]),
    'impflow_prep_weights': (_i, [_c_fp, _c_fp, _f, _i, _i, _i, _c_fp, _c_fp, _c_fp, _i, _i, _c_fp, _c_fp, _c_fp, _i, _i,
                                  _c_fp]),
    'impflow_sn_scale': (_i, [_c_fp, _c_fp, _f, _c_fp, _c_fp, _ll, _c_fp]),
    'impflow_sn_scale_grad': (_i, [_c_fp, _c_fp, _c_fp, _c_fp, _f, _c_fp, _ll, _c_fp]),
    'impflow_sn_scale_grad_layout': (_i, [_c_fp, _ll, _c_fp, _c_fp, _c_fp, _f, _i, _i, _i, _c_fp, _c_fp, _c_fp]),
    'impflow_prep_weights_lop': (_i, [_c_fp, _c_fp, _i, _f, _i, _i, _i, _c_fp, _c_fp, _c_fp, _i, _i, _c_fp, _c_fp,
                                      _c_fp, _i, _i, _c_fp]),
    'impflow_lop_norms': (_i, [_c_fp, _i, _i, _i, _i, _i, _c_fp, _c_fp, _c_fp]),
    'impflow_lop_scale_grad_layout': (_i, [_c_fp, _ll, _c_fp, _c_fp, _f, _i, _i, _i, _i, _i, _i, _c_fp, _c_fp,
                                           _c_fp]),
    'impflow_sn_conv_set_ctas': (_i, [_i]),
    'impflow_sn_conv_workspace_floats': (ctypes.c_size_t, [_i, _i, _i, _i]),
    'impflow_sn_power_iter_conv3x3': (_i, [_c_fp] * 5 + [_i, _i, _i, _i, _i, _f, _f, _c_fp, _c_fp, _c_fp]),
    'impflow_sn_power_iter_batch': (_i, [_c_fp, _i, _i, _i, _i, _f, _f, _c_fp]),
    'impflow_sn_power_iter': (_i, [_c_fp, _c_fp, _c_fp, _c_fp, _c_fp, _i, _i, _i, _f, _f, _c_fp]),
}



class SnDesc(ctypes.Structure):
    """impflow_sn_desc of include/impflow_b200.h (48 bytes)."""
    _fields_ = [('W', ctypes.c_void_p), ('u', ctypes.c_void_p), ('v', ctypes.c_void_p), ('sigma', ctypes.c_void_p),
                ('iters', ctypes.c_void_p), ('out_f', ctypes.c_int32), ('in_f', ctypes.c_int32)]


class Conv3Plan(ctypes.Structure):
    """impflow_conv3_plan of include/impflow_b200.h."""
    _fields_ = ([(n, ctypes.c_int32) for n in ('B', 'H', 'W', 'c', 'C', 'k0', 'act_kind', 'act0_kind', 'allow_fused',
                                               'reserved')] +
                [(n, ctypes.c_void_p) for n in ('beta0', 'beta1', 'beta2', 'W1f_hi', 'W1f_lo', 'W2f_hi', 'W2f_lo',
                                                'W3f_hi', 'W3f_lo', 'b1', 'b2', 'b3', 'W3b_hi', 'W3b_lo', 'W2b_hi',
                                                'W2b_lo', 'W1b_hi', 'W1b_lo', 'ws')])


_lib = None


def load():
    """Load (once) and type the shared library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError('libimpflow_b200.so is not built: run `python -c "import __graft_entry__ as g; g.build()"` '
                          '(there is no CPU / PyTorch fallback for the ImpFlow hot path)')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            continue   # test_cabi checks the export list against the header
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().impflow_last_error().decode()


def check(rc, what):
    if rc != 0:
        raise RuntimeError('%s failed (%d): %s' % (what, rc, last_error()))


def require_device(t, what='tensor'):
    """The product has no CPU execution path: every tensor handed to a kernel must be on a GPU."""
    if not t.is_cuda:
        raise RuntimeError('impflow_b200: %s must be a CUDA tensor (no CPU fallback exists for this path)' % what)


def pinned_bytes(n):
    return torch.zeros(n, dtype=torch.uint8).pin_memory()


def sync_stream():
    torch.cuda.current_stream().synchronize()


_F32 = torch.float32
_CHECK_DEVICE = [True]      # the CPU test-suite's C-ABI emulator switches the device check off (tests/cabi_emulator.py)


def ptr(t, name='tensor', allow_none=False):
    """Device pointer (int) of a dense fp32 CUDA tensor (memory order is the caller's business).  This sits on
    every kernel launch (~10 arguments each, thousands of launches per step), so it is kept to two attribute
    checks."""
    if t is None:
        if allow_none:
            return None
        raise ValueError('%s is None' % name)
    if t.dtype is not _F32:
        raise RuntimeError('impflow_b200: %s must be float32, got %s' % (name, t.dtype))
    if _CHECK_DEVICE[0] and not t.is_cuda:
        require_device(t, name)
    return t.data_ptr()


def iptr(t):
    if t is None:
        return None
    require_device(t, 'int tensor')
    return ctypes.c_void_p(t.data_ptr())


def stream():
    """Raw cudaStream_t of torch's current stream (the C-level getter: ~0.3 us instead of the
    ~15 us of torch.cuda.current_stream(), which matters at thousands of launches per step)."""
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


def launch_count():
    return int(load().impflow_launch_count())
