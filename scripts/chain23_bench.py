"""Micro-benchmark of the fused layer-2+3 kernel (csrc/chain23_fused.cu) at the CIFAR scale-1 / scale-2 shapes, next
to the two unfused tcgen05 GEMMs it replaces (CUDA events, L2 flushed).  `python scripts/chain23_bench.py [a32]`."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import impflow_b200 as pkg  # noqa: E402

ops = pkg.ops
dev = torch.device('cuda')
flush = torch.empty(64 * 1024 * 1024, device=dev)


def timeit(fn, reps=7):
    ts = []
    for i in range(reps + 1):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i:
            ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


A32 = 'a32' in sys.argv[1:]          # layer-2 input as one fp32 plane, split on chip
for M, C, N3 in [(16384, 512, 108), (4096, 512, 432)]:
    A = torch.randn(M, C, device=dev)
    if not A32:
        A = ops.split_tf32(A)
    W2 = ops.split_tf32(torch.randn(C, C, device=dev) / 22)
    W3 = ops.split_tf32(torch.randn(N3, C, device=dev) / 22)
    b2 = torch.randn(C, device=dev)
    beta = torch.full((1,), 0.97, device=dev)
    m2 = torch.randn(M, C, device=dev)
    flop = 2.0 * M * (C * C + C * N3)
    for tag, fn in [
        ('fwd (act)', lambda: ops.chain23_tc(A, W2, W3, N3, bias2=b2, act_kind=ops.ACT_LIPSWISH, beta2=beta)),
        ('fwd (act, save pre)', lambda: ops.chain23_tc(A, W2, W3, N3, bias2=b2, act_kind=ops.ACT_LIPSWISH, beta2=beta,
                                                       save_pre=True)),
        ('vjp (mul)', lambda: ops.chain23_tc(A, W2, W3, N3, mul2=m2)),
    ]:
        t = timeit(fn)
        print('chain23 M=%5d N3=%3d %-20s: %7.1f us  %6.1f TFLOP/s (fp32-equivalent)' % (M, N3, tag, t * 1e3,
                                                                                       flop / t / 1e9))
    # the two GEMMs it replaces: layer 2 with the split epilogue, layer 3 plain
    key2 = (M, C, C, False, False, False, True, False)
    key3 = (M, N3, C, True, False, False, False, False)
    t2, t3 = ops.time_gemm_shape(key2, reps=5, flush=flush), ops.time_gemm_shape(key3, reps=5, flush=flush)
    print('two GEMMs  M=%5d N3=%3d                     : %7.1f + %.1f us  %6.1f TFLOP/s' % (M, N3, t2 * 1e3, t3 * 1e3,
                                                                                         flop / (t2 + t3) / 1e9))
