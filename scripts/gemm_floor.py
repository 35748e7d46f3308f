import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import impflow_b200 as p
ops = p.ops
ops.set_gemm_backend('tc')
def t(M, N, K, reps=50, **kw):
    A = torch.randn(M, K, device='cuda'); B = torch.randn(N, K, device='cuda')
    As, Bs = ops.split_tf32(A), ops.split_tf32(B)
    lib = p._cabi.load(); st = p._cabi.stream()
    pre = torch.empty(M, N, device='cuda')
    def f():
        p._cabi.check(lib.impflow_gemm_nt_tc(As[0].data_ptr(), As[1].data_ptr(), K, Bs[0].data_ptr(), Bs[1].data_ptr(), K, None, pre.data_ptr(), None, None, None, None, N, M, N, K, 0, None, None, st), 'g')
    f(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): f()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3
for shp in [(128, 128, 32), (128, 256, 512), (4096, 512, 512), (16384, 512, 128), (16384, 512, 512), (16384, 128, 512), (18944, 256, 32), (18944, 256, 512)]:
    print(shp, '%.1f us back-to-back (warm L2)' % t(*shp))
