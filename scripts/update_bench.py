"""k_update (csrc/broyden.cu): for each shape, n iterations of impflow_broyden_step on fixed random residuals, timed
back to back (CUDA events between the iterations) and reported as a fraction of the HBM bandwidth.
Usage: python scripts/update_bench.py [B d n_iter] ...   (default: the classifier and bench shapes)"""
import ctypes
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import impflow_b200 as pkg                                   # noqa: E402
from impflow_b200.layers import broyden as _b                # noqa: E402


def run(B, d, T, n_iter, seed=0):
    cabi = pkg._cabi
    lib = cabi.load()
    dev = torch.device('cuda')
    gen = torch.Generator(device='cuda').manual_seed(seed)
    wk = _b._workspace(B, d, T, dev)
    wk.Ut.zero_()
    wk.Vt.zero_()
    gs = [torch.randn(B, d, device=dev, generator=gen) for _ in range(n_iter + 1)]
    wk.xa.copy_(torch.randn(B, d, device=dev, generator=gen))
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    cabi.check(lib.impflow_broyden_begin(vp(wk.xa), vp(gs[0]), vp(wk.xb), vp(wk.low_x), vp(wk.low_g), vp(wk.sample_sq),
                                         vp(wk.low_sq), vp(wk.partial), vp(wk.state), B, d, T, 1e-30, cabi.stream()),
               'begin')
    x_old, xn = wk.xa, wk.xb
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_iter + 1)]
    # back to back, as in the sync-free solver loop: the host runs ahead, the events sit between the iterations on the
    # stream; nothing is flushed (a 2 GB history exceeds L2 by itself, the iterate / residual vectors were just
    # written, as they are when a branch evaluation precedes the step)
    torch.cuda.synchronize()
    torch.cuda._sleep(2000000)            # keep the device busy while the host enqueues
    evs[0].record()
    for i in range(1, n_iter + 1):
        g_old, gn = gs[i - 1], gs[i]
        cabi.check(lib.impflow_broyden_step(vp(x_old), vp(g_old), vp(xn), vp(gn), vp(wk.Ut), vp(wk.Vt), vp(wk.low_x),
                                            vp(wk.low_g), vp(wk.sample_sq), vp(wk.low_sq), vp(wk.partial),
                                            vp(wk.state), B, d, T, cabi.stream()), 'step')
        evs[i].record()
        x_old, xn = xn, x_old
    torch.cuda.synchronize()
    return [evs[i - 1].elapsed_time(evs[i]) * 1e3 for i in range(1, n_iter + 1)]


def main():
    shapes = [(128, 65536, 15), (128, 16384, 15), (64, 3072, 15)]
    if len(sys.argv) > 3:
        a = [int(t) for t in sys.argv[1:]]
        shapes = [tuple(a[i:i + 3]) for i in range(0, len(a), 3)]
    hbm = 6543.1
    for B, d, n in shapes:
        run(B, d, 30, 2)          # warm-up
        times = run(B, d, 30, n)
        alg = [(6 + 2 * i) * d * 4.0 * B for i in range(1, n + 1)]
        frac = [a / (t * 1e-6) / 1e9 / hbm for a, t in zip(alg, times)]
        tot = sum(alg) / (sum(times) * 1e-6) / 1e9 / hbm
        print('B=%d d=%d back-to-back  us/iter: %s  frac@i=1,4,8,%d: %.2f %.2f %.2f %.2f  overall %.3f'
              % (B, d, ' '.join('%.0f' % t for t in times), n, frac[0], frac[3], frac[min(7, n - 1)], frac[-1], tot),
              flush=True)
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
