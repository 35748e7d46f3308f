"""iResBlock.inverse (the Banach fixed-point loop of iresblock.py:69-79) through the one-call solves of
BranchProgram.fixed_point (impflow_conv3_fixed_point / impflow_mlp_fixed_point) against the host loop over the
branch's forward (find_fixed_point, one stream drain per iteration), alternating the two in one run.

Shapes: the CIFAR ResidualFlow branch (3-1-3, idim 512, LipSwish, B = 64) at each of its three scales, the tabular
POWER (d = 6) and BSDS300 (d = 63) MLP branches (Sin, 4 x 128 hidden, B = 1000) and the toy branch (d = 2, 2 x 128,
B = 5000).  The per-layer bounds are raised above the recipes' (conv 3.0, MLP 2.0 instead of 0.9 / 0.99 on random,
untrained weights) so that each inverse takes a few to a few tens of iterations, as trained blocks do; the figure that
carries over between branches is ms per iteration, i.e. per branch evaluation (iterations + 1 of them per solve).
Every timed call ends in a device synchronise.
Usage: python scripts/fixed_point_bench.py [--reps N] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import impflow_b200 as pkg                                    # noqa: E402
from impflow_b200 import branch_program as bp                 # noqa: E402
from impflow_b200.layers import implicit_block as ib          # noqa: E402

SHAPES = [
    ('cifar-scale0', dict(kind='conv', c=3, hw=32, B=64)),
    ('cifar-scale1', dict(kind='conv', c=12, hw=16, B=64)),
    ('cifar-scale2', dict(kind='conv', c=48, hw=8, B=64)),
    ('power', dict(kind='mlp', d=6, hidden=[128] * 4, B=1000)),
    ('bsds300', dict(kind='mlp', d=63, hidden=[128] * 4, B=1000)),
    ('toy', dict(kind='mlp', d=2, hidden=[128] * 2, B=5000)),
]
CONV_COEFF, MLP_COEFF = 3.0, 2.0


def block(spec):
    L = pkg.layers.base
    torch.manual_seed(0)
    if spec['kind'] == 'conv':
        c = spec['c']
        mk = lambda a, b, k: L.get_conv2d(a, b, k, 1, k // 2, coeff=CONV_COEFF, n_iterations=None, domain=2,
                                          codomain=2, atol=1e-3, rtol=1e-3)
        net = torch.nn.Sequential(L.Swish(), mk(c, 512, 3), L.Swish(), mk(512, 512, 1), L.Swish(), mk(512, c, 3))
        x = torch.rand(spec['B'], c, spec['hw'], spec['hw'])
    else:
        dims = [spec['d']] + spec['hidden'] + [spec['d']]
        mods = []
        for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
            if i > 0:
                mods.append(L.Sin())
            mods.append(L.get_linear(a, b, coeff=MLP_COEFF, n_iterations=None, atol=1e-3, rtol=1e-3, domain=2,
                                     codomain=2))
        net = torch.nn.Sequential(*mods)
        x = torch.randn(spec['B'], spec['d'])
    blk = pkg.layers.iResBlock(net).cuda().eval()
    x = x.cuda()
    with torch.no_grad():
        blk(x)                                    # lazy u / v shaping
        for n, p in net.named_parameters():
            if n.endswith('weight'):
                p.mul_(10.0)
        L.update_lipschitz(net)
        y = blk(x)
    return blk, y


def host_loop(prog, rhs, start, atol, rtol, threshold):
    return ib.find_fixed_point(lambda x: pkg.ops.lincomb3(rhs, 1.0, prog.forward(x), -1.0), start, threshold, atol,
                               rtol)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, limit = [t.strip() for t in q[0].split(',')]
        return name, limit
    except Exception as e:          # the numbers are still printed; the card line says why it is missing
        return 'unknown (%s)' % e, 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'fixed_point_bench needs a GPU'
    name, limit = card()
    lines = ['# scripts/fixed_point_bench.py --reps %d' % args.reps,
             '# card: %s, power limit %s; torch %s' % (name, limit, torch.__version__),
             '# median over %d alternating reps; ms per solve / per iteration = host clock around the call + a device '
             'synchronise' % args.reps]
    rows = []
    native_fp = bp.BranchProgram.fixed_point
    for label, spec in SHAPES:
        blk, y = block(spec)
        prog = ib._program(blk.nnet)
        with torch.no_grad():
            for _ in range(2):                                   # warm both paths
                x_new = blk.inverse(y)
                n_new = blk.inverse_iterations
                bp.BranchProgram.fixed_point = host_loop
                try:
                    x_host = blk.inverse(y)
                    n_host = blk.inverse_iterations
                finally:
                    bp.BranchProgram.fixed_point = native_fp
            t_new, t_host = [], []
            for _ in range(args.reps):
                t, _ = timed(lambda: blk.inverse(y))
                t_new.append(t)
                bp.BranchProgram.fixed_point = host_loop
                try:
                    t, _ = timed(lambda: blk.inverse(y))
                finally:
                    bp.BranchProgram.fixed_point = native_fp
                t_host.append(t)
        one_call = (prog.native_plan(y) is not None) if spec['kind'] == 'conv' else \
            (prog.mlp_solver_spec(y) is not None)
        diff = float((x_new - x_host).abs().max() / x_host.abs().max().clamp_min(1e-30))
        agree = n_new == n_host and (bool(torch.equal(x_new, x_host)) if spec['kind'] == 'conv' else diff <= 1e-6)
        med = lambda v: sorted(v)[len(v) // 2]
        row = dict(shape=label, B=spec['B'], one_call=one_call, iterations=n_new, iterations_host=n_host,
                   ms_one_call=round(med(t_new), 3), ms_host_loop=round(med(t_host), 3),
                   ms_per_iter_one_call=round(med(t_new) / (n_new + 1), 4),
                   ms_per_iter_host_loop=round(med(t_host) / (n_host + 1), 4),
                   speedup=round(med(t_host) / med(t_new), 2), agree=agree, max_rel_diff=diff)
        rows.append(row)
        lines.append(json.dumps(row))
    text = '\n'.join(lines) + '\n'
    sys.stdout.write(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text)
    if not all(r['agree'] for r in rows):
        sys.exit(1)


if __name__ == '__main__':
    main()
