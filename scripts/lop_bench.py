"""Train-step time of the CIFAR-shape flow and the POWER-shape tabular flow with vnorms '2222' (every layer an
induced 2 -> 2 layer) and '122f' (first and last layer of every branch a closed-form operator-norm Lop layer), through
the package's public API only.  One JSON line per configuration: median and quartiles of the step time over --steps
steps after --warmup, and the card with its power limit.

    python scripts/lop_bench.py [--tree PATH] [--steps 20] [--warmup 5] [--only cifar-122f,...]

--tree imports the package from another checkout (e.g. the parent commit) so that two trees can be timed alternately
in one session."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

INF = float('inf')


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--tree', default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--only', default='cifar-2222,cifar-122f,power-2222,power-122f')
    ap.add_argument('--label', default='')
    return ap.parse_args()


def cifar_flow(pkg, vnorms, batch):
    """bench.py's CIFAR line (run_cifar10.sh: blocks 2-2-2, idim 512, k 3-1-3, LipSwish, 10 exact terms)."""
    return pkg.ImplicitFlow(
        (batch, 3, 32, 32), n_blocks=[2, 2, 2], intermediate_dim=512, factor_out=False, quadratic=False,
        init_layer=pkg.layers.LogitTransform(0.05), actnorm=True, fc_actnorm=False, batchnorm=False, dropout=0.,
        fc=False, coeff=0.9, vnorms=vnorms, n_lipschitz_iters=None, sn_atol=1e-3, sn_rtol=1e-3, n_power_series=None,
        n_dist='poisson', n_samples=1, kernels='3-1-3', activation_fn='swish', fc_end=False, fc_idim=128,
        n_exact_terms=10, preact=True, neumann_grad=True, grad_in_forward=True, first_resblock=True, learn_p=False,
        classification=False, classification_hdim=256, n_classes=10)


def power_flow(pkg, vnorms, d=6, hidden=(128,) * 4, n_blocks=20, scale_last=True):
    """train_tabular.py's POWER configuration: 20 imBlocks over Sin MLP branches d -> 128 x 4 -> d; layer i maps
    vnorms[i] -> vnorms[i + 1] (the last layer vnorms[-2] -> vnorms[-1]), as the script's build_nnet does.
    scale_last: move the zero-initialised last layers away from zero as bench.py does (else the flow is the
    identity)."""
    layers = pkg.layers
    norm = {'1': 1, '2': 2, 'f': INF}
    doms, cods = [norm[c] for c in vnorms[:-1]], [norm[c] for c in vnorms[1:]]
    dims = [d] + list(hidden) + [d]

    def net():
        mods = []
        for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
            j = min(i, len(doms) - 1) if i < len(dims) - 2 else -1
            if i > 0:
                mods.append(layers.base.Sin())
            mods.append(layers.base.get_linear(a, b, coeff=0.99, n_iterations=None, atol=1e-3, rtol=1e-3,
                                               domain=doms[j], codomain=cods[j], zero_init=(b == d)))
        return torch.nn.Sequential(*mods)
    blocks = [layers.imBlock(net(), net(), n_dist='geometric', n_power_series=None, exact_trace=False,
                             brute_force=False, n_samples=1, n_exact_terms=2, neumann_grad=False,
                             grad_in_forward=False, eps_forward=1e-5) for _ in range(n_blocks)]
    flow = layers.SequentialFlow(blocks)
    with torch.no_grad():
        for n_, p_ in flow.named_parameters():
            if scale_last and n_.endswith('weight') and p_.dim() == 2 and p_.shape[0] == d:
                p_.mul_(30.0)
    return flow


def normal_logprob(z):
    return -0.5 * (math.log(2 * math.pi) + z.pow(2))


def time_config(pkg, name, steps, warmup):
    workload, vnorms = name.split('-')
    dev = torch.device('cuda')
    torch.manual_seed(0)
    np.random.seed(0)
    gen = torch.Generator().manual_seed(1234)
    if workload == 'cifar':
        batch = 64
        model = cifar_flow(pkg, vnorms, batch).to(dev)
        x = torch.rand(batch, 3, 32, 32, generator=gen).to(dev)
        with torch.no_grad():
            model(x, restore=True)
        n_dims = 3 * 32 * 32

        def loss_fn():
            z, dlogp = model(x, 0)
            logpx = normal_logprob(z).reshape(batch, -1).sum(1, keepdim=True) - dlogp - math.log(256) * n_dims
            return -logpx.mean() / n_dims / math.log(2)
    else:
        batch = 1000
        model = power_flow(pkg, vnorms).to(dev)
        x = torch.randn(batch, 6, generator=gen).to(dev)
        with torch.no_grad():
            model(x)

        def loss_fn():
            z, dlogp = model(x, torch.zeros(batch, 1, device=dev))
            return -(normal_logprob(z).sum(1, keepdim=True) - dlogp).mean()
    model.train()
    params = [p for p in model.parameters() if p.requires_grad]
    bucket = pkg.parallel.FlatGradBucket(params)
    opt = pkg.optim.FusedAdam(params, lr=1e-3, betas=(0.9, 0.99), bucket=bucket, max_grad_norm=1., ema_decay=0.999)
    kinds = sorted({type(m).__name__ for m in model.modules() if 'Lop' in type(m).__name__ or 'InducedNorm' in
                    type(m).__name__})

    def step():
        bucket.zero()
        loss = loss_fn()
        loss.backward()
        opt.step()
        pkg.layers.base.update_lipschitz(model, None)
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        loss = step()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    q = np.percentile(times, [25, 50, 75])
    return {'config': name, 'batch': batch, 'layers': kinds, 'steps': steps, 'warmup': warmup,
            'ms_p25': round(float(q[0]), 2), 'ms_median': round(float(q[1]), 2), 'ms_p75': round(float(q[2]), 2),
            'samples_per_s': round(batch * 1e3 / float(q[1]), 1), 'loss': float(loss)}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        out = 'unknown'
    return {'gpu': name, 'power_limit,max_sm_clock': out}


if __name__ == '__main__':
    args = parse()
    sys.path.insert(0, os.path.abspath(args.tree))
    sys.dont_write_bytecode = True
    import impflow_b200 as pkg
    if not torch.cuda.is_available():
        raise SystemExit('lop_bench.py times the GPU: no CUDA device')
    info = card()
    for name in args.only.split(','):
        r = time_config(pkg, name, args.steps, args.warmup)
        r.update(info)
        r['tree'] = args.label or os.path.abspath(args.tree)
        print(json.dumps(r), flush=True)
