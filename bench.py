#!/usr/bin/env python
"""bench.py — ImpFlow hot-path benchmark (contract in the task brief, tier section ④).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W     # the reference algorithm on host cores

A "step" is one training step of the CIFAR-10-shape ImplicitFlow of run_cifar10.sh
(train_img.py:591-660): forward (6 imBlocks: Broyden solve + power-series log-det), bits/dim,
backward (implicit-differentiation Broyden solves), gradient all-reduce (N>1), clip, Adam,
update_lipschitz — on synthetic U[0,1) images (SURVEY.md §8d) with random-init weights.

Other configurations of BASELINE.json (`--workload`): toy / tabular-* (train_toy.py, train_tabular.py MLP flows),
classifier (train_classification.py ImplicitResNet18, solver + spectral-norm path, no log-det).
`--scaling strong` keeps the GLOBAL batch at the workload's batch and shards it over the ranks.

The reference arm (`--impl reference`, and the `cpu_baseline` key of this repo's line) runs the UNMODIFIED
reference from oracle/_ref (bytecode compiled by oracle/build_ref.py) on the host cores when it is present
(`kind: "reference"`), else the oracle port (`kind: "port"`); its config line states the batch it really ran.
"""
import argparse
import atexit
import contextlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: no bytecode caches next to the sources

METRIC = 'impflow_train_samples_per_sec'
UNIT = 'samples/s'
WORKLOADS = {
    # run_cifar10.sh:1-3 + train_img.py defaults
    'cifar': dict(input=(3, 32, 32), n_blocks=[2, 2, 2], idim=512, batch=64, n_exact_terms=10, coeff=0.9),
    # reduced-width debug variant (not a bench line)
    'cifar-small': dict(input=(3, 32, 32), n_blocks=[1, 1, 1], idim=64, batch=16, n_exact_terms=4, coeff=0.9),
    # run_tabular.sh / run_toy.sh shapes (parity-test configs; selectable, never the default bench line)
    'tabular-power': dict(kind='mlp', d=6, hidden=[128] * 4, n_blocks=20, batch=1000, coeff=0.99, sn_tol=1e-3,
                          n_lipschitz_iters=None, brute_force=False, eps_forward=1e-5),
    'tabular-miniboone': dict(kind='mlp', d=43, hidden=[128] * 4, n_blocks=20, batch=1000, coeff=0.99, sn_tol=1e-3,
                              n_lipschitz_iters=None, brute_force=False, eps_forward=1e-5),
    'tabular-bsds300': dict(kind='mlp', d=63, hidden=[128] * 4, n_blocks=20, batch=1000, coeff=0.99, sn_tol=1e-3,
                            n_lipschitz_iters=None, brute_force=False, eps_forward=1e-5),
    'toy': dict(kind='mlp', d=2, hidden=[128] * 2, n_blocks=6, batch=5000, coeff=0.99, sn_tol=None,
                n_lipschitz_iters=20, brute_force=True, eps_forward=1e-6),
    # run_classification.sh + train_classification.py:135-282: ImplicitResNet18, 4 imBlocks of 3x3-ReLU-3x3-ReLU
    # conv branches on (64ch,32x32), (64,32x32), (128,16x16), (256,8x8): d = 65536 / 65536 / 32768 / 16384, no log-det
    'classifier': dict(kind='cls', input=(3, 32, 32), batch=128, coeff=0.9, n_classes=100),
}
WORKLOAD_TEXT = {
    'cifar': 'cifar10-shape ImplicitFlow train step (run_cifar10.sh: nblocks 2-2-2, idim 512, k3-1-3, LipSwish, '
             '10 exact terms, Neumann grad, mem-eff)',
    'classifier': 'ImplicitResNet18 train step (run_classification.sh: 4 conv imBlocks, ReLU, coeff 0.9, '
                  'cross-entropy, no log-det)',
}


def std_normal_logprob(z):
    return -0.5 * np.log(2 * np.pi) - z.pow(2) / 2


def build_classifier(pkg, wl):
    """ImplicitResNet18 of train_classification.py:135-282 on the given layers namespace (this repo's package
    or the reference): conv stem, four BasicImplicitBlocks (imBlock over two 3x3-ReLU-3x3-ReLU induced-norm conv
    branches, then a strided 1x1 conv + BatchNorm + ReLU downsample), average pool, linear head."""
    import torch.nn as nn
    import torch.nn.functional as F
    layers = pkg.layers
    coeff = wl['coeff']

    class BasicImplicitBlock(nn.Module):
        def __init__(self, in_planes, hidden, planes, stride):
            super(BasicImplicitBlock, self).__init__()
            self.initialized = False
            conv = lambda a, b: layers.base.get_conv2d(a, b, kernel_size=3, stride=1, padding=1, bias=False,
                                                       coeff=coeff, n_iterations=None, domain=2, codomain=2,
                                                       atol=1e-3, rtol=1e-3)
            net = lambda: nn.Sequential(conv(in_planes, hidden), nn.ReLU(), conv(hidden, in_planes), nn.ReLU())
            self.block = layers.imBlock(net(), net())
            self.downsample = nn.Sequential()
            if stride != 1 or in_planes != planes:
                self.downsample = nn.Sequential(nn.Conv2d(in_planes, planes, kernel_size=1, stride=stride, bias=False),
                                                nn.BatchNorm2d(planes), nn.ReLU())

        def forward(self, x):
            out = self.block(x) if self.initialized else self.block(x, restore=True)
            self.initialized = True
            return self.downsample(out)

    class ImplicitResNet18(nn.Module):
        def __init__(self, num_classes):
            super(ImplicitResNet18, self).__init__()
            self.conv1 = nn.Conv2d(3, 64, kernel_size=3, stride=1, padding=1, bias=False)
            self.bn1 = nn.BatchNorm2d(64)
            self.layer1 = nn.Sequential(BasicImplicitBlock(64, 64, 64, 1))
            self.layer2 = nn.Sequential(BasicImplicitBlock(64, 128, 128, 2))
            self.layer3 = nn.Sequential(BasicImplicitBlock(128, 256, 256, 2))
            self.layer4 = nn.Sequential(BasicImplicitBlock(256, 512, 512, 2))
            self.linear = nn.Linear(512, num_classes)

        def forward(self, x, restore=False):
            out = F.relu(self.bn1(self.conv1(x)))
            out = self.layer4(self.layer3(self.layer2(self.layer1(out))))
            out = F.avg_pool2d(out, 4)
            return self.linear(out.view(out.size(0), -1))
    return ImplicitResNet18(wl['n_classes'])


def build_mlp_flow(pkg, wl):
    """train_tabular.py:292-336 / train_toy.py:146-171,224-242: n imBlocks over Sin MLP branches."""
    layers = pkg.layers
    d = wl['d']
    dims = [d] + list(wl['hidden']) + [d]

    def net():
        mods = []
        for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
            if i > 0:
                mods.append(layers.base.Sin())
            mods.append(layers.base.get_linear(a, b, coeff=wl['coeff'], n_iterations=wl['n_lipschitz_iters'],
                                               atol=wl['sn_tol'], rtol=wl['sn_tol'], domain=2, codomain=2,
                                               zero_init=(b == d)))
        return torch.nn.Sequential(*mods)
    blocks = [layers.imBlock(net(), net(), n_dist='geometric', n_power_series=None, exact_trace=False,
                             brute_force=wl['brute_force'], n_samples=1, n_exact_terms=2, neumann_grad=False,
                             grad_in_forward=False, eps_forward=wl['eps_forward']) for _ in range(wl['n_blocks'])]
    return layers.SequentialFlow(blocks)


def build_model(pkg, wl, batch):
    if wl.get('kind') == 'mlp':
        return build_mlp_flow(pkg, wl)
    if wl.get('kind') == 'cls':
        return build_classifier(pkg, wl)
    layers = pkg.layers
    c, h, w = wl['input']
    return pkg.ImplicitFlow(
        (batch, c, h, w), n_blocks=wl['n_blocks'], intermediate_dim=wl['idim'], factor_out=False, quadratic=False,
        init_layer=layers.LogitTransform(0.05), actnorm=True, fc_actnorm=False, batchnorm=False, dropout=0.,
        fc=False, coeff=wl['coeff'], vnorms='2222', n_lipschitz_iters=None, sn_atol=1e-3, sn_rtol=1e-3,
        n_power_series=None, n_dist='poisson', n_samples=1, kernels='3-1-3', activation_fn='swish', fc_end=False,
        fc_idim=128, n_exact_terms=wl['n_exact_terms'], preact=True, neumann_grad=True, grad_in_forward=True,
        first_resblock=True, learn_p=False, classification=False, classification_hdim=256, n_classes=10)


def update_lipschitz(pkg, model, n_iterations=None):
    """train_img.py:786-792 (train_toy.py:174-179 with n_iterations): power-iteration refresh of every
    induced-norm layer after the optimiser step; the package fans the independent layers out over side
    streams (the frozen *_copy twins are skipped, SURVEY.md quirk #11)."""
    pkg.layers.base.update_lipschitz(model, n_iterations)


class ClockSampler(object):
    """`nvidia-smi -lms 400` next to the benchmark.  The process is started BEFORE the warm-up steps: its start-up (NVML
    initialisation) holds driver locks for ~100 ms, which used to land in the first timed steps (per_step_ms showed
    150-300 ms there in one run out of three); only the samples taken between mark_begin() and stop() — the timed region —
    are reported."""
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp')

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix='.csv')
        self.proc = None
        self.gpu = gpu_index
        self.t_begin = None

    def mark_begin(self):
        import datetime
        self.t_begin = datetime.datetime.now()

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.QUERY,
                                          '--format=csv,noheader,nounits', '-lms', '400'],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
            atexit.register(self._reap)         # also when the run fails before stop(): no poller outlives it
        except Exception:
            self.proc = None

    def _reap(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.kill()
            self.proc.wait()

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        import datetime
        rows = []
        try:
            for line in open(self.path):
                f = [t.strip() for t in line.split(',')]
                if len(f) < 9:
                    continue
                try:
                    row = [float(f[1]), float(f[2])]
                except ValueError:
                    continue
                ts = None
                if len(f) >= 10:
                    try:
                        ts = datetime.datetime.strptime(f[9], '%Y/%m/%d %H:%M:%S.%f')
                    except ValueError:
                        ts = None
                rs = [name for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                                                 'sw_power_cap'), f[5:9]) if val.lower().startswith('active')]
                rows.append((ts, row[0], row[1], rs))
            os.unlink(self.path)
        except Exception:
            pass
        timed = [r for r in rows if self.t_begin is not None and r[0] is not None and r[0] >= self.t_begin]
        window = 'timed region'
        if not timed:           # region shorter than the sampling period (or no timestamps): everything since the start
            timed, window = rows, 'warm-up + timed region'
        if timed:
            out = {'sm_mhz': float(np.median([r[1] for r in timed])), 'sm_max_mhz': float(max(r[2] for r in timed)),
                   'reasons': sorted({n for r in timed for n in r[3]}), 'samples': len(timed), 'window': window}
        return out


def scale_mlp_last_layers(model, wl):
    """The zero-initialised last layers of the MLP branches (zero_init: weights / 1000) make a fresh flow the
    identity; move them away from zero so that the solves and estimators do real work (both arms)."""
    with torch.no_grad():
        for n_, p_ in model.named_parameters():
            if n_.endswith('weight') and p_.dim() == 2 and p_.requires_grad and p_.shape[0] == wl['d']:
                p_.mul_(30.0)


def synthetic_batch(wl, batch, gen):
    """Synthetic inputs of SURVEY.md section 8d: z-scored tabular rows, U[0,1) images (+ uniform labels)."""
    if wl.get('kind') == 'mlp':
        return torch.randn(batch, wl['d'], generator=gen), None
    c, h, w = wl['input']
    y = torch.randint(0, wl['n_classes'], (batch,), generator=gen) if wl.get('kind') == 'cls' else None
    return torch.rand(batch, c, h, w, generator=gen), y


def loss_of(model, wl, x, y, outputs=None):
    """The training objective of the three script families (train_img.py:517-549, train_tabular.py:398-407 /
    train_toy.py:108-116, train_classification.py:357-359).  `outputs`, when given, receives copies of what the model
    returned: the logits, or the latent `z` and the log-determinant `logdet`."""
    kind = wl.get('kind')
    if kind == 'cls':
        logits = model(x)
        if outputs is not None:
            outputs['logits'] = logits.detach().clone()
        return torch.nn.functional.cross_entropy(logits, y, reduction='sum')
    if kind == 'mlp':
        z, dlogp = model(x, torch.zeros(x.shape[0], 1, device=x.device))
        if outputs is not None:
            outputs['z'], outputs['logdet'] = z.detach().clone(), dlogp.detach().clone()
        logpz = std_normal_logprob(z).reshape(z.size(0), -1).sum(1, keepdim=True)
        return -(logpz - dlogp).mean()
    n_dims = int(np.prod(wl['input']))
    z, dlogp = model(x, 0)
    if outputs is not None:
        outputs['z'], outputs['logdet'] = z.detach().clone(), dlogp.detach().clone()
    logpz = std_normal_logprob(z).reshape(z.size(0), -1).sum(1, keepdim=True)
    logpx = logpz - dlogp - np.log(256) * n_dims
    return -torch.mean(logpx) / n_dims / np.log(2)


DUMP_BYTES = 64 * 1000 * 1000
DUMP_CAP = {'params': 6000000, 'grads': 6000000}      # elements; every other array: 1000000


def write_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float32 (float64 stays float64).  An array longer than its
    cap is replaced by a sample of its flattened elements at fixed positions (seed 0, so the same positions in every run
    of one configuration, and the same ones in `params` and `grads`); the directory stays under DUMP_BYTES."""
    out = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a if a.dtype == np.float64 else a.astype(np.float32)
        cap = DUMP_CAP.get(name, 1000000)
        if a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        out[name] = a
    assert sum(a.nbytes for a in out.values()) <= DUMP_BYTES - 4096 * len(out)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def run_reference_impl(wl_name, steps, warmup, batch, threads=None):
    """The UNMODIFIED reference (oracle/_ref, compiled from /root/reference by oracle/build_ref.py) on the host
    cores: the reference's own model classes, vendored Adam, EMA and update_lipschitz loop, one training step of
    the named workload per step (train_img.py:591-660 / train_tabular.py:447-500 / train_toy.py:283-297 /
    train_classification.py:352-366) on `batch` synthetic samples."""
    from oracle import ref_runner
    ns = ref_runner.load()
    wl = WORKLOADS[wl_name]
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    np.random.seed(0)
    model = build_model(ns, wl, batch)
    kind = wl.get('kind')
    if kind == 'mlp':
        scale_mlp_last_layers(model, wl)
    x, y = synthetic_batch(wl, batch, torch.Generator().manual_seed(1234))
    with torch.no_grad():
        model(x, restore=True)           # ActNorm data init + lazy u/v shaping (train_img.py:502-507)
    model.train()
    is_toy = wl_name == 'toy'
    opt = ns.optim.Adam(model.parameters(), lr=1e-3, **({} if (is_toy or kind == 'cls') else {'betas': (0.9, 0.99)}))
    ema = None if is_toy else ns.utils.ExponentialMovingAverage(model)
    times, fwd, bwd, loss = [], [], [], None
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        with ref_runner.SolveCounter(ns) as rec:
            loss = loss_of(model, wl, x, y)
            loss.backward()
            if kind != 'cls' and not is_toy:
                torch.nn.utils.clip_grad_norm_(model.parameters(), 1.)
            opt.step()
            opt.zero_grad()
            ref_runner.update_lipschitz(ns, model, wl.get('n_lipschitz_iters'))
            if ema is not None:
                ema.apply()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        fwd, bwd = rec.nsteps('forward'), rec.nsteps('backward')
    ms = float(np.mean(times) * 1e3)
    n_blocks = len(fwd)
    return {'value': batch / (ms / 1e3), 'ms_per_step': ms, 'cores': threads, 'batch': batch, 'bpd': float(loss),
            'fwd_nstep': fwd, 'bwd_nstep': bwd, 'kind': 'reference',
            'solves_per_step': 2 * n_blocks * batch}


def run_cpu_reference(wl_name, steps, warmup, batch, threads=None):
    """CPU arm: the unmodified reference when oracle/_ref is present, else the oracle port of the same step."""
    from oracle import ref_runner
    if ref_runner.available():
        return run_reference_impl(wl_name, steps, warmup, batch, threads)
    if WORKLOADS[wl_name].get('kind') == 'cls':
        raise RuntimeError('the classifier workload has no oracle port; build oracle/_ref (python oracle/build_ref.py)')
    res = run_cpu_port(wl_name, steps, warmup, batch, threads)
    res['kind'] = 'port'
    return res


def run_cpu_port(wl_name, steps, warmup, batch, threads=None):
    """The reference algorithm (oracle port, PyTorch CPU like the reference itself) on host cores."""
    from oracle import flow_oracle
    import impflow_b200 as pkg
    wl = WORKLOADS[wl_name]
    if wl.get('kind') == 'mlp':
        return run_cpu_reference_mlp(pkg, wl, steps, warmup, batch, threads)
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    np.random.seed(0)
    model = build_model(pkg, wl, batch)       # constructor only (CPU): same init path as the product
    sd = model.state_dict()
    c, h, w = wl['input']
    x = torch.rand(batch, c, h, w)
    # lazily shaped conv u/v buffers + data-dependent ActNorm init, as model(x, restore=True) would do
    sd = _host_init_lazy_buffers(sd, wl, x)
    cfg = dict(flow_oracle.CIFAR_CFG, n_exact_terms=wl['n_exact_terms'])
    flow = flow_oracle.OracleFlow(sd, wl['n_blocks'], cfg, coeff=wl['coeff'])
    opt = torch.optim.Adam(flow.params, lr=1e-3, betas=(0.9, 0.99))
    times, stats = [], {}
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        bpd = flow.train_step(x, opt, stats)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    ms = float(np.mean(times) * 1e3)
    return {'value': batch / (ms / 1e3), 'ms_per_step': ms, 'cores': threads, 'batch': batch, 'bpd': bpd,
            'fwd_nstep': stats.get('fwd_nstep', [])[-6:], 'bwd_nstep': stats.get('bwd_nstep', [])[-6:]}


def run_cpu_reference_mlp(pkg, wl, steps, warmup, batch, threads=None):
    """Oracle port of the tabular / toy training step on host cores."""
    from oracle import impflow_oracle as orc
    from tests.helpers import oracle_branch
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    np.random.seed(0)
    model = build_mlp_flow(pkg, wl)
    sd = model.state_dict()
    d = wl['d']
    blocks, params = [], []
    for i in range(wl['n_blocks']):
        sub = lambda pre: {k[len(pre):]: v.clone() for k, v in sd.items() if k.startswith(pre)}
        bx = oracle_branch(sub('chain.%d.nnet_x.' % i), 'sin', wl['coeff'], wl['sn_tol'], wl['n_lipschitz_iters'])
        bz = oracle_branch(sub('chain.%d.nnet_z.' % i), 'sin', wl['coeff'], wl['sn_tol'], wl['n_lipschitz_iters'])
        blocks.append((bx, bz))
        params += bx.parameters() + bz.parameters()
    cfg = dict(orc.DEFAULT_CFG, neumann_grad=False, grad_in_forward=False, eps_forward=wl['eps_forward'],
               brute_force=wl['brute_force'])
    opt = torch.optim.Adam(params, lr=1e-3)
    x = torch.randn(batch, d)
    times, stats = [], {}
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        h, logp = x, torch.zeros(batch, 1)
        for bx, bz in blocks:
            h, logp = orc.imblock_forward(bx, bz, h, logp, cfg, True, stats=stats)
        logpz = (-0.5 * np.log(2 * np.pi) - h.pow(2) / 2).sum(1, keepdim=True)
        loss = -(logpz - logp).mean()
        loss.backward()
        opt.step()
        for bx, bz in blocks:
            bx.update_lipschitz(wl['n_lipschitz_iters'])
            bz.update_lipschitz(wl['n_lipschitz_iters'])
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    ms = float(np.mean(times) * 1e3)
    return {'value': batch / (ms / 1e3), 'ms_per_step': ms, 'cores': threads, 'batch': batch, 'bpd': float(loss),
            'fwd_nstep': stats.get('fwd_nstep', [])[-6:], 'bwd_nstep': stats.get('bwd_nstep', [])[-6:]}


def solver_roofline(pkg, B, d, T, n_iter, flush, hbm_gbs, peak_src):
    """HBM roofline of the Broyden solver algebra (k_norm_decide + k_update, csrc/broyden.cu) at one (B, d):
    n_iter iterations of impflow_broyden_step on random residuals, each timed alone with CUDA events (L2
    flushed).  Algorithmic bytes of iteration i (history rank i-1): (6 + 2i) * d * 4 per sample
    (SURVEY.md section 8d)."""
    import ctypes
    from impflow_b200.layers import broyden as _b
    cabi = pkg._cabi
    lib = cabi.load()
    dev = torch.device('cuda', torch.cuda.current_device())
    wk = _b._workspace(B, d, T, dev)
    g = [torch.randn(B, d, device=dev) for _ in range(2)]
    wk.xa.normal_()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    cabi.check(lib.impflow_broyden_begin(vp(wk.xa), vp(g[0]), vp(wk.xb), vp(wk.low_x), vp(wk.low_g), vp(wk.sample_sq),
                                         vp(wk.low_sq), vp(wk.partial), vp(wk.state), B, d, T, 1e-30, cabi.stream()),
               'broyden_begin')
    x_old, xn, g_old, gn = wk.xa, wk.xb, g[0], g[1]
    t_ms, bytes_alg = 0.0, 0.0
    # a history larger than L2 (classifier shape: 2 GB) needs no flush: the iterations are enqueued back to back as the
    # sync-free solver loop does, one event between them; the iterate / residual vectors were just written, as they
    # are after a branch evaluation.  The bench shape (47 MB of history) is flushed between iterations.
    streamed = 8.0 * B * T * d > 256e6
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_iter + 1)]
    gs = [torch.randn(B, d, device=dev) for _ in range(n_iter)] if streamed else None
    if streamed:
        torch.cuda.synchronize()
        torch.cuda._sleep(2000000)        # the device stays busy while the host enqueues
        evs[0].record()
    for i in range(1, n_iter + 1):
        if streamed:
            gn = gs[i - 1]
        else:
            gn.normal_()
            flush.zero_()
            evs[i - 1].record()
        cabi.check(lib.impflow_broyden_step(vp(x_old), vp(g_old), vp(xn), vp(gn), vp(wk.Ut), vp(wk.Vt), vp(wk.low_x),
                                            vp(wk.low_g), vp(wk.sample_sq), vp(wk.low_sq), vp(wk.partial),
                                            vp(wk.state), B, d, T, cabi.stream()), 'broyden_step')
        evs[i].record()
        if not streamed:
            torch.cuda.synchronize()
            t_ms += evs[i - 1].elapsed_time(evs[i])
        bytes_alg += (6 + 2 * i) * d * 4.0 * B
        if streamed:
            x_old, xn, g_old = xn, x_old, gn
        else:
            x_old, xn, g_old, gn = xn, x_old, gn, g_old
    if streamed:
        torch.cuda.synchronize()
        t_ms = evs[0].elapsed_time(evs[n_iter])
    ach = bytes_alg / (t_ms / 1e3) / 1e9
    return {'kernel': 'k_norm_decide + k_update (Broyden rank-1 update and break rules, csrc/broyden.cu)',
            'bound': 'hbm', 'achieved': ach, 'peak': hbm_gbs, 'unit': 'GB/s', 'frac': ach / hbm_gbs, 'traffic': None,
            'peak_source': peak_src, 'shape': {'B': B, 'd': d, 'iterations': n_iter},
            'us_per_iteration': t_ms * 1e3 / n_iter,
            'l2': 'history %.0f MB > L2, iterations back to back, no flush' % (8.0 * B * T * d / 1e6) if streamed
                  else '256 MB flush between iterations',
            'note': 'algorithmic bytes (6+2i)*d*4 per sample for iteration i; the kernel reads the rank-(i-1) history '
                    'twice (dots, then combinations); the read-once variants measured slower, see '
                    'profiles/r02_update_bench.txt and DESIGN.md section 4'}


def _host_init_lazy_buffers(sd, wl, x):
    """Shape the conv u/v buffers and ActNorm parameters on the host the way the reference's first
    `model(x, restore=True)` does (mixed_lipschitz.py:195-239, act_norm.py:25-37)."""
    import torch.nn.functional as F
    from oracle import impflow_oracle as orc
    sd = {k: v.clone() for k, v in sd.items()}
    c, h, w = wl['input']
    feat = x
    alpha = 0.05
    s = alpha + (1 - 2 * alpha) * feat
    feat = torch.log(s) - torch.log(1 - s)
    n_scales = len(wl['n_blocks'])
    for sc, nb in enumerate(wl['n_blocks']):
        pre = 'transforms.%d.chain.' % sc
        i = 1 if sc == 0 else 0
        items = ([('actnorm', i)] if sc == 0 else [])
        i += len(items)
        for _ in range(nb):
            items.append(('imblock', i))
            items.append(('actnorm', i + 1))
            i += 2
        for kind, idx in items:
            if kind == 'actnorm':
                wgt, b = orc.actnorm_init(feat)
                sd['%s%d.weight' % (pre, idx)] = wgt
                sd['%s%d.bias' % (pre, idx)] = b
                sd['%s%d.initialized' % (pre, idx)] = torch.tensor(1)
                feat = (feat + b.view(1, -1, 1, 1)) * torch.exp(wgt.view(1, -1, 1, 1))
            else:
                for net in ('nnet_x', 'nnet_z', 'nnet_x_copy', 'nnet_z_copy'):
                    j = 0
                    while True:
                        key = '%s%d.%s.%d.' % (pre, idx, net, j)
                        if not any(k.startswith('%s%d.%s.' % (pre, idx, net)) and int(k.split('.')[5]) >= j
                                   for k in sd):
                            break
                        if key + 'weight' in sd and sd[key + 'weight'].dim() == 4:
                            Wt = sd[key + 'weight']
                            hh, ww = feat.shape[2], feat.shape[3]
                            sd[key + 'spatial_dims'] = torch.tensor([float(hh), float(ww)])
                            sd[key + 'initialized'] = torch.tensor(1)
                            if Wt.shape[-1] == 1:
                                u = F.normalize(torch.randn(Wt.shape[0]), dim=0)
                                v = F.normalize(torch.randn(Wt.shape[1]), dim=0)
                                u, v, _ = orc.power_iterate_matrix(Wt.view(Wt.shape[0], Wt.shape[1]), u, v, None,
                                                                   1e-3, 1e-3)
                            else:
                                v = F.normalize(torch.randn(Wt.shape[1] * hh * ww), dim=0)
                                u = F.normalize(torch.randn(Wt.shape[0] * hh * ww), dim=0)
                                u, v, _ = orc.power_iterate_conv(Wt, u, v, (Wt.shape[1], hh, ww), 1, 1, None, 1e-3,
                                                                 1e-3)
                            sd[key + 'u'], sd[key + 'v'] = u, v
                        j += 1
        if sc < n_scales - 1:
            feat = orc.squeeze2(feat)
    return sd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cifar', choices=list(WORKLOADS))
    ap.add_argument('--batch', type=int, default=None, help='per-GPU batch (weak scaling) / global batch (strong)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: per-GPU batch fixed; strong: global batch fixed and sharded over the ranks')
    ap.add_argument('--cpu-batch', type=int, default=None,
                    help='samples per step of the reference arm (bounded sample; default: a quarter of the batch, '
                         'capped so that K + W steps end within minutes)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--probe-mode', default='device', choices=['reference', 'device'])
    ap.add_argument('--unfused', action='store_true', help='disable the graph-free branch programs (A/B)')
    ap.add_argument('--roulette', default='shared', choices=['shared', 'per-rank'],
                    help='N > 1: the Russian-roulette term counts n are drawn from one seed on every rank (equal work '
                         'per rank; each rank\'s estimate stays unbiased, probes and data stay per-rank) or per rank '
                         '(what the reference\'s DataParallel threads do; the step then waits for the unluckiest rank)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last of them computed (loss, model outputs, updated '
                         'parameters, gradients) as DIR/<name>.npy; the inputs are seeded, so two builds run with the '
                         'same arguments can be compared output for output')
    args = ap.parse_args()

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    wl = WORKLOADS[args.workload]
    kind = wl.get('kind', 'img')
    wl_batch = args.batch or wl['batch']
    if args.scaling == 'strong':
        assert wl_batch % world == 0, 'strong scaling: the global batch must divide by the number of ranks'
        batch = wl_batch // world
    else:
        batch = wl_batch
    config = {'workload': WORKLOAD_TEXT.get(args.workload, args.workload),
              'per_gpu_batch': batch, 'global_batch': batch * world, 'parallelism': 'dp%d' % world,
              'l2': 'per-step working set (>1 GB of activations) exceeds the 126 MB L2; 256 MB flush between steps',
              'gemm': '3xTF32 on tcgen05 (fp32-accurate; ceiling = 1/6 of the bf16 peak)',
              'probe_mode': args.probe_mode, 'roulette_draws': args.roulette if world > 1 else 'single rank'}

    if args.impl == 'reference':
        if args.dump_outputs:
            ap.error('--dump-outputs writes the outputs of the GPU path (--impl b200)')
        if rank != 0:
            return
        # a bounded sample of the workload per step, stated in the line's own config: the metric is per sample
        default_cpu = {'img': 8, 'cls': 4, 'mlp': max(wl_batch // 8, 1)}[kind]
        cpu_batch = args.cpu_batch or min(default_cpu, wl_batch)
        res = run_cpu_reference(args.workload, max(args.steps, 1), max(args.warmup, 0), cpu_batch)
        ref_cfg = {'workload': config['workload'], 'per_gpu_batch': cpu_batch, 'global_batch': cpu_batch,
                   'parallelism': 'cpu', 'workload_batch': wl_batch,
                   'sample': 'each step trains on %d of the workload\'s %d samples (bounded CPU sample; the metric '
                             'is per sample)' % (cpu_batch, wl_batch),
                   'arithmetic': 'fp32 ATen on %d host threads' % res['cores']}
        solver = {'fwd': res['fwd_nstep'], 'bwd': res['bwd_nstep']}
        line = {'impl': 'reference', 'metric': METRIC, 'value': res['value'], 'unit': UNIT, 'n_gpus': 0,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': res['ms_per_step'],
                'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32',
                'data': 'synthetic', 'config': ref_cfg,
                'cpu_baseline': {'value': res['value'], 'unit': UNIT, 'cores': res['cores'], 'kind': res['kind'],
                                 'sample': '%d timed + %d warm-up steps of %d samples each of the same model'
                                           % (args.steps, args.warmup, cpu_batch)},
                'e2e': {'value': res['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'solver_iterations': solver}
        print(json.dumps(line))
        return
    if args.steps < 1:
        ap.error('--steps: at least one timed step')

    import torch.distributed as dist
    assert torch.cuda.is_available(), 'bench.py --impl b200 needs a GPU (there is no CPU fallback)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout while the communicator is created; rank 0's stdout is ONE JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    import __graft_entry__
    if rank == 0:
        with contextlib.redirect_stdout(sys.stderr):      # stdout carries the JSON line only
            __graft_entry__.build()
    if world > 1:
        dist.barrier()
    import impflow_b200 as pkg
    from impflow_b200.layers import implicit_block
    implicit_block.PROBE_MODE['mode'] = args.probe_mode
    implicit_block.FUSED['on'] = not args.unfused
    if os.environ.get('IMPFLOW_TMA_STORE', '') == '0':       # A/B: per-thread stores instead of bulk tensor stores
        pkg._cabi.load().impflow_gemm_tc_set_tma_store(0)
    if os.environ.get('IMPFLOW_PAIR', '') == '0':            # A/B: single-CTA GEMM tiles only (no cta_group::2)
        pkg._cabi.load().impflow_gemm_tc_set_pair(0)
    if os.environ.get('IMPFLOW_PDL', '') == '0':             # A/B: ordinary launches of the tile kernels
        pkg._cabi.load().impflow_set_pdl(0)
    if os.environ.get('IMPFLOW_CHAIN_FUSE', '') in ('0', '1'):    # A/B: power-series epilogue writes the next term's input
        pkg._cabi.load().impflow_conv3_set_chain_fuse(int(os.environ['IMPFLOW_CHAIN_FUSE']))
    if os.environ.get('IMPFLOW_SWEEP_MLP', '') in ('0', '1'):     # A/B: CUDA graphs of the MLP flows' batched sweeps
        pkg.branch_program.SWEEP_GRAPHS['mlp'] = os.environ['IMPFLOW_SWEEP_MLP'] == '1'
    if os.environ.get('IMPFLOW_SWEEP_GRAPHS', '') == '0':    # A/B: eager gradient sweeps instead of CUDA graphs
        pkg.branch_program.SWEEP_GRAPHS['on'] = False
    if os.environ.get('IMPFLOW_SWEEP_ROWS', ''):             # A/B: largest row count whose sweeps are graphed
        pkg.branch_program.SWEEP_GRAPHS['max_rows'] = int(os.environ['IMPFLOW_SWEEP_ROWS'])
    if os.environ.get('IMPFLOW_WGRAD_ORDER', '') == '0':     # A/B: tile-major weight-gradient work order
        pkg._cabi.load().impflow_wgrad_set_slice_major(0)
    if os.environ.get('IMPFLOW_SN_CTAS', ''):                # A/B: CTAs per 3x3 power-iteration launch
        pkg._cabi.load().impflow_sn_conv_set_ctas(int(os.environ['IMPFLOW_SN_CTAS']))
    if os.environ.get('IMPFLOW_SN_BATCH', '') == '0':        # A/B: one power-iteration launch per dense layer
        pkg.layers.base.mixed_lipschitz.BATCH_DENSE['on'] = False
    if os.environ.get('IMPFLOW_RUNAHEAD', ''):               # A/B: 0 = synchronise the solver loop every iteration
        pkg._cabi.load().impflow_conv3_set_runahead(int(os.environ['IMPFLOW_RUNAHEAD']))
    if os.environ.get('IMPFLOW_CHAIN23_A32', '') == '1':     # A/B: one fp32 plane between layer 1 and k_chain23
        pkg._cabi.load().impflow_conv3_set_chain23_a32(1)
    if os.environ.get('IMPFLOW_CHAIN23', '') == '0':         # A/B: two GEMM launches instead of k_chain23
        pkg._cabi.load().impflow_conv3_set_chain23(0)
        pkg.ops.CHAIN23['on'] = False

    torch.manual_seed(0)
    np.random.seed(0)
    model = build_model(pkg, wl, batch).to(dev)
    is_mlp = kind == 'mlp'
    is_cls = kind == 'cls'
    gen = torch.Generator().manual_seed(1234 + rank)
    if is_mlp:
        scale_mlp_last_layers(model, wl)      # move the near-zero last layers so the solves do real work
        n_dims = wl['d']
    else:
        n_dims = int(np.prod(wl['input']))
    x_host, y_host = synthetic_batch(wl, batch, gen)
    x_host = x_host.pin_memory()
    y_host = y_host.pin_memory() if y_host is not None else None
    x_dev = x_host.to(dev)
    y_dev = y_host.to(dev) if y_host is not None else None
    with torch.no_grad():
        model(x_dev, restore=True)           # ActNorm data init + lazy u/v shaping (train_img.py:502-507)
    if world > 1:
        pkg.parallel.broadcast_module(model, 0)
    np.random.seed(100 if args.roulette == 'shared' else 100 + rank)     # the roulette draws use the NumPy RNG
    torch.manual_seed(100 + rank)                                        # probes: per rank
    model.train()
    params = [p for p in model.parameters() if p.requires_grad]
    bucket = pkg.parallel.FlatGradBucket(params)
    # step tail of train_img.py:652-658 in one fused pass: clip_grad_norm_(1.) + the vendored Adam + parameter EMA
    # (train_toy.py: no clipping, no EMA; train_classification.py: EMA, no clipping)
    is_toy = args.workload == 'toy'
    opt = pkg.optim.FusedAdam(params, lr=1e-3, betas=(0.9, 0.999) if (is_toy or is_cls) else (0.9, 0.99),
                              bucket=bucket, max_grad_norm=None if (is_toy or is_cls) else 1.,
                              ema_decay=None if is_toy else 0.999)
    flush = torch.empty(64 * 1024 * 1024, device=dev, dtype=torch.float32)
    blocks = [m for m in model.modules() if isinstance(m, pkg.layers.imBlock)]

    def step(x, y=None, outputs=None):
        bucket.zero()
        loss = loss_of(model, wl, x, y, outputs)
        loss.backward()
        bucket.allreduce_mean()
        opt.step()
        update_lipschitz(pkg, model, wl.get('n_lipschitz_iters'))
        return loss

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the clock poller starts in front of the warm-up (its start-up stalls CUDA calls for ~100 ms, see ClockSampler)
    sampler = ClockSampler(local_rank)
    if rank == 0 and os.environ.get('IMPFLOW_BENCH_NOSAMPLER', '') != '1':     # diagnostic switch: cost of the poller
        sampler.start()
    trace = os.environ.get('IMPFLOW_TRACE_CAPTURE', '') == '1'
    if trace:                      # diagnostic: log every cyclic-GC pass (generation, duration) next to the captures
        import gc
        _gc_t = {}

        def _gc_cb(phase, info):
            if phase == 'start':
                _gc_t['t'] = time.perf_counter()
            elif info.get('generation', 0) >= 1:
                sys.stderr.write('[gc] t=%.3f gen=%d %.1f ms collected=%d\n' % (
                    time.perf_counter(), info['generation'], 1e3 * (time.perf_counter() - _gc_t.get('t', 0.0)),
                    info.get('collected', 0)))
        gc.callbacks.append(_gc_cb)
    for i_ in range(args.warmup):
        if trace:
            torch.cuda.synchronize()
            sys.stderr.write('[warm-up step %d] t=%.3f\n' % (i_, time.perf_counter()))
        step(x_dev, y_dev)
    sync_all()
    if trace:
        sys.stderr.write('[timed region] t=%.3f\n' % time.perf_counter())
    if os.environ.get('IMPFLOW_BENCH_GC', '') == 'freeze':      # diagnostic: cost of Python's cyclic GC in the loop
        import gc
        gc.collect()
        gc.freeze()
    elif os.environ.get('IMPFLOW_BENCH_GC', '') == 'off':
        import gc
        gc.disable()

    # ---------------- timed region: K steps, inputs resident in HBM ----------------
    sampler.mark_begin()
    launches0 = pkg._cabi.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    solves = 0
    fwd_its, bwd_its = [], []
    sync_all()
    torch.cuda.nvtx.range_push('timed')
    if os.environ.get('IMPFLOW_PROFILER_API', '') == '1':      # ncu --profile-from-start off: every thread's launches
        torch.cuda.cudart().cudaProfilerStart()
    dumped = {} if args.dump_outputs and rank == 0 else None
    ev0.record()
    step_evs = [ev0]
    for i_ in range(args.steps):
        if trace:
            sys.stderr.write('[timed step %d] t=%.3f\n' % (i_, time.perf_counter()))
        flush.zero_()
        loss_last = step(x_dev, y_dev, dumped if i_ == args.steps - 1 else None)
        step_evs.append(torch.cuda.Event(enable_timing=True))
        step_evs[-1].record()
        solves += 2 * len(blocks) * batch
        fwd_its.append([b.solver_stats['fwd']['nstep'] for b in blocks])
        bwd_its.append([b.solver_stats['bwd']['nstep'] if 'bwd' in b.solver_stats else None for b in blocks])
    ev1.record()
    sync_all()
    if os.environ.get('IMPFLOW_PROFILER_API', '') == '1':
        torch.cuda.cudart().cudaProfilerStop()
    torch.cuda.nvtx.range_pop()
    ms_total = ev0.elapsed_time(ev1)
    per_step_ms = [round(a.elapsed_time(b), 2) for a, b in zip(step_evs[:-1], step_evs[1:])]
    launches = pkg._cabi.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if dumped is not None:
        # besides the model outputs: the last timed step's loss, the parameters its optimiser step left and the
        # gradients it applied (taken now: the passes below train on)
        dumped['loss'] = loss_last.detach().reshape(1)
        dumped['params'] = torch.cat([p.detach().reshape(-1) for p in params])
        dumped['grads'] = torch.cat([g.reshape(-1) for g in bucket.views])
        write_outputs(args.dump_outputs, dumped)
        dumped = None

    # ---------------- instrumented pass (NOT the timed region): the same K steps again with the per-launch shape
    # recorder and CUDA events around every solve switched on.  The recorder costs host time per launch, and the step
    # is partly host-bound, so it stays out of the region `value` is measured on.
    pkg.ops.GEMM_PROFILE['on'] = True
    pkg.ops.GEMM_PROFILE['shapes'] = {}
    implicit_block.SOLVER_TIMING['on'], implicit_block.SOLVER_TIMING['events'] = True, []
    evi0, evi1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evi0.record()
    for _ in range(args.steps):
        flush.zero_()
        step(x_dev, y_dev)
    evi1.record()
    sync_all()
    ms_instr = evi0.elapsed_time(evi1)
    pkg.ops.GEMM_PROFILE['on'] = False
    implicit_block.SOLVER_TIMING['on'] = False
    solver_ms = {'fwd': 0.0, 'bwd': 0.0}
    for k_, e0_, e1_ in implicit_block.SOLVER_TIMING['events']:
        solver_ms[k_] += e0_.elapsed_time(e1_)
    implicit_block.SOLVER_TIMING['events'] = []
    t = torch.tensor([ms_total, solver_ms['fwd'] + solver_ms['bwd'], ms_instr], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, solver_ms_total, ms_instr = float(t[0].item()), float(t[1].item()), float(t[2].item())
    ms_step = ms_total / args.steps
    value = batch * world / (ms_step / 1e3)

    # roofline of the dominant kernel (tcgen05 3xTF32 GEMM): every launch of the timed region was
    # recorded by shape; each distinct shape is timed live here with CUDA events (L2 flushed, stream kept
    # busy so the events bracket the kernel alone) and weighted by its launch count.
    gemm_shapes = dict(pkg.ops.GEMM_PROFILE['shapes'])
    pkg.ops.GEMM_PROFILE['shapes'] = {}
    kern = {}      # kernel name -> dict(ms, flop, launches, shapes)
    if rank == 0:
        for key, cnt in gemm_shapes.items():
            if key[0] == 'branch3':
                _, M_, C_, N3_, is_vjp, save_pre = key
                name = 'k_branch3'
                t = pkg.ops.time_branch3_shape(key, reps=3, flush=flush)
                fl = 2.0 * M_ * (N3_ * C_ + C_ * C_ + C_ * N3_)      # algorithmic: unpadded 9c tap columns
                desc = {'M': M_, 'C': C_, 'taps': N3_, 'mode': 'vjp' if is_vjp else ('fwd+save' if save_pre else 'fwd')}
            elif key[0] == 'chain23':
                _, M_, C_, N3_, is_vjp, save_pre = key
                name = 'k_chain23'
                t = pkg.ops.time_chain23_shape(key, reps=3, flush=flush)
                fl = 2.0 * M_ * (C_ * C_ + C_ * N3_)
                desc = {'M': M_, 'C': C_, 'taps': N3_, 'mode': 'vjp' if is_vjp else ('fwd+save' if save_pre else 'fwd')}
            elif key[0] == 'wgrad':
                _, M_, N1_, N2_ = key
                name = 'k_wgrad_tc3'
                t = pkg.ops.time_wgrad_shape(key, reps=3, flush=flush)
                fl = 2.0 * M_ * N1_ * N2_
                desc = {'pixels': M_, 'N1': N1_, 'N2': N2_}
            else:
                name = 'k_gemm_tc3'
                t = pkg.ops.time_gemm_shape(key, reps=3, flush=flush)
                fl = 2.0 * key[0] * key[1] * key[2]
                desc = {'M': key[0], 'N': key[1], 'K': key[2]}
            k = kern.setdefault(name, {'ms': 0.0, 'flop': 0.0, 'launches': 0, 'shapes': []})
            k['ms'] += t * cnt
            k['flop'] += fl * cnt
            k['launches'] += cnt
            desc.update({'launches_per_step': cnt / args.steps, 'us': t * 1e3, 'tflops': fl / t / 1e9})
            k['shapes'].append((t * cnt, desc))

    # ---------------- e2e: same step through the public API from pinned host buffers ----------------
    # every step: H2D copy of its inputs from pinned memory, D2H copy of its loss into pinned memory (asynchronous, as a
    # training loop that logs the loss does it: the host does not stall on the value, so it keeps issuing the next step);
    # all K losses have arrived when the clock stops
    loss_host = torch.zeros(max(args.steps, 1), dtype=torch.float32).pin_memory()
    sync_all()
    t0 = time.perf_counter()
    for i_ in range(args.steps):
        xb = x_host.to(dev, non_blocking=True)
        yb = y_host.to(dev, non_blocking=True) if y_host is not None else None
        loss_host[i_:i_ + 1].copy_(step(xb, yb).detach().reshape(1), non_blocking=True)   # device -> host read of the loss
    sync_all()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    last = float(loss_host[args.steps - 1]) if args.steps > 0 else None
    te = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())

    # ---------------- generation path: forward-only Broyden solves (model.inverse, train_img.py:756-761) ----------
    inv = None
    if kind == 'img':
        model.eval()
        with torch.no_grad():
            zs = torch.randn(batch, n_dims, device=dev)
            for _ in range(2):
                model(zs, inverse=True)
            sync_all()
            i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_inv = max(2, min(args.steps, 5))
            i0.record()
            for _ in range(n_inv):
                model(zs, inverse=True)
            i1.record()
            sync_all()
        ti = torch.tensor([i0.elapsed_time(i1) / n_inv], device=dev)
        if world > 1:
            dist.all_reduce(ti, op=dist.ReduceOp.MAX)
        inv = {'ms_per_batch': float(ti.item()), 'samples_per_sec': batch * world / (float(ti.item()) / 1e3),
               'broyden_solves_per_sec': len(blocks) * batch * world / (float(ti.item()) / 1e3),
               'solver_iterations': [b.solver_stats['inv']['nstep'] for b in blocks if 'inv' in b.solver_stats]}
        model.train()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops_sustained', 1400.0)
    peak_src = 'MEASURED_PEAKS.json bf16_tflops_sustained' if peaks else 'fallback 1.4 PF sustained (B200_PROFILING.md)'
    KNAMES = {'k_branch3': 'k_branch3 (fused 3-layer residual-branch tile kernel, tcgen05 3xTF32, operands in TMEM)',
              'k_gemm_tc3': 'k_gemm_tc3 (tcgen05 3xTF32 residual-branch GEMM)',
              'k_chain23': 'k_chain23 (fused layers 2+3 of the wider-scale conv branches, tcgen05 3xTF32, layer-2 output '
                           'kept in TMEM)',
              'k_wgrad_tc3': 'k_wgrad_tc3 (tcgen05 3xTF32 weight gradient, MN-major operands)'}

    # DRAM bytes per launch of each kernel from the committed `ncu --set full` captures (profiles/)
    try:
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
    except Exception:
        traffic = {}

    def roof(name):
        k = kern[name]
        ach = k['flop'] / (k['ms'] / 1e3) / 1e12 if k['ms'] > 0 else 0.0
        tr = traffic.get(name)
        return {'kernel': KNAMES[name], 'bound': 'tensor', 'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s',
                'frac': ach / peak_tf, 'traffic': tr['dram_bytes_per_launch'] if tr else None,
                'traffic_detail': tr, 'peak_source': peak_src, 'launches': k['launches'],
                'share_of_step': k['ms'] / ms_instr if ms_instr > 0 else None,
                'top_shapes': [d for _, d in sorted(k['shapes'], key=lambda x: -x[0])[:4]],
                'frac_of_3xtf32_ceiling': ach / (peak_tf / 6.0),
                'note': 'achieved = sum(algorithmic flops) / sum(kernel time) over every launch of this kernel in '
                        'the timed region; per-shape kernel times measured live with CUDA events (L2 flushed). '
                        'Each product is 3 tf32 MMAs (fp32-accurate 3xTF32), so the mode ceiling is peak/6 = '
                        '%.0f TFLOP/s' % (peak_tf / 6.0)}

    order = sorted(kern, key=lambda n: -kern[n]['ms'])
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'config': config, 'clocks': clocks,
        'e2e': {'value': batch * world / (e2e_ms / 1e3), 'unit': UNIT, 'ms_per_step': e2e_ms,
                'h2d_bytes_per_step': int(x_host.numel() * 4 + (y_host.numel() * 8 if y_host is not None else 0)),
                'd2h_bytes_per_step': 4, 'last_loss': last},
        'gpu_launches': int(launches),
        # SURVEY.md section 8d: solves (samples x imBlocks x [forward + implicit-backward]) / time inside the solver
        # phases (CUDA events around every solve); the whole-step figure beside it
        'broyden_solves_per_sec': solves * world / (solver_ms_total / 1e3) if solver_ms_total > 0 else None,
        'broyden_solves_per_sec_whole_step': solves * world / (ms_total / 1e3),
        'per_step_ms': per_step_ms,
        'instrumented_pass': {'ms_per_step': ms_instr / args.steps,
                              'note': 'the K steps repeated with the per-launch shape recorder and solver events on; '
                                      'roofline shares and solver_phase come from this pass, value from the clean one'},
        'solver_phase': {'ms_per_step': solver_ms_total / args.steps, 'share_of_step': solver_ms_total / ms_instr,
                         'fwd_ms_per_step': solver_ms['fwd'] / args.steps,
                         'bwd_ms_per_step': solver_ms['bwd'] / args.steps},
        'solver_iterations_fwd_last_step': fwd_its[-1] if fwd_its else None,
        'solver_iterations_bwd_last_step': bwd_its[-1] if bwd_its else None,
        'inverse_sampling': inv,
        'roofline': roof(order[0]) if order else None,
    }
    if len(order) > 1:
        line['roofline_secondary'] = roof(order[1])
    if len(order) > 2:
        line['roofline_tertiary'] = roof(order[2])
    hbm = peaks.get('hbm_gbs', 6650.0)
    hsrc = 'MEASURED_PEAKS.json hbm_gbs' if peaks else 'fallback 6.65 TB/s (B200_PROFILING.md)'
    if kind != 'mlp':
        # the solver-algebra phase against the HBM roofline: the bench shape (latency-bound: 0.8 MB per
        # vector) and the classifier shape of SURVEY.md section 8 (B=128, d=65536: 2 GB of history)
        try:
            d_solver = n_dims if kind == 'img' else 65536
            line['roofline_solver'] = [solver_roofline(pkg, batch, d_solver, 30, 6, flush, hbm, hsrc)] + \
                ([solver_roofline(pkg, 128, 65536, 30, 8, flush, hbm, hsrc)] if kind == 'img' else [])
        except Exception as exc:
            line['roofline_solver'] = 'failed: %r' % (exc,)
    if not order and line.get('roofline') is None and isinstance(line.get('roofline_solver'), list):
        line['roofline'] = line['roofline_solver'][0]       # no tensor-core launch in this workload: HBM-bound solver
    if world == 1 and not args.no_cpu_baseline:
        try:
            # one warm-up + one timed step on a bounded sample of the batch (about 15-30 s of CPU work: the unmodified
            # reference needs > 1 min per 64-image step of the CIFAR flow; DESIGN.md lists its measured per-image
            # throughput at batch 4 / 8 / 16 / 32 / 64)
            cb = {'img': min(16, wl_batch), 'cls': 8, 'mlp': max(wl_batch // 4, 1)}[kind]
            cb = args.cpu_batch or cb
            res = run_cpu_reference(args.workload, 1, 1, cb)
            line['cpu_baseline'] = {'value': res['value'], 'unit': UNIT, 'cores': res['cores'], 'kind': res['kind'],
                                    'sample': '1 timed + 1 warm-up step of %d samples (workload batch %d) of the same '
                                              'model on host cores' % (cb, wl_batch),
                                    'solver_iterations': {'fwd': res['fwd_nstep'], 'bwd': res['bwd_nstep']}}
        except Exception as exc:      # the baseline must never hide the GPU number
            line['cpu_baseline'] = {'value': None, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': 'reference',
                                    'sample': 'failed: %r' % (exc,)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
