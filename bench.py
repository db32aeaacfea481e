#!/usr/bin/env python
"""Benchmark of the BCNN VGG-16 448x448 train step (BASELINE.json metric) on N B200s, one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload bcnn_s2|bcnn_s1|cbcnn8192|mpn] [--batch 32]
                  [--impl native|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).
  value         device-timed images/s, inputs resident in HBM (CUDA events, max over ranks)
  e2e           the same step through hawkeye_b200.train.Trainer.batch_training with pinned HOST inputs (H2D copy and the
                loss / accuracy read-back inside the timed region)
  roofline      hk_bilinear_pool_fwd (K1, the kernel BASELINE.json names) against the measured HBM peak, at the workload's
                batch 32 and at 256 / 1024; roofline_bwd = hk_bilinear_pool_bwd (K1b); roofline_cbp = hk_cbp_fwd (K2);
                roofline_mpncov = covariance + Newton-Schulz fwd+bwd (K3/K4) against the TF32 tensor peak
  roofline_conv whole-step TF32 TFLOP/s against measured bf16-sustained / 2
  eager_gpu     informational: the same BCNN step in stock PyTorch eager (torch.nn, cuDNN/cuBLAS with TF32 allowed) on the
                same GPU — the practical bar (SURVEY 2a), not the reference arm
  cpu_baseline  the reference step on the host cores: the UNMODIFIED reference when its tree is importable
                ($HAWKEYE_REF, baseline/_ref, /root/reference; kind "reference"), else the oracle port (kind "port")
`--impl reference` times that CPU path only and reports the steps it actually timed.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import torch  # noqa: E402

K1_FWD_BYTES_PER_IMG = 1449984      # read X 512*196*4 + write Y 512*512*4 (SURVEY.md 8(d))
K1_BWD_BYTES_PER_IMG = 1851392      # read dY + read X + write dX (z recomputed)
VGG16_FWD_GFLOP_PER_IMG = 122.9
RESNET50_MPN_FWD_GFLOP_PER_IMG = 32.9
MPNCOV_GFLOP_PER_IMG = 1.77         # covariance + 5-iteration Newton-Schulz, forward + backward (SURVEY.md 8(d))
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the ncu --set full captures under profiles/ (see
# profiles/README.md for the file each number comes from); None = not captured for this build
K1_DRAM_TRAFFIC = {32: 12.89e6 + 0.01e6, 256: 102.83e6 + 210.72e6}   # profiles/gram_r3_metrics.txt (tests/prof_bilinear.py 32 / 256)
WORKLOADS = {
    'bcnn_s2': dict(cfg='BCNN_S2.yaml', trainer='BCNN', model='BCNN VGG-16 stage 2', fwd_gflop=VGG16_FWD_GFLOP_PER_IMG, bwd_mult=3.0),
    'bcnn_s1': dict(cfg='BCNN_S1.yaml', trainer='BCNN', model='BCNN VGG-16 stage 1 (classifier only)', fwd_gflop=VGG16_FWD_GFLOP_PER_IMG, bwd_mult=1.0),
    'cbcnn8192': dict(cfg='CBCNN_S1.yaml', trainer='CBCNN', model='CBCNN VGG-16 d=8192 stage 1', fwd_gflop=VGG16_FWD_GFLOP_PER_IMG, bwd_mult=1.0),
    'mpn': dict(cfg='MPN.yaml', trainer='MPN', model='Fast MPN-COV ResNet-50', fwd_gflop=RESNET50_MPN_FWD_GFLOP_PER_IMG, bwd_mult=3.0),
    # BASELINE.json config 5 (OSME half): ResNet-101 trunk (4 x 7.8 GFLOP at 448x448) + two 401408 -> 1024 attention FCs; MAMC loss
    'osmenet': dict(cfg='OSMENet.yaml', trainer='OSMENet', model='OSMENet ResNet-101 + OSME (2 attentions) + MAMC loss',
                    fwd_gflop=32.9, bwd_mult=3.0),
}


def metric_name(w):
    if w == 'bcnn_s2':
        return '448x448 images/sec, BCNN VGG-16 train step (fwd+CE+bwd+grad all-reduce+SGD), device-timed, max over ranks'
    return f'448x448 images/sec, {WORKLOADS[w]["model"]} train step (fwd+CE+bwd+grad all-reduce+optimizer), device-timed, max over ranks'


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('hbm_gbs', 6650.0), d.get('bf16_tflops_sustained', 1400.0), 'measured'
    return 6650.0, 1400.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference step on the host cores
# ----------------------------------------------------------------------------------------------------------------------
def _cpu_state_and_forward(workload):
    """(state dict, forward(x, state), trainable keys) of the oracle port for `workload`."""
    import detgen
    from oracle import hop_oracle as O
    if workload in ('bcnn_s1', 'bcnn_s2'):
        stage = 1 if workload == 'bcnn_s1' else 2
        state = detgen.vgg_bcnn_state(O.VGG16_D, 200, seed=100)
        keys = None if stage == 2 else {'classifier.weight', 'classifier.bias'}
        return state, (lambda xx, st: O.bcnn_forward(xx, st, stage)), keys
    if workload == 'cbcnn8192':
        state = detgen.vgg_bcnn_state(O.VGG16_D, 200, seed=100, head_in=8192)
        return state, (lambda xx, st: O.cbcnn_forward(xx, st, 8192, 1)), {'classifier.weight', 'classifier.bias'}
    import hawkeye_b200 as hb

    class Cfg(dict):
        __getattr__ = dict.__getitem__
    net = hb.MODEL.get('MPN')(Cfg(name='MPN', iter_num=5, is_sqrt=True, is_vec=True, input_dim=2048,
                                  dimension_reduction=256, num_classes=200))
    state = detgen.state_like(net)
    keys = {k for k, _ in net.named_parameters()}
    return state, (lambda xx, st: O.mpn_forward(xx, st, 5)), keys


def cpu_step_port(workload, B, threads, steps):
    """The oracle port of the reference step (test/bench infrastructure, never the product)."""
    from oracle import hop_oracle as O
    torch.set_num_threads(threads)
    state, fwd, keys = _cpu_state_and_forward(workload)
    x = torch.randn(B, 3, 448, 448, generator=torch.Generator().manual_seed(1234))
    labels = torch.randint(0, 200, (B,), generator=torch.Generator().manual_seed(1))
    bufs = {}

    def step():
        _, loss, grads = O.loss_and_grads(fwd, x, labels, state, keys)
        for k, g in grads.items():
            if g is not None:
                state[k], bufs[k] = O.sgd_momentum_step(state[k], g, bufs.get(k), 0.005, 0.9, 1e-5, k not in bufs)
        return loss

    step()  # warm-up
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / steps


def cpu_step_reference(workload, B, threads, steps):
    """The UNMODIFIED reference (model/registry.MODEL + nn.CrossEntropyLoss(label_smoothing=0.1) + torch.optim, i.e. what
    train.py:310-325 runs) imported from $HAWKEYE_REF / baseline/_ref / /root/reference.  Raises if the tree is absent."""
    from oracle import ref_harness as rh
    if not rh.available():
        raise RuntimeError('reference tree not importable')
    rh.load_reference()
    from model.registry import MODEL
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    if workload in ('bcnn_s1', 'bcnn_s2'):
        net = MODEL.get('BCNN')(rh.cfg(name='BCNN', stage=1 if workload == 'bcnn_s1' else 2, num_classes=200))
    elif workload == 'cbcnn8192':
        net = MODEL.get('CBCNN')(rh.cfg(name='CBCNN', stage=1, num_classes=200, input_channel=512, output_channel=8192))
        for p in net.backbone.parameters():                          # Examples/CBCNN.py:13-15
            p.requires_grad = False
    else:
        net = MODEL.get('MPN')(rh.cfg(name='MPN', iter_num=5, is_sqrt=True, is_vec=True, input_dim=2048,
                                      dimension_reduction=256, num_classes=200))
    net.train()
    params = [p for p in net.parameters() if p.requires_grad]
    opt = torch.optim.SGD(params, lr=0.005, momentum=0.9, weight_decay=1e-5) if workload != 'mpn' else \
        torch.optim.Adam(params, lr=8e-5, weight_decay=2e-5)
    crit = torch.nn.CrossEntropyLoss(label_smoothing=0.1)
    x = torch.randn(B, 3, 448, 448, generator=torch.Generator().manual_seed(1234))
    labels = torch.randint(0, 200, (B,), generator=torch.Generator().manual_seed(1))

    def step():
        loss = crit(net(x), labels)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss

    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / steps


def cpu_baseline(workload, steps):
    """-> dict(value img/s, cores, kind, sample, dt).  Batch 2 (BASELINE.json configs[0]); all host threads it can use:
    a batch-2 step stops scaling around 32 threads, so 32 and os.cpu_count() are both probed and the faster one is kept."""
    B = 2
    ncpu = os.cpu_count() or 1
    for fn, kind in ((cpu_step_reference, 'reference'), (cpu_step_port, 'port')):
        try:
            cands = sorted({min(32, ncpu), ncpu})
            best = None
            for th in cands:
                dt = fn(workload, B, th, 1)
                if best is None or dt < best[1]:
                    best = (th, dt)
            threads = best[0]
            dt = fn(workload, B, threads, steps) if steps > 1 else best[1]
            what = ('UNMODIFIED reference modules (model.registry.MODEL) + torch.optim' if kind == 'reference'
                    else 'torch-CPU oracle port of the reference step')
            return dict(value=B / dt, unit='img/s', cores=threads, kind=kind, dt=dt,
                        sample=f'{max(steps, 1)} timed step(s) of batch {B} ({dt:.2f} s/step; fwd+CE+bwd+optimizer), {what}, '
                               f'{threads} of {ncpu} host threads')
        except Exception as e:  # reference tree absent on the GPU box -> port
            last = e
    raise last


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.workload == 'osmenet':      # the reference OSME hard-codes a 7x7 trunk output (OSME.py:57): no 448x448 reference step exists
        print(json.dumps({'impl': 'reference', 'unavailable': 'reference OSMENet is fixed to 224x224 inputs (OSME.py:57)'}), flush=True)
        return
    timed = max(1, min(args.steps, 3))
    cb = cpu_baseline(args.workload, timed)
    dt = cb.pop('dt')
    line = {
        'impl': 'reference', 'metric': metric_name(args.workload), 'value': cb['value'], 'unit': 'img/s', 'n_gpus': args.gpus,
        'steps': timed, 'steps_requested': args.steps, 'warmup': 1, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{WORKLOADS[args.workload]["model"]}, 448x448, 200 classes; CPU sample batch 2 '
                               f'(BASELINE.json configs[0])'},
        'cpu_baseline': cb,
        'e2e': {'value': cb['value'], 'unit': 'img/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# kernel micro-benchmarks (rank 0, one GPU)
# ----------------------------------------------------------------------------------------------------------------------
def _timed_calls(call, nset, reps):
    for i in range(min(nset, 3)):
        call(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(int(4e6))        # ~2 ms of device-side spin so the host enqueues ahead of the GPU (no launch gaps)
    e0.record()
    for _ in range(reps):
        for i in range(nset):
            call(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / (reps * nset)


def time_bilinear_kernel(B, bwd=False, min_footprint=640 << 20, reps=4):
    """Average device time per call of hk_bilinear_pool_fwd (or _bwd): `reps` passes over a ring of buffer sets whose
    total footprint is >= 5x the 126 MB L2, launched back to back and bracketed by one CUDA-event pair on the launching
    stream.  Every call therefore reads inputs that are not L2-resident and runs while its predecessors' outputs are
    still being written back — the steady state of the kernel, with no separate flush kernel in the timed region."""
    from hawkeye_b200 import _lib
    per_set = B * (K1_BWD_BYTES_PER_IMG + 401408 if bwd else K1_FWD_BYTES_PER_IMG)
    nset = max(2, -(-min_footprint // per_set))
    xs = [torch.rand(B, 512, 14, 14, device='cuda') for _ in range(nset)]
    ys = [torch.empty(B, 512 * 512, device='cuda') for _ in range(nset)]
    if bwd:
        for y in ys:
            y.normal_()
        dxs = [torch.empty_like(x) for x in xs]
    name = 'hk_bilinear_pool_bwd' if bwd else 'hk_bilinear_pool_fwd'
    nb = _lib.query(name + '_workspace_bytes', B, 512, 196)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    s = _lib.stream_ptr()

    def call(i):
        if bwd:
            _lib.call(name, xs[i], ys[i], dxs[i], B, 512, 196, ws, nb, s)
        else:
            _lib.call(name, xs[i], ys[i], None, B, 512, 196, ws, nb, s)

    return _timed_calls(call, nset, reps)


def time_cbp_kernel(B, d=8192, min_footprint=640 << 20, reps=4):
    """hk_cbp_fwd (K2): algorithmic traffic 401 408 B in + 4 d B out per image."""
    import numpy as np
    from hawkeye_b200 import _lib, ops
    per_set = B * (401408 + 8 * d)
    nset = max(2, min(64, -(-min_footprint // per_set)))
    h1, s1, h2, s2 = ops.count_sketch_hashes(512, d)
    dev = 'cuda'
    h1, h2 = torch.from_numpy(h1.astype(np.int32)).to(dev), torch.from_numpy(h2.astype(np.int32)).to(dev)
    s1, s2 = torch.from_numpy(s1.astype(np.float32)).to(dev), torch.from_numpy(s2.astype(np.float32)).to(dev)
    xs = [torch.rand(B, 512, 14, 14, device=dev) for _ in range(nset)]
    ys = [torch.empty(B, d, device=dev) for _ in range(nset)]
    pres = [torch.empty(B, d, device=dev) for _ in range(nset)]
    s = _lib.stream_ptr()
    return _timed_calls(lambda i: _lib.call('hk_cbp_fwd', xs[i], h1, h2, s1, s2, ys[i], pres[i], B, 512, 196, d, s), nset, reps)


def time_mpncov_head(B, reps=3):
    """covariance pooling + 5-iteration Newton-Schulz + triu-vec, forward + backward, on [B,256,14,14] (K3/K4)."""
    from hawkeye_b200 import ops
    x = torch.rand(B, 256, 14, 14, device='cuda', requires_grad=True)

    def fb():
        v = ops.TriuvecLayer(ops.SqrtmLayer(ops.CovpoolLayer(x), 5))
        v.backward(torch.ones_like(v))
        x.grad = None

    for _ in range(2):
        fb()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fb()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def eager_gpu_bcnn(stage, B, steps):
    """Stock PyTorch eager on this GPU: torch.nn VGG-16 'D' features + the reference's BilinearPooling arithmetic +
    nn.Linear, CE(label_smoothing=0.1), SGD(momentum) — cuDNN / cuBLAS kernels with TF32 allowed.  Informational."""
    import torch.nn as nn
    import torch.nn.functional as F
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    layers, cin = [], 3
    for v in [64, 64, 'M', 128, 128, 'M', 256, 256, 256, 'M', 512, 512, 512, 'M', 512, 512, 512, 'M']:
        if v == 'M':
            layers.append(nn.MaxPool2d(2, 2))
        else:
            layers += [nn.Conv2d(cin, v, 3, padding=1), nn.ReLU(inplace=True)]
            cin = v
    feats = nn.Sequential(*layers).cuda()
    cls = nn.Linear(512 * 512, 200).cuda()
    if stage == 1:
        for p in feats.parameters():
            p.requires_grad = False
    params = [p for p in list(feats.parameters()) + list(cls.parameters()) if p.requires_grad]
    opt = torch.optim.SGD(params, lr=0.005, momentum=0.9, weight_decay=1e-5)
    x = torch.randn(B, 3, 448, 448, device='cuda')
    y = torch.randint(0, 200, (B,), device='cuda')

    def step():
        f = feats(x)
        if stage == 1:
            f = f.detach()
        f = f.view(B, 512, -1)
        g = torch.bmm(f, f.transpose(1, 2)) / f.shape[2]                 # BCNN.py:17-18
        z = F.normalize(torch.sqrt(g.view(B, -1) + 1e-5))                # BCNN.py:21,26
        loss = F.cross_entropy(cls(z), y, label_smoothing=0.1)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del feats, cls, opt
    torch.cuda.empty_cache()
    return dict(value=B / ms * 1e3, unit='img/s', ms_per_step=ms,
                note='stock PyTorch eager (torch.nn + cuDNN/cuBLAS, allow_tf32=True, cudnn.benchmark) on the same GPU, same '
                     'batch; informational practical bar, not the reference arm')


DUMP_SAMPLE = 1 << 15      # elements kept per tensor above this size: --dump-outputs writes ~28 MB for osmenet, less for the rest


def _sample(t, seed):
    """float32 numpy copy of `t`; above DUMP_SAMPLE elements, its flattened elements at DUMP_SAMPLE positions drawn with
    `seed`, so that two runs (or two builds) keep the same positions."""
    t = t.detach()
    if t.numel() > DUMP_SAMPLE:
        idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(seed))
        t = t.flatten()[idx.to(t.device)]
    return t.float().cpu().numpy()


def dump_outputs(d, outputs, loss, model):
    """Writes what the last timed step handed its caller as d/<name>.npy: the model outputs (`outputs.npy`, or
    `outputs_<i>.npy` for a tuple), `loss.npy`, and the state after the optimizer step: `state.npy` (every floating-point
    state_dict entry, i.e. updated parameters and running statistics) and `grads.npy` (every parameter gradient), each the
    concatenation in state_dict / named_parameters order of per-tensor samples (_sample, seeded by position)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    outs = outputs if isinstance(outputs, (tuple, list)) else (outputs,)
    arrays = {'outputs' if len(outs) == 1 else f'outputs_{i}': _sample(o, i) for i, o in enumerate(outs)}
    arrays['loss'] = _sample(loss, 0)
    arrays['state'] = np.concatenate([_sample(v, i).ravel() for i, v in enumerate(model.state_dict().values())
                                      if v.is_floating_point()])
    arrays['grads'] = np.concatenate([_sample(p.grad, i).ravel() for i, (_, p) in enumerate(model.named_parameters())
                                      if p.grad is not None])
    for name, a in arrays.items():
        np.save(os.path.join(d, name + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default=None, choices=sorted(WORKLOADS))
    ap.add_argument('--stage', type=int, default=2, help='BCNN stage (kept for compatibility; --workload wins)')
    ap.add_argument('--batch', type=int, default=32)
    ap.add_argument('--impl', default='native')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true', help='profiling runs only')
    ap.add_argument('--no-micro', action='store_true', help='skip the kernel micro-benchmarks (roofline legs)')
    ap.add_argument('--no-eager', action='store_true', help='skip the stock-PyTorch eager GPU leg')
    ap.add_argument('--graph', default='auto', choices=['auto', '0', '1'],
                    help='replay forward+backward from a CUDA graph (Trainer cuda_graph mode); auto = only for the '
                         'host-launch-bound ResNet-50 workload')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs, loss, updated state and gradients of the last timed step to DIR/<name>.npy '
                         '(float32; tensors above %d elements sampled at seeded positions)' % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.workload is None:
        args.workload = f'bcnn_s{args.stage}'
    if args.impl == 'reference':
        return run_reference_arm(args)

    import torch.distributed as dist
    from hawkeye_b200 import _lib, engine, examples
    from hawkeye_b200.config import load_config

    os.environ.setdefault('HAWKEYE_ALLOW_RANDOM_INIT', '1')     # random-init weights are the benchmark's contract
    use_graph = args.graph == '1' or (args.graph == 'auto' and args.workload == 'mpn')
    os.environ['HK_CUDA_GRAPH'] = '1' if use_graph else '0' 
    W = WORKLOADS[args.workload]
    rank, local, world = engine.init_distributed()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    cfg = load_config(os.path.join(ROOT, 'configs', W['cfg']))
    torch.manual_seed(0)                                   # random-init weights, reference initialisers
    tr = examples.TRAINERS[W['trainer']](cfg, dataloaders={})
    tr.model.train()
    B = args.batch
    g = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(B, 3, 448, 448, generator=g).pin_memory()
    y_host = torch.randint(0, 200, (B,), generator=g).pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)

    def step_resident():
        if tr._graph_wanted():           # eager for three steps, captured on the third, replayed from then on
            out, loss = tr._graph_step(x_dev, y_dev)
        else:
            out = tr.model(x_dev)
            loss = tr.criterion(out, y_dev)
            tr.optimizer.zero_grad()
            loss.backward()
            tr.allreduce.finish()
        tr.optimizer.step()
        return out, loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), res

    warm = max(args.warmup, 5 if use_graph else 3)
    for _ in range(warm):
        _, loss = step_resident()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _lib.reset_launch_count()
    ms, (last_out, last_loss) = timed(step_resident, args.steps)
    launches = _lib.launch_count()
    if use_graph and getattr(tr, '_graph', None) is not None:       # replayed kernels are not seen by the host-side counter
        launches += args.steps * tr._graph['kernels']
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:     # before the e2e leg below trains further (and overwrites graph outputs)
        dump_outputs(args.dump_outputs, last_out, last_loss, tr.model)
    value = B * world * args.steps / (ms * 1e-3)

    # end to end through the public Trainer API with host inputs
    data = {'img': x_host, 'label': y_host}
    if args.no_e2e:
        ms_e2e = float('nan')
    else:
        for _ in range(2):
            tr.batch_training(data)
        ms_e2e, _ = timed(lambda: tr.batch_training(data), args.steps)
    e2e = B * world * args.steps / (ms_e2e * 1e-3)
    final_loss = float(loss.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm_peak, tf_peak, which = measured_peaks()
    conv_tf = W['fwd_gflop'] * W['bwd_mult'] * 1e9 * B * args.steps / (ms * 1e-3) / 1e12
    line = {
        'metric': metric_name(args.workload), 'value': value, 'unit': 'img/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': warm, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'tf32 (fp32 storage, fp32 accumulate)', 'data': 'synthetic',
        'config': {'workload': f'{W["model"]}, 448x448, batch {B}/GPU, 200 classes ({W["cfg"]})',
                   'global_batch': B * world, 'parallelism': f'dp{world}', 'cuda_graph': bool(use_graph),
                   'l2': 'per-step working set (GBs of activations) >> 126 MB L2; kernel microbenches rotate through buffer '
                         'sets totalling >= 640 MB (5x L2), so every launch reads cold inputs',
                   'final_loss': final_loss},
        'clocks': clocks,
        'e2e': {'value': e2e, 'unit': 'img/s', 'ms_per_step': ms_e2e / args.steps,
                'h2d_bytes_per_step': x_host.numel() * 4 + y_host.numel() * 8, 'd2h_bytes_per_step': 8},
        'gpu_launches': launches,
        'roofline_conv': {'bound': 'tensor', 'achieved': conv_tf, 'unit': 'TFLOP/s (tf32, whole step incl. non-conv time)',
                          'peak': tf_peak / 2, 'frac': conv_tf / (tf_peak / 2),
                          'note': 'peak = measured bf16 sustained / 2 (tf32 runs at half the bf16 rate)'},
    }
    del tr
    torch.cuda.empty_cache()
    if not args.no_micro:
        t32, t256, t1024 = time_bilinear_kernel(32), time_bilinear_kernel(256), time_bilinear_kernel(1024)

        def bw(B_, t, per_img):
            a = B_ * per_img / t / 1e9
            return {'achieved': a, 'frac': a / hbm_peak, 'us_per_launch': t * 1e6}
        r32 = bw(32, t32, K1_FWD_BYTES_PER_IMG)
        line['roofline'] = {
            'kernel': 'hk_bilinear_pool_fwd, one launch: Gram + sqrt + L2 normalise.  B=32 (the per-GPU batch of this workload, '
                      'C=512, HW=196) = bcnn_super_fwd_kernel<true>: one wave of 4-CTA clusters, four operand-sharing items per '
                      'image, DSMEM norm exchange; b256 / b1024 = bcnn_gram_fwd_kernel<512>: persistent 128x128 tiles, '
                      'bounded-wait norm exchange',
            'bound': 'hbm', 'achieved': r32['achieved'], 'peak': hbm_peak, 'unit': 'GB/s', 'frac': r32['frac'],
            'traffic': K1_DRAM_TRAFFIC[32], 'traffic_note': 'ncu dram read+write per launch: the 33.5 MB output of a B=32 launch stays in the 126 MB L2 under ncu (serialised launches); in the timed back-to-back series it is written back while later launches run', 'peak_source': which, 'us_per_launch': r32['us_per_launch'],
            'algorithmic_bytes_per_launch': 32 * K1_FWD_BYTES_PER_IMG,
            'b256': dict(bw(256, t256, K1_FWD_BYTES_PER_IMG), traffic=K1_DRAM_TRAFFIC[256]),
            'b1024': bw(1024, t1024, K1_FWD_BYTES_PER_IMG)}
    if not args.no_micro and world == 1:
        tb32, tb256 = time_bilinear_kernel(32, bwd=True), time_bilinear_kernel(256, bwd=True)
        line['roofline_bwd'] = {'kernel': 'hk_bilinear_pool_bwd (K1b), B=32, C=512, HW=196', 'bound': 'hbm', 'peak': hbm_peak,
                                'unit': 'GB/s', 'algorithmic_bytes_per_launch': 32 * K1_BWD_BYTES_PER_IMG,
                                **bw(32, tb32, K1_BWD_BYTES_PER_IMG), 'b256': bw(256, tb256, K1_BWD_BYTES_PER_IMG)}
        tc32, tc256 = time_cbp_kernel(32), time_cbp_kernel(256)
        line['roofline_cbp'] = {'kernel': 'hk_cbp_fwd (K2: Gram -> signed scatter into d=8192 bins -> signed sqrt + L2), B=32',
                                'bound': 'hbm', 'peak': hbm_peak, 'unit': 'GB/s',
                                'algorithmic_bytes_per_launch': 32 * (401408 + 4 * 8192),
                                **bw(32, tc32, 401408 + 4 * 8192), 'b256': bw(256, tc256, 401408 + 4 * 8192)}
        tm = time_mpncov_head(32)
        mtf = 32 * MPNCOV_GFLOP_PER_IMG * 1e9 / tm / 1e12
        line['roofline_mpncov'] = {'kernel': 'covpool + sqrtm(5) + triuvec, fwd+bwd (K3/K4), B=32, C=256, HW=196', 'bound': 'tensor',
                                   'achieved': mtf, 'unit': 'TFLOP/s (algorithmic tf32 flops; executed 3x as 3xTF32)',
                                   'peak': tf_peak / 2, 'frac': mtf / (tf_peak / 2), 'ms_per_call': tm * 1e3}
    if not args.no_eager and world == 1 and args.workload in ('bcnn_s1', 'bcnn_s2'):
        try:
            line['eager_gpu'] = eager_gpu_bcnn(1 if args.workload == 'bcnn_s1' else 2, B, max(3, min(args.steps, 10)))
        except Exception as e:          # e.g. out of memory next to a large resident workload
            line['eager_gpu'] = {'unavailable': repr(e)[:200]}
    if not args.no_cpu_baseline:
        if args.workload == 'osmenet':     # the reference OSME hard-codes a 7x7 map (OSME.py:57): it cannot run at 448x448
            line['cpu_baseline'] = {'unavailable': 'reference OSMENet is fixed to 224x224 inputs (OSME.py:57)'}
        else:
            cb = cpu_baseline(args.workload, 2)
            cb.pop('dt')
            line['cpu_baseline'] = cb
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
