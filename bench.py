#!/usr/bin/env python
"""Benchmark of the few-shot-detection meta-training hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on the host CPU

One "step" = one meta-training iteration on one synthetic batch per GPU:
Darknet(darknet_dynamic + reweighting_net).forward -> RegionLossV2 (decode,
build_targets, loss) -> backward -> (gradient all-reduce) -> SGD, at the
configuration BASELINE.json's metric is quoted on (configs[1]): 416x416, batch 64
per GPU, 20 classes, 5 anchors.  Prints ONE JSON line on rank 0.
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
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'images/sec (416x416, 20-cls) meta-training step; build_targets ms/batch'
# kernels launched per C-ABI call (lower bounds, for the gpu_launches claim)
LAUNCHES = {'fsdet_weight_prep': 2, 'fsdet_conv_wgrad': 2, 'fsdet_bn_finalize': 2, 'fsdet_bn_bwd_finalize': 2, 'fsdet_head_bias_grad': 2,
            'fsdet_region_loss_grad': 3}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=64, help='query images per GPU')
    ap.add_argument('--ncls', type=int, default=20)
    ap.add_argument('--side', type=int, default=416)
    ap.add_argument('--ref-batch', type=int, default=8, help='query images per CPU reference step (bounded sample)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel eagerly instead of replaying a CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)')
    return ap.parse_args()


def synth_batch(B, ncls, side, seed):
    from seeding import synth_targets, synth_masks
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, side, side, generator=g)
    metax = torch.rand(ncls, 3, 416, 416, generator=g)
    mask = torch.from_numpy(synth_masks(ncls, 416, seed + 1))
    target = torch.from_numpy(synth_targets(B, ncls, seed + 2, max_gt=5))
    return x, metax, mask, target


def arch_costs(blocks, side, n_cls=1):
    """(forward FLOPs, fused activation elements read + written) per image of a cfg network at input `side`, by
    SURVEY.md 8d's rule: every convolution reads its input once and writes its output once, pooling / BN / leaky /
    reorg / concat are fused into producers or consumers, the dynamic convolution + head count as ONE layer that reads
    its input once and writes n_cls * 30 channels."""
    C, H = int(blocks[0]['channels']), side
    flops = elems = 0
    hist = []
    body = blocks[1:]
    for idx, b in enumerate(body):
        t = b['type']
        if t == 'convolutional':
            if 'dynamic' in b and int(b['dynamic']) == 1:
                hist.append((C, H))
                continue
            k, f = int(b['size']), int(b['filters'])
            rep = n_cls if (idx > 0 and 'dynamic' in body[idx - 1] and int(body[idx - 1]['dynamic']) == 1) else 1
            flops += 2 * H * H * f * k * k * C * rep
            elems += H * H * C + H * H * f * rep
            C = f
        elif t == 'maxpool' and int(b['stride']) == 2:
            H //= 2
        elif t == 'reorg':
            C, H = C * 4, H // 2
        elif t == 'route':
            ls = [int(x) for x in b['layers'].split(',')]
            ls = [l if l > 0 else l + idx for l in ls]
            C, H = sum(hist[l][0] for l in ls), hist[ls[0]][1]
        elif t == 'globalmax':
            H = 1
        hist.append((C, H))
    return flops, elems


def step_costs(B, ncls, side):
    """Algorithmic FLOPs and HBM bytes of one training step per GPU (SURVEY 8d): 3x the forward of B query and n_cls
    support images (fp32 activations), weights read twice + written once + 5 SGD passes."""
    from fewshot_detection_b200 import netcfg
    fq, eq = arch_costs(netcfg.darknet_dynamic_blocks(side, side), side, ncls)
    fs, es = arch_costs(netcfg.reweighting_net_blocks(), 416)
    return 3.0 * (B * fq + ncls * fs), 3.0 * 4 * (B * eq + ncls * es) + 8 * 265.2e6


class ClockSampler(object):
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            f = [c.strip() for c in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def cpu_threads():
    """Host threads for the CPU arm: all cores up to 32.  torch/oneDNN throughput on this workload peaks at 16-32
    threads and collapses beyond (measured on the 128-core GPU box with tools/cpu_threads.py: 2.5 s/step at 16, 2.9 s at
    32, 4.4 s at 64, 50 s at 128 threads), so using more threads would only handicap the reference arm."""
    return min(os.cpu_count() or 1, 32)


def cpu_step_factory(ncls, side, B, threads):
    """The reference's algorithm on the host CPU: oracle port (torch-CPU ops +
    Python build_targets), one full training step."""
    from fewshot_detection_b200 import netcfg
    from oracle import darknet as ODK, region_loss as ORL
    from seeding import seeded_init
    torch.set_num_threads(threads)
    m = ODK.MetaDarknet(netcfg.darknet_dynamic_blocks(side, side), netcfg.reweighting_net_blocks())
    seeded_init(m, 0)
    m.train()
    factor = 15.0
    opt = torch.optim.SGD(m.parameters(), lr=1e-3 / factor / B, momentum=0.9, dampening=0, weight_decay=0.0005 * B * factor)
    x, metax, mask, target = synth_batch(B, ncls, side, 1234)
    state = {'seen': 20000, 'bt_ms': None}

    def step():
        opt.zero_grad()
        out = m(x, metax, mask)
        state['seen'] += B
        t0 = time.perf_counter()
        loss = ORL.region_loss_v2(out, target, m.anchors, m.num_anchors, m.num_classes, seen=state['seen'])
        state['loss_ms'] = (time.perf_counter() - t0) * 1e3
        loss.backward()
        opt.step()
        return float(loss.item())

    def support_only():
        """forward + backward of the support branch alone (its cost is per STEP, not per query image)"""
        opt.zero_grad()
        dw = m.meta_forward(metax, mask)
        dw[0].sum().backward()
    state['support_only'] = support_only
    return step, state


DUMP_SAMPLE = 65536      # values kept per parameter tensor: 89 tensors -> 1.6 M values, 13 MB for params + grads
DUMP_SEED = 20240


def dump_outputs(out_dir, model, region_loss):
    """What one training step hands its caller, as float32 / float64 .npy files in out_dir:
      loss.npy          the float32 loss the step returns
      loss_terms.npy    float64 [x, y, w, h, conf, cls, total] of RegionLossV2 (the reference's log line)
      counts.npy        float64 [nGT, nCorrect, nProposals]
      param.<name>.npy  the parameter after the SGD update, flattened in logical (OIHW) order
      grad.<name>.npy   its gradient, same order
    Tensors larger than DUMP_SAMPLE values are sampled at sorted positions drawn from a generator seeded with
    (DUMP_SEED, parameter index), so two runs or two builds sample the same positions."""
    os.makedirs(out_dir, exist_ok=True)

    def save(name, a):
        np.save(os.path.join(out_dir, name + '.npy'), a)
    losses = region_loss.last['losses'].cpu().numpy()
    counters = region_loss.last['counters'].cpu().numpy()
    save('loss', losses[6].astype(np.float32))     # the returned loss is losses[6] cast to float32
    save('loss_terms', losses[:7])
    save('counts', np.array([counters[0], counters[1], losses[7]], dtype=np.float64))
    for i, (name, p) in enumerate(model.named_parameters()):
        n = p.numel()
        idx = None
        if n > DUMP_SAMPLE:
            pos = np.sort(np.random.default_rng([DUMP_SEED, i]).choice(n, DUMP_SAMPLE, replace=False))
            idx = torch.from_numpy(pos).to(p.device)
        for tag, t in (('param', p), ('grad', p.grad)):
            if t is None:
                continue
            v = t.detach().reshape(-1)
            if idx is not None:
                v = v[idx]
            save('%s.%s' % (tag, name), v.float().cpu().numpy())


def fair_cpu_rate(B_ref, B_full, t_step, t_support):
    """images/s of the CPU arm at the GPU arm's query:support ratio.  The CPU step is a bounded sample of B_ref query
    images but pays the whole support branch (n_cls images) every step, which the GPU arm amortises over B_full query
    images: time per full step = (t_step - t_support) * B_full / B_ref + t_support."""
    t_full = (t_step - t_support) * B_full / B_ref + t_support
    return B_full / t_full


def cpu_build_targets_ms(B, ncls, G=13):
    """Reference-side value of the metric's second half: build_targets on the host."""
    from fewshot_detection_b200 import netcfg
    from oracle import region_loss as ORL
    from seeding import synth_targets
    anchors = [float(a) for a in netcfg.VOC_ANCHORS.split(',')]
    nB = B * ncls
    tgt = synth_targets(B, ncls, 77, max_gt=5).reshape(nB, 250)
    rs = np.random.RandomState(5)
    n = nB * 5 * G * G
    pred = np.abs(rs.randn(n, 4)).astype(np.float32) * 3 + 0.1
    t0 = time.perf_counter()
    ORL.build_targets(pred, tgt, anchors, 5, G, G, 1.0, 5.0, 0.6, 20000)
    return (time.perf_counter() - t0) * 1e3


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    threads = cpu_threads()
    B = args.ref_batch
    step, state = cpu_step_factory(args.ncls, args.side, B, threads)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    state['support_only']()
    t1 = time.perf_counter()
    for _ in range(2):
        state['support_only']()
    t_sup = (time.perf_counter() - t1) / 2
    raw = B * args.steps / dt
    val = fair_cpu_rate(B, args.batch, dt / args.steps, t_sup)
    sample = '%d query + %d support images per step, oracle port, torch %s CPU, %d threads; value = images/s at the GPU ' \
             "arm's ratio of %d query : %d support images per step, i.e. the support branch (%.2f s of the %.2f s sample step) " \
             'charged once per %d query images (raw sample rate %.3f img/s)' % (
                 B, args.ncls, torch.__version__, threads, args.batch, args.ncls, t_sup, dt / args.steps, args.batch, raw)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'images/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'configs[1]: darknet_dynamic + reweighting_net base-train step, %dx%d, %d classes, 5 anchors'
                               % (args.side, args.side, args.ncls), 'batch_per_step': B, 'n_cls': args.ncls,
                   'neg': 'full', 'host': 'cpu', 'support_branch': 'pro-rated to %d query images per step' % args.batch},
        'cpu_baseline': {'value': val, 'unit': 'images/s', 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': val, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


_JSON_FD = None


def quiet_stdout():
    """Point fd 1 at stderr for the whole run and keep the original for the JSON line: NCCL's version / INFO lines,
    the reference-style 'class_scale' print and anything a library writes to stdout would otherwise sit beside the
    one line the driver parses."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + '\n').encode()
    fd = _JSON_FD if _JSON_FD is not None else 1
    while data:
        data = data[os.write(fd, data):]


def teardown(dist, holders):
    """Leave the process group without hanging: CUDA graphs that captured NCCL work must be destroyed BEFORE their
    communicator, and a watchdog ends the process if the teardown itself stalls (the JSON line is already out)."""
    import gc
    sys.stdout.flush()
    sys.stderr.flush()
    wd = threading.Timer(30.0, lambda: os._exit(0))
    wd.daemon = True
    wd.start()
    try:
        for h in holders:
            if h is not None and hasattr(h, 'entries'):
                h.entries.clear()
        holders.clear()
        gc.collect()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    except Exception as e:
        sys.stderr.write('destroy_process_group: %r\n' % (e,))
    wd.cancel()


def main():
    args = parse()
    quiet_stdout()
    if args.impl == 'reference':
        return run_reference(args)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the hot path has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    import torch.distributed as dist
    if world > 1:
        if rank == 0:      # communicator / algorithm lines (NVLS, rings, trees) of rank 0 - on STDERR: stdout carries the JSON line
            if not os.environ.get('FSDET_NCCL_QUIET'):
                os.environ['NCCL_DEBUG'] = 'INFO'
                os.environ.setdefault('NCCL_DEBUG_SUBSYS', 'INIT,GRAPH,TUNING')
        dist.init_process_group('nccl', device_id=dev)
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    from fewshot_detection_b200 import netcfg, _lib, engine as _engine
    engine_terms = dict(_engine.TC_TERMS, persist=_engine.TC_PERSIST, cluster=_engine.TC_CLUSTER)
    from fewshot_detection_b200.cfg import cfg
    from fewshot_detection_b200.darknet_meta import Darknet
    from fewshot_detection_b200.optim import FusedSGD
    from fewshot_detection_b200.distributed import GradAllReducer
    from fewshot_detection_b200.graph import GraphedTrainStep
    from fewshot_detection_b200.region_loss import build_targets
    from seeding import seeded_init

    B, ncls, side = args.batch, args.ncls, args.side
    cfg.neg_ratio = 'full'
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):  # the reference's RegionLossV2.__init__ prints 'class_scale'
        model = Darknet(netcfg.darknet_dynamic_blocks(side, side), netcfg.reweighting_net_blocks())
    seeded_init(model, 0)            # identical replicas on every rank
    model = model.to(dev).train()
    region_loss = model.loss
    region_loss.verbose = False
    region_loss.seen = 20000
    global_batch = B * world
    factor = 15.0                    # train_meta.py:124-135 for neg='full'
    opt = FusedSGD(model.parameters(), lr=1e-3 / factor / global_batch, momentum=0.9, dampening=0,
                   weight_decay=0.0005 * global_batch * factor)
    reducer = GradAllReducer(model, bucket_mb=32)

    # two distinct host batches (pinned) per rank, alternated
    host = []
    for i in range(2):
        x, metax, mask, target = synth_batch(B, ncls, side, 1000 * rank + 10 * i)
        host.append((x.pin_memory(), metax.pin_memory(), mask.pin_memory(), target.pin_memory()))
    resident = [tuple(t.to(dev) for t in hb) for hb in host]
    h2d = sum(t.numel() * t.element_size() for t in host[0])

    def eager_step(x, metax, mask, target):
        reducer.begin_step()
        out = model(x, metax, mask)
        region_loss.seen += global_batch
        loss = region_loss(out, target)
        loss.backward()
        reducer.finish()
        opt.step()
        return loss

    graphed = None if args.no_graph else GraphedTrainStep(model, region_loss, opt, reducer)

    def step(x, metax, mask, target):
        if graphed is None:
            return eager_step(x, metax, mask, target)
        region_loss.seen += global_batch
        return graphed(x, metax, mask, target)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = {}

    def timed(fn, steps, tag=None, flush=None):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            fn(i)
        if flush is not None:
            flush()
        e1.record()
        if tag:
            host_ms[tag] = (time.perf_counter() - t0) * 1e3 / steps   # host-side enqueue time per step
        sync()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    # ---- device-resident throughput (value)
    for i in range(args.warmup):
        step(*resident[i % 2])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(lambda i: step(*resident[i % 2]), args.steps, 'value')
    clocks = sampler.stop() if rank == 0 else None
    value = global_batch * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:     # before the untimed steps below move the parameters on
        dump_outputs(args.dump_outputs, model, region_loss)

    # per-kernel timing + launch count: the same kernels launched eagerly (a CUDA-graph replay has no per-kernel
    # CUDA events), in the same run, right after the timed region
    prof = {}
    model._det.profile = prof
    model._ler.profile = prof
    reducer.overlap = world > 1 and graphed is None
    calls0 = dict(_lib.CALLS)
    prof_steps = 2
    for i in range(prof_steps):
        eager_step(*resident[i % 2])
    torch.cuda.synchronize()
    calls1 = dict(_lib.CALLS)
    model._det.profile = None
    model._ler.profile = None
    launches = sum((calls1.get(k, 0) - calls0.get(k, 0)) * LAUNCHES.get(k, 1) for k in calls1) * args.steps // prof_steps

    # per-kernel roofline of the dominant kernel (CUDA events recorded on the launching stream)
    launches_tbl = prof.pop('_launches', [])
    if os.environ.get('FSDET_DUMP_LAUNCHES') and rank == 0:
        rows = [(a.elapsed_time(b2) * 1e3, n, f, d) for (n, f, a, b2, d) in launches_tbl[len(launches_tbl) // 2:]]
        for us, n, f, d in sorted(rows, key=lambda r: -r[0]):
            sys.stderr.write('%9.1f us %-12s %7.1f TF/s  %s\n' % (us, n, f / us / 1e6, d[-9:]))
    kern = {}
    for name, (flops, evs) in prof.items():
        t = sum(a.elapsed_time(b) for a, b in evs)
        kern[name] = {'launches_per_step': len(evs) / prof_steps, 'ms_per_step': t / prof_steps,
                      'tflops_algorithmic': flops / (t / 1e3) / 1e12 if t > 0 else None}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops_sustained', 1400.0)
    peak_src = 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)' if peaks else 'fallback 1.4 PF (B200_PROFILING.md)'
    dom = max(kern, key=lambda k: kern[k]['ms_per_step']) if kern else None
    traffic = None
    try:
        rj = json.load(open(os.path.join(ROOT, 'profiles', 'roofline_r02.json' if os.path.exists(os.path.join(ROOT, 'profiles', 'roofline_r02.json')) else 'roofline_r01.json')))
        if rj.get('kernel') == dom:
            traffic = rj['traffic_bytes_per_launch']
    except Exception:
        pass
    roofline = None
    if dom:
        a = kern[dom]['tflops_algorithmic']
        roofline = {'kernel': dom, 'bound': 'tensor', 'achieved': a, 'peak': peak_tf, 'unit': 'TFLOP/s',
                    'frac': a / peak_tf, 'traffic': traffic, 'peak_source': peak_src,
                    'share_of_step': kern[dom]['ms_per_step'] / (ms / args.steps), 'kernels': kern,
                    'note': 'tcgen05 implicit GEMM (forward + input gradient) with fp16 hi/lo operand splitting: 3 tensor-core MMAs '
                            'per fp32-equivalent MAC, i.e. the tensor pipe does 3x the algorithmic FLOPs; measured against the bf16 peak. '
                            'Per-kernel times are CUDA-event timed eager launches in this run (the timed region '
                            'replays the same kernels from a CUDA graph)'}

    # Whole-step rooflines (SURVEY.md 8d): the north star asks for images/s as a fraction of the conv-stack HBM roofline
    # (fused algorithmic bytes: every layer reads its input and writes its output once, x3 for a training step, + 8
    # passes over the 265 MB of parameters) next to the tensor-pipe figure of the MMA layers.
    step_rooflines = None
    hbm_gbs = float(peaks.get('hbm_gbs', 6577.7))

    def whole_step(Bq, nc, sd, ms_step):
        alg_flops, alg_bytes = step_costs(Bq, nc, sd)
        t = ms_step / 1e3
        return {'hbm_frac': alg_bytes / t / 1e9 / hbm_gbs, 'tensor_frac': alg_flops / t / 1e12 / peak_tf,
                'algorithmic_GB': alg_bytes / 1e9, 'algorithmic_TFLOP': alg_flops / 1e12}
    try:
        if True:
            alg_flops, alg_bytes = step_costs(B, ncls, side)
            t = ms / args.steps / 1e3
            step_rooflines = {
                'hbm': {'algorithmic_bytes_per_step_per_gpu': alg_bytes, 'achieved_GBps': alg_bytes / t / 1e9,
                        'peak_GBps': hbm_gbs, 'frac': alg_bytes / t / 1e9 / hbm_gbs, 'floor_ms': alg_bytes / hbm_gbs / 1e6},
                'tensor': {'algorithmic_flops_per_step_per_gpu': alg_flops, 'achieved_TFLOPs': alg_flops / t / 1e12,
                           'peak_TFLOPs': peak_tf, 'frac': alg_flops / t / 1e12 / peak_tf,
                           'note': 'forward / input-gradient GEMMs: fp32-equivalent arithmetic = 3 tensor-core MACs per MAC; '
                                   'weight-gradient GEMMs: 1 (engine.TC_TERMS, profiles/precision_budget_r02.log)'}}
            if roofline is not None:
                roofline['whole_step'] = step_rooflines
    except Exception as e:  # never lose the bench line over a derived figure
        sys.stderr.write('step rooflines skipped: %r\n' % (e,))

    # ---- end-to-end through the public API with HOST buffers (e2e)
    # Every step: the step's inputs travel from pinned host memory to the device (DevicePrefetcher: the copy of
    # batch i+1 is issued on a side stream while step i computes - what DataLoader(pin_memory=True) + .cuda() does
    # serially in train_meta.py:209-213); the float64 target travels with them (the reference keeps it on the host
    # because its build_targets runs there; RegionLoss here takes either).  It must NOT be uploaded on the training
    # stream: a small H2D copy queued behind the 190 MB prefetch on the same copy engine delays the step by the whole
    # transfer (measured with tools/e2e_probe.py: +2.9 ms/step).  The prefetcher is primed before the timed region,
    # so the region contains exactly `steps` input copies.
    # The loss of every step is read back to the host (AsyncLossReader: a 4-byte copy into pinned memory behind the
    # step, consumed one step late so that the launch of step i+1 does not wait for step i; the last value is
    # drained inside the timed region).
    from fewshot_detection_b200.prefetch import DevicePrefetcher, AsyncLossReader
    pf = DevicePrefetcher((host[i % 2] for i in range(args.steps + 4)), dev)
    reader = AsyncLossReader(depth=2)
    e2e_losses = []

    def e2e_step(i):
        x, metax, mask, tgt = next(pf)
        loss = step(x, metax, mask, tgt)
        reader.push(loss)                     # device -> host read of the step's result ...
        if reader.count == 2:
            e2e_losses.append(reader.pop())   # ... consumed while the next step is already queued
    for i in range(3):                        # untimed: staging buffers allocated, pipeline primed
        e2e_step(i)
    e2e_losses.extend(reader.drain())
    ms_e2e = timed(e2e_step, args.steps, flush=lambda: e2e_losses.extend(reader.drain()))
    assert len(e2e_losses) == args.steps + 3 and all(np.isfinite(v) for v in e2e_losses)
    e2e_value = global_batch * args.steps / (ms_e2e / 1e3)

    # ---- the reference's real training regimes and the other BASELINE configs, same model / optimizer / graph cache
    # (extra keys; each is a device-resident CUDA-graph replay loop like `value`, inputs larger than L2):
    #   neg1     configs[1] with cfg.neg_ratio = 1 (cfg/metayolo.data: base training; rows sampled on the host per step)
    #   eager    configs[1] with every kernel launched eagerly through ctypes (--no-graph path, host-bound)
    #   configs3 fine-tuning regime: 20 classes, cfg.neg_ratio = 0 (cfg/metatune.data)
    #   configs4 608x608, 80 classes (largest single-GPU variant: B = 64 per GPU)
    extras = {}

    def extra_line(tag, Bq, nc, sd, neg, nsteps, graph=True):
        try:
            hb = [synth_batch(Bq, nc, sd, 7000 + 1000 * rank + 10 * i) for i in range(2)]
            rb = [tuple(t.to(dev) for t in b[:3]) + (b[3],) for b in hb]       # labels stay on the host (neg_filter)
            cfg.neg_ratio = neg
            fn = (lambda i: step(*rb[i % 2])) if graph else (lambda i: eager_step(*rb[i % 2]))
            for i in range(4):      # first call of a new regime = graph capture; then three replays
                fn(i)
            # every step between its own pair of events as well: a one-off stall (allocator, first replay) shows as max >> min
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nsteps)]

            def fn_ev(i):
                evs[i][0].record()
                fn(i)
                evs[i][1].record()
            m_ = timed(fn_ev, nsteps)
            per = [a.elapsed_time(b) for a, b in evs]
            v = Bq * world * nsteps / (m_ / 1e3)
            extras[tag] = {'value': v, 'unit': 'images/s', 'ms_per_step': m_ / nsteps, 'steps': nsteps,
                           'ms_per_step_min_max': [min(per), max(per)],
                           'config': {'batch_per_gpu': Bq, 'n_cls': nc, 'side': sd, 'neg': str(neg),
                                      'launch': 'cuda-graph replay' if graph else 'eager'},
                           'roofline_whole_step': whole_step(Bq, nc, sd, m_ / nsteps)}
            del hb, rb
        except Exception as e:      # an extra line must never cost the headline
            extras[tag] = {'error': repr(e)}
            sys.stderr.write('extra line %s failed: %r\n' % (tag, e))
        finally:
            cfg.neg_ratio = 'full'
            torch.cuda.empty_cache()

    if graphed is not None and world == 1 and not os.environ.get('FSDET_BENCH_NO_EXTRAS'):
        extra_line('neg1', B, ncls, side, 1, max(4, args.steps // 2))
        extra_line('eager', B, ncls, side, 'full', 3, graph=False)
        extra_line('configs3', B, 20, 416, 0, max(4, args.steps // 2))
        extra_line('configs4', B, 80, 608, 'full', 4)

    # ---- build_targets ms/batch (decode output -> 9 target tensors + counters, device resident)
    nB = B * ncls
    G = side // 32
    pred = torch.rand(nB * 5 * G * G, 4, device=dev) * 3 + 0.1
    tgt_dev = resident[0][3].view(nB, 250)
    anchors = model.anchors
    for _ in range(3):
        build_targets(pred, tgt_dev, anchors, 5, 1, G, G, 1.0, 5.0, 0.6, 20000, sync=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        build_targets(pred, tgt_dev, anchors, 5, 1, G, G, 1.0, 5.0, 0.6, 20000, sync=False)
    e1.record()
    torch.cuda.synchronize()
    bt_gpu_ms = e0.elapsed_time(e1) / 20

    # ---- evaluation decode + NMS (SURVEY 8f row 1): head output -> thresholded candidates -> NMS survivors for all
    # B*n_cls (image, class) rows, device resident (valid_ensemble.py:145-162 does this in Python loops on the host)
    from fewshot_detection_b200.utils import region_detections
    gdet = torch.Generator().manual_seed(5)
    head = torch.randn(nB, 30, G, G, generator=gdet)
    head.view(nB, 5, 6, G, G)[:, :, 4] -= 2.0
    head_dev = head.to(dev)
    for _ in range(2):
        dets = region_detections(head_dev, 0.005, 1, anchors, 5, 0, 1, n_models=ncls).nms(0.45)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        dets = region_detections(head_dev, 0.005, 1, anchors, 5, 0, 1, n_models=ncls).nms(0.45)
    e1.record()
    torch.cuda.synchronize()
    det_gpu_ms = e0.elapsed_time(e1) / 10
    det_kept = int(dets.keep_count.sum().item())

    # ---- training-input augmentation ms/batch (SURVEY 8f row 3): B decoded 375x500 uint8 images -> crop, PIL-exact
    # bicubic resize, flip, HSV jitter, /255 -> [B,3,side,side] float32, device resident.  Kept LAST among the GPU work and
    # guarded: the newest kernel must never cost the bench line.
    aug = None
    try:
        if world != 1:
            raise RuntimeError('single-GPU runs only')
        import random as _random
        from fewshot_detection_b200 import image as IMG
        rsa = np.random.RandomState(17)
        _random.seed(17)
        srcs = [torch.from_numpy(rsa.randint(0, 256, (375, 500, 3)).astype(np.uint8)).to(dev) for _ in range(B)]
        aps = [IMG.draw_augmentation(500, 375, 0.2, 0.1, 1.5, 1.5) for _ in range(B)]
        aug_out = torch.empty(B, 3, side, side, device=dev)
        for _ in range(2):
            IMG.augment_batch(srcs, (side, side), aps, out=aug_out)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(10):
            IMG.augment_batch(srcs, (side, side), aps, out=aug_out)
        a1.record()
        torch.cuda.synchronize()
        aug = {'gpu_ms_per_batch': a0.elapsed_time(a1) / 10, 'images': B, 'source': '375x500 uint8 RGB', 'out': side,
               'filter': 'PIL BICUBIC', 'out_mean': float(aug_out.mean().item())}
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            try:
                from PIL import Image as _PILImage      # what the reference's worker processes run per image
                t0 = time.perf_counter()
                for k in range(8):
                    pim = _PILImage.fromarray(srcs[k].cpu().numpy(), 'RGB')
                    p = aps[k]
                    pim = pim.crop((p['pleft'], p['ptop'], p['pleft'] + p['cw'], p['ptop'] + p['ch'])).resize((side, side))
                    pim = pim.convert('HSV').convert('RGB')
                    np.asarray(pim, dtype=np.float32) / 255
                aug['cpu_pil_ms_per_image'] = (time.perf_counter() - t0) * 1e3 / 8
                aug['cpu_note'] = 'Pillow crop + resize + HSV round trip + ToTensor on one host core, 8 images (the reference ' \
                                  'runs this in 10 DataLoader workers, utils.py:463)'
            except Exception as e:
                aug['cpu_note'] = 'Pillow timing skipped: %r' % (e,)
    except Exception as e:
        if world == 1:
            sys.stderr.write('augment timing skipped: %r\n' % (e,))

    if rank != 0:
        if world > 1:
            teardown(dist, [graphed])
        return

    cpu_baseline = None
    bt_cpu_ms = None
    det_cpu_ms = None
    if world == 1 and not args.no_cpu_baseline:
        threads = cpu_threads()
        cstep, cstate = cpu_step_factory(ncls, side, args.ref_batch, threads)
        cstep()                                   # warm-up (oneDNN primitive creation)
        t0 = time.perf_counter()
        cstep()
        cstep()
        dt = (time.perf_counter() - t0) / 2
        cstate['support_only']()
        t0 = time.perf_counter()
        cstate['support_only']()
        t_sup = time.perf_counter() - t0
        cpu_baseline = {'value': fair_cpu_rate(args.ref_batch, B, dt, t_sup), 'unit': 'images/s', 'cores': threads, 'kind': 'port',
                        'raw_sample_rate': args.ref_batch / dt, 'support_branch_s': t_sup, 'sample_step_s': dt,
                        'sample': '2 full training steps (after 1 warm-up) of %d query + %d support images at %dx%d (oracle '
                                  'port: torch-CPU ops + Python build_targets); %d of %d host cores used, see cpu_threads(); '
                                  'value = images/s with the support branch charged once per %d query images, the GPU '
                                  "arm's query:support ratio (fair_cpu_rate)"
                                  % (args.ref_batch, ncls, side, side, threads, os.cpu_count() or 1, B)}
        bt_cpu_ms = cpu_build_targets_ms(B, ncls, G)
        # decode + NMS of ONE image's n_cls rows with the oracle port (Python loops, as the reference's)
        from oracle import utils as OU
        t0 = time.perf_counter()
        ob = OU.get_region_boxes_v2(head[:ncls], ncls, 0.005, 1, anchors, 5, 0, 1)
        for row in ob:
            OU.nms(row, 0.45)
        det_cpu_ms = (time.perf_counter() - t0) * 1e3

    line = {
        'metric': METRIC, 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms / args.steps, 'host_enqueue_ms_per_step': host_ms.get('value'), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'configs[1]: darknet_dynamic + reweighting_net base-train step (fwd + RegionLossV2 + bwd + '
                               'SGD), %dx%d, %d classes, 5 anchors' % (side, side, ncls),
                   'batch_per_gpu': B, 'global_batch': global_batch, 'n_cls': ncls, 'neg': 'full',
                   'parallelism': 'dp%d' % world, 'weights': 'seeded random init (no checkpoint offline)',
                   'launch': 'eager' if graphed is None else 'cuda-graph replay of the whole step',
                   'l2': 'inputs larger than L2: ~%.1f GB of activations are streamed per step (L2 = 126 MB)'
                         % (B * 105e6 / 1e9)},
        'e2e': {'value': e2e_value, 'unit': 'images/s', 'ms_per_step': ms_e2e / args.steps,
                'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                'input_staging': 'pinned host -> device on a copy stream, one batch ahead (prefetch.DevicePrefetcher)',
                'loss_readback': 'every step, 4 bytes into pinned memory, read one step late (prefetch.AsyncLossReader)'},
        'gpu_launches': int(launches),
        'clocks': clocks,
        'roofline': roofline,
        'cpu_baseline': cpu_baseline,
        'build_targets_ms': {'gpu': bt_gpu_ms, 'cpu_oracle': bt_cpu_ms, 'rows': nB, 'grid': G},
        'augment': aug,
        'extras': extras,
        'precision_policy': dict(engine_terms),
        'detect_nms_ms': {'gpu': det_gpu_ms, 'rows': nB, 'survivors': det_kept, 'cpu_oracle_one_image': det_cpu_ms,
                          'cpu_rows': ncls, 'note': 'decode + threshold 0.005 + NMS 0.45 of all (image, class) rows; the CPU '
                                                    'figure is the oracle port on the first image only (n_cls rows)'},
    }
    emit(line)
    if world > 1:
        teardown(dist, [graphed])


if __name__ == '__main__':
    main()
