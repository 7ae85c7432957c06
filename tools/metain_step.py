"""Cost of the cropped-object support inputs (metain_type 3 / 4) on one GPU, against the default image + mask (type 2).

    python tools/metain_step.py [--steps 20 --warmup 5 --rounds 3] [--out FILE.json]

Three measurements, each alternating the variants it compares and repeating them (`--rounds`):
  step    graphed meta-training step (darknet_dynamic + reweighting_net, RegionLossV2, backward, SGD) at B = 64 query
          images of 416 x 416 and 20 support images of 416 x 416, for metain_type 2, 3 and 4: images/s
  first   the support net's first convolution (+ BatchNorm partial rows) and its weight gradient at 7 input channels,
          20 x 416 x 416 -> 32: the direct NCHW kernels (fsdet_conv_first_fwd_stats + fsdet_conv_first_wgrad) against
          the generic path the engine took before (fsdet_nchw_to_nhwc + fsdet_conv_fwd + fsdet_conv_wgrad), same call
  finish  MetaBatcher.finish (the device half of a support batch: augmentation launches + masks) for 20 training
          images of 500 x 375, type 2 against type 3
Times come from CUDA events (step, first) or a host clock around work that ends in a device synchronise (finish).
The card's name, power limit and maximum SM clock are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))

import numpy as np  # noqa: E402
import torch  # noqa: E402

CHANNELS = {2: 4, 3: 7, 4: 6}


def card():
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()),
                            '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except Exception:
        q = ''
    f = [c.strip() for c in q.split(',')] if q else []
    return {'name': torch.cuda.get_device_name(), 'power_limit': f[1] if len(f) > 1 else None,
            'sm_max_clock': f[2] if len(f) > 2 else None}


def events_ms(fn, n):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def measure_steps(args, dev):
    from fewshot_detection_b200 import netcfg
    from fewshot_detection_b200.cfg import cfg
    from fewshot_detection_b200.darknet_meta import Darknet
    from fewshot_detection_b200.optim import FusedSGD
    from fewshot_detection_b200.distributed import GradAllReducer
    from fewshot_detection_b200.graph import GraphedTrainStep
    from seeding import seeded_init, synth_targets, synth_masks
    B, ncls, side = 64, 20, 416
    cfg.neg_ratio = 'full'
    runs = {}
    for t in (2, 3, 4):
        cfg.metain_type = t
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):
            model = Darknet(netcfg.darknet_dynamic_blocks(side, side), netcfg.reweighting_net_blocks(channels=CHANNELS[t]))
        seeded_init(model, 0)
        model = model.to(dev).train()
        L = model.loss
        L.verbose = False
        L.seen = 20000
        opt = FusedSGD(model.parameters(), lr=1e-3 / 15 / B, momentum=0.9, dampening=0, weight_decay=0.0005 * B * 15)
        red = GradAllReducer(model, bucket_mb=32)
        g = torch.Generator().manual_seed(10 + t)
        x = torch.rand(B, 3, side, side, generator=g).to(dev)
        metax = torch.rand(ncls, 3 if t == 2 else 6, 416, 416, generator=g).to(dev)
        mask = torch.from_numpy(synth_masks(ncls, 416, 11)).to(dev)
        tgt = torch.from_numpy(synth_targets(B, ncls, 12, max_gt=5)).to(dev)
        gs = GraphedTrainStep(model, L, opt, red)
        runs[t] = (gs, (x, metax, mask, tgt), L, model)
    for t, (gs, batch, L, _) in runs.items():      # warm-up (and capture) of every variant before any timing
        cfg.metain_type = t
        for _ in range(args.warmup):
            L.seen += 64
            gs(*batch)
    torch.cuda.synchronize()
    res = {t: [] for t in runs}
    for r in range(args.rounds):
        for t, (gs, batch, L, _) in runs.items():
            cfg.metain_type = t

            def one(i):
                L.seen += 64
                gs(*batch)
            ms = events_ms(one, args.steps)
            res[t].append({'ms_per_step': ms, 'images_per_s': 64 / ms * 1e3})
    cfg.metain_type = 2
    # the support net's first layer really takes the direct kernels at types 3 / 4: one profiled eager forward
    routes = {}
    for t, (_, batch, _, model) in runs.items():
        cfg.metain_type = t
        model._ler.profile = {}
        with torch.no_grad():
            model.meta_forward(batch[1], batch[2])
        routes[t] = sorted(k for k in model._ler.profile if not k.startswith('_'))[:6]
        model._ler.profile = None
    cfg.metain_type = 2
    out = {}
    for t in runs:
        ms = [v['ms_per_step'] for v in res[t]]
        out['type%d' % t] = {'rounds': res[t], 'median_ms': float(np.median(ms)), 'median_images_per_s': 64 / float(np.median(ms)) * 1e3,
                             'support_first_layer_kernels': routes[t]}
    base = out['type2']['median_ms']
    for t in (3, 4):
        out['type%d' % t]['extra_ms_vs_type2'] = out['type%d' % t]['median_ms'] - base
    return out


def measure_first(args, dev):
    from fewshot_detection_b200 import _lib
    call, lib = _lib.call, _lib.lib
    st = torch.cuda.current_stream().cuda_stream
    B, H, W, Cout, C0, C1 = 20, 416, 416, 32, 6, 1
    C, CP = C0 + C1, 8
    g = torch.Generator(device=dev).manual_seed(3)
    a = torch.rand(B, C0, H, W, device=dev, generator=g)
    m = (torch.rand(B, C1, H, W, device=dev, generator=g) > 0.5).float()
    w = torch.zeros(Cout, 9, CP, device=dev)
    w[:, :, :C] = torch.randn(Cout, 9, C, device=dev, generator=g) * 0.2
    dz = torch.randn(B * H * W, Cout, device=dev, generator=g)
    npix = B * H * W
    z_new = torch.empty(npix, Cout, device=dev)
    part_new = torch.empty(lib.fsdet_conv_first_stat_rows(B, H, W), 4 * Cout, device=dev)
    nws_new = lib.fsdet_conv_first_wgrad_workspace_floats_cin(B, H, W, C, Cout)
    ws_new = torch.empty(nws_new, device=dev)
    dw_new = torch.empty(Cout, 9, CP, device=dev)
    xin = torch.empty(npix, CP, device=dev)
    z_gen = torch.empty(npix, Cout, device=dev)
    part_gen = torch.empty(lib.fsdet_conv_stat_rows(npix), 4 * Cout, device=dev)
    nws_gen = lib.fsdet_conv_wgrad_workspace_floats(B, H, W, CP, Cout, 3)
    ws_gen = torch.empty(max(nws_gen, 4), device=dev)
    dw_gen = torch.empty(Cout, 9, CP, device=dev)

    def new_fwd(_):
        call('fsdet_conv_first_fwd_stats', a.data_ptr(), C0, m.data_ptr(), C1, w.data_ptr(), z_new.data_ptr(), Cout, B, H, W, Cout,
             part_new.data_ptr(), st)

    def new_wgrad(_):
        call('fsdet_conv_first_wgrad', a.data_ptr(), C0, m.data_ptr(), C1, dz.data_ptr(), Cout, dw_new.data_ptr(), ws_new.data_ptr(),
             nws_new, B, H, W, Cout, st)

    def gen_fwd(_):
        call('fsdet_nchw_to_nhwc', a.data_ptr(), C0, m.data_ptr(), C1, xin.data_ptr(), CP, CP, B, H * W, st)
        call('fsdet_conv_fwd', xin.data_ptr(), CP, w.data_ptr(), None, z_gen.data_ptr(), Cout, part_gen.data_ptr(), B, H, W, CP, Cout,
             3, 0, st)

    def gen_wgrad(_):
        call('fsdet_conv_wgrad', xin.data_ptr(), CP, dz.data_ptr(), Cout, dw_gen.data_ptr(), ws_gen.data_ptr(), nws_gen, B, H, W, CP,
             Cout, 3, st)

    fns = {'new_fwd_stats': new_fwd, 'new_wgrad': new_wgrad, 'generic_fwd_stats': gen_fwd, 'generic_wgrad': gen_wgrad}
    for fn in fns.values():
        for i in range(3):
            fn(i)
    torch.cuda.synchronize()
    same = {'z_rel': ((z_new - z_gen).norm() / z_gen.norm()).item(), 'dw_rel': ((dw_new - dw_gen).norm() / dw_gen.norm()).item(),
            'dw_padding_zero': bool((dw_new[:, :, C:] == 0).all())}
    res = {k: [] for k in fns}
    for r in range(args.rounds):
        for k, fn in fns.items():
            res[k].append(events_ms(fn, 20))
    med = {k: float(np.median(v)) for k, v in res.items()}
    return {'shape': {'B': B, 'H': H, 'W': W, 'Cin': C, 'Cout': Cout}, 'ms_rounds': res, 'median_ms': med,
            'new_total_ms': med['new_fwd_stats'] + med['new_wgrad'], 'generic_total_ms': med['generic_fwd_stats'] + med['generic_wgrad'],
            'agreement': same}


def measure_finish(args, dev):
    from fewshot_detection_b200.cfg import cfg
    from fewshot_detection_b200.dataset import MetaBatcher
    keys = ('meta_width', 'meta_height', 'mask_width', 'mask_height', 'base_classes', 'metain_type')
    old = {k: cfg.get(k) for k in keys}
    cfg.meta_width = cfg.meta_height = cfg.mask_width = cfg.mask_height = 416
    ncls = 20
    cfg.base_classes = cfg.voc_classes[:ncls]
    rs = np.random.RandomState(0)
    pool = [[(rs.randint(0, 256, (375, 500, 3)).astype(np.uint8), np.array([[0.5, 0.5, 0.4, 0.5]]))] * 2 for _ in range(ncls)]
    inds = [(c, 0) for c in range(ncls)]
    res = {2: [], 3: []}
    batchers = {}
    for t in (2, 3):
        cfg.metain_type = t
        batchers[t] = MetaBatcher(pool, inds, train=True)
    random.seed(1)
    for r in range(args.rounds + 1):
        for t in (2, 3):
            cfg.metain_type = t
            mb = batchers[t]
            preps = [mb.prepare(range(ncls)) for _ in range(10)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for p in preps:
                mb.finish(p)
            torch.cuda.synchronize()
            if r:                                  # round 0 warms up
                res[t].append((time.perf_counter() - t0) * 1e3 / len(preps))
    for k, v in old.items():
        if v is None:
            cfg.pop(k, None)
        else:
            cfg[k] = v
    return {'images': ncls, 'source': [375, 500], 'size': 416, 'ms_rounds': {'type%d' % t: v for t, v in res.items()},
            'median_ms': {'type%d' % t: float(np.median(v)) for t, v in res.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None, help='also write the JSON result here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('metain_step.py measures on a GPU; none found')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    res = {'card': card(), 'first_layer_7ch': measure_first(args, dev), 'finish': measure_finish(args, dev),
           'step_B64_ncls20_416': measure_steps(args, dev)}
    res['card_after'] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()
