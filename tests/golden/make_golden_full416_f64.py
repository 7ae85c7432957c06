#!/usr/bin/env python
"""Mint tests/golden/meta_full416_f64.npz: the REFERENCE's darknet_dynamic + reweighting_net meta-model at 416x416
(the case of meta_full416.npz: seed 61, 1 query image, 2 classes) run in float64, imported through
make_golden.load_ref (mechanical Py3 patches only) - build container only:

    python tests/golden/make_golden_full416_f64.py

The network runs in float64; the region loss stays float32 as in the reference (it is applied to the float32 cast of the
head output and its gradient is fed back in float64).  The float32 gradients of this network move by up to ~4e-3 with
the CPU's convolution kernels (thread count, instruction set), so a float32 digest only reproduces on a CPU that picks
the kernels of the one that minted it; the float64 digest reproduces to ~1e-9 with AVX2 or AVX-512 kernels at any
thread count.  Stored: the head output, the loss, and per parameter the gradient's norm and first 64 values.
"""
import io
import os
import sys
from contextlib import redirect_stdout

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as MG                                # noqa: E402  (sets sys.path for the reference and the shims)
from seeding import seeded_init, synth_targets, synth_masks  # noqa: E402
from fewshot_detection_b200 import netcfg               # noqa: E402


def main():
    with redirect_stdout(io.StringIO()):
        MG.importlib.import_module('utils')
        ref_cfg = MG.importlib.import_module('cfg')
    RL = MG.load_ref('region_loss')
    DM = MG.load_ref('darknet_meta')
    ref_cfg.cfg.neg_ratio = 'full'
    bs, cs, side, seed, seen = 1, 2, 416, 61, 20000
    with redirect_stdout(io.StringIO()):
        m = DM.Darknet(netcfg.darknet_dynamic_blocks(), netcfg.reweighting_net_blocks())
    seeded_init(m, seed)
    m.double().train()
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(bs, 3, side, side, generator=g)
    metax = torch.rand(cs, 3, side, side, generator=g)
    mask = torch.from_numpy(synth_masks(cs, side, seed + 2))
    tgt = synth_targets(bs, cs, seed + 3, max_gt=4)
    out = m(x.double(), metax.double(), mask.double())
    o32 = out.detach().float().requires_grad_(True)
    L = m.models[len(m.models) - 1]
    L.seen = seen
    orig_bt = RL.build_targets
    RL.build_targets = lambda pb, tg, *a: orig_bt(MG._Legacy2D(pb), MG._Legacy2D(tg), *a)
    buf = io.StringIO()
    try:
        with redirect_stdout(buf):
            loss = L(o32, torch.from_numpy(tgt))
    finally:
        RL.build_targets = orig_bt
    loss.backward()
    out.backward(o32.grad.double())
    r = dict(target=tgt, output=out.detach().numpy(), bs=bs, cs=cs, side=side, meta_side=side, seed=seed, seen=seen,
             loss=np.float64(loss.item()), log_line=buf.getvalue().strip().splitlines()[-1])
    for name, p in m.named_parameters():
        r['gradnorm/' + name] = np.float64(p.grad.norm().item())
        r['gradhead/' + name] = p.grad.reshape(-1)[:64].numpy().copy()
    np.savez_compressed(os.path.join(HERE, 'meta_full416_f64.npz'), **r)
    print('wrote meta_full416_f64.npz: loss %.9f, %d parameters' % (loss.item(), len(list(m.parameters()))))


if __name__ == '__main__':
    main()
