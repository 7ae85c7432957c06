#!/usr/bin/env python
"""Mint tests/golden/metain.npz from the REFERENCE's own code for the support-input forms metain_type 1, 3 and 4
(build container only; the reference is imported read-only, as in make_golden.py / make_golden_dataset.py):

    python tests/golden/make_golden_metain.py

(a) MetaDataset.__getitem__ (dataset.py:400-445, 519-530) at metain_type 3 and 4 - image + cropped object
    (`img.crop(mask rect).resize(img.size)`, dataset.py:386-390) and the mask - in training mode (augmented, with
    the re-draw loop) and in ensemble mode (identity transform, `filter`ed inds, with class ids), on the 48-pixel
    synthetic VOC-shaped directory of make_golden_dataset.py.  Both types return the same tensors (checked here), so
    they are stored once, under crop/: source pixels, label rows, pools, inds and the returned tensors (images as the
    uint8 bytes ToTensor divided by 255, masks as bytes).
(b) darknet_meta.Darknet on the mini architectures of make_golden.py's run_meta at metain_type 1, 3 and 4
    (learnet channels 3 / 7 / 6), inputs regenerated from the seed: output, RegionLossV2 loss and log line, the full
    gradient of the support net's small tensors (first convolution, BatchNorm vectors), and the norm and first 64
    values of every other gradient.
"""
import io
import os
import random
import sys
import tempfile
from contextlib import redirect_stdout

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
import make_golden as MG                                   # noqa: E402  (sets sys.path: shims, reference, repo)
from make_golden_augment import synth_image               # noqa: E402
from seeding import seeded_init, synth_targets, synth_masks  # noqa: E402
from fewshot_detection_b200 import netcfg                  # noqa: E402

CHANNELS = {1: 3, 2: 4, 3: 7, 4: 6}                        # reference cfg.py:158-178 (feat_layer 0)
FULL_GRAD = 2048


def regen_inputs(t, bs, cs, side, meta_side, seed):
    """(x, metax, mask) of the model fixture at metain_type t, from its seed (3 support channels for type 1, 6 else)."""
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(bs, 3, side, side, generator=g)
    metax = torch.rand(cs, 3 if t == 1 else 6, meta_side, meta_side, generator=g)
    return x, metax, torch.from_numpy(synth_masks(cs, meta_side, seed + 2))


def mint_dataset(out):
    with redirect_stdout(io.StringIO()):
        import dataset as RD                               # the reference's dataset.py
    from cfg import cfg as RC
    from PIL import Image
    tmp = tempfile.mkdtemp()
    os.makedirs(os.path.join(tmp, 'JPEGImages'))
    classes = RC.voc_classes
    RC.data, RC.multiscale, RC.metayolo, RC.yolo_joint = 'voc', 0, True, False
    RC.classes = classes
    RC.num_gpus, RC.batch_size, RC.randmeta = 1, 64, False
    RC.meta_width = RC.meta_height = RC.mask_width = RC.mask_height = 48
    ncls = 3
    RC.base_classes = classes[:ncls]
    RC.base_ids = list(range(ncls))
    rs = np.random.RandomState(71)
    for i in range(8):
        h, w = int(rs.randint(40, 64)), int(rs.randint(48, 80))
        a = synth_image(h, w, 700 + i, smooth=(i % 2 == 0))
        Image.fromarray(a, 'RGB').save(os.path.join(tmp, 'JPEGImages', '%06d.png' % i))
        out['src%d' % i] = a
    metadict = os.path.join(tmp, 'metadict.txt')
    with open(metadict, 'w') as f:
        for c in range(ncls):
            lst = os.path.join(tmp, 'meta_%s.txt' % classes[c])
            os.makedirs(os.path.join(tmp, 'labels_1c', classes[c]), exist_ok=True)
            with open(lst, 'w') as g:
                for i in range(8):
                    if (i + c) % 3 == 0:
                        continue
                    g.write(os.path.join(tmp, 'JPEGImages', '%06d.png' % i) + '\n')
                    rows = []
                    for k in range(int(rs.randint(0, 4))):
                        # tiny boxes (no mask at 48 pixels), 1-pixel-wide ones, the full image, ordinary ones
                        kind = rs.randint(0, 4)
                        if kind == 0:
                            bw, bh = rs.uniform(0.004, 0.012, 2)
                        elif kind == 1:
                            bw, bh = 1.0 / 48, rs.uniform(0.1, 0.6)
                        elif kind == 2:
                            bw, bh = 1.0, 1.0
                        else:
                            bw, bh = rs.uniform(0.05, 0.7, 2)
                        rows.append([c, rs.uniform(bw / 2, 1 - bw / 2) if bw < 1 else 0.5,
                                     rs.uniform(bh / 2, 1 - bh / 2) if bh < 1 else 0.5, bw, bh])
                    with open(os.path.join(tmp, 'labels_1c', classes[c], '%06d.txt' % i), 'w') as lf:
                        for r in rows:
                            lf.write('%d %.6f %.6f %.6f %.6f\n' % tuple(r))
                    out['meta_lab/%d/%d' % (c, i)] = np.loadtxt(
                        os.path.join(tmp, 'labels_1c', classes[c], '%06d.txt' % i)).reshape(-1, 5) if rows else np.zeros((0, 5))
            f.write('%s %s\n' % (classes[c], lst))
    got = {}
    for t in (3, 4):
        RC.metain_type = t
        for mode in ('train', 'ensemble'):
            np.random.seed(81)
            random.seed(82)
            with redirect_stdout(io.StringIO()):
                if mode == 'train':
                    ms = RD.MetaDataset(metadict, train=True, num_workers=0)
                else:
                    RC.classes = classes[:ncls]
                    ms = RD.MetaDataset(metadict, train=False, num_workers=0, ensemble=True, with_ids=True)
                    RC.classes = classes
            inds = list(ms.inds)[:2 * ncls] if mode == 'train' else list(ms.inds)
            r = {'inds': np.array(inds, dtype=np.int64),
                 'pool': np.array([[int(os.path.basename(l.strip())[:6]) for l in ms.metalines[c]]
                                   + [-1] * (8 - len(ms.metalines[c])) for c in range(ncls)], dtype=np.int64)}
            imgs, masks, ids = [], [], []
            random.seed(83)
            for k in range(len(inds)):
                item = ms[k]
                imgs.append(item[0].numpy())
                masks.append(item[1].numpy())
                if mode == 'ensemble':
                    ids.append(item[2])
            img, mask = np.stack(imgs), np.stack(masks)
            r['img_u8'] = np.rint(img * 255).astype(np.uint8)          # ToTensor of uint8 pixels: stored as those bytes
            assert np.array_equal(r['img_u8'].astype(np.float32) / np.float32(255), img)
            r['mask_u8'] = mask.astype(np.uint8)
            assert np.array_equal(r['mask_u8'].astype(np.float32), mask)
            if ids:
                r['ids'] = np.array(ids, dtype=np.int64)
            if t == 3:
                got[mode] = r
                for k, v in r.items():
                    out['crop/%s/%s' % (mode, k)] = v
            else:   # the reference crops for both types (dataset.py:386): the same draws give the same tensors
                assert set(r) == set(got[mode]) and all(np.array_equal(v, got[mode][k]) for k, v in r.items()), mode
            print(t, mode, 'inds', len(inds), 'img', img.shape)
    RC.metain_type = 2


def mint_models(out):
    with redirect_stdout(io.StringIO()):
        import cfg as ref_cfg
    RL = MG.load_ref('region_loss')
    DM = MG.load_ref('darknet_meta')
    cfg = ref_cfg.cfg
    cfg.neg_ratio = 'full'
    bs, cs, side, meta_side, seed, seen = 2, 3, 128, 64, 51, 20000
    for t in (1, 3, 4):
        cfg.metain_type = t
        det = netcfg.mini_dynamic_blocks(128, 4)
        ler = netcfg.mini_reweighting_blocks(64, 4, 128, channels=CHANNELS[t])
        with redirect_stdout(io.StringIO()):
            m = DM.Darknet([dict(b) for b in det], [dict(b) for b in ler])
        seeded_init(m, seed)
        m.train()
        g = torch.Generator().manual_seed(seed + 1)
        x = torch.rand(bs, 3, side, side, generator=g)
        metax = torch.rand(cs, 3 if t == 1 else 6, meta_side, meta_side, generator=g)
        mask = torch.from_numpy(synth_masks(cs, meta_side, seed + 2))
        tgt = synth_targets(bs, cs, seed + 3, max_gt=4)
        out_t = m(x, metax, mask)
        L = m.models[len(m.models) - 1]
        L.seen = seen
        orig_bt = RL.build_targets
        RL.build_targets = lambda pb, tg, *a: orig_bt(MG._Legacy2D(pb), MG._Legacy2D(tg), *a)
        buf = io.StringIO()
        try:
            with redirect_stdout(buf):
                loss = L(out_t, torch.from_numpy(tgt))
        finally:
            RL.build_targets = orig_bt
        loss.backward()
        key = 'model/in%d/' % t
        out.update({key + 'output': out_t.detach().numpy(), key + 'loss': np.float64(loss.item()),
                    key + 'log_line': buf.getvalue().strip().splitlines()[-1]})
        # inputs are regenerated from `seed` by the tests (regen_inputs below).  Gradients: in full for the support-net
        # tensors of up to FULL_GRAD values (its first convolution, whose input the type changes, and every BatchNorm
        # vector); norm + first 64 values for the rest
        assert all(torch.equal(a, b) for a, b in zip((x, metax, mask), regen_inputs(t, bs, cs, side, meta_side, seed)))
        for name, p in m.named_parameters():
            if name.startswith('learnet_models') and p.numel() <= FULL_GRAD:
                out[key + 'grad/' + name] = p.grad.numpy()
            else:
                out[key + 'gradnorm/' + name] = np.float64(p.grad.double().norm().item())
                out[key + 'gradhead/' + name] = p.grad.reshape(-1)[:64].numpy().copy()
        print('model', t, 'loss', loss.item())
    cfg.metain_type = 2
    out['model/dims'] = np.array([bs, cs, side, meta_side, seed, seen], dtype=np.int64)


def main():
    out = {}
    mint_models(out)
    mint_dataset(out)
    np.savez_compressed(os.path.join(HERE, 'metain.npz'), **out)
    print('wrote metain.npz', os.path.getsize(os.path.join(HERE, 'metain.npz')))


if __name__ == '__main__':
    main()
