#!/usr/bin/env python
"""End-to-end run of the command-line driver (tools/train_meta_b200.py = the reference's train_meta.py loop) on a
throw-away VOC-shaped directory: JPEG files + Darknet label files + image list + per-class support dict + .data file +
.cfg files, base-training protocol of cfg/metayolo.data (15 base classes, novel split 0, neg = 1, multi-scale on).

    python tools/e2e_train_synth.py [n_images] [epochs] [out.json] [--metain-type N]  (one GPU; N = 2 by default)
    torchrun --nproc-per-node 2 tools/e2e_train_synth.py ...                    (one process per GPU)

Prints the driver's log, then one JSON line: images/s of the whole loop (file decode, augmentation, graph-replayed
steps, weight saves) and of its steady state (after the first epoch: graphs captured, files in the page cache).
"""
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
VOC = ["aeroplane", "bicycle", "bird", "boat", "bottle", "bus", "car", "cat", "chair", "cow", "diningtable", "dog", "horse",
       "motorbike", "person", "pottedplant", "sheep", "sofa", "train", "tvmonitor"]


def make_dataset(root, n, seed=0):
    from PIL import Image
    rs = np.random.RandomState(seed)
    for d in ('JPEGImages', 'labels', 'lists'):
        os.makedirs(os.path.join(root, d), exist_ok=True)
    imgs, per_class = [], {c: [] for c in VOC}
    for i in range(n):
        h, w = (375, 500) if i % 3 else (500, 375)
        base = rs.randint(0, 256, (h // 25 + 1, w // 25 + 1, 3)).astype(np.uint8)
        a = np.kron(base, np.ones((25, 25, 1), dtype=np.uint8))[:h, :w]
        a = np.clip(a.astype(np.int16) + rs.randint(-20, 20, a.shape), 0, 255).astype(np.uint8)
        p = os.path.join(root, 'JPEGImages', '%06d.jpg' % i)
        Image.fromarray(a, 'RGB').save(p, quality=90)
        imgs.append(p)
        rows = []
        for _ in range(int(rs.randint(1, 4))):
            c = int(rs.randint(0, 20))
            bw, bh = rs.uniform(0.15, 0.6, 2)
            rows.append((c, rs.uniform(bw / 2, 1 - bw / 2), rs.uniform(bh / 2, 1 - bh / 2), bw, bh))
            per_class[VOC[c]].append((p, rows[-1]))
        with open(os.path.join(root, 'labels', '%06d.txt' % i), 'w') as f:
            f.write(''.join('%d %.6f %.6f %.6f %.6f\n' % r for r in rows))
    with open(os.path.join(root, 'lists', 'train.txt'), 'w') as f:
        f.write(''.join(p + '\n' for p in imgs))
    # support dictionary: per class a list of images + per-class single-class label files (labels_1c/<class>/)
    lines = []
    for ci, c in enumerate(VOC):
        os.makedirs(os.path.join(root, 'labels_1c', c), exist_ok=True)
        if not per_class[c]:
            per_class[c] = [(imgs[ci], (ci, 0.5, 0.5, 0.4, 0.4))]
        lp = os.path.join(root, 'lists', 'support_%s.txt' % c)
        with open(lp, 'w') as f:
            for p, row in per_class[c]:
                f.write(p + '\n')
                with open(os.path.join(root, 'labels_1c', c, os.path.basename(p).replace('.jpg', '.txt')), 'a') as g:
                    g.write('%d %.6f %.6f %.6f %.6f\n' % row)
        lines.append('%s %s' % (c, lp))
    with open(os.path.join(root, 'lists', 'dict_full.txt'), 'w') as f:
        f.write('\n'.join(lines) + '\n')
    with open(os.path.join(root, 'novels.txt'), 'w') as f:
        f.write('bird,bus,cow,motorbike,sofa\naeroplane,bottle,cow,horse,sofa\n')


def main():
    metain_type = 2                 # --metain-type N: the support-input form written to the .data file (1..4)
    if '--metain-type' in sys.argv:
        i = sys.argv.index('--metain-type')
        metain_type = int(sys.argv[i + 1])
        del sys.argv[i:i + 2]
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 512
    epochs = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    outp = sys.argv[3] if len(sys.argv) > 3 else None
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    root = os.environ.get('FSDET_SYNTH_ROOT') or os.path.join(tempfile.gettempdir(), 'fsdet_synth_voc_%d' % n)
    if rank == 0 and not os.path.exists(os.path.join(root, 'novels.txt')):
        make_dataset(root, n)
    if world > 1:
        time.sleep(0 if rank == 0 else 8)
        while not os.path.exists(os.path.join(root, 'novels.txt')):
            time.sleep(1)
    from fewshot_detection_b200 import netcfg
    batch = 64 * world
    det = netcfg.darknet_dynamic_blocks()
    det[0]['batch'] = str(batch)
    with open(os.path.join(root, 'lists', 'train.txt')) as f:
        nsamples_all = len(f.readlines())
    det[0]['max_batches'] = str(max(1, (epochs - 1) * nsamples_all // batch))     # max_epochs = max_batches*batch//nsamples + 1
    netcfg.write_cfg(det, os.path.join(root, 'dyn.cfg'))
    netcfg.write_cfg(netcfg.reweighting_net_blocks(), os.path.join(root, 'rw.cfg'))   # channels follow metain_type
    backup = os.path.join(root, 'backup')
    with open(os.path.join(root, 'meta.data'), 'w') as f:
        f.write('metayolo=1\nmetain_type=%d\ndata=voc\nneg = 1\nrand = 0\nnovel = %s\nnovelid = 0\nmeta = %s\ntrain = %s\n'
                'backup = %s\ngpus=%s\n' % (metain_type, os.path.join(root, 'novels.txt'), os.path.join(root, 'lists', 'dict_full.txt'),
                                           os.path.join(root, 'lists', 'train.txt'), backup, ','.join(str(i) for i in range(world))))
    import importlib.util
    spec = importlib.util.spec_from_file_location('train_meta_b200', os.path.join(ROOT, 'tools', 'train_meta_b200.py'))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    from fewshot_detection_b200 import trainer as T
    marks = []
    orig = T.MetaTrainer.train_epoch

    def timed_epoch(self, epoch, max_epochs=None):
        import torch
        torch.cuda.synchronize()
        t0 = time.time()
        nb = orig(self, epoch, max_epochs)
        torch.cuda.synchronize()
        marks.append((nb, time.time() - t0))
        return nb
    T.MetaTrainer.train_epoch = timed_epoch
    # initial weights: the reference starts from a pretrained trunk; a purely random detector emits box sizes e^N(0, s)
    # that blow the w/h loss up within a few steps.  Write a Darknet weight file (exercises save_weights / load_weights)
    # whose head convolution is scaled down so that training starts from near-zero box offsets.
    wfile = os.path.join(root, 'init.weights' if metain_type == 2 else 'init_in%d.weights' % metain_type)
    if rank == 0 and not os.path.exists(wfile):
        import torch
        from fewshot_detection_b200.darknet_meta import Darknet
        torch.manual_seed(0)
        m0 = Darknet(det, netcfg.reweighting_net_blocks(channels={1: 3, 2: 4, 3: 7, 4: 6}[metain_type]))
        head = [mod for mod in m0.models if isinstance(mod, torch.nn.Sequential)][-1][0]
        with torch.no_grad():
            head.weight.mul_(0.02)
            head.bias.zero_()
        m0.save_weights(wfile + '.tmp')
        os.replace(wfile + '.tmp', wfile)
        del m0
    while not os.path.exists(wfile):
        time.sleep(1)
    sys.argv = ['train_meta_b200.py', os.path.join(root, 'meta.data'), os.path.join(root, 'dyn.cfg'), os.path.join(root, 'rw.cfg'), wfile]
    os.environ.setdefault('FSDET_SEED', '1')
    from fewshot_detection_b200.cfg import cfg as _cfg
    _cfg.save_interval = 2          # write a weight file inside a 3-epoch run (the default of 10 never would)
    t0 = time.time()
    rc = cli.main()
    total = time.time() - t0
    if rank == 0:
        from fewshot_detection_b200.cfg import _backup_dir
        bdir = _backup_dir({'backup': backup}, 0)
        steps = sum(nb for nb, _ in marks)
        steady = marks[1:] if len(marks) > 1 else marks
        line = {'rc': rc, 'world': world, 'images': n, 'metain_type': metain_type, 'backup_dir': bdir, 'global_batch': batch, 'epochs': len(marks), 'steps': steps,
                'loop_images_per_s': steps * batch / sum(t for _, t in marks),
                'steady_images_per_s': sum(nb for nb, _ in steady) * batch / sum(t for _, t in steady),
                'epoch_seconds': [round(t, 3) for _, t in marks], 'wall_s_incl_setup': total,
                'weights_saved': sorted(os.listdir(bdir)) if os.path.isdir(bdir) else
                sorted(os.listdir(backup)) if os.path.isdir(backup) else []}
        print(json.dumps(line))
        if outp:
            with open(outp, 'w') as f:
                json.dump(line, f)
    return rc


if __name__ == '__main__':
    sys.exit(main())
