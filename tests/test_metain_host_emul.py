"""The cropped-object support inputs (metain_type 3 / 4) on the CPU: the crop channels of the host-emulated
augmentation kernel against Pillow, MetaBatcher against the reference's MetaDataset (tests/golden/metain.npz, minted by
tests/golden/make_golden_metain.py), and the oracle's support-input rule against the reference model at types 1/3/4."""
import ctypes
import os
import random

import numpy as np
import pytest
import torch

from emul_util import build_emul, route_image_calls_to_emulation

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
NCLS = 3
CHANNELS = {1: 3, 2: 4, 3: 7, 4: 6}


def oracle_meta(det_blocks, learnet_blocks, metain_type):
    """oracle.darknet.MetaDarknet (which restates metain_type 2) with the reference's support-input rule for any type
    (darknet_meta.py:117-118): the mask is concatenated for types 2 and 3, `metax` goes in alone for 1 and 4."""
    from oracle import darknet as ODK

    class MetainDarknet(ODK.MetaDarknet):
        def meta_forward(self, metax, mask):
            if metain_type in (2, 3):
                return super().meta_forward(metax, mask)
            for model in self.learnet_models:
                metax = model(metax)
            return [metax]
    return MetainDarknet(det_blocks, learnet_blocks)


def regen_inputs(gold, t):
    """(x, metax, mask, target) of the fixture's mini-model run at metain_type t, regenerated from its seed."""
    from seeding import synth_masks, synth_targets
    bs, cs, side, ms, seed, _ = (int(v) for v in gold['model/dims'])
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(bs, 3, side, side, generator=g)
    metax = torch.rand(cs, 3 if t == 1 else 6, ms, ms, generator=g)
    mask = torch.from_numpy(synth_masks(cs, ms, seed + 2))
    return x, metax, mask, torch.from_numpy(synth_targets(bs, cs, seed + 3, max_gt=4))


@pytest.fixture(scope='module')
def emul():
    return build_emul('augment', 'augment.cu')


@pytest.fixture(scope='module')
def gold():
    return np.load(os.path.join(G, 'metain.npz'), allow_pickle=False)


def _route(monkeypatch, emul):
    """image.* C-ABI calls -> emulated kernels, including the pitched entry point."""
    I = route_image_calls_to_emulation(monkeypatch, emul)
    plain = I.call
    V = ctypes.c_void_p

    def call(name, *a):
        if name != 'fsdet_augment_batch_pitched':
            return plain(name, *a)
        src, geom, color, n, W, H, kmax, filt, ws, ws_bytes, out, pitch, out_u8, status, stream = a
        tbytes = n * 2 * max(W, H) * (2 + kmax) * 4
        assert ws_bytes >= tbytes + n * 768
        emul.emul_augment_batch_pitched(V(src), V(geom), V(color), n, W, H, kmax, filt, V(ws), V(ws + tbytes), V(out),
                                        ctypes.c_longlong(pitch), V(out_u8) if out_u8 else None, V(status))
        return 0
    monkeypatch.setattr(I, 'call', call)
    return I


def _pil_crop_resize(u8, rect, size, filt):
    from PIL import Image
    im = Image.fromarray(u8, 'RGB').crop(rect).resize(size, filt)
    return np.asarray(im, dtype=np.uint8)


@pytest.mark.parametrize('filt', [0, 3])
def test_crop_channels_equal_pillow(emul, gold, monkeypatch, filt):
    """Second launch of the cropped-object pipeline: uint8 image -> crop(rect).resize(size) -> /255 into channels 3..5
    of a 6-channel tensor, bit for bit what Pillow 12.2 computes (1-pixel-wide and -high crops, the full image -
    Pillow returns a copy - and up- and down-scaling)."""
    I = _route(monkeypatch, emul)
    cases = [((48, 48), (0, 0, 48, 48), (48, 48)),      # full image: a copy
             ((48, 48), (17, 3, 18, 40), (48, 48)),     # 1 pixel wide
             ((48, 48), (2, 30, 45, 31), (48, 48)),     # 1 pixel high
             ((48, 48), (5, 9, 12, 30), (48, 48)),      # up-scaling
             ((60, 70), (3, 4, 66, 57), (24, 20)),      # down-scaling in both axes
             ((60, 70), (10, 0, 30, 60), (48, 96))]     # down in one axis, up in the other
    for k, ((h, w), rect, size) in enumerate(cases):
        src = np.ascontiguousarray(gold['src%d' % k][:h, :w])
        W, H = size
        out = torch.full((2, 6, H, W), -1.0)
        srcs = [torch.from_numpy(src), torch.from_numpy(src[::-1].copy())]
        I.augment_batch(srcs, size, [I.crop_params(rect)] * 2, filter=filt, out=out[:, 3:])
        for i in range(2):
            want = _pil_crop_resize(srcs[i].numpy(), rect, size, filt)
            got = out[i, 3:].permute(1, 2, 0).numpy()
            assert np.array_equal(got, want.astype(np.float32) / np.float32(255)), (k, rect, size, i)
        assert (out[:, :3] == -1).all()                 # the pitched launch leaves the other channels alone


def _batcher(gold, cfg, metain_type, mode):
    from fewshot_detection_b200.dataset import MetaBatcher
    key = 'crop/%s/' % mode                   # the reference returns the same tensors for types 3 and 4
    cfg.metain_type = metain_type
    pool = gold[key + 'pool']
    metalines = [[(gold['src%d' % i], gold['meta_lab/%d/%d' % (c, i)]) for i in pool[c] if i >= 0] for c in range(NCLS)]
    inds = [tuple(int(v) for v in r) for r in gold[key + 'inds']]
    if mode == 'train':
        return MetaBatcher(metalines, inds, train=True, with_ids=True), inds, key
    return MetaBatcher(metalines, inds, classes=cfg.voc_classes[:NCLS], ensemble=True, with_ids=True), inds, key


@pytest.fixture()
def cfg48():
    from fewshot_detection_b200.cfg import cfg
    keys = ('data', 'multiscale', 'metayolo', 'yolo_joint', 'classes', 'base_classes', 'base_ids', 'metain_type',
            'meta_width', 'meta_height', 'mask_width', 'mask_height')
    old = {k: cfg.get(k) for k in keys}
    cfg.data, cfg.multiscale, cfg.metayolo, cfg.yolo_joint = 'voc', 0, True, False
    cfg.classes = cfg.voc_classes
    cfg.base_classes, cfg.base_ids = cfg.voc_classes[:NCLS], list(range(NCLS))
    cfg.meta_width = cfg.meta_height = cfg.mask_width = cfg.mask_height = 48
    yield cfg
    for k, v in old.items():
        if v is None:
            cfg.pop(k, None)
        else:
            cfg[k] = v


def run_batcher(gold, cfg, metain_type, mode):
    """All of the fixture's samples, one support image per class per batch: (metax, mask, ids) as numpy."""
    mb, inds, key = _batcher(gold, cfg, metain_type, mode)
    random.seed(83)
    xs, ms, ids = [], [], []
    for b in range(0, len(inds), NCLS):
        metax, mask, clsids = mb.batch(range(b, min(b + NCLS, len(inds))))
        assert tuple(metax.shape[1:]) == (6, 48, 48) and tuple(mask.shape[1:]) == (1, 48, 48)
        xs.append(metax.cpu().numpy())
        ms.append(mask.cpu().numpy())
        ids += clsids
    return np.concatenate(xs), np.concatenate(ms), ids, key


@pytest.mark.parametrize('metain_type', [3, 4])
@pytest.mark.parametrize('mode', ['train', 'ensemble'])
def test_meta_batcher_equals_reference(emul, gold, cfg48, monkeypatch, metain_type, mode):
    _route(monkeypatch, emul)
    metax, mask, ids, key = run_batcher(gold, cfg48, metain_type, mode)
    assert ids == [int(r[0]) for r in gold[key + 'inds']]
    if mode == 'ensemble':
        assert ids == gold[key + 'ids'].tolist()
    assert np.array_equal(mask, gold[key + 'mask_u8'].astype(np.float32))
    assert np.array_equal(metax, gold[key + 'img_u8'].astype(np.float32) / np.float32(255))


def run_oracle(gold, metain_type, double=False):
    from oracle import region_loss as ORL
    from fewshot_detection_b200 import netcfg
    from seeding import seeded_init
    bs, cs, side, ms, seed, seen = (int(v) for v in gold['model/dims'])
    key = 'model/in%d/' % metain_type
    ler = netcfg.mini_reweighting_blocks(ms, 4, 128, channels=CHANNELS[metain_type])
    m = oracle_meta(netcfg.mini_dynamic_blocks(side, 4), ler, metain_type)
    seeded_init(m, seed)
    x, metax, mask, target = regen_inputs(gold, metain_type)
    if double:
        m.double()
        x, metax, mask = x.double(), metax.double(), mask.double()
    m.train()
    out = m(x, metax, mask)
    o = out.detach().float().requires_grad_(True) if double else out
    loss = ORL.region_loss_v2(o, target, m.anchors, m.num_anchors, m.num_classes, seen=seen)
    loss.backward()
    if double:
        out.backward(o.grad.double())
    return m, out, loss, key


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


@pytest.mark.parametrize('metain_type', [1, 3, 4])
def test_oracle_follows_reference_support_input(gold, metain_type):
    m, out, loss, key = run_oracle(gold, metain_type)
    assert _rel(out.detach().numpy(), gold[key + 'output']) < 1e-6
    assert abs(loss.item() - float(gold[key + 'loss'])) < 1e-5 * abs(float(gold[key + 'loss']))
    n = 0
    for name, p in m.named_parameters():
        if key + 'grad/' + name in gold.files:
            assert _rel(p.grad.numpy(), gold[key + 'grad/' + name]) < 1e-5, name
            n += 1
        else:
            assert abs(p.grad.double().norm().item() - float(gold[key + 'gradnorm/' + name])) \
                < 1e-5 * float(gold[key + 'gradnorm/' + name]), name
            assert _rel(p.grad.reshape(-1)[:64].numpy(), gold[key + 'gradhead/' + name]) < 1e-4, name
    assert n == len([k for k in gold.files if k.startswith(key + 'grad/')])
    assert key + 'grad/learnet_models.0.conv1.weight' in gold.files     # the first convolution, in full
    assert m.learnet_models[0][0].weight.shape[1] == CHANNELS[metain_type]
