"""Batch-at-a-time input pipeline: the per-sample work of the reference's dataset.py with the pixels on the device
(SURVEY.md 8f row 3).

The reference builds a batch from 64 `listDataset.__getitem__` calls (dataset.py:219-263) and n_cls
`MetaDataset.__getitem__` calls (dataset.py:519-530) spread over DataLoader worker processes, each doing PIL crop /
resize / flip / HSV work per image.  Here the host only decodes the files, draws the random numbers (same order as
the reference's single-process loader, so a seeded run sees the same crops) and transforms the labels; the pixel
work of the WHOLE batch is one `fsdet_augment_batch` launch (+ one `fsdet_box_masks` launch for the support masks).

  DetectionBatcher   query images + targets: multi-scale schedule (dataset.py:223-245), data_augmentation,
                     fill_truth_detection(_meta)
  MetaBatcher        support images + masks: get_metain (dataset.py:423-445) incl. its re-draw loop, get_img_mask
                     (dataset.py:378-398) for metain_type 1/2 and the cropped-object inputs 3/4 (a second augmentation
                     launch resizes the mask rectangle of each augmented image to full size)

The few-shot list construction (build_dataset / load_metadict / build_fewset, MetaDataset's index) lives in lists.py;
both classes here take already-built lists.  Entries may be image
paths (decoded on the host with PIL, label path derived like listDataset.get_labpath) or in-memory
(uint8 array, label array) pairs.
"""
import random

import numpy as np
import torch

from .cfg import cfg
from . import image as I

JITTER, HUE, SATURATION, EXPOSURE = 0.2, 0.1, 1.5, 1.5      # dataset.py:247-250, :401-404


def get_labpath(imgpath):
    """listDataset.get_labpath (dataset.py:265-271)."""
    return imgpath.replace('images', 'labels').replace('JPEGImages', 'labels').replace('.jpg', '.txt').replace('.png', '.txt')


def get_meta_labpath(imgpath, cls_name):
    """MetaDataset.get_labpath (dataset.py:532-548)."""
    sub = 'labels_1c/{}'.format(cls_name)
    if cfg.get('data', 'voc') == 'voc':
        return imgpath.replace('images', sub).replace('JPEGImages', sub).replace('.jpg', '.txt').replace('.png', '.txt')
    if 'train2014' in imgpath:
        return imgpath.replace('images/train2014', 'labels_1c/train2014/{}'.format(cls_name)) \
            .replace('.jpg', '.txt').replace('.png', '.txt')
    if 'val2014' in imgpath:
        return imgpath.replace('images/val2014', 'labels_1c/val2014/{}'.format(cls_name)) \
            .replace('.jpg', '.txt').replace('.png', '.txt')
    raise NotImplementedError('Image path note recognized!')


def multiscale_width(seen, first_batch=False, bs=64, batchs=4000):
    """The size schedule of dataset.py:226-245 (one draw from `random` per call past the first 4000 batches)."""
    if first_batch:
        return 19 * 32
    if seen < batchs * bs:
        return 13 * 32
    if seen < 2 * batchs * bs:
        return (random.randint(0, 3) + 13) * 32
    if seen < 3 * batchs * bs:
        return (random.randint(0, 5) + 12) * 32
    if seen < 4 * batchs * bs:
        return (random.randint(0, 7) + 11) * 32
    return (random.randint(0, 9) + 10) * 32


class _Entry(object):
    """An image given as a path or as a decoded array; the size is available without decoding a file twice."""

    def __init__(self, item, label=None):
        self.item, self.label, self._arr = item, label, None
        if not isinstance(item, str):
            self._arr = item

    def size(self):
        if self._arr is not None:
            return int(self._arr.shape[1]), int(self._arr.shape[0])
        hit = I._CACHE.get(self.item)
        if hit is not None:
            return int(hit.shape[1]), int(hit.shape[0])
        from PIL import Image
        with Image.open(self.item) as im:
            return im.size

    def pixels(self):
        if self._arr is None:
            self._arr = I._decode(self.item)
        return self._arr


class DetectionBatcher(object):
    """listDataset (dataset.py:182-263) a batch at a time.

    lines: image paths, or (uint8 [h, w, 3] array, label array [k, 5]) pairs.  `batch(indices)` returns
    (data float32 CUDA [B, 3, H, W], target float64 CPU [B, n_cls, 250] (cfg.metayolo) or [B, 250])."""

    def __init__(self, lines, shape=None, shuffle=True, train=False, seen=0, batch_size=64, num_workers=4, filter=None,
                 seen_step=None):
        """seen_step: by how much `seen` (the GLOBAL sample count that drives the multi-scale schedule) advances per
        sample of THIS batcher.  The reference adds `num_workers` per sample inside every DataLoader worker's private
        dataset copy, each of which sees 1/num_workers of the samples (dataset.py:262) - i.e. its copies track the
        global count.  One batcher that sees every sample must add 1 (single process) or the world size (one process
        per GPU, each batcher seeing 1/world of the global batch).  `num_workers` is kept for signature compatibility
        and only used as the step when seen_step is None and a legacy caller relies on it (tests pass 1)."""
        self.lines = list(lines)
        if shuffle:
            random.shuffle(self.lines)
        self.nSamples = len(self.lines)
        self.shape, self.train, self.seen = shape, train, seen
        self.batch_size, self.num_workers, self.filter = batch_size, num_workers, filter
        self.seen_step = num_workers if seen_step is None else seen_step
        self.first_batch = False

    def __len__(self):
        return self.nSamples

    def _entry(self, index):
        line = self.lines[index]
        if isinstance(line, str):
            path = line.rstrip()
            return _Entry(path, get_labpath(path))
        return _Entry(line[0], line[1])

    def batch(self, indices):
        return self.finish(self.prepare(indices))

    def prepare(self, indices):
        """Host half of a batch (may run in a background thread while the GPU trains on the previous batch): the
        random draws in the reference's order, file decode, label transforms.  Returns what finish() needs."""
        entries, params = [], []
        for index in indices:
            assert index <= len(self), 'index range error'
            if self.train and index % 64 == 0 and cfg.get('data', 'voc') != 'coco' and cfg.multiscale:
                width = multiscale_width(self.seen, self.first_batch)
                self.first_batch = False
                self.shape = (width, width)
            e = self._entry(index)
            ow, oh = e.size()
            p = I.draw_augmentation(ow, oh, JITTER, HUE, SATURATION, EXPOSURE) if self.train else I.identity_augmentation(ow, oh)
            p['shape'] = self.shape
            entries.append(e)
            params.append(p)
            self.seen = self.seen + self.seen_step
        shapes = set(p['shape'] for p in params)
        if len(shapes) != 1:
            raise ValueError('a batch must not straddle a multi-scale boundary (indices %r)' % (list(indices),))
        W, H = params[0]['shape']
        pixels = I.PackedImages(I.decode_many([e.item if e._arr is None else e._arr for e in entries])).marshal(params, W, H)
        fill = I.fill_truth_detection_meta if cfg.metayolo else I.fill_truth_detection
        labels = [fill(e.label, W, H, p['flip'], p['dx'], p['dy'], 1. / p['sx'], 1. / p['sy']) for e, p in zip(entries, params)]
        target = torch.from_numpy(np.stack(labels))
        try:
            target = target.pin_memory()          # the step uploads it asynchronously
        except RuntimeError:
            pass
        return pixels, (W, H), params, target

    def finish(self, prepared):
        """Device half: one augmentation launch for the whole batch."""
        pixels, shape, params, target = prepared
        return I.augment_batch(pixels, shape, params, filter=self.filter), target

    def batch_ranges(self):
        return [range(start, start + self.batch_size) for start in range(0, self.nSamples - self.batch_size + 1, self.batch_size)]

    def __iter__(self):
        for r in self.batch_ranges():
            yield self.batch(r)


class MetaBatcher(object):
    """MetaDataset.__getitem__ / get_metain (dataset.py:400-445, 519-530) a batch at a time.

    metalines[c]: the support pool of class c - image paths, or (uint8 array, boxes [k, 4..5] of that class) pairs;
    inds: sequence of (clsid, metaind) like MetaDataset.inds.  `batch(indices)` returns (metax float32 CUDA
    [n, C, S, S], mask float32 CUDA [n, 1, S, S][, clsids]).  C = 3 for metain_type 1 / 2 (the image); 6 for 3 / 4
    (the image, then its mask rectangle cropped and resized to S x S: dataset.py:386-390).  The mask comes back for
    every type, as in the reference; the network concatenates it for types 2 and 3 only."""

    def __init__(self, metalines, inds, classes=None, train=False, ensemble=False, with_ids=False, filter=None):
        if cfg.metain_type not in (1, 2, 3, 4):
            raise NotImplementedError('metain_type %r' % cfg.metain_type)
        self.crop = cfg.metain_type in (3, 4)
        self.metalines, self.inds = metalines, list(inds)
        self.classes = classes if classes is not None else (cfg.base_classes if train else cfg.classes)
        self.train, self.ensemble, self.with_ids, self.filter = train, ensemble, with_ids, filter
        self.meta_shape = (cfg.meta_width, cfg.meta_height)
        self.mask_shape = (cfg.mask_width, cfg.mask_height)
        self.batch_size = len(self.classes)      # one support image per class per process (MetaDataset.batch_size / num_gpus)

    def __len__(self):
        return len(self.inds)

    def _entry(self, clsid, item):
        if isinstance(item, int):
            item = self.metalines[clsid][item]
        if isinstance(item, str):
            path = item.rstrip()
            return _Entry(path, get_meta_labpath(path, self.classes[clsid]))
        boxes = np.asarray(item[1], dtype=np.float64)
        if boxes.size == 0:
            boxes = np.zeros((0, 5))
        elif boxes.reshape(len(boxes), -1).shape[1] == 4:         # (x, y, w, h) -> label rows with a class column
            boxes = np.concatenate([np.zeros((len(boxes), 1)), boxes.reshape(len(boxes), 4)], 1)
        return _Entry(item[0], boxes)

    def _try(self, e):
        """get_metaimg + the first box with a non-empty mask (dataset.py:400-432): (params, rect) or None."""
        ow, oh = e.size()
        p = I.draw_augmentation(ow, oh, JITTER, HUE, SATURATION, EXPOSURE) if self.train else I.identity_augmentation(ow, oh)
        W, H = self.meta_shape
        labs = I.load_label(e.label, W, H, p['flip'], p['dx'], p['dy'], 1. / p['sx'], 1. / p['sy'])
        for lab in labs:
            x1, y1, x2, y2 = I.mask_rect(lab, self.mask_shape[0], self.mask_shape[1])
            if x1 == x2 or y1 == y2:
                continue
            return p, (x1, y1, x2, y2)
        return None

    def get_metain(self, clsid, metaind):
        """(entry, params, rect), or None where the reference returns (None, None)."""
        e = self._entry(clsid, metaind)
        r = self._try(e)
        if r is not None:
            return (e,) + r
        while not self.ensemble:      # the selected image has only degenerate objects: draw another one (dataset.py:434-444)
            e = self._entry(clsid, random.sample(self.metalines[clsid], 1)[0])
            r = self._try(e)
            if r is not None:
                return (e,) + r
        return None

    def batch(self, indices):
        return self.finish(self.prepare(indices))

    def prepare(self, indices):
        """Host half (draws, decode, label transforms); see DetectionBatcher.prepare."""
        chosen, clsids = [], []
        for index in indices:
            clsid, metaind = self.inds[index]
            r = self.get_metain(clsid, metaind)
            if r is None:
                raise ValueError('support image (%d, %r) has no usable box (the reference returns (None, None))' % (clsid, metaind))
            chosen.append(r)
            clsids.append(clsid)
        pixels = I.PackedImages(I.decode_many([e.item if e._arr is None else e._arr for e, _, _ in chosen]))
        pixels.marshal([p for _, p, _ in chosen], self.meta_shape[0], self.meta_shape[1])
        rects = torch.from_numpy(np.array([r for _, _, r in chosen], dtype=np.int32).reshape(len(chosen), 4))
        try:
            rects = rects.pin_memory()
        except RuntimeError:
            pass
        return pixels, [p for _, p, _ in chosen], rects, clsids

    def finish(self, prepared):
        pixels, params, rects, clsids = prepared
        n = len(pixels)
        if self.crop:
            W, H = self.meta_shape
            metax = torch.empty(n, 6, H, W, dtype=torch.float32, device=I._default_device())
            _, u8 = I.augment_batch(pixels, self.meta_shape, params, filter=self.filter, out=metax[:, :3], return_uint8=True)
            # img.crop(mask rect).resize(img.size) of the augmented uint8 image, same resampling filter
            I.augment_batch([u8[i] for i in range(n)], self.meta_shape, [I.crop_params(r) for r in rects.tolist()],
                            filter=self.filter, out=metax[:, 3:])
        else:
            metax = I.augment_batch(pixels, self.meta_shape, params, filter=self.filter)
        w, h = self.mask_shape
        mask = torch.empty(n, 1, h, w, dtype=torch.float32, device=metax.device)
        I.call('fsdet_box_masks', I.ptr(rects.to(metax.device, non_blocking=True)), n, h, w, I.ptr(mask), I._st())
        if self.with_ids:
            return metax, mask, clsids
        return metax, mask
