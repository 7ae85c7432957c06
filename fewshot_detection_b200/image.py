"""Training-input augmentation: the reference's image.py with the pixel work on the device (SURVEY.md 8f row 3).

Same names, arguments and random-number consumption as the reference (image.py:39-87, 90-260), so that a run seeded
like the reference's draws the same crops / flips / colour jitters:

  data_augmentation(img, shape, jitter, hue, saturation, exposure, flag=True) -> (img, flip, dx, dy, sx, sy)
  fill_truth_detection / fill_truth_detection_meta / load_label (label transforms, host numpy exactly as the
  reference: a few dozen float64 operations per image)
  load_data_detection / load_data_with_label

What changed: `img` may be a decoded uint8 RGB array / tensor [h, w, 3] (or a PIL image, or - in the load_* functions -
a path, decoded on the host with PIL like the reference), and the returned `img` is the float32 CUDA tensor [3, H, W]
that the reference obtains later from `transforms.ToTensor()` (train_meta.py:176-178) - crop, resize, flip, HSV jitter
and the /255 run in ONE kernel launch (csrc/augment.cu), bit-identical to Pillow's uint8 pipeline.  `augment_batch`
does a whole batch in that one launch (what the reference spreads over 10 DataLoader worker processes,
utils.py:463).  CUDA only: no host fallback.

Resize filter: the reference calls `cropped.resize(shape)` without a filter, i.e. Pillow's default - BICUBIC since
Pillow 7.0 (the container's 12.2), NEAREST in the Pillow of the reference's 2018 environment.  `DEFAULT_FILTER`
follows the installed behaviour (BICUBIC); pass `filter=NEAREST` for the old one.
"""
import math
import os
import random

import collections
import threading

import numpy as np
import torch

from .cfg import cfg
from ._lib import call, ptr, lib

NEAREST, BICUBIC = 0, 3        # PIL.Image.Resampling values
DEFAULT_FILTER = BICUBIC


def _st():
    return torch.cuda.current_stream().cuda_stream


def _default_device():
    return torch.device('cuda', torch.cuda.current_device())


def rand_scale(s):
    """image.py:39-43."""
    scale = random.uniform(1, s)
    if random.randint(1, 10000) % 2:
        return scale
    return 1. / scale


def draw_augmentation(ow, oh, jitter, hue, saturation, exposure):
    """The random draws of data_augmentation + random_distort_image (image.py:45-70) in the reference's order:
    pleft, pright, ptop, pbot, flip, dhue, dsat (2 draws), dexp (2 draws)."""
    dw = int(ow * jitter)
    dh = int(oh * jitter)
    pleft = random.randint(-dw, dw)
    pright = random.randint(-dw, dw)
    ptop = random.randint(-dh, dh)
    pbot = random.randint(-dh, dh)
    flip = random.randint(1, 10000) % 2
    swidth = ow - pleft - pright
    sheight = oh - ptop - pbot
    sx = float(swidth) / ow
    sy = float(sheight) / oh
    dx = (float(pleft) / ow) / sx
    dy = (float(ptop) / oh) / sy
    dhue = random.uniform(-hue, hue)
    dsat = rand_scale(saturation)
    dexp = rand_scale(exposure)
    return dict(pleft=pleft, ptop=ptop, cw=swidth - 1, ch=sheight - 1, flip=flip, distort=1, dhue=dhue, dsat=dsat,
                dexp=dexp, dx=dx, dy=dy, sx=sx, sy=sy)


def identity_augmentation(ow, oh):
    """flag=False branch (image.py:83-86): plain resize, no crop, no flip, no colour jitter."""
    return dict(pleft=0, ptop=0, cw=ow, ch=oh, flip=0, distort=0, dhue=0.0, dsat=1.0, dexp=1.0, dx=0, dy=0, sx=1, sy=1)


class PackedImages(object):
    """The decoded uint8 images of a batch back to back in ONE pinned host buffer (offsets / shapes on the side), so
    that they travel to the device in one asynchronous copy instead of one small copy per image."""

    def __init__(self, arrays):
        arrays = [np.ascontiguousarray(np.asarray(a)) for a in arrays]
        for a in arrays:
            if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
                raise TypeError('image must be uint8 [h, w, 3] RGB, got %s %s' % (a.dtype, a.shape))
        self.shapes = [a.shape for a in arrays]
        self.offsets = []
        total = 0
        for a in arrays:
            self.offsets.append(total)
            total += (a.size + 255) // 256 * 256             # 256-byte aligned starts
        try:
            buf = torch.empty(max(total, 1), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
        except RuntimeError:
            buf = torch.empty(max(total, 1), dtype=torch.uint8)
        flat = buf.numpy()
        for a, o in zip(arrays, self.offsets):
            flat[o:o + a.size] = a.reshape(-1)
        self.buf = buf

        self.tables = None

    def __len__(self):
        return len(self.shapes)

    def to_device(self, device):
        d = self.buf.to(device, non_blocking=True)
        return [d[o:o + h * w * 3].view(h, w, 3) for o, (h, w, _) in zip(self.offsets, self.shapes)]

    def marshal(self, params, W, H):
        """Build the per-image argument tables of the augmentation launch NOW (host side, possibly in the background
        thread), in pinned memory, so that the device half of the batch issues only asynchronous copies."""
        geom, color, kmax = marshal_params([(h, w) for h, w, _ in self.shapes], params, W, H)

        def pin(t):
            try:
                return t.pin_memory()
            except RuntimeError:
                return t
        self.tables = (pin(torch.from_numpy(geom)), pin(torch.from_numpy(color)), kmax, pin(torch.empty(len(self.shapes), dtype=torch.int64)),
                       (int(W), int(H)))
        return self


def _as_u8_hwc(img, device):
    """uint8 [h, w, 3] CUDA tensor from a tensor / ndarray / PIL image."""
    if not torch.is_tensor(img):
        img = torch.from_numpy(np.ascontiguousarray(np.asarray(img)))
    if img.dtype != torch.uint8 or img.dim() != 3 or img.size(2) != 3:
        raise TypeError('image must be uint8 [h, w, 3] RGB, got %s %s' % (img.dtype, tuple(img.shape)))
    return img.to(device, non_blocking=True).contiguous()


def kmax_for(params, W, H):
    """Upper bound of the resampling taps per output coordinate (Resample.c: 2*ceil(support) + 1, support = 2*max(scale,1))."""
    k = 5
    for p in params:
        for insize, outsize in ((p['cw'], W), (p['ch'], H)):
            scale = max(float(insize) / outsize, 1.0)
            k = max(k, int(math.ceil(2.0 * scale)) * 2 + 1)
    return k


def marshal_params(sizes, params, W, H):
    """The per-image argument tables of fsdet_augment_batch: geom int32 [n, 8], color float64 [n, 3], kmax.
    sizes[i] = (h, w) of source image i."""
    n = len(params)
    geom = np.zeros((n, 8), dtype=np.int32)
    color = np.zeros((n, 3), dtype=np.float64)
    for i, ((h, w), p) in enumerate(zip(sizes, params)):
        if p['cw'] <= 0 or p['ch'] <= 0:
            raise ValueError('empty crop for image %d' % i)
        geom[i] = [w, h, p['pleft'], p['ptop'], p['cw'], p['ch'], p['flip'], p['distort']]
        color[i] = [p['dhue'], p['dsat'], p['dexp']]
    kmax = kmax_for(params, W, H)
    if kmax > 254:
        raise ValueError('down-scaling factor too large for the resampler tables (kmax=%d)' % kmax)
    return geom, color, kmax


def augment_batch(images, shape, params, filter=None, device=None, out=None, return_uint8=False):
    """One launch for a batch: images[i] (uint8 [h, w, 3]) -> out[i] float32 [3, H, W] under params[i] (a dict from
    draw_augmentation / identity_augmentation).  shape = (W, H) like the reference's `shape` argument.
    `out` may be a channel slice of a larger NCHW tensor (e.g. t[:, 3:6]): each out[i] must be contiguous."""
    if not torch.cuda.is_available():
        raise RuntimeError('augment_batch runs on the GPU only (no CPU fallback)')
    device = _default_device() if device is None else torch.device(device)
    filter = DEFAULT_FILTER if filter is None else filter
    W, H = int(shape[0]), int(shape[1])
    n = len(images)
    assert len(params) == n
    srcs = images.to_device(device) if isinstance(images, PackedImages) else [_as_u8_hwc(im, device) for im in images]
    if isinstance(images, PackedImages) and images.tables is not None and images.tables[4] == (W, H):
        # tables prepared on the host side in pinned memory: nothing here blocks the launching thread
        geom_h, color_h, kmax, ptr_h, _ = images.tables
        for i, s_ in enumerate(srcs):
            ptr_h[i] = s_.data_ptr()
        ptrs = ptr_h.to(device, non_blocking=True)
        geom_d = geom_h.to(device, non_blocking=True)
        color_d = color_h.to(device, non_blocking=True)
    else:
        geom, color, kmax = marshal_params([(int(s.size(0)), int(s.size(1))) for s in srcs], params, W, H)
        ptrs = torch.tensor([s.data_ptr() for s in srcs], dtype=torch.int64).to(device)
        geom_d = torch.from_numpy(geom).to(device)
        color_d = torch.from_numpy(color).to(device)
    ws_bytes = int(lib.fsdet_augment_workspace_bytes(n, W, H, kmax))
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=device)
    status = torch.zeros(1, dtype=torch.int32, device=device)
    if out is None:
        out = torch.empty(n, 3, H, W, dtype=torch.float32, device=device)
    else:
        assert out.device.type == device.type and out.dtype == torch.float32 and tuple(out.shape) == (n, 3, H, W) \
            and out.stride()[1:] == (H * W, W, 1) and (n <= 1 or out.stride(0) >= 3 * H * W)
    u8 = torch.empty(n, H, W, 3, dtype=torch.uint8, device=device) if return_uint8 else None
    if out.is_contiguous():
        call('fsdet_augment_batch', ptr(ptrs), ptr(geom_d), ptr(color_d), n, W, H, kmax, int(filter), ptr(ws), ws_bytes,
             ptr(out), ptr(u8), ptr(status), _st())
    else:
        call('fsdet_augment_batch_pitched', ptr(ptrs), ptr(geom_d), ptr(color_d), n, W, H, kmax, int(filter), ptr(ws),
             ws_bytes, ptr(out), int(out.stride(0)), ptr(u8), ptr(status), _st())
    if return_uint8:
        return out, u8
    return out


def data_augmentation(img, shape, jitter, hue, saturation, exposure, flag=True, filter=None):
    """image.py:52-87.  Returns (float32 CUDA tensor [3, H, W], flip, dx, dy, sx, sy)."""
    src = img if torch.is_tensor(img) else torch.from_numpy(np.ascontiguousarray(np.asarray(img)))
    oh, ow = int(src.size(0)), int(src.size(1))
    p = draw_augmentation(ow, oh, jitter, hue, saturation, exposure) if flag else identity_augmentation(ow, oh)
    out = augment_batch([src], shape, [p], filter=filter)[0]
    return out, p['flip'], p['dx'], p['dy'], p['sx'], p['sy']


# ------------------------------------------------------------------------------------------------- label transforms
def _load_boxes(lab):
    """`np.loadtxt(labpath)` reshaped to [-1, 5] (image.py:94-98), or an array passed directly."""
    if isinstance(lab, str):
        hit = _LABELS.get(lab)
        if hit is None:
            if not (os.path.exists(lab) and os.path.getsize(lab)):
                hit = False
            else:
                hit = np.reshape(np.loadtxt(lab), (-1, 5))
            if len(_LABELS) < 1000000:
                _LABELS[lab] = hit                  # label files are parsed once per process
        if hit is False:
            return None
        bs = hit.copy()                             # callers transform the rows in place
    else:
        bs = np.array(lab, dtype=np.float64)
        if bs.size == 0:
            return None
    if bs is None:
        return None
    return np.reshape(bs, (-1, 5))


def _transform_box(b, flip, dx, dy, sx, sy):
    """image.py:116-134: clamp the corners into the crop, re-centre, flip.  In place; returns False if degenerate."""
    x1 = b[1] - b[3] / 2
    y1 = b[2] - b[4] / 2
    x2 = b[1] + b[3] / 2
    y2 = b[2] + b[4] / 2
    x1 = min(0.999, max(0, x1 * sx - dx))
    y1 = min(0.999, max(0, y1 * sy - dy))
    x2 = min(0.999, max(0, x2 * sx - dx))
    y2 = min(0.999, max(0, y2 * sy - dy))
    b[1] = (x1 + x2) / 2
    b[2] = (y1 + y2) / 2
    b[3] = (x2 - x1)
    b[4] = (y2 - y1)
    if flip:
        b[1] = 0.999 - b[1]
    return not (b[3] < 0.001 or b[4] < 0.001)


def fill_truth_detection(labpath, w, h, flip, dx, dy, sx, sy):
    """image.py:90-141 -> float64 [max_boxes * 5]."""
    max_boxes = cfg.max_boxes
    label = np.zeros((max_boxes, 5))
    bs = _load_boxes(labpath)
    if bs is not None:
        imgid = labpath.split('/')[-1].split('.')[0] if isinstance(labpath, str) else None
        cc = 0
        for i in range(bs.shape[0]):
            clsid = int(bs[i][0])
            if clsid in cfg.base_ids:
                keepit = True
            elif cfg.yolo_joint and imgid in cfg.metaids:
                keepit = True
            else:
                keepit = False
            if not keepit:
                continue
            if not _transform_box(bs[i], flip, dx, dy, sx, sy):
                continue
            label[cc] = bs[i]
            cc += 1
            if cc >= 50:
                break
    return np.reshape(label, (-1))


def fill_truth_detection_meta(labpath, w, h, flip, dx, dy, sx, sy):
    """image.py:144-192 -> float64 [n_cls, max_boxes * 5] (one row per base class, class index = row)."""
    max_boxes = cfg.max_boxes
    n_cls = len(cfg.base_classes)
    label = np.zeros((n_cls, max_boxes, 5))
    bs = _load_boxes(labpath)
    if bs is not None:
        ccs = [0] * n_cls
        for i in range(bs.shape[0]):
            clsid = int(bs[i][0])
            if clsid not in cfg.base_ids:
                continue
            if not _transform_box(bs[i], flip, dx, dy, sx, sy):
                continue
            ind = cfg.base_ids.index(clsid)
            if ind >= n_cls or ccs[ind] >= cfg.max_boxes:
                raise IndexError('more than max_boxes boxes of one class (the reference drops into pdb here)')
            label[ind][ccs[ind]] = bs[i]
            label[ind][ccs[ind]][0] = ind
            ccs[ind] += 1
            if sum(ccs) >= 50:
                break
    return np.reshape(label, (n_cls, -1))


def load_label(labpath, w, h, flip, dx, dy, sx, sy):
    """image.py:195-232 -> list of [x, y, w, h] arrays."""
    label = []
    bs = _load_boxes(labpath)
    if bs is not None:
        cc = 0
        for i in range(bs.shape[0]):
            if not _transform_box(bs[i], flip, dx, dy, sx, sy):
                continue
            label.append(bs[i, 1:])
            cc += 1
            if cc >= 50:
                break
    return label


# decoded-image cache: the reference decodes every file again in every epoch (10 DataLoader worker processes hide
# it); here a decoded VOC train set (16.5 k images, ~9 GB of uint8 RGB) simply stays in host memory after its first
# use.  FSDET_DECODE_CACHE_MB bounds it (0 disables); eviction is oldest first.
_CACHE = collections.OrderedDict()
_CACHE_BYTES = [0]
_CACHE_LIMIT = int(os.environ.get('FSDET_DECODE_CACHE_MB', '16384')) * (1 << 20)
_CACHE_LOCK = threading.Lock()


def _decode(img):
    if isinstance(img, str):
        with _CACHE_LOCK:
            hit = _CACHE.get(img)
        if hit is not None:
            return hit
        from PIL import Image            # host JPEG decode, as the reference (image.py:240)
        arr = np.array(Image.open(img).convert('RGB'))
        if _CACHE_LIMIT > 0 and arr.nbytes <= _CACHE_LIMIT:
            with _CACHE_LOCK:
                if img not in _CACHE:
                    _CACHE[img] = arr
                    _CACHE_BYTES[0] += arr.nbytes
                    while _CACHE_BYTES[0] > _CACHE_LIMIT:
                        _, old = _CACHE.popitem(last=False)
                        _CACHE_BYTES[0] -= old.nbytes
        return arr
    return img


_POOL = [None]
_LABELS = {}


def decode_many(items):
    """Decode a batch of files with a small thread pool (Pillow releases the GIL while it decodes)."""
    todo = [i for i in items if isinstance(i, str)]
    if len(todo) > 1:
        if _POOL[0] is None:
            from concurrent.futures import ThreadPoolExecutor
            _POOL[0] = ThreadPoolExecutor(max_workers=int(os.environ.get('FSDET_DECODE_THREADS', '16')))
        done = dict(zip(todo, _POOL[0].map(_decode, todo)))
        return [done[i] if isinstance(i, str) else i for i in items]
    return [_decode(i) for i in items]


def load_data_detection(imgpath, labpath, shape, jitter, hue, saturation, exposure, data_aug=True, filter=None):
    """image.py:235-246."""
    img, flip, dx, dy, sx, sy = data_augmentation(_decode(imgpath), shape, jitter, hue, saturation, exposure,
                                                  flag=data_aug, filter=filter)
    W, H = int(shape[0]), int(shape[1])
    if cfg.metayolo:
        label = fill_truth_detection_meta(labpath, W, H, flip, dx, dy, 1. / sx, 1. / sy)
    else:
        label = fill_truth_detection(labpath, W, H, flip, dx, dy, 1. / sx, 1. / sy)
    return img, label


def load_data_with_label(imgpath, labpath, shape, jitter, hue, saturation, exposure, data_aug=True, filter=None):
    """image.py:248-253."""
    img, flip, dx, dy, sx, sy = data_augmentation(_decode(imgpath), shape, jitter, hue, saturation, exposure,
                                                  flag=data_aug, filter=filter)
    label = load_label(labpath, int(shape[0]), int(shape[1]), flip, dx, dy, 1. / sx, 1. / sy)
    return img, label


# ------------------------------------------------------------------------------------------------- support masks
def mask_rect(box, w, h):
    """dataset.py:381-384: pixel rectangle of a normalised (x, y, w, h) box, Python round() like the reference."""
    x1 = int(max(0, round((box[0] - box[2] / 2) * w)))
    y1 = int(max(0, round((box[1] - box[3] / 2) * h)))
    x2 = int(min(w, round((box[0] + box[2] / 2) * w)))
    y2 = int(min(h, round((box[1] + box[3] / 2) * h)))
    return x1, y1, x2, y2


def crop_params(rect):
    """Augmentation parameters of `img.crop(rect).resize(img.size)` (dataset.py:387, the cropped-object input of
    metain_type 3 / 4) for the augmented uint8 support image: crop at the mask rectangle, no flip, no colour change."""
    x1, y1, x2, y2 = (int(v) for v in rect)
    p = identity_augmentation(x2 - x1, y2 - y1)
    p['pleft'], p['ptop'] = x1, y1
    return p


def box_masks(boxes, w, h, device=None):
    """dataset.MetaDataset.get_img_mask's masks (dataset.py:378-398) for n support images at once:
    float32 CUDA [n, 1, h, w], ones inside each box's rectangle.  Rows whose rectangle is empty come back all zero
    (the reference returns mask=None for those and re-draws the support image; see `mask_rect`)."""
    if not torch.cuda.is_available():
        raise RuntimeError('box_masks runs on the GPU only (no CPU fallback)')
    device = _default_device() if device is None else torch.device(device)
    n = len(boxes)
    rects = np.array([mask_rect(b, w, h) for b in boxes], dtype=np.int32).reshape(n, 4)
    out = torch.empty(n, 1, h, w, dtype=torch.float32, device=device)
    call('fsdet_box_masks', ptr(torch.from_numpy(rects).to(device)), n, h, w, ptr(out), _st())
    return out
