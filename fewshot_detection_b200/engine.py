"""Host-side executor of the cfg-driven networks on libfsdet.so.

The reference interprets its block list with one torch module per block
(darknet_meta.py:130-195, darknet.py:80-129) and lets autograd + cuDNN do the
rest.  Here the same block list is walked, but every block launches hand-written
sm_100a kernels through the C ABI (include/fsdet.h) on NHWC fp32 buffers, and a
small tape replays the blocks in reverse for the backward pass.

Memory comes from torch's caching allocator (`torch.empty`): torch is used for
device memory, streams and autograd plumbing only -- no torch compute op runs on
the hot path.
"""
import torch

from . import _lib
from ._lib import call, ptr

import os

# tensor-core (tcgen05) convolution path for layers with Cin % 64 == 0; FSDET_TC=0 selects the exact-fp32 SIMT kernels
USE_TC = os.environ.get('FSDET_TC', '1') != '0'
# 'first' = the recomputing first-block kernels (csrc/conv_first_tc.cuh): correct but, as measured on a B200, slower than the
# store-z path they were meant to replace (instruction-bound epilogues, DESIGN.md section 3) - opt-in only
TC_PARTS = set(os.environ.get('FSDET_TC_PARTS', 'fwd,dgrad,wgrad,head').split(','))  # debugging: which GEMMs may use it


def _parse_terms(spec):
    """'fwd=3,dgrad=3,wgrad=0,head=3' -> dict.  Operand-term mode of each GEMM class (include/fsdet.h,
    fsdet_conv_tc_fwd `mode` bits 0-1): 3 = hi*hi + lo*hi + hi*lo (fp32 grade), 1 / 2 = one operand exact and the
    other rounded to fp16, 0 = fp16 x fp16.  The defaults are the measured per-class decision (DESIGN.md section 3,
    profiles/precision_budget_r02.*): the forward chain amplifies per-layer rounding ~1000x through 23 train-mode BN
    layers (2-term forward: 9e-3 at the head output) and the input-gradient chain accumulates it towards the first
    layers (2-term: 1.4e-3), so both keep the fp32-grade 3-term scheme; the weight gradient feeds SGD only, does not
    compound, and its plain fp16 x fp16 form stays within 2.3e-4 ... 5.7e-4 of the fp32-grade value on every tensor."""
    d = {'fwd': 3, 'dgrad': 3, 'wgrad': 0, 'head': 3}
    for item in filter(None, (spec or '').split(',')):
        k, v = item.split('=')
        if k not in d or int(v) not in (0, 1, 2, 3):
            raise ValueError('FSDET_TC_TERMS: bad item %r' % item)
        d[k] = int(v)
    return d


TC_TERMS = _parse_terms(os.environ.get('FSDET_TC_TERMS'))
# persistent tile loop (one CTA per SM, double-buffered TMEM accumulators) for the short-K layers
TC_PERSIST = os.environ.get('FSDET_TC_PERSIST', '0') == '1'


# thread-block clusters of two CTAs sharing the weight tile through TMA multicast (one-tile-per-CTA flavours)
TC_CLUSTER = os.environ.get('FSDET_TC_CLUSTER', '0') == '1'


# halo-tile kernel for the high-resolution 3x3 layers (csrc/conv_halo_kernels.cuh): on unless FSDET_TC_HALO=0
TC_HALO = os.environ.get('FSDET_TC_HALO', '1') != '0'


# A_hi * [B_hi | B_lo] as one MMA of width 2*BN (two MMAs per K step instead of three): on unless FSDET_TC_FUSE=0
TC_FUSE = os.environ.get('FSDET_TC_FUSE', '1') != '0'


def tc_mode(name):
    return (TC_TERMS[name] | (16 if TC_PERSIST else 0) | (32 if TC_CLUSTER else 0) | (0 if TC_HALO else 64)
            | (0 if TC_FUSE else 128))

# Weight gradients on a second stream: after a block's BatchNorm backward, its weight-gradient GEMM (tensor-bound, one
# CTA per SM) and the rest of the backward chain (input gradient, then the next block's HBM-bound BatchNorm passes) are
# independent - the weight gradient is only needed by the optimizer.  FSDET_WGRAD_STREAM=0 keeps everything on one stream.
WGRAD_STREAM = os.environ.get('FSDET_WGRAD_STREAM', '1') != '0'

LEAKY_SLOPE = 0.1
BN_EPS = 1e-5
BN_MOMENTUM = 0.1


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _empty(*shape, dtype=torch.float32, device=None):
    return torch.empty(*shape, dtype=dtype, device=device)


def _round_up(v, m):
    return (v + m - 1) // m * m


def same_layout(a, b):
    """Same shape and same strides on every dimension of extent > 1."""
    if a.shape != b.shape:
        return False
    return all(sa == sb for n, sa, sb in zip(a.shape, a.stride(), b.stride()) if n > 1)


class Act(object):
    """A view [B*H*W pixels] x [C channels at column `off`] of a 2-D NHWC fp32 buffer, and/or the fp16 hi/lo
    planes of the same activation for the tensor-core kernels (`buf` is None when only the planes exist)."""
    __slots__ = ('buf', 'off', 'C', 'B', 'H', 'W', 'g', 'needs_grad', 'parent', 'planes', 'amax', 'dev', 'nchw')

    def __init__(self, buf, off, C, B, H, W, needs_grad=True, parent=None, dev=None):
        self.buf, self.off, self.C, self.B, self.H, self.W = buf, off, C, B, H, W
        self.g = None            # gradient Act (same geometry) once some consumer wrote it
        self.needs_grad = needs_grad
        self.parent = parent     # concat buffer this view is a slice of
        self.planes = None       # (hi, lo, amax) fp16 planes of this activation for the tensor-core path
        self.amax = None         # device scalar |max| if already known (skips the amax pass before splitting)
        self.dev = buf.device if buf is not None else dev
        self.nchw = None         # (in0, C0, in1, C1): the network input, still in the reference's NCHW tensors

    @property
    def ld(self):
        return self.buf.shape[1]

    @property
    def npix(self):
        return self.B * self.H * self.W

    @property
    def ptr(self):
        if self.buf is None:
            raise RuntimeError('this activation only exists as fp16 planes (internal planning error)')
        return self.buf.data_ptr() + 4 * self.off

    @staticmethod
    def new(B, H, W, C, device, needs_grad=True):
        return Act(_empty(B * H * W, C, device=device), 0, C, B, H, W, needs_grad)

    @staticmethod
    def planes_only(B, H, W, C, device, planes):
        a = Act(None, 0, C, B, H, W, True, dev=device)
        a.planes = planes
        return a

    def slice(self, off, C):
        return Act(self.buf, self.off + off, C, self.B, self.H, self.W, self.needs_grad, parent=(self, off))

    def grad_for_write(self):
        """Returns (grad Act, accumulate flag) for a consumer about to write its
        contribution to d(loss)/d(this activation)."""
        if self.g is not None:
            return self.g, 1
        if self.parent is not None:
            par, off = self.parent
            if par.g is None:
                raise NotImplementedError('gradient of a concat slice written before the concat buffer')
            self.g = par.g.slice(off, self.C)
            return self.g, 1
        self.g = Act.new(self.B, self.H, self.W, self.C, self.dev, needs_grad=False)
        return self.g, 0

    def grad_for_read(self):
        if self.g is None and self.parent is not None:
            par, off = self.parent
            if par.g is not None:
                self.g = par.g.slice(off, self.C)
        return self.g


# ----------------------------------------------------------------- plan
class Spec(object):
    def __init__(self, kind, idx, **kw):
        self.kind = kind
        self.idx = idx
        self.__dict__.update(kw)


def is_dynamic(block):
    return 'dynamic' in block and int(block['dynamic']) == 1


def compile_blocks(blocks):
    """Block list -> list of Spec (one per module index, the reference's `ind`).

    Fusions decided here:
      * conv(+BN+leaky) followed by maxpool 2/2: the pool is computed in the
        conv block's activation pass; the full-resolution activation is only
        materialised if a route refers to the conv.
      * dynamic conv followed by a linear 1x1 conv: one GEMM with per-class
        effective weights (the [B*n_cls,1024,G,G] tensor is never built).
      * two-layer routes: producers write straight into slices of one buffer.
    """
    specs = []
    in_ch = 3
    out_ch = []
    ind = -1
    body = []
    for block in blocks:
        t = block['type']
        if t in ('net', 'learnet'):
            in_ch = int(block['channels'])
            continue
        body.append(block)
    prev = in_ch
    for block in body:
        ind += 1
        t = block['type']
        if t == 'convolutional':
            filters = int(block['filters'])
            k = int(block['size'])
            if int(block['stride']) != 1:
                raise NotImplementedError('convolutional stride %s' % block['stride'])
            if k not in (1, 3) or not int(block['pad']) and k != 1:
                raise NotImplementedError('convolutional size=%d pad=%s' % (k, block['pad']))
            act = block['activation']
            if act not in ('leaky', 'linear'):
                raise NotImplementedError('activation %s' % act)
            specs.append(Spec('conv', ind, cin=prev, cout=filters, k=k, bn=int(block['batch_normalize']),
                              slope=LEAKY_SLOPE if act == 'leaky' else 1.0, dynamic=is_dynamic(block),
                              fuse_pool=False, head=False))
            prev = filters
        elif t == 'maxpool':
            size, stride = int(block['size']), int(block['stride'])
            if size != 2 or stride not in (1, 2):
                raise NotImplementedError('maxpool size=%d stride=%d' % (size, stride))
            specs.append(Spec('maxpool', ind, stride=stride, fused=False))
        elif t == 'reorg':
            s = int(block['stride'])
            if s != 2:
                raise NotImplementedError('reorg stride %d' % s)
            specs.append(Spec('reorg', ind))
            prev = 4 * prev
        elif t == 'route':
            layers = [int(i) for i in block['layers'].split(',')]
            layers = [i if i > 0 else i + ind for i in layers]
            if len(layers) == 1:
                prev = out_ch[layers[0]]
            elif len(layers) == 2:
                if 'concat' in block and int(block['concat']) == 0:
                    raise NotImplementedError('route concat=0')
                prev = out_ch[layers[0]] + out_ch[layers[1]]
            else:
                raise NotImplementedError('route with %d layers' % len(layers))
            specs.append(Spec('route', ind, layers=layers))
        elif t == 'globalmax':
            specs.append(Spec('globalmax', ind))
        elif t in ('region', 'cost'):
            specs.append(Spec('skip', ind))
        else:
            raise NotImplementedError('block type %s' % t)
        out_ch.append(prev)
    # ---- fusion passes
    routed = set()
    for s in specs:
        if s.kind == 'route':
            routed.update(s.layers)
    for i, s in enumerate(specs):
        nxt = specs[i + 1] if i + 1 < len(specs) else None
        if s.kind == 'conv' and not s.dynamic and nxt is not None and nxt.kind == 'maxpool' and nxt.stride == 2:
            s.fuse_pool = True
            s.keep_full = s.idx in routed
            nxt.fused = True
        if s.kind == 'conv' and s.dynamic:
            ok = (nxt is not None and nxt.kind == 'conv' and not nxt.dynamic and nxt.k == 1 and not nxt.bn and
                  nxt.slope == 1.0 and s.k == 1 and not s.bn and s.slope == 1.0)
            if not ok:
                raise NotImplementedError('dynamic conv must be 1x1/linear and followed by a linear 1x1 conv')
            s.kind = 'dyn'
            nxt.head = True
    # ---- zero-copy concat planning: producer idx -> (route idx, channel offset)
    placement = {}
    for s in specs:
        if s.kind == 'route' and len(s.layers) == 2:
            off = 0
            ok = all(l not in placement and specs[l].kind in ('conv', 'reorg', 'maxpool') for l in s.layers) \
                and s.layers[0] != s.layers[1]
            for l in s.layers:
                if ok:
                    placement[l] = (s.idx, off)
                off += out_ch[l]
            s.zero_copy = ok
            s.total = off
    return specs, out_ch, placement, in_ch


# ------------------------------------------------------------- executor
class Tape(object):
    def __init__(self):
        self.records = []


class NetRunner(object):
    """Executes one cfg network (detector or support net) for a Darknet module."""

    def __init__(self, blocks, models):
        self.blocks = blocks
        self.models = models  # nn.ModuleList aligned with spec.idx
        self.specs, self.out_ch, self.placement, self.in_ch = compile_blocks(blocks)
        self.routed = set(l for sp in self.specs if sp.kind == 'route' for l in sp.layers)
        self.in_cpad = _round_up(self.in_ch, 4)
        self.grad_hook = None   # optional callable(param) invoked when a parameter gradient has been enqueued
        self.profile = None     # optional dict name -> [flops, [(start_event, end_event), ...]]
        self.side = None        # second stream for the weight gradients (created by the first backward pass)
        self._side_used = False
        self._keep = []         # tensors allocated on the main stream that the side stream still reads (until the join)

    # -- helpers ---------------------------------------------------------
    @staticmethod
    def _conv_modules(seq):
        conv = bn = None
        for m in seq.children():
            if isinstance(m, torch.nn.BatchNorm2d):
                bn = m
            elif hasattr(m, 'weight') or getattr(m, 'is_dynamic_conv', False):
                if conv is None:
                    conv = m
        return conv, bn

    @staticmethod
    def _ohwi(w):
        """Physical OHWI view of a conv weight Parameter (converted in place once)."""
        if w.dim() == 4 and not w.is_contiguous(memory_format=torch.channels_last):
            w.data = w.data.contiguous(memory_format=torch.channels_last)
        return w

    # -- tensor-core helpers ------------------------------------------------
    @staticmethod
    def _tc_ok(cin, cout, k):
        """Tensor-core path: >= 32 input channels (planes are zero-padded to a multiple of 64)."""
        return USE_TC and cin >= 32 and cin % 4 == 0 and cout % 4 == 0 and bool(
            _lib.lib.fsdet_conv_tc_supported(_round_up(cin, 32), cout, k))

    @staticmethod
    def _split_tensor(t2d_ptr, ld, C, rows, dev, st, cpad=None, amax=None):
        """fp32 [rows][ld] -> (hi, lo, amax): scaled fp16 planes [rows][cpad] + the device scalar they were scaled by
        (computed here unless the producer already provided it)."""
        cpad = cpad or C
        if amax is None:
            amax = torch.empty(1, dtype=torch.float32, device=dev)
            call('fsdet_amax', t2d_ptr, ld, C, rows, ptr(amax), st)
        hi = torch.empty(rows, cpad, dtype=torch.float16, device=dev)
        lo = torch.empty(rows, cpad, dtype=torch.float16, device=dev)
        call('fsdet_split_f16', t2d_ptr, ld, C, cpad, rows, ptr(amax), ptr(hi), ptr(lo), st)
        return hi, lo, amax

    def _planes(self, act, st):
        """fp16 hi/lo planes [npix][round_up(C, 64)] (+ amax) of an activation (cached: the forward /
        input-gradient GEMM and the weight-gradient GEMM read the same planes)."""
        if act.planes is None:
            act.planes = self._split_tensor(act.ptr, act.ld, act.C, act.npix, act.dev, st, _round_up(act.C, 64), act.amax)
        return act.planes

    def _consumer_takes_planes(self, spec_pos, cin):
        """True if the block at position `spec_pos` is a convolution that will read its input only through the
        tensor-core kernels (forward and weight gradient), so the producer may skip the fp32 activation."""
        if not USE_TC or not {'fwd', 'dgrad', 'wgrad', 'head'} <= TC_PARTS or spec_pos >= len(self.specs):
            return False
        c = self.specs[spec_pos]
        if c.kind == 'dyn':
            return cin >= 32 and cin % 4 == 0
        if c.kind != 'conv' or c.head or not c.bn:
            return False
        return self._tc_ok(cin, c.cout, c.k) and c.cout >= 32 and bool(
            _lib.lib.fsdet_conv_tc_wgrad_supported(_round_up(cin, 64), _round_up(c.cout, 64), c.k))

    def _conv(self, name, x, w_ohwi, bias, z, stat_rows_out, cin, cout, k, acc, st, w_amax=None, wplanes=None):
        """z = conv(x, w) through the tensor-core kernel when the shape allows, else SIMT.
        Returns the number of BN partial rows written to `stat_rows_out` (a float tensor or None).
        wplanes: (hi, lo, amax) of the weight operand when fsdet_weight_prep already produced them."""
        flops = 2.0 * x.npix * cout * k * k * cin
        if x.nchw is not None:
            in0, c0, in1, c1 = x.nchw
            assert bias is None and not acc and cin == _round_up(c0 + c1, 4) and cin <= 8 and k == 3
            if stat_rows_out is not None:   # BatchNorm partial rows straight from the kernel's registers (no pass over z)
                self._timed('first_fwd', flops, 'fsdet_conv_first_fwd_stats', ptr(in0), c0, ptr(in1), c1, ptr(w_ohwi), z.ptr, z.ld,
                            x.B, x.H, x.W, cout, ptr(stat_rows_out), st)
                return _lib.lib.fsdet_conv_first_stat_rows(x.B, x.H, x.W)
            self._timed('first_fwd', flops, 'fsdet_conv_first_fwd', ptr(in0), c0, ptr(in1), c1, ptr(w_ohwi), z.ptr, z.ld, x.B, x.H,
                        x.W, cout, st)
            return 0
        if bias is None and name in TC_PARTS and self._tc_ok(cin, cout, k):
            cpad = _round_up(cin, 64)
            xh, xl, xa = self._planes(x, st)
            if wplanes is not None:
                wh, wl, wa = wplanes
            else:
                wh, wl, wa = self._split_tensor(ptr(w_ohwi), cin, cin, cout * k * k, x.dev, st, cpad, w_amax)
                if name == 'fwd':   # the flip-transposed copy used by the input-gradient GEMM has the same absolute maximum
                    w_ohwi._fsdet_amax = (wa, w_ohwi._version)
            mode = tc_mode(name)
            self._timed('conv_tc', flops, 'fsdet_conv_tc_fwd', ptr(xh), ptr(xl), ptr(wh), ptr(wl), ptr(xa), ptr(wa), z.ptr, z.ld,
                        x.B, x.H, x.W, _round_up(cin, 32), cpad, cout, k, acc, mode, ptr(stat_rows_out), st)
            if stat_rows_out is not None:   # BatchNorm partial rows come out of the convolution's epilogue
                return _lib.lib.fsdet_conv_tc_stat_rows(x.B, x.H, x.W, _round_up(cin, 32), cout, k, mode)
            return 0
        self._timed('conv_igemm', flops, 'fsdet_conv_fwd', x.ptr, x.ld, ptr(w_ohwi), ptr(bias), z.ptr, z.ld,
                    ptr(stat_rows_out), x.B, x.H, x.W, cin, cout, k, acc, st)
        return _lib.lib.fsdet_conv_stat_rows(x.npix) if stat_rows_out is not None else 0

    def _done(self, *params):
        if self.grad_hook is not None:
            if self._side_used:
                # a bucket's collective is ordered behind the CURRENT stream only: make it see the other stream's gradients too
                cur = torch.cuda.current_stream()
                cur.wait_stream(self.side if cur != self.side else self._main)
            for p in params:
                if p is not None:
                    self.grad_hook(p)

    def _side_ok(self):
        """Weight gradients go to the second stream unless disabled or per-kernel timing is on (profiled durations must
        not include a concurrent kernel's share of the SMs)."""
        if not WGRAD_STREAM or self.profile is not None:
            return False
        if self.grad_hook is not None and os.environ.get('FSDET_WGRAD_STREAM') != '2':
            # data-parallel runs launch their bucket collectives from the backward pass: keep one compute stream there
            # (the overlap is worth ~0.6 % of a step; FSDET_WGRAD_STREAM=2 forces it for experiments)
            return False
        if self.side is None:
            if torch.cuda.is_current_stream_capturing():
                return False            # streams are created outside captures (the first eager step does it)
            self.side = torch.cuda.Stream()
        return True

    def _timed(self, name, flops, fn, *args):
        """call() bracketed by CUDA events on the launching stream when profiling."""
        if self.profile is None:
            return call(fn, *args)
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        call(fn, *args)
        e1.record()
        ent = self.profile.setdefault(name, [0.0, []])
        ent[0] += flops
        ent[1].append((e0, e1))
        self.profile.setdefault('_launches', []).append((name, flops, e0, e1, tuple(a for a in args if isinstance(a, int) and a < 100000)))

    @staticmethod
    def _param_grad(p):
        """Returns (tensor to write the gradient into, finish callback)."""
        if p.grad is not None and getattr(p, '_fsdet_overwrite', False) and same_layout(p.grad, p):
            return p.grad, None
        if p.grad is None:
            p.grad = torch.empty_like(p)  # preserve_format: same (OHWI) strides as p
            return p.grad, None
        if not same_layout(p.grad, p):
            p.grad = p.grad.contiguous(memory_format=torch.channels_last if p.dim() == 4 else torch.contiguous_format)
        tmp = torch.empty_like(p)
        return tmp, (lambda: p.grad.add_(tmp))

    # -- weight operands of all tensor-core layers, two launches per step ----------------------------------------
    def _weight_plan(self, dev):
        """Device tables for fsdet_weight_prep (built once; rebuilt when a weight tensor moved): one descriptor per
        BatchNorm convolution that runs on the tensor cores, persistent zero-initialised fp16 planes for its forward
        GEMM and - when its input needs a gradient - for its input-gradient GEMM."""
        import struct
        import numpy as np
        layers = []
        prev = self.in_cpad
        first = True
        for s in self.specs:
            if s.kind == 'conv' and not s.head:
                conv, bn = self._conv_modules(self.models[s.idx])
                cin_p = _round_up(s.cin, 4)
                if bn is not None and not first and self._tc_ok(cin_p, s.cout, s.k) and cin_p == s.cin:
                    layers.append((s, self._ohwi(conv.weight), cin_p))
            first = False if s.kind == 'conv' else first
        key = (str(dev), USE_TC, tuple(sorted(TC_PARTS)), tuple(w.data_ptr() for _, w, _ in layers))
        plan = getattr(self, '_wplan', None)
        if plan is not None and plan['key'] == key:
            return plan
        plan = {'key': key, 'by_id': {}, 'n': len(layers)}
        if not layers:
            self._wplan = plan
            return plan
        amax_all = torch.zeros(len(layers), dtype=torch.float32, device=dev)
        descs = b''
        tiles = []
        for li, (s, w, cin_p) in enumerate(layers):
            kk = s.k * s.k
            fp, bp = _round_up(cin_p, 64), _round_up(s.cout, 64)
            want_fwd = 'fwd' in TC_PARTS
            want_bwd = 'dgrad' in TC_PARTS and self._tc_ok(s.cout, cin_p, s.k)
            fh = fl = bh = bl = None
            if want_fwd:
                fh = torch.zeros(s.cout, kk * fp, dtype=torch.float16, device=dev)
                fl = torch.zeros(s.cout, kk * fp, dtype=torch.float16, device=dev)
            if want_bwd:
                bh = torch.zeros(cin_p, kk * bp, dtype=torch.float16, device=dev)
                bl = torch.zeros(cin_p, kk * bp, dtype=torch.float16, device=dev)
            tci, tco = (cin_p + 31) // 32, (s.cout + 31) // 32
            am = amax_all[li:li + 1]
            descs += struct.pack('<6Q8i', w.data_ptr(), ptr(fh) or 0, ptr(fl) or 0, ptr(bh) or 0, ptr(bl) or 0, am.data_ptr(),
                                 s.cout, kk, cin_p, fp, bp, tci, tco, 0)
            n_t = kk * tci * tco
            t = np.empty((n_t, 2), dtype=np.int32)
            t[:, 0] = li
            t[:, 1] = np.arange(n_t, dtype=np.int32)
            tiles.append(t)
            plan['by_id'][id(w)] = {'fwd': (fh, fl, am) if want_fwd else None, 'bwd': (bh, bl, am) if want_bwd else None}
        tiles = np.concatenate(tiles, 0)
        plan['descs'] = torch.frombuffer(bytearray(descs), dtype=torch.uint8).to(dev)
        plan['tiles'] = torch.from_numpy(tiles).to(dev)
        plan['n_tiles'] = int(tiles.shape[0])
        plan['amax'] = amax_all
        self._wplan = plan
        return plan

    def _prepare_weights(self, dev, st):
        """Planes of every tensor-core layer's weights for this step (the weights change once per step)."""
        self._wp = {}
        if not USE_TC:
            return
        plan = self._weight_plan(dev)
        if plan['n']:
            call('fsdet_weight_prep', ptr(plan['descs']), ptr(plan['tiles']), plan['n_tiles'], ptr(plan['amax']), plan['n'], st)
            self._wp = plan['by_id']

    # -- forward -----------------------------------------------------------
    def forward(self, inputs, extra=None, training=True, record=True):
        """inputs: list of NCHW tensors concatenated along channels (image[, mask]).
        extra: reweighting vectors [n_cls, K(,1,1)] for a dynamic head.
        Returns (output tensor, tape)."""
        x0 = inputs[0]
        dev = x0.device
        B, _, H, W = x0.shape
        st = _stream()
        tape = Tape() if record else None
        c0 = x0.shape[1]
        c1 = inputs[1].shape[1] if len(inputs) > 1 else 0
        if c0 + c1 != self.in_ch:
            raise ValueError('network expects %d input channels, got %d' % (self.in_ch, c0 + c1))
        for t in inputs:
            if t.dtype != torch.float32 or not t.is_cuda:
                raise TypeError('inputs must be float32 CUDA tensors (no CPU fallback)')
        self._prepare_weights(dev, st)
        first = self.specs[0] if self.specs else None
        in0 = inputs[0].contiguous()
        in1 = inputs[1].contiguous() if c1 else None
        if (first is not None and first.kind == 'conv' and not first.dynamic and first.k == 3 and first.cout <= 32
                and first.cout % 4 == 0 and self.in_ch <= 8 and _lib.lib.fsdet_conv_first_wgrad_supported(self.in_ch, W)):
            # the first convolution reads the NCHW input directly (no NHWC copy of the images); weights and their
            # gradient carry in_cpad channels (4 for image + mask, 8 for the cropped-object inputs of metain_type 3 / 4,
            # whose weight-gradient staging outgrows shared memory past W = 518: those take the NHWC path)
            xin = Act(None, 0, self.in_cpad, B, H, W, needs_grad=False, dev=dev)
            xin.nchw = (in0, c0, in1, c1)
        else:
            xin = Act.new(B, H, W, self.in_cpad, dev, needs_grad=False)
            call('fsdet_nchw_to_nhwc', ptr(in0), c0, ptr(in1), c1, xin.ptr, xin.ld, self.in_cpad, B, H * W, st)
        outputs = {}
        cat_bufs = {}
        cur = xin
        result = None
        specs = self.specs
        i = 0

        def out_act(idx, B_, H_, W_, C_):
            """Allocate (or place into a concat buffer) the output of module idx."""
            if idx in self.placement:
                ridx, off = self.placement[idx]
                rs = specs[ridx]
                if ridx not in cat_bufs:
                    cat_bufs[ridx] = Act.new(B_, H_, W_, rs.total, dev)
                return cat_bufs[ridx].slice(off, C_)
            return Act.new(B_, H_, W_, C_, dev)

        while i < len(specs):
            s = specs[i]
            if s.kind == 'conv' and not s.head:
                cur, rec = self._conv_fwd(s, cur, training, out_act, st)
                if s.fuse_pool:
                    full, pooled = cur
                    outputs[s.idx] = full
                    outputs[s.idx + 1] = pooled
                    cur = pooled
                    i += 1  # the fused maxpool spec
                else:
                    outputs[s.idx] = cur
                if tape is not None:
                    tape.records.append(rec)
            elif s.kind == 'dyn':
                head = specs[i + 1]
                result, rec = self._head_fwd(s, head, cur, extra, st)
                if tape is not None:
                    tape.records.append(rec)
                outputs[s.idx] = None
                outputs[head.idx] = None
                cur = None
                i += 1
            elif s.kind == 'maxpool':
                Ho, Wo = (cur.H // 2, cur.W // 2) if s.stride == 2 else (cur.H, cur.W)
                y = out_act(s.idx, cur.B, Ho, Wo, cur.C)
                call('fsdet_maxpool_fwd', cur.ptr, cur.ld, y.ptr, y.ld, cur.B, cur.H, cur.W, cur.C, s.stride, st)
                if tape is not None:
                    tape.records.append(('maxpool', s, cur, y))
                cur = y
                outputs[s.idx] = cur
            elif s.kind == 'reorg':
                y = out_act(s.idx, cur.B, cur.H // 2, cur.W // 2, cur.C * 4)
                call('fsdet_reorg_fwd', cur.ptr, cur.ld, y.ptr, y.ld, cur.B, cur.H, cur.W, cur.C, st)
                if tape is not None:
                    tape.records.append(('reorg', s, cur, y))
                cur = y
                outputs[s.idx] = cur
            elif s.kind == 'route':
                if len(s.layers) == 1:
                    cur = outputs[s.layers[0]]
                    if cur is None:
                        raise NotImplementedError('route to a fused-away layer %d' % s.layers[0])
                else:
                    a0, a1 = outputs[s.layers[0]], outputs[s.layers[1]]
                    if a0 is None or a1 is None:
                        raise NotImplementedError('route to a fused-away layer')
                    if s.zero_copy:
                        cur = cat_bufs[s.idx]
                    else:
                        if (a0.B, a0.H, a0.W) != (a1.B, a1.H, a1.W):
                            raise NotImplementedError('route of different geometries (maybe_repeat)')
                        cur = Act.new(a0.B, a0.H, a0.W, a0.C + a1.C, dev)
                        call('fsdet_copy_channels', a0.ptr, a0.ld, cur.ptr, cur.ld, a0.npix, a0.C, 0, st)
                        call('fsdet_copy_channels', a1.ptr, a1.ld, cur.ptr + 4 * a0.C, cur.ld, a1.npix, a1.C, 0, st)
                        if tape is not None:
                            tape.records.append(('cat', s, a0, a1, cur))
                outputs[s.idx] = cur
            elif s.kind == 'globalmax':
                if cur.H != cur.W:
                    raise NotImplementedError('GlobalMaxPool2d uses kernel = W; non-square maps unsupported')
                y = _empty(cur.B, cur.C, device=dev)
                arg = _empty(cur.B, cur.C, dtype=torch.int32, device=dev)
                call('fsdet_globalmax_fwd', cur.ptr, cur.ld, ptr(y), ptr(arg), cur.B, cur.H * cur.W, cur.C, st)
                if tape is not None:
                    tape.records.append(('globalmax', s, cur, arg))
                result = y.view(cur.B, cur.C, 1, 1)
                cur = None
                outputs[s.idx] = None
            elif s.kind == 'skip':
                pass
            else:
                raise NotImplementedError(s.kind)
            i += 1
        if result is None:
            # network ends in an ordinary activation: hand it back as NCHW
            if cur is None:
                raise RuntimeError('network produced no output')
            c_true = self.out_ch[[sp.idx for sp in specs if sp.kind != 'skip'][-1]]
            result = _empty(cur.B, c_true, cur.H, cur.W, device=dev)
            call('fsdet_nhwc_to_nchw', cur.ptr, cur.ld, None, ptr(result), cur.B, c_true, cur.H * cur.W, st)
            if tape is not None:
                tape.records.append(('output', cur, c_true))
        return result, tape

    def _conv_fwd(self, s, x, training, out_act, st):
        seq = self.models[s.idx]
        conv, bn = self._conv_modules(seq)
        dev = x.dev
        B, H, W = x.B, x.H, x.W
        npix = x.npix
        w = self._ohwi(conv.weight)
        kk = s.k * s.k
        cin_p = x.C  # activation channel count (input padded to a multiple of 4)
        if cin_p != s.cin:
            wuse = _empty(s.cout, kk, cin_p, device=dev)
            call('fsdet_pad_channels', ptr(w), s.cin, ptr(wuse), cin_p, s.cout * kk, st)
        else:
            wuse = w
        cout_p = _round_up(s.cout, 4)
        if (bn is not None and x.nchw is not None and s.fuse_pool and not s.keep_full and USE_TC and 'first' in TC_PARTS
                and cin_p == 4 and s.k == 3 and _lib.lib.fsdet_conv_first_tc_supported(H, W, s.cout)):
            return self._first_tc_fwd(s, x, wuse, conv, bn, training, out_act, st)
        if bn is not None:
            assert cout_p == s.cout, 'BatchNorm conv with Cout % 4 != 0 is unsupported'
            z = Act.new(B, H, W, s.cout, dev)
            use_batch_stats = training or not bn.track_running_stats
            rows_cap = max(_lib.lib.fsdet_conv_stat_rows(npix), _lib.lib.fsdet_colstats_rows(npix), (npix + 127) // 128 + 1, 3 * 148)
            stat = _empty(rows_cap + _lib.lib.fsdet_bn_stat_scratch_rows(), 4 * s.cout, device=dev) if use_batch_stats else None
            wp = getattr(self, '_wp', {}).get(id(wuse))
            rows = self._conv('fwd', x, wuse, None, z, stat, cin_p, s.cout, s.k, 0, st, wplanes=wp['fwd'] if wp else None)
            vec = _empty(5, s.cout, device=dev)  # mean, invstd, scale, shift, max|xhat| (batch statistics only)
            vec.xh_ok = bool(use_batch_stats)
            amax_y = _empty(1, device=dev) if use_batch_stats else None
            upd = training and bn.track_running_stats
            call('fsdet_bn_finalize', ptr(stat), rows, float(npix), ptr(bn.weight), ptr(bn.bias),
                 ptr(bn.running_mean) if (upd or not use_batch_stats) else None,
                 ptr(bn.running_var) if (upd or not use_batch_stats) else None,
                 BN_MOMENTUM if bn.momentum is None else float(bn.momentum), float(bn.eps),
                 ptr(vec[0]), ptr(vec[1]), ptr(vec[2]), ptr(vec[3]), s.slope, ptr(amax_y), ptr(vec[4]), s.cout,
                 1 if use_batch_stats else 0, st)
            if upd and bn.num_batches_tracked is not None:
                bn.num_batches_tracked += 1
            # which outputs exist, and in which representation (fp32 and / or fp16 planes)
            pos = self.specs.index(s)
            cp64 = _round_up(s.cout, 64)
            want_full = (not s.fuse_pool) or s.keep_full
            want_pool = s.fuse_pool
            full = pooled = None
            fpl = ppl = None
            if want_full:
                planes_ok = (amax_y is not None and not s.fuse_pool and s.idx not in self.placement
                             and s.idx not in self.routed and self._consumer_takes_planes(pos + 1, s.cout))
                if planes_ok:
                    fpl = (torch.empty(npix, cp64, dtype=torch.float16, device=dev),
                           torch.empty(npix, cp64, dtype=torch.float16, device=dev), amax_y)
                    full = Act.planes_only(B, H, W, s.cout, dev, fpl)
                else:
                    full = out_act(s.idx, B, H, W, s.cout)
                    full.amax = amax_y
            if want_pool:
                Hp, Wp = H // 2, W // 2
                planes_ok = (amax_y is not None and (s.idx + 1) not in self.placement and (s.idx + 1) not in self.routed
                             and self._consumer_takes_planes(pos + 2, s.cout))
                if planes_ok:
                    ppl = (torch.empty(B * Hp * Wp, cp64, dtype=torch.float16, device=dev),
                           torch.empty(B * Hp * Wp, cp64, dtype=torch.float16, device=dev), amax_y)
                    pooled = Act.planes_only(B, Hp, Wp, s.cout, dev, ppl)
                else:
                    pooled = out_act(s.idx + 1, B, Hp, Wp, s.cout)
                    pooled.amax = amax_y   # upper bound (max-pool of y): still a valid plane scale
            f32 = full if (full is not None and full.buf is not None) else None
            p32 = pooled if (pooled is not None and pooled.buf is not None) else None
            call('fsdet_bn_act_fwd', z.ptr, z.ld, ptr(vec[2]), ptr(vec[3]), s.slope,
                 f32.ptr if f32 else None, f32.ld if f32 else 0, p32.ptr if p32 else None, p32.ld if p32 else 0,
                 ptr(fpl[0]) if fpl else None, ptr(fpl[1]) if fpl else None, ptr(ppl[0]) if ppl else None,
                 ptr(ppl[1]) if ppl else None, cp64, ptr(amax_y) if (fpl or ppl) else None, B, H, W, s.cout, st)
            rec = ('convbn', s, x, wuse, z, vec, full, pooled, conv, bn)
            return ((full, pooled) if s.fuse_pool else full), rec
        # conv + bias (+ leaky), no BN
        if cout_p != s.cout:
            wp = torch.zeros(cout_p, kk, cin_p, device=dev)
            wp[:s.cout].copy_(wuse.detach().reshape(s.cout, kk, cin_p) if wuse is not w else
                              w.detach().permute(0, 2, 3, 1).reshape(s.cout, kk, cin_p))
            bp = torch.zeros(cout_p, device=dev)
            if conv.bias is not None:
                bp[:s.cout].copy_(conv.bias.detach())
        else:
            wp = wuse
            bp = conv.bias
        z = Act.new(B, H, W, cout_p, dev)
        self._timed('conv_igemm', 2.0 * npix * cout_p * kk * cin_p, 'fsdet_conv_fwd', x.ptr, x.ld, ptr(wp), ptr(bp), z.ptr,
                    z.ld, None, B, H, W, cin_p, cout_p, s.k, 0, st)
        ones = zeros = None
        if s.slope != 1.0:
            ones = torch.ones(cout_p, device=dev)
            zeros = torch.zeros(cout_p, device=dev)
        full = pooled = None
        if s.fuse_pool or s.slope != 1.0:
            if ones is None:
                ones = torch.ones(cout_p, device=dev)
                zeros = torch.zeros(cout_p, device=dev)
            if s.fuse_pool:
                pooled = out_act(s.idx + 1, B, H // 2, W // 2, cout_p)
                if s.keep_full:
                    full = out_act(s.idx, B, H, W, cout_p)
            else:
                full = out_act(s.idx, B, H, W, cout_p)
            call('fsdet_bn_act_fwd', z.ptr, z.ld, ptr(ones), ptr(zeros), s.slope, full.ptr if full else None,
                 full.ld if full else 0, pooled.ptr if pooled else None, pooled.ld if pooled else 0, None, None, None, None,
                 cout_p, None, B, H, W, cout_p, st)
        else:
            full = z  # linear: the conv output is the block output
        rec = ('convbias', s, x, wp, z, (ones, zeros), full, pooled, conv, cout_p)
        return ((full, pooled) if s.fuse_pool else full), rec

    # -- first block without its pre-BN tensor (csrc/conv_first_tc.cuh) ------------------------------------------
    def _first_tc_fwd(self, s, x, w4, conv, bn, training, out_act, st):
        """conv 3x3 from the NCHW images + BatchNorm + LeakyReLU + max-pool in two recomputing passes: the layer's
        pre-BN output (the largest tensor of the network) is never written; backward recomputes it too."""
        dev = x.dev
        B, H, W = x.B, x.H, x.W
        in0, c0, in1, c1 = x.nchw
        npix = x.npix
        amax_x = torch.empty(1, dtype=torch.float32, device=dev)
        call('fsdet_amax', ptr(in0), W, W, in0.numel() // W, ptr(amax_x), st)
        if in1 is not None:
            call('fsdet_amax_acc', ptr(in1), W, W, in1.numel() // W, ptr(amax_x), st)
        use_batch_stats = training or not bn.track_running_stats
        rows = _lib.lib.fsdet_conv_first_tc_rows(B, H, W)
        stat = None
        if use_batch_stats:
            stat = _empty(rows + _lib.lib.fsdet_bn_stat_scratch_rows(), 4 * s.cout, device=dev)
            self._timed('first_tc', 2.0 * npix * s.cout * 36, 'fsdet_conv_first_tc_stats', ptr(in0), c0, ptr(in1), c1, ptr(w4),
                        ptr(amax_x), ptr(stat), B, H, W, s.cout, st)
        vec = _empty(5, s.cout, device=dev)
        vec.xh_ok = bool(use_batch_stats)
        amax_y = _empty(1, device=dev) if use_batch_stats else None
        upd = training and bn.track_running_stats
        call('fsdet_bn_finalize', ptr(stat), rows, float(npix), ptr(bn.weight), ptr(bn.bias),
             ptr(bn.running_mean) if (upd or not use_batch_stats) else None,
             ptr(bn.running_var) if (upd or not use_batch_stats) else None,
             BN_MOMENTUM if bn.momentum is None else float(bn.momentum), float(bn.eps),
             ptr(vec[0]), ptr(vec[1]), ptr(vec[2]), ptr(vec[3]), s.slope, ptr(amax_y), ptr(vec[4]), s.cout,
             1 if use_batch_stats else 0, st)
        if upd and bn.num_batches_tracked is not None:
            bn.num_batches_tracked += 1
        pos = self.specs.index(s)
        Hp, Wp = H // 2, W // 2
        cp64 = _round_up(s.cout, 64)
        planes_ok = (amax_y is not None and (s.idx + 1) not in self.placement and (s.idx + 1) not in self.routed
                     and self._consumer_takes_planes(pos + 2, s.cout))
        ppl = None
        if planes_ok:
            ppl = (torch.empty(B * Hp * Wp, cp64, dtype=torch.float16, device=dev),
                   torch.empty(B * Hp * Wp, cp64, dtype=torch.float16, device=dev), amax_y)
            pooled = Act.planes_only(B, Hp, Wp, s.cout, dev, ppl)
        else:
            pooled = out_act(s.idx + 1, B, Hp, Wp, s.cout)
            pooled.amax = amax_y
        p32 = pooled if pooled.buf is not None else None
        self._timed('first_tc', 2.0 * npix * s.cout * 36, 'fsdet_conv_first_tc_apply', ptr(in0), c0, ptr(in1), c1, ptr(w4),
                    ptr(amax_x), ptr(vec[2]), ptr(vec[3]), s.slope, p32.ptr if p32 else None, p32.ld if p32 else 0,
                    ptr(ppl[0]) if ppl else None, ptr(ppl[1]) if ppl else None, cp64 if ppl else 0, ptr(amax_y) if ppl else None,
                    B, H, W, s.cout, st)
        rec = ('first_tc', s, x, w4, vec, pooled, conv, bn, amax_x)
        return (None, pooled), rec

    def _first_tc_bwd(self, rec, st):
        _, s, x, w4, vec, pooled, conv, bn, amax_x = rec
        dev = x.dev
        B, H, W = x.B, x.H, x.W
        in0, c0, in1, c1 = x.nchw
        gp = pooled.grad_for_read()
        gw, fin_w = self._param_grad(conv.weight)
        gg, fin_g = self._param_grad(bn.weight)
        gb, fin_b = self._param_grad(bn.bias)
        if gp is None:
            for t in (gw, gg, gb):
                t.zero_()
        else:
            rows = _lib.lib.fsdet_conv_first_tc_rows(B, H, W)
            part = _empty(rows + 1, 3 * s.cout, dtype=torch.float64, device=dev)
            coef = _empty(2, s.cout, dtype=torch.float64, device=dev)
            flops = 2.0 * x.npix * s.cout * 36
            self._timed('first_tc', flops, 'fsdet_conv_first_tc_bwd_reduce', ptr(in0), c0, ptr(in1), c1, ptr(w4), ptr(amax_x),
                        ptr(vec[2]), ptr(vec[3]), ptr(vec[0]), ptr(vec[1]), s.slope, gp.ptr, gp.ld, ptr(part), B, H, W, s.cout, st)
            amax_dz = _empty(1, device=dev)
            call('fsdet_bn_bwd_finalize', ptr(part), rows, float(x.npix), ptr(bn.weight), ptr(vec[1]), ptr(vec[4]), ptr(gg), ptr(gb),
                 ptr(coef), ptr(amax_dz), s.cout, 1, st)
            nws = _lib.lib.fsdet_conv_first_tc_wgrad_workspace_floats(B, H, W)
            ws = _empty(max(nws, 4), device=dev)
            gw4 = gw if s.cin == 4 else _empty(s.cout, 9, 4, device=dev)
            self._timed('first_tc', 2 * flops, 'fsdet_conv_first_tc_bwd_wgrad', ptr(in0), c0, ptr(in1), c1, ptr(w4), ptr(amax_x),
                        ptr(vec[2]), ptr(vec[3]), ptr(vec[0]), ptr(vec[1]), ptr(coef), s.slope, gp.ptr, gp.ld, ptr(amax_dz),
                        ptr(gw4), ptr(ws), nws, B, H, W, s.cout, st)
            if s.cin != 4:
                call('fsdet_pad_channels', ptr(gw4), 4, ptr(gw), s.cin, s.cout * 9, st)
        for f in (fin_w, fin_g, fin_b):
            if f:
                f()
        self._done(conv.weight, bn.weight, bn.bias)

    def _head_fwd(self, s, head, x, rw, st):
        """dynamic_conv.DynamicConv2d.forward (dynamic_conv.py:125-164) + the
        following nn.Conv2d(K, O, 1): out[b*n_cls+c] = (W (.) rw[c]) x[b] + bias."""
        if rw is None:
            raise ValueError('this network has a dynamic convolution: dynamic weights are required')
        dev = x.dev
        conv, _ = self._conv_modules(self.models[head.idx])
        K = x.C
        n_cls = rw.shape[0]
        if rw.numel() != n_cls * K:
            raise ValueError('dynamic weights must be [n_cls, %d, 1, 1], got %s' % (K, tuple(rw.shape)))
        rw2 = rw.detach().reshape(n_cls, K).contiguous()
        O = head.cout
        N = n_cls * O
        Npad = _round_up(N, 64)
        W = conv.weight  # [O, K, 1, 1]: OIHW == OHWI storage for 1x1
        weff = _empty(Npad, K, device=dev)
        beff = _empty(Npad, device=dev)
        call('fsdet_head_weff', ptr(W), ptr(conv.bias), ptr(rw2), ptr(weff), ptr(beff), n_cls, O, K, Npad, st)
        z = Act.new(x.B, x.H, x.W, Npad, dev)
        self._conv('head', x, weff, None, z, None, K, Npad, 1, 0, st)
        out = _empty(x.B * n_cls, O, x.H, x.W, device=dev)
        call('fsdet_nhwc_to_nchw', z.ptr, z.ld, ptr(beff), ptr(out), x.B, N, x.H * x.W, st)  # + bias[o]
        rec = ('head', s, head, x, rw2, weff, conv, n_cls, O, Npad)
        return out, rec

    # -- backward ----------------------------------------------------------
    def backward(self, tape, gout):
        """Replays the tape in reverse. gout: gradient of the NCHW result.
        Parameter gradients are written into `.grad` directly. Returns the
        gradient w.r.t. the dynamic weights (or None)."""
        st = _stream()
        gout = gout.contiguous()
        drw = None
        self._side_used = False
        self._main = torch.cuda.current_stream()
        try:
            drw = self._backward_records(tape, gout, st)
        finally:
            if self._side_used:         # join: everything after the backward pass sees the weight gradients
                self._main.wait_stream(self.side)
                self._side_used = False
            self._keep = []
        return drw

    def _backward_records(self, tape, gout, st):
        drw = None
        for rec in reversed(tape.records):
            kind = rec[0]
            if kind == 'head':
                drw = self._head_bwd(rec, gout, st)
            elif kind == 'output':
                _, act, c_true = rec
                g, acc = act.grad_for_write()
                if acc:
                    raise NotImplementedError('network output consumed elsewhere')
                call('fsdet_nchw_to_nhwc', ptr(gout), c_true, None, 0, g.ptr, g.ld, g.C, act.B, act.H * act.W, st)
            elif kind == 'globalmax':
                _, s, x, arg = rec
                g, acc = x.grad_for_write()
                tgt = g if not acc else Act.new(x.B, x.H, x.W, x.C, x.buf.device, False)
                gy = gout.reshape(x.B, x.C)
                call('fsdet_globalmax_bwd', ptr(gy), ptr(arg), tgt.ptr, tgt.ld, x.B, x.H * x.W, x.C, st)
                if acc:
                    call('fsdet_copy_channels', tgt.ptr, tgt.ld, g.ptr, g.ld, x.npix, x.C, 1, st)
            elif kind == 'convbn':
                self._convbn_bwd(rec, st)
            elif kind == 'first_tc':
                self._first_tc_bwd(rec, st)
            elif kind == 'convbias':
                self._convbias_bwd(rec, st)
            elif kind == 'maxpool':
                _, s, x, y = rec
                gy = y.grad_for_read()
                if gy is None or not x.needs_grad:
                    continue
                g, acc = x.grad_for_write()
                tgt = g if not acc else Act.new(x.B, x.H, x.W, x.C, x.buf.device, False)
                call('fsdet_maxpool_bwd', x.ptr, x.ld, gy.ptr, gy.ld, tgt.ptr, tgt.ld, x.B, x.H, x.W, x.C, s.stride, st)
                if acc:
                    call('fsdet_copy_channels', tgt.ptr, tgt.ld, g.ptr, g.ld, x.npix, x.C, 1, st)
            elif kind == 'reorg':
                _, s, x, y = rec
                gy = y.grad_for_read()
                if gy is None or not x.needs_grad:
                    continue
                g, acc = x.grad_for_write()
                tgt = g if not acc else Act.new(x.B, x.H, x.W, x.C, x.buf.device, False)
                call('fsdet_reorg_bwd', gy.ptr, gy.ld, tgt.ptr, tgt.ld, x.B, x.H, x.W, x.C, st)
                if acc:
                    call('fsdet_copy_channels', tgt.ptr, tgt.ld, g.ptr, g.ld, x.npix, x.C, 1, st)
            elif kind == 'cat':
                _, s, a0, a1, cat = rec
                gc = cat.grad_for_read()
                if gc is None:
                    continue
                off = 0
                for a in (a0, a1):
                    if a.needs_grad:
                        g, acc = a.grad_for_write()
                        call('fsdet_copy_channels', gc.ptr + 4 * off, gc.ld, g.ptr, g.ld, a.npix, a.C, acc, st)
                    off += a.C
            else:
                raise NotImplementedError(kind)
        return drw

    def _dgrad(self, x, dz, w_ohwi, cin_p, cout, k, st):
        """dX = conv(dZ, flip-transposed W) accumulated into x's gradient."""
        if not x.needs_grad:
            return
        dev = x.dev
        kk = k * k
        g, acc = x.grad_for_write()
        wp = getattr(self, '_wp', {}).get(id(w_ohwi))
        if wp is not None and wp['bwd'] is not None and dz.planes is not None:
            # flip-transposed planes prepared at the start of the step; `w_ohwi` only names the layer here
            self._conv('dgrad', dz, w_ohwi, None, g, None, cout, cin_p, k, acc, st, wplanes=wp['bwd'])
            return
        wt = _empty(cin_p, kk, cout, device=dev)
        call('fsdet_weight_flip_transpose', ptr(w_ohwi), ptr(wt), cout, kk, cin_p, st)
        known = getattr(w_ohwi, '_fsdet_amax', None)
        w_amax = known[0] if (known is not None and known[1] == w_ohwi._version) else None
        self._conv('dgrad', dz, wt, None, g, None, cout, cin_p, k, acc, st, w_amax)

    @staticmethod
    def _wgrad_tc_ok(cin_p, cout, k):
        return bool(USE_TC and 'wgrad' in TC_PARTS and cin_p >= 32 and cout >= 32 and _lib.lib.fsdet_conv_tc_wgrad_supported(
            _round_up(cin_p, 64), _round_up(cout, 64), k))

    def _wgrad(self, x, dz, out_tensor, cin_p, cout, k, st):
        dev = x.dev
        flops = 2.0 * x.npix * cout * k * k * cin_p
        ci64, co64 = _round_up(cin_p, 64), _round_up(cout, 64)
        if x.nchw is None and self._wgrad_tc_ok(cin_p, cout, k):
            xh, xl, xa = self._planes(x, st)
            dh, dl, da = self._planes(dz, st)
            mode = TC_TERMS['wgrad']
            nws = _lib.lib.fsdet_conv_tc_wgrad_workspace_floats(x.B, x.H, x.W, ci64, co64, k, mode)
            ws = _empty(max(nws, 4), device=dev)
            padded = (ci64 != cin_p) or (co64 != cout)
            tgt = _empty(co64, k * k, ci64, device=dev) if padded else out_tensor
            self._timed('wgrad_tc', flops, 'fsdet_conv_tc_wgrad', ptr(xh), ptr(xl), ptr(dh), ptr(dl), ptr(xa), ptr(da),
                        ptr(tgt), ptr(ws), nws, x.B, x.H, x.W, ci64, co64, k, mode, st)
            if padded:  # crop the zero channels / rows: rows [0, cout) are contiguous, channels via pad_channels
                call('fsdet_pad_channels', ptr(tgt), ci64, ptr(out_tensor), cin_p, cout * k * k, st)
            return
        if x.nchw is not None:
            in0, c0, in1, c1 = x.nchw
            nws = _lib.lib.fsdet_conv_first_wgrad_workspace_floats_cin(x.B, x.H, x.W, c0 + c1, cout)
            ws = _empty(max(nws, 4), device=dev)
            self._timed('first_wgrad', flops, 'fsdet_conv_first_wgrad', ptr(in0), c0, ptr(in1), c1, dz.ptr, dz.ld, ptr(out_tensor),
                        ptr(ws), nws, x.B, x.H, x.W, cout, st)
            return
        nws = _lib.lib.fsdet_conv_wgrad_workspace_floats(x.B, x.H, x.W, cin_p, cout, k)
        ws = _empty(max(nws, 4), device=dev)
        self._timed('conv_wgrad', flops, 'fsdet_conv_wgrad', x.ptr, x.ld, dz.ptr, dz.ld, ptr(out_tensor), ptr(ws), nws, x.B,
                    x.H, x.W, cin_p, cout, k, st)

    def _convbn_bwd(self, rec, st):
        _, s, x, wuse, z, vec, full, pooled, conv, bn = rec
        dev = x.dev
        B, H, W = x.B, x.H, x.W
        gf = full.grad_for_read() if full is not None else None
        gp = pooled.grad_for_read() if pooled is not None else None
        gw, fin_w = self._param_grad(conv.weight)
        gg, fin_g = self._param_grad(bn.weight)
        gb, fin_b = self._param_grad(bn.bias)
        if gf is None and gp is None:
            for t in (gw, gg, gb):
                t.zero_()
            for f in (fin_w, fin_g, fin_b):
                if f:
                    f()
            self._done(conv.weight, bn.weight, bn.bias)
            return
        rows = _lib.lib.fsdet_bn_bwd_rows(B, H, W)
        part = _empty(rows + 1, 3 * s.cout, dtype=torch.float64, device=dev)
        coef = _empty(2, s.cout, dtype=torch.float64, device=dev)
        a_gf = (gf.ptr, gf.ld) if gf is not None else (None, 0)
        a_gp = (gp.ptr, gp.ld) if gp is not None else (None, 0)
        call('fsdet_bn_act_bwd_reduce', z.ptr, z.ld, a_gf[0], a_gf[1], a_gp[0], a_gp[1], ptr(vec[2]), ptr(vec[3]),
             ptr(vec[0]), ptr(vec[1]), s.slope, ptr(part), B, H, W, s.cout, 1, st)
        # which GEMMs will read dz, and in which form: the tensor-core ones take fp16 planes, written directly by
        # the apply pass (scaled by the bound of max|dz| from the finalize step); fp32 dz only if a SIMT kernel needs it
        cin_p = x.C
        wg_tc = self._wgrad_tc_ok(cin_p, s.cout, s.k)
        dg_tc = x.needs_grad and 'dgrad' in TC_PARTS and self._tc_ok(s.cout, cin_p, s.k)
        want_planes = USE_TC and s.cout % 64 == 0 and (wg_tc or dg_tc) and getattr(vec, 'xh_ok', False)
        want_f32 = (not want_planes) or (not wg_tc) or (x.needs_grad and not dg_tc)
        amax = _empty(1, device=dev) if want_planes else None
        call('fsdet_bn_bwd_finalize', ptr(part), rows, float(x.npix), ptr(bn.weight), ptr(vec[1]), ptr(vec[4]), ptr(gg), ptr(gb),
             ptr(coef), ptr(amax), s.cout, 1, st)
        planes = None
        if want_planes:
            planes = (torch.empty(x.npix, s.cout, dtype=torch.float16, device=dev),
                      torch.empty(x.npix, s.cout, dtype=torch.float16, device=dev), amax)
        if want_f32:
            dz = Act.new(B, H, W, s.cout, dev, False)
            dz.planes = planes
        else:
            dz = Act.planes_only(B, H, W, s.cout, dev, planes)
        call('fsdet_bn_act_bwd_apply', z.ptr, z.ld, a_gf[0], a_gf[1], a_gp[0], a_gp[1], ptr(vec[2]), ptr(vec[3]),
             ptr(vec[0]), ptr(vec[1]), ptr(coef), s.slope, dz.ptr if want_f32 else None, dz.ld if want_f32 else 0,
             ptr(planes[0]) if planes else None, ptr(planes[1]) if planes else None, s.cout, ptr(amax), B, H, W, s.cout, 1, st)
        cin_p = x.C

        def weight_grad(sw):
            if cin_p != s.cin:
                gwp = _empty(s.cout, s.k * s.k, cin_p, device=dev)
                self._wgrad(x, dz, gwp, cin_p, s.cout, s.k, sw)
                call('fsdet_pad_channels', ptr(gwp), cin_p, ptr(gw), s.cin, s.cout * s.k * s.k, sw)
            else:
                self._wgrad(x, dz, gw, cin_p, s.cout, s.k, sw)
            if fin_w:
                fin_w()
            self._done(conv.weight, bn.weight, bn.bias)

        for f in (fin_g, fin_b):
            if f:
                f()
        if self._side_ok():
            # fork behind the apply pass; dz (and the activation planes) were allocated on the main stream: keep them alive
            # until the join at the end of the backward pass, the allocator only orders their reuse on the main stream
            self.side.wait_stream(self._main)
            self._side_used = True
            self._keep.append((dz, planes, x))
            with torch.cuda.stream(self.side):
                weight_grad(self.side.cuda_stream)
        else:
            weight_grad(st)
        self._dgrad(x, dz, wuse, cin_p, s.cout, s.k, st)

    def _convbias_bwd(self, rec, st):
        _, s, x, wp, z, onez, full, pooled, conv, cout_p = rec
        dev = x.dev
        B, H, W = x.B, x.H, x.W
        gf = full.grad_for_read() if full is not None else None
        gp = pooled.grad_for_read() if pooled is not None else None
        gw, fin_w = self._param_grad(conv.weight)
        gb, fin_b = self._param_grad(conv.bias) if conv.bias is not None else (None, None)
        if gf is None and gp is None:
            gw.zero_()
            if gb is not None:
                gb.zero_()
            for f in (fin_w, fin_b):
                if f:
                    f()
            self._done(conv.weight, conv.bias)
            return
        ones, zeros = onez
        if ones is None:
            ones = torch.ones(cout_p, device=dev)
            zeros = torch.zeros(cout_p, device=dev)
        rows = _lib.lib.fsdet_bn_bwd_rows(B, H, W)
        part = _empty(rows + 1, 3 * cout_p, dtype=torch.float64, device=dev)
        dbp = _empty(cout_p, device=dev)
        a_gf = (gf.ptr, gf.ld) if gf is not None else (None, 0)
        a_gp = (gp.ptr, gp.ld) if gp is not None else (None, 0)
        call('fsdet_bn_act_bwd_reduce', z.ptr, z.ld, a_gf[0], a_gf[1], a_gp[0], a_gp[1], ptr(ones), ptr(zeros), None, None,
             s.slope, ptr(part), B, H, W, cout_p, 0, st)
        call('fsdet_bn_bwd_finalize', ptr(part), rows, float(x.npix), None, None, None, None, ptr(dbp), None, None, cout_p, 0, st)
        if full is z and gp is None:
            dz = gf  # linear, unpooled: dZ is the incoming gradient itself
        else:
            dz = Act.new(B, H, W, cout_p, dev, False)
            call('fsdet_bn_act_bwd_apply', z.ptr, z.ld, a_gf[0], a_gf[1], a_gp[0], a_gp[1], ptr(ones), ptr(zeros), None,
                 None, None, s.slope, dz.ptr, dz.ld, None, None, 0, None, B, H, W, cout_p, 0, st)
        cin_p = x.C
        kk = s.k * s.k
        gwp = _empty(cout_p, kk, cin_p, device=dev)
        self._wgrad(x, dz, gwp, cin_p, cout_p, s.k, st)
        if cin_p != s.cin:
            call('fsdet_pad_channels', ptr(gwp), cin_p, ptr(gw), s.cin, s.cout * kk, st)
        else:
            # rows [0, cout) of the padded gradient, OHWI order == gw's storage order
            gw.permute(0, 2, 3, 1).copy_(gwp[:s.cout].view(s.cout, s.k, s.k, cin_p))
        if gb is not None:
            gb.copy_(dbp[:s.cout])
        for f in (fin_w, fin_b):
            if f:
                f()
        self._done(conv.weight, conv.bias)
        self._dgrad(x, dz, wp, cin_p, cout_p, s.k, st)

    def _head_bwd(self, rec, gout, st):
        _, s, head, x, rw2, weff, conv, n_cls, O, Npad = rec
        dev = x.dev
        K = x.C
        N = n_cls * O
        HW = x.H * x.W
        dzh = Act.new(x.B, x.H, x.W, Npad, dev, False)
        call('fsdet_nchw_to_nhwc', ptr(gout), N, None, 0, dzh.ptr, dzh.ld, Npad, x.B, HW, st)
        gw, fin_w = self._param_grad(conv.weight)
        gb, fin_b = self._param_grad(conv.bias) if conv.bias is not None else (None, None)
        if gb is not None:
            nws = _lib.lib.fsdet_head_bias_grad_workspace_floats(x.npix, n_cls, O)
            ws = _empty(max(nws, 1), device=dev)
            call('fsdet_head_bias_grad', dzh.ptr, dzh.ld, ptr(gb), ptr(ws), x.npix, n_cls, O, st)
        dweff = _empty(Npad, K, device=dev)
        self._wgrad(x, dzh, dweff, K, Npad, 1, st)
        drw = _empty(n_cls, K, device=dev)
        call('fsdet_head_param_grads', ptr(dweff), ptr(conv.weight), ptr(rw2), ptr(gw), ptr(drw), n_cls, O, K, st)
        for f in (fin_w, fin_b):
            if f:
                f()
        self._done(conv.weight, conv.bias)
        self._dgrad(x, dzh, weff, K, Npad, 1, st)
        return drw


class _NetFunction(torch.autograd.Function):
    """Autograd boundary of one network. Parameters are passed so that autograd
    schedules the backward; their gradients are written into `.grad` by the
    executor (None is returned for them)."""

    @staticmethod
    def forward(ctx, runner, training, n_in, has_extra, *tensors):
        inputs = list(tensors[:n_in])
        extra = tensors[n_in] if has_extra else None
        out, tape = runner.forward(inputs, extra, training=training, record=True)
        ctx.runner = runner
        ctx.tape = tape
        ctx.n_in = n_in
        ctx.has_extra = has_extra
        ctx.n_tensors = len(tensors)
        ctx.extra_shape = tuple(extra.shape) if has_extra else None
        return out

    @staticmethod
    def backward(ctx, gout):
        tape = ctx.tape
        ctx.tape = None
        drw = ctx.runner.backward(tape, gout)
        grads = [None] * ctx.n_tensors
        if ctx.has_extra and drw is not None:
            grads[ctx.n_in] = drw.view(ctx.extra_shape)
        return (None, None, None, None) + tuple(grads)


def run_network(runner, inputs, extra, params, training):
    """Forward through `runner`; differentiable when grad mode is on."""
    need_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in params) or
                                             (extra is not None and extra.requires_grad))
    if not need_grad:
        out, _ = runner.forward(list(inputs), extra, training=training, record=False)
        return out
    tensors = list(inputs) + ([extra] if extra is not None else []) + list(params)
    return _NetFunction.apply(runner, training, len(inputs), extra is not None, *tensors)
