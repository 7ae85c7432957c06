"""ctypes binding of libfsdet.so (declared in include/fsdet.h).

There is NO fallback: if the shared library is missing or a symbol cannot be
resolved the import fails loudly.  `call(name, *args)` raises RuntimeError with
`fsdet_last_error()` on a non-zero return code.
"""
import collections
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libfsdet.so')

_P, _I, _F, _D, _Z, _Q = (ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_size_t,
                          ctypes.c_longlong)
_T = {'p': _P, 'i': _I, 'f': _F, 'd': _D, 'z': _Z, 'q': _Q}

# name -> (argument codes, restype code)   [must match include/fsdet.h]
SIGNATURES = {
    'fsdet_version': ('', 'i'),
    'fsdet_last_error': ('', 's'),
    'fsdet_compiled_arch': ('', 'i'),
    'fsdet_nchw_to_nhwc': ('pipipiiiip', 'i'),
    'fsdet_nhwc_to_nchw': ('pippiiip', 'i'),
    'fsdet_conv_fwd': ('pipppip iiiiiii p'.replace(' ', ''), 'i'),
    'fsdet_conv_stat_rows': ('i', 'i'),
    'fsdet_conv_wgrad': ('pipippz iiiiii p'.replace(' ', ''), 'i'),
    'fsdet_conv_wgrad_workspace_floats': ('iiiiii', 'z'),
    'fsdet_conv_first_fwd': ('pipippiiiiip', 'i'),
    'fsdet_conv_first_stat_rows': ('iii', 'i'),
    'fsdet_conv_first_fwd_stats': ('pipippiiiiipp', 'i'),
    'fsdet_conv_first_wgrad': ('pipipippziiiip', 'i'),
    'fsdet_conv_first_wgrad_workspace_floats': ('iiii', 'z'),
    'fsdet_conv_first_wgrad_workspace_floats_cin': ('iiiii', 'z'),
    'fsdet_conv_first_wgrad_supported': ('ii', 'i'),
    'fsdet_conv_first_tc_supported': ('iii', 'i'),
    'fsdet_conv_first_tc_rows': ('iii', 'i'),
    'fsdet_conv_first_tc_stats': ('pipipppiiiip', 'i'),
    'fsdet_conv_first_tc_apply': ('pipipp pp f pi pp i p iiii p'.replace(' ', ''), 'i'),
    'fsdet_conv_first_tc_bwd_reduce': ('pipipp pppp f pi p iiii p'.replace(' ', ''), 'i'),
    'fsdet_conv_first_tc_wgrad_workspace_floats': ('iii', 'z'),
    'fsdet_conv_first_tc_bwd_wgrad': ('pipipp pppp p f pi p p pz iiii p'.replace(' ', ''), 'i'),
    'fsdet_weight_flip_transpose': ('ppiiip', 'i'),
    'fsdet_pad_channels': ('pipizp', 'i'),
    'fsdet_conv_tc_supported': ('iii', 'i'),
    'fsdet_conv_tc_stat_rows': ('iiiiiii', 'i'),
    'fsdet_conv_tc_uses_halo': ('iiiiiii', 'i'),
    'fsdet_conv_tc_fwd': ('pppppppiiiiiiiiiipp', 'i'),
    'fsdet_conv_tc_wgrad_supported': ('iii', 'i'),
    'fsdet_conv_tc_wgrad_workspace_floats': ('iiiiiii', 'z'),
    'fsdet_conv_tc_wgrad': ('ppppppppziiiiiiip', 'i'),
    'fsdet_weight_prep': ('ppipip', 'i'),
    'fsdet_amax': ('piizpp', 'i'),
    'fsdet_amax_acc': ('piizpp', 'i'),
    'fsdet_split_f16': ('piiizpppp', 'i'),
    'fsdet_colstats': ('pizipp', 'i'),
    'fsdet_colstats_rows': ('z', 'i'),
    'fsdet_debug_im2col_tile': ('piiiiiqiipp', 'i'),
    'fsdet_bn_finalize': ('pidppppffppppfppiip', 'i'),
    'fsdet_bn_stat_scratch_rows': ('', 'i'),
    'fsdet_bn_act_fwd': ('pippfpipippppipiiiip', 'i'),
    'fsdet_bn_act_bwd_reduce': ('pipipippppfpiiiiip', 'i'),
    'fsdet_bn_bwd_rows': ('iii', 'i'),
    'fsdet_bn_bwd_finalize': ('pidpppppppiip', 'i'),
    'fsdet_bn_act_bwd_apply': ('pipipipppppfpippipiiiiip', 'i'),
    'fsdet_maxpool_fwd': ('pipiiiiiip', 'i'),
    'fsdet_maxpool_bwd': ('pipipiiiiiip', 'i'),
    'fsdet_reorg_fwd': ('pipiiiiip', 'i'),
    'fsdet_reorg_bwd': ('pipiiiiip', 'i'),
    'fsdet_globalmax_fwd': ('pippiiip', 'i'),
    'fsdet_globalmax_bwd': ('pppiiiip', 'i'),
    'fsdet_copy_channels': ('pipiziip', 'i'),
    'fsdet_head_weff': ('pppppiiiip', 'i'),
    'fsdet_head_param_grads': ('pppppiiip', 'i'),
    'fsdet_head_bias_grad': ('pippziip', 'i'),
    'fsdet_head_bias_grad_workspace_floats': ('zii', 'z'),
    'fsdet_region_decode': ('ppipiiiippp', 'i'),
    'fsdet_build_targets': ('pppiiiiifffqppppppppppppp', 'i'),
    'fsdet_region_loss_grad': ('ppppp iiiiiiii ppppppppp ff ii p p'.replace(' ', ''), 'i'),
    'fsdet_sgd_step': ('ppppppiiffffipp', 'i'),
    'fsdet_fill': ('pfzp', 'i'),
    'fsdet_region_detect': ('ppiiiiiiiidpppp', 'i'),
    'fsdet_nms': ('ppiiiidppp', 'i'),
    'fsdet_nms_boxes64': ('ppiidppp', 'i'),
    'fsdet_rw_running_mean': ('pppppiiip', 'i'),
    'fsdet_augment_workspace_bytes': ('iiii', 'z'),
    'fsdet_augment_batch': ('pppiiiiipzpppp', 'i'),
    'fsdet_augment_batch_pitched': ('pppiiiiipzpzppp', 'i'),
    'fsdet_box_masks': ('piiipp', 'i'),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'libfsdet.so not found at %s. Build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU or PyTorch fallback.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (args, res) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.argtypes = [_T[c] for c in args]
        fn.restype = ctypes.c_char_p if res == 's' else _T[res]
    return lib


lib = _load()


def last_error():
    e = lib.fsdet_last_error()
    return e.decode() if e else ''


CALLS = collections.Counter()  # C-ABI calls made so far, by entry point (bench.py's gpu_launches)


def call(name, *args):
    CALLS[name] += 1
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError('%s failed (rc=%d): %s' % (name, rc, last_error()))
    return rc


def ptr(t, offset_elems=0):
    """Device pointer of a torch tensor (or None) plus an element offset."""
    if t is None:
        return None
    return t.data_ptr() + offset_elems * t.element_size()
