"""ctypes binding of libffc_b200.so (include/ffc_b200.h).  No CPU fallback: a missing library is fatal."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('FFC_B200_LIB', os.path.join(_HERE, 'libffc_b200.so'))   # override: kernel-variant experiments only

LOSS_TYPES = {'AM': 0, 'Arc': 1, 'SV': 2}
PRECISIONS = {'bf16': 0, 'fp32': 1}
LRU_MAX_BATCH = 1024     # keys per chunk of the resolve CTA
LRU_MAX_KEYS = 65536     # keys per ffc_lru_assign call
TOPK_MAX = 10
IDENTIFY_MAX_ROWS = 65536  # query rows per ffc_identify call
KEY_RESERVED = (-(1 << 63), -(1 << 63) + 1)

c_void_p, c_int, c_int32, c_int64, c_float = C.c_void_p, C.c_int, C.c_int32, C.c_int64, C.c_float


class HeadConfig(C.Structure):
    _fields_ = [('max_rows', c_int32), ('q_local', c_int64), ('q_total', c_int64), ('col_offset', c_int64),
                ('feat_dim', c_int32), ('loss_type', c_int32), ('scale', c_float), ('margin', c_float),
                ('topk', c_int32), ('precision', c_int32)]


class HeadPass(C.Structure):
    _fields_ = [('p_f32', c_void_p), ('queue_f32', c_void_p), ('queue_bf16', c_void_p), ('label', c_void_p),
                ('ones_list', c_void_p), ('n_ones', c_void_p), ('cmask', c_void_p), ('n_rows', c_int32)]


class HeadStats(C.Structure):
    _fields_ = [('lsum', c_void_p), ('osum', c_void_p), ('tgt', c_void_p), ('topv', c_void_p), ('topi', c_void_p)]


class FinalizeOpts(C.Structure):
    _fields_ = [('overlay_map', c_void_p), ('overlay_g', c_void_p), ('overlay_undo', c_void_p), ('dp_peer', c_void_p),
                ('dp_rows_per_rank', c_int32), ('dp_slot_offset', c_int64)]


class TailArgs(C.Structure):
    _fields_ = [('x', c_void_p), ('p', c_void_p), ('p_stride', c_int64), ('inv_norm', c_void_p), ('n_rows', c_int32), ('feat_dim', c_int32),
                ('mode', c_int32), ('eps', c_float), ('momentum', c_float), ('gamma', c_void_p), ('beta', c_void_p),
                ('running_mean', c_void_p), ('running_var', c_void_p), ('save_mean', c_void_p), ('save_invstd', c_void_p),
                ('workspace', c_void_p), ('workspace_bytes', c_int64)]


# name -> (restype, argtypes); every symbol include/ffc_b200.h declares
PROTOTYPES = {
    'ffc_last_error': (C.c_char_p, []),
    'ffc_version': (C.c_char_p, []),
    'ffc_launch_count': (c_int64, []),
    'ffc_lru_create': (c_int, [c_int64, c_int64, C.POINTER(c_void_p)]),
    'ffc_lru_destroy': (c_int, [c_void_p]),
    'ffc_lru_clear': (c_int, [c_void_p, c_void_p]),
    'ffc_lru_assign': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    'ffc_lru_view': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    'ffc_lru_undo': (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    'ffc_lru_maintain': (c_int, [c_void_p, c_void_p]),
    'ffc_lru_size': (c_int, [c_void_p, C.POINTER(c_int64), C.POINTER(c_int64), c_void_p]),
    'ffc_lru_export': (c_int, [c_void_p, c_void_p, c_void_p, C.POINTER(c_int64), c_void_p]),
    'ffc_lru_import': (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    'ffc_queue_scatter': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p]),
    'ffc_queue_restore': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p]),
    'ffc_queue_restore_packed': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p]),
    'ffc_cast_bf16': (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    'ffc_head_create': (c_int, [C.POINTER(HeadConfig), C.POINTER(c_void_p)]),
    'ffc_head_destroy': (c_int, [c_void_p]),
    'ffc_head_sweep': (c_int, [c_void_p, C.POINTER(HeadPass), C.POINTER(HeadStats), c_void_p]),
    'ffc_head_prep': (c_int, [c_void_p, C.POINTER(HeadPass), C.POINTER(HeadStats), c_void_p]),
    'ffc_head_sweep_prepared': (c_int, [c_void_p, C.POINTER(HeadPass), C.POINTER(HeadStats), c_void_p]),
    'ffc_head_finalize': (c_int, [c_void_p, C.POINTER(HeadPass), C.POINTER(HeadStats), c_int, c_void_p, c_void_p, c_void_p]),
    'ffc_head_pass_single': (c_int, [c_void_p, C.POINTER(HeadPass), C.POINTER(HeadStats), c_void_p, c_void_p, c_void_p]),
    'ffc_head_record_words': (c_int, [C.POINTER(HeadConfig), c_int, C.POINTER(c_int64)]),
    'ffc_head_sweep_record': (c_int, [c_void_p, C.POINTER(HeadPass), c_void_p, c_void_p]),
    'ffc_head_finalize_gathered': (c_int, [c_void_p, C.POINTER(HeadPass), c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    'ffc_queue_scatter_indexed': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p]),
    'ffc_queue_scatter_overlay': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    'ffc_overlay_clear': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_void_p]),
    'ffc_sum_slabs': (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p]),
    'ffc_sum_slabs_barrier': (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int, c_int, c_int32, c_void_p, c_void_p]),
    'ffc_head_push_record': (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    'ffc_peer_barrier': (c_int, [c_void_p, c_int, c_int, c_int32, c_void_p, c_void_p]),
    'ffc_head_finalize_gathered_ex': (c_int, [c_void_p, C.POINTER(HeadPass), c_void_p, c_int, c_int64, C.POINTER(FinalizeOpts), c_void_p, c_void_p, c_void_p]),
    'ffc_route_keys': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'ffc_ema_chunk_elems': (c_int, []),
    'ffc_ema_update': (c_int, [c_void_p, c_int, c_float, c_float, c_void_p]),
    'ffc_tail_workspace_bytes': (c_int, [c_int, c_int, C.POINTER(c_int64)]),
    'ffc_tail_forward': (c_int, [C.POINTER(TailArgs), c_void_p]),
    'ffc_tail_backward': (c_int, [C.POINTER(TailArgs), c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    'ffc_head_set_dqueue': (c_int, [c_void_p, c_int]),
    'ffc_head_dqueue': (c_int, [c_void_p, C.POINTER(HeadPass), c_void_p, c_void_p]),
    'ffc_head_set_timing': (c_int, [c_void_p, c_int]),
    'ffc_head_get_timing': (c_int, [c_void_p, C.POINTER(C.c_double), C.POINTER(c_int64)]),
    'ffc_head_stats_bytes': (c_int, [C.POINTER(HeadConfig), c_int, C.POINTER(c_int64)]),
    'ffc_identify_workspace_bytes': (c_int, [c_void_p, c_int, c_int, C.POINTER(c_int64)]),
    'ffc_identify': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
}

_lib = None


class FFCError(RuntimeError):
    pass


def lib():
    """Load the library (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise FFCError(f'{LIB_PATH} is missing: build it with `python very-large-scale-face-recognition_b200/build.py` '
                           '(the FFC head has no CPU or PyTorch fallback)')
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int):
    if rc != 0:
        raise FFCError(lib().ffc_last_error().decode())


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def side_stream_priority():
    """Priority of the bookkeeping streams (LRU / label kernels that run underneath the sweeps): -1 = above the caller's stream, so
    that their pending blocks are placed before the sweep's pending CTAs whenever an SM frees up.  FFC_SIDE_PRIORITY overrides (0 =
    default priority: the behaviour before this switch existed; for A/B timing)."""
    return int(os.environ.get('FFC_SIDE_PRIORITY', '-1'))
