"""ctypes binding of libb200tts.so (C ABI declared in include/b200tts.h).

There is deliberately no fallback: if the library is missing or no CUDA device is
visible, the first compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from .build import LIB

OK = 0
RNG_PHILOX, RNG_EXT_EXPONENTIAL = 0, 1
KERNEL_AUTO, KERNEL_UTTERANCE, KERNEL_GRID, KERNEL_TC = 0, 1, 2, 3
KERNELS = {'auto': KERNEL_AUTO, 'utterance': KERNEL_UTTERANCE, 'grid': KERNEL_GRID, 'tc': KERNEL_TC}


class B200TTSError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f'libb200tts error {code}: {msg}')
        self.code = code


class WaveRNNCfg(C.Structure):
    _fields_ = [('rnn_dims', C.c_int32), ('fc_dims', C.c_int32), ('bits', C.c_int32), ('pad', C.c_int32),
                ('feat_dims', C.c_int32), ('compute_dims', C.c_int32), ('res_out_dims', C.c_int32),
                ('res_blocks', C.c_int32), ('n_upsample', C.c_int32), ('upsample_factors', C.c_int32 * 4),
                ('hop_length', C.c_int32)]


class Tensor(C.Structure):
    _fields_ = [('name', C.c_char_p), ('data', C.c_void_p), ('ndim', C.c_int32), ('shape', C.c_int64 * 4)]


class Rng(C.Structure):
    _fields_ = [('mode', C.c_int32), ('seed', C.c_uint64), ('utterance_offset', C.c_uint64), ('d_q', C.c_void_p),
                ('d_utterance_ids', C.c_void_p)]


class GenOpts(C.Structure):
    _fields_ = [('kernel', C.c_int32), ('mu_law', C.c_int32), ('d_teacher', C.c_void_p), ('d_logits', C.c_void_p),
                ('max_steps', C.c_int32), ('fold_target', C.c_int32), ('fold_overlap', C.c_int32), ('d_utt_frames', C.c_void_p),
                ('d_pack_utt', C.c_void_p), ('d_pack_start', C.c_void_p), ('pack_rows', C.c_int32), ('pack_segs', C.c_int32),
                ('pack_steps', C.c_int32)]


class TacoCfg(C.Structure):
    _fields_ = [('num_mels', C.c_int32), ('prenet_units', C.c_int32), ('lstm_units', C.c_int32), ('enc_dim', C.c_int32),
                ('attn_dim', C.c_int32), ('attn_filters', C.c_int32), ('attn_kernel', C.c_int32), ('zoneout', C.c_float)]


class TacoDropout(C.Structure):
    _fields_ = [('mode', C.c_int32), ('seed', C.c_uint64), ('utterance_offset', C.c_uint64), ('d_masks', C.c_void_p)]


# every symbol include/b200tts.h declares: (restype, argtypes)
SIGNATURES = {
    'b200tts_abi_version': (C.c_int, []),
    'b200tts_last_error': (C.c_char_p, []),
    'b200tts_device_count': (C.c_int, []),
    'b200tts_wavernn_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(WaveRNNCfg), C.POINTER(Tensor), C.c_int]),
    'b200tts_wavernn_destroy': (None, [C.c_void_p]),
    'b200tts_wavernn_upsample': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]),
    'b200tts_wavernn_generate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(Rng), C.POINTER(GenOpts),
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    'b200tts_wavernn_generate_stream': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(Rng), C.POINTER(GenOpts),
                                                  C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'b200tts_wavernn_stream_wait': (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_int64)]),
    'b200tts_wavernn_fold_geometry': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'b200tts_wavernn_generate_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(Rng),
                                                C.POINTER(GenOpts), C.c_void_p, C.c_void_p]),
    'b200tts_philox_exponential': (C.c_int, [C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_void_p]),
    'b200tts_wavernn_launch_count': (C.c_int64, [C.c_void_p]),
    'b200tts_wavernn_last_kernel_ms': (C.c_double, [C.c_void_p]),
    'b200tts_wavernn_last_kernel': (C.c_int, [C.c_void_p]),
    'b200tts_wavernn_debug_phase_cycles': (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    'b200tts_wavernn_check': (C.c_int, [C.c_void_p]),
    'b200tts_debug_fp32_peak': (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    'b200tts_taco_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(TacoCfg), C.POINTER(Tensor), C.c_int]),
    'b200tts_taco_destroy': (None, [C.c_void_p]),
    'b200tts_taco_decode': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(TacoDropout), C.c_int,
                                      C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'b200tts_taco_state_floats': (C.c_int, [C.c_void_p, C.c_int]),
    'b200tts_taco_decode_forced': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(TacoDropout), C.c_int,
                                             C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'b200tts_taco_encode': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    'b200tts_taco_postnet': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    'b200tts_taco_philox_masks': (C.c_int, [C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
}

_lib = None
_lock = threading.Lock()


def lib_path() -> str:
    return os.environ.get('B200TTS_LIB', LIB)


def load():
    """Loads the shared library once and declares every prototype."""
    global _lib
    with _lock:
        if _lib is None:
            path = lib_path()
            if not os.path.isfile(path):
                raise RuntimeError(f'{path} not found: the CUDA library is not built and there is no CPU fallback. '
                                   f'Run `python -m tacotronv2_wavernn_chinese_b200.build` '
                                   f'(or `python -c "import __graft_entry__ as g; g.build()"`).')
            lib = C.CDLL(path)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            if lib.b200tts_abi_version() != 3:
                raise RuntimeError('libb200tts.so ABI version mismatch; rebuild it')
            _lib = lib
    return _lib


def check(rc: int):
    if rc != OK:
        raise B200TTSError(rc, load().b200tts_last_error().decode('utf-8', 'replace'))


def make_tensor_array(state: dict):
    """dict name -> float32 C-contiguous numpy array  ->  (ctypes array, keep-alive list)."""
    items = [(k, v) for k, v in state.items() if v.dtype == np.float32]
    arr = (Tensor * len(items))()
    keep = []
    for i, (k, v) in enumerate(items):
        v = np.ascontiguousarray(v)
        keep.append(v)
        name = k.encode()
        keep.append(name)
        arr[i].name = name
        arr[i].data = v.ctypes.data
        arr[i].ndim = v.ndim
        for d in range(v.ndim):
            arr[i].shape[d] = v.shape[d]
    return arr, keep
