"""CPU-side checks of the streaming entry points (include/b200tts.h): argument checks come before any CUDA call, a call without a
device fails loudly, and the host-only wait helper sees a progress word that another thread raises."""
import ctypes
import threading
import time

import numpy as np

EINVAL, ECUDA = -1, -2


def _lib():
    from tacotronv2_wavernn_chinese_b200 import build, _lib
    build.build_lib()
    return _lib.load(), _lib


def _buf(n, dtype):
    a = np.zeros(n, dtype=dtype)
    return a, ctypes.c_void_p(a.ctypes.data)


def test_generate_stream_argument_checks_come_first():
    lib, L = _lib()
    fake = ctypes.create_string_buffer(4096)           # never dereferenced: every call below is refused before that
    ctx, mel = ctypes.cast(fake, ctypes.c_void_p), ctypes.c_void_p(16)
    w, wp = _buf(20 * 275, np.float64)
    p, pp = _buf(1, np.int64)
    gen = lib.b200tts_wavernn_generate_stream
    assert gen(None, mel, 1, 21, None, None, 275, wp, pp, None, None, None) == EINVAL
    assert b'null argument' in lib.b200tts_last_error()
    assert gen(ctx, None, 1, 21, None, None, 275, wp, pp, None, None, None) == EINVAL
    assert gen(ctx, mel, 1, 21, None, None, 275, None, pp, None, None, None) == EINVAL
    assert gen(ctx, mel, 1, 21, None, None, 275, wp, None, None, None, None) == EINVAL
    for chunk in (0, -5):
        assert gen(ctx, mel, 1, 21, None, None, chunk, wp, pp, None, None, None) == EINVAL
        assert b'chunk_steps' in lib.b200tts_last_error()
    for B in (0, 33):
        assert gen(ctx, mel, B, 21, None, None, 275, wp, pp, None, None, None) == EINVAL
    assert gen(ctx, mel, 1, 20, None, None, 275, wp, pp, None, None, None) == EINVAL          # shorter than the fade-out
    assert gen(ctx, mel, 1, 21, None, None, 275, wp, ctypes.c_void_p(pp.value + 4), None, None, None) == EINVAL
    refused = [dict(fold_target=11000, fold_overlap=550), dict(d_pack_utt=8, pack_rows=1, pack_segs=1, pack_steps=1),
               dict(max_steps=100), dict(kernel=L.KERNEL_TC), dict(kernel=L.KERNEL_UTTERANCE)]
    for fields in refused:
        o = L.GenOpts(mu_law=1)
        for k, v in fields.items():
            setattr(o, k, v)
        assert gen(ctx, mel, 1, 21, None, ctypes.byref(o), 275, wp, pp, None, None, None) == EINVAL, fields
    assert p[0] == 0                                    # nothing was written


def test_generate_stream_without_a_device_is_ecuda():
    import torch
    if torch.cuda.is_available():
        return
    lib, L = _lib()
    fake = ctypes.create_string_buffer(4096)
    w, wp = _buf(20 * 275, np.float64)
    p, pp = _buf(1, np.int64)
    p[0] = 7
    rc = lib.b200tts_wavernn_generate_stream(ctypes.cast(fake, ctypes.c_void_p), ctypes.c_void_p(16), 1, 21, None, None, 275, wp, pp,
                                             None, None, None)
    assert rc == ECUDA and lib.b200tts_last_error()
    assert p[0] == 7                                    # refused before it touched the progress word


def test_stream_wait():
    lib, L = _lib()
    wait = lib.b200tts_wavernn_stream_wait
    p, pp = _buf(1, np.int64)
    out = ctypes.c_int64()
    assert wait(None, 1, 10, ctypes.byref(out)) == EINVAL
    assert wait(pp, 1, 10, None) == EINVAL
    assert wait(pp, 1, -1, ctypes.byref(out)) == EINVAL
    p[0] = 550                                          # already at the target: returns at once
    t0 = time.perf_counter()
    assert wait(pp, 550, 10_000, ctypes.byref(out)) == 0 and out.value == 550
    assert time.perf_counter() - t0 < 1.0
    p[0] = -1                                           # the kernel gave up: returns at once with the negative value
    t0 = time.perf_counter()
    assert wait(pp, 10 ** 9, 10_000, ctypes.byref(out)) == 0 and out.value == -1
    assert time.perf_counter() - t0 < 1.0
    p[0] = 275                                          # timeout: the last value seen
    t0 = time.perf_counter()
    assert wait(pp, 550, 200, ctypes.byref(out)) == 0 and out.value == 275
    assert 0.15 < time.perf_counter() - t0 < 5.0


def test_stream_wait_wakes_when_another_thread_raises_the_word():
    lib, L = _lib()
    p, pp = _buf(1, np.int64)
    out = ctypes.c_int64()

    def raise_it():
        time.sleep(0.2)
        p[0] = 825

    th = threading.Thread(target=raise_it)
    t0 = time.perf_counter()
    th.start()                                          # (ctypes releases the GIL for the duration of the wait)
    assert lib.b200tts_wavernn_stream_wait(pp, 800, 10_000, ctypes.byref(out)) == 0
    dt = time.perf_counter() - t0
    th.join()
    assert out.value == 825 and 0.15 < dt < 5.0
