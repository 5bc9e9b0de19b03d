"""Streaming WaveRNN generation (b200tts_wavernn_generate_stream / WaveRNNEngine.generate_stream / pipeline.synthesize_stream):
the chunks handed out while the push kernel runs are, concatenated, bit for bit the wave of a plain generate call."""
import ctypes
import time

import numpy as np
import pytest

from tacotronv2_wavernn_chinese_b200 import synth

pytestmark = pytest.mark.gpu

EINVAL = -1


@pytest.fixture(scope='module')
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.fail('GPU tests need a CUDA device (and there is no CPU fallback to hide behind)')
    from tacotronv2_wavernn_chinese_b200.engine import WaveRNNEngine
    return WaveRNNEngine(synth.synth_state_dict(0), synth.DEFAULT_DIMS)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _collect(eng, mels, **kw):
    dev = {}
    chunks = list(eng.generate_stream(mels, device_out=dev, **kw))
    starts = [s for s, _ in chunks]
    assert starts == sorted(starts) and starts[0] == 0
    pos = 0
    for s, c in chunks:
        assert s == pos and c.dtype == np.float64 and c.shape[0] == mels.shape[0] and c.shape[1] > 0
        pos += c.shape[1]
    return np.concatenate([c for _, c in chunks], axis=1), dev, chunks


CASES = [   # rows, frames, chunk_steps, extra generate() arguments
    (1, 24, 275, {}),                                                               # <8>
    (5, 22, 1, {}),                                                                 # <8>, a publish every lock-step
    (12, 23, 1000, dict(seed=9)),                                                   # <16>, chunk that does not divide the length
    (32, 21, 275, dict(utterance_offset=40)),                                       # <32>
    (5, 24, 275, dict(utt_frames=[24, 21, 22, 24, 23])),                            # ragged rows shorter than the launch
    (4, 22, 333, dict(utterance_ids=[7, 3, 100, 42])),                              # non-consecutive noise keys
    (2, 21, 275, dict(mu_law=False)),
    (3, 25, 500, dict(utt_frames=[25, 21, 23], utterance_ids=[5, 1, 9], mu_law=False, seed=4)),
]


@pytest.mark.parametrize('B,T,chunk,kw', CASES, ids=[f'B{c[0]}_T{c[1]}_chunk{c[2]}_{"_".join(c[3]) or "plain"}' for c in CASES])
def test_stream_equals_generate_bit_for_bit(eng, B, T, chunk, kw):
    mels = synth.synth_mels(100 + B, B, T)
    ref = eng.generate(mels, **kw)
    want_wave = ref['wave'].cpu().numpy()
    want_labels = ref['labels'].cpu().numpy()
    got, dev, _ = _collect(eng, mels, chunk_steps=chunk, **kw)
    assert eng.last_kernel() == 'wavernn_push_kernel'
    assert got.shape == want_wave.shape == (B, (T - 1) * 275)
    assert np.array_equal(_bits(got), _bits(want_wave))
    assert np.array_equal(dev['labels'].cpu().numpy(), want_labels)
    # the device wave of the streaming call (finish_wave_kernel) equals what the kernel wrote to the host buffer
    assert np.array_equal(_bits(dev['wave'].cpu().numpy()), _bits(got))
    if 'utt_frames' in kw:
        for b, f in enumerate(kw['utt_frames']):
            assert not got[b, (f - 1) * 275:].any()


def test_stream_delivery_is_progressive(eng):
    """One 402-frame sentence (BASELINE config 2) at one row: chunks arrive while the kernel runs, the first within the first
    quarter of the call."""
    import torch
    mels = synth.synth_mels(1235, 1, 402)
    list(eng.generate_stream(mels, seed=1, chunk_steps=275))          # warm-up (module load, buffers)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    arrivals = []
    for start, c in eng.generate_stream(mels, seed=1, chunk_steps=275):
        arrivals.append((time.perf_counter() - t0, start, start + c.shape[1]))
    total = time.perf_counter() - t0
    ends = [e for _, _, e in arrivals]
    assert ends == sorted(set(ends)) and ends[-1] == 401 * 275
    assert len(arrivals) - 1 >= 10, arrivals                          # intermediate progress values seen
    assert arrivals[0][0] < 0.25 * total, (arrivals[0], total)


def test_abandoned_stream_waits_for_its_launch(eng):
    """A consumer that stops after the first chunk: closing the generator waits for the launch, and the context is usable."""
    mels = synth.synth_mels(5, 2, 30)
    g = eng.generate_stream(mels, seed=2, chunk_steps=275)
    s, c = next(g)
    assert s == 0 and c.shape[0] == 2
    g.close()
    ref = eng.generate(mels, seed=2)['wave'].cpu().numpy()
    got, _, _ = _collect(eng, mels, seed=2)
    assert np.array_equal(_bits(got), _bits(ref))


def _raw_stream(eng, mels, opts=None, h_wave=None, h_prog=None, B=None, T=None):
    import torch
    from tacotronv2_wavernn_chinese_b200 import _lib
    m = torch.as_tensor(mels).cuda().contiguous()
    B = m.shape[0] if B is None else B
    T = m.shape[2] if T is None else T
    rng = _lib.Rng(mode=_lib.RNG_PHILOX, seed=1)
    o = opts if opts is not None else _lib.GenOpts(mu_law=1)
    hw = torch.empty(m.shape[0], (m.shape[2] - 1) * 275, dtype=torch.float64, pin_memory=True) if h_wave is None else h_wave
    hp = torch.zeros(1, dtype=torch.int64, pin_memory=True) if h_prog is None else h_prog
    ptr = lambda x: ctypes.c_void_p(x.data_ptr() if hasattr(x, 'data_ptr') else x.ctypes.data)
    rc = eng.lib.b200tts_wavernn_generate_stream(eng._h, ptr(m), B, T, ctypes.byref(rng), ctypes.byref(o), 275, ptr(hw), ptr(hp),
                                                 None, None, None)
    torch.cuda.synchronize()
    return rc, eng.lib.b200tts_last_error()


def test_stream_refusals(eng):
    import torch
    from tacotronv2_wavernn_chinese_b200 import _lib
    mels = synth.synth_mels(3, 2, 22)
    before = eng.generate(mels, seed=1)
    G = _lib.GenOpts
    pk_u = torch.zeros(1, 1, dtype=torch.int32, device='cuda')
    pk_s = torch.tensor([[0, 22 * 275]], dtype=torch.int32, device='cuda')
    for o, what in [(G(mu_law=1, fold_target=2750, fold_overlap=550), b'fold'),
                    (G(mu_law=1, d_pack_utt=pk_u.data_ptr(), d_pack_start=pk_s.data_ptr(), pack_rows=1, pack_segs=1, pack_steps=22 * 275), b'packed'),
                    (G(mu_law=1, kernel=_lib.KERNEL_TC), b'push kernel'),
                    (G(mu_law=1, kernel=_lib.KERNEL_UTTERANCE), b'push kernel'),
                    (G(mu_law=1, max_steps=1000), b'max_steps')]:
        rc, msg = _raw_stream(eng, mels, opts=o)
        assert rc == EINVAL and what in msg, (what, msg)
    rc, msg = _raw_stream(eng, synth.synth_mels(3, 33, 22))
    assert rc == EINVAL and b'1..32 rows' in msg
    # pageable host memory cannot be written by a running kernel
    rc, msg = _raw_stream(eng, mels, h_wave=np.zeros((2, 21 * 275)))
    assert rc == EINVAL and b'PINNED' in msg and b'h_wave' in msg
    rc, msg = _raw_stream(eng, mels, h_prog=np.zeros(1, dtype=np.int64))
    assert rc == EINVAL and b'PINNED' in msg and b'h_progress' in msg
    with pytest.raises(ValueError):
        next(eng.generate_stream(mels, chunk_steps=0))
    # a plain generate on the same context after streaming calls gives its usual result
    list(eng.generate_stream(mels, seed=1))
    after = eng.generate(mels, seed=1)
    assert np.array_equal(after['labels'].cpu().numpy(), before['labels'].cpu().numpy())
    assert np.array_equal(_bits(after['wave'].cpu().numpy()), _bits(before['wave'].cpu().numpy()))
    eng.check()


def test_synthesize_stream_equals_synthesize_batch():
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from taco_common import real_taco_weights, sentences
    w = real_taco_weights()
    if w is None:
        pytest.skip('shipped Tacotron checkpoint not available on this box')
    from tacotronv2_wavernn_chinese_b200.engine import WaveRNNEngine
    from tacotronv2_wavernn_chinese_b200.pipeline import synthesize_batch, synthesize_stream
    from tacotronv2_wavernn_chinese_b200.tacotron.engine import TacoDecoderEngine
    from tacotronv2_wavernn_chinese_b200.tacotron.synthesizer import Synthesizer
    from tacotronv2_wavernn_chinese_b200.tacotron.text import Symbols
    s = sentences()
    syn = Synthesizer()
    syn.symbols = Symbols(s['symbols'])
    syn.engine = TacoDecoderEngine(w)
    syn.step = 206500
    text = syn.symbols.sequence_to_text(s['sentences']['241']['ids'][:-1])
    voc = WaveRNNEngine(synth.synth_state_dict(0), synth.DEFAULT_DIMS)
    want = synthesize_batch(syn, voc, [text], seed=3, utterance_offset=2)[0][0]
    parts = list(synthesize_stream(syn, voc, text, seed=3, utterance_offset=2))
    got = np.concatenate([c for _, c in parts])
    assert len(parts) > 1 and parts[0][0] == 0
    assert got.shape == want.shape and np.array_equal(_bits(got), _bits(want))
