"""CPU checks of the Tacotron side: TF-bundle reader, and whole-sentence behaviour of the oracle (its per-step arithmetic is pinned in test_tacotron_*_pins.py)."""
import os

import numpy as np
import pytest

from oracle import tacotron_oracle as to
from conftest import GOLDEN
from taco_common import SHAPES, real_taco_weights, sentences, synth_taco_weights


def _checkpoint_dir(d):
    """The shipped checkpoint directory rebuilt from tests/golden/ (oracle/make_golden_reference_files.py): the real `checkpoint`
    pointer file and .index, and a sparse stand-in for the 62 MB data shard that holds the sampled tensors' bytes where the
    index places them (zeros elsewhere).  -> {name: raw bytes} of the sampled tensors."""
    import shutil
    prefix = d / 'tacotron_model.ckpt-206500'
    shutil.copyfile(os.path.join(GOLDEN, 'taco_ckpt_checkpoint.txt'), d / 'checkpoint')
    shutil.copyfile(os.path.join(GOLDEN, 'taco_ckpt.index'), str(prefix) + '.index')
    z = np.load(os.path.join(GOLDEN, 'taco_ckpt_data_sample.npz'))
    sampled = {}
    with open(str(prefix) + '.data-00000-of-00001', 'wb') as f:
        f.truncate(int(z['data_size']))
        for i, name in enumerate(z['names']):
            f.seek(int(z[f'offset_{i}']))
            f.write(z[f'bytes_{i}'].tobytes())
            sampled[str(name)] = z[f'bytes_{i}'].tobytes()
    return sampled


def test_bundle_reader_shapes_and_step(tmp_path):
    from tacotronv2_wavernn_chinese_b200.tacotron import ckpt
    sampled = _checkpoint_dir(tmp_path)
    w = ckpt.load_tacotron_weights(str(tmp_path))          # resolves the TF `checkpoint` pointer file, skips Adam slots
    assert int(w['global_step']) == 206500
    for k, shp in SHAPES.items():
        assert w[k].shape == shp and w[k].dtype == np.float32, k
    assert not any(k.endswith('/Adam') or k.endswith('/Adam_1') for k in w)
    n = sum(v.size for k, v in w.items() if k != 'global_step')
    assert n == 5166370
    idx = ckpt.read_index(ckpt.resolve_checkpoint(str(tmp_path)) + '.index')
    assert idx['Tacotron_model/inference/inputs_embedding']['shape'] == (191, 128)
    for name, raw in sampled.items():                      # the bytes come back from where the index says they are
        key = name[len(ckpt.PREFIX):] if name.startswith(ckpt.PREFIX) else name
        assert w[key].tobytes() == raw, name


def test_symbol_table_pin():
    s = sentences()
    assert len(s['symbols']) == 191 and s['symbols'][:2] == ['_', '~']
    assert s['symbols'][2:] == sorted(s['symbols'][2:])
    assert all(len(s['sentences'][k]['ids']) == 51 for k in ('241', '378', '407'))      # the 50-token sentences of config 4
    assert len(s['sentences']) == 67 and all(v['ids'][-1] == 1 and min(v['ids']) >= 1 for v in s['sentences'].values())


def test_oracle_aligns_and_stops_on_a_training_sentence():
    """Weak pin of the restated semantics (gate order, forget bias, BN eps, attention recursion): on train.txt line 241
    (444 ground-truth frames) the decoder must walk the 51 tokens monotonically and stop in the right neighbourhood."""
    w = real_taco_weights()
    if w is None:
        pytest.skip('shipped Tacotron checkpoint not available')
    ids = sentences()['sentences']['241']['ids']
    mem = to.encoder(w, ids)
    assert mem.shape == (51, 512) and np.abs(mem).max() <= 1.0
    d = to.decode(w, mem, seed=1238, max_iters=800)
    n = d['n_steps']
    assert 300 <= n <= 600, n
    path = d['alignments'].argmax(1)
    assert path[0] <= 2 and path[-1] >= 48 and (np.diff(path) >= -1).all()
    assert d['stop'][-1] > 0.5 and (d['stop'][:-1] <= 0.5).all()
    np.testing.assert_allclose(d['alignments'].sum(1), 1.0, atol=1e-5)
    mel = to.postnet(w, d['frames'])
    assert mel.shape == (n, 80) and mel.min() >= -4.1 - 1e-6 and mel.max() <= 4.0 + 1e-6
    out, info = to.synthesize(w, ids, seed=1238, max_iters=800)
    assert out.shape == (n - 1, 80) and 0.0 <= out.min() and out.max() <= 1.0      # cut before the stop frame (:104-107)


def test_oracle_window_mode_runs():
    w = synth_taco_weights(3)
    mem = np.random.RandomState(1).uniform(-1, 1, (23, 512)).astype(np.float32)
    d = to.decode(w, mem, seed=5, max_iters=40, window=True)
    np.testing.assert_allclose(d['alignments'].sum(1), 1.0, atol=1e-5)
    assert (d['alignments'] > 0).sum(1).max() <= 5        # at most the 5-wide window [max-2, max+3) survives


def test_real_checkpoint_decoder_is_chaotic():
    """Why the GPU parity test uses a horizon: the SAME oracle evaluated in float32 and in float64 on the shipped checkpoint
    agrees to ~2e-5 for the first ~80 decoder steps (3.5e-4 by step 120) and then diverges to O(1) (LSTM kernel entries reach 30); no two
    fp32 implementations with different summation orders can match over a whole utterance."""
    w = real_taco_weights()
    if w is None:
        pytest.skip('shipped Tacotron checkpoint not available')
    ids = sentences()['sentences']['241']['ids']
    mem = to.encoder(w, ids)
    masks = (np.random.RandomState(1238).uniform(size=(700, 2, 256)) >= 0.5).astype(np.uint8)
    r32 = to.decode(w, mem, dropout_masks=masks, max_iters=700)
    old = to.F32
    try:
        to.F32 = np.float64
        r64 = to.decode({k: v.astype(np.float64) for k, v in w.items()}, mem.astype(np.float64), dropout_masks=masks,
                        max_iters=700)
    finally:
        to.F32 = old
    n = min(r32['n_steps'], r64['n_steps'])
    err = np.abs(r32['frames'][:n] - r64['frames'][:n]).max(1)
    assert err[:80].max() < 5e-5             # agreement over the horizon the GPU test asserts (measured 1.8e-5)
    assert err[min(n - 1, 300):].max() > 1e-2  # ... and genuine divergence afterwards
