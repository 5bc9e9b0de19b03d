"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every declared symbol,
the hparams singleton / dsp / paths mirrors behave like the reference's, the CLI validates its input.
No GPU compute is invoked here."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np

from tacotronv2_wavernn_chinese_b200 import synth as synth_mod
import pytest

from conftest import ROOT
from oracle import wavernn_oracle as wo


def _lib():
    from tacotronv2_wavernn_chinese_b200 import build, _lib
    build.build_lib()
    return _lib.load(), _lib


def test_library_exports_every_declared_symbol():
    lib, L = _lib()
    header = open(os.path.join(ROOT, 'include', 'b200tts.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    declared = set(re.findall(r'\b(b200tts_\w+)\s*\(', header))
    assert declared, 'no prototypes parsed from include/b200tts.h'
    for name in sorted(declared):
        assert hasattr(lib, name), f'{name} declared in b200tts.h but not exported'
    assert declared == set(L.SIGNATURES), declared ^ set(L.SIGNATURES)
    assert lib.b200tts_abi_version() == 3


def test_library_is_sm100a_and_has_no_cpu_path():
    lib, L = _lib()
    out = subprocess.run(['cuobjdump', '--list-elf', L.lib_path()], capture_output=True, text=True).stdout
    assert 'sm_100a' in out, out
    import torch
    if not torch.cuda.is_available():
        # without a device every compute entry point must fail loudly, never fall back
        assert lib.b200tts_device_count() <= 0
        from tacotronv2_wavernn_chinese_b200 import synth
        from tacotronv2_wavernn_chinese_b200.engine import WaveRNNEngine
        with pytest.raises(RuntimeError):
            WaveRNNEngine(synth.synth_state_dict(0), synth.DEFAULT_DIMS)


def test_struct_layouts_match_header():
    _, L = _lib()
    assert ctypes.sizeof(L.WaveRNNCfg) == 14 * 4
    assert ctypes.sizeof(L.Tensor) == 8 + 8 + 8 + 32
    assert ctypes.sizeof(L.Rng) == 40          # ABI 2: + d_utterance_ids
    assert ctypes.sizeof(L.GenOpts) == 80          # ABI 3: + packed-row schedule


def test_hparams_singleton_contract(tmp_path):
    code = f'''
import sys
sys.path.insert(0, {ROOT!r})
from tacotronv2_wavernn_chinese_b200.wavernn.utils import hparams as hp
try:
    hp.bits
    raise SystemExit("no AttributeError before configure")
except AttributeError:
    pass
try:
    hp.configure("/nonexistent/hp.py"); raise SystemExit("missing file accepted")
except FileNotFoundError:
    pass
try:
    hp.configure({str(tmp_path / "x.txt")!r}); raise SystemExit("non-.py accepted")
except ValueError:
    pass
hp.configure({os.path.join(ROOT, "wavernn_hparams.py")!r})
assert (hp.bits, hp.hop_length, hp.voc_upsample_factors, hp.voc_rnn_dims, hp.voc_pad, hp.voc_mode) == (10, 275, (5, 5, 11), 512, 2, "RAW")
assert (hp.sample_rate, hp.num_mels, hp.voc_target, hp.voc_overlap, hp.mu_law) == (22050, 80, 11000, 550, True)
try:
    hp.configure({os.path.join(ROOT, "wavernn_hparams.py")!r}); raise SystemExit("reconfigure accepted")
except RuntimeError:
    pass
print("OK")
'''
    (tmp_path / 'x.txt').write_text('a = 1')
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert r.returncode == 0 and 'OK' in r.stdout, r.stdout + r.stderr


def test_hparams_file_matches_reference_values():
    """Every value of wavernn_hparams.py equals the reference's (tests/golden/wavernn_hparams_from_reference.json,
    oracle/make_golden_reference_files.py)."""
    from oracle.make_golden_reference_files import hparams_values
    ref = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'wavernn_hparams_from_reference.json')))
    assert hparams_values(os.path.join(ROOT, 'wavernn_hparams.py')) == ref


def test_dsp_mirror_matches_oracle():
    from tacotronv2_wavernn_chinese_b200.wavernn.utils import dsp
    y = np.linspace(-1, 1, 1024)
    np.testing.assert_array_equal(dsp.decode_mu_law(y, 1024, from_labels=False), wo.decode_mu_law(y, 1024))
    lab = np.arange(1024)
    np.testing.assert_allclose(dsp.decode_mu_law(lab, 1024), wo.decode_mu_law(dsp.label_2_float(lab, 10), 1024))
    x = np.linspace(-1, 1, 101)
    enc = dsp.encode_mu_law(x, 1024)
    assert enc.min() == 0 and enc.max() == 1023
    assert np.abs(dsp.decode_mu_law(enc, 1024) - x).max() < 0.01


def test_save_wav_float32(tmp_path):
    from scipy.io import wavfile
    from tacotronv2_wavernn_chinese_b200.wavernn.utils import dsp
    x = np.sin(np.arange(2205) / 10.0) * 0.5
    dsp.save_wav(x, tmp_path / 'a.wav', 22050)
    sr, y = wavfile.read(tmp_path / 'a.wav')
    assert sr == 22050 and y.dtype == np.float32
    np.testing.assert_array_equal(y, x.astype(np.float32))


def test_paths(tmp_path):
    from tacotronv2_wavernn_chinese_b200.wavernn.utils.paths import Paths
    p = Paths('wavernn', base=tmp_path)
    assert p.voc_latest_weights == tmp_path / 'logs_wavernn/checkpoints/latest_weights.pyt'
    assert p.voc_checkpoints.is_dir() and p.voc_output.is_dir()
    assert p.get_voc_named_weights('x').name == 'x_weights.pyt'


def test_model_keys_and_cpu_refusal():
    import torch
    from tacotronv2_wavernn_chinese_b200 import synth
    from tacotronv2_wavernn_chinese_b200.wavernn.models.fatchord_version import WaveRNN
    m = WaveRNN(512, 512, 10, 2, (5, 5, 11), 80, 128, 128, 10, 275, 22050)
    sd = synth.synth_state_dict(3)
    assert set(sd) == set(m.state_dict())
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == sd[k].shape, k
    with pytest.raises(ValueError):
        m.generate(torch.zeros(1, 80, 20), None, False, 11000, 550, True) if torch.cuda.is_available() else (_ for _ in ()).throw(ValueError())
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            m.generate(torch.zeros(1, 80, 30), None, False, 11000, 550, True)


def test_cli_rejects_bad_mel(tmp_path):
    import importlib
    sys.path.insert(0, ROOT)
    code = f'''
import sys, numpy as np
sys.path.insert(0, {ROOT!r})
import wavernn_gen as g
from tacotronv2_wavernn_chinese_b200.wavernn.utils import hparams as hp
hp.configure({os.path.join(ROOT, "wavernn_hparams.py")!r})
class M:
    def get_step(self): return 617000
    def generate(self, *a, **k): raise SystemExit("generate reached")
np.save({str(tmp_path / "bad_range.npy")!r}, np.full((30, 80), 1.5, np.float32))
np.save({str(tmp_path / "bad_shape.npy")!r}, np.zeros((30, 81), np.float32))
for f in ("bad_range.npy", "bad_shape.npy", "x.wav"):
    try:
        g.gen_from_file(M(), {str(tmp_path)!r} + "/" + f, {str(tmp_path)!r}, False, 11000, 550)
        raise SystemExit("accepted " + f)
    except ValueError:
        pass
print("OK")
'''
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert r.returncode == 0 and 'OK' in r.stdout, r.stdout + r.stderr


def test_fold_geometry_matches_reference_formula():
    """b200tts_wavernn_fold_geometry needs no GPU: (n_folds, fold_len) of fold_with_overlap (fatchord_version.py:319-330)."""
    lib, L = _lib()
    for T, target, overlap in [(80, 11000, 550), (30, 2750, 550), (30, 2700, 500), (402, 11000, 550), (21, 100, 20)]:
        S = T * 275
        nf = (S - overlap) // (target + overlap)
        if S - (nf * (target + overlap) + overlap) != 0:
            nf += 1
        a, b = ctypes.c_int(), ctypes.c_int()
        assert lib.b200tts_wavernn_fold_geometry(T, 275, target, overlap, ctypes.byref(a), ctypes.byref(b)) == 0
        assert (a.value, b.value) == (nf, target + 2 * overlap)
        x = np.zeros((1, S, 1), dtype=np.float32)
        assert wo.fold_with_overlap(x, target, overlap).shape[:2] == (nf, target + 2 * overlap)
    assert lib.b200tts_wavernn_fold_geometry(2, 275, 100, 600, ctypes.byref(a), ctypes.byref(b)) != 0     # shorter than the overlap
    assert b'overlap' in lib.b200tts_last_error()


def test_bench_cpu_arm_helpers():
    """bench.py's CPU arms (cpu_baseline / --impl reference): same config object as the GPU arm; a time-bounded sample of the
    UNMODIFIED reference's generate loop when its travel copy is present (kind "reference", source oracle/_ref), the numpy port beside it."""
    import argparse
    import bench
    args = argparse.Namespace(batch=4, frames=80)
    cfg = bench.workload_config(args, 2, 'test weights')
    assert cfg['utterances_per_gpu'] == 4 and cfg['global_batch'] == 8 and cfg['steps_per_utterance'] == 80 * 275
    assert cfg['workload'].startswith('BASELINE config 3')
    bench._PORT[('t', 4)] = 2                                # skip the thread probe in the test
    pr = bench.port_sample(4, 0.3)
    assert pr['value'] > 0 and pr['steps'] >= 10 and pr['threads'] == 2
    if bench.ref_model() is not None:                        # the reference's sources are present (oracle/_ref/reference_src.zip)
        import torch
        bench._REF[('threads', 4)] = 2
        r = bench.ref_sample(4, 0.3)
        assert r['value'] > 0 and r['steps'] >= 8 and r['threads'] == 2
        base = bench.cpu_baseline(4, 80, 0.3)
        assert base['kind'] == 'reference' and base['source'] == 'oracle/_ref' and 'UNMODIFIED reference' in base['sample'] and base['port']['kind'] == 'port'
        torch.set_num_threads(min(4, torch.get_num_threads()))


def test_reference_travel_copy_times_the_reference_loop():
    """oracle/ref_harness.timed_generate_sample drives the reference's OWN generate() (hooks only): step count, bounded
    sample, and the memoised conditioning network returning what the reference module computed."""
    from oracle import ref_harness as rh
    if not rh.available():
        pytest.skip('the reference sources are not present (oracle/_ref/reference_src.zip is made by __graft_entry__.build())')
    import torch
    m = rh.build_model()
    mel = torch.as_tensor(synth_mod.synth_mels(3, 2, 21))
    full = rh.timed_generate_sample(m, mel, max_steps=40)
    assert full['steps'] == 40 and full['batch'] == 2 and full['loop_seconds'] > 0
    rh.memoize_upsample(m)
    a = rh.timed_generate_sample(m, mel, max_steps=8)
    b = rh.timed_generate_sample(m, mel, max_steps=8)
    assert a['steps'] == b['steps'] == 8 and b['upsample_seconds'] < max(0.05, 0.5 * full['upsample_seconds'])
    assert m.training                                         # generate() leaves the module in train() mode (:262)


def test_error_codes_and_messages_without_a_device():
    """Status-code contract of include/b200tts.h: 0 / negative B200TTS_E* + a thread-local message, nothing throws across the ABI.
    Argument checks come before any CUDA call, so they can be exercised on a box without a GPU."""
    lib, L = _lib()
    EINVAL, ECUDA = -1, -2
    h = ctypes.c_void_p()
    cfg = L.WaveRNNCfg()
    assert lib.b200tts_wavernn_create(ctypes.byref(h), 0, ctypes.byref(cfg), None, 0) == EINVAL        # null weights
    assert b'null argument' in lib.b200tts_last_error() and not h.value
    dims = dict(synth_mod.DEFAULT_DIMS)
    arr, keep = L.make_tensor_array({k: np.asarray(v, dtype=np.float32) for k, v in
                                     wo.as_params(synth_mod.synth_state_dict(0)).items() if np.asarray(v).dtype.kind == 'f'})
    from tacotronv2_wavernn_chinese_b200.engine import _cfg_from_dims
    bad = _cfg_from_dims(dict(dims, upsample_factors=(5, 5, 10)))                                     # prod != hop_length
    assert lib.b200tts_wavernn_create(ctypes.byref(h), 0, ctypes.byref(bad), arr, len(arr)) == EINVAL
    assert b'hop_length' in lib.b200tts_last_error()
    bad = _cfg_from_dims(dict(dims, bits=16))                                                         # labels are int16
    assert lib.b200tts_wavernn_create(ctypes.byref(h), 0, ctypes.byref(bad), arr, len(arr)) == EINVAL
    nf, fl = ctypes.c_int(), ctypes.c_int()
    assert lib.b200tts_wavernn_fold_geometry(80, 275, 11000, 1, ctypes.byref(nf), ctypes.byref(fl)) == EINVAL   # overlap < 2
    assert lib.b200tts_wavernn_fold_geometry(1, 275, 11000, 550, ctypes.byref(nf), ctypes.byref(fl)) == EINVAL  # shorter than the overlap
    assert lib.b200tts_wavernn_generate(None, None, 1, 21, None, None, None, None, None) == EINVAL
    assert lib.b200tts_wavernn_check(None) == EINVAL
    assert lib.b200tts_wavernn_launch_count(None) == -1 and lib.b200tts_wavernn_last_kernel(None) == 0
    lib.b200tts_wavernn_destroy(None)                                                                 # no-op, must not crash
    import torch
    if not torch.cuda.is_available():
        good = _cfg_from_dims(dims)
        rc = lib.b200tts_wavernn_create(ctypes.byref(h), 0, ctypes.byref(good), arr, len(arr))
        assert rc == ECUDA and lib.b200tts_last_error() and not h.value                               # no device: loud, no fallback
        v = ctypes.c_double()
        assert lib.b200tts_debug_fp32_peak(0, ctypes.byref(v)) == ECUDA
    del keep


def test_taco_error_codes_without_a_device():
    lib, L = _lib()
    h = ctypes.c_void_p()
    cfg = L.TacoCfg()
    assert lib.b200tts_taco_create(ctypes.byref(h), 0, ctypes.byref(cfg), None, 0) == -1 and not h.value
    assert lib.b200tts_last_error()
    lib.b200tts_taco_destroy(None)
    assert lib.b200tts_taco_decode(None, None, None, 1, 5, None, 10, 0, None, None, None, None, None) == -1
    assert lib.b200tts_taco_encode(None, None, None, 1, 5, None, None) == -1
    assert lib.b200tts_taco_postnet(None, None, None, 1, 10, None, None) == -1
