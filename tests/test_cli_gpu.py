"""The two drop-in command lines, run as a user would (subprocess), on the GPU box with the travel copies of the shipped
checkpoints: tacotron_synthesize.py writes the .npy that wavernn_gen.py --file consumes (reference flow, SURVEY 3.3)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, REF_CKPT_COPY, ROOT
from taco_common import TRAVEL_COPY, sentences

pytestmark = pytest.mark.gpu


def _run(args, cwd):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get('PYTHONPATH', ''))
    return subprocess.run([sys.executable] + args, cwd=cwd, env=env, capture_output=True, text=True, timeout=600)


def test_tacotron_synthesize_then_wavernn_gen(tmp_path):
    wav_ckpt = REF_CKPT_COPY
    if not (os.path.isfile(TRAVEL_COPY) and os.path.isfile(wav_ckpt)):
        pytest.skip('shipped checkpoints not available on this box')
    s = sentences()
    text = '宝马配挂跛骡鞍，貂蝉怨枕董翁榻。'                       # train.txt line 3 as HANZI: the CLI runs it through get_pyin (:187)
    from tacotronv2_wavernn_chinese_b200.tacotron.pinyin import get_pyin
    assert get_pyin(text)[0] == ' '.join(s['symbols'][i] for i in s['sentences']['3']['ids'][:-1])
    r = _run([os.path.join(ROOT, 'tacotron_synthesize.py'), '--text', text, '--checkpoint', TRAVEL_COPY,
              '--symbols_json', os.path.join(GOLDEN, 'taco_symbols.json'), '--seed', '5'], str(tmp_path))
    assert r.returncode == 0, r.stdout + r.stderr
    out_dir = tmp_path / 'tacotron_inference_output'
    mels = [f for f in os.listdir(out_dir) if f.endswith('-mel-pred.npy')]
    assert len(mels) == 1 and mels[0].startswith('step-206500-')
    mel = np.load(out_dir / mels[0])
    gt = s['sentences']['3']['frames']
    assert mel.dtype == np.float32 and mel.shape[1] == 80 and abs(mel.shape[0] - gt) < 0.3 * gt and 0 <= mel.min() and mel.max() <= 1
    # vocode it with the drop-in wavernn_gen.py (same flags as the reference), unbatched then --batched
    for extra, tag in (([], 'gen_NOT_BATCHED'), (['--batched', '-t', '5500', '-o', '550'], 'gen_batched_target5500_overlap550')):
        r = _run([os.path.join(ROOT, 'wavernn_gen.py'), '--file', str(out_dir / mels[0]), '--voc_weights', wav_ckpt,
                  '--hp_file', os.path.join(ROOT, 'wavernn_hparams.py'), '--seed', '3'] + extra, str(tmp_path))
        assert r.returncode == 0, r.stdout + r.stderr
        name = mels[0].split('.')[0] + f'_{tag}_step=617k.wav'
        path = tmp_path / 'wavernn_inference_output' / name
        assert path.is_file(), os.listdir(tmp_path / 'wavernn_inference_output')
        from scipy.io import wavfile
        sr, y = wavfile.read(path)
        assert sr == 22050 and y.dtype == np.float32 and y.shape == ((mel.shape[0] - 1) * 275,) and np.abs(y).max() <= 1.0
        assert y.std() > 1e-3            # it is audio, not silence


def test_wavernn_gen_rejects_bad_input(tmp_path):
    np.save(tmp_path / 'bad.npy', np.full((30, 80), 2.0, np.float32))
    r = _run([os.path.join(ROOT, 'wavernn_gen.py'), '--file', str(tmp_path / 'bad.npy'), '--voc_weights', 'nonexistent.pyt',
              '--hp_file', os.path.join(ROOT, 'wavernn_hparams.py')], str(tmp_path))
    assert r.returncode != 0
