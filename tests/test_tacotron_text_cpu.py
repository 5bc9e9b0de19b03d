"""TF-free text front-end mirror (tacotron/utils/symbols.py + text.py of the reference) and the CLI plumbing."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from taco_common import sentences
from tacotronv2_wavernn_chinese_b200.tacotron.text import Symbols, build_symbols


def test_symbols_roundtrip_and_eos():
    s = sentences()
    sym = Symbols(s['symbols'])
    assert len(sym) == 191
    ids = s['sentences']['241']['ids']
    text = sym.sequence_to_text(ids[:-1])
    assert sym.text_to_sequence(text) == ids and ids[-1] == 1
    assert sym.text_to_sequence('zz_unknown ' + text) == ids          # unknown tokens are dropped like the reference


def test_build_symbols_matches_reference_scan(tmp_path):
    # the train.txt lines that introduce every symbol (oracle/make_golden_reference_files.py)
    assert build_symbols(os.path.join(GOLDEN, 'train_symbol_lines.txt')) == sentences()['symbols']
    p = tmp_path / 't.txt'
    p.write_text('a|b|1|2|x|b a1 c\na|b|1|2|y|a1 d\n', encoding='utf-8')
    assert build_symbols(str(p)) == ['_', '~', 'a1', 'b', 'c', 'd']


def test_tacotron_hparams_shim():
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location('tacotron_hparams', os.path.join(root, 'tacotron_hparams.py'))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    hp = m.hparams
    assert (hp.num_mels, hp.outputs_per_step, hp.max_iters, hp.decoder_lstm_units, hp.attention_dim) == (80, 1, 2000, 256, 128)
    assert (hp.tacotron_zoneout_rate, hp.tacotron_dropout_rate, hp.max_abs_value, hp.symmetric_mels) == (0.1, 0.5, 4.0, True)
    hp2 = hp.parse('max_iters=500,stop_at_any=False')
    assert hp2.max_iters == 500 and hp2.stop_at_any is False and hp.max_iters == 2000
    with pytest.raises(KeyError):
        hp.parse('no_such_key=1')
