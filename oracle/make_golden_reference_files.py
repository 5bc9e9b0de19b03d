"""Small data fixtures taken from files of the reference, so that the tests comparing with them need only the repository.

  tests/golden/wavernn_hparams_from_reference.json   every value the reference's wavernn_hparams.py defines
  tests/golden/train_symbol_lines.txt                the lines of train.txt that first introduce each symbol of its last
                                                      column (in file order): scanning them builds the same 191-entry table
                                                      as scanning the whole 2 MB file (tacotron/utils/symbols.py:12-28)
  tests/golden/taco_ckpt_checkpoint.txt              the `checkpoint` pointer file of logs-Tacotron-2/taco_pretrained/
  tests/golden/taco_ckpt.index                       its tensor-bundle index tacotron_model.ckpt-206500.index (10 KB)
  tests/golden/taco_ckpt_data_sample.npz             the size of the 62 MB data shard and the bytes of a few of its tensors
                                                      (global_step and small decoder biases) with their offsets: a sparse
                                                      stand-in for the shard holds exactly these bytes where the index says

    B200TTS_REFERENCE=<reference checkout> python oracle/make_golden_reference_files.py
"""
import json
import os
import shutil

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
REF = os.environ.get('B200TTS_REFERENCE', '/root/reference')
TACO_CKPT = 'logs-Tacotron-2/taco_pretrained'
TACO_SAMPLED = ['global_step'] + ['Tacotron_model/inference/decoder/' + k for k in (
    'Location_Sensitive_Attention/attention_bias', 'Location_Sensitive_Attention/attention_variable_projection',
    'Location_Sensitive_Attention/location_features_convolution/bias', 'dense/bias',
    'linear_transform_projection/projection_linear_transform_projection/bias',
    'stop_token_projection/projection_stop_token_projection/bias')]


def hparams_values(path):
    """Name -> repr() of each value a hparams file defines (repr keeps the type: a tuple does not equal a list)."""
    ns = {}
    exec(open(path).read(), ns)
    return {k: repr(v) for k, v in ns.items() if not k.startswith('__')}


def taco_ckpt_files():
    """Pointer file and index of the Tacotron checkpoint, and the sampled bytes of its data shard."""
    import sys
    sys.path.insert(0, ROOT)
    from tacotronv2_wavernn_chinese_b200.tacotron import ckpt
    d = os.path.join(REF, TACO_CKPT)
    prefix = ckpt.resolve_checkpoint(d)
    shutil.copyfile(os.path.join(d, 'checkpoint'), os.path.join(GOLDEN, 'taco_ckpt_checkpoint.txt'))
    shutil.copyfile(prefix + '.index', os.path.join(GOLDEN, 'taco_ckpt.index'))
    entries = ckpt.read_index(prefix + '.index')
    data = prefix + '.data-00000-of-00001'
    raw = np.memmap(data, dtype=np.uint8, mode='r')
    out = {'data_size': np.int64(os.path.getsize(data)), 'names': np.array(TACO_SAMPLED)}
    for i, n in enumerate(TACO_SAMPLED):
        e = entries[n]
        out[f'offset_{i}'] = np.int64(e['offset'])
        out[f'bytes_{i}'] = np.array(raw[e['offset']:e['offset'] + e['size']])
    np.savez_compressed(os.path.join(GOLDEN, 'taco_ckpt_data_sample.npz'), **out)


def main():
    hp = hparams_values(os.path.join(REF, 'wavernn_hparams.py'))
    json.dump(hp, open(os.path.join(GOLDEN, 'wavernn_hparams_from_reference.json'), 'w'), indent=1, sort_keys=True)
    seen, keep = set(), []
    with open(os.path.join(REF, 'train.txt'), encoding='utf-8') as f:
        for line in f:
            toks = set(line.strip().split('|')[-1].strip().split(' '))
            if toks - seen:
                keep.append(line if line.endswith('\n') else line + '\n')
                seen |= toks
    with open(os.path.join(GOLDEN, 'train_symbol_lines.txt'), 'w', encoding='utf-8') as f:
        f.writelines(keep)
    taco_ckpt_files()
    print(len(hp), 'hparams;', len(keep), 'train.txt lines cover', len(seen), 'symbols')


if __name__ == '__main__':
    main()
