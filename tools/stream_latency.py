"""Time to first audio and real-time margin of streaming WaveRNN generation on one GPU (DESIGN 3.7).

    python tools/stream_latency.py [--out profiles/r03_stream_latency.json] [--reps 3]

Shipped checkpoint (oracle/_ref travel copy; synthetic weights if absent, stated in the output), 402-frame mels (BASELINE
config 2 length, 5.0 s of audio) at 1, 8 and 32 rows, chunk_steps = 275 (one mel frame).  In one process:
  * time from the generate_stream call (first next()) to the first chunk;
  * every chunk's arrival against a playback clock started at the first chunk (22 050 samples/s): worst slack, underruns;
  * time to the first chunk of pipeline.synthesize_stream on the config-4 sentence (Tacotron included; needs the Tacotron
    travel copy);
  * the step kernel's time (CUDA events) of streaming against plain generate, alternated `--reps` times each, per lock-step;
  * the card's name, power limit and max SM clock, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import numpy as np
import torch

from tacotronv2_wavernn_chinese_b200 import synth
from tacotronv2_wavernn_chinese_b200.engine import WaveRNNEngine

SR, HOP, FRAMES, CHUNK = 22050, 275, 402, 275


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def stream_once(eng, mels, seed):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    arr = []
    for start, c in eng.generate_stream(mels, seed=seed, chunk_steps=CHUNK):
        arr.append((time.perf_counter() - t0, start, c.shape[1]))
    total = time.perf_counter() - t0
    first = arr[0][0]
    # playback starts with the first chunk; chunk k is needed when the player reaches its first sample
    slack = [start / SR - (t - first) for t, start, _ in arr[1:]]      # > 0: the chunk was there before playback needed it
    return dict(first_chunk_ms=first * 1e3, first_chunk_samples=arr[0][2], call_s=total, chunks=len(arr),
                audio_s=(arr[-1][1] + arr[-1][2]) / SR, worst_slack_ms=min(slack) * 1e3, underruns=sum(s < 0 for s in slack),
                kernel_ms=eng.last_kernel_ms())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r03_stream_latency.json'))
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    torch.cuda.set_device(0)
    from conftest import load_ckpt_state_dict
    sd = load_ckpt_state_dict()
    weights = 'shipped checkpoint (oracle/_ref/latest_weights.pyt)' if sd is not None else 'synthetic (synth_state_dict(0))'
    eng = WaveRNNEngine(sd if sd is not None else synth.synth_state_dict(0), synth.DEFAULT_DIMS, device=0)
    out = dict(card=card(), weights=weights, frames=FRAMES, chunk_steps=CHUNK, sample_rate=SR, rows={})
    steps = FRAMES * HOP
    for B in (1, 8, 32):
        mels = synth.synth_mels(1235, B, FRAMES)
        eng.generate(mels, seed=1)                                      # warm-up of both paths
        list(eng.generate_stream(mels, seed=1, chunk_steps=CHUNK))
        plain, stream, runs = [], [], []
        for _ in range(a.reps):                                         # alternated: plain, streaming, plain, streaming, ...
            eng.generate(mels, seed=1)
            plain.append(eng.last_kernel_ms() * 1e3 / steps)
            r = stream_once(eng, mels, seed=1)
            stream.append(r['kernel_ms'] * 1e3 / steps)
            runs.append(r)
        best = min(runs, key=lambda r: r['first_chunk_ms'])
        row = dict(first_chunk_ms=[r['first_chunk_ms'] for r in runs], worst_slack_ms=[r['worst_slack_ms'] for r in runs],
                   underruns=[r['underruns'] for r in runs], call_s=[r['call_s'] for r in runs], chunks=best['chunks'],
                   audio_s=best['audio_s'], step_us_plain=plain, step_us_stream=stream,
                   stream_over_plain=float(np.median(stream) / np.median(plain)))
        out['rows'][str(B)] = row
        print(B, json.dumps(row), flush=True)
    from taco_common import real_taco_weights, sentences
    w = real_taco_weights()
    if w is None:
        out['synthesize_stream'] = 'not measured: Tacotron travel copy (oracle/_ref/tacotron_weights.npz) absent'
    else:
        from tacotronv2_wavernn_chinese_b200.pipeline import synthesize_stream
        from tacotronv2_wavernn_chinese_b200.tacotron.engine import TacoDecoderEngine
        from tacotronv2_wavernn_chinese_b200.tacotron.synthesizer import Synthesizer
        from tacotronv2_wavernn_chinese_b200.tacotron.text import Symbols
        s = sentences()
        syn = Synthesizer()
        syn.symbols = Symbols(s['symbols'])
        syn.engine = TacoDecoderEngine(w, device=0)
        syn.step = 206500
        text = syn.symbols.sequence_to_text(s['sentences']['241']['ids'][:-1])   # BASELINE config 4 sentence
        res = []
        for rep in range(a.reps + 1):                                   # first one is warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            g = synthesize_stream(syn, eng, text, seed=1238)
            start, c = next(g)
            first = time.perf_counter() - t0
            n = c.shape[0]
            for _, c in g:
                n += c.shape[0]
            if rep:
                res.append(dict(first_chunk_ms=first * 1e3, call_s=time.perf_counter() - t0, audio_s=n / SR))
        out['synthesize_stream'] = dict(sentence='241 (config 4)', seed=1238, runs=res)
        print('synthesize_stream', json.dumps(res), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print('wrote', a.out)


if __name__ == '__main__':
    main()
