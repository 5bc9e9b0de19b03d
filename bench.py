#!/usr/bin/env python
"""Benchmark of the WaveRNN generation hot path (BASELINE.json metric: audio samples/sec, batched utterances).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...       # the UNMODIFIED reference's generate() on the host cores
    python bench.py ... --dump-outputs DIR     # also write the last timed step's outputs as DIR/*.npy (compare two builds)

One "step" = one full pass of the hot path (conditioning network + all T*hop autoregressive sample steps + mu-law
decode/fade) over this rank's batch of synthetic 80-frame mels, on the SHIPPED checkpoint when its travel copy is present
(oracle/_ref/latest_weights.pyt, made by __graft_entry__.build()), else on random-init weights of the same architecture.

Headline line (`value`, `scaling: weak`): BASELINE config 3 with 256 utterances PER GPU -- utterances are sharded with no
data-path collective and for N > 1 every timed step ends with the NCCL all-gather of the int16 labels.  BASELINE config 3 AS
WRITTEN is a 256-utterance GLOBAL batch over 8 GPUs: that is the `strong` object of the same JSON line (256/N per GPU,
measured in the same run with the same timing rules).

Prints ONE JSON line (rank 0).  `value` is measured with inputs resident in HBM; `e2e` goes through the C-ABI host entry
point (b200tts_wavernn_generate_host: pinned H2D of the mels, generation, D2H of labels + float64 wave).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HOP, FEAT, NCLS = 275, 80, 1024
STEP_WEIGHT_BYTES = 17_371_136          # all per-step weights + biases, fp32, touched once per lock-step (SURVEY 8d)
COND_BYTES_PER_UTT = 836                # 80 mel + 128 aux fp32 in, 4 B out, per utterance-sample
FLOP_PER_SAMPLE = 8_668_160             # 2 * 4 334 080 MAC per utterance-sample
CKPT_TRAVEL = os.path.join(ROOT, 'oracle', '_ref', 'latest_weights.pyt')
DUMP_BUDGET = 64_000_000                # bytes --dump-outputs may write in all


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', choices=('b200', 'reference'), default='b200')
    ap.add_argument('--batch', type=int, default=256, help='utterances per GPU (weak line) = global batch of the strong line')
    ap.add_argument('--frames', type=int, default=80)
    ap.add_argument('--kernel', default='auto', choices=('auto', 'grid', 'utterance', 'tc'))
    ap.add_argument('--weights', default='auto', choices=('auto', 'shipped', 'synthetic'))
    ap.add_argument('--workload', default='config3', choices=('config3', 'text2audio', 'tacotron'),
                    help='config3 (default, the BASELINE metric) | text2audio: BASELINE config 5, 64 sentences text->mel->audio sharded '
                         'over the GPUs | tacotron: BASELINE config 4, the decoder loop on the 50-token sentence')
    ap.add_argument('--no-strong', action='store_true', help='skip the strong-scaling (global batch) measurement')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 or float64, '
                         'at most 64 MB in all: larger outputs keep a fixed, seeded sample of their rows, listed in <name>_rows.npy)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs: the reference arm only times bounded samples of its loop')
    return args


def dump_outputs(path, arrays):
    """Writes each array as path/<name>.npy: float64 stays float64, every other dtype becomes float32 (exact for the int16
    labels).  When they would exceed DUMP_BUDGET bytes together, each keeps the same fraction of its rows (axis 0), chosen
    with a fixed seed and recorded in <name>_rows.npy, so that the same arguments always dump the same elements."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v.cpu() if hasattr(v, 'cpu') else v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    need = sum(v.nbytes + 8 * len(v) + 256 for v in arrays.values())          # + row indices and .npy headers
    frac = min(1.0, DUMP_BUDGET / need)
    for name, v in arrays.items():
        if frac < 1.0:
            rows = np.sort(np.random.RandomState(0).choice(len(v), int(len(v) * frac), replace=False))
            v = v[rows]
            np.save(os.path.join(path, name + '_rows.npy'), rows.astype(np.float64))
        np.save(os.path.join(path, name + '.npy'), v)


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self._stop_evt, self.max_mhz = index, [], set(), threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
                 getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
                 getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
                 getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap'}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ------------------------------------------------------------------------------------------------
# weights: the drop-in checkpoint when it is on the box
# ------------------------------------------------------------------------------------------------
def load_weights(which):
    from tacotronv2_wavernn_chinese_b200 import synth
    if which in ('auto', 'shipped'):
        if os.path.isfile(CKPT_TRAVEL):
            import torch
            sd = torch.load(CKPT_TRAVEL, map_location='cpu', weights_only=True)
            return {k: v.numpy() for k, v in sd.items()}, 'shipped checkpoint latest_weights.pyt (step 617k)'
        if which == 'shipped':
            raise SystemExit('--weights shipped: no travel copy of the checkpoint (run __graft_entry__.build() in the container)')
    return synth.synth_state_dict(0), 'random-init weights of the shipped architecture (synth.synth_state_dict(0))'


# ------------------------------------------------------------------------------------------------
# CPU arms.  kind "reference" (source oracle/_ref): the UNMODIFIED reference WaveRNN.generate (fatchord_version.py:169), imported from the git-ignored
# travel copy oracle/_ref/reference_src.zip through oracle/ref_harness.py, shipped checkpoint, torch CPU.
# kind "port": the numpy oracle port (oracle/wavernn_oracle.py), kept beside it for continuity with round 1.
# ------------------------------------------------------------------------------------------------
_REF = {}


def ref_model():
    if 'model' not in _REF:
        from oracle import ref_harness as rh
        if not rh.available():
            _REF['model'] = None
        else:
            m = rh.build_model()
            rh.memoize_upsample(m)
            _REF['model'], _REF['rh'] = m, rh
    return _REF['model']


def ref_pick_threads(batch, mels):
    """"All the host threads it can USE": probe a few torch intra-op pool sizes on the actual batch, keep the fastest."""
    import torch
    key = ('threads', batch)
    if key in _REF:
        return _REF[key]
    rh, m = _REF['rh'], _REF['model']
    ncpu = os.cpu_count() or 1
    best, best_rate = 1, 0.0
    rh.timed_generate_sample(m, mels, max_steps=4)                         # conditioning network once (memoised afterwards)
    for nt in sorted({1, 8, 16, 32, 64, ncpu} & set(range(1, ncpu + 1))):
        torch.set_num_threads(nt)
        r = rh.timed_generate_sample(m, mels, max_seconds=1.0 if batch > 1 else 0.5)
        rate = r['steps'] / r['loop_seconds']
        if rate > best_rate:
            best, best_rate = nt, rate
    torch.set_num_threads(best)
    _REF[key] = best
    return best


def ref_sample(batch, max_seconds):
    """One bounded sample of the reference's own sampling loop on `batch` utterances -> dict(value samples/s, steps, threads)."""
    import torch
    from tacotronv2_wavernn_chinese_b200 import synth
    m = ref_model()
    rh = _REF['rh']
    key = ('mels', batch)
    if key not in _REF:
        _REF[key] = torch.as_tensor(synth.synth_mels(1236, batch, 21))     # minimum length: per-step cost is length-independent
    mels = _REF[key]
    threads = ref_pick_threads(batch, mels)
    torch.set_num_threads(threads)
    r = rh.timed_generate_sample(m, mels, max_seconds=max_seconds)
    return dict(value=batch * r['steps'] / r['loop_seconds'], steps=r['steps'], threads=threads, seconds=r['loop_seconds'])


def ref_config1():
    """BASELINE config 1: what the reference's CLI does -- ONE 80-frame utterance, all 22 000 steps, conditioning included."""
    import torch
    from tacotronv2_wavernn_chinese_b200 import synth
    m = ref_model()
    rh = _REF['rh']
    mel = torch.as_tensor(synth.synth_mels(1234, 1, 80))
    threads = ref_pick_threads(1, torch.as_tensor(synth.synth_mels(1234, 1, 21)))
    torch.set_num_threads(threads)
    m.upsample._b200_memo.clear()
    t0 = time.perf_counter()
    r = rh.timed_generate_sample(m, mel)
    wall = time.perf_counter() - t0
    S = 80 * HOP
    return dict(samples_per_s=S / wall, rtf=wall / ((79 * HOP) / 22050.0), seconds=wall, loop_seconds=r['loop_seconds'],
                conditioning_seconds=r['upsample_seconds'], steps=r['steps'], threads=threads,
                what='unmodified reference WaveRNN.generate(mel[1,80,80], batched=False), shipped checkpoint, torch CPU')


_PORT = {}


def port_sample(batch, max_seconds):
    """The numpy oracle port on the same batch (sampling loop only), BLAS threads chosen by probe."""
    import contextlib
    from oracle import wavernn_oracle as wo
    from tacotronv2_wavernn_chinese_b200 import synth
    if batch not in _PORT:
        p = {k: (v.astype(np.float32) if v.dtype.kind == 'f' else v) for k, v in wo.as_params(synth.synth_state_dict(0)).items()}
        distinct = min(8, batch)
        mels = synth.synth_mels(1234, distinct, 21)
        mp = wo.pad_tensor(mels.transpose(0, 2, 1), wo._dims(p)['pad'], 'both').transpose(0, 2, 1)
        m_up, aux = wo.upsample(p, mp)
        reps = (batch + distinct - 1) // distinct
        tile = lambda a: np.ascontiguousarray(np.tile(a, (reps, 1, 1))[:batch])
        _PORT[batch] = (wo, p, tile(mels), (tile(m_up), tile(aux)))
    wo, p, mels, cond = _PORT[batch]
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        threadpool_limits = None
    ncpu = os.cpu_count() or 1
    if ('t', batch) not in _PORT:
        best, best_rate = ncpu, 0.0
        if threadpool_limits is not None:
            for nt in sorted({1, 8, 16, 32, ncpu} & set(range(1, ncpu + 1))):
                with threadpool_limits(limits=nt):
                    wo.generate(p, mels, max_steps=3, seed=0, cond=cond)
                    r = wo.generate(p, mels, max_steps=20 if batch > 1 else 100, seed=0, cond=cond)
                rate = r['steps'] / r['loop_seconds']
                if rate > best_rate:
                    best, best_rate = nt, rate
        _PORT[('t', batch)] = best
    threads = _PORT[('t', batch)]
    ctx = threadpool_limits(limits=threads) if threadpool_limits is not None else contextlib.nullcontext()
    with ctx:
        probe = wo.generate(p, mels, max_steps=10, seed=0, cond=cond)
        per_step = max(probe['loop_seconds'] / 10, 1e-6)
        steps = int(min(mels.shape[2] * HOP, max(10, max_seconds / per_step)))
        r = wo.generate(p, mels, max_steps=steps, seed=0, cond=cond)
    return dict(value=batch * steps / r['loop_seconds'], steps=steps, threads=threads)


def cpu_baseline(batch, frames, seconds):
    """cpu_baseline object of the b200 line / the reference arm: `_ref` when the travel copy is there, the port otherwise."""
    if ref_model() is not None:
        r = ref_sample(batch, seconds)
        out = {'value': r['value'], 'unit': 'samples/s', 'cores': r['threads'], 'kind': 'reference', 'source': 'oracle/_ref',
               'sample': f"{batch} utterances x {r['steps']} of {frames * HOP} lock-steps of the UNMODIFIED reference "
                         f"WaveRNN.generate loop (fatchord_version.py:201-241, shipped checkpoint, torch CPU, {r['threads']} intra-op "
                         f"threads picked by probe on a {os.cpu_count()}-thread host); the one-shot conditioning network is "
                         f"outside the timed region (21-frame mels: the per-step cost does not depend on the length)"}
        try:
            pr = port_sample(batch, min(seconds, 6.0))
            out['port'] = {'value': pr['value'], 'cores': pr['threads'], 'kind': 'port',
                           'sample': f"{batch} utterances x {pr['steps']} lock-steps, numpy oracle port, random-init weights"}
        except Exception as e:                                               # the port is a side note, never fatal
            out['port'] = {'error': str(e)[:200]}
        return out
    pr = port_sample(batch, seconds)
    return {'value': pr['value'], 'unit': 'samples/s', 'cores': pr['threads'], 'kind': 'port',
            'sample': f"{batch} utterances x {pr['steps']} of {frames * HOP} lock-steps, numpy oracle port of generate() "
                      f"(the reference's travel copy oracle/_ref/reference_src.zip is absent: run __graft_entry__.build() in the container)"}


def workload_config(args, N, wdesc):
    B, T = args.batch, args.frames
    return {'workload': f'BASELINE config 3: WaveRNN generate(), batch={B} utterances/GPU of {T}-frame synthetic mels '
                        f'(voc_mode=RAW bits=10 hop=275), {wdesc}',
            'utterances_per_gpu': B, 'global_batch': N * B, 'frames': T, 'steps_per_utterance': T * HOP}


def run_reference(args):
    """--impl reference: the reference's own generate() loop on the host cores, on the b200 arm's batch.  Each bench step
    is a time-bounded sample of the 22 000 lock-steps of the 256-utterance batch; BASELINE config 1 (what the reference's
    CLI does: one utterance, all steps) is measured once and reported beside it."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    have_ref = ref_model() is not None
    per_step_budget = max(1.5, min(8.0, 110.0 / max(1, args.steps + args.warmup)))
    rates, last = [], None
    for i in range(args.warmup + args.steps):
        last = ref_sample(args.batch, per_step_budget) if have_ref else port_sample(args.batch, per_step_budget)
        if i >= args.warmup:
            rates.append(last['value'])
    v = float(np.mean(rates))
    cfg = workload_config(args, 1, 'shipped checkpoint' if have_ref else 'random-init weights')
    cfg['parallelism'] = f"host CPU, {last['threads']} threads (rank 0 only)"
    base = cpu_baseline(args.batch, args.frames, 4.0)
    base['value'] = v
    line = {
        'impl': 'reference', 'metric': 'wavernn_audio_samples_per_sec', 'value': v, 'unit': 'samples/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * args.batch * last['steps'] / last['value'],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': cfg, 'cpu_baseline': base,
        'e2e': {'value': v, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0, 'rtf': 22050.0 / (v / args.batch), 'host_threads': os.cpu_count(),
    }
    if have_ref:
        try:
            line['config1_reference_cli'] = ref_config1()
        except Exception as e:
            line['config1_reference_cli'] = {'error': str(e)[:200]}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def _taco_setup(local):
    """Synthesizer on the shipped Tacotron checkpoint (travel copy oracle/_ref/tacotron_weights.npz, read without TensorFlow)
    + the 191-entry symbol table and the train.txt sentences 1-64 / 241 kept as ids in tests/golden/taco_symbols.json."""
    from tacotronv2_wavernn_chinese_b200.tacotron.engine import TacoDecoderEngine
    from tacotronv2_wavernn_chinese_b200.tacotron.synthesizer import Synthesizer
    from tacotronv2_wavernn_chinese_b200.tacotron.text import Symbols
    npz = os.path.join(ROOT, 'oracle', '_ref', 'tacotron_weights.npz')
    if not os.path.isfile(npz):
        raise SystemExit(f'no Tacotron checkpoint: {npz} is made by __graft_entry__.build() from the reference checkout')
    w = dict(np.load(npz))
    s = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'taco_symbols.json'), encoding='utf-8'))
    syn = Synthesizer()
    syn.symbols = Symbols(s['symbols'])
    syn.engine = TacoDecoderEngine(w, device=local)
    syn.step = 206500
    text_of = lambda k: syn.symbols.sequence_to_text(s['sentences'][str(k)]['ids'][:-1])
    return syn, text_of, w, s


def run_text2audio(args):
    """BASELINE config 5: train.txt sentences 1-64 -> Tacotron-2 -> WaveRNN, one process per GPU, sentences dealt round-robin by
    length, length-sorted chunks per launch (pipeline.synthesize_sharded).  value = audio samples of all 64 sentences / wall time
    of the whole text->audio call (max over ranks), host strings in, host float64 waves out."""
    import torch
    import torch.distributed as dist
    from tacotronv2_wavernn_chinese_b200 import synth
    from tacotronv2_wavernn_chinese_b200.engine import WaveRNNEngine
    from tacotronv2_wavernn_chinese_b200.pipeline import MIN_FRAMES, deal_round_robin, padded_lockstep_rows, plan_ragged, synthesize_sharded
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    syn, text_of, _, _ = _taco_setup(local)
    sd, wdesc = load_weights(args.weights)
    voc = WaveRNNEngine(sd, synth.DEFAULT_DIMS, device=local)
    texts = [text_of(k) for k in range(1, 65)]
    times, waves, mels = [], None, None
    for i in range(args.warmup + args.steps):
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        waves, mels = synthesize_sharded(syn, voc, texts, seed=7)
        torch.cuda.synchronize(dev)
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        if i >= args.warmup:
            times.append(float(dt.item()))
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {'wave': np.concatenate(waves), 'wave_lengths': [len(w) for w in waves],
                                         'mel': np.concatenate(mels), 'mel_frames': [len(m) for m in mels]})
    if rank == 0:
        total = int(sum(len(w) for w in waves))
        frames = [int(m.shape[0]) for m in mels]
        shares = deal_round_robin(frames, world)
        done = need = 0
        plans = []
        for sh in shares:
            fr = [frames[i] for i in sh]
            kind, plan = plan_ragged(fr, 32)
            if kind == 'pack':
                d, n = plan['rows'] * plan['steps'], sum(max(f, MIN_FRAMES) for f in fr) * HOP
                plans.append(f"packed {plan['rows']} rows")
            else:
                d, n = padded_lockstep_rows(fr, plan)
                plans.append(f'{len(plan)} chunk(s)')
            done, need = done + d, need + n
        dt = float(np.mean(times))
        print(json.dumps({
            'metric': 'text_to_audio_samples_per_sec', 'value': total / dt, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * dt, 'higher_is_better': True, 'scaling': 'strong', 'dtype': 'f32',
            'data': 'train.txt sentences 1-64 (pinyin ids from tests/golden/taco_symbols.json), shipped Tacotron checkpoint, ' + wdesc,
            'config': {'workload': 'BASELINE config 5: tacotron_synthesize -> wavernn_gen in process, 64 sentences', 'sentences': 64,
                       'audio_seconds': total / 22050.0, 'mel_frames_min_max': [min(frames), max(frames)],
                       'parallelism': f'sentences dealt round-robin by length over {world} GPU(s); per rank the cheaper of length-sorted chunks '
                                      f'(<= 32 rows per launch) and packed rows (queues of utterances per kernel row): rank 0 = {plans[0]}',
                       'scheduler_rowsteps_computed_over_needed': done / max(1, need)},
            'rtf': dt / (total / 22050.0)}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_tacotron(args):
    """BASELINE config 4: Tacotron-2 forward-attention decoder on the 50-token sentence (train.txt line 241): one step = encoder +
    the whole decoder loop (until its stop token) + postnet on one GPU.  value = decoder steps (mel frames) per second.
    Roofline: all decoder weights once per step = 6.9 MB (SURVEY 8d), streamed from L2 by the one-CTA-per-sentence kernel."""
    import torch
    from oracle import tacotron_oracle as to
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if int(os.environ.get('RANK', '0')) != 0:
        return
    torch.cuda.set_device(local)
    syn, text_of, w, s = _taco_setup(local)
    text = text_of(241)
    nst, times = 0, []
    for i in range(args.warmup + args.steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mels, info = syn.mels([text], seed=1238, max_iters=800)
        torch.cuda.synchronize()
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
        nst = int(info['decode']['nsteps'][0])
    dt = float(np.mean(times))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'mel': mels[0]})
    # the decoder loop alone (CUDA events on the launch stream), encoder / postnet / host copies excluded
    ids = np.array([s['sentences']['241']['ids']], dtype=np.int32)
    mem = syn.engine.encode(ids, np.array([ids.shape[1]], dtype=np.int32))
    loop_ms = []
    for i in range(args.warmup + args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dec = syn.engine.decode(mem, np.array([ids.shape[1]], dtype=np.int32), seed=1238, max_steps=800, want_align=False)
        e1.record()
        torch.cuda.synchronize()
        if i >= args.warmup:
            loop_ms.append(e0.elapsed_time(e1))
    loop_steps = int(dec['nsteps'][0])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    step_bytes = 4 * sum(int(np.prod(v.shape)) for k, v in w.items() if k.startswith('decoder/'))
    line = {'metric': 'tacotron_decoder_steps_per_sec', 'value': nst / dt, 'unit': 'mel frames/s', 'n_gpus': 1, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * dt, 'higher_is_better': True, 'dtype': 'f32', 'scaling': 'replicas only',
            'data': 'train.txt line 241 (50 pinyin tokens + EOS), shipped checkpoint step 206500',
            'config': {'workload': 'BASELINE config 4: Tacotron-2 decoder inference, 50-token sentence, 1 GPU', 'decoder_steps': nst},
            'us_per_decoder_step': 1e6 * dt / max(1, nst),
            'decoder_loop_only': {'us_per_step': 1e3 * float(np.mean(loop_ms)) / max(1, loop_steps), 'steps': loop_steps,
                                  'kernel': 'taco_grid_kernel (128 blocks, weights resident in shared memory) unless B200TTS_TACO_GRID=0'},
            'roofline': {'bound': 'hbm', 'achieved': step_bytes * nst / dt / 1e9, 'peak': float(peaks.get('hbm_gbs', 6650.0)), 'unit': 'GB/s',
                         'frac': step_bytes * nst / dt / 1e9 / float(peaks.get('hbm_gbs', 6650.0)), 'traffic': None,
                         'algorithmic_bytes_per_step': step_bytes,
                         'note': 'single sentence: weights are shared-memory resident across 128 blocks (taco_grid.cuh), so neither HBM nor L2 '
                                 're-streams them; the step is bound by the six L2-mediated exchanges of its dependency chain'}}
    if not args.no_cpu_baseline:
        mem = to.encoder(w, s['sentences']['241']['ids'])
        t0 = time.perf_counter()
        d = to.decode(w, mem, seed=1238, max_iters=800)
        cpu = time.perf_counter() - t0
        line['cpu_baseline'] = {'value': d['n_steps'] / cpu, 'unit': 'mel frames/s', 'cores': 1, 'kind': 'port',
                                'sample': f"the whole decoder loop ({d['n_steps']} steps) of the numpy oracle (TensorFlow 1.14, which the "
                                          f"reference needs, cannot run here)"}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    if args.workload == 'text2audio':
        return run_text2audio(args)
    if args.workload == 'tacotron':
        return run_tacotron(args)
    import torch
    import torch.distributed as dist
    from tacotronv2_wavernn_chinese_b200 import synth
    from tacotronv2_wavernn_chinese_b200.engine import WaveRNNEngine

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the B200 path has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    N = world
    B, T = args.batch, args.frames
    S, wave_len = T * HOP, (T - 1) * HOP

    sd, wdesc = load_weights(args.weights)
    eng = WaveRNNEngine(sd, synth.DEFAULT_DIMS, device=local)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)   # > 126 MB L2

    def sync_all():
        torch.cuda.synchronize(dev)
        if N > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def measure(per_gpu, global_offset, steps, warmup):
        """Times `steps` passes over this rank's `per_gpu` utterances (rows global_offset ... of the global batch)."""
        mels_dev = torch.as_tensor(synth.synth_mels(1236 + global_offset, per_gpu, T)).to(dev)
        # NCCL has no int16: the labels travel as raw bytes
        gathered = [torch.empty(per_gpu, S * 2, device=dev, dtype=torch.uint8) for _ in range(N)] if N > 1 else None

        def one_step(i):
            flush.fill_(float(i))                                          # evict L2 between iterations
            out = eng.generate(mels_dev, seed=20260923, utterance_offset=global_offset, kernel=args.kernel)
            if N > 1:
                dist.all_gather(gathered, out['labels'].view(torch.uint8))
            return out

        for i in range(warmup):
            one_step(i)
        sync_all()
        launches0 = eng.launch_count
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            measure.last = one_step(i)
        ev1.record()
        sync_all()
        eng.check()
        ms = ev0.elapsed_time(ev1)
        launches = eng.launch_count - launches0 + steps           # + the L2 flush fill per step
        kms = []
        for i in range(min(3, max(1, steps))):                    # the dominant kernel's own duration (events inside the library)
            one_step(i)
            kms.append(eng.last_kernel_ms())
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if N > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        measure.kernel = eng.last_kernel()
        return float(t.item()), float(np.mean(kms)), int(launches)

    sampler = ClockSampler(local)
    sampler.start()
    ms, gen_ms, launches = measure(B, rank * B, args.steps, args.warmup)
    weak_kernel, weak_out = measure.kernel, measure.last
    clocks = sampler.stop()
    value = N * B * S * args.steps / (ms / 1e3)

    # ---- BASELINE config 3 as written: the SAME 256 utterances as a global batch, 256/N per GPU ("strong") ----------
    strong = None
    if not args.no_strong:
        if N == 1:
            strong = {'global_batch': B, 'utterances_per_gpu': B, 'value': value, 'ms_per_step': ms / args.steps,
                      'us_per_lockstep': 1e3 * gen_ms / S, 'note': 'N = 1: identical to the weak line'}
        elif B % N == 0:
            per = B // N
            sms, sgen, _ = measure(per, rank * per, args.steps, max(3, args.warmup))
            strong = {'global_batch': B, 'utterances_per_gpu': per, 'value': B * S * args.steps / (sms / 1e3), 'unit': 'samples/s',
                      'ms_per_step': sms / args.steps, 'us_per_lockstep': 1e3 * sgen / S,
                      'note': 'BASELINE config 3 as written (256 utterances sharded over the GPUs); efficiency = value / (N x the N=1 value)'}

    # ---- end to end through the C-ABI host entry point --------------------------------------------------
    e2e = None
    if not args.no_e2e:
        mels_host = synth.synth_mels(1236 + rank * B, B, T)
        eng.generate_host(mels_host, seed=1)                                # warm the pinned staging buffers
        sync_all()
        t0 = time.perf_counter()
        for i in range(args.steps):
            res = eng.generate_host(mels_host, seed=20260923 + i, utterance_offset=rank * B, kernel=args.kernel)
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=dev, dtype=torch.float64)
        if N > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        assert res['wave'].shape == (B, wave_len) and np.isfinite(res['wave'][:, :8]).all()
        e2e = {'value': N * B * S * args.steps / dt, 'unit': 'samples/s',
               'h2d_bytes_per_step': int(N * B * FEAT * T * 4),
               'd2h_bytes_per_step': int(N * B * (S * 2 + wave_len * 8))}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
        peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s'
        alg_bytes = S * (STEP_WEIGHT_BYTES + B * COND_BYTES_PER_UTT)       # per launch of the generation kernel
        achieved = alg_bytes / (gen_ms / 1e3) / 1e9
        sm_mhz = clocks.get('sm_mhz') or 1965.0
        nominal_fp32 = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
        try:
            fp32_measured = eng.fp32_peak_tflops()
        except Exception:
            fp32_measured = None
        flops = B * S * FLOP_PER_SAMPLE / (gen_ms / 1e3) / 1e12
        traffic, traffic_note = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
            traffic, traffic_note = tj.get('dram_bytes_per_launch'), tj.get('captured_on')
        except Exception:
            pass
        fpeak = fp32_measured or nominal_fp32
        # tensor-core pipeline (wavernn_tc_kernel): every fp32 operand is two fp16 planes and a dot product is three kind::f16
        # MMA products, so the tensor cores EXECUTE 3x the algorithmic GEMM work (6656 x 512 MAC per sample; the conditioning
        # and the fed-back sample column stay on the CUDA cores).  The kernel is bound by the latency of its five-exchange
        # dependency chain, not by either ceiling; both forms are reported.
        tensor_form = None
        if weak_kernel == 'wavernn_tc_kernel':
            tf = 3 * 2 * 6656 * 512 * B * S / (gen_ms / 1e3) / 1e12
            tpeak = float(peaks.get('bf16_tflops_sustained', peaks.get('bf16_tflops', 1437.7)))
            tensor_form = {'executed': tf, 'peak': tpeak, 'unit': 'TFLOP/s (kind::f16 tcgen05.mma, fp32 accumulate)', 'frac': tf / tpeak,
                           'peak_source': 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)' if 'bf16_tflops_sustained' in peaks
                           else 'fallback', 'products_per_dot': 3,
                           'note': 'latency-bound pipeline: 2 groups of 128 rows in flight over 144 layer-stationary CTAs'}
        line = {
            'metric': 'wavernn_audio_samples_per_sec', 'value': value, 'unit': 'samples/s', 'n_gpus': N,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': dict(workload_config(args, N, wdesc), kernel=args.kernel, l2='flushed between timed iterations (256 MiB fill)',
                           parallelism=f'utterance-sharded x{N}, NCCL all-gather of labels' if N > 1 else 'single GPU'),
            'rtf': 22050.0 / (value / (N * B)),
            'us_per_lockstep': 1e3 * gen_ms / S,
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': achieved / hbm_peak,
                         'traffic': traffic, 'traffic_captured_on': traffic_note, 'peak_source': peak_src,
                         'note': 'weights are SMEM-stationary, so the HBM form is small by construction; the binding resources are '
                                 'fp32 FMA issue + the L2->SM broadcast of the activations (wide CUDA-core mapping) or the latency of '
                                 'the per-step exchange chain (tensor-core pipeline); see flop_form / tensor_form',
                         'kernel': weak_kernel, 'kernel_ms': gen_ms, 'algorithmic_bytes_per_launch': alg_bytes, 'tensor_form': tensor_form,
                         'flop_form': {'achieved': flops, 'peak': fpeak, 'unit': 'TFLOP/s fp32 CUDA-core',
                                       'frac': flops / fpeak,
                                       'peak_source': 'measured: register-only FFMA2 loop on all SMs (b200tts_debug_fp32_peak)'
                                       if fp32_measured else 'nominal 148 SM x 128 FMA/clk x 2 x SM clock',
                                       'nominal_peak': nominal_fp32, 'frac_of_nominal': flops / nominal_fp32}},
            'clocks': clocks,
            'gpu_launches': int(launches),
            'e2e': e2e,
            'strong': strong,
        }
        if not args.no_cpu_baseline and N == 1:        # reported baseline: rank 0, single-GPU runs only
            line['cpu_baseline'] = cpu_baseline(B, T, 12.0)
        if args.dump_outputs:                          # rank 0's utterances: labels [B, S], wave [B, (T - 1) * hop]
            dump_outputs(args.dump_outputs, {'labels': weak_out['labels'], 'wave': weak_out['wave']})
        print(json.dumps(line), flush=True)
    if N > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
