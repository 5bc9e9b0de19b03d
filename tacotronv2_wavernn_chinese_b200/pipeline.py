"""Text -> mel -> audio in one process on the GPU(s) (BASELINE config 5; SURVEY.md 8f rank 2, 8e).

The reference couples its two halves only through a `.npy` file on disk (tacotron_synthesize.py:114-116 ->
wavernn_gen.py:22, float32 (T, 80) = clip((mel + 4) / 8, 0, 1)).  Here the same array goes straight from the Tacotron
postnet to the WaveRNN conditioning network.

Ragged sets are scheduled, not just padded.  A lock-step costs the same whether a row still has samples to produce or not,
and below ~32 rows it barely depends on the row count at all, so
  * the vocoder runs LENGTH-SORTED CHUNKS of at most `max_rows` rows (one launch each, padded only to the longest mel of the
    chunk; every row is truncated / faded at its own length, `gen_opts.d_utt_frames`) -- the padded lock-steps of a 64-sentence
    set drop from (longest - mean) x 64 to the spread inside each chunk;
  * or, when cheaper by the measured step times, PACKED ROWS: one launch whose 8 / 16 / 32 kernel rows each run a queue of
    utterances back to back (longest-processing-time list scheduling, `gen_opts.d_pack_*`), the row restarting from the zero
    state at every utterance start -- no lock-step is spent on padding and a short queue can use a faster, narrower kernel;
  * across ranks the sentences are dealt round-robin in order of decreasing length (SURVEY 8e), so every rank gets the same
    length profile and the makespan is the longest sentence's;
  * the sampling noise and the prenet dropout are keyed by the GLOBAL sentence index (`rng.d_utterance_ids`), so a
    sentence's audio depends neither on the chunking nor on the number of ranks.
Tacotron itself is replicated on every rank: one thread block decodes one sentence, all sentences of a set decode
concurrently (<= 148 per GPU), so sharding it would not shorten anything -- and it removes the mel exchange.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

MIN_FRAMES = 21          # shorter than the 20-hop fade-out cannot be faded (the reference raises, fatchord_version.py:256-258)


def plan_chunks(frames, max_rows=32):
    """Indices of `frames` grouped into launches: sorted by decreasing length, cut every `max_rows`."""
    order = sorted(range(len(frames)), key=lambda i: (-int(frames[i]), i))
    return [order[i:i + max_rows] for i in range(0, len(order), max_rows)]


def deal_round_robin(frames, world):
    """Sentence indices of every rank: the length-sorted list dealt like cards (rank r gets positions r, r+world, ...)."""
    order = sorted(range(len(frames)), key=lambda i: (-int(frames[i]), i))
    return [order[r::world] for r in range(world)]


def padded_lockstep_rows(frames, chunks, hop=275):
    """(row-steps computed, row-steps needed) of a chunk plan: the scheduler's efficiency."""
    done = sum(len(c) * max(max(int(frames[i]) for i in c), MIN_FRAMES) for c in chunks) * hop
    need = sum(max(int(f), MIN_FRAMES) for f in frames) * hop
    return done, need


# us per lock-step of the push kernel by row count (B200, profiles/r02_push_v5_phase_cycles.txt): the scheduler's cost model
STEP_US = {8: 9.0, 16: 14.5, 32: 20.6}


def pack_schedule(frames, rows, hop=275):
    """Longest-processing-time list scheduling of utterances onto `rows` kernel rows: every utterance (longest first) goes to
    the row that frees first.  Returns dict(rows, utt [rows, segs], start [rows, segs + 1], steps) for gen_opts.d_pack_*:
    row r runs utterance utt[r, k] during lock-steps [start[r, k], start[r, k+1]); unused slots: utt = -1, start = 2^31 - 1."""
    order = sorted(range(len(frames)), key=lambda i: (-int(frames[i]), i))
    queue = [[] for _ in range(rows)]
    load = [0] * rows
    for i in order:
        r = min(range(rows), key=lambda j: (load[j], j))
        queue[r].append(i)
        load[r] += max(int(frames[i]), MIN_FRAMES) * hop
    segs = max(1, max(len(q) for q in queue))
    big = 2 ** 31 - 1
    utt = np.full((rows, segs), -1, dtype=np.int32)
    start = np.full((rows, segs + 1), big, dtype=np.int32)
    for r, q in enumerate(queue):
        t = 0
        start[r, 0] = 0
        for k, i in enumerate(q):
            utt[r, k] = i
            t += max(int(frames[i]), MIN_FRAMES) * hop
            start[r, k + 1] = t
    return dict(rows=rows, utt=utt, start=start, steps=int(max(load)), queue=queue)


def plan_ragged(frames, max_rows=32, hop=275):
    """Cheapest of: length-sorted chunks (one utterance per row, padded to the chunk's longest) and packed rows at 8 / 16 / 32
    rows, by the measured step times.  Returns ('chunks', chunk list) or ('pack', schedule)."""
    step = lambda rows: STEP_US[8 if rows <= 8 else (16 if rows <= 16 else 32)]
    chunks = plan_chunks(frames, max_rows)
    best = ('chunks', chunks)
    best_us = sum(max(max(int(frames[i]) for i in c), MIN_FRAMES) * hop * step(len(c)) for c in chunks)
    for rows in (8, 16, 32):
        if rows > max_rows or rows >= 2 * len(frames):
            continue
        sch = pack_schedule(frames, rows, hop)
        us = sch['steps'] * step(rows)
        if us < 0.97 * best_us:
            best, best_us = ('pack', sch), us
    return best


def vocode_ragged(voc, mels, ids, seed=0, max_rows=32, kernel='auto', allow_pack=True):
    """mels: list of float32 [T_b, 80] in [0, 1]; ids: global sentence index of each (keys the sampling noise).
    Returns the list of float64 waves [(max(T_b, 21) - 1) * hop] in the order given."""
    n = len(mels)
    if n == 0:
        return []
    frames = [int(m.shape[0]) for m in mels]
    kind, plan = plan_ragged(frames, max_rows, voc.hop) if allow_pack else ('chunks', plan_chunks(frames, max_rows))
    if kind == 'pack':
        # ONE launch: `rows` kernel rows run queues of utterances back to back (state reset at every utterance start)
        T = max(max(frames), MIN_FRAMES)
        feat = mels[0].shape[1]
        batch = np.zeros((n, feat, T), dtype=np.float32)
        uf = np.zeros(n, dtype=np.int32)
        for i, m in enumerate(mels):
            batch[i, :, :frames[i]] = m.T
            uf[i] = max(frames[i], MIN_FRAMES)
        out = voc.generate(torch.as_tensor(batch), seed=seed, utterance_ids=[int(i) for i in ids], kernel=kernel, utt_frames=uf,
                           pack=plan)
        wave = out['wave'].cpu().numpy()
        voc.check()
        return [wave[i, :(uf[i] - 1) * voc.hop].copy() for i in range(n)]
    waves = [None] * n
    feat = mels[0].shape[1]
    for chunk in plan:
        T = max(max(frames[i] for i in chunk), MIN_FRAMES)
        batch = np.zeros((len(chunk), feat, T), dtype=np.float32)      # zero frames past the end == the reference's own padding
        uf = np.zeros(len(chunk), dtype=np.int32)
        for r, i in enumerate(chunk):
            batch[r, :, :frames[i]] = mels[i].T
            uf[r] = max(frames[i], MIN_FRAMES)
        out = voc.generate(torch.as_tensor(batch), seed=seed, utterance_ids=[int(ids[i]) for i in chunk], kernel=kernel,
                           utt_frames=uf)
        wave = out['wave'].cpu().numpy()
        voc.check()
        for r, i in enumerate(chunk):
            waves[i] = wave[r, :(uf[r] - 1) * voc.hop].copy()
    return waves


def synthesize_batch(synth, wavernn_engine, texts, seed=0, utterance_offset=0, kernel='auto', max_rows=32, allow_pack=True):
    """synth: tacotron.synthesizer.Synthesizer (loaded); wavernn_engine: engine.WaveRNNEngine; texts: pinyin strings.
    Returns (list of float64 waves, list of mels [T_b, 80]) for sentences utterance_offset ... of a larger set."""
    mels, _ = synth.mels(texts, seed=seed, utterance_offset=utterance_offset)
    ids = [utterance_offset + b for b in range(len(mels))]
    return vocode_ragged(wavernn_engine, mels, ids, seed=seed, max_rows=max_rows, kernel=kernel, allow_pack=allow_pack), list(mels)


def synthesize_sharded(synth, wavernn_engine, texts, seed=0, group=None, kernel='auto', max_rows=32):
    """All ranks call this with the SAME `texts`; every rank returns all waves (input order) and all mels.
    One process per GPU (`torch.distributed`); the only collective is the final all-gather of the padded waves."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    mels, _ = synth.mels(texts, seed=seed, utterance_offset=0)           # replicated (see module docstring)
    n = len(mels)
    frames = [int(m.shape[0]) for m in mels]
    mine = deal_round_robin(frames, world)[rank]
    local = vocode_ragged(wavernn_engine, [mels[i] for i in mine], mine, seed=seed, max_rows=max_rows, kernel=kernel)
    if world == 1:
        out = [None] * n
        for i, w in zip(mine, local):
            out[i] = w
        return out, list(mels)
    hop = wavernn_engine.hop
    lens = [(max(f, MIN_FRAMES) - 1) * hop for f in frames]
    per_rank = (n + world - 1) // world
    nccl = dist.get_backend(group) == 'nccl'
    dev = torch.device('cuda', torch.cuda.current_device()) if nccl else torch.device('cpu')
    buf = torch.zeros((per_rank, max(lens) if lens else 1), dtype=torch.float64, device=dev)
    for r, w in enumerate(local):
        buf[r, :len(w)] = torch.as_tensor(w, device=dev)
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf, group=group)
    shares = deal_round_robin(frames, world)
    out = [None] * n
    for r, share in enumerate(shares):
        host = parts[r].cpu().numpy()
        for k, i in enumerate(share):
            out[i] = host[k, :lens[i]].copy()
    return out, list(mels)


def synthesize_stream(synth, wavernn_engine, text, seed=0, utterance_offset=0, chunk_steps=None):
    """Text -> audio for ONE sentence, handed out while the vocoder runs: Tacotron decodes the whole mel first, then the
    push kernel streams the wave (WaveRNNEngine.generate_stream).  Yields (start, float64 chunk [n]) until the sentence's
    (max(T, 21) - 1) * hop samples are out; concatenated they are bit for bit synthesize_batch(synth, eng, [text])[0][0]
    (same noise key: the sentence is global utterance `utterance_offset`, padded to MIN_FRAMES like vocode_ragged)."""
    mels, _ = synth.mels([text], seed=seed, utterance_offset=utterance_offset)
    mel = mels[0]
    frames = int(mel.shape[0])
    T = max(frames, MIN_FRAMES)
    batch = np.zeros((1, mel.shape[1], T), dtype=np.float32)
    batch[0, :, :frames] = mel.T
    for start, chunk in wavernn_engine.generate_stream(torch.as_tensor(batch), seed=seed, utterance_ids=[int(utterance_offset)],
                                                       utt_frames=np.array([T], dtype=np.int32), chunk_steps=chunk_steps):
        yield start, chunk[0]
