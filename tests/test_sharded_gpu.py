"""N-rank sharded generation == single-rank generation, BIT FOR BIT, on the real kernels (VERDICT r1 weak #9).

The property rests on two things the kernels guarantee: the sampling noise is keyed by the GLOBAL utterance index, and the push
kernels (<= 32 rows per launch) add the 128 block products of every output in one fixed order whatever the row count, so a row's
arithmetic does not depend on the batch it sits in.  (Above 32 rows per GPU the wide mapping of wavernn_grid.cuh runs, whose
summation order depends on its tile shape: there a shard reproduces the single-rank rows up to sampling near-ties only.)
  * test_shards_equal_single_rank_one_gpu: the shards of 2-, 4- and 8-rank runs computed one after the other on ONE GPU through
    dist.shard_bounds + the same engine call dist.generate_sharded makes (runs everywhere, incl. the driver's 1-GPU box);
  * test_generate_sharded_nccl_world2: the real thing over NCCL with one process per GPU (skipped with fewer than 2 GPUs)."""
import os
import socket

import numpy as np
import pytest

from tacotronv2_wavernn_chinese_b200 import synth
from tacotronv2_wavernn_chinese_b200.dist import shard_bounds

pytestmark = pytest.mark.gpu
STEPS = 3000


def _engine():
    from conftest import load_ckpt_state_dict
    from tacotronv2_wavernn_chinese_b200.engine import WaveRNNEngine
    sd = load_ckpt_state_dict() or synth.synth_state_dict(3)
    return WaveRNNEngine(sd, synth.DEFAULT_DIMS)


@pytest.mark.parametrize('n', [24, 32])      # <= 32 rows in total: every shard AND the single-rank run take the push kernels
def test_shards_equal_single_rank_one_gpu(n):
    import torch
    if not torch.cuda.is_available():
        pytest.fail('GPU tests need a CUDA device')
    eng = _engine()
    mels = synth.synth_mels(4321, n, 21)
    ref = eng.generate(mels, seed=9, max_steps=STEPS, kernel='grid')['labels'].cpu().numpy()
    for world in (2, 4, 8):
        for rank in range(world):
            lo, hi = shard_bounds(n, world, rank)
            part = eng.generate(mels[lo:hi], seed=9, utterance_offset=lo, max_steps=STEPS, kernel='grid')['labels'].cpu().numpy()
            assert np.array_equal(part[:, :STEPS], ref[lo:hi, :STEPS]), f'n={n}: shard {rank}/{world} differs from the single-rank rows {lo}:{hi}'


def _nccl_worker(rank, world, port, n, out):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        from tacotronv2_wavernn_chinese_b200.dist import generate_sharded
        eng = _engine()
        mels = torch.as_tensor(synth.synth_mels(4321, n, 21))
        labels, (lo, hi) = generate_sharded(eng.generate, mels, seed=9, max_steps=STEPS, kernel='grid')
        ref = eng.generate(mels, seed=9, max_steps=STEPS, kernel='grid')['labels']
        out[rank] = bool(torch.equal(labels[:, :STEPS].cpu(), ref[:, :STEPS].cpu()) and (lo, hi) == shard_bounds(n, world, rank))
    finally:
        dist.destroy_process_group()


def test_generate_sharded_nccl_world2():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_nccl_worker, args=(2, port, 24, out), nprocs=2, join=True)
    assert dict(out) == {0: True, 1: True}
