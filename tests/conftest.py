import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a real B200 (run with -m gpu on the GPU box)')


@pytest.fixture(scope='session', autouse=True)
def _bounded_blas_pool():
    """The oracles run thousands of tiny matvecs; more than 4 BLAS threads buys nothing (measured: 61 s with 4, 64 s with 8)
    and, on a busy or over-committed host, spinning worker threads can stretch the suite from one minute to tens of minutes."""
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        yield
        return
    with threadpool_limits(limits=min(4, os.cpu_count() or 1)):
        yield


GOLDEN = os.path.join(ROOT, 'tests', 'golden')
REF_CKPT_COPY = os.path.join(ROOT, 'oracle', '_ref', 'latest_weights.pyt')


def load_ckpt_state_dict():
    """The shipped checkpoint, from the git-ignored copy that __graft_entry__.build() makes under oracle/_ref/, or None."""
    import torch
    if not os.path.isfile(REF_CKPT_COPY):
        return None
    sd = torch.load(REF_CKPT_COPY, map_location='cpu', weights_only=False)
    return {k: v.numpy() for k, v in sd.items()}


@pytest.fixture(scope='session')
def ckpt_state_dict():
    sd = load_ckpt_state_dict()
    if sd is None:
        pytest.skip('shipped checkpoint not available (no oracle/_ref/ copy)')
    return sd
