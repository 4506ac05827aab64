"""CPU tests of the host-side logic added in round 2 (no GPU, no compute calls into the library)."""
import numpy as np
import pytest

from snekmer_b200 import dist as D
from snekmer_b200 import engine as E
from snekmer_b200 import pipeline as P


def test_push_plan_layout_matches_all_to_all_order():
    """Receive buffers hold the senders' runs in rank order; a sender's run starts behind the runs of the lower ranks."""
    m = np.array([[5, 0, 2], [1, 7, 0], [3, 4, 9]], dtype=np.int64)        # m[s, r] = entries rank s sends to rank r
    for rank in range(3):
        dst_off, runs, words = D.push_plan(m, rank)
        assert dst_off.tolist() == m[:rank].sum(axis=0).tolist()
        assert runs.tolist() == m[:, rank].tolist()
        assert words == int(m.sum(axis=0).max()) == 11
    # every receiver's buffer is tiled exactly by the runs written into it
    for r in range(3):
        spans = sorted((int(D.push_plan(m, s)[0][r]), int(m[s, r])) for s in range(3))
        pos = 0
        for off, n in spans:
            assert off == pos
            pos += n
        assert pos == int(m[:, r].sum())
    assert D.push_plan(np.zeros((1, 1), dtype=np.int64), 0)[2] == 0


def test_learn_methods_are_checked():
    """An unknown learn method is an error, not a silent switch to another algorithm."""
    with pytest.raises(ValueError, match="hybrid"):
        E.learn_sparse_with_totals(None, "miqs", 3, None, 4, method="typo")
    with pytest.raises(ValueError, match="grouped"):
        E.learn_sparse(None, "miqs", 3, None, 4, method="sorted")


def test_host_coo_unpacks_the_exchange_format():
    rng = np.random.default_rng(0)
    bits = 29
    keys = np.sort(rng.choice(1 << 34, size=1000, replace=False)).astype(np.int64)
    vals = rng.integers(1, 1 << 20, size=1000, dtype=np.int64)
    packed = (keys.astype(np.uint64) << np.uint64(bits)) | vals.astype(np.uint64)
    h = P.HostCOO(S=6 ** 8, n_ann=20000, count_bits=bits, packed=packed)
    assert h.nnz == 1000 and np.array_equal(h.keys(), keys) and np.array_equal(h.vals(), vals)
    raw = P.HostCOO(S=6 ** 8, n_ann=20000, count_bits=bits, raw=(keys, vals))
    assert raw.nnz == 1000 and raw.keys() is keys and raw.vals() is vals


def test_bind_to_local_cpus_is_harmless_without_a_gpu():
    import os

    before = os.sched_getaffinity(0)
    r = D.bind_to_local_cpus(0)
    assert r is None or set(r) <= before
    os.sched_setaffinity(0, before)


def test_peer_exchange_is_off_outside_nccl():
    import torch

    assert not E.peer_exchange_enabled(torch.zeros(1))       # CPU tensor, no process group: the collective path
    assert D.peer_buffers().words == 0 and not D.peer_buffers().disabled
