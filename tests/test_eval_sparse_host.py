"""Host side of the sparse evaluate path: the .skme side-car, the name table of skm_confidence_classify and the rank
merge of the evaluate crosstabs (dist.allreduce_confidence_tables) under gloo."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from snekmer_b200 import confidence as CF
from snekmer_b200 import dist as D
from snekmer_b200 import sidecar as SC


def test_evalscores_roundtrip(tmp_path):
    rng = np.random.default_rng(1)
    q = 1000
    anns = ["TIGR00001", "ünï", ""]
    names = anns + ["file-only", "β"]
    arrays = dict(top1=rng.integers(-1, 3, q).astype(np.int32), top2=rng.integers(-1, 3, q).astype(np.int32),
                  score1=rng.random(q), score2=np.where(rng.random(q) < 0.1, np.nan, rng.random(q)),
                  truth=rng.integers(-1, 5, q).astype(np.int32))
    p = str(tmp_path / "seq-annotation-scores-x.skme")
    SC.write_evalscores(p, anns, names, row_base=123456789012, **arrays)
    for mmap in (True, False):
        d = SC.read_evalscores(p, mmap)
        assert d["annotations"] == anns and d["names"] == names and d["row_base"] == 123456789012
        for k, v in arrays.items():
            assert d[k].dtype == v.dtype and np.array_equal(d[k], v, equal_nan=True), k
    # an empty file
    e = str(tmp_path / "empty.skme")
    SC.write_evalscores(e, [], [], *(np.zeros(0),) * 5, row_base=0)
    d = SC.read_evalscores(e)
    assert d["names"] == [] and d["top1"].dtype == np.int32 and d["top1"].size == 0
    # another container kind is refused
    SC.write_counts(str(tmp_path / "c.skmc"), ["Totals"], ["AAA"], np.zeros(1), np.zeros(1), np.zeros((1, 1)))
    with pytest.raises(ValueError):
        SC.read_evalscores(str(tmp_path / "c.skmc"))


def test_joint_name_table():
    anns = ["b", "a", "c"]
    table, idx = CF.joint_name_table(anns, ["a", None, "x", "c", "x", "", None, "y", "b"])
    assert table == ["b", "a", "c", "x", "", "y"]
    assert idx.dtype == np.int32 and idx.tolist() == [1, -1, 3, 2, 3, 4, -1, 5, 0]
    assert all(idx[i] < 0 or table[idx[i]] == n for i, n in enumerate(["a", None, "x", "c", "x", "", None, "y", "b"]))
    # non-string annotation values are named by str(), as the label f-string names them
    table, idx = CF.joint_name_table(["1"], [1, 2.5])
    assert table == ["1", "2.5"] and idx.tolist() == [0, 1]
    table, idx = CF.joint_name_table([], [])
    assert table == [] and idx.size == 0


# ---- rank merge under gloo -------------------------------------------------------------------------------------------
N_ANN, NROWS = 7, 3000


def _rows():
    """One file's rows as the device produces them: prediction, Difference bin (255 = none), class, exact tie."""
    rng = np.random.default_rng(11)
    pred = rng.integers(0, N_ANN, NROWS)
    bins = np.where(rng.random(NROWS) < 0.05, 255, rng.integers(0, 101, NROWS))
    bins[rng.random(NROWS) < 0.02] = 0
    cls = rng.integers(0, 3, NROWS).astype(np.uint8)
    tie = rng.random(NROWS) < 0.5
    return pred, bins, cls, tie


def _tables(pred, bins, cls, tie, row_base):
    """Crosstabs (what skm_confidence_hist accumulates) and the zero-bin key of ConfidenceAccumulator.add_device."""
    ok = bins != 255
    ht = np.bincount((pred * 101 + bins)[ok & (cls == 1)], minlength=N_ANN * 101).reshape(N_ANN, 101)
    hf = np.bincount((pred * 101 + bins)[ok & (cls == 2)], minlength=N_ANN * 101).reshape(N_ANN, 101)
    z = np.flatnonzero((cls == 1) & (bins == 0))
    key = 2 * (row_base + int(z[0])) + int(tie[z[0]]) if z.size else CF.NO_ZERO_ROW
    return torch.from_numpy(ht.astype(np.int64)), torch.from_numpy(hf.astype(np.int64)), torch.tensor([key], dtype=torch.int64)


def _worker(rank, world, port, tmp, cut):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    D.init("gloo")
    try:
        pred, bins, cls, tie = _rows()
        lo, hi = (0, cut) if rank == 0 else (cut, NROWS)
        base, total = D.exclusive_prefix(hi - lo)
        assert base == lo and total == NROWS
        ht, hf, key = _tables(pred[lo:hi], bins[lo:hi], cls[lo:hi], tie[lo:hi], base)
        D.allreduce_confidence_tables(ht, hf, key)
        wt, wf, wkey = _tables(pred, bins, cls, tie, 0)
        assert torch.equal(ht, wt) and torch.equal(hf, wf) and torch.equal(key, wkey)
        with open(os.path.join(tmp, f"ok{rank}-{cut}"), "w") as fh:
            fh.write(str(int(key)))
    finally:
        torch.distributed.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_rank_merge_equals_one_process(tmp_path):
    pred, bins, cls, tie = _rows()
    first = int(np.flatnonzero((cls == 1) & (bins == 0))[0])
    # the first qualifying row on rank 0, on rank 1 (rank 0 has none), and rank 0 empty
    for cut in (NROWS // 2, first, 0):
        mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), cut), nprocs=2, join=True)
        keys = {open(tmp_path / f"ok{r}-{cut}").read() for r in range(2)}
        assert keys == {str(2 * first + int(tie[first]))}
    # one process: nothing to exchange
    ht, hf, key = _tables(pred, bins, cls, tie, 0)
    h0, f0, k0 = ht.clone(), hf.clone(), key.clone()
    D.allreduce_confidence_tables(ht, hf, key)
    assert torch.equal(ht, h0) and torch.equal(hf, f0) and torch.equal(key, k0)
