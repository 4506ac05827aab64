"""CPU: the association side-car (.skma, sidecar.AssociationsWriter) and the streamed seq-annotation-scores CSV writer
against one-shot numpy / pyarrow references."""
import numpy as np
import pytest

from snekmer_b200 import sidecar as SC

ANNS = ["TIGR00001", 'fam,"quoted"', "with space", "α", ""]


def _table(Q, A, seed=0):
    rng = np.random.default_rng(seed)
    S = rng.random((Q, A))
    S[rng.random((Q, A)) < 0.3] = np.nan
    if Q > 3:
        S[3] = 0.0
    if Q and A:
        S[0, 0] = 1.0 / 3.0
    labels = [f"{ANNS[q % len(ANNS)]}_known_{q}" if q % 3 else f"acc{q}_unknown_{q}" for q in range(Q)]
    return S, labels


def _cuts(Q, sizes):
    q0, out = 0, []
    i = 0
    while q0 < Q:
        n = min(sizes[i % len(sizes)], Q - q0)
        out.append((q0, n))
        q0 += n
        i += 1
    return out


@pytest.mark.parametrize("Q,A", [(0, 5), (1, 1), (23, 5), (40, 0), (257, 3)])
def test_skma_roundtrip_in_uneven_blocks(Q, A, tmp_path):
    S, labels = _table(Q, A)
    anns = (ANNS * 2)[:A]
    p = str(tmp_path / "a.skma")
    with SC.AssociationsWriter(p, anns, labels) as w:
        for q0, n in reversed(_cuts(Q, [7, 1, 13])):          # any order: blocks land at their offsets
            w.write(q0, S[q0:q0 + n])
    one = str(tmp_path / "b.skma")
    with SC.associations_writer(one, anns, labels) as w:
        w.write(0, S)
    assert open(p, "rb").read() == open(one, "rb").read()
    for mmap in (True, False):
        d = SC.read_associations(p, mmap)
        assert d["annotations"] == anns and d["rows"] == labels
        assert d["scores"].dtype == np.float64 and d["scores"].shape == (Q, A)
        assert np.array_equal(d["scores"], S, equal_nan=True)
    kind, attrs, _ = SC.read_container(p)
    assert kind == "associations" and attrs == {"n_ann": A, "nrows": Q}
    with pytest.raises(ValueError):
        SC.read_evalscores(p)


@pytest.mark.parametrize("Q,A", [(0, 5), (1, 1), (23, 5), (40, 0), (257, 3)])
def test_csv_export_matches_pyarrow_write_csv(Q, A, tmp_path):
    import pyarrow as pa
    from pyarrow import csv as pacsv

    S, labels = _table(Q, A, seed=1)
    anns = (ANNS * 2)[:A]
    cols = {a: S[:, j] for j, a in enumerate(anns)}
    cols[SC.INDEX_COL] = pa.array(labels, type=pa.string())
    want = str(tmp_path / "want.csv")
    pacsv.write_csv(pa.table(cols), want)
    direct = str(tmp_path / "direct.csv")
    with SC.associations_writer(direct, anns, labels) as w:
        for q0, n in _cuts(Q, [5, 11, 2]):
            w.write(q0, S[q0:q0 + n])
    side = str(tmp_path / "a.skma")
    with SC.associations_writer(side, anns, labels) as w:
        w.write(0, S)
    exported = str(tmp_path / "exported.csv")
    SC.export_associations_csv(side, exported, block_rows=4)
    ref = open(want, "rb").read()
    assert open(direct, "rb").read() == ref and open(exported, "rb").read() == ref
    if Q:
        assert b"nan" in ref or not np.isnan(S).any()


def test_csv_writer_needs_rows_in_order(tmp_path):
    S, labels = _table(10, 2)
    with SC.AssociationsCSVWriter(str(tmp_path / "x.csv"), ANNS[:2], labels) as w:
        w.write(0, S[:4])
        with pytest.raises(AssertionError):
            w.write(6, S[6:])
