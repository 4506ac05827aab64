"""CPU only: the sparse learn oracle (learn_coo_oracle.learn_coo, the checker of the wide learn) equals the golden-pinned
dense oracle (oracle/skm_oracle.py::learn_matrix) on the golden rule inputs and on a small wide-space case."""
import os

import numpy as np
import pytest

from learn_coo_oracle import annotation_ids, coo_dense, learn_coo
from oracle import skm_oracle as O
from util import GOLDEN, RULE_CONFIGS, read_ann, read_fasta


def _alpha(a):
    return None if a == "None" else (int(a) if str(a).isdigit() else a)


def _check(ids, seqs, a, k, mf, seq_annot):
    lut, syms = O.build_lut(a)
    res, offs = O.pack(seqs)
    si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
    basis, _ = O.basis_codes(si, pos, code, valid, mf)
    C = O.count_matrix(si, code, valid, len(seqs), basis)
    anns, M, nseq, totals, total_seqs = O.learn_matrix(ids, C, seq_annot)
    ann_id, got_anns = annotation_ids(ids, seq_annot)
    keys, vals, got_totals = learn_coo(si, code, valid, ann_id, len(got_anns), basis)
    assert got_anns == anns
    assert np.all(np.diff(keys) > 0) and np.all(vals > 0)
    assert np.array_equal(coo_dense(keys, vals, len(anns), len(basis)), M)
    assert np.array_equal(got_totals, totals)
    assert np.array_equal(np.bincount(ann_id[ann_id >= 0], minlength=len(anns)), nseq)


@pytest.mark.parametrize("name", sorted(RULE_CONFIGS))
def test_learn_coo_equals_learn_matrix_on_golden_rules(name):
    a, k, mf = RULE_CONFIGS[name]
    seq_annot = read_ann(os.path.join(GOLDEN, "syn.ann"))
    for nb in ("synA", "synB"):
        ids, seqs = read_fasta(os.path.join(GOLDEN, f"{nb}.fasta"))
        _check(ids, seqs, _alpha(a), k, mf, seq_annot)


@pytest.mark.parametrize("mf", [0, 1])
def test_learn_coo_equals_learn_matrix_wide(mf):
    """20 letters at k = 8 (20^8 > 2^27): a dense [N, K] matrix is still cheap at 300 sequences.  Repeated ids, ids
    without an annotation and a min_filter basis (windows outside it count nowhere, Totals included)."""
    rng = np.random.default_rng(11 + mf)
    aa = np.array(list("ACDEFGHIKLMNPQRSTVWYX"))
    n = 300
    seqs = ["".join(rng.choice(aa, size=int(rng.integers(0, 200)))) for _ in range(n)]
    # low-complexity copies so that some k-mers repeat across sequences and survive the filter
    seqs += [s[: len(s) // 2] * 2 for s in seqs[:60]]
    accs = [f"P{i % 250:04d}" for i in range(len(seqs))]                    # repeated accessions -> repeated ids
    ids = [f"sp|{acc}|x" for acc in accs]
    seq_annot = {f"P{i:04d}": f"TIGR{int(rng.integers(0, 12)):05d}" for i in range(0, 250) if rng.random() < 0.7}
    _check(ids, seqs, None, 8, mf, seq_annot)
