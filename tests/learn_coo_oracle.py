"""Sparse numpy restatement of the learn step (learn.smk:306-326,359-408) for matrices keyed by basis column, the
checker of engine.learn_wide and the wide rule bodies.  Built on oracle/skm_oracle.py's window codes; pinned against
its dense learn_matrix (itself pinned on the reference's CSVs) by tests/test_learn_coo_oracle.py."""
from typing import Dict, List, Sequence, Tuple

import numpy as np

from oracle import skm_oracle as O


def annotation_ids(ids: Sequence[str], seq_annot: Dict[str, str]) -> Tuple[np.ndarray, List[str]]:
    """(ann_id int32 [N], annotations in first-appearance order): learn.smk:316-326 keys a dict by sequence id, so a
    repeated id keeps its first position but only its LAST record joins an annotation row; the others get -1."""
    last: Dict[str, int] = {}
    for i, sid in enumerate(ids):
        last[sid] = i
    index: Dict[str, int] = {}
    ann_id = np.full(len(ids), -1, dtype=np.int32)
    for sid, i in last.items():
        acc = O.accession(sid)
        if acc in seq_annot:
            ann_id[i] = index.setdefault(seq_annot[acc], len(index))
    return ann_id, list(index)


def basis_columns(code: np.ndarray, basis: np.ndarray) -> np.ndarray:
    """Column of every code in `basis` (uint64, distinct), -1 when absent."""
    K = len(basis)
    if K == 0:
        return np.full(len(code), -1, dtype=np.int64)
    order = np.argsort(basis, kind="stable")
    sb = basis[order]
    j = np.minimum(np.searchsorted(sb, code), K - 1)
    return np.where(sb[j] == code, order[j], -1)


def learn_coo(seq_idx, code, valid, ann_id: np.ndarray, n_ann: int, basis: np.ndarray):
    """-> (keys int64 sorted, key = ann * K + col; vals int64; totals int64 [K]).  (ann, col) pairs of every valid window
    whose code the basis holds -> np.unique counts; a sequence with ann_id outside [0, n_ann) joins no row.  Totals
    (learn.smk:380) = occurrences of every column over ALL sequences, by bincount."""
    K = len(basis)
    col = basis_columns(code[valid], np.asarray(basis, dtype=np.uint64))
    hit = col >= 0
    col = col[hit]
    a = ann_id[seq_idx[valid][hit]].astype(np.int64)
    totals = np.bincount(col, minlength=K).astype(np.int64)
    ann = (a >= 0) & (a < n_ann)
    keys, vals = np.unique(a[ann] * K + col[ann], return_counts=True)
    return keys.astype(np.int64), vals.astype(np.int64), totals


def coo_dense(keys: np.ndarray, vals: np.ndarray, n_ann: int, K: int) -> np.ndarray:
    M = np.zeros((n_ann, K), dtype=np.int64)
    if K:
        M[keys // K, keys % K] = vals
    return M


def merge(parts):
    """learn.smk:467-494 on (annotations, kmers, M, seq_count, totals, total_seqs) tuples: rows and columns in order of
    first appearance, element-wise sums."""
    rows: Dict[str, int] = {}
    cols: Dict[str, int] = {}
    for anns, kmers, *_ in parts:
        for a in anns:
            rows.setdefault(a, len(rows))
        for km in kmers:
            cols.setdefault(km, len(cols))
    M = np.zeros((len(rows), len(cols)), dtype=np.int64)
    seq_count = np.zeros(len(rows), dtype=np.int64)
    totals = np.zeros(len(cols), dtype=np.int64)
    total_seqs = 0
    for anns, kmers, Mp, sc, tp, ts in parts:
        ri = np.array([rows[a] for a in anns], dtype=np.int64)
        ci = np.array([cols[km] for km in kmers], dtype=np.int64)
        if len(ri) and len(ci):
            M[np.ix_(ri, ci)] += Mp
        np.add.at(seq_count, ri, sc)
        totals[ci] += tp
        total_seqs += ts
    return list(rows), list(cols), M, seq_count, totals, total_seqs
