"""GPU: full association rows from the SpMM (skm_apply_sparse_rows, engine.apply_sparse(rows_out=) /
apply_sparse_tiled(rows_sink=)) and the association files of the sparse apply / eval_apply rule bodies, against the
float64 numpy cosine, the top-2-only path, the reference's cosine matrices and the CSV Evaluator."""
import os

import numpy as np
import pandas as pd
import pytest
import torch

from learn_coo_oracle import annotation_ids, basis_columns, coo_dense, learn_coo, merge
from oracle import skm_oracle as O
from util import GOLDEN, RULE_CONFIGS, load_rule, read_fasta

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from snekmer_b200 import engine as E
    from snekmer_b200 import io as skio
    from snekmer_b200 import rules as R
    from snekmer_b200 import rules_sparse as RS
    from snekmer_b200 import sidecar as SC

ALPHA, K = 2, 6
C1 = os.path.join(GOLDEN, "c1")
C1_FILES = ["UP000322080_2603819", "UP000322981_424902"]


# ---- kernel and engine against the numpy cosine ---------------------------------------------------------------------
def _seqs(rng, n, lo, hi):
    aa = np.array(list("ACDEFGHIKLMNPQRSTVWYX"))
    p = np.array([1.0] * 20 + [0.05])
    return ["".join(rng.choice(aa, size=int(rng.integers(lo, hi)), p=p / p.sum())) for _ in range(n)]


def _problem(seed, n_ann, vmax=50, big=None, long_query=False):
    """A random sorted COO matrix over the codes of (ALPHA, K) — annotation 0 and the middle one all zero — and
    queries including an empty one, one shorter than k and one of invalid residues only."""
    rng = np.random.default_rng(seed)
    S = len(O.build_lut(ALPHA)[1]) ** K
    keys = []
    for a in range(n_ann):
        if n_ann > 2 and a in (0, n_ann // 2):
            continue
        codes = np.unique(rng.integers(0, S, size=int(rng.integers(1, 120))))
        keys.append(a * S + codes)
    key = np.concatenate(keys).astype(np.int64) if keys else np.zeros(0, np.int64)
    val = rng.integers(1, vmax, size=key.size).astype(np.int64)
    if big is not None and key.size:
        val[key.size // 3] = big
    queries = _seqs(rng, 150, 0, 300) + ["", "ACD", "X" * 10, "XA" * 8]
    if long_query:
        queries.append(_seqs(rng, 1, 70100, 70101)[0].replace("X", "A"))
    qb = E.SequenceBatch.from_strings(queries)
    rowptr, cols, cvals = E.count_csr(qb, ALPHA, K, None)
    lut, syms = O.build_lut(ALPHA)
    res, offs = O.pack(queries)
    si, _, code, valid = O.window_codes(res, offs, lut, len(syms), K)
    Q = O.count_matrix(si, code, valid, len(queries), np.arange(S, dtype=np.uint64))
    M = np.zeros((n_ann, S), dtype=np.int64)
    M[key // S, key % S] = val
    return (rowptr, cols, cvals, torch.from_numpy(key).cuda(), torch.from_numpy(val).cuda(), S), O.cosine_scores(Q, M)


class Sink:
    def __init__(self, nq, n_ann):
        self.rows = np.full((nq, n_ann), np.nan)
        self.calls = []

    def __call__(self, q0, block):
        assert block.dtype == np.float64 and block.shape[1] == self.rows.shape[1]
        self.calls.append((q0, block.shape[0]))
        self.rows[q0:q0 + block.shape[0]] = block


def _same_top2(a, b):
    assert torch.equal(a.top1, b.top1) and torch.equal(a.top2, b.top2)
    for f in ("score1", "score2"):                  # NaN where a query has no candidate (no annotations)
        assert np.array_equal(getattr(a, f).cpu().numpy(), getattr(b, f).cpu().numpy(), equal_nan=True)


def _check_rows(rows, r, Sc):
    nq = rows.shape[0]
    assert not np.isnan(rows).any()
    assert np.max(np.abs(rows - Sc), initial=0.0) < 1e-12
    q = np.arange(nq)
    t1, t2 = r.top1.cpu().numpy(), r.top2.cpu().numpy()
    assert np.array_equal(rows[q, t1], r.score1.cpu().numpy())          # bit for bit
    k2 = t2 >= 0
    assert np.array_equal(rows[q[k2], t2[k2]], r.score2.cpu().numpy()[k2])
    zero = ~Sc.any(axis=1)
    assert zero.sum() >= 4 and np.all(rows[zero] == 0.0)                # no valid window: exact zeros, no NaN


@pytest.mark.parametrize("n_ann,vmax,big,long_query,tile,chunk,acc_bits", [
    (1, 50, None, False, None, None, 32),
    (2, 50, None, False, None, 1, 32),
    (7, 50, None, False, 3, 5, 32),
    (403, 50, None, False, 100, 37, 32),
    (403, 50, 70000, False, 64, 64, 32),             # an entry >= 65,536: unpacked CSC, 32-bit dots
    (7, 50, 1 << 26, False, 2, 13, 64),              # unpacked, 64-bit accumulators
    (403, 65535, None, True, 150, 40, 64),           # packed, 64-bit accumulators (a 70,100-residue query)
])
def test_rows_match_numpy_cosine(n_ann, vmax, big, long_query, tile, chunk, acc_bits):
    (rowptr, cols, cvals, keys, vals, S), Sc = _problem(n_ann + int(vmax) + (big or 0), n_ann, vmax, big, long_query)
    nq = rowptr.numel() - 1
    row_total = E.query_row_total_max(rowptr, cvals)
    assert E.sparse_acc_bits(int(vals.max().item()), row_total) == acc_bits
    want = E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann, tile)
    sink = Sink(nq, n_ann)
    got = E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann, tile, rows_sink=sink, chunk_rows=chunk)
    _same_top2(got, want)
    step = chunk or nq
    assert sink.calls == [(q0, min(step, nq - q0)) for q0 in range(0, nq, step)]
    _check_rows(sink.rows, got, Sc)


@pytest.mark.parametrize("use_packed", [True, False])
def test_one_tile_rows_out_into_a_wider_buffer(use_packed):
    n_ann = 7
    (rowptr, cols, cvals, keys, vals, S), Sc = _problem(5, n_ann)
    nq = rowptr.numel() - 1
    csc = E.csc_build(keys, vals, S, n_ann, 0)
    assert csc.packed is not None
    want = E.apply_sparse(rowptr, cols, cvals, csc, use_packed=use_packed)
    buf = torch.full((nq, n_ann + 6), -7.0, dtype=torch.float64, device="cuda")
    got = E.apply_sparse(rowptr, cols, cvals, csc, use_packed=use_packed, rows_out=buf[:, 3:3 + n_ann])
    _same_top2(got, want)
    h = buf.cpu().numpy()
    assert np.all(h[:, :3] == -7.0) and np.all(h[:, 3 + n_ann:] == -7.0)       # nothing outside the slice
    _check_rows(h[:, 3:3 + n_ann], got, Sc)
    with pytest.raises(E.SkmError):
        E.apply_sparse(rowptr, cols, cvals, csc, rows_out=buf[:, :n_ann - 1])
    with pytest.raises(E.SkmError):
        E.apply_sparse(rowptr, cols, cvals, csc, rows_out=buf[:, :n_ann].to(torch.float32))


def test_empty_query_set_and_no_annotations():
    (rowptr, cols, cvals, keys, vals, S), _ = _problem(9, 7)
    nq = rowptr.numel() - 1
    calls = []
    e = E.apply_sparse_tiled(rowptr[:1], cols, cvals, keys, vals, S, 7, rows_sink=lambda q0, b: calls.append(q0))
    assert calls == [] and e.top1.numel() == 0
    sink = Sink(nq, 0)
    r = E.apply_sparse_tiled(rowptr, cols, cvals, keys[:0], vals[:0], S, 0, rows_sink=sink, chunk_rows=60)
    assert sink.calls == [(q0, min(60, nq - q0)) for q0 in range(0, nq, 60)]
    _same_top2(r, E.apply_sparse_tiled(rowptr, cols, cvals, keys[:0], vals[:0], S, 0))


# ---- a column-keyed code space ---------------------------------------------------------------------------------------
def test_wide_rows_match_oracle(tmp_path):
    a, k = None, 7
    seq_annot = R.load_annotations([os.path.join(GOLDEN, "syn.ann")])
    lut, syms = O.build_lut(a)
    files, parts = {}, []
    for nb in ("synA", "synB"):
        ids, seqs = read_fasta(os.path.join(GOLDEN, f"{nb}.fasta"))
        reduced = [O.reduce_str(s, a) for s in seqs]
        res, offs = O.pack(seqs)
        si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
        basis, _ = O.basis_codes(si, pos, code, valid, 0)
        ann_id, anns = annotation_ids(ids, seq_annot)
        keys, vals, totals = learn_coo(si, code, valid, ann_id, len(anns), basis)
        seq_count = np.bincount(ann_id[ann_id >= 0], minlength=len(anns)).astype(np.int64)
        kmers = [str(x) for x in O.decode(basis, syms, k)]
        files[nb] = dict(ids=ids, reduced=reduced, windows=(si, code, valid), basis=basis, n=len(seqs),
                         part=(anns, kmers, coo_dense(keys, vals, len(anns), len(basis)), seq_count, totals, len(set(ids))))
        parts.append(RS.learn_counts_sparse(ids, reduced, "".join(sorted(set("".join(kmers)))), k, seq_annot))
    merged = RS.merge_counts_sparse(parts)
    assert merged.columns is not None
    rows, cols, Mm, *_ = merge([f["part"] for f in files.values()])
    code_of = {}
    for f in files.values():
        code_of.update(zip(f["part"][1], f["basis"]))
    col_codes = np.array([code_of[km] for km in cols], dtype=np.uint64)
    for nb, f in files.items():
        side = str(tmp_path / f"{nb}.skma")
        ev = RS.eval_counts_sparse(f["ids"], f["reduced"], merged, seq_annot, out_scores=side, save_associations=True, chunk_rows=17)
        plain = RS.eval_counts_sparse(f["ids"], f["reduced"], merged, seq_annot)
        _same_top2(ev.result(), plain.result())
        uniq, pick = R._unique_last(f["ids"])
        si, code, valid = f["windows"]
        C_all = O.count_matrix(si, code, valid, f["n"], f["basis"])[pick].astype(np.int64)
        at = basis_columns(col_codes, f["basis"])
        Q = np.zeros((len(pick), len(cols)), dtype=np.int64)
        Q[:, at >= 0] = C_all[:, at[at >= 0]]
        d = SC.read_associations(side)
        assert d["annotations"] == rows and len(d["rows"]) == len(uniq)
        assert np.max(np.abs(d["scores"] - O.cosine_scores(Q, Mm, (C_all * C_all).sum(axis=1)))) < 1e-12
        q = np.arange(len(uniq))
        assert np.array_equal(d["scores"][q, ev.top1.cpu().numpy()], ev.score1.cpu().numpy())


# ---- rule bodies against the reference's cosine matrices -------------------------------------------------------------
def _read_scores(path):
    df = pd.read_csv(path, index_col="__index_level_0__")
    return [str(x) for x in df.index], [str(c) for c in df.columns], df.values.astype(np.float64)


def _check_eval_files(tmp_path, tag, ids, seqs, merged, seq_annot, kmerlist, ref_rows, ref_cols, ref_S, chunk):
    full = str(tmp_path / f"seq-annotation-scores-{tag}.csv")
    ev = RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist, out_scores=full, save_associations=True,
                               chunk_rows=chunk)
    rows, cols, S = _read_scores(full)
    assert rows == [str(x) for x in ref_rows] and cols == [str(x) for x in ref_cols]
    assert np.max(np.abs(S - ref_S)) < 1e-12
    side = str(tmp_path / f"{tag}.skma")
    RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist, out_scores=side, save_associations=True)
    back = str(tmp_path / f"{tag}.export.csv")
    SC.export_associations_csv(side, back)
    assert open(back, "rb").read() == open(full, "rb").read()
    masked = str(tmp_path / f"seq-annotation-scores-{tag}-top2.csv")
    ev2 = RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist, out_scores=masked)
    _same_top2(ev.result(), ev2.result())
    rows2, cols2, S2 = _read_scores(masked)
    assert rows2 == rows and cols2 == cols
    fin = np.isfinite(S2)
    assert np.all(fin.sum(axis=1) == min(2, len(cols)))
    assert np.max(np.abs(S2[fin] - ref_S[fin])) < 1e-12
    assert np.max(np.abs(np.nanmax(S2, axis=1) - ref_S.max(axis=1))) < 1e-12
    return ev, masked


@pytest.mark.parametrize("name", ["hydro_k8", "miqs_k3", "solvacc_k4"])
def test_rule_association_files_match_reference(name, tmp_path):
    a, k, mf = RULE_CONFIGS[name]
    a = None if a == "None" else (int(a) if str(a).isdigit() else a)
    d = load_rule(name)
    seq_annot = R.load_annotations([os.path.join(GOLDEN, "syn.ann")])
    parts, frames = [], {}
    for nb in ("synA", "synB"):
        npz = str(tmp_path / f"{nb}.npz")
        R.vectorize_rule(os.path.join(GOLDEN, f"{nb}.fasta"), npz, None, a, k, min_filter=mf)
        kl, df = skio.load_npz(npz)
        kmerlist = [str(x) for x in kl[0]]
        frames[nb] = (df, kmerlist)
        parts.append(RS.learn_counts_sparse(list(df["sequence_id"]), list(df["sequence"]), "".join(sorted(set("".join(kmerlist)))), k,
                                            seq_annot))
    merged = RS.merge_counts_sparse(parts)
    for nb, chunk in (("synA", 7), ("synB", None)):
        df, kmerlist = frames[nb]
        _check_eval_files(tmp_path, nb, list(df["sequence_id"]), list(df["sequence"]), merged, seq_annot, kmerlist,
                          d[f"{nb}_eval_rows"], d[f"{nb}_eval_cols"], d[f"{nb}_eval_scores"], chunk)
    # apply: synB against the matrix learned on synA
    df, kmerlist = frames["synB"]
    ids, seqs = list(df["sequence_id"]), list(df["sequence"])
    out = str(tmp_path / "seq-annotation-scores-apply.csv")
    r = RS.apply_counts_sparse(ids, seqs, parts[0], out_scores=out, save_associations=True, chunk_rows=9, query_kmers=kmerlist)
    rows, cols, S = _read_scores(out)
    assert rows == [str(x) for x in d["apply_rows"]] and cols == [str(x) for x in d["apply_cols"]] == r.annotations
    assert np.max(np.abs(S - d["apply_scores"])) < 1e-12
    plain = RS.apply_counts_sparse(ids, seqs, parts[0], query_kmers=kmerlist)
    assert np.array_equal(plain.top1, r.top1) and np.array_equal(plain.score1, r.score1)
    assert np.array_equal(plain.score2, r.score2, equal_nan=True)
    side = str(tmp_path / "apply.skma")
    RS.apply_counts_sparse(ids, seqs, parts[0], out_scores=side, save_associations=True, query_kmers=kmerlist)
    SC.export_associations_csv(side, str(tmp_path / "apply.export.csv"))
    assert open(tmp_path / "apply.export.csv", "rb").read() == open(out, "rb").read()
    # without save_associations there is no association file
    none = str(tmp_path / "none.csv")
    RS.apply_counts_sparse(ids, seqs, parts[0], out_scores=none, query_kmers=kmerlist)
    assert not os.path.exists(none)


def _edge(s1, s2):
    return np.abs(((s1 - s2) * 100) % 1 - 0.5) < 1e-7


def test_c1_association_files_and_csv_evaluator(tmp_path):
    d = np.load(os.path.join(C1, "c1_golden.npz"))
    seq_annot = R.load_annotations([os.path.join(C1, "c1.ann")])
    a, k = 2, 8
    parts, frames = [], {}
    for nb in C1_FILES:
        npz = str(tmp_path / f"{nb}.npz")
        R.vectorize_rule(os.path.join(C1, nb + ".fasta.gz"), npz, None, a, k)
        kl, df = skio.load_npz(npz)
        kmerlist = [str(x) for x in kl[0]]
        frames[nb] = (df, kmerlist)
        parts.append(RS.learn_counts_sparse(list(df["sequence_id"]), list(df["sequence"]), "".join(sorted(set("".join(kmerlist)))), k,
                                            seq_annot))
    merged = RS.merge_counts_sparse(parts)
    evs, masked, edge = [], [], False
    for nb in C1_FILES:
        df, kmerlist = frames[nb]
        ev, m = _check_eval_files(tmp_path, nb, list(df["sequence_id"]), list(df["sequence"]), merged, seq_annot, kmerlist,
                                  d[f"{nb}_eval_rows"], d[f"{nb}_eval_cols"], d[f"{nb}_eval_scores"], 1000)
        evs.append(ev)
        masked.append(m)
        edge |= bool(_edge(ev.score1.cpu().numpy(), ev.score2.cpu().numpy()).any())
    df, kmerlist = frames[C1_FILES[1]]
    out = str(tmp_path / "apply.csv")
    RS.apply_counts_sparse(list(df["sequence_id"]), list(df["sequence"]), parts[0], out_scores=out, save_associations=True,
                           query_kmers=kmerlist)
    rows, cols, S = _read_scores(out)
    assert rows == [str(x) for x in d["apply_rows"]] and cols == [str(x) for x in d["apply_cols"]]
    assert np.max(np.abs(S - d["apply_scores"])) < 1e-12
    # the stock CSV Evaluator over the sparse-written top-2 files == evaluate_sparse over the same rows
    c_csv, g_csv = str(tmp_path / "confidence-matrix-csv.csv"), str(tmp_path / "global-confidence-scores-csv.csv")
    c_sp, g_sp = str(tmp_path / "confidence-matrix-sparse.csv"), str(tmp_path / "global-confidence-scores-sparse.csv")
    got = R.evaluate_rule(masked, c_csv, g_csv)
    want = RS.evaluate_sparse(evs, c_sp, g_sp)
    assert want.weight[0] > 0
    if not edge:
        assert got.rows == want.rows
        for f in ("ratio", "confidence", "weight", "sum"):
            assert np.array_equal(getattr(got, f), getattr(want, f), equal_nan=True), f
        assert open(g_csv, "rb").read() == open(g_sp, "rb").read()
        assert open(c_csv, "rb").read() == open(c_sp, "rb").read()
    else:
        assert abs(got.weight[0] - want.weight[0]) <= 8
