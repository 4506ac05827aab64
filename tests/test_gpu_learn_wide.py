"""GPU: learn and apply over code spaces beyond the 2^27 tables (engine.learn_wide / query_csr_wide / apply_wide, the
wide dispatch of the sparse rule bodies, skm_csc_build over more than 2^27 columns) against the numpy oracle.
Bit-exact unless stated."""
import os

import numpy as np
import pytest
import torch

from learn_coo_oracle import annotation_ids, basis_columns, coo_dense, learn_coo, merge
from oracle import skm_oracle as O
from util import GOLDEN, read_ann, read_fasta

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from snekmer_b200 import engine as E
    from snekmer_b200 import rules as R
    from snekmer_b200 import rules_sparse as RS
    from snekmer_b200 import sidecar as SC


def _rand_seqs(rng, n, lo=0, hi=500, p_x=0.002):
    aa = np.array(list("ACDEFGHIKLMNPQRSTVWYXBZUO*acd"))
    p = np.array([1.0] * 20 + [p_x * 20] * 9)
    p /= p.sum()
    return ["".join(rng.choice(aa, size=int(rng.integers(lo, hi)), p=p)) for _ in range(n)]


def _windows(seqs, a, k):
    lut, syms = O.build_lut(a)
    res, offs = O.pack(seqs)
    return O.window_codes(res, offs, lut, len(syms), k)


def _np(t):
    return t.cpu().numpy()


def _check(got, want):
    keys, vals, totals = got
    wk, wv, wt = want
    assert np.array_equal(_np(keys), wk)
    assert np.array_equal(_np(vals), wv)
    assert np.array_equal(_np(totals), wt)


# (alphabet, k): 20^7 just past the tables, 20^8, 20^14, 30^12 (ptm), 2^32 (hydro: the all-ones fill's low bits tie
# with the largest code of a power-of-two space), 3^40 (> 2^63)
CASES = [(None, 7), (None, 8), (None, 14), ("ptm", 12), (0, 32), (3, 40)]


@pytest.mark.parametrize("a,k", CASES)
@pytest.mark.parametrize("mf", [0, 2])
def test_learn_wide_matches_oracle(a, k, mf):
    rng = np.random.default_rng(k * 13 + mf)
    seqs = _rand_seqs(rng, 500, 0, 500)
    seqs += [s[: len(s) // 3] * 3 for s in seqs[:80]] + ["", "A", "ACDEFG"]       # repeats, short and empty sequences
    n_ann = 37
    ann = rng.integers(-1, n_ann + 3, size=len(seqs)).astype(np.int32)          # -1 and >= n_ann: the rest row
    si, pos, code, valid = _windows(seqs, a, k)
    basis_o, _ = O.basis_codes(si, pos, code, valid, mf)
    want = learn_coo(si, code, valid, ann, n_ann, basis_o)
    batch = E.SequenceBatch.from_strings(seqs)
    basis = E.build_basis_wide(batch, a, k, mf)
    assert np.array_equal(basis.codes_host(), basis_o)
    got = E.learn_wide(batch, a, k, basis, torch.from_numpy(ann), n_ann)
    _check(got, want)
    # a chunked shard (lists of the chunks merged) == one chunk
    _check(E.learn_wide(batch, a, k, basis, torch.from_numpy(ann), n_ann, max_chunk_res=9000), want)


def test_learn_wide_degenerate_inputs():
    a, k = None, 8
    rng = np.random.default_rng(4)
    seqs = _rand_seqs(rng, 200, 0, 300)
    si, pos, code, valid = _windows(seqs, a, k)
    batch = E.SequenceBatch.from_strings(seqs)
    basis = E.build_basis_wide(batch, a, k, 0)
    basis_o, _ = O.basis_codes(si, pos, code, valid, 0)
    # all unannotated: an empty matrix, Totals over everything
    none = np.full(len(seqs), -1, dtype=np.int32)
    _check(E.learn_wide(batch, a, k, basis, torch.from_numpy(none), 5), learn_coo(si, code, valid, none, 5, basis_o))
    # n_ann = 0: every sequence is in the rest row
    ann = rng.integers(0, 4, size=len(seqs)).astype(np.int32)
    _check(E.learn_wide(batch, a, k, basis, torch.from_numpy(ann), 0), learn_coo(si, code, valid, ann, 0, basis_o))
    # no sequences
    empty = E.SequenceBatch.from_strings([])
    keys, vals, totals = E.learn_wide(empty, a, k, basis, torch.zeros(0, dtype=torch.int32), 3)
    assert keys.numel() == 0 and vals.numel() == 0 and torch.equal(totals, torch.zeros(basis.K, dtype=torch.int64, device="cuda"))
    # sequences shorter than k
    short = E.SequenceBatch.from_strings(["ACDEFGH", "", "AC"])
    keys, vals, totals = E.learn_wide(short, a, k, basis, torch.zeros(3, dtype=torch.int32), 1)
    assert keys.numel() == 0 and int(totals.sum()) == 0
    # an empty basis
    b0 = E.build_basis_wide(short, a, k, 0)
    assert b0.K == 0
    keys, vals, totals = E.learn_wide(batch, a, k, b0, torch.from_numpy(ann), 4)
    assert keys.numel() == 0 and totals.numel() == 0


@pytest.mark.parametrize("a,k,mf", [(None, 8, 1), ("ptm", 12, 0), (5, 3, 0), (2, 8, 1)])
def test_learn_wide_equals_existing_compositions(a, k, mf):
    """learn_wide == count_csr_wide over the basis -> ann * K + col per entry in torch -> coo_merge (the composition of
    existing entry points), and on table-space alphabets == learn_sparse_with_totals gathered onto the basis columns."""
    rng = np.random.default_rng(k + 31)
    seqs = _rand_seqs(rng, 800, 0, 500)
    n_ann = 60
    ann = rng.integers(-1, n_ann, size=len(seqs)).astype(np.int32)
    batch = E.SequenceBatch.from_strings(seqs)
    basis = E.build_basis_wide(batch, a, k, mf)
    K = basis.K
    keys, vals, totals = E.learn_wide(batch, a, k, basis, torch.from_numpy(ann), n_ann)
    rowptr, _, cols, cvals = E.count_csr_wide(batch, a, k, basis)
    d_ann = torch.from_numpy(ann).cuda().to(torch.int64)
    row = torch.repeat_interleave(torch.arange(len(seqs), device="cuda"), rowptr[1:] - rowptr[:-1])
    ra = d_ann[row]
    ra = torch.where(ra < 0, torch.full_like(ra, n_ann), ra)
    bk, bv = E.coo_merge(ra * K + cols.to(torch.int64), cvals.to(torch.int64), key_bound=(n_ann + 1) * K)
    m = int((bk < n_ann * K).sum())
    assert torch.equal(keys, bk[:m]) and torch.equal(vals, bv[:m])
    bt = torch.zeros(K, dtype=torch.int64, device="cuda").index_add_(0, bk % K, bv)
    assert torch.equal(totals, bt)
    tab = E.alphabet_tables(a)
    S = E.code_space(tab.nsym, k)
    if S <= E._native.SKM_DENSE_MAX_SPACE:
        tk, tv, tt = E.learn_sparse_with_totals(batch, a, k, torch.from_numpy(ann), n_ann)
        col_of_code = torch.full((S,), -1, dtype=torch.int64, device="cuda")
        col_of_code[basis.codes] = torch.arange(K, device="cuda")
        c = col_of_code[tk % S]
        keep = c >= 0
        gk = (tk // S)[keep] * K + c[keep]
        order = torch.argsort(gk)
        assert torch.equal(keys, gk[order]) and torch.equal(vals, tv[keep][order])
        assert torch.equal(totals, tt[basis.codes])


def test_csc_build_beyond_table_columns():
    """skm_csc_build with S > 2^27 columns (a matrix keyed by basis column) against numpy."""
    rng = np.random.default_rng(9)
    S, n_ann, nnz = (1 << 28) + 3, 40, 300000
    ann = rng.integers(0, n_ann, size=nnz)
    col = np.concatenate([rng.integers(0, S, size=nnz - 3), [0, S - 1, S - 1]])
    keys = np.unique(ann * S + col)
    vals = rng.integers(1, 1000, size=keys.size).astype(np.int64)
    d_keys, d_vals = torch.from_numpy(keys).cuda(), torch.from_numpy(vals).cuda()
    csc = E.csc_build(d_keys, d_vals, S, n_ann, 0, pack=False)
    a, c = keys // S, keys % S
    order = np.lexsort((a, c))
    assert np.array_equal(_np(csc.rows), a[order]) and np.array_equal(_np(csc.mvals), vals[order])
    probe = np.unique(np.concatenate([c, c + 1, [0, S], rng.integers(0, S + 1, size=1000)]))
    probe = probe[probe <= S]
    colptr = _np(csc.colptr[torch.from_numpy(probe).cuda()])
    assert np.array_equal(colptr, np.searchsorted(np.sort(c), probe, side="left"))
    assert int(csc.colptr[-1]) == keys.size
    n2 = np.zeros(n_ann, dtype=np.float64)
    np.add.at(n2, a, (vals * vals).astype(np.float64))
    assert np.array_equal(_np(csc.mnorm2), n2)
    # the slice of annotations [10, 30)
    sl = E.csc_build(d_keys, d_vals, S, 20, 10, pack=False)
    m = (a >= 10) & (a < 30)
    o2 = np.lexsort((a[m], c[m]))
    assert np.array_equal(_np(sl.rows), (a[m] - 10)[o2]) and int(sl.colptr[-1]) == int(m.sum())


# ---- the rule bodies at (None, 8) on the golden files -----------------------------------------------------------
def _oracle_file(nb, a, k, seq_annot, mf=0):
    ids, seqs = read_fasta(os.path.join(GOLDEN, f"{nb}.fasta"))
    lut, syms = O.build_lut(a)
    si, pos, code, valid = _windows(seqs, a, k)
    basis, _ = O.basis_codes(si, pos, code, valid, mf)
    ann_id, anns = annotation_ids(ids, seq_annot)
    keys, vals, totals = learn_coo(si, code, valid, ann_id, len(anns), basis)
    M = coo_dense(keys, vals, len(anns), len(basis))
    seq_count = np.bincount(ann_id[ann_id >= 0], minlength=len(anns)).astype(np.int64)
    kmers = [str(x) for x in O.decode(basis, syms, k)]
    return dict(ids=ids, seqs=seqs, reduced=[O.reduce_str(s, a) for s in seqs], anns=anns, kmers=kmers, M=M,
                seq_count=seq_count, totals=totals, total_seqs=len(set(ids)), windows=(si, code, valid), basis=basis)


def _dense_of(sc, kmers):
    """M [A, len(kmers)] and totals of a wide SparseCounts over the given k-mer strings."""
    learned = [str(x) for x in sc.columns.kmers()]
    pos = {km: i for i, km in enumerate(learned)}
    full = coo_dense(_np(sc.keys), _np(sc.vals), len(sc.annotations), sc.columns.K)
    idx = np.array([pos[km] for km in kmers], dtype=np.int64)
    return full[:, idx], _np(sc.totals)[idx], learned


def test_wide_rule_bodies_match_oracle(tmp_path):
    a, k = None, 8
    seq_annot = R.load_annotations([os.path.join(GOLDEN, "syn.ann")])
    assert seq_annot == read_ann(os.path.join(GOLDEN, "syn.ann"))
    files = {nb: _oracle_file(nb, a, k, seq_annot) for nb in ("synA", "synB")}
    parts = []
    for nb, f in files.items():
        symbols = "".join(sorted(set("".join(f["kmers"]))))
        assert len(symbols) ** k > E._native.SKM_DENSE_MAX_SPACE
        sc = RS.learn_counts_sparse(f["ids"], f["reduced"], symbols, k, seq_annot)
        assert sc.columns is not None and sc.stride == sc.columns.K == len(f["kmers"])
        assert sc.annotations == f["anns"] and np.array_equal(sc.seq_count, f["seq_count"]) and sc.total_seqs == f["total_seqs"]
        # the columns are the k-mers that occur, in first-occurrence order: the file's kmerlist
        M, totals, learned = _dense_of(sc, f["kmers"])
        assert learned == f["kmers"]
        assert np.array_equal(M, f["M"]) and np.array_equal(totals, f["totals"])
        # .skmc with the file's kmerlist -> the learn rule's CSV == the oracle's, byte for byte
        side = str(tmp_path / f"{nb}.skmc")
        RS.write_counts_sidecar(side, sc, kmers=f["kmers"])
        out, ref = tmp_path / f"kmer-counts-{nb}.csv", tmp_path / f"oracle-{nb}.csv"
        SC.export_counts_csv(side, str(out))
        R.write_counts_csv(str(ref), R.LearnResult(f["anns"], f["seq_count"], f["M"], f["totals"], f["total_seqs"], f["kmers"]))
        assert out.read_bytes() == ref.read_bytes()
        # the side-car round trip: back to the device unchanged
        side2 = str(tmp_path / f"{nb}.cols.skmc")
        RS.write_counts_sidecar(side2, sc)
        back = RS.read_counts_sidecar(side2, symbols=sc.symbols)
        assert back.columns is not None and torch.equal(back.columns.codes, sc.columns.codes)
        assert back.annotations == sc.annotations and torch.equal(back.keys, sc.keys) and torch.equal(back.vals, sc.vals)
        assert torch.equal(back.totals, sc.totals) and back.total_seqs == sc.total_seqs and np.array_equal(back.seq_count, sc.seq_count)
        parts.append(sc)
    # merge == the oracle merge: row order, column order, values
    merged = RS.merge_counts_sparse(parts)
    rows, cols, Mm, seq_count, totals, total_seqs = merge([(f["anns"], f["kmers"], f["M"], f["seq_count"], f["totals"], f["total_seqs"])
                                                           for f in files.values()])
    assert merged.annotations == rows and np.array_equal(merged.seq_count, seq_count) and merged.total_seqs == total_seqs
    got_M, got_t, learned = _dense_of(merged, cols)
    assert learned == cols
    assert np.array_equal(got_M, Mm) and np.array_equal(got_t, totals)
    # apply against the matrix learned on synA: cosine over the union columns, query norm over all valid windows.  synB
    # shares almost no 8-mer with synA (every score ties at 0); synA's own records have clear winners.
    A = files["synA"]
    for nb, clear_winners in (("synB", False), ("synA", True)):
        Q_ = files[nb]
        uniq, pick = R._unique_last(Q_["ids"])
        r = RS.apply_counts_sparse(Q_["ids"], Q_["reduced"], parts[0])
        si, code, valid = Q_["windows"]
        C_all = O.count_matrix(si, code, valid, len(Q_["seqs"]), Q_["basis"])[pick].astype(np.int64)
        Q = O.count_matrix(si, code, valid, len(Q_["seqs"]), A["basis"])[pick]
        _assert_scores(r, O.cosine_scores(Q, A["M"], (C_all * C_all).sum(axis=1)), uniq, A["anns"], clear_winners)
    # synA's queries restricted to their own kmerlist (a min_filter = 1 list): norm and dots over that list only
    si, code, valid = A["windows"]
    uniq, pick = R._unique_last(A["ids"])
    kl_codes, _ = O.basis_codes(si, None, code, valid, 1)
    kl = [str(x) for x in O.decode(kl_codes, O.build_lut(a)[1], k)]
    r2 = RS.apply_counts_sparse(A["ids"], A["reduced"], parts[0], query_kmers=kl)
    C_kl = O.count_matrix(si, code, valid, len(A["seqs"]), kl_codes)[pick].astype(np.int64)
    in_a = basis_columns(kl_codes, A["basis"])
    Q = np.zeros((len(pick), len(A["basis"])), dtype=np.int64)          # the learned matrix keeps all its columns
    Q[:, in_a[in_a >= 0]] = C_kl[:, in_a >= 0]
    S2 = O.cosine_scores(Q, A["M"], (C_kl * C_kl).sum(axis=1))
    _assert_scores(r2, S2, uniq, A["anns"], True)
    assert not np.allclose(r.score1, r2.score1)


def _assert_scores(r, S, rows, anns, clear_winners):
    assert r.rows == rows and r.annotations == anns
    order = np.argsort(-S, axis=1, kind="stable")
    s1 = S[np.arange(len(S)), order[:, 0]]
    s2 = S[np.arange(len(S)), order[:, 1]]
    assert np.max(np.abs(r.score1 - s1)) < 1e-12 and np.max(np.abs(r.score2 - s2)) < 1e-12
    clear = (s1 - s2) > 1e-9
    assert clear.any() or not clear_winners
    assert np.array_equal(r.top1[clear], order[:, 0][clear])
