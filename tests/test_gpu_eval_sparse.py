"""GPU: the sparse eval_apply / evaluate rule bodies (rules_sparse.eval_counts_sparse, evaluate_sparse) and the row
classes decided on the device (skm_confidence_classify) against the host classifier, the dense rule chain, the
reference's C1 files and the numpy oracle."""
import os

import numpy as np
import pandas as pd
import pytest
import torch

from learn_coo_oracle import annotation_ids, basis_columns, coo_dense, learn_coo, merge
from oracle import skm_evaluator as EV
from oracle import skm_oracle as O
from util import GOLDEN, read_fasta

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from snekmer_b200 import confidence as CF
    from snekmer_b200 import engine as E
    from snekmer_b200 import io as skio
    from snekmer_b200 import rules as R
    from snekmer_b200 import rules_sparse as RS

C1 = os.path.join(GOLDEN, "c1")
C1_FILES = ["UP000322080_2603819", "UP000322981_424902"]

# names whose substring relations with each other and with "_known_<digits>" are the hard cases of learn.smk:997-1008
ADVERSARIAL = ["TIGR0001", "TIGR00012", "1", "_k", "known_1", "n_", "7_", "", "unknown", "xunknownx", "α", "αβ",
               "Z" * 150 + "αβ" * 25 + "Y" * 50, "TIGR00010", "0", "_known_", "wn_12"]
FILE_ONLY = ["TIGR000123", "β", "known", "TIGR0001x", "unknownTIGR0001"]     # eval-file annotations no matrix row has


def adversarial_rows(n, seed=0, row_base=999_999_999_000):
    """(names, A, top1, truth, row_base, labels): names = the matrix's A annotations + file-only names."""
    rng = np.random.default_rng(seed)
    names, A = ADVERSARIAL + FILE_ONLY, len(ADVERSARIAL)
    top1 = rng.integers(-1, A, size=n).astype(np.int32)
    truth = rng.integers(-1, len(names), size=n).astype(np.int32)
    same = rng.random(n) < 0.3
    truth[same] = np.maximum(top1[same], -1)
    labels = [f"{names[t]}_known_{row_base + q}" if t >= 0 else f"TIGR0001{q % 7}_unknown_{row_base + q}"
              for q, t in enumerate(truth)]
    return names, A, top1, truth, row_base, labels


def test_classify_kernel_equals_classify_rows():
    n = 120_000
    names, A, top1, truth, row_base, labels = adversarial_rows(n)
    d_top1, d_truth = torch.from_numpy(top1).cuda(), torch.from_numpy(truth).cuda()
    got = CF.classify_device(d_top1, d_truth, row_base, names).cpu().numpy()
    want = CF.classify_rows(top1, labels, names[:A])
    assert np.array_equal(got, want)
    assert (want == 0).any() and (want == 1).any() and (want == 2).any()
    # the truth shortcut (rows whose label comes from a matrix annotation or is unknown)
    m = truth < A
    assert np.array_equal(got[m], CF.classify_rows(top1[m], [labels[i] for i in np.flatnonzero(m)], names[:A], truth[m]))
    # row numbers near 2^63 - 1 (19 digits), a shard that starts mid-file, one row
    for base in ((1 << 63) - 1 - 5000, 17, 0):
        q = 5000
        lab = [f"{names[t]}_known_{base + i}" if t >= 0 else f"x_unknown_{base + i}" for i, t in enumerate(truth[:q])]
        got = CF.classify_device(d_top1[:q], d_truth[:q], base, names).cpu().numpy()
        assert np.array_equal(got, CF.classify_rows(top1[:q], lab, names[:A]))
    assert CF.classify_device(d_top1[:0], d_truth[:0], 0, names).numel() == 0
    # no names at all: every row unknown
    none = torch.full((10,), -1, dtype=torch.int32, device="cuda")
    assert CF.classify_device(none, none, 0, []).sum().item() == 0


# ---- helpers -------------------------------------------------------------------------------------------------------
def _labels(ev, ids, seq_annot):
    """The eval_apply labels of an EvalScores' rows, built the way the dense rule builds them."""
    uniq, _ = R._unique_last(list(ids))
    out = []
    for n, sid in enumerate(uniq):
        acc = R._ACCESSION.findall(sid)[0]
        out.append(f"{seq_annot[acc]}_known_{ev.row_base + n}" if acc in seq_annot else f"{acc}_unknown_{ev.row_base + n}")
    return out


def _score_result(ev, labels):
    return R.ScoreResult(labels, list(ev.annotations), ev.top1.cpu().numpy(), ev.top2.cpu().numpy(), ev.score1.cpu().numpy(),
                         ev.score2.cpu().numpy(), None)


def _same_result(a, b):
    assert a.rows == b.rows and a.zero_negative == b.zero_negative
    assert a.weight_is_int == b.weight_is_int and a.sum_is_int == b.sum_is_int
    for f in ("ratio", "confidence", "weight", "sum"):
        assert np.array_equal(getattr(a, f), getattr(b, f), equal_nan=True), f


def _files(tmp_path, tag):
    return str(tmp_path / f"confidence-matrix-{tag}.csv"), str(tmp_path / f"global-confidence-scores-{tag}.csv")


def _edge(s1, s2):
    """Rows whose Difference sits on a rounding boundary of round(., 2)."""
    return np.abs(((s1 - s2) * 100) % 1 - 0.5) < 1e-7


def _bins(top1, s1, s2, n_ann):
    return CF.difference_bins(torch.from_numpy(np.ascontiguousarray(top1, dtype=np.int32)).cuda(),
                              torch.from_numpy(np.ascontiguousarray(s1)).cuda(), torch.from_numpy(np.ascontiguousarray(s2)).cuda(),
                              n_ann).cpu().numpy()


# ---- C1: the sparse chain against the dense chain and the reference's files ----------------------------------------
def test_c1_sparse_chain_matches_dense_chain_and_reference(tmp_path):
    d = np.load(os.path.join(C1, "c1_golden.npz"))
    ann = [os.path.join(C1, "c1.ann")]
    seq_annot = R.load_annotations(ann[:1])
    a, k = 2, 8
    parts, counts, frames = [], [], {}
    for nb in C1_FILES:
        npz = str(tmp_path / f"{nb}.npz")
        R.vectorize_rule(os.path.join(C1, nb + ".fasta.gz"), npz, None, a, k)
        kl, df = skio.load_npz(npz)
        kmerlist = [str(x) for x in kl[0]]
        frames[nb] = (df, kmerlist)
        symbols = "".join(sorted(set("".join(kmerlist))))
        parts.append(RS.learn_counts_sparse(list(df["sequence_id"]), list(df["sequence"]), symbols, k, seq_annot))
        out = str(tmp_path / f"kmer-counts-{nb}.csv")
        R.learn_rule(npz, ann, out)
        counts.append(out)
    merged = RS.merge_counts_sparse(parts)
    tot = str(tmp_path / "kmer-counts-total.csv")
    R.merge_rule(counts, tot)
    evs, dense = [], []
    moved = 0
    for nb in C1_FILES:
        df, kmerlist = frames[nb]
        ids = list(df["sequence_id"])
        ev = RS.eval_counts_sparse(ids, list(df["sequence"]), merged, seq_annot, query_kmers=kmerlist)
        dr = R.eval_apply_rule(str(tmp_path / f"{nb}.npz"), ann, tot, str(tmp_path / f"seq-annotation-scores-{nb}.csv"))
        assert ev.annotations == dr.annotations and ev.row_base == 0
        labels = _labels(ev, ids, seq_annot)
        assert labels == dr.rows
        evs.append(ev)
        dense.append(dr)
        t1, s1, s2 = ev.top1.cpu().numpy(), ev.score1.cpu().numpy(), ev.score2.cpu().numpy()
        assert np.max(np.abs(s1 - dr.score1)) < 1e-12 and np.nanmax(np.abs(s2 - dr.score2)) < 1e-12
        clear = (dr.score1 - dr.score2) > 1e-9
        assert np.array_equal(t1[clear], dr.top1[clear])
        cls = CF.classify_device(ev.top1, ev.truth, ev.row_base, ev.names).cpu().numpy()
        dcls = CF.classify_rows(dr.top1, dr.rows, dr.annotations)
        assert np.array_equal(cls[clear], dcls[clear])
        bins = _bins(t1, s1, s2, len(ev.annotations))
        dbins = _bins(dr.top1, dr.score1, dr.score2, len(ev.annotations))
        edge = _edge(s1, s2) | _edge(dr.score1, dr.score2)
        assert np.array_equal(bins[~edge], dbins[~edge])
        counted = ((cls > 0) & (bins != 255)) | ((dcls > 0) & (dbins != 255))
        moved += int((((bins != dbins) | (t1 != dr.top1) | (cls != dcls)) & counted).sum())
    conf, glob = _files(tmp_path, "sparse")
    got = RS.evaluate_sparse(evs, conf, glob, modifier=20)
    dconf, dglob = _files(tmp_path, "dense")
    want = R.evaluate_results(dense, dconf, dglob, modifier=20)
    if moved == 0:
        _same_result(got, want)
        assert open(glob, "rb").read() == open(dglob, "rb").read()
        assert open(conf, "rb").read() == open(dconf, "rb").read()
    # the reference's own files (the assertions of test_c1_rule_chain_reproduces_reference)
    g = pd.read_csv(glob)
    w = pd.read_csv(pd.io.common.BytesIO(d["global_confidence_csv"].tobytes()))
    ref_moved = int(np.abs(g["sum"].values - w["sum"].values).sum())
    assert ref_moved <= 8, ref_moved
    assert np.array_equal(g["weight"].values, w["weight"].values)
    assert np.nanmax(np.abs(g["confidence"].values - w["confidence"].values)) < 5e-3
    if ref_moved == 0:
        assert open(glob, "rb").read() == d["global_confidence_csv"].tobytes()
        assert open(conf, "rb").read() == d["confidence_matrix_csv"].tobytes()


# ---- a column-keyed code space against the numpy oracle --------------------------------------------------------------
def test_wide_sparse_chain_matches_oracle(tmp_path):
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
        symbols = "".join(sorted(set("".join(kmers))))
        assert len(symbols) ** k > E._native.SKM_DENSE_MAX_SPACE
        parts.append(RS.learn_counts_sparse(ids, reduced, symbols, k, seq_annot))
    merged = RS.merge_counts_sparse(parts)
    assert merged.columns is not None
    rows, cols, Mm, *_ = merge([f["part"] for f in files.values()])
    assert merged.annotations == rows
    code_of = {}
    for f in files.values():
        code_of.update(zip(f["part"][1], f["basis"]))
    col_codes = np.array([code_of[km] for km in cols], dtype=np.uint64)
    evs, oracle_files, edge_any = [], [], False
    for nb, f in files.items():
        ev = RS.eval_counts_sparse(f["ids"], f["reduced"], merged, seq_annot)
        uniq, pick = R._unique_last(f["ids"])
        si, code, valid = f["windows"]
        C_all = O.count_matrix(si, code, valid, f["n"], f["basis"])[pick].astype(np.int64)
        at = basis_columns(col_codes, f["basis"])                 # union column -> this file's basis column
        Q = np.zeros((len(pick), len(cols)), dtype=np.int64)
        Q[:, at >= 0] = C_all[:, at[at >= 0]]
        S = O.cosine_scores(Q, Mm, (C_all * C_all).sum(axis=1))
        labels = _labels(ev, f["ids"], seq_annot)
        oracle_files.append((S, labels, rows))
        ht, hf, pred, bins, tf, known, diff = EV.file_tables(S, labels, rows)
        _, top, second = EV.top_two_values(S)
        s1, s2, t1 = ev.score1.cpu().numpy(), ev.score2.cpu().numpy(), ev.top1.cpu().numpy()
        assert np.max(np.abs(s1 - top)) < 1e-12 and np.nanmax(np.abs(s2 - second)) < 1e-12
        clear = (top - second) > 1e-9
        assert clear.any() and np.array_equal(t1[clear], pred[clear])
        cls = CF.classify_device(ev.top1, ev.truth, ev.row_base, ev.names).cpu().numpy()
        ocls = np.where(known, np.where(tf, 1, 2), 0).astype(np.uint8)
        assert np.array_equal(cls[clear], ocls[clear])
        gbins = _bins(t1, s1, s2, len(rows))
        edge = _edge(s1, s2) | _edge(top, second)
        obins = np.where(bins < 0, 255, bins)
        assert np.array_equal(gbins[~edge & clear], obins[~edge & clear])
        edge_any |= bool((edge | ~clear)[ocls > 0].any())
        evs.append(ev)
    got = RS.evaluate_sparse(evs)
    want = EV.evaluate(oracle_files)
    assert got.weight[0] > 0
    if not edge_any:
        assert got.rows == want["rows"] and got.zero_negative == want["zero_negative"]
        for f in ("ratio", "confidence", "weight", "sum"):
            assert np.array_equal(getattr(got, f), want[f], equal_nan=True), f
    else:
        assert abs(got.weight[0] - want["weight"][0]) <= 8


# ---- side-cars, prior confidence, edge cases -------------------------------------------------------------------------
def _syn_files(a=2):
    syms = O.build_lut(a)[1]
    out = {}
    for nb in ("synA", "synB"):
        ids, seqs = read_fasta(os.path.join(GOLDEN, f"{nb}.fasta"))
        out[nb] = (ids, [O.reduce_str(s, a) for s in seqs])
    return out, syms, R.load_annotations([os.path.join(GOLDEN, "syn.ann")])


def _chain(files, symbols, k, learn_annot, eval_annot, tmp_path=None):
    parts = [RS.learn_counts_sparse(ids, red, symbols, k, learn_annot) for ids, red in files.values()]
    merged = RS.merge_counts_sparse(parts)
    evs = []
    for nb, (ids, red) in files.items():
        side = str(tmp_path / f"{nb}.skme") if tmp_path is not None else None
        evs.append(RS.eval_counts_sparse(ids, red, merged, eval_annot, out_sidecar=side))
    return merged, evs


def _dense_twin(evs, ids_and_annots):
    """The same rows as ScoreResults with their labels as strings, for the host classifier (evaluate_results)."""
    return [_score_result(ev, _labels(ev, ids, annot)) for ev, (ids, annot) in zip(evs, ids_and_annots)]


def test_sidecars_and_prior_confidence(tmp_path):
    files, symbols, seq_annot = _syn_files()
    _, evs = _chain(files, symbols, 4, seq_annot, seq_annot, tmp_path)
    sides = [str(tmp_path / f"{nb}.skme") for nb in files]
    back = RS.read_eval_sidecar(sides[0])
    assert back.annotations == evs[0].annotations and back.names == evs[0].names and back.row_base == evs[0].row_base
    for f in ("top1", "top2", "score1", "score2", "truth"):
        assert torch.equal(getattr(back, f), getattr(evs[0], f)), f
    c_mem, g_mem = _files(tmp_path, "mem")
    c_side, g_side = _files(tmp_path, "side")
    r_mem = RS.evaluate_sparse(evs, c_mem, g_mem)
    r_side = RS.evaluate_sparse(sides, c_side, g_side)
    _same_result(r_mem, r_side)
    assert open(g_mem, "rb").read() == open(g_side, "rb").read() and open(c_mem, "rb").read() == open(c_side, "rb").read()
    assert r_mem.weight[0] > 0
    # the same rows through the host classifier (labels as strings): identical results and files
    twin = _dense_twin(evs, [(ids, seq_annot) for ids, _ in files.values()])
    c_d, g_d = _files(tmp_path, "dense")
    _same_result(r_mem, R.evaluate_results(twin, c_d, g_d))
    assert open(g_mem, "rb").read() == open(g_d, "rb").read() and open(c_mem, "rb").read() == open(c_d, "rb").read()
    # prior confidence merged with weight modifier 3.5 (the prior: synB's curve alone)
    prior = str(tmp_path / "prior.csv")
    RS.evaluate_sparse(sides[1:], None, prior)
    c_p, g_p = _files(tmp_path, "prior-sparse")
    c_q, g_q = _files(tmp_path, "prior-dense")
    rp = RS.evaluate_sparse(sides, c_p, g_p, base_confidence=[prior], modifier=3.5)
    rq = R.evaluate_results(twin, c_q, g_q, base_confidence=[prior], modifier=3.5)
    _same_result(rp, rq)
    assert open(g_p, "rb").read() == open(g_q, "rb").read() and open(c_p, "rb").read() == open(c_q, "rb").read()
    assert not np.array_equal(rp.weight, r_mem.weight)


def test_edge_cases_match_dense_path(tmp_path):
    files, symbols, seq_annot = _syn_files()
    k = 4

    def both(evs, ids_and_annots, tag):
        c_s, g_s = _files(tmp_path, tag + "-s")
        c_d, g_d = _files(tmp_path, tag + "-d")
        rs = RS.evaluate_sparse(evs, c_s, g_s)
        rd = R.evaluate_results(_dense_twin(evs, ids_and_annots), c_d, g_d)
        _same_result(rs, rd)
        assert open(g_s, "rb").read() == open(g_d, "rb").read() and open(c_s, "rb").read() == open(c_d, "rb").read()
        return rs

    merged, evs = _chain(files, symbols, k, seq_annot, seq_annot)
    known = [(ids, seq_annot) for ids, _ in files.values()]
    # an empty file, first and alone
    empty = RS.eval_counts_sparse([], [], merged, seq_annot)
    assert empty.top1.numel() == 0 and empty.row_base == 0
    r = both([empty] + evs, [([], seq_annot)] + known, "empty-first")
    assert r.weight[0] > 0
    r = both([empty], [([], seq_annot)], "empty-only")
    assert r.rows == [] and r.weight[0] == 0
    # a file without a Known row (its accessions are in no annotation file): alone, and first of three
    ids_b, red_b = files["synB"]
    none = RS.eval_counts_sparse(ids_b, red_b, merged, {})
    assert int(none.truth.max()) == -1 and none.names == merged.annotations
    r = both([none], [(ids_b, {})], "no-known")
    assert r.weight[0] == 0
    both([none] + evs, [(ids_b, {})] + known, "no-known-first")
    # every row Unknown: every annotation name contains "unknown"
    renamed = {acc: f"unknown-{a}" for acc, a in seq_annot.items()}
    _, evs_u = _chain(files, symbols, k, renamed, renamed)
    r = both(evs_u, [(ids, renamed) for ids, _ in files.values()], "all-unknown")
    assert r.weight[0] == 0 and r.rows == []
    # one annotation: no runner-up, every Difference undefined (bin 255) as in the dense path and the oracle
    single = {acc: "TIGR00001" for acc in seq_annot}
    _, evs_1 = _chain(files, symbols, k, single, single)
    assert len(evs_1[0].annotations) == 1 and int(evs_1[0].top2.max()) == -1
    r = both(evs_1, [(ids, single) for ids, _ in files.values()], "one-annotation")
    want = EV.evaluate([(ev.score1.cpu().numpy()[:, None], _labels(ev, ids, single), ev.annotations)
                        for ev, (ids, _) in zip(evs_1, files.values())])
    assert r.weight[0] == want["weight"][0] == 0 and r.rows == want["rows"] == []
