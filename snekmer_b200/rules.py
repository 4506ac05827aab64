"""rules: the ``run:`` bodies of Snekmer's vectorize / learn / merge / eval_apply /
apply rules on the batch GPU API (same inputs, same output files).

  vectorize_rule   rules/kmerize.smk:67-142
  learn_rule       rules/learn.smk:247-422   (class Library)
  merge_rule       rules/learn.smk:443-594   (class Merge)
  eval_apply_rule  rules/learn.smk:628-887   (class KmerCompare of the learn workflow)
  apply_rule       rules/apply.smk:147-353   (class KmerCompare of the apply workflow)
  evaluate_rule    rules/learn.smk:923-1348  (class Evaluator; device side in confidence.py)

Each rule has an in-memory core (``vectorize_records``, ``learn_counts``,
``merge_tables``, ``cosine_top2``) that returns arrays, and a thin file layer
that reads / writes the reference's formats (``.npz`` keys kmerlist / ids / seqs /
vecs / lengths, ``kmer-counts-*.csv`` with blank zeros and an
``__index_level_0__`` column, pyarrow-written totals / score / summary CSVs).
All arithmetic on sequences and count matrices happens on the device through
``engine``; pandas / pyarrow appear only at the file boundary.
"""
from __future__ import annotations

import csv as _csv
import io as _io
import itertools
import os
import pickle
import re
import sys
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import engine as E
from . import io as skio
from .vectorize import KmerVec

_ACCESSION = re.compile(r"\|(.*?)\|")
INDEX_COL = "__index_level_0__"


# ---------------------------------------------------------------------------
# vectorize
# ---------------------------------------------------------------------------
DENSE_MAX_K = 51200         # widest basis the dense kernels hold (a 200 KB shared-memory row of int32 counters)
VECS_MAX_BYTES = 32 << 30   # largest float64 presence matrix vecs() will materialise on the host


def _dense_envelope_error(what: str, K: int) -> E.SkmError:
    return E.SkmError(-3, f"{what}: a basis of {K} k-mers is outside the dense envelope of the rule bodies (K <= {DENSE_MAX_K}); "
                          "the reference's dense CSV / matrix layout does not scale there either — use the sparse rule bodies "
                          "snekmer_b200.rules_sparse.learn_counts_sparse / merge_counts_sparse / apply_counts_sparse with the "
                          ".skmc / .skmv side-cars (sidecar.py)")


@dataclass
class VectorizeResult:
    kmerlist: np.ndarray        # '<Uk' [K] (or the supplied list)
    ids: List[str]
    seqs: List[str]             # reduced sequences (trailing '*' removed)
    lengths: np.ndarray         # raw lengths, int64 [N]
    counts: Optional[torch.Tensor]      # device int32 [N, K]; vecs = counts > 0 (None when the basis is too wide: see csr)
    csr: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None   # (rowptr int64 [N+1], cols int32 [nnz], vals int32 [nnz])

    def vecs(self) -> np.ndarray:
        """float64 0/1 presence matrix, as the rule stores it (kmerize.smk:112-120)."""
        if self.counts is not None:
            return (self.counts > 0).to(torch.float64).cpu().numpy()
        n, K = len(self.ids), len(self.kmerlist)
        if n * K * 8 > VECS_MAX_BYTES:
            raise MemoryError(f"the dense float64 presence matrix of this shard is {n} x {K} ({n * K * 8 / 2 ** 30:.0f} GiB); "
                              "write the CSR side-car instead (vectorize_rule(out_npz=None, out_sidecar=...))")
        rowptr, cols, _ = (t.cpu().numpy() for t in self.csr)
        out = np.zeros((n, K), dtype=np.float64)
        out[np.repeat(np.arange(n), np.diff(rowptr)), cols] = 1.0
        return out

    def write_sidecar(self, path: str, alphabet, k: int) -> None:
        """Binary side-car (.skmv, sidecar.py) of this shard: COUNTS as CSR instead of the dense float64 presence
        matrix; ``sidecar.export_npz`` turns it back into the rule's .npz."""
        from . import alphabet as _alpha
        from . import sidecar

        name = _alpha.get_alphabet_name(alphabet)
        symbols = _alpha.symbols(name)
        codes, ok = E.encode_kmers([str(x) for x in self.kmerlist], symbols, k)
        assert bool(ok.all()), "a k-mer of the basis does not belong to the alphabet"
        if self.counts is None:
            rowptr, cols, vals = self.csr
            sidecar.write_vectors(path, name, k, symbols, codes, self.ids, self.seqs, self.lengths, rowptr.cpu().numpy(),
                                  cols.to(torch.int32).cpu().numpy(), vals.to(torch.int32).cpu().numpy())
            return
        nz = self.counts.nonzero()
        rowptr = torch.zeros(self.counts.shape[0] + 1, dtype=torch.int64, device=self.counts.device)
        if nz.numel():
            rowptr[1:] = torch.cumsum(torch.bincount(nz[:, 0], minlength=self.counts.shape[0]), 0)
        vals = self.counts[nz[:, 0], nz[:, 1]] if nz.numel() else self.counts.new_zeros(0)
        sidecar.write_vectors(path, name, k, symbols, codes, self.ids, self.seqs, self.lengths, rowptr.cpu().numpy(),
                              nz[:, 1].to(torch.int32).cpu().numpy(), vals.to(torch.int32).cpu().numpy())


def _reduced_strings(batch: E.SequenceBatch, alphabet) -> List[str]:
    red = bytes(E.reduce_bytes(batch, alphabet).cpu().numpy()).decode("latin-1") if batch.nres else ""
    off = batch.offsets_host
    return [red[off[i]:off[i + 1]].rstrip("*") for i in range(batch.n)]


def vectorize_records(ids: Sequence[str], seqs: Sequence[str], alphabet, k: int, min_filter: int = 0,
                      kmerbasis: Optional[Sequence[str]] = None) -> VectorizeResult:
    """Both passes of the vectorize rule for one FASTA shard held in memory as strings."""
    residues, offsets = E.SequenceBatch.pack_host([str(s) for s in seqs])
    return vectorize_packed(ids, residues, offsets, alphabet, k, min_filter, kmerbasis)


def vectorize_packed(ids: Sequence[str], residues: np.ndarray, offsets: np.ndarray, alphabet, k: int, min_filter: int = 0,
                     kmerbasis: Optional[Sequence[str]] = None, pinned: bool = False) -> VectorizeResult:
    """Both passes of the vectorize rule for a packed shard (io.read_fasta_packed's layout): no per-record
    Python objects on the way to the device."""
    batch = E.SequenceBatch.from_packed(residues, offsets, pinned=pinned)
    lengths = np.diff(np.asarray(offsets, dtype=np.int64))
    csr = None
    if kmerbasis is not None:                       # basis.txt branch, kmerize.smk:72-78
        kmerlist = list(kmerbasis)
        if len(kmerlist) > DENSE_MAX_K:
            raise _dense_envelope_error("vectorize with a basis file", len(kmerlist))
        counts = E.count_over_kmers(batch, alphabet, k, kmerlist)
    else:                                           # kmerize.smk:85-104
        tab = E.alphabet_tables(alphabet, batch.device)
        if E.code_space(tab.nsym, k) <= E._native.SKM_DENSE_MAX_SPACE:
            # the occurrence counts only serve the `count > min_filter` test: without a filter the basis ORDER is enough
            basis = E.build_basis(batch, alphabet, k, min_filter, counts=min_filter > 0)
            if basis.K <= DENSE_MAX_K:
                counts = E.count_dense(batch, alphabet, k, basis)
            else:                                   # too wide for dense rows: CSR over the basis columns
                counts, csr = None, E.count_csr(batch, alphabet, k, basis)
        else:                                       # code spaces beyond 2^27: sort-based basis, CSR counts
            v = E.vectorize(batch, alphabet, k, min_filter)
            basis, counts, csr = v.basis, None, (v.rowptr, v.cols, v.vals)
        kmerlist = basis.kmers() if basis.K else np.array([])
    return VectorizeResult(kmerlist, list(ids), _reduced_strings(batch, alphabet), lengths, counts, csr)


def vectorize_rule(fasta: str, out_npz: Optional[str], out_kmerobj: Optional[str], alphabet, k: int, min_filter: int = 0,
                   basis_file: Optional[str] = None, out_sidecar: Optional[str] = None) -> VectorizeResult:
    kmer = KmerVec(alphabet=alphabet, k=k)
    ids, residues, offsets = skio.read_fasta_packed(fasta, pinned=True)      # native multithreaded parser
    kmerbasis = skio.read_kmers(basis_file) if (basis_file and os.path.exists(basis_file)) else None
    r = vectorize_packed(ids, residues, offsets, alphabet, k, 0 if kmerbasis is not None else min_filter, kmerbasis, pinned=True)
    kmer.set_kmer_set(r.kmerlist)
    if out_npz:
        np.savez_compressed(out_npz, kmerlist=r.kmerlist, ids=r.ids, seqs=r.seqs, vecs=r.vecs(), lengths=r.lengths)
    if out_sidecar:
        r.write_sidecar(out_sidecar, alphabet, k)
    if out_kmerobj:
        with open(out_kmerobj, "wb") as f:
            pickle.dump(kmer, f)
    return r


# ---------------------------------------------------------------------------
# learn (Library)
# ---------------------------------------------------------------------------
def load_annotations(files: Sequence[str]) -> Dict[str, str]:
    """accession -> annotation from TSV files with `id` and `TIGRFAMs` columns (learn.smk:277-291)."""
    import pandas as pd

    table = pd.concat([pd.read_table(f) for f in files])
    return dict(zip(table["id"].tolist(), table["TIGRFAMs"].tolist()))


def _kmer_tables(*kmerlists):
    """Device tables for counting windows of REDUCED text against k-mer lists: the symbols
    are the characters the lists use; k is the length of the first k-mer of the first list."""
    chars = set(itertools.chain.from_iterable(itertools.chain.from_iterable(kl) for kl in kmerlists))
    k = len(str(kmerlists[0][0]))
    return E.alphabet_tables_from_symbols("".join(sorted(chars))), k


@dataclass
class LearnResult:
    annotations: List[str]      # row labels in first-appearance order
    seq_count: np.ndarray       # int64 [A]
    M: np.ndarray               # int64 [A, K]
    totals: np.ndarray          # int64 [K], over ALL sequences of the file
    total_seqs: int             # number of distinct sequence ids
    kmerlist: List[str]


def learn_counts(ids: Sequence[str], reduced_seqs: Sequence[str], kmerlist: Sequence[str],
                 seq_annot: Dict[str, str]) -> LearnResult:
    """Per-annotation summed k-mer counts of one file (Library.generate_kmer_counts +
    filter_and_construct, learn.smk:306-326,359-408).

    The reference keys a dict by sequence id: a repeated id keeps its FIRST position but
    its LAST counts, while every copy has already been added to the totals.  Annotation
    rows appear in the order their first (distinct) sequence does."""
    kmerlist = [str(x) for x in kmerlist]
    if len(kmerlist) > DENSE_MAX_K:
        raise _dense_envelope_error("learn", len(kmerlist))
    tab, k = _kmer_tables(kmerlist)
    batch = E.SequenceBatch.from_strings([str(s) for s in reduced_seqs])
    last = {}
    for i, sid in enumerate(ids):
        last[sid] = i
    ann_index: Dict[str, int] = {}
    ann_id = np.full(len(ids), -1, dtype=np.int32)
    seq_count: List[int] = []
    for sid, i in last.items():
        acc = _ACCESSION.findall(sid)[0]          # IndexError without two pipes, like learn.smk:322
        if acc not in seq_annot:
            continue
        a = seq_annot[acc]
        if a not in ann_index:
            ann_index[a] = len(ann_index)
            seq_count.append(0)
        ann_id[i] = ann_index[a]
        seq_count[ann_index[a]] += 1
    M, totals = E.learn_over_kmers(batch, tab, k, kmerlist, torch.from_numpy(ann_id), len(ann_index))
    return LearnResult(list(ann_index), np.array(seq_count, dtype=np.int64), M, totals, len(last), kmerlist)


def _csv_field(text: str) -> str:
    buf = _io.StringIO()
    _csv.writer(buf, lineterminator="").writerow([text])
    return buf.getvalue()


def write_counts_csv(path: str, r: LearnResult) -> None:
    """kmer-counts-{nb}.csv exactly as Library.format_and_write_output writes it
    (learn.smk:328-357): zeros blank, `Totals` first, index column first."""
    with open(path, "w", newline="") as f:
        f.write(",".join([INDEX_COL, "Sequence count", "Kmer Count"] + [_csv_field(km) for km in r.kmerlist]) + "\n")

        def row(label, nseq, values):
            cells = [str(v) if v else "" for v in values.tolist()]
            total = int(values.sum())
            f.write(",".join([_csv_field(str(label)), str(nseq) if nseq else "", str(total) if total else ""] + cells) + "\n")

        row("Totals", r.total_seqs, r.totals)
        for a, n, m in zip(r.annotations, r.seq_count.tolist(), r.M):
            row(a, n, m)


def learn_rule(npz: str, annotation_files: Sequence[str], out_csv: str) -> LearnResult:
    kmerlists, df = skio.load_npz(npz)
    r = learn_counts(list(df["sequence_id"]), list(df["sequence"]), list(kmerlists[0]), load_annotations(annotation_files))
    write_counts_csv(out_csv, r)
    return r


# ---------------------------------------------------------------------------
# merge (Merge)
# ---------------------------------------------------------------------------
@dataclass
class CountsTable:
    """A kmer-counts CSV in memory: rows (`Totals` + annotations) x (Sequence count, Kmer Count, k-mers)."""
    rows: List[str]
    kmers: List[str]
    seq_count: np.ndarray       # int64 [R]
    kmer_count: np.ndarray      # int64 [R]
    M: np.ndarray               # int64 [R, K]


def read_counts_csv(path: str) -> CountsTable:
    """Reads either writer's layout (index column first or last; blanks are zeros)."""
    with open(path, newline="") as f:
        reader = _csv.reader(f)
        header = next(reader)
        ix = header.index(INDEX_COL)
        cols = [c for i, c in enumerate(header) if i != ix]
        rows, data = [], []
        for rec in reader:
            if not rec:
                continue
            rows.append(rec[ix])
            data.append([int(float(v)) if v else 0 for i, v in enumerate(rec) if i != ix])
    arr = np.array(data, dtype=np.int64).reshape(len(rows), len(cols))
    sc, kc = cols.index("Sequence count"), cols.index("Kmer Count")
    km = [i for i in range(len(cols)) if i not in (sc, kc)]
    return CountsTable(rows, [cols[i] for i in km], arr[:, sc].copy(), arr[:, kc].copy(), np.ascontiguousarray(arr[:, km]))


def merge_tables(tables: Sequence[CountsTable]) -> CountsTable:
    """Outer join on k-mer columns + row-wise sum (``concat -> groupby(sort=False).sum``,
    learn.smk:467-494): rows and columns in order of first appearance."""
    rows: Dict[str, int] = {}
    kmers: Dict[str, int] = {}
    for t in tables:
        for r in t.rows:
            rows.setdefault(r, len(rows))
        for c in t.kmers:
            kmers.setdefault(c, len(kmers))
    dev = E._require_cuda()
    # two extra columns carry Sequence count / Kmer Count through the same scatter-add
    dst = torch.zeros((len(rows), len(kmers) + 2), dtype=torch.int64, device=dev)
    for t in tables:
        src = np.concatenate([t.seq_count[:, None], t.kmer_count[:, None], t.M], axis=1)
        row_map = np.array([rows[r] for r in t.rows], dtype=np.int64)
        col_map = np.array([0, 1] + [kmers[c] + 2 for c in t.kmers], dtype=np.int64)
        E.scatter_add(dst, torch.from_numpy(np.ascontiguousarray(src)).to(dev), row_map, col_map)
    out = dst.cpu().numpy()
    return CountsTable(list(rows), list(kmers), out[:, 0].copy(), out[:, 1].copy(), np.ascontiguousarray(out[:, 2:]))


def write_totals_csv(path: str, t: CountsTable) -> None:
    """kmer-counts-total.csv in the layout pyarrow gives the reference (learn.smk:583-594):
    quoted header, integer cells, index column last."""
    q = lambda s: '"' + str(s).replace('"', '""') + '"'
    with open(path, "w", newline="") as f:
        f.write(",".join([q("Sequence count"), q("Kmer Count")] + [q(k) for k in t.kmers] + [q(INDEX_COL)]) + "\n")
        for i, label in enumerate(t.rows):
            f.write(",".join([str(int(t.seq_count[i])), str(int(t.kmer_count[i]))] + [str(v) for v in t.M[i].tolist()]
                             + [q(label)]) + "\n")


def _letters(names) -> set:
    return set(itertools.chain.from_iterable(list(str(x)) for x in names))


def merge_rule(count_files: Sequence[str], out_csv: str, base_counts: Optional[str] = None) -> CountsTable:
    merged = merge_tables([read_counts_csv(f) for f in count_files])
    if base_counts and "csv" in str(base_counts):
        base = read_counts_csv(str(base_counts))
        # learn.smk:517-554: same letters in the columns from position 3 on, same k-mer length
        cols_new = ["Sequence count", "Kmer Count"] + merged.kmers
        cols_base = ["Sequence count", "Kmer Count"] + base.kmers
        n = len(cols_new)
        ok = _letters(cols_new[3:n]) == _letters(cols_base[3:n]) and len(cols_new[1]) == len(cols_base[1])
        if ok:
            merged = merge_tables([base, merged])
    write_totals_csv(out_csv, merged)
    return merged


# ---------------------------------------------------------------------------
# cosine scoring shared by eval_apply and apply
# ---------------------------------------------------------------------------
def _compare_check(query_cols: Sequence[str], total_cols: Sequence[str]) -> None:
    """apply.smk:224-260 / learn.smk:761-788: 11th column names of equal length and the same
    letters from the 11th column on; otherwise the rule prints and exits."""
    ok = len(str(query_cols[10])) == len(str(total_cols[10]))
    if ok:
        n = len(query_cols)
        ok = _letters(query_cols[10:n]) == _letters(total_cols[10:n])
    if not ok:
        print("Compare Check Failed. ")
        sys.exit()


@dataclass
class ScoreResult:
    rows: List[str]             # query labels
    annotations: List[str]
    top1: np.ndarray
    top2: np.ndarray
    score1: np.ndarray
    score2: np.ndarray
    scores: Optional[np.ndarray]    # float64 [Q, A] when requested


def cosine_top2(reduced_seqs: Sequence[str], query_kmers: Sequence[str], totals: CountsTable,
                full: bool = False) -> E.ApplyResult:
    """Cosine of every query against every annotation row of `totals` + top-2.

    Reference semantics (apply.smk:262-289): both frames are re-indexed onto the UNION of
    their k-mer columns, so the query norm runs over the query file's own k-mer list while
    the dot product only sees k-mers present in both lists."""
    query_kmers = [str(x) for x in query_kmers]
    if max(len(query_kmers), len(totals.kmers)) > DENSE_MAX_K:
        raise _dense_envelope_error("apply", max(len(query_kmers), len(totals.kmers)))
    keep = [i for i, r in enumerate(totals.rows) if r != "Totals"]
    M = torch.from_numpy(np.ascontiguousarray(totals.M[keep])).to(E._require_cuda())
    tab, k = _kmer_tables(query_kmers, totals.kmers) if totals.kmers else _kmer_tables(query_kmers)
    batch = E.SequenceBatch.from_strings([str(s) for s in reduced_seqs])
    q_basis, _ = E.basis_from_kmers(query_kmers, tab, k, batch.device)
    t_basis, t_keep = E.basis_from_kmers(totals.kmers, tab, k, batch.device)
    both = E.intersect_basis(t_basis, q_basis)
    Q = E.count_dense(batch, tab, k, both)                 # columns = encodable learned k-mers
    qn2 = E.row_norm2(E.count_dense(batch, tab, k, q_basis))
    Mk = M[:, torch.from_numpy(t_keep).to(M.device)].contiguous() if len(t_keep) != M.shape[1] else M
    # learned k-mers that cannot be encoded never match a window but still count in ||m||
    return E.apply_dense(Q, Mk, qnorm2=qn2, mnorm2=E.row_norm2(M), full=full)


def _unique_last(ids: Sequence[str]) -> Tuple[List[str], np.ndarray]:
    """dict(id -> value) semantics: first position, last value."""
    last = {}
    for i, sid in enumerate(ids):
        last[sid] = i
    return list(last), np.fromiter(last.values(), dtype=np.int64, count=len(last))


def _write_arrow_csv(path: str, columns: Dict[str, object]) -> None:
    import pyarrow as pa
    from pyarrow import csv as pacsv

    pacsv.write_csv(pa.table(columns), path)


def eval_apply_rule(npz: str, annotation_files: Sequence[str], counts_csv: str, out_csv: str,
                    save_associations: bool = False) -> ScoreResult:
    """learn.smk:628-887: score the training sequences against the merged matrix; rows are
    tagged ``<annotation>_known_<i>`` / ``<accession>_unknown_<i>``; unless
    `save_associations`, only the two best scores of a row are kept (the rest NaN)."""
    totals = read_counts_csv(counts_csv)
    import pandas as pd

    first = pd.read_table(annotation_files[0])               # the reference uses the first file only here
    seq_annot = dict(zip(first["id"].tolist(), first["TIGRFAMs"].tolist()))
    kmerlists, df = skio.load_npz(npz)
    kmerlist = [str(x) for x in kmerlists[0]]
    _compare_check(["Sequence count"] + kmerlist, ["Sequence count", "Kmer Count"] + totals.kmers)
    ids, pick = _unique_last(list(df["sequence_id"]))
    labels = []
    for n, sid in enumerate(ids):
        acc = _ACCESSION.findall(sid)[0]
        labels.append(f"{seq_annot[acc]}_known_{n}" if acc in seq_annot else f"{acc}_unknown_{n}")
    seqs = [df["sequence"][int(i)] for i in pick]
    r = cosine_top2(seqs, kmerlist, totals, full=True)
    S = r.scores.cpu().numpy()
    anns = [x for x in totals.rows if x != "Totals"]
    if not save_associations and S.shape[1] > 0:
        keep = np.zeros_like(S, dtype=bool)
        rows = np.arange(S.shape[0])
        keep[rows, r.top1.cpu().numpy()] = True
        t2 = r.top2.cpu().numpy()
        keep[rows[t2 >= 0], t2[t2 >= 0]] = True
        S = np.where(keep, S, np.nan)
    cols: Dict[str, object] = {a: S[:, j] for j, a in enumerate(anns)}
    cols[INDEX_COL] = labels
    _write_arrow_csv(out_csv, cols)
    return ScoreResult(labels, anns, r.top1.cpu().numpy(), r.top2.cpu().numpy(), r.score1.cpu().numpy(),
                       r.score2.cpu().numpy(), S)


def read_confidence_csv(path: str) -> Dict[float, float]:
    """global-confidence-scores.csv: first column = delta key, second = confidence (apply.smk:301-310)."""
    import pandas as pd

    t = pd.read_csv(str(path))
    return dict(zip(t.iloc[:, 0].astype(float).tolist(), t.iloc[:, 1].astype(float).tolist()))


def delta_and_confidence(r: E.ApplyResult, conf: Dict[float, float], n_ann: int) -> Tuple[np.ndarray, np.ndarray]:
    """delta = round(top1 - top2, 2) and Confidence = lookup of delta (apply.smk:312-335) for all queries at once:
    the Difference bin of every query comes from the device (skm_confidence_hist without histograms, numpy's
    rint(x * 100) / 100), delta and the confidence are table look-ups over the 101 values.  Rows whose bin is
    undefined (a single annotation: no runner-up) fall back to the scalar formula."""
    from . import confidence as CF

    bins = CF.difference_bins(r.top1, r.score1, r.score2, n_ann).cpu().numpy()
    vals = np.array(CF.POSSIBLE_VALS + [np.nan], dtype=np.float64)
    table = np.array([conf.get(v, np.nan) for v in CF.POSSIBLE_VALS] + [np.nan], dtype=np.float64)
    idx = np.where(bins == 255, len(CF.POSSIBLE_VALS), bins).astype(np.int64)
    delta, confidence = vals[idx], table[idx]
    odd = np.flatnonzero(bins == 255)
    if odd.size:
        d = np.round(r.score1[torch.from_numpy(odd).to(r.score1.device)].cpu().numpy()
                     - r.score2[torch.from_numpy(odd).to(r.score2.device)].cpu().numpy(), 2)
        delta[odd] = d
        confidence[odd] = [conf.get(float(x), np.nan) for x in d]
    return delta, confidence


def apply_rule(npz: str, counts_csv: str, confidence_csv: str, out_summary: str, out_scores: Optional[str] = None,
               save_associations: bool = False) -> ScoreResult:
    """apply.smk:147-353: Prediction = best annotation, Score = its cosine,
    delta = round(top1 - top2, 2), Confidence = lookup of delta."""
    totals = read_counts_csv(counts_csv)
    kmerlists, df = skio.load_npz(npz)
    kmerlist = [str(x) for x in kmerlists[0]]
    _compare_check(["Sequence count"] + kmerlist, ["Sequence count", "Kmer Count"] + totals.kmers)
    ids, pick = _unique_last(list(df["sequence_id"]))
    seqs = [df["sequence"][int(i)] for i in pick]
    r = cosine_top2(seqs, kmerlist, totals, full=bool(save_associations))
    anns = [x for x in totals.rows if x != "Totals"]
    top1, s1, s2 = r.top1.cpu().numpy(), r.score1.cpu().numpy(), r.score2.cpu().numpy()
    if save_associations and out_scores:
        S = r.scores.cpu().numpy()
        cols: Dict[str, object] = {a: S[:, j] for j, a in enumerate(anns)}
        cols[INDEX_COL] = ids
        _write_arrow_csv(out_scores, cols)
    conf = read_confidence_csv(confidence_csv)
    delta, confidence = delta_and_confidence(r, conf, len(anns))
    import pyarrow as pa

    _write_arrow_csv(out_summary, {
        "index": ids,
        "Prediction": [str(anns[i]) for i in top1],
        "Score": s1,
        "delta": delta,
        "Confidence": pa.array(confidence, from_pandas=True),      # NaN -> null, like DataFrame.map misses
    })
    return ScoreResult(ids, anns, top1, r.top2.cpu().numpy(), s1, s2, r.scores.cpu().numpy() if r.scores is not None else None)


# ---------------------------------------------------------------------------
# evaluate (Evaluator)
# ---------------------------------------------------------------------------
def evaluate_rule(score_csvs: Sequence[str], out_conf: str, out_glob: str, base_confidence: Sequence[str] = (),
                  modifier: float = 1.0):
    """learn.smk:897-1360: seq-annotation-scores files -> confidence-matrix.csv + global-confidence-scores.csv
    (optionally merged with ONE prior global-confidence file, weight modifier = conf_weight_modifier)."""
    from .confidence import Evaluator

    ev = Evaluator(list(score_csvs), out_conf, out_glob, list(base_confidence), modifier=modifier)
    return ev.execute_all()


def evaluate_results(results: Sequence[ScoreResult], out_conf: Optional[str] = None, out_glob: Optional[str] = None,
                     base_confidence: Sequence[str] = (), modifier: float = 1.0):
    """The same evaluation fed by eval_apply_rule's in-memory results (top-2 per row): no Q x A file is read back."""
    from . import confidence as CF

    dev = E._require_cuda()
    acc = CF.ConfidenceAccumulator()
    for r in results:
        res = E.ApplyResult(torch.from_numpy(np.ascontiguousarray(r.top1, dtype=np.int32)).to(dev),
                            torch.from_numpy(np.ascontiguousarray(r.top2, dtype=np.int32)).to(dev),
                            torch.from_numpy(np.ascontiguousarray(r.score1, dtype=np.float64)).to(dev),
                            torch.from_numpy(np.ascontiguousarray(r.score2, dtype=np.float64)).to(dev))
        acc.add(res, r.rows, r.annotations)
    return _write_evaluation(acc, out_conf, out_glob, base_confidence, modifier)


def _write_evaluation(acc, out_conf: Optional[str], out_glob: Optional[str], base_confidence: Sequence[str], modifier: float):
    """The end of Evaluator.execute_all: the curve of the accumulated crosstabs, merged with ONE prior
    global-confidence file when given, and the two files."""
    from . import confidence as CF

    prior = CF.read_global_confidence(str(base_confidence[0])) if len(base_confidence) == 1 else None
    out = acc.finalize(prior, modifier)
    if out_glob:
        CF.write_global_confidence(out_glob, out)
    if out_conf:
        CF.write_confidence_matrix(out_conf, out)
    return out
