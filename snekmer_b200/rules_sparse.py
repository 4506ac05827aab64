"""rules_sparse: the learn / merge / apply rule bodies for bases that do not fit dense matrices.

``rules.py`` mirrors the reference one to one: a dense ``[annotations, K]`` matrix in memory and wide CSV files
(learn.smk:306-357, apply.smk:147-353).  At the benchmark shapes (C3 / C4: 20 k - 50 k annotations x 1.68 M k-mers) that
matrix is 100+ GB dense and its CSV far larger, so the same three steps are offered on the sparse device paths with the
binary ``.skmc`` side-car (sidecar.py) as the file between them:

  learn_counts_sparse   Library (learn.smk:306-408)      -> COO matrix + Totals on the device
  merge_counts_sparse   Merge (learn.smk:467-494)        -> outer join on annotations, sum (skm_coo_merge)
  eval_counts_sparse    KmerCompare of learn (learn.smk:628-887) -> SpMM cosine, top-2 + each row's annotation
                        (EvalScores; the ``.skme`` side-car, and seq-annotation-scores-*.csv or its ``.skma`` when asked)
  evaluate_sparse       Evaluator (learn.smk:923-1348)   -> row classes and crosstabs on the device, the confidence files
  apply_counts_sparse   KmerCompare (apply.smk:224-342)  -> SpMM cosine, top-2, delta, Confidence

Row / column conventions are the reference's: annotation rows in order of first appearance, ``Totals`` over ALL
sequences, a repeated sequence id keeps its first position and last value, the query norm runs over all valid windows of
the query (its own k-mer list), ties go to the lowest annotation index.  ``sidecar.export_counts_csv`` /
``export_totals_csv`` turn a side-car back into the reference's CSV when the matrix is small enough to be one.

Code spaces beyond the tables (``len(symbols)^k > 2^27``) are keyed by basis column instead of code: the matrix carries
its column table (``SparseCounts.columns``), the k-mers that occur in first-occurrence order (engine.learn_wide).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import confidence as CF
from . import dist as D
from . import engine as E
from . import sidecar
from .rules import (_ACCESSION, ScoreResult, _unique_last, _write_arrow_csv, _write_evaluation, delta_and_confidence,
                    read_confidence_csv)


@dataclass
class SparseCounts:
    """A learned count matrix on the device: sorted COO keys ``ann * S + code`` over the reduced alphabet ``symbols``,
    or, with a column table (code spaces beyond 2^27), ``ann * K + col`` over the K columns of ``columns``."""
    annotations: List[str]
    seq_count: np.ndarray           # int64 [A]
    symbols: str
    k: int
    keys: torch.Tensor              # int64 [nnz], sorted
    vals: torch.Tensor              # int64 [nnz]
    totals: torch.Tensor            # int64 [S] (or [K] with columns): occurrences over ALL sequences
    total_seqs: int
    columns: Optional[E.WideBasis] = None   # column table: column j holds the k-mer code columns.codes[j]

    @property
    def S(self) -> int:
        return len(self.symbols) ** self.k

    @property
    def stride(self) -> int:
        """Key stride: S, or the number of columns K of a matrix keyed by column."""
        return self.S if self.columns is None else self.columns.K


def _wide(symbols: str, k: int) -> bool:
    return len(symbols) ** int(k) > E._native.SKM_DENSE_MAX_SPACE


def annotation_ids(ids: Sequence[str], seq_annot: Dict[str, str]):
    """(ann_id int32 [N], annotations in first-appearance order, sequences per annotation, distinct ids): the dict
    semantics of learn.smk:316-326 — a repeated id keeps its first position but only its LAST record counts."""
    last = {}
    for i, sid in enumerate(ids):
        last[sid] = i
    index: Dict[str, int] = {}
    ann_id = np.full(len(ids), -1, dtype=np.int32)
    seq_count: List[int] = []
    for sid, i in last.items():
        acc = _ACCESSION.findall(sid)[0]              # IndexError without two pipes, like learn.smk:322
        if acc not in seq_annot:
            continue
        a = seq_annot[acc]
        if a not in index:
            index[a] = len(index)
            seq_count.append(0)
        ann_id[i] = index[a]
        seq_count[index[a]] += 1
    return ann_id, list(index), np.array(seq_count, dtype=np.int64), len(last)


def learn_counts_sparse(ids: Sequence[str], reduced_seqs: Sequence[str], symbols: str, k: int,
                        seq_annot: Dict[str, str]) -> SparseCounts:
    """Library.generate_kmer_counts + filter_and_construct for one file, sparse.  NOTE the reference adds EVERY record
    to the totals but only the last record of a repeated id to its annotation row; so does this (records that lost to a
    later duplicate are counted as unannotated)."""
    tab = E.alphabet_tables_from_symbols(symbols)
    batch = E.SequenceBatch.from_strings([str(s) for s in reduced_seqs])
    ann_id, annotations, seq_count, total = annotation_ids(ids, seq_annot)
    if _wide(tab.symbols, k):
        # columns: every k-mer that occurs, in first-occurrence order (the wide analogue of "every code")
        columns = E.build_basis_wide(batch, tab, int(k), 0)
        keys, vals, totals = E.learn_wide(batch, tab, int(k), columns, torch.from_numpy(ann_id), len(annotations))
        return SparseCounts(annotations, seq_count, tab.symbols, int(k), keys, vals, totals, total, columns)
    keys, vals, totals = E.learn_sparse_with_totals(batch, tab, int(k), torch.from_numpy(ann_id), len(annotations))
    return SparseCounts(annotations, seq_count, tab.symbols, int(k), keys, vals, totals, total)


def _file_csr(sc: SparseCounts, kmers: Optional[Sequence[str]] = None):
    """A learned matrix as CSR over the columns of a counts file: (kmers, rowptr int64 [A + 2], cols int32, vals int64,
    seq_count int64 [A + 1] on the host, kmer_count int64 [A + 1]), rows ``Totals`` + annotations, columns ascending in
    a row, zeros left out; device tensors.  kmers: the file's columns (default: the k-mers that occur, in code order;
    the vectorize rule's kmerlist gives the reference's column order).  The key -> file-column remap and the row sort
    (skm_coo_merge over annotation * K + column) run on the device."""
    S = sc.stride
    dev = sc.keys.device
    totals = sc.totals
    # col_of_code: file column of every key % S (a code, or a learned column when the matrix has a column table)
    if sc.columns is not None:
        learned = sc.columns.codes_host()
        col_of_code = np.full(S, -1, dtype=np.int64)
        if kmers is None:
            occ = np.flatnonzero(totals.cpu().numpy())
            kmers = list(E.decode_kmers(learned[occ], sc.symbols, sc.k))
            col_of_code[occ] = np.arange(len(occ))
        else:
            kmers = [str(x) for x in kmers]
            codes, ok = E.encode_kmers(kmers, sc.symbols, sc.k)
            fcol = np.flatnonzero(ok)
            order = np.argsort(codes[fcol], kind="stable")
            fcodes = codes[fcol][order]
            j = np.minimum(np.searchsorted(fcodes, learned), max(len(fcodes) - 1, 0))
            hit = (fcodes[j] == learned) if len(fcodes) else np.zeros(len(learned), dtype=bool)
            col_of_code[hit] = fcol[order][j[hit]]
    elif kmers is None:
        codes = np.flatnonzero(totals.cpu().numpy()).astype(np.uint64)
        kmers = list(E.decode_kmers(codes, sc.symbols, sc.k))
        col_of_code = np.full(S, -1, dtype=np.int64)
        col_of_code[codes.astype(np.int64)] = np.arange(len(codes))
    else:
        kmers = [str(x) for x in kmers]
        codes, ok = E.encode_kmers(kmers, sc.symbols, sc.k)
        col_of_code = np.full(S, -1, dtype=np.int64)
        col_of_code[codes[ok].astype(np.int64)] = np.flatnonzero(ok)
    K, A = len(kmers), len(sc.annotations)
    cmap = torch.from_numpy(col_of_code).to(dev)
    z = torch.zeros(0, dtype=torch.int64, device=dev)
    col = cmap[sc.keys % S] if sc.keys.numel() else z
    keep = col >= 0
    fkeys, fvals = (sc.keys // S)[keep] * K + col[keep], sc.vals[keep]
    if fkeys.numel():
        fkeys, fvals = E.coo_merge(fkeys, fvals, key_bound=A * K)    # rows by annotation, columns ascending in a row
    tkeep = (cmap >= 0) & (totals != 0) if S else torch.zeros(0, dtype=torch.bool, device=dev)
    tcols, tvals = cmap[tkeep], totals[tkeep]
    if tcols.numel():
        tcols, tvals = E.coo_merge(tcols, tvals, key_bound=K)
    rowptr = torch.zeros(A + 2, dtype=torch.int64, device=dev)
    rowptr[1:] = tcols.numel()
    if A:
        rowptr[2:] += torch.searchsorted(fkeys, torch.arange(1, A + 1, dtype=torch.int64, device=dev) * K)
    vals = torch.cat([tvals, fvals])
    csum = torch.zeros(vals.numel() + 1, dtype=torch.int64, device=dev)
    torch.cumsum(vals, 0, out=csum[1:])
    kmer_count = csum[rowptr[1:]] - csum[rowptr[:-1]]
    cols = torch.cat([tcols, fkeys % K if K else fkeys]).to(torch.int32)
    seq_count = np.concatenate([[sc.total_seqs], sc.seq_count]).astype(np.int64)
    return kmers, rowptr, cols, vals, seq_count, kmer_count


def write_counts_sidecar(path: str, sc: SparseCounts, kmers: Optional[Sequence[str]] = None) -> None:
    """``.skmc`` of a learned matrix: rows ``Totals`` + annotations, columns = `kmers` (default: the k-mers that occur, in
    code order; pass the vectorize rule's kmerlist to get the reference's column order), CSR values."""
    kmers, rowptr, cols, vals, seq_count, kmer_count = _file_csr(sc, kmers)
    sidecar.write_counts_csr(path, ["Totals"] + list(sc.annotations), kmers, seq_count, kmer_count.cpu().numpy(),
                             rowptr.cpu().numpy(), cols.cpu().numpy(), vals.cpu().numpy())


def write_counts_csv(path: str, sc: SparseCounts, kmers: Optional[Sequence[str]] = None, layout: str = "learn") -> None:
    """The reference's count file of a learned matrix, its rows formatted on the device from the file-column CSR —
    no dense matrix: ``layout="learn"`` kmer-counts-{nb}.csv as the learn rule writes it (learn.smk:328-357: index
    first, zeros blank), ``"total"`` kmer-counts-total.csv as the merge rule writes it (learn.smk:583-594: quoted header,
    zeros as 0, index last).  Byte for byte write_counts_sidecar followed by sidecar.export_counts_csv /
    export_totals_csv; `kmers` as in write_counts_sidecar."""
    from .rules import INDEX_COL, _csv_field

    if layout not in ("learn", "total"):
        raise ValueError(f"layout must be 'learn' or 'total', not {layout!r}")
    kmers, rowptr, cols, vals, seq_count, kmer_count = _file_csr(sc, kmers)
    rows = ["Totals"] + [str(a) for a in sc.annotations]
    d_seq = torch.from_numpy(seq_count).to(rowptr.device)
    with open(path, "wb") as f:
        if layout == "learn":
            f.write((",".join([INDEX_COL, "Sequence count", "Kmer Count"] + [_csv_field(km) for km in kmers]) + "\n").encode("utf-8"))
            E.write_counts_csv_rows(f, rowptr, cols, vals, len(kmers), d_seq, kmer_count, [_csv_field(r) for r in rows], E.CSV_LEARN)
        else:
            f.write((",".join(E.pyarrow_quote(x) for x in ["Sequence count", "Kmer Count"] + list(kmers) + [INDEX_COL]) + "\n").encode("utf-8"))
            E.write_counts_csv_rows(f, rowptr, cols, vals, len(kmers), d_seq, kmer_count, rows, E.CSV_TOTAL)


def read_counts_sidecar(path: str, symbols: Optional[str] = None) -> SparseCounts:
    """``.skmc`` -> device COO.  The reduced alphabet is the set of characters of the k-mer columns unless given.  In a
    code space beyond 2^27 the matrix is keyed by column: the file's k-mers (those of the alphabet) in file order."""
    d = sidecar.read_counts_csr(path)
    dev = E._require_cuda()
    return _counts_from_file_csr(path, d["rows"], d["kmers"], d["seq_count"], torch.from_numpy(d["rowptr"]).to(dev),
                                 torch.from_numpy(d["cols"]).to(dev), torch.from_numpy(d["vals"]).to(dev), symbols)


def read_counts_csv(path: str, symbols: Optional[str] = None, block_bytes: int = E.CSV_PARSE_BLOCK) -> SparseCounts:
    """A kmer-counts CSV of either layout (a stock ``kmer-counts-total.csv`` or ``base/counts`` file, learn.smk:496-579)
    parsed on the device (engine.parse_counts_csv) straight into the device COO: what
    ``read_counts_sidecar(import_counts_csv(path))`` returns, without a dense matrix.  Cells follow a stated grammar —
    empty, [0-9]+, [0-9]+.0*, pyarrow's exponent form of an integer — and anything else raises SkmError."""
    labels, kmers, seq_count, _, rowptr, cols, vals = E.parse_counts_csv(path, block_bytes)
    return _counts_from_file_csr(path, labels, kmers, seq_count, rowptr, cols, vals, symbols)


def _counts_from_file_csr(path: str, rows: Sequence[str], kmers: Sequence[str], seq_count: np.ndarray, rowptr: torch.Tensor,
                          cols: torch.Tensor, vals: torch.Tensor, symbols: Optional[str]) -> SparseCounts:
    """A counts file's rows (``Totals`` first) as device CSR over its k-mer columns -> device COO: the file column -> key
    conversion of read_counts_sidecar and read_counts_csv."""
    if not rows or rows[0] != "Totals":
        raise ValueError(f"{path}: a counts table starts with its Totals row")
    k = len(kmers[0]) if kmers else 1
    symbols = "".join(sorted(set("".join(kmers)))) if symbols is None else "".join(sorted(set(symbols)))
    codes, ok = E.encode_kmers(kmers, symbols, k)
    dev = rowptr.device
    columns = None
    if _wide(symbols, k):
        columns = E.wide_basis_from_codes(codes[ok], E.alphabet_tables_from_symbols(symbols, dev), k, dev)
        key_of_col = np.cumsum(ok) - 1                   # file column -> learned column
        S = columns.K
    else:
        key_of_col = codes.astype(np.int64)
        S = len(symbols) ** k
    kc = torch.from_numpy(np.ascontiguousarray(key_of_col, dtype=np.int64)).to(dev)
    okd = torch.from_numpy(np.asarray(ok, dtype=bool)).to(dev)
    cols = cols.to(torch.int64)
    rows_of = torch.repeat_interleave(torch.arange(len(rows), dtype=torch.int64, device=dev), rowptr[1:] - rowptr[:-1])
    good = okd[cols] if cols.numel() else torch.zeros(0, dtype=torch.bool, device=dev)
    totals = torch.zeros(S, dtype=torch.int64, device=dev)
    t = (rows_of == 0) & good
    totals[kc[cols[t]]] = vals[t].to(torch.int64)
    m = (rows_of > 0) & good
    keys = (rows_of[m] - 1) * S + kc[cols[m]]
    keys, order = torch.sort(keys, stable=True)
    return SparseCounts(list(rows[1:]), np.asarray(seq_count[1:], dtype=np.int64), symbols, k, keys,
                        vals[m][order].to(torch.int64).contiguous(), totals, int(seq_count[0]), columns)


def merge_counts_sparse(parts: Sequence[SparseCounts]) -> SparseCounts:
    """Merge.merge_dataframes (learn.smk:467-494): outer join on the annotation rows (first appearance), element-wise sum."""
    assert parts and all(p.symbols == parts[0].symbols and p.k == parts[0].k for p in parts), "same reduced alphabet and k"
    index: Dict[str, int] = {}
    for p in parts:
        for a in p.annotations:
            index.setdefault(a, len(index))
    if parts[0].columns is not None:
        return _merge_wide(parts, index)
    S = parts[0].S
    seq_count = np.zeros(len(index), dtype=np.int64)
    ks, vs = [], []
    totals = torch.zeros_like(parts[0].totals)
    total_seqs = 0
    for p in parts:
        remap = torch.tensor([index[a] for a in p.annotations] + [0], dtype=torch.int64, device=p.keys.device)
        ks.append(remap[p.keys // S] * S + p.keys % S)
        vs.append(p.vals)
        np.add.at(seq_count, [index[a] for a in p.annotations], p.seq_count)
        totals += p.totals
        total_seqs += p.total_seqs
    keys, vals = E.coo_merge(torch.cat(ks), torch.cat(vs), key_bound=len(index) * S)
    return SparseCounts(list(index), seq_count, parts[0].symbols, parts[0].k, keys, vals, totals, total_seqs)


def _merge_wide(parts: Sequence[SparseCounts], index: Dict[str, int]) -> SparseCounts:
    """merge_counts_sparse of matrices keyed by column: the union of the columns in first-appearance order (the first
    part's columns, then each later part's new ones: learn.smk:467-494), every part re-keyed onto it, summed."""
    assert all(p.columns is not None for p in parts), "all parts keyed by column"
    tab = E.alphabet_tables_from_symbols(parts[0].symbols)
    codes = torch.cat([p.columns.codes for p in parts])
    n = codes.numel()
    dev = codes.device
    union = E.basis_table_finalize(tab, parts[0].k, codes, torch.ones(n, dtype=torch.int64, device=dev),
                                   torch.arange(n, dtype=torch.int64, device=dev), merged=False, min_filter=0, first_bound=n)
    KU = union.K
    seq_count = np.zeros(len(index), dtype=np.int64)
    ks, vs = [], []
    totals = torch.zeros(KU, dtype=torch.int64, device=dev)
    total_seqs = 0
    for p in parts:
        Kp = p.columns.K
        col = E.codes_to_columns(p.columns.codes, union).to(torch.int64)
        remap = torch.tensor([index[a] for a in p.annotations] + [0], dtype=torch.int64, device=dev)
        if Kp:
            ks.append(remap[p.keys // Kp] * KU + col[p.keys % Kp])
            vs.append(p.vals)
            totals.index_add_(0, col, p.totals)
        np.add.at(seq_count, [index[a] for a in p.annotations], p.seq_count)
        total_seqs += p.total_seqs
    keys, vals = (E.coo_merge(torch.cat(ks), torch.cat(vs), key_bound=len(index) * KU) if ks
                  else (torch.zeros(0, dtype=torch.int64, device=dev),) * 2)
    return SparseCounts(list(index), seq_count, parts[0].symbols, parts[0].k, keys, vals, totals, total_seqs, union)


def restrict_csr_to_kmers(rowptr: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, symbols: str, k: int,
                          kmers: Sequence[str]):
    """Drop the CSR entries (codes) that are not in `kmers` — the query file's own kmerlist: the reference takes the
    query norm over that list only (apply.smk:262-289), which matters when the vectorize step ran with min_filter > 0 or
    a basis.txt."""
    S = len(symbols) ** int(k)
    codes, ok = E.encode_kmers([str(x) for x in kmers], symbols, int(k))
    member = torch.zeros(S, dtype=torch.bool, device=cols.device)
    member[torch.from_numpy(codes[ok].astype(np.int64)).to(cols.device)] = True
    keep = member[cols.to(torch.int64)]
    csum = torch.zeros(keep.numel() + 1, dtype=torch.int64, device=cols.device)
    torch.cumsum(keep, 0, out=csum[1:])
    return csum[rowptr], cols[keep].contiguous(), vals[keep].contiguous()


def _score_sparse(seqs: Sequence[str], sc: SparseCounts, tile: Optional[int], query_kmers: Optional[Sequence[str]],
                  rows_sink=None, chunk_rows: Optional[int] = None) -> E.ApplyResult:
    """Cosine of every sequence against every annotation row of `sc` as SpMM, top-2 on the device (see
    apply_counts_sparse for `query_kmers` and `tile`); rows_sink / chunk_rows: the full rows as well
    (engine.apply_sparse_tiled)."""
    tab = E.alphabet_tables_from_symbols(sc.symbols)
    batch = E.SequenceBatch.from_strings(list(seqs))
    A = len(sc.annotations)
    if sc.columns is not None:
        restrict = None
        if query_kmers is not None:
            qcodes, ok = E.encode_kmers([str(x) for x in query_kmers], tab.symbols, sc.k)
            restrict = E.wide_basis_from_codes(np.unique(qcodes[ok]), tab, sc.k, batch.device)
        rowptr, cols, cvals = E.query_csr_wide(batch, tab, sc.k, sc.columns, restrict)
        return E.apply_wide(rowptr, cols, cvals, sc.keys, sc.vals, sc.columns.K, A, tile, rows_sink, chunk_rows)
    rowptr, cols, cvals = E.count_csr(batch, tab, sc.k, None)
    if query_kmers is not None:
        rowptr, cols, cvals = restrict_csr_to_kmers(rowptr, cols, cvals, tab.symbols, sc.k, query_kmers)
    return E.apply_sparse_tiled(rowptr, cols, cvals, sc.keys, sc.vals, sc.S, A, tile, rows_sink, chunk_rows)


MASK_BLOCK_ROWS = 65536     # rows per block of a top-2-only association side-car


def _associations_file(path: str, annotations: Sequence[str], labels: Sequence[str]):
    """``.skma`` side-car for a path ending in .skma, else the CSV with its text formatted on the device."""
    if str(path).endswith(".skma"):
        return sidecar.AssociationsWriter(path, annotations, labels)
    return E.AssociationsCSVText(path, annotations, labels)


def _write_top2_rows(w, r: E.ApplyResult, A: int) -> None:
    """The masked association rows of eval_apply without save_associations (learn.smk:831-849): each row keeps its
    top-2 scores, every other entry NaN — built from the top-2, block by block."""
    top1, top2 = r.top1.cpu().numpy(), r.top2.cpu().numpy()
    s1, s2 = r.score1.cpu().numpy(), r.score2.cpu().numpy()
    for q0 in range(0, len(top1), MASK_BLOCK_ROWS):
        q1 = min(q0 + MASK_BLOCK_ROWS, len(top1))
        block = np.full((q1 - q0, A), np.nan)
        rows = np.arange(q1 - q0)
        t1, t2 = top1[q0:q1], top2[q0:q1]
        k1, k2 = t1 >= 0, t2 >= 0
        block[rows[k1], t1[k1]] = s1[q0:q1][k1]
        block[rows[k2], t2[k2]] = s2[q0:q1][k2]
        w.write(q0, block)


def apply_counts_sparse(ids: Sequence[str], reduced_seqs: Sequence[str], sc: SparseCounts, confidence_csv: Optional[str] = None,
                        out_summary: Optional[str] = None, tile: Optional[int] = None,
                        query_kmers: Optional[Sequence[str]] = None, out_scores: Optional[str] = None,
                        save_associations: bool = False, chunk_rows: Optional[int] = None) -> ScoreResult:
    """KmerCompare of the apply workflow (apply.smk:224-342) as SpMM: cosine of every query against every annotation
    row, top-2, delta, Confidence; writes kmer-summary CSV when asked.  A repeated id keeps its last record.
    query_kmers: the query file's kmerlist (from its .npz / side-car).  The reference's query norm and dot run over that
    list; without it every valid window of the query counts — the same thing when the vectorize step ran with
    min_filter = 0 and no basis file, which is the only case the two differ in.  The annotation tile follows the
    accumulator width the data needs (engine.apply_sparse_tiled).
    out_scores with save_associations (learnapp: save_apply_associations, apply.smk:295-299): the association file,
    every query's cosine against every annotation (columns = the annotations, ``__index_level_0__`` = the distinct
    query ids last), streamed from the device `chunk_rows` queries at a time; a path ending in ``.skma`` writes the
    side-car (sidecar.export_associations_csv turns it into the CSV)."""
    uniq, pick = _unique_last(list(ids))
    seqs = [str(reduced_seqs[int(i)]) for i in pick]
    A = len(sc.annotations)
    if out_scores and save_associations:
        with _associations_file(out_scores, sc.annotations, uniq) as w:
            r = _score_sparse(seqs, sc, tile, query_kmers, w if isinstance(w, E.AssociationsCSVText) else w.write, chunk_rows)
    else:
        r = _score_sparse(seqs, sc, tile, query_kmers)
    top1, top2 = r.top1.cpu().numpy(), r.top2.cpu().numpy()
    s1, s2 = r.score1.cpu().numpy(), r.score2.cpu().numpy()
    if out_summary:
        conf = read_confidence_csv(confidence_csv) if confidence_csv else {}
        delta, confidence = delta_and_confidence(r, conf, A)
        import pyarrow as pa

        _write_arrow_csv(out_summary, {"index": uniq, "Prediction": [str(sc.annotations[i]) for i in top1], "Score": s1,
                                       "delta": delta, "Confidence": pa.array(confidence, from_pandas=True)})
    return ScoreResult(uniq, list(sc.annotations), top1, top2, s1, s2, None)


@dataclass
class EvalScores:
    """eval_apply of one training file on the sparse path: top-2 of every row on the device and, in place of the row
    label ``<annotation>_known_<n>`` / ``<accession>_unknown_<n>`` (learn.smk:712-732), its parts — the entry of
    `names` it was built from (`truth`, -1 for an unknown row) and n = row_base + row.  `names` starts with the
    matrix's `annotations` (the columns top1 / top2 index), then the file's other annotation names."""
    annotations: List[str]
    names: List[str]
    top1: torch.Tensor              # int32 [Q]
    top2: torch.Tensor              # int32 [Q]
    score1: torch.Tensor            # float64 [Q]
    score2: torch.Tensor            # float64 [Q]
    truth: torch.Tensor             # int32 [Q]
    row_base: int

    def result(self) -> E.ApplyResult:
        return E.ApplyResult(self.top1, self.top2, self.score1, self.score2)


def eval_counts_sparse(ids: Sequence[str], reduced_seqs: Sequence[str], sc: SparseCounts, seq_annot: Dict[str, str],
                       out_sidecar: Optional[str] = None, tile: Optional[int] = None,
                       query_kmers: Optional[Sequence[str]] = None, out_scores: Optional[str] = None,
                       save_associations: bool = False, chunk_rows: Optional[int] = None) -> EvalScores:
    """KmerCompare of the learn workflow (learn.smk:628-887) as SpMM: the training sequences of one file against the
    merged matrix.  Rows as eval_apply_rule: the distinct ids (a repeated id keeps its first position and last record),
    numbered in that order; a row is known when its accession is in `seq_annot` — the caller passes the FIRST
    annotation file only, as the rule reads only that one.  Top-2 stay on the device; `out_sidecar` writes the
    ``.skme`` that evaluate_sparse reads.  With several ranks (matrix replicated), each passes a contiguous share of the
    file's distinct ids, in order; row numbers continue across ranks.
    out_scores: the rule's seq-annotation-scores file (``.skma`` side-car for a path ending in .skma), rows labelled
    ``<annotation>_known_<n>`` / ``<accession>_unknown_<n>`` (learn.smk:712-732): with save_associations every score,
    streamed from the device `chunk_rows` rows at a time; without, each row's top-2 and NaN elsewhere
    (learn.smk:831-849).  Each rank writes its own rows."""
    uniq, pick = _unique_last(list(ids))
    dev = E._require_cuda()
    accs = [_ACCESSION.findall(sid)[0] for sid in uniq]         # IndexError without two pipes, like learn.smk:714
    row_base, _ = D.exclusive_prefix(len(uniq), dev)
    w = None
    if out_scores:
        labels = [f"{seq_annot[a]}_known_{row_base + n}" if a in seq_annot else f"{a}_unknown_{row_base + n}"
                  for n, a in enumerate(accs)]
        w = _associations_file(out_scores, sc.annotations, labels)
    try:
        if uniq:
            sink = None
            if w is not None and save_associations:
                sink = w if isinstance(w, E.AssociationsCSVText) else w.write
            r = _score_sparse([str(reduced_seqs[int(i)]) for i in pick], sc, tile, query_kmers, sink, chunk_rows)
        else:
            e32, e64 = torch.zeros(0, dtype=torch.int32, device=dev), torch.zeros(0, dtype=torch.float64, device=dev)
            r = E.ApplyResult(e32, e32.clone(), e64, e64.clone())
        if w is not None and not save_associations:
            if isinstance(w, E.AssociationsCSVText):
                E.write_top2_csv(w, r, chunk_rows)
            else:
                _write_top2_rows(w, r, len(sc.annotations))
    finally:
        if w is not None:
            w.close()
    names, truth = CF.joint_name_table(sc.annotations, [seq_annot[a] if a in seq_annot else None for a in accs])
    ev = EvalScores(list(sc.annotations), names, r.top1, r.top2, r.score1, r.score2, torch.from_numpy(truth).to(r.top1.device),
                    row_base)
    if out_sidecar:
        write_eval_sidecar(out_sidecar, ev)
    return ev


def write_eval_sidecar(path: str, ev: EvalScores) -> None:
    sidecar.write_evalscores(path, ev.annotations, ev.names, ev.top1.cpu().numpy(), ev.top2.cpu().numpy(),
                             ev.score1.cpu().numpy(), ev.score2.cpu().numpy(), ev.truth.cpu().numpy(), ev.row_base)


def read_eval_sidecar(path: str) -> EvalScores:
    d = sidecar.read_evalscores(path)
    dev = E._require_cuda()
    t = {k: torch.from_numpy(d[k]).to(dev) for k in ("top1", "top2", "score1", "score2", "truth")}
    return EvalScores(d["annotations"], d["names"], t["top1"], t["top2"], t["score1"], t["score2"], t["truth"], d["row_base"])


def evaluate_sparse(evals: Sequence, out_conf: Optional[str] = None, out_glob: Optional[str] = None,
                    base_confidence: Sequence[str] = (), modifier: float = 1.0) -> CF.EvalResult:
    """Evaluator.execute_all (learn.smk:923-1348) over eval_counts_sparse results or their ``.skme`` side-cars, in file
    order: row classes (skm_confidence_classify) and crosstabs (skm_confidence_hist) on the device, then the same
    curve, prior-confidence merge (ONE base file, weight `modifier`) and files as evaluate_rule."""
    acc = CF.ConfidenceAccumulator()
    for ev in evals:
        if not isinstance(ev, EvalScores):
            ev = read_eval_sidecar(str(ev))
        acc.add_device(ev.result(), ev.truth, ev.row_base, ev.names, ev.annotations)
    return _write_evaluation(acc, out_conf, out_glob, base_confidence, modifier)
