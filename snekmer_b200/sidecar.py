"""sidecar: binary side-cars for the two big artefacts of the path, with lossless export to / import from the
reference's own formats.

The reference hands vectors between rules as ``.npz`` with a dense float64 presence matrix
(kmerize.smk:132-139, read by io.py:46-96) and count matrices as wide CSVs (learn.smk:328-357 writer,
:496-579 merge reader).  At the benchmark shapes those files are hundreds of GB and CSV parsing dwarfs
every kernel, so the GPU path keeps

  *.skmv   vectors of one FASTA shard: basis codes, ids, reduced sequences, raw lengths and the per-sequence
           counts as CSR (rowptr int64, cols int32, vals int32)
  *.skmc   a learned count matrix: row labels (annotations, ``Totals`` first), sequence counts, k-mer list and the
           matrix as CSR (int64 values)
  *.skme   eval_apply scores of one training file for the evaluate rule (in place of seq-annotation-scores-*.csv):
           the matrix's annotations, the name table of the row labels, top-2 columns and scores and the label's
           annotation (truth) of every row, and the global number of the first row
  *.skma   an association matrix (apply.smk:295-299, learn.smk:821-849): the annotation names, the row labels and
           the float64 [Q, A] cosine table, written block by block while the rows stream off the device;
           ``export_associations_csv`` writes the reference's seq-annotation-scores CSV from it

in one flat container (below), whose arrays can be memory-mapped and uploaded without parsing.  ``export_npz`` /
``export_counts_csv`` / ``export_totals_csv`` write exactly what the reference's rules write; ``import_counts_csv``
reads either CSV layout.  Host-only module (file formats); device work stays in engine.

Container:  b"SKMB200\\0" | u32 version | u32 reserved | u64 meta_len | meta (UTF-8 JSON, padded to 64 bytes) |
            arrays, each 64-byte aligned.  meta = {"kind": ..., "attrs": {...},
            "arrays": [{"name", "dtype", "shape", "offset", "nbytes"}, ...]} with offsets from the file start.
"""
from __future__ import annotations

import json
import struct
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

MAGIC = b"SKMB200\0"
VERSION = 1
_ALIGN = 64


def _pad(n: int) -> int:
    return (n + _ALIGN - 1) // _ALIGN * _ALIGN


def _strings_to_arrays(strings: Sequence[str]) -> Tuple[np.ndarray, np.ndarray]:
    enc = [str(s).encode("utf-8") for s in strings]
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    if enc:
        np.cumsum([len(b) for b in enc], out=off[1:])
    return np.frombuffer(b"".join(enc), dtype=np.uint8), off


def _arrays_to_strings(buf: np.ndarray, off: np.ndarray) -> List[str]:
    raw = buf.tobytes()
    return [raw[off[i]:off[i + 1]].decode("utf-8") for i in range(len(off) - 1)]


def _layout(kind: str, attrs: Dict, specs: Sequence[Tuple[str, np.dtype, Tuple[int, ...]]]) -> Tuple[bytes, List[Dict]]:
    """(file header with its meta, array entries with their offsets) of a container holding arrays (name, dtype, shape)."""
    entries = [{"name": k, "dtype": np.dtype(dt).str, "shape": list(shape), "offset": 0,
                "nbytes": int(np.prod(shape, dtype=np.int64)) * np.dtype(dt).itemsize} for k, dt, shape in specs]
    # offsets depend on the meta length, which depends on the offsets' digits: reserve, then fix
    meta_len = _pad(len(json.dumps({"kind": kind, "attrs": attrs, "arrays": entries}).encode()) + 24 * len(entries) + 64)
    pos = _pad(len(MAGIC) + 16 + meta_len)
    for e in entries:
        e["offset"] = pos
        pos = _pad(pos + e["nbytes"])
    meta = json.dumps({"kind": kind, "attrs": attrs, "arrays": entries}).encode()
    assert len(meta) <= meta_len
    return MAGIC + struct.pack("<IIQ", VERSION, 0, meta_len) + meta + b" " * (meta_len - len(meta)), entries


def write_container(path: str, kind: str, attrs: Dict, arrays: Dict[str, np.ndarray]) -> None:
    arrs = {k: np.ascontiguousarray(v) for k, v in arrays.items()}
    head, entries = _layout(kind, attrs, [(k, v.dtype, v.shape) for k, v in arrs.items()])
    with open(path, "wb") as f:
        f.write(head)
        for e in entries:
            f.write(b"\0" * (e["offset"] - f.tell()))
            f.write(arrs[e["name"]].tobytes())


def read_container(path: str, mmap: bool = True) -> Tuple[str, Dict, Dict[str, np.ndarray]]:
    with open(path, "rb") as f:
        head = f.read(len(MAGIC) + 16)
        if head[:len(MAGIC)] != MAGIC:
            raise ValueError(f"{path}: not a snekmer_b200 side-car")
        version, _, meta_len = struct.unpack("<IIQ", head[len(MAGIC):])
        if version != VERSION:
            raise ValueError(f"{path}: side-car version {version}, this reader handles {VERSION}")
        meta = json.loads(f.read(meta_len).decode())
    arrays = {}
    for e in meta["arrays"]:
        shape, dt = tuple(e["shape"]), np.dtype(e["dtype"])
        if e["nbytes"] == 0:
            arrays[e["name"]] = np.zeros(shape, dtype=dt)
        elif mmap:
            arrays[e["name"]] = np.memmap(path, dtype=dt, mode="r", offset=e["offset"], shape=shape)
        else:
            with open(path, "rb") as f:
                f.seek(e["offset"])
                arrays[e["name"]] = np.frombuffer(f.read(e["nbytes"]), dtype=dt).reshape(shape)
    return meta["kind"], meta["attrs"], arrays


# ---------------------------------------------------------------------------
# vectors (.skmv)  <->  .npz of the vectorize rule
# ---------------------------------------------------------------------------
def write_vectors(path: str, alphabet: str, k: int, symbols: str, basis_codes: np.ndarray, ids: Sequence[str],
                  seqs: Sequence[str], lengths: np.ndarray, rowptr: np.ndarray, cols: np.ndarray, vals: np.ndarray) -> None:
    ib, io_ = _strings_to_arrays(ids)
    sb, so = _strings_to_arrays(seqs)
    write_container(path, "vectors", {"alphabet": str(alphabet), "k": int(k), "symbols": symbols, "nseq": len(ids), "K": int(len(basis_codes))},
                    {"basis_codes": np.asarray(basis_codes, dtype=np.uint64), "ids": ib, "id_offsets": io_, "seqs": sb, "seq_offsets": so,
                     "lengths": np.asarray(lengths, dtype=np.int64), "rowptr": np.asarray(rowptr, dtype=np.int64),
                     "cols": np.asarray(cols, dtype=np.int32), "vals": np.asarray(vals, dtype=np.int32)})


def dense_to_csr(counts: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    counts = np.asarray(counts)
    r, c = np.nonzero(counts)
    rowptr = np.zeros(counts.shape[0] + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=counts.shape[0]), out=rowptr[1:])
    return rowptr, c.astype(np.int32), counts[r, c].astype(np.int32)


def read_vectors(path: str, mmap: bool = True) -> Dict:
    kind, attrs, a = read_container(path, mmap)
    if kind != "vectors":
        raise ValueError(f"{path}: holds '{kind}', not vectors")
    out = dict(attrs)
    out.update(basis_codes=a["basis_codes"], ids=_arrays_to_strings(a["ids"], a["id_offsets"]),
               seqs=_arrays_to_strings(a["seqs"], a["seq_offsets"]), lengths=a["lengths"], rowptr=a["rowptr"], cols=a["cols"], vals=a["vals"])
    return out


def decode_kmers(codes: np.ndarray, symbols: str, k: int) -> np.ndarray:
    codes = np.asarray(codes, dtype=np.uint64)
    if codes.size == 0:
        return np.array([])
    n = np.uint64(len(symbols))
    sym = np.frombuffer(symbols.encode("latin-1"), dtype=np.uint8)
    chars = np.empty((codes.size, k), dtype=np.uint8)
    c = codes.copy()
    for i in range(k - 1, -1, -1):
        chars[:, i] = sym[(c % n).astype(np.int64)]
        c //= n
    return chars.view(f"S{k}").ravel().astype(f"<U{k}")


def export_npz(skmv_path: str, npz_path: str) -> None:
    """The .npz the vectorize rule writes (kmerize.smk:132-139): kmerlist, ids, seqs, vecs (float64 presence), lengths."""
    v = read_vectors(skmv_path)
    n, K = v["nseq"], v["K"]
    vecs = np.zeros((n, K), dtype=np.float64)
    rows = np.repeat(np.arange(n), np.diff(v["rowptr"]))
    vecs[rows, np.asarray(v["cols"], dtype=np.int64)] = 1.0
    np.savez_compressed(npz_path, kmerlist=decode_kmers(v["basis_codes"], v["symbols"], v["k"]), ids=v["ids"], seqs=v["seqs"],
                        vecs=vecs, lengths=np.asarray(v["lengths"]))


# ---------------------------------------------------------------------------
# count matrices (.skmc)  <->  kmer-counts-*.csv
# ---------------------------------------------------------------------------
def write_counts_csr(path: str, rows: Sequence[str], kmers: Sequence[str], seq_count: np.ndarray, kmer_count: np.ndarray,
                     rowptr: np.ndarray, cols: np.ndarray, vals: np.ndarray) -> None:
    """rows include ``Totals`` (first) exactly like the CSV; the matrix is given as CSR over the k-mer list."""
    rb, ro = _strings_to_arrays(rows)
    kb, ko = _strings_to_arrays(kmers)
    write_container(path, "counts", {"nrows": len(rows), "K": len(kmers)},
                    {"rows": rb, "row_offsets": ro, "kmers": kb, "kmer_offsets": ko, "seq_count": np.asarray(seq_count, dtype=np.int64),
                     "kmer_count": np.asarray(kmer_count, dtype=np.int64), "rowptr": np.asarray(rowptr, dtype=np.int64),
                     "cols": np.asarray(cols, dtype=np.int32), "vals": np.asarray(vals, dtype=np.int64)})


def write_counts(path: str, rows: Sequence[str], kmers: Sequence[str], seq_count: np.ndarray, kmer_count: np.ndarray, M: np.ndarray) -> None:
    """Dense int64 [R, K] in, CSR on disk."""
    M = np.asarray(M, dtype=np.int64)
    r, c = np.nonzero(M)
    rowptr = np.zeros(M.shape[0] + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=M.shape[0]), out=rowptr[1:])
    write_counts_csr(path, rows, kmers, seq_count, kmer_count, rowptr, c.astype(np.int32), M[r, c])


def read_counts_csr(path: str, mmap: bool = True) -> Dict:
    """The side-car as stored (no dense matrix): rows, kmers, seq_count, kmer_count, rowptr, cols, vals."""
    kind, attrs, a = read_container(path, mmap)
    if kind != "counts":
        raise ValueError(f"{path}: holds '{kind}', not counts")
    return dict(rows=_arrays_to_strings(a["rows"], a["row_offsets"]), kmers=_arrays_to_strings(a["kmers"], a["kmer_offsets"]),
                seq_count=np.array(a["seq_count"]), kmer_count=np.array(a["kmer_count"]), rowptr=np.array(a["rowptr"]),
                cols=np.array(a["cols"]), vals=np.array(a["vals"]))


# ---------------------------------------------------------------------------
# eval_apply scores (.skme)
# ---------------------------------------------------------------------------
def write_evalscores(path: str, annotations: Sequence[str], names: Sequence[str], top1: np.ndarray, top2: np.ndarray,
                     score1: np.ndarray, score2: np.ndarray, truth: np.ndarray, row_base: int) -> None:
    """names: the label name table (the annotations first); truth int32 [Q]: entry of names the row's label was built
    from, -1 for an ``_unknown_`` row; row q is row ``row_base + q`` of the file."""
    ab, ao = _strings_to_arrays(annotations)
    nb, no = _strings_to_arrays(names)
    write_container(path, "evalscores", {"n_ann": len(annotations), "nrows": int(len(top1)), "row_base": int(row_base)},
                    {"annotations": ab, "annotation_offsets": ao, "names": nb, "name_offsets": no,
                     "top1": np.asarray(top1, dtype=np.int32), "top2": np.asarray(top2, dtype=np.int32),
                     "score1": np.asarray(score1, dtype=np.float64), "score2": np.asarray(score2, dtype=np.float64),
                     "truth": np.asarray(truth, dtype=np.int32)})


def read_evalscores(path: str, mmap: bool = True) -> Dict:
    kind, attrs, a = read_container(path, mmap)
    if kind != "evalscores":
        raise ValueError(f"{path}: holds '{kind}', not evalscores")
    return dict(annotations=_arrays_to_strings(a["annotations"], a["annotation_offsets"]),
                names=_arrays_to_strings(a["names"], a["name_offsets"]), row_base=int(attrs["row_base"]),
                **{k: np.array(a[k]) for k in ("top1", "top2", "score1", "score2", "truth")})


def read_counts(path: str, mmap: bool = True):
    """-> rules.CountsTable (dense int64 M rebuilt from the CSR)."""
    from .rules import CountsTable

    kind, attrs, a = read_container(path, mmap)
    if kind != "counts":
        raise ValueError(f"{path}: holds '{kind}', not counts")
    R, K = attrs["nrows"], attrs["K"]
    M = np.zeros((R, K), dtype=np.int64)
    rows = np.repeat(np.arange(R), np.diff(a["rowptr"]))
    M[rows, np.asarray(a["cols"], dtype=np.int64)] = a["vals"]
    return CountsTable(_arrays_to_strings(a["rows"], a["row_offsets"]), _arrays_to_strings(a["kmers"], a["kmer_offsets"]),
                       np.array(a["seq_count"]), np.array(a["kmer_count"]), M)


def import_counts_csv(csv_path: str, skmc_path: str) -> None:
    """Either CSV layout (learn.smk:328-357 pandas writer, :583-594 pyarrow writer) -> side-car."""
    from .rules import read_counts_csv

    t = read_counts_csv(csv_path)
    write_counts(skmc_path, t.rows, t.kmers, t.seq_count, t.kmer_count, t.M)


def export_totals_csv(skmc_path: str, csv_path: str) -> None:
    """kmer-counts-total.csv as the merge rule writes it (pyarrow layout, index column last)."""
    from .rules import write_totals_csv

    write_totals_csv(csv_path, read_counts(skmc_path))


def export_counts_csv(skmc_path: str, csv_path: str, total_seqs: Optional[int] = None) -> None:
    """kmer-counts-{nb}.csv as the learn rule writes it (pandas layout: index first, zeros blank)."""
    from .rules import LearnResult, write_counts_csv

    t = read_counts(skmc_path)
    assert t.rows and t.rows[0] == "Totals", "a per-file counts table starts with its Totals row"
    r = LearnResult(t.rows[1:], t.seq_count[1:], t.M[1:], t.M[0], int(t.seq_count[0]) if total_seqs is None else total_seqs, t.kmers)
    write_counts_csv(csv_path, r)


# ---------------------------------------------------------------------------
# association matrices (.skma)  ->  seq-annotation-scores-*.csv
# ---------------------------------------------------------------------------
INDEX_COL = "__index_level_0__"


class AssociationsWriter:
    """``.skma`` written block by block: the names and labels go first and the [Q, A] float64 array is laid out behind
    them up front, so write(q0, block) puts rows [q0, q0 + len(block)) straight at their place."""

    def __init__(self, path: str, annotations: Sequence[str], labels: Sequence[str]):
        ab, ao = _strings_to_arrays(annotations)
        lb, lo = _strings_to_arrays(labels)
        small = {"annotations": ab, "annotation_offsets": ao, "rows": lb, "row_offsets": lo}
        self.Q, self.A = len(labels), len(annotations)
        head, entries = _layout("associations", {"n_ann": self.A, "nrows": self.Q},
                                [(k, v.dtype, v.shape) for k, v in small.items()] + [("scores", np.dtype(np.float64), (self.Q, self.A))])
        self._f = open(path, "wb")
        self._f.write(head)
        for e in entries[:-1]:
            self._f.write(b"\0" * (e["offset"] - self._f.tell()))
            self._f.write(small[e["name"]].tobytes())
        self._base = entries[-1]["offset"]
        self._f.truncate(self._base + entries[-1]["nbytes"])

    def write(self, q0: int, block: np.ndarray) -> None:
        block = np.ascontiguousarray(block, dtype=np.float64)
        assert block.ndim == 2 and block.shape[1] == self.A and 0 <= q0 and q0 + block.shape[0] <= self.Q
        self._f.seek(self._base + q0 * self.A * 8)
        self._f.write(block.tobytes())

    def close(self) -> None:
        self._f.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class AssociationsCSVWriter:
    """The seq-annotation-scores CSV (annotations as float64 columns, the row labels last under ``__index_level_0__``)
    streamed through pyarrow's CSVWriter, one record batch per block: the bytes of one ``pyarrow.csv.write_csv`` of the
    whole table, which is how the reference and rules.apply_rule / eval_apply_rule write it.  Blocks come in row order."""

    def __init__(self, path: str, annotations: Sequence[str], labels: Sequence[str]):
        import pyarrow as pa
        from pyarrow import csv as pacsv

        self._pa = pa
        self._labels = [str(x) for x in labels]
        self.A = len(annotations)
        self._schema = pa.schema([(str(a), pa.float64()) for a in annotations] + [(INDEX_COL, pa.string())])
        self._w = pacsv.CSVWriter(path, self._schema)
        self._next = 0

    def write(self, q0: int, block: np.ndarray) -> None:
        assert q0 == self._next and block.ndim == 2 and block.shape[1] == self.A, "blocks in row order"
        n = block.shape[0]
        pa = self._pa
        arrays = [pa.array(np.ascontiguousarray(block[:, j], dtype=np.float64)) for j in range(self.A)]
        self._w.write_batch(pa.record_batch(arrays + [pa.array(self._labels[q0:q0 + n], type=pa.string())], schema=self._schema))
        self._next = q0 + n

    def close(self) -> None:
        self._w.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def associations_writer(path: str, annotations: Sequence[str], labels: Sequence[str]):
    """``.skma`` side-car for a path ending in .skma, the CSV otherwise."""
    cls = AssociationsWriter if str(path).endswith(".skma") else AssociationsCSVWriter
    return cls(path, annotations, labels)


def read_associations(path: str, mmap: bool = True) -> Dict:
    """annotations, rows (labels) and scores float64 [Q, A] (memory-mapped)."""
    kind, attrs, a = read_container(path, mmap)
    if kind != "associations":
        raise ValueError(f"{path}: holds '{kind}', not associations")
    return dict(annotations=_arrays_to_strings(a["annotations"], a["annotation_offsets"]),
                rows=_arrays_to_strings(a["rows"], a["row_offsets"]), scores=a["scores"])


def export_associations_csv(skma_path: str, csv_path: str, block_rows: int = 65536) -> None:
    """The seq-annotation-scores CSV of a ``.skma``, byte for byte what the direct writer gives."""
    d = read_associations(skma_path)
    S = d["scores"]
    with AssociationsCSVWriter(csv_path, d["annotations"], d["rows"]) as w:
        for q0 in range(0, S.shape[0], block_rows):
            w.write(q0, S[q0:q0 + block_rows])
