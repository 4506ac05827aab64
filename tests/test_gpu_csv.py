"""CSV interchange text formatted on the device (skm_csv.cu): float64 cells against pyarrow's CSV writer, association
rows and top-2-masked rows against sidecar.AssociationsCSVWriter / export_associations_csv, and count files against
the host writers (rules.write_counts_csv / write_totals_csv through the .skmc side-car) and the reference's files."""
import ctypes
import io
import os

import numpy as np
import pyarrow as pa
import pyarrow.csv as pacsv
import pytest
import torch

from util import GOLDEN, RULE_CONFIGS, load_rule

if torch.cuda.is_available():
    from snekmer_b200 import engine as E
    from snekmer_b200 import io as skio
    from snekmer_b200 import rules as R
    from snekmer_b200 import rules_sparse as RS
    from snekmer_b200 import sidecar as SC

LABELS_ODD = ["", "a,b", 'q"uote', "two\nlines", "é✓ü", '"', ",,", "plain"]


def _pyarrow_cells(values: np.ndarray) -> list:
    b = io.BytesIO()
    pacsv.write_csv(pa.table({"x": pa.array(values, type=pa.float64())}), b, pacsv.WriteOptions(include_header=False))
    return b.getvalue().split(b"\n")[:-1]


def _edge_values() -> np.ndarray:
    vals = []
    for e in range(-324, 309):
        v = float(f"1e{e}")
        vals += [v, np.nextafter(v, 0.0), np.nextafter(v, np.inf)]
    for k in range(-1074, 1024):
        vals += [np.ldexp(1.0, k), -np.ldexp(1.0, k)]
    vals += [2.2250738585072014e-308, 1.7976931348623157e308, 5e-324, 0.0, -0.0, np.inf, -np.inf, np.nan,
             2.0 ** 53 - 1, 2.0 ** 53 + 1, 2.0 ** 53, -1.2345678901234567e-06, 9999999999.5, 1e10, 0.30000000000000004]
    return np.array(vals, dtype=np.float64)


def test_host_formatter_matches_pyarrow():
    """The same __host__ __device__ formatter through its host entry point (no GPU needed)."""
    from snekmer_b200 import _native, build

    build.build()
    lib = _native.lib()
    buf = ctypes.create_string_buffer(32)
    rng = np.random.default_rng(7)
    for values in (_edge_values(), rng.integers(0, 2 ** 64, size=50000, dtype=np.uint64).view(np.float64), rng.random(50000)):
        want = _pyarrow_cells(values)
        got = []
        for v in values:
            n = lib.skm_csv_f64_host(float(v), buf)
            got.append(buf.raw[:n])
        assert got == want


def test_pow5_tables_match_generator():
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    assert subprocess.run([sys.executable, os.path.join(root, "scripts", "gen_csv_pow5.py"), "--check"]).returncode == 0


# ---- on the device ---------------------------------------------------------------------------------------------------
def _device_csv(block: np.ndarray, labels, chunk=None) -> bytes:
    """block float64 [Q, A] written through engine.AssociationsCSVText as an apply chunk would be."""
    import tempfile

    Q, A = block.shape
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "x.csv")
        w = E.AssociationsCSVText(path, [f"a{j}" for j in range(A)], labels)
        dblock = torch.from_numpy(np.ascontiguousarray(block)).cuda()
        chunk = chunk or max(Q, 1)
        pipe = w.pipe(chunk)
        for q0 in range(0, Q, chunk):
            s = pipe.slot()
            pipe.push(s, w.format_rows(q0, dblock[q0:q0 + chunk], pipe.text[s]))
        w.close()
        return open(path, "rb").read()


def _host_csv(block: np.ndarray, labels) -> bytes:
    b = io.BytesIO()
    Q, A = block.shape
    names = [f"a{j}" for j in range(A)]
    schema = pa.schema([(n, pa.float64()) for n in names] + [("__index_level_0__", pa.string())])
    tab = pa.table([pa.array(block[:, j]) for j in range(A)] + [pa.array(list(labels), type=pa.string())], schema=schema)
    pacsv.write_csv(tab, b)
    return b.getvalue()


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", [("bits", 10_000_000), ("unit", 10_000_000), ("edge", 0)])
def test_device_formatter_matches_pyarrow(name, n):
    rng = np.random.default_rng(11)
    if name == "bits":
        v = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64).view(np.float64)
    elif name == "unit":
        v = rng.random(n)
    else:
        v = _edge_values()
    labels = [""] * len(v)
    got = _device_csv(v[:, None], labels, chunk=3_000_001)
    assert got == _host_csv(v[:, None], labels)


@pytest.mark.gpu
@pytest.mark.parametrize("Q,A,chunk", [(37, 5, 10), (64, 1, None), (0, 4, None), (9, 0, 4), (200, 33, 7)])
def test_association_rows_match_host_writer(Q, A, chunk, tmp_path):
    rng = np.random.default_rng(Q * 100 + A)
    block = rng.random((Q, A))
    block[rng.random((Q, A)) < 0.2] = np.nan
    block[rng.random((Q, A)) < 0.1] = 0.0
    labels = [LABELS_ODD[q % len(LABELS_ODD)] + str(q) * (q % 3) for q in range(Q)]
    host = str(tmp_path / "host.csv")
    with SC.AssociationsCSVWriter(host, [f"a{j}" for j in range(A)], labels) as w:
        step = chunk or max(Q, 1)
        for q0 in range(0, Q, step):
            w.write(q0, block[q0:q0 + step])
    assert _device_csv(block, labels, chunk) == open(host, "rb").read()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [None, 5])
def test_top2_rows_match_host_masking(chunk, tmp_path):
    rng = np.random.default_rng(3)
    Q, A = 41, 6
    top1 = rng.integers(-1, A, size=Q).astype(np.int32)
    top2 = np.where(rng.random(Q) < 0.3, -1, (top1 + 1) % A).astype(np.int32)
    s1, s2 = rng.random(Q), rng.random(Q)
    r = E.ApplyResult(*(torch.from_numpy(x).cuda() for x in (top1, top2, s1, s2)))
    labels = [LABELS_ODD[q % len(LABELS_ODD)] for q in range(Q)]
    anns = [f"ann{j}" for j in range(A)]
    host, dev = str(tmp_path / "host.csv"), str(tmp_path / "dev.csv")
    with SC.AssociationsCSVWriter(host, anns, labels) as w:
        RS._write_top2_rows(w, r, A)
    with E.AssociationsCSVText(dev, anns, labels) as w:
        E.write_top2_csv(w, r, chunk)
    assert open(dev, "rb").read() == open(host, "rb").read()


def _learn_rule_files(name, tmp_path):
    a, k, mf = RULE_CONFIGS[name]
    a = None if a == "None" else (int(a) if str(a).isdigit() else a)
    seq_annot = R.load_annotations([os.path.join(GOLDEN, "syn.ann")])
    out = {}
    for nb in ("synA", "synB"):
        npz = str(tmp_path / f"{nb}.npz")
        R.vectorize_rule(os.path.join(GOLDEN, f"{nb}.fasta"), npz, None, a, k, min_filter=mf)
        kl, df = skio.load_npz(npz)
        kmerlist = [str(x) for x in kl[0]]
        sc = RS.learn_counts_sparse(list(df["sequence_id"]), list(df["sequence"]), "".join(sorted(set("".join(kmerlist)))), k, seq_annot)
        out[nb] = (df, kmerlist, sc)
    return out, seq_annot


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hydro_k8", "miqs_k3", "solvacc_k4"])
def test_rule_files_match_reference_and_export(name, tmp_path):
    d = load_rule(name)
    files, seq_annot = _learn_rule_files(name, tmp_path)
    for nb, (df, kmerlist, sc) in files.items():
        out = tmp_path / f"kmer-counts-{nb}.csv"
        RS.write_counts_csv(str(out), sc, kmers=kmerlist)
        assert out.read_bytes() == d[f"{nb}_counts_csv"].tobytes()
    merged = RS.merge_counts_sparse([f[2] for f in files.values()])
    side = str(tmp_path / "merged.skmc")
    RS.write_counts_sidecar(side, merged)
    for layout, export in (("total", SC.export_totals_csv), ("learn", SC.export_counts_csv)):
        want, got = tmp_path / f"want-{layout}.csv", tmp_path / f"got-{layout}.csv"
        export(side, str(want))
        RS.write_counts_csv(str(got), merged, layout=layout)
        assert got.read_bytes() == want.read_bytes()
    # the merged matrix in the reference's merged column order gives its kmer-counts-total.csv
    ref = tmp_path / "ref-total.csv"
    ref.write_bytes(d["totals_csv"].tobytes())
    t = R.read_counts_csv(str(ref))
    got = tmp_path / "total.csv"
    RS.write_counts_csv(str(got), merged, kmers=t.kmers, layout="total")
    assert got.read_bytes() == ref.read_bytes()
    # synA alone through the merge rule: kmer-counts-total.csv of the one-file merge
    refA = tmp_path / "ref-totalA.csv"
    refA.write_bytes(d["totalsA_csv"].tobytes())
    gotA = tmp_path / "totalA.csv"
    RS.write_counts_csv(str(gotA), RS.merge_counts_sparse([files["synA"][2]]), kmers=R.read_counts_csv(str(refA)).kmers, layout="total")
    assert gotA.read_bytes() == refA.read_bytes()
    # association files of the sparse rule bodies: the device CSV == export of the same call's .skma, top-2 bit-equal
    df, kmerlist, _ = files["synB"]
    ids, seqs = list(df["sequence_id"]), list(df["sequence"])
    for save in (True, False):
        csv, skma = str(tmp_path / f"e{save}.csv"), str(tmp_path / f"e{save}.skma")
        a = RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist, out_scores=csv, save_associations=save, chunk_rows=6)
        b = RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist, out_scores=skma, save_associations=save)
        c = RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist)
        SC.export_associations_csv(skma, str(tmp_path / "back.csv"))
        assert open(csv, "rb").read() == open(tmp_path / "back.csv", "rb").read()
        for x in (b, c):
            for f in ("top1", "top2", "score1", "score2"):
                assert np.array_equal(getattr(a, f).cpu().numpy(), getattr(x, f).cpu().numpy(), equal_nan=True)
    csv, skma = str(tmp_path / "apply.csv"), str(tmp_path / "apply.skma")
    r1 = RS.apply_counts_sparse(ids, seqs, files["synA"][2], out_scores=csv, save_associations=True, chunk_rows=5, query_kmers=kmerlist)
    r2 = RS.apply_counts_sparse(ids, seqs, files["synA"][2], out_scores=skma, save_associations=True, query_kmers=kmerlist)
    SC.export_associations_csv(skma, str(tmp_path / "apply.back.csv"))
    assert open(csv, "rb").read() == open(tmp_path / "apply.back.csv", "rb").read()
    assert np.array_equal(r1.top1, r2.top1) and np.array_equal(r1.top2, r2.top2)
    assert np.array_equal(r1.score1, r2.score1) and np.array_equal(r1.score2, r2.score2, equal_nan=True)


def _random_counts(seed, A, symbols, k, vmax, wide=False):
    """A random SparseCounts over (symbols, k): empty annotation rows, values up to vmax."""
    rng = np.random.default_rng(seed)
    dev = torch.device("cuda")
    S = len(symbols) ** k
    if wide:
        K = 300
        codes = np.unique(rng.integers(0, S, size=K, dtype=np.uint64))
        columns = E.wide_basis_from_codes(codes, E.alphabet_tables_from_symbols(symbols, dev), k, dev)
        stride = columns.K
    else:
        columns, stride = None, S
    keys = []
    for a in range(A):
        if a % 3 == 1:
            continue
        n = 1 if a == 0 else int(rng.integers(1, 40))        # row 0 holds the one 2^63 - 1 entry alone
        keys.append(a * stride + np.unique(rng.integers(0, stride, size=n)))
    key = np.concatenate(keys).astype(np.int64) if keys else np.zeros(0, np.int64)
    val = rng.integers(1, vmax, size=key.size, dtype=np.int64)
    if key.size:
        val[0] = (1 << 63) - 1
    totals = np.zeros(stride, dtype=np.int64)
    np.add.at(totals, key % stride if key.size else key, np.minimum(val, 1 << 40))
    totals[rng.integers(0, stride, size=5)] += 3
    return RS.SparseCounts([f'ann"{a},x' if a % 4 == 0 else f"a{a}" for a in range(A)], rng.integers(0, 9, size=A).astype(np.int64),
                           symbols, k, torch.from_numpy(key).to(dev), torch.from_numpy(val).to(dev), torch.from_numpy(totals).to(dev),
                           int(rng.integers(0, 100)), columns)


@pytest.mark.gpu
@pytest.mark.parametrize("A,symbols,k,wide", [(9, "ACDE", 3, False), (1, "AC", 2, False), (0, "ACD", 2, False), (7, "ACDEFGHIKLMNPQRSTVWY", 7, True)])
def test_random_counts_match_host_export(A, symbols, k, wide, tmp_path):
    sc = _random_counts(A * 10 + k, A, symbols, k, 1000, wide)
    side = str(tmp_path / "m.skmc")
    RS.write_counts_sidecar(side, sc)
    for layout, export in (("learn", SC.export_counts_csv), ("total", SC.export_totals_csv)):
        want, got = tmp_path / f"want-{layout}.csv", tmp_path / f"got-{layout}.csv"
        export(side, str(want))
        RS.write_counts_csv(str(got), sc, layout=layout)
        assert got.read_bytes() == want.read_bytes(), layout


@pytest.mark.gpu
def test_c1_files(tmp_path):
    """C1 (two UniProt proteomes, alphabet 2, k = 8): count files against the host exports, association CSVs of
    eval_apply with and without save_associations and of apply against the exports of the same calls' .skma."""
    C1 = os.path.join(GOLDEN, "c1")
    seq_annot = R.load_annotations([os.path.join(C1, "c1.ann")])
    parts, frames = [], []
    for nb in ("UP000322080_2603819", "UP000322981_424902"):
        npz = str(tmp_path / f"{nb}.npz")
        R.vectorize_rule(os.path.join(C1, nb + ".fasta.gz"), npz, None, 2, 8)
        kl, df = skio.load_npz(npz)
        kmerlist = [str(x) for x in kl[0]]
        frames.append((df, kmerlist))
        sc = RS.learn_counts_sparse(list(df["sequence_id"]), list(df["sequence"]), "".join(sorted(set("".join(kmerlist)))), 8, seq_annot)
        parts.append(sc)
        side, want, got = str(tmp_path / f"{nb}.skmc"), tmp_path / f"{nb}.want.csv", tmp_path / f"{nb}.got.csv"
        RS.write_counts_sidecar(side, sc, kmers=kmerlist)
        SC.export_counts_csv(side, str(want))
        RS.write_counts_csv(str(got), sc, kmers=kmerlist)
        assert got.read_bytes() == want.read_bytes()
    merged = RS.merge_counts_sparse(parts)
    side, want, got = str(tmp_path / "m.skmc"), tmp_path / "m.want.csv", tmp_path / "m.got.csv"
    RS.write_counts_sidecar(side, merged)
    SC.export_totals_csv(side, str(want))
    RS.write_counts_csv(str(got), merged, layout="total")
    assert got.read_bytes() == want.read_bytes()
    _same_counts(RS.read_counts_csv(str(got)), RS.read_counts_sidecar(side))
    df, kmerlist = frames[1]
    ids, seqs = list(df["sequence_id"]), list(df["sequence"])
    for save in (True, False):
        csv, skma = str(tmp_path / f"e{save}.csv"), str(tmp_path / f"e{save}.skma")
        a = RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist, out_scores=csv, save_associations=save, chunk_rows=300)
        b = RS.eval_counts_sparse(ids, seqs, merged, seq_annot, query_kmers=kmerlist, out_scores=skma, save_associations=save)
        SC.export_associations_csv(skma, str(tmp_path / "back.csv"))
        assert open(csv, "rb").read() == open(tmp_path / "back.csv", "rb").read()
        for f in ("top1", "top2", "score1", "score2"):
            assert np.array_equal(getattr(a, f).cpu().numpy(), getattr(b, f).cpu().numpy(), equal_nan=True)
    csv, skma = str(tmp_path / "apply.csv"), str(tmp_path / "apply.skma")
    r1 = RS.apply_counts_sparse(ids, seqs, parts[0], out_scores=csv, save_associations=True, query_kmers=kmerlist)
    r2 = RS.apply_counts_sparse(ids, seqs, parts[0], out_scores=skma, save_associations=True, query_kmers=kmerlist)
    SC.export_associations_csv(skma, str(tmp_path / "apply.back.csv"))
    assert open(csv, "rb").read() == open(tmp_path / "apply.back.csv", "rb").read()
    for f in ("top1", "top2", "score1", "score2"):
        assert np.array_equal(getattr(r1, f), getattr(r2, f), equal_nan=True)


# ---- the count-CSV parser ---------------------------------------------------------------------------------------------
def _same_counts(a, b):
    assert a.annotations == b.annotations and a.symbols == b.symbols and a.k == b.k and a.total_seqs == b.total_seqs
    assert np.array_equal(a.seq_count, b.seq_count)
    assert torch.equal(a.keys, b.keys) and torch.equal(a.vals, b.vals) and torch.equal(a.totals, b.totals)
    assert (a.columns is None) == (b.columns is None)
    if a.columns is not None:
        assert torch.equal(a.columns.codes, b.columns.codes)


def _golden_csvs():
    out = []
    for name in ("hydro_k8", "miqs_k3", "solvacc_k4"):
        d = load_rule(name)
        out += [(f"{name}:{key}", d[key]) for key in ("synA_counts_csv", "synB_counts_csv", "totals_csv", "totalsA_csv")]
    d = np.load(os.path.join(GOLDEN, "merge_base.npz"))
    out += [(f"merge_base:{key}", d[key]) for key in d.files]
    return out


@pytest.mark.gpu
def test_parser_matches_host_import_on_golden_csvs(tmp_path):
    for name, raw in _golden_csvs():
        p = tmp_path / (name.replace(":", "_") + ".csv")
        p.write_bytes(raw.tobytes())
        side = str(tmp_path / "x.skmc")
        SC.import_counts_csv(str(p), side)
        want = RS.read_counts_sidecar(side)
        _same_counts(RS.read_counts_csv(str(p)), want)
        _same_counts(RS.read_counts_csv(str(p), block_bytes=64), want)       # rows straddle many blocks


@pytest.mark.gpu
@pytest.mark.parametrize("A,symbols,k,wide", [(9, "ACDE", 3, False), (7, "ACDEFGHIKLMNPQRSTVWY", 7, True)])
def test_parser_round_trips_device_files(A, symbols, k, wide, tmp_path):
    sc = _random_counts(A * 7 + k, A, symbols, k, 1000, wide)
    sc.annotations[1] = 'line\nbreak, "quoted"'
    sc.annotations[2] = ""
    side = str(tmp_path / "m.skmc")
    RS.write_counts_sidecar(side, sc)
    want = RS.read_counts_sidecar(side, symbols=symbols)
    for layout in ("learn", "total"):
        p = str(tmp_path / f"{layout}.csv")
        RS.write_counts_csv(p, sc, layout=layout)
        for block in (E.CSV_PARSE_BLOCK, 5, 333):
            _same_counts(RS.read_counts_csv(p, symbols=symbols, block_bytes=block), want)


def _write(tmp_path, text):
    p = tmp_path / "c.csv"
    p.write_bytes(text.encode("utf-8"))
    return str(p)


@pytest.mark.gpu
def test_parser_grammar(tmp_path):
    head = '__index_level_0__,Sequence count,Kmer Count,AC,CA,"A""C"\n'
    p = _write(tmp_path, head + "Totals,3,12.0,1e+10,,1.2345678901e+10\n\"x,\ny\",1,2.000,,2,\n")
    labels, kmers, sq, kc, rowptr, cols, vals = E.parse_counts_csv(p)
    assert labels == ["Totals", "x,\ny"] and kmers == ["AC", "CA", 'A"C']
    assert sq.tolist() == [3, 1] and kc.tolist() == [12, 2]
    assert rowptr.tolist() == [0, 2, 3] and cols.tolist() == [0, 2, 1] and vals.tolist() == [10 ** 10, 12345678901, 2]
    for cell, col in (("1.5", "AC"), ("abc", "AC"), ("-3", "AC"), ("1e-1", "AC"), ("9223372036854775808", "AC"), ("1 ", "AC")):
        p = _write(tmp_path, head + "Totals,1,1,1,1,1\n" + f"a,1,1,{cell},1,1\n")
        with pytest.raises(E.SkmError, match=f"line 3, column '{col}'"):
            E.parse_counts_csv(p)
    p = _write(tmp_path, head + "Totals,1,1,1,1\n")
    with pytest.raises(E.SkmError, match="line 2"):
        E.parse_counts_csv(p)
    p = _write(tmp_path, head)
    labels, kmers, sq, kc, rowptr, cols, vals = E.parse_counts_csv(p)
    assert labels == [] and kmers == ["AC", "CA", 'A"C'] and rowptr.tolist() == [0] and cols.numel() == 0
    # the largest value and a file without a final newline
    p = _write(tmp_path, head + "Totals,1,9223372036854775807,9223372036854775807,0,0")
    assert E.parse_counts_csv(p)[6].tolist() == [(1 << 63) - 1]
