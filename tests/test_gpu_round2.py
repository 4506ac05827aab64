"""GPU parity tests added in round 2: order-only basis walk with device-side early exit, per-row fallback of the
tensor-core scoring, compact count transports, host pipelines."""
import numpy as np
import pytest
import torch

from oracle import skm_oracle as O
from snekmer_b200 import engine as E

pytestmark = pytest.mark.gpu

AA = np.array(list("ACDEFGHIKLMNPQRSTVWYX"))


def _rand_seqs(rng, n, lo, hi, p_x=0.02):
    p = np.full(21, (1 - p_x) / 20)
    p[-1] = p_x
    return ["".join(rng.choice(AA, size=int(rng.integers(lo, hi)), p=p)) for _ in range(n)]


def _oracle_basis(seqs, a, k, mf=0):
    lut, syms = O.build_lut(a)
    res, offs = O.pack(seqs)
    si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
    basis, cnt = O.basis_codes(si, pos, code, valid, mf)
    return basis, cnt, (si, code, valid)


@pytest.mark.parametrize("a,k,n,first_chunk", [("miqs", 3, 3000, 1 << 12), ("miqs", 3, 3000, 1 << 30), (2, 8, 4000, 1 << 14),
                                               (0, 9, 2500, 1 << 10), ("standard", 4, 500, 1 << 9), (None, 3, 1500, 1 << 13)])
def test_order_only_basis_equals_full_basis(a, k, n, first_chunk, monkeypatch):
    """build_basis(counts=False): same basis (order included) as the full pass and as the oracle, whether the space
    saturates in the first chunk, in a later one, or never."""
    rng = np.random.default_rng(k * 100 + n)
    seqs = _rand_seqs(rng, n, 0, 300)
    seqs[5] = ""
    batch = E.SequenceBatch.from_strings(seqs)
    want, _, _ = _oracle_basis(seqs, a, k)
    monkeypatch.setattr(E, "ORDER_FIRST_CHUNK_RES", first_chunk)
    monkeypatch.setattr(E, "ORDER_GROWTH", 2)
    b = E.build_basis(batch, a, k, 0, counts=False)
    assert b.counts is None
    assert np.array_equal(b.codes_host(), want)
    full = E.build_basis(batch, a, k, 0)
    assert torch.equal(full.codes, b.codes) and torch.equal(full.col_of_code, b.col_of_code)
    C = E.count_dense(batch, a, k, b)
    assert torch.equal(C.sum(dim=0, dtype=torch.int64), full.counts)


def test_order_only_basis_early_exit_state():
    """The walk really stops: a saturated space leaves state[0] = 1 and first positions inside the scanned prefix;
    k-mers that only occur at the very end are still found when the space never saturates."""
    rng = np.random.default_rng(7)
    seqs = _rand_seqs(rng, 6000, 50, 300, p_x=0.0)
    batch = E.SequenceBatch.from_strings(seqs)
    tab = E.alphabet_tables("hydro", batch.device)       # 2 letters, k = 4: 16 codes, saturated within a few residues
    S = tab.nsym ** 4
    first = torch.full((S,), -1, dtype=torch.int64, device=batch.device)
    state = torch.zeros(4, dtype=torch.int32, device=batch.device)
    old = E.ORDER_FIRST_CHUNK_RES
    try:
        E.ORDER_FIRST_CHUNK_RES = 1 << 12
        E.basis_first_progressive(batch, "hydro", 4, first, state, 0)
    finally:
        E.ORDER_FIRST_CHUNK_RES = old
    st = state.cpu().numpy()
    assert st[0] == 1 and st[2] == S and st[1] == 0
    assert int(first.max().item()) < (1 << 12) + 400
    # rare k-mer at the end of the shard: 'W' only in the last sequence (None alphabet, k = 2 -> WW)
    seqs2 = ["".join(rng.choice(AA[:18], size=200)) for _ in range(3000)] + ["AWWA"]
    b2 = E.build_basis(E.SequenceBatch.from_strings(seqs2), None, 2, 0, counts=False)
    want, _, _ = _oracle_basis(seqs2, None, 2)
    assert np.array_equal(b2.codes_host(), want)


def test_apply_tc_per_row_fallback_long_homopolymer():
    """One 60k-residue homopolymer (a count of ~60,000 in one column) inside a large batch: only that row leaves the
    tensor-core path; every row equals the exact CUDA-core result bit for bit."""
    rng = np.random.default_rng(3)
    a, k = "miqs", 3
    seqs = _rand_seqs(rng, 20000, 30, 400)
    seqs[777] = "A" * 60000
    seqs[12345] = "L" * 300 + "".join(rng.choice(AA[:20], size=100))          # a count of 298: just over 255
    batch = E.SequenceBatch.from_strings(seqs)
    Q = E.count_dense(batch, a, k, None)
    M = torch.from_numpy(rng.integers(0, 50, size=(300, Q.shape[1]), dtype=np.int64) * (rng.random((300, Q.shape[1])) < 0.4)).cuda()
    prep = E.prepare_annotations(M)
    bad = E.rows_out_of_range(Q, 0, 255)
    assert bad.tolist() == [777, 12345]
    tc = E.apply_tc(Q, prep)
    exact = E.apply_dense(Q, M, tensor_cores=False)
    assert torch.equal(tc.top1, exact.top1) and torch.equal(tc.top2, exact.top2)
    assert torch.allclose(tc.score1, exact.score1, rtol=1e-14, atol=0) and torch.allclose(tc.score2, exact.score2, rtol=1e-14, atol=0)
    assert torch.equal(tc.score1[bad], exact.score1[bad])


@pytest.mark.parametrize("dtype", [torch.int32, torch.uint16])
@pytest.mark.parametrize("rows,cols", [(1, 1), (37, 1000), (200, 6561), (513, 27), (64, 3)])
def test_pack_counts_u8_and_presence_bits(dtype, rows, cols):
    from snekmer_b200 import pipeline as P

    rng = np.random.default_rng(rows * cols)
    X = (rng.integers(0, 40, size=(rows, cols)) * (rng.random((rows, cols)) < 0.3)).astype(np.int64)
    X[rng.integers(0, rows), rng.integers(0, cols)] = 255
    X[rng.integers(0, rows), rng.integers(0, cols)] = 254
    X[rng.integers(0, rows), rng.integers(0, cols)] = 60000
    X[0, 0] = 256
    d = torch.from_numpy(X.astype(np.int32)).cuda().to(dtype) if dtype == torch.int32 else torch.from_numpy(X.astype(np.uint16)).cuda()
    u8, er, ec, evv = P.pack_counts_u8(d)
    got = P.unpack_counts_u8(u8.cpu().numpy(), er.cpu().numpy(), ec.cpu().numpy(), evv.cpu().numpy())
    assert np.array_equal(got, X)
    assert int((u8 == 255).sum().item()) == er.numel() == int((X >= 255).sum())
    bits = P.pack_presence_bits(d)
    assert tuple(bits.shape) == (rows, (cols + 7) // 8)
    assert np.array_equal(np.unpackbits(bits.cpu().numpy(), axis=1, bitorder="little")[:, :cols], (X > 0).astype(np.uint8))


@pytest.mark.parametrize("transport", ["int32", "uint16", "uint8", "bits"])
def test_vectorize_host_transports_match_oracle(transport):
    from snekmer_b200 import pipeline as P

    rng = np.random.default_rng(11)
    seqs = _rand_seqs(rng, 5000, 0, 500)
    seqs[17] = "G" * 1000                                                  # a count of 998 -> escape list of the uint8 transport
    a, k = "miqs", 3
    res, offs = E.SequenceBatch.pack_host(seqs)
    want_basis, _, (si, code, valid) = _oracle_basis(seqs, a, k)
    want = O.count_matrix(si, code, valid, len(seqs), want_basis)
    h_res = torch.from_numpy(res.copy()).pin_memory()
    r = P.vectorize_host(h_res, offs, a, k, transport=transport, n_chunks=5)
    assert np.array_equal(r.basis.codes_host(), want_basis)
    if transport == "bits":
        assert np.array_equal(r.presence(), (want > 0))
    else:
        assert np.array_equal(r.counts(), want)
        assert r.counts().dtype == np.int32


def test_apply_host_matches_device_path():
    from snekmer_b200 import pipeline as P

    rng = np.random.default_rng(5)
    a, k = "miqs", 3
    train = _rand_seqs(rng, 3000, 30, 300)
    ann = rng.integers(0, 200, size=len(train)).astype(np.int32)
    tb = E.SequenceBatch.from_strings(train)
    M, _ = E.learn_dense(tb, a, k, None, torch.from_numpy(ann), 200)
    M = M[:200].contiguous()
    prep = E.prepare_annotations(M)
    queries = _rand_seqs(rng, 7000, 0, 400)
    queries[3] = "A" * 3000
    res, offs = E.SequenceBatch.pack_host(queries)
    h = P.apply_host(torch.from_numpy(res.copy()).pin_memory(), offs, a, k, prep, n_chunks=3)
    qb = E.SequenceBatch.from_strings(queries)
    Q = E.count_dense(qb, a, k, None)
    want = E.apply_dense(Q, M, tensor_cores=False)
    assert np.array_equal(h.top1, want.top1.cpu().numpy()) and np.array_equal(h.top2, want.top2.cpu().numpy())
    assert np.allclose(h.score1, want.score1.cpu().numpy(), rtol=1e-14, atol=0)
    assert np.allclose(h.score2, want.score2.cpu().numpy(), rtol=1e-14, atol=0)
    S = O.cosine_scores(Q.cpu().numpy(), M.cpu().numpy())
    i1, _, s1, _ = O.top2(S)
    assert np.array_equal(h.top1, i1) and np.max(np.abs(h.score1 - s1)) < 1e-12


def test_apply_sparse_64bit_accumulators_with_many_annotations():
    """ADVICE r1: more than 25,600 annotations AND dots that need 64-bit accumulators (max(M) * query total >= 2^32):
    the annotation tile follows the accumulator width; results equal the dense float64 oracle."""
    rng = np.random.default_rng(64)
    a, k = "hydro", 10                                   # 2 letters: S = 1024
    S, n_ann = 1024, 30000
    nnz = 200000
    ann = np.sort(rng.integers(0, n_ann, size=nnz))
    code = rng.integers(0, S, size=nnz)
    key = np.unique(ann.astype(np.int64) * S + code)
    val = rng.integers(1, 50, size=key.size).astype(np.int64)
    val[5] = 70000                                       # >= 65536: unpacked CSC, and 70000 * 70000 >= 2^32
    keys, vals = torch.from_numpy(key).cuda(), torch.from_numpy(val).cuda()
    queries = _rand_seqs(rng, 300, 0, 300, p_x=0.0) + ["".join(rng.choice(list("AV"), size=70100))]
    qb = E.SequenceBatch.from_strings(queries)
    rowptr, cols, cvals = E.count_csr(qb, a, k, None)
    row_total = E.query_row_total_max(rowptr, cvals)
    assert E.sparse_acc_bits(70000, row_total) == 64 and E.sparse_max_ann(64) < n_ann
    with pytest.raises(E.SkmError):
        E.apply_sparse(rowptr, cols, cvals, E.csc_build(keys, vals, S, n_ann, 0), row_total)
    r = E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann)
    lut, syms = O.build_lut(a)
    res, offs = O.pack(queries)
    si, pos, codes, valid = O.window_codes(res, offs, lut, len(syms), k)
    Q = O.count_matrix(si, codes, valid, len(queries), np.arange(S, dtype=np.uint64))
    M = np.zeros((n_ann, S), dtype=np.int64)
    M[key // S, key % S] = val
    Sc = O.cosine_scores(Q, M)
    i1, i2, s1, s2 = O.top2(Sc)
    assert np.allclose(r.score1.cpu().numpy(), s1, rtol=1e-12, atol=1e-15) and np.allclose(r.score2.cpu().numpy(), s2, rtol=1e-12, atol=1e-15)
    clear = (s1 - s2) > 1e-12 * np.maximum(s1, 1e-30)
    assert np.array_equal(r.top1.cpu().numpy()[clear], i1[clear])
    # empty inputs give -1 / NaN on both sparse entry points
    e = E.apply_sparse_tiled(rowptr, cols, cvals, keys[:0], vals[:0], S, 0)
    assert int(e.top1.max().item()) == -1 and bool(torch.isnan(e.score1).all())


def test_apply_counts_sparse_query_kmerlist_restriction():
    """ADVICE r1: with the query file's kmerlist (min_filter > 0) the sparse rule's norm runs over that list only, like
    the dense rule and the reference (apply.smk:262-289)."""
    from snekmer_b200 import rules as R
    from snekmer_b200 import rules_sparse as RS

    rng = np.random.default_rng(9)
    a, k = 2, 6
    ids = [f"tr|T{i:04d}|x" for i in range(400)]
    seqs = _rand_seqs(rng, 400, 20, 200, p_x=0.0)
    ann = {f"T{i:04d}": f"FAM{int(rng.integers(0, 9))}" for i in range(400) if rng.random() < 0.8}
    red = [O.reduce_str(s, a) for s in seqs]
    syms = "".join(sorted(O.symbols_of(a)))
    sc = RS.learn_counts_sparse(ids, red, syms, k, ann)
    q_ids = [f"tr|Q{i:04d}|y" for i in range(150)]
    q_seqs = _rand_seqs(rng, 150, 10, 200, p_x=0.0)
    q_red = [O.reduce_str(s, a) for s in q_seqs]
    qb = E.SequenceBatch.from_strings(q_seqs)
    q_basis = E.build_basis(qb, a, k, 12)                                   # min_filter = 12 drops the rarer k-mers
    q_kmers = list(q_basis.kmers())
    assert 0 < len(q_kmers) < len(syms) ** k
    all_kmers = list(E.decode_kmers(np.arange(len(syms) ** k, dtype=np.uint64), syms, k))
    lr = R.learn_counts(ids, red, all_kmers, ann)
    table = R.CountsTable(["Totals"] + lr.annotations, all_kmers, np.concatenate([[lr.total_seqs], lr.seq_count]),
                          np.concatenate([[lr.totals.sum()], lr.M.sum(axis=1)]), np.concatenate([lr.totals[None], lr.M]))
    want = R.cosine_top2(q_red, q_kmers, table)
    got = RS.apply_counts_sparse(q_ids, q_red, sc, query_kmers=q_kmers)
    assert got.annotations == lr.annotations
    assert np.allclose(got.score1, want.score1.cpu().numpy(), rtol=1e-12, atol=1e-15)
    assert np.allclose(got.score2, want.score2.cpu().numpy(), rtol=1e-12, atol=1e-15)
    loose = RS.apply_counts_sparse(q_ids, q_red, sc)                        # without the list: norm over all windows
    assert not np.allclose(loose.score1, got.score1)


@pytest.mark.parametrize("a,k,n", [(None, 4, 300), (None, 8, 200)])
def test_vectorize_rule_beyond_the_dense_envelope(a, k, n, tmp_path):
    """ADVICE r1: the vectorize rule body no longer hard-fails when the basis has more than 51,200 k-mers (table space,
    CSR counts) or the code space exceeds 2^27 (sort-based wide path): same kmerlist / presence matrix as the oracle;
    learn / apply on such a basis name the sparse rule bodies."""
    from snekmer_b200 import rules as R

    rng = np.random.default_rng(k)
    seqs = _rand_seqs(rng, n, 100, 500, p_x=0.01)
    ids = [f"tr|W{i:04d}|w" for i in range(n)]
    r = R.vectorize_records(ids, seqs, a, k)
    want_basis, _, (si, code, valid) = _oracle_basis(seqs, a, k)
    lut, syms = O.build_lut(a)
    assert r.counts is None and r.csr is not None and len(r.kmerlist) == len(want_basis) > R.DENSE_MAX_K
    assert list(r.kmerlist) == list(O.decode(want_basis, syms, k))
    C = O.count_matrix(si, code, valid, n, want_basis)
    assert np.array_equal(r.vecs(), (C > 0).astype(np.float64))
    rowptr, cols, vals = (t.cpu().numpy() for t in r.csr)
    dense = np.zeros_like(C)
    dense[np.repeat(np.arange(n), np.diff(rowptr)), cols] = vals
    assert np.array_equal(dense, C)
    side = str(tmp_path / "w.skmv")
    r.write_sidecar(side, a, k)
    from snekmer_b200 import sidecar as SC
    SC.export_npz(side, str(tmp_path / "w.npz"))
    z = np.load(str(tmp_path / "w.npz"))
    assert list(z["kmerlist"]) == list(r.kmerlist) and np.array_equal(z["vecs"], r.vecs())
    with pytest.raises(E.SkmError, match="rules_sparse"):
        R.learn_counts(ids, r.seqs, list(r.kmerlist), {})


@pytest.mark.parametrize("a,k,n_seq,n_ann,zipf,frac_un,div", [
    ("hydro", 10, 3000, 50, 1.1, 0.3, 4),       # S = 1024: almost every annotation is heavy
    (2, 8, 4000, 300, 1.1, 0.3, 4),             # S = 6561: a heavy head, a light tail, adjacent heavy ids
    (2, 8, 4000, 300, 0.0, 0.0, 4),             # uniform sizes: nothing heavy without the rest row
    ("miqs", 3, 2000, 40, 1.5, 0.5, 1),         # S = 1000, threshold S: only the biggest families
    (5, 4, 1500, 7, 1.1, 0.9, 4),               # few annotations, mostly unannotated
    (2, 8, 600, 5, 1.1, 0.0, 1 << 30),          # threshold 0: EVERY annotation is heavy, the light list is empty
    (2, 8, 600, 300, 0.0, 0.2, 4),              # no heavy annotation: the light list alone, Totals added on the way
])
def test_learn_sparse_hybrid_equals_sorted(a, k, n_seq, n_ann, zipf, frac_un, div):
    """Dense-row counting of the heavy annotations + sort of the light ones == the all-sorted path, bit for bit (keys,
    values, Totals), and == the oracle's dense matrix."""
    rng = np.random.default_rng(n_seq + n_ann)
    seqs = _rand_seqs(rng, n_seq, 0, 300)
    w = 1.0 / np.arange(1, n_ann + 1) ** zipf
    ann = rng.permutation(n_ann)[rng.choice(n_ann, size=n_seq, p=w / w.sum())].astype(np.int32)      # heavy ids scattered
    ann[rng.random(n_seq) < frac_un] = -1
    ann[:3] = [n_ann + 5, -7, n_ann]                                      # ids outside [0, n_ann) count as unannotated
    lut, syms = O.build_lut(a)
    S = len(syms) ** k
    ok = (ann >= 0) & (ann < n_ann)
    per_ann = np.bincount(ann[ok], weights=np.array([len(s) for s in seqs])[ok], minlength=n_ann)
    if (n_seq, n_ann) == (600, 300):
        assert per_ann.max() <= S // div
    batch = E.SequenceBatch.from_strings(seqs)
    d_ann = torch.from_numpy(ann)
    k1, v1, t1 = E.learn_sparse_with_totals(batch, a, k, d_ann, n_ann, method="sorted")
    k2, v2, t2 = E.learn_sparse_hybrid(batch, a, k, d_ann, n_ann, want_totals=True, heavy_div=div)
    assert torch.equal(k1, k2) and torch.equal(v1, v2) and torch.equal(t1, t2)
    k3, v3 = E.learn_sparse_hybrid(batch, a, k, d_ann, n_ann, want_totals=False, heavy_div=div)
    assert torch.equal(k1, k3) and torch.equal(v1, v3)
    res, offs = O.pack(seqs)
    si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
    C = O.count_matrix(si, code, valid, n_seq, np.arange(S, dtype=np.uint64)).astype(np.int64)
    M = np.zeros((n_ann, S), dtype=np.int64)
    np.add.at(M, ann[ok], C[ok])
    got = np.zeros_like(M)
    kk = k2.cpu().numpy()
    got[kk // S, kk % S] = v2.cpu().numpy()
    assert np.array_equal(got, M) and np.array_equal(t2.cpu().numpy(), C.sum(axis=0))
    assert bool((k2[1:] > k2[:-1]).all()) if k2.numel() > 1 else True


def test_learn_sparse_hybrid_falls_back_to_sorted(monkeypatch):
    """Inputs the grouped sort cannot take get the all-sorted result, bit for bit: a slice of GROUP_MAX_RES residues or
    more (the limit lowered below one slice; heavy rows are counted first), an empty batch, no annotations."""
    a, k, n_ann = 2, 8, 300
    rng = np.random.default_rng(77)
    seqs = _rand_seqs(rng, 4000, 0, 300)
    w = 1.0 / np.arange(1, n_ann + 1) ** 1.1
    ann = rng.permutation(n_ann)[rng.choice(n_ann, size=len(seqs), p=w / w.sum())].astype(np.int32)
    ann[rng.random(len(seqs)) < 0.3] = -1
    S = len(O.build_lut(a)[1]) ** k
    ok = ann >= 0
    per_ann = np.bincount(ann[ok], weights=np.array([len(s) for s in seqs])[ok], minlength=n_ann)
    assert per_ann.max() > S // E.HEAVY_ROW_DIV                          # the input has heavy rows
    batch, d_ann = E.SequenceBatch.from_strings(seqs), torch.from_numpy(ann)
    empty, no_ids = E.SequenceBatch.from_strings([]), torch.zeros(0, dtype=torch.int32)
    k1, v1, t1 = E.learn_sparse_with_totals(batch, a, k, d_ann, n_ann, method="sorted")
    edge_cases = [(empty, no_ids, n_ann), (batch, d_ann, 0)]
    want_edge = [E.learn_sparse_with_totals(b, a, k, ids, n, method="sorted") for b, ids, n in edge_cases]
    calls = []
    sorted_path = E._learn_sorted
    monkeypatch.setattr(E, "_learn_sorted", lambda *args: calls.append(1) or sorted_path(*args))
    monkeypatch.setattr(E, "GROUP_MAX_RES", 1000)
    k2, v2, t2 = E.learn_sparse_hybrid(batch, a, k, d_ann, n_ann, want_totals=True)
    assert torch.equal(k1, k2) and torch.equal(v1, v2) and torch.equal(t1, t2)
    k3, v3 = E.learn_sparse_hybrid(batch, a, k, d_ann, n_ann, want_totals=False)
    assert torch.equal(k1, k3) and torch.equal(v1, v3)
    k4, v4, t4 = E.learn_sparse_with_totals(batch, a, k, d_ann, n_ann)
    assert torch.equal(k1, k4) and torch.equal(v1, v4) and torch.equal(t1, t4)
    assert len(calls) == 3
    for (b, ids, n), want in zip(edge_cases, want_edge):
        got = E.learn_sparse_with_totals(b, a, k, ids, n)
        assert all(torch.equal(x, y) for x, y in zip(got, want))


def _syn6():
    from snekmer_b200 import alphabet as A

    syn6 = {"AGILMV": "A", "FWY": "F", "NQSTC": "N", "DE": "D", "KRH": "K", "P": "P"}
    A.register_alphabet("syn6", syn6)
    return {"syn6": [(k, v) for k, v in syn6.items()]}


def _uniref_like(rng, n, mean_len=350.0, sigma=0.6):
    bg = dict(A=.122, L=.105, G=.084, R=.074, V=.071, D=.060, E=.057, P=.053, T=.050, S=.047, I=.047, F=.034, Q=.034,
              K=.025, M=.024, N=.022, Y=.022, H=.021, W=.014, C=.009)
    letters = np.array(list(bg) + ["X"])
    p = np.append(np.array(list(bg.values())) / sum(bg.values()) * 0.999, 0.001)
    lens = np.clip(np.rint(rng.lognormal(np.log(mean_len) - sigma * sigma / 2, sigma, size=n)), 30, 5000).astype(int)
    return ["".join(rng.choice(letters, size=L, p=p)) for L in lens]


def test_c3_shaped_learn_against_the_oracle():
    """VERDICT r1: a C3-SHAPED learn (6-letter alphabet, k = 8, S = 1,679,616, Zipf(1.1) annotations, 30 % unannotated,
    UniRef-like lengths) at a size the numpy oracle still does — 50,000 sequences, 2,000 annotations — compared with the
    oracle's (annotation, k-mer) counts and Totals, for both device methods."""
    extra = _syn6()
    rng = np.random.default_rng(33)
    n, n_ann, k = 50000, 2000, 8
    seqs = _uniref_like(rng, n)
    w = 1.0 / np.arange(1, n_ann + 1) ** 1.1
    ann = rng.choice(n_ann, size=n, p=w / w.sum()).astype(np.int32)
    ann[rng.random(n) < 0.3] = -1
    lut, syms = O.build_lut("syn6", extra)
    S = len(syms) ** k
    res, offs = O.pack(seqs)
    si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
    a = ann[si]
    keep = valid & (a >= 0)
    want_k, want_v = np.unique(a[keep].astype(np.int64) * S + code[keep].astype(np.int64), return_counts=True)
    want_t = np.bincount(code[valid].astype(np.int64), minlength=S)
    batch = E.SequenceBatch.from_strings(seqs)
    d_ann = torch.from_numpy(ann)
    for method in ("hybrid", "sorted"):
        keys, vals, totals = E.learn_sparse_with_totals(batch, "syn6", k, d_ann, n_ann, method=method)
        assert np.array_equal(keys.cpu().numpy(), want_k), method
        assert np.array_equal(vals.cpu().numpy(), want_v), method
        assert np.array_equal(totals.cpu().numpy(), want_t), method


def test_c4_shaped_sparse_apply_against_the_oracle():
    """A C4-SHAPED apply (S = 1,679,616, matrix learned from Zipf families, half of the queries mutated copies of training
    sequences): top-2 and scores of the SpMM path against exact sparse integer products (scipy) + float64 scaling."""
    import scipy.sparse as sp

    extra = _syn6()
    rng = np.random.default_rng(44)
    k, n_ann, n_train, nq = 8, 3000, 12000, 4000
    train = _uniref_like(rng, n_train)
    w = 1.0 / np.arange(1, n_ann + 1) ** 1.1
    t_ann = rng.choice(n_ann, size=n_train, p=w / w.sum()).astype(np.int32)
    queries = _uniref_like(rng, nq // 2)
    aa = np.array(list("ACDEFGHIKLMNPQRSTVWY"))
    for i in rng.choice(n_train, size=nq - nq // 2, replace=False):      # mutated copies: 10 % substitutions
        s = np.array(list(train[int(i)]))
        m = rng.random(len(s)) < 0.1
        s[m] = rng.choice(aa, size=int(m.sum()))
        queries.append("".join(s))
    lut, syms = O.build_lut("syn6", extra)
    S = len(syms) ** k

    def csr_counts(seqs, rows_of=None, n_rows=None):
        res, offs = O.pack(seqs)
        si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
        r = si[valid] if rows_of is None else rows_of[si[valid]]
        m = sp.coo_matrix((np.ones(int(valid.sum()), dtype=np.int64), (r, code[valid].astype(np.int64))),
                          shape=(len(seqs) if n_rows is None else n_rows, S)).tocsr()
        m.sum_duplicates()
        return m
    M = csr_counts(train, t_ann, n_ann)
    Q = csr_counts(queries)
    dots = (Q @ M.T).toarray().astype(np.float64)                         # exact: integer products far below 2^53
    qn = np.sqrt(np.asarray(Q.multiply(Q).sum(axis=1)).ravel().astype(np.float64))
    mn = np.sqrt(np.asarray(M.multiply(M).sum(axis=1)).ravel().astype(np.float64))
    qn[qn == 0] = 1.0
    mn[mn == 0] = 1.0
    Sc = dots / qn[:, None] / mn[None, :]
    i1, i2, s1, s2 = O.top2(Sc)
    tb = E.SequenceBatch.from_strings(train)
    keys, vals = E.learn_sparse(tb, "syn6", k, torch.from_numpy(t_ann), n_ann)
    qb = E.SequenceBatch.from_strings(queries)
    rowptr, cols, cvals = E.count_csr(qb, "syn6", k, None)
    r = E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann)
    assert np.allclose(r.score1.cpu().numpy(), s1, rtol=1e-12, atol=1e-15) and np.allclose(r.score2.cpu().numpy(), s2, rtol=1e-12, atol=1e-15)
    clear = (s1 - s2) > 1e-12 * np.maximum(s1, 1e-30)
    assert np.array_equal(r.top1.cpu().numpy()[clear], i1[clear])
    # the long queries are the point: 512 or more distinct k-mers fill a whole staging block of the SpMM kernel
    assert int((np.diff(rowptr.cpu().numpy()) >= 512).sum()) > 100


@pytest.mark.parametrize("n_runs,count_bits,n", [(1, 29, 5000), (2, 29, 40000), (5, 20, 30000), (8, 29, 100000), (3, 40, 0)])
def test_packed_exchange_format_merges_like_the_unpacked_one(n_runs, count_bits, n):
    """skm_coo_pack + skm_coo_merge_runs_packed (the multi-GPU fan-in's wire format: key << count_bits | count) against
    numpy and against skm_coo_merge_runs on the unpacked lists; overflow of either field is flagged."""
    rng = np.random.default_rng(n_runs * 1000 + count_bits)
    key_bits = min(64 - count_bits, 36)
    runs_k, runs_v = [], []
    for r in range(n_runs):
        m = int(rng.integers(0, 2 * n // n_runs + 1)) if n else 0
        k = np.unique(rng.integers(0, 1 << key_bits, size=m, dtype=np.int64) // 3)       # collisions between runs
        runs_k.append(k)
        runs_v.append(rng.integers(1, 1 << min(count_bits - 4, 30), size=k.size, dtype=np.int64))
    keys = torch.from_numpy(np.concatenate(runs_k)).cuda()
    vals = torch.from_numpy(np.concatenate(runs_v)).cuda()
    sizes = [int(k.size) for k in runs_k]
    packed, bad = E.coo_pack(keys, vals, count_bits)
    assert not bad
    assert np.array_equal(packed.cpu().numpy().view(np.uint64), (keys.cpu().numpy().astype(np.uint64) << np.uint64(count_bits)) | vals.cpu().numpy().astype(np.uint64))
    ok, ov, dn = E.coo_merge_runs_packed(packed.data_ptr(), sizes, count_bits, keys.device)
    m = int(dn.item())
    uk, inv = np.unique(np.concatenate(runs_k), return_inverse=True)
    uv = np.zeros(uk.size, dtype=np.int64)
    np.add.at(uv, inv, np.concatenate(runs_v))
    assert m == uk.size and np.array_equal(ok[:m].cpu().numpy(), uk) and np.array_equal(ov[:m].cpu().numpy(), uv)
    if keys.numel():
        k2, v2 = E.coo_merge_runs(keys, vals, sizes)
        assert torch.equal(k2, ok[:m]) and torch.equal(v2, ov[:m])
        big = vals.clone()
        big[-1] = 1 << count_bits
        assert E.coo_pack(keys, big, count_bits)[1]
        if count_bits > 28:
            bigk = keys.clone()
            bigk[0] = 1 << (64 - count_bits)
            assert E.coo_pack(bigk, vals, count_bits)[1]


@pytest.mark.parametrize("a,k,n", [("miqs", 3, 3000), ("miqs", 3, 12), (2, 4, 400), ("hydro", 10, 2000), (0, 3, 40)])
def test_vectorize_order_only_overlapped_readback(a, k, n):
    """vectorize_order_only (count pass launched over S columns before K is read back) == basis + counts of the two
    separate calls and of the oracle, for saturated spaces (K = S) and unsaturated ones (K < S: compacted)."""
    rng = np.random.default_rng(n + k)
    seqs = _rand_seqs(rng, n, 0, 120)
    batch = E.SequenceBatch.from_strings(seqs)
    basis, counts = E.vectorize_order_only(batch, a, k)
    ref = E.build_basis(batch, a, k, 0, counts=False)
    want_codes, _, (si, code, valid) = _oracle_basis(seqs, a, k)
    assert basis.K == ref.K == len(want_codes)
    assert np.array_equal(basis.codes_host(), want_codes) and torch.equal(basis.col_of_code, ref.col_of_code)
    assert tuple(counts.shape) == (n, basis.K) and counts.is_contiguous()
    assert torch.equal(counts, E.count_dense(batch, a, k, ref))
    assert np.array_equal(counts.cpu().numpy(), O.count_matrix(si, code, valid, n, want_codes))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    out = torch.empty((n, basis.S), dtype=torch.int32, device="cuda")
    b2, c2 = E.vectorize_order_only(batch, a, k, out=out, count_events=ev)
    assert torch.equal(c2, counts) and (c2.data_ptr() == out.data_ptr()) == (basis.K == basis.S)
    plan = E.OrderOnlyPlan(batch, a, k)                  # the front of the step as one CUDA-graph launch, replayed twice
    assert plan.graph is not None
    for _ in range(2):
        out.fill_(-7)
        b3, c3 = E.vectorize_order_only(batch, a, k, out=out, plan=plan)
        assert b3.K == basis.K and torch.equal(b3.codes, basis.codes) and torch.equal(c3, counts)


def test_learn_host_packed_download_equals_device_path(monkeypatch):
    """pipeline.learn_host: host residues + annotation ids -> host COO in the packed 8-byte format == the device lists of
    learn_sparse; a count beyond the packed word's count bits comes back unpacked."""
    from snekmer_b200 import pipeline as P

    rng = np.random.default_rng(21)
    seqs = _rand_seqs(rng, 1500, 0, 200)
    ann = rng.integers(-1, 30, size=len(seqs)).astype(np.int32)
    res, offs = O.pack(seqs)
    batch = E.SequenceBatch.from_strings(seqs)
    k1, v1 = E.learn_sparse(batch, 2, 8, torch.from_numpy(ann), 30)
    h = P.learn_host(torch.from_numpy(res).pin_memory(), offs, ann, 2, 8, 30)
    assert h.packed is not None and h.nnz == k1.numel()
    assert np.array_equal(h.keys(), k1.cpu().numpy()) and np.array_equal(h.vals(), v1.cpu().numpy())
    out = torch.empty(h.nnz + 5, dtype=torch.int64, pin_memory=True)
    h2 = P.learn_host(torch.from_numpy(res), offs, torch.from_numpy(ann), 2, 8, 30, out=out)
    assert np.array_equal(h2.keys(), h.keys()) and np.array_equal(h2.vals(), h.vals())
    monkeypatch.setattr(E, "coo_pack", lambda keys, vals, bits: (None, True))       # a count that does not fit: unpacked download
    h3 = P.learn_host(torch.from_numpy(res), offs, ann, 2, 8, 30)
    assert h3.packed is None and np.array_equal(h3.keys(), k1.cpu().numpy()) and np.array_equal(h3.vals(), v1.cpu().numpy())
