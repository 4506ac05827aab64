"""GPU parity tests: every CUDA kernel (through the C-ABI) against the CPU oracle
and the reference-generated golden vectors.  Bit-exact for codes / bases /
counts / learn matrices; cosine within 1e-12 absolute (float64 both sides; the
stated tolerance of the path is 1e-5 relative)."""
import os

import numpy as np
import pytest
import torch

from oracle import skm_oracle as O
from util import GOLDEN, RULE_CONFIGS, csv_frame, edge_cases, load_rule, read_ann, read_fasta, unpack_vecs

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from snekmer_b200 import engine as E
    from snekmer_b200 import alphabet as A


def _alpha(a):
    return None if a == "None" else (int(a) if str(a).isdigit() else a)


def _rand_seqs(rng, n, lo=0, hi=600, p_x=0.002):
    aa = np.array(list("ACDEFGHIKLMNPQRSTVWYXBZUO*acd"))
    p = np.array([1.0] * 20 + [p_x * 20] * 9)
    p /= p.sum()
    return ["".join(rng.choice(aa, size=int(rng.integers(lo, hi)), p=p)) for _ in range(n)]


def _codes_oracle(seqs, a, k):
    lut, syms = O.build_lut(a)
    res, offs = O.pack(seqs)
    si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
    full = np.full(len(res), np.uint64(0xFFFFFFFFFFFFFFFF), dtype=np.uint64)
    g = offs[si] + pos
    full[g[valid]] = code[valid]
    return full, (si, pos, code, valid), (res, offs, lut, syms)


def test_lut_matches_oracle():
    for a in (0, 1, 2, 3, 4, 5, "ptm", None):
        lut, syms = O.build_lut(a)
        assert A.symbols(a) == syms
        assert np.array_equal(np.frombuffer(A.lut(a), dtype=np.uint8), lut)


@pytest.mark.parametrize("a", [0, 1, 2, 3, 4, 5, "ptm", "None"])
def test_encode_edge_cases(a):
    a = _alpha(a)
    fx = edge_cases()
    seqs = [s for _, s in fx["sequences"]]
    batch = E.SequenceBatch.from_strings(seqs)
    nsym = len(A.symbols(a))
    for k in (1, 2, 3, 5, 8, 14):
        if nsym ** k >= 2 ** 64:
            with pytest.raises(E.SkmError):
                E.encode_windows(batch, a, k)
            continue
        want, _, _ = _codes_oracle(seqs, a, k)
        got = E.encode_windows(batch, a, k).cpu().numpy()
        got = got.view(np.uint32).astype(np.uint64) if got.dtype == np.int32 else got.view(np.uint64)
        if nsym ** k < 2 ** 32:
            want = np.where(want == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), want)
        assert np.array_equal(got, want), (a, k)
        # and the strings the reference API returns
        case = fx["cases"][f"{'None' if a is None else a}:{k}"]
        offs = batch.offsets_host
        inv = np.uint64(0xFFFFFFFF if nsym ** k < 2 ** 32 else 0xFFFFFFFFFFFFFFFF)
        for i in range(len(seqs)):
            c = got[offs[i]:offs[i + 1]]
            assert list(E.decode_kmers(c[c != inv], A.symbols(a), k)) == case["kmers"][i]


@pytest.mark.parametrize("a,k", [(0, 1), (0, 16), (0, 31), (2, 8), (2, 20), (5, 3), (5, 9), (5, 19), (None, 2),
                                 (None, 7), (None, 14), ("ptm", 6), ("ptm", 13), (1, 11), (3, 17), (4, 40), (0, 63)])
def test_encode_random(a, k):
    rng = np.random.default_rng(k * 131 + 7)
    seqs = _rand_seqs(rng, 300, 0, 700)
    seqs[5] = ""
    seqs[17] = "A" * 1500
    batch = E.SequenceBatch.from_strings(seqs)
    want, _, (_, _, _, syms) = _codes_oracle(seqs, a, k)
    got = E.encode_windows(batch, a, k).cpu().numpy()
    if got.dtype == np.int32:
        got = got.view(np.uint32).astype(np.uint64)
        want = np.where(want == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), want)
    else:
        got = got.view(np.uint64)
    assert np.array_equal(got, want)


def test_reduce_bytes():
    rng = np.random.default_rng(3)
    seqs = _rand_seqs(rng, 100, 0, 300)
    batch = E.SequenceBatch.from_strings(seqs)
    for a in (0, 3, 4, 5, None):
        got = bytes(E.reduce_bytes(batch, a).cpu().numpy()).decode("latin-1")
        want = "".join(O.reduce_str(s + "|", a)[:-1] for s in seqs)   # '|' guards rstrip: kernel keeps '*'
        assert got == want


@pytest.mark.parametrize("name", sorted(RULE_CONFIGS))
def test_golden_rule_fixtures(name):
    """vectorize → learn → apply on the reference-generated fixtures."""
    a, k, mf = RULE_CONFIGS[name]
    a = _alpha(a)
    d = load_rule(name)
    ann = read_ann(os.path.join(GOLDEN, "syn.ann"))
    res_files = {}
    for nb in ("synA", "synB"):
        ids, seqs = read_fasta(os.path.join(GOLDEN, f"{nb}.fasta"))
        batch = E.SequenceBatch.from_strings(seqs)
        basis = E.build_basis(batch, a, k, mf)
        assert list(basis.kmers()) == list(d[f"{nb}_kmerlist"])
        C = E.count_dense(batch, a, k, basis)
        assert np.array_equal((C.cpu().numpy() > 0).astype(np.uint8), unpack_vecs(d, f"{nb}_"))
        C16 = E.count_dense(batch, a, k, basis, dtype=torch.uint16)
        assert np.array_equal(C16.cpu().numpy().astype(np.int32), C.cpu().numpy())
        # learn (learn.smk:306-357)
        anns_o, M_o, nseq_o, tot_o, _ = O.learn_matrix(ids, C.cpu().numpy(), ann)
        ann_index = {x: i for i, x in enumerate(anns_o)}
        ann_id = np.array([ann_index.get(ann.get(O.accession(s), None), -1) for s in ids], dtype=np.int32)
        M, totals = E.learn_dense(batch, a, k, basis, torch.from_numpy(ann_id), len(anns_o))
        ref = csv_frame(d[f"{nb}_counts_csv"]).values.astype(np.int64)
        assert np.array_equal(M[:-1].cpu().numpy(), ref[1:, 2:])
        assert np.array_equal(totals.cpu().numpy(), ref[0, 2:])
        assert np.array_equal(M[:-1].cpu().numpy(), M_o)
        res_files[nb] = (ids, basis, C, anns_o, M[:-1].clone())
    # apply (apply.smk:224-289): synB queries against the matrix learned on synA
    idsB, basisB, CB, _, _ = res_files["synB"]
    _, basisA, _, annsA, MA = res_files["synA"]
    _, seqsB = read_fasta(os.path.join(GOLDEN, "synB.fasta"))
    batchB = E.SequenceBatch.from_strings(seqsB)
    # query counts live on the query file's OWN basis (min_filter applies to it), re-indexed onto the
    # learned columns: a k-mer contributes to the dot only if it is in both bases (apply.smk:268-276)
    both = E.intersect_basis(basisA, basisB)
    QA = E.count_dense(batchB, a, k, both)
    qn2 = E.row_norm2(CB)                                    # norm over the query file's own basis
    r = E.apply_dense(QA, MA, qnorm2=qn2, full=True)
    ref = d["apply_scores"]
    got = r.scores.cpu().numpy()
    assert got.shape == ref.shape
    assert np.max(np.abs(got - ref)) < 1e-12
    i1, i2, s1, s2 = O.top2(got)
    assert np.array_equal(r.top1.cpu().numpy(), i1) and np.array_equal(r.top2.cpu().numpy(), i2)
    assert np.array_equal(r.score1.cpu().numpy(), s1) and np.array_equal(r.score2.cpu().numpy(), s2)
    # predictions identical to the reference wherever its own top-2 gap is not a float tie
    ri1, ri2, rs1, rs2 = O.top2(ref)
    clear = (rs1 - rs2) > 1e-9
    assert np.array_equal(r.top1.cpu().numpy()[clear], ri1[clear])
    assert np.allclose(r.score1.cpu().numpy(), rs1, rtol=1e-5, atol=0)


# Between them, the int32 and uint16 counts of these cases reach every dense count kernel: the tile kernel with and
# without a column map, and both warp kernels (words: k <= 5, bytes: k > 5) with each column-map mode (identity, map in
# shared memory for S <= 16384, map in global memory beyond; the last two filtered down to a few thousand columns).
@pytest.mark.parametrize("a,k,mf", [(5, 3, 0), (2, 8, 0), (0, 12, 2), (None, 3, 0), (1, 4, 5), ("ptm", 2, 0), (4, 9, 0),
                                    (0, 11, 0), (None, 4, 6), (2, 10, 14)])
def test_basis_and_dense_counts_random(a, k, mf):
    rng = np.random.default_rng(hash((str(a), k)) % 2 ** 32)
    seqs = _rand_seqs(rng, 700, 0, 900)
    seqs[0] = ""
    seqs[3] = "ACD"
    batch = E.SequenceBatch.from_strings(seqs)
    _, (si, pos, code, valid), (res, offs, lut, syms) = _codes_oracle(seqs, a, k)
    want_basis, want_tot = O.basis_codes(si, pos, code, valid, mf)
    basis = E.build_basis(batch, a, k, mf)
    assert np.array_equal(basis.codes_host(), want_basis)
    assert np.array_equal(basis.counts.cpu().numpy(), want_tot)
    want = O.count_matrix(si, code, valid, len(seqs), want_basis)
    for dtype in (torch.int32, torch.uint16):
        got = E.count_dense(batch, a, k, basis, dtype=dtype).cpu().numpy()
        assert np.array_equal(got, want)
    if len(syms) ** k <= 20000:
        full = O.count_matrix(si, code, valid, len(seqs), np.arange(len(syms) ** k, dtype=np.uint64))
        for dtype in (torch.int32, torch.uint16):
            ident = E.count_dense(batch, a, k, None, dtype=dtype).cpu().numpy()
            assert np.array_equal(ident, full)


def test_dense_counts_long_sequences_use_32bit_counters():
    # > 65535 residues: the 16-bit shared-memory counters would overflow
    seqs = ["A" * 70000, "ACDEFGHIKL" * 7000, "MKV"]
    batch = E.SequenceBatch.from_strings(seqs)
    got = E.count_dense(batch, 0, 2, None).cpu().numpy()
    _, (si, pos, code, valid), _ = _codes_oracle(seqs, 0, 2)
    want = O.count_matrix(si, code, valid, 3, np.arange(4, dtype=np.uint64))
    assert np.array_equal(got, want) and got.max() == 69999
    with pytest.raises(E.SkmError):
        E.count_dense(batch, 0, 2, None, dtype=torch.uint16)


@pytest.mark.parametrize("a,k", [(5, 3), (2, 8), (None, 5), (1, 6)])
def test_count_csr(a, k):
    rng = np.random.default_rng(k)
    seqs = _rand_seqs(rng, 500, 0, 800)
    seqs[7] = ""
    batch = E.SequenceBatch.from_strings(seqs)
    _, (si, pos, code, valid), (res, offs, lut, syms) = _codes_oracle(seqs, a, k)
    rp, cc, cv = O.count_csr(si, code, valid, len(seqs))
    rowptr, cols, vals = E.count_csr(batch, a, k, None)
    assert np.array_equal(rowptr.cpu().numpy(), rp)
    assert np.array_equal(cols.cpu().numpy().view(np.uint32).astype(np.uint64), cc)
    assert np.array_equal(vals.cpu().numpy(), cv)
    # over a filtered basis: columns instead of codes
    basis = E.build_basis(batch, a, k, 1)
    rowptr, cols, vals = E.count_csr(batch, a, k, basis)
    dense = E.count_dense(batch, a, k, basis).cpu().numpy()
    rp2 = rowptr.cpu().numpy()
    for r in range(len(seqs)):
        nz = np.flatnonzero(dense[r])
        assert np.array_equal(cols.cpu().numpy()[rp2[r]:rp2[r + 1]], nz)
        assert np.array_equal(vals.cpu().numpy()[rp2[r]:rp2[r + 1]], dense[r, nz])


def test_learn_and_apply_random():
    rng = np.random.default_rng(99)
    seqs = _rand_seqs(rng, 3000, 0, 500)
    a, k = 2, 5
    batch = E.SequenceBatch.from_strings(seqs)
    basis = E.build_basis(batch, a, k, 0)
    n_ann = 37
    ann_id = rng.integers(-1, n_ann, size=len(seqs)).astype(np.int32)
    C = E.count_dense(batch, a, k, basis).cpu().numpy().astype(np.int64)
    M, totals = E.learn_dense(batch, a, k, basis, torch.from_numpy(ann_id), n_ann)
    want = np.zeros((n_ann + 1, basis.K), dtype=np.int64)
    np.add.at(want, np.where(ann_id < 0, n_ann, ann_id), C)
    assert np.array_equal(M.cpu().numpy(), want)
    assert np.array_equal(totals.cpu().numpy(), C.sum(axis=0))
    Q = torch.from_numpy(C[:777].astype(np.int32)).cuda()
    r = E.apply_dense(Q, M[:-1].contiguous(), full=True, chunk=300)
    S = O.cosine_scores(C[:777], want[:-1])
    assert np.max(np.abs(r.scores.cpu().numpy() - S)) < 1e-12
    i1, i2, s1, s2 = O.top2(r.scores.cpu().numpy())
    assert np.array_equal(r.top1.cpu().numpy(), i1) and np.array_equal(r.top2.cpu().numpy(), i2)


def test_apply_ties_and_zero_rows():
    Q = torch.tensor([[0, 0, 0], [1, 1, 0], [2, 0, 0]], dtype=torch.int32).cuda()
    M = torch.tensor([[1, 1, 0], [1, 1, 0], [0, 0, 0], [5, 0, 0]], dtype=torch.int64).cuda()
    r = E.apply_dense(Q, M, full=True)
    assert r.top1.tolist() == [0, 0, 3] and r.top2.tolist() == [1, 1, 0]
    assert r.score1.tolist()[0] == 0.0 and abs(r.score1.tolist()[1] - 1.0) < 1e-15


def test_errors_are_loud():
    batch = E.SequenceBatch.from_strings(["ACD"])
    with pytest.raises(E.SkmError):
        E.encode_windows(batch, "ptm", 14)      # 30^14 > 2^64
    with pytest.raises(E.SkmError):
        E.build_basis(batch, None, 8)           # 20^8 > table limit
    with pytest.raises(ValueError):
        E.encode_windows(batch, "nope", 3)


# ---------------------------------------------------------------------------------------------
# sparse paths
# ---------------------------------------------------------------------------------------------
def _dense_from_coo(keys, vals, S, n_ann):
    k = keys.cpu().numpy().view(np.uint64)
    M = np.zeros((n_ann, S), dtype=np.int64)
    M[(k // np.uint64(S)).astype(np.int64), (k % np.uint64(S)).astype(np.int64)] = vals.cpu().numpy()
    return M


@pytest.mark.parametrize("a,k,chunk", [(2, 5, 1 << 28), (5, 3, 20000), (0, 10, 7000), (None, 3, 1 << 28)])
def test_learn_sparse_matches_dense(a, k, chunk):
    rng = np.random.default_rng(k * 7 + 1)
    seqs = _rand_seqs(rng, 900, 0, 300)
    seqs[4] = ""
    batch = E.SequenceBatch.from_strings(seqs)
    n_ann = 29
    ann = rng.integers(-1, n_ann, size=len(seqs)).astype(np.int32)
    keys, vals = E.learn_sparse(batch, a, k, torch.from_numpy(ann), n_ann, max_chunk_res=chunk)
    kk = keys.cpu().numpy().view(np.uint64)
    assert np.all(kk[1:] > kk[:-1])                      # sorted, distinct
    _, (si, pos, code, valid), (res, offs, lut, syms) = _codes_oracle(seqs, a, k)
    S = len(syms) ** k
    full = O.count_matrix(si, code, valid, len(seqs), np.arange(S, dtype=np.uint64)).astype(np.int64)
    want = np.zeros((n_ann, S), dtype=np.int64)
    sel = ann >= 0
    np.add.at(want, ann[sel], full[sel])
    assert np.array_equal(_dense_from_coo(keys, vals, S, n_ann), want)
    assert int(vals.min().item()) > 0
    # merging a list with itself doubles every count
    k2, v2 = E.coo_merge(torch.cat([keys, keys]), torch.cat([vals, vals]))
    assert torch.equal(k2, keys) and torch.equal(v2, 2 * vals)
    # the grouped 32-bit-key build (default) and the global 64-bit sort give the same list
    kg, vg = E.learn_sparse(batch, a, k, torch.from_numpy(ann), n_ann, max_chunk_res=chunk, method="global")
    assert torch.equal(kg, keys) and torch.equal(vg, vals)


def test_learn_sparse_grouped_many_slices():
    """C3 shape in small: 6-letter alphabet, k = 8 (S = 1,679,616 -> 2,556 annotations per 32-bit slice), 6,000
    annotations -> 3 slices, some annotations empty, 30 % unannotated; equal to the global sort."""
    from snekmer_b200 import alphabet as A

    A.register_alphabet("syn6", {"AGILMV": "A", "FWY": "F", "NQSTC": "N", "DE": "D", "KRH": "K", "P": "P"})
    rng = np.random.default_rng(8)
    seqs = _rand_seqs(rng, 5000, 0, 200)
    batch = E.SequenceBatch.from_strings(seqs)
    n_ann = 6000
    w = 1.0 / np.arange(1, n_ann + 1) ** 1.1
    ann = rng.choice(n_ann, size=len(seqs), p=w / w.sum()).astype(np.int32)
    ann[rng.random(len(seqs)) < 0.3] = -1
    k1, v1 = E.learn_sparse(batch, "syn6", 8, torch.from_numpy(ann), n_ann)
    k2, v2 = E.learn_sparse(batch, "syn6", 8, torch.from_numpy(ann), n_ann, method="global")
    assert k1.numel() > 0 and torch.equal(k1, k2) and torch.equal(v1, v2)
    # gather_sequences on its own
    sel = torch.from_numpy(rng.permutation(len(seqs))[:777].astype(np.int64))
    g_res, g_off = E.gather_sequences(batch, sel)
    raw = bytes(g_res.cpu().numpy())
    off = g_off.cpu().numpy()
    assert [raw[off[i]:off[i + 1]].decode("latin-1") for i in range(len(sel))] == [seqs[int(j)] for j in sel]


@pytest.mark.parametrize("a,k,tile", [(2, 6, 8192), (5, 3, 7), (1, 4, 16)])
def test_apply_sparse_matches_dense_oracle(a, k, tile):
    rng = np.random.default_rng(k + 100)
    train = _rand_seqs(rng, 1200, 20, 300)
    n_ann = 37
    ann = rng.integers(-1, n_ann, size=len(train)).astype(np.int32)
    tb = E.SequenceBatch.from_strings(train)
    keys, vals = E.learn_sparse(tb, a, k, torch.from_numpy(ann), n_ann)
    queries = _rand_seqs(rng, 400, 0, 250) + train[:50] + ["", "AC"]
    qb = E.SequenceBatch.from_strings(queries)
    rowptr, cols, cvals = E.count_csr(qb, a, k, None)
    _, (si, pos, code, valid), (res, offs, lut, syms) = _codes_oracle(queries, a, k)
    S = len(syms) ** k
    r = E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann, tile=tile)
    Q = O.count_matrix(si, code, valid, len(queries), np.arange(S, dtype=np.uint64))
    M = _dense_from_coo(keys, vals, S, n_ann)
    Sc = O.cosine_scores(Q, M)
    i1, i2, s1, s2 = O.top2(Sc)
    g1, g2 = r.top1.cpu().numpy(), r.top2.cpu().numpy()
    gs1, gs2 = r.score1.cpu().numpy(), r.score2.cpu().numpy()
    # exact integer dots, float64 scaling: the scores agree with the float64 oracle to rounding
    assert np.allclose(gs1, s1, rtol=1e-12, atol=1e-15) and np.allclose(gs2, s2, rtol=1e-12, atol=1e-15)
    rows = np.arange(len(queries))
    # identical predictions wherever the oracle's own ranking is not a rounding-level tie
    clear1 = (s1 - s2) > 1e-12 * np.maximum(s1, 1e-30)
    assert np.array_equal(g1[clear1], i1[clear1])
    assert np.allclose(Sc[rows, g1], s1, rtol=1e-12, atol=1e-15) and np.allclose(Sc[rows, g2], s2, rtol=1e-12, atol=1e-15)
    zero = s1 == 0
    assert np.array_equal(g1[zero], np.zeros(zero.sum(), dtype=g1.dtype))     # all-zero rows: prediction = column 0


# ---------------------------------------------------------------------------------------------
# tensor-core scoring (tcgen05 int8 GEMM): bit-for-bit the same top-2 as the exact CUDA-core path
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nq,A,K,mmax", [(300, 40, 1000, 200), (1000, 513, 257, 70000), (129, 128, 128, 2 ** 24 + 5),
                                         (64, 3, 3000, 2 ** 31 - 1), (257, 700, 6561, 5000)])
def test_apply_tensor_cores_match_exact_path(nq, A, K, mmax):
    rng = np.random.default_rng(nq + A + K)
    Q = rng.integers(0, 6, size=(nq, K)).astype(np.int32) * (rng.random((nq, K)) < 0.3)
    Q[0] = 0
    Q[1, :5] = 255
    M = (rng.integers(0, mmax + 1, size=(A, K), dtype=np.int64) * (rng.random((A, K)) < 0.5)).astype(np.int64)
    M[A // 2] = M[0]                       # an exact tie between two annotations
    if A > 2:
        M[A - 1] = 0                       # a zero-norm annotation
    M[0, 0] = mmax
    dQ, dM = torch.from_numpy(Q.astype(np.int32)).cuda(), torch.from_numpy(M).cuda()
    exact = E.apply_dense(dQ, dM, full=True, tensor_cores=False)
    prep = E.prepare_annotations(dM)
    assert prep is not None and prep.n_planes == max(1, (int(mmax).bit_length() + 7) // 8)
    tc = E.apply_tc(dQ, prep, full=True)
    assert tc is not None
    torch.cuda.synchronize()
    # integer dots are exact on both paths; the scaling differs by <= 2 ulp
    assert torch.allclose(tc.scores, exact.scores, rtol=1e-14, atol=0)
    S = O.cosine_scores(Q, M)
    assert np.max(np.abs(tc.scores.cpu().numpy() - S)) < 1e-12
    i1, i2, s1, s2 = O.top2(tc.scores.cpu().numpy())
    assert np.array_equal(tc.top1.cpu().numpy(), i1) and np.array_equal(tc.top2.cpu().numpy(), i2)
    assert np.array_equal(tc.score1.cpu().numpy(), s1) and np.array_equal(tc.score2.cpu().numpy(), s2)
    assert tc.top1[0].item() == 0 and tc.score1[0].item() == 0.0
    # via the dispatcher, and without the full matrix
    r = E.apply_dense(dQ, dM, tensor_cores=True, prepared=prep)
    assert torch.equal(r.top1, tc.top1) and torch.equal(r.score2, tc.score2)


def test_apply_tensor_cores_envelope_fallbacks():
    Q = torch.zeros((10, 64), dtype=torch.int32).cuda()
    Q[3, 7] = 300                                        # does not fit 8 bits -> exact path
    M = torch.ones((5, 64), dtype=torch.int64).cuda()
    prep = E.prepare_annotations(M)
    rt = E.apply_tc(Q, prep)                             # row 3 alone is re-scored by the exact path
    assert rt is not None and rt.top1[3].item() == 0 and abs(rt.score1[3].item() - 300 / (300 * 8.0)) < 1e-15
    prep.M = None                                        # a prepared matrix without M cannot re-score: None
    assert E.apply_tc(Q, prep) is None
    r = E.apply_dense(Q, M, tensor_cores=True)
    assert r.top1[3].item() == 0 and abs(r.score1[3].item() - 300 / (300 * 8.0)) < 1e-15
    M[2, 2] = 2 ** 40                                    # needs 6 digit planes
    assert E.prepare_annotations(M) is None


@pytest.mark.parametrize("a,k", [(5, 3), (2, 9), (None, 5)])
def test_kmer_totals_counts_only(a, k):
    """skm_basis_accumulate without the first-position table == the count column of the full tables."""
    rng = np.random.default_rng(k)
    seqs = _rand_seqs(rng, 700, 0, 400)
    batch = E.SequenceBatch.from_strings(seqs)
    tab = E.alphabet_tables(a)
    count, first = E.basis_tables(tab.nsym ** k, batch.device)
    E.basis_accumulate(batch, a, k, count, first, 0)
    assert torch.equal(E.kmer_totals(batch, a, k), count)
    _, (si, pos, code, valid), _ = _codes_oracle(seqs, a, k)
    assert np.array_equal(count.cpu().numpy(), np.bincount(code[valid].astype(np.int64), minlength=tab.nsym ** k))


@pytest.mark.parametrize("nruns", [1, 2, 3, 4, 7, 8])
def test_coo_merge_runs_equals_sort_merge(nruns):
    """Merge tree over sorted runs (the multi-GPU fan-in) == sort + reduce-by-key, including empty runs."""
    rng = np.random.default_rng(nruns)
    runs_k, runs_v, sizes = [], [], []
    for r in range(nruns):
        n = 0 if (r == 2 and nruns > 3) else int(rng.integers(1, 5000))
        k = np.unique(rng.integers(0, 20000, size=n)).astype(np.int64)           # sorted, distinct inside a run
        runs_k.append(k)
        runs_v.append(rng.integers(1, 100, size=len(k)).astype(np.int64))
        sizes.append(len(k))
    keys = torch.from_numpy(np.concatenate(runs_k)).cuda()
    vals = torch.from_numpy(np.concatenate(runs_v)).cuda()
    k1, v1 = E.coo_merge(keys, vals, key_bound=20000)
    k2, v2 = E.coo_merge_runs(keys, vals, sizes)
    assert torch.equal(k1, k2) and torch.equal(v1, v2)
    want = np.zeros(20000, np.int64)
    np.add.at(want, keys.cpu().numpy(), vals.cpu().numpy())
    assert np.array_equal(k2.cpu().numpy(), np.flatnonzero(want)) and np.array_equal(v2.cpu().numpy(), want[want > 0])


@pytest.mark.parametrize("a,k", [(5, 3), (2, 8), (None, 4)])
def test_learn_sparse_with_totals(a, k):
    """Totals from the matrix's column sums + the unannotated sequences == the occurrence table over all sequences."""
    rng = np.random.default_rng(k + 31)
    seqs = _rand_seqs(rng, 1500, 0, 300)
    batch = E.SequenceBatch.from_strings(seqs)
    n_ann = 17
    ann = rng.integers(-1, n_ann + 2, size=len(seqs)).astype(np.int32)       # -1 and ids >= n_ann are both "unannotated"
    keys, vals, totals = E.learn_sparse_with_totals(batch, a, k, torch.from_numpy(ann), n_ann)
    assert torch.equal(totals, E.kmer_totals(batch, a, k))
    k2, v2 = E.learn_sparse(batch, a, k, torch.from_numpy(ann), n_ann, method="global")
    assert torch.equal(keys, k2) and torch.equal(vals, v2)
    # all sequences annotated / none annotated
    _, _, t_all = E.learn_sparse_with_totals(batch, a, k, torch.zeros(len(seqs), dtype=torch.int32), n_ann)
    _, _, t_none = E.learn_sparse_with_totals(batch, a, k, torch.full((len(seqs),), -1, dtype=torch.int32), n_ann)
    assert torch.equal(t_all, totals) and torch.equal(t_none, totals)


@pytest.mark.parametrize("a,k", [(2, 6), (5, 3), (1, 4)])
def test_apply_sparse_packed_csc_identical(a, k):
    """The 4-byte packed CSC (value << 16 | annotation, pipelined loads) gives bit-identical results to the 8-byte one,
    and csc_build refuses to pack entries that do not fit 16 bits."""
    rng = np.random.default_rng(k + 300)
    train = _rand_seqs(rng, 1500, 20, 300)
    n_ann = 41
    ann = rng.integers(0, n_ann, size=len(train)).astype(np.int32)
    tb = E.SequenceBatch.from_strings(train)
    keys, vals = E.learn_sparse(tb, a, k, torch.from_numpy(ann), n_ann)
    S = E.alphabet_tables(a).nsym ** k
    queries = _rand_seqs(rng, 500, 0, 900) + ["", "ACD", "A" * 2000]
    qb = E.SequenceBatch.from_strings(queries)
    rowptr, cols, cvals = E.count_csr(qb, a, k, None)
    csc = E.csc_build(keys, vals, S, n_ann, 0)
    assert csc.packed is not None and csc.packed.numel() == csc.rows.numel()
    r0 = E.apply_sparse(rowptr, cols, cvals, csc, use_packed=False)
    r1 = E.apply_sparse(rowptr, cols, cvals, csc, use_packed=True)
    assert torch.equal(r0.top1, r1.top1) and torch.equal(r0.top2, r1.top2) and torch.equal(r0.score1, r1.score1)
    assert np.array_equal(r0.score2.cpu().numpy(), r1.score2.cpu().numpy(), equal_nan=True)
    big = E.csc_build(keys, vals * 70000, S, n_ann, 0)           # entries beyond 16 bits: stays unpacked
    assert big.packed is None
    r2 = E.apply_sparse(rowptr, cols, cvals, big)
    assert torch.equal(r2.top1, r0.top1)
