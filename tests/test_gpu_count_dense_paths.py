"""Dense count paths of count_dense_warp_kernel against the CPU oracle, bit-exact: the lane-striped column map (small
code spaces, one CTA of up to 32 warps per SM) and the uint16 map just above its threshold, the residue translation in
registers (every built-in alphabet but ptm) and through the shared LUT (ptm), int32 and uint16 counts, the compacted
output of an unsaturated order-only vectorize, and the sequence shapes a warp's walk has to get right."""
import numpy as np
import pytest
import torch

from oracle import skm_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from snekmer_b200 import alphabet as A
    from snekmer_b200 import engine as E

# 11 and 12 output symbols: S = 11^3 = 1,331 still takes the striped map (25 warps of 5.8 KB next to 85 KB of map),
# S = 12^3 = 1,728 does not (16 warps would fit) and keeps the uint16 map
SYN = {
    "syn11": {"A": "A", "C": "C", "DE": "D", "FWY": "F", "G": "G", "H": "H", "ILV": "I", "KR": "K", "MQ": "M", "P": "P", "NST": "S"},
    "syn12": {"A": "A", "C": "C", "D": "D", "E": "E", "FWY": "F", "G": "G", "H": "H", "ILV": "I", "KR": "K", "MQ": "M", "P": "P",
              "NST": "S"},
}


def _lut(a):
    if a in SYN:
        A.register_alphabet(a, SYN[a])
        return O.build_lut(a, {a: list(SYN[a].items())})
    return O.build_lut(a)


def _seqs(rng, n, lo, hi):
    aa = np.array(list("ACDEFGHIKLMNPQRSTVWYXBZ*ac@^_-"))
    p = np.array([1.0] * 20 + [0.05] * 10)
    seqs = ["".join(rng.choice(aa, size=int(rng.integers(lo, hi)), p=p / p.sum())) for _ in range(n)]
    # empty, shorter than k, a run of X, longer than one 384-residue segment, several segments with X at their edges
    seqs[:6] = ["", "AC", "X" * 50, "ACDEFGHIKLMNPQRSTVWY" * 30, "MKV" + "X" * 400 + "MKVLA", ("W" * 383 + "X") * 3 + "ACD"]
    return seqs


def _oracle(seqs, a, k, basis_codes):
    lut, syms = _lut(a)
    res, offs = O.pack(seqs)
    si, pos, code, valid = O.window_codes(res, offs, lut, len(syms), k)
    return O.count_matrix(si, code, valid, len(seqs), basis_codes), (si, pos, code, valid)


@pytest.mark.parametrize("a,k,n", [("miqs", 3, 900), ("syn11", 3, 900), ("syn12", 3, 900), ("ptm", 2, 900), ("miqs", 3, 5),
                                   ("hydro", 5, 300)])
def test_dense_counts_match_oracle(a, k, n):
    rng = np.random.default_rng(hash((a, k, n)) % 2 ** 32)
    seqs = _seqs(rng, max(n, 6), 0, 1200)[:max(n, 6)]
    _lut(a)
    batch = E.SequenceBatch.from_strings(seqs)
    basis = E.build_basis(batch, a, k, 0)
    want, _ = _oracle(seqs, a, k, basis.codes_host())
    for dtype in (torch.int32, torch.uint16):
        got = E.count_dense(batch, a, k, basis, dtype=dtype).cpu().numpy()
        assert np.array_equal(got, want), dtype
    full, _ = _oracle(seqs, a, k, np.arange(basis.S, dtype=np.uint64))
    assert np.array_equal(E.count_dense(batch, a, k, None).cpu().numpy(), full)


@pytest.mark.parametrize("dtype", ["int32", "uint16"])
def test_order_only_unsaturated_compacts(dtype):
    # a handful of sequences leave most of the 1,000 miqs 3-mers unseen: K < S, the count pass runs with S columns
    # through the striped map and the result is compacted to K
    rng = np.random.default_rng(11)
    seqs = _seqs(rng, 40, 0, 60)
    batch = E.SequenceBatch.from_strings(seqs)
    basis, counts = E.vectorize_order_only(batch, "miqs", 3, dtype=getattr(torch, dtype))
    assert basis.K < basis.S
    codes = basis.codes_host()
    want, (si, pos, code, valid) = _oracle(seqs, "miqs", 3, codes)
    ob, _ = O.basis_codes(si, pos, code, valid, 0)
    assert np.array_equal(np.sort(codes), np.sort(ob))
    assert tuple(counts.shape) == (len(seqs), basis.K)
    assert np.array_equal(counts.cpu().numpy().astype(np.int64), want)
