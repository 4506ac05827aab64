"""engine: batch entry points of the B200 hot path (host side of the C-ABI).

PyTorch is used for device memory, streams and (elsewhere) torch.distributed
only; every computation below is a call into libskm_b200.so with raw device
pointers.  All functions raise if CUDA or the library is unavailable — there is
no CPU fallback.

Data layout in HBM
  residues  uint8 [R]    all sequences back to back (ASCII), 16-byte aligned
  offsets   int64 [N+1]  sequence s is residues[offsets[s]:offsets[s+1]]
  codes     uint32/uint64 base-|A| k-mer codes (symbols in sorted order)
  basis     uint64 [K] codes in first-occurrence order (kmerize.smk:89-104)
  col_of_code int32 [|A|^k]  code → basis column, -1 if filtered out
  counts    int32/uint16 [N, K] row-major, or CSR (rowptr int64, cols uint32, vals int32)
  M         int64 [A+1, K] annotation rows + one "rest" row; totals int64 [K]
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Callable, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _native
from . import alphabet as _alphabet
from ._native import SkmError, check, lib

INT64_MAX = (1 << 63) - 1

AlphabetT = Union[str, int, None]


def _require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise SkmError(-101, "no CUDA device: snekmer_b200 has no CPU path (the oracle lives in oracle/ and is test-only)")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise SkmError(-101, f"device {dev} is not a CUDA device")
    return dev


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


@dataclass
class AlphabetTables:
    name: str
    symbols: str
    nsym: int
    lut_host: bytes
    lut: torch.Tensor          # uint8 [256] on device
    charmap: torch.Tensor      # uint8 [256] on device


_tables_cache = {}


def alphabet_tables(alphabet, device=None) -> AlphabetTables:
    """Device tables of an alphabet given by name / index / None — or an AlphabetTables
    object, which is passed through (lets callers use ad-hoc symbol sets)."""
    if isinstance(alphabet, AlphabetTables):
        return alphabet
    dev = _require_cuda(device)
    name = _alphabet.get_alphabet_name(alphabet)
    key = (name, dev.index, tuple(sorted(_alphabet.residue_map(name).items())))
    hit = _tables_cache.get(key)
    if hit is not None:
        return hit
    syms = _alphabet.symbols(name)
    lut_host = _alphabet.lut(name)
    t = AlphabetTables(
        name=name, symbols=syms, nsym=len(syms), lut_host=lut_host,
        lut=torch.frombuffer(bytearray(lut_host), dtype=torch.uint8).to(dev),
        charmap=torch.frombuffer(bytearray(_alphabet.charmap(name)), dtype=torch.uint8).to(dev),
    )
    _tables_cache[key] = t
    return t


def alphabet_tables_from_symbols(symbols: str, device=None) -> AlphabetTables:
    """Identity alphabet over already REDUCED text: every character of `symbols` is its own
    symbol, everything else is invalid.  This is what the learn / apply rules need: they
    count windows of the reduced strings stored in the .npz against a k-mer list
    (learn.smk:359-383, apply.smk:188-206), so a window can only match when all its
    characters occur in that list."""
    dev = _require_cuda(device)
    syms = "".join(sorted(set(symbols)))
    key = ("=" + syms, dev.index)
    hit = _tables_cache.get(key)
    if hit is not None:
        return hit
    lut_host = _native.lut_build(syms, syms, syms)
    t = AlphabetTables(name="=" + syms, symbols=syms, nsym=len(syms), lut_host=lut_host,
                       lut=torch.frombuffer(bytearray(lut_host), dtype=torch.uint8).to(dev),
                       charmap=torch.arange(256, dtype=torch.uint8, device=dev))
    _tables_cache[key] = t
    return t


def code_space(nsym: int, k: int) -> int:
    return nsym ** k


class SequenceBatch:
    """Packed sequences resident in HBM."""

    def __init__(self, residues: torch.Tensor, offsets: torch.Tensor, offsets_host: np.ndarray):
        assert residues.dtype == torch.uint8 and offsets.dtype == torch.int64
        self.residues = residues
        self.offsets = offsets
        self.offsets_host = offsets_host
        self.n = len(offsets_host) - 1
        self.nres = int(offsets_host[-1]) if self.n >= 0 and len(offsets_host) else 0
        lens = np.diff(offsets_host) if self.n > 0 else np.zeros(0, np.int64)
        self.max_len = int(lens.max()) if lens.size else 0

    @property
    def device(self):
        return self.residues.device

    @staticmethod
    def pack_host(seqs: Sequence[str]) -> Tuple[np.ndarray, np.ndarray]:
        offs = np.zeros(len(seqs) + 1, dtype=np.int64)
        if len(seqs):
            np.cumsum([len(s) for s in seqs], out=offs[1:])
        buf = np.frombuffer("".join(seqs).encode("latin-1", "replace"), dtype=np.uint8)
        return buf, offs

    @classmethod
    def from_packed(cls, residues: np.ndarray, offsets: np.ndarray, device=None, pinned: bool = False) -> "SequenceBatch":
        dev = _require_cuda(device)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        residues = np.ascontiguousarray(residues, dtype=np.uint8)
        nres = int(offsets[-1]) if len(offsets) else 0
        # +16 bytes of slack keeps the buffer 16-byte granular; kernels never read past nres
        d_res = torch.empty(max(nres, 1) + 16, dtype=torch.uint8, device=dev)
        if nres:
            src = torch.from_numpy(residues[:nres] if residues.flags.writeable else residues[:nres].copy())
            d_res[:nres].copy_(src, non_blocking=pinned)
        d_off = torch.from_numpy(offsets).to(dev)
        return cls(d_res, d_off, offsets)

    @classmethod
    def from_strings(cls, seqs: Sequence[str], device=None) -> "SequenceBatch":
        buf, offs = cls.pack_host([str(s) for s in seqs])
        return cls.from_packed(buf, offs, device)


# ---------------------------------------------------------------------------
# (a) encode
# ---------------------------------------------------------------------------
def encode_windows(batch: SequenceBatch, alphabet: AlphabetT, k: int) -> torch.Tensor:
    """Code of the window starting at every residue (KmerVec.reduce_vectorize,
    vectorize.py:292-328, for the whole batch).  Returns uint32-as-int32 or
    uint64-as-int64 tensor [nres]; invalid windows are all-ones (-1)."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    bits = 32 if S < 2 ** 32 else 64
    out = torch.empty(max(batch.nres, 1), dtype=torch.int32 if bits == 32 else torch.int64, device=batch.device)
    check(lib().skm_encode_windows(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), batch.n, _ptr(tab.lut),
                                   tab.nsym, int(k), bits, _ptr(out), _stream()))
    return out[:batch.nres]


def reduce_bytes(batch: SequenceBatch, alphabet: AlphabetT) -> torch.Tensor:
    """reduce() (vectorize.py:173-195) on the packed buffer: translated bytes [nres]."""
    tab = alphabet_tables(alphabet, batch.device)
    out = torch.empty_like(batch.residues)
    check(lib().skm_reduce_bytes(_ptr(batch.residues), batch.nres, _ptr(tab.charmap), _ptr(out), _stream()))
    return out[:batch.nres]


# ---------------------------------------------------------------------------
# (b') basis
# ---------------------------------------------------------------------------
@dataclass
class Basis:
    """k-mer basis in first-occurrence order + the code→column map."""
    alphabet: str
    k: int
    symbols: str
    codes: torch.Tensor                 # int64 (uint64 bit pattern) [K]
    counts: Optional[torch.Tensor]      # int64 [K] total occurrences, None for a supplied basis
    col_of_code: torch.Tensor           # int32 [S]
    K: int
    S: int

    def codes_host(self) -> np.ndarray:
        return self.codes.cpu().numpy().view(np.uint64)

    def kmers(self) -> np.ndarray:
        return decode_kmers(self.codes_host(), self.symbols, self.k)


def decode_kmers(codes: np.ndarray, symbols: str, k: int) -> np.ndarray:
    """uint64 codes → '<Uk' strings (host-side formatting of the basis)."""
    codes = np.asarray(codes, dtype=np.uint64)
    if codes.size == 0:
        return np.array([], dtype=f"<U{max(k, 1)}")
    n = np.uint64(len(symbols))
    sym = np.frombuffer(symbols.encode("latin-1"), dtype=np.uint8)
    chars = np.empty((codes.size, k), dtype=np.uint8)
    c = codes.copy()
    for i in range(k - 1, -1, -1):
        chars[:, i] = sym[(c % n).astype(np.int64)]
        c //= n
    return chars.view(f"S{k}").ravel().astype(f"<U{k}")


def encode_kmers(kmers: Sequence[str], symbols: str, k: int) -> Tuple[np.ndarray, np.ndarray]:
    """k-mer strings → (uint64 codes, ok mask).  ok is False for k-mers of the
    wrong length or with foreign symbols (they can never match a window)."""
    arr = np.asarray(list(kmers), dtype=str)
    ok = np.ones(arr.size, dtype=bool)
    codes = np.zeros(arr.size, dtype=np.uint64)
    if arr.size == 0:
        return codes, ok
    idx = np.full(256, -1, dtype=np.int64)
    for i, ch in enumerate(symbols):
        idx[ord(ch)] = i
    lens = np.char.str_len(arr)
    ok &= lens == k
    n = np.uint64(len(symbols))
    safe = np.where(ok, arr, symbols[0] * k)
    try:
        raw = np.char.encode(safe, "latin-1")
    except UnicodeEncodeError:
        raw = np.array([s.encode("latin-1", "replace") for s in safe])
    mat = np.frombuffer(raw.astype(f"S{k}").tobytes(), dtype=np.uint8).reshape(arr.size, k)
    d = idx[mat]
    ok &= (d >= 0).all(axis=1)
    d = np.where(d < 0, 0, d).astype(np.uint64)
    for i in range(k):
        codes = codes * n + d[:, i]
    return codes, ok


def basis_tables(S: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
    """Fresh (count, first) accumulation tables over the code space."""
    count = torch.zeros(S, dtype=torch.int64, device=device)
    first = torch.full((S,), -1, dtype=torch.int64, device=device)   # all-ones = +inf as uint64
    return count, first


def basis_accumulate(batch: SequenceBatch, alphabet: AlphabetT, k: int, count: torch.Tensor, first: Optional[torch.Tensor],
                     res_base: int = 0) -> None:
    """count[c] += occurrences of code c; first[c] = min(first[c], global position) unless first is None
    (occurrence counts only: the Totals row of learn.smk:380)."""
    tab = alphabet_tables(alphabet, batch.device)
    check(lib().skm_basis_accumulate(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), batch.n, _ptr(tab.lut),
                                     tab.nsym, int(k), int(res_base), _ptr(count), _ptr(first), _stream()))


def kmer_totals(batch: SequenceBatch, alphabet: AlphabetT, k: int) -> torch.Tensor:
    """int64 [nsym^k]: occurrences of every k-mer code over ALL sequences of the batch (learn.smk:380 Totals)."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    if S > _native.SKM_DENSE_MAX_SPACE:
        raise SkmError(-3, f"code space {tab.nsym}^{k} exceeds the table limit 2^27")
    count = torch.zeros(S, dtype=torch.int64, device=batch.device)
    basis_accumulate(batch, alphabet, k, count, None, 0)
    return count


def basis_finalize(alphabet: AlphabetT, k: int, count: Optional[torch.Tensor], first: torch.Tensor, min_filter: int = 0) -> Basis:
    """Tables -> basis in first-occurrence order.  count may be None (order-only tables, min_filter 0): every code
    with a first position is kept and Basis.counts is None."""
    dev = first.device
    tab = alphabet_tables(alphabet, dev)
    S = first.numel()
    ws_bytes = lib().skm_basis_finalize_workspace(S)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    codes = torch.empty(S, dtype=torch.int64, device=dev)
    counts = torch.empty(S, dtype=torch.int64, device=dev) if count is not None else None
    col = torch.empty(S, dtype=torch.int32, device=dev)
    dK = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().skm_basis_finalize(_ptr(count), _ptr(first), S, int(min_filter), _ptr(codes), _ptr(counts), _ptr(col),
                                   _ptr(dK), _ptr(ws), ws_bytes, _stream()))
    K = int(dK.item())
    return Basis(tab.name, int(k), tab.symbols, codes[:K], None if counts is None else counts[:K], col, K, S)


ORDER_FIRST_CHUNK_RES = 4 << 20     # residues in the first chunk of the order-only basis walk
ORDER_GROWTH = 4                    # every further chunk is this many times longer


def basis_first_progressive(batch: SequenceBatch, alphabet: AlphabetT, k: int, first: torch.Tensor, state: torch.Tensor,
                            res_base: int = 0) -> None:
    """first[c] = min(first[c], global position of the first window with code c), walking the shard front to back
    and stopping on the device once every code of the space has been seen (state int32[4], zeroed by the caller)."""
    tab = alphabet_tables(alphabet, batch.device)
    oh = np.ascontiguousarray(batch.offsets_host, dtype=np.int64)
    check(lib().skm_basis_first_progressive(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), oh.ctypes.data, batch.n,
                                            _ptr(tab.lut), tab.nsym, int(k), int(res_base), _ptr(first), _ptr(state),
                                            ORDER_FIRST_CHUNK_RES, ORDER_GROWTH, _stream()))


def order_only_supported(S: int) -> bool:
    return S <= lib().skm_basis_order_max_space()


def build_basis(batch: SequenceBatch, alphabet: AlphabetT, k: int, min_filter: int = 0, counts: bool = True) -> Basis:
    """Pass 1 of the vectorize rule (kmerize.smk:89-104) for one shard.

    counts=False with min_filter <= 0 asks for the basis ORDER only (Basis.counts is None): the reference uses the
    occurrence counts for nothing but the `count > min_filter` test, and with min_filter = 0 the basis is determined
    by the first positions alone, so the walk stops as soon as every code of the space has been seen (small code
    spaces; others take the full pass)."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    if S > _native.SKM_DENSE_MAX_SPACE:
        raise SkmError(-3, f"code space {tab.nsym}^{k} exceeds the table limit 2^27")
    if not counts and min_filter <= 0 and order_only_supported(S):
        first = torch.full((S,), -1, dtype=torch.int64, device=batch.device)
        state = torch.zeros(4, dtype=torch.int32, device=batch.device)
        basis_first_progressive(batch, alphabet, k, first, state, 0)
        return basis_finalize(alphabet, k, None, first, 0)
    count, first = basis_tables(S, batch.device)
    basis_accumulate(batch, alphabet, k, count, first, 0)
    return basis_finalize(alphabet, k, count, first, min_filter)


class OrderOnlyPlan:
    """The launch-bound front of the vectorize rule for ONE resident batch — table reset, order-only basis walk
    (4 chunk launches), key build, sort and emit of the finalisation: ten tiny kernels, ~0.15 ms of host-paced launches in
    front of a 0.85 ms count pass — captured once into a CUDA graph and replayed as a single launch.  The graph holds
    the batch's pointers and chunk geometry, so a plan belongs to its batch (a resident upload buffer that is refilled
    with batches of the same layout keeps its plan only if the offsets are the same; otherwise build a new one or run
    without).  Capture failure (a driver that refuses a node) leaves `graph = None`: the calls then run eagerly."""

    def __init__(self, batch: SequenceBatch, alphabet: AlphabetT, k: int, capture: bool = True):
        tab = alphabet_tables(alphabet, batch.device)
        dev = batch.device
        S = code_space(tab.nsym, k)
        if not order_only_supported(S):
            raise SkmError(-3, f"OrderOnlyPlan: code space {tab.nsym}^{k} exceeds {lib().skm_basis_order_max_space()}")
        self.batch, self.alphabet, self.k, self.tab, self.S = batch, alphabet, int(k), tab, S
        self.first = torch.empty(S, dtype=torch.int64, device=dev)
        self.state = torch.empty(4, dtype=torch.int32, device=dev)
        self.ws_bytes = lib().skm_basis_finalize_workspace(S)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.codes = torch.empty(S, dtype=torch.int64, device=dev)
        self.col = torch.empty(S, dtype=torch.int32, device=dev)
        self.dK = torch.empty(1, dtype=torch.int64, device=dev)
        self.graph = None
        if capture:
            self.enqueue()                               # eager once: function attributes, lazy module loading
            torch.cuda.synchronize(dev)
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self.enqueue()
                self.graph = g
            except Exception:                            # noqa: BLE001 — stay on the eager path
                self.graph = None
                torch.cuda.synchronize(dev)

    def enqueue(self) -> None:
        self.first.fill_(-1)
        self.state.zero_()
        self.dK.zero_()
        basis_first_progressive(self.batch, self.alphabet, self.k, self.first, self.state, 0)
        check(lib().skm_basis_finalize(None, _ptr(self.first), self.S, 0, _ptr(self.codes), None, _ptr(self.col), _ptr(self.dK),
                                       _ptr(self.ws), self.ws_bytes, _stream()))

    def launch(self) -> None:
        if self.graph is not None:
            self.graph.replay()
        else:
            self.enqueue()


def vectorize_order_only(batch: SequenceBatch, alphabet: AlphabetT, k: int, out: Optional[torch.Tensor] = None,
                         dtype: torch.dtype = torch.int32, count_events=None, plan: Optional[OrderOnlyPlan] = None) -> Tuple[Basis, torch.Tensor]:
    """Both passes of the vectorize rule (kmerize.smk:89-120) for min_filter = 0 over a small code space
    (order_only_supported): order-only basis walk + dense counts, with the read-back of K taken OFF the critical path.
    K only sizes the output, and K <= S: the count pass is launched with S columns (the column map sends every basis
    k-mer below K, the columns from K on stay zero) before the host asks for K, so the 8-byte read-back and the host
    latency around it overlap the count kernel instead of leaving the GPU idle between the passes (~0.07 ms of a
    1.04 ms C2 step).  Returns (basis, counts [N, K]); when the space is not saturated (K < S) the counts are compacted
    to K columns.  `out`: optional [N, S] buffer; `count_events`: optional (start, end) CUDA events recorded around the
    count launch; `plan`: an OrderOnlyPlan of THIS batch (the front of the step as one CUDA-graph launch).  The basis
    tensors of the result alias the plan's buffers: they are valid until the plan is launched again."""
    tab = alphabet_tables(alphabet, batch.device)
    dev = batch.device
    S = code_space(tab.nsym, k)
    if plan is None:
        plan = OrderOnlyPlan(batch, alphabet, k, capture=False)
    else:
        assert plan.batch is batch and plan.S == S and plan.k == int(k) and plan.tab.name == tab.name
    plan.launch()
    codes, col, dK = plan.codes, plan.col, plan.dK
    bits = {torch.int32: 32, torch.uint16: 16, torch.int16: 16}[dtype]
    if out is None:
        out = torch.empty((batch.n, S), dtype=dtype, device=dev)
    else:
        assert out.is_contiguous() and tuple(out.shape) == (batch.n, S) and out.dtype == dtype
    if count_events:
        count_events[0].record()
    check(lib().skm_count_dense(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), batch.n, _ptr(tab.lut), tab.nsym,
                                int(k), _ptr(col), S, S, bits, _ptr(out), batch.max_len, _stream()))
    if count_events:
        count_events[1].record()
    K = int(dK.item())                                  # the count pass is already running
    basis = Basis(tab.name, int(k), tab.symbols, codes[:K], None, col, K, S)
    if K < S:
        out = out[:, :K].contiguous()
    return basis, out


def basis_from_kmers(kmers: Sequence[str], alphabet: AlphabetT, k: int, device=None) -> Tuple[Basis, np.ndarray]:
    """A supplied basis (basis.txt branch, kmerize.smk:72-78, or a learned
    kmerlist).  Returns (Basis over the encodable k-mers, index of each of them
    in the supplied list)."""
    dev = _require_cuda(device)
    tab = alphabet_tables(alphabet, dev)
    S = code_space(tab.nsym, k)
    if S > _native.SKM_DENSE_MAX_SPACE:
        raise SkmError(-3, f"code space {tab.nsym}^{k} exceeds the table limit 2^27")
    codes, ok = encode_kmers(kmers, tab.symbols, k)
    keep = np.flatnonzero(ok)
    d_codes = torch.from_numpy(codes[keep].view(np.int64)).to(dev)
    col = torch.empty(S, dtype=torch.int32, device=dev)
    check(lib().skm_basis_colmap(_ptr(d_codes), len(keep), S, _ptr(col), _stream()))
    return Basis(tab.name, int(k), tab.symbols, d_codes, None, col, len(keep), S), keep


def gather_columns(matrix, index) -> "np.ndarray | torch.Tensor":
    """out[:, j] = matrix[:, index[j]], zero where index[j] is outside [0, n) — the column
    gather of KmerBasis.transform (vectorize.py:54-119).  numpy in → numpy out, tensor in → tensor out."""
    as_numpy = not isinstance(matrix, torch.Tensor)
    dev = _require_cuda(None if as_numpy else matrix.device)
    if as_numpy:
        arr = np.ascontiguousarray(matrix)
        if arr.ndim == 1:
            arr = arr.reshape(1, -1)
        if arr.dtype.itemsize not in (1, 2, 4, 8) or arr.dtype.kind not in "iufb":
            raise TypeError(f"gather_columns: unsupported dtype {arr.dtype}")
        d_in = torch.from_numpy(arr.view(f"u{arr.dtype.itemsize}").view(np.dtype(f"i{arr.dtype.itemsize}"))).to(dev)
    else:
        d_in = matrix.contiguous()
    rows, n = d_in.shape
    idx = torch.as_tensor(np.asarray(index, dtype=np.int64) if not isinstance(index, torch.Tensor) else index,
                          dtype=torch.int64, device=dev).contiguous()
    out = torch.empty((rows, idx.numel()), dtype=d_in.dtype, device=dev)
    check(lib().skm_gather_columns(_ptr(d_in), rows, n, d_in.element_size(), _ptr(idx), idx.numel(), _ptr(out), _stream()))
    if as_numpy:
        return out.cpu().numpy().view(arr.dtype)
    return out


def scatter_add(dst: torch.Tensor, src: torch.Tensor, row_map, col_map) -> None:
    """dst[row_map[r], col_map[c]] += src[r, c] for int64 matrices (negative map entries are dropped):
    the outer-join-and-sum of Merge.merge_dataframes (learn.smk:467-494)."""
    dev = dst.device
    assert dst.dtype == torch.int64 and src.dtype == torch.int64 and dst.is_contiguous()
    src = src.contiguous()
    rm = torch.as_tensor(row_map, dtype=torch.int64, device=dev).contiguous()
    cm = torch.as_tensor(col_map, dtype=torch.int64, device=dev).contiguous()
    assert rm.numel() == src.shape[0] and cm.numel() == src.shape[1]
    check(lib().skm_scatter_add_i64(_ptr(src), src.shape[0], src.shape[1], _ptr(rm), _ptr(cm), _ptr(dst), dst.shape[0],
                                    dst.shape[1], _stream()))


def basis_from_codes(codes: np.ndarray, alphabet, k: int, device=None) -> Tuple[Basis, np.ndarray]:
    """Basis whose column j holds code codes[j] (uint64, distinct)."""
    dev = _require_cuda(device)
    tab = alphabet_tables(alphabet, dev)
    S = code_space(tab.nsym, k)
    if S > _native.SKM_DENSE_MAX_SPACE:
        raise SkmError(-3, f"code space {tab.nsym}^{k} exceeds the table limit 2^27")
    codes = np.ascontiguousarray(codes, dtype=np.uint64)
    d_codes = torch.from_numpy(codes.view(np.int64)).to(dev)
    col = torch.empty(S, dtype=torch.int32, device=dev)
    check(lib().skm_basis_colmap(_ptr(d_codes), len(codes), S, _ptr(col), _stream()))
    return Basis(tab.name, int(k), tab.symbols, d_codes, None, col, len(codes), S), np.arange(len(codes))


def intersect_basis(target: Basis, other: Basis) -> Basis:
    """Columns of `target`, restricted to codes that `other` also holds.

    apply.smk:268-276 re-indexes query counts (columns = the query file's own
    basis) onto the union of columns: a learned column receives a query count
    only if the k-mer is in both bases."""
    assert target.S == other.S
    minus1 = torch.full_like(target.col_of_code, -1)
    col = torch.where(other.col_of_code >= 0, target.col_of_code, minus1)
    return Basis(target.alphabet, target.k, target.symbols, target.codes, target.counts, col, target.K, target.S)


# ---------------------------------------------------------------------------
# (b) counts
# ---------------------------------------------------------------------------
def count_dense(batch: SequenceBatch, alphabet: AlphabetT, k: int, basis: Optional[Basis] = None,
                dtype: torch.dtype = torch.int32, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-sequence k-mer counts [N, K] over `basis` (None = identity basis: column = code)."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    K = S if basis is None else basis.K
    bits = {torch.int32: 32, torch.uint16: 16, torch.int16: 16}[dtype]
    if out is None:
        out = torch.empty((batch.n, K), dtype=dtype, device=batch.device)
    else:
        assert out.is_contiguous() and tuple(out.shape) == (batch.n, K) and out.dtype == dtype
    check(lib().skm_count_dense(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), batch.n, _ptr(tab.lut), tab.nsym,
                                int(k), None if basis is None else _ptr(basis.col_of_code), S, K, bits, _ptr(out),
                                batch.max_len, _stream()))
    return out


def count_over_kmers(batch: SequenceBatch, alphabet, k: int, kmerlist: Sequence[str], dtype: torch.dtype = torch.int32) -> torch.Tensor:
    """Counts [N, len(kmerlist)] with one column per LIST ENTRY, in list order
    (``[k_counts.get(kmer, 0) for kmer in kmerlist]``, learn.smk:377-382): entries that
    cannot be encoded (wrong length, foreign characters) are zero columns, repeated
    entries repeat the column."""
    basis, keep = basis_from_kmers(kmerlist, alphabet, k, batch.device)
    n_list = len(kmerlist)
    codes = basis.codes_host()
    if basis.K == n_list and np.unique(codes).size == n_list:
        return count_dense(batch, alphabet, k, basis, dtype=dtype)
    # distinct codes -> dense columns, then expand to the list
    uniq, inverse = np.unique(codes, return_inverse=True)
    ub, _ = basis_from_codes(uniq, alphabet, k, batch.device)
    C = count_dense(batch, alphabet, k, ub, dtype=dtype)
    index = np.full(n_list, -1, dtype=np.int64)
    index[keep] = inverse
    return gather_columns(C, index)


def count_csr(batch: SequenceBatch, alphabet: AlphabetT, k: int, basis: Optional[Basis] = None, method: str = "warp"):
    """Per-sequence sorted (column, count) pairs as CSR: (rowptr int64 [N+1], cols int32 [nnz], vals int32 [nnz]).
    method "warp" (default): a warp sorts one sequence's keys in shared memory (skm_count_csr_sorted);
    "segsort": window keys in HBM + cub::DeviceSegmentedSort (skm_count_csr, the first implementation, kept as a
    cross-check)."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    dev = batch.device
    rowptr = torch.empty(batch.n + 1, dtype=torch.int64, device=dev)
    cols = torch.empty(max(batch.nres, 1), dtype=torch.int32, device=dev)
    vals = torch.empty(max(batch.nres, 1), dtype=torch.int32, device=dev)
    if method == "segsort":
        ws_bytes = lib().skm_count_csr_workspace(batch.nres, batch.n)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(lib().skm_count_csr(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), batch.n, _ptr(tab.lut), tab.nsym,
                                  int(k), None if basis is None else _ptr(basis.col_of_code), S, _ptr(rowptr), _ptr(cols),
                                  _ptr(vals), _ptr(ws), ws_bytes, _stream()))
    else:
        ws_bytes = lib().skm_count_csr_sorted_workspace(batch.nres, batch.n, batch.max_len, 32)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(lib().skm_count_csr_sorted(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), batch.n, _ptr(tab.lut), tab.nsym,
                                         int(k), 32, None if basis is None else _ptr(basis.col_of_code), S, None, None, 0,
                                         batch.max_len, _ptr(rowptr), _ptr(cols), None, _ptr(vals), _ptr(ws), ws_bytes, _stream()))
    nnz = int(rowptr[-1].item()) if batch.n else 0
    return rowptr, cols[:nnz].clone(), vals[:nnz].clone()


# ---------------------------------------------------------------------------
# (c) learn
# ---------------------------------------------------------------------------
def learn_dense(batch: SequenceBatch, alphabet: AlphabetT, k: int, basis: Optional[Basis], ann_id: torch.Tensor,
                n_ann: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-annotation summed counts.  ann_id int32 [N] (<0 = not in any row).
    Returns (M int64 [n_ann+1, K] with the "rest" row last, totals int64 [K])."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    K = S if basis is None else basis.K
    dev = batch.device
    ann_id = ann_id.to(device=dev, dtype=torch.int32).contiguous()
    assert ann_id.numel() == batch.n
    # group equal ids: stable sort so that each annotation is one contiguous run
    order = torch.sort(torch.where(ann_id < 0, torch.full_like(ann_id, n_ann), ann_id), stable=True).indices.contiguous()
    M = torch.empty((n_ann + 1, K), dtype=torch.int64, device=dev)
    totals = torch.empty(K, dtype=torch.int64, device=dev)
    check(lib().skm_learn_dense(_ptr(batch.residues), batch.nres, _ptr(batch.offsets), batch.n, _ptr(tab.lut), tab.nsym,
                                int(k), None if basis is None else _ptr(basis.col_of_code), S, K, _ptr(ann_id),
                                _ptr(order), int(n_ann), _ptr(M), _ptr(totals), _stream()))
    return M, totals


def learn_over_kmers(batch: SequenceBatch, alphabet, k: int, kmerlist: Sequence[str], ann_id: torch.Tensor,
                     n_ann: int) -> Tuple[np.ndarray, np.ndarray]:
    """learn_dense over a k-mer LIST: (M int64 [n_ann, len(kmerlist)], totals int64 [len(kmerlist)]) on the
    host, one column per list entry (zero columns for entries no window can match)."""
    basis, keep = basis_from_kmers(kmerlist, alphabet, k, batch.device)
    codes = basis.codes_host()
    n_list = len(kmerlist)
    plain = basis.K == n_list and np.unique(codes).size == n_list
    if not plain:
        uniq, inverse = np.unique(codes, return_inverse=True)
        basis, _ = basis_from_codes(uniq, alphabet, k, batch.device)
    M, totals = learn_dense(batch, alphabet, k, basis, ann_id, n_ann)
    if not plain:
        index = np.full(n_list, -1, dtype=np.int64)
        index[keep] = inverse
        M = gather_columns(M, index)
        totals = gather_columns(totals.reshape(1, -1), index).reshape(-1)
    return M[:n_ann].cpu().numpy(), totals.cpu().numpy()


# ---------------------------------------------------------------------------
# (d) apply
# ---------------------------------------------------------------------------
def row_norm2(X: torch.Tensor) -> torch.Tensor:
    X = X.contiguous()
    out = torch.empty(X.shape[0], dtype=torch.float64, device=X.device)
    fn = {torch.int32: lib().skm_row_norm2_i32, torch.int64: lib().skm_row_norm2_i64}[X.dtype]
    check(fn(_ptr(X), X.shape[0], X.shape[1], _ptr(out), _stream()))
    return out


@dataclass
class ApplyResult:
    top1: torch.Tensor      # int32 [Q]
    top2: torch.Tensor      # int32 [Q] (-1 if fewer than 2 annotations)
    score1: torch.Tensor    # float64 [Q]
    score2: torch.Tensor    # float64 [Q]
    scores: Optional[torch.Tensor] = None   # float64 [Q, A] when requested


TC_MAX_K = 32768


@dataclass
class PreparedAnnotations:
    """An annotation matrix split into base-256 digit planes for the tensor-core scoring kernel."""
    planes: torch.Tensor        # uint8 buffer [n_planes, pad128(A), pad128(K)]
    n_planes: int
    n_ann: int
    K: int
    mnorm2: torch.Tensor        # float64 [A]
    M: Optional[torch.Tensor] = None    # the int64 matrix itself (a reference, not a copy): per-row fallback of apply_tc

    def tiles(self) -> np.ndarray:
        """The annotation tiles of the prepared matrix as int32 [n_tiles, 3] = (first sorted row, width, digit planes)
        (blob header: n_tiles, rows per plane; TileDesc records follow the row permutation)."""
        hdr = self.planes[:8].view(torch.int32).cpu().numpy()
        n_tiles, rows = int(hdr[0]), int(hdr[1])
        off = 1024 + rows * 4
        return self.planes[off:off + 16 * n_tiles].view(torch.int32).cpu().numpy().reshape(-1, 4)[:, :3].copy()

    def issued_macs_per_query(self) -> int:
        """int8 multiply-accumulates apply_tc issues per query row: sum over tiles of width x planes x padded K."""
        t = self.tiles()
        return int((t[:, 1].astype(np.int64) * t[:, 2]).sum()) * ((self.K + 127) // 128 * 128)


def prepare_annotations(M: torch.Tensor, mnorm2: Optional[torch.Tensor] = None) -> Optional[PreparedAnnotations]:
    """Digit planes of M for apply_tc, or None when M is outside the tensor-core envelope
    (K > 32768, entries >= 2^32 or negative).  Do this once per learned matrix."""
    M = M.contiguous()
    A, K = M.shape
    if A == 0 or K == 0 or K > TC_MAX_K:
        return None
    dev = _require_cuda(M.device)
    nbytes = lib().skm_apply_tc_planes_bytes(A, K)
    planes = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    n_planes = _native.C.c_int(0)
    rc = lib().skm_apply_tc_prepare(_ptr(M), A, K, _ptr(planes), nbytes, _native.C.byref(n_planes), _stream())
    if rc == -3:            # SKM_ERR_UNSUPPORTED: too many digit planes
        return None
    check(rc)
    return PreparedAnnotations(planes, int(n_planes.value), A, K, row_norm2(M) if mnorm2 is None else mnorm2, M)


def rows_out_of_range(X: torch.Tensor, lo: int, hi: int) -> torch.Tensor:
    """Sorted indices (int64) of the rows of an int32 matrix that hold an element outside [lo, hi]."""
    dev = _require_cuda(X.device)
    X = X.contiguous()
    rows, cols = X.shape
    out = torch.empty(max(rows, 1), dtype=torch.int32, device=dev)
    dn = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().skm_rows_out_of_range_i32(_ptr(X), rows, cols, int(lo), int(hi), _ptr(out), rows, _ptr(dn), _stream()))
    n = int(dn.item())
    return torch.sort(out[:n].to(torch.int64)).values


def apply_tc(Q: torch.Tensor, prep: PreparedAnnotations, qnorm2: Optional[torch.Tensor] = None,
             full: bool = False) -> Optional[ApplyResult]:
    """Tensor-core scoring (tcgen05 int8 GEMM, exact integer dots).  Query rows holding a count above 255 (a
    5,000-residue low-complexity protein) do not fit the uint8 operand: they — and only they — are re-scored by the
    exact CUDA-core path (skm_apply_dense) against prep.M.  Returns None only when such rows exist and the
    prepared matrix does not carry M."""
    dev = _require_cuda(Q.device)
    Q = Q.contiguous()
    nq, K = Q.shape
    assert K == prep.K and Q.dtype == torch.int32
    if qnorm2 is None:
        qnorm2 = row_norm2(Q)
    A = prep.n_ann
    top1 = torch.empty(nq, dtype=torch.int32, device=dev)
    top2 = torch.empty(nq, dtype=torch.int32, device=dev)
    s1 = torch.empty(nq, dtype=torch.float64, device=dev)
    s2 = torch.empty(nq, dtype=torch.float64, device=dev)
    scores = torch.empty((nq, A), dtype=torch.float64, device=dev) if full else None
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = lib().skm_apply_tc_workspace(nq, K, A)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(lib().skm_apply_tc(_ptr(Q), nq, K, _ptr(prep.planes), prep.n_planes, A, _ptr(qnorm2), _ptr(prep.mnorm2), _ptr(top1),
                             _ptr(top2), _ptr(s1), _ptr(s2), _ptr(scores), _ptr(status), _ptr(ws), ws_bytes, _stream()))
    if int(status.item()) != 0:
        if prep.M is None:
            return None
        bad = rows_out_of_range(Q, 0, 255)
        r = apply_dense(Q[bad].contiguous(), prep.M, qnorm2=qnorm2[bad].contiguous(), mnorm2=prep.mnorm2, full=full,
                        tensor_cores=False)
        top1[bad], top2[bad], s1[bad], s2[bad] = r.top1, r.top2, r.score1, r.score2
        if full:
            scores[bad] = r.scores
    return ApplyResult(top1, top2, s1, s2, scores)


def apply_dense(Q: torch.Tensor, M: torch.Tensor, qnorm2: Optional[torch.Tensor] = None,
                mnorm2: Optional[torch.Tensor] = None, full: bool = False, chunk: int = 1 << 16,
                tensor_cores: Optional[bool] = None, prepared: Optional[PreparedAnnotations] = None) -> ApplyResult:
    """Cosine of every query count row against every annotation row + top-2
    (apply.smk:278-335).  Q int32 [nq, K], M int64 [A, K]; qnorm2 defaults to the
    norm over Q's own columns.  tensor_cores: None = use the tcgen05 path when the
    operands fit its exactness envelope and the problem is large enough to pay for the
    operand split; True / False force the choice (True still falls back when the envelope
    is violated)."""
    dev = Q.device
    Q = Q.contiguous()
    M = M.contiguous()
    nq, K = Q.shape
    A = M.shape[0]
    assert M.shape[1] == K and Q.dtype == torch.int32 and M.dtype == torch.int64
    if qnorm2 is None:
        qnorm2 = row_norm2(Q)
    if mnorm2 is None:
        mnorm2 = row_norm2(M) if prepared is None else prepared.mnorm2
    want_tc = tensor_cores if tensor_cores is not None else (nq * A * K >= (1 << 24))
    if want_tc and nq > 0 and A > 0 and 0 < K <= TC_MAX_K:
        prep = prepared if prepared is not None else prepare_annotations(M, mnorm2)
        if prep is not None:
            r = apply_tc(Q, prep, qnorm2, full)
            if r is not None:
                return r
    top1 = torch.empty(nq, dtype=torch.int32, device=dev)
    top2 = torch.empty(nq, dtype=torch.int32, device=dev)
    s1 = torch.empty(nq, dtype=torch.float64, device=dev)
    s2 = torch.empty(nq, dtype=torch.float64, device=dev)
    scores = torch.empty((nq, A), dtype=torch.float64, device=dev) if full else None
    chunk = max(1, min(chunk, nq, (1 << 31) // max(1, A * 8)))      # dots workspace <= 2 GiB
    ws_bytes = lib().skm_apply_dense_workspace(chunk, A, K)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    for q0 in range(0, nq, chunk):
        q1 = min(nq, q0 + chunk)
        check(lib().skm_apply_dense(_ptr(Q[q0:q1]), q1 - q0, K, _ptr(M), A, _ptr(qnorm2[q0:q1]), _ptr(mnorm2),
                                    _ptr(top1[q0:q1]), _ptr(top2[q0:q1]), _ptr(s1[q0:q1]), _ptr(s2[q0:q1]),
                                    None if scores is None else _ptr(scores[q0:q1]), _ptr(ws), ws_bytes, _stream()))
    return ApplyResult(top1, top2, s1, s2, scores)


def merge_top2(idx: torch.Tensor, score: torch.Tensor) -> ApplyResult:
    """Global top-2 from stacked per-shard top-2 lists (idx int64 [W, 2, Q] global annotation
    indices or -1, score float64 [W, 2, Q]) — the fan-in of annotation-sharded apply."""
    dev = _require_cuda(idx.device)
    idx = idx.contiguous()
    score = score.contiguous()
    W, two, nq = idx.shape
    assert two == 2 and tuple(score.shape) == (W, 2, nq) and idx.dtype == torch.int64 and score.dtype == torch.float64
    top1 = torch.empty(nq, dtype=torch.int32, device=dev)
    top2 = torch.empty(nq, dtype=torch.int32, device=dev)
    s1 = torch.empty(nq, dtype=torch.float64, device=dev)
    s2 = torch.empty(nq, dtype=torch.float64, device=dev)
    check(lib().skm_top2_merge(_ptr(idx), _ptr(score), W, nq, _ptr(top1), _ptr(top2), _ptr(s1), _ptr(s2), _stream()))
    return ApplyResult(top1, top2, s1, s2, None)


# ---------------------------------------------------------------------------
# sparse paths (large bases): sort-based learn, CSC, SpMM apply
# ---------------------------------------------------------------------------
def _sub_batch(batch: SequenceBatch, lo: int, hi: int) -> SequenceBatch:
    """Sequences [lo, hi) of a batch as a self-contained shard (same HBM buffer, rebased offsets)."""
    oh = batch.offsets_host
    base = int(oh[lo]) & ~15                      # keep the 16-byte alignment of the residue pointer
    sub = SequenceBatch(batch.residues[base:], batch.offsets[lo:hi + 1] - base, oh[lo:hi + 1] - base)
    sub.nres = int(oh[hi]) - base
    return sub


def _chunks_by_residues(offsets_host: np.ndarray, max_res: int):
    n = len(offsets_host) - 1
    out, lo = [], 0
    while lo < n:
        hi = int(np.searchsorted(offsets_host, offsets_host[lo] + max_res, side="right")) - 1
        hi = min(max(hi, lo + 1), n)
        out.append((lo, hi))
        lo = hi
    return out


def coo_merge(keys: torch.Tensor, vals: torch.Tensor, key_bound: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """Sum entries with equal keys; result sorted by key (Merge.merge_dataframes for sparse matrices).
    key_bound: exclusive upper bound of the keys (n_ann * S) when known — the sort then runs over its bits only."""
    dev = _require_cuda(keys.device)
    n = keys.numel()
    keys, vals = keys.contiguous(), vals.contiguous()
    ws_bytes = lib().skm_coo_merge_workspace(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    ok = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    ov = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    dn = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().skm_coo_merge(_ptr(keys), _ptr(vals), n, int(key_bound), _ptr(ok), _ptr(ov), _ptr(dn), _ptr(ws), ws_bytes, _stream()))
    m = int(dn.item())
    return ok[:m].clone(), ov[:m].clone()


def gather_sequences(batch: SequenceBatch, sel: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Sequences sel[0], sel[1], ... of a batch packed back to back: (residues uint8 [R' + 16], offsets int64 [n_sel + 1])."""
    dev = batch.device
    sel = sel.to(device=dev, dtype=torch.int64).contiguous()
    lens = (batch.offsets[1:] - batch.offsets[:-1])[sel]
    out_off = torch.zeros(sel.numel() + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lens, 0, out=out_off[1:])
    total = int(out_off[-1].item()) if sel.numel() else 0
    out_res = torch.empty(total + 32, dtype=torch.uint8, device=dev)
    check(lib().skm_gather_sequences(_ptr(batch.residues), _ptr(batch.offsets), _ptr(sel), sel.numel(), _ptr(out_res), _ptr(out_off), _stream()))
    return out_res, out_off


def coo_merge_runs(keys: torch.Tensor, vals: torch.Tensor, run_sizes: Sequence[int]) -> Tuple[torch.Tensor, torch.Tensor]:
    """coo_merge for an input that is a concatenation of SORTED runs (run_sizes entries each): merge tree + reduce-by-key."""
    dev = _require_cuda(keys.device)
    n = keys.numel()
    assert sum(run_sizes) == n
    keys, vals = keys.contiguous(), vals.contiguous()
    offs = np.zeros(len(run_sizes) + 1, dtype=np.int64)
    np.cumsum(np.asarray(run_sizes, dtype=np.int64), out=offs[1:])
    ws_bytes = lib().skm_coo_merge_runs_workspace(n, len(run_sizes))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    ok = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    ov = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    dn = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().skm_coo_merge_runs(_ptr(keys), _ptr(vals), offs.ctypes.data, len(run_sizes), _ptr(ok), _ptr(ov), _ptr(dn), _ptr(ws),
                                   ws_bytes, _stream()))
    m = int(dn.item())
    return ok[:m].clone(), ov[:m].clone()


def coo_merge_runs_packed(packed_ptr: int, run_sizes: Sequence[int], count_bits: int, device) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """coo_merge_runs for SORTED runs of packed words (key << count_bits | count, skm_coo_pack's format) lying back to
    back at device address `packed_ptr` (a peer-memory receive buffer).  Returns (keys, vals, n) with n a device scalar:
    the first n entries are the merged list — the caller slices after its own synchronisation."""
    dev = _require_cuda(device)
    n = int(sum(run_sizes))
    offs = np.zeros(len(run_sizes) + 1, dtype=np.int64)
    np.cumsum(np.asarray(run_sizes, dtype=np.int64), out=offs[1:])
    ws_bytes = lib().skm_coo_merge_runs_packed_workspace(n, len(run_sizes))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    ok = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    ov = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    dn = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().skm_coo_merge_runs_packed(packed_ptr, offs.ctypes.data, len(run_sizes), int(count_bits), _ptr(ok), _ptr(ov), _ptr(dn),
                                          _ptr(ws), ws_bytes, _stream()))
    return ok, ov, dn


def coo_pack(keys: torch.Tensor, vals: torch.Tensor, count_bits: int) -> Tuple[torch.Tensor, bool]:
    """(packed words int64, overflow) — skm_coo_pack; the single-GPU half of the exchange format (tests, side-cars)."""
    dev = _require_cuda(keys.device)
    out = torch.empty(keys.numel(), dtype=torch.int64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    check(lib().skm_coo_pack(_ptr(keys.contiguous()), _ptr(vals.contiguous()), keys.numel(), int(count_bits), _ptr(out), _ptr(flag), _stream()))
    return out, bool(flag.item())


GROUP_MAX_RES = (1 << 31) - 64      # residues per skm_learn_sparse_group call (its 32-bit window keys need < 2^31)


@dataclass
class _Placement:
    """Room for H foreign blocks (the dense rows of learn_sparse_hybrid's heavy annotations) inside the grouped list:
    skm_learn_sparse_group_place writes every entry straight to its place in the larger list."""
    ins_ann: torch.Tensor               # int64 [H] ascending annotation ids of the blocks
    ins_cum: Optional[torch.Tensor]     # int64 [H] inclusive prefix of the block sizes (None when H = 0)
    ins_pos: torch.Tensor               # int64 [H] INT64_MAX on entry; skm_learn_sparse_group_place's candidates per block
    totals: Optional[torch.Tensor]      # int64 [S] += counts per code, or None
    extra: int                          # entries of all blocks


def _learn_grouped(batch: SequenceBatch, tab: AlphabetTables, k: int, ann_id: torch.Tensor, n_ann: int,
                   place: Optional[_Placement] = None):
    """The grouped path of learn_sparse: the annotated sequences are gathered in annotation order and sorted one
    annotation slice at a time with 32-bit keys (skm_learn_sparse_group; with `place`, skm_learn_sparse_group_place).
    ann_id: int32 on the device.  Returns (keys buffer, vals buffer, entries of the grouped list) without slicing — with
    `place` the buffers also have room for its blocks — or None when the path does not apply (no sequences, no
    annotations, a code space beyond 32-bit slice keys, or a slice of GROUP_MAX_RES residues or more)."""
    dev = batch.device
    S = code_space(tab.nsym, k)
    per_group = ((1 << 32) - 2) // S
    if per_group < 1 or batch.n == 0 or n_ann == 0:
        return None
    extra = place.extra if place is not None else 0
    key = torch.where((ann_id >= 0) & (ann_id < n_ann), ann_id, torch.full_like(ann_id, n_ann))
    sk, order = torch.sort(key, stable=True)
    starts = list(range(0, n_ann, per_group)) + [n_ann]
    bounds = torch.searchsorted(sk, torch.tensor(starts, dtype=torch.int32, device=dev)).tolist()     # one sync
    n_sel = bounds[-1]
    if n_sel == 0:
        cap = max(extra, 1)
        return torch.empty(cap, dtype=torch.int64, device=dev), torch.empty(cap, dtype=torch.int64, device=dev), 0
    g_res, g_off = gather_sequences(batch, order[:n_sel])
    g_ann = sk[:n_sel].contiguous()
    edge = g_off[torch.tensor(bounds, dtype=torch.int64, device=dev)].tolist()
    if max(edge[i + 1] - (edge[i] & ~15) for i in range(len(starts) - 1)) >= GROUP_MAX_RES:
        return None
    total = edge[-1] + extra
    keys = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
    vals = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
    dn = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = None
    for gi in range(len(starts) - 1):
        s0, s1 = bounds[gi], bounds[gi + 1]
        if s1 == s0:
            continue
        base = edge[gi] & ~15
        nres = edge[gi + 1] - base
        ws_bytes = lib().skm_learn_sparse_group_workspace(nres)
        if ws is None or ws.numel() < ws_bytes:
            ws = None
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        offs = (g_off[s0:s1 + 1] - base).contiguous()
        args = (_ptr(g_res[base:]), nres, _ptr(offs), s1 - s0, _ptr(tab.lut), tab.nsym, int(k), _ptr(g_ann[s0:s1]), starts[gi],
                starts[gi + 1] - starts[gi], _ptr(keys), _ptr(vals), total, _ptr(dn))
        if place is not None:
            check(lib().skm_learn_sparse_group_place(*args, _ptr(place.ins_ann), _ptr(place.ins_cum), int(place.ins_pos.numel()),
                                                     _ptr(place.ins_pos), _ptr(place.totals), _ptr(ws), ws.numel(), _stream()))
        else:
            check(lib().skm_learn_sparse_group(*args, _ptr(ws), ws.numel(), _stream()))
    m = int(dn.item())
    assert m <= total
    return keys, vals, m


def learn_sparse(batch: SequenceBatch, alphabet, k: int, ann_id: torch.Tensor, n_ann: int,
                 max_chunk_res: int = 1 << 28, method: str = "grouped") -> Tuple[torch.Tensor, torch.Tensor]:
    """Annotation x k-mer count matrix as a COO list sorted by key = ann * S + code
    (keys int64 holding the uint64 pattern, vals int64).  Sequences with ann_id < 0 do not
    contribute (Totals come from the basis tables).

    method "grouped" (default): the annotated sequences are gathered in annotation order and sorted one annotation
    slice at a time with 32-bit keys (skm_learn_sparse_group); "global": one 64-bit radix sort over all window keys of
    the shard (skm_learn_sparse, the first implementation, kept as a cross-check and for slices whose keys need more
    than 32 bits)."""
    if method not in ("grouped", "global"):
        raise ValueError(f"learn_sparse: method must be 'grouped' or 'global', not {method!r}")
    tab = alphabet_tables(alphabet, batch.device)
    dev = batch.device
    ann_id = ann_id.to(device=dev, dtype=torch.int32).contiguous()
    assert ann_id.numel() == batch.n
    S = code_space(tab.nsym, k)
    grouped = _learn_grouped(batch, tab, k, ann_id, n_ann) if method == "grouped" else None
    if grouped is not None:
        keys, vals, m = grouped
        return keys[:m].clone(), vals[:m].clone()
    parts_k, parts_v = [], []
    for lo, hi in _chunks_by_residues(batch.offsets_host, max_chunk_res):
        sub = _sub_batch(batch, lo, hi)
        ws_bytes = lib().skm_learn_sparse_workspace(sub.nres)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        ok = torch.empty(max(sub.nres, 1), dtype=torch.int64, device=dev)
        ov = torch.empty(max(sub.nres, 1), dtype=torch.int64, device=dev)
        dn = torch.zeros(1, dtype=torch.int64, device=dev)
        check(lib().skm_learn_sparse(_ptr(sub.residues), sub.nres, _ptr(sub.offsets), sub.n, _ptr(tab.lut), tab.nsym, int(k),
                                     _ptr(ann_id[lo:hi]), int(n_ann), _ptr(ok), _ptr(ov), _ptr(dn), _ptr(ws), ws_bytes,
                                     _stream()))
        m = int(dn.item())
        parts_k.append(ok[:m].clone())
        parts_v.append(ov[:m].clone())
        del ws, ok, ov
    if len(parts_k) == 1:
        return parts_k[0], parts_v[0]
    if not parts_k:
        z = torch.zeros(0, dtype=torch.int64, device=dev)
        return z, z.clone()
    return coo_merge(torch.cat(parts_k), torch.cat(parts_v), key_bound=n_ann * S)


def _learn_sorted(batch: SequenceBatch, tab: AlphabetTables, k: int, ann_id: torch.Tensor, n_ann: int, want_totals: bool):
    """The all-sorted path (the reference of the hybrid one): learn_sparse, and with want_totals the Totals row — the
    annotated share is the column sums of the matrix (one atomic per entry instead of one per window), the unannotated
    sequences are counted window by window.  ann_id: int32 on the device."""
    keys, vals = learn_sparse(batch, tab, k, ann_id, n_ann)
    if not want_totals:
        return keys, vals
    dev = batch.device
    S = code_space(tab.nsym, k)
    totals = torch.zeros(S, dtype=torch.int64, device=dev)
    check(lib().skm_coo_colsum(_ptr(keys), _ptr(vals), keys.numel(), S, _ptr(totals), _stream()))
    rest = torch.nonzero((ann_id < 0) | (ann_id >= n_ann)).reshape(-1)
    if rest.numel():
        g_res, g_off = gather_sequences(batch, rest)
        basis_accumulate(SequenceBatch(g_res, g_off, g_off.cpu().numpy()), tab, k, totals, None, 0)
    return keys, vals, totals


HEAVY_ROW_DIV = 4                   # an annotation is "heavy" when it has more residues than S / HEAVY_ROW_DIV ...
HEAVY_ROWS_MAX_BYTES = 8 << 30      # ... as long as the dense rows of all heavy annotations stay below this
ROWS_L2_BYTES = 100 << 20           # rows counted by one skm_rows_accumulate launch (L2-resident counters): ~0.8 of the 126 MB L2, from a sweep (profiles/R2al_*)


def _learn_rows(batch: SequenceBatch, tab: AlphabetTables, k: int, ann_id: torch.Tensor, n_ann: int, S: int,
                want_totals: bool, heavy_div: int):
    """Dense-row part of learn_sparse_hybrid: returns (rows uint32 [R, S] or None when R = 0, heavy annotation ids
    int64 [H] ascending).  Rows 0..H-1 are the heavy annotations, row H (when want_totals) the unannotated sequences."""
    dev = batch.device
    lens = (batch.offsets[1:] - batch.offsets[:-1])
    valid = (ann_id >= 0) & (ann_id < n_ann)
    per_ann = torch.zeros(n_ann + 1, dtype=torch.int64, device=dev)
    per_ann.index_add_(0, torch.where(valid, ann_id, torch.full_like(ann_id, n_ann)).to(torch.int64), lens)
    thr = max(S // max(int(heavy_div), 1), 1)
    max_rows = max(int(HEAVY_ROWS_MAX_BYTES // (4 * S)) - 1, 0)
    heavy = torch.nonzero(per_ann[:n_ann] > thr).reshape(-1)
    if heavy.numel() > max_rows:                         # keep the largest ones
        order = torch.argsort(per_ann[heavy], descending=True)[:max_rows]
        heavy = torch.sort(heavy[order]).values
    H = int(heavy.numel())                               # one sync
    rest_row = H if want_totals else -1
    R = H + (1 if want_totals else 0)
    if R == 0:
        return None, heavy
    row_of_ann = torch.full((n_ann + 1,), -1, dtype=torch.int32, device=dev)
    row_of_ann[heavy] = torch.arange(H, dtype=torch.int32, device=dev)
    row_of_ann[n_ann] = rest_row
    row_of_seq = row_of_ann[torch.where(valid, ann_id, torch.full_like(ann_id, n_ann)).to(torch.int64)].contiguous()
    # the sequences of a row next to each other: the row stays in L2 while they stream past
    sel = torch.nonzero(row_of_seq >= 0).reshape(-1)
    order = torch.sort(row_of_seq[sel].to(torch.int64), stable=True).indices
    sel = sel[order]
    rows = torch.zeros((R, S), dtype=torch.int32, device=dev)
    if sel.numel():
        g_res, g_off = gather_sequences(batch, sel)
        g_row = row_of_seq[sel].contiguous()
        total = int(g_off[-1].item())
        # One launch per group of rows whose counters fit L2 together (ROWS_L2_BYTES): a launch spreads its CTAs over the
        # whole residue range it is given, so a single launch over all rows touches every row at once (C3: 66 rows =
        # 442 MB) and the atomics run at DRAM speed.  Also < 2^32 residues per call.
        per_launch = max(int(ROWS_L2_BYTES // (4 * S)), 1)
        row_edges = torch.searchsorted(g_row, torch.arange(R + 1, dtype=torch.int32, device=dev)).tolist()
        g_off_host = None
        bounds = [0]
        for r0 in range(0, R, per_launch):
            lo, hi = row_edges[r0], row_edges[min(r0 + per_launch, R)]
            if hi == lo:
                continue
            if total >= (1 << 32) - 64:                  # a huge group: cut it by sequences
                if g_off_host is None:
                    g_off_host = g_off.cpu().numpy()
                while g_off_host[hi] - g_off_host[bounds[-1]] >= (1 << 31):
                    bounds.append(int(np.searchsorted(g_off_host, g_off_host[bounds[-1]] + (1 << 31), side="right")) - 1)
            bounds.append(hi)
        edges = g_off[torch.tensor(bounds, dtype=torch.int64, device=dev)].tolist()
        for i, (lo, hi) in enumerate(zip(bounds[:-1], bounds[1:])):
            if hi == lo:
                continue
            e0, e1 = edges[i], edges[i + 1]
            base = e0 & ~15
            offs = (g_off[lo:hi + 1] - base).contiguous()
            check(lib().skm_rows_accumulate(_ptr(g_res[base:]), e1 - base, _ptr(offs), hi - lo, _ptr(tab.lut), tab.nsym, int(k),
                                            _ptr(g_row[lo:hi]), int(S), _ptr(rows), _stream()))
    return rows, heavy


def _row_blocks(rows: Optional[torch.Tensor], H: int, S: int):
    """Layout of the heavy rows' entries in the COO list: (blk_off int64 [H, nblk] exclusive non-zeros in front of each
    block inside its row, row_nnz int64 [H], cum int64 [H] inclusive prefix of row_nnz, heavy_total); all None / 0 when
    H == 0."""
    if H == 0:
        return None, None, None, 0
    blk = lib().skm_rows_block()
    counts = torch.empty((H, (S + blk - 1) // blk), dtype=torch.int32, device=rows.device)
    check(lib().skm_rows_block_counts(_ptr(rows), H, S, _ptr(counts), _stream()))
    c64 = counts.to(torch.int64)
    incl = torch.cumsum(c64, dim=1)
    blk_off = (incl - c64).contiguous()
    row_nnz = incl[:, -1].contiguous()
    cum = torch.cumsum(row_nnz, 0).contiguous()
    return blk_off, row_nnz, cum, int(cum[-1].item())    # one sync


def _learn_hybrid(batch: SequenceBatch, tab: AlphabetTables, k: int, ann_id: torch.Tensor, n_ann: int, S: int,
                  want_totals: bool, heavy_div: int):
    dev = batch.device
    if batch.n == 0 or n_ann == 0:
        return _learn_sorted(batch, tab, k, ann_id, n_ann, want_totals)
    rows, heavy = _learn_rows(batch, tab, k, ann_id, n_ann, S, want_totals, heavy_div)
    H = int(heavy.numel())
    totals = torch.zeros(S, dtype=torch.int64, device=dev) if want_totals else None
    # light part: the heavy annotations (and, with totals, nothing else) leave the sorted path
    if H:
        is_heavy = torch.zeros(n_ann + 1, dtype=torch.bool, device=dev)
        is_heavy[heavy] = True
        safe = torch.where((ann_id >= 0) & (ann_id < n_ann), ann_id, torch.full_like(ann_id, n_ann)).to(torch.int64)
        ann_light = torch.where(is_heavy[safe], torch.full_like(ann_id, -1), ann_id)
    else:
        ann_light = ann_id
    # The heavy blocks' sizes first (the rows are counted already), then the light list is sorted slice by slice and
    # written STRAIGHT to its final places between the heavy blocks, adding its counts to the Totals on the way
    # (skm_learn_sparse_group_place): no column-sum pass over the light list and no copy of it.
    blk_off, row_nnz, cum, heavy_total = _row_blocks(rows, H, S)
    ins_pos = torch.full((H,), INT64_MAX, dtype=torch.int64, device=dev)
    placed = _learn_grouped(batch, tab, k, ann_light, n_ann, _Placement(heavy, cum, ins_pos, totals, heavy_total))
    if placed is None:
        return _learn_sorted(batch, tab, k, ann_id, n_ann, want_totals)
    keys, vals, m_light = placed
    if want_totals:
        check(lib().skm_rows_colsum(_ptr(rows), rows.shape[0], S, _ptr(totals), _stream()))
    total = m_light + heavy_total
    if H:
        # light entries in front of block h = the smallest recorded index over the blocks from h on (none: all of them)
        tail = torch.cat([ins_pos, torch.tensor([m_light], dtype=torch.int64, device=dev)])
        before = torch.flip(torch.cummin(torch.flip(tail, [0]), 0).values, [0])[:H]
        row_dst = (before + cum - row_nnz).contiguous()
        check(lib().skm_rows_emit(_ptr(rows), H, S, _ptr(blk_off), _ptr(row_dst), _ptr(heavy.contiguous()), _ptr(keys), _ptr(vals), total, _stream()))
    keys, vals = keys[:total], vals[:total]
    return (keys, vals, totals) if want_totals else (keys, vals)


def learn_sparse_hybrid(batch: SequenceBatch, alphabet, k: int, ann_id: torch.Tensor, n_ann: int, want_totals: bool = False,
                        heavy_div: int = HEAVY_ROW_DIV):
    """learn_sparse for heavy-tailed family sizes: annotations with more residues than S / heavy_div are COUNTED into
    dense L2-resident rows (skm_rows_accumulate; their sequences gathered together), the others are sorted
    (skm_learn_sparse_group_place) straight into the gaps between the heavy rows' entries.  Same result as learn_sparse,
    bit for bit; inputs the grouped sort cannot take (a slice of GROUP_MAX_RES residues or more, no sequences, no
    annotations) get the all-sorted result.  want_totals: also return the Totals row (int64 [S], occurrences over ALL
    sequences, learn.smk:380) — the unannotated sequences are then counted into a row of their own and the totals are
    column sums."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    if S > _native.SKM_DENSE_MAX_SPACE:
        raise SkmError(-3, f"code space {tab.nsym}^{k} exceeds the table limit 2^27")
    ann_id = ann_id.to(device=batch.device, dtype=torch.int32).contiguous()
    assert ann_id.numel() == batch.n
    return _learn_hybrid(batch, tab, k, ann_id, n_ann, S, want_totals, heavy_div)


def learn_sparse_with_totals(batch: SequenceBatch, alphabet, k: int, ann_id: torch.Tensor, n_ann: int, method: str = "hybrid"):
    """learn_sparse + the Totals row (k-mer occurrences over ALL sequences, learn.smk:380) -> (keys, vals, totals int64 [S]).
    method "hybrid" (default): heavy annotations and the unannotated sequences are counted into dense rows, the Totals are
    column sums (learn_sparse_hybrid).  "sorted": everything through the sort; the annotated share of the totals is the
    column sums of the matrix and the unannotated sequences are counted window by window (the round-1 path, kept as the
    cross-check)."""
    if method not in ("hybrid", "sorted"):
        raise ValueError(f"learn_sparse_with_totals: method must be 'hybrid' or 'sorted', not {method!r}")
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    if S > _native.SKM_DENSE_MAX_SPACE:
        raise SkmError(-3, f"code space {tab.nsym}^{k} exceeds the table limit 2^27")
    ann_id = ann_id.to(device=batch.device, dtype=torch.int32).contiguous()
    assert ann_id.numel() == batch.n
    if method == "hybrid":
        return _learn_hybrid(batch, tab, k, ann_id, n_ann, S, True, HEAVY_ROW_DIV)
    return _learn_sorted(batch, tab, k, ann_id, n_ann, True)


@dataclass
class AnnotationCSC:
    """k-mer-major view of an annotation slice [ann_lo, ann_lo + n_ann) of a learned matrix."""
    colptr: torch.Tensor    # int64 [S+1]
    rows: torch.Tensor      # int32 [nnz] annotation index relative to ann_lo
    mvals: torch.Tensor     # int32 [nnz] = M[a, c]
    mnorm2: torch.Tensor    # float64 [n_ann], exact integer sums
    inv_m32: torch.Tensor   # float32 [n_ann] = 1 / ||m_a|| (screening pass)
    max_m: int              # largest entry
    n_ann: int
    ann_lo: int
    S: int
    packed: Optional[torch.Tensor] = None   # int32 (uint32 pattern) [nnz]: value << 16 | row, when n_ann <= 65536 and max_m < 65536


def csc_build(keys: torch.Tensor, vals: torch.Tensor, S: int, n_ann: int, ann_lo: int = 0, pack: bool = True) -> AnnotationCSC:
    """CSC of the annotation slice [ann_lo, ann_lo + n_ann) of a sorted COO matrix.  pack: also keep the entries as one
    32-bit word each (value << 16 | annotation) when they fit — apply_sparse then reads half the bytes."""
    dev = _require_cuda(keys.device)
    if keys.numel():
        # the slice is contiguous because the list is sorted by ann * S + code
        bounds = torch.tensor([ann_lo * S, (ann_lo + n_ann) * S], dtype=torch.int64, device=dev)
        i0, i1 = torch.searchsorted(keys, bounds).tolist()
        keys = (keys[i0:i1] - ann_lo * S).contiguous()
        vals = vals[i0:i1].contiguous()
    nnz = keys.numel()
    ws_bytes = lib().skm_csc_build_workspace_cols(nnz, n_ann, int(S))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    colptr = torch.empty(S + 1, dtype=torch.int64, device=dev)
    rows = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    mvals = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    mn2 = torch.zeros(max(n_ann, 1), dtype=torch.float64, device=dev)
    inv32 = torch.zeros(max(n_ann, 1), dtype=torch.float32, device=dev)
    max_m = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().skm_csc_build(_ptr(keys), _ptr(vals), nnz, int(S), int(n_ann), _ptr(colptr), _ptr(rows), _ptr(mvals), _ptr(mn2),
                              _ptr(inv32), _ptr(max_m), _ptr(ws), ws_bytes, _stream()))
    mx = int(max_m.item())
    if mx >= 2 ** 31:
        raise SkmError(-3, f"csc_build: an annotation count of {mx} does not fit the 32-bit CSC values")
    csc = AnnotationCSC(colptr, rows[:nnz], mvals[:nnz], mn2[:n_ann], inv32[:n_ann], mx, int(n_ann), int(ann_lo), int(S))
    if pack and nnz and n_ann <= 65536 and mx < 65536:
        csc.packed = torch.empty(nnz, dtype=torch.int32, device=dev)
        check(lib().skm_csc_pack(_ptr(csc.rows), _ptr(csc.mvals), nnz, _ptr(csc.packed), _stream()))
    return csc


SPARSE_MAX_ANN = 50 * 1024          # annotations per apply_sparse call with 32-bit accumulators (half with 64-bit)


def apply_sparse(rowptr: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, csc: AnnotationCSC,
                 max_row_total: Optional[int] = None, use_packed: bool = True,
                 rows_out: Optional[torch.Tensor] = None) -> ApplyResult:
    """SpMM scoring of CSR queries (codes + counts, count_csr with basis=None) against one annotation slice.
    max_row_total bounds the sum of a query's counts (default: the largest row total, one reduction); it decides
    whether the exact integer dots fit 32-bit accumulators.  rows_out: a float64 device view [nq, >= n_ann] with unit
    column stride (any row stride) that receives every query's full cosine row, entry for entry the value the top-2
    scores are taken from (skm_apply_sparse_rows)."""
    dev = _require_cuda(rowptr.device)
    nq = rowptr.numel() - 1
    if nq == 0 or csc.n_ann == 0:               # no candidates: -1 / NaN, like apply_dense
        return ApplyResult(torch.full((nq,), -1, dtype=torch.int32, device=dev), torch.full((nq,), -1, dtype=torch.int32, device=dev),
                           torch.full((nq,), float("nan"), dtype=torch.float64, device=dev),
                           torch.full((nq,), float("nan"), dtype=torch.float64, device=dev), None)
    top1 = torch.empty(nq, dtype=torch.int32, device=dev)
    top2 = torch.empty(nq, dtype=torch.int32, device=dev)
    s1 = torch.empty(nq, dtype=torch.float64, device=dev)
    s2 = torch.empty(nq, dtype=torch.float64, device=dev)
    if max_row_total is None:
        max_row_total = query_row_total_max(rowptr, vals)
    acc_bits = sparse_acc_bits(csc.max_m, max_row_total)
    if csc.n_ann > sparse_max_ann(acc_bits):
        raise SkmError(-3, f"apply_sparse: {csc.n_ann} annotations with {acc_bits}-bit accumulators exceed one pass "
                           f"({sparse_max_ann(acc_bits)}); use apply_sparse_tiled")
    args = (_ptr(rowptr), _ptr(cols), _ptr(vals), nq, _ptr(csc.colptr), _ptr(csc.rows), _ptr(csc.mvals),
            _ptr(csc.packed) if use_packed else None, _ptr(csc.mnorm2), _ptr(csc.inv_m32), csc.n_ann, acc_bits, _ptr(top1), _ptr(top2),
            _ptr(s1), _ptr(s2), None)
    if rows_out is None:
        check(lib().skm_apply_sparse(*args, _stream()))
    else:
        if (rows_out.dtype != torch.float64 or rows_out.device != dev or rows_out.dim() != 2 or rows_out.shape[0] != nq
                or rows_out.shape[1] < csc.n_ann or rows_out.stride(1) != 1):
            raise SkmError(-2, f"apply_sparse: rows_out must be a float64 [{nq}, >= {csc.n_ann}] view with unit column stride on {dev}")
        check(lib().skm_apply_sparse_rows(*args, _ptr(rows_out), rows_out.stride(0), _stream()))
    return ApplyResult(top1, top2, s1, s2, None)


def query_row_total_max(rowptr: torch.Tensor, vals: torch.Tensor) -> int:
    """Largest sum of counts over a CSR row (= number of valid windows of the longest query)."""
    if vals.numel() == 0:
        return 0
    csum = torch.zeros(vals.numel() + 1, dtype=torch.int64, device=vals.device)
    torch.cumsum(vals, 0, out=csum[1:])
    return int((csum[rowptr[1:]] - csum[rowptr[:-1]]).max().item())


def sparse_acc_bits(max_m: int, max_row_total: int) -> int:
    """Width of the exact integer accumulators of apply_sparse: a dot is at most max_m * (sum of the query's counts)."""
    return 32 if int(max_m) * max(int(max_row_total), 1) < 2 ** 32 else 64


def sparse_max_ann(acc_bits: int) -> int:
    """Annotations one apply_sparse pass holds in shared memory (200 KB of accumulators)."""
    return SPARSE_MAX_ANN if acc_bits == 32 else SPARSE_MAX_ANN // 2


ROWS_CHUNK_BYTES = 1 << 30         # device buffer of one query chunk of association rows (two are in flight)


def apply_sparse_tiled(rowptr, cols, vals, keys, mvals, S: int, n_ann: int, tile: Optional[int] = None,
                       rows_sink: Optional[Callable[[int, np.ndarray], None]] = None,
                       chunk_rows: Optional[int] = None) -> ApplyResult:
    """All annotations of a sorted COO matrix, `tile` at a time, merged with the top-2 merge (the same fan-in as the
    multi-GPU annotation sharding).  The tile defaults to what one pass can hold, which depends on the accumulator
    width: 51,200 annotations with 32-bit accumulators, 25,600 when max(M) * (largest query total) needs 64 bits.

    rows_sink(q0, block): also stream the full cosine rows (the association matrix) to the host, `chunk_rows` queries
    at a time (default: a ~1 GiB float64 block), in query order: block is float64 [rows, n_ann] for queries
    [q0, q0 + rows), a view of pinned memory that is reused once the call returns.  An AssociationsCSVText sink
    instead gets every chunk as CSV text formatted on the device (chunks of ~1 GiB of worst-case text), and only the
    text is copied to the host.  The result is bit-identical to the call without a sink."""
    dev = rowptr.device
    nq = rowptr.numel() - 1
    if rows_sink is not None and nq > 0:
        return _apply_sparse_rows_tiled(rowptr, cols, vals, keys, mvals, S, n_ann, tile, rows_sink, chunk_rows)
    if n_ann <= 0 or nq <= 0:
        return ApplyResult(torch.full((nq,), -1, dtype=torch.int32, device=dev), torch.full((nq,), -1, dtype=torch.int32, device=dev),
                           torch.full((nq,), float("nan"), dtype=torch.float64, device=dev),
                           torch.full((nq,), float("nan"), dtype=torch.float64, device=dev), None)
    row_total = query_row_total_max(rowptr, vals)
    max_m = int(mvals.max().item()) if mvals.numel() else 0
    cap = sparse_max_ann(sparse_acc_bits(max_m, row_total))
    tile = cap if tile is None else max(1, min(int(tile), cap))
    idxs, scs = [], []
    for a0 in range(0, n_ann, tile):
        na = min(tile, n_ann - a0)
        r = apply_sparse(rowptr, cols, vals, csc_build(keys, mvals, S, na, a0), row_total)
        if n_ann <= tile:
            return r
        i = torch.stack([r.top1.to(torch.int64), r.top2.to(torch.int64)])
        idxs.append(torch.where(i >= 0, i + a0, i))
        scs.append(torch.stack([r.score1, r.score2]))
    return merge_top2(torch.stack(idxs), torch.stack(scs))


def _apply_sparse_rows_tiled(rowptr, cols, vals, keys, mvals, S: int, n_ann: int, tile: Optional[int], rows_sink,
                             chunk_rows: Optional[int]) -> ApplyResult:
    """apply_sparse_tiled with a rows sink (nq > 0).  The annotation-tile CSCs are built once; every query chunk runs
    each tile into its column slice of a [chunk, n_ann] device block (the kernel reads absolute CSR offsets, so a chunk
    is rowptr[q0:q1 + 1] without a copy).  Two device and two pinned host blocks: the copy of chunk i (side stream,
    events) and the sink's work on it overlap the kernels of chunk i + 1."""
    dev = rowptr.device
    nq = rowptr.numel() - 1
    n_ann = max(int(n_ann), 0)
    csv = rows_sink if isinstance(rows_sink, AssociationsCSVText) else None
    row_bytes = csv.row_bound() if csv is not None else 8 * max(n_ann, 1)
    chunk = int(chunk_rows) if chunk_rows is not None else ROWS_CHUNK_BYTES // row_bytes
    chunk = max(1, min(chunk, nq))
    tiles = []
    row_total = 0
    if n_ann > 0:
        row_total = query_row_total_max(rowptr, vals)
        max_m = int(mvals.max().item()) if mvals.numel() else 0
        cap = sparse_max_ann(sparse_acc_bits(max_m, row_total))
        tile = cap if tile is None else max(1, min(int(tile), cap))
        tiles = [(a0, csc_build(keys, mvals, S, min(tile, n_ann - a0), a0)) for a0 in range(0, n_ann, tile)]
    main = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(dev)
    dbuf = [torch.empty((chunk, n_ann), dtype=torch.float64, device=dev) for _ in range(2 if csv is None else 1)]
    outs = [[] for _ in tiles]                      # per tile: the chunks' ApplyResults
    if csv is not None:
        # the block is formatted on the device right behind its kernels; only the text is copied (TextPipe)
        pipe = csv.pipe(chunk)
        for q0 in range(0, nq, chunk):
            n = min(chunk, nq - q0)
            rp = rowptr[q0:q0 + n + 1]
            for t, (a0, csc) in enumerate(tiles):
                outs[t].append(apply_sparse(rp, cols, vals, csc, row_total, rows_out=dbuf[0][:n, a0:a0 + csc.n_ann]))
            s = pipe.slot()
            pipe.push(s, csv.format_rows(q0, dbuf[0][:n], pipe.text[s]))
        pipe.close()
    else:
        hbuf = [torch.empty((chunk, n_ann), dtype=torch.float64, pin_memory=True) for _ in range(2)]
        copied = [torch.cuda.Event() for _ in range(2)]
        pending = None                              # (slot, q0, rows) whose copy is in flight
        for i, q0 in enumerate(range(0, nq, chunk)):
            s, n = i % 2, min(chunk, nq - q0)
            main.wait_event(copied[s])              # the copy of chunk i - 2 has left dbuf[s]
            rp = rowptr[q0:q0 + n + 1]
            for t, (a0, csc) in enumerate(tiles):
                outs[t].append(apply_sparse(rp, cols, vals, csc, row_total, rows_out=dbuf[s][:n, a0:a0 + csc.n_ann]))
            side.wait_stream(main)
            with torch.cuda.stream(side):
                hbuf[s][:n].copy_(dbuf[s][:n], non_blocking=True)
                copied[s].record(side)
            if pending is not None:
                _rows_flush(pending, hbuf, copied, rows_sink)
            pending = (s, q0, n)
        _rows_flush(pending, hbuf, copied, rows_sink)
    if not tiles:
        return apply_sparse_tiled(rowptr, cols, vals, keys, mvals, S, 0)
    res = [ApplyResult(*(torch.cat([getattr(r, f) for r in o]) for f in ("top1", "top2", "score1", "score2"))) for o in outs]
    if len(res) == 1:
        return res[0]
    idxs, scs = [], []
    for (a0, _), r in zip(tiles, res):
        i = torch.stack([r.top1.to(torch.int64), r.top2.to(torch.int64)])
        idxs.append(torch.where(i >= 0, i + a0, i))
        scs.append(torch.stack([r.score1, r.score2]))
    return merge_top2(torch.stack(idxs), torch.stack(scs))


def _rows_flush(pending, hbuf, copied, rows_sink) -> None:
    s, q0, n = pending
    copied[s].synchronize()
    rows_sink(q0, hbuf[s][:n].numpy())


# ---------------------------------------------------------------------------
# CSV text on the device (skm_csv.cu): the reference's interchange files, formatted where the data is
# ---------------------------------------------------------------------------
CSV_CELL_MAX = 26                  # a float64 cell as pyarrow prints it (<= 25 bytes) and its separator
CSV_INDEX_COL = "__index_level_0__"


def pyarrow_quote(text: str) -> str:
    """A string cell or header name as pyarrow's CSV writer quotes it."""
    return '"' + str(text).replace('"', '""') + '"'


def labels_device(labels: Sequence[str], device=None) -> Tuple[torch.Tensor, torch.Tensor, np.ndarray]:
    """(UTF-8 bytes uint8, offsets int64 [n + 1]) on the device, and the offsets on the host."""
    dev = _require_cuda(device)
    enc = [str(x).encode("utf-8") for x in labels]
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    if enc:
        np.cumsum([len(b) for b in enc], out=off[1:])
    raw = np.frombuffer(b"".join(enc), dtype=np.uint8)
    return torch.from_numpy(raw.copy()).to(dev), torch.from_numpy(off).to(dev), off


def _csv_measure(fn, rows: int, *args) -> torch.Tensor:
    """Row offsets int64 [rows + 1] of a *_measure entry point (args: everything before d_row_offsets)."""
    dev = _require_cuda()
    row_off = torch.empty(rows + 1, dtype=torch.int64, device=dev)
    ws_bytes = lib().skm_csv_rows_workspace(rows)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(fn(*args, _ptr(row_off), _ptr(ws), ws_bytes, _stream()))
    return row_off


class TextPipe:
    """Chunks of text written on the device into two device buffers, copied to two pinned host buffers and appended to
    a file: the copy and the file write of one chunk run while the next chunk is computed and formatted."""

    def __init__(self, f, capacity: int, device=None):
        dev = _require_cuda(device)
        self.f = f
        self.main = torch.cuda.current_stream(dev)
        self.side = torch.cuda.Stream(dev)
        self.text = [torch.empty(max(int(capacity), 1), dtype=torch.uint8, device=dev) for _ in range(2)]
        self.host = [torch.empty(max(int(capacity), 1), dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        self.nbytes = [torch.zeros(1, dtype=torch.int64, pin_memory=True) for _ in range(2)]
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.copied = [torch.cuda.Event() for _ in range(2)]
        self.i = 0
        self.pending = None

    def slot(self) -> int:
        """The buffer for the next chunk; its previous text has left the device before the main stream writes it."""
        s = self.i % 2
        self.main.wait_event(self.copied[s])
        return s

    def push(self, s: int, row_off: torch.Tensor) -> None:
        """text[s][:row_off[-1]] holds the chunk (written on the main stream).  Flushes the previous chunk first, so
        its copy is not queued behind this chunk's kernels."""
        if self.pending is not None:
            self._flush(self.pending)
        self.side.wait_stream(self.main)
        with torch.cuda.stream(self.side):
            self.nbytes[s].copy_(row_off[-1:], non_blocking=True)
            self.ready[s].record(self.side)
        row_off.record_stream(self.side)        # the allocator keeps it until the side stream's copy has read it
        self.pending = s
        self.i += 1

    def _flush(self, s: int) -> None:
        self.ready[s].synchronize()
        n = int(self.nbytes[s][0])
        with torch.cuda.stream(self.side):
            self.host[s][:n].copy_(self.text[s][:n], non_blocking=True)
            self.copied[s].record(self.side)
        self.copied[s].synchronize()
        self.f.write(memoryview(self.host[s][:n].numpy()))

    def close(self) -> None:
        if self.pending is not None:
            self._flush(self.pending)
            self.pending = None


class AssociationsCSVText:
    """The seq-annotation-scores CSV (apply.smk:295-299, learn.smk:821-849) with its rows formatted on the device
    (skm_csv_assoc_*): byte for byte what sidecar.AssociationsCSVWriter writes through pyarrow.  Passed as the
    rows_sink of apply_sparse_tiled, or filled by write_top2_csv."""

    def __init__(self, path: str, annotations: Sequence[str], labels: Sequence[str], device=None):
        self.A = len(annotations)
        self.Q = len(labels)
        self.labels, self.label_off, off = labels_device(labels, device)
        self.max_label = int(np.diff(off).max()) if len(labels) else 0
        self.f = open(path, "wb")
        self.f.write((",".join(pyarrow_quote(x) for x in list(annotations) + [CSV_INDEX_COL]) + "\n").encode("utf-8"))
        self._pipe = None

    def row_bound(self) -> int:
        """Most bytes a row can take: every cell at its longest, every label byte a quote."""
        return CSV_CELL_MAX * self.A + 2 * self.max_label + 3

    def pipe(self, rows: int) -> TextPipe:
        self._pipe = TextPipe(self.f, rows * self.row_bound(), self.label_off.device)
        return self._pipe

    def format_rows(self, q0: int, block: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
        """Rows q0 .. q0 + len(block) of a float64 device block [n, A] (unit column stride) into out; -> row offsets."""
        n = block.shape[0]
        assert block.dtype == torch.float64 and block.shape[1] == self.A and (n == 0 or block.stride(1) == 1 or self.A <= 1)
        assert out.numel() >= n * self.row_bound() and 0 <= q0 and q0 + n <= self.Q
        lo = self.label_off[q0:q0 + n + 1]
        ld = block.stride(0) if self.A else 0
        row_off = _csv_measure(lib().skm_csv_assoc_measure, n, _ptr(block), n, self.A, ld, _ptr(self.labels), _ptr(lo))
        check(lib().skm_csv_assoc_write(_ptr(block), n, self.A, ld, _ptr(self.labels), _ptr(lo), _ptr(row_off), _ptr(out), _stream()))
        return row_off

    def close(self) -> None:
        if self._pipe is not None:
            self._pipe.close()
            self._pipe = None
        self.f.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def write_top2_csv(w: AssociationsCSVText, r: ApplyResult, chunk_rows: Optional[int] = None) -> None:
    """The top-2-masked association rows of eval_apply without save_associations (learn.smk:831-849) into w: each
    row's two best scores and "nan" elsewhere, formatted on the device straight from the top-2 (skm_csv_top2_*)."""
    nq = r.top1.numel()
    assert nq == w.Q
    if nq == 0:
        return
    chunk = max(1, min(int(chunk_rows) if chunk_rows is not None else ROWS_CHUNK_BYTES // w.row_bound(), nq))
    pipe = w.pipe(chunk)
    t1, t2, s1, s2 = (x.contiguous() for x in (r.top1, r.top2, r.score1, r.score2))
    for q0 in range(0, nq, chunk):
        n = min(chunk, nq - q0)
        lo = w.label_off[q0:q0 + n + 1]
        ptrs = [_ptr(x) + q0 * x.element_size() for x in (t1, t2, s1, s2)]
        row_off = _csv_measure(lib().skm_csv_top2_measure, n, *ptrs, n, w.A, _ptr(w.labels), _ptr(lo))
        s = pipe.slot()
        check(lib().skm_csv_top2_write(*ptrs, n, w.A, _ptr(w.labels), _ptr(lo), _ptr(row_off), _ptr(pipe.text[s]), _stream()))
        pipe.push(s, row_off)
    pipe.close()


CSV_PARSE_BLOCK = 1 << 30          # bytes of a count CSV on the device at a time


def _csv_header(f) -> Tuple[bytes, int]:
    """(the header line's bytes without its '\n', bytes consumed): the first newline outside quotes."""
    head, parity = b"", 0
    while True:
        piece = f.read(1 << 20)
        if not piece:
            return head, len(head)
        a = np.frombuffer(piece, dtype=np.uint8)
        par = (np.cumsum(a == ord('"')) + parity) & 1
        hit = np.flatnonzero((a == ord("\n")) & (par == 0))
        if hit.size:
            cut = int(hit[0])
            f.seek(len(head) + cut + 1)
            return head + piece[:cut], len(head) + cut + 1
        head += piece
        parity = int(par[-1])


def _csv_label(raw: bytes) -> str:
    if len(raw) >= 2 and raw[:1] == b'"' and raw[-1:] == b'"':
        raw = raw[1:-1].replace(b'""', b'"')
    return raw.decode("utf-8")


def parse_counts_csv(path: str, block_bytes: int = CSV_PARSE_BLOCK, device=None):
    """A kmer-counts CSV of either layout (learn.smk:328-357 / :583-594) parsed on the device (skm_csv_parse_*), read
    in blocks of `block_bytes`, each cut at its last row end with the rest carried into the next block.  Header and
    labels are decoded on the host.  -> (labels, kmers, seq_count int64 [R], kmer_count int64 [R], rowptr int64 [R + 1],
    cols int32 (file columns, ascending in a row), vals int64) with the CSR on the device; zeros are left out.
    A cell outside the grammar (empty, [0-9]+, [0-9]+.0*, pyarrow's exponent form of an integer below 2^63) raises
    SkmError naming the line and the column."""
    import csv as _csv
    import io as _io

    dev = _require_cuda(device)
    with open(path, "rb") as f:
        head, consumed = _csv_header(f)
        header = next(_csv.reader(_io.StringIO(head.decode("utf-8")))) if head else []
        if CSV_INDEX_COL not in header:
            raise SkmError(-1, f"{path}: no {CSV_INDEX_COL} column in the header")
        role = np.empty(len(header), dtype=np.int32)
        kmers = []
        for j, name in enumerate(header):
            if name == CSV_INDEX_COL:
                role[j] = -1
            elif name == "Sequence count":
                role[j] = -2
            elif name == "Kmer Count":
                role[j] = -3
            else:
                role[j] = len(kmers)
                kmers.append(name)
        if (role == -2).sum() != 1 or (role == -3).sum() != 1 or (role == -1).sum() != 1:
            raise SkmError(-1, f"{path}: the header needs one each of {CSV_INDEX_COL}, Sequence count and Kmer Count")
        d_role = torch.from_numpy(role).to(dev)
        labels, seqs, kcs, nnzs, colss, valss = [], [], [], [], [], []
        line = 2                                    # line number of the next row
        carry, block, eof = b"", max(int(block_bytes), 1), False
        while not eof or carry:
            piece = f.read(max(block - len(carry), 1)) if not eof else b""
            eof = eof or not piece
            buf = carry + piece
            if eof and buf and not buf.endswith(b"\n"):
                buf += b"\n"
            if not buf:
                break
            n = len(buf)
            text = torch.from_numpy(np.frombuffer(buf, dtype=np.uint8).copy()).to(dev)
            parity = torch.empty(n, dtype=torch.uint8, device=dev)
            ends = torch.empty(n, dtype=torch.int64, device=dev)
            d_n = torch.zeros(1, dtype=torch.int64, device=dev)
            ws_bytes = lib().skm_csv_parse_workspace(n)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            check(lib().skm_csv_parse_rows(_ptr(text), n, _ptr(parity), _ptr(ends), _ptr(d_n), _ptr(ws), ws_bytes, _stream()))
            m = int(d_n.item())
            if m == 0:                              # a row longer than the block: read on with a larger one
                carry, block = buf, 2 * block
                if eof:
                    raise SkmError(-1, f"{path}: line {line}: a quoted field is not closed")
                continue
            ends = ends[:m]
            last_nl = int(ends[-1].item())          # the block is cut after its last row end
            starts = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), ends[:-1] + 1])
            keep = ends > starts                    # blank lines are skipped, like csv.reader
            starts, ends = starts[keep].contiguous(), ends[keep].contiguous()
            R = starts.numel()
            if R:
                nnz = torch.empty(R, dtype=torch.int64, device=dev)
                sq = torch.zeros(R, dtype=torch.int64, device=dev)
                kc = torch.zeros(R, dtype=torch.int64, device=dev)
                ls = torch.zeros(R, dtype=torch.int64, device=dev)
                le = torch.zeros(R, dtype=torch.int64, device=dev)
                err = torch.full((1,), -1, dtype=torch.int64, device=dev)
                check(lib().skm_csv_parse_cells(_ptr(text), _ptr(parity), _ptr(starts), _ptr(ends), R, _ptr(d_role), len(header), None,
                                                _ptr(nnz), _ptr(sq), _ptr(kc), _ptr(ls), _ptr(le), None, None, _ptr(err), _stream()))
                e = int(err.item()) & 0xFFFFFFFFFFFFFFFF
                if e != 0xFFFFFFFFFFFFFFFF:
                    r, fld = e >> 32, e & 0xFFFFFFFF
                    at = line + buf.count(b"\n", 0, int(starts[r].item()))
                    if fld == 0xFFFFFFFF:
                        raise SkmError(-1, f"{path}: line {at}: the row does not have the header's {len(header)} fields")
                    raise SkmError(-1, f"{path}: line {at}, column {header[fld]!r}: the cell is not an integer count")
                off = torch.zeros(R + 1, dtype=torch.int64, device=dev)
                torch.cumsum(nnz, 0, out=off[1:])
                tot = int(off[-1].item())
                cols = torch.empty(max(tot, 1), dtype=torch.int32, device=dev)
                vals = torch.empty(max(tot, 1), dtype=torch.int64, device=dev)
                check(lib().skm_csv_parse_cells(_ptr(text), _ptr(parity), _ptr(starts), _ptr(ends), R, _ptr(d_role), len(header),
                                                _ptr(off), None, None, None, None, None, _ptr(cols), _ptr(vals), _ptr(err), _stream()))
                lsh, leh = ls.cpu().numpy(), le.cpu().numpy()
                labels += [_csv_label(buf[a:b]) for a, b in zip(lsh.tolist(), leh.tolist())]
                seqs.append(sq.cpu().numpy())
                kcs.append(kc.cpu().numpy())
                nnzs.append(nnz)
                colss.append(cols[:tot])
                valss.append(vals[:tot])
            line += buf.count(b"\n", 0, last_nl + 1)
            carry = buf[last_nl + 1:]
            if eof and carry:
                raise SkmError(-1, f"{path}: line {line}: a quoted field is not closed")
    R = len(labels)
    rowptr = torch.zeros(R + 1, dtype=torch.int64, device=dev)
    if R:
        torch.cumsum(torch.cat(nnzs), 0, out=rowptr[1:])
    cols = torch.cat(colss) if colss else torch.zeros(0, dtype=torch.int32, device=dev)
    vals = torch.cat(valss) if valss else torch.zeros(0, dtype=torch.int64, device=dev)
    cat = lambda xs: np.concatenate(xs) if xs else np.zeros(0, dtype=np.int64)
    return labels, kmers, cat(seqs), cat(kcs), rowptr, cols, vals


CSV_LEARN, CSV_TOTAL = 0, 1        # count-file layouts: learn.smk:328-357 (pandas) and :583-594 (pyarrow)


def write_counts_csv_rows(f, rowptr: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, K: int, seq_count: torch.Tensor,
                          kmer_count: torch.Tensor, labels: Sequence[str], layout: int) -> None:
    """Rows of a kmer-counts CSV from device CSR over the file's K k-mer columns (skm_csv_counts_*), appended to the
    open binary file f.  labels: written verbatim with CSV_LEARN (escape them first), quoted with CSV_TOTAL."""
    dev = rowptr.device
    R = rowptr.numel() - 1
    if R == 0:
        return
    lab, lab_off, _ = labels_device(labels, dev)
    row_off = _csv_measure(lib().skm_csv_counts_measure, R, _ptr(rowptr), _ptr(vals), R, int(K), _ptr(seq_count), _ptr(kmer_count),
                           _ptr(lab), _ptr(lab_off), int(layout))
    off = row_off.cpu().numpy()
    # chunks of whole rows of about ROWS_CHUNK_BYTES of text (a longer row is a chunk of its own)
    cuts = [0]
    while cuts[-1] < R:
        r0 = cuts[-1]
        r1 = int(np.searchsorted(off, off[r0] + ROWS_CHUNK_BYTES, side="right")) - 1
        cuts.append(min(max(r1, r0 + 1), R))
    cap = max(int(off[b] - off[a]) for a, b in zip(cuts[:-1], cuts[1:]))
    pipe = TextPipe(f, cap, dev)
    for r0, r1 in zip(cuts[:-1], cuts[1:]):
        n = r1 - r0
        s = pipe.slot()
        check(lib().skm_csv_counts_write(_ptr(rowptr) + 8 * r0, _ptr(cols), _ptr(vals), n, int(K), _ptr(seq_count) + 8 * r0,
                                         _ptr(kmer_count) + 8 * r0, _ptr(lab), _ptr(lab_off) + 8 * r0, int(layout),
                                         _ptr(row_off) + 8 * r0, _ptr(pipe.text[s]), _stream()))
        pipe.push(s, row_off[r0:r1 + 1] - row_off[r0])
    pipe.close()


# ---------------------------------------------------------------------------
# wide path: code spaces beyond the table limit (nsym^k > 2^27, up to 2^64 - 1) — sort-based
# ---------------------------------------------------------------------------
WIDE_MAX_CHUNK_RES = (1 << 30) - 16


@dataclass
class WideBasis:
    """Basis over a code space too large for tables: codes in first-occurrence order plus the
    ascending code list with the column of each entry (binary-search lookup)."""
    alphabet: str
    k: int
    symbols: str
    codes: torch.Tensor             # int64 (uint64 pattern) [K], first-occurrence order
    counts: Optional[torch.Tensor]  # int64 [K]
    sorted_codes: torch.Tensor      # int64 (uint64 pattern) [K], ascending (unsigned)
    col_of_sorted: torch.Tensor     # int32 [K]
    K: int

    def codes_host(self) -> np.ndarray:
        return self.codes.cpu().numpy().view(np.uint64)

    def kmers(self) -> np.ndarray:
        return decode_kmers(self.codes_host(), self.symbols, self.k)


def basis_table_local(batch: SequenceBatch, alphabet: AlphabetT, k: int, res_base: int = 0,
                      max_chunk_res: int = WIDE_MAX_CHUNK_RES) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, bool]:
    """(codes, counts, first) of a shard: distinct window codes sorted by code, their occurrence counts and
    the global position of their first occurrence.  Returns a 4th item: True when the table is one merged
    list (a single chunk), False when it is the concatenation of several chunks' tables."""
    tab = alphabet_tables(alphabet, batch.device)
    dev = batch.device
    parts = []
    for lo, hi in _chunks_by_residues(batch.offsets_host, max_chunk_res):
        sub = batch if (lo == 0 and hi == batch.n) else _sub_batch(batch, lo, hi)
        shift = 0 if sub is batch else (int(batch.offsets_host[lo]) & ~15)
        n_cap = max(sub.nres, 1)
        ws_bytes = lib().skm_basis_sorted_local_workspace(sub.nres)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        codes = torch.empty(n_cap, dtype=torch.int64, device=dev)
        counts = torch.empty(n_cap, dtype=torch.int64, device=dev)
        first = torch.empty(n_cap, dtype=torch.int64, device=dev)
        dn = torch.zeros(1, dtype=torch.int64, device=dev)
        check(lib().skm_basis_sorted_local(_ptr(sub.residues), sub.nres, _ptr(sub.offsets), sub.n, _ptr(tab.lut), tab.nsym, int(k),
                                           int(res_base) + shift, _ptr(codes), _ptr(counts), _ptr(first), _ptr(dn), _ptr(ws),
                                           ws_bytes, _stream()))
        m = int(dn.item())
        parts.append((codes[:m].clone(), counts[:m].clone(), first[:m].clone()))
        del ws, codes, counts, first
    if not parts:
        z = torch.zeros(0, dtype=torch.int64, device=dev)
        return z, z.clone(), z.clone(), True
    if len(parts) == 1:
        return parts[0] + (True,)
    return (torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts]), torch.cat([p[2] for p in parts]), False)


def basis_table_finalize(alphabet: AlphabetT, k: int, codes: torch.Tensor, counts: torch.Tensor, first: torch.Tensor,
                         merged: bool, min_filter: int = 0, first_bound: int = 0) -> WideBasis:
    """Tables of one or more shards -> the basis in the reference's order (kmerize.smk:89-104).
    first_bound: exclusive upper bound of the first positions (total residues of all shards), 0 = unknown."""
    dev = _require_cuda(codes.device)
    tab = alphabet_tables(alphabet, dev)
    n = codes.numel()
    codes, counts, first = codes.contiguous(), counts.contiguous(), first.contiguous()
    ws_bytes = lib().skm_basis_sorted_finalize_workspace(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    cap = max(n, 1)
    basis = torch.empty(cap, dtype=torch.int64, device=dev)
    bcnt = torch.empty(cap, dtype=torch.int64, device=dev)
    scodes = torch.empty(cap, dtype=torch.int64, device=dev)
    scol = torch.empty(cap, dtype=torch.int32, device=dev)
    dK = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().skm_basis_sorted_finalize(_ptr(codes), _ptr(counts), _ptr(first), n, 1 if merged else 0, int(min_filter), int(first_bound),
                                          _ptr(basis), _ptr(bcnt), _ptr(scodes), _ptr(scol), _ptr(dK), _ptr(ws), ws_bytes, _stream()))
    K = int(dK.item())
    return WideBasis(tab.name, int(k), tab.symbols, basis[:K].clone(), bcnt[:K].clone(), scodes[:K].clone(), scol[:K].clone(), K)


def build_basis_wide(batch: SequenceBatch, alphabet: AlphabetT, k: int, min_filter: int = 0) -> WideBasis:
    """Pass 1 of the vectorize rule (kmerize.smk:89-104) for any nsym^k <= 2^64 - 1: sort-based."""
    codes, counts, first, merged = basis_table_local(batch, alphabet, k, 0)
    return basis_table_finalize(alphabet, k, codes, counts, first, merged, min_filter, first_bound=batch.nres + 16)


def wide_basis_from_codes(codes: np.ndarray, alphabet: AlphabetT, k: int, device=None) -> WideBasis:
    """Basis whose column j holds code codes[j] (uint64, distinct): a supplied / learned k-mer list."""
    dev = _require_cuda(device)
    tab = alphabet_tables(alphabet, dev)
    codes = np.ascontiguousarray(codes, dtype=np.uint64)
    order = np.argsort(codes, kind="stable")
    d_codes = torch.from_numpy(codes.view(np.int64)).to(dev)
    return WideBasis(tab.name, int(k), tab.symbols, d_codes, None, torch.from_numpy(codes[order].view(np.int64)).to(dev),
                     torch.from_numpy(order.astype(np.int32)).to(dev), len(codes))


def codes_to_columns(codes: torch.Tensor, basis: WideBasis) -> torch.Tensor:
    """Basis column of every code (int32, -1 = not in the basis)."""
    dev = _require_cuda(codes.device)
    codes = codes.contiguous()
    out = torch.empty(codes.numel(), dtype=torch.int32, device=dev)
    check(lib().skm_codes_to_columns(_ptr(codes), codes.numel(), _ptr(basis.sorted_codes), _ptr(basis.col_of_sorted), basis.K,
                                     _ptr(out), _stream()))
    return out


def count_csr_wide(batch: SequenceBatch, alphabet: AlphabetT, k: int, basis: Optional[WideBasis] = None,
                   max_chunk_res: int = WIDE_MAX_CHUNK_RES, method: str = "warp"):
    """Per-sequence distinct k-mers and their counts for any nsym^k <= 2^64 - 1.
    Returns (rowptr int64 [N+1], codes int64 (uint64 pattern) [nnz], cols int32 [nnz] or None, vals int32 [nnz]);
    a row's entries are ordered by code; with a basis, entries outside it are dropped and cols holds columns."""
    tab = alphabet_tables(alphabet, batch.device)
    dev = batch.device
    if basis is not None and basis.K == 0:           # nothing can match an empty basis
        return (torch.zeros(batch.n + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int64, device=dev),
                torch.zeros(0, dtype=torch.int32, device=dev), torch.zeros(0, dtype=torch.int32, device=dev))
    b_codes = None if basis is None else _ptr(basis.sorted_codes)
    b_cols = None if basis is None else _ptr(basis.col_of_sorted)
    b_K = 0 if basis is None else basis.K

    def count(sub: SequenceBatch):
        cap = max(sub.nres, 1)
        rowptr = torch.empty(sub.n + 1, dtype=torch.int64, device=dev)
        codes = torch.empty(cap, dtype=torch.int64, device=dev)
        cols = torch.empty(cap, dtype=torch.int32, device=dev) if basis is not None else None
        vals = torch.empty(cap, dtype=torch.int32, device=dev)
        if method == "segsort":          # the first implementation (window keys in HBM + cub::DeviceSegmentedSort), a cross-check
            ws_bytes = lib().skm_count_csr_wide_workspace(sub.nres, sub.n)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            check(lib().skm_count_csr_wide(_ptr(sub.residues), sub.nres, _ptr(sub.offsets), sub.n, _ptr(tab.lut), tab.nsym, int(k),
                                           b_codes, b_cols, b_K, _ptr(rowptr), _ptr(codes), _ptr(cols), _ptr(vals), _ptr(ws), ws_bytes, _stream()))
        else:                            # a warp sorts one sequence's keys in shared memory
            max_len = int(np.diff(sub.offsets_host).max()) if sub.n else 0
            ws_bytes = lib().skm_count_csr_sorted_workspace(sub.nres, sub.n, max_len, 64)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            check(lib().skm_count_csr_sorted(_ptr(sub.residues), sub.nres, _ptr(sub.offsets), sub.n, _ptr(tab.lut), tab.nsym, int(k), 64,
                                             None, 0, b_codes, b_cols, b_K, max_len, _ptr(rowptr), _ptr(codes), _ptr(cols), _ptr(vals),
                                             _ptr(ws), ws_bytes, _stream()))
        nnz = int(rowptr[-1].item()) if sub.n else 0
        return rowptr, codes[:nnz].clone(), (cols[:nnz].clone() if cols is not None else None), vals[:nnz].clone()

    return _csr_by_chunks(batch, max_chunk_res, (torch.int64, torch.int32 if basis is not None else None, torch.int32), count)


def _csr_by_chunks(batch: SequenceBatch, max_chunk_res: int, dtypes, count):
    """CSR of `batch` from `count(sub) -> (rowptr, *entry arrays)` run on every chunk of at most `max_chunk_res`
    residues: the chunks' rowptrs are rebased onto one running nnz and their entry arrays concatenated (an array that
    is None stays None).  `dtypes` are the entry arrays' dtypes (None: the array is None) for a batch with no chunk."""
    dev = batch.device
    rowptrs, parts, base = [], [], 0
    for lo, hi in _chunks_by_residues(batch.offsets_host, max_chunk_res):
        sub = batch if (lo == 0 and hi == batch.n) else _sub_batch(batch, lo, hi)
        rowptr, *arrays = count(sub)
        rowptrs.append(rowptr[(1 if rowptrs else 0):] + base)
        parts.append(arrays)
        base += int(arrays[-1].numel())
    if not rowptrs:
        return (torch.zeros(1, dtype=torch.int64, device=dev),
                *(None if dt is None else torch.zeros(0, dtype=dt, device=dev) for dt in dtypes))
    cat = (lambda xs: xs[0] if len(xs) == 1 else torch.cat(xs))
    return (cat(rowptrs), *(None if xs[0] is None else cat(list(xs)) for xs in zip(*parts)))


def learn_wide(batch: SequenceBatch, alphabet: AlphabetT, k: int, basis: WideBasis, ann_id: torch.Tensor, n_ann: int,
               max_chunk_res: int = WIDE_MAX_CHUNK_RES) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """learn_sparse_with_totals for any nsym^k <= 2^64 - 1, with the matrix keyed by BASIS COLUMN:
    -> (keys int64 [nnz] sorted, key = ann * K + col; vals int64 [nnz]; totals int64 [K]: occurrences of every basis
    column over ALL sequences, learn.smk:380).  Windows outside the basis count nowhere.  Sequences with ann_id
    outside [0, n_ann) go to a rest row that only feeds the Totals (skm_learn_wide)."""
    tab = alphabet_tables(alphabet, batch.device)
    dev = batch.device
    ann_id = ann_id.to(device=dev, dtype=torch.int32).contiguous()
    assert ann_id.numel() == batch.n
    K, n_ann = int(basis.K), int(n_ann)
    if (n_ann + 2) * K >= 2 ** 63:
        raise SkmError(-3, f"learn_wide: (n_ann + 2) * K = {(n_ann + 2) * K} does not fit 63 bits")
    parts_k, parts_v = [], []
    for lo, hi in _chunks_by_residues(batch.offsets_host, max_chunk_res):
        sub = batch if (lo == 0 and hi == batch.n) else _sub_batch(batch, lo, hi)
        ws_bytes = lib().skm_learn_wide_workspace(sub.nres)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        ok = torch.empty(max(sub.nres, 1), dtype=torch.int64, device=dev)
        ov = torch.empty(max(sub.nres, 1), dtype=torch.int64, device=dev)
        dn = torch.zeros(1, dtype=torch.int64, device=dev)
        check(lib().skm_learn_wide(_ptr(sub.residues), sub.nres, _ptr(sub.offsets), sub.n, _ptr(tab.lut), tab.nsym, int(k),
                                   _ptr(ann_id[lo:hi]), n_ann, _ptr(basis.sorted_codes), _ptr(basis.col_of_sorted), K,
                                   _ptr(ok), _ptr(ov), _ptr(dn), _ptr(ws), ws_bytes, _stream()))
        m = int(dn.item())
        parts_k.append(ok[:m].clone())
        parts_v.append(ov[:m].clone())
        del ws, ok, ov
    if not parts_k:
        keys = vals = torch.zeros(0, dtype=torch.int64, device=dev)
    elif len(parts_k) == 1:
        keys, vals = parts_k[0], parts_v[0]
    else:
        keys, vals = coo_merge_runs(torch.cat(parts_k), torch.cat(parts_v), [p.numel() for p in parts_k])
    totals = torch.zeros(max(K, 1), dtype=torch.int64, device=dev)
    if keys.numel():
        check(lib().skm_coo_colsum(_ptr(keys), _ptr(vals), keys.numel(), K, _ptr(totals), _stream()))
    m = int(torch.searchsorted(keys, torch.tensor([n_ann * K], dtype=torch.int64, device=dev)).item()) if keys.numel() else 0
    return keys[:m], vals[:m], totals[:K]


def query_csr_wide(batch: SequenceBatch, alphabet: AlphabetT, k: int, basis: WideBasis,
                   restrict: Optional[WideBasis] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Queries for apply against a matrix keyed by the columns of `basis`: (rowptr int64 [N+1], cols int32, vals int32)
    over EVERY valid window (the query norm runs over all of them, apply.smk:268-276).  An entry the basis does not hold
    gets the empty column K: it adds to the norm and to no dot.  restrict: keep only the codes this basis holds (the
    query file's own kmerlist, apply.smk:262-289)."""
    rowptr, codes, _, vals = count_csr_wide(batch, alphabet, k)
    if restrict is not None:
        keep = codes_to_columns(codes, restrict) >= 0
        csum = torch.zeros(keep.numel() + 1, dtype=torch.int64, device=codes.device)
        torch.cumsum(keep, 0, out=csum[1:])
        rowptr, codes, vals = csum[rowptr], codes[keep].contiguous(), vals[keep].contiguous()
    cols = codes_to_columns(codes, basis)
    cols = torch.where(cols < 0, torch.full_like(cols, basis.K), cols)
    return rowptr, cols, vals


def apply_wide(rowptr: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, keys: torch.Tensor, mvals: torch.Tensor, K: int,
               n_ann: int, tile: Optional[int] = None, rows_sink: Optional[Callable[[int, np.ndarray], None]] = None,
               chunk_rows: Optional[int] = None) -> ApplyResult:
    """apply_sparse_tiled for a matrix keyed by basis column (learn_wide, key = ann * K + col) and queries from
    query_csr_wide: the matrix is re-keyed to the stride K + 1, whose last column is the empty one."""
    return apply_sparse_tiled(rowptr, cols, vals, keys + keys // K if K else keys, mvals, K + 1, n_ann, tile, rows_sink, chunk_rows)


def build_basis_wide_distributed(batch: SequenceBatch, alphabet, k: int, min_filter: int = 0,
                                 res_base: Optional[int] = None) -> WideBasis:
    """The wide basis of the CONCATENATION of all ranks' shards, identical on every rank: local tables with
    global first positions, all_gather of the tables, one finalisation (sort by code, sum / min, order)."""
    from . import dist as D

    total = 0
    if res_base is None:
        res_base, total = D.exclusive_prefix(batch.nres, batch.device)
    codes, counts, first, merged = basis_table_local(batch, alphabet, k, res_base)
    _, w = D.world()
    if w > 1:
        codes, counts, first = D.allgather_tables(codes, counts, first)
        merged = False
    return basis_table_finalize(alphabet, k, codes, counts, first, merged, min_filter, first_bound=(total + 16 * w) if total else 0)


DENSE_ROW_MAX_K = 4096          # widest basis whose per-sequence counts are kept as dense rows by vectorize()


@dataclass
class Vectorized:
    """Result of vectorize(): the basis and the per-sequence counts in the layout the basis size calls for."""
    path: str                               # "dense" | "csr" | "wide"
    basis: "Basis | WideBasis"
    counts: Optional[torch.Tensor] = None   # dense: int32 [N, K]
    rowptr: Optional[torch.Tensor] = None   # csr / wide: int64 [N+1]
    cols: Optional[torch.Tensor] = None     #             int32 [nnz] basis column of every entry
    vals: Optional[torch.Tensor] = None     #             int32 [nnz]
    codes: Optional[torch.Tensor] = None    # wide only: int64 (uint64 pattern) [nnz]

    @property
    def K(self) -> int:
        return self.basis.K

    @property
    def nnz(self) -> int:
        return int(self.vals.numel()) if self.vals is not None else int((self.counts != 0).sum().item())


def vectorize(batch: SequenceBatch, alphabet: AlphabetT, k: int, min_filter: int = 0,
              dense_max_K: int = DENSE_ROW_MAX_K) -> Vectorized:
    """Both passes of the vectorize rule (kmerize.smk:85-120) for ANY alphabet / k with nsym^k <= 2^64 - 1:
    first-occurrence basis + per-sequence counts.  Code spaces up to 2^27 use the table kernels (dense rows while
    the basis has at most `dense_max_K` columns, CSR beyond); larger ones the sort-based wide path."""
    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    if S <= _native.SKM_DENSE_MAX_SPACE:
        basis = build_basis(batch, alphabet, k, min_filter)
        if basis.K <= dense_max_K:
            return Vectorized("dense", basis, counts=count_dense(batch, alphabet, k, basis))
        rowptr, cols, vals = _csr_by_chunks(batch, (1 << 30) - 16, (torch.int32, torch.int32),
                                            lambda sub: count_csr(sub, alphabet, k, basis))
        return Vectorized("csr", basis, rowptr=rowptr, cols=cols, vals=vals)
    basis = build_basis_wide(batch, alphabet, k, min_filter)
    rowptr, codes, cols, vals = count_csr_wide(batch, alphabet, k, basis)
    return Vectorized("wide", basis, rowptr=rowptr, cols=cols, vals=vals, codes=codes)


# ---------------------------------------------------------------------------
# multi-GPU compositions (one process per GPU; collectives in dist.py)
# ---------------------------------------------------------------------------
def build_basis_distributed(batch: SequenceBatch, alphabet, k: int, min_filter: int = 0, res_base: Optional[int] = None) -> Basis:
    """The basis of the CONCATENATION of all ranks' shards (rank order), identical on every rank:
    local tables with global first positions, all_reduce(SUM / MIN), local finalisation."""
    from . import dist as D

    tab = alphabet_tables(alphabet, batch.device)
    S = code_space(tab.nsym, k)
    if S > _native.SKM_DENSE_MAX_SPACE:
        raise SkmError(-3, f"code space {tab.nsym}^{k} exceeds the table limit 2^27")
    if res_base is None:
        res_base, _ = D.exclusive_prefix(batch.nres, batch.device)
    count, first = basis_tables(S, batch.device)
    basis_accumulate(batch, alphabet, k, count, first, res_base)
    D.allreduce_basis_tables(count, first)
    return basis_finalize(alphabet, k, count, first, min_filter)


def learn_dense_distributed(batch: SequenceBatch, alphabet, k: int, basis: Optional[Basis], ann_id: torch.Tensor,
                            n_ann: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """learn_dense on the local shard followed by the NCCL sum over ranks (the reference's
    serial Merge step, learn.smk:467-494); every rank ends with the full matrix."""
    from . import dist as D

    M, totals = learn_dense(batch, alphabet, k, basis, ann_id, n_ann)
    D.allreduce_sum_(M, totals)
    return M, totals


def apply_dense_annotation_sharded(Q: torch.Tensor, M_local: torch.Tensor, ann_base: int,
                                   qnorm2: Optional[torch.Tensor] = None) -> ApplyResult:
    """Every rank scores all queries against ITS rows of the annotation matrix; the per-shard
    top-2 are all-gathered and merged (identical result on every rank)."""
    from . import dist as D

    r = apply_dense(Q, M_local, qnorm2=qnorm2)
    idx, sc = D.allgather_top2(r.top1, r.top2, r.score1, r.score2, ann_base)
    return merge_top2(idx, sc)


def peer_exchange_enabled(t: torch.Tensor) -> bool:
    """The sparse-learn fan-in goes through NVLink peer memory when the ranks are CUDA processes of one node (NCCL
    backend); SKM_EXCHANGE=nccl selects the all_to_all_single baseline."""
    import torch.distributed as dist
    from . import dist as D
    return (t.is_cuda and dist.is_initialized() and dist.get_backend() == "nccl" and dist.get_world_size() <= 16
            and os.environ.get("SKM_EXCHANGE", "peer") != "nccl" and not D.peer_buffers().disabled)


def exchange_coo_by_annotation(keys: torch.Tensor, vals: torch.Tensor, S: int, n_ann: int,
                               balance: bool = True) -> Tuple[torch.Tensor, torch.Tensor, Tuple[int, int]]:
    """Multi-GPU fan-in of sparse learn: annotations are split into W contiguous ranges, rank r ends up with the merged
    rows [a_lo, a_hi) of the matrix — the annotation sharding apply uses.  Returns (keys, vals, (a_lo, a_hi)).

    balance=True cuts the ranges by ENTRY count (one all_reduce of the per-annotation entry histogram): family sizes
    are Zipf-distributed, so equal id ranges would send ~90 % of all entries to rank 0.  Cuts stay at annotation
    boundaries (a rank owns whole rows), so a single annotation larger than 1/W of the matrix still limits the balance."""
    from . import dist as D

    rank, w = D.world()
    if w == 1:
        return keys, vals, (0, n_ann)
    if balance:
        ann_bounds = D.balanced_annotation_bounds(keys, S, n_ann)
    else:
        ann_bounds = [n_ann * r // w for r in range(w)] + [n_ann]
    key_bounds = [a * int(S) for a in ann_bounds]
    count_bits = 64 - max(int(n_ann) * int(S) - 1, 1).bit_length()
    if peer_exchange_enabled(keys) and count_bits >= 16:
        # fused pack + all_to_all over NVLink peer memory (skm_coo_pack_push); the histogram all_reduce above (or the
        # barrier below) is the fence that says no rank still reads its receive buffer
        if not balance:
            D.barrier()
        pushed = D.push_coo_by_key_range(keys, vals, key_bounds, count_bits)
        if pushed is not None:
            ptr, runs, flag = pushed
            k3, v3, dn = coo_merge_runs_packed(ptr, runs, count_bits, keys.device)
            m, bad = torch.cat([dn, flag.to(torch.int64)]).tolist()
            if not bad:
                return k3[:m].clone(), v3[:m].clone(), (ann_bounds[rank], ann_bounds[rank + 1])
        # a count beyond count_bits somewhere: the unpacked NCCL exchange below
    k2, v2, runs = D.alltoall_coo_by_key_range(keys, vals, key_bounds, return_runs=True)
    k3, v3 = coo_merge_runs(k2, v2, runs)           # W sorted runs, one per sender: merge tree + reduce-by-key
    return k3, v3, (ann_bounds[rank], ann_bounds[rank + 1])
