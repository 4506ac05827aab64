"""dist: one process per GPU, ``torch.distributed`` (NCCL over NVLink; gloo in CPU tests).

The reference fans out one Snakemake job per input FASTA (learn.smk:105-106,
apply.smk:107-111) and fans in with one serial pandas merge (learn.smk:467-494).
Here sequences are sharded by contiguous ranges balanced by residue count; the path
has exactly three exchange steps, each a plain collective on integer / top-2 buffers:

  basis   (kmerize.smk:89-104)   all_reduce(SUM) of per-code counts + all_reduce(MIN)
                                 of first positions (global residue positions)
                                 (code spaces without tables: all_gather of the per-rank
                                 (code, count, first) tables, merged by one sort)
  learn   (learn.smk:467-494)    all_reduce(SUM) of the dense count matrix / totals
  apply   (apply.smk:312-335)    when the annotation matrix is row-(annotation-)sharded:
                                 all_gather of per-shard (top1, top2, score1, score2) and a
                                 2-way merge — top-2, not top-1: delta needs the runner-up
  evaluate (learn.smk:1052-1110) training rows sharded, matrix replicated: all_reduce(SUM) of
                                 the True / False crosstabs, all_reduce(MIN) of the zero-bin key

encode / count / apply-with-replicated-M need no collective (weak scaling).
Every function works on whatever device the tensors live on, so the collective
plumbing is exercised on CPU with gloo (tests/test_dist_gloo.py); the compute around
it is CUDA-only as everywhere else.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

INT64_MAX = np.iinfo(np.int64).max


def init(backend: Optional[str] = None, device: Optional[torch.device] = None) -> Tuple[int, int]:
    """Initialise the default process group from RANK / WORLD_SIZE / MASTER_* (torchrun). Returns (rank, world)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1 and not dist.is_initialized():
        backend = backend or ("nccl" if torch.cuda.is_available() else "gloo")
        kw = {"device_id": device} if (backend == "nccl" and device is not None) else {}
        dist.init_process_group(backend, rank=rank, world_size=world, **kw)
    return rank, world


def bind_to_local_cpus(device_index: int) -> Optional[List[int]]:
    """Pin this process to the CPUs NVML reports as local to its GPU (same NUMA node / PCIe root), so that the pinned host
    buffers it allocates afterwards — first touch — and the threads that fill them sit next to the GPU's PCIe link.
    With one process per GPU on a two-socket host this keeps half of the ranks from copying across the socket
    interconnect.  Returns the CPU list, or None when NVML or the affinity call is not available (nothing is changed)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        p = torch.cuda.get_device_properties(device_index)
        bus = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus)
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        local = {i for i in range(ncpu) if (int(mask[i // 64]) >> (i % 64)) & 1}
        use = sorted(local & os.sched_getaffinity(0))
        if not use:
            return None
        os.sched_setaffinity(0, use)
        return use
    except Exception:                                    # noqa: BLE001 — NVML missing, containers without the call
        return None


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_bounds(offsets: np.ndarray, parts: int) -> List[Tuple[int, int]]:
    """Cut N sequences into `parts` contiguous ranges with ~equal residue counts, only at
    sequence boundaries (SURVEY 8e).  Ranges may be empty; together they cover [0, N)."""
    offsets = np.asarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    if n <= 0:
        return [(0, 0)] * parts
    span = offsets[-1] - offsets[0]
    targets = offsets[0] + (span * np.arange(1, parts, dtype=np.float64) / parts)
    cuts = np.searchsorted(offsets[:-1], targets, side="left")
    cuts = np.concatenate([[0], np.clip(cuts, 0, n), [n]]).astype(np.int64)
    cuts = np.maximum.accumulate(cuts)
    return [(int(cuts[i]), int(cuts[i + 1])) for i in range(parts)]


def allreduce_basis_tables(count: torch.Tensor, first: torch.Tensor) -> None:
    """Merge per-rank (count, first) tables of skm_basis_accumulate in place.

    `first` holds uint64 bit patterns in int64 with all-ones (-1) = "never seen"; positions
    are < 2^63, so mapping -1 to INT64_MAX makes a signed MIN correct."""
    if world()[1] == 1:
        return
    dist.all_reduce(count, op=dist.ReduceOp.SUM)
    f = torch.where(first < 0, torch.full_like(first, INT64_MAX), first)
    dist.all_reduce(f, op=dist.ReduceOp.MIN)
    first.copy_(torch.where(f == INT64_MAX, torch.full_like(f, -1), f))


def allreduce_sum_(*tensors: torch.Tensor) -> None:
    """Learn-mode fan-in: integer sums of the per-rank count matrices / totals / sequence counts."""
    if world()[1] == 1:
        return
    for t in tensors:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)


def allreduce_confidence_tables(hist_true: torch.Tensor, hist_false: torch.Tensor, zero_key: torch.Tensor) -> None:
    """Evaluate fan-in over ranks that scored disjoint rows of one file, in place: the int64 [A, 101] crosstabs are
    summed; zero_key (int64 [1], 2 * global row + exact-tie flag of a rank's first Known & True row in the zero bin,
    INT64_MAX for none) becomes the minimum, i.e. the lowest such row of the file."""
    if world()[1] == 1:
        return
    allreduce_sum_(hist_true, hist_false)
    dist.all_reduce(zero_key, op=dist.ReduceOp.MIN)


def exclusive_prefix(value: int, device=None) -> Tuple[int, int]:
    """(sum of `value` over lower ranks, sum over all ranks): global residue / sequence bases."""
    rank, w = world()
    if w == 1:
        return 0, int(value)
    t = torch.zeros(w, dtype=torch.int64, device=device)
    t[rank] = int(value)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    v = t.cpu().numpy()
    return int(v[:rank].sum()), int(v.sum())


def allgather_top2(top1: torch.Tensor, top2: torch.Tensor, s1: torch.Tensor, s2: torch.Tensor,
                   ann_base: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Annotation-sharded apply: every rank scored ALL queries against its slice of annotations.
    Returns (idx [W, 2, Q] int64 global annotation indices or -1, score [W, 2, Q] float64)
    stacked over ranks, ready for the 2-way merge (engine.merge_top2)."""
    rank, w = world()
    idx = torch.stack([top1.to(torch.int64), top2.to(torch.int64)])
    idx = torch.where(idx >= 0, idx + int(ann_base), idx)
    sc = torch.stack([s1.to(torch.float64), s2.to(torch.float64)])
    if w == 1:
        return idx.unsqueeze(0), sc.unsqueeze(0)
    all_idx = [torch.empty_like(idx) for _ in range(w)]
    all_sc = [torch.empty_like(sc) for _ in range(w)]
    dist.all_gather(all_idx, idx.contiguous())
    dist.all_gather(all_sc, sc.contiguous())
    return torch.stack(all_idx), torch.stack(all_sc)


def gather_rows(local: torch.Tensor, dst: int = 0) -> Optional[torch.Tensor]:
    """Concatenate per-rank row blocks (different lengths) on `dst` in rank order (query-sharded outputs)."""
    rank, w = world()
    if w == 1:
        return local
    n = torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device)
    sizes = [torch.zeros_like(n) for _ in range(w)]
    dist.all_gather(sizes, n)
    sizes = [int(s.item()) for s in sizes]
    m = max(sizes)
    pad = torch.zeros((m,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    parts = [torch.empty_like(pad) for _ in range(w)]
    dist.all_gather(parts, pad)
    if rank != dst:
        return None
    return torch.cat([p[:s] for p, s in zip(parts, sizes)])


def allgather_tables(*columns: torch.Tensor) -> Tuple[torch.Tensor, ...]:
    """Wide-basis fan-in (kmerize.smk:89-104 over code spaces without tables): every rank contributes the
    columns (codes, counts, first) of its local table — equal lengths on one rank, different lengths across
    ranks — and receives the concatenation over ranks in rank order."""
    rank, w = world()
    if w == 1:
        return tuple(columns)
    dev = columns[0].device
    n = torch.tensor([columns[0].numel()], dtype=torch.int64, device=dev)
    sizes = [torch.zeros_like(n) for _ in range(w)]
    dist.all_gather(sizes, n)
    sizes = [int(x.item()) for x in sizes]
    m = max(sizes + [1])
    out = []
    for c in columns:
        pad = torch.zeros(m, dtype=c.dtype, device=dev)
        pad[:c.numel()] = c
        parts = [torch.empty_like(pad) for _ in range(w)]
        dist.all_gather(parts, pad)
        out.append(torch.cat([q[:sz] for q, sz in zip(parts, sizes)]))
    return tuple(out)


def alltoall_coo_by_key_range(keys: torch.Tensor, vals: torch.Tensor, key_bounds: Sequence[int], return_runs: bool = False):
    """Sparse learn fan-in (learn.smk:467-494 for COO matrices): rank r receives from every rank the
    entries whose key lies in [key_bounds[r], key_bounds[r+1]).  `keys` must be sorted (int64 holding
    non-negative keys), so each destination is one contiguous run.  The received runs still have to be
    merged (engine.coo_merge / coo_merge_runs).  key_bounds has world+1 entries.  return_runs: also return the
    sizes of the W received runs (each sorted), in rank order."""
    rank, w = world()
    if w == 1:
        return (keys, vals, [keys.numel()]) if return_runs else (keys, vals)
    b = torch.tensor(list(key_bounds), dtype=torch.int64, device=keys.device)
    cut = torch.searchsorted(keys, b)
    send = (cut[1:] - cut[:-1]).contiguous()
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv, send)
    send_l, recv_l = send.tolist(), recv.tolist()
    lo, hi = int(cut[0].item()), int(cut[-1].item())
    out_k = torch.empty(sum(recv_l), dtype=keys.dtype, device=keys.device)
    out_v = torch.empty(sum(recv_l), dtype=vals.dtype, device=vals.device)
    dist.all_to_all_single(out_k, keys[lo:hi].contiguous(), recv_l, send_l)
    dist.all_to_all_single(out_v, vals[lo:hi].contiguous(), recv_l, send_l)
    return (out_k, out_v, recv_l) if return_runs else (out_k, out_v)


def push_plan(count_matrix: np.ndarray, rank: int) -> Tuple[np.ndarray, np.ndarray, int]:
    """Layout of the peer-memory exchange.  count_matrix[s, r] = entries rank s sends to rank r (identical on every
    rank).  Rank r's receive buffer holds the runs of the senders in rank order — the layout all_to_all_single gives —
    so sender s starts at sum(count_matrix[:s, r]).  Returns (dst_off [W]: where THIS rank's run starts in every
    receiver's buffer, runs [W]: sizes of the runs this rank receives, words: the largest receive buffer of any rank)."""
    m = np.asarray(count_matrix, dtype=np.int64)
    dst_off = m[:rank].sum(axis=0)
    return dst_off.astype(np.int64), m[:, rank].copy(), int(m.sum(axis=0).max()) if m.size else 0


class PeerBuffers:
    """One receive buffer of 64-bit words per rank, mapped into every rank of the node through CUDA IPC
    (skm_peer_alloc / skm_peer_open): the target of skm_coo_pack_push.  Grown collectively on demand."""

    def __init__(self):
        self.words = 0
        self.own = None                  # int: device pointer of this rank's buffer
        self.ptrs: List[Optional[int]] = []
        self.disabled = False            # set (on every rank) when a buffer could not be allocated or mapped

    def ensure(self, words: int) -> bool:
        """Collective: every rank passes the SAME `words` (push_plan's third value).  Returns False — on every rank — when
        any rank could not allocate or map a buffer (no peer access between the GPUs, CUDA IPC closed off by the
        container): the buffers are then released, `disabled` is set and the callers use the NCCL exchange."""
        import ctypes as C

        from ._native import SkmError, check, lib
        if self.disabled:
            return False
        if words <= self.words:
            return True
        rank, w = world()
        self.release()
        words = max(int(words * 1.25), 1 << 16)
        own = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        ok = not os.environ.get("SKM_PEER_FAIL")          # test hook: behave as if the allocation had failed
        if ok:
            try:
                check(lib().skm_peer_alloc(words * 8, C.byref(own), handle))
            except SkmError:
                ok = False
        handles = [None] * w
        dist.all_gather_object(handles, (bytes(handle), ok))
        opened: List[Optional[int]] = []
        ok = all(h[1] for h in handles)
        if ok:
            for r in range(w):
                if r == rank:
                    opened.append(own.value)
                    continue
                q = C.c_void_p()
                try:
                    check(lib().skm_peer_open((C.c_ubyte * 64).from_buffer_copy(handles[r][0]), C.byref(q)))
                except SkmError:
                    ok = False
                    break
                opened.append(q.value)
        flags = [None] * w
        dist.all_gather_object(flags, ok)
        if not all(flags):
            for r, q in enumerate(opened):
                if r != rank and q:
                    lib().skm_peer_close(q)
            dist.barrier()
            if own.value:
                lib().skm_peer_free(own.value)
            self.disabled = True
            return False
        self.ptrs, self.own, self.words = opened, own.value, words
        return True

    def release(self) -> None:
        from ._native import lib
        if self.own is None:
            return
        torch.cuda.synchronize()
        rank, w = world()
        for r, q in enumerate(self.ptrs):
            if r != rank and q:
                lib().skm_peer_close(q)
        if w > 1:
            dist.barrier()               # nobody maps the buffer any more
        lib().skm_peer_free(self.own)
        self.own, self.words, self.ptrs = None, 0, []


_peer_buffers: Optional[PeerBuffers] = None


def peer_buffers() -> PeerBuffers:
    global _peer_buffers
    if _peer_buffers is None:
        _peer_buffers = PeerBuffers()
    return _peer_buffers


def push_coo_by_key_range(keys: torch.Tensor, vals: torch.Tensor, key_bounds: Sequence[int], count_bits: int):
    """alltoall_coo_by_key_range over NVLink peer memory: ONE kernel packs the entries (key << count_bits | count) and
    stores them into the receive buffers of their owners (skm_coo_pack_push) — no NCCL send/recv, 8 instead of 16 bytes
    per entry on the wire.  Returns (own buffer pointer, runs [W] received run sizes in sender order, flag: int32 device
    tensor, non-zero when any rank saw a key / count that does not fit the packed word — the buffer content is then
    unusable and the caller falls back to alltoall_coo_by_key_range).  The all_reduce of the flag is also the fence that
    says every rank's stores have landed; the CALLER provides the fence before this call (any collective issued after
    the previous step's last read of the buffer — balanced_annotation_bounds does).  Returns None (on every rank) when the
    peer buffers cannot be set up; the caller then exchanges through alltoall_coo_by_key_range."""
    import ctypes as C

    from ._native import check, lib
    rank, w = world()
    dev = keys.device
    b = torch.tensor(list(key_bounds), dtype=torch.int64, device=dev)
    cut = torch.searchsorted(keys, b)
    send = (cut[1:] - cut[:-1]).contiguous()
    mat = torch.empty(w * w, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(mat, send)
    host = torch.cat([mat, cut]).cpu().numpy()                     # the step's one host synchronisation before the push
    mat_h, cut_h = host[:w * w].reshape(w, w), np.ascontiguousarray(host[w * w:])
    dst_off, runs, words = push_plan(mat_h, rank)
    pb = peer_buffers()
    if not pb.ensure(words):
        return None
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    ptrs = (C.c_void_p * w)(*pb.ptrs)
    dst_off = np.ascontiguousarray(dst_off)
    st = torch.cuda.current_stream(dev).cuda_stream
    check(lib().skm_coo_pack_push(keys.data_ptr(), vals.data_ptr(), cut_h.ctypes.data, w, int(count_bits), ptrs, dst_off.ctypes.data,
                                  flag.data_ptr(), st))
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    return pb.own, [int(x) for x in runs], flag


def balanced_annotation_bounds(keys: torch.Tensor, S: int, n_ann: int, weights: Optional[torch.Tensor] = None) -> List[int]:
    """W+1 annotation indices cutting [0, n_ann) into contiguous ranges with ~equal numbers of COO entries summed over
    all ranks (`keys` = this rank's sorted keys ann * S + code).  One all_reduce of the per-annotation entry histogram;
    identical on every rank.  Family sizes are Zipf-distributed: equal id ranges would give rank 0 most of the matrix.
    weights (int64 [nnz], optional): balance the SUM OF WEIGHTS per range instead of the entry count — e.g. how often an
    entry's k-mer occurs, which is what an annotation slice costs in the scoring SpMM."""
    rank, w = world()
    dev = keys.device
    if weights is None:
        edges = torch.arange(n_ann + 1, dtype=torch.int64, device=dev) * int(S)
        per_ann = torch.diff(torch.searchsorted(keys, edges))                  # local entries of every annotation
    else:
        per_ann = torch.zeros(n_ann, dtype=torch.int64, device=dev)
        per_ann.index_add_(0, torch.div(keys, int(S), rounding_mode="floor"), weights.to(torch.int64))
    allreduce_sum_(per_ann)
    csum = torch.cumsum(per_ann, 0)
    total = int(csum[-1].item()) if n_ann else 0
    targets = torch.tensor([total * r // w for r in range(1, w)], dtype=torch.int64, device=dev)
    cuts = torch.searchsorted(csum, targets, right=False).tolist() if w > 1 and n_ann else []
    bounds = [0] + [min(c + 1, n_ann) for c in cuts] + [n_ann]                  # the annotation that reaches the target closes its range
    for i in range(1, len(bounds)):
        bounds[i] = max(bounds[i], bounds[i - 1])
    return bounds


def barrier() -> None:
    if world()[1] > 1:
        dist.barrier()
