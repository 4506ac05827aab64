"""Full association rows on the sparse path at the C4 shape, per phase, with CUDA events: the top-2-only SpMM kernel
against the same kernel writing every query's cosine row (skm_apply_sparse_rows) on the same queries and tiles, the
device -> host copy of the rows, and the wall time of engine.apply_sparse_tiled with a rows sink that discards the
blocks, one that writes the .skma side-car and one that writes the seq-annotation-scores CSV (the CSV on a subsample:
pyarrow's CSV formatting, not the GPU, bounds it).  In-run parity: the top-2 of every sink run are bit-equal to
apply_sparse_tiled without a sink, sampled rows are within 1e-12 of a float64 numpy cosine built from the host COO
matrix, the rows at top1 / top2 equal score1 / score2 bit for bit and the .skma holds the device's rows bit for bit.

Shape: bench.py's apply_sparse workload (syn6, k = 8, S = 1,679,616; 50,000 annotations learned from 400,000
synthetic proteins) scored for 20,000 queries: 8 GB of float64 rows, far more than L2.

usage: python scripts/sparse_associations.py [--out DIR] [--nq N] [--reps R] [--csv-queries N] [--scale F]
Writes one JSON line to stdout and DIR/sparse_associations.json."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from snekmer_b200 import alphabet as AL  # noqa: E402
from snekmer_b200 import engine as E  # noqa: E402
from snekmer_b200 import sidecar as SC  # noqa: E402

K_MER, S = 8, 6 ** 8


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def events_ms(fn, reps):
    """Median device time of fn() over reps launches (one warm-up first)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    out = []
    for _ in range(reps):
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return float(np.median(out)), [round(x, 3) for x in out]


def wall_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def same_top2(a, b):
    return (torch.equal(a.top1, b.top1) and torch.equal(a.top2, b.top2) and torch.equal(a.score1, b.score1)
            and bool(np.array_equal(a.score2.cpu().numpy(), b.score2.cpu().numpy(), equal_nan=True)))


def numpy_rows(sample, rowptr, cols, cvals, keys, vals, n_ann):
    """float64 cosine rows of the sampled queries from the host COO matrix: exact int64 dots over the query's codes."""
    ann, code = keys // S, keys % S
    mn2 = np.bincount(ann, weights=vals.astype(np.float64) ** 2, minlength=n_ann)
    order = np.argsort(code, kind="stable")
    code_sorted = code[order]
    out = np.zeros((len(sample), n_ann))
    for i, q in enumerate(sample):
        c, v = cols[rowptr[q]:rowptr[q + 1]].astype(np.int64), cvals[rowptr[q]:rowptr[q + 1]].astype(np.int64)
        dot = np.zeros(n_ann, dtype=np.int64)
        lo, hi = np.searchsorted(code_sorted, c), np.searchsorted(code_sorted, c, side="right")
        for cnt, a0, a1 in zip(v, lo, hi):
            idx = order[a0:a1]
            np.add.at(dot, ann[idx], cnt * vals[idx])
        qn = np.sqrt(float((v * v).sum()))
        nz = dot != 0
        out[i, nz] = dot[nz] / qn / np.sqrt(mn2[nz])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--nq", type=int, default=20_000)
    ap.add_argument("--n-ann", type=int, default=50_000)
    ap.add_argument("--ntrain", type=int, default=400_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--csv-queries", type=int, default=400, help="queries written through the CSV sink")
    ap.add_argument("--samples", type=int, default=48, help="rows checked against the numpy cosine")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of nq / ntrain (rehearsal at small size)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    AL.register_alphabet("syn6", bench.SYN6)
    nq, ntrain, n_ann = max(64, int(args.nq * args.scale)), max(1000, int(args.ntrain * args.scale)), args.n_ann
    rec = {"device": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "shape": "C4 (syn6, k = 8)", "nq": nq,
           "ntrain": ntrain, "n_ann": n_ann, "reps": args.reps}

    tr_res, tr_off = bench.synth_proteins(ntrain, 79)
    tr_ann = bench.zipf_annotations(ntrain, n_ann, 0.0, 80)
    tb = E.SequenceBatch.from_packed(tr_res, tr_off)
    keys, vals = E.learn_sparse(tb, "syn6", K_MER, torch.from_numpy(tr_ann), n_ann)
    del tb
    res, off = bench.synth_proteins(nq, 5)
    qb = E.SequenceBatch.from_packed(res, off)
    rowptr, cols, cvals = E.count_csr(qb, "syn6", K_MER, None)
    row_total = E.query_row_total_max(rowptr, cvals)
    acc_bits = E.sparse_acc_bits(int(vals.max().item()), row_total)
    tile = E.sparse_max_ann(acc_bits)
    tiles = [(a0, E.csc_build(keys, vals, S, min(tile, n_ann - a0), a0)) for a0 in range(0, n_ann, tile)]
    rec.update(nnz_matrix=int(keys.numel()), nnz_queries=int(cols.numel()), acc_bits=acc_bits, tiles=len(tiles),
               row_bytes=nq * n_ann * 8)

    # ---- kernels: top-2 only against ROWS on the same queries and tiles, alternated ----
    rows = torch.empty((nq, n_ann), dtype=torch.float64, device="cuda")

    def top2_only():
        for _, c in tiles:
            E.apply_sparse(rowptr, cols, cvals, c, row_total)

    def with_rows():
        for a0, c in tiles:
            E.apply_sparse(rowptr, cols, cvals, c, row_total, rows_out=rows[:, a0:a0 + c.n_ann])

    t2, r2 = [], []
    for _ in range(args.reps):
        t2.append(events_ms(top2_only, 1)[0])
        r2.append(events_ms(with_rows, 1)[0])
    rec["kernel_top2_ms"], rec["kernel_rows_ms"] = round(float(np.median(t2)), 3), round(float(np.median(r2)), 3)
    rec["kernel_top2_ms_all"], rec["kernel_rows_ms_all"] = [round(x, 3) for x in t2], [round(x, 3) for x in r2]
    rec["rows_over_top2"] = round(rec["kernel_rows_ms"] / rec["kernel_top2_ms"], 3)
    rec["rows_extra_GBps"] = round(nq * n_ann * 8 / ((rec["kernel_rows_ms"] - rec["kernel_top2_ms"]) * 1e-3) / 1e9, 1) \
        if rec["kernel_rows_ms"] > rec["kernel_top2_ms"] else None

    # ---- device -> host copy of the rows, in the engine's default blocks ----
    chunk = max(1, min(nq, E.ROWS_CHUNK_BYTES // (8 * n_ann)))
    host = torch.empty((chunk, n_ann), dtype=torch.float64, pin_memory=True)

    def d2h():
        for q0 in range(0, nq, chunk):
            n = min(chunk, nq - q0)
            host[:n].copy_(rows[q0:q0 + n], non_blocking=True)

    rec["d2h_ms"], rec["d2h_ms_all"] = events_ms(d2h, args.reps)
    rec["d2h_GBps"] = round(nq * n_ann * 8 / (rec["d2h_ms"] * 1e-3) / 1e9, 2)
    rec["chunk_rows"] = chunk
    del host

    # ---- parity of the rows kernel: sampled rows against numpy, top-2 entries against the scores ----
    ref = E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann)
    rng = np.random.default_rng(7)
    sample = np.sort(rng.choice(nq, size=min(args.samples, nq), replace=False))
    got = rows[torch.from_numpy(sample).cuda()].cpu().numpy()
    want = numpy_rows(sample, rowptr.cpu().numpy(), cols.cpu().numpy(), cvals.cpu().numpy(), keys.cpu().numpy(),
                      vals.cpu().numpy(), n_ann)
    rec["sample_rows"] = len(sample)
    rec["sample_max_abs_err"] = float(np.max(np.abs(got - want)))
    q = torch.arange(nq, device="cuda")
    t2d = ref.top2.to(torch.int64)
    ok_rows = bool(torch.equal(rows[q, ref.top1.to(torch.int64)], ref.score1)) and bool(
        torch.equal(rows[q[t2d >= 0], t2d[t2d >= 0]], ref.score2[t2d >= 0]))
    parity = {"rows_numpy_1e-12": rec["sample_max_abs_err"] < 1e-12, "rows_at_top2_bit_equal": ok_rows}
    del rows
    torch.cuda.empty_cache()

    # ---- wall time of the streamed paths ----
    def run(sink, n=nq):
        return E.apply_sparse_tiled(rowptr[:n + 1], cols, cvals, keys, vals, S, n_ann, rows_sink=sink)

    run(lambda q0, b: None, min(nq, 2 * chunk))                     # warm-up: pinned blocks, side stream
    r_dis, rec["wall_discard_ms"] = wall_ms(lambda: run(lambda q0, b: None))
    parity["top2_discard_bit_equal"] = same_top2(r_dis, ref)
    with tempfile.TemporaryDirectory() as tmp:
        skma = os.path.join(tmp, "rows.skma")
        try:
            with SC.AssociationsWriter(skma, [f"TIGR{i:05d}" for i in range(n_ann)], [f"q{i}" for i in range(nq)]) as w:
                r_sk, rec["wall_skma_ms"] = wall_ms(lambda: run(w.write))
            parity["top2_skma_bit_equal"] = same_top2(r_sk, ref)
            parity["skma_rows_bit_equal"] = bool(np.array_equal(SC.read_associations(skma)["scores"][sample], got))
        except OSError as e:                                       # a temporary directory too small for the rows
            rec["wall_skma_ms"] = f"not measured: {e}"
        nc = min(nq, args.csv_queries)
        csv = os.path.join(tmp, "rows.csv")
        with SC.AssociationsCSVWriter(csv, [f"TIGR{i:05d}" for i in range(n_ann)], [f"q{i}" for i in range(nc)]) as w:
            r_csv, rec["wall_csv_ms"] = wall_ms(lambda: run(w.write, nc))
        rec["csv_queries"], rec["csv_bytes"] = nc, os.path.getsize(csv)
        rec["csv_values_per_s"] = round(nc * n_ann / (rec["wall_csv_ms"] * 1e-3))
        parity["top2_csv_bit_equal"] = same_top2(r_csv, E.apply_sparse_tiled(rowptr[:nc + 1], cols, cvals, keys, vals, S, n_ann))
    rec["wall_discard_GBps"] = round(nq * n_ann * 8 / (rec["wall_discard_ms"] * 1e-3) / 1e9, 2)
    if isinstance(rec.get("wall_skma_ms"), float):
        rec["wall_skma_GBps"] = round(nq * n_ann * 8 / (rec["wall_skma_ms"] * 1e-3) / 1e9, 2)
    rec["parity_checks"] = parity
    rec["parity"] = "ok" if all(parity.values()) else "MISMATCH"
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "sparse_associations.json"), "w") as f:
            f.write(line + "\n")
    return 0 if rec["parity"] == "ok" else 1


if __name__ == "__main__":
    sys.exit(main())
