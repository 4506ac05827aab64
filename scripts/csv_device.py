"""CSV interchange text formatted on the device (skm_csv.cu), timed next to the host writers it stands in for.

  association CSV   apply_sparse_tiled at the C4 shape (syn6, k = 8; annotations learned from synthetic proteins) with
                    three sinks on the same queries: the device-formatted CSV (engine.AssociationsCSVText), the .skma
                    side-car and the host pyarrow CSV (sidecar.AssociationsCSVWriter, on a query subsample: its rate,
                    not the GPU, bounds it).  The formatter kernels alone (measure + write of one chunk) by CUDA events.
  count CSV         rules_sparse.write_counts_csv of a learned matrix in both layouts against rules.write_counts_csv /
                    write_totals_csv on a row subsample (the host writers need dense rows), and
                    rules_sparse.read_counts_csv (the device parser) reading each file back.
In-run parity: the host CSV of the subsample equals the device file's first rows byte for byte, the top-2 of every sink
run are bit-equal to the run without a sink, the sampled count rows equal the host writers' rows and the parsed
matrices equal the source matrix.

usage: python scripts/csv_device.py [--out DIR] [--nq N] [--n-ann A] [--ntrain N] [--count-ann A] [--scale F]
Writes one JSON line to stdout and DIR/csv_device.json.  The files go to a temporary directory (tens of GB at full
size: --scale shrinks the query and training counts)."""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import bench  # noqa: E402
from sparse_associations import events_ms, gpu_info, same_top2, wall_ms  # noqa: E402
from snekmer_b200 import alphabet as AL  # noqa: E402
from snekmer_b200 import engine as E  # noqa: E402
from snekmer_b200 import rules as R  # noqa: E402
from snekmer_b200 import rules_sparse as RS  # noqa: E402
from snekmer_b200 import sidecar as SC  # noqa: E402

K_MER, S = 8, 6 ** 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--nq", type=int, default=20_000)
    ap.add_argument("--n-ann", type=int, default=50_000)
    ap.add_argument("--ntrain", type=int, default=400_000)
    ap.add_argument("--count-ann", type=int, default=20_000, help="annotations of the count-file matrix (C3: 20,000)")
    ap.add_argument("--count-train", type=int, default=200_000)
    ap.add_argument("--csv-queries", type=int, default=200, help="queries written through the host CSV sink")
    ap.add_argument("--host-rows", type=int, default=8, help="count rows written by the host writers")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of nq / ntrain / count-ann / count-train")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    AL.register_alphabet("syn6", bench.SYN6)
    sc_ = lambda n, lo: max(lo, int(n * args.scale))
    nq, ntrain, n_ann = sc_(args.nq, 64), sc_(args.ntrain, 1000), args.n_ann
    rec = {"device": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "shape": "C4 (syn6, k = 8)", "nq": nq,
           "ntrain": ntrain, "n_ann": n_ann, "scale": args.scale}
    parity = []
    tmp = tempfile.mkdtemp(prefix="csv_device_")

    # ---- association CSV ----
    tr_res, tr_off = bench.synth_proteins(ntrain, 79)
    tr_ann = bench.zipf_annotations(ntrain, n_ann, 0.0, 80)
    tb = E.SequenceBatch.from_packed(tr_res, tr_off)
    keys, vals = E.learn_sparse(tb, "syn6", K_MER, torch.from_numpy(tr_ann), n_ann)
    del tb
    res, off = bench.synth_proteins(nq, 5)
    qb = E.SequenceBatch.from_packed(res, off)
    rowptr, cols, cvals = E.count_csr(qb, "syn6", K_MER, None)
    anns = [f"ann{a}" for a in range(n_ann)]
    labels = [f"q{q}|acc{q}|x" for q in range(nq)]
    plain = E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann)
    csv_path, skma_path, host_path = (os.path.join(tmp, x) for x in ("dev.csv", "rows.skma", "host.csv"))

    def run_csv():
        with E.AssociationsCSVText(csv_path, anns, labels) as w:
            return E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann, rows_sink=w)

    def run_skma():
        with SC.AssociationsWriter(skma_path, anns, labels) as w:
            return E.apply_sparse_tiled(rowptr, cols, cvals, keys, vals, S, n_ann, rows_sink=w.write)

    _, t_csv_first = wall_ms(run_csv)              # first call: includes allocating the pinned text buffers
    r_csv, t_csv = wall_ms(run_csv)                # steady state: the host allocator's pinned blocks are reused
    r_skma, t_skma = wall_ms(run_skma)
    nh = min(args.csv_queries, nq)
    t0 = time.perf_counter()
    with SC.AssociationsCSVWriter(host_path, anns, labels[:nh]) as w:
        E.apply_sparse_tiled(rowptr[:nh + 1], cols, cvals, keys, vals, S, n_ann, rows_sink=w.write)
    t_host = (time.perf_counter() - t0) * 1e3
    csv_bytes = os.path.getsize(csv_path)
    host_bytes = os.path.getsize(host_path)
    with open(csv_path, "rb") as f:
        head = f.read(host_bytes)
    parity.append(("association rows, host subsample byte-equal", head == open(host_path, "rb").read()))
    parity.append(("top-2 bit-equal, csv sink", same_top2(r_csv, plain)))
    parity.append(("top-2 bit-equal, skma sink", same_top2(r_skma, plain)))
    # formatter kernels on one chunk of rows (the engine's default chunk), device time by events
    w = E.AssociationsCSVText(os.path.join(tmp, "k.csv"), anns, labels)
    chunk = max(1, min(nq, E.ROWS_CHUNK_BYTES // w.row_bound()))
    block = torch.empty((chunk, n_ann), dtype=torch.float64, device="cuda")
    tile = E.sparse_max_ann(64)                    # the real cosine rows of the chunk's queries, every annotation tile
    for a0 in range(0, n_ann, tile):
        c = E.csc_build(keys, vals, S, min(tile, n_ann - a0), a0)
        E.apply_sparse(rowptr[:chunk + 1], cols, cvals, c, None, rows_out=block[:, a0:a0 + c.n_ann])
    text = torch.empty(chunk * w.row_bound(), dtype=torch.uint8, device="cuda")
    holder = {}
    k_ms, k_all = events_ms(lambda: holder.__setitem__("off", w.format_rows(0, block, text)), args.reps)
    k_bytes = int(holder["off"][-1].item())
    w.close()
    rec.update(assoc_csv_first_call_wall_s=round(t_csv_first / 1e3, 3), assoc_csv_wall_s=round(t_csv / 1e3, 3), assoc_csv_bytes=csv_bytes, assoc_csv_file_GBps=round(csv_bytes / t_csv / 1e6, 3),
               assoc_skma_wall_s=round(t_skma / 1e3, 3), assoc_skma_bytes=nq * n_ann * 8,
               assoc_skma_file_GBps=round(nq * n_ann * 8 / t_skma / 1e6, 3),
               assoc_host_csv_queries=nh, assoc_host_csv_wall_s=round(t_host / 1e3, 3),
               assoc_host_csv_Mvalues_per_s=round(nh * n_ann / t_host / 1e3, 2),
               assoc_device_csv_Mvalues_per_s=round(nq * n_ann / t_csv / 1e3, 2),
               formatter_chunk_rows=chunk, formatter_kernel_ms=round(k_ms, 3), formatter_kernel_ms_all=k_all,
               formatter_text_bytes=k_bytes, formatter_text_GBps=round(k_bytes / k_ms / 1e6, 2))
    for p in (csv_path, skma_path, host_path, os.path.join(tmp, "k.csv")):
        os.remove(p)
    del block, text, keys, vals, rowptr, cols, cvals, qb
    torch.cuda.empty_cache()

    # ---- count CSV of a learned matrix ----
    ca, ct = sc_(args.count_ann, 50), sc_(args.count_train, 2000)
    tr_res, tr_off = bench.synth_proteins(ct, 81)
    tr_ann = bench.zipf_annotations(ct, ca, 0.0, 82)
    tb = E.SequenceBatch.from_packed(tr_res, tr_off)
    keys, vals, totals = E.learn_sparse_with_totals(tb, "syn6", K_MER, torch.from_numpy(tr_ann), ca)
    seq_count = np.bincount(tr_ann[tr_ann >= 0], minlength=ca).astype(np.int64)
    m = RS.SparseCounts([f"ann{a}" for a in range(ca)], seq_count, AL.symbols("syn6"), K_MER, keys, vals, totals, ct)
    rec.update(count_ann=ca, count_train=ct, count_nnz=int(keys.numel()))
    kmers, rp, ccols, cv, sq, kc = RS._file_csr(m)
    rec["count_K"] = len(kmers)
    hr = min(args.host_rows, ca)
    for layout in ("learn", "total"):
        path = os.path.join(tmp, f"counts-{layout}.csv")
        _, t_dev = wall_ms(lambda: RS.write_counts_csv(path, m, layout=layout))
        nbytes = os.path.getsize(path)
        # host writer on the Totals row and the first hr annotation rows: dense rows from the same CSR
        rph, colh, vh = rp.cpu().numpy(), ccols.cpu().numpy(), cv.cpu().numpy()
        dense = np.zeros((hr + 1, len(kmers)), dtype=np.int64)
        for r in range(hr + 1):
            dense[r, colh[rph[r]:rph[r + 1]]] = vh[rph[r]:rph[r + 1]]
        hp = os.path.join(tmp, f"host-{layout}.csv")
        t0 = time.perf_counter()
        if layout == "learn":
            R.write_counts_csv(hp, R.LearnResult(m.annotations[:hr], sq[1:hr + 1], dense[1:], dense[0], int(sq[0]), kmers))
        else:
            R.write_totals_csv(hp, R.CountsTable(["Totals"] + m.annotations[:hr], kmers, sq[:hr + 1], kc[:hr + 1].cpu().numpy(), dense))
        t_host = time.perf_counter() - t0
        host_bytes = os.path.getsize(hp)
        with open(path, "rb") as f:
            head = f.read(host_bytes)
        parity.append((f"count rows ({layout}), host sample byte-equal", head == open(hp, "rb").read()))
        rec.update({f"count_{layout}_device_wall_s": round(t_dev / 1e3, 3), f"count_{layout}_bytes": nbytes,
                    f"count_{layout}_device_GBps": round(nbytes / t_dev / 1e6, 3),
                    f"count_{layout}_host_rows": hr + 1, f"count_{layout}_host_wall_s": round(t_host, 3),
                    f"count_{layout}_host_MBps": round(host_bytes / t_host / 1e6, 2)})
        # the parser reading back the file just written
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        back = RS.read_counts_csv(path, symbols=m.symbols)
        torch.cuda.synchronize()
        t_parse = time.perf_counter() - t0
        parity.append((f"parsed matrix ({layout}) equals the source", back.annotations == m.annotations and torch.equal(back.keys, m.keys)
                       and torch.equal(back.vals, m.vals) and torch.equal(back.totals, m.totals) and back.total_seqs == m.total_seqs
                       and np.array_equal(back.seq_count, m.seq_count)))
        rec.update({f"count_{layout}_parse_wall_s": round(t_parse, 3), f"count_{layout}_parse_GBps": round(nbytes / t_parse / 1e9, 3)})
        del back
        os.remove(path)
        os.remove(hp)
    os.rmdir(tmp)
    rec["parity_checks"] = {k: bool(v) for k, v in parity}
    rec["parity"] = "ok" if all(v for _, v in parity) else "FAILED"
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "csv_device.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
