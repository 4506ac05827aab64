"""Learn and apply over code spaces beyond the 2^27 tables (matrix keyed by basis column: engine.learn_wide,
query_csr_wide, apply_wide) at user scale, per phase, with CUDA events; plus the composition of existing entry points
as the baseline learn (count_csr_wide over the basis -> ann * K + col per entry in torch -> coo_merge), alternated with
the new path in the same process, and an in-run parity check of learn_wide against the numpy oracle on a sample.

Shapes: a learning set of 200,000 synthetic proteins (bench.synth_proteins), 2,000 annotations (Zipf 1.1, 30 %
unannotated), alphabets None at k = 8 and 14 and miqs at k = 10; 50,000 queries, half of them copies of training
proteins with 10 % substitutions.  Phases of the learn call (one C call) come from a torch.profiler run of their own:
key kernel (learn_wide_keys_kernel), sort (cub radix sort), run-length encode and finish, Totals (coo_colsum).

usage: python scripts/wide_learn_apply.py [--out DIR] [--n-train N] [--n-query N] [--reps R]
Writes one JSON line to stdout and DIR/wide_learn_apply.json."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from learn_coo_oracle import learn_coo  # noqa: E402
from oracle import skm_oracle as O  # noqa: E402
from snekmer_b200 import engine as E  # noqa: E402

SHAPES = [(None, 8), (None, 14), ("miqs", 10)]
N_ANN = 2000
AA = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", dtype=np.uint8)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def queries(res, off, n, seed):
    """n queries: half copies of random training proteins with 10 % substitutions, half fresh proteins."""
    rng = np.random.default_rng(seed)
    half = n // 2
    pick = rng.choice(len(off) - 1, size=half, replace=False)
    lens = off[pick + 1] - off[pick]
    q_off = np.zeros(n + 1, dtype=np.int64)
    fres, foff = bench.synth_proteins(n - half, seed + 1)
    np.cumsum(np.concatenate([lens, np.diff(foff)]), out=q_off[1:])
    src = np.concatenate([np.arange(off[i], off[i + 1]) for i in pick]) if half else np.zeros(0, np.int64)
    mut = res[src].copy()
    hit = rng.random(mut.size) < 0.10
    mut[hit] = rng.choice(AA, size=int(hit.sum()))
    return np.concatenate([mut, fres]), q_off


def timed(fn, *a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn(*a)
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1)


def baseline_learn(batch, a, k, basis, d_ann, n_ann):
    """The composition of existing entry points: per-sequence columns over the basis, one key per entry, coo_merge."""
    K = basis.K
    rowptr, _, cols, cvals = E.count_csr_wide(batch, a, k, basis)
    row = torch.repeat_interleave(torch.arange(batch.n, device=d_ann.device), rowptr[1:] - rowptr[:-1])
    ra = d_ann[row]
    ra = torch.where((ra < 0) | (ra >= n_ann), torch.full_like(ra, n_ann), ra)
    keys, vals = E.coo_merge(ra * K + cols.to(torch.int64), cvals.to(torch.int64), key_bound=(n_ann + 1) * K)
    totals = torch.zeros(K, dtype=torch.int64, device=keys.device).index_add_(0, keys % K, vals)
    m = int((keys < n_ann * K).sum())
    return keys[:m], vals[:m], totals


def apply_phases(qbatch, a, k, basis, keys, vals, n_ann):
    ms = {}
    (rowptr, cols, cvals), ms["query_count"] = timed(E.query_csr_wide, qbatch, a, k, basis)
    K = basis.K
    csc, ms["csc_build"] = timed(lambda: E.csc_build(keys + keys // K, vals, K + 1, n_ann))
    row_total = E.query_row_total_max(rowptr, cvals)
    r, ms["spmm"] = timed(E.apply_sparse, rowptr, cols, cvals, csc, row_total)
    return r, ms


def kernel_table(prof):
    """CUDA time per kernel name (ms), largest first."""
    agg = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t and ev.key not in ("cudaLaunchKernel",):
            agg[ev.key] = agg.get(ev.key, 0.0) + t / 1e3
    return dict(sorted(agg.items(), key=lambda kv: -kv[1])[:15])


def learn_phase_split(table):
    ph = {"key_kernel": 0.0, "sort": 0.0, "rle_finish": 0.0, "totals": 0.0, "other": 0.0}
    for name, t in table.items():
        if "learn_wide_keys_kernel" in name:
            ph["key_kernel"] += t
        elif "RadixSort" in name or "Onesweep" in name or "radix" in name.lower():
            ph["sort"] += t
        elif "RunLengthEncode" in name or "coo_finish" in name or "Rle" in name or "rle" in name:
            ph["rle_finish"] += t
        elif "coo_colsum" in name:
            ph["totals"] += t
        elif "bucket_index" in name or "Memset" in name or "memset" in name:
            ph["other"] += t
    return ph


def parity(res, off, ann, a, k, n_sample):
    n = min(n_sample, len(off) - 1)
    sres, soff = res[: off[n]], off[: n + 1]
    batch = E.SequenceBatch.from_packed(sres, soff)
    basis = E.build_basis_wide(batch, a, k, 0)
    keys, vals, totals = E.learn_wide(batch, a, k, basis, torch.from_numpy(ann[:n]), N_ANN)
    lut, syms = O.build_lut(a)
    si, pos, code, valid = O.window_codes(sres, soff, lut, len(syms), k)
    ob, _ = O.basis_codes(si, pos, code, valid, 0)
    wk, wv, wt = learn_coo(si, code, valid, ann[:n], N_ANN, ob)
    return bool(np.array_equal(basis.codes_host(), ob) and np.array_equal(keys.cpu().numpy(), wk)
                and np.array_equal(vals.cpu().numpy(), wv) and np.array_equal(totals.cpu().numpy(), wt))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--n-train", type=int, default=200000)
    ap.add_argument("--n-query", type=int, default=50000)
    ap.add_argument("--n-parity", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    res, off = bench.synth_proteins(args.n_train, 2024)
    ann = bench.zipf_annotations(args.n_train, N_ANN, 0.3, 2025)
    qres, qoff = queries(res, off, args.n_query, 2026)
    batch = E.SequenceBatch.from_packed(res, off)
    qbatch = E.SequenceBatch.from_packed(qres, qoff)
    d_ann = torch.from_numpy(ann).cuda()
    d_ann64 = d_ann.to(torch.int64)
    out = {"device": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "n_train": args.n_train,
           "residues_train": int(off[-1]), "n_query": args.n_query, "residues_query": int(qoff[-1]), "n_ann": N_ANN,
           "reps": args.reps, "shapes": []}
    ok_all = True
    for a, k in SHAPES:
        rec = {"alphabet": str(a), "k": k}
        basis, rec["basis_ms"] = timed(E.build_basis_wide, batch, a, k, 0)
        rec["K"] = basis.K
        # warm-up of every shape the timed runs use
        keys, vals, totals = E.learn_wide(batch, a, k, basis, d_ann, N_ANN)
        bk, bv, bt = baseline_learn(batch, a, k, basis, d_ann64, N_ANN)
        rec["baseline_equal"] = bool(torch.equal(keys, bk) and torch.equal(vals, bv) and torch.equal(totals, bt))
        del bk, bv, bt
        apply_phases(qbatch, a, k, basis, keys, vals, N_ANN)
        new_ms, base_ms, ph = [], [], []
        for _ in range(args.reps):
            _, t = timed(E.learn_wide, batch, a, k, basis, d_ann, N_ANN)
            new_ms.append(t)
            r = timed(baseline_learn, batch, a, k, basis, d_ann64, N_ANN)
            base_ms.append(r[1])
            del r
            _, p = apply_phases(qbatch, a, k, basis, keys, vals, N_ANN)
            ph.append(p)
        rec["nnz"] = int(keys.numel())
        rec["learn_ms"] = float(np.median(new_ms))
        rec["learn_ms_all"] = [round(x, 3) for x in new_ms]
        rec["baseline_learn_ms"] = float(np.median(base_ms))
        rec["baseline_learn_ms_all"] = [round(x, 3) for x in base_ms]
        rec["learn_seq_per_s"] = args.n_train / (rec["learn_ms"] / 1e3)
        rec["apply_phases_ms"] = {kk: float(np.median([p[kk] for p in ph])) for kk in ph[0]}
        rec["apply_ms"] = sum(rec["apply_phases_ms"].values())
        rec["apply_seq_per_s"] = args.n_query / (rec["apply_ms"] / 1e3)
        # kernel names and the learn call's phases: a profiled run of its own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            E.learn_wide(batch, a, k, basis, d_ann, N_ANN)
            torch.cuda.synchronize()
        lt = kernel_table(prof)
        rec["learn_kernels_ms"] = lt
        rec["learn_phases_ms"] = learn_phase_split(lt)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            apply_phases(qbatch, a, k, basis, keys, vals, N_ANN)
            torch.cuda.synchronize()
        rec["apply_kernels_ms"] = kernel_table(prof)
        t0 = time.time()
        rec["parity"] = "ok" if parity(res, off, ann, a, k, args.n_parity) else "MISMATCH"
        rec["parity_s"] = round(time.time() - t0, 1)
        ok_all &= rec["parity"] == "ok" and rec["baseline_equal"]
        out["shapes"].append(rec)
        del keys, vals, totals, basis
        torch.cuda.empty_cache()
        print(json.dumps({kk: rec[kk] for kk in ("alphabet", "k", "K", "learn_ms", "baseline_learn_ms", "apply_ms", "parity")}),
              file=sys.stderr, flush=True)
    out["parity"] = "ok" if ok_all else "MISMATCH"
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "wide_learn_apply.json"), "w") as f:
            f.write(line + "\n")
    return 0 if ok_all else 1


if __name__ == "__main__":
    sys.exit(main())
