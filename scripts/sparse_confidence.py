"""The evaluate step of the sparse path (eval_apply + evaluate over a learned matrix) at user scale, per phase, with
CUDA events: query CSR, SpMM top-2, row classes (skm_confidence_classify), crosstabs (skm_confidence_hist), and the
host finalize (histograms to the host, the 101-point curve).  Beside them, the host classifier that the device one
replaces (confidence.classify_rows) on the same rows: building the eval_apply labels, then classifying with the truth
shortcut and from the labels alone.  In-run parity: the device classes equal classify_rows on every row, and the
crosstabs equal a numpy bincount of (prediction, Difference bin, class) with the bins computed in numpy.

Shapes (engine level, no Python strings on the device path): C3 — syn6, k = 8, 1,000,000 training proteins
(bench.synth_proteins), 20,000 annotations (bench.zipf_annotations, 30 % unannotated); wide — alphabet None, k = 8
(20^8 > 2^27, matrix keyed by basis column), 200,000 proteins, 2,000 annotations.  The training set is scored against
the matrix learned from it, as the learn workflow's eval_apply does.

usage: python scripts/sparse_confidence.py [--out DIR] [--reps R] [--scale F]
Writes one JSON line to stdout and DIR/sparse_confidence.json."""
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
import bench  # noqa: E402
from oracle.skm_evaluator import POSSIBLE  # noqa: E402
from snekmer_b200 import alphabet as AL  # noqa: E402
from snekmer_b200 import confidence as CF  # noqa: E402
from snekmer_b200 import engine as E  # noqa: E402
from snekmer_b200._native import check, lib  # noqa: E402
from snekmer_b200.sidecar import _strings_to_arrays  # noqa: E402

SHAPES = [("C3", "syn6", 8, 1_000_000, 20_000), ("wide", None, 8, 200_000, 2_000)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def timed(fn, *a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn(*a)
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1)


def host_timed(fn, *a):
    t0 = time.perf_counter()
    out = fn(*a)
    return out, (time.perf_counter() - t0) * 1e3


def learn(batch, a, k, d_ann, n_ann):
    if a is None:
        basis = E.build_basis_wide(batch, a, k, 0)
        keys, vals, _ = E.learn_wide(batch, a, k, basis, d_ann, n_ann)
        return basis, keys, vals
    keys, vals, _ = E.learn_sparse_with_totals(batch, a, k, d_ann, n_ann)
    return None, keys, vals


def query_csr(batch, a, k, basis):
    return E.query_csr_wide(batch, a, k, basis) if basis is not None else E.count_csr(batch, a, k, None)


def spmm(csr, basis, keys, vals, S, n_ann):
    if basis is not None:
        return E.apply_wide(*csr, keys, vals, basis.K, n_ann)
    return E.apply_sparse_tiled(*csr, keys, vals, S, n_ann)


def numpy_tables(pred, s1, s2, cls, n_ann):
    """Crosstabs by bincount, Difference bins as learn.smk:1052-1110 computes them (numpy round, the 101 values)."""
    with np.errstate(invalid="ignore"):
        diff = -(np.round(s2 - s1, 2))
        j = np.rint(diff * 100.0)
    ok = (pred >= 0) & ~np.isnan(diff) & (j >= 0) & (j <= 100)
    ji = np.where(ok, j, 0).astype(np.int64)
    ok &= np.asarray(POSSIBLE)[ji] == diff
    idx = pred.astype(np.int64) * 101 + ji
    ht = np.bincount(idx[ok & (cls == 1)], minlength=n_ann * 101).reshape(n_ann, 101)
    hf = np.bincount(idx[ok & (cls == 2)], minlength=n_ann * 101).reshape(n_ann, 101)
    return ht, hf, np.where(ok, ji, 255)


def run_shape(name, a, k, n, n_ann, reps):
    res, off = bench.synth_proteins(n, 4242)
    ann = bench.zipf_annotations(n, n_ann, 0.3, 4243)
    batch = E.SequenceBatch.from_packed(res, off)
    d_ann = torch.from_numpy(ann).cuda()
    tab = E.alphabet_tables(a)
    S = E.code_space(tab.nsym, k)
    (basis, keys, vals), learn_ms = timed(learn, batch, a, k, d_ann, n_ann)
    names = [f"TIGR{i:05d}" for i in range(n_ann)]          # matrix row i = annotation i, the label's name
    buf, noff = _strings_to_arrays(names)
    d_buf, d_off = torch.from_numpy(buf.copy()).cuda(), torch.from_numpy(noff).cuda()
    d_truth = d_ann.clone()                                 # -1: an unannotated sequence, an `_unknown_` row
    cls = torch.empty(n, dtype=torch.uint8, device="cuda")
    ht = torch.zeros((n_ann, 101), dtype=torch.int64, device="cuda")
    hf = torch.zeros_like(ht)
    bins = torch.empty(n, dtype=torch.uint8, device="cuda")

    def classify(r):
        check(lib().skm_confidence_classify(E._ptr(r.top1), E._ptr(d_truth), n, 0, E._ptr(d_buf), E._ptr(d_off), n_ann,
                                            E._ptr(cls), E._stream()))

    def hist(r):
        check(lib().skm_confidence_hist(E._ptr(r.top1), E._ptr(r.score1), E._ptr(r.score2), E._ptr(cls), n, n_ann,
                                        E._ptr(ht), E._ptr(hf), E._ptr(bins), E._stream()))

    def finalize():
        acc = CF.ConfidenceAccumulator()
        acc.add_histograms(ht.cpu().numpy(), hf.cpu().numpy(), names)
        return acc.finalize()

    phases = {"query_csr": [], "spmm_top2": [], "classify": [], "histogram": [], "host_finalize": []}
    for rep in range(reps + 1):                              # rep 0 warms every shape up
        csr, t_csr = timed(query_csr, batch, a, k, basis)
        r, t_spmm = timed(spmm, csr, basis, keys, vals, S, n_ann)
        del csr
        _, t_cls = timed(classify, r)
        ht.zero_()
        hf.zero_()
        _, t_hist = timed(hist, r)
        ev, t_fin = host_timed(finalize)
        if rep:
            for key, t in zip(phases, (t_csr, t_spmm, t_cls, t_hist, t_fin)):
                phases[key].append(t)
    rec = {"shape": name, "alphabet": str(a), "k": k, "n_train": n, "residues": int(off[-1]), "n_ann": n_ann,
           "key_space": "basis column" if basis is not None else "code", "K": basis.K if basis is not None else S,
           "nnz": int(keys.numel()), "learn_ms": round(learn_ms, 3),
           "phases_ms": {kk: round(float(np.median(v)), 4) for kk, v in phases.items()},
           "phases_ms_all": {kk: [round(x, 4) for x in v] for kk, v in phases.items()}}
    rec["device_evaluate_ms"] = round(sum(rec["phases_ms"][kk] for kk in ("classify", "histogram")), 4)
    # the host classifier on the same rows
    top1 = r.top1.cpu().numpy()
    labels, rec["host_labels_ms"] = host_timed(
        lambda: [f"{names[t]}_known_{q}" if t >= 0 else f"ACC{q}_unknown_{q}" for q, t in enumerate(ann.tolist())])
    want_t, rec["host_classify_truth_ms"] = host_timed(CF.classify_rows, top1, labels, names, ann)
    want_l, rec["host_classify_labels_ms"] = host_timed(CF.classify_rows, top1, labels, names)
    rec["host_classify_rows"] = n
    got = cls.cpu().numpy()
    rec["class_counts"] = np.bincount(got, minlength=3).tolist()
    nt, nf, nbins = numpy_tables(top1, r.score1.cpu().numpy(), r.score2.cpu().numpy(), got, n_ann)
    rec["bins_equal_numpy"] = bool(np.array_equal(bins.cpu().numpy(), nbins))
    ok = (np.array_equal(got, want_t) and np.array_equal(got, want_l) and np.array_equal(ht.cpu().numpy(), nt)
          and np.array_equal(hf.cpu().numpy(), nf))
    rec["parity"] = "ok" if ok else "MISMATCH"
    rec["weight"] = float(ev.weight[0])
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the training sets (rehearsal at small size)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    AL.register_alphabet("syn6", bench.SYN6)
    out = {"device": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "reps": args.reps, "shapes": []}
    for name, a, k, n, n_ann in SHAPES:
        rec = run_shape(name, a, k, max(1000, int(n * args.scale)), n_ann, args.reps)
        out["shapes"].append(rec)
        print(json.dumps({kk: rec[kk] for kk in ("shape", "phases_ms", "host_classify_labels_ms", "parity")}), file=sys.stderr, flush=True)
        torch.cuda.empty_cache()
    out["parity"] = "ok" if all(s["parity"] == "ok" for s in out["shapes"]) else "MISMATCH"
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "sparse_confidence.json"), "w") as f:
            f.write(line + "\n")
    return 0 if out["parity"] == "ok" else 1


if __name__ == "__main__":
    sys.exit(main())
