#!/usr/bin/env python
"""The dense count kernel at the C2 shape (1 M synthetic proteins of bench.synth_proteins seed 2, miqs k = 3, S = K =
1,000, int32 [N, K] output = 4 GB) beside the two floors it is judged against, all in one process with CUDA events
(mean of 50 launches after warm-up):
  * write floor: fill_ of the same [1 M, 1000] int32 buffer (4 GB written, nothing read);
  * copy: a 4 GB device-to-device copy (4 GB read + 4 GB written);
  * count: skm_count_dense of this build (through engine.count_dense, the order-only basis' column map).
Writes one JSON line to stdout (and to DIR/count_dense_ab.json with --out DIR), with the card name and power limit.

    python scripts/count_dense_ab.py [--out DIR] [--nseq N] [--reps R]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from snekmer_b200 import engine as E  # noqa: E402


def mean_ms(fn, reps, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def card():
    idx = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0] or "0"
    try:
        r = subprocess.run(["nvidia-smi", "-i", idx, "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clock = [f.strip() for f in r.stdout.strip().split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # the numbers stand without it, but say why it is missing
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--nseq", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "count_dense_ab.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res_np, offsets = bench.synth_proteins(args.nseq, 2)
    batch = E.SequenceBatch.from_packed(res_np, offsets, dev)
    a, k = "miqs", 3
    out = torch.empty((batch.n, 1000), dtype=torch.int32, device=dev)
    basis, _ = E.vectorize_order_only(batch, a, k, out=out)
    assert basis.K == basis.S == 1000
    nbytes = out.numel() * out.element_size()
    fill_ms = mean_ms(lambda: out.fill_(0), args.reps)
    src = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    src.fill_(1)
    copy_ms = mean_ms(lambda: dst.copy_(src), args.reps)
    del src, dst
    count_ms = mean_ms(lambda: E.count_dense(batch, a, k, basis, out=out), args.reps)
    nres = int(offsets[-1])
    alg = nres + 8 * (batch.n + 1) + nbytes
    line = {
        "metric": "count_dense C2 against the write floor", "card": card(), "nseq": batch.n, "nres": nres, "reps": args.reps,
        "write_floor": {"ms": fill_ms, "gbs": nbytes / (fill_ms * 1e-3) / 1e9, "bytes": nbytes, "what": "torch fill_ of the [N, 1000] int32 output"},
        "d2d_copy": {"ms": copy_ms, "gbs": 2 * nbytes / (copy_ms * 1e-3) / 1e9, "bytes_moved": 2 * nbytes, "what": "4 GB device-to-device copy (read + write)"},
        "count_dense": {"ms": count_ms, "gbs": alg / (count_ms * 1e-3) / 1e9, "algorithmic_bytes": alg,
                        "over_write_floor": count_ms / fill_ms},
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "count_dense_ab.json"), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
