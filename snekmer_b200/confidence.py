"""confidence: the evaluate rule (class Evaluator, rules/learn.smk:923-1348) on the GPU path.

The reference reads every ``seq-annotation-scores-*.csv`` (Q x A), takes the top two scores of each row,
bins ``Difference = round(Top - Second, 2)`` and cross-tabulates Known rows by (Prediction, Difference) for
True and False predictions; the ratio T / (T + F) per bin, interpolated, is the global confidence curve that
the apply rule looks up (apply.smk:301-335).

Here the per-row work (top-2 of a score matrix, Difference bins, the two histograms) runs on the device
(``skm_top2_rows_f64``, ``skm_confidence_hist``); when the scores come straight from ``engine.apply_*`` the
Q x A matrix never exists.  The reference decides a row's class with string tests on its label (T iff the predicted
name is a substring of the label, Known iff the label lacks "unknown", learn.smk:997-1008): ``classify_rows`` does
that on the host for labels read from a file; for the rows of eval_apply, whose labels are built from the annotation
name and the row number, ``skm_confidence_classify`` does it on the device from a name table (``add_device``).  The
101-point curve arithmetic stays on the host (float64, same operation order as the reference).
Multi-GPU: histograms are summed with one all_reduce (dist.allreduce_confidence_tables).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import dist as D
from . import engine as E
from .sidecar import _strings_to_arrays
from ._native import check, lib

NBINS = 101
POSSIBLE_VALS = [round(x * 0.01, 2) for x in range(NBINS)]      # learn.smk:1063
INDEX_COL = "__index_level_0__"


def top2_rows(scores: torch.Tensor) -> E.ApplyResult:
    """Column of the maximum and the two largest values of every row of a float64 matrix with NaN holes
    (idxmax + argpartition of learn.smk:964-981)."""
    dev = E._require_cuda(scores.device)
    scores = scores.contiguous()
    assert scores.dtype == torch.float64 and scores.dim() == 2
    nq, a = scores.shape
    top1 = torch.empty(nq, dtype=torch.int32, device=dev)
    top2 = torch.empty(nq, dtype=torch.int32, device=dev)
    s1 = torch.empty(nq, dtype=torch.float64, device=dev)
    s2 = torch.empty(nq, dtype=torch.float64, device=dev)
    check(lib().skm_top2_rows_f64(E._ptr(scores), nq, a, E._ptr(top1), E._ptr(top2), E._ptr(s1), E._ptr(s2), E._stream()))
    return E.ApplyResult(top1, top2, s1, s2, None)


def difference_bins(top1: torch.Tensor, s1: torch.Tensor, s2: torch.Tensor, n_ann: int) -> torch.Tensor:
    """uint8 [Q]: 100 * round(score1 - score2, 2), 255 where undefined."""
    dev = E._require_cuda(top1.device)
    nq = top1.numel()
    out = torch.empty(nq, dtype=torch.uint8, device=dev)
    check(lib().skm_confidence_hist(E._ptr(top1.contiguous()), E._ptr(s1.contiguous()), E._ptr(s2.contiguous()), None, nq, int(n_ann),
                                    None, None, E._ptr(out), E._stream()))
    return out


def classify_rows(pred: np.ndarray, labels: Sequence[str], annotations: Sequence[str],
                  truth: Optional[np.ndarray] = None) -> np.ndarray:
    """uint8 [Q]: 0 = Unknown row (not counted), 1 = Known & True, 2 = Known & False (learn.smk:997-1008).
    `truth` (optional, int [Q]): index of the annotation the label was built from (``<annotation>_known_<i>``),
    -1 for ``<accession>_unknown_<i>`` rows; it only short-cuts the substring tests of rows predicted right."""
    names = [str(a) for a in annotations]
    q = len(labels)
    cls = np.zeros(q, dtype=np.uint8)
    if truth is not None:
        truth = np.asarray(truth)
        name_unknown = np.array(["unknown" in n for n in names] + [True], dtype=bool)
        known = ~name_unknown[truth]                      # truth == -1 -> the appended True
        right = known & (pred == truth) & (pred >= 0)
        cls[right] = 1
        todo = np.flatnonzero(known & ~right)
    else:
        todo = np.arange(q)
    for i in todo:
        lab = str(labels[i])
        if "unknown" in lab:
            continue
        p = int(pred[i])
        cls[i] = 1 if (p >= 0 and names[p] in lab) else 2
    return cls


def joint_name_table(annotations: Sequence[str], names: Sequence[Optional[str]]):
    """(table, index int32 [len(names)]): the name table of ``skm_confidence_classify`` — the matrix's annotations
    in matrix order, then every other name of `names` once, in order of first appearance — and the entry of each of
    `names` in it (-1 for None: an ``_unknown_`` row)."""
    table = [str(a) for a in annotations]
    index: Dict[str, int] = {}
    for i, a in enumerate(table):
        index.setdefault(a, i)
    idx = np.full(len(names), -1, dtype=np.int32)
    for j, n in enumerate(names):
        if n is None:
            continue
        n = str(n)
        i = index.get(n)
        if i is None:
            i = index[n] = len(table)
            table.append(n)
        idx[j] = i
    return table, idx


def classify_device(top1: torch.Tensor, truth: torch.Tensor, row_base: int, names: Sequence[str]) -> torch.Tensor:
    """uint8 [Q], the classes of ``classify_rows`` for the eval_apply labels ``names[truth[q]]_known_<row_base + q>``
    (``<accession>_unknown_<n>`` where truth[q] < 0), without the labels.  top1 indexes the first A entries of
    `names` (joint_name_table)."""
    dev = E._require_cuda(top1.device)
    nq = top1.numel()
    assert truth.numel() == nq
    buf, off = _strings_to_arrays(names)
    d_buf = torch.from_numpy(buf.copy()).to(dev) if buf.size else None
    d_off = torch.from_numpy(off).to(dev)
    cls = torch.empty(nq, dtype=torch.uint8, device=dev)
    check(lib().skm_confidence_classify(E._ptr(top1.to(dev, torch.int32).contiguous()), E._ptr(truth.to(dev, torch.int32).contiguous()),
                                        nq, int(row_base), E._ptr(d_buf), E._ptr(d_off), len(names), E._ptr(cls), E._stream()))
    return cls


# zero-bin key of a rank with no qualifying row (dist.allreduce_confidence_tables takes the minimum)
NO_ZERO_ROW = np.iinfo(np.int64).max


@dataclass
class EvalResult:
    rows: List[str]                 # sorted names of the predictions that occur among Known rows
    ratio: np.ndarray               # float64 [R, 101], NaN where T + F = 0
    confidence: np.ndarray          # float64 [101]
    weight: np.ndarray              # float64 [101]
    sum: np.ndarray                 # float64 [101]
    zero_negative: bool             # the zero bin is labelled -0.0 (see ConfidenceAccumulator.add)
    weight_is_int: bool = False     # pandas keeps integer columns for ONE input file (crosstab counts); the running
    sum_is_int: bool = False        # tables of several files are float (concat + groupby.sum + fillna)

    def labels(self) -> List[float]:
        out = list(POSSIBLE_VALS)
        if self.zero_negative:
            out[0] = -0.0
        return out


class ConfidenceAccumulator:
    """Running True / False crosstabs over files (handle_running_crosstabs, learn.smk:1063-1176), kept on the
    device as int64 [A, 101] per distinct annotation list."""

    def __init__(self):
        self._names: Dict[str, int] = {}
        self._t: List[np.ndarray] = []
        self._f: List[np.ndarray] = []
        self._files = 0
        self.zero_negative = False

    def add(self, result: E.ApplyResult, labels: Sequence[str], annotations: Sequence[str],
            truth: Optional[np.ndarray] = None) -> None:
        """One file / shard: top-2 of every row (device tensors) + row labels + column names."""
        dev = E._require_cuda(result.top1.device)
        a, nq = len(annotations), result.top1.numel()
        pred = result.top1.cpu().numpy()
        cls = classify_rows(pred, labels, annotations, truth)
        ht = torch.zeros((max(a, 1), NBINS), dtype=torch.int64, device=dev)
        hf = torch.zeros((max(a, 1), NBINS), dtype=torch.int64, device=dev)
        bins = torch.empty(max(nq, 1), dtype=torch.uint8, device=dev)
        d_cls = torch.from_numpy(cls).to(dev)
        check(lib().skm_confidence_hist(E._ptr(result.top1.contiguous()), E._ptr(result.score1.contiguous()),
                                        E._ptr(result.score2.contiguous()), E._ptr(d_cls), nq, a, E._ptr(ht), E._ptr(hf),
                                        E._ptr(bins), E._stream()))
        if self._files == 0 and nq:
            # label of the zero bin = first zero Difference among the Known & True rows of the first file:
            # -(round(0.0)) = -0.0 for an exact tie, +0.0 otherwise (pd.crosstab keeps the first-seen one)
            z = np.flatnonzero((cls == 1) & (bins[:nq].cpu().numpy() == 0))
            if z.size:
                i = int(z[0])
                self.zero_negative = bool(result.score1[i].item() == result.score2[i].item())
        self._files += 1
        self.add_histograms(ht.cpu().numpy(), hf.cpu().numpy(), annotations)

    def add_device(self, result: E.ApplyResult, truth: torch.Tensor, row_base: int, names: Sequence[str],
                   annotations: Sequence[str]) -> None:
        """One eval_apply file (or one rank's contiguous rows of it) with the classes decided on the device
        (classify_device): row q is global row ``row_base + q``, labelled from ``names[truth[q]]``; `names` starts with
        the A `annotations` that result.top1 indexes.  With several ranks every rank calls this for every file: the
        histograms are summed over ranks and the zero-bin label comes from the lowest global row that qualifies."""
        dev = E._require_cuda(result.top1.device)
        a, nq = len(annotations), result.top1.numel()
        top1 = result.top1.contiguous()
        cls = classify_device(top1, truth, row_base, names)
        ht = torch.zeros((max(a, 1), NBINS), dtype=torch.int64, device=dev)
        hf = torch.zeros((max(a, 1), NBINS), dtype=torch.int64, device=dev)
        bins = torch.empty(max(nq, 1), dtype=torch.uint8, device=dev)
        s1, s2 = result.score1.contiguous(), result.score2.contiguous()
        check(lib().skm_confidence_hist(E._ptr(top1), E._ptr(s1), E._ptr(s2), E._ptr(cls), nq, a, E._ptr(ht), E._ptr(hf),
                                        E._ptr(bins), E._stream()))
        # zero-bin label (see add): key 2 * row + (exact tie) of the first Known & True row in bin 0
        zero = torch.full((1,), NO_ZERO_ROW, dtype=torch.int64, device=dev)
        if self._files == 0 and nq:
            key = (torch.arange(nq, dtype=torch.int64, device=dev) + int(row_base)) * 2 + (s1 == s2)
            zero = torch.where((cls == 1) & (bins[:nq] == 0), key, zero).min().reshape(1)
        D.allreduce_confidence_tables(ht, hf, zero)
        if self._files == 0:
            z = int(zero.item())
            if z != NO_ZERO_ROW:
                self.zero_negative = bool(z & 1)
        self._files += 1
        self.add_histograms(ht.cpu().numpy(), hf.cpu().numpy(), annotations)

    def add_histograms(self, hist_true: np.ndarray, hist_false: np.ndarray, annotations: Sequence[str]) -> None:
        for j, name in enumerate(annotations):
            if hist_true[j].any() or hist_false[j].any():
                i = self._names.setdefault(str(name), len(self._names))
                if i == len(self._t):
                    self._t.append(np.zeros(NBINS, np.int64))
                    self._f.append(np.zeros(NBINS, np.int64))
                self._t[i] += hist_true[j]
                self._f[i] += hist_false[j]

    def add_scores_csv(self, path: str) -> None:
        """A seq-annotation-scores CSV exactly as the reference reads it (read_and_transform_input_data,
        learn.smk:964-970): pandas' C parser — its default float converter is not round-trip exact (about a third of
        17-digit values come back one ulp off), and exact ties / bin edges depend on it."""
        import pandas as pd

        frame = pd.read_csv(path, index_col=INDEX_COL, header=0, engine="c")
        S = np.ascontiguousarray(frame.values, dtype=np.float64)
        self.add(top2_rows(torch.from_numpy(S).to(E._require_cuda())), [str(x) for x in frame.index], [str(c) for c in frame.columns])

    def finalize(self, prior: Optional[Dict[str, np.ndarray]] = None, modifier: float = 1.0) -> EvalResult:
        rows = sorted(self._names)
        T = np.array([self._t[self._names[r]] for r in rows], dtype=np.float64).reshape(len(rows), NBINS)
        F = np.array([self._f[self._names[r]] for r in rows], dtype=np.float64).reshape(len(rows), NBINS)
        with np.errstate(invalid="ignore", divide="ignore"):
            ratio = T / (T + F)                                         # generate_global_crosstab
            tt, ff = T.sum(axis=0), F.sum(axis=0)                       # calculate_distributions
            conf = _interpolate_linear(tt / (tt + ff))                  # compute_ratio_distribution
        sum_series = tt + ff
        weight = float(T.sum() + F.sum())
        out_w, out_sum = np.full(NBINS, weight), sum_series
        w_int = s_int = self._files == 1
        if prior is not None:
            w_int = w_int and bool(prior.get("weight_is_int", False))
            s_int = s_int and bool(prior.get("sum_is_int", False))
        if prior is not None:                                           # check_confidence_merge
            pw = np.asarray(prior["weight"], dtype=np.float64)
            k_factor = 1 + modifier * (weight / (weight + pw))
            out_w = pw + weight
            weighted_current = k_factor * weight
            total_weight = pw + weighted_current
            conf = (np.asarray(prior["confidence"], np.float64) * pw + conf * weighted_current) / total_weight
            out_sum = sum_series + np.asarray(prior["sum"], np.float64)
        return EvalResult(rows, ratio, conf, out_w, out_sum, self.zero_negative, w_int, s_int)


def _interpolate_linear(y: np.ndarray) -> np.ndarray:
    """Series.interpolate(method="linear") over equally spaced bins: gaps filled linearly, the tail repeats the
    last value, leading NaNs stay."""
    y = np.asarray(y, dtype=np.float64).copy()
    ok = np.flatnonzero(~np.isnan(y))
    if ok.size:
        x = np.arange(len(y), dtype=np.float64)
        m = x >= ok[0]
        y[m] = np.interp(x[m], ok.astype(np.float64), y[ok])
    return y


def read_global_confidence(path: str) -> Dict[str, np.ndarray]:
    """global-confidence-scores.csv (Difference, confidence, weight, sum; 101 rows) as the reference reads its
    prior (``pd.read_csv(..., index_col="Difference")``, learn.smk:1264-1266): same parser, same integer / float
    column typing."""
    import pandas as pd

    t = pd.read_csv(path, index_col="Difference")
    return {"Difference": t.index.to_numpy(dtype=np.float64), "confidence": t["confidence"].to_numpy(dtype=np.float64),
            "weight": t["weight"].to_numpy(dtype=np.float64), "sum": t["sum"].to_numpy(dtype=np.float64),
            "weight_is_int": t["weight"].dtype.kind in "iu", "sum_is_int": t["sum"].dtype.kind in "iu"}


def _num(v: float, as_int: bool = False) -> str:
    if np.isnan(v):
        return ""
    return str(int(v)) if as_int else repr(float(v))


def write_global_confidence(path: str, r: EvalResult) -> None:
    """``ratio_total_dist.to_csv`` (learn.smk:1314): index Difference, float repr, empty for NaN."""
    with open(path, "w", newline="") as f:
        f.write("Difference,confidence,weight,sum\n")
        for lab, c, w, s in zip(r.labels(), r.confidence, r.weight, r.sum):
            f.write(f"{lab!r},{_num(c)},{_num(w, r.weight_is_int)},{_num(s, r.sum_is_int)}\n")


def write_confidence_matrix(path: str, r: EvalResult) -> None:
    """confidence-matrix.csv as pyarrow writes the crosstab ratio (learn.smk:1315-1316): one column per
    Difference value, the Prediction index last, empty cells for 0 / 0."""
    import pyarrow as pa
    from pyarrow import csv as pacsv

    cols = {str(lab): pa.array(r.ratio[:, j], from_pandas=True) for j, lab in enumerate(r.labels())}
    cols["Prediction"] = pa.array(r.rows, type=pa.string())
    pacsv.write_csv(pa.table(cols), path)


class Evaluator:
    """Same constructor and ``execute_all`` as the reference's class (learn.smk:926-1340)."""

    def __init__(self, input_data, output_conf_path, output_glob_path, confidence_data=None, modifier: float = 1.0):
        self.input_data = list(input_data)
        self.confidence_data = list(confidence_data) if confidence_data else []
        self.output_conf = output_conf_path
        self.output_glob = output_glob_path
        self.modifier = modifier
        self.result: Optional[EvalResult] = None

    def execute_all(self) -> EvalResult:
        acc = ConfidenceAccumulator()
        for f in self.input_data:
            acc.add_scores_csv(str(f))
        prior = None
        if len(self.confidence_data) == 1:
            prior = read_global_confidence(str(self.confidence_data[0]))
        else:
            print("Base confidence file not found. Only one file is allowed in base/confidence.")
        self.result = acc.finalize(prior, self.modifier)
        write_global_confidence(self.output_glob, self.result)
        write_confidence_matrix(self.output_conf, self.result)
        return self.result
