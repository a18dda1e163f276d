"""Host definition of LOFOutlierErrorDetector, written for clarity, not speed: the specification that
``dr_lof_flag`` reproduces bit for bit.

1. NULL cells take the median of the column's non-NULL values (``np.median``); -0.0 becomes +0.0.
2. Stable sort by (value, row position) -> s[0..n).
3. For sorted position i, the windows [l, l + k] with max(0, i - k) <= l <= min(i, n - 1 - k); the one
   minimising d(l) = max(s[i] - s[l], s[l + k] - s[i]) wins, the leftmost on ties.  kdist[i] = d(l*), the
   neighbours are the window without i.
4. scikit-learn's formulas (sklearn/neighbors/_lof.py) with the sums in ascending sorted position:
   reach(i, j) = max(|s[i] - s[j]|, kdist[j]),  lrd[i] = 1 / (sum_j reach(i, j) / k + 1e-10),
   lof[i] = (sum_j lrd[j] / lrd[i]) / k.
5. A cell is an error iff lof > 1.5 (``negative_outlier_factor_ < offset_`` with contamination="auto").
An all-NULL column, or one with fewer than 2 rows, is not scored.
"""
import numpy as np

LOF_K = 20
LOF_THRESHOLD = 1.5


def lof_scores_1d(values, k):
    """-> float64 scores in row order; all NaN when nothing is scored (n < 2 or every value NULL)."""
    v = np.array(values, dtype=np.float64)
    n = len(v)
    out = np.full(n, np.nan)
    null = np.isnan(v)
    if n < 2 or null.all():
        return out
    assert 1 <= k <= n - 1
    v[null] = np.median(v[~null])
    v[v == 0.0] = 0.0
    order = np.lexsort((np.arange(n), v))
    s = v[order]
    i = np.arange(n)
    lo = np.maximum(0, i - k)
    hi = np.minimum(i, n - 1 - k)
    kdist = np.full(n, np.inf)
    first = lo.copy()
    for o in range(k + 1):          # every candidate window, left to right; strict < keeps the leftmost
        l = np.minimum(lo + o, hi)
        d = np.maximum(s - s[l], s[l + k] - s)
        better = (lo + o <= hi) & (d < kdist)
        kdist = np.where(better, d, kdist)
        first = np.where(better, l, first)
    acc = np.zeros(n)
    for o in range(k + 1):
        j = first + o
        acc = np.where(j != i, acc + np.maximum(np.abs(s - s[j]), kdist[j]), acc)
    lrd = 1.0 / (acc / k + 1e-10)
    acc = np.zeros(n)
    for o in range(k + 1):
        j = first + o
        acc = np.where(j != i, acc + lrd[j] / lrd, acc)
    out[order] = acc / k
    return out


def lof_flags(values, k=LOF_K):
    """bool per row: flagged by the detector (k = min(k, n - 1))."""
    n = len(values)
    if n < 2:
        return np.zeros(n, dtype=bool)
    with np.errstate(invalid="ignore"):
        return lof_scores_1d(values, min(k, n - 1)) > LOF_THRESHOLD


def lof_cells(tbl, row_id, continuous, targets):
    """{(row position, attribute)} of an oracle table (``oracle.table.OTable``)."""
    out = set()
    for attr in [a for a in continuous if a in targets]:
        if attr not in tbl.cols:
            continue
        for r in np.nonzero(lof_flags(np.asarray(tbl.cols[attr], dtype=np.float64)))[0]:
            out.add((int(r), attr))
    return out


def with_lof(run_detectors):
    """The oracle's ``run_detectors`` extended with {"type": "lof"} specs."""
    def run(tbl, row_id, targets, detectors, continuous):
        lof = [d for d in detectors if d["type"] == "lof"]
        rest = [d for d in detectors if d["type"] != "lof"]
        cells = run_detectors(tbl, row_id, targets, rest, continuous) if rest or not detectors else set()
        target_attrs = [c for c in tbl.names if c != row_id and (not targets or c in set(targets))]
        for _ in lof[:1]:
            cells |= lof_cells(tbl, row_id, continuous, target_attrs)
        return cells
    return run
