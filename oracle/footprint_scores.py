"""Plain float64 restatement of the footprint observations (``footprint_mean_kernel`` and the footprint stage of
``misfit_finish_kernel`` in nesosim_abi.cu, DESIGN.md §4.2), down to the order of every addition, so that the GPU's
footprint means and fp_chi2 can be compared bit for bit.  The point operators and the 256-thread sum are those of
``observation_scores``.

A footprint is a weighted set of (day, row, col) points of one kind.  Its points on land or lake cells are dropped at
registration; the kept point j (input order) belongs to lane j % 32 of one warp, which adds w*v to sw and w to s, in
order from 0.0, where the point's model value v is finite; lane 0 collects both with a[l] += a[l + off] for off = 16,
8, 4, 2, 1, and the mean is sw / s (NaN when no point was finite).  Per kind, over a season's footprints of that kind in
input order, fp_chi2 is the ``fixed_order_sum`` of the finite ((mean - value)/sigma)^2 and fp_count their number.
"""
import numpy as np

from .observation_scores import KINDS, WARP, fixed_order_sum, model_values, ocean


def footprint_values(snowDepths, density, conc, fps, mask):
    """The model value of every footprint of one member's season (``fps``: dict of kind, value, sigma per footprint,
    begin [n_fp+1] and day, row, col, weight per point; ``ensemble.normalize_footprints``), restating
    ``footprint_mean_kernel``: the points on ocean cells, in input order, point j to lane j % 32, which adds w*v to sw and
    w to s in order from 0.0 where v is finite; then lane l += lane l + off for off = 16, 8, 4, 2, 1; mean = sw / s
    (NaN when no point was finite, all points on land included)."""
    begin = np.asarray(fps["begin"], dtype=np.int64)
    kind = np.repeat(np.asarray(fps["kind"]), np.diff(begin))
    pts = {"day": fps["day"], "row": fps["row"], "col": fps["col"], "kind": kind}
    v = model_values(snowDepths, density, conc, pts, mask)
    w = np.asarray(fps["weight"], dtype=np.float64)
    kept = ocean(mask)[np.asarray(fps["row"]), np.asarray(fps["col"])]
    out = np.empty(len(begin) - 1)
    for g in range(len(out)):
        sel = np.arange(begin[g], begin[g + 1])
        sel = sel[kept[sel]]
        rows = -(-len(sel) // WARP) * WARP
        vv, ww = np.full(rows, np.nan), np.ones(rows)
        vv[:len(sel)], ww[:len(sel)] = v[sel], w[sel]
        sw, s = np.zeros(WARP), np.zeros(WARP)
        with np.errstate(all="ignore"):
            for vr, wr in zip(vv.reshape(-1, WARP), ww.reshape(-1, WARP)):   # round i: lane l takes point i*32 + l
                ok = np.isfinite(vr)
                sw = np.where(ok, sw + wr * vr, sw)
                s = np.where(ok, s + wr, s)
            off = WARP // 2
            while off:
                sw = sw[:off] + sw[off:2 * off]
                s = s[:off] + s[off:2 * off]
                off //= 2
            out[g] = sw[0] / s[0]
    return out


def footprint_scores(fp_model, fps):
    """(fp_chi2[KINDS], fp_count[KINDS]) of one member: per kind, over its footprints in input order, the finite
    ((model - value)/sigma)^2 summed with ``fixed_order_sum``."""
    kind = np.asarray(fps["kind"])
    with np.errstate(all="ignore"):
        r = (np.asarray(fp_model) - np.asarray(fps["value"], dtype=np.float64)) / np.asarray(fps["sigma"])
        sq = r * r
    ok = np.isfinite(r)
    chi2 = np.zeros(KINDS)
    used = np.zeros(KINDS, dtype=np.int64)
    for k in range(KINDS):
        sel = kind == k
        with np.errstate(over="ignore"):
            chi2[k] = fixed_order_sum(np.where(ok[sel], sq[sel], 0.0))
        used[k] = ok[sel].sum()
    return chi2, used
