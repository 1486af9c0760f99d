"""Plain float64 restatement of the fused calibration scores (``misfit_finish_kernel`` in nesosim_abi.cu, DESIGN.md
§4.2), down to the order of every addition, so that the GPU's chi2 can be compared bit for bit.

For one member, the observations of its season are kept only where the cell is ocean (mask 1..10: land and lake
observations are dropped at registration) and ordered by a stable sort on (row*nx + col, day).  The native tables sort
by (owner, day) with owner = ocean_off[strip] + index in the strip's row-major ocean list; ocean_off grows with the
strip, so the owner is monotone in row*nx + col for every strip cut and the order does not depend on the cut.  Per kind,
in that order, with r = (model - value)/sigma and only finite r counted:

* observation i of the kind goes to thread i % 256, which adds r*r in order starting from 0.0 (an observation whose r is
  not finite keeps its place i and adds nothing);
* within each warp of 32 threads, lane 0 collects a[l] += a[l + off] for off = 16, 8, 4, 2, 1;
* chi2 = (((0.0 + warp[0]) + warp[1]) + ...) + warp[7]; used = the number of finite r.

Plain IEEE double everywhere, as the library is built with --fmad=false.
"""
import numpy as np

DEPTH, VOLUME, DENSITY, KINDS = 0, 1, 2, 3
THREADS, WARP = 256, 32


def ocean(mask):
    mask = np.asarray(mask)
    return (mask >= 1) & (mask <= 10)


def model_values(snowDepths, density, conc, obs, mask):
    """The model value of every observation from one member's season arrays (``snowDepths`` (T,2,ny,nx), ``density``
    (T,ny,nx), ``conc`` (T,ny,nx)): depth over ice (h0+h1)/conc[day], volume h0+h1, or density; NaN on land and lake."""
    d, r, c, k = (np.asarray(obs[n]) for n in ("day", "row", "col", "kind"))
    vol = snowDepths[d, 0, r, c] + snowDepths[d, 1, r, c]
    with np.errstate(all="ignore"):
        v = np.where(k == DEPTH, vol / conc[d, r, c], np.where(k == VOLUME, vol, density[d, r, c]))
    v[~ocean(mask)[r, c]] = np.nan
    return v


def order(obs, mask):
    """Indices of the observations on ocean cells in the order the library sums them: a stable sort on (cell, day)."""
    nx = np.asarray(mask).shape[1]
    r, c, d = (np.asarray(obs[n]).astype(np.int64) for n in ("row", "col", "day"))
    keep = np.flatnonzero(ocean(mask)[r, c])
    return keep[np.lexsort((d[keep], r[keep] * nx + c[keep]))]


def fixed_order_sum(terms):
    """The epilogue's sum of ``terms`` (one kind's r*r in summation order, 0.0 where r is not finite: adding 0.0 leaves
    a non-negative sum as it is): 256 thread sums, a shuffle tree per warp, then the warps one after the other."""
    terms = np.asarray(terms, dtype=np.float64)
    rows = np.zeros(-(-len(terms) // THREADS) * THREADS)
    rows[:len(terms)] = terms
    acc = np.zeros(THREADS)
    for row in rows.reshape(-1, THREADS):                     # round j: thread t adds term j*256 + t
        acc = acc + row
    warps = acc.reshape(THREADS // WARP, WARP)
    off = WARP // 2
    while off:
        warps = warps[:, :off] + warps[:, off:2 * off]
        off //= 2
    total = 0.0
    for w in warps[:, 0]:
        total += w
    return total


def scores(model, obs, mask):
    """(chi2[KINDS], used[KINDS]) of one member: ``model`` = the model value of every input observation
    (``model_values``), ``obs`` = dict of day, row, col, value, sigma, kind arrays."""
    idx = order(obs, mask)
    kind = np.asarray(obs["kind"])[idx]
    with np.errstate(all="ignore"):
        r = (np.asarray(model)[idx] - np.asarray(obs["value"], dtype=np.float64)[idx]) / np.asarray(obs["sigma"])[idx]
        sq = r * r
    ok = np.isfinite(r)
    chi2 = np.zeros(KINDS)
    used = np.zeros(KINDS, dtype=np.int64)
    for k in range(KINDS):
        sel = kind == k
        with np.errstate(over="ignore"):                      # a finite r whose square overflows: inf, as on the GPU
            chi2[k] = fixed_order_sum(np.where(ok[sel], sq[sel], 0.0))
        used[k] = ok[sel].sum()
    return chi2, used
