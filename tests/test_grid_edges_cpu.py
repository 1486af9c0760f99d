"""CPU: the restatements (oracle/score_adjoint.py, oracle/score_gradients.py, oracle/forcing_adjoint.py) on forcing with
ice and finite drift up to the grid edge, where np.gradient takes one-sided differences with divisor dx: the IC/theta
and forcing dot-product identities to 1e-12 and ic_grad against central differences at corner and edge cells.  The
forcing helper (``edge_season``), the observations and the grids are the ones tests/test_grid_edges_gpu.py holds the
kernels to, so these tests keep the reference honest on exactly those shapes."""
import functools

import numpy as np
import pytest
from scipy.ndimage import gaussian_filter

from nesosim_b200 import ensemble as ENS
from nesosim_b200 import synthetic as S
from oracle import footprint_scores as F
from oracle import forcing_adjoint as FA
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_adjoint as A
from oracle import score_gradients as G
from test_general_scores_gpu import DENSITY, DEPTH, VOLUME, cat_footprints, make_footprints, make_obs, one, oracle_params

W, FW = (1.0, 0.5, 2.0), (0.25, 1.0, 0.0)    # test_score_adjoint_gpu's weights: not all one
FLAGS = O.Flags(atmlossInc=1)
FLAVOURS = ("land_nan", "land_finite")       # drift NaN over land (as real products) or finite there too


def all_ocean(shape):
    return np.full(shape, 8, dtype=np.uint8)


def coast(shape):
    """Ocean (codes 8 and 9) with a land block across the tile corner at row 16 / column 32 (tiles are 32 x 16), a
    coast strip across the row-tile boundary at 16, a lake by the bottom edge, the upper half of the first column land
    (an edge partly land) and the grid's last tile cell land where that tile is ragged."""
    ny, nx = shape
    m = np.full(shape, 8, dtype=np.uint8)
    m[:, nx // 2:] = 9
    m[14:19, 28:37] = 11
    m[12:min(20, ny - 1), nx // 2 - 3:nx // 2 + 2] = 12
    m[ny - 3:ny - 1, 5:9] = 0
    m[:ny // 2, 0] = 11
    if ny % 16 and nx % 32:
        m[16 * (ny // 16):, 32 * (nx // 32):] = 11
    return m


# name: (mask, dx, days).  33 = 2*16+1 and 65 = 2*32+1 put the grid edge one cell into a tile; 34 and 66 put it exactly
# at the bound of the day kernel's `interior` test; 32 x 64 ends on a tile boundary; 97 and 98 = 3*32 + 1, + 2.
GRIDS = {
    "ocean_2x2": (lambda: all_ocean((2, 2)), 100000, 8),
    "ocean_2x7": (lambda: all_ocean((2, 7)), 100000, 8),
    "ocean_7x2": (lambda: all_ocean((7, 2)), 100000, 8),
    "ocean_3x3": (lambda: all_ocean((3, 3)), 100000, 8),
    "coast_33x65": (lambda: coast((33, 65)), 50000, 7),
    "coast_34x66": (lambda: coast((34, 66)), 50000, 7),
    "coast_32x64": (lambda: coast((32, 64)), 50000, 7),
    "coast_17x97": (lambda: coast((17, 97)), 50000, 6),
    "coast_50x98": (lambda: coast((50, 98)), 50000, 6),
    "100km": (lambda: S.region_mask(dx=100000), 100000, 8),
    "25km": (lambda: S.region_mask(dx=25000), 25000, 4),
}
CPU_GRIDS = [g for g in GRIDS if g not in ("100km", "25km")]


def land_ic(mask, ic):
    return np.where(R.ocean(mask), ic, 0.3)               # finite IC on land: day 0's dynamics read it


def _unit(a):
    return (a - a.min()) / max(a.max() - a.min(), 1e-12)


def edge_season(mask, T, seed, drift_over_land):
    """(forcing, ic): ``make_season`` with ice (conc in [0.3, 1]) on every ocean cell, an open-water patch (conc 0.05 <
    minConc) on the top edge on days 1-2, smooth finite drift on every ocean cell (and on land if ``drift_over_land``)
    with one missing-drift day and a NaN strip on the upper half of the last column on day 1, finite snowfall but for
    one NaN corner day, wind exactly 5.0 on edge cells; the IC finite on every ocean cell and, where conc[0] >= minConc
    keeps it, on land."""
    mask = np.asarray(mask)
    ny, nx = mask.shape
    f = S.make_season(mask, T, seed=seed)
    rng = np.random.default_rng(seed + 1)
    wet = R.ocean(mask)
    sig = max(1.0, ny / 20.0)

    conc = 0.3 + 0.7 * _unit(gaussian_filter(rng.random((T, ny, nx)), (0, sig, sig), mode="nearest"))
    conc[1:3, :max(1, ny // 6), nx // 3:nx // 3 + max(1, nx // 5)] = 0.05
    conc[:, ~wet] = 0.0
    conc[0][~wet] = 0.9                                   # keeps the IC on land (conc[0] >= minConc)
    f["conc"] = conc

    yy, xx = np.mgrid[0:ny, 0:nx]
    trend = (0.03 * (xx / max(nx - 1, 1) - 0.5), 0.03 * (yy / max(ny - 1, 1) - 0.5))
    drift = np.empty((T, 2, ny, nx))
    for t in range(T):
        for c in range(2):
            g = gaussian_filter(rng.standard_normal((ny, nx)), sig, mode="nearest")
            drift[t, c] = 0.1 * g / max(g.std(), 1e-12) + trend[c]
    if not drift_over_land:
        drift[:, :, ~wet] = np.nan
    drift[min(3, T - 2)] = np.nan                         # a whole missing-drift day
    drift[1, :, :max(1, ny // 2), nx - 1] = np.nan        # a NaN strip along the last column: mixed finite bits there
    f["drift"] = drift

    f["precip"] = rng.gamma(0.5, 2.0, size=(T, ny, nx))
    f["precip"][T - 2, ny - 1, nx - 1] = np.nan           # one NaN corner day
    f["wind"][1, 0, ::2] = 5.0
    f["wind"][2, ::2, nx - 1] = 5.0
    f["wind"][0, ny - 1, 1::3] = 5.0

    ic = land_ic(mask, 0.02 + 0.08 * _unit(gaussian_filter(rng.random((ny, nx)), sig, mode="nearest")))
    return f, ic


def edge_cells(mask):
    """Every corner and up to five cells along each edge."""
    ny, nx = mask.shape
    cols, rows = np.unique(np.linspace(0, nx - 1, 5).astype(int)), np.unique(np.linspace(0, ny - 1, 5).astype(int))
    cells = [(0, c) for c in cols] + [(ny - 1, c) for c in cols] + [(r, 0) for r in rows] + [(r, nx - 1) for r in rows]
    return sorted(set(cells))


def edge_obs(mask, T, rng, n=400):
    """``make_obs`` plus every kind on every cell of ``edge_cells`` on two days (density from day 1 on)."""
    obs = make_obs(mask, T, rng, n)
    cells = np.array(edge_cells(mask))
    kind = np.tile(np.repeat(np.arange(R.KINDS), 2), len(cells))
    rc = np.repeat(cells, 2 * R.KINDS, axis=0)
    day = np.where(np.arange(len(kind)) % 2, T - 1, rng.integers(1, T, len(kind)))
    value = np.where(kind == DENSITY, 250.0 + 50.0 * rng.random(len(kind)), 0.2 * rng.random(len(kind)))
    sigma = np.where(kind == DENSITY, 30.0, 0.05)
    extra = {"day": day, "row": rc[:, 0], "col": rc[:, 1], "value": value, "kind": kind, "sigma": sigma}
    return {k: np.concatenate([np.asarray(obs[k]), np.asarray(extra[k])]) for k in obs}


def edge_footprints(mask, T, rng):
    """``make_footprints`` (on grids with land; regional means and a one-point footprint on all-ocean grids), a depth
    footprint over the whole top row and a volume footprint down the last column."""
    ny, nx = mask.shape
    if (~R.ocean(mask)).any():
        parts = [make_footprints(mask, T, rng)]
    else:
        codes = [k for k in range(1, 11) if (mask == k).any()]
        parts = [ENS.region_footprints(mask, codes, [(1, T // 2), (T // 2, T)], DEPTH, [0.2, 0.25], 0.05),
                 ENS.region_footprints(mask, codes, [(1, T)], DENSITY, 300.0, 30.0),
                 one(VOLUME, 0.1, [T - 1], [ny - 1], [0])]
    parts.append(one(DEPTH, 0.12, np.full(nx, T // 2), np.zeros(nx, np.int64), np.arange(nx), 2.0 ** rng.uniform(-2, 2, nx)))
    parts.append(one(VOLUME, 0.1, 1 + np.arange(ny) % (T - 1), np.arange(ny), np.full(ny, nx - 1)))
    return cat_footprints(parts)


@functools.lru_cache(maxsize=None)
def edge_case(grid, flavour, M=2, seed=0):
    """(mask, dx, T, forcing, ic (M, ny, nx), params (M, 4), obs, fps) of one grid and drift flavour."""
    make, dx, T = GRIDS[grid]
    mask = make()
    seed = seed + 10 * list(GRIDS).index(grid) + 1000 * FLAVOURS.index(flavour)
    rng = np.random.default_rng(seed)
    forcing, ic = edge_season(mask, T, seed + 1, flavour == "land_finite")
    ic = ic[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=seed + 2)
    return mask, dx, T, forcing, ic, params, edge_obs(mask, T, rng), edge_footprints(mask, T, rng)


def edges(shape):
    """Boolean masks of the four grid edges: first row, last row, first column, last column."""
    out = []
    for axis, idx in ((0, 0), (0, -1), (1, 0), (1, -1)):
        e = np.zeros(shape, dtype=bool)
        if axis == 0:
            e[idx, :] = True
        else:
            e[:, idx] = True
        out.append(e)
    return out


# --------------------------------------------------------------------------------------------------------- the tests

@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("grid", list(GRIDS))
def test_the_edge_code_runs(grid, flavour):
    """On every grid edge an ocean cell has finite raw adv and div terms (the record build's finite bits) on some day,
    and ic_grad is nonzero: the one-sided differences compute finite values there, not zeros."""
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, flavour)
    p = oracle_params(params[0])
    _, rec = A.run_season_record(forcing, ic[0], mask, dx, p, FLAGS)
    _, icg, _ = A.score_adjoint(forcing, ic[0], mask, dx, p, FLAGS, obs, fps, W, FW)
    wet = R.ocean(mask)
    for e in edges(mask.shape):
        if not (e & wet).any():                           # the bundled masks' last column is land
            continue
        fin = [(fa & fd)[:, e & wet].any() for _, _, fa, fd in rec]
        assert any(fin), fin
        assert np.abs(icg[e & wet]).max() > 0
    assert sum((e & wet).any() for e in edges(mask.shape)) >= 3
    if wet[:, -1].all():                                  # the NaN strip leaves the last column's finite bits mixed
        fa = rec[1][2][:, :, -1]
        assert fa.any() and not fa.all()

def objective_tangent(forcing, ic, mask, dx, p, f, obs, fps, v):
    """dJ along the IC direction v, and per parameter (forward mode of score_gradients)."""
    s, tan = A.run_season_tangent_ic(forcing, ic, v, mask, dx, p, f)
    tan3 = np.repeat(tan[:, None], G.DIRS, axis=1)
    _, ptan = G.run_season_tangent(forcing, ic, mask, dx, p, f)
    out = []
    for t in (tan3, ptan):
        mv = R.model_values(s["snowDepths"], s["density"], forcing["conc"], obs, mask)
        dv = G.model_tangents(s["snowDepths"], t, forcing["conc"], obs, mask, p)
        mean, dmean = G.footprint_tangents(s["snowDepths"], s["density"], t, forcing["conc"], fps, mask, p)
        out.append(np.asarray(W) @ G.score_gradients(mv, dv, obs, mask) + np.asarray(FW) @ G.footprint_gradients(mean, dmean, fps))
    return out[0][0], out[1]


@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("grid", CPU_GRIDS)
def test_ic_and_theta_dot_product_identity(grid, flavour):
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, flavour)
    p = oracle_params(params[0])
    theta, icg, _ = A.score_adjoint(forcing, ic[0], mask, dx, p, FLAGS, obs, fps, W, FW)
    for e in edges(mask.shape):
        assert np.abs(icg[e & R.ocean(mask)]).max() > 0
    rng = np.random.default_rng(7)
    v = rng.standard_normal(mask.shape)
    e = rng.standard_normal(G.DIRS)
    d_ic, d_th = objective_tangent(forcing, ic[0], mask, dx, p, FLAGS, obs, fps, v)
    lhs = float(np.sum(icg * v) + theta @ e)
    rhs = float(d_ic + d_th @ e)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs), 1e-300), (lhs, rhs)
    assert np.allclose(theta, d_th, rtol=1e-12, atol=1e-12 * np.abs(d_th).max())


def directions(forcing, seed=11):
    rng = np.random.default_rng(seed)
    out = []
    for n in FA.FIELDS:
        d = rng.standard_normal(forcing[n].shape) * np.nanstd(forcing[n])
        out.append(np.where(np.isfinite(forcing[n]), d, 0.0))
    return out


@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("grid", CPU_GRIDS)
def test_forcing_dot_product_identity(grid, flavour):
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, flavour)
    p = oracle_params(params[1])
    got = FA.score_adjoint_forcing(forcing, ic[1], mask, dx, p, FLAGS, obs, fps, W, FW)
    d = directions(forcing)
    lhs = float(sum(np.sum(got[n + "_day_grad"] * d[i]) for i, n in enumerate(FA.FIELDS)))
    rhs = FA.objective_tangent_forcing(forcing, ic[1], mask, dx, p, FLAGS, obs, fps, W, FW, *d)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs), 1e-300), (lhs, rhs)
    wet = R.ocean(mask)
    for n in FA.FIELDS:
        g = got[n + "_day_grad"]
        assert np.isfinite(g).all() and all(np.abs(g[:, e & wet]).max() > 0 for e in edges(mask.shape)), n


def objective(forcing, ic, mask, dx, p, obs, fps):
    st = O.run_season(forcing, ic, mask, dx, p, FLAGS)
    mv = R.model_values(st["snowDepths"], st["density"], forcing["conc"], obs, mask)
    chi2, used = R.scores(mv, obs, mask)
    fm = F.footprint_values(st["snowDepths"], st["density"], forcing["conc"], fps, mask)
    fchi2, fused = F.footprint_scores(fm, fps)
    kinks = (np.isnan(st["snowDepths"]), st["snowDepths"] == 0.0, used, fused)
    return float(np.dot(W, chi2) + np.dot(FW, fchi2)), kinks


@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("grid", CPU_GRIDS)
def test_ic_grad_matches_central_differences_on_the_edges(grid, flavour):
    """At every corner and edge cell of ``edge_cells`` that is ocean and carries a gradient, where the kink pattern
    (NaN and zero depths, counted observations) is the same on both sides of the step."""
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, flavour)
    obs = {k: v[obs["kind"] != DENSITY] for k, v in obs.items()}
    p = oracle_params(params[0])
    ic = ic[0]
    _, icg, _ = A.score_adjoint(forcing, ic, mask, dx, p, FLAGS, obs, fps, W, FW)
    _, base = objective(forcing, ic, mask, dx, p, obs, fps)
    scale = np.abs(icg).max()
    checked, corners = 0, 0
    ny, nx = mask.shape
    for r, c in edge_cells(mask):
        if not R.ocean(mask)[r, c] or abs(icg[r, c]) <= 1e-6 * scale:
            continue
        h = 1e-4 * max(abs(ic[r, c]), 1e-3)
        vals, ok = [], True
        for sg in (1, -1):
            q = ic.copy()
            q[r, c] += sg * h
            val, k = objective(forcing, q, mask, dx, p, obs, fps)
            ok = ok and all(np.array_equal(a, b) for a, b in zip(base, k))
            vals.append(val)
        if not ok:
            continue
        fd = (vals[0] - vals[1]) / (2 * h)
        assert np.isclose(icg[r, c], fd, rtol=1e-6, atol=1e-9 * scale), (r, c, icg[r, c], fd)
        checked += 1
        corners += r in (0, ny - 1) and c in (0, nx - 1)
    assert checked >= 4 and corners >= 1, (checked, corners)
