"""CPU: the calibration restatements (oracle/score_adjoint.py, oracle/forcing_adjoint.py, oracle/score_gradients.py) on
the configurations the GPU's calibration builds are compared with in test_calibration_switches_gpu.py: pre-normalised
smoothing, every loss and packing switch off (with and without dynamics), NaN wind where it does not kill the cell,
NaN and inf concentration (day 0 included) and inf precipitation.  The adjoints hold the dot-product identity with the
forward tangents, the tangents agree with central differences, and a switched-off term gives exact zeros."""
import dataclasses

import numpy as np
import pytest

from oracle import forcing_adjoint as FA
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_adjoint as A
from oracle import score_gradients as G
from test_score_adjoint_cpu import DX, make_case as adj_case, objective_tangent
from test_score_gradients_cpu import RTOL, STEP, kinks, point_obs, season, values

NAMES = FA.FIELDS
NAN_WIND = (2, slice(5, 8), slice(6, 10))          # day, rows, cols: ocean cells of the 20 x 26 disc
NAN_CONC = (4, slice(8, 10), slice(12, 15))
NAN_CONC0 = (0, slice(10, 12), slice(6, 9))
INF_CONC = (3, slice(11, 13), slice(16, 18))
INF_PRECIP = (5, 9, 11)

CASES = {
    "pre_normalised": dict(f={"conv_variant": "pre_normalised"}),
    "budget_only": dict(f={"windpackInc": 0, "leadlossInc": 0, "atmlossInc": 0}),
    "all_off": dict(f={"windpackInc": 0, "leadlossInc": 0, "atmlossInc": 0, "dynamicsInc": 0}),
    "nan_wind_no_lead_no_atm": dict(f={"leadlossInc": 0, "atmlossInc": 0}, nan_wind=True),
    "nonfinite_conc": dict(f={}, conc=True),
    "inf_precip": dict(f={}, inf_precip=True),
}


def make_case(name, T=8, seed=3):
    """test_score_adjoint_cpu's "disc_land_ic" case with the switches and non-finite forcing of ``CASES[name]``."""
    c = CASES[name]
    mask, forcing, ic, p, f, obs, fps, w, fw = adj_case("disc_land_ic", T, seed)
    f = dataclasses.replace(f, **c["f"])
    if c.get("nan_wind"):
        forcing["wind"][NAN_WIND] = np.nan
    if c.get("conc"):
        forcing["conc"][NAN_CONC] = np.nan
        forcing["conc"][NAN_CONC0] = np.nan
        forcing["conc"][INF_CONC] = np.inf
    if c.get("inf_precip"):
        forcing["precip"][INF_PRECIP] = np.inf
    return mask, forcing, ic, p, f, obs, fps, w, fw


def patch_cells(mask, patch):
    cells = np.zeros(mask.shape, dtype=bool)
    cells[patch[1:]] = True
    return cells


def directions(forcing, seed=11):
    """Random forcing directions, 0 where the forcing is not finite (test_forcing_adjoint_cpu.directions scaled by
    the spread of the finite values, which inf would make NaN)."""
    rng = np.random.default_rng(seed)
    out = []
    for n in NAMES:
        fin = np.isfinite(forcing[n])
        d = rng.standard_normal(forcing[n].shape) * np.std(forcing[n][fin])
        out.append(np.where(fin, d, 0.0))
    return out


def identity(forcing, ic, mask, p, f, obs, fps, w, fw):
    got = FA.score_adjoint_forcing(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    d = directions(forcing)
    lhs = float(sum(np.sum(got[n + "_day_grad"] * d[i]) for i, n in enumerate(NAMES)))
    rhs = FA.objective_tangent_forcing(forcing, ic, mask, DX, p, f, obs, fps, w, fw, *d)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs), 1e-300), (lhs, rhs)
    return got


@pytest.mark.parametrize("name", list(CASES))
def test_dot_product_identity(name):
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case(name)
    ocean = R.ocean(mask)
    # the initial condition and the parameters (score_adjoint against the IC- and parameter-seeded tangents)
    theta, icg, _ = A.score_adjoint(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    rng = np.random.default_rng(7)
    v = rng.standard_normal(mask.shape)
    e = rng.standard_normal(G.DIRS)
    d_ic, d_th = objective_tangent(forcing, ic, mask, p, f, obs, fps, w, fw, v)
    lhs = float(np.sum(icg * v) + theta @ e)
    rhs = float(d_ic + d_th @ e)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs), 1e-300), (lhs, rhs)
    assert np.allclose(theta, d_th, rtol=1e-12, atol=1e-12 * np.abs(d_th).max())
    assert np.isfinite(icg).all() and np.abs(icg).max() > 0
    # the forcing
    got = identity(forcing, ic, mask, p, f, obs, fps, w, fw)
    assert np.array_equal(got["theta_grad"], theta) and np.array_equal(got["ic_grad"], icg)
    for n in NAMES:
        assert np.isfinite(got[n + "_day_grad"]).all() and np.isfinite(got["forcing_scale_grad"]).all()
    assert np.abs(got["precip_day_grad"]).max() > 0 and np.abs(got["conc_day_grad"]).max() > 0
    if f.leadlossInc == 0 and f.atmlossInc == 0:
        assert not got["wind_day_grad"].any() and not got["forcing_scale_grad"][1].any()
        assert got["forcing_scale_total"][1] == 0.0
    else:
        assert np.abs(got["wind_day_grad"]).max() > 0
    for j, sw in enumerate(("windpackInc", "leadlossInc", "atmlossInc")):
        assert (theta[j] == 0.0) == (getattr(f, sw) == 0), (j, theta)
    c = CASES[name]
    if c.get("nan_wind"):
        x, cells = NAN_WIND[0], patch_cells(mask, NAN_WIND)
        assert ocean[cells].all()
        # NaN wind gives windT = 0: wind packing stays finite, and only the lead loss (NaN * 0) kills the cell
        rec = A.run_season_record(forcing, ic, mask, DX, p, f)[1]
        lead_on = A.run_season_record(forcing, ic, mask, DX, p, dataclasses.replace(f, leadlossInc=1))[1]
        assert not rec[x][0][cells].any() and lead_on[x][0][cells].all()
        assert np.abs(got["precip_day_grad"][x][cells]).max() > 0
    if c.get("conc"):
        for patch in (NAN_CONC, NAN_CONC0, INF_CONC):
            x, cells = patch[0], patch_cells(mask, patch)
            assert ocean[cells].all()
            rec = A.run_season_record(forcing, ic, mask, DX, p, f)[1]
            assert rec[x][0][cells].all()                     # the new h0 is not finite: killed
            assert not got["precip_day_grad"][x][cells].any()
        # NaN < minConc is false: the IC is kept under NaN concentration on day 0
        assert np.abs(icg[patch_cells(mask, NAN_CONC0)]).max() > 0
    if c.get("inf_precip"):
        x, r, cc = INF_PRECIP
        assert ocean[r, cc] and not got["precip_day_grad"][x, r, cc]
        assert np.isfinite(got["forcing_scale_total"]).all()


def test_pre_normalised_tangents_match_central_differences():
    mask, forcing, ic = season()
    dx, T = 100000, forcing["precip"].shape[0]
    f = O.Flags(atmlossInc=1, conv_variant="pre_normalised")
    p = O.Params(windPackFactor=5.8e-7, windPackThresh=4.0, leadLossFactor=2.9e-7, atmLossFactor=2.2e-8)
    obs = point_obs(mask, T, np.random.default_rng(2))
    s, tan = G.run_season_tangent(forcing, ic, mask, dx, p, f)
    ref, v = values(forcing, ic, mask, dx, p, f, obs)
    assert np.array_equal(s["snowDepths"], ref["snowDepths"], equal_nan=True)
    post = O.run_season(forcing, ic, mask, dx, p, O.Flags(atmlossInc=1))
    assert not np.array_equal(post["snowDepths"], ref["snowDepths"], equal_nan=True)    # the variants differ
    dv = G.model_tangents(s["snowDepths"], tan, forcing["conc"], obs, mask, p)
    chi2_grad = G.score_gradients(v, dv, obs, mask)
    for j, name in enumerate(G.PARAM_FIELDS):
        h = STEP * getattr(p, name)
        sp, vp = values(forcing, ic, mask, dx, dataclasses.replace(p, **{name: getattr(p, name) + h}), f, obs)
        sm, vm = values(forcing, ic, mask, dx, dataclasses.replace(p, **{name: getattr(p, name) - h}), f, obs)
        for a, b, c in zip(kinks(s, p), kinks(sp, p), kinks(sm, p)):
            assert np.array_equal(a, b) and np.array_equal(a, c), name
        fd = (vp - vm) / (2 * h)
        ok = np.isfinite(v)
        assert ok.sum() > 100 and np.array_equal(np.isfinite(dv[j]), ok)
        scale = np.abs(fd[ok]).max()
        assert scale > 0, name
        assert np.allclose(dv[j][ok], fd[ok], rtol=RTOL, atol=RTOL * scale), name
        fd_chi2 = (R.scores(vp, obs, mask)[0] - R.scores(vm, obs, mask)[0]) / (2 * h)
        assert np.allclose(chi2_grad[:, j], fd_chi2, rtol=RTOL, atol=RTOL * np.abs(fd_chi2).max()), name


@pytest.mark.parametrize("off", [("windpackInc",), ("leadlossInc",), ("atmlossInc",), ("leadlossInc", "atmlossInc"),
                                 ("windpackInc", "leadlossInc", "atmlossInc")])
def test_switched_off_terms_have_exact_zeros(off):
    """A disabled parameter's theta_grad component, d chi2 column and Jacobian row are exactly 0, the enabled ones
    are not; with lead and atm loss off the wind derivatives are exactly 0."""
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case("pre_normalised")
    f = dataclasses.replace(f, **{k: 0 for k in off})
    cols = [j for j, sw in enumerate(("windpackInc", "leadlossInc", "atmlossInc")) if sw in off]
    on = [j for j in range(G.DIRS) if j not in cols]
    s, tan = G.run_season_tangent(forcing, ic, mask, DX, p, f)
    v = R.model_values(s["snowDepths"], s["density"], forcing["conc"], obs, mask)
    dv = G.model_tangents(s["snowDepths"], tan, forcing["conc"], obs, mask, p)
    grad = G.score_gradients(v, dv, obs, mask)
    mean, dmean = G.footprint_tangents(s["snowDepths"], s["density"], tan, forcing["conc"], fps, mask, p)
    fgrad = G.footprint_gradients(mean, dmean, fps)
    got = FA.score_adjoint_forcing(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    fin = np.isfinite(v)
    for j in cols:
        assert not tan[:, j].any() and not grad[:, j].any() and not fgrad[:, j].any(), j
        assert not dv[j][fin].any() and np.array_equal(np.isfinite(dv[j]), fin), j
        assert not np.nan_to_num(dmean[j]).any() and got["theta_grad"][j] == 0.0, j
    for j in on:
        assert np.abs(grad[:, j]).max() > 0 and np.abs(dv[j][fin]).max() > 0 and got["theta_grad"][j] != 0.0, j
    if "leadlossInc" in off and "atmlossInc" in off:
        assert not got["wind_day_grad"].any() and not got["forcing_scale_grad"][1].any()
        assert got["forcing_scale_total"][1] == 0.0
    else:
        assert np.abs(got["wind_day_grad"]).max() > 0
