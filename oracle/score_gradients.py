"""Plain float64 restatement of the calibration gradients (``nesosim_run_season_score_grads``: the GRAD builds of the
scoring day kernel, ``footprint_mean_kernel`` and ``misfit_finish_kernel`` in nesosim_b200/csrc, DESIGN.md §4.1), down to
the order of every operation, so that the GPU's tangents, Jacobian rows and gradients can be compared bit for bit.

Directions j = 0 windPackFactor, 1 leadLossFactor, 2 atmLossFactor (parameter-row columns 0, 2, 3).  The tangent state
is t[x] = d snowDepths[x] / d theta_j, shape (DIRS, 2, ny, nx); t[0] = 0.  The step x -> x+1 (``tangent_step``):

* raw dynamics: ``calc_dynamics``' stencils on t (the drift does not depend on theta), each term replaced by 0 where the
  primal raw term was not finite (``fill_mask_nan_zero`` made the primal a constant there);
* smoothing: ``convolve_fill0`` of each raw tangent plane (no NaN: the plain branch, same tap order), 0 on land;
* point terms: each primal term applied to t0, plus -- in the parameter's own direction only -- the primal term of h0
  with that parameter set to 1; a term whose switch is off is 0.0;
* new tangents t0 + wpl + lead + atm + adv0 + div0 and t1 + wpg + adv1 + div1 (left to right), set to 0 where the
  primal ``fill_nan_no_negative`` replaced the new depth (not finite, land, or the clamp of a negative value to 0).

Observation operators (``model_tangents``): depth (t0+t1)/conc, volume t0+t1, density ((t0*rhoF + t1*rhoO) - q*(t0+t1)) /
den from the primal quotient q = (h0*rhoF + h1*rhoO)/den, den = h0+h1, and 0 where a clamp changed q; NaN wherever the
model value is not finite.  d chi2/d theta_j of a kind is the ``fixed_order_sum`` of 2*r*(dv/sigma) over the terms chi2
counts; a footprint's derivative is the footprint lane order of w*dv over its points with finite v, over the primal s.
"""
import dataclasses

import numpy as np

from . import nesosim_oracle as O
from .footprint_scores import footprint_values
from .observation_scores import DENSITY, DEPTH, KINDS, VOLUME, WARP, fixed_order_sum, model_values, ocean, order

DIRS = 3
PARAM_FIELDS = ("windPackFactor", "leadLossFactor", "atmLossFactor")


def land(mask):
    mask = np.asarray(mask)
    return (mask > 10) | (mask < 1)


def raw_dynamics(drift, h, dx, p):
    """``calc_dynamics`` before ``fill_mask_nan_zero``: (adv, div), each (2, ny, nx)."""
    with np.errstate(all="ignore"):
        divx = h * np.gradient(drift[0] * p.deltaT, dx, axis=(1))
        divy = h * np.gradient(drift[1] * p.deltaT, dx, axis=(0))
        div = -(divx + divy)
        advx = drift[0] * p.deltaT * np.gradient(h, dx, axis=(2))
        advy = drift[1] * p.deltaT * np.gradient(h, dx, axis=(1))
        adv = -(advx + advy)
    return adv, div


def tangent_step(hx, tx, conc, precip, drift, wind, mask, dx, p, f):
    """The tangents of slot x+1 (DIRS, 2, ny, nx) from the primal depths ``hx`` (2, ny, nx) and tangents ``tx`` of slot
    x; the primal is recomputed here exactly as ``calc_budget`` forms it."""
    lnd = land(mask)
    zeros = lambda: np.zeros(conc.shape)
    with np.errstate(all="ignore"):
        acc = (precip / p.snowDensityFresh) * conc
        if f.dynamicsInc == 1:
            adv_r, div_r = raw_dynamics(drift, hx, dx, p)
            fin_a, fin_d = np.isfinite(adv_r), np.isfinite(div_r)
            adv, div = O.calc_dynamics(drift, hx, dx, p)
            adv = np.stack([O.smooth_snow(a, f.conv_variant) for a in adv])
            div = np.stack([O.smooth_snow(d, f.conv_variant) for d in div])
            for plane in (adv[0], adv[1], div[0], div[1]):
                O.fill_nan_no_negative(plane, mask, negative_to_zero=False)
        else:
            adv = np.zeros((2,) + conc.shape)
            div = np.zeros((2,) + conc.shape)
        lead = O.lead_loss(hx[0], wind, conc, p) if f.leadlossInc == 1 else zeros()
        atm = O.atm_loss(hx[0], wind, p) if f.atmlossInc == 1 else zeros()
        wpl, wpg, _ = O.wind_packing(wind, hx[0], p) if f.windpackInc == 1 else (zeros(), zeros(), zeros())
        h0n = hx[0] + acc + wpl + lead + atm + adv[0] + div[0]
        h1n = hx[1] + wpg + adv[1] + div[1]
        kill0 = ~np.isfinite(h0n) | lnd | (h0n < 0.)
        kill1 = ~np.isfinite(h1n) | lnd | (h1n < 0.)

        out = np.zeros_like(tx)
        for j in range(DIRS):
            t = tx[j]
            one = dataclasses.replace(p, **{PARAM_FIELDS[j]: 1.0})
            if f.dynamicsInc == 1:
                ta, td = raw_dynamics(drift, t, dx, p)
                ta, td = np.where(fin_a, ta, 0.0), np.where(fin_d, td, 0.0)
                dadv = np.stack([np.where(lnd, 0.0, O.smooth_snow(a, f.conv_variant)) for a in ta])
                ddiv = np.stack([np.where(lnd, 0.0, O.smooth_snow(d, f.conv_variant)) for d in td])
            else:
                dadv = np.zeros((2,) + conc.shape)
                ddiv = np.zeros((2,) + conc.shape)
            dlead, datm, dwpl, dwpg = zeros(), zeros(), zeros(), zeros()
            if f.leadlossInc == 1:
                dlead = O.lead_loss(t[0], wind, conc, p)
                if j == 1:
                    dlead = dlead + O.lead_loss(hx[0], wind, conc, one)
            if f.atmlossInc == 1:
                datm = O.atm_loss(t[0], wind, p)
                if j == 2:
                    datm = datm + O.atm_loss(hx[0], wind, one)
            if f.windpackInc == 1:
                dwpl, dwpg, _ = O.wind_packing(wind, t[0], p)
                if j == 0:
                    l1, g1, _ = O.wind_packing(wind, hx[0], one)
                    dwpl, dwpg = dwpl + l1, dwpg + g1
            out[j, 0] = np.where(kill0, 0.0, t[0] + dwpl + dlead + datm + dadv[0] + ddiv[0])
            out[j, 1] = np.where(kill1, 0.0, t[1] + dwpg + dadv[1] + ddiv[1])
    return out


def run_season_tangent(forcing, ic, mask, dx, p=None, f=None, num_steps=None):
    """``nesosim_oracle.run_season`` (variable density) with the tangents alongside: returns (state dict, tangents
    (T, DIRS, 2, ny, nx))."""
    p = p or O.Params()
    f = f or O.Flags()
    T, ny, nx = forcing["precip"].shape
    s = O.gen_empty_arrays(T, ny, nx)
    temp = np.full((ny, nx), np.nan)
    if ic is not None:
        half = O.initial_depths(ic, forcing["conc"][0], p)
        s["snowDepths"][0, 0] = half
        s["snowDepths"][0, 1] = half
    tan = np.zeros((T, DIRS, 2, ny, nx))
    steps = T - 1 if num_steps is None else num_steps
    for x in range(steps):
        args = (forcing["conc"][x], forcing["precip"][x], forcing["drift"][x], forcing["wind"][x])
        tan[x + 1] = tangent_step(s["snowDepths"][x], tan[x], *args, mask, dx, p, f)
        O.calc_budget(s, args[0], args[1], args[2], args[3], temp, mask, dx, x, p, f)
    return s, tan


def model_tangents(snowDepths, tan, conc, obs, mask, p):
    """dv [DIRS, n] at every input observation (dict of day, row, col, kind arrays), NaN where the model value
    (``model_values``) is not finite."""
    d, r, c, k = (np.asarray(obs[n]) for n in ("day", "row", "col", "kind"))
    density = np.full(conc.shape, np.nan)
    with np.errstate(all="ignore"):
        for t in np.unique(d[k == DENSITY]):
            density[t] = O.density_calc(snowDepths[t], conc[t], mask, p)
    v = model_values(snowDepths, density, conc, obs, mask)
    h0, h1 = snowDepths[d, 0, r, c], snowDepths[d, 1, r, c]
    out = np.empty((DIRS, len(d)))
    with np.errstate(all="ignore"):
        den = h0 + h1
        q = ((h0 * p.snowDensityFresh) + (h1 * p.snowDensityOld)) / den
        clamped = (q > p.snowDensityOld) | (q < p.snowDensityFresh)
        for j in range(DIRS):
            t0, t1 = tan[d, j, 0, r, c], tan[d, j, 1, r, c]
            dens = (((t0 * p.snowDensityFresh) + (t1 * p.snowDensityOld)) - (q * (t0 + t1))) / den
            dens = np.where(clamped, 0.0, dens)
            dv = np.where(k == DEPTH, (t0 + t1) / conc[d, r, c], np.where(k == VOLUME, t0 + t1, dens))
            out[j] = np.where(np.isfinite(v), dv, np.nan)
    return out


def gradient_terms(model, dmodel, values, sigma, kind, idx):
    """Per kind and direction, ``fixed_order_sum`` of 2*r*(dv/sigma) over the observations ``idx`` (summation order)
    whose r = (model - value)/sigma is finite: [KINDS, DIRS]."""
    kind = np.asarray(kind)[idx]
    with np.errstate(all="ignore"):
        r = (np.asarray(model)[idx] - np.asarray(values, dtype=np.float64)[idx]) / np.asarray(sigma)[idx]
        ok = np.isfinite(r)
        out = np.zeros((KINDS, DIRS))
        for j in range(DIRS):
            term = 2.0 * r * (np.asarray(dmodel[j])[idx] / np.asarray(sigma)[idx])
            for kk in range(KINDS):
                sel = kind == kk
                out[kk, j] = fixed_order_sum(np.where(ok[sel], term[sel], 0.0))
    return out


def score_gradients(model, dmodel, obs, mask):
    """d chi2 / d theta [KINDS, DIRS] of one member (``model``: ``model_values``; ``dmodel``: ``model_tangents``)."""
    return gradient_terms(model, dmodel, obs["value"], obs["sigma"], obs["kind"], order(obs, mask))


def footprint_tangents(snowDepths, density, tan, conc, fps, mask, p):
    """(mean [n_fp], dmean [DIRS, n_fp]) of one member: ``footprint_values`` and, in the same lane order and shuffle
    tree over the points with finite v, sum w*dv divided by the primal s (NaN where the mean is not finite)."""
    begin = np.asarray(fps["begin"], dtype=np.int64)
    kind = np.repeat(np.asarray(fps["kind"]), np.diff(begin))
    pts = {"day": fps["day"], "row": fps["row"], "col": fps["col"], "kind": kind}
    v = model_values(snowDepths, density, conc, pts, mask)
    dv = model_tangents(snowDepths, tan, conc, pts, mask, p)
    w = np.asarray(fps["weight"], dtype=np.float64)
    kept = ocean(mask)[np.asarray(fps["row"]), np.asarray(fps["col"])]
    mean = footprint_values(snowDepths, density, conc, fps, mask)
    out = np.empty((DIRS, len(begin) - 1))
    for g in range(len(begin) - 1):
        sel = np.arange(begin[g], begin[g + 1])
        sel = sel[kept[sel]]
        rows = -(-len(sel) // WARP) * WARP
        vv, ww, dd = np.full(rows, np.nan), np.ones(rows), np.zeros((DIRS, rows))
        vv[:len(sel)], ww[:len(sel)], dd[:, :len(sel)] = v[sel], w[sel], dv[:, sel]
        s, sdw = np.zeros(WARP), np.zeros((DIRS, WARP))
        with np.errstate(all="ignore"):
            for i in range(rows // WARP):                     # round i: lane l takes point i*32 + l
                lo = i * WARP
                ok = np.isfinite(vv[lo:lo + WARP])
                s = np.where(ok, s + ww[lo:lo + WARP], s)
                sdw = np.where(ok, sdw + ww[lo:lo + WARP] * dd[:, lo:lo + WARP], sdw)
            off = WARP // 2
            while off:
                s = s[:off] + s[off:2 * off]
                sdw = sdw[:, :off] + sdw[:, off:2 * off]
                off //= 2
            out[:, g] = np.where(np.isfinite(mean[g]), sdw[:, 0] / s[0], np.nan)
    return mean, out


def footprint_gradients(fp_model, fp_dmodel, fps):
    """d fp_chi2 / d theta [KINDS, DIRS] of one member: per kind over its footprints in input order."""
    return gradient_terms(fp_model, fp_dmodel, fps["value"], fps["sigma"], fps["kind"], np.arange(len(fps["value"])))
