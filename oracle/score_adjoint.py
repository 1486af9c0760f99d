"""Plain float64 restatement of the calibration adjoint (``nesosim_run_season_score_adjoint``: the record build of the
scoring day kernel, ``adjoint_seed_kernel``, ``adjoint_init_kernel``, ``day_step_adjoint_kernel`` and
``adjoint_finish_kernel`` in nesosim_b200/csrc, DESIGN.md §4.1), down to the order of every operation, so that the GPU's
``ic_grad`` and ``theta_grad`` can be compared bit for bit.

Objective of one member: J = sum_k w[k] chi2[k] + sum_k fw[k] fp_chi2[k].  The adjoint state lam[x] = dJ/d snowDepths[x]
(2, ny, nx) is the transpose of ``score_gradients.tangent_step``, taken pathwise on the primal's side of every kink:

* forward record: per day x and cell, kill0/kill1 (``fill_nan_no_negative`` replaced the new depth: not finite, land, or
  the clamp of a negative value) and whether each raw term adv0, adv1, div0, div1 was finite;
* seeds (``seeds``): per observed (day, cell) slot, from 0.0, first every point observation chi2 counts in chi2's order
  (kinds in turn, ``order`` within a kind) adding a*dv/d(h0, h1) with a = ((2 r) w[k]) / sigma, then every kept
  footprint point with finite v in footprint input order, with a = b * w_p, b = (((2 r_g) fw[k]) / sigma_g) / s_g;
  depth dv = (a/C, a/C), volume (a, a), density ((a (rhoF - q)) / den, (a (rhoO - q)) / den), 0 where a clamp set q;
* backward step x+1 -> x (``adjoint_step``): mu = kill ? 0 : lam[x+1]; the point terms applied to mu0 (kill0 off) and
  wpg to mu1 (kill1 off), then the transposed dynamics: nu = the transposed 3x3 smoothing of mu/divisor on every grid
  cell, px = (nu_adv * ut) / d_x and py = (nu_adv * vt) / d_y (d = dx on the grid edge of that axis, else 2 dx) where
  the raw adv term was finite, and per cell dd = -((nu_div gxu) + (nu_div gyv)) where the raw div term was finite,
  dyn = dd - ((px[c-1] - px[c+1] + E_x) + (py[c-1] - py[c+1] + E_y)), E = (last ? p[c] : 0) - (first ? p[c] : 0);
  lam0 = ((((mu0 + wpl) + lead) + atm) + wpg) + dyn0, lam1 = mu1 + dyn1; then the day's seeds at its slots;
* theta: per cell and day (x descending), acc_j += the parameter's source term times mu (0 where killed; windpack adds
  its two layers' terms first); theta_grad_j = ``fixed_order_sum`` of acc_j over the cells in row-major order;
* ic_grad = (lam0[0] + lam1[0]) * 0.5 where conc[0] >= minConc, else 0.
"""
import dataclasses

import numpy as np

from . import nesosim_oracle as O
from .astropy_restated import gaussian2d_kernel
from .observation_scores import DENSITY, DEPTH, KINDS, VOLUME, WARP, fixed_order_sum, model_values, ocean, order
from .score_gradients import DIRS, PARAM_FIELDS, land, raw_dynamics


def conv_weights(f):
    """The 3x3 kernel and the divisor applied after the sum (the smoothing's two variants)."""
    g = gaussian2d_kernel(x_stddev=1, x_size=3, y_size=3)
    return (g, g.sum()) if f.conv_variant == "post_divide" else (g / g.sum(), 1.0)


def step_record(hx, conc, precip, drift, wind, mask, dx, p, f):
    """What the record build stores for day x: (kill0, kill1, fin_adv (2, ny, nx), fin_div (2, ny, nx))."""
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
            fin_a = fin_d = np.zeros((2,) + conc.shape, dtype=bool)
        lead = O.lead_loss(hx[0], wind, conc, p) if f.leadlossInc == 1 else zeros()
        atm = O.atm_loss(hx[0], wind, p) if f.atmlossInc == 1 else zeros()
        wpl, wpg, _ = O.wind_packing(wind, hx[0], p) if f.windpackInc == 1 else (zeros(), zeros(), zeros())
        h0n = hx[0] + acc + wpl + lead + atm + adv[0] + div[0]
        h1n = hx[1] + wpg + adv[1] + div[1]
        kill0 = ~np.isfinite(h0n) | lnd | (h0n < 0.)
        kill1 = ~np.isfinite(h1n) | lnd | (h1n < 0.)
    return kill0, kill1, fin_a, fin_d


def run_season_record(forcing, ic, mask, dx, p, f, num_steps=None):
    """The primal season (``nesosim_oracle.run_season``, variable density) and the record of every step."""
    T, ny, nx = forcing["precip"].shape
    s = O.gen_empty_arrays(T, ny, nx)
    temp = np.full((ny, nx), np.nan)
    if ic is not None:
        half = O.initial_depths(ic, forcing["conc"][0], p)
        s["snowDepths"][0, 0] = half
        s["snowDepths"][0, 1] = half
    rec = []
    steps = T - 1 if num_steps is None else num_steps
    for x in range(steps):
        args = (forcing["conc"][x], forcing["precip"][x], forcing["drift"][x], forcing["wind"][x])
        rec.append(step_record(s["snowDepths"][x], *args, mask, dx, p, f))
        O.calc_budget(s, args[0], args[1], args[2], args[3], temp, mask, dx, x, p, f)
    return s, rec


def _partials(kind, h0, h1, C, a, p):
    """a * dv/d(h0, h1) of one model value (``adjoint_seed_kernel``)."""
    if kind == DEPTH:
        d = a / C
        return d, d
    if kind == VOLUME:
        return a, a
    den = h0 + h1
    q = ((h0 * p.snowDensityFresh) + (h1 * p.snowDensityOld)) / den
    if q > p.snowDensityOld or q < p.snowDensityFresh:
        return 0.0, 0.0
    return (a * (p.snowDensityFresh - q)) / den, (a * (p.snowDensityOld - q)) / den


def footprint_sums(snowDepths, density, conc, fps, mask):
    """(mean, s) of every footprint: ``footprint_values`` and the weight sum s of its points with finite v."""
    begin = np.asarray(fps["begin"], dtype=np.int64)
    kind = np.repeat(np.asarray(fps["kind"]), np.diff(begin))
    pts = {"day": fps["day"], "row": fps["row"], "col": fps["col"], "kind": kind}
    v = model_values(snowDepths, density, conc, pts, mask)
    w = np.asarray(fps["weight"], dtype=np.float64)
    kept = ocean(mask)[np.asarray(fps["row"]), np.asarray(fps["col"])]
    mean, ssum = np.empty(len(begin) - 1), np.empty(len(begin) - 1)
    for g in range(len(mean)):
        sel = np.arange(begin[g], begin[g + 1])
        sel = sel[kept[sel]]
        rows = -(-len(sel) // WARP) * WARP
        vv, ww = np.full(rows, np.nan), np.ones(rows)
        vv[:len(sel)], ww[:len(sel)] = v[sel], w[sel]
        sw, s = np.zeros(WARP), np.zeros(WARP)
        with np.errstate(all="ignore"):
            for vr, wr in zip(vv.reshape(-1, WARP), ww.reshape(-1, WARP)):
                ok = np.isfinite(vr)
                sw = np.where(ok, sw + wr * vr, sw)
                s = np.where(ok, s + wr, s)
            off = WARP // 2
            while off:
                sw = sw[:off] + sw[off:2 * off]
                s = s[:off] + s[off:2 * off]
                off //= 2
            mean[g], ssum[g] = sw[0] / s[0], s[0]
    return mean, ssum, v


def seeds(snowDepths, density, conc, obs, fps, mask, p, w, fw):
    """dJ/d snowDepths at the observed cell-days of one member: (S (T, 2, ny, nx), slot (T, ny, nx) bool), S summed
    per slot from 0.0 in the fixed order of the module docstring."""
    T, _, ny, nx = snowDepths.shape
    S = np.zeros((T, 2, ny, nx))
    slot = np.zeros((T, ny, nx), dtype=bool)
    w, fw = np.asarray(w, dtype=np.float64), np.asarray(fw, dtype=np.float64)
    with np.errstate(all="ignore"):
        if obs is not None and len(obs["day"]):
            d, r, c, k = (np.asarray(obs[n]) for n in ("day", "row", "col", "kind"))
            val, sig = np.asarray(obs["value"], dtype=np.float64), np.asarray(obs["sigma"], dtype=np.float64)
            v = model_values(snowDepths, density, conc, obs, mask)
            idx = order(obs, mask)
            slot[d[idx], r[idx], c[idx]] = True
            for kk in range(KINDS):
                for q in idx[k[idx] == kk]:
                    res = (v[q] - val[q]) / sig[q]
                    if not np.isfinite(res):
                        continue
                    a = ((2.0 * res) * w[kk]) / sig[q]
                    h0, h1 = snowDepths[d[q], 0, r[q], c[q]], snowDepths[d[q], 1, r[q], c[q]]
                    g0, g1 = _partials(kk, h0, h1, conc[d[q], r[q], c[q]], a, p)
                    S[d[q], 0, r[q], c[q]] += g0
                    S[d[q], 1, r[q], c[q]] += g1
        if fps is not None and len(fps["value"]):
            mean, ssum, v = footprint_sums(snowDepths, density, conc, fps, mask)
            begin = np.asarray(fps["begin"], dtype=np.int64)
            d, r, c = (np.asarray(fps[n]) for n in ("day", "row", "col"))
            pw = np.asarray(fps["weight"], dtype=np.float64)
            kept = ocean(mask)[r, c]
            slot[d[kept], r[kept], c[kept]] = True
            for g in range(len(mean)):
                kk = int(fps["kind"][g])
                res = (mean[g] - float(fps["value"][g])) / float(fps["sigma"][g])
                if not np.isfinite(res):
                    continue
                b = (((2.0 * res) * fw[kk]) / float(fps["sigma"][g])) / ssum[g]
                for j in range(begin[g], begin[g + 1]):
                    if not kept[j] or not np.isfinite(v[j]):
                        continue
                    a = b * pw[j]
                    h0, h1 = snowDepths[d[j], 0, r[j], c[j]], snowDepths[d[j], 1, r[j], c[j]]
                    g0, g1 = _partials(kk, h0, h1, conc[d[j], r[j], c[j]], a, p)
                    S[d[j], 0, r[j], c[j]] += g0
                    S[d[j], 1, r[j], c[j]] += g1
    return S, slot


def _smooth_t(m, g):
    """The transposed 3x3 smoothing at every grid cell of the already divided plane ``m`` (0 outside the grid)."""
    ny, nx = m.shape
    mp = np.zeros((ny + 2, nx + 2))
    mp[1:-1, 1:-1] = m
    acc = np.zeros((ny, nx))
    for ii in range(3):
        for jj in range(3):
            acc = acc + mp[2 - ii:2 - ii + ny, 2 - jj:2 - jj + nx] * g[2 - ii, 2 - jj]
    return acc


def _grad_t(pl, axis):
    """Transposed np.gradient of one axis for the divided, gated plane ``pl``: p[c-1] - p[c+1] + E."""
    pm = np.moveaxis(pl, axis, 0)
    n = pm.shape[0]
    pad = np.zeros((n + 2,) + pm.shape[1:])
    pad[1:-1] = pm
    first = np.zeros(n, dtype=bool)
    last = np.zeros(n, dtype=bool)
    first[0], last[-1] = True, True
    shape = (n,) + (1,) * (pm.ndim - 1)
    e = np.where(last.reshape(shape), pm, 0.0) - np.where(first.reshape(shape), pm, 0.0)
    return np.moveaxis((pad[:-2] - pad[2:]) + e, 0, axis)


def adjoint_step(lam, hx, rec, conc, drift, wind, mask, dx, p, f, acc):
    """lam[x] (2, ny, nx) from lam[x+1] and day x's primal depths ``hx`` and record ``rec``; adds day x's parameter
    terms to ``acc`` (DIRS, ny, nx) in place.  The day's seeds are added by the caller."""
    kill0, kill1, fin_a, fin_d = rec
    ny, nx = conc.shape
    with np.errstate(all="ignore"):
        mu0 = np.where(kill0, 0.0, lam[0])
        mu1 = np.where(kill1, 0.0, lam[1])
        a0 = mu0
        if f.windpackInc == 1:
            a0 = np.where(kill0, a0, a0 + O.wind_packing(wind, mu0, p)[0])
        if f.leadlossInc == 1:
            a0 = np.where(kill0, a0, a0 + O.lead_loss(mu0, wind, conc, p))
        if f.atmlossInc == 1:
            a0 = np.where(kill0, a0, a0 + O.atm_loss(mu0, wind, p))
        if f.windpackInc == 1:
            a0 = np.where(kill1, a0, a0 + O.wind_packing(wind, mu1, p)[1])
        out = np.stack([a0, mu1])
        if f.dynamicsInc == 1:
            g, cd = conv_weights(f)
            ut, vt = drift[0] * p.deltaT, drift[1] * p.deltaT
            gxu = np.gradient(ut, dx, axis=1)
            gyv = np.gradient(vt, dx, axis=0)
            dxc = np.full(nx, 2. * dx)
            dxc[0] = dxc[-1] = dx
            dyc = np.full(ny, 2. * dx)
            dyc[0] = dyc[-1] = dx
            for l, mu in enumerate((mu0, mu1)):
                nu = _smooth_t(mu / cd, g)
                px = np.where(fin_a[l], (nu * ut) / dxc[None, :], 0.0)
                py = np.where(fin_a[l], (nu * vt) / dyc[:, None], 0.0)
                dd = np.where(fin_d[l], -((nu * gxu) + (nu * gyv)), 0.0)
                out[l] = out[l] + (dd - (_grad_t(px, 1) + _grad_t(py, 0)))
        h0 = hx[0]
        one = [dataclasses.replace(p, **{PARAM_FIELDS[j]: 1.0}) for j in range(DIRS)]
        s0 = s1 = np.zeros((ny, nx))
        if f.windpackInc == 1:
            l1, g1, _ = O.wind_packing(wind, h0, one[0])
            s0 = np.where(kill0, 0.0, mu0 * l1)
            s1 = np.where(kill1, 0.0, mu1 * g1)
        acc[0] = acc[0] + (s0 + s1)
        s = np.where(kill0, 0.0, mu0 * O.lead_loss(h0, wind, conc, one[1])) if f.leadlossInc == 1 else np.zeros((ny, nx))
        acc[1] = acc[1] + s
        s = np.where(kill0, 0.0, mu0 * O.atm_loss(h0, wind, one[2])) if f.atmlossInc == 1 else np.zeros((ny, nx))
        acc[2] = acc[2] + s
    return out


def score_adjoint(forcing, ic, mask, dx, p, f, obs=None, fps=None, w=(1.0,) * KINDS, fw=(1.0,) * KINDS, num_steps=None):
    """(theta_grad [DIRS], ic_grad (ny, nx), s) of one member whose season takes ``num_steps`` steps (default T-1)."""
    T, ny, nx = forcing["precip"].shape
    L = T - 1 if num_steps is None else num_steps
    s, rec = run_season_record(forcing, ic, mask, dx, p, f, L)
    S, slot = seeds(s["snowDepths"][:L + 1], s["density"][:L + 1], forcing["conc"][:L + 1], obs, fps, mask, p, w, fw)
    lam = np.where(slot[L], 0.0 + S[L], 0.0)
    acc = np.zeros((DIRS, ny, nx))
    for x in range(L - 1, -1, -1):
        args = (forcing["conc"][x], forcing["drift"][x], forcing["wind"][x])
        lam = adjoint_step(lam, s["snowDepths"][x], rec[x], *args, mask, dx, p, f, acc)
        lam = np.where(slot[x], lam + S[x], lam)
    theta = np.array([fixed_order_sum(acc[j].ravel()) for j in range(DIRS)])
    with np.errstate(invalid="ignore"):
        keep = ~(forcing["conc"][0] < p.minConc)
    ic_grad = np.where(keep, (lam[0] + lam[1]) * 0.5, 0.0)
    return theta, ic_grad, s


def tangent_step_ic(hx, tx, conc, precip, drift, wind, mask, dx, p, f):
    """``score_gradients.tangent_step`` of one direction without parameter source terms: the tangent (2, ny, nx) of
    slot x+1 for an initial-condition direction."""
    lnd = land(mask)
    zeros = lambda: np.zeros(conc.shape)
    kill0, kill1, fin_a, fin_d = step_record(hx, conc, precip, drift, wind, mask, dx, p, f)
    with np.errstate(all="ignore"):
        if f.dynamicsInc == 1:
            ta, td = raw_dynamics(drift, tx, dx, p)
            ta, td = np.where(fin_a, ta, 0.0), np.where(fin_d, td, 0.0)
            dadv = np.stack([np.where(lnd, 0.0, O.smooth_snow(a, f.conv_variant)) for a in ta])
            ddiv = np.stack([np.where(lnd, 0.0, O.smooth_snow(d, f.conv_variant)) for d in td])
        else:
            dadv = ddiv = np.zeros((2,) + conc.shape)
        dlead = O.lead_loss(tx[0], wind, conc, p) if f.leadlossInc == 1 else zeros()
        datm = O.atm_loss(tx[0], wind, p) if f.atmlossInc == 1 else zeros()
        dwpl, dwpg, _ = O.wind_packing(wind, tx[0], p) if f.windpackInc == 1 else (zeros(), zeros(), zeros())
        out = np.empty_like(tx)
        out[0] = np.where(kill0, 0.0, tx[0] + dwpl + dlead + datm + dadv[0] + ddiv[0])
        out[1] = np.where(kill1, 0.0, tx[1] + dwpg + dadv[1] + ddiv[1])
    return out


def run_season_tangent_ic(forcing, ic, v, mask, dx, p, f, num_steps=None):
    """Tangents (T, 2, ny, nx) of the season in the initial-condition direction ``v`` (ny, nx): t[0] is
    ``initial_depths``' derivative, 0.5 v in both layers where conc[0] >= minConc."""
    T, ny, nx = forcing["precip"].shape
    s = O.gen_empty_arrays(T, ny, nx)
    temp = np.full((ny, nx), np.nan)
    half = O.initial_depths(ic, forcing["conc"][0], p)
    s["snowDepths"][0, 0] = half
    s["snowDepths"][0, 1] = half
    tan = np.zeros((T, 2, ny, nx))
    tan[0, 0] = tan[0, 1] = O.initial_depths(v, forcing["conc"][0], p)
    steps = T - 1 if num_steps is None else num_steps
    for x in range(steps):
        args = (forcing["conc"][x], forcing["precip"][x], forcing["drift"][x], forcing["wind"][x])
        tan[x + 1] = tangent_step_ic(s["snowDepths"][x], tan[x], *args, mask, dx, p, f)
        O.calc_budget(s, args[0], args[1], args[2], args[3], temp, mask, dx, x, p, f)
    return s, tan
