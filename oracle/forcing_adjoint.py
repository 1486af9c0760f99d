"""Plain float64 restatement of the calibration adjoint with respect to the forcing
(``nesosim_run_season_score_adjoint_forcing``: the forcing builds of ``adjoint_seed_kernel``, ``adjoint_init_kernel``,
``day_step_adjoint_kernel`` and ``adjoint_finish_kernel`` in nesosim_b200/csrc, DESIGN.md §4.1), down to the order of
every operation, so that the GPU's per-day gradients, scale fields and totals can be compared bit for bit.  It runs
``score_adjoint``'s sweep unchanged and forms, for day x <= L - 1 (L the member's last slot), per cell with
mu0 = kill0 ? 0 : lam0[x+1], pd = P / rhoF, wt = (W > windPackThresh) and X = (((wt llf) dT) h0) W:

* g_P = kill0 ? 0 : (mu0 C) / rhoF;
* g_W = kill0 ? 0 : (lead ? mu0 lead_loss(W := 1) : 0) + (atm ? mu0 atm_loss(W := 1) : 0);
* g_C = (kill0 ? 0 : mu0 pd + (lead ? mu0 X : 0)) + cseed(x), cseed summed per sample slot from 0.0 in the order of
  ``score_adjoint.seeds`` over the depth items alone, each adding -((a v) / C) with v = (h0 + h1) / C (0 without a
  slot); g_C(L) = 0 + cseed(L); every gradient is 0 after L, and g_P, g_W are 0 on L.

The scale field of F is sum over x = L, L-1, ..., 0 of (finite(F) ? F g_F : 0) from 0.0; the total is its
``fixed_order_sum`` over the cells in row-major order.  The step W > windPackThresh and the IC zeroing where
conc[0] < minConc have no derivative.
"""
import numpy as np

from . import nesosim_oracle as O
from . import score_gradients as G
from .footprint_scores import footprint_values
from .observation_scores import DEPTH, KINDS, fixed_order_sum, model_values, ocean, order
from .score_adjoint import adjoint_step, footprint_sums, run_season_record, seeds, step_record, tangent_step_ic

FIELDS = ("precip", "wind", "conc")


def conc_seeds(snowDepths, density, conc, obs, fps, mask, p, w, fw):
    """dJ/dC at the observed cell-days of one member (T, ny, nx): the depth items of ``score_adjoint.seeds`` in its
    order, each adding -((a v) / C)."""
    T, _, ny, nx = snowDepths.shape
    CS = np.zeros((T, ny, nx))
    w, fw = np.asarray(w, dtype=np.float64), np.asarray(fw, dtype=np.float64)
    with np.errstate(all="ignore"):
        if obs is not None and len(obs["day"]):
            d, r, c, k = (np.asarray(obs[n]) for n in ("day", "row", "col", "kind"))
            val, sig = np.asarray(obs["value"], dtype=np.float64), np.asarray(obs["sigma"], dtype=np.float64)
            v = model_values(snowDepths, density, conc, obs, mask)
            idx = order(obs, mask)
            for q in idx[k[idx] == DEPTH]:
                res = (v[q] - val[q]) / sig[q]
                if not np.isfinite(res):
                    continue
                a = ((2.0 * res) * w[DEPTH]) / sig[q]
                CS[d[q], r[q], c[q]] += -((a * v[q]) / conc[d[q], r[q], c[q]])
        if fps is not None and len(fps["value"]):
            mean, ssum, v = footprint_sums(snowDepths, density, conc, fps, mask)
            begin = np.asarray(fps["begin"], dtype=np.int64)
            d, r, c = (np.asarray(fps[n]) for n in ("day", "row", "col"))
            pw = np.asarray(fps["weight"], dtype=np.float64)
            kept = ocean(mask)[r, c]
            for g in range(len(mean)):
                if int(fps["kind"][g]) != DEPTH:
                    continue
                res = (mean[g] - float(fps["value"][g])) / float(fps["sigma"][g])
                if not np.isfinite(res):
                    continue
                b = (((2.0 * res) * fw[DEPTH]) / float(fps["sigma"][g])) / ssum[g]
                for j in range(begin[g], begin[g + 1]):
                    if not kept[j] or not np.isfinite(v[j]):
                        continue
                    a = b * pw[j]
                    CS[d[j], r[j], c[j]] += -((a * v[j]) / conc[d[j], r[j], c[j]])
    return CS


def forcing_terms(mu0, kill0, h0, P, W, C, p, f):
    """(g_P, g_W, step_C) of one day from mu0 = kill0 ? 0 : lam0[x+1] and the primal h0 of day x."""
    with np.errstate(all="ignore"):
        wt = np.where(W > p.windPackThresh, 1.0, 0.0)
        gP = np.where(kill0, 0.0, (mu0 * C) / p.snowDensityFresh)
        lead1 = -((((wt * p.leadLossFactor) * p.deltaT) * h0) * (1.0 - C))            # lead_loss with W = 1
        atm1 = -(((wt * p.deltaT) * h0) * p.atmLossFactor)                            # atm_loss with W = 1
        wl = mu0 * lead1 if f.leadlossInc == 1 else np.zeros(C.shape)
        wa = mu0 * atm1 if f.atmlossInc == 1 else np.zeros(C.shape)
        gW = np.where(kill0, 0.0, wl + wa)
        X = (((wt * p.leadLossFactor) * p.deltaT) * h0) * W
        sC = (mu0 * (P / p.snowDensityFresh)) + (mu0 * X if f.leadlossInc == 1 else 0.0)
        sC = np.where(kill0, 0.0, sC)
    return gP, gW, sC


def score_adjoint_forcing(forcing, ic, mask, dx, p, f, obs=None, fps=None, w=(1.0,) * KINDS, fw=(1.0,) * KINDS,
                          num_steps=None):
    """One member's adjoint with the forcing: dict of "theta_grad" [DIRS], "ic_grad" (ny, nx), "<field>_day_grad"
    (T, ny, nx) for each of ``FIELDS``, "forcing_scale_grad" (3, ny, nx) and "forcing_scale_total" [3]."""
    T, ny, nx = forcing["precip"].shape
    L = T - 1 if num_steps is None else num_steps
    s, rec = run_season_record(forcing, ic, mask, dx, p, f, L)
    args = (s["snowDepths"][:L + 1], s["density"][:L + 1], forcing["conc"][:L + 1], obs, fps, mask, p, w, fw)
    S, slot = seeds(*args)
    CS = conc_seeds(*args)
    day = {n: np.zeros((T, ny, nx)) for n in FIELDS}
    day["conc"][L] = 0.0 + CS[L]
    lam = np.where(slot[L], 0.0 + S[L], 0.0)
    acc = np.zeros((G.DIRS, ny, nx))
    with np.errstate(invalid="ignore"):
        for x in range(L - 1, -1, -1):
            P, C, W = forcing["precip"][x], forcing["conc"][x], forcing["wind"][x]
            kill0 = rec[x][0]
            mu0 = np.where(kill0, 0.0, lam[0])
            gP, gW, sC = forcing_terms(mu0, kill0, s["snowDepths"][x][0], P, W, C, p, f)
            day["precip"][x], day["wind"][x], day["conc"][x] = gP, gW, sC + CS[x]
            args = (forcing["conc"][x], forcing["drift"][x], forcing["wind"][x])
            lam = adjoint_step(lam, s["snowDepths"][x], rec[x], *args, mask, dx, p, f, acc)
            lam = np.where(slot[x], lam + S[x], lam)
        scale = np.zeros((3, ny, nx))
        for x in range(L, -1, -1):
            for i, n in enumerate(FIELDS):
                F = forcing[n][x]
                scale[i] = scale[i] + np.where(np.isfinite(F), F * day[n][x], 0.0)
        keep = ~(forcing["conc"][0] < p.minConc)
    out = {n + "_day_grad": day[n] for n in FIELDS}
    out["theta_grad"] = np.array([fixed_order_sum(acc[j].ravel()) for j in range(G.DIRS)])
    out["ic_grad"] = np.where(keep, (lam[0] + lam[1]) * 0.5, 0.0)
    out["forcing_scale_grad"] = scale
    out["forcing_scale_total"] = np.array([fixed_order_sum(scale[i].ravel()) for i in range(3)])
    return out


def run_season_tangent_forcing(forcing, ic, mask, dx, p, f, dP, dW, dC, num_steps=None):
    """Tangents (T, 2, ny, nx) of the season in the forcing direction (dP, dW, dC), each (T, ny, nx): the transported
    tangent of ``score_adjoint.tangent_step_ic`` plus the forcing's own terms d acc = (dP / rhoF) C + pd dC,
    d lead = -((((wt llf) dT) h0) dW (1 - C)) + X dC and d atm = -((((wt dT) h0) dW) alf), 0 where the primal killed
    the new h0.  The IC does not depend on the forcing (conc[0] acts on it through a step)."""
    T, ny, nx = forcing["precip"].shape
    s = O.gen_empty_arrays(T, ny, nx)
    temp = np.full((ny, nx), np.nan)
    half = O.initial_depths(ic, forcing["conc"][0], p)
    s["snowDepths"][0, 0] = half
    s["snowDepths"][0, 1] = half
    tan = np.zeros((T, 2, ny, nx))
    steps = T - 1 if num_steps is None else num_steps
    for x in range(steps):
        P, C, W = forcing["precip"][x], forcing["conc"][x], forcing["wind"][x]
        hx = s["snowDepths"][x]
        args = (C, P, forcing["drift"][x], W)
        tan[x + 1] = tangent_step_ic(hx, tan[x], *args, mask, dx, p, f)
        kill0 = step_record(hx, *args, mask, dx, p, f)[0]
        with np.errstate(all="ignore"):
            wt = np.where(W > p.windPackThresh, 1.0, 0.0)
            K = ((wt * p.leadLossFactor) * p.deltaT) * hx[0]
            src = (dP[x] / p.snowDensityFresh) * C + (P / p.snowDensityFresh) * dC[x]
            if f.leadlossInc == 1:
                src = src + (-(K * dW[x] * (1.0 - C)) + (K * W) * dC[x])
            if f.atmlossInc == 1:
                src = src - (((wt * p.deltaT) * hx[0]) * dW[x]) * p.atmLossFactor
            tan[x + 1, 0] = np.where(kill0, 0.0, tan[x + 1, 0] + src)
        O.calc_budget(s, C, P, forcing["drift"][x], W, temp, mask, dx, x, p, f)
    return s, tan


def _dv(snowDepths, tan, conc, dC, pts, mask, p):
    """d model value of every point (dict of day, row, col, kind): the state tangent through ``model_tangents`` plus,
    for depth, dv/dC dC = -(v / C) dC; NaN where v is not finite."""
    t3 = np.repeat(tan[:, None], G.DIRS, axis=1)
    dv = G.model_tangents(snowDepths, t3, conc, pts, mask, p)[0]
    d, r, c, k = (np.asarray(pts[n]) for n in ("day", "row", "col", "kind"))
    density = np.full(conc.shape, np.nan)
    v = model_values(snowDepths, density, conc, {**pts, "kind": np.where(k == DEPTH, DEPTH, 1)}, mask)
    with np.errstate(all="ignore"):
        return np.where(k == DEPTH, dv - (v / conc[d, r, c]) * dC[d, r, c], dv)


def objective_tangent_forcing(forcing, ic, mask, dx, p, f, obs, fps, w, fw, dP, dW, dC, num_steps=None):
    """dJ of one member along the forcing direction (dP, dW, dC) by the forward mode, for the dot-product identity."""
    T = forcing["precip"].shape[0]
    L = T - 1 if num_steps is None else num_steps
    s, tan = run_season_tangent_forcing(forcing, ic, mask, dx, p, f, dP, dW, dC, L)
    conc = forcing["conc"]
    sd, tan = s["snowDepths"][:L + 1], tan[:L + 1]
    density = s["density"][:L + 1]
    dJ = 0.0
    with np.errstate(all="ignore"):
        if obs is not None and len(obs["day"]):
            v = model_values(sd, density, conc, obs, mask)
            dv = _dv(sd, tan, conc, dC, obs, mask, p)
            r = (v - np.asarray(obs["value"], dtype=np.float64)) / np.asarray(obs["sigma"], dtype=np.float64)
            idx = order(obs, mask)
            k = np.asarray(obs["kind"])
            for q in idx:
                if np.isfinite(r[q]):
                    dJ += w[k[q]] * (2.0 * r[q] * dv[q] / obs["sigma"][q])
        if fps is not None and len(fps["value"]):
            begin = np.asarray(fps["begin"], dtype=np.int64)
            kind = np.repeat(np.asarray(fps["kind"]), np.diff(begin))
            pts = {"day": fps["day"], "row": fps["row"], "col": fps["col"], "kind": kind}
            v = model_values(sd, density, conc, pts, mask)
            dv = _dv(sd, tan, conc, dC, pts, mask, p)
            pw = np.asarray(fps["weight"], dtype=np.float64)
            kept = ocean(mask)[np.asarray(fps["row"]), np.asarray(fps["col"])]
            mean = footprint_values(sd, density, conc, fps, mask)
            for g in range(len(mean)):
                sel = np.arange(begin[g], begin[g + 1])
                sel = sel[kept[sel] & np.isfinite(v[sel])]
                res = (mean[g] - float(fps["value"][g])) / float(fps["sigma"][g])
                if not np.isfinite(res) or not len(sel):
                    continue
                dmean = np.sum(pw[sel] * dv[sel]) / np.sum(pw[sel])
                dJ += fw[int(fps["kind"][g])] * (2.0 * res * dmean / float(fps["sigma"][g]))
    return dJ
