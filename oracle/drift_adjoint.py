"""Plain float64 restatement of the calibration adjoint with respect to the ice drift
(``nesosim_run_season_score_adjoint_drift``: the drift builds of ``day_step_adjoint_kernel`` and
``adjoint_finish_kernel`` in nesosim_b200/csrc, DESIGN.md §4.1), down to the order of every operation, so that the
GPU's per-day gradients, scale fields and totals can be compared bit for bit.  It runs ``score_adjoint``'s sweep
unchanged and forms, for day x <= L - 1 (L the member's last slot), with ut = u dT, vt = v dT, h_l the primal depth of
day x, m_l = (kill_l ? 0 : lam_l[x+1]) / divisor, nu_l its transposed 3x3 smoothing and A_l, D_l the record's finite
bits of the raw adv_l and div_l:

* Qx = (D_0 ? (nu_0 h_0) / d_x : 0) + (D_1 ? (nu_1 h_1) / d_x : 0), d_x = dx on the first and last column, else 2 dx;
  Qy alike along the rows;
* Gx = (A_0 ? nu_0 gx(h_0) : 0) + (A_1 ? nu_1 gx(h_1) : 0) with np.gradient's gx; Gy alike with gy;
* g_u = -((Gx + ((Qx[c-1] - Qx[c+1]) + E_x)) dT), E_x = (last ? Qx[c] : 0) - (first ? Qx[c] : 0); g_v alike;
* g = 0 on days L..T-1 and without dynamics.

The scale field of component k is the sum over x = L-1, ..., 0 of (finite(F) ? F g_F : 0) from 0.0 with F the raw
drift component; the total is its ``fixed_order_sum`` over the cells in row-major order.
"""
import numpy as np

from . import nesosim_oracle as O
from . import score_gradients as G
from .footprint_scores import footprint_values
from .forcing_adjoint import _dv
from .observation_scores import KINDS, fixed_order_sum, model_values, ocean, order
from .score_adjoint import (_grad_t, _smooth_t, adjoint_step, conv_weights, run_season_record, seeds, step_record,
                            tangent_step_ic)

COMPONENTS = ("u", "v")


def edge_divisors(ny, nx, dx):
    """d_x (nx,) and d_y (ny,): dx on the grid edge of that axis, 2 dx elsewhere."""
    dxc = np.full(nx, 2. * dx)
    dxc[0] = dxc[-1] = dx
    dyc = np.full(ny, 2. * dx)
    dyc[0] = dyc[-1] = dx
    return dxc, dyc


def drift_terms(lam, hx, rec, dx, p, f):
    """(g_u, g_v) of day x from lam[x+1] (2, ny, nx), the primal depths ``hx`` of day x and its record ``rec``."""
    kill0, kill1, fin_a, fin_d = rec
    ny, nx = hx.shape[1:]
    if f.dynamicsInc != 1:
        return np.zeros((2, ny, nx))
    g, cd = conv_weights(f)
    dxc, dyc = edge_divisors(ny, nx, dx)
    with np.errstate(all="ignore"):
        qx, qy, ax, ay = [], [], [], []
        for l, kill in enumerate((kill0, kill1)):
            nu = _smooth_t(np.where(kill, 0.0, lam[l]) / cd, g)
            nh = nu * hx[l]
            qx.append(np.where(fin_d[l], nh / dxc[None, :], 0.0))
            qy.append(np.where(fin_d[l], nh / dyc[:, None], 0.0))
            ax.append(np.where(fin_a[l], nu * np.gradient(hx[l], dx, axis=1), 0.0))
            ay.append(np.where(fin_a[l], nu * np.gradient(hx[l], dx, axis=0), 0.0))
        Qx, Qy = qx[0] + qx[1], qy[0] + qy[1]
        Gx, Gy = ax[0] + ax[1], ay[0] + ay[1]
        gu = -((Gx + _grad_t(Qx, 1)) * p.deltaT)
        gv = -((Gy + _grad_t(Qy, 0)) * p.deltaT)
    return np.stack([gu, gv])


def score_adjoint_drift(forcing, ic, mask, dx, p, f, obs=None, fps=None, w=(1.0,) * KINDS, fw=(1.0,) * KINDS,
                        num_steps=None):
    """One member's adjoint with the drift: dict of "theta_grad" [DIRS], "ic_grad" (ny, nx), "drift_day_grad"
    (T, 2, ny, nx), "drift_scale_grad" (2, ny, nx) and "drift_scale_total" [2]."""
    T, ny, nx = forcing["precip"].shape
    L = T - 1 if num_steps is None else num_steps
    s, rec = run_season_record(forcing, ic, mask, dx, p, f, L)
    S, slot = seeds(s["snowDepths"][:L + 1], s["density"][:L + 1], forcing["conc"][:L + 1], obs, fps, mask, p, w, fw)
    day = np.zeros((T, 2, ny, nx))
    scale = np.zeros((2, ny, nx))
    lam = np.where(slot[L], 0.0 + S[L], 0.0)
    acc = np.zeros((G.DIRS, ny, nx))
    with np.errstate(invalid="ignore"):
        for x in range(L - 1, -1, -1):
            day[x] = drift_terms(lam, s["snowDepths"][x], rec[x], dx, p, f)
            if f.dynamicsInc == 1:
                F = forcing["drift"][x]
                scale = scale + np.where(np.isfinite(F), F * day[x], 0.0)
            args = (forcing["conc"][x], forcing["drift"][x], forcing["wind"][x])
            lam = adjoint_step(lam, s["snowDepths"][x], rec[x], *args, mask, dx, p, f, acc)
            lam = np.where(slot[x], lam + S[x], lam)
        keep = ~(forcing["conc"][0] < p.minConc)
    return {"theta_grad": np.array([fixed_order_sum(acc[j].ravel()) for j in range(G.DIRS)]),
            "ic_grad": np.where(keep, (lam[0] + lam[1]) * 0.5, 0.0),
            "drift_day_grad": day, "drift_scale_grad": scale,
            "drift_scale_total": np.array([fixed_order_sum(scale[k].ravel()) for k in range(2)])}


def run_season_tangent_drift(forcing, ic, mask, dx, p, f, dD, num_steps=None):
    """Tangents (T, 2, ny, nx) of the season in the drift direction ``dD`` (T, 2, ny, nx): the transported tangent of
    ``score_adjoint.tangent_step_ic`` plus the drift's own raw terms d adv_l = -((dut gx(h_l)) + (dvt gy(h_l))) and
    d div_l = -((h_l gx(dut)) + (h_l gy(dvt))) (dut = du dT), each 0 where the primal raw term was not finite, smoothed,
    0 on land and where the primal killed the new depth.  The IC does not depend on the drift."""
    T, ny, nx = forcing["precip"].shape
    s = O.gen_empty_arrays(T, ny, nx)
    temp = np.full((ny, nx), np.nan)
    half = O.initial_depths(ic, forcing["conc"][0], p)
    s["snowDepths"][0, 0] = half
    s["snowDepths"][0, 1] = half
    tan = np.zeros((T, 2, ny, nx))
    steps = T - 1 if num_steps is None else num_steps
    for x in range(steps):
        P, C, W, D = forcing["precip"][x], forcing["conc"][x], forcing["wind"][x], forcing["drift"][x]
        hx = s["snowDepths"][x]
        tan[x + 1] = tangent_step_ic(hx, tan[x], C, P, D, W, mask, dx, p, f)
        if f.dynamicsInc == 1:
            kill0, kill1, fin_a, fin_d = step_record(hx, C, P, D, W, mask, dx, p, f)
            with np.errstate(all="ignore"):
                dut, dvt = dD[x, 0] * p.deltaT, dD[x, 1] * p.deltaT
                gxu, gyv = np.gradient(dut, dx, axis=1), np.gradient(dvt, dx, axis=0)
                for l, kill in enumerate((kill0, kill1)):
                    da = np.where(fin_a[l], -((dut * np.gradient(hx[l], dx, axis=1)) +
                                              (dvt * np.gradient(hx[l], dx, axis=0))), 0.0)
                    dd = np.where(fin_d[l], -((hx[l] * gxu) + (hx[l] * gyv)), 0.0)
                    src = O.smooth_snow(da, f.conv_variant) + O.smooth_snow(dd, f.conv_variant)
                    tan[x + 1, l] = np.where(kill, 0.0, tan[x + 1, l] + src)
        O.calc_budget(s, C, P, D, W, temp, mask, dx, x, p, f)
    return s, tan


def objective_tangent_drift(forcing, ic, mask, dx, p, f, obs, fps, w, fw, dD, num_steps=None):
    """dJ of one member along the drift direction ``dD`` (T, 2, ny, nx) by the forward mode, for the dot-product
    identity."""
    T = forcing["precip"].shape[0]
    L = T - 1 if num_steps is None else num_steps
    s, tan = run_season_tangent_drift(forcing, ic, mask, dx, p, f, dD, L)
    conc = forcing["conc"]
    sd, tan, density = s["snowDepths"][:L + 1], tan[:L + 1], s["density"][:L + 1]
    dC = np.zeros(conc.shape)
    dJ = 0.0
    with np.errstate(all="ignore"):
        if obs is not None and len(obs["day"]):
            v = model_values(sd, density, conc, obs, mask)
            dv = _dv(sd, tan, conc, dC, obs, mask, p)
            r = (v - np.asarray(obs["value"], dtype=np.float64)) / np.asarray(obs["sigma"], dtype=np.float64)
            k = np.asarray(obs["kind"])
            for q in order(obs, mask):
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
