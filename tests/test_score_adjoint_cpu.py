"""CPU: the calibration adjoint without a device -- the reverse-mode restatement (oracle/score_adjoint.py) against the
initial-condition and parameter tangents (dot-product identity), central differences of the primal oracle and the
forward-mode gradients; the driver's argument checks and the gather of the adjoint results over two gloo ranks."""
import dataclasses
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nesosim_b200 import _lib
from nesosim_b200 import ensemble as ENS
from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_adjoint as A
from oracle import score_gradients as G

FIELDS = G.PARAM_FIELDS
DX = 100000


def season(T=9, seed=1, shape=(20, 26), kind="disc"):
    mask = S.region_mask(shape=shape, kind="disc")
    if kind == "all_ocean":                               # ocean on every grid edge: the one-sided differences
        mask = np.full(shape, 8, np.uint8)
        mask[5:8, 6:9] = 11
    forcing = S.make_season(mask, T, seed=seed)
    forcing["wind"] = forcing["wind"] * 1.5
    ic = 0.05 + S.make_ic(mask, seed=seed)
    return mask, forcing, ic


def point_obs(mask, T, rng, n=300, day0=1):
    wet = np.argwhere(R.ocean(mask))
    cell = wet[rng.integers(len(wet), size=n)]
    day = rng.integers(day0, T, n)
    kind = rng.integers(0, R.KINDS, n)
    day = np.where(kind == R.DENSITY, np.maximum(day, 1), day)
    value = np.where(kind == R.DENSITY, 250.0 + 50 * rng.random(n), 0.2 * rng.random(n))
    return {"day": day, "row": cell[:, 0], "col": cell[:, 1], "kind": kind, "value": value,
            "sigma": rng.uniform(0.01, 1.0, n) * np.where(kind == R.DENSITY, 100.0, 1.0)}


def footprints(mask, T):
    regions = [k for k in range(1, 11) if (mask == k).any()][:2]
    a = ENS.region_footprints(mask, regions, [(1, T // 2), (T // 2, T)], R.DEPTH, [0.2, 0.25], 0.05)
    b = ENS.region_footprints(mask, regions[:1], [(1, T)], R.DENSITY, [300.0], 30.0)
    return _concat(a, b)


def _concat(a, b):
    n = len(a["begin"]) - 1
    out = {k: np.concatenate([np.asarray(a[k]), np.asarray(b[k])]) for k in ("kind", "value", "sigma", "day", "row",
                                                                                 "col", "weight")}
    out["begin"] = np.concatenate([np.asarray(a["begin"]), np.asarray(b["begin"])[1:] + np.asarray(a["begin"])[n]])
    return out


def objective_tangent(forcing, ic, mask, p, f, obs, fps, w, fw, v):
    """dJ along the IC direction v, and per parameter (forward mode of score_gradients)."""
    s, tan = A.run_season_tangent_ic(forcing, ic, v, mask, DX, p, f)
    tan3 = np.repeat(tan[:, None], G.DIRS, axis=1)
    s2, ptan = G.run_season_tangent(forcing, ic, mask, DX, p, f)
    out = []
    for t in (tan3, ptan):
        g = np.zeros(G.DIRS)
        if obs is not None:
            mv = R.model_values(s["snowDepths"], s["density"], forcing["conc"], obs, mask)
            dv = G.model_tangents(s["snowDepths"], t, forcing["conc"], obs, mask, p)
            g += np.asarray(w) @ G.score_gradients(mv, dv, obs, mask)
        if fps is not None:
            mean, dmean = G.footprint_tangents(s["snowDepths"], s["density"], t, forcing["conc"], fps, mask, p)
            g += np.asarray(fw) @ G.footprint_gradients(mean, dmean, fps)
        out.append(g)
    return out[0][0], out[1]


CASES = {
    "edge_ocean": dict(shape=(14, 18), kind="all_ocean", f={}),
    "disc_land_ic": dict(shape=(20, 26), kind="disc", f={}),
    "nan_patch": dict(shape=(20, 26), kind="disc", f={}, nan=True),
    "no_dynamics": dict(shape=(20, 26), kind="disc", f={"dynamicsInc": 0}),
    "no_windpack": dict(shape=(20, 26), kind="disc", f={"windpackInc": 0}),
    "no_leadloss": dict(shape=(20, 26), kind="disc", f={"leadlossInc": 0}),
    "no_atmloss": dict(shape=(20, 26), kind="disc", f={"atmlossInc": 0}),
    "zero_weights": dict(shape=(20, 26), kind="disc", f={}, w=(1.0, 0.0, 2.0), fw=(0.0, 1.0, 0.5)),
    "density_near_min": dict(shape=(20, 26), kind="disc", f={}, near_min=True),
}


def density_near_min_snow(forcing, ic, mask, p, f, rng, n=120):
    """Density observations on ocean cell-days whose total depth lies within a factor 2 of minSnowD, on both sides:
    some counted (h0 + h1 >= minSnowD, near the operator's NaN edge), some not (below it)."""
    s = O.run_season(forcing, ic, mask, DX, p, f)
    tot = s["snowDepths"][1:, 0] + s["snowDepths"][1:, 1]
    with np.errstate(invalid="ignore"):
        near = np.argwhere((tot > 0.5 * p.minSnowD) & (tot < 2.0 * p.minSnowD) & R.ocean(mask)[None])
    pick = near[rng.choice(len(near), size=min(n, len(near)), replace=False)]
    picked = tot[pick[:, 0], pick[:, 1], pick[:, 2]]
    assert (picked >= p.minSnowD).sum() >= 5 and (picked < p.minSnowD).sum() >= 5
    m = len(pick)
    return {"day": pick[:, 0] + 1, "row": pick[:, 1], "col": pick[:, 2], "kind": np.full(m, R.DENSITY),
            "value": 250.0 + 50 * rng.random(m), "sigma": rng.uniform(10.0, 100.0, m)}


def make_case(name, T=8, seed=3):
    c = CASES[name]
    mask, forcing, ic = season(T, seed, c["shape"], c["kind"])
    ic = np.where(R.ocean(mask), ic, 0.3)                 # finite IC on land: day 0's dynamics read it ...
    forcing["conc"][0][G.land(mask)] = 0.9                # ... where conc[0] >= minConc keeps it
    forcing["drift"] = np.where(np.isnan(forcing["drift"]), 0.01, forcing["drift"])   # drift up to the coast
    if c.get("nan"):
        forcing["wind"][2, 5:8, 6:10] = np.nan
        forcing["drift"][3, :, 9:11, 12:15] = np.nan
    # a strong loss so that the clamp at 0 fires on some days
    p = O.Params(windPackThresh=4.0, leadLossFactor=2.9e-6, atmLossFactor=2.2e-7)
    f = dataclasses.replace(O.Flags(atmlossInc=1), **c["f"])
    rng = np.random.default_rng(seed)
    if c.get("near_min"):      # a thin snowpack: many cell-days near minSnowD
        ic = ic * 0.3
    obs = point_obs(mask, T, rng, day0=0)
    if c.get("near_min"):
        near = density_near_min_snow(forcing, ic, mask, p, f, rng)
        obs = {k: np.concatenate([np.asarray(obs[k]), np.asarray(near[k])]) for k in obs}
    fps = footprints(mask, T)
    return mask, forcing, ic, p, f, obs, fps, c.get("w", (1.0, 1.0, 1.0)), c.get("fw", (1.0, 1.0, 1.0))


@pytest.mark.parametrize("name", list(CASES))
def test_dot_product_identity(name):
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case(name)
    theta, icg, s = A.score_adjoint(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    rec = A.run_season_record(forcing, ic, mask, DX, p, f)[1]
    assert any(r[0][~G.land(mask)].any() for r in rec[1:]) or name == "no_leadloss"   # kills on ocean cells
    if f.dynamicsInc:
        assert np.abs(icg[G.land(mask)]).max() > 0        # finite IC on land reaches the objective
    rng = np.random.default_rng(7)
    v = rng.standard_normal(mask.shape)
    e = rng.standard_normal(G.DIRS)
    d_ic, d_th = objective_tangent(forcing, ic, mask, p, f, obs, fps, w, fw, v)
    lhs = float(np.sum(icg * v) + theta @ e)
    rhs = float(d_ic + d_th @ e)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs), 1e-300), (lhs, rhs)
    assert np.allclose(theta, d_th, rtol=1e-12, atol=1e-12 * np.abs(d_th).max())


def test_ic_grad_matches_central_differences():
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case("disc_land_ic")
    obs = {k: v[obs["kind"] != R.DENSITY] for k, v in obs.items()}
    theta, icg, s = A.score_adjoint(forcing, ic, mask, DX, p, f, obs, fps, w, fw)

    def J(ic_, p_):
        st = O.run_season(forcing, ic_, mask, DX, p_, f)
        mv = R.model_values(st["snowDepths"], st["density"], forcing["conc"], obs, mask)
        out = np.dot(w, R.scores(mv, obs, mask)[0])
        from oracle import footprint_scores as F
        fm = F.footprint_values(st["snowDepths"], st["density"], forcing["conc"], fps, mask)
        return out + np.dot(fw, F.footprint_scores(fm, fps)[0]), st

    def kinks(st):
        return np.isnan(st["snowDepths"]), st["snowDepths"] == 0.0

    base = kinks(s)
    cells = np.argwhere(np.abs(icg) > 1e-3 * np.abs(icg).max())
    checked = 0
    for r, c in cells[:: max(1, len(cells) // 12)]:
        h = 1e-4 * max(abs(ic[r, c]), 1e-3)
        vals = []
        ok = True
        for sg in (1, -1):
            q = ic.copy()
            q[r, c] += sg * h
            val, st = J(q, p)
            ok = ok and all(np.array_equal(a, b) for a, b in zip(base, kinks(st)))
            vals.append(val)
        if not ok:
            continue
        fd = (vals[0] - vals[1]) / (2 * h)
        assert np.isclose(icg[r, c], fd, rtol=1e-6, atol=1e-6 * np.abs(icg).max()), (r, c)
        checked += 1
    assert checked >= 5
    checked = 0
    for j, name in enumerate(FIELDS):
        h = 1e-4 * getattr(p, name)
        jp, sp = J(ic, dataclasses.replace(p, **{name: getattr(p, name) + h}))
        jm, sm = J(ic, dataclasses.replace(p, **{name: getattr(p, name) - h}))
        if not all(np.array_equal(a, b) and np.array_equal(a, cc) for a, b, cc in zip(base, kinks(sp), kinks(sm))):
            continue
        fd = (jp - jm) / (2 * h)
        assert np.isclose(theta[j], fd, rtol=1e-6, atol=1e-6 * np.abs(theta).max()), name
        checked += 1
    assert checked >= 2


def test_short_season_and_last_day_observations():
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case("disc_land_ic", T=8)
    L = 5
    keep = obs["day"] <= L
    obs = {k: v[keep] for k, v in obs.items()}
    obs["day"][:20] = L                                  # observed on the season's last day
    theta, icg, _ = A.score_adjoint(forcing, ic, mask, DX, p, f, obs, None, w, fw, num_steps=L)
    short = {k: (v[:L + 1] if k != "drift" else v[:L + 1]) for k, v in forcing.items()}
    theta2, icg2, _ = A.score_adjoint(short, ic, mask, DX, p, f, obs, None, w, fw)
    assert np.array_equal(theta, theta2) and np.array_equal(icg, icg2)


def test_driver_rejects_bad_adjoint_requests():
    mask, forcing, ic = season(T=4)
    seasons = [{"forcing": forcing, "ic": ic, "obs": point_obs(mask, 4, np.random.default_rng(5), 20)}]
    params = S.ensemble_params(2, seed=6)
    with pytest.raises(ValueError, match="adjoint"):
        ENS.run_calibration_scores(mask, seasons, params, DX, adjoint=True, grad=True)
    for fused in (True, False):
        with pytest.raises(ValueError, match="adjoint"):
            ENS.run_calibration_scores(mask, seasons, params, DX, adjoint=True, fused=fused)
    for bad in ([1.0, -1.0, 1.0], [1.0, np.nan, 1.0], [1.0, 1.0], [np.inf, 0.0, 0.0]):
        with pytest.raises(ValueError, match="weights"):
            ENS.run_calibration_scores(mask, seasons, params, DX, adjoint=True, weights=bad)
        with pytest.raises(ValueError, match="weights"):
            ENS.run_calibration_scores(mask, seasons, params, DX, adjoint=True, fp_weights=bad)
    with pytest.raises(ValueError, match="adjoint=True"):
        ENS.run_calibration_scores(mask, seasons, params, DX, weights=[1.0, 1.0, 1.0])


def test_native_entry_point_validates_its_arguments(lib):
    assert lib.nesosim_run_season_score_adjoint(None, None, None, 0, None, None, None, None, None, 0, None, None,
                                                None, 0, None, None, None) == _lib.ERR_ARG
    assert "nesosim_run_season_score_adjoint" in _lib.EXPORTED_SYMBOLS


def member_rows(p, s, shape):
    th = np.array([1.0, 2.0, 3.0]) + 10.0 * p + s
    icg = np.full(shape, 100.0 * p + s) + np.arange(np.prod(shape)).reshape(shape) / 1000.0
    return th, icg


def _worker(rank, world, port, P, S_, shape, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rows = [member_rows(p, s, shape) for p, s in ENS.calibration_plan(P, S_, rank, world)["pairs"]]
    th = torch.tensor(np.array([r[0] for r in rows]).reshape(-1, 3))
    icg = torch.tensor(np.array([r[1] for r in rows]).reshape((-1,) + shape))
    got = ENS.gather_adjoint(th, icg, P, S_, rank, world)
    q.put((rank, got))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_gather_the_same_adjoint():
    P, S_, world, shape = 3, 3, 2, (4, 5)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, P, S_, shape, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, got in results:
        assert got["adjoint_grad"].shape == (P, S_, 3) and got["ic_grad"].shape == (P, S_) + shape
        for p in range(P):
            for s in range(S_):
                th, icg = member_rows(p, s, shape)
                assert np.array_equal(got["adjoint_grad"][p, s], th)
                assert np.array_equal(got["ic_grad"][p, s], icg)
