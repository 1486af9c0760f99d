"""CPU: the calibration adjoint with respect to the forcing without a device -- the reverse-mode restatement
(oracle/forcing_adjoint.py) against the forward tangent in random forcing directions (dot-product identity) and
against central differences of the primal objective; the scale fields against the per-day stacks; the engine's, the
driver's and the native entry point's argument checks; the gather of the forcing derivatives over two gloo ranks."""
import dataclasses
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nesosim_b200 import _lib
from nesosim_b200 import ensemble as ENS
from nesosim_b200 import synthetic as S
from nesosim_b200.engine import SnowBudgetEngine
from oracle import footprint_scores as F
from oracle import forcing_adjoint as FA
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_adjoint as A
from oracle import score_gradients as G
from test_score_adjoint_cpu import make_case as adj_case
from test_score_adjoint_cpu import point_obs, season

DX = 100000
NAMES = FA.FIELDS

CASES = {
    "nan_precip": dict(base="disc_land_ic", nan_precip=True),
    "low_conc0": dict(base="disc_land_ic", low_conc0=True),
    "edge_ocean": dict(base="edge_ocean"),
    "no_dynamics": dict(base="no_dynamics"),
    "no_windpack": dict(base="no_windpack"),
    "no_leadloss": dict(base="no_leadloss"),
    "no_atmloss": dict(base="no_atmloss"),
    "no_lead_no_atm": dict(base="disc_land_ic", f={"leadlossInc": 0, "atmlossInc": 0}),
    "zero_weights": dict(base="zero_weights"),
    "density_near_min": dict(base="density_near_min"),
}


def make_case(name, T=8, seed=3):
    c = CASES[name]
    mask, forcing, ic, p, f, obs, fps, w, fw = adj_case(c["base"], T, seed)
    if c.get("f"):
        f = dataclasses.replace(f, **c["f"])
    if c.get("nan_precip"):
        forcing["precip"][3, 4:7, 8:12] = np.nan
        forcing["precip"][0, 10:12, 3:6] = np.nan
    if c.get("low_conc0"):
        forcing["conc"][0, 6:9, 6:12] = 0.1
    return mask, forcing, ic, p, f, obs, fps, w, fw


def directions(forcing, seed=11):
    rng = np.random.default_rng(seed)
    out = []
    for n in NAMES:
        d = rng.standard_normal(forcing[n].shape) * np.nanstd(forcing[n])
        out.append(np.where(np.isfinite(forcing[n]), d, 0.0))
    return out


def identity(forcing, ic, mask, p, f, obs, fps, w, fw, num_steps=None):
    got = FA.score_adjoint_forcing(forcing, ic, mask, DX, p, f, obs, fps, w, fw, num_steps=num_steps)
    d = directions(forcing)
    lhs = float(sum(np.sum(got[n + "_day_grad"] * d[i]) for i, n in enumerate(NAMES)))
    rhs = FA.objective_tangent_forcing(forcing, ic, mask, DX, p, f, obs, fps, w, fw, *d, num_steps=num_steps)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs), 1e-300), (lhs, rhs)
    return got


@pytest.mark.parametrize("name", list(CASES))
def test_dot_product_identity(name):
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case(name)
    assert set(range(R.KINDS)) <= set(np.asarray(obs["kind"]).tolist())
    assert set(range(R.KINDS)) - {R.VOLUME} <= set(np.asarray(fps["kind"]).tolist())
    got = identity(forcing, ic, mask, p, f, obs, fps, w, fw)
    for n in NAMES:
        assert np.isfinite(got[n + "_day_grad"]).all()
    assert not got["precip_day_grad"][-1].any() and not got["wind_day_grad"][-1].any()
    if f.leadlossInc == 0 and f.atmlossInc == 0:
        assert not got["wind_day_grad"].any()
    else:
        assert np.abs(got["wind_day_grad"]).max() > 0
    assert np.abs(got["precip_day_grad"]).max() > 0 and np.abs(got["conc_day_grad"]).max() > 0
    if CASES[name].get("nan_precip"):
        assert not got["precip_day_grad"][3, 4:7, 8:12].any()
        assert np.isfinite(got["forcing_scale_grad"]).all()
    # the existing outputs are those of score_adjoint
    theta, icg, _ = A.score_adjoint(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    assert np.array_equal(theta, got["theta_grad"]) and np.array_equal(icg, got["ic_grad"])


def test_scale_fields_are_the_per_day_stacks_resummed():
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case("nan_precip")
    got = FA.score_adjoint_forcing(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    T = forcing["precip"].shape[0]
    for i, n in enumerate(NAMES):
        acc = np.zeros(mask.shape)
        with np.errstate(invalid="ignore"):
            for x in range(T - 1, -1, -1):
                acc = acc + np.where(np.isfinite(forcing[n][x]), forcing[n][x] * got[n + "_day_grad"][x], 0.0)
        assert np.array_equal(acc.view(np.int64), got["forcing_scale_grad"][i].view(np.int64)), n
        assert got["forcing_scale_total"][i] == R.fixed_order_sum(acc.ravel())


def objective(forcing, ic, mask, p, f, obs, fps, w, fw):
    st = O.run_season(forcing, ic, mask, DX, p, f)
    mv = R.model_values(st["snowDepths"], st["density"], forcing["conc"], obs, mask)
    chi2, used = R.scores(mv, obs, mask)
    fm = F.footprint_values(st["snowDepths"], st["density"], forcing["conc"], fps, mask)
    fchi2, fused = F.footprint_scores(fm, fps)
    kinks = (np.isnan(st["snowDepths"]), st["snowDepths"] == 0.0, used, fused)
    return float(np.dot(w, chi2) + np.dot(fw, fchi2)), kinks


def same_kinks(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def test_central_differences():
    mask, forcing, ic, p, f, obs, fps, w, fw = adj_case("disc_land_ic")
    p = dataclasses.replace(p, leadLossFactor=2.9e-7, atmLossFactor=2.2e-8)   # no clamp moves at 1 +- h
    obs = {k: v[obs["kind"] != R.DENSITY] for k, v in obs.items()}
    # winds on both sides of the threshold, none within a relative 1e-3 of it
    W = forcing["wind"]
    near = np.abs(W - p.windPackThresh) < 1e-3 * p.windPackThresh
    forcing["wind"] = np.where(near, p.windPackThresh * 1.01, W)
    assert (forcing["wind"] > p.windPackThresh).any() and (forcing["wind"] < p.windPackThresh).any()
    forcing["conc"] = np.where(np.abs(forcing["conc"] - p.minConc) < 1e-3, p.minConc + 0.01, forcing["conc"])
    got = FA.score_adjoint_forcing(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    _, base = objective(forcing, ic, mask, p, f, obs, fps, w, fw)
    h = 1e-4
    checked = 0
    for i, n in enumerate(NAMES):
        vals = []
        ok = True
        for sg in (1, -1):
            fc = dict(forcing)
            fc[n] = forcing[n] * (1.0 + sg * h)
            val, k = objective(fc, ic, mask, p, f, obs, fps, w, fw)
            ok = ok and same_kinks(base, k)
            vals.append(val)
        if not ok:
            continue
        fd = (vals[0] - vals[1]) / (2 * h)
        assert np.isclose(got["forcing_scale_total"][i], fd, rtol=1e-6, atol=1e-9 * abs(fd)), (n, got["forcing_scale_total"][i], fd)
        checked += 1
    assert checked == 3
    # per-cell factors on a few cells with the largest snowfall sensitivity
    sg0 = got["forcing_scale_grad"][0]
    cells = np.argsort(-np.abs(sg0).ravel())[:6]
    checked = 0
    for cell in cells:
        r, c = np.unravel_index(cell, mask.shape)
        vals = []
        ok = True
        for sg in (1, -1):
            fc = dict(forcing)
            fc["precip"] = forcing["precip"].copy()
            fc["precip"][:, r, c] *= 1.0 + sg * h
            val, k = objective(fc, ic, mask, p, f, obs, fps, w, fw)
            ok = ok and same_kinks(base, k)
            vals.append(val)
        if not ok:
            continue
        fd = (vals[0] - vals[1]) / (2 * h)
        assert np.isclose(sg0[r, c], fd, rtol=1e-6, atol=1e-6 * np.abs(sg0).max()), (r, c, sg0[r, c], fd)
        checked += 1
    assert checked >= 3


def test_short_season_with_last_day_observed():
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case("nan_precip", T=8)
    L = 5
    keep = obs["day"] <= L
    obs = {k: v[keep] for k, v in obs.items()}
    obs["day"][:20] = L
    obs["kind"][:20] = R.DEPTH
    got = identity(forcing, ic, mask, p, f, obs, None, w, fw, num_steps=L)
    short = {k: v[:L + 1] for k, v in forcing.items()}
    ref = FA.score_adjoint_forcing(short, ic, mask, DX, p, f, obs, None, w, fw)
    for k in ("theta_grad", "ic_grad", "forcing_scale_grad", "forcing_scale_total"):
        assert np.array_equal(got[k], ref[k]), k
    for n in NAMES:
        assert np.array_equal(got[n + "_day_grad"][:L + 1], ref[n + "_day_grad"])
        assert not got[n + "_day_grad"][L + 1:].any()
    assert np.abs(got["conc_day_grad"][L]).max() > 0 and not got["precip_day_grad"][L].any()


def test_engine_and_driver_reject_bad_requests():
    fake = types.SimpleNamespace()       # no context: the checks run before any device work
    for kw in (dict(forcing_days=("precip",)), dict(forcing=True, forcing_days=("snow",)),
               dict(forcing_days=("wind", "ice"))):
        with pytest.raises(ValueError, match="forcing_days"):
            SnowBudgetEngine.run_season_score_adjoint(fake, np.zeros((1, 4)), None, **kw)
    mask, forcing, ic = season(T=4)
    seasons = [{"forcing": forcing, "ic": ic, "obs": point_obs(mask, 4, np.random.default_rng(5), 20)}]
    params = S.ensemble_params(2, seed=6)
    with pytest.raises(ValueError, match="forcing_grad"):
        ENS.run_calibration_scores(mask, seasons, params, DX, forcing_grad=True)
    with pytest.raises(ValueError, match="forcing_grad"):
        ENS.run_calibration_scores(mask, seasons, params, DX, grad=True, forcing_grad=True)


def test_native_entry_point_validates_its_arguments(lib):
    assert lib.nesosim_run_season_score_adjoint_forcing(None, None, None, 0, None, None, None, None, None, 0, None,
                                                        None, None, 0, None, None, None, None, None, None, None,
                                                        None) == _lib.ERR_ARG
    assert "nesosim_run_season_score_adjoint_forcing" in _lib.EXPORTED_SYMBOLS
    assert _lib.FORCING_DIRS == len(_lib.FORCING_FIELDS) == 3 and _lib.FORCING_FIELDS == NAMES


def member_rows(p, s, shape):
    g = np.full((3,) + shape, 100.0 * p + s) + np.arange(3 * np.prod(shape)).reshape((3,) + shape) / 1000.0
    return g, np.array([1.0, 2.0, 3.0]) + 10.0 * p + s


def _worker(rank, world, port, P, S_, shape, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rows = [member_rows(p, s, shape) for p, s in ENS.calibration_plan(P, S_, rank, world)["pairs"]]
    g = torch.tensor(np.array([r[0] for r in rows]).reshape((-1, 3) + shape))
    t = torch.tensor(np.array([r[1] for r in rows]).reshape(-1, 3))
    got = ENS.gather_forcing_grad(g, t, P, S_, rank, world)
    q.put((rank, got))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_gather_the_same_forcing_gradients():
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
        assert got["forcing_scale_grad"].shape == (P, S_, 3) + shape and got["forcing_scale_total"].shape == (P, S_, 3)
        for p in range(P):
            for s in range(S_):
                g, t = member_rows(p, s, shape)
                assert np.array_equal(got["forcing_scale_grad"][p, s], g)
                assert np.array_equal(got["forcing_scale_total"][p, s], t)
