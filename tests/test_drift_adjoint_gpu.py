"""GPU: the calibration adjoint with respect to the ice drift (nesosim_run_season_score_adjoint_drift: the drift builds
of the backward day and finish kernels).  The drift scale fields, their totals and the per-day stacks are bit-identical
to the restatement (oracle/drift_adjoint.py) for both CTA shapes, the land-tile shortcut on and off, dynamics on and
off and the drift NaN or finite over land (where land cells next to the ocean, all-land tiles included, carry
derivatives); the outputs the plain adjoint gives are bit-identical to it, and with the forcing terms too the forcing
outputs are bit-identical to nesosim_run_season_score_adjoint_forcing's; the scale outputs do not depend on the per-day
buffers.  Also forcing sets with short seasons, a wide ragged grid, the 100 km and 25 km edge grids, the driver, the
launch count, determinism and the errors."""
import ctypes as C
import functools

import numpy as np
import pytest

from nesosim_b200 import _lib
from nesosim_b200 import ensemble as ENS
from nesosim_b200 import synthetic as S
from oracle import drift_adjoint as DA
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_gradients as G
from test_calibration_switches_gpu import driver_seasons
from test_forcing_adjoint_gpu import DAY_KEYS, bits
from test_general_scores_gpu import WIDE, clear_env, engine, make_footprints, make_obs, oracle_params, same
from test_grid_edges_cpu import edge_case, edges
from test_score_adjoint_gpu import FLAGS, FW, W, disc_case, land_ic

pytestmark = pytest.mark.gpu

DRIFT_KEYS = ("drift_scale_grad", "drift_scale_total", "drift_day_grad")
FORCING_KEYS = ("forcing_scale_grad", "forcing_scale_total") + DAY_KEYS


def run(eng, params, ic, drift=True, drift_days=True, forcing=False):
    r = eng.run_season_score_adjoint(params, ic, W, FW, model=True, forcing=forcing,
                                     forcing_days=_lib.FORCING_FIELDS if forcing else (), drift=drift,
                                     drift_days=drift and drift_days)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in r.items()}


@functools.lru_cache(maxsize=None)
def drift_case(flavour):
    """disc_case with the drift NaN over land (as make_season leaves it) or finite there too."""
    mask, dx, T, M, forcing, ic, params, obs, fps = disc_case()
    forcing = dict(forcing)
    if flavour == "land_finite":
        yy, xx = np.mgrid[0:mask.shape[0], 0:mask.shape[1]]
        fill = np.stack([0.02 + 0.01 * np.sin(xx / 7.0), -0.01 + 0.01 * np.cos(yy / 5.0)])[None]
        forcing["drift"] = np.where(np.isnan(forcing["drift"]) & G.land(mask)[None, None], fill, forcing["drift"])
    return mask, dx, T, M, forcing, ic, params, obs, fps


@functools.lru_cache(maxsize=None)
def oracle_member(flavour, dynamics, m):
    mask, dx, T, M, forcing, ic, params, obs, fps = drift_case(flavour)
    f = O.Flags(dynamicsInc=dynamics, atmlossInc=1)
    return DA.score_adjoint_drift(forcing, ic[m], mask, dx, oracle_params(params[m]), f, obs, fps, W, FW)


def check_drift(got, m, want, T, days=True):
    for k in ("theta_grad", "ic_grad", "drift_scale_grad", "drift_scale_total") + (("drift_day_grad",) if days else ()):
        g = got[k][m]
        if k == "drift_day_grad":
            assert not g[T:].any(), k
            g = g[:T]
        assert bits(g, want[k]), (m, k, np.abs(g - want[k]).max())


def land_tiles(mask):
    """Cells of the day kernel's all-land tiles (32 x 16)."""
    ny, nx = mask.shape
    out = np.zeros(mask.shape, dtype=bool)
    wet = R.ocean(mask)
    for y in range(0, ny, 16):
        for x in range(0, nx, 32):
            if not wet[y:y + 16, x:x + 32].any():
                out[y:y + 16, x:x + 32] = True
    return out


@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("land", [0, 1])
@pytest.mark.parametrize("dynamics", [0, 1])
@pytest.mark.parametrize("flavour", ["land_nan", "land_finite"])
def test_drift_adjoint_bit_for_bit_against_the_oracle(cuda, monkeypatch, threads, land, dynamics, flavour):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_DAY_THREADS", str(threads))
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", str(land))
    mask, dx, T, M, forcing, ic, params, obs, fps = drift_case(flavour)
    eng = engine(mask, dx, T, M, [forcing], path="general", dynamicsInc=dynamics, **FLAGS)
    eng.set_observations_fp(obs, fps)
    got = run(eng, params, ic)
    both = run(eng, params, ic, forcing=True)
    scale_only = run(eng, params, ic, drift_days=False)
    plain = run(eng, params, ic, drift=False)
    with_forcing = run(eng, params, ic, drift=False, forcing=True)
    eng.close()
    for k, v in plain.items():                      # everything the plain adjoint gives, bit for bit
        for r in (got, both, scale_only):
            assert v is None or same(r[k], v), k
    for k in FORCING_KEYS:
        assert bits(both[k], with_forcing[k]), k
    for k in DRIFT_KEYS:
        assert bits(both[k], got[k]), k
    for k in ("drift_scale_grad", "drift_scale_total"):
        assert bits(got[k], scale_only[k]), k
    assert "drift_day_grad" not in scale_only
    for m in range(M):
        check_drift(got, m, oracle_member(flavour, dynamics, m), T)
    g = got["drift_day_grad"]
    if not dynamics:
        assert not any(got[k].any() or np.signbit(got[k]).any() for k in DRIFT_KEYS)
        return
    assert all(np.abs(got[k]).max() > 0 for k in DRIFT_KEYS)
    lnd = G.land(mask)
    on_land = (np.abs(g[:, 1:T - 1]) > 0).any(axis=(0, 1, 2)) & lnd
    if flavour == "land_finite":                    # the land-tile shortcut must not drop these
        assert on_land.sum() > 50
    else:
        assert not on_land.any()


def test_forcing_sets_with_short_seasons(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    days, member_set = [9, 13, 6], [2, 0, 1, 1, 0]
    T, M = max(days), len(member_set)
    rng = np.random.default_rng(380)
    seasons = [S.make_season(mask, d, seed=381 + s) for s, d in enumerate(days)]
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=384))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=385)
    obs = [make_obs(mask, d, rng, 300) for d in days]
    fps = [make_footprints(mask, d, rng) for d in days]
    cat = {k: np.concatenate([o[k] for o in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(obs)])
    fcat = {k: np.concatenate([np.asarray(f[k]) for f in fps]) for k in ("kind", "value", "sigma", "day", "row", "col",
                                                                          "weight")}
    fcat["begin"] = np.concatenate([[0], np.cumsum(np.concatenate([np.diff(f["begin"]) for f in fps]))]).astype(np.int64)
    ftag = np.concatenate([np.full(len(f["value"]), i, dtype=np.int32) for i, f in enumerate(fps)])
    eng = engine(mask, dx, T, M, seasons, member_set, days, path="general", **FLAGS)
    eng.set_observations_fp(cat, fcat, obs_set=tag, fp_set=ftag)
    got = run(eng, params, ic)
    eng.close()
    f = O.Flags(atmlossInc=1)
    for m, s in enumerate(member_set):
        assert (obs[s]["day"] == days[s] - 1).any()
        want = DA.score_adjoint_drift(seasons[s], ic[m], mask, dx, oracle_params(params[m]), f, obs[s], fps[s], W, FW)
        check_drift(got, m, want, days[s])
        assert not got["drift_day_grad"][m, days[s] - 1:].any()


def grid_case(grid):
    if grid in WIDE:
        make, dx, T = WIDE[grid]
        mask = make()
        rng = np.random.default_rng(390)
        forcing = S.make_season(mask, T, seed=391)
        ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=392))[None] * rng.uniform(0.5, 2.0, (2, 1, 1))
        return mask, dx, T, forcing, ic, S.ensemble_params(2, seed=393), make_obs(mask, T, rng, 600), \
            make_footprints(mask, T, rng)
    name, flavour = grid.split(":")
    return edge_case(name, flavour)


@pytest.mark.parametrize("grid", ["ragged", "coast_50x98:land_finite", "100km:land_nan", "100km:land_finite",
                                  "25km:land_nan", "25km:land_finite"])
def test_grids_bit_for_bit_against_the_oracle(cuda, monkeypatch, grid):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", "1")
    mask, dx, T, forcing, ic, params, obs, fps = grid_case(grid)
    M = len(params)
    eng = engine(mask, dx, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    got = run(eng, params, ic, forcing=True)
    eng.close()
    f = O.Flags(atmlossInc=1)
    for m in range(M):
        want = DA.score_adjoint_drift(forcing, ic[m], mask, dx, oracle_params(params[m]), f, obs, fps, W, FW)
        check_drift(got, m, want, T)
    wet = R.ocean(mask)
    g = got["drift_day_grad"]
    for e in edges(mask.shape) if ":" in grid else ():     # the edge grids' edge cells reached the objective
        if (e & wet).any():
            assert np.abs(g[..., e & wet]).max() > 0
    if grid == "coast_50x98:land_finite":           # an all-land tile next to the ocean, behind the land-tile shortcut
        on_land = (np.abs(g[:, 1:T - 1]) > 0).any(axis=(0, 1, 2)) & land_tiles(mask)
        assert on_land.sum() >= 2


def test_driver(cuda, monkeypatch):
    """run_calibration_scores(adjoint=True, drift_grad=True) gives, per pair, what the engine gives."""
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    seasons = [driver_seasons(mask, 660, days=(8, 9, 10))[s] for s in (0, 2)]
    params = S.ensemble_params(3, seed=661)
    res = ENS.run_calibration_scores(mask, seasons, params, dx, adjoint=True, forcing_grad=True, drift_grad=True,
                                     model=True)
    assert res["drift_scale_grad"].shape == (3, 2, 2) + mask.shape and res["drift_scale_total"].shape == (3, 2, 2)
    for s, season in enumerate(seasons):
        f = season["forcing"]
        eng = engine(mask, dx, len(f["precip"]), len(params), [f], path="general")
        eng.set_observations_fp(ENS.normalize_observations(season["obs"]), ENS.normalize_footprints(season["footprints"]))
        ad = {k: v.cpu().numpy() for k, v in eng.run_season_score_adjoint(params, season["ic"], forcing=True,
                                                                          drift=True).items() if v is not None}
        eng.close()
        for p in range(len(params)):
            assert same(res["adjoint_grad"][p, s], ad["theta_grad"][p]) and same(res["ic_grad"][p, s], ad["ic_grad"][p])
            for k in ("forcing_scale_grad", "forcing_scale_total", "drift_scale_grad", "drift_scale_total"):
                assert bits(res[k][p, s], ad[k][p]), (k, p, s)
        assert np.abs(ad["drift_scale_total"]).max() > 0


def test_launches_determinism_and_errors(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask = S.region_mask(shape=(40, 130), kind="disc")
    T, M = 7, 3
    rng = np.random.default_rng(400)
    forcing = S.make_season(mask, T, seed=401)
    params = S.ensemble_params(M, seed=402)
    ic = S.make_ic(mask, seed=403)
    obs, fps = make_obs(mask, T, rng, 300), make_footprints(mask, T, rng)
    eng = engine(mask, 50000, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    l0 = eng.launch_count()
    a = run(eng, params, ic, forcing=True)
    assert eng.launch_count() - l0 == 2 * T + 5          # the plain adjoint's 2T+4, 2T+5 with footprints
    b = run(eng, params, ic, forcing=True)
    assert all(bits(a[k], b[k]) for k in DRIFT_KEYS + FORCING_KEYS)
    assert all(same(a[k], b[k]) for k in a if k not in DRIFT_KEYS + FORCING_KEYS)
    assert a["drift_scale_grad"].shape == (M, 2) + mask.shape and a["drift_scale_total"].shape == (M, 2)
    assert a["drift_day_grad"].shape == (M, T, 2) + mask.shape
    lib, h = eng.lib, eng.handle
    p = _lib.member_params_array(params)
    buf = {k: eng._dev(np.zeros_like(v)) for k, v in a.items() if v is not None}
    ptr = lambda k: buf[k].data_ptr()
    cw, cfw = (C.c_double * 3)(*W), (C.c_double * 3)(*FW)

    def call(fscale=True, ftotal=True, fday=False, dscale=True, dtotal=True, dday=True, fp_chi2=True):
        return lib.nesosim_run_season_score_adjoint_drift(
            h, p, None, 0, cw, cfw, ptr("chi2"), ptr("used"), None, 0, ptr("fp_chi2") if fp_chi2 else None,
            ptr("fp_used"), None, 0, ptr("theta_grad"), ptr("ic_grad"), ptr("forcing_scale_grad") if fscale else None,
            ptr("forcing_scale_total") if ftotal else None, None, ptr("wind_day_grad") if fday else None, None,
            ptr("drift_scale_grad") if dscale else None, ptr("drift_scale_total") if dtotal else None,
            ptr("drift_day_grad") if dday else None, None)
    assert call() == _lib.OK and call(fscale=False, ftotal=False, dday=False) == _lib.OK
    assert call(dscale=False) == _lib.ERR_ARG and call(dtotal=False) == _lib.ERR_ARG
    assert call(fscale=False) == _lib.ERR_ARG and call(ftotal=False) == _lib.ERR_ARG
    assert call(fscale=False, ftotal=False, fday=True) == _lib.ERR_ARG
    assert call(fp_chi2=False) == _lib.ERR_STATE
    c = run(eng, params, ic, forcing=True)               # the registration and the state are intact
    assert all(bits(a[k], c[k]) for k in DRIFT_KEYS + FORCING_KEYS)
    eng.set_path("ensemble")
    with pytest.raises(_lib.NesosimError) as e:
        eng.run_season_score_adjoint(params, ic, drift=True)
    assert e.value.code == _lib.ERR_STATE
    eng.close()
