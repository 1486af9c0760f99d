"""GPU: the calibration adjoint (nesosim_run_season_score_adjoint: the record build of the scoring day kernel, the
seeds, the backward day kernel and the finish).  ic_grad and theta_grad are bit-identical to the restatement
(oracle/score_adjoint.py) for both CTA shapes, the land-tile shortcut on and off, dynamics on and off, per-member ICs
finite on land, forcing sets with short seasons (each season's last day observed) and wide, ragged and coastline grids;
the scores are bit-identical to nesosim_run_season_scores_fp; theta_grad agrees with the forward-mode gradients; also
determinism, the launch count and the errors.  Ice and finite drift on the grid edges (the one-sided differences, the
backward kernel's edge divisors and E term): test_grid_edges_gpu.py."""
import functools

import numpy as np
import pytest

from nesosim_b200 import _lib
from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_adjoint as A
from test_general_scores_gpu import (WIDE, clear_env, engine, make_footprints, make_obs, oracle_params, same)

pytestmark = pytest.mark.gpu

FLAGS = dict(atmlossInc=1)
W, FW = (1.0, 0.5, 2.0), (0.25, 1.0, 0.0)


def land_ic(mask, ic):
    return np.where(R.ocean(mask), ic, 0.3)               # finite IC on land: day 0's dynamics read it


def adjoint(eng, params, ic, obs, fps, obs_set=None, fp_set=None):
    eng.set_observations_fp(obs, fps, obs_set=obs_set, fp_set=fp_set)
    r = eng.run_season_score_adjoint(params, ic, W, FW, model=True)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in r.items()}


def check_member(got, m, forcing, ic_m, mask, dx, prow, obs, fps, dynamics=1):
    p = oracle_params(prow)
    f = O.Flags(dynamicsInc=dynamics, atmlossInc=1)
    theta, icg, _ = A.score_adjoint(forcing, ic_m, mask, dx, p, f, obs, fps, W, FW)
    assert same(got["theta_grad"][m], theta), (m, got["theta_grad"][m], theta)
    assert same(got["ic_grad"][m], icg), (m, np.abs(got["ic_grad"][m] - icg).max())
    return icg


@functools.lru_cache(maxsize=None)
def disc_case():
    mask, dx, T, M = S.region_mask(dx=100000), 100000, 12, 3
    rng = np.random.default_rng(170)
    forcing = S.make_season(mask, T, seed=171)
    forcing["conc"][0][~R.ocean(mask)] = 0.9              # keeps the IC on land (conc[0] >= minConc)
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=172))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=173)
    return mask, dx, T, M, forcing, ic, params, make_obs(mask, T, rng, 700), make_footprints(mask, T, rng)


@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("land", [0, 1])
@pytest.mark.parametrize("dynamics", [0, 1])
def test_adjoint_bit_for_bit_against_the_oracle(cuda, monkeypatch, threads, land, dynamics):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_DAY_THREADS", str(threads))
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", str(land))
    mask, dx, T, M, forcing, ic, params, obs, fps = disc_case()
    eng = engine(mask, dx, T, M, [forcing], path="general", dynamicsInc=dynamics, **FLAGS)
    got = adjoint(eng, params, ic, obs, fps)
    eng.set_observations_fp(obs, fps)
    plain = [t.cpu().numpy() for t in eng.run_season_scores_fp(params, ic, model=True)]
    eng.close()
    for name, want in zip(("chi2", "used", "model", "fp_chi2", "fp_used", "fp_model"), plain):
        assert same(got[name], want), name
    for m in range(M):
        icg = check_member(got, m, forcing, ic[m], mask, dx, params[m], obs, fps, dynamics)
        if dynamics:
            assert np.abs(icg[~R.ocean(mask)]).max() > 0
    assert np.abs(got["theta_grad"]).max() > 0


def test_forcing_sets_with_short_seasons(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    days, member_set = [9, 13, 6], [2, 0, 1, 1, 0]
    T, M = max(days), len(member_set)
    rng = np.random.default_rng(180)
    seasons = [S.make_season(mask, d, seed=181 + s) for s, d in enumerate(days)]
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=184))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=185)
    obs = [make_obs(mask, d, rng, 300) for d in days]
    fps = [make_footprints(mask, d, rng) for d in days]
    cat = {k: np.concatenate([o[k] for o in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(obs)])
    fcat = {k: np.concatenate([np.asarray(f[k]) for f in fps]) for k in ("kind", "value", "sigma", "day", "row", "col",
                                                                          "weight")}
    fcat["begin"] = np.concatenate([[0], np.cumsum(np.concatenate([np.diff(f["begin"]) for f in fps]))]).astype(np.int64)
    ftag = np.concatenate([np.full(len(f["value"]), i, dtype=np.int32) for i, f in enumerate(fps)])
    eng = engine(mask, dx, T, M, seasons, member_set, days, path="general", **FLAGS)
    got = adjoint(eng, params, ic, cat, fcat, tag, ftag)
    eng.close()
    for m, s in enumerate(member_set):
        assert (obs[s]["day"] == days[s] - 1).any()
        check_member(got, m, seasons[s], ic[m], mask, dx, params[m], obs[s], fps[s])


@pytest.mark.parametrize("grid", list(WIDE))
def test_wide_grids_bit_for_bit_against_the_oracle(cuda, monkeypatch, grid):
    clear_env(monkeypatch)
    make, dx, T = WIDE[grid]
    mask = make()
    M = 2
    rng = np.random.default_rng(190)
    forcing = S.make_season(mask, T, seed=191)
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=192))[None] * rng.uniform(0.5, 2.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=193)
    obs, fps = make_obs(mask, T, rng, 600), make_footprints(mask, T, rng)
    eng = engine(mask, dx, T, M, [forcing], path="general", **FLAGS)
    got = adjoint(eng, params, ic, obs, fps)
    eng.close()
    for m in range(M):
        check_member(got, m, forcing, ic[m], mask, dx, params[m], obs, fps)


def test_against_forward_mode(cuda, monkeypatch):
    """theta_grad = sum_k w_k grad[k] + sum_k fw_k fp_grad[k] of the tangent build, up to summation order."""
    clear_env(monkeypatch)
    mask, dx, T, M, forcing, ic, params, obs, fps = disc_case()
    eng = engine(mask, dx, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    fwd = {k: (None if v is None else v.cpu().numpy()) for k, v in eng.run_season_score_grads(params, ic).items()}
    adj = eng.run_season_score_adjoint(params, ic, W, FW)["theta_grad"].cpu().numpy()
    eng.close()
    want = np.einsum("k,mkd->md", W, fwd["grad"]) + np.einsum("k,mkd->md", FW, fwd["fp_grad"])
    rel = np.abs(adj - want).max(axis=1) / np.abs(want).max(axis=1)
    assert (rel <= 1e-10).all(), rel


def test_launches_determinism_and_errors(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask = S.region_mask(shape=(40, 130), kind="disc")
    T, M = 7, 3
    rng = np.random.default_rng(200)
    forcing = S.make_season(mask, T, seed=201)
    params = S.ensemble_params(M, seed=202)
    ic = S.make_ic(mask, seed=203)
    obs, fps = make_obs(mask, T, rng, 300), make_footprints(mask, T, rng)
    eng = engine(mask, 50000, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    l0 = eng.launch_count()
    a = {k: v.cpu().numpy() for k, v in eng.run_season_score_adjoint(params, ic, W, FW, model=True).items()}
    assert eng.launch_count() - l0 == 2 * T + 5          # documented: 2T+4, 2T+5 with footprints
    b = eng.run_season_score_adjoint(params, ic, W, FW, model=True)
    assert all(same(a[k], v.cpu().numpy()) for k, v in b.items())
    assert a["theta_grad"].shape == (M, 3) and a["ic_grad"].shape == (M,) + mask.shape
    lib, h = eng.lib, eng.handle
    p = _lib.member_params_array(params)
    buf = {k: eng._dev(np.zeros_like(v)) for k, v in a.items()}
    ptr = lambda k: buf[k].data_ptr()
    K = _lib.OBS_KINDS
    ok = (C_double3(W), C_double3(FW))

    def call(w=ok[0], fw=ok[1], theta=True, icg=True, fp_chi2=True, model_stride=a["model"].shape[-1]):
        return lib.nesosim_run_season_score_adjoint(
            h, p, None, 0, w, fw, ptr("chi2"), ptr("used"), ptr("model"), model_stride,
            ptr("fp_chi2") if fp_chi2 else None, ptr("fp_used"), None, 0, ptr("theta_grad") if theta else None,
            ptr("ic_grad") if icg else None, None)
    assert call() == _lib.OK
    assert call(theta=False) == _lib.ERR_ARG and call(icg=False) == _lib.ERR_ARG
    assert call(w=C_double3((1.0, -1.0, 1.0))) == _lib.ERR_ARG
    assert call(fw=C_double3((1.0, float("nan"), 1.0))) == _lib.ERR_ARG
    assert call(model_stride=a["model"].shape[-1] - 1) == _lib.ERR_ARG
    assert call(fp_chi2=False) == _lib.ERR_STATE
    c = eng.run_season_score_adjoint(params, ic, W, FW, model=True)     # the registration is intact
    assert all(same(a[k], v.cpu().numpy()) for k, v in c.items())
    assert K == 3
    for path in ("auto", "ensemble"):
        eng.set_path(path)
        with pytest.raises(_lib.NesosimError) as e:
            eng.run_season_score_adjoint(params, ic)
        assert e.value.code == _lib.ERR_STATE
    eng.close()


def C_double3(v):
    import ctypes as C
    return (C.c_double * 3)(*v)


@pytest.mark.parametrize("km,M", [(100, 128), (25, 16)])
def test_against_forward_mode_at_scale(cuda, monkeypatch, km, M):
    """The same agreement on 260-day seasons with 20 000 observations and footprints, where theta_grad sums every
    member-cell-day in an order unlike the forward mode's."""
    clear_env(monkeypatch)
    mask, dx, T = S.region_mask(dx=km * 1000), km * 1000, 260
    rng = np.random.default_rng(210 + km)
    forcing = S.make_season(mask, T, seed=211)
    params = S.ensemble_params(M, seed=212)
    ic = S.make_ic(mask, seed=213)
    obs, fps = make_obs(mask, T, rng, 20000), make_footprints(mask, T, rng)
    eng = engine(mask, dx, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    fwd = {k: (None if v is None else v.cpu().numpy()) for k, v in eng.run_season_score_grads(params, ic).items()}
    adj = eng.run_season_score_adjoint(params, ic, W, FW)["theta_grad"].cpu().numpy()
    eng.close()
    want = np.einsum("k,mkd->md", W, fwd["grad"]) + np.einsum("k,mkd->md", FW, fwd["fp_grad"])
    rel = np.abs(adj - want).max(axis=1) / np.abs(want).max(axis=1)
    print("largest relative difference to forward mode at %d km, M = %d: %.3e" % (km, M, rel.max()))
    assert (rel <= 1e-10).all(), rel
