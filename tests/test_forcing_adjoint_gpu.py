"""GPU: the calibration adjoint with respect to the forcing (nesosim_run_season_score_adjoint_forcing: the forcing
builds of the seed, init, backward day and finish kernels).  The scale fields, their totals and the three per-day
gradient stacks are bit-identical to the restatement (oracle/forcing_adjoint.py) for both CTA shapes, the land-tile
shortcut on and off, dynamics on and off, forcing sets with short seasons and a wide, ragged grid; the outputs the
plain adjoint also gives are bit-identical to it; the scale outputs do not depend on the per-day buffers; also
determinism, the launch count and the errors.  Ice and finite drift on the grid edges: test_grid_edges_gpu.py."""
import ctypes as C

import numpy as np
import pytest

from nesosim_b200 import _lib
from nesosim_b200 import synthetic as S
from oracle import forcing_adjoint as FA
from oracle import nesosim_oracle as O
from test_general_scores_gpu import WIDE, clear_env, engine, make_footprints, make_obs, oracle_params, same
from test_score_adjoint_gpu import FLAGS, FW, W, disc_case, land_ic

pytestmark = pytest.mark.gpu

NAMES = _lib.FORCING_FIELDS
DAY_KEYS = tuple(n + "_day_grad" for n in NAMES)
FORCING_KEYS = ("forcing_scale_grad", "forcing_scale_total") + DAY_KEYS


def bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def run(eng, params, ic, days=NAMES, forcing=True):
    r = eng.run_season_score_adjoint(params, ic, W, FW, model=True, forcing=forcing, forcing_days=days)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in r.items()}


def check_member(got, m, forcing, ic_m, mask, dx, prow, obs, fps, dynamics=1, num_steps=None, days=True):
    f = O.Flags(dynamicsInc=dynamics, atmlossInc=1)
    want = FA.score_adjoint_forcing(forcing, ic_m, mask, dx, oracle_params(prow), f, obs, fps, W, FW, num_steps)
    for k in ("theta_grad", "ic_grad", "forcing_scale_grad", "forcing_scale_total") + (DAY_KEYS if days else ()):
        g = got[k][m]
        if k in DAY_KEYS:
            T = forcing["precip"].shape[0]
            assert not g[T:].any(), k
            g = g[:T]
        assert bits(g, want[k]), (m, k, np.abs(g - want[k]).max())
    return want


@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("land", [0, 1])
@pytest.mark.parametrize("dynamics", [0, 1])
def test_forcing_adjoint_bit_for_bit_against_the_oracle(cuda, monkeypatch, threads, land, dynamics):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_DAY_THREADS", str(threads))
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", str(land))
    mask, dx, T, M, forcing, ic, params, obs, fps = disc_case()
    eng = engine(mask, dx, T, M, [forcing], path="general", dynamicsInc=dynamics, **FLAGS)
    eng.set_observations_fp(obs, fps)
    got = run(eng, params, ic)
    plain = run(eng, params, ic, days=(), forcing=False)
    scale_only = run(eng, params, ic, days=())
    eng.close()
    for k, v in plain.items():                      # everything the plain adjoint gives, bit for bit
        assert v is None or same(got[k], v), k
    for k in ("forcing_scale_grad", "forcing_scale_total"):
        assert bits(got[k], scale_only[k]), k
    assert not any(k in scale_only for k in DAY_KEYS)
    for m in range(M):
        check_member(got, m, forcing, ic[m], mask, dx, params[m], obs, fps, dynamics)
    for k in FORCING_KEYS:
        assert np.abs(got[k]).max() > 0, k
    # the scale fields are the per-day stacks re-summed (days descending, non-finite forcing skipped)
    for i, n in enumerate(NAMES):
        acc = np.zeros((M,) + mask.shape)
        with np.errstate(invalid="ignore"):
            for x in range(T - 1, -1, -1):
                F = forcing[n][x][None]
                acc = acc + np.where(np.isfinite(F), F * got[n + "_day_grad"][:, x], 0.0)
        assert bits(acc, got["forcing_scale_grad"][:, i]), n


def test_forcing_sets_with_short_seasons(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    days, member_set = [9, 13, 6], [2, 0, 1, 1, 0]
    T, M = max(days), len(member_set)
    rng = np.random.default_rng(280)
    seasons = [S.make_season(mask, d, seed=281 + s) for s, d in enumerate(days)]
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=284))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=285)
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
    for m, s in enumerate(member_set):
        assert (obs[s]["day"] == days[s] - 1).any()
        L = days[s] - 1
        check_member(got, m, seasons[s], ic[m], mask, dx, params[m], obs[s], fps[s])
        assert not got["precip_day_grad"][m, L:].any() and not got["conc_day_grad"][m, L + 1:].any()
        assert np.abs(got["conc_day_grad"][m, L]).max() > 0


@pytest.mark.parametrize("grid", list(WIDE)[:1])
def test_wide_grid_bit_for_bit_against_the_oracle(cuda, monkeypatch, grid):
    clear_env(monkeypatch)
    make, dx, T = WIDE[grid]
    mask = make()
    M = 2
    rng = np.random.default_rng(290)
    forcing = S.make_season(mask, T, seed=291)
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=292))[None] * rng.uniform(0.5, 2.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=293)
    obs, fps = make_obs(mask, T, rng, 600), make_footprints(mask, T, rng)
    eng = engine(mask, dx, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    got = run(eng, params, ic)
    eng.close()
    for m in range(M):
        check_member(got, m, forcing, ic[m], mask, dx, params[m], obs, fps)


def test_launches_determinism_and_errors(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask = S.region_mask(shape=(40, 130), kind="disc")
    T, M = 7, 3
    rng = np.random.default_rng(300)
    forcing = S.make_season(mask, T, seed=301)
    params = S.ensemble_params(M, seed=302)
    ic = S.make_ic(mask, seed=303)
    obs, fps = make_obs(mask, T, rng, 300), make_footprints(mask, T, rng)
    eng = engine(mask, 50000, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    l0 = eng.launch_count()
    a = run(eng, params, ic)
    assert eng.launch_count() - l0 == 2 * T + 5          # the plain adjoint's 2T+4, 2T+5 with footprints
    b = run(eng, params, ic)
    assert all(bits(a[k], b[k]) for k in FORCING_KEYS)
    assert all(same(a[k], b[k]) for k in a if k not in FORCING_KEYS)
    assert a["forcing_scale_grad"].shape == (M, 3) + mask.shape and a["forcing_scale_total"].shape == (M, 3)
    assert all(a[k].shape == (M, T) + mask.shape for k in DAY_KEYS)
    lib, h = eng.lib, eng.handle
    p = _lib.member_params_array(params)
    buf = {k: eng._dev(np.zeros_like(v)) for k, v in a.items() if v is not None}
    ptr = lambda k: buf[k].data_ptr()
    cw, cfw = (C.c_double * 3)(*W), (C.c_double * 3)(*FW)

    def call(scale=True, total=True, fp_chi2=True):
        return lib.nesosim_run_season_score_adjoint_forcing(
            h, p, None, 0, cw, cfw, ptr("chi2"), ptr("used"), None, 0, ptr("fp_chi2") if fp_chi2 else None,
            ptr("fp_used"), None, 0, ptr("theta_grad"), ptr("ic_grad"), ptr("forcing_scale_grad") if scale else None,
            ptr("forcing_scale_total") if total else None, None, ptr("wind_day_grad"), None, None)
    assert call() == _lib.OK
    assert call(scale=False) == _lib.ERR_ARG and call(total=False) == _lib.ERR_ARG
    assert call(fp_chi2=False) == _lib.ERR_STATE
    c = run(eng, params, ic)                             # the registration and the state are intact
    assert all(bits(a[k], c[k]) for k in FORCING_KEYS)
    eng.set_path("ensemble")
    with pytest.raises(_lib.NesosimError) as e:
        eng.run_season_score_adjoint(params, ic, forcing=True)
    assert e.value.code == _lib.ERR_STATE
    eng.close()
