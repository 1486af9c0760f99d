"""GPU: calibration gradients (nesosim_run_season_score_grads, the tangent-linear build of the scoring day kernel and of
both epilogues).  Jacobian rows, d chi2 / d theta, footprint derivatives and footprint gradients are bit-identical to
the restatement (oracle/score_gradients.py) for both CTA shapes, the land-tile shortcut on and off, dynamics on and off,
every loss switch on, per-member ICs, forcing sets with short seasons (each season's last day observed) and wide,
ragged and coastline grids.  The primal outputs are bit-identical to nesosim_run_season_scores_fp; also determinism,
the launch count, the errors, agreement with finite differences through extra members and the calibration driver."""
import functools

import numpy as np
import pytest

from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_gradients as G
from test_general_scores_gpu import (WIDE, clear_env, engine, make_footprints, make_obs, oracle_params, same)

pytestmark = pytest.mark.gpu

FLAGS = dict(atmlossInc=1)


def grads(eng, params, ic, obs, fps, obs_set=None, fp_set=None):
    eng.set_observations_fp(obs, fps, obs_set=obs_set, fp_set=fp_set)
    r = eng.run_season_score_grads(params, ic, model=True, jac=True)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in r.items()}


_ORACLE = {}


def check_member(got, m, forcing, ic_m, mask, dx, prow, obs, fps, dynamics=1):
    """One member's gradient outputs against the oracle (seasons of the disc case are shared by several tests)."""
    p = oracle_params(prow)
    f = O.Flags(dynamicsInc=dynamics, atmlossInc=1)
    key = (id(forcing), id(ic_m) if ic_m.base is None else (id(ic_m.base), m), tuple(prow), dynamics)
    if key not in _ORACLE:
        _ORACLE[key] = G.run_season_tangent(forcing, ic_m, mask, dx, p, f)
    s, tan = _ORACLE[key]
    arrays = (s["snowDepths"], s["density"], forcing["conc"])
    v = R.model_values(*arrays, obs, mask)
    dv = G.model_tangents(s["snowDepths"], tan, forcing["conc"], obs, mask, p)
    n = len(v)
    assert same(got["model"][m, :n], v), m
    assert same(got["jac"][m, :, :n], dv), m
    assert same(got["grad"][m], G.score_gradients(v, dv, obs, mask)), m
    mean, dmean = G.footprint_tangents(*arrays[:2], tan, forcing["conc"], fps, mask, p)
    k = len(mean)
    assert same(got["fp_model"][m, :k], mean) and same(got["fp_jac"][m, :, :k], dmean), m
    assert same(got["fp_grad"][m], G.footprint_gradients(mean, dmean, fps)), m
    return dv


@functools.lru_cache(maxsize=None)
def disc_case(dynamics):
    mask, dx, T, M = S.region_mask(dx=100000), 100000, 14, 3
    rng = np.random.default_rng(70 + dynamics)
    forcing = S.make_season(mask, T, seed=71)
    ic = (0.02 + S.make_ic(mask, seed=72))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=73)
    return mask, dx, T, M, forcing, ic, params, make_obs(mask, T, rng, 900), make_footprints(mask, T, rng)


@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("land", [0, 1])
@pytest.mark.parametrize("dynamics", [0, 1])
def test_gradients_bit_for_bit_against_the_oracle(cuda, monkeypatch, threads, land, dynamics):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_DAY_THREADS", str(threads))
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", str(land))
    mask, dx, T, M, forcing, ic, params, obs, fps = disc_case(dynamics)
    eng = engine(mask, dx, T, M, [forcing], path="general", dynamicsInc=dynamics, **FLAGS)
    got = grads(eng, params, ic, obs, fps)
    eng.set_observations_fp(obs, fps)
    plain = [t.cpu().numpy() for t in eng.run_season_scores_fp(params, ic, model=True)]
    eng.close()
    for name, want in zip(("chi2", "used", "model", "fp_chi2", "fp_used", "fp_model"), plain):
        assert same(got[name], want), name
    for m in range(M):
        dv = check_member(got, m, forcing, ic[m], mask, dx, params[m], obs, fps, dynamics)
        assert np.isfinite(dv).any() and np.abs(dv[np.isfinite(dv)]).max() > 0
    assert np.abs(got["grad"]).max() > 0 and np.abs(got["fp_grad"]).max() > 0


def test_forcing_sets_with_short_seasons(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    days, member_set = [9, 13, 6], [2, 0, 1, 1, 0]
    T, M = max(days), len(member_set)
    rng = np.random.default_rng(80)
    seasons = [S.make_season(mask, d, seed=81 + s) for s, d in enumerate(days)]
    ic = (0.02 + S.make_ic(mask, seed=84))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=85)
    obs = [make_obs(mask, d, rng, 300) for d in days]
    fps = [make_footprints(mask, d, rng) for d in days]
    cat = {k: np.concatenate([o[k] for o in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(obs)])
    fcat = {k: np.concatenate([np.asarray(f[k]) for f in fps]) for k in ("kind", "value", "sigma", "day", "row", "col",
                                                                          "weight")}
    fcat["begin"] = np.concatenate([[0], np.cumsum(np.concatenate([np.diff(f["begin"]) for f in fps]))]).astype(np.int64)
    ftag = np.concatenate([np.full(len(f["value"]), i, dtype=np.int32) for i, f in enumerate(fps)])
    eng = engine(mask, dx, T, M, seasons, member_set, days, path="general", **FLAGS)
    got = grads(eng, params, ic, cat, fcat, tag, ftag)
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
    rng = np.random.default_rng(90)
    forcing = S.make_season(mask, T, seed=91)
    ic = (0.02 + S.make_ic(mask, seed=92))[None] * rng.uniform(0.5, 2.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=93)
    obs, fps = make_obs(mask, T, rng, 600), make_footprints(mask, T, rng)
    eng = engine(mask, dx, T, M, [forcing], path="general", **FLAGS)
    got = grads(eng, params, ic, obs, fps)
    eng.close()
    for m in range(M):
        check_member(got, m, forcing, ic[m], mask, dx, params[m], obs, fps)


def test_launches_determinism_and_errors(cuda, monkeypatch):
    from nesosim_b200 import _lib
    clear_env(monkeypatch)
    mask = S.region_mask(shape=(40, 130), kind="disc")
    T, M = 7, 3
    rng = np.random.default_rng(100)
    forcing = S.make_season(mask, T, seed=101)
    params = S.ensemble_params(M, seed=102)
    ic = S.make_ic(mask, seed=103)
    obs, fps = make_obs(mask, T, rng, 300), make_footprints(mask, T, rng)
    eng = engine(mask, 50000, T, M, [forcing], path="general", **FLAGS)
    eng.set_observations_fp(obs, fps)
    l0 = eng.launch_count()
    a = eng.run_season_score_grads(params, ic, model=True, jac=True)
    a = {k: v.cpu().numpy() for k, v in a.items()}
    # init, T-1 gradient day kernels, the last-day samples, the footprint means, the epilogue
    assert eng.launch_count() - l0 == 1 + (T - 1) + 1 + 1 + 1
    b = eng.run_season_score_grads(params, ic, model=True, jac=True)
    assert all(same(a[k], v.cpu().numpy()) for k, v in b.items())
    lib, h = eng.lib, eng.handle
    p = _lib.member_params_array(params)
    buf = {k: eng._dev(np.zeros_like(v)) for k, v in a.items()}
    ptr = lambda k: buf[k].data_ptr()
    K = _lib.OBS_KINDS

    def call(jac_stride=a["jac"].shape[-1], fp_grad=True, fp_jac_stride=a["fp_jac"].shape[-1], grad=True):
        return lib.nesosim_run_season_score_grads(
            h, p, None, 0, ptr("chi2"), ptr("used"), None, 0, ptr("grad") if grad else None, ptr("jac"), jac_stride,
            ptr("fp_chi2"), ptr("fp_used"), None, 0, ptr("fp_grad") if fp_grad else None, ptr("fp_jac"), fp_jac_stride,
            None)
    assert call(jac_stride=a["jac"].shape[-1] - 1) == _lib.ERR_ARG
    assert call(fp_jac_stride=a["fp_jac"].shape[-1] - 1) == _lib.ERR_ARG
    assert call(grad=False) == _lib.ERR_ARG
    assert call(fp_grad=False) == _lib.ERR_STATE
    c = eng.run_season_score_grads(params, ic, model=True, jac=True)       # the registration is intact
    assert all(same(a[k], v.cpu().numpy()) for k, v in c.items())
    assert a["grad"].shape == (M, K, 3) and a["jac"].shape == (M, 3, len(obs["day"]))
    for path in ("auto", "ensemble"):
        eng.set_path(path)
        with pytest.raises(_lib.NesosimError) as e:
            eng.run_season_score_grads(params, ic)
        assert e.value.code == _lib.ERR_STATE and "register" in str(e.value)
    eng.close()
    # season-kernel observations: no tangent build
    mask100 = S.region_mask(dx=100000)
    eng = engine(mask100, 100000, T, M, [S.make_season(mask100, T, seed=104)], **FLAGS)
    o = make_obs(mask100, T, rng, 100)
    eng.set_observations_ex(o["day"], o["row"], o["col"], o["value"], o["kind"], o["sigma"])
    with pytest.raises(_lib.NesosimError) as e:
        eng.run_season_score_grads(params, None)
    assert e.value.code == _lib.ERR_STATE and "general path" in str(e.value)
    eng.close()


def test_agreement_with_finite_differences_through_extra_members(cuda, monkeypatch):
    """Central differences of the model values, from 1 + 6 members of one scores call, on the 100 km grid."""
    from nesosim_b200 import _lib
    clear_env(monkeypatch)
    mask, dx, T = S.region_mask(dx=100000), 100000, 20
    rng = np.random.default_rng(110)
    forcing = S.make_season(mask, T, seed=111)
    ic = 0.02 + S.make_ic(mask, seed=112)
    base = S.ensemble_params(1, seed=113)[0]
    rows = [base]
    for col in _lib.GRAD_PARAMS:
        for sign in (1, -1):
            r = base.copy()
            r[col] *= 1 + sign * 1e-4
            rows.append(r)
    params = np.array(rows)
    wet = np.argwhere(R.ocean(mask))                 # ocean cells only: land observations have no model value
    cell = wet[rng.integers(len(wet), size=1500)]
    kind = rng.integers(0, R.KINDS, 1500)
    obs = {"day": rng.integers(1, T, 1500), "row": cell[:, 0], "col": cell[:, 1], "kind": kind,
           "value": np.where(kind == R.DENSITY, 300.0, 0.1), "sigma": np.where(kind == R.DENSITY, 30.0, 0.05)}
    eng = engine(mask, dx, T, len(params), [forcing], path="general", **FLAGS)
    eng.set_observations_ex(obs["day"], obs["row"], obs["col"], obs["value"], obs["kind"], obs["sigma"])
    r = eng.run_season_score_grads(params, ic, model=True, jac=True)
    model, jac = r["model"].cpu().numpy(), r["jac"].cpu().numpy()
    eng.close()
    ok = np.isfinite(model[0]) & np.isfinite(model[1:]).all(axis=0)
    assert ok.sum() > 500
    for j, col in enumerate(_lib.GRAD_PARAMS):
        fd = (model[1 + 2 * j] - model[2 + 2 * j]) / (2e-4 * base[col])
        scale = np.abs(fd[ok]).max()
        assert scale > 0
        # step straddles no kink for most observations; those that do differ at O(1) -- allow 1% of them
        good = np.isclose(jac[0, j][ok], fd[ok], rtol=1e-5, atol=1e-5 * scale)
        assert good.mean() > 0.99, (j, good.mean())


def test_driver_gradients_leave_the_scores_unchanged(cuda, monkeypatch):
    from nesosim_b200 import ensemble as ENS
    from test_general_scores_gpu import driver_seasons
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    seasons = driver_seasons(mask, 120, days=(8, 9, 10))
    params = S.ensemble_params(2, seed=121)
    plain = ENS.run_calibration_scores(mask, seasons, params, dx, atmlossInc=1, model=True)
    res = ENS.run_calibration_scores(mask, seasons, params, dx, atmlossInc=1, model=True, grad=True, jac=True)
    for k in ("chi2", "used", "fp_chi2", "fp_used"):
        assert same(res[k], plain[k]), k
    for k in ("model", "fp_model"):
        assert all(same(a, b) for a, b in zip(res[k], plain[k])), k
    assert res["grad"].shape == (2, 3, 3, 3) and res["fp_grad"].shape == (2, 3, 3, 3)
    for p in range(2):
        for s in range(3):
            f = seasons[s]["forcing"]
            o = ENS.normalize_observations(seasons[s]["obs"])
            st, tan = G.run_season_tangent(f, seasons[s]["ic"], mask, dx, oracle_params(params[p]), O.Flags(atmlossInc=1))
            v = R.model_values(st["snowDepths"], st["density"], f["conc"], o, mask)
            dv = G.model_tangents(st["snowDepths"], tan, f["conc"], o, mask, oracle_params(params[p]))
            assert same(res["jac"][s][p], dv) and same(res["grad"][p, s], G.score_gradients(v, dv, o, mask))
            if s != 1:
                fps = ENS.normalize_footprints(seasons[s]["footprints"])
                mean, dmean = G.footprint_tangents(st["snowDepths"], st["density"], tan, f["conc"], fps, mask,
                                                   oracle_params(params[p]))
                assert same(res["fp_jac"][s][p], dmean)
                assert same(res["fp_grad"][p, s], G.footprint_gradients(mean, dmean, fps))
            else:
                assert res["fp_jac"][s].shape == (2, 3, 0) and not res["fp_grad"][p, s].any()
