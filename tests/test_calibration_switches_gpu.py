"""GPU: the calibration builds (scores, tangent, record / adjoint and forcing adjoint) on every process-switch
configuration the API accepts, not only the all-on one: the reference's default (atm loss off), each loss or packing
term off, the budget alone with and without dynamics, pre-normalised smoothing, and divisors without the fast-division
proof.  The forcing carries NaN wind, NaN concentration (day 0 included), inf and subnormal precipitation on observed
ocean cells.  Scores, gradients and the forcing adjoint are bit-identical to the restatements (oracle/score_gradients.py,
oracle/forcing_adjoint.py) for both CTA shapes and the land-tile shortcut on and off; a switched-off term gives exact
zeros next to nonzero enabled terms; the season kernel scores as the general path does; two-day seasons, the
calibration driver in the reference default, and 128 members of 260-day seasons."""
import dataclasses
import functools
import time

import numpy as np
import pytest

from nesosim_b200 import _lib
from nesosim_b200 import ensemble as ENS
from nesosim_b200 import synthetic as S
from oracle import footprint_scores as F
from oracle import forcing_adjoint as FA
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_gradients as G
from test_general_scores_gpu import (DENSITY, DEPTH, clear_env, driver_seasons, engine, make_footprints, make_obs,
                                     misfit, oracle_params, same)
from test_score_adjoint_gpu import FW, W, land_ic

pytestmark = pytest.mark.gpu

NAMES = _lib.FORCING_FIELDS
DAY_KEYS = tuple(n + "_day_grad" for n in NAMES)
SWITCHES = ("windpackInc", "leadlossInc", "atmlossInc")     # the theta columns _lib.GRAD_PARAMS, in order

# Every divisor tried in [1e-100, 1e100] (grid spacings, densities, 4e5 random values) carries the fast-division proof;
# const_div_host gives none outside that range, so these two are the divisors that take div_generic everywhere.
INEXACT_DX = 1e101
INEXACT_RHO = 1e101


def config(dx=100000, consts=None, **switches):
    return {"dx": dx, "consts": consts or {}, "switches": switches}


CONFIGS = {
    "reference_default": config(atmlossInc=0),
    "no_windpack": config(windpackInc=0, atmlossInc=1),
    "no_leadloss": config(leadlossInc=0, atmlossInc=1),
    "no_lead_no_atm": config(leadlossInc=0, atmlossInc=0),
    "budget_only": config(windpackInc=0, leadlossInc=0, atmlossInc=0),
    "all_off": config(windpackInc=0, leadlossInc=0, atmlossInc=0, dynamicsInc=0),
    "pre_normalised": config(conv_variant="pre_normalised", atmlossInc=1),
    "inexact_dx": config(dx=INEXACT_DX, atmlossInc=1),
    "inexact_rho_fresh": config(consts={"snowDensityFresh": INEXACT_RHO}, atmlossInc=1),
}


def flags_of(name):
    return O.Flags(**CONFIGS[name]["switches"])


def params_of(name, row):
    return dataclasses.replace(oracle_params(row), **CONFIGS[name]["consts"])


def make_engine(name, mask, T, M, seasons, member_set=None, days=None, path="general"):
    c = CONFIGS[name]
    return engine(mask, c["dx"], T, M, seasons, member_set, days, path=path, **c["switches"], **c["consts"])


def enabled(name):
    f = flags_of(name)
    return [getattr(f, sw) == 1 for sw in SWITCHES]


def bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def test_inexact_configs_lack_the_proof(cuda):
    lib = _lib.load()
    dx = CONFIGS["inexact_dx"]["dx"]
    assert lib.nesosim_const_div_is_fast(dx) == 0 or lib.nesosim_const_div_is_fast(2 * dx) == 0
    assert lib.nesosim_const_div_is_fast(CONFIGS["inexact_rho_fresh"]["consts"]["snowDensityFresh"]) == 0
    assert lib.nesosim_const_div_is_fast(CONFIGS["inexact_rho_fresh"]["dx"]) == 1
    assert all(lib.nesosim_const_div_is_fast(c) == 1 for c in (100000., 200000., 200.))


# ------------------------------------------------------------------------------------------------------------ the case

# (day, rows, cols) of the non-finite forcing, on ocean cells of the 100 km grid away from the NaN precip corners
NAN_WIND = (4, slice(42, 45), slice(30, 33))
NAN_CONC = (6, slice(44, 46), slice(40, 42))
NAN_CONC0 = (0, slice(46, 48), slice(26, 28))
INF_PRECIP = (5, slice(43, 44), slice(45, 46))
TINY_PRECIP = (3, slice(50, 52), slice(30, 32))             # subnormal: P / rho_new takes div_generic
PATCHES = {"nan_wind": NAN_WIND, "nan_conc": NAN_CONC, "nan_conc0": NAN_CONC0, "inf_precip": INF_PRECIP,
           "tiny_precip": TINY_PRECIP}


def inject(forcing):
    forcing["wind"][NAN_WIND] = np.nan
    forcing["conc"][NAN_CONC] = np.nan
    forcing["conc"][NAN_CONC0] = np.nan
    forcing["precip"][INF_PRECIP] = np.inf
    forcing["precip"][TINY_PRECIP] = 1e-310
    return forcing


def patch_obs(rng):
    """Depth, volume and density observations on every patch, on its day and the day after."""
    rows, cols, days = [], [], []
    for x, r, c in PATCHES.values():
        rr, cc = np.mgrid[r, c]
        for d in (x, x + 1):
            rows.append(rr.ravel())
            cols.append(cc.ravel())
            days.append(np.full(rr.size, d))
    row, col, day = np.concatenate(rows), np.concatenate(cols), np.concatenate(days)
    kind = np.arange(len(day)) % R.KINDS
    kind[(day == 0) & (kind == DENSITY)] = DEPTH
    value = np.where(kind == DENSITY, 300.0, 0.1)
    return {"day": day, "row": row, "col": col, "value": value, "kind": kind, "sigma": np.where(kind == DENSITY, 30., .05)}


def cat_obs(a, b):
    return {k: np.concatenate([np.asarray(a[k]), np.asarray(b[k])]) for k in a}


@functools.lru_cache(maxsize=None)
def disc_case():
    """test_score_adjoint_gpu's 100 km case with the non-finite forcing of PATCHES, each patch observed."""
    mask, dx, T, M = S.region_mask(dx=100000), 100000, 12, 3
    rng = np.random.default_rng(500)
    forcing = S.make_season(mask, T, seed=501)
    forcing["conc"][0][~R.ocean(mask)] = 0.9              # keeps the IC on land (conc[0] >= minConc)
    inject(forcing)
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=502))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=503)
    obs = cat_obs(make_obs(mask, T, rng, 700), patch_obs(rng))
    fps = make_footprints(mask, T, rng)
    ocean = R.ocean(mask)
    for x, r, c in PATCHES.values():
        assert ocean[r, c].all() and np.isfinite(forcing["precip"][:, r, c]).any()
        assert ((obs["day"] == x + 1) & np.isin(obs["row"], np.arange(90)[r]) & np.isin(obs["col"], np.arange(90)[c])).any()
    return mask, T, M, forcing, ic, params, obs, fps


@functools.lru_cache(maxsize=None)
def oracle(name, m):
    """Member m of the disc case under config ``name``: the scores, the tangent outputs and the forcing adjoint."""
    mask, T, M, forcing, ic, params, obs, fps = disc_case()
    return oracle_member(name, forcing, ic[m], mask, params[m], obs, fps)


def oracle_member(name, forcing, ic_m, mask, prow, obs, fps, num_steps=None):
    dx, p, f = CONFIGS[name]["dx"], params_of(name, prow), flags_of(name)
    s, tan = G.run_season_tangent(forcing, ic_m, mask, dx, p, f, num_steps)
    arrays = (s["snowDepths"], s["density"], forcing["conc"])
    v = R.model_values(*arrays, obs, mask)
    chi2, used = R.scores(v, obs, mask)
    mean = F.footprint_values(*arrays, fps, mask)
    fchi2, fused = F.footprint_scores(mean, fps)
    dv = G.model_tangents(s["snowDepths"], tan, forcing["conc"], obs, mask, p)
    _, dmean = G.footprint_tangents(*arrays[:2], tan, forcing["conc"], fps, mask, p)
    out = {"chi2": chi2, "used": used, "model": v, "fp_chi2": fchi2, "fp_used": fused, "fp_model": mean, "jac": dv,
           "grad": G.score_gradients(v, dv, obs, mask), "fp_jac": dmean, "fp_grad": G.footprint_gradients(mean, dmean, fps)}
    out.update(FA.score_adjoint_forcing(forcing, ic_m, mask, dx, p, f, obs, fps, W, FW, num_steps))
    return out


def run_all(eng, params, ic, obs, fps, obs_set=None, fp_set=None):
    """The four entry points on one registration: scores, grads, and the adjoint with the three per-day stacks."""
    eng.set_observations_fp(obs, fps, obs_set=obs_set, fp_set=fp_set)
    host = lambda r: {k: (None if v is None else v.cpu().numpy()) for k, v in r.items()}
    sc = dict(zip(("chi2", "used", "model", "fp_chi2", "fp_used", "fp_model"),
                  (t.cpu().numpy() for t in eng.run_season_scores_fp(params, ic, model=True))))
    gr = host(eng.run_season_score_grads(params, ic, model=True, jac=True))
    ad = host(eng.run_season_score_adjoint(params, ic, W, FW, model=True, forcing=True, forcing_days=NAMES))
    return sc, gr, ad


def check_member(sc, gr, ad, m, want):
    n, k = len(want["model"]), len(want["fp_model"])
    for key in ("chi2", "used", "fp_chi2", "fp_used"):
        assert same(sc[key][m], want[key]), (m, key)
    assert same(sc["model"][m, :n], want["model"]) and same(sc["fp_model"][m, :k], want["fp_model"]), m
    for key in ("chi2", "used", "model", "fp_chi2", "fp_used", "fp_model"):       # the builds score alike
        assert same(gr[key], sc[key]) and same(ad[key], sc[key]), key
    assert same(gr["jac"][m, :, :n], want["jac"]) and same(gr["fp_jac"][m, :, :k], want["fp_jac"]), m
    assert same(gr["grad"][m], want["grad"]) and same(gr["fp_grad"][m], want["fp_grad"]), m
    T = len(want["precip_day_grad"])
    for key in ("theta_grad", "ic_grad", "forcing_scale_grad", "forcing_scale_total") + DAY_KEYS:
        g = ad[key][m][:T] if key in DAY_KEYS else ad[key][m]
        if key in DAY_KEYS:
            assert not ad[key][m][T:].any(), key
        assert bits(g, want[key]), (m, key, np.abs(g - want[key]).max())


def check_structure(name, gr, ad):
    """Exact zeros of every switched-off term, each next to a nonzero enabled one."""
    on = enabled(name)
    for j in range(G.DIRS):
        cols = (gr["grad"][..., j], np.nan_to_num(gr["jac"][:, j]), gr["fp_grad"][..., j],
                np.nan_to_num(gr["fp_jac"][:, j]), ad["theta_grad"][:, j])
        if on[j]:
            assert all(np.abs(c).max() > 0 for c in cols), (name, j)
        else:
            assert not any(c.any() for c in cols), (name, j)
    if not on[1] and not on[2]:
        assert not ad["wind_day_grad"].any() and not ad["forcing_scale_grad"][:, 1].any()
        assert not ad["forcing_scale_total"][:, 1].any()
    else:
        assert np.abs(ad["wind_day_grad"]).max() > 0 and np.abs(ad["forcing_scale_total"][:, 1]).min() > 0
    for key in ("precip_day_grad", "conc_day_grad", "ic_grad"):
        assert np.abs(ad[key]).max() > 0, key


def forward_mode_rel(gr, ad, on):
    """max relative difference of theta_grad to the weighted forward-mode gradients over the enabled columns."""
    want = np.einsum("k,mkd->md", W, gr["grad"]) + np.einsum("k,mkd->md", FW, gr["fp_grad"])
    want, got = want[:, on], ad["theta_grad"][:, on]
    return (np.abs(got - want).max(axis=1) / np.abs(want).max(axis=1)) if on.any() else np.zeros(len(got))


@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("land", [0, 1])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_every_entry_point_bit_for_bit_against_the_oracle(cuda, monkeypatch, name, land, threads):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_DAY_THREADS", str(threads))
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", str(land))
    mask, T, M, forcing, ic, params, obs, fps = disc_case()
    eng = make_engine(name, mask, T, M, [forcing])
    sc, gr, ad = run_all(eng, params, ic, obs, fps)
    eng.close()
    for m in range(M):
        check_member(sc, gr, ad, m, oracle(name, m))
    check_structure(name, gr, ad)
    rel = forward_mode_rel(gr, ad, np.array(enabled(name)))
    assert (rel <= 1e-10).all(), rel
    # the patches reached the scores: NaN model values where the forcing killed the cell
    assert np.isnan(sc["model"]).any() and np.isfinite(sc["model"]).any()


# ----------------------------------------------------------------------------------- season kernel = general path

SET_DAYS, SET_MEMBERS = [12, 9, 10], [2, 0, 1, 1, 0]


def sets_case():
    mask = S.region_mask(dx=100000)
    rng = np.random.default_rng(520)
    seasons = [inject(S.make_season(mask, d, seed=521 + s)) for s, d in enumerate(SET_DAYS)]
    M = len(SET_MEMBERS)
    ic = (0.02 + S.make_ic(mask, seed=524))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=525)
    obs = [make_obs(mask, d, rng, 300) for d in SET_DAYS]
    fps = [make_footprints(mask, d, rng) for d in SET_DAYS]
    return mask, seasons, ic, params, obs, fps


def concat_sets(obs, fps):
    cat = {k: np.concatenate([o[k] for o in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(obs)])
    fcat, ftag = ENS.concat_footprints(fps)
    return cat, tag, fcat, ftag


@pytest.mark.parametrize("name", list(CONFIGS))
def test_season_kernel_equals_general_path(cuda, monkeypatch, name):
    clear_env(monkeypatch)
    mask, T, M, forcing, ic, params, obs, fps = disc_case()
    depth = {k: obs[k] for k in ("day", "row", "col", "value")}
    smask, seasons, sic, sparams, sobs, sfps = sets_case()
    cat, tag, fcat, ftag = concat_sets(sobs, sfps)
    if name == "inexact_dx":
        # the season kernel needs proven grid divisors: "auto" refuses the registration, and the calibration drivers
        # take that refusal as their cue to score on the general path (checked above for this config)
        for eng, args in ((make_engine(name, mask, T, M, [forcing], path="auto"), (obs, fps, None, None)),
                          (make_engine(name, smask, max(SET_DAYS), len(SET_MEMBERS), seasons, SET_MEMBERS, SET_DAYS,
                                       path="auto"), (cat, fcat, tag, ftag))):
            with pytest.raises(_lib.NesosimError) as e:
                eng.set_observations_fp(*args)
            assert e.value.code == _lib.ERR_ARG and "fast-division proof" in str(e.value)
            eng.close()
        return
    if name == "inexact_rho_fresh":
        # the season kernel takes this grid and divides P by rho_new through div_generic, but with rho_new = 1e101
        # the accumulated snowfall (~1e-101) leaves the range its bare divisions are proven for: the scoring call
        # refuses, as misfit mode has no fallback (the general path's builds were checked above for this config)
        eng = make_engine(name, mask, T, M, [forcing], path="auto")
        eng.set_observations_fp(obs, fps)
        with pytest.raises(_lib.NesosimError) as e:
            eng.run_season_scores_fp(params, ic, model=True)
        assert e.value.code == _lib.ERR_ARG and "left the range" in str(e.value)
        eng.close()
        return
    got = {}
    for path in ("auto", "general"):
        eng = make_engine(name, mask, T, M, [forcing], path=path)
        eng.set_observations_fp(obs, fps)
        one = [t.cpu().numpy() for t in eng.run_season_scores_fp(params, ic, model=True)]
        assert eng.last_path() == ("ensemble" if path == "auto" else "general"), path
        one += list(misfit(eng, params, ic, depth))
        eng.close()
        eng = make_engine(name, smask, max(SET_DAYS), len(SET_MEMBERS), seasons, SET_MEMBERS, SET_DAYS, path=path)
        eng.set_observations_fp(cat, fcat, obs_set=tag, fp_set=ftag)
        sets = [t.cpu().numpy() for t in eng.run_season_scores_fp(sparams, sic, model=True)]
        assert eng.last_path() == ("ensemble" if path == "auto" else "general"), path
        eng.close()
        got[path] = one + sets
    for i, (a, b) in enumerate(zip(got["auto"], got["general"])):
        assert same(a, b), i
    assert (got["general"][1] > 0).all() and np.isnan(got["general"][2]).any()


# ----------------------------------------------------------------------------------------------- two-day seasons

def short_footprints(mask, d):
    codes = [k for k in range(1, 11) if (mask == k).any()]
    return ENS.concat_footprints([ENS.region_footprints(mask, codes[:2], [(0, d)], DEPTH, [0.2], 0.05),
                                  ENS.region_footprints(mask, codes[-1:], [(1, d)], DENSITY, 300.0, 30.0)])[0]


@pytest.mark.parametrize("name", ["reference_default", "all_off"])
def test_two_day_seasons(cuda, monkeypatch, name):
    clear_env(monkeypatch)
    mask = S.region_mask(dx=100000)
    rng = np.random.default_rng(540)
    # one forcing of 2 days: a single backward day (x = 0)
    T, M = 2, 3
    forcing = S.make_season(mask, T, seed=541)
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=542))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=543)
    obs, fps = make_obs(mask, T, rng, 400), short_footprints(mask, T)
    assert set(obs["day"].tolist()) == {0, 1}
    eng = make_engine(name, mask, T, M, [forcing])
    sc, gr, ad = run_all(eng, params, ic, obs, fps)
    l0 = eng.launch_count()
    eng.run_season_score_adjoint(params, ic, W, FW, forcing=True, forcing_days=NAMES)
    assert eng.launch_count() - l0 == 2 * T + 5
    eng.close()
    for m in range(M):
        check_member(sc, gr, ad, m, oracle_member(name, forcing, ic[m], mask, params[m], obs, fps))
    # forcing sets of 2, 3 and 9 days, each set's last day observed
    days, member_set = [2, 3, 9], [0, 2, 1, 0, 2]
    T, M = max(days), len(member_set)
    seasons = [S.make_season(mask, d, seed=545 + s) for s, d in enumerate(days)]
    ic = land_ic(mask, 0.02 + S.make_ic(mask, seed=548))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=549)
    obs = [make_obs(mask, d, rng, 300) for d in days]
    fps = [short_footprints(mask, d) for d in days]
    cat, tag, fcat, ftag = concat_sets(obs, fps)
    eng = make_engine(name, mask, T, M, seasons, member_set, days)
    sc, gr, ad = run_all(eng, params, ic, cat, fcat, tag, ftag)
    eng.close()
    for m, s in enumerate(member_set):
        assert (obs[s]["day"] == days[s] - 1).any()
        padded = {k: np.concatenate([v, np.zeros((T - days[s],) + v.shape[1:])]) for k, v in seasons[s].items()}
        want = oracle_member(name, padded, ic[m], mask, params[m], obs[s], fps[s], num_steps=days[s] - 1)
        # rows of one set's observations within the concatenated registration
        sub = {k: v[m:m + 1] for k, v in sc.items()}
        check_member(sub, {k: v[m:m + 1] for k, v in gr.items()}, {k: v[m:m + 1] for k, v in ad.items()}, 0, want)


# --------------------------------------------------------------------------------- the driver, reference default

def test_driver_in_the_reference_default(cuda, monkeypatch):
    """run_calibration_scores without switch keywords (atmlossInc=0) gives, per pair, what the engine gives."""
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    seasons = [driver_seasons(mask, 560, days=(8, 9, 10))[s] for s in (0, 2)]      # both with footprints
    params = S.ensemble_params(3, seed=561)
    res = ENS.run_calibration_scores(mask, seasons, params, dx, adjoint=True, forcing_grad=True, model=True)
    gres = ENS.run_calibration_scores(mask, seasons, params, dx, grad=True, model=True)
    assert not res["adjoint_grad"][..., 2].any() and np.abs(res["adjoint_grad"][..., :2]).min() > 0
    assert not gres["grad"][..., 2].any() and np.abs(gres["grad"][..., :2]).max() > 0
    for s, season in enumerate(seasons):
        f = season["forcing"]
        eng = engine(mask, dx, len(f["precip"]), len(params), [f], path="general")
        eng.set_observations_fp(ENS.normalize_observations(season["obs"]), ENS.normalize_footprints(season["footprints"]))
        ad = {k: v.cpu().numpy() for k, v in eng.run_season_score_adjoint(params, season["ic"], forcing=True).items()
              if v is not None}
        gr = eng.run_season_score_grads(params, season["ic"])["grad"].cpu().numpy()
        eng.close()
        for p in range(len(params)):
            assert same(res["adjoint_grad"][p, s], ad["theta_grad"][p]) and same(res["ic_grad"][p, s], ad["ic_grad"][p])
            assert bits(res["forcing_scale_grad"][p, s], ad["forcing_scale_grad"][p])
            assert bits(res["forcing_scale_total"][p, s], ad["forcing_scale_total"][p])
            assert same(gres["grad"][p, s], gr[p]), (p, s)


# ---------------------------------------------------------------------------------------------------------- at scale

SCALE_MEMBERS = (0, 64, 127)


@functools.lru_cache(maxsize=None)
def at_scale():
    """128 members of a 260-day season at 100 km, 20 000 points and footprints, the reference default: the adjoint
    with all three per-day stacks (members SCALE_MEMBERS copied back) and theta_grad's agreement with forward mode."""
    mask, dx, T, M = S.region_mask(dx=100000), 100000, 260, 128
    rng = np.random.default_rng(580)
    forcing = S.make_season(mask, T, seed=581)
    params = S.ensemble_params(M, seed=582)
    ic = S.make_ic(mask, seed=583)
    obs, fps = make_obs(mask, T, rng, 20000), make_footprints(mask, T, rng)
    eng = make_engine("reference_default", mask, T, M, [forcing])
    eng.set_observations_fp(obs, fps)
    fwd = {k: (None if v is None else v.cpu().numpy()) for k, v in eng.run_season_score_grads(params, ic).items()}
    r = eng.run_season_score_adjoint(params, ic, W, FW, forcing=True, forcing_days=NAMES)
    sel = list(SCALE_MEMBERS)
    got = {k: v[sel].cpu().numpy() for k, v in r.items() if v is not None and v.dim() > 1}
    theta = r["theta_grad"].cpu().numpy()
    del r
    eng.close()
    rel = forward_mode_rel(fwd, {"theta_grad": theta}, np.array(enabled("reference_default")))
    return mask, forcing, ic, params, obs, fps, got, rel


@pytest.mark.parametrize("i", range(len(SCALE_MEMBERS)))
def test_at_scale_in_the_reference_default(cuda, monkeypatch, i):
    clear_env(monkeypatch)
    mask, forcing, ic, params, obs, fps, got, rel = at_scale()
    assert (rel <= 1e-10).all(), rel.max()
    m = SCALE_MEMBERS[i]
    t0 = time.perf_counter()
    want = FA.score_adjoint_forcing(forcing, ic, mask, 100000, params_of("reference_default", params[m]),
                                    flags_of("reference_default"), obs, fps, W, FW)
    print("oracle of member %d: %.1f s; largest relative difference to forward mode: %.3e"
          % (m, time.perf_counter() - t0, rel.max()))
    for key in ("theta_grad", "ic_grad", "forcing_scale_grad", "forcing_scale_total") + DAY_KEYS:
        assert bits(got[key][i], want[key]), (m, key)
    assert got["theta_grad"][i][2] == 0.0 and np.abs(got["precip_day_grad"][i]).max() > 0
