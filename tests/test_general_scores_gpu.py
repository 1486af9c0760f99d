"""GPU: fused calibration scores on the general day-kernel path (nesosim_set_path(ctx, 1) before registering; the
scoring build of the day kernel samples the observed cells, the epilogues are the season kernel's).  The scores are
bit-identical to the season kernel's on the grids it takes -- every CTA shape, the land-tile shortcut on and off,
dynamics on and off, per-member ICs, forcing sets -- and to the fixed-order restatement (oracle/observation_scores.py,
oracle/footprint_scores.py) on grids it does not take: wider than 96 columns, ragged tiles, the 25 km coastline.  Also
the launch count, determinism, errors and the calibration drivers' default on a wide grid."""
import numpy as np
import pytest

from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O
from oracle import footprint_scores as F
from oracle import observation_scores as R

pytestmark = pytest.mark.gpu

DEPTH, VOLUME, DENSITY, KINDS = R.DEPTH, R.VOLUME, R.DENSITY, R.KINDS
ENV = ("NESOSIM_ENS_VARIANT", "NESOSIM_ENS_CLUSTER", "NESOSIM_ENS_CLUSTERS", "NESOSIM_ENS_ROWS", "NESOSIM_ENS_COST",
       "NESOSIM_ENS_DBG", "NESOSIM_ENS_TIMING", "NESOSIM_DAY_THREADS", "NESOSIM_LAND_SHORTCUT", "NESOSIM_PDL")


def clear_env(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)


def oracle_params(row):
    return O.Params(windPackFactor=row[0], windPackThresh=row[1], leadLossFactor=row[2], atmLossFactor=row[3])


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def make_obs(mask, days, rng, n):
    """n point observations of all kinds on land and ocean, with NaN values, some on day 0 and on the last day, and
    ten of every kind at one ocean cell and day; density only from day 1 on."""
    ny, nx = mask.shape
    row, col, day = rng.integers(0, ny, n), rng.integers(0, nx, n), rng.integers(0, days, n)
    day[:n // 20] = 0
    day[n // 20:n // 10] = days - 1
    kind = rng.integers(0, KINDS, n)
    wet = np.argwhere(R.ocean(mask))
    r, c = wet[rng.integers(len(wet))]
    row[-10:], col[-10:], day[-10:] = r, c, max(1, days // 2)
    kind[(day == 0) & (kind == DENSITY)] = VOLUME
    value = np.where(kind == DENSITY, 200.0 + 150.0 * rng.random(n), 0.3 * rng.random(n))
    value[rng.random(n) < 0.05] = np.nan
    return {"day": day, "row": row, "col": col, "value": value, "kind": kind, "sigma": 10.0 ** rng.uniform(-3, 1, n)}


def cat_footprints(parts):
    out = {k: np.concatenate([np.asarray(p[k]) for p in parts]) for k in ("kind", "value", "sigma", "day", "row", "col",
                                                                           "weight")}
    out["begin"] = np.concatenate([[0], np.cumsum(np.concatenate([np.diff(p["begin"]) for p in parts]))]).astype(np.int64)
    return out


def one(kind, value, day, row, col, weight=None):
    n = len(day)
    return {"kind": np.array([kind]), "value": np.array([value]), "sigma": np.array([0.5]), "begin": np.array([0, n]),
            "day": np.asarray(day), "row": np.asarray(row), "col": np.asarray(col),
            "weight": np.ones(n) if weight is None else np.asarray(weight)}


def make_footprints(mask, days, rng):
    """Regional means (region_footprints), a one-point footprint, one partly and one entirely on land."""
    from nesosim_b200 import ensemble as ENS
    codes = [k for k in range(1, 11) if (mask == k).any()]
    parts = [ENS.region_footprints(mask, codes[:2], [(1, days // 2), (days // 2, days)], DEPTH, [0.2, 0.25], 0.05),
             ENS.region_footprints(mask, codes[-1:], [(1, days)], DENSITY, 300.0, 30.0)]
    wet, land = np.argwhere(R.ocean(mask)), np.argwhere(~R.ocean(mask))
    w = wet[rng.integers(len(wet), size=40)]
    parts.append(one(VOLUME, 0.1, [days - 1], [w[0, 0]], [w[0, 1]]))
    mixed = np.concatenate([w[1:31], land[:10]])
    parts.append(one(DEPTH, 0.15, rng.integers(0, days, 40), mixed[:, 0], mixed[:, 1], 2.0 ** rng.uniform(-3, 3, 40)))
    parts.append(one(DEPTH, 0.1, np.arange(4) % days, land[:4, 0], land[:4, 1]))
    return cat_footprints(parts)


def engine(mask, dx, T, M, seasons=None, member_set=None, days=None, path="auto", **flags):
    from nesosim_b200.engine import SnowBudgetEngine
    eng = SnowBudgetEngine(mask, T, dx, n_members=M, **flags)
    if member_set is None:
        f = seasons[0]
        eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
    else:
        st = {k: np.stack([np.concatenate([f[k], np.zeros((T - len(f[k]),) + f[k].shape[1:])]) for f in seasons])
              for k in ("precip", "conc", "wind", "drift")}
        eng.set_forcing_sets(st["precip"], st["conc"], st["wind"], st["drift"], member_set, days)
    if path != "auto":
        eng.set_path(path)
    return eng


def scores(eng, params, ic, obs, fps, obs_set=None, fp_set=None):
    eng.set_observations_fp(obs, fps, obs_set=obs_set, fp_set=fp_set)
    return tuple(t.cpu().numpy() for t in eng.run_season_scores_fp(params, ic, model=True))


def misfit(eng, params, ic, obs):
    eng.set_observations((obs["day"], obs["row"], obs["col"], obs["value"]))
    return tuple(t.cpu().numpy() for t in eng.run_season_misfit(params, ic))


# ---------------------------------------------------------------------------------------- same grid, two producers

@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("land", [0, 1])
@pytest.mark.parametrize("dynamics", [0, 1])
@pytest.mark.parametrize("per_member_ic", [False, True])
def test_general_path_equals_season_kernel(cuda, monkeypatch, threads, land, dynamics, per_member_ic):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_DAY_THREADS", str(threads))
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", str(land))
    mask, dx, T, M = S.region_mask(dx=100000), 100000, 30, 9
    rng = np.random.default_rng(10 + dynamics)
    seasons = [S.make_season(mask, T, seed=11)]
    ic = S.make_ic(mask, seed=12)
    if per_member_ic:
        ic = (0.02 + ic)[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=13)
    obs, fps = make_obs(mask, T, rng, 1500), make_footprints(mask, T, rng)
    depth = {k: obs[k] for k in ("day", "row", "col", "value")}
    got = {}
    for path in ("auto", "general"):
        eng = engine(mask, dx, T, M, seasons, path=path, dynamicsInc=dynamics, atmlossInc=1)
        got[path] = scores(eng, params, ic, obs, fps) + misfit(eng, params, ic, depth)
        assert eng.last_path() == ("general" if path == "general" else "ensemble")
        eng.close()
    names = ("chi2", "used", "model", "fp_chi2", "fp_used", "fp_model", "misfit", "misfit_used")
    for name, a, b in zip(names, got["auto"], got["general"]):
        assert same(a, b), name
    chi2, used, model = got["general"][:3]
    assert (used > 0).all() and np.isnan(model).any() and np.isfinite(model).any()
    assert (got["general"][4][:, DEPTH] == 3).all()         # two regional means and the partly-on-land footprint


def test_forcing_sets_general_equals_season_kernel(cuda, monkeypatch):
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    days, member_set = [12, 17, 21], [2, 0, 1, 1, 0, 2, 1]
    T, M = max(days), len(member_set)
    rng = np.random.default_rng(20)
    seasons = [S.make_season(mask, d, seed=21 + s) for s, d in enumerate(days)]
    ic = (0.02 + S.make_ic(mask, seed=24))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=25)
    obs = [make_obs(mask, d, rng, 300 + 40 * s) for s, d in enumerate(days)]
    for o, d in zip(obs, days):
        assert (o["day"] == d - 1).sum() > 10                 # every season's last day is observed
    fps = [make_footprints(mask, d, rng) for d in days]
    cat = {k: np.concatenate([o[k] for o in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(obs)])
    ftag = np.concatenate([np.full(len(f["value"]), i, dtype=np.int32) for i, f in enumerate(fps)])
    got = {}
    for path in ("auto", "general"):
        eng = engine(mask, dx, T, M, seasons, member_set, days, path=path, atmlossInc=1)
        got[path] = scores(eng, params, ic, cat, cat_footprints(fps), tag, ftag)
        eng.close()
    for a, b in zip(got["auto"], got["general"]):
        assert same(a, b)
    # the last day of every short season against the oracle's season arrays
    model = got["general"][2]
    for m, s in enumerate(member_set):
        f = seasons[s]
        ref = O.run_season(f, ic[m], mask, dx, oracle_params(params[m]), O.Flags(atmlossInc=1))
        want = R.model_values(ref["snowDepths"], ref["density"], f["conc"], obs[s], mask)
        last = obs[s]["day"] == days[s] - 1
        assert same(model[m, :len(want)][last], want[last]), m


# ------------------------------------------------------------------------------------ wide grids against the oracle

def ragged_mask():
    m = S.region_mask(dx=50000)
    return np.ascontiguousarray(m[40:85, 20:121])           # 45 x 101: partial tiles in both directions


WIDE = {"disc": (lambda: S.region_mask(shape=(40, 130), kind="disc"), 50000, 9),
        "ragged": (ragged_mask, 50000, 9),
        "25km": (lambda: S.region_mask(dx=25000), 25000, 4)}


@pytest.mark.parametrize("grid", list(WIDE))
def test_wide_grids_bit_for_bit_against_the_oracle(cuda, monkeypatch, grid):
    clear_env(monkeypatch)
    make, dx, T = WIDE[grid]
    mask = make()
    assert mask.shape[1] > 96
    M = 2
    rng = np.random.default_rng(30)
    seasons = [S.make_season(mask, T, seed=31)]
    ic = (0.02 + S.make_ic(mask, seed=32))[None] * rng.uniform(0.5, 2.0, (M, 1, 1))
    params = S.ensemble_params(M, seed=33)
    obs, fps = make_obs(mask, T, rng, 800), make_footprints(mask, T, rng)
    eng = engine(mask, dx, T, M, seasons, path="general", atmlossInc=1)
    chi2, used, model, fchi2, fused, fmodel = scores(eng, params, ic, obs, fps)
    eng.close()
    f = seasons[0]
    for m in range(M):
        ref = O.run_season(f, ic[m], mask, dx, oracle_params(params[m]), O.Flags(atmlossInc=1))
        arrays = (ref["snowDepths"], ref["density"], f["conc"])
        wm = R.model_values(*arrays, obs, mask)
        wc, wu = R.scores(wm, obs, mask)
        wfm = F.footprint_values(*arrays, fps, mask)
        wfc, wfu = F.footprint_scores(wfm, fps)
        assert same(model[m], wm) and same(chi2[m], wc) and np.array_equal(used[m], wu), m
        assert same(fmodel[m], wfm) and same(fchi2[m], wfc) and np.array_equal(fused[m], wfu), m
        assert wu.sum() > 0 and wfu.sum() > 0


# --------------------------------------------------------------------------------------------------------- contract

def test_launches_determinism_and_path_changes(cuda, monkeypatch):
    from nesosim_b200 import _lib
    clear_env(monkeypatch)
    mask = S.region_mask(shape=(40, 130), kind="disc")
    T, M = 7, 3
    rng = np.random.default_rng(40)
    seasons = [S.make_season(mask, T, seed=41)]
    params = S.ensemble_params(M, seed=42)
    ic = S.make_ic(mask, seed=43)
    obs, fps = make_obs(mask, T, rng, 300), make_footprints(mask, T, rng)
    eng = engine(mask, 50000, T, M, seasons, path="general")
    eng.set_observations_fp(obs, fps)
    l0 = eng.launch_count()
    a = [t.cpu().numpy() for t in eng.run_season_scores_fp(params, ic, model=True)]
    # init, T-1 scoring day kernels, the last-day samples, the footprint means, the epilogue
    assert eng.launch_count() - l0 == 1 + (T - 1) + 1 + 1 + 1
    b = [t.cpu().numpy() for t in eng.run_season_scores_fp(params, ic, model=True)]
    assert all(same(x, y) for x, y in zip(a, b))
    eng.set_observations_ex(obs["day"], obs["row"], obs["col"], obs["value"], obs["kind"], obs["sigma"])
    l0 = eng.launch_count()
    eng.run_season_scores(params, ic)
    assert eng.launch_count() - l0 == 1 + (T - 1) + 1 + 1
    for path in ("auto", "ensemble"):
        eng.set_path(path)
        with pytest.raises(_lib.NesosimError) as e:
            eng.run_season_scores(params, ic)
        assert e.value.code == _lib.ERR_STATE and "register" in str(e.value)
    eng.set_path("general")
    c = [t.cpu().numpy() for t in eng.run_season_scores(params, ic, model=True)]
    assert same(c[0], a[0]) and same(c[1], a[1]) and same(c[2], a[2])
    eng.close()


def test_rejected_registrations_keep_the_previous_one(cuda, monkeypatch):
    from nesosim_b200 import _lib
    from nesosim_b200.engine import SnowBudgetEngine
    clear_env(monkeypatch)
    mask = S.region_mask(shape=(40, 130), kind="disc")
    T, M = 6, 2
    rng = np.random.default_rng(50)
    seasons = [S.make_season(mask, T, seed=51)]
    params = S.ensemble_params(M, seed=52)
    obs = make_obs(mask, T, rng, 200)
    eng = engine(mask, 50000, T, M, seasons, path="general")
    eng.set_observations_ex(obs["day"], obs["row"], obs["col"], obs["value"], obs["kind"], obs["sigma"])
    a = [t.cpu().numpy() for t in eng.run_season_scores(params, None, model=True)]
    bad_day = dict(obs, day=np.where(np.arange(len(obs["day"])) == 7, T, obs["day"]))
    bad_sigma = dict(obs, sigma=np.where(np.arange(len(obs["day"])) == 3, 0.0, obs["sigma"]))
    for bad in (bad_day, bad_sigma):
        with pytest.raises(_lib.NesosimError) as e:
            eng.set_observations_ex(bad["day"], bad["row"], bad["col"], bad["value"], bad["kind"], bad["sigma"])
        assert e.value.code == _lib.ERR_ARG
        b = [t.cpu().numpy() for t in eng.run_season_scores(params, None, model=True)]
        assert all(same(x, y) for x, y in zip(a, b))
    eng.close()
    clim = SnowBudgetEngine(mask, T, 50000, n_members=M, densityType="clim")
    clim.set_path("general")
    with pytest.raises(_lib.NesosimError) as e:
        clim.set_observations(([1], [20], [60], [0.1]))
    assert e.value.code == _lib.ERR_ARG and "clim" in str(e.value)
    clim.close()
    strip = SnowBudgetEngine(mask, T, 50000, n_members=1)
    strip.strip_setup(0, 1)
    strip.set_path("general")
    with pytest.raises(_lib.NesosimError) as e:
        strip.set_observations(([1], [20], [60], [0.1]))
    assert e.value.code == _lib.ERR_ARG and "strip" in str(e.value)
    strip.close()


# --------------------------------------------------------------------------------------------- drivers, wide grid

def driver_seasons(mask, seed, days):
    from nesosim_b200 import ensemble as ENS
    rng = np.random.default_rng(seed)
    out = []
    for s, d in enumerate(days):
        season = {"forcing": S.make_season(mask, d, seed=seed + s), "ic": S.make_ic(mask, seed=seed + s) * (1 + s),
                  "obs": make_obs(mask, d, rng, 200)}
        if s != 1:
            season["footprints"] = ENS.region_footprints(mask, [8], [(1, d // 2), (d // 2, d)], DEPTH, [0.2, 0.25], 0.05)
        out.append(season)
    return out


def oracle_season(season, mask, dx, p):
    f = season["forcing"]
    ref = O.run_season(f, season["ic"], mask, dx, oracle_params(p), O.Flags(atmlossInc=1))
    return ref["snowDepths"], ref["density"], f["conc"]


def depth_obs(o):
    n = len(o["day"])
    return {"day": o["day"], "row": o["row"], "col": o["col"], "value": o["value"], "kind": np.zeros(n, np.int64),
            "sigma": np.ones(n)}


def test_drivers_default_to_the_general_fused_path_on_a_wide_grid(cuda, monkeypatch):
    from nesosim_b200 import ensemble as ENS
    clear_env(monkeypatch)
    mask, dx = S.region_mask(shape=(40, 130), kind="disc"), 50000
    seasons = driver_seasons(mask, 60, days=(8, 9, 10))
    params = S.ensemble_params(2, seed=61)
    ref = {(p, s): oracle_season(seasons[s], mask, dx, params[p]) for p in range(2) for s in range(3)}

    res = ENS.run_calibration_scores(mask, seasons, params, dx, atmlossInc=1, model=True)
    hbm = ENS.run_calibration_scores(mask, seasons, params, dx, atmlossInc=1, model=True, fused=False)
    for (p, s), arrays in ref.items():
        o = ENS.normalize_observations(seasons[s]["obs"])
        wm = R.model_values(*arrays, o, mask)
        wc, wu = R.scores(wm, o, mask)
        assert same(res["model"][s][p], wm) and same(res["chi2"][p, s], wc) and np.array_equal(res["used"][p, s], wu)
        if s != 1:
            fps = ENS.normalize_footprints(seasons[s]["footprints"])
            wfm = F.footprint_values(*arrays, fps, mask)
            wfc, wfu = F.footprint_scores(wfm, fps)
            assert same(res["fp_model"][s][p], wfm) and same(res["fp_chi2"][p, s], wfc)
            assert np.array_equal(res["fp_used"][p, s], wfu) and wfu.sum() > 0
    for k in ("used", "fp_used"):
        assert np.array_equal(res[k], hbm[k])
    for k in ("chi2", "fp_chi2"):
        assert np.allclose(res[k], hbm[k], rtol=1e-12, atol=0.0)

    cal_seasons = [dict(s, obs=(s["obs"]["day"], s["obs"]["row"], s["obs"]["col"], s["obs"]["value"])) for s in seasons]
    mis, used = ENS.run_calibration(mask, cal_seasons, params, dx, atmlossInc=1)
    mis_h, used_h = ENS.run_calibration(mask, cal_seasons, params, dx, atmlossInc=1, fused=False)
    for (p, s), arrays in ref.items():
        o = depth_obs(seasons[s]["obs"])
        wc, wu = R.scores(R.model_values(*arrays, o, mask), o, mask)
        assert same(mis[p, s], wc[DEPTH]) and used[p, s] == wu[DEPTH]
    assert np.array_equal(used, used_h) and np.allclose(mis, mis_h, rtol=1e-12, atol=0.0)

    s0 = seasons[0]
    obs = cal_seasons[0]["obs"]
    mis, used = ENS.run_ensemble(mask, s0["forcing"], s0["ic"], params, dx, obs, atmlossInc=1)
    mis_h, used_h = ENS.run_ensemble(mask, s0["forcing"], s0["ic"], params, dx, obs, atmlossInc=1, fused=False)
    for p in range(2):
        o = depth_obs(s0["obs"])
        wc, wu = R.scores(R.model_values(*ref[(p, 0)], o, mask), o, mask)
        assert same(mis[p], wc[DEPTH]) and used[p] == wu[DEPTH]
    assert np.array_equal(used, used_h) and np.allclose(mis, mis_h, rtol=1e-12, atol=0.0)
