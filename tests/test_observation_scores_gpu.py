"""GPU: calibration scores -- observations of snow depth over ice, snow volume and bulk density with an error each
(nesosim_set_observations_ex), scored per kind inside the fused path with the model value at every observation
(nesosim_run_season_scores), on one shared forcing and on forcing sets, and the driver ensemble.run_calibration_scores."""
import ctypes as C

import numpy as np
import pytest

from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O

pytestmark = pytest.mark.gpu

DX = 100000
T = 20
DAYS = [14, 17, 20]                    # forcing sets: three seasons of different length in a T = 20 context
MEMBER_SET = [2, 0, 1, 0, 2, 1, 2]
DEPTH, VOLUME, DENSITY, KINDS = 0, 1, 2, 3


def oracle_params(row):
    return O.Params(windPackFactor=row[0], windPackThresh=row[1], leadLossFactor=row[2], atmLossFactor=row[3])


def oracle_run(season, ic, row):
    return O.run_season(season, ic, np.asarray(S.region_mask(dx=DX)), DX, oracle_params(row), O.Flags(atmlossInc=1))


def make_obs(mask, days, rng, n, thin=()):
    """n observations of all kinds: on land and ocean, depth and volume on day 0, the last day, one cell-day observed ten
    times across the three kinds, log-uniform sigma, some NaN values; `thin` (day, row, col) cell-days get a density
    observation (total depth below minSnowD there: the model value is NaN)."""
    ny, nx = mask.shape
    row, col, day = rng.integers(0, ny, n), rng.integers(0, nx, n), rng.integers(0, days, n)
    kind = rng.integers(0, KINDS, n)
    day[:30] = 0
    day[30:60] = days - 1
    row[100:110], col[100:110], day[100:110] = row[100], col[100], max(day[100], 1)
    kind[100:110] = [0, 1, 2, 0, 1, 2, 0, 1, 2, 0]
    kind[(day == 0) & (kind == DENSITY)] = VOLUME
    value = np.where(kind == DENSITY, 200.0 + 150.0 * rng.random(n), 0.3 * rng.random(n))
    value[rng.random(n) < 0.05] = np.nan
    sigma = 10.0 ** rng.uniform(-3, 1, n)
    if len(thin):
        t = np.asarray(thin)
        day, row, col = (np.concatenate([a, t[:, j]]) for j, a in enumerate((day, row, col)))
        kind = np.concatenate([kind, np.full(len(t), DENSITY)])
        value = np.concatenate([value, np.full(len(t), 300.0)])
        sigma = np.concatenate([sigma, np.full(len(t), 50.0)])
    return {"day": day, "row": row, "col": col, "value": value, "kind": kind, "sigma": sigma}


def thin_cells(mask, ref, days, k=5):
    """Ocean cell-days (day >= 1) whose total depth is below minSnowD in an oracle run."""
    tot = ref["snowDepths"][1:days, 0] + ref["snowDepths"][1:days, 1]
    ocean = (mask >= 1) & (mask <= 10)
    d, r, c = np.nonzero((tot < O.Params().minSnowD) & ocean[None])
    assert len(d) >= k
    return [(d[i] + 1, r[i], c[i]) for i in np.linspace(0, len(d) - 1, k).astype(int)]


def model_values(depths, dens, conc, o, mask):
    """The model value of every observation gathered from the arrays of one member's season (NaN on land and lake)."""
    d, r, c, k = o["day"], o["row"], o["col"], o["kind"]
    vol = depths[d, 0, r, c] + depths[d, 1, r, c]
    with np.errstate(all="ignore"):
        v = np.where(k == DEPTH, vol / conc[d, r, c], np.where(k == VOLUME, vol, dens[d, r, c]))
    v[~((mask[r, c] >= 1) & (mask[r, c] <= 10))] = np.nan
    return v


def scores(model, o):
    with np.errstate(all="ignore"):
        res = (model - o["value"]) / o["sigma"]
    ok = np.isfinite(res)
    return (np.array([np.sum(res[ok & (o["kind"] == k)] ** 2) for k in range(KINDS)]),
            np.array([np.sum(ok & (o["kind"] == k)) for k in range(KINDS)]))


def make_case(layout):
    """(mask, forcing per set, member_set, days per set, params, ic [M], observations per set)"""
    mask = S.region_mask(dx=DX)
    rng = np.random.default_rng(170)
    if layout == "single":
        member_set, days = [0, 0, 0, 0], [T]
    else:
        member_set, days = MEMBER_SET, DAYS
    M = len(member_set)
    seasons = [S.make_season(mask, d, seed=171 + s) for s, d in enumerate(days)]
    params = S.ensemble_params(M, seed=172)
    ic = S.make_ic(mask, seed=173)[None] * rng.uniform(0.2, 3.0, (M, 1, 1))
    obs = []
    for s, d in enumerate(days):
        m0 = member_set.index(s)
        thin = thin_cells(mask, oracle_run(seasons[s], ic[m0], params[m0]), d)
        obs.append(make_obs(mask, d, rng, 700 + 100 * s, thin))
    return mask, seasons, member_set, days, params, ic, obs


def engine(mask, seasons, member_set, days):
    from nesosim_b200.engine import SnowBudgetEngine
    eng = SnowBudgetEngine(mask, T, DX, n_members=len(member_set), atmlossInc=1)
    if len(days) == 1:
        f = seasons[0]
        eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
    else:
        st = {k: np.stack([np.concatenate([f[k], np.zeros((T - len(f[k]),) + f[k].shape[1:])]) for f in seasons])
              for k in ("precip", "conc", "wind", "drift")}
        eng.set_forcing_sets(st["precip"], st["conc"], st["wind"], st["drift"], member_set, days)
    return eng


def register(eng, obs, kinds=None, sigma=True):
    """All sets' observations (only `kinds` if given; sigma 1 unless `sigma`), tagged with their set on forcing sets."""
    sel = [np.isin(o["kind"], kinds if kinds is not None else range(KINDS)) for o in obs]
    cat = {k: np.concatenate([o[k][s] for o, s in zip(obs, sel)]) for k in obs[0]}
    tag = np.concatenate([np.full(s.sum(), i, dtype=np.int32) for i, s in enumerate(sel)]) if len(obs) > 1 else None
    eng.set_observations_ex(cat["day"], cat["row"], cat["col"], cat["value"], cat["kind"],
                            cat["sigma"] if sigma else None, obs_set=tag)


def run(eng, params, ic, model=True):
    return tuple(None if t is None else t.cpu().numpy() for t in eng.run_season_scores(params, ic, model=model))


@pytest.mark.parametrize("cluster", [None, "8"])
@pytest.mark.parametrize("layout", ["single", "sets"])
def test_model_rows_and_scores(cuda, layout, cluster, monkeypatch):
    """Model rows equal bit for bit the quantities gathered from nesosim_run_season of the same context; chi2 equals the
    oracle's to 1e-12 (another summation order) with exact counts; two runs are bit-identical in four launches each."""
    if cluster:
        monkeypatch.setenv("NESOSIM_ENS_CLUSTER", cluster)
    mask, seasons, member_set, days, params, ic, obs = make_case(layout)
    eng = engine(mask, seasons, member_set, days)
    register(eng, obs)
    assert eng.observation_row_length() == max(len(o["day"]) for o in obs)
    l0 = eng.launch_count()
    chi2, used, model = run(eng, params, ic)
    assert eng.launch_count() - l0 == 4
    chi2b, usedb, modelb = run(eng, params, ic)
    assert np.array_equal(chi2, chi2b) and np.array_equal(used, usedb) and np.array_equal(model, modelb, equal_nan=True)
    out = eng.run_season(params, ic, eng.alloc_outputs(names=("snowDepths", "density")))
    depths, dens = out["snowDepths"].cpu().numpy(), out["density"].cpu().numpy()
    eng.close()
    for m, s in enumerate(member_set):
        o, n = obs[s], len(obs[s]["day"])
        want = model_values(depths[m], dens[m], seasons[s]["conc"], o, mask)
        assert np.array_equal(model[m, :n], want, equal_nan=True), m
        assert np.isnan(model[m, n:]).all()
        thin = slice(n - 5, n)                          # the density observations below minSnowD (in member m0's run)
        if m == member_set.index(s):
            assert np.isnan(model[m, thin]).all()
        ref = oracle_run(seasons[s], ic[m], params[m])
        want_chi2, want_used = scores(model_values(ref["snowDepths"], ref["density"], seasons[s]["conc"], o, mask), o)
        assert np.array_equal(used[m], want_used) and (want_used > 10).all(), (m, used[m], want_used)
        assert np.allclose(chi2[m], want_chi2, rtol=1e-12, atol=0.0), (m, chi2[m], want_chi2)


@pytest.mark.parametrize("cluster", [None, "8"])
@pytest.mark.parametrize("layout", ["single", "sets"])
def test_each_kind_is_summed_as_if_registered_alone(cuda, layout, cluster, monkeypatch):
    """Depth observations through nesosim_set_observations(_sets): chi2[:, DEPTH] is run_season_misfit's misfit bit for
    bit, the other kinds 0.  A mixed registration with sigma 1: each kind's chi2 is that of the kind registered alone."""
    if cluster:
        monkeypatch.setenv("NESOSIM_ENS_CLUSTER", cluster)
    mask, seasons, member_set, days, params, ic, obs = make_case(layout)
    eng = engine(mask, seasons, member_set, days)
    depth = [tuple(o[k][o["kind"] == DEPTH] for k in ("day", "row", "col", "value")) for o in obs]
    if layout == "single":
        eng.set_observations(depth[0])
    else:
        tag = np.concatenate([np.full(len(d[0]), i, dtype=np.int32) for i, d in enumerate(depth)])
        eng.set_observations_sets(tag, *(np.concatenate([d[j] for d in depth]) for j in range(4)))
    mis, mused = (t.cpu().numpy() for t in eng.run_season_misfit(params, ic))
    chi2, used, _ = run(eng, params, ic, model=False)
    assert np.array_equal(chi2[:, DEPTH], mis) and np.array_equal(used[:, DEPTH], mused)
    assert (chi2[:, 1:] == 0).all() and (used[:, 1:] == 0).all() and (mused > 20).all()
    register(eng, obs, sigma=False)
    mixed, mixed_used, _ = run(eng, params, ic, model=False)
    for k in range(KINDS):
        register(eng, obs, kinds=[k], sigma=False)
        alone, alone_used, _ = run(eng, params, ic, model=False)
        assert np.array_equal(mixed[:, k], alone[:, k]) and np.array_equal(mixed_used[:, k], alone_used[:, k]), k
        assert (np.delete(alone, k, axis=1) == 0).all()
    eng.close()


def test_errors_keep_the_registered_observations(cuda):
    from nesosim_b200 import _lib
    mask, seasons, member_set, days, params, ic, obs = make_case("sets")
    eng = engine(mask, seasons, member_set, days)
    register(eng, obs)
    chi2, used, model = run(eng, params, ic)
    o = {k: np.concatenate([x[k] for x in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(x["day"]), i, dtype=np.int32) for i, x in enumerate(obs)])

    def code(fn, *a, **kw):
        with pytest.raises(_lib.NesosimError) as e:
            fn(*a, **kw)
        return e.value.code

    def ex(**over):
        a = dict(o, **over)
        return code(eng.set_observations_ex, a["day"], a["row"], a["col"], a["value"], a["kind"], a["sigma"], obs_set=tag)

    for bad in (3, -1):
        k = o["kind"].copy()
        k[5] = bad
        assert ex(kind=k) == _lib.ERR_ARG
    k, d = o["kind"].copy(), o["day"].copy()
    k[5], d[5] = DENSITY, 0
    assert ex(kind=k, day=d) == _lib.ERR_ARG                                  # density on day 0
    for bad in (0.0, -1.0, np.nan, np.inf):
        sg = o["sigma"].copy()
        sg[7] = bad
        assert ex(sigma=sg) == _lib.ERR_ARG
    # a short model row
    torch = pytest.importorskip("torch")
    M, n = len(member_set), eng.observation_row_length()
    c2 = torch.empty(M, KINDS, dtype=torch.float64, device="cuda")
    mod = torch.empty(M, n, dtype=torch.float64, device="cuda")
    ic_t = eng._dev(ic)
    rc = eng.lib.nesosim_run_season_scores(eng.handle, _lib.member_params_array(params), ic_t.data_ptr(), 1,
                                           c2.data_ptr(), None, mod.data_ptr(), n - 1, eng._stream())
    assert rc == _lib.ERR_ARG
    row_len = C.c_int64(0)
    assert eng.lib.nesosim_observation_row_length(None, C.byref(row_len)) == _lib.ERR_ARG
    # the earlier observations still score, unchanged
    chi2b, usedb, modelb = run(eng, params, ic)
    assert np.array_equal(chi2, chi2b) and np.array_equal(used, usedb) and np.array_equal(model, modelb, equal_nan=True)
    # misfit cannot report density or sigma != 1
    assert code(eng.run_season_misfit, params, ic) == _lib.ERR_STATE
    register(eng, obs, kinds=[DEPTH], sigma=False)
    eng.run_season_misfit(params, ic)
    # the forcing registered again with another layout
    f = {k: np.stack([np.concatenate([x[k], np.zeros((T - len(x[k]),) + x[k].shape[1:])]) for x in seasons])
         for k in ("precip", "conc", "wind", "drift")}
    eng.set_forcing_sets(f["precip"], f["conc"], f["wind"], f["drift"], member_set, [14, 17, 19])
    assert code(eng.run_season_scores, params, ic) == _lib.ERR_STATE
    eng.close()


def driver_seasons(mask, seed):
    rng = np.random.default_rng(seed)
    out = []
    for s, d in enumerate(DAYS):
        o = make_obs(mask, d, rng, 400 + 50 * s)
        out.append({"forcing": S.make_season(mask, d, seed=seed + s), "ic": S.make_ic(mask, seed=seed + s) * (1 + s),
                    "obs": o if s != 1 else (o["day"], o["row"], o["col"], o["value"])})   # season 1: a 4-tuple
    return out


def test_run_calibration_scores_fused_agrees_with_the_hbm_round_trip(cuda):
    from nesosim_b200 import ensemble as ENS
    mask = S.region_mask(dx=DX)
    seasons = driver_seasons(mask, 180)
    params = S.ensemble_params(3, seed=181)
    a = ENS.run_calibration_scores(mask, seasons, params, DX, atmlossInc=1, model=True)
    b = ENS.run_calibration_scores(mask, seasons, params, DX, atmlossInc=1, model=True, fused=False)
    assert a["chi2"].shape == (3, 3, KINDS) and a["used"].shape == (3, 3, KINDS)
    assert np.array_equal(a["used"], b["used"]) and np.allclose(a["chi2"], b["chi2"], rtol=1e-12, atol=0.0)
    for s in range(3):
        assert a["model"][s].shape == (3, len(seasons[s]["obs"][0] if s == 1 else seasons[s]["obs"]["day"]))
        assert np.array_equal(a["model"][s], b["model"][s], equal_nan=True), s
    assert (a["used"][:, 1, 1:] == 0).all() and (a["used"][:, [0, 2]] > 5).all()
    none = ENS.run_calibration_scores(mask, seasons, params, DX, atmlossInc=1)
    assert none["model"] is None and np.array_equal(none["chi2"], a["chi2"])


def test_run_calibration_scores_falls_back_on_grids_the_season_kernel_does_not_take(cuda):
    from nesosim_b200 import _lib
    from nesosim_b200 import ensemble as ENS
    mask = S.region_mask(shape=(40, 130), kind="disc")
    seasons = driver_seasons(mask, 190)
    params = S.ensemble_params(2, seed=191)
    with pytest.raises(_lib.NesosimError):
        ENS.run_calibration_scores(mask, seasons, params, DX, atmlossInc=1, fused=True)
    res = ENS.run_calibration_scores(mask, seasons, params, DX, atmlossInc=1, model=True)
    for p in range(2):
        for s in range(3):
            o = ENS.normalize_observations(seasons[s]["obs"])
            f = seasons[s]["forcing"]
            ref = O.run_season(f, seasons[s]["ic"], mask, DX, oracle_params(params[p]), O.Flags(atmlossInc=1))
            want_model = model_values(ref["snowDepths"], ref["density"], f["conc"], o, mask)
            want_chi2, want_used = scores(want_model, o)
            assert np.array_equal(res["used"][p, s], want_used)
            assert np.allclose(res["chi2"][p, s], want_chi2, rtol=1e-12, atol=0.0), (p, s)
            assert np.allclose(res["model"][s][p], want_model, rtol=1e-12, atol=0.0, equal_nan=True)
