"""GPU: the fused calibration scores (nesosim_set_observations_ex + nesosim_run_season_scores) bit for bit against the
float64 restatement of their fixed summation order (oracle/observation_scores.py) on the oracle's season arrays.

The summation order does not depend on the strip cut (the sort key is monotone in row*nx + col for every cut), so chi2
must be bit-identical on every build variant of the season kernel in its OBS and SETS && OBS instantiations, every
cluster size and any number of members per cluster.  Covered: every variant with one or two clusters running members
of different season lengths (odd and even step counts) one after the other; every variant of the plain SETS
instantiation; cluster sizes 2..8; masks with all-land rows at forced strip boundaries, ragged discs, an all-ocean grid,
a 30 000-observation case; scoring mode with operands outside the fast divisions' range (the drivers fall back); and
the drivers' range errors.  Every NESOSIM_ENS_* variable is set before the context builds its strip tables (at the
observation registration): a forced variant or cluster size that does not fit raises ERR_ARG, it never runs another."""
import functools

import numpy as np
import pytest

from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O
from oracle import observation_scores as R

pytestmark = pytest.mark.gpu

DEPTH, VOLUME, DENSITY, KINDS = R.DEPTH, R.VOLUME, R.DENSITY, R.KINDS
ENV = ("NESOSIM_ENS_VARIANT", "NESOSIM_ENS_CLUSTER", "NESOSIM_ENS_CLUSTERS", "NESOSIM_ENS_ROWS", "NESOSIM_ENS_COST",
       "NESOSIM_ENS_DBG", "NESOSIM_ENS_TIMING")
VARIANTS = ["t352r3o2", "t224r4o3", "t480r2o2", "t608r2o1", "t480r2o1", "t736r2o1", "t352r6o5"]
DAYS = [10, 13, 14]                    # forcing sets: 9, 12 and 13 steps
MEMBER_SET = [2, 0, 1, 1, 0, 2, 1]     # two clusters: members 0,2,4,6 (13,12,9,12 steps) and 1,3,5 (9,12,13 steps)
SINGLE_DAYS, SINGLE_M = 13, 5
BOUNDARY = [("5", "18,36,54,72", 3), ("6", "16,30,44,60,76", 55), ("6", "14,30,46,62,78", 55)]
CLUSTER_MASK = {2: "arctic:20:44", 3: "arctic:20:56", 4: "arctic:20:68"}   # smaller cuts for clusters of 2..4 CTAs


def clear_env(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)


def oracle_params(row):
    return O.Params(windPackFactor=row[0], windPackThresh=row[1], leadLossFactor=row[2], atmLossFactor=row[3])


def make_mask(name):
    """(mask, dx) by name: "arctic" (the 100 km grid), "arctic:a:b" (its rows a..b-1), "disc:ny:nx", "ocean" (90 x 90,
    all ocean), "boundary:rows:land_cols" (all-land row bands straddling the forced strip boundaries `rows`)."""
    kind, *arg = name.split(":")
    if kind == "arctic":
        m = S.region_mask(dx=100000)
        return (np.ascontiguousarray(m[int(arg[0]):int(arg[1])]) if arg else m), 100000
    if kind == "disc":
        return S.region_mask(shape=(int(arg[0]), int(arg[1])), kind="disc"), 50000
    if kind == "ocean":
        return np.full((90, 90), 8, dtype=np.uint8), 100000
    cuts, land_cols = [int(r) for r in arg[0].split(",")], int(arg[1])
    m = np.full((90, 90), 8, dtype=np.uint8)
    m[cuts[0] - 2:cuts[0] + 2] = 11               # land on both sides of the first boundary
    m[cuts[1]:cuts[1] + 2] = 11                   # only the lower strip's top rows are land
    m[cuts[2] - 2:cuts[2]] = 11                   # only the upper strip's bottom rows are land
    m[:, :land_cols] = 11
    m[40:43, 60:70] = 0
    return m, 100000


def make_obs(mask, days, rng, n, focus=(), kind_p=None, scale=1.0):
    """n observations of all kinds on land and ocean: depth and volume on day 0, every kind on the last day, one ocean
    cell-day observed ten times across the kinds, 30 more cell-days observed twice, sigma log-uniform over 1e-3..10,
    5 % NaN values.  `focus`: rows that get 60 % of the observations.  `scale` multiplies the depth and volume values
    and their sigmas."""
    ny, nx = mask.shape
    row, col, day = rng.integers(0, ny, n), rng.integers(0, nx, n), rng.integers(0, days, n)
    if len(focus):
        f = rng.random(n) < 0.6
        row[f] = rng.choice(np.asarray(focus), f.sum())
    kind = rng.choice(KINDS, n, p=kind_p)
    day[:30] = 0
    day[30:60] = days - 1
    wet = np.argwhere(R.ocean(mask))
    row[100:110], col[100:110] = wet[rng.integers(len(wet))]
    day[100:110] = max(day[100], 1)
    kind[100:110] = [0, 1, 2, 0, 1, 2, 0, 1, 2, 0]
    for a in (row, col, day):
        a[140:170] = a[110:140]
    kind[(day == 0) & (kind == DENSITY)] = VOLUME
    value = np.where(kind == DENSITY, 200.0 + 150.0 * rng.random(n), 0.3 * scale * rng.random(n))
    value[rng.random(n) < 0.05] = np.nan
    sigma = 10.0 ** rng.uniform(-3, 1, n) * np.where(kind == DENSITY, 1.0, scale)
    return {"day": day, "row": row, "col": col, "value": value, "kind": kind, "sigma": sigma}


@functools.lru_cache(maxsize=None)
def case(mask_name, layout, sizes=None, focus=(), kind_p=None, seed=0):
    """Inputs of one fused run: forcing per set, member_set, params, per-member ICs (snow on land too), observations per
    set.  Cached: the oracle runs (`expected`) are shared by every test on the same case."""
    mask, dx = make_mask(mask_name)
    if layout == "single":
        member_set, days = [0] * SINGLE_M, [SINGLE_DAYS]
    else:
        member_set, days = MEMBER_SET, DAYS
    sizes = sizes or tuple(700 + 100 * s for s in range(len(days)))
    rng = np.random.default_rng(seed)
    M = len(member_set)
    seasons = [S.make_season(mask, d, seed=seed + 1 + s) for s, d in enumerate(days)]
    ic = (0.02 + S.make_ic(mask, seed=seed + 5))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    obs = [make_obs(mask, d, rng, n, focus, kind_p) for d, n in zip(days, sizes)]
    return {"mask": mask, "dx": dx, "layout": layout, "member_set": member_set, "days": days, "seasons": seasons,
            "params": S.ensemble_params(M, seed=seed + 6), "ic": ic, "obs": obs}


def expected(c):
    """Per member: (oracle arrays of its own season, model row, chi2, used) from the restatement."""
    if "want" not in c:
        c["want"] = []
        for m, s in enumerate(c["member_set"]):
            f = c["seasons"][s]
            ref = O.run_season(f, c["ic"][m], c["mask"], c["dx"], oracle_params(c["params"][m]), O.Flags(atmlossInc=1))
            model = R.model_values(ref["snowDepths"], ref["density"], f["conc"], c["obs"][s], c["mask"])
            c["want"].append((ref, model) + R.scores(model, c["obs"][s], c["mask"]))
    return c["want"]


def engine(c):
    from nesosim_b200.engine import SnowBudgetEngine
    T = max(c["days"])
    eng = SnowBudgetEngine(c["mask"], T, c["dx"], n_members=len(c["member_set"]), atmlossInc=1)
    if c["layout"] == "single":
        f = c["seasons"][0]
        eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
    else:   # the sets stacked to the longest; days past a set's end are never read
        st = {k: np.stack([np.concatenate([f[k], np.zeros((T - len(f[k]),) + f[k].shape[1:])]) for f in c["seasons"]])
              for k in ("precip", "conc", "wind", "drift")}
        eng.set_forcing_sets(st["precip"], st["conc"], st["wind"], st["drift"], c["member_set"], c["days"])
    return eng


def register(eng, obs, sets):
    cat = {k: np.concatenate([o[k] for o in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(obs)]) if sets else None
    eng.set_observations_ex(cat["day"], cat["row"], cat["col"], cat["value"], cat["kind"], cat["sigma"], obs_set=tag)


def fused(c):
    """(chi2, used, model) of the fused path on the current NESOSIM_ENS_* settings."""
    eng = engine(c)
    register(eng, c["obs"], c["layout"] == "sets")
    got = tuple(t.cpu().numpy() for t in eng.run_season_scores(c["params"], c["ic"], model=True))
    eng.close()
    return got


def check_scores(c, got):
    chi2, used, model = got
    for m, s in enumerate(c["member_set"]):
        _, want_model, want_chi2, want_used = expected(c)[m]
        n = len(c["obs"][s]["day"])
        bad = np.flatnonzero(~((model[m, :n] == want_model) | (np.isnan(model[m, :n]) & np.isnan(want_model))))
        assert not len(bad), ("model row", m, bad[:5], model[m, bad[:5]], want_model[bad[:5]])
        assert np.isnan(model[m, n:]).all(), m
        assert np.array_equal(used[m], want_used), (m, used[m], want_used)
        assert np.array_equal(chi2[m], want_chi2), (m, chi2[m], want_chi2, chi2[m] - want_chi2)
    assert (used > 0).all()                      # every member scores every kind: the comparison is not vacuous


@functools.lru_cache(maxsize=None)
def default_run(mask_name, layout):
    """The fused run on automatic selection (call with every NESOSIM_ENS_* variable cleared)."""
    return fused(case(mask_name, layout))


@pytest.mark.parametrize("layout", ["single", "sets"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_every_variant_scores_bit_for_bit(cuda, variant, layout, monkeypatch):
    """OBS (one forcing) and SETS && OBS of every build variant, all members on one or two clusters: model rows, chi2
    and counts identical to the restatement and to the run on automatic selection (one member per cluster)."""
    clear_env(monkeypatch)
    auto = default_run("arctic", layout)
    clusters = 1 + (VARIANTS.index(variant) + (layout == "sets")) % 2
    monkeypatch.setenv("NESOSIM_ENS_VARIANT", variant)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTERS", str(clusters))
    c = case("arctic", layout)
    got = fused(c)
    check_scores(c, got)
    for a, b in zip(got, auto):
        assert np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("variant", VARIANTS)
def test_every_variant_of_the_plain_forcing_sets_kernel(cuda, variant, monkeypatch):
    """run_season on forcing sets (the plain SETS instantiation) of every build variant, members of three season
    lengths on two clusters: all 11 arrays value-identical to the oracle; slots past a member's season untouched."""
    from nesosim_b200 import _lib
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_ENS_VARIANT", variant)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTERS", "2")
    c = case("arctic", "sets")
    eng = engine(c)
    eng.set_path("ensemble")
    out = eng.alloc_outputs()
    for t in out.values():
        t.fill_(-5.0)
    out = {k: v.cpu().numpy() for k, v in eng.run_season(c["params"], c["ic"], out).items()}
    assert eng.last_path() == "ensemble" and eng.rerun_count() == 0
    eng.close()
    assert sorted(out) == sorted(_lib.OUTPUT_NAMES) and len(out) == 11
    for m, s in enumerate(c["member_set"]):
        d, ref = c["days"][s], expected(c)[m][0]
        for name in out:
            assert np.array_equal(out[name][m][:d], ref[name], equal_nan=True), (name, m)
            assert (out[name][m][d:] == -5.0).all(), (name, m)


@pytest.mark.parametrize("layout", ["single", "sets"])
@pytest.mark.parametrize("cluster", range(2, 9))
def test_every_cluster_size(cuda, cluster, layout, monkeypatch):
    """Clusters of 2..8 CTAs, several members per cluster; 2..4 on cuts of the 100 km grid small enough to fit."""
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTER", str(cluster))
    monkeypatch.setenv("NESOSIM_ENS_CLUSTERS", "2")
    c = case(CLUSTER_MASK.get(cluster, "arctic"), layout)
    check_scores(c, fused(c))


@pytest.mark.parametrize("layout", ["single", "sets"])
@pytest.mark.parametrize("cluster,rows,land_cols", BOUNDARY)
def test_all_land_rows_at_a_strip_boundary(cuda, cluster, rows, land_cols, layout, monkeypatch):
    """The strip-boundary masks of the season kernel's halo tests, most observations in the rows on both sides of
    each forced cut."""
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTERS", "2")
    monkeypatch.setenv("NESOSIM_ENS_CLUSTER", cluster)
    monkeypatch.setenv("NESOSIM_ENS_ROWS", rows)
    focus = tuple(r for cut in rows.split(",") for r in range(int(cut) - 4, int(cut) + 4))
    c = case("boundary:%s:%d" % (rows, land_cols), layout, focus=focus)
    check_scores(c, fused(c))


@pytest.mark.parametrize("layout", ["single", "sets"])
@pytest.mark.parametrize("mask_name", ["disc:45:70", "disc:94:33", "disc:9:96", "ocean"])
def test_ragged_and_all_ocean_grids(cuda, mask_name, layout, monkeypatch):
    """Ragged discs and an all-ocean 90 x 90 grid on automatic selection of the variant and the cluster size."""
    clear_env(monkeypatch)
    c = case(mask_name, layout)
    check_scores(c, fused(c))


def test_thirty_thousand_observations(cuda, monkeypatch):
    """30 000 observations in sets of 15 000, 5 000 and 10 000, 80 % depth and 5 % density: an epilogue thread sums
    up to 20 ocean observations of one kind, and the kinds' ranges differ by a factor of 15."""
    clear_env(monkeypatch)
    c = case("arctic", "sets", sizes=(15000, 5000, 10000), kind_p=(0.8, 0.15, 0.05), seed=7)
    got = fused(c)
    check_scores(c, got)
    assert (got[1][:, DEPTH] > 10 * got[1][:, DENSITY]).all() and got[1][:, DEPTH].max() > 2000


def test_scoring_mode_with_operands_outside_the_fast_divisions(cuda, monkeypatch):
    """Depths around 1e-300 leave the proven range of the season kernel's fast divisions.  Scoring mode has no general
    fall-back: nesosim_run_season_scores raises ERR_ARG, and the same context then scores an in-range season bit for
    bit.  The drivers fall back to the HBM round trip on fused=None (equal to the oracle to 1e-12: torch sums in another
    order) and raise on fused=True."""
    from nesosim_b200 import _lib
    from nesosim_b200 import ensemble as ENS
    from nesosim_b200.engine import SnowBudgetEngine
    clear_env(monkeypatch)
    mask, dx, T, M = S.region_mask(dx=100000), 100000, 6, 3
    rng = np.random.default_rng(31)
    tiny = S.make_season(mask, T, seed=31)
    tiny["precip"] = tiny["precip"] * 1e-300
    tiny_ic = S.make_ic(mask, seed=31) * 1e-298
    tiny_obs = make_obs(mask, T, rng, 600, scale=1e-300)
    params = S.ensemble_params(M, seed=31)
    eng = SnowBudgetEngine(mask, T, dx, n_members=M, atmlossInc=1)
    eng.set_forcing(tiny["precip"], tiny["conc"], tiny["wind"], tiny["drift"])
    register(eng, [tiny_obs], False)
    with pytest.raises(_lib.NesosimError) as e:
        eng.run_season_scores(params, tiny_ic, model=True)
    assert e.value.code == _lib.ERR_ARG and "fast divisions" in str(e.value)
    # the same context, an in-range season
    f = S.make_season(mask, T, seed=32)
    ic = S.make_ic(mask, seed=32)
    o = make_obs(mask, T, rng, 600)
    eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
    register(eng, [o], False)
    chi2, used, model = (t.cpu().numpy() for t in eng.run_season_scores(params, ic, model=True))
    eng.close()
    for m in range(M):
        ref = O.run_season(f, ic, mask, dx, oracle_params(params[m]), O.Flags(atmlossInc=1))
        want_model = R.model_values(ref["snowDepths"], ref["density"], f["conc"], o, mask)
        want_chi2, want_used = R.scores(want_model, o, mask)
        assert np.array_equal(model[m], want_model, equal_nan=True), m
        assert np.array_equal(chi2[m], want_chi2) and np.array_equal(used[m], want_used), m
    # the drivers on the out-of-range season
    depth = {k: v[tiny_obs["kind"] == DEPTH] for k, v in tiny_obs.items()}
    depth["value"] = 1e-150 * rng.random(len(depth["day"]))           # (model - value)^2 ~ 1e-300: not zero
    depth["sigma"] = np.ones(len(depth["day"]))
    tup = (depth["day"], depth["row"], depth["col"], depth["value"])
    want = []
    for m in range(M):
        ref = O.run_season(tiny, tiny_ic, mask, dx, oracle_params(params[m]), O.Flags(atmlossInc=1))
        wm = R.model_values(ref["snowDepths"], ref["density"], tiny["conc"], tiny_obs, mask)
        wd = R.model_values(ref["snowDepths"], ref["density"], tiny["conc"], depth, mask)
        want.append((wm, R.scores(wm, tiny_obs, mask), R.scores(wd, depth, mask)))
    season = {"forcing": tiny, "ic": tiny_ic, "obs": tiny_obs}
    res = ENS.run_calibration_scores(mask, [season], params, dx, atmlossInc=1, model=True)
    mis, mused = ENS.run_calibration(mask, [dict(season, obs=tup)], params, dx, atmlossInc=1)
    ens, eused = ENS.run_ensemble(mask, tiny, tiny_ic, params, dx, tup, atmlossInc=1)
    for m, (wm, (wc, wu), (dc, du)) in enumerate(want):
        assert np.array_equal(res["model"][0][m], wm, equal_nan=True), m
        assert np.array_equal(res["used"][m, 0], wu) and (wu[:DENSITY] > 20).all(), m
        assert np.allclose(res["chi2"][m, 0], wc, rtol=1e-12, atol=0.0), (m, res["chi2"][m, 0], wc)
        for got, n in ((mis[m, 0], mused[m, 0]), (ens[m], eused[m])):
            assert n == du[DEPTH] > 20 and dc[DEPTH] > 0.0, m
            assert np.isclose(got, dc[DEPTH], rtol=1e-12, atol=0.0), (m, got, dc[DEPTH])
    with pytest.raises(_lib.NesosimError):
        ENS.run_calibration_scores(mask, [season], params, dx, atmlossInc=1, fused=True)
    with pytest.raises(_lib.NesosimError):
        ENS.run_calibration(mask, [dict(season, obs=tup)], params, dx, atmlossInc=1, fused=True)
    with pytest.raises(_lib.NesosimError):
        ENS.run_ensemble(mask, tiny, tiny_ic, params, dx, tup, atmlossInc=1, fused=True)


def test_drivers_raise_on_observations_outside_the_grid_or_their_season(cuda, monkeypatch):
    """A day in [T_s, T) of a shorter season in the batch (a slot of the stacked context the season never writes) and
    row -1 (which would wrap around to the last row): ValueError on the fused and the HBM path."""
    from nesosim_b200 import ensemble as ENS
    clear_env(monkeypatch)
    mask, dx = S.region_mask(dx=100000), 100000
    rng = np.random.default_rng(41)
    days = [8, 11]
    seasons = [{"forcing": S.make_season(mask, d, seed=41 + s), "ic": S.make_ic(mask, seed=41),
                "obs": make_obs(mask, d, rng, 300)} for s, d in enumerate(days)]
    params = S.ensemble_params(2, seed=41)

    def tup(o):
        return (o["day"], o["row"], o["col"], o["value"])

    for field, value in (("day", days[0]), ("row", -1)):
        bad = [dict(s, obs=dict(s["obs"])) for s in seasons]
        bad[0]["obs"][field] = bad[0]["obs"][field].copy()
        bad[0]["obs"][field][200] = value
        for fused_ in (None, False):
            with pytest.raises(ValueError):
                ENS.run_calibration_scores(mask, bad, params, dx, atmlossInc=1, fused=fused_)
            with pytest.raises(ValueError):
                ENS.run_calibration(mask, [dict(s, obs=tup(s["obs"])) for s in bad], params, dx, atmlossInc=1,
                                    fused=fused_)
            if field == "row":
                with pytest.raises(ValueError):
                    ENS.run_ensemble(mask, bad[0]["forcing"], bad[0]["ic"], params, dx, tup(bad[0]["obs"]),
                                     atmlossInc=1, fused=fused_)
