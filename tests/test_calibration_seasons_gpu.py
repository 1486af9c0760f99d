"""GPU: multi-season calibration -- observations tagged with their season (nesosim_set_observations_sets) and the fused
misfit of every member against its own season's observations in one batched launch (nesosim_run_season_misfit on a
context with forcing sets), and the driver ensemble.run_calibration on top of it."""
import numpy as np
import pytest

from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O

pytestmark = pytest.mark.gpu

DX = 100000
T = 20
DAYS = [14, 17, 20]                    # three seasons of different length in a T = 20 context
MEMBER_SET = [2, 0, 1, 0, 2, 1, 2]     # not grouped by season
EMPTY = 1                              # the season without any observation


def oracle_params(row):
    return O.Params(windPackFactor=row[0], windPackThresh=row[1], leadLossFactor=row[2], atmLossFactor=row[3])


def make_case():
    mask = S.region_mask(dx=DX)
    ny, nx = mask.shape
    seasons = [S.make_season(mask, d, seed=70 + s) for s, d in enumerate(DAYS)]
    M = len(MEMBER_SET)
    params = S.ensemble_params(M, seed=71)
    rng = np.random.default_rng(72)
    ic = S.make_ic(mask, seed=72)[None] * rng.uniform(0.5, 3.0, (M, 1, 1))
    obs = []
    for s, d in enumerate(DAYS):
        n = 0 if s == EMPTY else 600 + 150 * s
        row, col = rng.integers(0, ny, n), rng.integers(0, nx, n)     # every strip; a good half of them on land
        day = rng.integers(0, d, n)
        if n:
            day[:30] = 0
            day[30:60] = d - 1                                       # the season's last day
            row[100:110], col[100:110], day[100:110] = row[100], col[100], day[100]   # one cell and day, ten times
            day[110:115] = day[100]                                   # ... and five more at other cells that day
        obs.append((day, row, col, 0.3 * rng.random(n)))
    return mask, seasons, params, ic, obs


def stacked(seasons):
    out = {}
    for k in ("precip", "conc", "wind", "drift"):
        a = np.zeros((len(seasons), T) + seasons[0][k].shape[1:])
        for s, f in enumerate(seasons):
            a[s, :len(f[k])] = f[k]
        out[k] = a
    return out


def tagged(obs):
    tag = np.concatenate([np.full(len(o[0]), s, dtype=np.int32) for s, o in enumerate(obs)])
    return (tag,) + tuple(np.concatenate([o[j] for o in obs]) for j in range(4))


def batch_engine(mask, seasons, obs, M=len(MEMBER_SET)):
    from nesosim_b200.engine import SnowBudgetEngine
    f = stacked(seasons)
    eng = SnowBudgetEngine(mask, T, DX, n_members=M, atmlossInc=1)
    eng.set_forcing_sets(f["precip"], f["conc"], f["wind"], f["drift"], MEMBER_SET[:M], DAYS)
    eng.set_observations_sets(*tagged(obs))
    return eng


def expected(mask, season, ic, row, obs):
    ref = O.run_season(season, ic, mask, DX, oracle_params(row), O.Flags(atmlossInc=1))
    day, r, c, depth = obs
    with np.errstate(all="ignore"):
        model = (ref["snowDepths"][day, 0, r, c] + ref["snowDepths"][day, 1, r, c]) / season["conc"][day, r, c]
    d = model - depth
    ok = np.isfinite(d)
    return np.sum(d[ok] ** 2), ok.sum()


@pytest.mark.parametrize("cluster", [None, "8"])
def test_batch_matches_the_oracle_deterministically_in_four_launches(cuda, cluster, monkeypatch):
    """Every member's misfit against its own season's observations equals the oracle's to 1e-12 (different summation
    order), counts exact; the season without observations gives 0 and 0; two runs are bit-identical and each is the
    pre-pass (2), the season kernel and the epilogue, however many seasons."""
    if cluster:
        monkeypatch.setenv("NESOSIM_ENS_CLUSTER", cluster)
    mask, seasons, params, ic, obs = make_case()
    eng = batch_engine(mask, seasons, obs)
    l0 = eng.launch_count()
    mis, used = (t.cpu().numpy() for t in eng.run_season_misfit(params, ic))
    assert eng.launch_count() - l0 == 4
    mis2, used2 = (t.cpu().numpy() for t in eng.run_season_misfit(params, ic))
    assert np.array_equal(mis, mis2) and np.array_equal(used, used2)
    eng.close()
    for m, s in enumerate(MEMBER_SET):
        want, n = expected(mask, seasons[s], ic[m], params[m], obs[s])
        if s == EMPTY:
            assert mis[m] == 0.0 and used[m] == 0
            continue
        assert used[m] == n and n > 100, (m, used[m], n)
        assert np.isclose(mis[m], want, rtol=1e-12, atol=0.0), (m, mis[m], want)


@pytest.mark.parametrize("cluster", ["8", "6"])
def test_each_member_equals_its_season_on_its_own(cuda, cluster, monkeypatch):
    """Same strips (cluster size pinned) -> every member's misfit is bit-identical to run_season_misfit on a
    single-forcing context of its season's length with that season's observations."""
    from nesosim_b200.engine import SnowBudgetEngine
    monkeypatch.setenv("NESOSIM_ENS_CLUSTER", cluster)
    mask, seasons, params, ic, obs = make_case()
    eng = batch_engine(mask, seasons, obs)
    mis, used = (t.cpu().numpy() for t in eng.run_season_misfit(params, ic))
    eng.close()
    for s, d in enumerate(DAYS):
        members = [m for m, ms in enumerate(MEMBER_SET) if ms == s]
        one = SnowBudgetEngine(mask, d, DX, n_members=len(members), atmlossInc=1)
        f = seasons[s]
        one.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
        ic_s = ic[members] if len(members) > 1 else ic[members[0]]
        m1, u1 = (t.cpu().numpy() for t in one.run_season_misfit(params[members], ic_s, obs[s]))
        one.close()
        assert np.array_equal(mis[members], m1), (s, mis[members], m1)
        assert np.array_equal(used[members], u1)


def test_errors_and_stale_observations(cuda):
    from nesosim_b200 import _lib
    from nesosim_b200.engine import SnowBudgetEngine
    mask, seasons, params, ic, obs = make_case()
    eng = batch_engine(mask, seasons, obs)
    tag, day, row, col, depth = tagged(obs)
    f = stacked(seasons)

    def code(fn, *a):
        with pytest.raises(_lib.NesosimError) as e:
            fn(*a)
        return e.value.code

    bad = tag.copy()
    bad[0] = 3
    assert code(eng.set_observations_sets, bad, day, row, col, depth) == _lib.ERR_ARG      # set index out of range
    bad[0] = -1
    assert code(eng.set_observations_sets, bad, day, row, col, depth) == _lib.ERR_ARG
    late = day.copy()
    late[0] = DAYS[tag[0]]                                                                  # at its set's set_days
    assert code(eng.set_observations_sets, tag, late, row, col, depth) == _lib.ERR_ARG
    off = row.copy()
    off[0] = mask.shape[0]
    assert code(eng.set_observations_sets, tag, day, off, col, depth) == _lib.ERR_ARG
    # plain observations on a context with forcing sets: unchanged
    eng.set_observations(obs[0])
    assert code(eng.run_season_misfit, params, ic) == _lib.ERR_ARG
    # the forcing registered again with another layout, or as one season: stale until registered again
    eng.set_observations_sets(tag, day, row, col, depth)
    eng.run_season_misfit(params, ic)
    eng.set_forcing_sets(f["precip"], f["conc"], f["wind"], f["drift"], MEMBER_SET, [14, 17, 19])
    assert code(eng.run_season_misfit, params, ic) == _lib.ERR_STATE
    eng.set_forcing_sets(f["precip"], f["conc"], f["wind"], f["drift"], MEMBER_SET, DAYS)
    eng.run_season_misfit(params, ic)                                                       # same layout again
    eng.set_forcing(f["precip"][2], f["conc"][2], f["wind"][2], f["drift"][2])
    assert code(eng.run_season_misfit, params, ic) == _lib.ERR_STATE
    assert code(eng.set_observations_sets, tag, day, row, col, depth) == _lib.ERR_STATE    # no forcing sets
    eng.close()
    one = SnowBudgetEngine(mask, T, DX, n_members=2, atmlossInc=1)
    one.set_forcing(f["precip"][2], f["conc"][2], f["wind"][2], f["drift"][2])
    assert code(one.set_observations_sets, tag, day, row, col, depth) == _lib.ERR_STATE
    one.close()


def driver_seasons(mask, seed):
    rng = np.random.default_rng(seed)
    ny, nx = mask.shape
    out = []
    for s, d in enumerate(DAYS):
        n = 0 if s == EMPTY else 500
        day = rng.integers(0, d, n)
        if n:
            day[:20], day[20:40] = 0, d - 1
        out.append({"forcing": S.make_season(mask, d, seed=seed + s), "ic": S.make_ic(mask, seed=seed + s) * (1 + s),
                    "obs": (day, rng.integers(0, ny, n), rng.integers(0, nx, n), 0.3 * rng.random(n))})
    return out


def test_run_calibration_fused_agrees_with_the_hbm_round_trip(cuda):
    from nesosim_b200 import ensemble as ENS
    mask = S.region_mask(dx=DX)
    seasons = driver_seasons(mask, 80)
    params = S.ensemble_params(3, seed=81)
    a = ENS.run_calibration(mask, seasons, params, DX, atmlossInc=1, fused=True)
    b = ENS.run_calibration(mask, seasons, params, DX, atmlossInc=1, fused=False)
    assert a[0].shape == (3, 3) and a[1].shape == (3, 3)
    assert np.allclose(a[0], b[0], rtol=1e-12, atol=0.0) and np.array_equal(a[1], b[1])
    assert (a[1][:, EMPTY] == 0).all() and (a[1][:, [0, 2]] > 50).all()
    for p in range(3):                                   # spot check against the oracle
        s = 2
        want, n = expected(mask, seasons[s]["forcing"], seasons[s]["ic"], params[p], seasons[s]["obs"])
        assert a[1][p, s] == n and np.isclose(a[0][p, s], want, rtol=1e-12, atol=0.0)


def test_run_calibration_falls_back_on_grids_the_season_kernel_does_not_take(cuda):
    from nesosim_b200 import _lib
    from nesosim_b200 import ensemble as ENS
    mask = S.region_mask(shape=(40, 130), kind="disc")
    seasons = driver_seasons(mask, 90)
    params = S.ensemble_params(2, seed=91)
    with pytest.raises(_lib.NesosimError):
        ENS.run_calibration(mask, seasons, params, DX, atmlossInc=1, fused=True)
    mis, used = ENS.run_calibration(mask, seasons, params, DX, atmlossInc=1)
    for p in range(2):
        for s in range(3):
            want, n = expected(mask, seasons[s]["forcing"], seasons[s]["ic"], params[p], seasons[s]["obs"])
            assert used[p, s] == n
            assert np.isclose(mis[p, s], want, rtol=1e-12, atol=0.0), (p, s)
