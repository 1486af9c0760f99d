"""CPU: the float64 restatement of the fused calibration scores (oracle/observation_scores.py) pinned against plain sums
and hand-made cases whose value depends on the summation order, and the drivers' range checks: an observation outside
the grid or outside its own season's days is rejected with ValueError before any engine exists, on every path."""
import numpy as np
import pytest

from nesosim_b200 import synthetic as S
from oracle import observation_scores as R

DEPTH, VOLUME, DENSITY, KINDS = R.DEPTH, R.VOLUME, R.DENSITY, R.KINDS
TINY = 2.0 ** -53                                   # half an ulp of 1.0


def grid_obs(mask, n, rng):
    ny, nx = mask.shape
    return {"day": rng.integers(0, 9, n), "row": rng.integers(0, ny, n), "col": rng.integers(0, nx, n),
            "kind": rng.integers(0, KINDS, n), "value": rng.random(n), "sigma": 10.0 ** rng.uniform(-3, 1, n)}


def test_fixed_order_sum_is_the_plain_sum_to_1e12():
    rng = np.random.default_rng(0)
    for n in (0, 1, 255, 256, 257, 5000, 30011):
        t = rng.random(n) * 10.0 ** rng.uniform(-6, 6, n)
        got = R.fixed_order_sum(t)
        assert got == pytest.approx(np.sum(t), rel=1e-12, abs=0.0), n
    assert R.fixed_order_sum([]) == 0.0 and R.fixed_order_sum([2.5]) == 2.5


def test_fixed_order_sum_follows_the_threads_and_the_warps():
    def at(positions, n=600):
        t = np.zeros(n)
        for p, v in positions.items():
            t[p] = v
        return R.fixed_order_sum(t)
    # 1, 2^-53, 2^-53 in one thread (observations 0, 256, 512): each small term rounds away
    assert at({0: 1.0, 256: TINY, 512: TINY}) == 1.0
    # the two small terms in another thread (observations 1 and 257): they add up first and survive
    assert at({0: 1.0, 1: TINY, 257: TINY}) == 1.0 + 2 * TINY
    # three warps combined one after the other from warp 0: (1 + 2^-53) + 2^-53 = 1 (reversed it would be 1 + 2^-52)
    assert at({0: 1.0, 32: TINY, 64: TINY}) == 1.0
    # inside a warp the shuffle tree pairs lane l with l + 16, then l + 8, ...: lanes 1 and 17 meet before lane 0
    assert at({0: 1.0, 1: TINY, 17: TINY}) == 1.0 + 2 * TINY
    assert at({0: 1.0, 1: TINY, 2: TINY}) == 1.0


def test_scores_sort_by_cell_then_day_whatever_the_input_order():
    """The same three terms r^2 = 1, 2^-54, 2^-54, 2^-54 (r = 1, 2^-27) placed by the (cell, day) order: all in thread 0
    gives 1; the small ones in thread 1 gives 1 + 2^-52.  The input order is shuffled and must not matter."""
    mask = np.full((30, 40), 8, dtype=np.uint8)
    n = 1000
    cells = np.arange(n)
    rng = np.random.default_rng(1)
    for small_at, want in (((256, 512, 768), 1.0), ((1, 257, 513), 1.0 + 2.0 ** -52)):
        model = np.zeros(n)
        model[0] = 1.0
        model[list(small_at)] = 2.0 ** -27
        perm = rng.permutation(n)
        obs = {"day": np.full(n, 3)[perm], "row": (cells // 40)[perm], "col": (cells % 40)[perm],
               "kind": np.full(n, VOLUME)[perm], "value": np.zeros(n), "sigma": np.ones(n)}
        chi2, used = R.scores(model[perm], obs, mask)
        assert chi2[VOLUME] == want and used.tolist() == [0, n, 0]
    # an observation whose r is not finite keeps its place: with a NaN value at position 1, the small terms at 257, 513
    # and 769 still meet in thread 1 (dropping the NaN first would move them to thread 0, where they round away)
    model = np.zeros(n)
    model[0] = 1.0
    model[[257, 513, 769]] = 2.0 ** -27
    value = np.zeros(n)
    value[1] = np.nan
    obs = {"day": np.full(n, 3), "row": cells // 40, "col": cells % 40, "kind": np.full(n, DEPTH), "value": value,
           "sigma": np.ones(n)}
    chi2, used = R.scores(model, obs, mask)
    assert chi2[DEPTH] == 1.0 + 2.0 ** -52 and used.tolist() == [n - 1, 0, 0]
    # one cell observed on several days: the day orders them, and equal (cell, day) keep their input order
    obs = {"day": np.array([5, 2, 2, 9]), "row": np.zeros(4, int), "col": np.zeros(4, int),
           "kind": np.zeros(4, int), "value": np.zeros(4), "sigma": np.ones(4)}
    assert R.order(obs, mask).tolist() == [1, 2, 0, 3]


def test_scores_separate_the_kinds_and_drop_land():
    mask = S.region_mask(shape=(40, 50), kind="disc")
    rng = np.random.default_rng(2)
    obs = grid_obs(mask, 3000, rng)
    model = rng.random(3000) * 2.0
    model[::13] = np.nan                                  # e.g. density below minSnowD
    obs["value"][::29] = np.nan
    chi2, used = R.scores(model, obs, mask)
    wet = R.ocean(mask)[obs["row"], obs["col"]]
    assert 300 < (~wet).sum() < 2700
    with np.errstate(all="ignore"):
        r = (model - obs["value"]) / obs["sigma"]
    for k in range(KINDS):
        sel = wet & (obs["kind"] == k) & np.isfinite(r)
        assert used[k] == sel.sum() > 100
        assert chi2[k] == pytest.approx(np.sum(r[sel] ** 2), rel=1e-12, abs=0.0)
    # land observations count for nothing, whatever their model value
    land = ~wet
    model2 = model.copy()
    model2[land] = 1e6
    assert np.array_equal(R.scores(model2, obs, mask)[0], chi2)
    # a kind's sum does not depend on the other kinds' observations
    only = {k: v[obs["kind"] == VOLUME] for k, v in obs.items()}
    alone, alone_used = R.scores(model[obs["kind"] == VOLUME], only, mask)
    assert alone[VOLUME] == chi2[VOLUME] and alone_used[VOLUME] == used[VOLUME] and alone[DEPTH] == 0.0


def test_model_values_gather_the_kinds_from_the_season_arrays():
    mask = S.region_mask(shape=(12, 10), kind="disc")
    rng = np.random.default_rng(3)
    T = 5
    depths = rng.random((T, 2, 12, 10))
    dens = 200.0 + 150.0 * rng.random((T, 12, 10))
    conc = rng.random((T, 12, 10))
    obs = grid_obs(mask, 400, rng)
    obs["day"] %= T
    v = R.model_values(depths, dens, conc, obs, mask)
    d, r, c, k = obs["day"], obs["row"], obs["col"], obs["kind"]
    wet = R.ocean(mask)[r, c]
    vol = depths[d, 0, r, c] + depths[d, 1, r, c]
    assert np.isnan(v[~wet]).all()
    for kind, want in ((DEPTH, vol / conc[d, r, c]), (VOLUME, vol), (DENSITY, dens[d, r, c])):
        sel = wet & (k == kind)
        assert sel.sum() > 20 and np.array_equal(v[sel], want[sel])


# ------------------------------------------------------------------------------------------------ the drivers

DX = 100000
DAYS = [6, 9]                                        # two seasons; the stacked context is 9 days long


class EngineReached(AssertionError):
    pass


def no_engine(*a, **kw):
    raise EngineReached("an engine was created: the observation was not rejected before device work")


def driver_inputs():
    mask = S.region_mask(shape=(12, 10), kind="disc")
    rng = np.random.default_rng(4)
    seasons = []
    for s, d in enumerate(DAYS):
        wet = np.argwhere(R.ocean(mask))[rng.integers(0, R.ocean(mask).sum(), 20)]
        o = {"day": rng.integers(1, d, 20), "row": wet[:, 0], "col": wet[:, 1], "value": rng.random(20)}
        seasons.append({"forcing": S.make_season(mask, d, seed=5 + s), "ic": S.make_ic(mask, seed=5), "obs": o})
    return mask, seasons, S.ensemble_params(2, seed=6)


def call(driver, mask, seasons, params, fused):
    from nesosim_b200 import ensemble as ENS
    tup = [(s["obs"]["day"], s["obs"]["row"], s["obs"]["col"], s["obs"]["value"]) for s in seasons]
    if driver == "run_ensemble":                     # one season: the first (the shorter)
        return ENS.run_ensemble(mask, seasons[0]["forcing"], seasons[0]["ic"], params, DX, tup[0], fused=fused)
    if driver == "run_calibration":
        return ENS.run_calibration(mask, [dict(s, obs=t) for s, t in zip(seasons, tup)], params, DX, fused=fused)
    return ENS.run_calibration_scores(mask, seasons, params, DX, fused=fused, model=True)


BAD = {
    "day_past_a_shorter_season": ("day", lambda ny, nx: DAYS[0]),      # in [T_s, T): a slot of the stacked context
    "day_past_every_season": ("day", lambda ny, nx: DAYS[1]),
    "negative_day": ("day", lambda ny, nx: -1),
    "negative_row": ("row", lambda ny, nx: -1),
    "row_past_the_grid": ("row", lambda ny, nx: ny),
    "negative_col": ("col", lambda ny, nx: -1),
    "col_past_the_grid": ("col", lambda ny, nx: nx),
}
DRIVERS = ["run_ensemble", "run_calibration", "run_calibration_scores"]


@pytest.mark.parametrize("bad", sorted(BAD))
@pytest.mark.parametrize("driver", DRIVERS)
def test_drivers_reject_observations_outside_the_grid_or_the_season(driver, bad, monkeypatch):
    import nesosim_b200.engine as E
    monkeypatch.setattr(E, "SnowBudgetEngine", no_engine)
    mask, seasons, params = driver_inputs()
    field, value = BAD[bad]
    seasons[0]["obs"][field][7] = value(*mask.shape)
    for fused in (None, True, False):
        with pytest.raises(ValueError):
            call(driver, mask, seasons, params, fused)


@pytest.mark.parametrize("driver", DRIVERS)
def test_drivers_pass_observations_on_the_edges_of_the_range(driver, monkeypatch):
    """Day 0, each season's last day, the first and last row and column reach the engine (here: the stub)."""
    import nesosim_b200.engine as E
    monkeypatch.setattr(E, "SnowBudgetEngine", no_engine)
    mask, seasons, params = driver_inputs()
    ny, nx = mask.shape
    for s, d in zip(seasons, DAYS):
        s["obs"]["day"][:2] = [0, d - 1]
        s["obs"]["row"][2:4], s["obs"]["col"][2:4] = [0, ny - 1], [0, nx - 1]
    for fused in (None, True, False):
        with pytest.raises(EngineReached):
            call(driver, mask, seasons, params, fused)
