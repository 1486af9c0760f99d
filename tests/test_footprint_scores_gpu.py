"""GPU: footprint observations (nesosim_set_observations_fp + nesosim_run_season_scores_fp) -- observed means over many
cells and/or days, scored in the fused calibration call -- bit for bit against the float64 restatement of their fixed
order (oracle/footprint_scores.py) on the oracle's season arrays, on one forcing
(OBS) and on forcing sets (SETS && OBS), every build variant, cluster sizes 2..8, strip-boundary, ragged and all-ocean
masks and a dense footprint set; the exact equalities the fixed order implies; determinism, launch count and errors;
and the driver ensemble.run_calibration_scores with footprints, fused against the HBM round trip."""
import ctypes as C
import functools

import numpy as np
import pytest

from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O
from oracle import footprint_scores as F
from oracle import observation_scores as R

pytestmark = pytest.mark.gpu

DEPTH, VOLUME, DENSITY, KINDS = R.DEPTH, R.VOLUME, R.DENSITY, R.KINDS
ENV = ("NESOSIM_ENS_VARIANT", "NESOSIM_ENS_CLUSTER", "NESOSIM_ENS_CLUSTERS", "NESOSIM_ENS_ROWS", "NESOSIM_ENS_COST",
       "NESOSIM_ENS_DBG", "NESOSIM_ENS_TIMING")
VARIANTS = ["t352r3o2", "t224r4o3", "t480r2o2", "t608r2o1", "t480r2o1", "t736r2o1", "t352r6o5"]
DAYS = [10, 13, 14]
MEMBER_SET = [2, 0, 1, 1, 0, 2, 1]
SINGLE_DAYS, SINGLE_M = 13, 5
BOUNDARY = [("5", "18,36,54,72", 3), ("6", "16,30,44,60,76", 55)]
CLUSTER_MASK = {2: "arctic:20:44", 3: "arctic:20:56", 4: "arctic:20:68"}


def clear_env(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)


def oracle_params(row):
    return O.Params(windPackFactor=row[0], windPackThresh=row[1], leadLossFactor=row[2], atmLossFactor=row[3])


def make_mask(name):
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
    m[cuts[0] - 2:cuts[0] + 2] = 11
    m[cuts[1]:cuts[1] + 2] = 11
    m[cuts[2] - 2:cuts[2]] = 11
    m[:, :land_cols] = 11
    m[40:43, 60:70] = 0
    return m, 100000


def make_obs(mask, days, rng, n):
    """n point observations of all kinds, on land and ocean, with some NaN values."""
    ny, nx = mask.shape
    row, col, day = rng.integers(0, ny, n), rng.integers(0, nx, n), rng.integers(0, days, n)
    kind = rng.integers(0, KINDS, n)
    kind[(day == 0) & (kind == DENSITY)] = VOLUME
    value = np.where(kind == DENSITY, 200.0 + 150.0 * rng.random(n), 0.3 * rng.random(n))
    value[rng.random(n) < 0.05] = np.nan
    return {"day": day, "row": row, "col": col, "value": value, "kind": kind, "sigma": 10.0 ** rng.uniform(-3, 1, n)}


def cat_footprints(parts):
    out = {k: np.concatenate([p[k] for p in parts]) for k in ("kind", "value", "sigma", "day", "row", "col", "weight")}
    out["begin"] = np.concatenate([[0], np.cumsum(np.concatenate([np.diff(p["begin"]) for p in parts]))])
    return out


def regional(mask, codes, *a):
    """ENS.region_footprints over the codes of `codes` the mask has (None if it has none)."""
    from nesosim_b200 import ensemble as ENS
    codes = [k for k in codes if (R.ocean(mask) & (mask == k)).any()]
    return ENS.region_footprints(mask, codes, *a) if codes else None


def make_footprints(mask, days, rng, zero_conc, dense=False):
    """Footprints of every kind: regional means over day windows (ENS.region_footprints), random scattered footprints
    with random weights that mix land and ocean points, the zero-concentration cell-days `zero_conc` and density
    points (some below minSnowD), one of 2000 points, and one entirely on land.  dense: every ocean region x three
    windows x depth and density instead of the regional part."""
    parts = []
    if dense:
        win = [(1, days // 3), (days // 3, 2 * days // 3), (2 * days // 3, days)]
        for code in range(1, 11):
            for k in (DEPTH, DENSITY):
                parts.append(regional(mask, [code], win, k, 0.2 if k == DEPTH else 300.0, 0.05 if k == DEPTH else 30.0))
    else:
        for codes, k in (([8], DEPTH), ([1, 2, 3], VOLUME), ([8, 9], DENSITY)):
            parts.append(regional(mask, codes, [(1, days // 2), (days // 2, days)], k,
                                  rng.random(2) * (300.0 if k == DENSITY else 0.3), rng.uniform(0.01, 10.0, 2)))
    parts = [p for p in parts if p is not None]
    ny, nx = mask.shape
    zc = np.asarray(zero_conc)
    sizes = [1, 3, 31, 32, 33, 65, 2000] + list(rng.integers(1, 200, 20))
    for i, n in enumerate(sizes):
        k = i % KINDS
        d, r, c = rng.integers(1 if k == DENSITY else 0, days, n), rng.integers(0, ny, n), rng.integers(0, nx, n)
        if k == DEPTH and n >= 3:                      # a zero-concentration cell-day among the points
            d[1], r[1], c[1] = zc[i % len(zc)]
        parts.append({"kind": np.array([k]), "value": np.array([rng.random() * (300.0 if k == DENSITY else 0.3)]),
                      "sigma": np.array([rng.uniform(0.01, 10.0)]), "begin": np.array([0, n]), "day": d, "row": r,
                      "col": c, "weight": 2.0 ** rng.uniform(-4, 4, n)})
    land = np.argwhere(~R.ocean(mask))
    if len(land) >= 4:
        parts.append({"kind": np.array([DEPTH]), "value": np.array([0.1]), "sigma": np.array([1.0]), "begin": np.array([0, 4]),
                      "day": np.arange(4) % days, "row": land[:4, 0], "col": land[:4, 1], "weight": np.ones(4)})
    order = rng.permutation(len(parts))                 # kinds interleaved in input order
    return cat_footprints([parts[i] for i in order])


@functools.lru_cache(maxsize=None)
def case(mask_name, layout, dense=False, seed=0):
    mask, dx = make_mask(mask_name)
    if layout == "single":
        member_set, days = [0] * SINGLE_M, [SINGLE_DAYS]
    else:
        member_set, days = MEMBER_SET, DAYS
    rng = np.random.default_rng(seed)
    M = len(member_set)
    seasons = [S.make_season(mask, d, seed=seed + 1 + s) for s, d in enumerate(days)]
    wet = np.argwhere(R.ocean(mask))
    zero_conc = []
    for f, d in zip(seasons, days):
        z = [(int(rng.integers(1, d)),) + tuple(wet[rng.integers(len(wet))]) for _ in range(4)]
        for dd, r, c in z:
            f["conc"][dd, r, c] = 0.0
        zero_conc.append(z)
    ic = (0.02 + S.make_ic(mask, seed=seed + 5))[None] * rng.uniform(0.3, 3.0, (M, 1, 1))
    obs = [make_obs(mask, d, rng, 300 + 50 * s) for s, d in enumerate(days)]
    fps = [make_footprints(mask, d, rng, zero_conc[s], dense) for s, d in enumerate(days)]
    return {"mask": mask, "dx": dx, "layout": layout, "member_set": member_set, "days": days, "seasons": seasons,
            "params": S.ensemble_params(M, seed=seed + 6), "ic": ic, "obs": obs, "fps": fps}


def expected(c):
    """Per member: (point model, chi2, used, footprint model, fp_chi2, fp_used) of the restatement."""
    if "want" not in c:
        c["want"] = []
        for m, s in enumerate(c["member_set"]):
            f = c["seasons"][s]
            ref = O.run_season(f, c["ic"][m], c["mask"], c["dx"], oracle_params(c["params"][m]), O.Flags(atmlossInc=1))
            arrays = (ref["snowDepths"], ref["density"], f["conc"])
            model = R.model_values(*arrays, c["obs"][s], c["mask"])
            fmodel = F.footprint_values(*arrays, c["fps"][s], c["mask"])
            c["want"].append((model,) + R.scores(model, c["obs"][s], c["mask"]) + (fmodel,)
                             + F.footprint_scores(fmodel, c["fps"][s]))
    return c["want"]


def engine(c):
    from nesosim_b200.engine import SnowBudgetEngine
    T = max(c["days"])
    eng = SnowBudgetEngine(c["mask"], T, c["dx"], n_members=len(c["member_set"]), atmlossInc=1)
    if c["layout"] == "single":
        f = c["seasons"][0]
        eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
    else:
        st = {k: np.stack([np.concatenate([f[k], np.zeros((T - len(f[k]),) + f[k].shape[1:])]) for f in c["seasons"]])
              for k in ("precip", "conc", "wind", "drift")}
        eng.set_forcing_sets(st["precip"], st["conc"], st["wind"], st["drift"], c["member_set"], c["days"])
    return eng


def register(eng, c, obs=None, fps=None):
    obs, fps = obs or c["obs"], fps or c["fps"]
    sets = c["layout"] == "sets"
    cat = {k: np.concatenate([o[k] for o in obs]) for k in obs[0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(obs)]) if sets else None
    ftag = np.concatenate([np.full(len(f["value"]), i, dtype=np.int32) for i, f in enumerate(fps)]) if sets else None
    eng.set_observations_fp(cat, cat_footprints(fps), obs_set=tag, fp_set=ftag)


def run(eng, c, model=True):
    return tuple(None if t is None else t.cpu().numpy() for t in eng.run_season_scores_fp(c["params"], c["ic"], model=model))


def fused(c):
    eng = engine(c)
    register(eng, c)
    got = run(eng, c)
    eng.close()
    return got


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def check(c, got):
    chi2, used, model, fchi2, fused_, fmodel = got
    for m, s in enumerate(c["member_set"]):
        wm, wc, wu, wfm, wfc, wfu = expected(c)[m]
        n, g = len(c["obs"][s]["day"]), len(c["fps"][s]["value"])
        assert same(model[m, :n], wm) and np.isnan(model[m, n:]).all(), m
        assert np.array_equal(used[m], wu) and np.array_equal(chi2[m], wc), (m, chi2[m], wc)
        bad = np.flatnonzero(~((fmodel[m, :g] == wfm) | (np.isnan(fmodel[m, :g]) & np.isnan(wfm))))
        assert not len(bad), ("footprint model", m, bad[:5], fmodel[m, bad[:5]], wfm[bad[:5]])
        assert np.isnan(fmodel[m, g:]).all(), m
        assert np.array_equal(fused_[m], wfu) and np.array_equal(fchi2[m], wfc), (m, fchi2[m], wfc, fused_[m], wfu)
        assert np.isnan(fmodel[m, :g]).any() or R.ocean(c["mask"]).all()     # the all-land footprint at least
    assert (fused_ > 0).all() and (used > 0).all()


@pytest.mark.parametrize("layout", ["single", "sets"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_every_variant_bit_for_bit(cuda, variant, layout, monkeypatch):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_ENS_VARIANT", variant)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTERS", str(1 + (VARIANTS.index(variant) + (layout == "sets")) % 2))
    c = case("arctic", layout)
    check(c, fused(c))


@pytest.mark.parametrize("cluster", range(2, 9))
def test_every_cluster_size(cuda, cluster, monkeypatch):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTER", str(cluster))
    monkeypatch.setenv("NESOSIM_ENS_CLUSTERS", "2")
    c = case(CLUSTER_MASK.get(cluster, "arctic"), "sets" if cluster % 2 else "single")
    check(c, fused(c))


@pytest.mark.parametrize("cluster,rows,land_cols", BOUNDARY)
def test_strip_boundary_masks(cuda, cluster, rows, land_cols, monkeypatch):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTERS", "2")
    monkeypatch.setenv("NESOSIM_ENS_CLUSTER", cluster)
    monkeypatch.setenv("NESOSIM_ENS_ROWS", rows)
    c = case("boundary:%s:%d" % (rows, land_cols), "sets")
    check(c, fused(c))


@pytest.mark.parametrize("mask_name,layout", [("disc:45:70", "sets"), ("disc:94:33", "single"), ("disc:9:96", "sets"),
                                              ("ocean", "single")])
def test_ragged_and_all_ocean_grids(cuda, mask_name, layout, monkeypatch):
    clear_env(monkeypatch)
    c = case(mask_name, layout)
    check(c, fused(c))


@pytest.mark.parametrize("layout", ["single", "sets"])
def test_dense_footprints(cuda, layout, monkeypatch):
    """Every ocean region x three windows x depth and density: nearly every ocean cell-day is a sample slot."""
    clear_env(monkeypatch)
    c = case("arctic", layout, dense=True)
    assert max(len(f["day"]) for f in c["fps"]) > 50000
    check(c, fused(c))


def test_points_unaffected_determinism_and_launches(cuda, monkeypatch):
    """The point outputs with footprints registered equal registering the points alone, bit for bit; two runs are
    bit-identical; the call takes five launches (pre-pass 2, season kernel, footprint means, epilogue)."""
    clear_env(monkeypatch)
    c = case("arctic", "sets")
    eng = engine(c)
    cat = {k: np.concatenate([o[k] for o in c["obs"]]) for k in c["obs"][0]}
    tag = np.concatenate([np.full(len(o["day"]), i, dtype=np.int32) for i, o in enumerate(c["obs"])])
    eng.set_observations_ex(cat["day"], cat["row"], cat["col"], cat["value"], cat["kind"], cat["sigma"], obs_set=tag)
    alone = tuple(t.cpu().numpy() for t in eng.run_season_scores(c["params"], c["ic"], model=True))
    register(eng, c)
    assert eng.footprint_row_length() == max(len(f["value"]) for f in c["fps"])
    l0 = eng.launch_count()
    a = run(eng, c)
    assert eng.launch_count() - l0 == 5
    b = run(eng, c)
    eng.close()
    assert all(same(x, y) for x, y in zip(a, b))
    assert all(same(x, y) for x, y in zip(a[:3], alone))


def test_exact_equalities(cuda, monkeypatch):
    """One-point weight-1 footprints given in (cell, day) order score exactly like the same point observations; weights
    scaled by 2^k give identical means; an all-land footprint is NaN and not counted."""
    clear_env(monkeypatch)
    c = case("arctic", "single")
    o = c["obs"][0]
    idx = R.order(o, c["mask"])                                         # ocean points in (cell, day) order
    o = {k: v[idx] for k, v in o.items()}
    n = len(o["day"])
    one = {"kind": o["kind"], "value": o["value"], "sigma": o["sigma"], "begin": np.arange(n + 1), "day": o["day"],
           "row": o["row"], "col": o["col"], "weight": np.ones(n)}
    eng = engine(c)
    register(eng, c, obs=[o], fps=[one])
    chi2, used, model, fchi2, fused_, fmodel = run(eng, c)
    assert np.array_equal(chi2, fchi2) and np.array_equal(used, fused_)
    fin = np.isfinite(model)                             # a non-finite point value (inf at zero concentration) is skipped
    assert np.array_equal(model[fin], fmodel[fin]) and np.isnan(fmodel[~fin]).all() and (~fin).any()
    fp = c["fps"][0]
    scaled = dict(fp, weight=fp["weight"] * 2.0 ** np.repeat(np.arange(len(fp["value"])) % 7 - 3, np.diff(fp["begin"])))
    register(eng, c, fps=[fp])
    base = run(eng, c)
    register(eng, c, fps=[scaled])
    got = run(eng, c)
    assert all(same(x, y) for x, y in zip(base, got))
    land = np.argwhere(~R.ocean(c["mask"]))[:5]
    only = {"kind": np.array([DEPTH]), "value": np.array([0.1]), "sigma": np.array([1.0]), "begin": np.array([0, 5]),
            "day": np.arange(5), "row": land[:, 0], "col": land[:, 1], "weight": np.ones(5)}
    register(eng, c, fps=[only])
    _, _, _, fchi2, fused_, fmodel = run(eng, c)
    eng.close()
    assert np.isnan(fmodel).all() and (fused_ == 0).all() and (fchi2 == 0).all()


def test_errors_keep_the_registration(cuda, monkeypatch):
    from nesosim_b200 import _lib
    clear_env(monkeypatch)
    c = case("arctic", "sets")
    eng = engine(c)
    register(eng, c)
    want = run(eng, c)

    def code(fn, *a, **kw):
        with pytest.raises(_lib.NesosimError) as e:
            fn(*a, **kw)
        return e.value.code

    def bad(**over):
        fps = [dict(f) for f in c["fps"]]
        for k, v in over.items():
            fps[1][k] = v(fps[1][k].copy())
        return code(register, eng, c, None, fps)

    def at(i, v):
        def f(a):
            a[i] = v
            return a
        return f

    fp = c["fps"][1]
    assert bad(begin=at(0, 1)) == _lib.ERR_ARG                               # fp_begin[0] != 0
    assert bad(begin=at(3, fp["begin"][2])) == _lib.ERR_ARG                  # an empty footprint
    for w in (0.0, -1.0, np.nan, np.inf):
        assert bad(weight=at(5, w)) == _lib.ERR_ARG
    for k in (3, -1):
        assert bad(kind=at(0, k)) == _lib.ERR_ARG
    for s in (0.0, np.nan):
        assert bad(sigma=at(0, s)) == _lib.ERR_ARG
    assert bad(row=at(7, -1)) == _lib.ERR_ARG and bad(col=at(7, 90)) == _lib.ERR_ARG
    assert bad(day=at(7, DAYS[1])) == _lib.ERR_ARG                           # outside its set's season
    g = int(np.flatnonzero(fp["kind"] == DENSITY)[0])
    assert bad(day=at(int(fp["begin"][g]), 0)) == _lib.ERR_ARG              # density point on day 0
    cat = cat_footprints(c["fps"])
    ftag = np.concatenate([np.full(len(f["value"]), i, dtype=np.int32) for i, f in enumerate(c["fps"])])
    ftag[0] = 3
    assert code(eng.set_observations_fp, None, cat, fp_set=ftag) == _lib.ERR_ARG    # set tag
    # a short footprint row
    torch = pytest.importorskip("torch")
    M, K, n = len(c["member_set"]), KINDS, eng.footprint_row_length()
    t = [torch.empty(M, K, dtype=torch.float64, device="cuda") for _ in range(2)]
    fm = torch.empty(M, n, dtype=torch.float64, device="cuda")
    rc = eng.lib.nesosim_run_season_scores_fp(eng.handle, _lib.member_params_array(c["params"]), eng._dev(c["ic"]).data_ptr(),
                                              1, t[0].data_ptr(), None, None, 0, t[1].data_ptr(), None, fm.data_ptr(),
                                              n - 1, eng._stream())
    assert rc == _lib.ERR_ARG
    row_len = C.c_int64(0)
    assert eng.lib.nesosim_footprint_row_length(None, C.byref(row_len)) == _lib.ERR_ARG
    # the registration in force is unchanged; the point-only calls refuse to drop the footprints
    assert all(same(x, y) for x, y in zip(want, run(eng, c)))
    assert code(eng.run_season_scores, c["params"], c["ic"]) == _lib.ERR_STATE
    assert code(eng.run_season_misfit, c["params"], c["ic"]) == _lib.ERR_STATE
    # the forcing registered again with another layout
    T = max(DAYS)
    f = {k: np.stack([np.concatenate([x[k], np.zeros((T - len(x[k]),) + x[k].shape[1:])]) for x in c["seasons"]])
         for k in ("precip", "conc", "wind", "drift")}
    eng.set_forcing_sets(f["precip"], f["conc"], f["wind"], f["drift"], c["member_set"], [10, 13, 13])
    assert code(eng.run_season_scores_fp, c["params"], c["ic"]) == _lib.ERR_STATE
    eng.close()


def driver_seasons(mask, seed, days=(14, 17, 20)):
    rng = np.random.default_rng(seed)
    out = []
    for s, d in enumerate(days):
        fp = cat_footprints([regional(mask, [8], [(1, d // 2), (d // 2, d)], DEPTH, [0.2, 0.25], 0.05),
                             regional(mask, [8, 9], [(1, d)], DENSITY, 300.0, 30.0)])
        season = {"forcing": S.make_season(mask, d, seed=seed + s), "ic": S.make_ic(mask, seed=seed + s) * (1 + s),
                  "obs": make_obs(mask, d, rng, 200)}
        if s != 1:
            season["footprints"] = fp
        out.append(season)
    return out


def test_driver_fused_agrees_with_the_hbm_round_trip(cuda, monkeypatch):
    from nesosim_b200 import ensemble as ENS
    clear_env(monkeypatch)
    mask = S.region_mask(dx=100000)
    seasons = driver_seasons(mask, 280)
    params = S.ensemble_params(3, seed=281)
    a = ENS.run_calibration_scores(mask, seasons, params, 100000, atmlossInc=1, model=True)
    b = ENS.run_calibration_scores(mask, seasons, params, 100000, atmlossInc=1, model=True, fused=False)
    assert a["fp_chi2"].shape == (3, 3, KINDS) and np.array_equal(a["fp_used"], b["fp_used"])
    assert np.allclose(a["fp_chi2"], b["fp_chi2"], rtol=1e-12, atol=0.0)
    assert np.array_equal(a["used"], b["used"]) and np.allclose(a["chi2"], b["chi2"], rtol=1e-12, atol=0.0)
    assert [m.shape for m in a["fp_model"]] == [(3, 3), (3, 0), (3, 3)]
    for s in range(3):
        assert np.allclose(a["fp_model"][s], b["fp_model"][s], rtol=1e-12, atol=0.0)
    assert (a["fp_used"][:, [0, 2]].sum(axis=2) == 3).all() and (a["fp_used"][:, 1] == 0).all()
    plain = ENS.run_calibration_scores(mask, [dict(s, footprints=None) for s in seasons], params, 100000, atmlossInc=1)
    assert "fp_chi2" not in plain and np.array_equal(plain["chi2"], a["chi2"])


def test_driver_falls_back_on_a_wide_grid(cuda, monkeypatch):
    from nesosim_b200 import _lib
    from nesosim_b200 import ensemble as ENS
    clear_env(monkeypatch)
    mask = S.region_mask(shape=(40, 130), kind="disc")
    seasons = driver_seasons(mask, 290, days=(8, 9, 10))
    seasons[1]["footprints"] = regional(mask, range(1, 11), [(1, 5)], DEPTH, 0.2)
    params = S.ensemble_params(2, seed=291)
    with pytest.raises(_lib.NesosimError):
        ENS.run_calibration_scores(mask, seasons, params, 50000, atmlossInc=1, fused=True)
    res = ENS.run_calibration_scores(mask, seasons, params, 50000, atmlossInc=1)
    for p in range(2):
        for s in range(3):
            f = seasons[s]["forcing"]
            fps = ENS.normalize_footprints(seasons[s]["footprints"])
            ref = O.run_season(f, seasons[s]["ic"], mask, 50000, oracle_params(params[p]), O.Flags(atmlossInc=1))
            wm = F.footprint_values(ref["snowDepths"], ref["density"], f["conc"], fps, mask)
            wc, wu = F.footprint_scores(wm, fps)
            assert np.array_equal(res["fp_used"][p, s], wu) and wu.sum() > 0
            assert np.allclose(res["fp_chi2"][p, s], wc, rtol=1e-12, atol=0.0), (p, s)
            assert np.allclose(res["fp_model"][s][p], wm, rtol=1e-12, atol=0.0, equal_nan=True)
