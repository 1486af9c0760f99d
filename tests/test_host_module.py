"""The drop-in host module ``nesosim_b200/NESOSIM.py``: forcing reader / season stager against what the reference's own
``loadData`` returned on the same files (CPU, stored in ``tests/golden/reference_contracts.npz``), the stager's
self-contained semantics (CPU) and ``main`` / ``calcBudget`` end to end on the GPU with the reference's out-of-scope
helpers (grid, mask, NetCDF writers, plots) replaced by recording fakes."""
import datetime
import os
import sys
import types

import numpy as np
import numpy.ma as ma
import pytest

import golden_util
from nesosim_b200 import NESOSIM as N
from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O

NY, NX = 12, 10
DXSTR = "100km"
EXTRA = "v11"


def write_forcing_tree(root, years_days, seed=0, with_temp_days=(), skip_drift_days=(), masked_drift_days=(),
                       bad_conc=True):
    """Forcing files in the layout the reference's gridding scripts write (ndarray.dump pickles)."""
    rng = np.random.default_rng(seed)
    base = os.path.join(root, DXSTR)
    made = {}
    for (year, day) in years_days:
        d = "%03d" % day
        P = rng.gamma(0.5, 2.0, (NY, NX))
        W = rng.gamma(4.0, 1.5, (NY, NX))
        C = np.clip(rng.random((NY, NX)), 0, 1)
        if bad_conc:
            C[0, 0] = np.nan
            C[1, 1] = np.inf
        U = 0.1 * rng.standard_normal((2, NY, NX))
        for sub, name, arr in (("Precip/ERA5/%d" % year, "ERA5sf%s-%d_d%s%s" % (DXSTR, year, d, EXTRA), P),
                               ("Winds/ERA5/%d" % year, "ERA5winds%s-%d_d%s%s" % (DXSTR, year, d, EXTRA), W),
                               ("IceConc/CDR/%d" % year, "iceConcG_CDR%s-%d_d%s%s" % (DXSTR, year, d, EXTRA), C)):
            os.makedirs(os.path.join(base, sub), exist_ok=True)
            arr.dump(os.path.join(base, sub, name))
        if (year, day) not in skip_drift_days:
            os.makedirs(os.path.join(base, "IceDrift/OSISAF/%d" % year), exist_ok=True)
            drift = U
            if (year, day) in masked_drift_days:
                drift = ma.masked_array(U, mask=U > 0.1)
            drift.dump(os.path.join(base, "IceDrift/OSISAF/%d" % year, "OSISAF_driftG%s-%d_d%s%s" % (DXSTR, year, d, EXTRA)))
        if (year, day) in with_temp_days:
            os.makedirs(os.path.join(base, "Temp/ERA5/t2m/%d" % year), exist_ok=True)
            (250 + rng.random((NY, NX))).dump(os.path.join(base, "Temp/ERA5/t2m/%d" % year, "t2m%s-%d_d%s%s" % (DXSTR, year, d, EXTRA)))
        made[(year, day)] = (C, P, U, W)
    return base + "/", made


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


@pytest.fixture
def quiet():
    N.VERBOSE = False
    yield
    N.VERBOSE = True


# ------------------------------------------------------------------------------------------ CPU, anywhere

def test_gen_empty_arrays_contract():
    arrs = N.genEmptyArrays(7, 5, 4)
    assert len(arrs) == 15
    for i, a in enumerate(arrs):
        assert a.dtype == np.float64 and not a.any()
        assert a.shape == ((7, 2, 5, 4) if i == 4 else (7, 5, 4))


def test_doy_to_month_keeps_the_reference_off_by_one():
    # the model's day counter is 0-based but the helper treats it as 1-based (NESOSIM.py:479):
    assert N.doyToMonth(0, 2019) == 12          # Jan 1 -> December of the previous year
    assert N.doyToMonth(31, 2019) == 1          # Feb 1 -> January
    assert N.doyToMonth(32, 2019) == 2
    assert N.doyToMonth(243, 2018) == 8         # Sep 1 (0-based 243) -> August


def test_load_data_semantics(tmp_path, quiet):
    days = [(2018, 100), (2018, 101), (2018, 364)]
    root, made = write_forcing_tree(str(tmp_path), days, with_temp_days=[(2018, 100)], skip_drift_days=[(2018, 101)],
                                    masked_drift_days=[(2018, 100)])
    N.forcingPath = root
    conc, precip, drift, wind, temp = N.loadData(2018, 100, "ERA5", "ERA5", "CDR", "OSISAF", DXSTR, EXTRA)
    C, P, U, W = made[(2018, 100)]
    assert conc[0, 0] == 0 and conc[1, 1] == 0 and same(conc[2:], C[2:])          # non-finite concentration -> 0
    assert same(precip, P) and same(wind, W)
    assert np.isnan(drift[U > 0.1]).all() and same(drift[U <= 0.1], U[U <= 0.1])   # masked drift -> NaN
    assert np.isfinite(temp).all()
    conc, precip, drift, wind, temp = N.loadData(2018, 101, "ERA5", "ERA5", "CDR", "OSISAF", DXSTR, EXTRA)
    assert drift.shape == (2, NY, NX) and np.isnan(drift).all() and np.isnan(temp).all()   # missing drift / temp
    with pytest.raises(SystemExit):
        N.loadData(2018, 102, "ERA5", "ERA5", "CDR", "OSISAF", DXSTR, EXTRA)               # missing snowfall ends the run


def test_stage_season_year_wrap_scaling_and_last_slot(tmp_path, quiet):
    start, ndays, ny1 = 362, 6, 365
    days = [(2018, 362), (2018, 363), (2018, 364), (2019, 0), (2019, 1), (2019, 2)]
    root, made = write_forcing_tree(str(tmp_path), days, seed=4, bad_conc=False)
    N.forcingPath = root
    sf = 1.0 + 0.1 * np.arange(12)[:, None, None] * np.ones((12, NY, NX))
    st = N.stage_season(2018, 2019, start, ndays, ny1, "ERA5", "ERA5", "CDR", "OSISAF", DXSTR, EXTRA, scale_factors=sf)
    for x, key in enumerate(days):
        C, P, U, W = made[key]
        assert same(st["conc"][x], C) and same(st["wind"][x], W)
        if x < ndays - 1:
            month = N.doyToMonth(key[1], key[0])
            assert same(st["precip"][x], P * sf[month - 1]) and same(st["drift"][x], U)
        else:                       # the slot after the last step: unscaled forcing copies, no drift
            assert same(st["precip"][x], P) and np.isnan(st["drift"][x]).all()
    assert st["rho_clim"] is None
    # Jan 1 (day 0) is scaled with December's factor -- the reference's off-by-one
    assert same(st["precip"][3], made[(2019, 0)][1] * sf[11])


# ------------------------------------------------------------------------------------------ CPU, against the reference
# The reference's own functions, run verbatim on the inputs below (oracle/ref_loader.py), returned the arrays stored in
# tests/golden/reference_contracts.npz (tests/golden/make_reference_contracts.py says how they were recorded).

CONTRACTS = "reference_contracts.npz"
LOAD_DATA_DAYS = (10, 11, 12, 365)
LOAD_DATA_NAMES = ("conc", "precip", "drift", "wind", "temp")
HELPER_YEARS = (2018, 2019, 2020)
HELPER_DAYS = (0, 1, 30, 31, 58, 59, 60, 243, 334, 364, 365)


def load_data_tree(root):
    """The forcing tree the reader is compared on: masked drift, a temperature file, a missing drift file, and the
    day-365 snowfall fallback, which the reference looks up under Precip/<var>/sf/<year>/ (NESOSIM.py:395)."""
    days = [(2018, d) for d in (10, 11, 12, 364)]
    root, _ = write_forcing_tree(root, days, seed=2, with_temp_days=[(2018, 11)], skip_drift_days=[(2018, 12)],
                                 masked_drift_days=[(2018, 10)])
    src = os.path.join(root, "Precip/ERA5/2018", "ERA5sf%s-2018_d364%s" % (DXSTR, EXTRA))
    os.makedirs(os.path.join(root, "Precip/ERA5/sf/2018"))
    np.load(src, allow_pickle=True).dump(os.path.join(root, "Precip/ERA5/sf/2018", os.path.basename(src)))
    return root


def load_data_outputs(root):
    N.forcingPath = root
    out = {}
    for day in LOAD_DATA_DAYS:
        got = N.loadData(2018, day, "ERA5", "ERA5", "CDR", "OSISAF", DXSTR, EXTRA)
        for g, name in zip(got, LOAD_DATA_NAMES):
            out["load_data__%s__%d" % (name, day)] = np.asarray(g)
    return out


def helper_outputs():
    out = {"helpers__doyToMonth": np.array([[N.doyToMonth(day, year) for day in HELPER_DAYS] for year in HELPER_YEARS]),
           "helpers__applyScaling": N.applyScaling(np.arange(6.).reshape(2, 3), 1.5)}
    for i, a in enumerate(N.genEmptyArrays(4, 3, 2)):
        out["helpers__genEmptyArrays__%d" % i] = a
    return out


def test_load_data_matches_reference(tmp_path, quiet, capsys):
    exp = golden_util.load(CONTRACTS)
    got = load_data_outputs(load_data_tree(str(tmp_path)))
    assert len(got) == len(LOAD_DATA_DAYS) * len(LOAD_DATA_NAMES)
    for key, g in got.items():
        assert same(g, exp[key]), key
    capsys.readouterr()


def test_helpers_match_reference():
    exp = golden_util.load(CONTRACTS)
    for key, g in helper_outputs().items():
        assert same(g, exp[key]), key
        assert np.asarray(g).dtype == exp[key].dtype, key


# ------------------------------------------------------------------------------------------ GPU

class FakeUtils(types.ModuleType):
    """Stands in for the reference's ``utils`` (pyproj / xarray / netCDF4 / cartopy are out of scope and absent):
    a tiny square grid whose region mask file IS the model grid, the reference's calendar rule, recording writers."""

    def __init__(self, mask):
        super().__init__("utils")
        self.mask = mask
        self.raw = None
        self.final = None
        self.plots = 0

    def create_grid(self, dxRes=50000):
        ny, nx = self.mask.shape
        y, x = np.mgrid[0:ny, 0:nx].astype(float)
        return x * dxRes, y * dxRes, y, x, "proj"

    def get_region_mask_pyproj(self, anc, proj, xypts_return=0):
        ny, nx = self.mask.shape
        y, x = np.mgrid[0:ny, 0:nx].astype(float)
        return self.mask.astype(np.uint8), x * 100000., y * 100000., x, y      # five values, like utils.py:1378

    def getDays(self, year1, month1, day1, year2, month2, day2):
        leap = [1976, 1980, 1984, 1988, 1992, 1996, 2000, 2004, 2008, 2012, 2016, 2020]
        d1 = datetime.datetime(year1, month1 + 1, day1 + 1)
        d2 = datetime.datetime(year2, month2 + 1, day2 + 1)
        return ((d1 - datetime.datetime(year1, 1, 1)).days, (d2 - d1).days + 1, 366 if year1 in leap else 365,
                d1.strftime('%d%m%Y') + '-' + d2.strftime('%d%m%Y'))

    def OutputSnowModelRaw(self, savePath, saveStr, *arrays):
        self.raw = (savePath, saveStr, [np.array(a) for a in arrays])

    def OutputSnowModelFinal(self, savePath, saveStr, lons, lats, xpts, ypts, snowVol, snowDepth, density, conc, precip, wind,
                             temp, dates):
        self.final = dict(savePath=savePath, saveStr=saveStr, snowVol=np.array(snowVol), snowDepth=np.array(snowDepth),
                          density=np.array(density), dates=list(dates), temp=np.array(temp))

    def plot_budgets_cartopy(self, *a, **k):
        self.plots += 1

    def plot_gridded_cartopy(self, *a, **k):
        self.plots += 1


@pytest.mark.gpu
def test_main_is_a_drop_in_for_the_reference_driver(cuda, tmp_path, quiet, monkeypatch):
    mask = S.region_mask(shape=(NY, NX), kind="disc")
    fake = FakeUtils(mask)
    monkeypatch.setitem(sys.modules, "utils", fake)
    # 2018-12-28 .. 2019-01-03 (month/day are 0-based like the reference's run scripts): 7 days, 6 steps, year wrap
    days = [(2018, 361), (2018, 362), (2018, 363), (2018, 364), (2019, 0), (2019, 1), (2019, 2), (2019, 3)]
    root, made = write_forcing_tree(str(tmp_path / "forcing"), days, seed=7, skip_drift_days=[(2018, 363)])
    ic = S.make_ic(mask, seed=7) * 3
    os.makedirs(os.path.join(root, "InitialConditions/ERA5"))
    ic.dump(os.path.join(root, "InitialConditions/ERA5", "ICsnow%s-2018%s" % (DXSTR, EXTRA)))
    out_root = str(tmp_path / "out") + "/"
    fig_root = str(tmp_path / "fig") + "/"
    ret = N.main(2018, 11, 27, 2019, 0, 2, outPathT=out_root, forcingPathT=str(tmp_path / "forcing") + "/",
                 anc_data_pathT="unused/", figPathT=fig_root, precipVar="ERA5", windVar="ERA5", driftVar="OSISAF",
                 concVar="CDR", icVar="ERA5", densityTypeT="variable", extraStr=EXTRA, outStr="test", IC=2,
                 windPackFactorT=5.8e-7, windPackThreshT=5, leadLossFactorT=2.9e-7, atmLossFactorT=2.2e-8,
                 dynamicsInc=1, leadlossInc=1, windpackInc=1, atmlossInc=1, saveData=1, plotBudgets=1, plotdaily=0,
                 dx=100000, scaleCS=False)
    assert ret is None and fake.plots == 1
    savePath, saveStr, arrays = fake.raw
    tag = "ERA5sfERA5windsOSISAFdriftsCDRsicrhovariable_IC2_DYN1_WP1_LL1_AL1_WPF5.8e-07_WPT5_LLF2.9e-07-100kmv11test"
    assert savePath == out_root + DXSTR + "//" + tag and saveStr == tag + "-28122018-03012019"
    assert os.path.isdir(savePath + "/budgets/") and os.path.isdir(savePath + "/final/")
    assert os.path.isdir(fig_root + "/Diagnostic/" + DXSTR + "/" + tag + "/daily_snow_depths/")

    # the same season through the oracle on the same staged forcing
    N.forcingPath = root
    st = N.stage_season(2018, 2019, 361, 7, 365, "ERA5", "ERA5", "CDR", "OSISAF", DXSTR, EXTRA)
    p = O.Params(windPackFactor=5.8e-7, windPackThresh=5, leadLossFactor=2.9e-7, atmLossFactor=2.2e-8)
    ref = O.run_season(st, ic, mask, 100000, p, O.Flags(atmlossInc=1))
    names = ("snowDepths", "density", "precipDays", "iceConcDays", "windDays", "snowAcc", "snowOcean", "snowAdv",
             "snowDiv", "snowLead", "snowAtm", "snowWindPack")       # argument order of OutputSnowModelRaw (utils.py:43)
    staged_names = {"precipDays": "precip", "iceConcDays": "conc", "windDays": "wind"}
    for name, got in zip(names, arrays):
        exp = st[staged_names[name]] if name in staged_names else ref[name]
        assert same(got, exp), name
    assert np.isnan(st["drift"][2]).all()                            # the missing drift file was an all-NaN day
    with np.errstate(all="ignore"):
        vol = ref["snowDepths"][:, 0] + ref["snowDepths"][:, 1]
        assert same(fake.final["snowVol"], vol) and same(fake.final["snowDepth"], vol / st["conc"])
    assert fake.final["dates"][0] == 20181228 and fake.final["dates"][-1] == 20190103 and len(fake.final["dates"]) == 7
    assert fake.final["saveStr"] == "NESOSIMv11_28122018-03012019"


@pytest.mark.gpu
def test_calc_budget_shim_has_the_reference_in_place_contract(cuda, quiet):
    mask = S.region_mask(shape=(NY, NX), kind="disc")
    T = 5
    forcing = S.make_season(mask, T, seed=9)
    ic = S.make_ic(mask, seed=9)
    p = O.Params(windPackFactor=5.8e-7, windPackThresh=5., leadLossFactor=1.45e-7, atmLossFactor=2.2e-8)
    ref = O.run_season(forcing, ic, mask, 50000, p, O.Flags(atmlossInc=1))
    N.windPackFactor, N.windPackThresh, N.leadLossFactor, N.atmLossFactor = 5.8e-7, 5., 1.45e-7, 2.2e-8
    (precipDays, iceConcDays, windDays, tempDays, snowDepths, density, snowDiv, snowAdv, snowAcc, snowOcean, snowWindPack,
     snowWindPackLoss, snowWindPackGain, snowLead, snowAtm) = N.genEmptyArrays(T, NY, NX)
    half = O.initial_depths(ic, forcing["conc"][0], p)
    snowDepths[0, 0] = half
    snowDepths[0, 1] = half
    temp = np.full((NY, NX), np.nan)
    for x in range(T - 1):
        N.calcBudget(None, None, snowDepths, forcing["conc"][x], forcing["precip"][x], forcing["drift"][x], forcing["wind"][x],
                     temp, density, precipDays, iceConcDays, windDays, tempDays, snowAcc, snowOcean, snowAdv, snowDiv,
                     snowLead, snowAtm, snowWindPackLoss, snowWindPackGain, snowWindPack, mask, 50000, x, 1 + x,
                     densityType='variable', dynamicsInc=1, leadlossInc=1, windpackInc=1, atmlossInc=1)
    got = dict(snowDepths=snowDepths, density=density, snowDiv=snowDiv, snowAdv=snowAdv, snowAcc=snowAcc,
               snowOcean=snowOcean, snowWindPack=snowWindPack, snowWindPackLoss=snowWindPackLoss,
               snowWindPackGain=snowWindPackGain, snowLead=snowLead, snowAtm=snowAtm)
    for name, arr in got.items():
        assert same(arr, ref[name]), name
    assert same(precipDays[:T - 1], forcing["precip"][:T - 1]) and not precipDays[T - 1].any()
    assert np.isnan(tempDays[:T - 1]).all()


def drift_regridder_outputs():
    """`drift_smoothing.int_smooth_drifts_v2/v3` (SURVEY 8f N4; utils.py:259-338 in the reference) on scattered source
    points with NaN drift and a model grid reaching outside their hull (NaN after interpolation -> the NaN-interpolating
    branch of the convolution and the final mask), both kernel widths the reference uses; astropy's pair is the
    restatement (oracle/astropy_restated.py), as it was for the reference.  Masked results as (filled with -9, mask)."""
    import numpy.ma as ma
    from scipy.spatial import Delaunay
    from nesosim_b200 import drift_smoothing as D
    from oracle import astropy_restated as ar

    def cpu_smoother(gx, gy, sigma_factor=1, x_size_val=3):
        k = ar.gaussian2d_kernel(x_stddev=sigma_factor, y_stddev=sigma_factor, theta=0.0, x_size=x_size_val, y_size=x_size_val)
        out = ma.masked_all((2,) + gx.shape)
        for i, c in enumerate((gx, gy)):
            out[i] = ma.masked_where(np.isnan(c), ar.convolve_fill0(c, k))
        return out

    rng = np.random.default_rng(11)
    jj, ii = np.meshgrid(np.arange(14.0), np.arange(12.0))
    xF = ii * 9.0 + rng.normal(0, 1.0, ii.shape) + 5.0          # scattered (jittered) source points
    yF = jj * 8.0 + rng.normal(0, 1.0, jj.shape) + 4.0
    latsF = 60.0 + 0.2 * ii
    drift = np.stack([np.sin(xF / 20.0) + 0.1 * rng.normal(size=xF.shape), np.cos(yF / 15.0) + 0.1 * rng.normal(size=xF.shape)])
    drift[:, 4:6, 5:8] = np.nan                                 # a data gap
    drift[1, 9, 2] = np.nan
    gj, gi = np.meshgrid(np.linspace(-5.0, 118.0, 24), np.linspace(-3.0, 112.0, 20))
    xG, yG = gi, gj
    tri = Delaunay(np.column_stack([xF.ravel(), yF.ravel()]))
    out = {}
    for sigma in (0.5, 1):
        for name, args in (("int_smooth_drifts_v2", ()), ("int_smooth_drifts_v3", (tri,))):
            got = getattr(D, name)(*args, xG, yG, xF, yF, latsF, drift, sigma_factor=sigma, smoother=cpu_smoother)
            key = "drift__%s__%s" % (name, sigma)
            out[key + "__filled"] = got.filled(-9.0)
            out[key + "__mask"] = ma.getmaskarray(got)
    return out


def test_drift_regridders_match_reference():
    exp = golden_util.load(CONTRACTS)
    got = drift_regridder_outputs()
    assert len(got) == 8
    for key, g in got.items():
        assert g.shape == exp[key].shape == (2, 20, 24), key
        assert np.array_equal(g, exp[key]), key
        if key.endswith("__mask"):
            assert exp[key].any() and not exp[key].all()


class _StandInOps:
    """CPU stand-in for the native per-function operators of `nesosim_b200.engine` (same signatures, checked below),
    backed by the oracle: lets the plumbing of the reference-named wrappers in `nesosim_b200.NESOSIM` be tested where
    there is no GPU.  The native operators themselves are tested on the GPU (`tests/test_gpu_parity.py::test_op_*`)."""

    @staticmethod
    def _p(params, deltaT, rhoFresh, rhoOld, minSnowD=0.02):
        from oracle import nesosim_oracle as O
        wpf, wpt, llf, alf = params[0]
        return O.Params(windPackFactor=wpf, windPackThresh=wpt, leadLossFactor=llf, atmLossFactor=alf, deltaT=deltaT,
                        snowDensityFresh=rhoFresh, snowDensityOld=rhoOld, minSnowD=minSnowD)

    @staticmethod
    def op_wind_terms(h0, wind, conc, params, deltaT=86400., rhoFresh=200., rhoOld=350., device=0):
        from oracle import nesosim_oracle as O
        p = _StandInOps._p(params, deltaT, rhoFresh, rhoOld)
        h0, wind, conc = (np.asarray(v, dtype=np.float64) for v in (h0, wind, conc))
        with np.errstate(all="ignore"):
            return [O.lead_loss(h0, wind, conc, p), O.atm_loss(h0, wind, p)] + list(O.wind_packing(wind, h0, p))

    @staticmethod
    def op_dynamics(drift, depths, dx, deltaT=86400., device=0):
        from oracle import nesosim_oracle as O
        return O.calc_dynamics(np.asarray(drift, dtype=np.float64), np.asarray(depths, dtype=np.float64), dx,
                               _StandInOps._p([[0, 0, 0, 0]], deltaT, 200., 350.))

    @staticmethod
    def op_fill_zero(arr, device=0):
        from oracle import nesosim_oracle as O
        a = np.array(arr, dtype=np.float64)
        O.fill_mask_nan_zero(a)
        return a

    @staticmethod
    def op_fill_nan_no_negative(arr, mask, negative_to_zero=True, device=0):
        from oracle import nesosim_oracle as O
        a = np.array(arr, dtype=np.float64)
        O.fill_nan_no_negative(a, np.asarray(mask), negative_to_zero)
        return a

    @staticmethod
    def op_density(depths, mask, rhoFresh=200., rhoOld=350., minSnowD=0.02, device=0):
        from oracle import nesosim_oracle as O
        return O.density_calc(np.asarray(depths, dtype=np.float64), None, np.asarray(mask),
                              _StandInOps._p([[0, 0, 0, 0]], 86400., rhoFresh, rhoOld, minSnowD))

    @staticmethod
    def smooth(arr, conv_variant="post_divide", device=0, stddev=1.0):
        from oracle import astropy_restated as ar
        k = ar.gaussian2d_kernel(x_stddev=stddev, y_stddev=stddev, theta=0.0, x_size=3, y_size=3)
        return ar.convolve_fill0(np.asarray(arr, dtype=np.float64), k, variant=conv_variant)


def use_stand_in_ops(monkeypatch):
    """The drop-in module on the oracle-backed stand-in operators, its module globals set as ``main`` sets them."""
    monkeypatch.setattr(N, "_ops", lambda: _StandInOps)
    for k, v in dict(windPackFactor=5.8e-7, windPackThresh=5., leadLossFactor=2.9e-7, atmLossFactor=2.2e-8).items():
        monkeypatch.setattr(N, k, v)


def operator_outputs():
    """`calcLeadLoss`, `calcAtmLoss`, `calcWindPacking`, `calcDynamics`, `densityCalc`, `smooth_snow`,
    `fill_nan_no_negative`, `fillMaskAndNaNWithZero` of the drop-in module on seeded inputs: return values, or the
    argument after the in-place call (those return None, as the reference's do)."""
    rng = np.random.default_rng(5)
    ny, nx = 9, 11
    mask = rng.choice(np.array([0, 3, 8, 8, 8, 11, 12]), size=(ny, nx)).astype(float)
    h = np.abs(rng.normal(0.1, 0.1, (2, ny, nx)))
    h[:, mask > 10] = np.nan
    h[0, 2, 3] = 0.0
    h[1, 2, 3] = 0.0
    W = rng.gamma(4.0, 1.5, (ny, nx))
    W[0, :3] = 5.0
    W[1, 1] = np.nan
    C = np.clip(rng.random((ny, nx)), 0, 1)
    drift = 0.1 * rng.normal(size=(2, ny, nx))
    drift[:, 4:6, 4:7] = np.nan
    out = {}
    with np.errstate(all="ignore"):
        out["ops__calcLeadLoss"] = N.calcLeadLoss(h[0], W, C)
        out["ops__calcAtmLoss"] = N.calcAtmLoss(h[0], W)
        for i, g in enumerate(N.calcWindPacking(W, h[0])):
            out["ops__calcWindPacking__%d" % i] = g
        for i, g in enumerate(N.calcDynamics(drift, h, 100000)):
            assert g.shape == (2, ny, nx)
            out["ops__calcDynamics__%d" % i] = g
        out["ops__densityCalc"] = N.densityCalc(h, C, mask)
        out["ops__smooth_snow__clean"] = N.smooth_snow(np.nan_to_num(h[0], nan=0.0))
        out["ops__smooth_snow__holes"] = N.smooth_snow(h[0].copy(), stddev_val=0.5)
        for negz in (True, False):
            a = rng.normal(size=(ny, nx))
            a[3, 3] = np.inf
            a[4, 4] = np.nan
            assert N.fill_nan_no_negative(a, mask, negative_to_zero=negz) is None
            out["ops__fill_nan_no_negative__%s" % negz] = a
        a = rng.normal(size=(ny, nx))
        a[1, 2], a[2, 1], a[0, 0] = np.nan, np.inf, -np.inf
        assert N.fillMaskAndNaNWithZero(a) is None
        out["ops__fillMaskAndNaNWithZero"] = a
    return out


def test_per_function_operators_have_the_reference_contracts(monkeypatch):
    """The eight functions calcBudget is made of (NESOSIM.py:51-222, 458-473 in the reference) against what the
    reference's own functions returned on the same arguments: same return values or in-place effect, the module
    globals as the parameters.  The arithmetic is the stand-in's here; what is tested is everything around it."""
    import inspect
    from nesosim_b200 import engine as E
    for name in ("op_wind_terms", "op_dynamics", "op_fill_zero", "op_fill_nan_no_negative", "op_density", "smooth"):
        assert inspect.signature(getattr(_StandInOps, name)) == inspect.signature(getattr(E, name)), name
    use_stand_in_ops(monkeypatch)
    exp = golden_util.load(CONTRACTS)
    got = operator_outputs()
    assert len(got) == 13
    for key, g in got.items():
        assert same(g, exp[key]), key
    assert np.isfinite(got["ops__fillMaskAndNaNWithZero"]).all()
    clean = np.zeros((9, 11))
    with pytest.raises(ValueError):
        N.smooth_snow(clean, x_size_val=5)
    with pytest.raises(TypeError):
        N.fillMaskAndNaNWithZero(np.ma.masked_invalid(got["ops__fillMaskAndNaNWithZero"]))
