"""Final-product diagnostics (SURVEY.md §8f N2): the fused GPU pass against the numpy oracle, and the oracle against what
the reference's own OutputSnowModelFinal wrote (run verbatim with a recording stand-in for netCDF4; stored in
tests/golden/reference_contracts.npz)."""
import numpy as np
import pytest

from golden_util import canon_sha, load
from nesosim_b200 import synthetic as S
from oracle import final_products as FP
from oracle import nesosim_oracle as O


def season(T=9, seed=13):
    mask = S.region_mask(dx=100000)
    forcing = S.make_season(mask, T, seed=seed)
    ic = S.make_ic(mask, seed=seed) * 4
    out = O.run_season(forcing, ic, mask, 100000, O.Params(), O.Flags(atmlossInc=1))
    conc = forcing["conc"].copy()
    conc[2, 40:44, 40:44] = 0.15            # thresholds exactly
    conc[3, 40:44, 40:44] = 0.5
    conc[4, 10, 10] = np.nan
    h = out["snowDepths"].copy()
    h[5, 0, 45, 45] = 0.123456789           # rounding cases: half-way and float32-inexact values
    h[5, 1, 45, 45] = 0.00005
    h[6, :, 46, 46] = [0.00125, 0.0]
    return h, out["density"], conc, forcing["precip"], forcing["wind"]


def same32(a, b):
    return a.dtype == np.float32 and b.dtype == np.float32 and a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


# the rows and columns of season() that hold the threshold and rounding cases
WINDOW = (slice(None), slice(38, 48), slice(38, 48))


def writer_digests():
    """The six float32 fields OutputSnowModelFinal writes (utils.py:161-179 in the reference), as the oracle computes
    them from season(): sha256 of each full field (golden_util.canon_sha) and the values in WINDOW."""
    h, dens, conc, precip, wind = season()
    out = {}
    for name, field in FP.final_fields(h, dens, conc, precip, wind).items():
        assert field.dtype == np.float32 and field.shape == conc.shape, name
        out["final__sha__" + name] = np.array(canon_sha(field))
        out["final__window__" + name] = field[WINDOW]
    return out


def test_oracle_matches_reference_writer():
    exp = load("reference_contracts.npz")
    got = writer_digests()
    names = ("snow_volume", "snow_depth", "snow_density", "ice_concentration", "precipitation", "wind_speed")
    assert len(got) == 2 * len(names)
    for name in names:
        assert str(got["final__sha__" + name]) == str(exp["final__sha__" + name]), name
        assert same32(got["final__window__" + name], exp["final__window__" + name]), name


def test_oracle_masks_and_rounding():
    h, dens, conc, precip, wind = season()
    f = FP.final_fields(h, dens, conc, precip, wind)
    assert all(v.dtype == np.float32 for v in f.values())
    with np.errstate(invalid="ignore"):
        low = conc < 0.5
    assert np.isnan(f["snow_volume"][low]).all() and np.isnan(f["snow_depth"][low]).all() and np.isnan(f["snow_density"][low]).all()
    assert not np.isnan(f["snow_volume"][3, 40:44, 40:44]).all()          # conc == 0.5 is kept
    assert np.isnan(f["ice_concentration"][conc < 0.15]).all() and f["ice_concentration"][2, 41, 41] == np.float32(0.15)
    assert np.isnan(f["snow_depth"][4, 10, 10])                              # NaN concentration: depth NaN, volume kept
    keep = FP.final_fields(h, dens, conc, precip, wind, ice_conc_mask=0)
    assert np.isfinite(keep["ice_concentration"][conc < 0.15]).all()


@pytest.mark.gpu
def test_gpu_final_products_match_oracle(cuda):
    from nesosim_b200 import engine as E
    h, dens, conc, precip, wind = season()
    for m in (0.5, 0.0, 0.3):
        exp = FP.final_fields(h, dens, conc, precip, wind, ice_conc_mask=m)
        got = {k: v.cpu().numpy() for k, v in E.final_products(h, dens, conc, precip, wind, ice_conc_mask=m).items()}
        for k in exp:
            assert same32(got[k], exp[k]), (k, m)
    # an ensemble: members stacked, one shared forcing
    h3 = np.stack([h, h * 0.5, h * 2.0])
    d3 = np.stack([dens, dens, dens])
    got = {k: v.cpu().numpy() for k, v in E.final_products(h3, d3, conc, precip, wind).items()}
    for m in range(3):
        exp = FP.final_fields(h3[m], d3[m], conc, precip, wind)
        for k in exp:
            assert same32(got[k][m], exp[k]), (k, m)
    # straight from a season still resident on the device
    from nesosim_b200.engine import SnowBudgetEngine
    mask = S.region_mask(dx=100000)
    forcing = S.make_season(mask, 9, seed=13)
    ic = S.make_ic(mask, seed=13) * 4
    eng = SnowBudgetEngine(mask, 9, 100000, atmlossInc=1)
    eng.set_forcing(forcing["precip"], forcing["conc"], forcing["wind"], forcing["drift"])
    out = eng.run_season([[5.8e-7, 5., 2.9e-7, 2.2e-8]], ic)
    got = E.final_products(out["snowDepths"][0], out["density"][0], forcing["conc"], forcing["precip"], forcing["wind"])
    ref = O.run_season(forcing, ic, mask, 100000, O.Params(), O.Flags(atmlossInc=1))
    exp = FP.final_fields(ref["snowDepths"], ref["density"], forcing["conc"], forcing["precip"], forcing["wind"])
    for k in exp:
        assert same32(got[k].cpu().numpy(), exp[k]), k
