"""GPU: the day kernels, the calibration scores, tangents and adjoints with ice and finite drift on the grid edges, where
np.gradient takes one-sided differences with divisor dx and each build has its own code: the forward day kernel's
non-interior tiles, the tangent build's raw tangents, the record build's finite bits, the backward kernel's edge divisors
and the E term of the transposed differences, the forcing builds, and the season kernel's grid-edge slots.

The forcing (test_grid_edges_cpu.edge_season) has conc in [0.3, 1] and smooth finite drift on every ocean cell up to the
grid edge -- NaN over land, or finite there too -- an open-water patch on the top edge, one missing-drift day, a NaN drift
strip along the last column and a NaN snowfall corner; observations of every kind sit on every corner and along every
edge, and one footprint covers the whole top row.  Grids: all-ocean 2x2, 2x7, 7x2 and 3x3; coasts whose edges fall one
cell into a 32 x 16 tile, exactly at the `interior` bound or on a tile boundary (33x65, 34x66, 32x64, 17x97, 50x98);
the bundled 100 km and 25 km masks.  On the general path, for both CTA shapes and the land shortcut on and off, the
eleven season arrays are value-identical to oracle/nesosim_oracle.py and every score, Jacobian, gradient, theta_grad,
ic_grad and forcing derivative is bit-identical to the restatements.  Two plausible edge bugs planted in the oracle
(no E term; edge differences over 2 dx) differ from the GPU, so these comparisons would catch them.  The season kernel,
every build variant and cluster size that fits, matches the oracle and the general path on the 100 km and an all-ocean
90 x 90 grid; the row-strip decomposition reproduces the oracle; theta_grad agrees with forward mode.
test_grid_edges_cpu.py checks that the edge code ran (finite adv/div bits on every edge) and the restatements' identities
on the same cases."""
import functools

import numpy as np
import pytest

from nesosim_b200 import _lib
from nesosim_b200 import domain
from nesosim_b200 import synthetic as S
from oracle import footprint_scores as F
from oracle import forcing_adjoint as FA
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_adjoint as A
from oracle import score_gradients as G
from test_calibration_switches_gpu import check_member, concat_sets, run_all
from test_fused_scores_matrix_gpu import VARIANTS
from test_fused_scores_matrix_gpu import make_mask as matrix_mask
from test_general_scores_gpu import clear_env, engine, oracle_params, same
from test_grid_edges_cpu import FLAGS, FLAVOURS, FW, GRIDS, W, edge_case, edge_footprints, edge_obs, edge_season, edges

pytestmark = pytest.mark.gpu

FLAG_KW = dict(atmlossInc=1)


def oracle_member(forcing, ic_m, mask, dx, prow, obs, fps):
    """One member's season arrays, scores, tangent outputs and forcing adjoint from the restatements."""
    p = oracle_params(prow)
    s, tan = G.run_season_tangent(forcing, ic_m, mask, dx, p, FLAGS)
    chi2, used, v, fchi2, fused, mean = footprint_and_point_scores(s, forcing["conc"], obs, fps, mask)
    dv = G.model_tangents(s["snowDepths"], tan, forcing["conc"], obs, mask, p)
    _, dmean = G.footprint_tangents(s["snowDepths"], s["density"], tan, forcing["conc"], fps, mask, p)
    out = {"chi2": chi2, "used": used, "model": v, "fp_chi2": fchi2, "fp_used": fused, "fp_model": mean, "jac": dv,
           "grad": G.score_gradients(v, dv, obs, mask), "fp_jac": dmean, "fp_grad": G.footprint_gradients(mean, dmean, fps)}
    out.update(FA.score_adjoint_forcing(forcing, ic_m, mask, dx, p, FLAGS, obs, fps, W, FW))
    out["season"] = O.run_season(forcing, ic_m, mask, dx, p, FLAGS)
    return out


@functools.lru_cache(maxsize=None)
def oracle(grid, flavour):
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, flavour)
    return [oracle_member(forcing, ic[m], mask, dx, params[m], obs, fps) for m in range(len(params))]


def edge_ocean(mask):
    """The ocean cells of every grid edge that has any (the bundled masks' last column is land)."""
    wet = R.ocean(mask)
    return [e & wet for e in edges(mask.shape) if (e & wet).any()]


# ------------------------------------------------------------------------------------------------- the general path

@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("land", [0, 1])
@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("grid", list(GRIDS))
def test_general_path_bit_for_bit_against_the_oracle(cuda, monkeypatch, grid, flavour, land, threads):
    clear_env(monkeypatch)
    monkeypatch.setenv("NESOSIM_DAY_THREADS", str(threads))
    monkeypatch.setenv("NESOSIM_LAND_SHORTCUT", str(land))
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, flavour)
    M = len(params)
    eng = engine(mask, dx, T, M, [forcing], path="general", **FLAG_KW)
    plain = {k: v.cpu().numpy() for k, v in eng.run_season(params, ic).items()}
    assert eng.last_path() == "general" and sorted(plain) == sorted(_lib.OUTPUT_NAMES) and len(plain) == 11
    sc, gr, ad = run_all(eng, params, ic, obs, fps)
    eng.close()
    want = oracle(grid, flavour)
    for m in range(M):
        for name, a in plain.items():
            assert same(a[m], want[m]["season"][name]), (name, m)
        check_member(sc, gr, ad, m, want[m])
        for e in edge_ocean(mask):                        # the edge cells reached the objective
            assert np.abs(ad["ic_grad"][m][e]).max() > 0
    assert (sc["used"] > 0).all()


# ------------------------------------------------------------------------- the comparison catches plausible edge bugs

def _grad_t_without_e(pl, axis):
    """score_adjoint._grad_t without the E term: the transposed central differences alone."""
    pm = np.moveaxis(pl, axis, 0)
    pad = np.zeros((pm.shape[0] + 2,) + pm.shape[1:])
    pad[1:-1] = pm
    return np.moveaxis(pad[:-2] - pad[2:], 0, axis)


def _gradient_over_two_dx_at_the_edges(real):
    def gradient(f, dx, axis):
        g = real(f, dx, axis=axis)
        fm, gm = np.moveaxis(np.asarray(f, dtype=float), axis, 0), np.moveaxis(g, axis, 0)
        with np.errstate(all="ignore"):
            gm[0] = (fm[1] - fm[0]) / (2. * dx)
            gm[-1] = (fm[-1] - fm[-2]) / (2. * dx)
        return g
    return gradient


@pytest.mark.parametrize("grid", ["ocean_2x7", "ocean_7x2", "coast_33x65", "coast_34x66"])
def test_planted_edge_bugs_differ_from_the_gpu(cuda, monkeypatch, grid):
    """The oracle with either bug gives another ic_grad on the grid edges than the GPU; the oracle without gives the
    GPU's bit for bit."""
    clear_env(monkeypatch)
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, "land_nan")
    eng = engine(mask, dx, T, len(params), [forcing], path="general", **FLAG_KW)
    eng.set_observations_fp(obs, fps)
    got = eng.run_season_score_adjoint(params, ic, W, FW)["ic_grad"].cpu().numpy()[0]
    eng.close()

    def ic_grad():
        return A.score_adjoint(forcing, ic[0], mask, dx, oracle_params(params[0]), FLAGS, obs, fps, W, FW)[1]

    assert same(got, ic_grad())
    with monkeypatch.context() as mp:
        mp.setattr(A, "_grad_t", _grad_t_without_e)
        no_e = ic_grad()
    with monkeypatch.context() as mp:
        mp.setattr(np, "gradient", _gradient_over_two_dx_at_the_edges(np.gradient))
        two_dx = ic_grad()
    assert np.array_equal(np.gradient(np.arange(3.0) ** 2, 1.0, axis=0), [1.0, 2.0, 3.0])   # restored
    for wrong in (no_e, two_dx):
        assert all((wrong[e] != got[e]).any() for e in edge_ocean(mask))


# ------------------------------------------------------------------------------------------------ the season kernel

SEASON_T, SEASON_M = 9, 3
SET_DAYS, SET_MEMBERS = [9, 6, 8], [2, 0, 1, 1, 0]
SEASON_MASKS = ("arctic", "ocean")      # the 100 km grid; 90 x 90 all ocean
SEASON_CLUSTERS = range(2, 9)


@functools.lru_cache(maxsize=None)
def season_case(mask_name, flavour):
    """One forcing (M members) and three forcing sets of 9, 6 and 8 days, every one an ``edge_season``; the oracle's
    arrays and the general path's scores of both."""
    mask, dx = matrix_mask(mask_name)
    seed = 300 + 10 * SEASON_MASKS.index(mask_name) + 100 * FLAVOURS.index(flavour)
    rng = np.random.default_rng(seed)
    land = flavour == "land_finite"
    forcing, ic1 = edge_season(mask, SEASON_T, seed + 1, land)
    ic = ic1[None] * rng.uniform(0.3, 3.0, (SEASON_M, 1, 1))
    params = S.ensemble_params(SEASON_M, seed=seed + 2)
    obs, fps = edge_obs(mask, SEASON_T, rng), edge_footprints(mask, SEASON_T, rng)
    one = {"forcing": forcing, "ic": ic, "params": params, "obs": obs, "fps": fps}
    seasons = [edge_season(mask, d, seed + 3 + s, land)[0] for s, d in enumerate(SET_DAYS)]
    sic = ic1[None] * rng.uniform(0.3, 3.0, (len(SET_MEMBERS), 1, 1))
    sparams = S.ensemble_params(len(SET_MEMBERS), seed=seed + 7)
    sobs = [edge_obs(mask, d, rng, 300) for d in SET_DAYS]
    sfps = [edge_footprints(mask, d, rng) for d in SET_DAYS]
    cat, tag, fcat, ftag = concat_sets(sobs, sfps)
    sets = {"seasons": seasons, "ic": sic, "params": sparams, "obs": cat, "fps": fcat, "tag": tag, "ftag": ftag,
            "per_set": (sobs, sfps)}
    c = {"mask": mask, "dx": dx, "one": one, "sets": sets}
    c["oracle"] = [O.run_season(forcing, ic[m], mask, dx, oracle_params(params[m]), FLAGS) for m in range(SEASON_M)]
    c["general"] = {"one": scores_one(c, "general"), "sets": scores_sets(c, "general")}
    check_against_the_oracle(c, c["general"])
    return c


def scores_one(c, path):
    o = c["one"]
    eng = engine(c["mask"], c["dx"], SEASON_T, SEASON_M, [o["forcing"]], path=path, **FLAG_KW)
    try:
        eng.set_observations_fp(o["obs"], o["fps"])
        got = [t.cpu().numpy() for t in eng.run_season_scores_fp(o["params"], o["ic"], model=True)]
        assert eng.last_path() == ("general" if path == "general" else "ensemble")
        assert eng.rerun_count() == 0
    finally:
        eng.close()
    return got


def scores_sets(c, path):
    s = c["sets"]
    eng = engine(c["mask"], c["dx"], max(SET_DAYS), len(SET_MEMBERS), s["seasons"], SET_MEMBERS, SET_DAYS, path=path,
                 **FLAG_KW)
    try:
        eng.set_observations_fp(s["obs"], s["fps"], obs_set=s["tag"], fp_set=s["ftag"])
        got = [t.cpu().numpy() for t in eng.run_season_scores_fp(s["params"], s["ic"], model=True)]
        assert eng.last_path() == ("general" if path == "general" else "ensemble")
        assert eng.rerun_count() == 0
    finally:
        eng.close()
    return got


def check_against_the_oracle(c, got):
    """chi2, used, model and the footprint outputs of both cases against the restatements."""
    mask, dx = c["mask"], c["dx"]
    o = c["one"]
    for m in range(SEASON_M):
        ref = c["oracle"][m]
        want = footprint_and_point_scores(ref, o["forcing"]["conc"], o["obs"], o["fps"], mask)
        for i, w in enumerate(want):
            assert same(got["one"][i][m][:len(w)], w), (m, i)
    s = c["sets"]
    sobs, sfps = s["per_set"]
    for m, k in enumerate(SET_MEMBERS):
        f = s["seasons"][k]
        ref = O.run_season(f, s["ic"][m], mask, dx, oracle_params(s["params"][m]), FLAGS)
        want = footprint_and_point_scores(ref, f["conc"], sobs[k], sfps[k], mask)
        chi2, used, model, fchi2, fused, fmodel = (g[m] for g in got["sets"])
        assert same(chi2, want[0]) and same(used, want[1]) and same(fchi2, want[3]) and same(fused, want[4]), m
        assert same(model[:len(want[2])], want[2]) and same(fmodel[:len(want[5])], want[5]), m


def footprint_and_point_scores(ref, conc, obs, fps, mask):
    arrays = (ref["snowDepths"], ref["density"], conc)
    v = R.model_values(*arrays, obs, mask)
    chi2, used = R.scores(v, obs, mask)
    mean = F.footprint_values(*arrays, fps, mask)
    fchi2, fused = F.footprint_scores(mean, fps)
    return chi2, used, v, fchi2, fused, mean


def season_kernel_run(c, monkeypatch, variant, cluster):
    """Plain run_season and both scoring cases on the season kernel forced to (variant, cluster); None if that build
    does not fit the grid (ERR_ARG "no strip decomposition fits")."""
    monkeypatch.setenv("NESOSIM_ENS_VARIANT", variant)
    monkeypatch.setenv("NESOSIM_ENS_CLUSTER", str(cluster))
    o = c["one"]
    eng = engine(c["mask"], c["dx"], SEASON_T, SEASON_M, [o["forcing"]], path="ensemble", **FLAG_KW)
    try:
        plain = {k: v.cpu().numpy() for k, v in eng.run_season(o["params"], o["ic"]).items()}
        assert eng.last_path() == "ensemble" and eng.rerun_count() == 0
    except _lib.NesosimError as e:
        assert e.code == _lib.ERR_ARG and "no strip decomposition fits" in str(e), str(e)
        return None
    finally:
        eng.close()
    return plain, {"one": scores_one(c, "ensemble"), "sets": scores_sets(c, "ensemble")}


# Builds that fit the all-ocean 90 x 90 grid: its 8100 ocean cells need KO * NTC >= 8100 / cluster owned-cell slots,
# which only t352r6o5 (1760) has, on 5..8 CTAs.  Every build fits the 100 km grid on some cluster size.
FITS_OCEAN = {"t352r6o5"}


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("mask_name", SEASON_MASKS)
def test_season_kernel_every_build_and_cluster_size(cuda, monkeypatch, mask_name, flavour, variant):
    clear_env(monkeypatch)
    c = season_case(mask_name, flavour)
    ran = []
    for cluster in SEASON_CLUSTERS:
        r = season_kernel_run(c, monkeypatch, variant, cluster)
        if r is None:
            continue
        plain, got = r
        ran.append(cluster)
        for m in range(SEASON_M):
            for name, a in plain.items():
                assert same(a[m], c["oracle"][m][name]), (cluster, name, m)
        for case in ("one", "sets"):
            for i, (a, b) in enumerate(zip(got[case], c["general"][case])):
                assert same(a, b), (cluster, case, i)
    print("%s %s %s: cluster sizes %s" % (mask_name, flavour, variant, ran))
    assert bool(ran) == (mask_name == "arctic" or variant in FITS_OCEAN), ran


# ------------------------------------------------------------------------------------------- strips, forward mode

@pytest.mark.parametrize("n_strips", [2, 3])
@pytest.mark.parametrize("flavour", FLAVOURS)
def test_gpu_strips_reproduce_the_oracle_with_ice_on_the_grid_edges(cuda, monkeypatch, flavour, n_strips):
    """The row-strip decomposition (test_domain's single-process strips): the grid's top and bottom edges sit in the
    first and the last strip."""
    clear_env(monkeypatch)
    mask, dx, T, forcing, ic, params, obs, fps = edge_case("100km", flavour)

    def make(local_mask, num_days, dx_, forcing_local, params_row, ic_local):
        return domain.GpuStripStepper(local_mask, num_days, dx_, forcing_local, params_row, ic_local, **FLAG_KW)

    got = domain.run_decomposed_season_one_process(mask, T, dx, forcing, params[0], ic[0], n_strips, make)
    want = oracle("100km", flavour)[0]["season"]
    assert sorted(got) == sorted(_lib.OUTPUT_NAMES)
    for k in got:
        assert same(got[k], want[k]), k


@pytest.mark.parametrize("grid", ["coast_33x65", "100km"])
def test_against_forward_mode(cuda, monkeypatch, grid):
    """theta_grad = sum_k w_k grad[k] + sum_k fw_k fp_grad[k] of the tangent build, up to summation order."""
    clear_env(monkeypatch)
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, "land_nan")
    eng = engine(mask, dx, T, len(params), [forcing], path="general", **FLAG_KW)
    eng.set_observations_fp(obs, fps)
    fwd = {k: (None if v is None else v.cpu().numpy()) for k, v in eng.run_season_score_grads(params, ic).items()}
    adj = eng.run_season_score_adjoint(params, ic, W, FW)["theta_grad"].cpu().numpy()
    eng.close()
    want = np.einsum("k,mkd->md", W, fwd["grad"]) + np.einsum("k,mkd->md", FW, fwd["fp_grad"])
    rel = np.abs(adj - want).max(axis=1) / np.abs(want).max(axis=1)
    assert (rel <= 1e-10).all(), rel
