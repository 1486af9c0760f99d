"""CPU: the calibration adjoint with respect to the ice drift without a device -- the reverse-mode restatement
(oracle/drift_adjoint.py) against the forward tangent in random drift directions (dot-product identity), on the
adjoint's cases and on every grid-edge case of test_grid_edges_cpu, and against central differences of the primal
objective; the scale fields against the per-day stacks; nonzero derivatives on land cells next to the ocean where the
drift is finite over land; zeros without dynamics; the engine's, the driver's and the native entry point's argument
checks; the gather of the drift derivatives over two gloo ranks."""
import dataclasses
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nesosim_b200 import _lib
from nesosim_b200 import ensemble as ENS
from nesosim_b200 import synthetic as S
from nesosim_b200.engine import SnowBudgetEngine
from oracle import drift_adjoint as DA
from oracle import observation_scores as R
from oracle import score_adjoint as A
from oracle import score_gradients as G
from test_forcing_adjoint_cpu import objective, same_kinks
from test_grid_edges_cpu import CPU_GRIDS, FLAGS, FLAVOURS, FW, W, edge_case, edges
from test_score_adjoint_cpu import make_case as adj_case
from test_score_adjoint_cpu import point_obs, season

DX = 100000

# make_case of test_score_adjoint_cpu finite-fills the drift up to the coast (finite over land) and puts a finite IC on
# land; these cases add the drift's non-finite shapes on top
CASES = {
    "disc_land_ic": dict(base="disc_land_ic"),
    "edge_ocean": dict(base="edge_ocean"),
    "nan_patch": dict(base="nan_patch"),
    "nan_day": dict(base="disc_land_ic", nan_day=3),
    "nan_edge_strip": dict(base="edge_ocean", nan_strip=True),
    "land_nan": dict(base="disc_land_ic", land_nan=True),
    "no_windpack": dict(base="no_windpack"),
    "no_leadloss": dict(base="no_leadloss"),
    "no_atmloss": dict(base="no_atmloss"),
    "zero_weights": dict(base="zero_weights"),
    "density_near_min": dict(base="density_near_min"),
}


def make_case(name, T=8, seed=3):
    c = CASES[name]
    mask, forcing, ic, p, f, obs, fps, w, fw = adj_case(c["base"], T, seed)
    if c.get("nan_day") is not None:
        forcing["drift"][c["nan_day"]] = np.nan
    if c.get("nan_strip"):
        forcing["drift"][2, :, :, -1] = np.nan
        forcing["drift"][4, 1, 0, 3:12] = np.nan
    if c.get("land_nan"):
        forcing["drift"][:, :, G.land(mask)] = np.nan
    return mask, forcing, ic, p, f, obs, fps, w, fw


def direction(forcing, seed=11):
    rng = np.random.default_rng(seed)
    D = forcing["drift"]
    return np.where(np.isfinite(D), rng.standard_normal(D.shape) * np.nanstd(D), 0.0)


def identity(forcing, ic, mask, dx, p, f, obs, fps, w, fw, num_steps=None):
    got = DA.score_adjoint_drift(forcing, ic, mask, dx, p, f, obs, fps, w, fw, num_steps=num_steps)
    d = direction(forcing)
    lhs = float(np.sum(got["drift_day_grad"] * d))
    rhs = DA.objective_tangent_drift(forcing, ic, mask, dx, p, f, obs, fps, w, fw, d, num_steps=num_steps)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs), 1e-300), (lhs, rhs)
    assert lhs != 0.0
    return got


@pytest.mark.parametrize("name", list(CASES))
def test_dot_product_identity(name):
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case(name)
    assert set(range(R.KINDS)) <= set(np.asarray(obs["kind"]).tolist())
    assert set(range(R.KINDS)) - {R.VOLUME} <= set(np.asarray(fps["kind"]).tolist())
    got = identity(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    g = got["drift_day_grad"]
    assert np.isfinite(g).all() and np.isfinite(got["drift_scale_grad"]).all()
    assert not g[-1].any() and np.abs(g[:, 0]).max() > 0 and np.abs(g[:, 1]).max() > 0
    # the existing outputs are those of score_adjoint
    theta, icg, _ = A.score_adjoint(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    assert np.array_equal(theta, got["theta_grad"]) and np.array_equal(icg, got["ic_grad"])


@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("grid", CPU_GRIDS)
def test_dot_product_identity_on_the_grid_edges(grid, flavour):
    mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, flavour)
    p = DA.O.Params(windPackFactor=params[0, 0], windPackThresh=params[0, 1], leadLossFactor=params[0, 2],
                    atmLossFactor=params[0, 3])
    got = identity(forcing, ic[0], mask, dx, p, FLAGS, obs, fps, W, FW)
    wet = R.ocean(mask)
    g = got["drift_day_grad"]
    for e in edges(mask.shape):
        if (e & wet).any():
            assert np.abs(g[:, 0][:, e & wet]).max() > 0 and np.abs(g[:, 1][:, e & wet]).max() > 0


def test_land_cells_next_to_the_ocean_get_drift_derivatives():
    """Where the drift is finite over land, an ocean cell's div term reads its land neighbour's drift: g_u and g_v are
    nonzero on land cells that border the ocean, on days x > 0 too (where every land depth is NaN)."""
    for grid in ("coast_50x98", "coast_33x65"):
        mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, "land_finite")
        p = DA.O.Params(windPackFactor=params[0, 0], windPackThresh=params[0, 1], leadLossFactor=params[0, 2],
                        atmLossFactor=params[0, 3])
        got = DA.score_adjoint_drift(forcing, ic[0], mask, dx, p, FLAGS, obs, fps, W, FW)
        lnd = G.land(mask)
        wet = R.ocean(mask)
        near = np.zeros_like(wet)
        near[1:] |= wet[:-1]
        near[:-1] |= wet[1:]
        near[:, 1:] |= wet[:, :-1]
        near[:, :-1] |= wet[:, 1:]
        g = got["drift_day_grad"][1:T - 1]
        assert (np.abs(g[:, :, lnd & near]) > 0).any(axis=(0, 1)).mean() > 0.5
        assert not g[:, :, lnd & ~near].any()
        # with the drift NaN over land, no ocean cell next to land has a finite div term: no land cell has any
        mask, dx, T, forcing, ic, params, obs, fps = edge_case(grid, "land_nan")
        got = DA.score_adjoint_drift(forcing, ic[0], mask, dx, p, FLAGS, obs, fps, W, FW)
        assert not got["drift_day_grad"][1:T - 1][:, :, lnd].any()


def test_scale_fields_are_the_per_day_stacks_resummed():
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case("nan_patch")
    got = DA.score_adjoint_drift(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    T = forcing["precip"].shape[0]
    for k in range(2):
        acc = np.zeros(mask.shape)
        with np.errstate(invalid="ignore"):
            for x in range(T - 1, -1, -1):
                F = forcing["drift"][x, k]
                acc = acc + np.where(np.isfinite(F), F * got["drift_day_grad"][x, k], 0.0)
        assert np.array_equal(acc.view(np.int64), got["drift_scale_grad"][k].view(np.int64)), k
        assert got["drift_scale_total"][k] == R.fixed_order_sum(acc.ravel())


def test_dynamics_off_gives_zeros():
    mask, forcing, ic, p, f, obs, fps, w, fw = adj_case("no_dynamics")
    got = DA.score_adjoint_drift(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    for k in ("drift_day_grad", "drift_scale_grad", "drift_scale_total"):
        assert not got[k].any() and not np.signbit(got[k]).any(), k
    theta, icg, _ = A.score_adjoint(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    assert np.array_equal(theta, got["theta_grad"]) and np.array_equal(icg, got["ic_grad"])


def test_central_differences():
    mask, forcing, ic, p, f, obs, fps, w, fw = adj_case("disc_land_ic")
    p = dataclasses.replace(p, leadLossFactor=2.9e-7, atmLossFactor=2.2e-8)   # no clamp moves at 1 +- h
    obs = {k: v[obs["kind"] != R.DENSITY] for k, v in obs.items()}
    got = DA.score_adjoint_drift(forcing, ic, mask, DX, p, f, obs, fps, w, fw)
    _, base = objective(forcing, ic, mask, p, f, obs, fps, w, fw)
    h = 1e-4

    def central(scale):
        vals = []
        for sg in (1, -1):
            fc = dict(forcing)
            fc["drift"] = forcing["drift"] * (1.0 + sg * h * scale)
            val, k = objective(fc, ic, mask, p, f, obs, fps, w, fw)
            assert same_kinks(base, k)
            vals.append(val)
        return (vals[0] - vals[1]) / (2 * h)

    tot = got["drift_scale_total"]
    for k in range(2):
        scale = np.zeros((1, 2, 1, 1))
        scale[0, k] = 1.0
        fd = central(scale)
        assert np.isclose(tot[k], fd, rtol=1e-6, atol=1e-9 * abs(fd)), (k, tot[k], fd)
    fd = central(np.ones((1, 2, 1, 1)))                  # one drift speed factor: the sum of the two totals
    assert np.isclose(tot[0] + tot[1], fd, rtol=1e-6, atol=1e-9 * abs(fd)), (tot, fd)
    # per-cell factors on a few cells with the largest sensitivity
    sg0 = got["drift_scale_grad"][0]
    for cell in np.argsort(-np.abs(sg0).ravel())[:4]:
        r, c = np.unravel_index(cell, mask.shape)
        scale = np.zeros((1, 2) + mask.shape)
        scale[0, 0, r, c] = 1.0
        fd = central(scale)
        assert np.isclose(sg0[r, c], fd, rtol=1e-6, atol=1e-6 * np.abs(sg0).max()), (r, c, sg0[r, c], fd)


def test_short_season_with_last_day_observed():
    mask, forcing, ic, p, f, obs, fps, w, fw = make_case("nan_day", T=8)
    L = 5
    keep = obs["day"] <= L
    obs = {k: v[keep] for k, v in obs.items()}
    obs["day"][:20] = L
    got = identity(forcing, ic, mask, DX, p, f, obs, None, w, fw, num_steps=L)
    short = {k: v[:L + 1] for k, v in forcing.items()}
    ref = DA.score_adjoint_drift(short, ic, mask, DX, p, f, obs, None, w, fw)
    for k in ("theta_grad", "ic_grad", "drift_scale_grad", "drift_scale_total"):
        assert np.array_equal(got[k], ref[k]), k
    assert np.array_equal(got["drift_day_grad"][:L + 1], ref["drift_day_grad"])
    assert not got["drift_day_grad"][L:].any()


def test_engine_and_driver_reject_bad_requests():
    fake = types.SimpleNamespace()       # no context: the checks run before any device work
    with pytest.raises(ValueError, match="drift_days"):
        SnowBudgetEngine.run_season_score_adjoint(fake, np.zeros((1, 4)), None, drift_days=True)
    with pytest.raises(ValueError, match="drift_days"):
        SnowBudgetEngine.run_season_score_adjoint(fake, np.zeros((1, 4)), None, forcing=True, drift_days=True)
    mask, forcing, ic = season(T=4)
    seasons = [{"forcing": forcing, "ic": ic, "obs": point_obs(mask, 4, np.random.default_rng(5), 20)}]
    params = S.ensemble_params(2, seed=6)
    with pytest.raises(ValueError, match="drift_grad"):
        ENS.run_calibration_scores(mask, seasons, params, DX, drift_grad=True)
    with pytest.raises(ValueError, match="drift_grad"):
        ENS.run_calibration_scores(mask, seasons, params, DX, forcing_grad=False, drift_grad=True, model=True)


def test_native_entry_point_validates_its_arguments(lib):
    assert lib.nesosim_run_season_score_adjoint_drift(*([None, None, None, 0, None, None, None, None, None, 0, None,
                                                         None, None, 0] + [None] * 11)) == _lib.ERR_ARG
    assert "nesosim_run_season_score_adjoint_drift" in _lib.EXPORTED_SYMBOLS
    assert _lib.DRIFT_DIRS == len(_lib.DRIFT_COMPONENTS) == 2 and _lib.DRIFT_COMPONENTS == DA.COMPONENTS


def member_rows(p, s, shape):
    g = np.full((2,) + shape, 100.0 * p + s) + np.arange(2 * np.prod(shape)).reshape((2,) + shape) / 1000.0
    return g, np.array([1.0, 2.0]) + 10.0 * p + s


def _worker(rank, world, port, P, S_, shape, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rows = [member_rows(p, s, shape) for p, s in ENS.calibration_plan(P, S_, rank, world)["pairs"]]
    g = torch.tensor(np.array([r[0] for r in rows]).reshape((-1, 2) + shape))
    t = torch.tensor(np.array([r[1] for r in rows]).reshape(-1, 2))
    got = ENS.gather_scale_grad(g, t, P, S_, rank, world, prefix="drift")
    q.put((rank, got))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_gather_the_same_drift_gradients():
    P, S_, world, shape = 3, 3, 2, (4, 5)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, P, S_, shape, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, got in results:
        assert set(got) == {"drift_scale_grad", "drift_scale_total"}
        assert got["drift_scale_grad"].shape == (P, S_, 2) + shape and got["drift_scale_total"].shape == (P, S_, 2)
        for p in range(P):
            for s in range(S_):
                g, t = member_rows(p, s, shape)
                assert np.array_equal(got["drift_scale_grad"][p, s], g)
                assert np.array_equal(got["drift_scale_total"][p, s], t)
