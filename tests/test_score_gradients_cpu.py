"""CPU: calibration gradients without a device -- the tangent-linear restatement (oracle/score_gradients.py) against
central finite differences of the primal oracle, the exact zeros of a switched-off parameter, the driver's argument
checks, the reassembly of the ranks' gradients and a two-rank gloo gather."""
import ctypes as C
import dataclasses
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nesosim_b200 import _lib
from nesosim_b200 import ensemble as ENS
from nesosim_b200 import synthetic as S
from oracle import nesosim_oracle as O
from oracle import observation_scores as R
from oracle import score_gradients as G

FIELDS = G.PARAM_FIELDS


def season(T=9, seed=1):
    mask = S.region_mask(shape=(20, 26), kind="disc")
    forcing = S.make_season(mask, T, seed=seed)
    forcing["wind"] = forcing["wind"] * 1.5             # most cells above the wind threshold: every term active
    ic = 0.05 + S.make_ic(mask, seed=seed)
    return mask, forcing, ic


def point_obs(mask, T, rng, n=400):
    wet = np.argwhere(R.ocean(mask))
    cell = wet[rng.integers(len(wet), size=n)]
    day = rng.integers(1, T, n)
    kind = rng.integers(0, R.KINDS, n)
    value = np.where(kind == R.DENSITY, 250.0 + 50 * rng.random(n), 0.2 * rng.random(n))
    return {"day": day, "row": cell[:, 0], "col": cell[:, 1], "kind": kind, "value": value,
            "sigma": rng.uniform(0.01, 1.0, n) * np.where(kind == R.DENSITY, 100.0, 1.0)}


def values(forcing, ic, mask, dx, p, f, obs):
    s = O.run_season(forcing, ic, mask, dx, p, f)
    return s, R.model_values(s["snowDepths"], s["density"], forcing["conc"], obs, mask)


def kinks(s, p):
    """Where the primal sits on a kink: NaN cells, depths clamped to (or at) 0, densities at a clamp."""
    h, d = s["snowDepths"], s["density"][1:]
    return np.isnan(h), h == 0.0, (d == p.snowDensityOld) | (d == p.snowDensityFresh)


# Relative step 1e-4 of each parameter: the season is polynomial in theta between kinks, so the central difference is
# exact up to O(step^2) (about 1e-8 relative here); the tangents must agree to 1e-6 relative to the column's scale.
STEP, RTOL = 1e-4, 1e-6


@pytest.mark.parametrize("dynamics", [0, 1])
def test_tangents_match_central_differences(dynamics):
    mask, forcing, ic = season()
    dx, T = 100000, forcing["precip"].shape[0]
    f = O.Flags(dynamicsInc=dynamics, atmlossInc=1)
    p = O.Params(windPackFactor=5.8e-7, windPackThresh=4.0, leadLossFactor=2.9e-7, atmLossFactor=2.2e-8)
    obs = point_obs(mask, T, np.random.default_rng(2))
    s, tan = G.run_season_tangent(forcing, ic, mask, dx, p, f)
    ref, v = values(forcing, ic, mask, dx, p, f, obs)
    assert np.array_equal(s["snowDepths"], ref["snowDepths"], equal_nan=True)     # the primal is calc_budget's
    dv = G.model_tangents(s["snowDepths"], tan, forcing["conc"], obs, mask, p)
    chi2_grad = G.score_gradients(v, dv, obs, mask)
    for j, name in enumerate(FIELDS):
        h = STEP * getattr(p, name)
        sp, vp = values(forcing, ic, mask, dx, dataclasses.replace(p, **{name: getattr(p, name) + h}), f, obs)
        sm, vm = values(forcing, ic, mask, dx, dataclasses.replace(p, **{name: getattr(p, name) - h}), f, obs)
        for a, b, c in zip(kinks(s, p), kinks(sp, p), kinks(sm, p)):   # no step straddles a kink
            assert np.array_equal(a, b) and np.array_equal(a, c), name
        fd = (vp - vm) / (2 * h)
        ok = np.isfinite(v)
        assert ok.sum() > 100 and np.array_equal(np.isfinite(dv[j]), ok)
        scale = np.abs(fd[ok]).max()
        assert scale > 0, name
        assert np.allclose(dv[j][ok], fd[ok], rtol=RTOL, atol=RTOL * scale), name
        cp = R.scores(vp, obs, mask)[0]
        cm = R.scores(vm, obs, mask)[0]
        fd_chi2 = (cp - cm) / (2 * h)
        assert np.allclose(chi2_grad[:, j], fd_chi2, rtol=RTOL, atol=RTOL * np.abs(fd_chi2).max()), name


def test_footprint_tangents_match_central_differences():
    mask, forcing, ic = season(T=8, seed=3)
    dx, T = 100000, 8
    f = O.Flags(atmlossInc=1)
    p = O.Params(windPackThresh=4.0)
    fps = ENS.region_footprints(mask, [k for k in range(1, 11) if (mask == k).any()][:2], [(1, 4), (4, 8)],
                                R.DEPTH, [0.2, 0.25], 0.05)
    s, tan = G.run_season_tangent(forcing, ic, mask, dx, p, f)
    mean, dmean = G.footprint_tangents(s["snowDepths"], s["density"], tan, forcing["conc"], fps, mask, p)
    for j, name in enumerate(FIELDS):
        h = STEP * getattr(p, name)
        fd = []
        for sign in (1, -1):
            q = dataclasses.replace(p, **{name: getattr(p, name) + sign * h})
            sq = O.run_season(forcing, ic, mask, dx, q, f)
            fd.append(G.footprint_tangents(sq["snowDepths"], sq["density"], tan, forcing["conc"], fps, mask, q)[0])
        fd = (fd[0] - fd[1]) / (2 * h)
        assert np.allclose(dmean[j], fd, rtol=RTOL, atol=RTOL * np.abs(fd).max()), name


@pytest.mark.parametrize("off", ["windpackInc", "leadlossInc", "atmlossInc"])
def test_a_switched_off_parameter_has_an_exactly_zero_column(off):
    mask, forcing, ic = season(T=6, seed=4)
    f = dataclasses.replace(O.Flags(atmlossInc=1), **{off: 0})
    j = {"windpackInc": 0, "leadlossInc": 1, "atmlossInc": 2}[off]
    s, tan = G.run_season_tangent(forcing, ic, mask, 100000, O.Params(windPackThresh=4.0), f)
    assert not tan[:, j].any()
    assert np.abs(tan[:, [k for k in range(3) if k != j]]).max() > 0


def test_driver_rejects_grad_off_the_general_path():
    mask, forcing, ic = season(T=4)
    seasons = [{"forcing": forcing, "ic": ic, "obs": point_obs(mask, 4, np.random.default_rng(5), 20)}]
    params = S.ensemble_params(2, seed=6)
    for fused in (True, False):
        with pytest.raises(ValueError, match="fused=None"):
            ENS.run_calibration_scores(mask, seasons, params, 100000, grad=True, fused=fused)
    with pytest.raises(ValueError, match="grad=True"):
        ENS.run_calibration_scores(mask, seasons, params, 100000, jac=True)


def test_native_entry_point_validates_its_arguments(lib):
    assert lib.nesosim_run_season_score_grads(None, None, None, 0, None, None, None, 0, None, None, 0, None, None, None,
                                              0, None, None, 0, None) == _lib.ERR_ARG
    assert "nesosim_run_season_score_grads" in _lib.EXPORTED_SYMBOLS
    assert _lib.GRAD_DIRS == 3 and _lib.GRAD_PARAMS == (0, 2, 3)
    assert [_lib.MemberParams._fields_[i][0] for i in _lib.GRAD_PARAMS] == list(FIELDS)


def member_grad(p, s, n_obs, width):
    g = np.arange(9, dtype=np.float64).reshape(3, 3) + 100.0 * p + s
    jac = np.full((3, width), np.nan)
    jac[:, :n_obs[s]] = 10.0 * p + s + np.arange(3 * n_obs[s]).reshape(3, -1) / 100.0
    return g, jac


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("P,S", [(1, 1), (3, 2), (2, 5)])
def test_gradients_land_at_their_place(world, P, S):
    n_obs = [2 + s % 3 for s in range(S)]
    width = max(n_obs)
    rows = [member_grad(p, s, n_obs, width) for r in range(world) for p, s in ENS.calibration_plan(P, S, r, world)["pairs"]]
    for prefix in ("", "fp_"):
        got = ENS.assemble_gradients(np.array([r[0] for r in rows]), np.array([r[1] for r in rows]), P, S, n_obs, prefix)
        assert got[prefix + "grad"].shape == (P, S, 3, 3) and len(got[prefix + "jac"]) == S
        for p in range(P):
            for s in range(S):
                g, jac = member_grad(p, s, n_obs, width)
                assert np.array_equal(got[prefix + "grad"][p, s], g)
                assert got[prefix + "jac"][s].shape == (P, 3, n_obs[s])
                assert np.array_equal(got[prefix + "jac"][s][p], jac[:, :n_obs[s]])
    assert ENS.assemble_gradients(np.zeros((P * S, 3, 3)), None, P, S, n_obs)["jac"] is None


def _worker(rank, world, port, P, S, n_obs, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rows = [member_grad(p, s, n_obs, max(n_obs)) for p, s in ENS.calibration_plan(P, S, rank, world)["pairs"]]
    g = torch.tensor(np.array([r[0] for r in rows]).reshape(-1, 3, 3))
    jac = torch.tensor(np.array([r[1] for r in rows]).reshape(-1, 3, max(n_obs)))
    got = ENS.gather_gradients(g, jac, P, S, n_obs, rank, world)
    got.update(ENS.gather_gradients(g, jac, P, S, n_obs, rank, world, prefix="fp_"))
    q.put((rank, got))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_gather_the_same_gradients():
    P, S, world = 3, 3, 2
    n_obs = [2, 0, 4]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, P, S, n_obs, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, got in results:
        for p in range(P):
            for s in range(S):
                g, jac = member_grad(p, s, n_obs, max(n_obs))
                for prefix in ("", "fp_"):
                    assert np.array_equal(got[prefix + "grad"][p, s], g)
                    assert np.array_equal(got[prefix + "jac"][s][p], jac[:, :n_obs[s]])
