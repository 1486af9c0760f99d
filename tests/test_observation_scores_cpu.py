"""CPU: calibration scores without a device -- the argument checks of the new entry points, the torch operator
ensemble.observation_scores against a numpy restatement (density through the oracle's densityCalc), the normalisation
of a season's observations, the reassembly of the ranks' scores and a two-rank gloo gather of padded model rows."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nesosim_b200 import _lib
from nesosim_b200 import ensemble as ENS
from oracle import nesosim_oracle as O


def test_new_entry_points_validate_their_arguments(lib):
    i32, f64 = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    one = (C.c_int32 * 1)(0)
    val = (C.c_double * 1)(0.1)
    assert lib.nesosim_set_observations_ex(None, 0, None, None, None, None, None, None, None) == _lib.ERR_ARG
    assert lib.nesosim_set_observations_ex(None, 1, None, C.cast(one, i32), C.cast(one, i32), C.cast(one, i32),
                                           C.cast(one, i32), C.cast(val, f64), C.cast(val, f64)) == _lib.ERR_ARG
    assert lib.nesosim_set_observations_ex(None, -1, None, None, None, None, None, None, None) == _lib.ERR_ARG
    n = C.c_int64(0)
    assert lib.nesosim_observation_row_length(None, C.byref(n)) == _lib.ERR_ARG
    assert lib.nesosim_run_season_scores(None, None, None, 0, None, None, None, 0, None) == _lib.ERR_ARG
    for name in ("nesosim_set_observations_ex", "nesosim_observation_row_length", "nesosim_run_season_scores"):
        assert name in _lib.EXPORTED_SYMBOLS
    assert (_lib.OBS_DEPTH, _lib.OBS_VOLUME, _lib.OBS_DENSITY, _lib.OBS_KINDS) == (0, 1, 2, 3)


def arrays(M=3, T=6, ny=5, nx=7, seed=0):
    rng = np.random.default_rng(seed)
    depths = rng.uniform(0.0, 0.2, (M, T, 2, ny, nx))
    depths[:, :, :, 0, 0] = np.nan                                 # a land cell
    depths[:, 2, :, 1, 1] = 0.004                                  # below minSnowD: density NaN
    conc = rng.uniform(0.0, 1.0, (T, ny, nx))
    conc[3, 2, 2] = 0.0                                            # zero concentration: depth over ice inf
    p = O.Params()
    mask = np.ones((ny, nx))
    mask[0, 0] = 0
    dens = np.stack([np.stack([O.density_calc(depths[m, d], conc[d], mask, p) if d else np.zeros((ny, nx))
                               for d in range(T)]) for m in range(M)])
    return depths, dens, conc


def restated(depths, dens, conc, o):
    d, r, c, k = o["day"], o["row"], o["col"], o["kind"]
    vol = depths[:, d, 0, r, c] + depths[:, d, 1, r, c]
    with np.errstate(all="ignore"):
        model = np.where(k == 0, vol / conc[d, r, c], np.where(k == 1, vol, dens[:, d, r, c]))
        res = (model - o["value"]) / o["sigma"]
    ok = np.isfinite(res)
    chi2 = np.stack([np.where(ok & (k == j), res * res, 0.0).sum(1) for j in range(3)], 1)
    used = np.stack([(ok & (k == j)).sum(1) for j in range(3)], 1)
    return chi2, used, model


def test_observation_scores_on_cpu_tensors_match_the_numpy_restatement():
    depths, dens, conc = arrays()
    rng = np.random.default_rng(1)
    n = 400
    o = {"day": rng.integers(1, 6, n), "row": rng.integers(0, 5, n), "col": rng.integers(0, 7, n),
         "kind": rng.integers(0, 3, n), "sigma": 10.0 ** rng.uniform(-3, 1, n)}
    o["day"][:20], o["kind"][:20] = 0, rng.integers(0, 2, 20)     # depth / volume on day 0
    o["day"][20:30], o["row"][20:30], o["col"][20:30] = 2, 1, 1    # below minSnowD
    o["day"][30:40], o["row"][30:40], o["col"][30:40] = 3, 2, 2    # zero concentration
    o["row"][40:50], o["col"][40:50] = 0, 0                        # land
    o["value"] = np.where(o["kind"] == 2, 250.0, 0.2) * rng.random(n)
    o["value"][::17] = np.nan
    chi2, used, model = ENS.observation_scores(torch.from_numpy(depths), torch.from_numpy(dens), torch.from_numpy(conc), o)
    want = restated(depths, dens, conc, ENS.normalize_observations(o))
    assert np.allclose(chi2.numpy(), want[0], rtol=1e-12, atol=0.0)
    assert np.array_equal(used.numpy(), want[1]) and (want[1] > 50).all()
    assert np.array_equal(model.numpy(), want[2], equal_nan=True)
    assert np.isnan(model.numpy()[:, 20:30][:, o["kind"][20:30] == 2]).all()


@pytest.mark.parametrize("field,bad", [("kind", 3), ("kind", -1), ("sigma", 0.0), ("sigma", -1.0), ("sigma", np.nan),
                                       ("sigma", np.inf), ("density_day0", None)])
def test_observation_scores_rejects_what_the_fused_path_rejects(field, bad):
    depths, dens, conc = arrays()
    o = {"day": np.array([1, 2]), "row": np.array([1, 2]), "col": np.array([1, 2]), "value": np.array([0.1, 0.2]),
         "kind": np.array([0, 2]), "sigma": np.array([1.0, 1.0])}
    if field == "density_day0":
        o["day"][1] = 0
    else:
        o[field] = o[field].astype(type(bad))
        o[field][0] = bad
    with pytest.raises(ValueError):
        ENS.observation_scores(torch.from_numpy(depths), torch.from_numpy(dens), torch.from_numpy(conc), o)


def test_a_four_tuple_is_depth_with_sigma_one():
    o = ENS.normalize_observations(([1, 2], [3, 4], [5, 6], [0.1, 0.2]))
    assert o["kind"].tolist() == [0, 0] and o["sigma"].tolist() == [1.0, 1.0]
    assert o["day"].dtype == np.int32 and o["value"].dtype == np.float64 and o["col"].tolist() == [5, 6]
    d = ENS.normalize_observations({"day": [1], "row": [2], "col": [3], "value": [0.5], "kind": [2]})
    assert d["kind"].tolist() == [2] and d["sigma"].tolist() == [1.0]
    with pytest.raises(ValueError):
        ENS.normalize_observations({"day": [1, 2], "row": [2], "col": [3], "value": [0.5]})


def member_scores(p, s, n_obs, width):
    chi2 = np.array([1000.0 * p + s, p + 0.5, s + 0.25])
    model = np.full(width, np.nan)
    model[:n_obs[s]] = 100.0 * p + s + np.arange(n_obs[s]) / 1000.0
    return chi2, model


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("P,S", [(1, 1), (3, 2), (4, 5), (2, 7)])
def test_scores_land_at_their_place(world, P, S):
    n_obs = [3 + 2 * s for s in range(S)]
    width = max(n_obs)
    chi2, model = [], []
    for rank in range(world):
        plan = ENS.calibration_plan(P, S, rank, world)
        for p, s in plan["pairs"]:
            c, m = member_scores(p, s, n_obs, width)
            chi2.append(c)
            model.append(m)
    chi2 = np.array(chi2).reshape(-1, 3)
    model = np.array(model).reshape(-1, width)
    got = ENS.assemble_scores(chi2, chi2.astype(np.int64), model, P, S, n_obs)
    assert got["chi2"].shape == (P, S, 3) and got["used"].shape == (P, S, 3)
    assert len(got["model"]) == S
    for p in range(P):
        for s in range(S):
            c, m = member_scores(p, s, n_obs, width)
            assert np.array_equal(got["chi2"][p, s], c)
            assert got["model"][s].shape == (P, n_obs[s]) and np.array_equal(got["model"][s][p], m[:n_obs[s]])
    assert ENS.assemble_scores(chi2, chi2, None, P, S, n_obs)["model"] is None


def _worker(rank, world, port, P, S, n_obs, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    plan = ENS.calibration_plan(P, S, rank, world)
    width = max(n_obs)
    rows = [member_scores(p, s, n_obs, width) for p, s in plan["pairs"]]
    chi2 = torch.tensor(np.array([r[0] for r in rows]).reshape(-1, 3))
    model = torch.tensor(np.array([r[1] for r in rows]).reshape(-1, width))
    got = ENS.gather_scores(chi2, chi2.to(torch.int64), model, P, S, n_obs, rank, world)
    q.put((rank, got))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_gather_the_same_scores_with_padded_rows():
    P, S, world = 3, 4, 2
    n_obs = [5, 2, 7, 0]
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
    for _, got in results:                                 # identical on every rank
        for p in range(P):
            for s in range(S):
                c, m = member_scores(p, s, n_obs, max(n_obs))
                assert np.array_equal(got["chi2"][p, s], c) and np.array_equal(got["used"][p, s], c.astype(np.int64))
                assert np.array_equal(got["model"][s][p], m[:n_obs[s]])
