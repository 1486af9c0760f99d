"""CPU: footprint observations without a device -- the restated fixed order (oracle footprint_values) against a plain
weighted mean and its lane assignment, the argument checks of the Python layer and of the native entry points,
ensemble.region_footprints, the torch operator ensemble.footprint_scores, the reassembly of the ranks' footprint scores
and a two-rank gloo gather."""
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
from oracle import footprint_scores as F
from oracle import observation_scores as R


def arrays(M=2, T=8, ny=6, nx=9, seed=0):
    rng = np.random.default_rng(seed)
    depths = rng.uniform(0.0, 0.2, (M, T, 2, ny, nx))
    depths[:, :, :, 0, 0] = np.nan                                 # a land cell
    depths[:, 2, :, 1, 1] = 0.004                                  # below minSnowD: density NaN
    conc = rng.uniform(0.1, 1.0, (T, ny, nx))
    conc[3, 2, 2] = 0.0                                            # zero concentration: depth over ice inf
    mask = np.full((ny, nx), 5)
    mask[0, 0] = 11
    p = O.Params()
    dens = np.stack([np.stack([O.density_calc(depths[m, d], conc[d], mask, p) if d else np.zeros((ny, nx))
                               for d in range(T)]) for m in range(M)])
    return depths, dens, conc, mask


def random_footprints(rng, sizes, T=8, ny=6, nx=9):
    n = int(np.sum(sizes))
    kind = np.arange(len(sizes)) % 3
    day = rng.integers(1, T, n)
    return ENS.normalize_footprints({
        "kind": kind, "value": np.where(kind == 2, 300.0, 0.1) * rng.random(len(sizes)),
        "sigma": rng.uniform(0.05, 5.0, len(sizes)), "begin": np.concatenate([[0], np.cumsum(sizes)]),
        "day": day, "row": rng.integers(0, ny, n), "col": rng.integers(0, nx, n), "weight": 2.0 ** rng.uniform(-3, 3, n)})


def test_restated_order_is_a_weighted_mean_with_lane_j_mod_32():
    depths, dens, conc, mask = arrays()
    rng = np.random.default_rng(1)
    fps = random_footprints(rng, [1, 5, 31, 32, 33, 64, 65, 300, 1000])
    fps["row"][:3], fps["col"][:3] = 0, 0                          # land points: dropped
    got = F.footprint_values(depths[0], dens[0], conc, fps, mask)
    for g in range(len(got)):
        sl = slice(fps["begin"][g], fps["begin"][g + 1])
        pts = {k: fps[k][sl] for k in ("day", "row", "col")}
        pts["kind"] = np.full(len(pts["day"]), fps["kind"][g])
        v, w = R.model_values(depths[0], dens[0], conc, pts, mask), fps["weight"][sl]
        ok = np.isfinite(v)
        want = np.sum(w[ok] * v[ok]) / np.sum(w[ok]) if ok.any() else np.nan   # footprint 0: its point is on land
        assert np.isclose(got[g], want, rtol=1e-13, atol=0.0, equal_nan=True), (g, got[g], want)
    # lane assignment: kept point j goes to lane j % 32.  Point 0 (lane 0) is 1.0, points 1 and 33 (lane 1) are 2^-53
    # each: lane 1 holds 2^-52 and the tree gives 1 + 2^-52; a single running sum would round both away.  A land
    # point in front is dropped before the lanes are assigned.
    d = np.zeros_like(depths[0])
    d[1, 0, 3, :3] = [1.0, 2.0 ** -53, 0.0]
    col = np.full(35, 2)
    col[[1, 2, 34]] = [0, 1, 1]
    one = {"kind": np.array([1]), "value": np.array([0.0]), "sigma": np.array([1.0]), "begin": np.array([0, 35]),
           "day": np.full(35, 1), "row": np.full(35, 3), "col": col, "weight": np.ones(35)}
    one["row"][0], one["col"][0] = 0, 0                            # land
    v = F.footprint_values(d, dens[0], conc, one, mask)[0]
    assert v == (1.0 + 2.0 ** -52) / 34.0 and v != 1.0 / 34.0


def test_region_footprints():
    mask = np.array([[1, 1, 11], [8, 0, 8], [8, 9, 3]], dtype=np.uint8)
    f = ENS.region_footprints(mask, [8, 11, 0], [(1, 3), (5, 6)], _lib.OBS_DENSITY, [300.0, 310.0], sigma=20.0)
    cells = [(1, 0), (1, 2), (2, 0)]                               # ocean cells with code 8, row-major; 11 and 0 are not ocean
    assert f["begin"].tolist() == [0, 6, 9]
    assert f["day"].tolist() == [1, 1, 1, 2, 2, 2, 5, 5, 5]
    assert list(zip(f["row"].tolist(), f["col"].tolist())) == cells * 3
    assert f["kind"].tolist() == [2, 2] and f["value"].tolist() == [300.0, 310.0] and f["sigma"].tolist() == [20.0, 20.0]
    assert (f["weight"] == 1.0).all() and f["begin"].dtype == np.int64
    ENS.check_footprints(f, mask.shape, 6)
    with pytest.raises(ValueError):
        ENS.region_footprints(mask, [5], [(1, 3)], 0, 0.1)        # no such ocean cell: an empty footprint
    with pytest.raises(ValueError):
        ENS.region_footprints(mask, [8], [(3, 3)], 0, 0.1)        # an empty window


@pytest.mark.parametrize("field,bad", [("begin0", 1), ("empty", None), ("end", None), ("kind", 3), ("kind", -1),
                                       ("sigma", 0.0), ("sigma", np.nan), ("weight", 0.0), ("weight", -2.0),
                                       ("weight", np.inf), ("density_day0", None), ("row", 6), ("col", -1),
                                       ("day", 8)])
def test_python_layer_rejects_what_the_native_registration_rejects(field, bad):
    depths, dens, conc, mask = arrays()
    fps = random_footprints(np.random.default_rng(2), [3, 4, 5])
    if field == "begin0":
        fps["begin"][0] = bad
    elif field == "empty":
        fps["begin"][2] = fps["begin"][1]
    elif field == "end":
        fps["begin"][-1] -= 1
    elif field == "density_day0":
        fps["day"][fps["begin"][2]] = 0                            # footprint 2 is density
    else:
        fps[field] = fps[field].astype(type(bad))
        fps[field][0] = bad
    with pytest.raises(ValueError):
        ENS.footprint_scores(torch.from_numpy(depths), torch.from_numpy(dens), torch.from_numpy(conc), fps, mask)
    with pytest.raises(ValueError):
        ENS.season_footprints(mask, [{"forcing": {"precip": np.zeros((8,) + mask.shape)}, "footprints": fps}])


def test_normalize_footprints_defaults_and_lengths():
    f = ENS.normalize_footprints({"value": [0.2], "begin": [0, 2], "day": [1, 2], "row": [0, 1], "col": [3, 4]})
    assert f["kind"].tolist() == [0] and f["sigma"].tolist() == [1.0] and f["weight"].tolist() == [1.0, 1.0]
    with pytest.raises(ValueError):
        ENS.normalize_footprints({"value": [0.2], "begin": [0, 2, 3], "day": [1, 2, 3], "row": [0, 1, 1], "col": [3, 4, 5]})
    with pytest.raises(ValueError):
        ENS.normalize_footprints({"value": [0.2], "begin": [0, 2], "day": [1, 2], "row": [0], "col": [3, 4]})


def test_footprint_scores_on_cpu_tensors_match_the_restatement():
    depths, dens, conc, mask = arrays()
    fps = random_footprints(np.random.default_rng(3), [1, 7, 40, 33, 200, 3])
    fps["row"][fps["begin"][5]:], fps["col"][fps["begin"][5]:] = 0, 0   # footprint 5: all on land
    fps["day"][fps["begin"][1]], fps["row"][fps["begin"][1]], fps["col"][fps["begin"][1]] = 2, 1, 1
    chi2, used, model = ENS.footprint_scores(torch.from_numpy(depths), torch.from_numpy(dens), torch.from_numpy(conc),
                                             fps, mask)
    for m in range(2):
        wm = F.footprint_values(depths[m], dens[m], conc, fps, mask)
        wc, wu = F.footprint_scores(wm, fps)
        assert np.allclose(model[m].numpy(), wm, rtol=1e-13, atol=0.0, equal_nan=True)
        assert np.isnan(wm[5]) and np.array_equal(used[m].numpy(), wu) and wu.sum() == 5
        assert np.allclose(chi2[m].numpy(), wc, rtol=1e-12, atol=0.0)


def test_native_entry_points_validate_their_arguments(lib):
    n = C.c_int64(0)
    assert lib.nesosim_set_observations_fp(None, 0, None, None, None, None, None, None, None, 0, None, None, None, None,
                                           None, None, None, None, None) == _lib.ERR_ARG
    assert lib.nesosim_footprint_row_length(None, C.byref(n)) == _lib.ERR_ARG
    assert lib.nesosim_run_season_scores_fp(None, None, None, 0, None, None, None, 0, None, None, None, 0,
                                            None) == _lib.ERR_ARG
    for name in ("nesosim_set_observations_fp", "nesosim_footprint_row_length", "nesosim_run_season_scores_fp"):
        assert name in _lib.EXPORTED_SYMBOLS


def member_fp(p, s, n_fp, width):
    chi2 = np.array([100.0 * p + s, p + 0.125, s + 0.5])
    model = np.full(width, np.nan)
    model[:n_fp[s]] = 10.0 * p + s + np.arange(n_fp[s]) / 100.0
    return chi2, model


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("P,S", [(1, 1), (3, 2), (2, 5)])
def test_footprint_scores_land_at_their_place(world, P, S):
    n_fp = [2 + s % 3 for s in range(S)]
    width = max(n_fp)
    rows = [member_fp(p, s, n_fp, width) for r in range(world) for p, s in ENS.calibration_plan(P, S, r, world)["pairs"]]
    chi2 = np.array([r[0] for r in rows])
    got = ENS.assemble_footprint_scores(chi2, chi2.astype(np.int64), np.array([r[1] for r in rows]), P, S, n_fp)
    assert got["fp_chi2"].shape == (P, S, 3) and got["fp_used"].shape == (P, S, 3) and len(got["fp_model"]) == S
    for p in range(P):
        for s in range(S):
            c, m = member_fp(p, s, n_fp, width)
            assert np.array_equal(got["fp_chi2"][p, s], c)
            assert np.array_equal(got["fp_model"][s][p], m[:n_fp[s]])


def _worker(rank, world, port, P, S, n_fp, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rows = [member_fp(p, s, n_fp, max(n_fp)) for p, s in ENS.calibration_plan(P, S, rank, world)["pairs"]]
    chi2 = torch.tensor(np.array([r[0] for r in rows]).reshape(-1, 3))
    model = torch.tensor(np.array([r[1] for r in rows]).reshape(-1, max(n_fp)))
    got = ENS.gather_footprint_scores(chi2, chi2.to(torch.int64), model, P, S, n_fp, rank, world)
    q.put((rank, got))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_gather_the_same_footprint_scores():
    P, S, world = 3, 3, 2
    n_fp = [2, 0, 4]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, P, S, n_fp, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, got in results:
        for p in range(P):
            for s in range(S):
                c, m = member_fp(p, s, n_fp, max(n_fp))
                assert np.array_equal(got["fp_chi2"][p, s], c) and np.array_equal(got["fp_used"][p, s], c.astype(np.int64))
                assert np.array_equal(got["fp_model"][s][p], m[:n_fp[s]])
