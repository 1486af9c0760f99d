"""CPU: bookkeeping of the multi-season calibration driver (ensemble.run_calibration) -- which (parameter set, season)
pairs a rank runs, which seasons it stages, the member -> forcing-set remap and the reassembly into [P, S] -- plus a
two-rank gloo run of its gather and the argument checks of nesosim_set_observations_sets that need no device."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nesosim_b200 import ensemble as ENS


def value(p, s):
    return 1000.0 * p + s


@pytest.mark.parametrize("world", [1, 2, 3, 5])
@pytest.mark.parametrize("P,S", [(1, 1), (1, 4), (3, 2), (8, 11), (13, 3), (2, 7)])
def test_every_pair_runs_once_and_lands_at_its_place(world, P, S):
    seen = []
    flat = []
    for rank in range(world):
        plan = ENS.calibration_plan(P, S, rank, world)
        pairs, staged, order, member_set = plan["pairs"], plan["seasons"], plan["order"], plan["member_set"]
        # a rank stages exactly the seasons its pairs use, in ascending order; its native call runs every pair once,
        # season by season, and every native member points at its own season
        assert staged == sorted({s for _, s in pairs})
        assert sorted(order.tolist()) == list(range(len(pairs)))
        run = [pairs[i] for i in order]
        assert [s for _, s in run] == sorted(s for _, s in pairs)
        assert len(member_set) == len(pairs) and member_set.dtype == np.int32
        assert all(staged[i] == s for i, (_, s) in zip(member_set, run))
        assert all(0 <= p < P and 0 <= s < S for p, s in pairs)
        seen += pairs
        native = np.array([value(p, s) for p, s in run])   # what the native call returns, in its member order
        flat += list(native[np.argsort(order)])           # back to the rank's pair order, as run_calibration does
    assert sorted(seen) == [(p, s) for p in range(P) for s in range(S)] and len(set(seen)) == P * S
    got = ENS.assemble_calibration(np.array(flat), P, S)  # the ranks' blocks concatenated in rank order (the gather)
    assert got.shape == (P, S)
    assert np.array_equal(got, np.array([[value(p, s) for s in range(S)] for p in range(P)]))


def test_a_rank_with_few_members_stages_few_seasons():
    # 4 parameter sets x 11 seasons over 8 ranks: 5 or 6 consecutive pairs per rank, hence at most 6 staged seasons
    for rank in range(8):
        plan = ENS.calibration_plan(4, 11, rank, 8)
        assert len(plan["seasons"]) == len(plan["pairs"]) <= 6
    # more ranks than pairs: the idle ranks stage nothing
    plan = ENS.calibration_plan(1, 2, 4, 5)
    assert plan["pairs"] == [] and plan["seasons"] == [] and len(plan["member_set"]) == 0


def _worker(rank, world, port, P, S, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    plan = ENS.calibration_plan(P, S, rank, world)
    mis = torch.tensor([value(p, s) for p, s in plan["pairs"]], dtype=torch.float64)
    used = torch.tensor([p + 10 * s for p, s in plan["pairs"]], dtype=torch.int64)
    got = ENS.gather_calibration(mis, used, P, S, rank, world)
    q.put((rank, got[0], got[1]))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_gather_the_same_calibration_table():
    P, S, world = 3, 5, 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, P, S, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want_mis = np.array([[value(p, s) for s in range(S)] for p in range(P)])
    want_used = np.array([[p + 10 * s for s in range(S)] for p in range(P)])
    for _, mis, used in results:                           # identical on every rank
        assert np.array_equal(mis, want_mis) and np.array_equal(used, want_used)


def test_set_observations_sets_validates_its_arguments(lib):
    from nesosim_b200 import _lib
    i32 = C.POINTER(C.c_int32)
    one = (C.c_int32 * 1)(0)
    dep = (C.c_double * 1)(0.1)
    assert lib.nesosim_set_observations_sets(None, 0, None, None, None, None, None) == _lib.ERR_ARG
    assert lib.nesosim_set_observations_sets(None, 1, C.cast(one, i32), C.cast(one, i32), C.cast(one, i32),
                                             C.cast(one, i32), dep) == _lib.ERR_ARG
    assert lib.nesosim_set_observations_sets(None, -1, None, None, None, None, None) == _lib.ERR_ARG
    assert "nesosim_set_observations_sets" in _lib.EXPORTED_SYMBOLS
