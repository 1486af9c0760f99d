"""Calibration-ensemble driver (SURVEY.md §8f N3; the reference has no counterpart -- it only runs one parameter set
per ``main`` call): M parameter sets over one forcing, sharded over the ranks of a box, with the outputs selected and
reduced ON THE DEVICE so that only what a calibration needs crosses PCIe (the full contract is 96 B per member-cell-day,
192 GB for 1024 members).

    misfit = run_ensemble(mask, forcing, ic, params, dx, obs=(day_idx, row_idx, col_idx, depth_obs))

Each rank runs its block of members through ``nesosim_run_season`` with only ``snowDepths`` requested, evaluates the
modelled snow depth over ice ``(h0+h1)/iceConc`` (what ``main`` writes as ``snow_depth``, NESOSIM.py:654) at the
observation points, and returns the per-member sum of squared differences; with ``world > 1`` the ranks' results are
all-gathered into member order (the only communication).

    misfit, used = run_calibration(mask, seasons, params, dx)      # [P, S]: every parameter set on every season

scores every parameter set on several observed seasons at once: the (parameter set, season) pairs are the members of one
batch of forcing sets, and the misfit of each pair is reduced against that season's observations.
"""
import numpy as np

from . import sharding


def depth_misfit(snowDepths, conc, obs):
    """Per-member sum of squared (modelled - observed) snow depth over ice at the observation points.
    ``snowDepths``: CUDA tensor (M,T,2,ny,nx); ``conc``: CUDA tensor (T,ny,nx); ``obs`` = (day, row, col, depth) arrays.
    NaN model values (land, missing forcing) are skipped, as a calibration against IceBridge-style data would."""
    import torch
    day, row, col, depth = (torch.as_tensor(np.asarray(a), device=snowDepths.device) for a in obs)
    day, row, col = day.long(), row.long(), col.long()
    h = snowDepths[:, day, 0, row, col] + snowDepths[:, day, 1, row, col]          # (M, n_obs)
    model = h / conc[day, row, col].unsqueeze(0)
    diff = model - depth.to(torch.float64).unsqueeze(0)
    ok = torch.isfinite(diff)
    return torch.where(ok, diff * diff, torch.zeros_like(diff)).sum(dim=1), ok.sum(dim=1)


def run_ensemble(mask, forcing, ic, params, dx, obs, rank=0, world=1, device=0, group=None, fused=None, **flags):
    """Returns (misfit[M], n_used[M]) as numpy arrays in member order (identical on every rank).  ``fused``: None =
    inside the season kernel where it applies, True = insist on it, False = depths to HBM + reduction there (the
    round-1 path, kept as the cross-check)."""
    import torch
    from .engine import SnowBudgetEngine
    params = np.asarray(params, dtype=np.float64).reshape(-1, 4)
    M = len(params)
    lo, hi = sharding.member_range(M, rank, world)
    T = forcing["precip"].shape[0]
    eng = SnowBudgetEngine(mask, T, dx, n_members=hi - lo, device=device, **flags)
    eng.set_forcing(forcing["precip"], forcing["conc"], forcing["wind"], forcing["drift"])
    from . import _lib
    try:
        # fused: the observation operator and the reduction run inside the season-resident kernel, nothing is stored
        mis, used = eng.run_season_misfit(params[lo:hi], ic, obs)
    except _lib.NesosimError as e:
        if fused is True or e.code != _lib.ERR_ARG:
            raise
        # grids the season-resident kernel does not take: depths to HBM, reduced there (still nothing crosses PCIe)
        out = eng.run_season(params[lo:hi], ic, eng.alloc_outputs(names=("snowDepths",)))
        mis, used = depth_misfit(out["snowDepths"], eng._forcing[1], obs)
    if fused is False:
        out = eng.run_season(params[lo:hi], ic, eng.alloc_outputs(names=("snowDepths",)))
        mis, used = depth_misfit(out["snowDepths"], eng._forcing[1], obs)
    eng.close()
    if world > 1:
        mis = sharding.gather_member_results(mis, M, rank, world, group)
        used = sharding.gather_member_results(used, M, rank, world, group)
    return mis.cpu().numpy(), used.cpu().numpy()


def calibration_plan(P, S, rank=0, world=1):
    """Bookkeeping of ``run_calibration`` (no device needed).  The P x S (parameter set, season) pairs are the members,
    parameter-major (member g = p*S + s), split over the ranks with ``sharding.member_range``.  Returns this rank's
    ``pairs`` [(p, s)] in member order, the seasons it stages (``seasons``, ascending: only those its pairs use) and
    the members of its native call: ``order`` (native member i is pair ``pairs[order[i]]``) and ``member_set`` (native
    member i's index into ``seasons``).  The native call takes its members season by season: the clusters that run at
    the same time then share one season's pre-digested forcing through L2 instead of each streaming another season's."""
    lo, hi = sharding.member_range(P * S, rank, world)
    pairs = [divmod(g, S) for g in range(lo, hi)]
    seasons = sorted({s for _, s in pairs})
    where = {s: i for i, s in enumerate(seasons)}
    order = np.array(sorted(range(len(pairs)), key=lambda i: (pairs[i][1], i)), dtype=np.int64)
    return {"pairs": pairs, "seasons": seasons, "order": order,
            "member_set": np.array([where[pairs[i][1]] for i in order], dtype=np.int32)}


def assemble_calibration(flat, P, S):
    """Results of all P*S members in member order -> array [P, S] (entry [p, s] = parameter set p on season s)."""
    return np.asarray(flat).reshape(P, S)


def gather_calibration(mis, used, P, S, rank=0, world=1, group=None):
    """All-gather the ranks' per-member results and reassemble them as numpy arrays (misfit[P,S], used[P,S]),
    identical on every rank."""
    if world > 1:
        mis = sharding.gather_member_results(mis, P * S, rank, world, group)
        used = sharding.gather_member_results(used, P * S, rank, world, group)
    return assemble_calibration(mis.cpu().numpy(), P, S), assemble_calibration(used.cpu().numpy(), P, S)


def run_calibration(mask, seasons, params, dx, rank=0, world=1, device=0, group=None, fused=None, **flags):
    """Multi-season calibration: every parameter set scored on every observed season in one native call per rank.
    ``seasons``: list of {"forcing": dict of (T_s,ny,nx) / drift (T_s,2,ny,nx) arrays, "ic": (ny,nx),
    "obs": (day, row, col, depth)}, each with its own length T_s.  Returns (misfit[P,S], used[P,S]) as numpy arrays,
    identical on every rank.  A rank stages only the seasons its (parameter set, season) pairs use, stacked as forcing
    sets of the longest of them, with each member's season IC as a per-member IC.  ``fused`` as in ``run_ensemble``:
    None = observations reduced inside the season kernel where it applies, True = insist on it, False = depths to HBM
    and a per-season reduction there."""
    import torch
    from . import _lib
    from .engine import SnowBudgetEngine
    params = np.asarray(params, dtype=np.float64).reshape(-1, 4)
    P, S = len(params), len(seasons)
    plan = calibration_plan(P, S, rank, world)
    pairs, staged, order, member_set = plan["pairs"], plan["seasons"], plan["order"], plan["member_set"]
    dev = "cuda:%d" % device
    if not pairs:   # more ranks than members: nothing to run, but the gather still needs this rank
        mis, used = torch.zeros(0, dtype=torch.float64, device=dev), torch.zeros(0, dtype=torch.int64, device=dev)
        return gather_calibration(mis, used, P, S, rank, world, group)
    days = [int(seasons[s]["forcing"]["precip"].shape[0]) for s in staged]
    T = max(days)

    def stack(name):   # [sets][T][...]; days past a season's end are never read (zero-filled)
        f0 = np.asarray(seasons[staged[0]]["forcing"][name])
        out = np.zeros((len(staged), T) + f0.shape[1:], dtype=np.float64)
        for i, s in enumerate(staged):
            out[i, :days[i]] = seasons[s]["forcing"][name]
        return out

    forcing = {k: stack(k) for k in ("precip", "conc", "wind", "drift")}
    run = [pairs[i] for i in order]                 # the native call's members, season by season
    ic = np.stack([np.asarray(seasons[s]["ic"], dtype=np.float64) for _, s in run])
    mine = params[[p for p, _ in run]]
    M = len(run)
    eng = SnowBudgetEngine(mask, T, dx, n_members=M, device=device, **flags)
    eng.set_forcing_sets(forcing["precip"], forcing["conc"], forcing["wind"], forcing["drift"], member_set, days)

    def hbm_round_trip():
        out = eng.run_season(mine, ic if M > 1 else ic[0], eng.alloc_outputs(names=("snowDepths",)))["snowDepths"]
        mis = torch.zeros(M, dtype=torch.float64, device=out.device)
        used = torch.zeros(M, dtype=torch.int64, device=out.device)
        for i, s in enumerate(staged):
            sel = torch.as_tensor(np.flatnonzero(member_set == i), device=out.device)
            m_i, u_i = depth_misfit(out[sel], eng._forcing[1][i], seasons[s]["obs"])
            mis[sel], used[sel] = m_i, u_i.to(torch.int64)
        return mis, used

    try:
        if fused is False:
            mis, used = hbm_round_trip()
        else:
            try:
                cols = [np.concatenate([np.asarray(seasons[s]["obs"][j]).ravel() for s in staged]) for j in range(4)]
                tag = np.concatenate([np.full(len(seasons[s]["obs"][0]), i, dtype=np.int32) for i, s in enumerate(staged)])
                eng.set_observations_sets(tag, *cols)
                mis, used = eng.run_season_misfit(mine, ic if M > 1 else ic[0])
            except _lib.NesosimError as e:
                if fused is True or e.code != _lib.ERR_ARG:
                    raise
                # grids the season-resident kernel does not take: depths to HBM, reduced there per season
                mis, used = hbm_round_trip()
    finally:
        eng.close()
    back = torch.as_tensor(np.argsort(order), device=mis.device)     # native member order -> this rank's pair order
    return gather_calibration(mis[back], used[back], P, S, rank, world, group)
