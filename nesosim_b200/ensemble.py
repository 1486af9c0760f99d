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

    res = run_calibration_scores(mask, seasons, params, dx, model=True)   # chi2/used [P, S, 3], model rows per season

does the same with observation errors and three observed quantities (snow depth over ice, snow volume, bulk density):
per kind the sum of ((model - observed)/sigma)^2, and optionally the model value at every observation.  A season's
``"footprints"`` (``region_footprints``) add observed means over many cells and/or days, scored in the same call.

    res = run_calibration_scores(mask, seasons, params, dx, grad=True, jac=True)  # + grad [P, S, 3, 3], jac per season

adds the exact derivatives of chi2 (and of every model value) with respect to windPackFactor, leadLossFactor and
atmLossFactor, from the tangent-linear build of the scoring day kernel.
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


def normalize_observations(obs):
    """A season's observations as a dict of numpy arrays day, row, col (int32), value, sigma (float64), kind (int32).
    ``obs``: a dict with day, row, col, value and optionally kind (default depth) and sigma (default 1), or the 4-tuple
    (day, row, col, depth), which means depth observations with sigma 1."""
    from . import _lib
    if not isinstance(obs, dict):
        day, row, col, value = obs
        obs = {"day": day, "row": row, "col": col, "value": value}
    out = {k: np.asarray(obs[k], dtype=np.int32).ravel() for k in ("day", "row", "col")}
    out["value"] = np.asarray(obs["value"], dtype=np.float64).ravel()
    n = len(out["day"])
    kind, sigma = obs.get("kind"), obs.get("sigma")
    out["kind"] = np.full(n, _lib.OBS_DEPTH, np.int32) if kind is None else np.asarray(kind, dtype=np.int32).ravel()
    out["sigma"] = np.ones(n) if sigma is None else np.asarray(sigma, dtype=np.float64).ravel()
    if any(len(v) != n for v in out.values()):
        raise ValueError("observation arrays of different lengths")
    return out


def check_observations(obs, shape=None, days=None):
    """Rejects what nesosim_set_observations_ex rejects: a kind outside [0, OBS_KINDS), a density observation on day 0
    (the model has no density there) and a sigma that is not finite and > 0; with ``shape`` = (ny, nx) a row or column
    outside the grid, with ``days`` a day outside [0, days) of the observations' own season.  (Indexing the model's
    arrays with such an observation would wrap around, read a slot past the season, or fault on the device.)"""
    from . import _lib
    if shape is not None:
        ny, nx = shape
        if ((obs["row"] < 0) | (obs["row"] >= ny) | (obs["col"] < 0) | (obs["col"] >= nx)).any():
            raise ValueError("observation outside the %d x %d grid" % (ny, nx))
    if days is not None and ((obs["day"] < 0) | (obs["day"] >= days)).any():
        raise ValueError("observation day outside its season [0, %d)" % days)
    kind, sigma = obs["kind"], obs["sigma"]
    if ((kind < 0) | (kind >= _lib.OBS_KINDS)).any():
        raise ValueError("observation kind outside [0, %d)" % _lib.OBS_KINDS)
    if ((kind == _lib.OBS_DENSITY) & (obs["day"] == 0)).any():
        raise ValueError("density observation on day 0: the model has no density there")
    if not (np.isfinite(sigma) & (sigma > 0)).all():
        raise ValueError("observation error sigma must be finite and > 0")


def season_observations(mask, seasons):
    """Every season's observations, normalized and checked against the grid and that season's own length -- all seasons
    on every rank, so that the ranks raise alike and before any device work."""
    out = []
    for s in seasons:
        o = normalize_observations(s["obs"])
        check_observations(o, np.shape(mask), np.shape(s["forcing"]["precip"])[0])
        out.append(o)
    return out


def observation_scores(snowDepths, density, conc, obs, mask=None):
    """Per-member scores of ``obs`` (see ``normalize_observations``) on grids the season kernel does not take, from the
    arrays ``run_season`` writes: ``snowDepths`` (M,T,2,ny,nx), ``density`` (M,T,ny,nx), ``conc`` (T,ny,nx), all on
    one device.  Returns (chi2[M, OBS_KINDS], used[M, OBS_KINDS], model[M, n_obs]): the model value of every observation
    (depth over ice (h0+h1)/conc, volume h0+h1, or density), and per kind the sum of the finite ((model - value)/sigma)^2
    and their number -- what nesosim_run_season_scores reduces on the fused path.  ``mask`` (ny,nx) given: observations on
    land or lake cells (outside 1..10) have the model value NaN and are skipped, as on the fused path."""
    import torch
    from . import _lib
    obs = normalize_observations(obs)
    check_observations(obs, tuple(snowDepths.shape[-2:]), snowDepths.shape[1])
    dev = snowDepths.device
    day, row, col, kind = (torch.as_tensor(obs[k], device=dev).long() for k in ("day", "row", "col", "kind"))
    value, sigma = (torch.as_tensor(obs[k], device=dev) for k in ("value", "sigma"))
    vol = snowDepths[:, day, 0, row, col] + snowDepths[:, day, 1, row, col]          # (M, n_obs)
    model = torch.where(kind == _lib.OBS_VOLUME, vol, density[:, day, row, col])
    model = torch.where(kind == _lib.OBS_DEPTH, vol / conc[day, row, col], model)
    if mask is not None:
        m = np.asarray(mask)[obs["row"], obs["col"]]
        model = torch.where(torch.as_tensor((m >= 1) & (m <= 10), device=dev), model, torch.full_like(model, float("nan")))
    r = (model - value) / sigma
    ok = torch.isfinite(r)
    sq = torch.where(ok, r * r, torch.zeros_like(r))
    chi2 = torch.stack([torch.where(kind == k, sq, torch.zeros_like(sq)).sum(dim=1) for k in range(_lib.OBS_KINDS)], 1)
    used = torch.stack([(ok & (kind == k)).sum(dim=1) for k in range(_lib.OBS_KINDS)], 1)
    return chi2, used, model


def normalize_footprints(fps):
    """A season's footprint observations as a dict of numpy arrays: per footprint kind (int32), value and sigma
    (float64); ``begin`` (int64, [n_fp+1]): footprint g's points are [begin[g], begin[g+1]) of the per-point arrays day,
    row, col (int32) and weight (float64).  ``fps``: a dict with value, begin, day, row, col and optionally kind (default
    depth), sigma and weight (default 1)."""
    from . import _lib
    out = {"value": np.asarray(fps["value"], dtype=np.float64).ravel()}
    n = len(out["value"])
    kind, sigma, weight = fps.get("kind"), fps.get("sigma"), fps.get("weight")
    out["kind"] = np.full(n, _lib.OBS_DEPTH, np.int32) if kind is None else np.asarray(kind, dtype=np.int32).ravel()
    out["sigma"] = np.ones(n) if sigma is None else np.asarray(sigma, dtype=np.float64).ravel()
    out["begin"] = np.asarray(fps["begin"], dtype=np.int64).ravel()
    for k in ("day", "row", "col"):
        out[k] = np.asarray(fps[k], dtype=np.int32).ravel()
    npt = len(out["day"])
    out["weight"] = np.ones(npt) if weight is None else np.asarray(weight, dtype=np.float64).ravel()
    if len(out["kind"]) != n or len(out["sigma"]) != n or len(out["begin"]) != n + 1:
        raise ValueError("footprint arrays of different lengths (begin needs n_fp + 1 entries)")
    if any(len(out[k]) != npt for k in ("row", "col", "weight")):
        raise ValueError("footprint point arrays of different lengths")
    return out


def check_footprints(fps, shape=None, days=None):
    """Rejects what nesosim_set_observations_fp rejects (``fps`` normalized): ``begin`` not starting at 0, not
    increasing (an empty footprint) or not ending at the number of points; a kind outside [0, OBS_KINDS); a sigma or a
    weight that is not finite and > 0; a density point on day 0; more points than int indices hold; with ``shape`` a
    point outside the grid, with ``days`` a point outside [0, days) of its season."""
    from . import _lib
    b = fps["begin"]
    if b[0] != 0 or (np.diff(b) <= 0).any() or b[-1] != len(fps["day"]):
        raise ValueError("footprint begin must start at 0, increase (no empty footprint) and end at the point count")
    if len(fps["day"]) >= 2 ** 31 - 1:
        raise ValueError("more footprint points than int indices hold")
    kind = fps["kind"]
    if ((kind < 0) | (kind >= _lib.OBS_KINDS)).any():
        raise ValueError("footprint kind outside [0, %d)" % _lib.OBS_KINDS)
    if not (np.isfinite(fps["sigma"]) & (fps["sigma"] > 0)).all():
        raise ValueError("footprint error sigma must be finite and > 0")
    if not (np.isfinite(fps["weight"]) & (fps["weight"] > 0)).all():
        raise ValueError("footprint point weight must be finite and > 0")
    pkind = np.repeat(kind, np.diff(b))
    if ((pkind == _lib.OBS_DENSITY) & (fps["day"] == 0)).any():
        raise ValueError("density footprint point on day 0: the model has no density there")
    if shape is not None:
        ny, nx = shape
        if ((fps["row"] < 0) | (fps["row"] >= ny) | (fps["col"] < 0) | (fps["col"] >= nx)).any():
            raise ValueError("footprint point outside the %d x %d grid" % (ny, nx))
    if days is not None and ((fps["day"] < 0) | (fps["day"] >= days)).any():
        raise ValueError("footprint point day outside its season [0, %d)" % days)


def empty_footprints():
    return normalize_footprints({"value": [], "begin": [0], "day": [], "row": [], "col": []})


def region_footprints(mask, codes, windows, kind, value, sigma=1.0):
    """One footprint per day window [d0, d1) over every ocean cell (mask 1..10) whose mask code is in ``codes``, all
    weights 1, points day by day in row-major cell order -- the shape of a drifting-station climatology or a monthly
    gridded product.  ``value`` and ``sigma``: one number or one per window.  Returns ``normalize_footprints``' dict."""
    mask = np.asarray(mask)
    cells = np.flatnonzero(np.isin(mask, list(codes)) & (mask >= 1) & (mask <= 10))
    if not len(cells) or any(d1 <= d0 for d0, d1 in windows):
        raise ValueError("a footprint needs a point: no ocean cell has one of the codes, or a window is empty")
    n = len(windows)
    day = [np.repeat(np.arange(d0, d1, dtype=np.int64), len(cells)) for d0, d1 in windows]
    cell = [np.tile(cells, d1 - d0) for d0, d1 in windows]
    npt = np.array([len(d) for d in day], dtype=np.int64)
    cell = np.concatenate(cell) if n else np.zeros(0, np.int64)
    return normalize_footprints({
        "kind": np.full(n, kind), "value": np.broadcast_to(np.asarray(value, dtype=np.float64), (n,)).copy(),
        "sigma": np.broadcast_to(np.asarray(sigma, dtype=np.float64), (n,)).copy(),
        "begin": np.concatenate([[0], np.cumsum(npt)]),
        "day": np.concatenate(day) if n else [], "row": cell // mask.shape[1], "col": cell % mask.shape[1]})


def footprint_scores(snowDepths, density, conc, fps, mask):
    """Per-member scores of the footprints ``fps`` (see ``normalize_footprints``) from the arrays ``run_season`` writes:
    ``snowDepths`` (M,T,2,ny,nx), ``density`` (M,T,ny,nx), ``conc`` (T,ny,nx), all on one device; ``mask`` (ny,nx):
    points on land or lake cells are dropped.  Returns (fp_chi2[M, OBS_KINDS], fp_used[M, OBS_KINDS], fp_model[M, n_fp]):
    every footprint's weighted mean of its points' finite model values (NaN when none is finite), and per kind the sum of
    the finite ((mean - value)/sigma)^2 and their number -- what nesosim_run_season_scores_fp computes on the fused path
    (in another summation order)."""
    import torch
    from . import _lib
    fps = normalize_footprints(fps)
    check_footprints(fps, tuple(snowDepths.shape[-2:]), snowDepths.shape[1])
    dev = snowDepths.device
    M, G = snowDepths.shape[0], len(fps["value"])
    seg = torch.as_tensor(np.repeat(np.arange(G), np.diff(fps["begin"])), device=dev)
    kind = torch.as_tensor(fps["kind"], device=dev).long()
    pts = {"day": fps["day"], "row": fps["row"], "col": fps["col"], "value": np.zeros(len(fps["day"])),
           "kind": np.repeat(fps["kind"], np.diff(fps["begin"]))}
    _, _, v = observation_scores(snowDepths, density, conc, pts, mask)                 # (M, points), NaN on land
    w = torch.as_tensor(fps["weight"], device=dev).unsqueeze(0).expand_as(v)
    ok = torch.isfinite(v)
    zero = torch.zeros_like(v)
    sw = torch.zeros(M, G, dtype=torch.float64, device=dev).index_add_(1, seg, torch.where(ok, w * v, zero))
    s = torch.zeros(M, G, dtype=torch.float64, device=dev).index_add_(1, seg, torch.where(ok, w, zero))
    model = sw / s
    r = (model - torch.as_tensor(fps["value"], device=dev)) / torch.as_tensor(fps["sigma"], device=dev)
    good = torch.isfinite(r)
    sq = torch.where(good, r * r, torch.zeros_like(r))
    chi2 = torch.stack([torch.where(kind == k, sq, torch.zeros_like(sq)).sum(dim=1) for k in range(_lib.OBS_KINDS)], 1)
    used = torch.stack([(good & (kind == k)).sum(dim=1) for k in range(_lib.OBS_KINDS)], 1)
    return chi2, used, model


def fused_on_general_path(eng, fused_call, hbm_round_trip):
    """The fused call again on the general day-kernel path, for grids the season-resident kernel does not take: the
    engine is switched to ``set_path("general")`` and ``fused_call`` registers the observations and runs the scoring
    call (bit-identical to the season kernel's fixed order).  Where that path does not apply either (densityType='clim'
    or a strip context), ``hbm_round_trip`` instead."""
    from . import _lib
    eng.set_path("general")
    try:
        return fused_call()
    except _lib.NesosimError as e:
        if e.code != _lib.ERR_ARG:
            raise
        return hbm_round_trip()


def run_ensemble(mask, forcing, ic, params, dx, obs, rank=0, world=1, device=0, group=None, fused=None, **flags):
    """Returns (misfit[M], n_used[M]) as numpy arrays in member order (identical on every rank).  ``fused``: None =
    inside the season kernel where it applies, else fused on the general day-kernel path; True = insist on the season
    kernel; False = depths to HBM + reduction there (the round-1 path, kept as the cross-check).  Observations outside
    the grid or the season's days raise ValueError before any device work, on either path."""
    import torch
    from .engine import SnowBudgetEngine
    params = np.asarray(params, dtype=np.float64).reshape(-1, 4)
    M = len(params)
    lo, hi = sharding.member_range(M, rank, world)
    T = forcing["precip"].shape[0]
    check_observations(normalize_observations(obs), np.shape(mask), T)
    eng = SnowBudgetEngine(mask, T, dx, n_members=hi - lo, device=device, **flags)
    eng.set_forcing(forcing["precip"], forcing["conc"], forcing["wind"], forcing["drift"])
    from . import _lib

    def hbm_round_trip():   # depths to HBM, reduced there (still nothing crosses PCIe)
        out = eng.run_season(params[lo:hi], ic, eng.alloc_outputs(names=("snowDepths",)))
        return depth_misfit(out["snowDepths"], eng._forcing[1], obs)

    try:
        # fused: the observation operator and the reduction run inside the season-resident kernel, nothing is stored
        mis, used = eng.run_season_misfit(params[lo:hi], ic, obs)
    except _lib.NesosimError as e:
        if fused is True or e.code != _lib.ERR_ARG:
            raise
        if fused is None:   # grids the season-resident kernel does not take: sampled by the general day kernel
            mis, used = fused_on_general_path(eng, lambda: eng.run_season_misfit(params[lo:hi], ic, obs), hbm_round_trip)
    if fused is False:
        mis, used = hbm_round_trip()
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


def assemble_scores(chi2, used, model, P, S, n_obs):
    """Scores of all P*S members in member order -> {"chi2": [P, S, OBS_KINDS], "used": [P, S, OBS_KINDS], "model": per
    season s the array [P, n_obs[s]] (rows padded to the largest season: the padding is dropped), or None}."""
    from . import _lib
    out = {"chi2": np.asarray(chi2).reshape(P, S, _lib.OBS_KINDS), "used": np.asarray(used).reshape(P, S, _lib.OBS_KINDS),
           "model": None}
    if model is not None:
        m = np.asarray(model).reshape(P, S, -1)
        out["model"] = [m[:, s, :n_obs[s]] for s in range(S)]
    return out


def gather_scores(chi2, used, model, P, S, n_obs, rank=0, world=1, group=None):
    """All-gather the ranks' per-member scores (model rows padded to the largest season) and reassemble them as numpy
    arrays (``assemble_scores``), identical on every rank."""
    if world > 1:
        chi2 = sharding.gather_member_results(chi2, P * S, rank, world, group)
        used = sharding.gather_member_results(used, P * S, rank, world, group)
        if model is not None:
            model = sharding.gather_member_results(model, P * S, rank, world, group)
    return assemble_scores(chi2.cpu().numpy(), used.cpu().numpy(), None if model is None else model.cpu().numpy(),
                           P, S, n_obs)


def assemble_footprint_scores(fp_chi2, fp_used, fp_model, P, S, n_fp):
    """Footprint scores of all P*S members in member order -> {"fp_chi2": [P, S, OBS_KINDS], "fp_used": [P, S,
    OBS_KINDS], "fp_model": per season s the array [P, n_fp[s]] (rows padded to the largest season: the padding is
    dropped)}."""
    from . import _lib
    m = np.asarray(fp_model).reshape(P, S, -1)
    return {"fp_chi2": np.asarray(fp_chi2).reshape(P, S, _lib.OBS_KINDS),
            "fp_used": np.asarray(fp_used).reshape(P, S, _lib.OBS_KINDS),
            "fp_model": [m[:, s, :n_fp[s]] for s in range(S)]}


def gather_footprint_scores(fp_chi2, fp_used, fp_model, P, S, n_fp, rank=0, world=1, group=None):
    """All-gather the ranks' per-member footprint scores (model rows padded to the largest season) and reassemble them
    (``assemble_footprint_scores``), identical on every rank."""
    if world > 1:
        fp_chi2 = sharding.gather_member_results(fp_chi2, P * S, rank, world, group)
        fp_used = sharding.gather_member_results(fp_used, P * S, rank, world, group)
        fp_model = sharding.gather_member_results(fp_model, P * S, rank, world, group)
    return assemble_footprint_scores(fp_chi2.cpu().numpy(), fp_used.cpu().numpy(), fp_model.cpu().numpy(), P, S, n_fp)


def assemble_gradients(grad, jac, P, S, n_obs, prefix=""):
    """Gradients of all P*S members in member order -> {prefix + "grad": [P, S, OBS_KINDS, GRAD_DIRS], prefix + "jac":
    per season s the array [P, GRAD_DIRS, n_obs[s]] (rows padded to the largest season: the padding is dropped), or
    None}; prefix "fp_" for the footprints."""
    from . import _lib
    out = {prefix + "grad": np.asarray(grad).reshape(P, S, _lib.OBS_KINDS, _lib.GRAD_DIRS), prefix + "jac": None}
    if jac is not None:
        j = np.asarray(jac).reshape(P, S, _lib.GRAD_DIRS, -1)
        out[prefix + "jac"] = [j[:, s, :, :n_obs[s]] for s in range(S)]
    return out


def gather_gradients(grad, jac, P, S, n_obs, rank=0, world=1, group=None, prefix=""):
    """All-gather the ranks' per-member gradients (Jacobian rows padded to the largest season) and reassemble them
    (``assemble_gradients``), identical on every rank."""
    if world > 1:
        grad = sharding.gather_member_results(grad, P * S, rank, world, group)
        if jac is not None:
            jac = sharding.gather_member_results(jac, P * S, rank, world, group)
    return assemble_gradients(grad.cpu().numpy(), None if jac is None else jac.cpu().numpy(), P, S, n_obs, prefix)


def gather_adjoint(theta_grad, ic_grad, P, S, rank=0, world=1, group=None):
    """All-gather the ranks' per-member adjoint results ([n, GRAD_DIRS] and [n, ny, nx] in this rank's pair order) ->
    {"adjoint_grad": [P, S, GRAD_DIRS], "ic_grad": [P, S, ny, nx]}, numpy, identical on every rank."""
    if world > 1:
        theta_grad = sharding.gather_member_results(theta_grad, P * S, rank, world, group)
        ic_grad = sharding.gather_member_results(ic_grad, P * S, rank, world, group)
    th, icg = theta_grad.cpu().numpy(), ic_grad.cpu().numpy()
    return {"adjoint_grad": th.reshape(P, S, th.shape[-1]), "ic_grad": icg.reshape((P, S) + icg.shape[-2:])}


def gather_scale_grad(scale_grad, scale_total, P, S, rank=0, world=1, group=None, prefix="forcing"):
    """All-gather the ranks' per-member scale derivatives of one group of inputs ([n, dirs, ny, nx] and [n, dirs] in this
    rank's pair order) -> {"<prefix>_scale_grad": [P, S, dirs, ny, nx], "<prefix>_scale_total": [P, S, dirs]}, numpy,
    identical on every rank.  ``prefix``: "forcing" (FORCING_DIRS) or "drift" (DRIFT_DIRS)."""
    if world > 1:
        scale_grad = sharding.gather_member_results(scale_grad, P * S, rank, world, group)
        scale_total = sharding.gather_member_results(scale_total, P * S, rank, world, group)
    g, t = scale_grad.cpu().numpy(), scale_total.cpu().numpy()
    return {prefix + "_scale_grad": g.reshape((P, S) + g.shape[-3:]), prefix + "_scale_total": t.reshape(P, S, t.shape[-1])}


def gather_forcing_grad(scale_grad, scale_total, P, S, rank=0, world=1, group=None):
    """``gather_scale_grad`` of the forcing derivatives ([n, FORCING_DIRS, ny, nx] and [n, FORCING_DIRS])."""
    return gather_scale_grad(scale_grad, scale_total, P, S, rank, world, group, "forcing")


def season_footprints(mask, seasons):
    """Every season's footprints (``"footprints"`` entry; none: no footprints), normalized and checked against the grid
    and that season's own length, on every rank before any device work."""
    out = []
    for s in seasons:
        f = s.get("footprints")
        f = empty_footprints() if f is None else normalize_footprints(f)
        check_footprints(f, np.shape(mask), np.shape(s["forcing"]["precip"])[0])
        out.append(f)
    return out


def concat_footprints(fps):
    """Several seasons' footprints as one registration: (footprints, set tag per footprint)."""
    out = {k: np.concatenate([f[k] for f in fps]) for k in ("kind", "value", "sigma", "day", "row", "col", "weight")}
    npt = np.concatenate([np.diff(f["begin"]) for f in fps])
    out["begin"] = np.concatenate([[0], np.cumsum(npt)]).astype(np.int64)
    tag = np.concatenate([np.full(len(f["value"]), i, dtype=np.int32) for i, f in enumerate(fps)])
    return out, tag


def stage_calibration(mask, seasons, params, dx, plan, device=0, **flags):
    """The native call of a calibration rank: the seasons its pairs use (``plan`` = ``calibration_plan``) stacked as
    forcing sets of the longest of them, on a context of one member per pair, season by season, with each member's season
    IC as a per-member IC.  Returns (engine, parameters [M, 4], IC) of those members."""
    from .engine import SnowBudgetEngine
    staged, member_set = plan["seasons"], plan["member_set"]
    days = [int(seasons[s]["forcing"]["precip"].shape[0]) for s in staged]
    T = max(days)

    def stack(name):   # [sets][T][...]; days past a season's end are never read (zero-filled)
        f0 = np.asarray(seasons[staged[0]]["forcing"][name])
        out = np.zeros((len(staged), T) + f0.shape[1:], dtype=np.float64)
        for i, s in enumerate(staged):
            out[i, :days[i]] = seasons[s]["forcing"][name]
        return out

    forcing = {k: stack(k) for k in ("precip", "conc", "wind", "drift")}
    run = [plan["pairs"][i] for i in plan["order"]]   # the native call's members, season by season
    ic = np.stack([np.asarray(seasons[s]["ic"], dtype=np.float64) for _, s in run])
    M = len(run)
    eng = SnowBudgetEngine(mask, T, dx, n_members=M, device=device, **flags)
    eng.set_forcing_sets(forcing["precip"], forcing["conc"], forcing["wind"], forcing["drift"], member_set, days)
    return eng, params[[p for p, _ in run]], (ic if M > 1 else ic[0])


def run_calibration(mask, seasons, params, dx, rank=0, world=1, device=0, group=None, fused=None, **flags):
    """Multi-season calibration: every parameter set scored on every observed season in one native call per rank.
    ``seasons``: list of {"forcing": dict of (T_s,ny,nx) / drift (T_s,2,ny,nx) arrays, "ic": (ny,nx),
    "obs": (day, row, col, depth)}, each with its own length T_s.  Returns (misfit[P,S], used[P,S]) as numpy arrays,
    identical on every rank.  A rank stages only the seasons its (parameter set, season) pairs use, stacked as forcing
    sets of the longest of them, with each member's season IC as a per-member IC.  ``fused`` as in ``run_ensemble``:
    None = observations reduced inside the season kernel where it applies, else fused on the general day-kernel path
    (``fused_on_general_path``), True = insist on the season kernel, False = depths to HBM and a per-season reduction
    there.  Observations outside the grid or outside their season's days raise ValueError
    before any device work, on either path."""
    import torch
    from . import _lib
    params = np.asarray(params, dtype=np.float64).reshape(-1, 4)
    P, S = len(params), len(seasons)
    season_observations(mask, seasons)
    plan = calibration_plan(P, S, rank, world)
    pairs, staged, order, member_set = plan["pairs"], plan["seasons"], plan["order"], plan["member_set"]
    dev = "cuda:%d" % device
    if not pairs:   # more ranks than members: nothing to run, but the gather still needs this rank
        mis, used = torch.zeros(0, dtype=torch.float64, device=dev), torch.zeros(0, dtype=torch.int64, device=dev)
        return gather_calibration(mis, used, P, S, rank, world, group)
    eng, mine, ic = stage_calibration(mask, seasons, params, dx, plan, device, **flags)
    M = len(mine)

    def hbm_round_trip():
        out = eng.run_season(mine, ic, eng.alloc_outputs(names=("snowDepths",)))["snowDepths"]
        mis = torch.zeros(M, dtype=torch.float64, device=out.device)
        used = torch.zeros(M, dtype=torch.int64, device=out.device)
        for i, s in enumerate(staged):
            sel = torch.as_tensor(np.flatnonzero(member_set == i), device=out.device)
            m_i, u_i = depth_misfit(out[sel], eng._forcing[1][i], seasons[s]["obs"])
            mis[sel], used[sel] = m_i, u_i.to(torch.int64)
        return mis, used

    def fused_call():
        cols = [np.concatenate([np.asarray(seasons[s]["obs"][j]).ravel() for s in staged]) for j in range(4)]
        tag = np.concatenate([np.full(len(seasons[s]["obs"][0]), i, dtype=np.int32) for i, s in enumerate(staged)])
        eng.set_observations_sets(tag, *cols)
        return eng.run_season_misfit(mine, ic)

    try:
        if fused is False:
            mis, used = hbm_round_trip()
        else:
            try:
                mis, used = fused_call()
            except _lib.NesosimError as e:
                if fused is True or e.code != _lib.ERR_ARG:
                    raise
                # grids the season-resident kernel does not take: sampled by the general day kernel
                mis, used = fused_on_general_path(eng, fused_call, hbm_round_trip)
    finally:
        eng.close()
    back = torch.as_tensor(np.argsort(order), device=mis.device)     # native member order -> this rank's pair order
    return gather_calibration(mis[back], used[back], P, S, rank, world, group)


def run_calibration_scores(mask, seasons, params, dx, rank=0, world=1, device=0, group=None, fused=None, model=False,
                           grad=False, jac=False, adjoint=False, weights=None, fp_weights=None, forcing_grad=False,
                           drift_grad=False, **flags):
    """``run_calibration`` with observation errors and three observed quantities.  A season's ``"obs"`` is a dict with
    day, row, col, value and optionally kind (``_lib.OBS_DEPTH`` / ``OBS_VOLUME`` / ``OBS_DENSITY``, default depth) and
    sigma (default 1), or the 4-tuple (day, row, col, depth).  Returns {"chi2": [P, S, OBS_KINDS], "used": [P, S,
    OBS_KINDS], "model": per season the array [P, n_obs] of model values (NaN on land), or None unless ``model``}, numpy,
    identical on every rank.  ``fused`` as in ``run_calibration``: None = scored inside the season kernel where it applies
    and on the general day-kernel path on grids wider than it takes (the same fixed order, bit for bit), True = insist
    on the season kernel, False = snowDepths and density to
    HBM and ``observation_scores`` there.  Observations outside the grid or outside their season's days, bad kinds,
    sigmas and density observations on day 0 raise ValueError before any device work, on either path.

    A season may also have ``"footprints"`` (``normalize_footprints``; e.g. ``region_footprints``): observed means over
    many cells and/or days.  When some season has any, the result also holds "fp_chi2" / "fp_used" [P, S, OBS_KINDS]
    and "fp_model" (per season the array [P, n_fp] of footprint model values); the fused path scores them in the same
    call (nesosim_run_season_scores_fp), the HBM path with ``footprint_scores``.  Without footprints the result is
    unchanged.

    ``grad=True`` adds "grad" [P, S, OBS_KINDS, GRAD_DIRS]: the exact derivative of every chi2 with respect to
    windPackFactor, leadLossFactor and atmLossFactor (parameter columns ``_lib.GRAD_PARAMS``; windPackThresh enters
    through a step function and has none), from the tangent-linear build of the scoring day kernel
    (nesosim_run_season_score_grads).  It always scores on the general day-kernel path, whose chi2, used and model are
    bit-identical to the season kernel's; ``fused`` must stay None (neither the HBM round trip nor the season kernel has
    tangents: ValueError before any device work).  ``jac=True`` (with ``grad``) adds "jac": per season the array [P,
    GRAD_DIRS, n_obs] of d model / d theta (NaN where the model value is not finite).  With footprints also "fp_grad"
    and, with ``jac``, "fp_jac" (per season [P, GRAD_DIRS, n_fp]).

    ``adjoint=True`` adds the reverse-mode derivatives of every pair's objective J = sum_k weights[k] chi2[k] + sum_k
    fp_weights[k] fp_chi2[k] (OBS_KINDS finite weights >= 0 each, default all ones; nesosim_run_season_score_adjoint):
    "adjoint_grad" [P, S, GRAD_DIRS] (dJ / d theta for the ``_lib.GRAD_PARAMS`` columns) and "ic_grad" [P, S, ny, nx]
    (dJ / d the season's IC).  Like ``grad`` it scores on the general day-kernel path; with ``grad=True``, with ``fused``
    not None or with bad weights it raises ValueError before any device work.

    ``forcing_grad=True`` (with ``adjoint``; nesosim_run_season_score_adjoint_forcing) also adds the derivatives of J
    with respect to the season's forcing fields ``_lib.FORCING_FIELDS`` (precip, wind, conc): "forcing_scale_grad" [P,
    S, FORCING_DIRS, ny, nx] (dJ / d alpha of a per-cell factor F -> alpha F over the whole season) and
    "forcing_scale_total" [P, S, FORCING_DIRS] (one factor for the whole grid; [..., 0] is the snowfall scaling
    factor).  The per-day derivatives are offered by ``SnowBudgetEngine.run_season_score_adjoint`` alone: they are 8 T
    bytes per member-cell and field, too large to gather on every rank.

    ``drift_grad=True`` (with ``adjoint``, and freely with ``forcing_grad``; nesosim_run_season_score_adjoint_drift)
    adds the derivatives of J with respect to the season's ice drift ``_lib.DRIFT_COMPONENTS`` (u, v):
    "drift_scale_grad" [P, S, DRIFT_DIRS, ny, nx] (dJ / d alpha of a per-cell factor scaling one component over the
    whole season) and "drift_scale_total" [P, S, DRIFT_DIRS]; [..., 0] + [..., 1] is the derivative with respect to one
    drift speed factor (u, v) -> alpha (u, v).  Without dynamics both are 0."""
    import torch
    from . import _lib
    from .engine import check_weights
    if adjoint and (grad or fused is not None):
        raise ValueError("adjoint=True needs grad=False and fused=None: it runs on the general day-kernel path alone")
    if not adjoint and (weights is not None or fp_weights is not None):
        raise ValueError("weights and fp_weights belong to adjoint=True")
    if forcing_grad and not adjoint:
        raise ValueError("forcing_grad=True needs adjoint=True")
    if drift_grad and not adjoint:
        raise ValueError("drift_grad=True needs adjoint=True")
    if adjoint:
        weights, fp_weights = check_weights(weights, "weights"), check_weights(fp_weights, "fp_weights")
    if grad and fused is not None:
        raise ValueError("grad=True needs fused=None: only the general day-kernel path has tangents")
    if jac and not grad:
        raise ValueError("jac=True needs grad=True")
    params = np.asarray(params, dtype=np.float64).reshape(-1, 4)
    P, S = len(params), len(seasons)
    obs = season_observations(mask, seasons)
    fps = season_footprints(mask, seasons)
    n_obs = [len(o["day"]) for o in obs]
    n_fp = [len(f["value"]) for f in fps]
    width, fp_width = max(n_obs, default=0), max(n_fp, default=0)
    with_fp = fp_width > 0
    plan = calibration_plan(P, S, rank, world)
    pairs, staged, order, member_set = plan["pairs"], plan["seasons"], plan["order"], plan["member_set"]
    dev = "cuda:%d" % device
    K = _lib.OBS_KINDS

    D = _lib.GRAD_DIRS

    def gather(chi2, used, mod, fp, g=None, adj=None):
        res = gather_scores(chi2, used, mod, P, S, n_obs, rank, world, group)
        if adjoint:
            res.update(gather_adjoint(adj[0], adj[1], P, S, rank, world, group))
        if forcing_grad:
            res.update(gather_scale_grad(adj[2], adj[3], P, S, rank, world, group, "forcing"))
        if drift_grad:
            res.update(gather_scale_grad(adj[4], adj[5], P, S, rank, world, group, "drift"))
        if with_fp:
            res.update(gather_footprint_scores(*fp, P, S, n_fp, rank, world, group))
        if grad:
            res.update(gather_gradients(g[0], g[1], P, S, n_obs, rank, world, group))
            if with_fp:
                res.update(gather_gradients(g[2], g[3], P, S, n_fp, rank, world, group, prefix="fp_"))
        return res

    if not pairs:   # more ranks than members: nothing to run, but the gather still needs this rank
        chi2, used = torch.zeros(0, K, dtype=torch.float64, device=dev), torch.zeros(0, K, dtype=torch.int64, device=dev)
        mod = torch.zeros(0, width, dtype=torch.float64, device=dev) if model else None
        fp = (chi2, used, torch.zeros(0, fp_width, dtype=torch.float64, device=dev))
        g0 = torch.zeros(0, K, D, dtype=torch.float64, device=dev)
        g = (g0, torch.zeros(0, D, width, dtype=torch.float64, device=dev) if jac else None,
             g0, torch.zeros(0, D, fp_width, dtype=torch.float64, device=dev) if jac else None)
        F, Dd = _lib.FORCING_DIRS, _lib.DRIFT_DIRS
        adj = (torch.zeros(0, D, dtype=torch.float64, device=dev),
               torch.zeros((0,) + tuple(np.shape(mask)), dtype=torch.float64, device=dev),
               torch.zeros((0, F) + tuple(np.shape(mask)), dtype=torch.float64, device=dev),
               torch.zeros(0, F, dtype=torch.float64, device=dev),
               torch.zeros((0, Dd) + tuple(np.shape(mask)), dtype=torch.float64, device=dev),
               torch.zeros(0, Dd, dtype=torch.float64, device=dev))
        return gather(chi2, used, mod, fp, g, adj)
    eng, mine, ic = stage_calibration(mask, seasons, params, dx, plan, device, **flags)
    M = len(mine)

    def hbm_round_trip():
        out = eng.run_season(mine, ic, eng.alloc_outputs(names=("snowDepths", "density")))
        chi2, fchi2 = (torch.zeros(M, K, dtype=torch.float64, device=dev) for _ in range(2))
        used, fused_ = (torch.zeros(M, K, dtype=torch.int64, device=dev) for _ in range(2))
        mod = torch.full((M, width), float("nan"), dtype=torch.float64, device=dev)
        fmod = torch.full((M, fp_width), float("nan"), dtype=torch.float64, device=dev)
        for i, s in enumerate(staged):
            sel = torch.as_tensor(np.flatnonzero(member_set == i), device=dev)
            arrays = (out["snowDepths"][sel], out["density"][sel], eng._forcing[1][i])
            c, u, m = observation_scores(*arrays, obs[s], mask)
            chi2[sel], used[sel], mod[sel, :n_obs[s]] = c, u.to(torch.int64), m
            if with_fp:
                c, u, m = footprint_scores(*arrays, fps[s], mask)
                fchi2[sel], fused_[sel], fmod[sel, :n_fp[s]] = c, u.to(torch.int64), m
        return chi2, used, mod, (fchi2, fused_, fmod)

    def fused_call():
        cols = {k: np.concatenate([obs[s][k] for s in staged]) for k in obs[0]}
        tag = np.concatenate([np.full(n_obs[s], i, dtype=np.int32) for i, s in enumerate(staged)])
        if with_fp:
            fcols, ftag = concat_footprints([fps[s] for s in staged])
            eng.set_observations_fp(cols, fcols, obs_set=tag, fp_set=ftag)
            chi2, used, m, fchi2, fused_, fm = eng.run_season_scores_fp(mine, ic, model=True)
            fmod = torch.full((M, fp_width), float("nan"), dtype=torch.float64, device=dev)
            fmod[:, :fm.shape[1]] = fm
            fp = (fchi2, fused_, fmod)
        else:
            eng.set_observations_ex(cols["day"], cols["row"], cols["col"], cols["value"], cols["kind"],
                                    cols["sigma"], obs_set=tag)
            chi2, used, m = eng.run_season_scores(mine, ic, model=model)
            fp = None
        mod = None
        if model:   # rows of the staged seasons' length -> the largest season's (NaN past a row's end)
            mod = torch.full((M, width), float("nan"), dtype=torch.float64, device=dev)
            mod[:, :m.shape[1]] = m
        return chi2, used, mod, fp

    def padded(t, n, rows):   # [M, ..., n_staged] -> [M, ..., n] with NaN past a row's end (or all NaN: no such rows)
        out = torch.full(rows + (n,), float("nan"), dtype=torch.float64, device=dev)
        if t is not None:
            out[..., :t.shape[-1]] = t
        return out

    def grad_call():   # the general path's tangent / adjoint build: registered after set_path("general")
        eng.set_path("general")
        cols = {k: np.concatenate([obs[s][k] for s in staged]) for k in obs[0]}
        tag = np.concatenate([np.full(n_obs[s], i, dtype=np.int32) for i, s in enumerate(staged)])
        if with_fp:
            fcols, ftag = concat_footprints([fps[s] for s in staged])
            eng.set_observations_fp(cols, fcols, obs_set=tag, fp_set=ftag)
        else:
            eng.set_observations_ex(cols["day"], cols["row"], cols["col"], cols["value"], cols["kind"], cols["sigma"],
                                    obs_set=tag)
        if adjoint:
            r = eng.run_season_score_adjoint(mine, ic, weights, fp_weights, model=model or with_fp, forcing=forcing_grad,
                                             drift=drift_grad)
        else:
            r = eng.run_season_score_grads(mine, ic, model=model or with_fp, jac=jac)
        mod = padded(r["model"], width, (M,)) if model else None
        fp, fg, fj = None, None, None
        if with_fp:   # the staged seasons may have no footprint at all: zero sums, NaN rows
            zk = lambda dt: torch.zeros(M, K, dtype=dt, device=dev)
            fp = (r.get("fp_chi2", zk(torch.float64)), r.get("fp_used", zk(torch.int64)),
                  padded(r.get("fp_model"), fp_width, (M,)))
            fg = r.get("fp_grad", torch.zeros(M, K, D, dtype=torch.float64, device=dev))
            fj = padded(r.get("fp_jac"), fp_width, (M, D)) if jac else None
        if adjoint:
            return r["chi2"], r["used"], mod, fp, (r["theta_grad"], r["ic_grad"], r.get("forcing_scale_grad"),
                                                   r.get("forcing_scale_total"), r.get("drift_scale_grad"),
                                                   r.get("drift_scale_total"))
        g = (r["grad"], padded(r["jac"], width, (M, D)) if jac else None, fg, fj)
        return r["chi2"], r["used"], mod, fp, g

    g = adj = None
    try:
        if adjoint:
            chi2, used, mod, fp, adj = grad_call()
        elif grad:
            chi2, used, mod, fp, g = grad_call()
        elif fused is False:
            chi2, used, mod, fp = hbm_round_trip()
        else:
            try:
                chi2, used, mod, fp = fused_call()
            except _lib.NesosimError as e:
                if fused is True or e.code != _lib.ERR_ARG:
                    raise
                # grids the season-resident kernel does not take: sampled by the general day kernel
                chi2, used, mod, fp = fused_on_general_path(eng, fused_call, hbm_round_trip)
    finally:
        eng.close()
    back = torch.as_tensor(np.argsort(order), device=chi2.device)    # native member order -> this rank's pair order
    if with_fp:
        fp = tuple(t[back] for t in fp)
    if grad:
        g = tuple(None if t is None else t[back] for t in g)
    if adjoint:
        adj = tuple(None if t is None else t[back] for t in adj)
    return gather(chi2[back], used[back], mod[back] if model else None, fp, g, adj)
