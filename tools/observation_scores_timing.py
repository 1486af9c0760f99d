"""Calibration-scores timing on the headline workload: 128 members, the 100 km season of bench.py (260 days), 20 000
point observations drawn as bench.py's run_misfit_mode draws them.

  (a) nesosim_run_season_misfit against nesosim_run_season_scores, all depth, and against run_season_scores with mixed
      kinds (depth, volume, density; log-uniform sigma) and the model row: CUDA events around the calls (each ends in a
      stream synchronise), warm-up then best of 5, with the season kernel's own device time (nesosim_season_kernel_time,
      mean of the 5) and the epilogue's device time (torch.profiler with CUDA activities, a run of its own, mean of 5)
  (b) the S = 11 batch of tools/calibration_seasons_timing.py at P = 8/32/128: misfit against scores (all depth)

--kernel-only prints just the season kernel's device time of the misfit mode on one forcing (the OBS instantiation)
and on forcing sets (SETS && OBS; two copies of the season, every member on set 0), through nesosim_set_observations /
_sets and nesosim_run_season_misfit only, so that it also runs on builds without the scores entry points: a copy of
this script in another checkout's tools/ measures that checkout's build, and alternating the two in one session
compares two builds of the season kernel.

The GPU's name and power limit are read in the same run.
usage: python tools/observation_scores_timing.py --out DIR [--P 8,32,128] | --kernel-only [--reps 10]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

DX = 100000
NUM_DAYS = 260
MEMBERS = 128
SEED = 2024
N_OBS = 20000


def headline(sets=False):
    """The bench season, its observations and an engine of MEMBERS members (forcing sets: two copies, all on set 0)."""
    from nesosim_b200 import synthetic as S
    from nesosim_b200.engine import SnowBudgetEngine
    mask = S.region_mask(dx=DX)
    f = S.make_season(mask, NUM_DAYS, seed=SEED)
    ic = S.make_ic(mask, seed=SEED)
    params = S.ensemble_params(MEMBERS, seed=SEED)
    rng = np.random.default_rng(SEED)
    ocean = np.argwhere((mask <= 10) & (mask >= 1))
    pick = ocean[rng.integers(0, len(ocean), N_OBS)]
    obs = (rng.integers(0, NUM_DAYS, N_OBS), pick[:, 0], pick[:, 1], 0.3 * rng.random(N_OBS))
    eng = SnowBudgetEngine(mask, NUM_DAYS, DX, n_members=MEMBERS, atmlossInc=1)
    if sets:
        st = {k: np.stack([f[k], f[k]]) for k in ("precip", "conc", "wind", "drift")}
        eng.set_forcing_sets(st["precip"], st["conc"], st["wind"], st["drift"], np.zeros(MEMBERS, np.int32),
                             [NUM_DAYS, NUM_DAYS])
    else:
        eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
    return eng, params, ic, obs


def mixed_kinds(obs, seed=SEED + 1):
    rng = np.random.default_rng(seed)
    day, row, col, depth = obs
    kind = rng.integers(0, 3, len(day)).astype(np.int32)
    kind[(kind == 2) & (day == 0)] = 1
    value = np.where(kind == 2, 200.0 + 150.0 * rng.random(len(day)), depth)
    return day, row, col, value, kind, 10.0 ** rng.uniform(-3, 1, len(day))


def timed(eng, fn, reps=5):
    import torch
    fn()
    k0, best = eng.season_kernel_time()[0], None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return {"ms": best, "season_kernel_ms": (eng.season_kernel_time()[0] - k0) / reps}


def epilogue_ms(fn, reps=5):
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = sum(e.device_time_total for e in prof.key_averages() if "misfit_finish_kernel" in e.key)
    return tot / reps / 1000.0


def kernel_only(reps):
    import torch
    out = {"tree": ROOT}
    for name, sets in (("obs", False), ("sets_obs", True)):
        eng, params, ic, obs = headline(sets)
        if sets:
            eng.set_observations_sets(np.zeros(N_OBS, np.int32), *obs)
        else:
            eng.set_observations(obs)
        ic_t = torch.from_numpy(np.ascontiguousarray(ic)).cuda()
        eng.run_season_misfit(params, ic_t)
        k0 = eng.season_kernel_time()[0]
        for _ in range(reps):
            mis, _ = eng.run_season_misfit(params, ic_t)
        out[name + "_season_kernel_ms"] = (eng.season_kernel_time()[0] - k0) / reps
        out[name + "_misfit_sum"] = float(mis.sum().item())
        eng.close()
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--P", default="8,32,128")
    ap.add_argument("--kernel-only", action="store_true")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU mode")
    if args.kernel_only:
        return kernel_only(args.reps)
    from calibration_seasons_timing import Batch, gpu_identity, make_seasons
    from nesosim_b200 import synthetic as S
    result = {"gpu": gpu_identity(), "torch_device": torch.cuda.get_device_name(0),
              "workload": "%d members, 100 km season of %d days, %d observations" % (MEMBERS, NUM_DAYS, N_OBS),
              "timing": "CUDA events around the calls, warm-up then best of 5; season kernel: mean device time of 5; "
                        "epilogue: torch.profiler device time, mean of 5 (a run of its own)"}
    eng, params, ic, obs = headline()
    ic_t = torch.from_numpy(np.ascontiguousarray(ic)).cuda()
    eng.set_observations(obs)
    mis = eng.run_season_misfit(params, ic_t)[0]
    runs = {"misfit": lambda: eng.run_season_misfit(params, ic_t),
            "scores_depth": lambda: eng.run_season_scores(params, ic_t)}
    head = {k: timed(eng, fn) for k, fn in runs.items()}
    head["misfit"]["epilogue_ms"] = epilogue_ms(runs["misfit"])
    head["scores_depth"]["epilogue_ms"] = epilogue_ms(runs["scores_depth"])
    head["scores_depth_equals_misfit"] = bool(torch.equal(eng.run_season_scores(params, ic_t)[0][:, 0], mis))
    day, row, col, value, kind, sigma = mixed_kinds(obs)
    eng.set_observations_ex(day, row, col, value, kind, sigma)
    fn = lambda: eng.run_season_scores(params, ic_t, model=True)   # noqa: E731
    head["scores_mixed_model_row"] = timed(eng, fn)
    head["scores_mixed_model_row"]["epilogue_ms"] = epilogue_ms(fn)
    head["scores_mixed_model_row"]["used_member0"] = eng.run_season_scores(params, ic_t)[1][0].tolist()
    eng.close()
    result["headline"] = head
    print(json.dumps(head), flush=True)
    mask = S.region_mask(dx=DX)
    seasons = make_seasons(mask)
    result["batch_S11"] = []
    for P in (int(p) for p in args.P.split(",")):
        x = Batch(mask, seasons, S.ensemble_params(P, seed=P))
        row = {"P": P, "members": P * len(seasons),
               "misfit": timed(x.eng, lambda: x.eng.run_season_misfit(x.params, x.ic)),
               "scores_depth": timed(x.eng, lambda: x.eng.run_season_scores(x.params, x.ic))}
        row["scores_depth_equals_misfit"] = bool(torch.equal(x.eng.run_season_scores(x.params, x.ic)[0][:, 0],
                                                             x.eng.run_season_misfit(x.params, x.ic)[0]))
        x.close()
        result["batch_S11"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "observation_scores_timing.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
