"""Fused calibration scores on the general day-kernel path (nesosim_set_path(ctx, 1), day_step_score_kernel) against the
HBM round trip, on grids the season kernel does not take: 260-day seasons at 50 km (synthetic.region_mask(dx=50000))
and 25 km (the bundled coastline), M in {16, 64, 128}, 20 000 mixed-kind point observations plus W99-like footprints
(region 8, November..April, depth and density; tools/footprint_scores_timing.py).

For each point: the fused call (nesosim_run_season_scores_fp) with CUDA events, warm-up then best of 5; the same scores
through the HBM round trip (run_season writing snowDepths and density, then ensemble.observation_scores /
footprint_scores), timed the same way, with the largest relative difference of the two and whether their counts agree;
the device bytes per member each arm needs, computed from shapes (an HBM point that would not fit in the free device
memory is skipped, never tried); and, in a torch.profiler run of its own, the scoring day kernel's device time per day.
Then 100 km, M = 128: the general path against the season kernel (both fused), with a bit-identity check.

The GPU's name and power limit are read in the same run.
usage: python tools/general_scores_timing.py --out DIR [--M 16,64,128] [--grids 50,25]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from footprint_scores_timing import device_ms, footprint_sets, hbm_scores, rel_diff   # noqa: E402

NUM_DAYS, N_OBS, SEED = 260, 20000, 606
NVAR = 12


def best_of(fn, reps=5):
    import torch
    fn()
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return best


def mixed_points(mask, rng):
    """N_OBS point observations of the three kinds, anywhere on the grid (land ones are dropped), any day."""
    ny, nx = mask.shape
    day, row, col = rng.integers(0, NUM_DAYS, N_OBS), rng.integers(0, ny, N_OBS), rng.integers(0, nx, N_OBS)
    kind = rng.integers(0, 3, N_OBS).astype(np.int32)
    kind[(kind == 2) & (day == 0)] = 1
    value = np.where(kind == 2, 200.0 + 150.0 * rng.random(N_OBS), 0.3 * rng.random(N_OBS))
    return {"day": day, "row": row, "col": col, "value": value, "kind": kind, "sigma": 10.0 ** rng.uniform(-3, 1, N_OBS)}


def sample_slots(mask, obs, fps):
    """Distinct observed ocean (cell, day) pairs plus one sentinel per ocean cell: a member's sample row."""
    nx = mask.shape[1]
    ocean = (mask >= 1) & (mask <= 10)
    day = np.concatenate([obs["day"], fps["day"]]).astype(np.int64)
    row = np.concatenate([obs["row"], fps["row"]]).astype(np.int64)
    col = np.concatenate([obs["col"], fps["col"]]).astype(np.int64)
    keep = ocean[row, col]
    return len(np.unique((row[keep] * nx + col[keep]) * NUM_DAYS + day[keep])) + int(ocean.sum())


def engine(mask, dx, M, forcing, path):
    from nesosim_b200.engine import SnowBudgetEngine
    eng = SnowBudgetEngine(mask, NUM_DAYS, dx, n_members=M, atmlossInc=1)
    eng.set_forcing(forcing["precip"], forcing["conc"], forcing["wind"], forcing["drift"])
    if path != "auto":
        eng.set_path(path)
    return eng


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--M", default="16,64,128")
    ap.add_argument("--grids", default="50,25")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU mode")
    from calibration_seasons_timing import gpu_identity
    from nesosim_b200 import synthetic as S
    result = {"gpu": gpu_identity(), "torch_device": torch.cuda.get_device_name(0),
              "workload": "%d-day seasons, %d mixed-kind point observations, W99-like footprints (region 8, Nov-Apr, "
                          "depth and density), atmlossInc=1" % (NUM_DAYS, N_OBS),
              "timing": "CUDA events around the calls, warm-up then best of 5; scoring day kernel: torch.profiler device "
                        "time, mean of 5 calls (a run of its own) / (T-1)",
              "bytes": "per member, from shapes: general = depth ring 32 B per cell + 16 B per sample slot; HBM = "
                       "snowDepths and density 24 B per cell-day + the day kernel's two-slot scratch of all twelve "
                       "arrays (192 B per cell) + about twelve float64 torch temporaries per observation and footprint "
                       "point (96 B each)",
              "points": []}
    rng = np.random.default_rng(SEED)
    for km in (int(g) for g in args.grids.split(",")):
        mask, dx = S.region_mask(dx=km * 1000), km * 1000
        forcing = S.make_season(mask, NUM_DAYS, seed=SEED + km)
        obs, fps = mixed_points(mask, rng), footprint_sets(mask, NUM_DAYS)["w99"]
        plane = mask.size
        slots = sample_slots(mask, obs, fps)
        general_b = 32 * plane + 16 * slots
        hbm_b = 24 * NUM_DAYS * plane + 2 * NVAR * 8 * plane + 96 * (len(obs["day"]) + len(fps["day"]))
        for M in (int(m) for m in args.M.split(",")):
            params = S.ensemble_params(M, seed=M)
            ic = torch.from_numpy(np.ascontiguousarray(S.make_ic(mask, seed=SEED))).cuda()
            r = {"grid_km": km, "shape": list(mask.shape), "M": M, "general_bytes_per_member": general_b,
                 "hbm_bytes_per_member": hbm_b}
            eng = engine(mask, dx, M, forcing, "general")
            eng.set_observations_fp(obs, fps)
            fn = lambda: eng.run_season_scores_fp(params, ic, model=True)      # noqa: E731
            r["general_fused_ms"] = best_of(fn)
            fused_res = [t.clone() for t in fn()]
            dm = device_ms(fn, ("day_step_score_kernel", "footprint_mean_kernel", "misfit_finish_kernel"))
            r["score_day_kernel_us_per_day"] = 1000.0 * dm["day_step_score_kernel"] / (NUM_DAYS - 1)
            r["epilogue_ms"] = dm["footprint_mean_kernel"] + dm["misfit_finish_kernel"]
            eng.close()
            torch.cuda.empty_cache()
            free = torch.cuda.mem_get_info()[0]
            if M * hbm_b > 0.8 * free:
                r["hbm_round_trip_ms"] = "skipped: %.1f GB needed, %.1f GB free" % (M * hbm_b / 1e9, free / 1e9)
            else:
                eng = engine(mask, dx, M, forcing, "auto")
                r["hbm_round_trip_ms"] = best_of(lambda: hbm_scores(eng, params, ic, obs, fps, mask))
                hbm = hbm_scores(eng, params, ic, obs, fps, mask)
                r["fused_vs_hbm_max_rel_diff"] = max(rel_diff(fused_res[i], hbm[i]) for i in (0, 2, 3, 5))
                r["fused_vs_hbm_counts_equal"] = bool(torch.equal(fused_res[1], hbm[1].to(fused_res[1].dtype))
                                                      and torch.equal(fused_res[4], hbm[4].to(fused_res[4].dtype)))
                r["speedup"] = r["hbm_round_trip_ms"] / r["general_fused_ms"]
                del hbm
                eng.close()
            result["points"].append(r)
            print(json.dumps(r), flush=True)
            torch.cuda.empty_cache()
    # 100 km, M = 128: the general path against the season kernel, both fused
    mask, dx, M = S.region_mask(dx=100000), 100000, 128
    forcing = S.make_season(mask, NUM_DAYS, seed=SEED + 100)
    obs, fps = mixed_points(mask, rng), footprint_sets(mask, NUM_DAYS)["w99"]
    params = S.ensemble_params(M, seed=M)
    ic = torch.from_numpy(np.ascontiguousarray(S.make_ic(mask, seed=SEED))).cuda()
    r, res = {"grid_km": 100, "shape": list(mask.shape), "M": M}, {}
    for path in ("auto", "general"):
        eng = engine(mask, dx, M, forcing, path)
        eng.set_observations_fp(obs, fps)
        fn = lambda: eng.run_season_scores_fp(params, ic, model=True)          # noqa: E731
        r[("season_kernel" if path == "auto" else "general") + "_fused_ms"] = best_of(fn)
        res[path] = [t.clone() for t in fn()]
        if path == "general":
            dm = device_ms(fn, ("day_step_score_kernel",))
            r["score_day_kernel_us_per_day"] = 1000.0 * dm["day_step_score_kernel"] / (NUM_DAYS - 1)
        eng.close()
    r["bit_identical"] = all(torch.equal(a.nan_to_num(7.5), b.nan_to_num(7.5)) and
                             torch.equal(torch.isnan(a), torch.isnan(b)) for a, b in zip(res["auto"], res["general"]))
    result["season_kernel_100km"] = r
    print(json.dumps(r), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "general_scores_timing.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
