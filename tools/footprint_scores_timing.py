"""Footprint-scores timing on the headline workload: 128 members, the 100 km season of bench.py (260 days), the 20 000
mixed-kind point observations of tools/observation_scores_timing.py, plus footprints:

  points  no footprints (nesosim_run_season_scores), for reference
  dense   every ocean region 1..10 x nine 30-day windows [1, 31) .. [241, 260) x depth and density: 180 footprints, every
          ocean cell observed on every day 1..259
  w99     region 8 x the months November..April (counted back from the season's last day, 30 April) x depth and density

For each: the call (nesosim_run_season_scores_fp) with CUDA events, warm-up then best of 5; the season kernel's device
time (nesosim_season_kernel_time, mean of 5); the epilogue's device time (footprint_mean_kernel and misfit_finish_kernel,
torch.profiler, a run of its own, mean of 5); the sample bytes per member; and the same scores through the HBM round
trip (run_season writing snowDepths and density, then ensemble.observation_scores / footprint_scores), timed the same
way, with the largest relative difference of the two.  Then the S = 11 batch of tools/calibration_seasons_timing.py at
P = 8 and 128 with W99-like footprints per season, against the same batch without footprints.

The GPU's name and power limit are read in the same run.
usage: python tools/footprint_scores_timing.py --out DIR [--P 8,128]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from observation_scores_timing import NUM_DAYS, headline, mixed_kinds, timed   # noqa: E402

MONTHS = (("nov", 30), ("dec", 31), ("jan", 31), ("feb", 28), ("mar", 31), ("apr", 30))


def w99_windows(days):
    """[d0, d1) of November..April, the season ending on the last day of April."""
    out, end = [], days
    for _, n in reversed(MONTHS):
        out.append((end - n, end))
        end -= n
    return out[::-1]


def footprint_sets(mask, days):
    from nesosim_b200 import ensemble as ENS
    from nesosim_b200._lib import OBS_DENSITY, OBS_DEPTH
    dense_win = [(1 + 30 * i, min(31 + 30 * i, days)) for i in range(9)]
    dense = [ENS.region_footprints(mask, [code], dense_win, k, 0.25 if k == OBS_DEPTH else 300.0,
                                   0.05 if k == OBS_DEPTH else 30.0)
             for code in range(1, 11) for k in (OBS_DEPTH, OBS_DENSITY)]
    w99 = [ENS.region_footprints(mask, [8], w99_windows(days), k, 0.25 if k == OBS_DEPTH else 300.0,
                                 0.05 if k == OBS_DEPTH else 30.0) for k in (OBS_DEPTH, OBS_DENSITY)]
    return {"dense": concat(dense), "w99": concat(w99)}


def concat(parts):
    from nesosim_b200 import ensemble as ENS
    return ENS.concat_footprints(parts)[0]


def sample_bytes(mask, obs, fps):
    """Bytes of one member's sample row: 16 B per distinct observed ocean (cell, day) plus one sentinel per ocean cell."""
    nx = mask.shape[1]
    ocean = (mask >= 1) & (mask <= 10)
    day = np.concatenate([obs[0], fps["day"] if fps else []]).astype(np.int64)
    row = np.concatenate([obs[1], fps["row"] if fps else []]).astype(np.int64)
    col = np.concatenate([obs[2], fps["col"] if fps else []]).astype(np.int64)
    keep = ocean[row, col]
    pairs = np.unique((row[keep] * nx + col[keep]) * 1000 + day[keep])
    return int(16 * (len(pairs) + ocean.sum()))


def device_ms(fn, names, reps=5):
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    return {n: sum(e.device_time_total for e in prof.key_averages() if n in e.key) / reps / 1000.0 for n in names}


def hbm_scores(eng, params, ic_t, obs, fps, mask):
    from nesosim_b200 import ensemble as ENS
    out = eng.run_season(params, ic_t, eng.alloc_outputs(names=("snowDepths", "density")))
    arrays = (out["snowDepths"], out["density"], eng._forcing[1])
    res = ENS.observation_scores(*arrays, obs, mask)
    if fps is not None:
        res = res + ENS.footprint_scores(*arrays, fps, mask)
    del out
    return res


def rel_diff(a, b):
    import torch
    a, b = a.double(), b.double()
    if not torch.equal(torch.isfinite(a), torch.isfinite(b)):
        return float("inf")                              # the finite entries differ: reported, not hidden
    ok = torch.isfinite(a)
    return float(((a[ok] - b[ok]).abs() / b[ok].abs().clamp_min(1e-300)).max().item()) if ok.any() else 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--P", default="8,128")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU mode")
    from calibration_seasons_timing import Batch, gpu_identity, make_seasons
    from nesosim_b200 import synthetic as S
    result = {"gpu": gpu_identity(), "torch_device": torch.cuda.get_device_name(0),
              "workload": "128 members, 100 km season of %d days, 20000 mixed-kind point observations" % NUM_DAYS,
              "timing": "CUDA events around the calls, warm-up then best of 5; season kernel: mean device time of 5; "
                        "epilogue kernels: torch.profiler device time, mean of 5 (a run of its own)"}
    eng, params, ic, obs4 = headline()
    mask = S.region_mask(dx=100000)
    day, row, col, value, kind, sigma = mixed_kinds(obs4)
    obs = {"day": day, "row": row, "col": col, "value": value, "kind": kind, "sigma": sigma}
    ic_t = torch.from_numpy(np.ascontiguousarray(ic)).cuda()
    head = {}
    for name, fps in [("points", None)] + sorted(footprint_sets(mask, NUM_DAYS).items()):
        if fps is None:
            eng.set_observations_ex(day, row, col, value, kind, sigma)
            fn = lambda: eng.run_season_scores(params, ic_t, model=True)        # noqa: E731
        else:
            eng.set_observations_fp(obs, fps)
            fn = lambda: eng.run_season_scores_fp(params, ic_t, model=True)     # noqa: E731
        r = timed(eng, fn)
        r.update(device_ms(fn, ("footprint_mean_kernel", "misfit_finish_kernel")))
        r["footprints"] = 0 if fps is None else len(fps["value"])
        r["footprint_points"] = 0 if fps is None else len(fps["day"])
        r["sample_bytes_per_member"] = sample_bytes(mask, obs4, fps)
        fused_res = [t.clone() for t in fn() if t is not None]
        r["hbm_round_trip"] = timed(eng, lambda: hbm_scores(eng, params, ic_t, obs, fps, mask))
        hbm = hbm_scores(eng, params, ic_t, obs, fps, mask)
        order = (0, 1, 2) if fps is None else (0, 1, 2, 3, 4, 5)
        r["fused_vs_hbm_max_rel_diff"] = max(rel_diff(fused_res[i], hbm[i]) for i in order)
        if fps is not None:
            r["fp_used_member0"] = fused_res[4][0].tolist()
        head[name] = r
        print(name, json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    eng.close()
    result["headline"] = head
    seasons = make_seasons(mask)
    result["batch_S11"] = []
    for P in (int(p) for p in args.P.split(",")):
        x = Batch(mask, seasons, S.ensemble_params(P, seed=P))
        row_ = {"P": P, "members": P * len(seasons), "points_only": timed(x.eng, lambda: x.eng.run_season_misfit(x.params, x.ic))}
        sets = np.repeat(np.arange(len(seasons), dtype=np.int32), [len(s["obs"][0]) for s in seasons])
        pts = {"day": np.concatenate([s["obs"][0] for s in seasons]), "row": np.concatenate([s["obs"][1] for s in seasons]),
               "col": np.concatenate([s["obs"][2] for s in seasons]), "value": np.concatenate([s["obs"][3] for s in seasons]),
               "kind": np.zeros(len(sets), np.int32), "sigma": np.ones(len(sets))}
        fps = [footprint_sets(mask, s["days"])["w99"] for s in seasons]
        fp_set = np.repeat(np.arange(len(seasons), dtype=np.int32), [len(f["value"]) for f in fps])
        x.eng.set_observations_fp(pts, concat(fps), obs_set=sets, fp_set=fp_set)
        row_["w99_footprints"] = timed(x.eng, lambda: x.eng.run_season_scores_fp(x.params, x.ic))
        x.close()
        result["batch_S11"].append(row_)
        print(json.dumps(row_), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "footprint_scores_timing.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
