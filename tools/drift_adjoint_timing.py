"""Cost of the calibration adjoint with respect to the ice drift (nesosim_run_season_score_adjoint_drift) against the
plain and the forcing adjoint calls, on the r08 workload (tools/score_adjoint_timing.py): 260-day seasons, 20 000
mixed-kind point observations and W99-like footprints, at 100 km with M = 128, 50 km and 25 km with M = 16 and 64.

Arms, each timed with CUDA events, warm-up then best of 5:
  adjoint        nesosim_run_season_score_adjoint, M members (model rows), all weights 1;
  forcing        nesosim_run_season_score_adjoint_forcing with the scale fields and totals only;
  drift          nesosim_run_season_score_adjoint_drift with the drift scale fields and totals only;
  forcing_drift  nesosim_run_season_score_adjoint_drift with both scale pairs (one sweep for snowfall and drift);
  drift_days     the drift arm with the per-day drift planes.
Per point also: the per-kernel device times of one call of each arm from torch.profiler in a separate pass, and
drift_scale_total[:, 0] + [:, 1] (dJ/d of one drift speed factor) against central differences of scores calls on the
drift scaled by 1 +- 1e-4 (J = the sum of chi2 and fp_chi2), over all members and over the members whose counts of
finite terms do not change between the two steps.  The GPU's name and power limit are read in the same run.
usage: python tools/drift_adjoint_timing.py --out DIR"""

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from footprint_scores_timing import footprint_sets                      # noqa: E402
from general_scores_timing import NUM_DAYS, SEED, best_of, engine, mixed_points   # noqa: E402
from score_adjoint_timing import WORKLOADS, kernel_times                 # noqa: E402

H = 1e-4


def objective(eng, params, ic):
    chi2, used, _, fchi2, fused, _ = eng.run_season_scores_fp(params, ic)
    return (chi2.sum(dim=1) + fchi2.sum(dim=1)).cpu().numpy(), np.concatenate([used.cpu().numpy(), fused.cpu().numpy()], 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sizes", default="all", help="'all' or a comma list of km:M, e.g. 100:128,25:16")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU mode")
    from calibration_seasons_timing import gpu_identity
    from nesosim_b200 import synthetic as S
    work = WORKLOADS if args.sizes == "all" else tuple(tuple(int(v) for v in s.split(":")) for s in args.sizes.split(","))
    result = {"gpu": gpu_identity(), "torch_device": torch.cuda.get_device_name(0),
              "workload": "%d-day seasons, 20000 mixed-kind point observations, W99-like footprints (region 8, Nov-Apr, "
                          "depth and density), atmlossInc=1, general day-kernel path" % NUM_DAYS,
              "timing": "CUDA events around each call, warm-up then best of 5; kernel times from torch.profiler in a "
                        "separate pass",
              "arms": {"adjoint_ms": "nesosim_run_season_score_adjoint, M members, weights 1",
                       "forcing_ms": "nesosim_run_season_score_adjoint_forcing, scale fields and totals only",
                       "drift_ms": "nesosim_run_season_score_adjoint_drift, drift scale fields and totals only",
                       "forcing_drift_ms": "nesosim_run_season_score_adjoint_drift with both scale pairs",
                       "drift_days_ms": "the drift arm with the per-day drift planes"},
              "points": []}
    rng = np.random.default_rng(SEED)
    for km, M in work:
        mask, dx = S.region_mask(dx=km * 1000), km * 1000
        forcing = S.make_season(mask, NUM_DAYS, seed=SEED + km)
        obs, fps = mixed_points(mask, rng), footprint_sets(mask, NUM_DAYS)["w99"]
        params = S.ensemble_params(M, seed=M)
        ic = torch.from_numpy(np.ascontiguousarray(S.make_ic(mask, seed=SEED))).cuda()
        r = {"grid_km": km, "shape": list(mask.shape), "M": M,
             "adjoint_state_bytes": int((17 * NUM_DAYS + 56) * M * mask.size),
             "drift_state_bytes": int((17 * NUM_DAYS + 72) * M * mask.size),
             "drift_day_bytes": int(16 * NUM_DAYS * M * mask.size)}
        eng = engine(mask, dx, M, forcing, "general")
        eng.set_observations_fp(obs, fps)
        arms = {"adjoint": lambda: eng.run_season_score_adjoint(params, ic, model=True),
                "forcing": lambda: eng.run_season_score_adjoint(params, ic, model=True, forcing=True),
                "drift": lambda: eng.run_season_score_adjoint(params, ic, model=True, drift=True),
                "forcing_drift": lambda: eng.run_season_score_adjoint(params, ic, model=True, forcing=True, drift=True),
                "drift_days": lambda: eng.run_season_score_adjoint(params, ic, model=True, drift=True, drift_days=True)}
        for name, fn in arms.items():
            r[name + "_ms"] = best_of(fn)
        a, b, c = arms["adjoint"](), arms["drift"](), arms["forcing_drift"]()
        r["existing_outputs_identical"] = all(torch.equal(a[k], b[k]) and torch.equal(a[k], c[k])
                                              for k in ("chi2", "used", "theta_grad", "ic_grad"))
        r["drift_outputs_identical_with_forcing"] = all(torch.equal(b[k], c[k]) for k in ("drift_scale_grad",
                                                                                         "drift_scale_total"))
        total = b["drift_scale_total"].sum(dim=1).cpu().numpy()
        for name, fn in arms.items():
            r[name + "_kernels"] = kernel_times(fn)
        eng.close()
        del a, b, c
        torch.cuda.empty_cache()
        vals, counts = [], []
        for sg in (1, -1):
            fc = dict(forcing)
            fc["drift"] = forcing["drift"] * (1.0 + sg * H)
            e = engine(mask, dx, M, fc, "general")
            e.set_observations_fp(obs, fps)
            v, cnt = objective(e, params, ic)
            vals.append(v)
            counts.append(cnt)
            e.close()
        fd = (vals[0] - vals[1]) / (2 * H)
        rel = np.abs(total - fd) / np.abs(fd)
        steady = (counts[0] == counts[1]).all(axis=1)
        r["drift_total_vs_central_difference"] = {
            "h": H, "max_rel_all": float(rel.max()), "median_rel_all": float(np.median(rel)),
            "max_rel_steady_counts": float(rel[steady].max()) if steady.any() else None,
            "members_with_changed_counts": int((~steady).sum())}
        for name in ("forcing", "drift", "forcing_drift", "drift_days"):
            r[name + "_over_adjoint"] = r[name + "_ms"] / r["adjoint_ms"]
        torch.cuda.empty_cache()
        result["points"].append(r)
        print(json.dumps({k: v for k, v in r.items() if not k.endswith("_kernels")}), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "drift_adjoint_timing.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
