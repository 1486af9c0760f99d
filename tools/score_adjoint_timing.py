"""Cost of the calibration adjoint (nesosim_run_season_score_adjoint: the record build, the seeds, the backward day
kernel and the finish) against the scores call and the forward-mode gradient call, on the general day-kernel path: the
r07 workload (tools/score_gradients_timing.py) -- 260-day seasons, 20 000 mixed-kind point observations and W99-like
footprints, at 100 km with M = 128, 50 km and 25 km with M = 16 and 64.

Arms, each timed with CUDA events, warm-up then best of 5:
  scores   nesosim_run_season_scores_fp, M members (model rows);
  grad     nesosim_run_season_score_grads, M members (model rows);
  adjoint  nesosim_run_season_score_adjoint, M members (model rows), all weights 1.
Per arm point also: the adjoint state's device bytes (by the header's formula), the per-kernel device times of one
adjoint call from torch.profiler in a separate pass (record day kernel, seeds, backward day kernel, finish, ...), and the
agreement of the adjoint's theta_grad with sum_k grad[k] + sum_k fp_grad[k] of the forward mode, as the largest
|difference| over the member's largest component.  The GPU's name and power limit are read in the same run.
usage: python tools/score_adjoint_timing.py --out DIR"""
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

WORKLOADS = ((100, 128), (50, 16), (50, 64), (25, 16), (25, 64))


def kernel_times(fn):
    """Device time per kernel name (ms summed over one call) from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            out[e.key] = {"ms": t / 1000.0, "calls": e.count}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms"]))


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
              "arms": {"scores_ms": "nesosim_run_season_scores_fp, M members", "grad_ms":
                       "nesosim_run_season_score_grads, M members", "adjoint_ms":
                       "nesosim_run_season_score_adjoint, M members, weights 1"},
              "points": []}
    rng = np.random.default_rng(SEED)
    for km, M in work:
        mask, dx = S.region_mask(dx=km * 1000), km * 1000
        forcing = S.make_season(mask, NUM_DAYS, seed=SEED + km)
        obs, fps = mixed_points(mask, rng), footprint_sets(mask, NUM_DAYS)["w99"]
        params = S.ensemble_params(M, seed=M)
        ic = torch.from_numpy(np.ascontiguousarray(S.make_ic(mask, seed=SEED))).cuda()
        r = {"grid_km": km, "shape": list(mask.shape), "M": M}
        eng = engine(mask, dx, M, forcing, "general")
        eng.set_observations_fp(obs, fps)
        r["adjoint_state_bytes"] = int((17 * NUM_DAYS + 56) * M * mask.size)
        r["scores_ms"] = best_of(lambda: eng.run_season_scores_fp(params, ic, model=True))
        r["grad_ms"] = best_of(lambda: eng.run_season_score_grads(params, ic, model=True))
        r["adjoint_ms"] = best_of(lambda: eng.run_season_score_adjoint(params, ic, model=True))
        g = eng.run_season_score_grads(params, ic)
        want = (g["grad"].sum(dim=1) + g["fp_grad"].sum(dim=1)).cpu().numpy()
        a = eng.run_season_score_adjoint(params, ic)
        got = a["theta_grad"].cpu().numpy()
        r["theta_grad_vs_forward_max_rel"] = float((np.abs(got - want).max(axis=1) / np.abs(want).max(axis=1)).max())
        r["adjoint_kernels"] = kernel_times(lambda: eng.run_season_score_adjoint(params, ic, model=True))
        r["grad_kernels"] = kernel_times(lambda: eng.run_season_score_grads(params, ic, model=True))
        eng.close()
        torch.cuda.empty_cache()
        r["adjoint_over_scores"] = r["adjoint_ms"] / r["scores_ms"]
        r["adjoint_over_grad"] = r["adjoint_ms"] / r["grad_ms"]
        result["points"].append(r)
        print(json.dumps({k: v for k, v in r.items() if not k.endswith("_kernels")}), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "score_adjoint_timing.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
