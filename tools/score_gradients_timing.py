"""Cost of the calibration gradients (nesosim_run_season_score_grads, the tangent build of the scoring day kernel)
against the scores call and against finite differences through extra members, on the general day-kernel path:
260-day seasons, 20 000 mixed-kind point observations and W99-like footprints (tools/general_scores_timing.py), at
100 km with M = 128, 50 km and 25 km with M = 16 and 64.

Arms, each timed with CUDA events, warm-up then best of 5:
  scores   nesosim_run_season_scores_fp, M members (model rows);
  grad     nesosim_run_season_score_grads, M members (model rows, gradients and Jacobian rows);
  forward  one scores call of 4M members (every parameter set and its three forward steps);
  central  one scores call of 7M members (every parameter set and its six central steps), where it fits.
The steps are 1e-4 of each parameter.  Agreement: the gradient of chi2 (points and footprints, per kind and direction)
against the forward and central differences of the difference arms, as the largest |grad - fd| over the largest
|grad| of the same kind and direction -- over every member, and over the members whose counts of finite terms are the
same at every step of the arm.  A term that appears or drops out between two steps (a density observation whose
h0 + h1 crosses minSnowD, a depth observation whose concentration crosses zero) is a jump of chi2 that no difference
quotient follows; "members_with_count_changes" says how many members had one.  The GPU's name and power limit are read
in the same run.
usage: python tools/score_gradients_timing.py --out DIR"""
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

STEP = 1e-4
WORKLOADS = ((100, 128), (50, 16), (50, 64), (25, 16), (25, 64))


def stepped(params, n_side):
    """[base; base with column c scaled by (1 + s*STEP) for c in GRAD_PARAMS, s in sides] per parameter set, member-major
    blocks: rows [k*M:(k+1)*M] are step k (k = 0 the base)."""
    from nesosim_b200 import _lib
    blocks = [params]
    for c in _lib.GRAD_PARAMS:
        for s in ((1,) if n_side == 1 else (1, -1)):
            b = params.copy()
            b[:, c] *= 1 + s * STEP
            blocks.append(b)
    return np.concatenate(blocks)


KIND_NAMES = ("depth", "volume", "density", "fp_depth", "fp_volume", "fp_density")


def agreement(grad, fd, members):
    """Per kind (points, then footprints): the largest |grad - fd| over the largest |grad| of the same kind and direction,
    over the given members ([DIRS] per kind; None where the kind has no non-zero gradient)."""
    out = {}
    for k, name in enumerate(KIND_NAMES):
        g, d = grad[members, k], fd[members, k]
        scale = np.abs(g).max(axis=0) if len(g) else np.zeros(grad.shape[-1])
        if not (scale > 0).any():
            out[name] = None
            continue
        out[name] = [float(x) for x in np.abs(g - d).max(axis=0) / np.where(scale > 0, scale, 1.0)]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU mode")
    from calibration_seasons_timing import gpu_identity
    from nesosim_b200 import _lib
    from nesosim_b200 import synthetic as S
    result = {"gpu": gpu_identity(), "torch_device": torch.cuda.get_device_name(0),
              "workload": "%d-day seasons, 20000 mixed-kind point observations, W99-like footprints (region 8, Nov-Apr, "
                          "depth and density), atmlossInc=1, general day-kernel path" % NUM_DAYS,
              "timing": "CUDA events around each call, warm-up then best of 5",
              "arms": {"scores_ms": "nesosim_run_season_scores_fp, M members", "grad_ms":
                       "nesosim_run_season_score_grads, M members, with model and Jacobian rows",
                       "forward_ms": "nesosim_run_season_scores_fp, 4M members", "central_ms":
                       "nesosim_run_season_scores_fp, 7M members"},
              "agreement": "per kind, max |grad - fd| / max |grad| per direction (windPackFactor, leadLossFactor, "
                           "atmLossFactor), over all members and over the members whose finite-term counts are the same "
                           "at every step of the arm; relative step %g" % STEP,
              "points": []}
    rng = np.random.default_rng(SEED)
    for km, M in WORKLOADS:
        mask, dx = S.region_mask(dx=km * 1000), km * 1000
        forcing = S.make_season(mask, NUM_DAYS, seed=SEED + km)
        obs, fps = mixed_points(mask, rng), footprint_sets(mask, NUM_DAYS)["w99"]
        params = S.ensemble_params(M, seed=M)
        ic = torch.from_numpy(np.ascontiguousarray(S.make_ic(mask, seed=SEED))).cuda()
        r = {"grid_km": km, "shape": list(mask.shape), "M": M}
        eng = engine(mask, dx, M, forcing, "general")
        eng.set_observations_fp(obs, fps)
        r["scores_ms"] = best_of(lambda: eng.run_season_scores_fp(params, ic, model=True))
        r["grad_ms"] = best_of(lambda: eng.run_season_score_grads(params, ic, model=True, jac=True))
        g = eng.run_season_score_grads(params, ic, model=True, jac=True)
        grad = np.concatenate([g["grad"].cpu().numpy(), g["fp_grad"].cpu().numpy()], axis=1)   # [M, 2*KINDS, DIRS]
        eng.close()
        torch.cuda.empty_cache()
        for arm, sides, n in (("forward", 1, 4), ("central", 2, 7)):
            free = torch.cuda.mem_get_info()[0]
            need = n * M * (32 * mask.size + 16 * (len(obs["day"]) + len(fps["day"])))
            if need > 0.8 * free:
                r[arm + "_ms"] = "skipped: %.1f GB needed, %.1f GB free" % (need / 1e9, free / 1e9)
                continue
            p = stepped(params, sides)
            eng = engine(mask, dx, n * M, forcing, "general")
            eng.set_observations_fp(obs, fps)
            r[arm + "_ms"] = best_of(lambda: eng.run_season_scores_fp(p, ic))
            res = eng.run_season_scores_fp(p, ic)
            chi2 = np.concatenate([res[0].cpu().numpy(), res[3].cpu().numpy()], axis=1).reshape(n, M, -1)
            used = np.concatenate([res[1].cpu().numpy(), res[4].cpu().numpy()], axis=1).reshape(n, M, -1)
            same_counts = (used == used[0]).all(axis=(0, 2))
            eng.close()
            fd = np.empty_like(grad)
            for j, c in enumerate(_lib.GRAD_PARAMS):
                h = STEP * params[:, c][:, None]
                if sides == 1:
                    fd[:, :, j] = (chi2[1 + j] - chi2[0]) / h
                else:
                    fd[:, :, j] = (chi2[1 + 2 * j] - chi2[2 + 2 * j]) / (2 * h)
            r[arm + "_agreement"] = agreement(grad, fd, np.arange(M))
            r[arm + "_agreement_same_counts"] = agreement(grad, fd, np.flatnonzero(same_counts))
            r[arm + "_members_with_count_changes"] = int(M - same_counts.sum())
            torch.cuda.empty_cache()
        r["grad_over_scores"] = r["grad_ms"] / r["scores_ms"]
        if isinstance(r.get("forward_ms"), float):
            r["grad_over_forward"] = r["grad_ms"] / r["forward_ms"]
        result["points"].append(r)
        print(json.dumps(r), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "score_gradients_timing.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
