"""Multi-season calibration timing: P parameter sets scored on S = 11 observed 100 km seasons (start years 2008-2018,
242/243 days, one seed per year, 2000 observations per season on ocean cells on days of March-April).

  (a) fused batch: one context of P*S members on forcing sets, one nesosim_run_season_misfit; members season-major
      (what ensemble.run_calibration stages), and parameter-major for comparison (clusters running at the same time
      then work on different seasons, so the seasons' pre-digested forcing no longer shares L2)
  (b) per-season loop: one single-forcing context of P members per season, one nesosim_run_season_misfit each, summed

Both are timed with CUDA events around the calls (every call ends in a stream synchronise), after a warm-up, best of 5;
the season kernel's own device time per call (nesosim_season_kernel_time, mean of the 5) is recorded beside it.  A third
measurement isolates the kernel instantiations: P*S members on ONE season, through a single-forcing context (the OBS
kernel) and through a forcing-sets context whose members all use set 0 (the SETS && OBS kernel).
The working set (forcing of 11 seasons, ~0.5 GB) is larger than L2.  The JSON also says whether (a) and (b) give
bit-identical misfit[P,S] -- with the cluster size each picks by itself, and with both pinned to the same size
(--cluster, the same strips for both) -- and the GPU's name and power limit, read in the same run.

usage: python tools/calibration_seasons_timing.py --out DIR [--P 8,32,128] [--cluster 8]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

DX = 100000
YEARS = list(range(2008, 2019))
N_OBS = 2000


def season_days(year):
    """Sep 1 of `year` .. Apr 30 of the next year (run_oneseason): 243 days when February has 29."""
    y = year + 1
    return 243 if (y % 4 == 0 and (y % 100 != 0 or y % 400 == 0)) else 242


def make_seasons(mask):
    from nesosim_b200 import synthetic as S
    ocean = np.argwhere((mask >= 1) & (mask <= 10))
    seasons = []
    for year in YEARS:
        d = season_days(year)
        rng = np.random.default_rng(year)
        cells = ocean[rng.integers(0, len(ocean), N_OBS)]
        march1 = d - 61                                  # March and April are the last 61 days of the season
        obs = (rng.integers(march1, d, N_OBS), cells[:, 0], cells[:, 1], 0.4 * rng.random(N_OBS))
        seasons.append({"days": d, "forcing": S.make_season(mask, d, seed=year), "ic": S.make_ic(mask, seed=year),
                        "obs": obs})
    return seasons


def gpu_identity():
    try:
        txt = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=30).stdout.strip()
    except Exception as e:                               # noqa: BLE001 -- recorded, not fatal
        txt = "nvidia-smi unavailable: %s" % e
    return txt.splitlines()


class Batch:
    """(a): one context, P*S members (season-major: member s*P + p, or parameter-major: p*S + s), forcing sets of the
    longest season."""

    def __init__(self, mask, seasons, params, season_major=True):
        from nesosim_b200.engine import SnowBudgetEngine
        P, S = len(params), len(seasons)
        T = max(s["days"] for s in seasons)
        stack = {}
        for k in ("precip", "conc", "wind", "drift"):
            a = np.zeros((S, T) + seasons[0]["forcing"][k].shape[1:])
            for i, s in enumerate(seasons):
                a[i, :s["days"]] = s["forcing"][k]
            stack[k] = a
        if season_major:
            member_set = np.repeat(np.arange(S, dtype=np.int32), P)
            self.params = np.tile(params, (S, 1))
        else:
            member_set = np.tile(np.arange(S, dtype=np.int32), P)
            self.params = np.repeat(params, S, axis=0)
        self.eng = SnowBudgetEngine(mask, T, DX, n_members=P * S, atmlossInc=1)
        self.eng.set_forcing_sets(stack["precip"], stack["conc"], stack["wind"], stack["drift"], member_set,
                                  [s["days"] for s in seasons])
        tag = np.concatenate([np.full(N_OBS, i, dtype=np.int32) for i in range(S)])
        self.eng.set_observations_sets(tag, *(np.concatenate([s["obs"][j] for s in seasons]) for j in range(4)))
        import torch
        # per-member ICs staged on the device once, as the forcing is (not a host upload inside every timed call)
        self.ic = torch.from_numpy(np.stack([seasons[i]["ic"] for i in member_set])).cuda()
        self.P, self.S, self.season_major = P, S, season_major

    def run(self):
        mis, used = self.eng.run_season_misfit(self.params, self.ic)
        if self.season_major:
            return mis.view(self.S, self.P).T, used.view(self.S, self.P).T
        return mis.view(self.P, self.S), used.view(self.P, self.S)

    def close(self):
        self.eng.close()


class Loop:
    """(b): one single-forcing context of P members per season."""

    def __init__(self, mask, seasons, params):
        import torch
        from nesosim_b200.engine import SnowBudgetEngine
        self.engs = []
        for s in seasons:
            e = SnowBudgetEngine(mask, s["days"], DX, n_members=len(params), atmlossInc=1)
            f = s["forcing"]
            e.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
            e.set_observations(s["obs"])
            self.engs.append((e, torch.from_numpy(np.ascontiguousarray(s["ic"], dtype=np.float64)).cuda()))
        self.params = params

    def run(self):
        import torch
        outs = [e.run_season_misfit(self.params, ic) for e, ic in self.engs]
        return torch.stack([o[0] for o in outs], dim=1), torch.stack([o[1] for o in outs], dim=1)

    def close(self):
        for e, _ in self.engs:
            e.close()


def engines(x):
    return [x.eng] if isinstance(x, Batch) else [e for e, _ in x.engs]


def launches(x):
    return sum(e.launch_count() for e in engines(x))


def kernel_ms(x):
    return sum(e.season_kernel_time()[0] for e in engines(x))


def timed(x, reps=5):
    import torch
    x.run()                                              # warm-up: module load, pre-pass buffers, the shapes timed below
    best, res = None, None
    k0 = kernel_ms(x)
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = launches(x)
        e0.record()
        res = x.run()
        e1.record()
        torch.cuda.synchronize()
        n = launches(x) - l0
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return best, n, (kernel_ms(x) - k0) / reps, tuple(r.cpu().numpy() for r in res)


class OneSeason(Batch):
    """P*S members on the first season only: through a single-forcing context (sets=False, the OBS kernel) or a
    forcing-sets context of two copies of the season, every member on set 0 (sets=True, the SETS && OBS kernel)."""

    def __init__(self, mask, seasons, params, sets):
        from nesosim_b200.engine import SnowBudgetEngine
        s0 = seasons[0]
        f, d, M = s0["forcing"], s0["days"], len(params)
        self.eng = SnowBudgetEngine(mask, d, DX, n_members=M, atmlossInc=1)
        if sets:
            st = {k: np.stack([f[k], f[k]]) for k in ("precip", "conc", "wind", "drift")}
            self.eng.set_forcing_sets(st["precip"], st["conc"], st["wind"], st["drift"], np.zeros(M, np.int32), [d, d])
            self.eng.set_observations_sets(np.zeros(N_OBS, np.int32), *s0["obs"])
        else:
            self.eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
            self.eng.set_observations(s0["obs"])
        import torch
        self.params, self.ic = params, torch.from_numpy(np.ascontiguousarray(s0["ic"], dtype=np.float64)).cuda()

    def run(self):
        return self.eng.run_season_misfit(self.params, self.ic)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--P", default="8,32,128")
    ap.add_argument("--cluster", default="8", help="cluster size pinned for the same-strips identity check")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU mode")
    from nesosim_b200 import build
    build.build(verbose=False)
    from nesosim_b200 import synthetic as S
    mask = S.region_mask(dx=DX)
    seasons = make_seasons(mask)
    cell_days = sum(s["days"] - 1 for s in seasons) * mask.size
    result = {"gpu": gpu_identity(), "torch_device": torch.cuda.get_device_name(0), "grid": list(mask.shape),
              "seasons": {str(y): s["days"] for y, s in zip(YEARS, seasons)}, "obs_per_season": N_OBS,
              "timing": "CUDA events around the calls, warm-up then best of 5", "runs": []}
    for P in (int(p) for p in args.P.split(",")):
        params = S.ensemble_params(P, seed=P)
        row = {"P": P, "S": len(seasons), "members": P * len(seasons)}
        os.environ.pop("NESOSIM_ENS_CLUSTER", None)
        runs = {}
        for name, mk in (("fused", Batch), ("loop", Loop), ("fused_parameter_major", lambda *a: Batch(*a, season_major=False))):
            x = mk(mask, seasons, params)
            ms, n, kms, res = timed(x)
            x.close()
            runs[name] = res
            row[name] = {"ms": ms, "launches_per_call": n, "season_kernel_ms": kms,
                         "member_cell_days_per_s": P * cell_days / (ms * 1e-3)}
        row["speedup_fused_over_loop"] = row["loop"]["ms"] / row["fused"]["ms"]
        row["bit_identical_auto_cluster"] = bool(np.array_equal(runs["fused"][0], runs["loop"][0]) and
                                                 np.array_equal(runs["fused"][1], runs["loop"][1]) and
                                                 np.array_equal(runs["fused_parameter_major"][0], runs["loop"][0]))
        os.environ["NESOSIM_ENS_CLUSTER"] = args.cluster
        pinned = []
        for cls in (Batch, Loop):
            x = cls(mask, seasons, params)
            pinned.append(tuple(r.cpu().numpy() for r in x.run()))
            x.close()
        os.environ.pop("NESOSIM_ENS_CLUSTER", None)
        row["bit_identical_pinned_cluster"] = bool(np.array_equal(pinned[0][0], pinned[1][0]) and
                                                   np.array_equal(pinned[0][1], pinned[1][1]))
        row["pinned_cluster"] = int(args.cluster)
        row["obs_used_min"] = int(runs["fused"][1].min())
        one = {}
        for name, sets in (("single_forcing_obs_kernel", False), ("forcing_sets_obs_kernel", True)):
            x = OneSeason(mask, seasons, np.tile(params, (len(seasons), 1)), sets)
            ms, _, kms, res = timed(x)
            x.close()
            one[name] = {"ms": ms, "season_kernel_ms": kms, "misfit": res[0]}
        row["one_season_%d_members" % (P * len(seasons))] = {
            "what": "every member on season %d: the cost of the forcing-sets instantiation itself" % YEARS[0],
            **{k: {"ms": v["ms"], "season_kernel_ms": v["season_kernel_ms"]} for k, v in one.items()},
            "bit_identical": bool(np.array_equal(one["single_forcing_obs_kernel"]["misfit"], one["forcing_sets_obs_kernel"]["misfit"]))}
        result["runs"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "calibration_seasons_timing.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
