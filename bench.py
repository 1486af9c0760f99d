#!/usr/bin/env python
"""bench.py -- grid-cell-days/s of the NESOSIM daily snow-budget hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): 100 km Arctic grid (90x90), one Aug 15 - May 1 season (260 days -> 259
steps), a 1024-member calibration ensemble sharded 128 members per GPU (weak scaling: each rank runs 128
members; N=8 is the named 1024-member job).  One "step" = one full season pass of this rank's 128 members =
128 x 8100 x 259 = 2.685e8 member-cell-days, synthetic forcing (nesosim_b200/synthetic.py, seeded).

Reported (one JSON line, rank 0):
  value      member-cell-days/s, all ranks, forcing resident in HBM, full 12-array output contract in HBM
  roofline   algorithmic HBM bytes (96 + 41/M per member-cell-day, SURVEY.md §8d) / device time, against the
             measured copy bandwidth in MEASURED_PEAKS.json
  e2e        the same metric through nesosim_run_season_host with HOST buffers (H2D + D2H inside the timing): all
             twelve arrays land in the caller's host memory; a single rank drains them compacted (ocean cells over
             the link, host threads scatter), several ranks plainly -- `e2e.drain` says which, and the host arrays are
             compared with the device-resident season
  cpu_baseline  the numpy oracle port of the reference's calcBudget loop on this box's host cores
`--impl reference` times only that CPU port (all host cores) and prints the same line shape.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DX = 100000
NUM_DAYS = 260                 # Aug 15 - May 1 (BASELINE.md §2)
MEMBERS_PER_GPU = 128          # 1024 members / 8 GPUs
METRIC = "grid-cell-days/s (members x cells x days)"
UNIT = "cell-days/s"
SEED = 2024


_T0 = time.perf_counter()


def stamp(label):
    """Progress line on stderr (rank 0): where the wall time of a bench run goes."""
    if int(os.environ.get("RANK", "0")) == 0:
        sys.stderr.write("[bench %7.1f s] %s\n" % (time.perf_counter() - _T0, label))
        sys.stderr.flush()


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def workload_config(members, n_gpus, extra=None):
    cfg = {"workload": "100 km Arctic season (90x90, Aug15-May1: 260 days, 259 steps), %d-member calibration "
                       "ensemble, %d members per GPU, full 12-array output" % (members * n_gpus, members),
           "grid": [90, 90], "dx_m": DX, "num_days": NUM_DAYS, "members_per_gpu": members,
           "members_total": members * n_gpus,
           "l2": "no flush: each step writes %.1f GB of outputs per GPU (>> 126 MB L2)"
                 % (members * NUM_DAYS * 8100 * 96 / 1e9)}
    if extra:
        cfg.update(extra)
    return cfg


# ----------------------------------------------------------------------------------------- CPU baseline

_CPU_CACHE = {}


def _cpu_member_season(args):
    """One member-season of the numpy oracle (= the reference's calcBudget loop, NESOSIM.py:614-639)."""
    os.environ["OMP_NUM_THREADS"] = "1"
    seed, row, num_days = args
    from nesosim_b200 import synthetic as S
    from oracle import nesosim_oracle as O
    key = (seed, num_days)
    if key not in _CPU_CACHE:
        mask = S.region_mask(dx=DX)
        _CPU_CACHE[key] = (mask, S.make_season(mask, num_days, seed=seed), S.make_ic(mask, seed=seed))
    mask, forcing, ic = _CPU_CACHE[key]
    p = O.Params(windPackFactor=row[0], windPackThresh=row[1], leadLossFactor=row[2], atmLossFactor=row[3])
    t0 = time.perf_counter()
    O.run_season(forcing, ic, mask, DX, p, O.Flags(atmlossInc=1))
    return time.perf_counter() - t0


class CpuPool:
    """One worker process per host core, each holding the synthetic forcing; reused across steps."""

    def __init__(self, cores=None, num_days=NUM_DAYS):
        import multiprocessing as mp
        self.cores = cores or os.cpu_count() or 1
        self.num_days = num_days
        self.pool = mp.get_context("spawn").Pool(self.cores)
        from nesosim_b200 import synthetic as S
        self.params = S.ensemble_params(self.cores * 8, seed=SEED)
        self.pool.map(_cpu_member_season, [(SEED, self.params[i], num_days) for i in range(self.cores)])   # warm the workers

    def step(self, members_per_core=1):
        """One bounded sample: members_per_core member-seasons on every core.  Returns (cell-days/s, seconds, text)."""
        n = self.cores * members_per_core
        jobs = [(SEED, self.params[i % len(self.params)], self.num_days) for i in range(n)]
        t0 = time.perf_counter()
        self.pool.map(_cpu_member_season, jobs)
        dt = time.perf_counter() - t0
        cells = 8100 * (self.num_days - 1) * n
        return cells / dt, dt, "%d member-seasons (90x90x%d steps each), %d processes" % (n, self.num_days - 1, self.cores)

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_baseline(members_per_core=1, cores=None, num_days=NUM_DAYS, target_seconds=12.0):
    """Process-parallel over members on all host cores, sized to about `target_seconds` of CPU work per core;
    returns (cell-days/s, cores, sample text, seconds)."""
    pool = CpuPool(cores, num_days)
    try:
        v, dt, sample = pool.step(members_per_core)
        reps = max(1, min(32, int(target_seconds / max(dt, 1e-3))))
        if reps > 1:
            v, dt, sample = pool.step(members_per_core * reps)
        return v, pool.cores, sample, dt
    finally:
        pool.close()


def verbatim_note():
    """The reference's own loop executed verbatim can only be timed where /root/reference exists (the build container):
    profiles/r02_reference_verbatim.json (tools/time_reference_verbatim.py) holds that figure next to the port's on the
    same core, with identical outputs -- the port this bench times is the faster of the two, i.e. a conservative baseline."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_reference_verbatim.json")) as f:
            d = json.load(f)
        return {"reference_verbatim_cell_days_per_s_per_core": d["reference_verbatim"]["cell_days_per_s_per_core"],
                "numpy_port_cell_days_per_s_per_core_same_core": d["numpy_port"]["cell_days_per_s_per_core"],
                "port_over_verbatim": d["port_over_verbatim"], "identical_outputs": d["identical_outputs"],
                "where": d["where"], "source": "profiles/r02_reference_verbatim.json"}
    except Exception:
        return None


def run_reference(args):
    """The reference's CPU path (the numpy port of its calcBudget loop: the reference itself is pure Python whose
    dependencies are absent) on all host cores.  One step = one bounded sample of the workload, sized so that
    steps + warmup stay within about two minutes."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    pool = CpuPool()
    try:
        _, dt1, _ = pool.step(1)
        per_step = 110.0 / max(args.steps + args.warmup, 1)
        mpc = max(1, min(32, int(per_step / max(dt1, 1e-3))))
        for _ in range(max(args.warmup, 0)):
            pool.step(mpc)
        vals, t_total, sample = [], 0.0, ""
        for _ in range(args.steps):
            v, dt, sample = pool.step(mpc)
            vals.append(v)
            t_total += dt
        cores = pool.cores
    finally:
        pool.close()
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(MEMBERS_PER_GPU, args.gpus),
            "reference_step": "bounded sample: " + sample,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "verbatim_reference": verbatim_note()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- clocks

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append(ln.strip())

    def wait_first(self, timeout=5.0):
        t0 = time.time()
        while self.proc and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.05)

    def mark(self):
        """Samples taken from now on belong to the timed region."""
        self.first = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows[getattr(self, "first", 0):]:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------- ours

def run_ours(args):
    import torch
    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the communicator comes up: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    from nesosim_b200 import build
    if rank == 0:
        build.build(verbose=False)
    if world > 1:
        dist.barrier()
    from nesosim_b200 import synthetic as S
    from nesosim_b200.engine import SnowBudgetEngine

    stamp("library ready")
    M = args.members
    T = args.days
    mask = S.region_mask(dx=DX)
    ny, nx = mask.shape
    forcing = S.make_season(mask, T, seed=SEED)
    ic = S.make_ic(mask, seed=SEED)
    from nesosim_b200 import sharding
    params = sharding.shard_params(S.ensemble_params(M * world, seed=SEED), rank, world)   # this rank's members

    if args.variant:
        os.environ["NESOSIM_ENS_VARIANT"] = args.variant
    eng = SnowBudgetEngine(mask, T, DX, n_members=M, atmlossInc=1, device=local)
    eng.set_path(args.path)
    eng.set_forcing(forcing["precip"], forcing["conc"], forcing["wind"], forcing["drift"])
    out = eng.alloc_outputs()
    cells_per_step = M * ny * nx * (T - 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # asynchronous mode: run_season never synchronises the stream, the K seasons of the timed region run back to back
    # and their operand-range flags are resolved by eng.sync() afterwards (nesosim_set_async / nesosim_sync)
    eng.set_async(True)
    ic_dev = eng._dev(ic)
    for _ in range(max(args.warmup, 0)):
        eng.run_season(params, ic_dev, out)
    eng.sync()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first()
    l0 = eng.launch_count()
    k0 = eng.season_kernel_time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark()
    ev0.record()
    for _ in range(args.steps):
        eng.run_season(params, ic_dev, out)
    ev1.record()
    barrier()
    redone = eng.sync()
    eng.set_async(False)
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - l0
    k1 = eng.season_kernel_time()
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * cells_per_step * args.steps / (ms * 1e-3)

    # roofline of the dominant kernel: algorithmic bytes per launch / average launch duration in the timed region
    # One launch of the season-resident kernel advances all M members by T-1 days, so the algorithmic bytes per
    # launch are cells_per_step * (96 + 41/M) (SURVEY.md 8d); its duration comes from CUDA events the library
    # records around that launch on the launching stream.  (General path: 259 day-step launches per step, timed
    # as the step.)
    b_alg = 96.0 + 41.0 / M
    bytes_per_step = cells_per_step * b_alg
    peak, peak_src = measured_peak()
    kn = k1[1] - k0[1]
    if kn > 0:
        kernel_ms = (k1[0] - k0[0]) / kn
        achieved = bytes_per_step / (kernel_ms * 1e-3) / 1e9
        launches_of_kernel = kn / max(args.steps, 1)
    else:
        kernel_ms = ms / max(launches, 1)
        achieved = bytes_per_step * args.steps / (ms * 1e-3) / 1e9
        launches_of_kernel = launches / max(args.steps, 1)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": eng.dominant_kernel(), "bytes_per_member_cell_day": b_alg,
                "bytes_per_launch": bytes_per_step if kn > 0 else bytes_per_step / max(launches_of_kernel, 1),
                "launches_per_step": launches_of_kernel, "peak_source": peak_src, "avg_launch_us": 1e3 * kernel_ms,
                "kernel_share_of_step": (k1[0] - k0[0]) / ms if kn > 0 else 1.0}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(prof):
        try:
            with open(prof) as f:
                roofline["traffic"] = json.load(f).get("dram_bytes_per_launch")
        except Exception:
            pass

    stamp("headline timed (%d steps)" % args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, mask, args.dump_outputs)
    # end to end through the host-buffer C-ABI call
    e2e = None
    try:
        if args.no_e2e:
            raise RuntimeError("skipped (--no-e2e)")
        e2e = run_e2e(args, eng, forcing, params, ic, rank, world, cells_per_step, barrier, out)
    except Exception as ex:   # keep the headline line even if the host path cannot allocate
        e2e = {"value": None, "unit": UNIT, "error": str(ex)[:200]}

    # the same season when only the final NetCDF product's six float32 fields go back to the host (labelled apart:
    # it is NOT the full 12-array contract the headline e2e figure keeps)
    stamp("e2e (host buffers) done")
    e2e_final = None
    try:
        if args.no_e2e:
            raise RuntimeError("skipped (--no-e2e)")
        e2e_final = run_e2e_final(args, eng, forcing, params, ic, out, world, cells_per_step, barrier)
    except Exception as ex:
        e2e_final = {"value": None, "unit": UNIT, "error": str(ex)[:200]}

    if isinstance(e2e, dict) and e2e.get("value") and not args.no_e2e:
        try:
            link = d2h_ceiling(world)
            e2e["link_d2h_gbs_per_gpu"] = link
            e2e["link_note"] = ("plain pinned device->host copy, one cudaMemcpyAsync stream per rank, all %d ranks at once; "
                                "fraction = this call's D2H bytes / its time / that ceiling" % world)
            e2e["d2h_fraction_of_link"] = e2e["d2h_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9 / link
        except Exception as ex:
            e2e["link_error"] = str(ex)[:200]

    stamp("e2e (final products) and link ceiling done")
    kernel_path = eng.last_path()
    failures = []
    if isinstance(e2e, dict) and e2e.get("host_arrays_identical_to_device_result") is False:
        failures.append("e2e: the host arrays differ from the device-resident season")
    if redone:
        failures.append("%d season(s) of the synthetic workload left the season kernel's operand range and were redone" % redone)

    # calibration mode (SURVEY 8f N3): the same 128-member season with the misfit against point observations reduced
    # inside the season kernel and NO output array stored
    misfit = None
    if not args.no_extra:
        try:
            misfit = run_misfit_mode(eng, mask, forcing, params, ic_dev, world, cells_per_step, barrier)
        except Exception as ex:
            misfit = {"error": str(ex)[:300]}
    del out
    eng.close()
    torch.cuda.empty_cache()

    stamp("calibration mode done")
    # BASELINE configs[3]: the 1980-2021 multi-season batch, seasons dealt over the ranks
    multi = None
    if not args.no_extra:
        try:
            multi = run_multiseason_41(rank, world, local, barrier, peak)
            if multi.get("identical_to_single_season_run") is False:
                failures.append("multiseason_41: batch result differs from the single-season run")
        except Exception as ex:
            multi = {"error": str(ex)[:300]}      # (a leg that could not run is reported, not fatal; a wrong result is)

    stamp("multi-season batch done")
    # BASELINE configs[4]: the 5 km grid as row strips over the ranks, ghost rows exchanged inside the day kernel
    dom = None
    if world > 1 and not args.no_extra:
        try:
            dom = run_domain_5km(rank, world, local, peak)
            if rank == 0 and dom.get("identical_to_one_gpu") is not True:
                failures.append("domain_5km: strips differ from the one-GPU run")
        except Exception as ex:
            dom = {"error": str(ex)[:300]}
            if "ghost rows" in str(ex):           # a strip timed out: its results are invalid (domain.check_strips)
                failures.append("domain_5km: " + str(ex)[:200])
    if world > 1:     # every rank learns whether any rank failed (rank 0 prints; all exit non-zero)
        flags = [None] * world
        dist.all_gather_object(flags, failures)
        failures = sorted({f for fl in flags for f in fl})

    stamp("5 km strips done" if world > 1 else "(5 km strips: N > 1 only)")
    # BASELINE configs[0]: the drop-in main() over a season of forcing files, next to the CPU loop over the same files
    dropin = None
    if rank == 0 and world == 1 and not args.no_cpu and not args.no_extra:
        try:
            dropin = run_main_dropin()
            if dropin.get("identical_to_cpu_loop") is False:
                failures.append("main_dropin: main() differs from the CPU loop on the same files")
        except Exception as ex:
            dropin = {"error": str(ex)[:300]}

    stamp("drop-in main done")
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, cores, sample, _ = cpu_baseline(1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
               "verbatim_reference": verbatim_note()}

    stamp("cpu baseline done")
    other = None
    if rank == 0 and world == 1 and not args.no_e2e and not args.no_other:
        try:
            other = run_other_grids(peak)
        except Exception as ex:
            other = {"error": str(ex)[:200]}

    stamp("other grids done")
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / max(args.steps, 1), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(M, world), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
                "kernel": {"path": kernel_path, "variant": args.variant or "default"},
                "roofline": roofline, "cpu_baseline": cpu, "e2e_final_products": e2e_final, "other_grids": other,
                "ensemble_misfit": misfit, "multiseason_41": multi, "domain_5km": dom, "main_dropin": dropin}
        if failures:
            line["failed"] = failures
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if failures:
        sys.stderr.write("bench.py: FAILED checks: %s\n" % "; ".join(failures))
        sys.exit(3)


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 18          # member-day-cells kept per array when the full outputs exceed DUMP_LIMIT_BYTES


def dump_outputs(out, mask, directory):
    """Write the device-resident season of the timed path (rank 0's members) under <directory>.

    NaN and +-inf are outputs of the model (land cells, density below minSnowD, days of NaN forcing), but the files stay
    finite so that two builds can be compared with a tolerance: <name>.npy (float64) holds 0 where the output is not
    finite, and <name>_nonfinite.npy (float32, same shape) says what is there: 0 finite, 1 NaN, 2 +inf, 3 -inf.
    Up to DUMP_LIMIT_BYTES the arrays are written whole.  Above it every array keeps the same DUMP_SAMPLE
    member-day-cells of the ocean (1 <= mask <= 10, the cells the model computes): sorted flat indices into
    (members * days, ocean cells in row-major order) drawn by np.random.default_rng(SEED).choice without replacement,
    so the sample depends only on the shape and the mask; snowDepths keeps both layers, shape (DUMP_SAMPLE, 2)."""
    import torch
    os.makedirs(directory, exist_ok=True)
    M, T, ny, nx = out["density"].shape
    plane = ny * nx
    total = sum(t.numel() for t in out.values()) * (8 + 4)
    mt = cell = None
    if total > DUMP_LIMIT_BYTES:
        ocean = np.flatnonzero((np.asarray(mask) >= 1) & (np.asarray(mask) <= 10))
        pick = np.sort(np.random.default_rng(SEED).choice(M * T * len(ocean), size=DUMP_SAMPLE, replace=False))
        dev = out["density"].device
        mt = torch.from_numpy(pick // len(ocean)).to(dev)
        cell = torch.from_numpy(ocean[pick % len(ocean)]).to(dev)
    for name, t in out.items():
        if mt is None:
            a = t
        elif name == "snowDepths":
            a = t.view(M * T, 2, plane)[mt, :, cell]
        else:
            a = t.view(M * T, plane)[mt, cell]
        a = a.cpu().numpy()
        code = np.zeros(a.shape, dtype=np.float32)
        code[np.isnan(a)] = 1
        code[np.isposinf(a)] = 2
        code[np.isneginf(a)] = 3
        np.save(os.path.join(directory, name + ".npy"), np.where(code == 0, a, 0.0))
        np.save(os.path.join(directory, name + "_nonfinite.npy"), code)
    stamp("outputs of the last timed step written to %s (%s)" % (directory, "whole" if mt is None else
                                                                 "%d sampled member-day-cells" % DUMP_SAMPLE))


def host_drain_settings(world, cores):
    """(host threads of this rank, compacted drain?) for nesosim_run_season_host.  Threads: this rank's share of the
    cores (the library's own default assumes a rank per visible GPU).  The compacted drain trades link bytes for host
    memory traffic, and the host's memory system is shared by the ranks of a box.  Measured
    (profiles/r02_e2e_compacted_drain.jsonl): one rank 330-345 ms against 425-455 ms plain; two ranks 402-420 against
    418 ms (the hybrid split keeps it from falling behind, but there is nothing to gain); eight ranks 2202 (all packed)
    against 2168 ms.  So a single rank takes it, several ranks stay on the plain drain."""
    threads = max(1, min(16, cores // world))      # (12 threads already saturate the host's memory system)
    return threads, (world == 1 and threads >= 4)


def run_e2e(args, eng, forcing, params, ic, rank, world, cells_per_step, barrier, dev_out=None):
    """Season through nesosim_run_season_host: pinned HOST forcing in, all 12 HOST arrays out, every step.  The
    library picks the drain: every byte of the arrays over the link, or -- when this rank has enough host threads --
    ocean cells only with the land cells filled in on the host (same arrays in the caller's memory either way; checked
    below against the device-resident result of the headline run)."""
    import torch
    M, T, ny, nx = eng.M, eng.T, eng.ny, eng.nx
    threads, compact = host_drain_settings(world, os.cpu_count() or 1)
    os.environ.setdefault("NESOSIM_HOST_THREADS", str(threads))
    os.environ.setdefault("NESOSIM_HOST_COMPACT", "1" if compact else "0")
    names = list(__import__("nesosim_b200._lib", fromlist=["x"]).OUTPUT_NAMES)
    need = 12 * M * T * ny * nx * 8
    avail = None
    try:
        with open("/proc/meminfo") as f:
            for ln in f:
                if ln.startswith("MemAvailable"):
                    avail = int(ln.split()[1]) * 1024
    except OSError:
        pass
    note = "all 12 arrays to pinned host memory"
    if avail is not None and need * world > 0.6 * avail:
        names = ["snowDepths", "density"]
        note = "host RAM too small for the full contract x %d ranks: snowDepths+density only" % world
    host_out = {}
    for n in names:
        shape = (M, T, 2, ny, nx) if n == "snowDepths" else (M, T, ny, nx)
        host_out[n] = torch.empty(shape, dtype=torch.float64, pin_memory=True)
    hf = {k: torch.from_numpy(np.ascontiguousarray(forcing[k])).pin_memory() for k in ("precip", "conc", "wind", "drift")}
    ic_h = torch.from_numpy(np.ascontiguousarray(ic)).pin_memory()
    steps = max(1, min(args.steps, args.e2e_steps))
    eng.run_season_host(hf, params, ic_h, host_out)      # warm-up (allocates device staging)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        _, up, down = eng.run_season_host(hf, params, ic_h, host_out)
    barrier()
    dt = time.perf_counter() - t0
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    compacted, full_chunks = eng.host_drain_info()
    blocks_packed, blocks_plain = eng.host_drain_blocks()
    res = {"value": world * cells_per_step * steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(up),
           "d2h_bytes_per_step": int(down), "steps": steps, "ms_per_step": 1e3 * dt / steps, "outputs": note,
           "host_array_bytes_per_step": int(sum(v.numel() * 8 for v in host_out.values())),
           "drain": ("compacted: ocean cells of the nine member-dependent arrays + the land cells of the first three time slots "
                     "cross the link, %s host threads scatter them into the caller's arrays" % os.environ["NESOSIM_HOST_THREADS"])
           if compacted else "full: every byte of the arrays crosses the link",
           "host_threads": int(os.environ["NESOSIM_HOST_THREADS"]), "chunks_copied_in_full": full_chunks,
           "blocks_packed": blocks_packed, "blocks_copied_whole_by_the_link": blocks_plain}
    if dev_out is not None:       # the caller's arrays against the device-resident season of the headline run
        same = True
        for n in host_out:
            for m in sorted({0, M // 2, M - 1}):
                same = same and bool(torch.equal(host_out[n][m].nan_to_num(nan=-7.0), dev_out[n][m].cpu().nan_to_num(nan=-7.0)))
        res["host_arrays_identical_to_device_result"] = same
    return res


def run_e2e_final(args, eng, forcing, params, ic, dev_out, world, cells_per_step, barrier):
    """Host forcing in (pinned, H2D every step), season on the device, fused final-product pass
    (nesosim_final_products), six float32 (M,T,ny,nx) fields back to pinned host memory."""
    import torch
    from nesosim_b200 import engine as E
    M, T, ny, nx = eng.M, eng.T, eng.ny, eng.nx
    hf = {k: torch.from_numpy(np.ascontiguousarray(forcing[k])).pin_memory() for k in ("precip", "conc", "wind", "drift")}
    ic_h = torch.from_numpy(np.ascontiguousarray(ic)).pin_memory()
    host = {n: torch.empty((M, T, ny, nx), dtype=torch.float32, pin_memory=True) for n in E.FINAL_NAMES}
    dev_f = {n: torch.empty((M, T, ny, nx), dtype=torch.float32, device="cuda") for n in E.FINAL_NAMES}
    steps = max(1, min(args.steps, args.e2e_steps))

    def one():
        d = {k: v.cuda(non_blocking=True) for k, v in hf.items()}
        eng.set_forcing(d["precip"], d["conc"], d["wind"], d["drift"])
        eng.run_season(params, ic_h.cuda(non_blocking=True), dev_out)
        E.final_products(dev_out["snowDepths"], dev_out["density"], d["conc"], d["precip"], d["wind"], out=dev_f)
        for n in E.FINAL_NAMES:
            host[n].copy_(dev_f[n], non_blocking=True)
        torch.cuda.synchronize()

    one()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    h2d = sum(v.numel() * 8 for v in hf.values()) + ic_h.numel() * 8
    return {"value": world * cells_per_step * steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(6 * M * T * ny * nx * 4), "steps": steps, "ms_per_step": 1e3 * dt / steps,
            "outputs": "the six float32 fields of final/NESOSIMv11_*.nc (snow depth, volume, density, ice concentration, "
                       "precipitation, wind), masked and rounded on the device"}


def d2h_ceiling(world, gib=1.0, reps=3):
    """GB/s of a plain pinned device->host cudaMemcpyAsync on this rank while every other rank does the same
    (max time over ranks): the ceiling any end-to-end figure of this box can reach per GPU."""
    import torch
    n = int(gib * (1 << 30)) // 8
    d = torch.empty(n, dtype=torch.float64, device="cuda")
    h = torch.empty(n, dtype=torch.float64, pin_memory=True)
    h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return reps * n * 8 / float(t.item()) / 1e9


def run_misfit_mode(eng, mask, forcing, params, ic, world, cells_per_step, barrier, n_obs=20000, reps=5):
    """nesosim_run_season_misfit: every member's sum of squared differences to `n_obs` point observations of snow depth
    over ice; the season-resident kernel stores only the depths of the observed cell-days (8 B each), a per-member
    epilogue reduces them to M scalars.  Labelled apart from the
    headline: without the 96 B per member-cell-day of output stores the algorithmic HBM bytes are 41/M per member-cell-day,
    so the bound of this mode is the kernel's fp64 / shared-memory work, not HBM."""
    import torch
    rng = np.random.default_rng(SEED)
    ocean = np.argwhere((mask <= 10) & (mask >= 1))
    pick = ocean[rng.integers(0, len(ocean), n_obs)]
    obs = (rng.integers(0, eng.T, n_obs), pick[:, 0], pick[:, 1], 0.3 * rng.random(n_obs))
    eng.set_observations(obs)                      # compiled against the kernel's cell ownership once, kept on the device
    mis, used = eng.run_season_misfit(params, ic)
    ref = mis.clone()
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        mis, used = eng.run_season_misfit(params, ic)
        e1.record()
        torch.cuda.synchronize()
        best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
    t = torch.tensor([best], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    M = eng.M
    return {"workload": "the headline season in calibration mode: %d point observations sampled inside the season kernel, no output "
                        "array stored, per-member misfit from a one-CTA-per-member epilogue" % n_obs,
            "ms_per_season": ms, "value": world * cells_per_step / (ms * 1e-3), "unit": UNIT,
            "bytes_per_member_cell_day": 41.0 / M, "bound": "fp64 / shared memory of the season kernel (not HBM: no output stores)",
            "d2h_bytes": 16 * M, "observations_used_member0": int(used[0].item()), "deterministic": bool(torch.equal(ref, mis)),
            "includes": "pre-pass, season kernel, epilogue (the observations are registered once, outside the timing)"}


MULTI_YEARS = list(range(1980, 2021))      # 41 start years, Sep 1 - Apr 30 (run_multiseason.py:30-50)


def season_days(year):
    """numDays of the Sep 1 (year) - Apr 30 (year+1) season: 242, or 243 when February of year+1 has 29 days."""
    import datetime
    return (datetime.date(year + 1, 4, 30) - datetime.date(year, 9, 1)).days + 1


def run_multiseason_41(rank, world, local, barrier, peak):
    """The loop of run_multiseason.py as ONE native call per rank: the 41 seasons are dealt round-robin over the ranks
    (sharding.season_assignment), each rank stacks its seasons' forcing with nesosim_set_forcing_sets (one member per
    season, the script's parameters, seasons of 242 or 243 days) and runs them together.  Strong scaling: the job is
    the 41 seasons = 9891 steps whatever N is.  Device time (CUDA events), max over ranks."""
    import torch
    from nesosim_b200 import sharding, synthetic as S
    from nesosim_b200.engine import SnowBudgetEngine
    mine = sharding.season_assignment(MULTI_YEARS, rank, world)
    mask = S.region_mask(dx=DX)
    ny, nx = mask.shape
    days = [season_days(y) for y in mine]
    T = max(season_days(y) for y in MULTI_YEARS)
    total_steps = sum(season_days(y) - 1 for y in MULTI_YEARS)
    Sn = len(mine)
    stack = {k: np.zeros((Sn, T) + ((2,) if k == "drift" else ()) + (ny, nx)) for k in ("precip", "conc", "wind", "drift")}
    ics = np.zeros((Sn, ny, nx))
    for i, y in enumerate(mine):
        f = S.make_season(mask, days[i], seed=y)
        for k in stack:
            stack[k][i, :days[i]] = f[k]
        ics[i] = S.make_ic(mask, seed=y)
    params = [[5.8e-7, 5., 1.45e-7, 2.2e-8]] * Sn           # run_multiseason.py:42-50
    eng = SnowBudgetEngine(mask, T, DX, n_members=Sn, atmlossInc=1, device=local)
    eng.set_forcing_sets(stack["precip"], stack["conc"], stack["wind"], stack["drift"], np.arange(Sn), days)
    out = eng.alloc_outputs(zero=True)
    ic_dev = eng._dev(ics)
    l0 = eng.launch_count()
    best = None
    for rep in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        eng.run_season(params, ic_dev, out)
        e1.record()
        torch.cuda.synchronize()
        if rep:
            best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
    launches = (eng.launch_count() - l0) // 4
    path = eng.last_path()
    t = torch.tensor([best], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # the batch against the same season run alone (plain single-season context): rank 0, its first season
    same = None
    if rank == 0:
        y, d = mine[0], days[0]
        one = SnowBudgetEngine(mask, d, DX, n_members=1, atmlossInc=1, device=local)
        one.set_forcing(stack["precip"][0, :d], stack["conc"][0, :d], stack["wind"][0, :d], stack["drift"][0, :d])
        ref = one.run_season(params[:1], ics[0])
        same = all(bool(torch.equal(torch.nan_to_num(out[k][0, :d], nan=-7.0), torch.nan_to_num(ref[k][0], nan=-7.0)))
                   for k in out)
        one.close()
    eng.close()
    del out
    torch.cuda.empty_cache()
    cells = total_steps * ny * nx
    b_alg = 96.0 + 41.0            # every season has its own forcing: nothing is shared between members
    return {"workload": "multi-season 1980-2021 batch: 41 seasons (Sep 1 - Apr 30, 242/243 days), 100 km grid, one native call "
                        "per rank over its seasons (nesosim_set_forcing_sets)",
            "seasons_total": len(MULTI_YEARS), "seasons_this_rank": Sn, "steps_total": total_steps, "n_gpus": world,
            "ms": ms, "steps_per_s": total_steps / (ms * 1e-3), "value": cells / (ms * 1e-3), "unit": UNIT,
            "scaling": "strong", "kernel_path": path, "launches_per_rank": launches,
            "roofline_frac_algorithmic_per_gpu": cells * b_alg / world / (ms * 1e-3) / 1e9 / peak,
            "identical_to_single_season_run": same, "data": "synthetic, one seed per start year"}


def nvlink_tx_kib(index):
    """Sum of the NVLink data-transmit counters of one GPU (nvidia-smi nvlink -gt d), KiB; None if unavailable."""
    import re
    try:
        txt = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(index)], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, text=True, timeout=20).stdout
        vals = [int(v) for v in re.findall(r"Data Tx:\s*(\d+)\s*KiB", txt)]
        return sum(vals) if vals else None
    except Exception:
        return None


def run_domain_5km(rank, world, local, peak, steps=40, gen_days=4, reps=3):
    """5 km pan-Arctic grid (1785 x 1785, real coastline) as `world` row strips, one per GPU, the ghost-row exchange
    fused into the day kernel over peer memory (nesosim_strip_*; domain.run_decomposed_season_peer).  Also runs the
    same season on ONE GPU of the same box (rank 0) and compares EVERY owned row of all eleven arrays with it."""
    import torch
    import torch.distributed as dist
    from nesosim_b200 import domain, synthetic as S
    from nesosim_b200.engine import SnowBudgetEngine
    dx, T = 5000, steps + 1
    mask = S.region_mask(dx=dx)
    n = mask.shape[0]
    gen = S.make_season(mask, gen_days, seed=7)
    gen = {k: v for k, v in gen.items() if k != "temp"}
    idx = np.arange(T) % gen_days
    ic = S.make_ic(mask, seed=7)
    params = [5.8e-7, 5., 1.45e-7, 2.2e-8]
    cells = n * n * steps

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- one GPU, the whole grid (rank 0; the others wait)
    ref, one_ms = None, 0.0
    if rank == 0:
        eng1 = SnowBudgetEngine(mask, T, dx, n_members=1, device=local, atmlossInc=1)
        eng1.set_path("general")
        it = torch.as_tensor(idx, device="cuda", dtype=torch.long)
        f = {k: eng1._dev(v)[it].contiguous() for k, v in gen.items()}
        eng1.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
        ref = eng1.alloc_outputs()
        best = None
        for r in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            eng1.run_season([params], ic, ref)
            e1.record()
            torch.cuda.synchronize()
            if r:
                best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
        one_ms = best
        eng1.close()
        del f
        torch.cuda.empty_cache()
    dist.barrier()

    # ---- the strips
    lo, hi, part, eng = domain.run_decomposed_season_peer(mask, T, dx, gen, params, ic, rank, world, device=local,
                                                          day_index=idx, atmlossInc=1, timeout_s=20.0, balance=True)
    outs = eng._keep[1]
    lo_, hi_, elo, ehi = eng._strip_rows
    ic_dev = eng._dev(np.ascontiguousarray(ic[elo:ehi]))
    best = None
    tx0 = nvlink_tx_kib(local) if rank == 0 else None
    for r in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        eng.run_season([params], ic_dev, outs)
        e1.record()
        torch.cuda.synchronize()
        domain.check_strips(eng, rank, world)            # raises on every rank if any strip timed out
        ms = max_over_ranks(e0.elapsed_time(e1))
        best = ms if best is None else min(best, ms)

    tx1 = nvlink_tx_kib(local) if rank == 0 else None
    nvlink = None
    if tx0 is not None and tx1 is not None:
        nvlink = {"rank0_tx_bytes_per_day_measured": (tx1 - tx0) * 1024.0 / (reps * steps),
                  "rank0_tx_bytes_per_day_algorithmic": 2 * 2 * n * 8 + 8,
                  "note": "rank 0 has one neighbour: 2 layers x 2 rows x nx doubles + the 8-byte flag per day, stored by the day "
                          "kernel straight into the neighbour GPU's memory (nvidia-smi nvlink -gt d, KiB resolution)"}
    # ---- every owned row of every array against the one-GPU run (gathered to rank 0 over NCCL, compared on the device)
    own = slice(lo - elo, lo - elo + (hi - lo))
    names = sorted(outs)
    ok = True
    bounds = [None] * world
    dist.all_gather_object(bounds, (lo, hi))
    for k in names:
        mine = outs[k][0][..., own, :].contiguous()
        if rank == 0:
            ok = ok and bool(torch.equal(torch.nan_to_num(mine, nan=-7.0), torch.nan_to_num(ref[k][0][..., lo:hi, :], nan=-7.0)))
            for r in range(1, world):
                rl, rh = bounds[r]
                shape = list(ref[k][0].shape)
                shape[-2] = rh - rl
                buf = torch.empty(shape, dtype=torch.float64, device="cuda")
                dist.recv(buf, src=r)
                ok = ok and bool(torch.equal(torch.nan_to_num(buf, nan=-7.0), torch.nan_to_num(ref[k][0][..., rl:rh, :], nan=-7.0)))
                del buf
        else:
            dist.send(mine, dst=0)
    eng.close()
    del outs, ref
    torch.cuda.empty_cache()
    dist.barrier()
    if rank != 0:
        return {}
    gbs = cells * 137.0 / (best * 1e-3) / 1e9
    return {"workload": "5 km pan-Arctic grid (1785x1785, real coastline), %d steps, %d row strips (one per GPU), ghost rows "
                        "stored into the neighbour GPU's memory by the day kernel (peer memory, flags); no collective" % (steps, world),
            "grid": [n, n], "steps": steps, "n_gpus": world, "ms": best, "us_per_day": 1e3 * best / steps,
            "value": cells / (best * 1e-3), "unit": UNIT, "scaling": "strong",
            "roofline_frac_algorithmic_per_gpu": gbs / world / peak,
            "one_gpu_same_box": {"ms": one_ms, "us_per_day": 1e3 * one_ms / steps, "value": cells / (one_ms * 1e-3),
                                 "roofline_frac_algorithmic": cells * 137.0 / (one_ms * 1e-3) / 1e9 / peak},
            "speedup_vs_one_gpu": one_ms / best, "identical_to_one_gpu": bool(ok),
            "compared": "all 11 arrays, every owned row, every time slot (NaN patterns and values) on the device",
            "strip_status": "no time-out on any rank", "launches_per_day": 1, "nvlink": nvlink,
            "strip_rows": [b[1] - b[0] for b in bounds], "strip_cut": "rows cut for equal modelled cost (domain.balanced_cuts)",
            "data": "synthetic (%d generated days repeated)" % gen_days}


class _StandInUtils:
    """What ``nesosim_b200.NESOSIM.main`` needs from the reference's ``utils`` module (grid, mask, calendar) when the
    reference's own dependencies (pyproj, netCDF4, cartopy) are not installed: the closed-form EPSG:3413 grid and the
    bundled regrid of region_n.msk from nesosim_b200.grid.  The writers are not called (saveData=0)."""

    def __init__(self, dx):
        from nesosim_b200 import grid
        self.grid = grid
        self.mask = grid.bundled_region_mask(dx)
        self.getDays = grid.getDays

    def create_grid(self, dxRes=50000):
        return self.grid.create_grid(dxRes=dxRes)

    def get_region_mask_pyproj(self, anc, proj, xypts_return=0):
        x, y, lats, lons, _ = self.grid.create_grid(dxRes=DX)       # the mask "file" is already on the model grid
        return self.mask, x, y, lons, lats


def run_main_dropin():
    """BASELINE configs[0]: one 100 km season (run_oneseason.py:40-48 dates and parameters) from forcing FILES.
    A synthetic season is written as the pickle tree the reference's gridding scripts produce; timed are (ours)
    nesosim_b200.NESOSIM.main(saveData=0, plotBudgets=0, plotdaily=0) -- read 5 files per day, stage, one GPU season
    call, all arrays back on the host -- and (CPU) the reference's loop over the same files: loadData + calcBudget per
    day (the numpy port).  Best of two passes each (the files are in the page cache for both)."""
    import shutil
    import tempfile
    import types
    from nesosim_b200 import NESOSIM as N, synthetic as S, grid
    from oracle import nesosim_oracle as O           # the CPU loop below is the reference's path, not the product
    y1, m1, d1, y2, m2, d2 = 2018, 8, 0, 2019, 3, 29          # run_oneseason.py: Sep 1 2018 - Apr 30 2019 (0-based)
    startDay, numDays, nDaysY1, dateOut = grid.getDays(y1, m1, d1, y2, m2, d2)
    mask = S.region_mask(dx=DX)
    ny, nx = mask.shape
    f = S.make_season(mask, numDays, seed=SEED)
    ic = S.make_ic(mask, seed=SEED)
    root = tempfile.mkdtemp(prefix="nesosim_dropin_")
    try:
        base = os.path.join(root, "forcing", "100km")
        day, year = startDay, y1
        for x in range(numDays):
            if x < numDays - 1:
                day = x + startDay
                year = y1
                if day >= nDaysY1:
                    day -= nDaysY1
                    year = y2
                d = day
            else:
                d = day + 1
            ds = "%03d" % d
            for sub, name, arr in (("Precip/ERA5/%d" % year, "ERA5sf100km-%d_d%sv11" % (year, ds), f["precip"][x]),
                                   ("Winds/ERA5/%d" % year, "ERA5winds100km-%d_d%sv11" % (year, ds), f["wind"][x]),
                                   ("IceConc/CDR/%d" % year, "iceConcG_CDR100km-%d_d%sv11" % (year, ds), f["conc"][x]),
                                   ("IceDrift/OSISAF/%d" % year, "OSISAF_driftG100km-%d_d%sv11" % (year, ds), f["drift"][x])):
                os.makedirs(os.path.join(base, sub), exist_ok=True)
                if not (sub.startswith("IceDrift") and np.isnan(arr).all()):      # an all-NaN day = a missing drift file
                    np.ascontiguousarray(arr).dump(os.path.join(base, sub, name))
        os.makedirs(os.path.join(base, "InitialConditions/ERA5"))
        ic.dump(os.path.join(base, "InitialConditions/ERA5", "ICsnow100km-%dv11" % y1))
        stand_in = types.ModuleType("utils")
        su = _StandInUtils(DX)
        for name in ("create_grid", "get_region_mask_pyproj", "getDays"):
            setattr(stand_in, name, getattr(su, name))
        saved = sys.modules.get("utils")
        sys.modules["utils"] = stand_in
        N.VERBOSE = False
        kw = dict(outPathT=os.path.join(root, "out") + "/", forcingPathT=os.path.join(root, "forcing") + "/",
                  anc_data_pathT="unused/", figPathT=os.path.join(root, "fig") + "/", precipVar="ERA5", windVar="ERA5",
                  driftVar="OSISAF", concVar="CDR", icVar="ERA5", densityTypeT="variable", extraStr="v11", outStr="bench",
                  IC=2, windPackFactorT=5.8e-7, windPackThreshT=5, leadLossFactorT=2.9e-7, atmLossFactorT=2.2e-8,
                  dynamicsInc=1, leadlossInc=1, windpackInc=1, atmlossInc=0, saveData=0, plotBudgets=0, plotdaily=0, dx=DX)
        ours = []
        try:
            for _ in range(3):
                t0 = time.perf_counter()
                N.main(y1, m1, d1, y2, m2, d2, **kw)
                ours.append(time.perf_counter() - t0)
            # where main's time goes: the stager alone, and the season + copies alone
            t0 = time.perf_counter()
            st = N.stage_season(y1, y2, startDay, numDays, nDaysY1, "ERA5", "ERA5", "CDR", "OSISAF", "100km", "v11")
            t_stage = time.perf_counter() - t0
            eng = N._engine(su.mask, numDays, DX, "variable", 1, 1, 1, 0)
            import torch
            t0 = time.perf_counter()
            eng.set_forcing(st["precip"], st["conc"], st["wind"], st["drift"], None)
            out = eng.run_season([[5.8e-7, 5., 2.9e-7, 2.2e-8]], ic)
            got = {k: v[0].cpu().numpy() for k, v in out.items()}
            t_gpu = time.perf_counter() - t0
        finally:
            if saved is None:
                sys.modules.pop("utils", None)
            else:
                sys.modules["utils"] = saved
        # ---- the reference's loop on the CPU over the same files (NESOSIM.py:614-649)
        p = O.Params(windPackFactor=5.8e-7, windPackThresh=5., leadLossFactor=2.9e-7, atmLossFactor=2.2e-8)
        fl = O.Flags(atmlossInc=0)
        N.forcingPath = base + "/"
        cpu = []
        s = None
        for _ in range(2):
            t0 = time.perf_counter()
            s = O.gen_empty_arrays(numDays, ny, nx)
            icm = np.load(os.path.join(base, "InitialConditions/ERA5", "ICsnow100km-%dv11" % y1), allow_pickle=True)
            day, year = startDay, y1
            for x in range(numDays - 1):
                day = x + startDay
                year = y1
                if day >= nDaysY1:
                    day -= nDaysY1
                    year = y2
                conc, precip, drift, wind, temp = N.loadData(year, day, "ERA5", "ERA5", "CDR", "OSISAF", "100km", "v11")
                if x == 0:
                    half = O.initial_depths(icm, conc, p)
                    s["snowDepths"][0, 0] = half
                    s["snowDepths"][0, 1] = half
                O.calc_budget(s, conc, precip, drift, wind, temp, mask, DX, x, p, fl)
            cpu.append(time.perf_counter() - t0)
        same = all(bool(np.array_equal(got[k], s[k], equal_nan=True)) for k in got)
        cells = ny * nx * (numDays - 1)
        return {"workload": "one 100 km season (Sep 1 2018 - Apr 30 2019, %d days) from forcing files through the drop-in "
                            "main(saveData=0, plotBudgets=0, plotdaily=0)" % numDays,
                "files": 4 * numDays, "ours_ms": 1e3 * min(ours), "ours_first_call_ms": 1e3 * ours[0],
                "ours_stage_files_ms": 1e3 * t_stage, "ours_h2d_season_d2h_ms": 1e3 * t_gpu,
                "cpu_loop_ms": 1e3 * min(cpu), "cpu_loop": "loadData + calcBudget per day (numpy port), 1 process",
                "speedup": min(cpu) / min(ours), "value": cells / min(ours), "cpu_value": cells / min(cpu), "unit": UNIT,
                "identical_to_cpu_loop": bool(same)}
    finally:
        shutil.rmtree(root, ignore_errors=True)



def run_other_grids(peak):
    """The other single-GPU configurations of BASELINE.json on the general per-day path (one member, full 12-array
    output, forcing resident): the 25 km season and a short stretch of the 5 km grid.  Reported as an extra key next to
    the headline workload, not as bench lines of their own; algorithmic bytes = 96 + 41 per cell-day (M = 1)."""
    import torch
    from nesosim_b200 import synthetic as S
    from nesosim_b200.engine import SnowBudgetEngine
    rows = []
    for name, n, dx, T, gen_days in (("25 km Arctic grid, single season (general day kernel)", 357, 25000, NUM_DAYS, 8),
                                     ("5 km pan-Arctic grid, 40 steps (general day kernel)", 1785, 5000, 41, 4)):
        mask = S.region_mask(dx=dx)      # the real coastline (5 km: the 25 km regrid sampled at the 5 km cell centres)
        gen = S.make_season(mask, gen_days, seed=7)
        idx = np.arange(T) % gen_days
        f = {k: torch.from_numpy(v[idx]).cuda() for k, v in gen.items() if v is not None}
        ic = S.make_ic(mask, seed=7)
        eng = SnowBudgetEngine(mask, T, dx, n_members=1, atmlossInc=1)
        eng.set_path("general")
        eng.set_forcing(f["precip"], f["conc"], f["wind"], f["drift"])
        out = eng.alloc_outputs()
        best = None
        for rep in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            eng.run_season([[5.8e-7, 5., 1.45e-7, 2.2e-8]], ic, out)
            e1.record()
            torch.cuda.synchronize()
            if rep:
                best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
        cells = n * n * (T - 1)
        gbs = cells * 137.0 / (best * 1e-3) / 1e9
        rows.append({"workload": name, "grid": [n, n], "num_days": T, "value": cells / (best * 1e-3), "unit": UNIT,
                     "us_per_day": 1e3 * best / (T - 1), "kernel": "day_step_kernel", "launches": T - 1,
                     "roofline_frac_algorithmic": gbs / peak, "mask": "region_n.msk regridded (grid.bundled_region_mask)",
                     "data": "synthetic (%d generated days repeated)" % gen_days})
        del out, f
        eng.close()
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--members", type=int, default=MEMBERS_PER_GPU)
    ap.add_argument("--days", type=int, default=NUM_DAYS)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--path", default="auto", choices=["auto", "general", "ensemble"])
    ap.add_argument("--variant", default="", help="season-resident kernel build variant (NESOSIM_ENS_VARIANT)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--no-other", action="store_true", help="skip the 25 km / 5 km general-path figures")
    ap.add_argument("--no-extra", action="store_true", help="skip the multi-season, 5 km strips and drop-in main legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the arrays of the last one as DIR/<name>.npy, non-finite "
                         "values as 0 and flagged in DIR/<name>_nonfinite.npy (a fixed sample when they exceed 64 MiB; "
                         "see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
