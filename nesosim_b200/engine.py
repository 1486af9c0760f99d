"""Python handle on the native snow-budget context.  PyTorch is used only to own device memory and streams;
every number is computed by ``libnesosim_b200.so`` through the C ABI in ``include/nesosim_b200.h``.
"""
import ctypes as C

import numpy as np

from . import _lib

DEFAULTS = dict(snowDensityFresh=200., snowDensityOld=350., minSnowD=0.02, minConc=0.15, deltaT=60. * 60. * 24.)


def gaussian_kernel_3x3(stddev=1.0, size=3):
    """Host-side weights of ``Gaussian2DKernel(x_stddev=stddev, x_size=size, y_size=size)`` (smooth_snow,
    NESOSIM.py:184).  astropy's own array is used when astropy is installed; otherwise the same closed form
    (amplitude 1/(2*pi*s^2) times exp(-(0.5*x^2/s^2 + 0.5*y^2/s^2)) sampled at integer offsets)."""
    try:   # pragma: no cover - astropy is absent from the build image
        from astropy.convolution import Gaussian2DKernel
        return np.array(Gaussian2DKernel(x_stddev=stddev, x_size=size, y_size=size).array, dtype=np.float64)
    except Exception:
        pass
    s = float(stddev)
    r = np.arange(-(int(size) // 2), int(size) // 2 + 1)
    x, y = np.meshgrid(r, r)
    x = x.astype(float)
    y = y.astype(float)
    a = 0.5 * ((1.0 / s ** 2) + (0.0 / s ** 2))
    c = 0.5 * ((0.0 / s ** 2) + (1.0 / s ** 2))
    return (1. / (2 * np.pi * s * s)) * np.exp(-((a * x ** 2) + (0.0 * x * y) + (c * y ** 2)))


def conv_constants(variant="post_divide", stddev=1.0):
    """(weights[9], divisor) handed to the device.  ``post_divide`` = astropy 3.1-4.x order (raw kernel, then
    ``result /= kernel.sum()``); ``pre_normalised`` = kernel divided by its sum first (divisor 1)."""
    g = gaussian_kernel_3x3(stddev)
    ksum = g.sum()
    if variant == "post_divide":
        return g.reshape(-1).copy(), float(ksum)
    if variant == "pre_normalised":
        return (g / ksum).reshape(-1).copy(), 1.0
    raise ValueError("conv_variant must be 'post_divide' or 'pre_normalised'")


def check_weights(w, name="weights"):
    """The per-kind weights of the adjoint's objective as a tuple of OBS_KINDS floats (None: all ones); ValueError
    unless there are OBS_KINDS of them, each finite and >= 0."""
    if w is None:
        return (1.0,) * _lib.OBS_KINDS
    a = np.asarray(w, dtype=np.float64).ravel()
    if a.shape != (_lib.OBS_KINDS,) or not (np.isfinite(a) & (a >= 0)).all():
        raise ValueError("%s must be %d finite numbers >= 0" % (name, _lib.OBS_KINDS))
    return tuple(float(x) for x in a)


def _torch():
    import torch
    return torch


def region_codes_u8(region_mask):
    """Any numeric mask -> uint8 codes preserving the only two predicates the model tests (>10, <1)."""
    m = np.asarray(region_mask)
    out = np.full(m.shape, 5, dtype=np.uint8)
    with np.errstate(invalid="ignore"):
        out[m > 10] = 11
        out[m < 1] = 0
    return np.ascontiguousarray(out)


class SnowBudgetEngine:
    """One native context: grid + constants + switches for ``n_members`` parameter sets sharing one forcing."""

    def __init__(self, region_mask, num_days, dx, n_members=1, dynamicsInc=1, leadlossInc=1, windpackInc=1,
                 atmlossInc=0, densityType="variable", conv_variant="post_divide", device=0, **consts):
        self.lib = _lib.load()
        mask = region_codes_u8(region_mask)
        self.ny, self.nx = mask.shape
        self.T = int(num_days)
        self.M = int(n_members)
        self.device = int(device)
        k = dict(DEFAULTS)
        k.update(consts)
        cfg = _lib.Config()
        cfg.ny, cfg.nx, cfg.num_days, cfg.n_members = self.ny, self.nx, self.T, self.M
        cfg.dx = float(dx)
        for name in DEFAULTS:
            setattr(cfg, name, float(k[name]))
        w, div = conv_constants(conv_variant)
        cfg.conv_weights = (C.c_double * 9)(*w.tolist())
        cfg.conv_divisor = div
        cfg.dynamicsInc, cfg.leadlossInc, cfg.windpackInc, cfg.atmlossInc = (int(dynamicsInc), int(leadlossInc),
                                                                            int(windpackInc), int(atmlossInc))
        cfg.density_clim = 1 if densityType == "clim" else 0
        cfg.device = self.device
        self.cfg = cfg
        self._weights = w
        self._divisor = div
        handle = C.c_void_p()
        _lib.check(self.lib.nesosim_create(C.byref(cfg), mask.ctypes.data_as(C.c_void_p), C.byref(handle)))
        self.handle = handle
        self._forcing = None

    def close(self):
        if getattr(self, "handle", None):
            self.lib.nesosim_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------ device API
    def _dev(self, a):
        torch = _torch()
        if isinstance(a, torch.Tensor):
            t = a
        else:
            t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
        return t.to(device="cuda:%d" % self.device, dtype=torch.float64).contiguous()

    def set_forcing(self, precip, conc, wind, drift, rho_clim=None):
        """Stage a season of forcing in HBM (arrays (T,ny,nx), drift (T,2,ny,nx); numpy or CUDA tensors)."""
        f = [self._dev(precip), self._dev(conc), self._dev(wind), self._dev(drift)]
        T, ny, nx = self.T, self.ny, self.nx
        assert tuple(f[0].shape) == (T, ny, nx) and tuple(f[3].shape) == (T, 2, ny, nx), "forcing shape"
        rc = None if rho_clim is None else self._dev(rho_clim)
        self._forcing = f + [rc]
        _lib.check(self.lib.nesosim_set_forcing(self.handle, f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr(),
                                                f[3].data_ptr(), None if rc is None else rc.data_ptr()))

    def set_forcing_sets(self, precip, conc, wind, drift, member_set, set_days):
        """A batch of independent seasons: forcing (S,T,ny,nx) / drift (S,T,2,ny,nx); member m runs season
        ``member_set[m]`` for ``set_days[s]`` days (run_multiseason.py as one call; see nesosim_set_forcing_sets)."""
        f = [self._dev(precip), self._dev(conc), self._dev(wind), self._dev(drift)]
        S = f[0].shape[0]
        assert tuple(f[0].shape) == (S, self.T, self.ny, self.nx) and tuple(f[3].shape) == (S, self.T, 2, self.ny, self.nx)
        ms = np.ascontiguousarray(member_set, dtype=np.int32)
        sd = np.ascontiguousarray(set_days, dtype=np.int32)
        assert ms.shape == (self.M,) and sd.shape == (S,)
        self._forcing = f
        _lib.check(self.lib.nesosim_set_forcing_sets(self.handle, S, f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr(),
                                                     f[3].data_ptr(), ms.ctypes.data_as(C.POINTER(C.c_int32)),
                                                     sd.ctypes.data_as(C.POINTER(C.c_int32))))

    def alloc_outputs(self, names=_lib.OUTPUT_NAMES, zero=False):
        """Device tensors shaped like genEmptyArrays (NESOSIM.py:350-376) with a leading member axis."""
        torch = _torch()
        mk = torch.zeros if zero else torch.empty
        dev = "cuda:%d" % self.device
        out = {}
        for n in names:
            shape = (self.M, self.T, 2, self.ny, self.nx) if n == "snowDepths" else (self.M, self.T, self.ny, self.nx)
            out[n] = mk(shape, dtype=torch.float64, device=dev)
        return out

    def _outputs_struct(self, outputs):
        o = _lib.Outputs()
        plane = self.ny * self.nx
        for n in _lib.OUTPUT_NAMES:
            t = outputs.get(n)
            if t is None:
                setattr(o, n, None)
                continue
            assert t.is_contiguous() and t.dtype == _torch().float64
            setattr(o, n, t.data_ptr())
        o.depth_member_stride = self.T * 2 * plane
        o.plane_member_stride = self.T * plane
        return o

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def run_season(self, params, ic=None, outputs=None, first_step=0, num_steps=-1):
        """All members, steps ``first_step .. first_step+num_steps-1``; returns the dict of device tensors."""
        if outputs is None:
            outputs = self.alloc_outputs()
        p = _lib.member_params_array(params)
        assert len(p) == self.M, "need one parameter row per member"
        ic_t = None if ic is None else self._dev(ic)
        per_member = 0
        if ic_t is not None:
            per_member = 1 if (ic_t.dim() == 3 and self.M > 1) else 0
            assert tuple(ic_t.shape[-2:]) == (self.ny, self.nx)
        o = self._outputs_struct(outputs)
        _lib.check(self.lib.nesosim_run_season(self.handle, p, None if ic_t is None else ic_t.data_ptr(), per_member,
                                               C.byref(o), int(first_step), int(num_steps), self._stream()))
        self._keep = (ic_t, outputs)
        return outputs

    def step_day(self, x, conc, precip, drift, wind, params, outputs, rho_new=200.):
        """One ``calcBudget`` (NESOSIM.py:224-347) on explicit day planes; mutates slot x+1 of ``outputs``."""
        p = _lib.member_params_array(params)
        planes = [self._dev(conc), self._dev(precip), self._dev(drift), self._dev(wind)]
        o = self._outputs_struct(outputs)
        _lib.check(self.lib.nesosim_step_day(self.handle, int(x), planes[0].data_ptr(), planes[1].data_ptr(),
                                             planes[2].data_ptr(), planes[3].data_ptr(), float(rho_new), p,
                                             C.byref(o), self._stream()))
        self._keep = (planes, outputs)

    def launch_count(self):
        return int(self.lib.nesosim_launch_count(self.handle))

    def rerun_count(self):
        """Seasons the season-resident kernel handed back to the general kernels (operand-range flag)."""
        return int(self.lib.nesosim_rerun_count(self.handle))

    def host_drain_info(self):
        """(compacted, full_chunks): whether the last `run_season_host` shipped ocean cells only, and how many chunks
        of members had to be copied in full since creation because their land cells were not constant."""
        c, n = C.c_int(0), C.c_int64(0)
        _lib.check(self.lib.nesosim_host_drain_info(self.handle, C.byref(c), C.byref(n)))
        return bool(c.value), int(n.value)

    def host_drain_blocks(self):
        """(packed, plain): the (member, array) blocks of the last `run_season_host` that crossed the link packed (ocean
        cells, scattered by host threads) and whole (copy engine, straight into the caller's arrays)."""
        a, b = C.c_int64(0), C.c_int64(0)
        _lib.check(self.lib.nesosim_host_drain_blocks(self.handle, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def season_kernel_time(self):
        """(total device ms, launches) of the season-resident kernel so far."""
        ms, n = C.c_double(0), C.c_int64(0)
        _lib.check(self.lib.nesosim_season_kernel_time(self.handle, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # ------------------------------------------------------------- strips of a decomposed grid (peer memory)
    def strip_setup(self, has_up, has_down, timeout_s=None):
        """Declare this context a row strip with neighbours above / below (see nesosim_strip_setup)."""
        _lib.check(self.lib.nesosim_strip_setup(self.handle, int(bool(has_up)), int(bool(has_down))))
        if timeout_s is not None:
            _lib.check(self.lib.nesosim_strip_set_timeout(self.handle, float(timeout_s)))

    def strip_export(self):
        """The exchange block as a 64-byte CUDA IPC handle (for a neighbour in another process)."""
        buf = C.create_string_buffer(64)
        _lib.check(self.lib.nesosim_strip_export(self.handle, buf))
        return buf.raw

    def strip_block(self):
        """The exchange block as a device address (for a neighbour in this process)."""
        ptr, n = C.c_void_p(), C.c_int64(0)
        _lib.check(self.lib.nesosim_strip_block(self.handle, C.byref(ptr), C.byref(n)))
        return ptr.value

    def strip_connect(self, up_handle=None, down_handle=None):
        _lib.check(self.lib.nesosim_strip_connect(self.handle, up_handle, down_handle))

    def strip_connect_local(self, up_block=None, down_block=None):
        _lib.check(self.lib.nesosim_strip_connect_local(self.handle, up_block, down_block))

    def strip_timed_out(self):
        v = C.c_int(0)
        _lib.check(self.lib.nesosim_strip_status(self.handle, C.byref(v)))
        return bool(v.value)

    def set_observations(self, obs):
        """Register point observations ``(day, row, col, depth)`` for ``run_season_misfit`` (copied to the device once)."""
        day, row, col = (np.ascontiguousarray(np.asarray(a), dtype=np.int32) for a in obs[:3])
        depth = np.ascontiguousarray(np.asarray(obs[3]), dtype=np.float64)
        n = len(day)
        assert len(row) == n and len(col) == n and len(depth) == n
        i32 = C.POINTER(C.c_int32)
        _lib.check(self.lib.nesosim_set_observations(self.handle, n, day.ctypes.data_as(i32), row.ctypes.data_as(i32),
                                                     col.ctypes.data_as(i32), depth.ctypes.data_as(C.POINTER(C.c_double))))

    def set_observations_sets(self, obs_set, day, row, col, depth):
        """Register observations tagged with the forcing set (season) they belong to, for ``run_season_misfit`` on a
        context with forcing sets (``set_forcing_sets`` first): member m is then scored against the observations of set
        ``member_set[m]`` only (see nesosim_set_observations_sets)."""
        s, day, row, col = (np.ascontiguousarray(np.asarray(a), dtype=np.int32) for a in (obs_set, day, row, col))
        depth = np.ascontiguousarray(np.asarray(depth), dtype=np.float64)
        n = len(day)
        assert len(s) == n and len(row) == n and len(col) == n and len(depth) == n
        i32 = C.POINTER(C.c_int32)
        _lib.check(self.lib.nesosim_set_observations_sets(self.handle, n, s.ctypes.data_as(i32), day.ctypes.data_as(i32),
                                                          row.ctypes.data_as(i32), col.ctypes.data_as(i32),
                                                          depth.ctypes.data_as(C.POINTER(C.c_double))))

    def set_observations_ex(self, day, row, col, value, kind=None, sigma=None, obs_set=None):
        """Register observations of any kind (``_lib.OBS_DEPTH`` / ``OBS_VOLUME`` / ``OBS_DENSITY``; None: all depth) with
        an error each (``sigma``; None: all 1), on one shared forcing or (``obs_set`` given) tagged with their forcing set,
        for ``run_season_scores`` (see nesosim_set_observations_ex)."""
        day, row, col = (np.ascontiguousarray(np.asarray(a), dtype=np.int32) for a in (day, row, col))
        value = np.ascontiguousarray(np.asarray(value), dtype=np.float64)
        n = len(day)
        opt = []
        for a, dt in ((obs_set, np.int32), (kind, np.int32), (sigma, np.float64)):
            a = None if a is None else np.ascontiguousarray(np.asarray(a), dtype=dt)
            assert a is None or len(a) == n
            opt.append(a)
        assert len(row) == n and len(col) == n and len(value) == n
        i32, f64 = C.POINTER(C.c_int32), C.POINTER(C.c_double)
        s, k, sg = (None if a is None else a.ctypes.data_as(t) for a, t in zip(opt, (i32, i32, f64)))
        _lib.check(self.lib.nesosim_set_observations_ex(self.handle, n, s, day.ctypes.data_as(i32), row.ctypes.data_as(i32),
                                                        col.ctypes.data_as(i32), k, value.ctypes.data_as(f64), sg))

    def observation_row_length(self):
        """Entries of a member's model row: the largest number of input observations of one set."""
        n = C.c_int64(0)
        _lib.check(self.lib.nesosim_observation_row_length(self.handle, C.byref(n)))
        return int(n.value)

    def run_season_scores(self, params, ic, model=False):
        """The season with the registered observations scored inside the fused path (nesosim_run_season_scores); returns
        CUDA tensors (chi2[M, OBS_KINDS] float64, used[M, OBS_KINDS] int64, model[M, row_len] float64 or None): per kind
        the sum of ((model - observed)/sigma)^2 and its number of finite terms, and the model value at every input
        observation (NaN on land)."""
        torch = _torch()
        p = _lib.member_params_array(params)
        assert len(p) == self.M
        ic_t = None if ic is None else self._dev(ic)
        per_member = 1 if (ic_t is not None and ic_t.dim() == 3 and self.M > 1) else 0
        dev = "cuda:%d" % self.device
        chi2 = torch.empty(self.M, _lib.OBS_KINDS, dtype=torch.float64, device=dev)
        used = torch.empty(self.M, _lib.OBS_KINDS, dtype=torch.int64, device=dev)
        mod = torch.empty(self.M, self.observation_row_length(), dtype=torch.float64, device=dev) if model else None
        _lib.check(self.lib.nesosim_run_season_scores(self.handle, p, None if ic_t is None else ic_t.data_ptr(), per_member,
                                                      chi2.data_ptr(), used.data_ptr(),
                                                      None if mod is None else mod.data_ptr(),
                                                      0 if mod is None else mod.shape[1], self._stream()))
        self._keep = (ic_t, chi2, used, mod)
        return chi2, used, mod

    def set_observations_fp(self, obs, footprints, obs_set=None, fp_set=None):
        """Register point observations and footprint observations together, for ``run_season_scores_fp`` (see
        nesosim_set_observations_fp).  ``obs``: dict of day, row, col, value, kind, sigma arrays (``ensemble.
        normalize_observations``), or None for no points; ``footprints``: dict of kind, value, sigma (per footprint),
        begin (int64, [n_fp+1]) and day, row, col, weight (per point) arrays (``ensemble.normalize_footprints``);
        ``obs_set`` / ``fp_set``: forcing-set tags of the points / footprints on a context with forcing sets."""
        i32, i64, f64 = C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_double)

        def arr(a, dt, t):
            if a is None:
                return None, None
            a = np.ascontiguousarray(np.asarray(a), dtype=dt)
            return a, a.ctypes.data_as(t)

        n = 0 if obs is None else len(obs["day"])
        po = [arr(None if obs is None else obs[k], dt, t) for k, dt, t in
              (("day", np.int32, i32), ("row", np.int32, i32), ("col", np.int32, i32), ("kind", np.int32, i32),
               ("value", np.float64, f64), ("sigma", np.float64, f64))]
        fp = footprints
        n_fp = len(fp["value"])
        fo = [arr(fp[k], dt, t) for k, dt, t in
              (("kind", np.int32, i32), ("value", np.float64, f64), ("sigma", np.float64, f64), ("begin", np.int64, i64),
               ("day", np.int32, i32), ("row", np.int32, i32), ("col", np.int32, i32), ("weight", np.float64, f64))]
        os_, fs = arr(obs_set, np.int32, i32), arr(fp_set, np.int32, i32)
        assert len(fo[3][0]) == n_fp + 1
        (_, day), (_, row), (_, col), (_, kind), (_, value), (_, sigma) = po
        (_, fkind), (_, fval), (_, fsig), (_, begin), (_, pday), (_, prow), (_, pcol), (_, pw) = fo
        _lib.check(self.lib.nesosim_set_observations_fp(self.handle, n, os_[1], day, row, col, kind, value, sigma,
                                                        n_fp, fs[1], fkind, fval, fsig, begin, pday, prow, pcol, pw))

    def footprint_row_length(self):
        """Entries of a member's footprint model row: the largest number of input footprints of one set."""
        n = C.c_int64(0)
        _lib.check(self.lib.nesosim_footprint_row_length(self.handle, C.byref(n)))
        return int(n.value)

    def run_season_scores_fp(self, params, ic, model=False):
        """``run_season_scores`` with the registered footprints scored too (nesosim_run_season_scores_fp); returns CUDA
        tensors (chi2, used, model) of the point observations as ``run_season_scores`` and (fp_chi2[M, OBS_KINDS]
        float64, fp_used[M, OBS_KINDS] int64, fp_model[M, fp_row_len] float64 or None): per kind the sum of
        ((mean - observed)/sigma)^2 over the footprints and its number of finite terms, and every footprint's model
        value (the weighted mean of its points' model values, NaN when none is finite)."""
        torch = _torch()
        p = _lib.member_params_array(params)
        assert len(p) == self.M
        ic_t = None if ic is None else self._dev(ic)
        per_member = 1 if (ic_t is not None and ic_t.dim() == 3 and self.M > 1) else 0
        dev = "cuda:%d" % self.device
        K = _lib.OBS_KINDS
        chi2 = torch.empty(self.M, K, dtype=torch.float64, device=dev)
        used = torch.empty(self.M, K, dtype=torch.int64, device=dev)
        fp_chi2 = torch.empty(self.M, K, dtype=torch.float64, device=dev)
        fp_used = torch.empty(self.M, K, dtype=torch.int64, device=dev)
        mod = torch.empty(self.M, self.observation_row_length(), dtype=torch.float64, device=dev) if model else None
        fmod = torch.empty(self.M, self.footprint_row_length(), dtype=torch.float64, device=dev) if model else None
        _lib.check(self.lib.nesosim_run_season_scores_fp(
            self.handle, p, None if ic_t is None else ic_t.data_ptr(), per_member, chi2.data_ptr(), used.data_ptr(),
            None if mod is None else mod.data_ptr(), 0 if mod is None else mod.shape[1], fp_chi2.data_ptr(),
            fp_used.data_ptr(), None if fmod is None else fmod.data_ptr(), 0 if fmod is None else fmod.shape[1],
            self._stream()))
        self._keep = (ic_t, chi2, used, mod, fp_chi2, fp_used, fmod)
        return chi2, used, mod, fp_chi2, fp_used, fmod

    def run_season_score_grads(self, params, ic, model=False, jac=False):
        """``run_season_scores_fp`` with the exact derivatives of the scores with respect to windPackFactor,
        leadLossFactor and atmLossFactor (``_lib.GRAD_PARAMS``) of every member (nesosim_run_season_score_grads; needs
        observations registered after ``set_path('general')``).  Returns a dict of CUDA tensors: "chi2", "used",
        "model" (or None) as ``run_season_scores`` and bit-identical to it; "grad" [M, OBS_KINDS, GRAD_DIRS] (d chi2 /
        d theta per kind); with ``jac`` "jac" [M, GRAD_DIRS, row_len] (d model / d theta per observation, NaN where the
        model value is not finite).  With footprints registered also "fp_chi2", "fp_used", "fp_model" (or None),
        "fp_grad" and, with ``jac``, "fp_jac" [M, GRAD_DIRS, fp_row_len].  windPackThresh enters through a step
        function only and has no derivative here."""
        torch = _torch()
        p = _lib.member_params_array(params)
        assert len(p) == self.M
        ic_t = None if ic is None else self._dev(ic)
        per_member = 1 if (ic_t is not None and ic_t.dim() == 3 and self.M > 1) else 0
        dev = "cuda:%d" % self.device
        K, D = _lib.OBS_KINDS, _lib.GRAD_DIRS
        n_row, n_fp = self.observation_row_length(), self.footprint_row_length()
        f64 = dict(dtype=torch.float64, device=dev)
        r = {"chi2": torch.empty(self.M, K, **f64), "used": torch.empty(self.M, K, dtype=torch.int64, device=dev),
             "model": torch.empty(self.M, n_row, **f64) if model else None, "grad": torch.empty(self.M, K, D, **f64),
             "jac": torch.empty(self.M, D, n_row, **f64) if jac else None}
        if n_fp:
            r.update({"fp_chi2": torch.empty(self.M, K, **f64), "fp_used": torch.empty(self.M, K, dtype=torch.int64, device=dev),
                      "fp_model": torch.empty(self.M, n_fp, **f64) if model else None,
                      "fp_grad": torch.empty(self.M, K, D, **f64),
                      "fp_jac": torch.empty(self.M, D, n_fp, **f64) if jac else None})

        def ptr(name):
            t = r.get(name)
            return None if t is None else t.data_ptr()

        def width(name):
            t = r.get(name)
            return 0 if t is None else t.shape[-1]

        _lib.check(self.lib.nesosim_run_season_score_grads(
            self.handle, p, None if ic_t is None else ic_t.data_ptr(), per_member, ptr("chi2"), ptr("used"), ptr("model"),
            width("model"), ptr("grad"), ptr("jac"), width("jac"), ptr("fp_chi2"), ptr("fp_used"), ptr("fp_model"),
            width("fp_model"), ptr("fp_grad"), ptr("fp_jac"), width("fp_jac"), self._stream()))
        self._keep = (ic_t, r)
        return r

    def run_season_score_adjoint(self, params, ic, weights=None, fp_weights=None, model=False, forcing=False,
                                 forcing_days=(), drift=False, drift_days=False):
        """``run_season_scores_fp`` with the reverse-mode derivatives of every member's objective J = sum_k weights[k]
        chi2[k] + sum_k fp_weights[k] fp_chi2[k] (nesosim_run_season_score_adjoint; needs observations registered after
        ``set_path('general')``).  ``weights``, ``fp_weights``: OBS_KINDS finite numbers >= 0 (default all ones).
        Returns a dict of CUDA tensors: "chi2", "used", "model" (or None) and, with footprints registered, "fp_chi2",
        "fp_used", "fp_model" (or None), bit-identical to ``run_season_scores_fp``; "theta_grad" [M, GRAD_DIRS] (dJ /
        d theta for ``_lib.GRAD_PARAMS``) and "ic_grad" [M, ny, nx] (dJ / d ic of each member, also when the IC is
        shared).

        ``forcing=True`` (nesosim_run_season_score_adjoint_forcing) adds the derivatives with respect to the forcing
        fields ``_lib.FORCING_FIELDS`` (precip, wind, conc): "forcing_scale_grad" [M, FORCING_DIRS, ny, nx] (dJ / d alpha
        of a per-cell factor F -> alpha F applied to the whole season) and "forcing_scale_total" [M, FORCING_DIRS] (one
        factor for the whole grid).  ``forcing_days``: any of those names, each adding "<name>_day_grad" [M, T, ny, nx]
        = dJ / d F of every day (8 T bytes per member-cell each).  ``forcing_days`` without ``forcing=True`` or with an
        unknown name raises ValueError before any device work.

        ``drift=True`` (nesosim_run_season_score_adjoint_drift; combines freely with ``forcing``) adds the derivatives
        with respect to the ice drift components ``_lib.DRIFT_COMPONENTS`` (u, v): "drift_scale_grad" [M, DRIFT_DIRS,
        ny, nx] (dJ / d alpha of a per-cell factor scaling one component over the whole season) and "drift_scale_total"
        [M, DRIFT_DIRS]; the derivative for one drift speed factor (u, v) -> alpha (u, v) is the sum of the two totals.
        ``drift_days=True`` also adds "drift_day_grad" [M, T, DRIFT_DIRS, ny, nx] = dJ / d drift of every day, in the
        staged drift's layout (16 T bytes per member-cell).  ``drift_days`` without ``drift=True`` raises ValueError
        before any device work.  Without dynamics (dynamicsInc=0) the drift outputs are 0."""
        torch = _torch()
        K, D = _lib.OBS_KINDS, _lib.GRAD_DIRS
        forcing_days = tuple(forcing_days)
        bad = [n for n in forcing_days if n not in _lib.FORCING_FIELDS]
        if bad:
            raise ValueError("forcing_days: unknown field(s) %s; expected any of %s" % (bad, _lib.FORCING_FIELDS))
        if forcing_days and not forcing:
            raise ValueError("forcing_days needs forcing=True")
        if drift_days and not drift:
            raise ValueError("drift_days needs drift=True")
        w = check_weights(weights, "weights")
        fw = check_weights(fp_weights, "fp_weights")
        p = _lib.member_params_array(params)
        assert len(p) == self.M
        ic_t = None if ic is None else self._dev(ic)
        per_member = 1 if (ic_t is not None and ic_t.dim() == 3 and self.M > 1) else 0
        dev = "cuda:%d" % self.device
        n_row, n_fp = self.observation_row_length(), self.footprint_row_length()
        f64 = dict(dtype=torch.float64, device=dev)
        r = {"chi2": torch.empty(self.M, K, **f64), "used": torch.empty(self.M, K, dtype=torch.int64, device=dev),
             "model": torch.empty(self.M, n_row, **f64) if model else None,
             "theta_grad": torch.empty(self.M, D, **f64), "ic_grad": torch.empty(self.M, self.ny, self.nx, **f64)}
        if n_fp:
            r.update({"fp_chi2": torch.empty(self.M, K, **f64), "fp_used": torch.empty(self.M, K, dtype=torch.int64, device=dev),
                      "fp_model": torch.empty(self.M, n_fp, **f64) if model else None})

        def ptr(name):
            t = r.get(name)
            return None if t is None else t.data_ptr()

        def width(name):
            t = r.get(name)
            return 0 if t is None else t.shape[-1]

        cw, cfw = (C.c_double * K)(*w), (C.c_double * K)(*fw)
        args = (self.handle, p, None if ic_t is None else ic_t.data_ptr(), per_member, cw, cfw, ptr("chi2"), ptr("used"),
                ptr("model"), width("model"), ptr("fp_chi2"), ptr("fp_used"), ptr("fp_model"), width("fp_model"),
                ptr("theta_grad"), ptr("ic_grad"))
        if forcing:
            F = _lib.FORCING_DIRS
            r["forcing_scale_grad"] = torch.empty(self.M, F, self.ny, self.nx, **f64)
            r["forcing_scale_total"] = torch.empty(self.M, F, **f64)
            for n in forcing_days:
                r[n + "_day_grad"] = torch.empty(self.M, self.T, self.ny, self.nx, **f64)
        days = [ptr(n + "_day_grad") for n in _lib.FORCING_FIELDS]
        if drift:
            Dd = _lib.DRIFT_DIRS
            r["drift_scale_grad"] = torch.empty(self.M, Dd, self.ny, self.nx, **f64)
            r["drift_scale_total"] = torch.empty(self.M, Dd, **f64)
            if drift_days:
                r["drift_day_grad"] = torch.empty(self.M, self.T, Dd, self.ny, self.nx, **f64)
            _lib.check(self.lib.nesosim_run_season_score_adjoint_drift(
                *args, ptr("forcing_scale_grad"), ptr("forcing_scale_total"), *days, ptr("drift_scale_grad"),
                ptr("drift_scale_total"), ptr("drift_day_grad"), self._stream()))
        elif forcing:
            _lib.check(self.lib.nesosim_run_season_score_adjoint_forcing(
                *args, ptr("forcing_scale_grad"), ptr("forcing_scale_total"), *days, self._stream()))
        else:
            _lib.check(self.lib.nesosim_run_season_score_adjoint(*args, self._stream()))
        self._keep = (ic_t, r)
        return r

    def run_season_misfit(self, params, ic, obs=None):
        """The season with the calibration misfit reduced INSIDE the season-resident kernel (nesosim_run_season_misfit;
        after ``set_path('general')``: sampled by the general day kernel, on any grid) against the registered
        observations (``obs`` given: registered first); returns CUDA tensors (misfit[M] float64, used[M] int64).  No
        output array is written."""
        torch = _torch()
        if obs is not None:
            self.set_observations(obs)
        p = _lib.member_params_array(params)
        assert len(p) == self.M
        ic_t = None if ic is None else self._dev(ic)
        per_member = 1 if (ic_t is not None and ic_t.dim() == 3 and self.M > 1) else 0
        dev = "cuda:%d" % self.device
        mis = torch.empty(self.M, dtype=torch.float64, device=dev)
        used = torch.empty(self.M, dtype=torch.int64, device=dev)
        _lib.check(self.lib.nesosim_run_season_misfit(self.handle, p, None if ic_t is None else ic_t.data_ptr(), per_member,
                                                      mis.data_ptr(), used.data_ptr(), self._stream()))
        self._keep = (ic_t, mis, used)
        return mis, used

    def set_async(self, on=True):
        """Asynchronous mode (nesosim_set_async): ``run_season`` never synchronises its stream; call ``sync()`` before
        using a season's outputs or reusing its buffers."""
        _lib.check(self.lib.nesosim_set_async(self.handle, int(bool(on))))

    def sync(self):
        """Wait for every season enqueued in asynchronous mode; returns how many had to be redone by the general
        kernels (operand-range flag; 0 on physical data)."""
        n = C.c_int(0)
        _lib.check(self.lib.nesosim_sync(self.handle, C.byref(n)))
        return n.value

    PATHS = {"auto": 0, "general": 1, "ensemble": 2}

    def set_path(self, path):
        """'auto' | 'general' (per-day kernel) | 'ensemble' (season-resident cluster kernel).  Observations registered
        after ``set_path('general')`` are scored by the general day kernel on any grid (``run_season_misfit``,
        ``run_season_scores``, ``run_season_scores_fp``: the same fixed order as the season kernel, bit for bit);
        changing the path afterwards makes those calls fail until the observations are registered again."""
        _lib.check(self.lib.nesosim_set_path(self.handle, self.PATHS[path]))

    def last_path(self):
        return {0: None, 1: "general", 2: "ensemble"}[int(self.lib.nesosim_last_path(self.handle))]

    def dominant_kernel(self):
        return {"general": "day_step_kernel", "ensemble": "ensemble_season_kernel"}.get(self.last_path(), "?")

    # -------------------------------------------------------------------------------------------- host API
    def run_season_host(self, forcing, params, ic=None, outputs=None, names=_lib.OUTPUT_NAMES):
        """End-to-end call on HOST numpy arrays (H2D + season + D2H inside).  Returns (outputs, h2d, d2h)."""
        T, ny, nx, M = self.T, self.ny, self.nx, self.M
        if outputs is None:
            outputs = {}
            for n in names:
                shape = (M, T, 2, ny, nx) if n == "snowDepths" else (M, T, ny, nx)
                outputs[n] = np.empty(shape, dtype=np.float64)

        def hp(a):
            if a is None:
                return None
            if hasattr(a, "data_ptr"):      # pinned torch CPU tensor
                return C.c_void_p(a.data_ptr())
            assert a.dtype == np.float64 and a.flags.c_contiguous
            return a.ctypes.data_as(C.c_void_p)

        o = _lib.Outputs()
        for n in _lib.OUTPUT_NAMES:
            setattr(o, n, hp(outputs.get(n)))
        plane = ny * nx
        o.depth_member_stride = T * 2 * plane
        o.plane_member_stride = T * plane
        p = _lib.member_params_array(params)
        per_member = 0
        if ic is not None and getattr(ic, "ndim", 2) == 3 and M > 1:
            per_member = 1
        up, down = C.c_int64(0), C.c_int64(0)
        _lib.check(self.lib.nesosim_run_season_host(self.handle, hp(forcing["precip"]), hp(forcing["conc"]),
                                                    hp(forcing["wind"]), hp(forcing["drift"]),
                                                    hp(forcing.get("rho_clim")), p, hp(ic), per_member,
                                                    C.byref(o), C.byref(up), C.byref(down)))
        return outputs, up.value, down.value


# -------------------------------------------------------------------------------- per-function device ops

def _cuda(a, device=0, dtype=None):
    torch = _torch()
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
    return t.to(device="cuda:%d" % device, dtype=dtype or t.dtype).contiguous()


def _cur_stream(device=0):
    return C.c_void_p(_torch().cuda.current_stream(device).cuda_stream)


def smooth(arr, conv_variant="post_divide", device=0, stddev=1.0):
    """``smooth_snow`` (NESOSIM.py:170-187) on the GPU; numpy in, numpy out (new array, as the reference).
    ``stddev`` is the Gaussian's sigma (1 in smooth_snow; ``sigma_factor`` in utils.int_smooth_drifts_v2/v3)."""
    torch = _torch()
    lib = _lib.load()
    a = _cuda(np.asarray(arr, dtype=np.float64), device)
    out = torch.empty_like(a)
    w, div = conv_constants(conv_variant, stddev)
    wc = (C.c_double * 9)(*w.tolist())
    _lib.check(lib.nesosim_smooth(a.data_ptr(), out.data_ptr(), a.shape[0], a.shape[1], wc, div, _cur_stream(device)))
    return out.cpu().numpy()


def op_dynamics(drift, depths, dx, deltaT=86400., device=0):
    torch = _torch()
    lib = _lib.load()
    d = _cuda(np.asarray(drift, dtype=np.float64), device)
    h = _cuda(np.asarray(depths, dtype=np.float64), device)
    adv = torch.empty_like(h)
    div = torch.empty_like(h)
    _lib.check(lib.nesosim_op_dynamics(d.data_ptr(), h.data_ptr(), float(dx), float(deltaT), h.shape[1], h.shape[2],
                                       adv.data_ptr(), div.data_ptr(), _cur_stream(device)))
    return adv.cpu().numpy(), div.cpu().numpy()


def op_wind_terms(h0, wind, conc, params, deltaT=86400., rhoFresh=200., rhoOld=350., device=0):
    torch = _torch()
    lib = _lib.load()
    a = [_cuda(np.asarray(v, dtype=np.float64), device) for v in (h0, wind, conc)]
    outs = [torch.empty_like(a[0]) for _ in range(5)]
    p = _lib.member_params_array(params)
    _lib.check(lib.nesosim_op_wind_terms(a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(), a[0].numel(), p,
                                         float(deltaT), float(rhoFresh), float(rhoOld),
                                         *[o.data_ptr() for o in outs], _cur_stream(device)))
    return [o.cpu().numpy() for o in outs]


def op_fill_zero(arr, device=0):
    lib = _lib.load()
    a = _cuda(np.array(arr, dtype=np.float64), device)
    _lib.check(lib.nesosim_op_fill_zero(a.data_ptr(), a.numel(), _cur_stream(device)))
    return a.cpu().numpy()


def op_fill_nan_no_negative(arr, mask, negative_to_zero=True, device=0):
    lib = _lib.load()
    a = _cuda(np.array(arr, dtype=np.float64), device)
    m = _cuda(region_codes_u8(mask), device)
    _lib.check(lib.nesosim_op_fill_nan_no_negative(a.data_ptr(), m.data_ptr(), a.numel(), int(bool(negative_to_zero)),
                                                   _cur_stream(device)))
    return a.cpu().numpy()


def op_density(depths, mask, rhoFresh=200., rhoOld=350., minSnowD=0.02, device=0):
    torch = _torch()
    lib = _lib.load()
    h = _cuda(np.asarray(depths, dtype=np.float64), device)
    m = _cuda(region_codes_u8(mask), device)
    rho = torch.empty_like(h[0])
    _lib.check(lib.nesosim_op_density(h.data_ptr(), m.data_ptr(), rho.numel(), float(rhoFresh), float(rhoOld),
                                      float(minSnowD), rho.data_ptr(), _cur_stream(device)))
    return rho.cpu().numpy()


FINAL_NAMES = ("snow_depth", "snow_volume", "snow_density", "ice_concentration", "precipitation", "wind_speed")


def final_products(snowDepths, density, iceConc, precip, wind, ice_conc_mask=0.5, device=0, out=None):
    """The float32 fields of ``final/NESOSIMv11_*.nc`` (``OutputSnowModelFinal``, utils.py:161-179, fed as ``main`` feeds
    it, NESOSIM.py:654) computed in one fused pass on the GPU.  Inputs: (T,2,ny,nx) depths and (T,ny,nx) arrays of one
    member, or an ensemble's (M,T,2,ny,nx) / (M,T,ny,nx) depths and density with the (T,ny,nx) forcing all members
    share; numpy or CUDA tensors.  Returns a dict of float32 CUDA tensors shaped like ``density``."""
    torch = _torch()
    lib = _lib.load()
    d = _cuda(snowDepths, device, torch.float64)
    rho = _cuda(density, device, torch.float64)
    forcing = [_cuda(a, device, torch.float64) for a in (iceConc, precip, wind)]
    T, ny, nx = forcing[0].shape
    days = rho.numel() // (ny * nx)
    assert d.numel() == 2 * rho.numel() and days % T == 0
    if out is None:
        out = {n: torch.empty(tuple(rho.shape), dtype=torch.float32, device=d.device) for n in FINAL_NAMES}
    _lib.check(lib.nesosim_final_products(d.data_ptr(), rho.data_ptr(), forcing[0].data_ptr(), forcing[1].data_ptr(),
                                          forcing[2].data_ptr(), days, T, ny * nx, float(ice_conc_mask),
                                          out["snow_depth"].data_ptr(), out["snow_volume"].data_ptr(),
                                          out["snow_density"].data_ptr(), out["ice_concentration"].data_ptr(),
                                          out["precipitation"].data_ptr(), out["wind_speed"].data_ptr(), _cur_stream(device)))
    return out


def smooth_gridded_drift(driftFGx, driftFGy, sigma_factor=1, x_size_val=3, conv_variant="post_divide", device=0):
    """The smoothing tail of the reference's offline drift regridders ``utils.int_smooth_drifts_v2/v3``
    (utils.py:283-291, 328-336): ``convolve(component, Gaussian2DKernel(sigma_factor, x_size=3))`` -- here NaNs DO reach
    the convolution, so astropy's NaN-interpolating branch runs -- then masked where the gridded input was NaN.
    Returns the (2, nx, ny) masked array the reference returns.  (The Delaunay / griddata interpolation before it
    stays on the CPU.)"""
    import numpy.ma as ma
    if int(x_size_val) != 3:
        raise ValueError("the native smoother is the reference's 3x3 kernel (x_size_val=3)")
    out = ma.masked_all((2,) + tuple(np.shape(driftFGx)))
    for i, comp in enumerate((driftFGx, driftFGy)):
        comp = np.asarray(comp, dtype=np.float64)
        out[i] = ma.masked_where(np.isnan(comp), smooth(comp, conv_variant, device, stddev=float(sigma_factor)))
    return out
