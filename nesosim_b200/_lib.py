"""ctypes binding of ``libnesosim_b200.so`` (include/nesosim_b200.h).

The library is the product: if it is missing this module raises -- there is no Python/numpy fallback for any
compute entry point.  ``python __graft_entry__.py`` (or ``nesosim_b200.build.build()``) compiles it in-tree.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# NESOSIM_B200_LIB: development override (A/B timing of two builds); the default is the in-tree build
LIB_PATH = os.environ.get("NESOSIM_B200_LIB") or os.path.join(_HERE, "libnesosim_b200.so")

OK = 0
ERR_ARG, ERR_CUDA, ERR_STATE, ERR_NOMEM = -1, -2, -3, -4

# observed quantities of nesosim_set_observations_ex (NESOSIM_OBS_*): snow depth over ice, snow volume, bulk density
OBS_DEPTH, OBS_VOLUME, OBS_DENSITY, OBS_KINDS = 0, 1, 2, 3
# parameter directions of nesosim_run_season_score_grads (NESOSIM_GRAD_DIRS): windPackFactor, leadLossFactor,
# atmLossFactor -- the columns GRAD_PARAMS of a parameter row [WPF, WPT, LLF, ALF] (windPackThresh has no derivative)
GRAD_DIRS = 3
GRAD_PARAMS = (0, 2, 3)
# forcing fields of nesosim_run_season_score_adjoint_forcing (NESOSIM_FORCING_DIRS), in the order of its outputs
FORCING_DIRS = 3
FORCING_FIELDS = ("precip", "wind", "conc")
# drift components of nesosim_run_season_score_adjoint_drift (NESOSIM_DRIFT_DIRS), in the order of its outputs
DRIFT_DIRS = 2
DRIFT_COMPONENTS = ("u", "v")


class NesosimError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("nesosim_b200 error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("ny", C.c_int32), ("nx", C.c_int32), ("num_days", C.c_int32), ("n_members", C.c_int32),
                ("dx", C.c_double), ("deltaT", C.c_double), ("snowDensityFresh", C.c_double),
                ("snowDensityOld", C.c_double), ("minSnowD", C.c_double), ("minConc", C.c_double),
                ("conv_weights", C.c_double * 9), ("conv_divisor", C.c_double),
                ("dynamicsInc", C.c_int32), ("leadlossInc", C.c_int32), ("windpackInc", C.c_int32),
                ("atmlossInc", C.c_int32), ("density_clim", C.c_int32), ("device", C.c_int32)]


class MemberParams(C.Structure):
    _fields_ = [("windPackFactor", C.c_double), ("windPackThresh", C.c_double),
                ("leadLossFactor", C.c_double), ("atmLossFactor", C.c_double)]


OUTPUT_NAMES = ("snowDepths", "density", "snowAcc", "snowOcean", "snowAdv", "snowDiv", "snowLead", "snowAtm",
                "snowWindPackLoss", "snowWindPackGain", "snowWindPack")


class Outputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in OUTPUT_NAMES] + [("depth_member_stride", C.c_int64),
                                                           ("plane_member_stride", C.c_int64)]


_SIGNATURES = {
    "nesosim_abi_version": (C.c_int, []),
    "nesosim_last_error": (C.c_char_p, []),
    "nesosim_device_count": (C.c_int, []),
    "nesosim_create": (C.c_int, [C.POINTER(Config), C.c_void_p, C.POINTER(C.c_void_p)]),
    "nesosim_destroy": (C.c_int, [C.c_void_p]),
    "nesosim_set_forcing": (C.c_int, [C.c_void_p] + [C.c_void_p] * 5),
    "nesosim_set_forcing_sets": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "nesosim_run_season": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int,
                                     C.POINTER(Outputs), C.c_int, C.c_int, C.c_void_p]),
    "nesosim_step_day": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_double, C.POINTER(MemberParams), C.POINTER(Outputs), C.c_void_p]),
    "nesosim_run_season_host": (C.c_int, [C.c_void_p] + [C.c_void_p] * 5 + [C.POINTER(MemberParams), C.c_void_p,
                                                                             C.c_int, C.POINTER(Outputs),
                                                                             C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "nesosim_smooth": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_double,
                                 C.c_void_p]),
    "nesosim_op_dynamics": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "nesosim_op_wind_terms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(MemberParams),
                                        C.c_double, C.c_double, C.c_double] + [C.c_void_p] * 6),
    "nesosim_op_fill_zero": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "nesosim_op_fill_nan_no_negative": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "nesosim_op_density": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_double,
                                     C.c_void_p, C.c_void_p]),
    "nesosim_final_products": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_int64, C.c_double] + [C.c_void_p] * 7),
    "nesosim_launch_count": (C.c_int64, [C.c_void_p]),
    "nesosim_rerun_count": (C.c_int64, [C.c_void_p]),
    "nesosim_unpack_member_array": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "nesosim_host_drain_blocks": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "nesosim_host_drain_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "nesosim_season_kernel_time": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "nesosim_strip_setup": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "nesosim_strip_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nesosim_strip_block": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "nesosim_strip_connect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nesosim_strip_connect_local": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nesosim_strip_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "nesosim_strip_set_timeout": (C.c_int, [C.c_void_p, C.c_double]),
    "nesosim_set_observations": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                           C.POINTER(C.c_int32), C.POINTER(C.c_double)]),
    "nesosim_run_season_misfit": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_void_p]),
    "nesosim_set_observations_sets": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                                C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_double)]),
    "nesosim_set_observations_ex": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                              C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                              C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "nesosim_observation_row_length": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "nesosim_run_season_scores": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "nesosim_set_observations_fp": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                              C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                              C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int64,
                                              C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                              C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                              C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_double)]),
    "nesosim_footprint_row_length": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "nesosim_run_season_scores_fp": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_int64, C.c_void_p]),
    "nesosim_run_season_score_grads": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int, C.c_void_p,
                                                 C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                                 C.c_int64, C.c_void_p]),
    "nesosim_run_season_score_adjoint": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int,
                                                   C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "nesosim_run_season_score_adjoint_forcing": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int,
                                                           C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p,
                                                           C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                                           C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                           C.c_void_p]),
    "nesosim_run_season_score_adjoint_drift": (C.c_int, [C.c_void_p, C.POINTER(MemberParams), C.c_void_p, C.c_int,
                                                         C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p,
                                                         C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, C.c_void_p, C.c_void_p]),
    "nesosim_set_async": (C.c_int, [C.c_void_p, C.c_int]),
    "nesosim_sync": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "nesosim_set_path": (C.c_int, [C.c_void_p, C.c_int]),
    "nesosim_last_path": (C.c_int, [C.c_void_p]),
    "nesosim_const_div_is_fast": (C.c_int, [C.c_double]),
    "nesosim_const_div_eval_host": (C.c_double, [C.c_double, C.c_double]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load the shared library (once) and attach the prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError("libnesosim_b200.so is not built (%s); run `python __graft_entry__.py build`. "
                          "nesosim_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != OK:
        raise NesosimError(code, load().nesosim_last_error().decode("utf-8", "replace"))


def member_params_array(params):
    """(M,4) array-like [WPF, WPT, LLF, ALF] -> ctypes array of MemberParams."""
    p = np.ascontiguousarray(np.asarray(params, dtype=np.float64).reshape(-1, 4))
    arr = (MemberParams * p.shape[0])()
    C.memmove(arr, p.ctypes.data, p.nbytes)
    return arr
