"""ctypes binding of libtsg.so (include/tsg.h).  There is NO CPU path: loading fails loudly if the
CUDA library is missing, and tsg_create fails if there is no sm_100 device."""
import ctypes as C
import os

from . import build as _build
from . import model as _M
from .model import TsgEnvConfig, TsgModel

STATE_STRIDE, INFO_DIM, NDRAW, HEADING_SLOTS = 96, 32, 10, 32
CTRL_F64, CTRL_F32 = 0, 1
INFO = dict(rew_fwd=0, rew_ctrl=1, rew_survive=2, x=3, y=4, psi=5, xvel=6, yvel=7, ten=8, terminated=17,
            truncated=18, ncon=19, niter=20, nls=21, barforce=22, maxcfrc=23, waypt=24, ori=26, overflow=28,
            bad=29, nmpr=30, reset_psi=31)
# per-env parameter row (TSG_PARAM_*): field -> slice of the TSG_NPARAM doubles
NPARAM = _M.NPARAM
PARAM = {name: slice(off, off + w) for name, off, w in _M.PARAM_FIELDS}

SYMBOLS = ["tsg_last_error", "tsg_version", "tsg_device_count", "tsg_create", "tsg_create_pooled", "tsg_pool_stats_host", "tsg_destroy", "tsg_num_envs",
           "tsg_obs_dim", "tsg_launches", "tsg_kernel_config", "tsg_reset", "tsg_step", "tsg_forward",
           "tsg_get_state_host", "tsg_set_state_host", "tsg_get_records_host", "tsg_set_records_host",
           "tsg_get_draws_host", "tsg_step_host", "tsg_reset_host", "tsg_set_real_obs", "tsg_get_real_obs_host",
           "tsg_create_opts", "tsg_precision", "tsg_forward_host", "tsg_get_heading_host", "tsg_set_heading_host",
           "tsg_set_param_ranges", "tsg_set_env_params", "tsg_get_env_params"]
PRECISION = {"f64": 0, "f32": 1}


class TsgError(RuntimeError):
    pass


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    so = os.environ.get("TSG_LIB", _build.SO)  # alternative builds for A/B measurements
    if not os.path.isfile(so):
        raise TsgError(f"{so} not built: run `python -m tensegrity_rl_b200.build` (needs nvcc); "
                       "there is no CPU fallback")
    if so == _build.SO and _build.is_stale():   # an .so built from other sources would load with a silent ABI skew
        raise TsgError(f"{so} is stale (sources or flags changed since it was built): "
                       "run `python -m tensegrity_rl_b200.build`")
    L = C.CDLL(so)
    vp, dp, fp, u8p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
    L.tsg_last_error.restype = C.c_char_p
    L.tsg_create.argtypes = [C.POINTER(TsgModel), C.POINTER(TsgEnvConfig), C.c_int, C.c_int, C.c_longlong, C.POINTER(vp)]
    L.tsg_create_pooled.argtypes = [C.POINTER(TsgModel), C.POINTER(TsgEnvConfig), C.c_int, C.c_int, C.c_int, C.c_longlong, C.POINTER(vp)]
    L.tsg_create_opts.argtypes = [C.POINTER(TsgModel), C.POINTER(TsgEnvConfig), C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, C.POINTER(vp)]
    L.tsg_pool_stats_host.argtypes = [vp, C.POINTER(C.c_int)]
    L.tsg_destroy.argtypes = [vp]
    for f in ("tsg_num_envs", "tsg_obs_dim", "tsg_launches", "tsg_precision"):
        getattr(L, f).argtypes = [vp]
    L.tsg_kernel_config.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.tsg_reset.argtypes = [vp, u8p, C.c_ulonglong, dp, dp, fp, dp, vp]
    L.tsg_step.argtypes = [vp, vp, C.c_int, dp, fp, dp, u8p, dp, C.c_int, C.c_ulonglong, dp, vp]
    L.tsg_forward.argtypes = [vp, dp, dp, vp]
    L.tsg_get_state_host.argtypes = [vp, dp, dp, dp, dp, dp]
    L.tsg_set_state_host.argtypes = [vp, dp, dp, dp, dp, dp]
    L.tsg_get_records_host.argtypes = [vp, dp]
    L.tsg_set_records_host.argtypes = [vp, dp]
    L.tsg_get_draws_host.argtypes = [vp, dp]
    L.tsg_forward_host.argtypes = [vp, dp, dp]
    L.tsg_get_heading_host.argtypes = [vp, dp]
    L.tsg_set_heading_host.argtypes = [vp, dp]
    L.tsg_step_host.argtypes = [vp, dp, dp, dp, u8p, dp, C.c_int, C.c_ulonglong, dp]
    L.tsg_reset_host.argtypes = [vp, u8p, C.c_ulonglong, dp, dp]
    L.tsg_set_real_obs.argtypes = [vp, dp]
    L.tsg_get_real_obs_host.argtypes = [vp, dp]
    L.tsg_set_param_ranges.argtypes = [vp, dp, dp]
    L.tsg_set_env_params.argtypes = [vp, dp, u8p, vp]
    L.tsg_get_env_params.argtypes = [vp, dp, vp]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise TsgError(load().tsg_last_error().decode())
