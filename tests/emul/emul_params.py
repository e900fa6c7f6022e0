"""ctypes driver of the per-env-parameter variant of the CUDA source in the host warp emulator (TEST HARNESS ONLY).

tests/emul/tb_emul_params.cpp is tb_emul.cpp plus the variant's entry points (tbp_*).  `EmulWarpP` / `EmulP` are the
`EmulWarp` / `Emul` views of emul.py running that variant with caller-owned parameter rows."""
import ctypes as C
import os
import subprocess

import numpy as np

from emul import emul as E
from tensegrity_rl_b200 import model as M

HERE = os.path.dirname(os.path.abspath(__file__))
NPARAM = 41
_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(HERE, "libtb_emul_params.so")
        csrc = os.path.join(os.path.dirname(os.path.dirname(HERE)), "tensegrity_rl_b200", "csrc")
        deps = [os.path.join(HERE, f) for f in ("tb_emul.cpp", "tb_emul_params.cpp")] + [
            os.path.join(csrc, f) for f in os.listdir(csrc) if f.startswith("tb_")]
        if not os.path.isfile(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off",
                                   "-Wno-unknown-pragmas", "-o", so, os.path.join(HERE, "tb_emul_params.cpp")])
        L = C.CDLL(so)
        L.tbe_create.restype = C.c_char_p
        L.tbp_create.restype = C.c_void_p
        L.tbp_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.tbp_destroy.argtypes = [C.c_void_p]
        _lib = L
    return _lib


P = E.P


class EmulWarpP(E.EmulWarp):
    """n <= 10 envs of the per-env variant in one emulated warp.  rows [n (+ pool slots)][41] are kept and updated in
    place (self.params), as the device keeps d_params; prange [3][41] = nominal, lo, hi of the reset draws (None =
    rows kept at resets)."""

    def __init__(self, xml_file="flat", n=1, rows=None, prange=None, **env_kwargs):
        super().__init__(xml_file, n, **env_kwargs)
        self.L.tbe_destroy(self.h)          # the handle of emul.py's library; this variant lives in its own
        self.L = lib()
        h = C.c_void_p()
        err = self.L.tbe_create(C.byref(self.model), C.byref(self.cfg), C.byref(h))
        if err:
            raise RuntimeError(err.decode())
        self.h = h
        if rows is None:
            rows = np.tile(nominal_params(self.md), (n, 1))
        self.params = np.ascontiguousarray(rows, np.float64)
        self.prange = None if prange is None else np.ascontiguousarray(prange, np.float64)
        self.hp = C.c_void_p(self.L.tbp_create(self.h, P(self.params), P(self.prange)))

    def __del__(self):
        try:
            self.L.tbp_destroy(self.hp)
        except Exception:
            pass
        super().__del__()

    def mj_step(self, ctrl, nstep=1):
        ten = np.zeros((self.n, 9)); cfrc = np.zeros((self.n, 24)); stats = np.zeros((self.n, 6), np.int32)
        c = np.ascontiguousarray(np.broadcast_to(ctrl, (self.n, 6)), np.float64)
        self.L.tbp_mj_step(self.hp, self.n, P(self.rec), P(c), int(nstep), P(ten), P(cfrc), P(stats, C.c_int))
        return ten, cfrc.reshape(self.n, 4, 6), stats

    def mj_step_f32(self, ctrl, nstep=1):
        ten = np.zeros((self.n, 9)); stats = np.zeros((self.n, 6), np.int32)
        c = np.ascontiguousarray(np.broadcast_to(ctrl, (self.n, 6)), np.float64)
        self.L.tbp_mj_step_f32(self.hp, self.n, P(self.rec), P(c), int(nstep), P(ten), P(stats, C.c_int))
        return ten, stats

    def step(self, action):
        a = np.ascontiguousarray(np.broadcast_to(action, (self.n, 6)), np.float64)
        rew = np.zeros(self.n); done = np.zeros(self.n, np.uint8)
        self.L.tbp_step(self.hp, self.n, P(self.rec), P(self.heading), P(a), P(self.obs), P(rew), P(done, C.c_uint8), P(self.info))
        return self.obs.copy(), rew, done.astype(bool), self.info.copy()

    def reset(self, draws=None, seed=0, env_id=0, mask=None):
        if draws is not None:
            self.draws[:] = draws
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self.L.tbp_reset(self.hp, self.n, P(self.rec), P(self.heading), P(self.draws), int(draws is not None),
                         C.c_ulonglong(seed), C.c_longlong(env_id), P(self.obs), P(mk, C.c_uint8))
        return self.obs.copy()

    def forward(self):
        self.L.tbp_forward(self.hp, self.n, P(self.rec), P(self.heading), P(self.obs), P(self.info))
        return self.obs.copy(), self.info.copy()

    def pool(self, n_pool, rec, heading, draws, pool_obs, seed, finish_now=False):
        """one pool advance over records [n + n_pool] (self.params then holds n + n_pool rows)"""
        self.L.tbp_pool(self.hp, self.n, int(n_pool), P(rec), P(heading), P(draws), P(pool_obs), C.c_ulonglong(seed),
                        int(finish_now))


class EmulP(E.Emul):
    """single env of the per-env variant with its parameter row"""

    def __init__(self, xml_file="flat", row=None, **env_kwargs):
        self.w = EmulWarpP(xml_file, 1, rows=None if row is None else np.asarray(row)[None, :], **env_kwargs)
        self.md, self.cfg, self.L = self.w.md, self.w.cfg, self.w.L
        self.rec = self.w.rec[0]
        self.heading = self.w.heading[0]
        self.info = self.w.info[0]
        self.obs = self.w.obs[0]


def nominal_params(md):
    """the nominal parameter row as the CUDA source builds it from the TsgModel struct"""
    m, _keep = M.model_struct(md)
    out = np.zeros(NPARAM)
    lib().tbp_nominal_params(C.byref(m), P(out))
    return out


def param_draws(prange, seed, stream0, nreset, n=1):
    """the parameter rows [n][41] that reset `nreset` of streams stream0 .. stream0 + n - 1 draws"""
    pr = np.ascontiguousarray(prange, np.float64)
    out = np.zeros((n, NPARAM))
    lib().tbp_param_draws(P(out), P(pr), C.c_ulonglong(seed), C.c_ulonglong(stream0), C.c_ulonglong(nreset), int(n))
    return out
