"""ctypes driver of the host warp emulator of the CUDA source (TEST HARNESS ONLY).

tests/emul/tb_emul.cpp compiles csrc/tb_*.cuh as plain C++ and runs one 32-lane warp of it as cooperative fibres.
`Emul` is the single-env view the parity tests use; `EmulWarp` steps up to 10 envs in one warp, which exercises the
predication of envs that need different numbers of Newton iterations / line-search evaluations / contacts.  Both run
the per-env-parameter variant of the kernels when given parameter rows, the default variant otherwise."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from tensegrity_rl_b200 import model as M

HERE = os.path.dirname(os.path.abspath(__file__))
STATE_STRIDE, INFO_DIM, HEADING_SLOTS, NDRAW = 96, 32, 32, 10
EPW = 10
NPARAM = 41
_lib = None


def lib():
    """libtb_emul.so, compiled on first use into the temporary directory (the test tree may be read-only), under a
    name that hashes the sources and flags it is built from"""
    global _lib
    if _lib is None:
        csrc = os.path.join(os.path.dirname(os.path.dirname(HERE)), "tensegrity_rl_b200", "csrc")
        src = os.path.join(HERE, "tb_emul.cpp")
        cmd = ["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-Wno-unknown-pragmas"]
        h = hashlib.sha256(" ".join(cmd).encode())
        for d in [src] + sorted(os.path.join(csrc, f) for f in os.listdir(csrc) if f.startswith("tb_")):
            h.update(open(d, "rb").read())
        so = os.path.join(tempfile.gettempdir(), "libtb_emul-%d-%s.so" % (os.getuid(), h.hexdigest()[:16]))
        if not os.path.isfile(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(cmd + ["-o", tmp, src])
            os.replace(tmp, so)      # whole files only, for concurrent test processes
        L = C.CDLL(so)
        L.tbe_create.restype = C.c_char_p
        assert L.tbe_envs_per_warp() == EPW
        _lib = L
    return _lib


def P(a, t=C.c_double):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


class EmulWarp:
    """n <= 10 envs stepped together by one emulated warp.  With rows [n (+ pool slots)][41] the per-env variant runs:
    the rows are kept and updated in place (self.params), as the device keeps d_params; prange [3][41] = nominal, lo,
    hi of the reset draws (None = rows kept at resets)."""

    def __init__(self, xml_file="flat", n=1, rows=None, prange=None, **env_kwargs):
        assert 1 <= n <= EPW
        if prange is not None and rows is None:
            raise ValueError("prange needs parameter rows")
        self.n = n
        self.md = M.load_model(xml_file)
        self.model, self._keep = M.model_struct(self.md)
        self.cfg = M.env_config(self.md, **env_kwargs)
        self.L = lib()
        h = C.c_void_p()
        err = self.L.tbe_create(C.byref(self.model), C.byref(self.cfg), C.byref(h))
        if err:
            raise RuntimeError(err.decode())
        self.h = h
        self.rec = np.zeros((n, STATE_STRIDE))
        self.heading = np.zeros((n, HEADING_SLOTS))
        self.obs = np.zeros((n, self.cfg.obs_dim))
        self.info = np.zeros((n, INFO_DIM))
        self.draws = np.zeros((n, NDRAW))
        self.rec[:, 0:21] = self.md["qpos0"]
        self.real_obs = None
        self.params = None if rows is None else np.ascontiguousarray(rows, np.float64)
        self.prange = None if prange is None else np.ascontiguousarray(prange, np.float64)
        self.L.tbe_set_params(self.h, P(self.params), P(self.prange))

    def __del__(self):
        try:
            self.L.tbe_destroy(self.h)
        except Exception:
            pass

    def mj_step(self, ctrl, nstep=1):
        ten = np.zeros((self.n, 9)); cfrc = np.zeros((self.n, 24)); stats = np.zeros((self.n, 6), np.int32)
        c = np.ascontiguousarray(np.broadcast_to(ctrl, (self.n, 6)), np.float64)
        self.L.tbe_mj_step(self.h, self.n, P(self.rec), P(c), int(nstep), P(ten), P(cfrc), P(stats, C.c_int))
        return ten, cfrc.reshape(self.n, 4, 6), stats

    def mj_step_f32(self, ctrl, nstep=1):
        """the same through the optional fp32 mode (fp32 kinematics / tendons / collision / integration, fp64 narrow
        phase and constraint solver); the records stay fp64"""
        ten = np.zeros((self.n, 9)); stats = np.zeros((self.n, 6), np.int32)
        c = np.ascontiguousarray(np.broadcast_to(ctrl, (self.n, 6)), np.float64)
        self.L.tbe_mj_step_f32(self.h, self.n, P(self.rec), P(c), int(nstep), P(ten), P(stats, C.c_int))
        return ten, stats

    def step(self, action):
        a = np.ascontiguousarray(np.broadcast_to(action, (self.n, 6)), np.float64)
        rew = np.zeros(self.n); done = np.zeros(self.n, np.uint8)
        self.L.tbe_step(self.h, self.n, P(self.rec), P(self.heading), P(a), P(self.obs), P(rew), P(done, C.c_uint8), P(self.info))
        return self.obs.copy(), rew, done.astype(bool), self.info.copy()

    def reset(self, draws=None, seed=0, env_id=0, mask=None):
        if draws is not None:
            self.draws[:] = draws
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self.L.tbe_reset(self.h, self.n, P(self.rec), P(self.heading), P(self.draws), int(draws is not None),
                         C.c_ulonglong(seed), C.c_longlong(env_id), P(self.obs), P(mk, C.c_uint8))
        return self.obs.copy()

    def set_noise(self, seed, env_id=0):
        """observation-noise keys; the true observation of every step / reset then lands in self.real_obs"""
        self.real_obs = np.zeros((self.n, self.cfg.obs_dim))
        self.L.tbe_set_noise(self.h, C.c_ulonglong(seed), C.c_longlong(env_id), P(self.real_obs))

    def forward(self):
        self.L.tbe_forward(self.h, self.n, P(self.rec), P(self.heading), P(self.obs), P(self.info))
        return self.obs.copy(), self.info.copy()

    def pool(self, n_pool, rec, heading, draws, pool_obs, seed, finish_now=False):
        """one pool advance over records [n + n_pool] (self.params, if set, then holds n + n_pool rows)"""
        self.L.tbe_pool(self.h, self.n, int(n_pool), P(rec), P(heading), P(draws), P(pool_obs), C.c_ulonglong(seed),
                        int(finish_now))


class Emul:
    """single env (the other 9 env slots of the warp idle), with its parameter row if one is given"""

    def __init__(self, xml_file="flat", row=None, **env_kwargs):
        self.w = EmulWarp(xml_file, 1, rows=None if row is None else np.asarray(row)[None, :], **env_kwargs)
        self.md, self.cfg, self.L = self.w.md, self.w.cfg, self.w.L
        self.rec = self.w.rec[0]
        self.heading = self.w.heading[0]
        self.info = self.w.info[0]
        self.obs = self.w.obs[0]

    # state record views
    @property
    def qpos(self): return self.rec[0:21]
    @property
    def qvel(self): return self.rec[21:39]
    @property
    def warm(self): return self.rec[39:57]
    @property
    def ctrl(self): return self.rec[57:63]
    @property
    def act(self): return self.rec[63:69]
    @property
    def real_obs(self): return self.w.real_obs[0]

    def mj_step(self, ctrl, nstep=1):
        ten, cfrc, stats = self.w.mj_step(ctrl, nstep)
        return ten[0], cfrc[0], stats[0]

    def step(self, action):
        o, r, d, i = self.w.step(action)
        return o[0], float(r[0]), bool(d[0]), i[0]

    def reset(self, draws=None, seed=0, env_id=0):
        return self.w.reset(draws, seed, env_id)[0]

    def set_noise(self, seed, env_id=0):
        self.w.set_noise(seed, env_id)

    def forward(self):
        o, i = self.w.forward()
        return o[0], i[0]


def reset_noise(seed, stream, nreset):
    """the 21 uniform(-1, 1) qpos offsets and 18 standard-normal qvel values of reset `nreset` of stream `stream`"""
    out = np.zeros(39)
    lib().tbe_reset_noise(C.c_ulonglong(seed), C.c_ulonglong(stream), C.c_ulonglong(nreset), P(out))
    return out[:21], out[21:]


def obs_normals(seed, stream, nreset, step, n):
    """the standard-normal draws the CUDA source uses for the observation of (stream, reset count, episode step)"""
    out = np.zeros(n + 1)
    lib().tbe_obs_normals(C.c_ulonglong(seed), C.c_ulonglong(stream), C.c_ulonglong(nreset), C.c_ulonglong(step),
                          int(n), P(out))
    return out[:n]


def nominal_params(md):
    """the nominal parameter row as the CUDA source builds it from the TsgModel struct"""
    m, _keep = M.model_struct(md)
    out = np.zeros(NPARAM)
    lib().tbe_nominal_params(C.byref(m), P(out))
    return out


def param_draws(prange, seed, stream0, nreset, n=1):
    """the parameter rows [n][41] that reset `nreset` of streams stream0 .. stream0 + n - 1 draws"""
    pr = np.ascontiguousarray(prange, np.float64)
    out = np.zeros((n, NPARAM))
    lib().tbe_param_draws(P(out), P(pr), C.c_ulonglong(seed), C.c_ulonglong(stream0), C.c_ulonglong(nreset), int(n))
    return out
