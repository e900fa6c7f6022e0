"""Single-env classes with the reference's names and signatures, backed by the CUDA library.

    tr_env(xml_file=..., is_test=..., desired_action=..., desired_direction=..., terminate_when_unhealthy=...)
    tensegrity_env(...)

mirror /root/reference/tr_env/tr_env/envs/tr_env.py:20 and
/root/reference/tensegrity_env/tensegrity_env/envs/tensegrity_env.py:20 as seen through gym 0.26:
`reset(seed=None, options=None) -> (obs, info)`, `step(a) -> (obs, reward, terminated, truncated, info)`,
`dt`, `observation_space`, `action_space`, `data.contact` / `model` (shims for run.py:155-160).
Each call goes through the C ABI with HOST buffers (tsg_step_host / tsg_reset_host): N = 1 view of the
same kernels the batched `TensegrityVecEnv` launches.  `make(id, **kwargs)` stands in for `gym.make`
(adds the TimeLimit of the registration, tr_env/tr_env/__init__.py:3-7); when gym is importable the ids
`tr_env-v0` / `tensegrity_env-v0` are registered too.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import lib as _lib
from . import model as M
from .spaces import Box


class _Contact:
    def __init__(self, geom1, geom2, force):
        self.geom1, self.geom2, self._force = geom1, geom2, force


class _DataShim:
    """The slice of mjData the reference scripts read."""

    def __init__(self, env):
        self._env = env
        self.contact = []

    def _state(self):
        return self._env._get_state()

    qpos = property(lambda s: s._state()["qpos"][0])
    qvel = property(lambda s: s._state()["qvel"][0])
    ctrl = property(lambda s: s._state()["ctrl"][0])
    act = property(lambda s: s._state()["act"][0])
    ten_length = property(lambda s: np.array(s._env._last_info[_lib.INFO["ten"]:_lib.INFO["ten"] + 9]))


def mj_contactForce(model, data, j, out):
    """Stand-in for mujoco.mj_contactForce on the shim contacts (run.py:158): the bar-bar contacts of a
    step are aggregated into one entry carrying their summed force magnitude."""
    out[:] = 0
    out[0] = data.contact[j]._force


class _SingleEnv:
    env_kind = "tr_env"
    metadata = {"render_modes": ["human", "rgb_array", "depth_array"], "render_fps": 50}

    def __init__(self, xml_file=os.path.join(os.getcwd(), "3prism_jonathan_steady_side.xml"), device=0, seed=0,
                 max_episode_steps=0, render_mode=None, param_ranges=None, **kwargs):
        """param_ranges: per-env tendon and actuator parameters redrawn at every reset, {field: (lo, hi)} scale
        factors (TensegrityVecEnv.set_param_ranges)"""
        self.L = _lib.load()
        for k in ("width", "height", "camera_id", "camera_name", "contact_with_self_penalty",
                  "use_cap_size_noise", "cap_size_noise_range", "threshold_waypt"):
            v = kwargs.pop(k, None)
            if k == "use_cap_size_noise" and v:   # tr_env.py:685-706 calls model.geom_names / geom_name2id, which the
                # `mujoco` 2.3.7 bindings do not have (mujoco-py API): the reference itself raises AttributeError here
                raise NotImplementedError("use_cap_size_noise=True fails in the reference too (mujoco-py-only API, tr_env.py:689-699)")
        self.render_mode = render_mode
        self.md = M.load_model(xml_file)
        self._model, self._keep = M.model_struct(self.md)
        self.cfg = M.env_config(self.md, env_kind=self.env_kind, max_episode_steps=max_episode_steps, **kwargs)
        self.obs_dim = int(self.cfg.obs_dim)
        self.frame_skip = int(self.cfg.frame_skip)
        self.dt = self.md["timestep"] * self.frame_skip
        h = C.c_void_p()
        _lib.check(self.L.tsg_create(C.byref(self._model), C.byref(self.cfg), 1, int(device), 0, C.byref(h)))
        self.h = h
        if param_ranges is not None:
            lo, hi = M.param_scale_ranges(param_ranges)
            _lib.check(self.L.tsg_set_param_ranges(self.h, self._p(lo), self._p(hi)))
        lo, hi = self.md["ctrlrange"]
        self.action_space = Box(np.full(6, lo, np.float32), np.full(6, hi, np.float32), dtype=np.float32)
        # use_contact_forces: the reference DECLARES 84 more observation slots (tr_env.py:263-264) but its _get_obs never
        # fills them (:529-646), so the vectors it returns keep obs_dim entries; the declared space follows the reference
        declared = self.obs_dim + (84 if self.cfg.use_contact_forces else 0)
        self.observation_space = Box(-np.inf, np.inf, shape=(declared,), dtype=np.float64)
        self.init_qpos = np.array(self.md["qpos0"])
        self.init_qvel = np.zeros(18)
        self.model = self.md
        self.data = _DataShim(self)
        self._seed = int(seed)
        self._nreset = 0
        self._obs = np.zeros((1, self.obs_dim))
        self._rew = np.zeros(1)
        self._done = np.zeros(1, np.uint8)
        self._info = np.zeros((1, _lib.INFO_DIM))
        self._last_info = self._info[0]
        self.np_random = np.random.default_rng(seed)

    @staticmethod
    def _p(a):
        return C.c_void_p(a.ctypes.data) if a is not None else None

    def reset(self, seed=None, options=None, draws=None):
        if seed is not None:
            self._seed = int(seed)
            self.np_random = np.random.default_rng(seed)
        d = None if draws is None else np.ascontiguousarray(np.asarray(draws, np.float64).reshape(1, _lib.NDRAW))
        _lib.check(self.L.tsg_reset_host(self.h, None, self._seed, self._p(d), self._p(self._obs)))
        self.data.contact = []
        return self._obs[0].copy(), {}

    def step(self, action):
        a = np.asarray(action, np.float64)
        if a.shape != (6,):
            raise ValueError("Action dimension mismatch")  # gym MujocoEnv.do_simulation
        a = np.ascontiguousarray(a.reshape(1, 6))
        _lib.check(self.L.tsg_step_host(self.h, self._p(a), self._p(self._obs), self._p(self._rew), self._p(self._done),
                                        self._p(self._info), 0, self._seed, None))
        row = self._info[0]
        self._last_info = row
        I = _lib.INFO
        obs = self._obs[0].copy()
        x, y = float(row[I["x"]]), float(row[I["y"]])
        info = {
            "reward_forward": float(row[I["rew_fwd"]]), "reward_ctrl": float(row[I["rew_ctrl"]]),
            "reward_survive": float(row[I["rew_survive"]]), "x_position": x, "y_position": y,
            "psi": float(row[I["psi"]]), "distance_from_origin": float(np.hypot(x, y)),
            "x_velocity": float(row[I["xvel"]]), "y_velocity": float(row[I["yvel"]]),
            "forward_reward": float(row[I["rew_fwd"]]),
        }
        if self.env_kind == "tr_env":
            real = obs.copy()
            if self.cfg.use_obs_noise:   # obs is the noisy observation (tr_env.py:524-527), info carries the true one (:505)
                buf = np.zeros((1, self.obs_dim))
                _lib.check(self.L.tsg_get_real_obs_host(self.h, self._p(buf)))
                real = buf[0]
            info.update(tendon_length=np.array(row[I["ten"]:I["ten"] + 9]), real_observation=real,
                        waypt=np.array(row[I["waypt"]:I["waypt"] + 2]) if self.cfg.task in (2, 3) else np.array([]),
                        oripoint=np.array(row[I["ori"]:I["ori"] + 2]))
        bf = float(row[I["barforce"]])
        self.data.contact = [_Contact(1, 6, bf)] if bf > 0 else []
        terminated, truncated = bool(row[I["terminated"]]), bool(row[I["truncated"]])
        return obs, float(self._rew[0]), terminated, truncated, info

    def _get_state(self):
        out = {k: np.zeros((1, w)) for k, w in (("qpos", 21), ("qvel", 18), ("act", 6), ("qacc_warmstart", 18), ("ctrl", 6))}
        _lib.check(self.L.tsg_get_state_host(self.h, *[self._p(out[k]) for k in ("qpos", "qvel", "act", "qacc_warmstart", "ctrl")]))
        return out

    def state_vector(self):
        s = self._get_state()
        return np.concatenate([s["qpos"][0], s["qvel"][0]])

    def set_state(self, qpos, qvel):
        q = np.ascontiguousarray(np.asarray(qpos, np.float64).reshape(1, 21))
        v = np.ascontiguousarray(np.asarray(qvel, np.float64).reshape(1, 18))
        _lib.check(self.L.tsg_set_state_host(self.h, self._p(q), self._p(v), None, None, None))
        _lib.check(self.L.tsg_forward_host(self.h, None, None))   # own stream, synchronous: ordered with step / reset

    def render(self):
        return None

    def close(self):
        if getattr(self, "h", None):
            self.L.tsg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def unwrapped(self):
        return self


class tr_env(_SingleEnv):
    env_kind = "tr_env"


class tensegrity_env(_SingleEnv):
    env_kind = "tensegrity_env"


_REGISTRY = {"tr_env-v0": (tr_env, 5000), "tensegrity_env-v0": (tensegrity_env, 5000)}


def make(env_id, **kwargs):
    """Stand-in for gym.make(env_id, **kwargs): TimeLimit(max_episode_steps=5000) folded into the env."""
    cls, limit = _REGISTRY[env_id]
    kwargs.setdefault("max_episode_steps", limit)
    return cls(**kwargs)


def register_with_gym():
    """Register the reference ids when gym / gymnasium is importable (it is not in this image)."""
    done = []
    for modname in ("gym", "gymnasium"):
        try:
            mod = __import__(modname)
            from importlib import import_module
            reg = import_module(modname + ".envs.registration").register
            for env_id, (cls, limit) in _REGISTRY.items():
                if env_id not in getattr(mod.envs.registration, "registry", {}):
                    reg(id=env_id, entry_point=f"tensegrity_rl_b200.envs:{cls.__name__}", max_episode_steps=limit)
            done.append(modname)
        except Exception:  # noqa: BLE001
            pass
    return done
