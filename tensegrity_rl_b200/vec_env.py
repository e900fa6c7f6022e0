"""Batched env front end: N independent tensegrity envs stepped by one CUDA launch.

`TensegrityVecEnv` follows the stable-baselines3 `VecEnv` protocol (num_envs, observation_space,
action_space, reset(), step_async(), step_wait(), auto reset with `terminal_observation` /
`TimeLimit.truncated`) so SB3 algorithms can consume it, and adds a zero-copy torch path
(`reset_tensor`, `step_tensor`) where ctrl / obs / reward / done stay on the GPU.

Constructor kwargs are the reference env kwargs (tr_env.py:137-173, tensegrity_env.py:160-181).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib as _lib
from . import model as M
from .spaces import Box


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class TensegrityVecEnv:
    metadata = {"render_modes": []}

    def __init__(self, num_envs, xml_file=None, env="tr_env", device=0, seed=0, env_id_base=0,
                 auto_reset=True, info_mode="auto", max_episode_steps=5000, reset_pool=0, precision="f64",
                 param_ranges=None, **env_kwargs):
        """reset_pool: number of background reset slots (0 = every reset runs synchronously, bit-reproducible per
        env id; "auto" = num_envs // 4, at least 32).  With a pool, an env that is done receives a slot that has
        already been through the reference's 50-step reset warm-up, so resets add no latency to a step.
        precision: "f64" (the reference's arithmetic, default) or "f32" (optional fp32 physics).
        param_ranges: per-env tendon and actuator parameters redrawn at every reset (domain randomisation), as
        {field: (lo, hi)} scale factors of the nominal value; fields are those of `lib.PARAM`, each bound a scalar or an
        array of the field's width, fields not given keep scale 1.  See set_param_ranges."""
        import torch

        if not torch.cuda.is_available():
            raise _lib.TsgError("TensegrityVecEnv needs a CUDA device (sm_100a); there is no CPU path")
        self.L = _lib.load()
        self.torch = torch
        self.num_envs = int(num_envs)
        self.env_name = env
        self.md = M.load_model(xml_file)
        self._model, self._keep = M.model_struct(self.md)
        for k in ("render_mode", "width", "height", "camera_id", "camera_name"):
            env_kwargs.pop(k, None)
        self.cfg = M.env_config(self.md, env_kind=env, max_episode_steps=max_episode_steps, **env_kwargs)
        self.obs_dim = int(self.cfg.obs_dim)
        self.dt = self.md["timestep"] * self.cfg.frame_skip
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        self.seed_value = int(seed)
        self.auto_reset = bool(auto_reset)
        self.info_mode = info_mode
        h = C.c_void_p()
        if reset_pool == "auto":
            reset_pool = max(32, self.num_envs // 4) if auto_reset else 0
        self.reset_pool = int(reset_pool)
        self.precision = precision
        _lib.check(self.L.tsg_create_opts(C.byref(self._model), C.byref(self.cfg), self.num_envs, self.reset_pool,
                                          self.device_index, int(env_id_base), _lib.PRECISION[precision], C.byref(h)))
        self.h = h
        lo, hi = self.md["ctrlrange"]
        self.action_space = Box(np.full(6, lo, np.float32), np.full(6, hi, np.float32), dtype=np.float32)
        self.observation_space = Box(-np.inf, np.inf, shape=(self.obs_dim,), dtype=np.float64)
        n, dev = self.num_envs, self.device
        with torch.cuda.device(dev):
            self.obs = torch.zeros(n, self.obs_dim, dtype=torch.float64, device=dev)
            self.obs32 = torch.zeros(n, self.obs_dim, dtype=torch.float32, device=dev)
            self.reward = torch.zeros(n, dtype=torch.float64, device=dev)
            self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
            self.info = torch.zeros(n, _lib.INFO_DIM, dtype=torch.float64, device=dev)
            self.term_obs = torch.zeros(n, self.obs_dim, dtype=torch.float64, device=dev)
            self.real_obs = None
            if self.cfg.use_obs_noise:   # obs rows are noisy (tr_env.py:524-527); the true ones land here
                self.real_obs = torch.zeros(n, self.obs_dim, dtype=torch.float64, device=dev)
                _lib.check(self.L.tsg_set_real_obs(self.h, _ptr(self.real_obs)))
        self._actions = None
        self.n_steps = 0
        if param_ranges is not None:
            self.set_param_ranges(param_ranges)

    # ------------------------------------------------------------------ torch (device) path
    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def reset_tensor(self, mask=None, draws=None, seed=None):
        """Reset all envs (or those with mask != 0).  Returns the obs tensor [N, D] (float64, device)."""
        t = self.torch
        if mask is not None:
            mask = mask.to(device=self.device, dtype=t.uint8).contiguous()
        if draws is not None:
            draws = t.as_tensor(draws, dtype=t.float64, device=self.device).contiguous()
            assert draws.shape == (self.num_envs, _lib.NDRAW)
        with t.cuda.device(self.device):
            _lib.check(self.L.tsg_reset(self.h, _ptr(mask), self.seed_value if seed is None else int(seed),
                                        _ptr(draws), _ptr(self.obs), _ptr(self.obs32), None, self._stream()))
        return self.obs

    def step_tensor(self, ctrl, want_info=True, auto_reset=None):
        """ctrl: CUDA tensor [N, 6] float64 or float32.  Returns (obs, reward, done) device tensors
        (views of internal buffers, overwritten by the next call); `self.info`, `self.obs32`,
        `self.term_obs` are filled too."""
        t = self.torch
        assert ctrl.is_cuda and ctrl.shape == (self.num_envs, 6)
        ctrl = ctrl.contiguous()
        dtype = _lib.CTRL_F64 if ctrl.dtype == t.float64 else _lib.CTRL_F32
        if dtype == _lib.CTRL_F32 and ctrl.dtype != t.float32:
            ctrl = ctrl.float()
        ar = self.auto_reset if auto_reset is None else auto_reset
        with t.cuda.device(self.device):
            _lib.check(self.L.tsg_step(self.h, _ptr(ctrl), dtype, _ptr(self.obs), _ptr(self.obs32), _ptr(self.reward),
                                       _ptr(self.done), _ptr(self.info) if want_info else None, int(ar),
                                       self.seed_value, _ptr(self.term_obs) if ar else None, self._stream()))
        self.n_steps += 1
        return self.obs, self.reward, self.done

    def forward_tensor(self):
        with self.torch.cuda.device(self.device):
            _lib.check(self.L.tsg_forward(self.h, _ptr(self.obs), _ptr(self.info), self._stream()))
        return self.obs

    # ------------------------------------------------------------------ per-env parameters
    def set_param_ranges(self, param_ranges):
        """From now on every reset draws each env's parameter row as nominal * U(lo, hi) per field (the lower and upper
        ten_lengthspring of a tendon share one draw).  None stops the draws; rows then stay as they are.  The first
        call switches the handle to the per-env kernels."""
        if param_ranges is None:
            _lib.check(self.L.tsg_set_param_ranges(self.h, None, None))
            return
        lo, hi = M.param_scale_ranges(param_ranges)
        _lib.check(self.L.tsg_set_param_ranges(self.h, C.c_void_p(lo.ctypes.data), C.c_void_p(hi.ctypes.data)))

    def set_env_params(self, params, mask=None):
        """explicit parameter rows [N, 41] (absolute values, layout `lib.PARAM`) for all envs or those with mask != 0,
        from the next step on; with param_ranges set they last until the env's next reset.  Not on a handle with a
        reset pool (an env that receives a pool slot takes the slot's row)."""
        t = self.torch
        params = t.as_tensor(params, dtype=t.float64, device=self.device).contiguous()
        if params.shape != (self.num_envs, _lib.NPARAM):
            raise ValueError(f"params must have shape ({self.num_envs}, {_lib.NPARAM}), got {tuple(params.shape)}")
        if mask is not None:
            mask = t.as_tensor(mask, device=self.device).to(t.uint8).contiguous()
        with t.cuda.device(self.device):
            _lib.check(self.L.tsg_set_env_params(self.h, _ptr(params), _ptr(mask), self._stream()))
            if params.device.type == "cuda":   # the copy is stream ordered: keep the source alive until it ran
                params.record_stream(t.cuda.current_stream(self.device))

    def get_env_params(self):
        """every env's parameter row, a cuda float64 tensor [N, 41] (the nominal row until per-env parameters are on)"""
        t = self.torch
        out = t.empty(self.num_envs, _lib.NPARAM, dtype=t.float64, device=self.device)
        with t.cuda.device(self.device):
            _lib.check(self.L.tsg_get_env_params(self.h, _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ SB3 VecEnv protocol (host numpy)
    def reset(self):
        obs = self.reset_tensor()
        return obs.cpu().numpy()

    def step_async(self, actions):
        self._actions = np.asarray(actions)

    def step_wait(self):
        t = self.torch
        a = t.as_tensor(np.ascontiguousarray(self._actions, np.float64)).to(self.device, non_blocking=True)
        obs, rew, done = self.step_tensor(a.reshape(self.num_envs, 6), want_info=True)
        obs_h, rew_h, done_h, info_h = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy().astype(bool), self.info.cpu().numpy()
        full = self.info_mode == "full" or (self.info_mode == "auto" and self.num_envs <= 64)
        term_h = self.term_obs.cpu().numpy() if (self.auto_reset and done_h.any()) else None
        real_h = self.real_obs.cpu().numpy() if (full and self.real_obs is not None) else obs_h
        infos = []
        for e in range(self.num_envs):
            d = self.info_dict(info_h[e], real_h[e]) if full else {}
            if done_h[e]:
                d["TimeLimit.truncated"] = bool(info_h[e, _lib.INFO["truncated"]]) and not bool(info_h[e, _lib.INFO["terminated"]])
                if term_h is not None:
                    d["terminal_observation"] = term_h[e]
            infos.append(d)
        return obs_h, rew_h, done_h, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def info_dict(self, row, obs_row=None):
        """info dict of one env with the reference's keys (tr_env.py:496-512)."""
        I = _lib.INFO
        x, y = float(row[I["x"]]), float(row[I["y"]])
        d = {
            "reward_forward": float(row[I["rew_fwd"]]), "reward_ctrl": float(row[I["rew_ctrl"]]),
            "reward_survive": float(row[I["rew_survive"]]), "x_position": x, "y_position": y,
            "psi": float(row[I["psi"]]), "distance_from_origin": float(np.hypot(x, y)),
            "x_velocity": float(row[I["xvel"]]), "y_velocity": float(row[I["yvel"]]),
            "forward_reward": float(row[I["rew_fwd"]]),
            "total_bar_contact": float(row[I["barforce"]]),
        }
        if self.env_name == "tr_env":
            d["tendon_length"] = np.array(row[I["ten"]:I["ten"] + 9])
            d["real_observation"] = None if obs_row is None else np.array(obs_row)
            d["waypt"] = np.array(row[I["waypt"]:I["waypt"] + 2]) if self.cfg.task in (2, 3) else np.array([])
            d["oripoint"] = np.array(row[I["ori"]:I["ori"] + 2])
        return d

    # raw state (host numpy), for parity tests and env-state checkpoints
    def get_state(self):
        n = self.num_envs
        out = {k: np.zeros((n, w)) for k, w in (("qpos", 21), ("qvel", 18), ("act", 6), ("qacc_warmstart", 18), ("ctrl", 6))}
        P = lambda a: C.c_void_p(a.ctypes.data)
        _lib.check(self.L.tsg_get_state_host(self.h, P(out["qpos"]), P(out["qvel"]), P(out["act"]),
                                             P(out["qacc_warmstart"]), P(out["ctrl"])))
        return out

    def set_state(self, qpos=None, qvel=None, act=None, qacc_warmstart=None, ctrl=None):
        n = self.num_envs
        arrs = []
        for a, w in ((qpos, 21), (qvel, 18), (act, 6), (qacc_warmstart, 18), (ctrl, 6)):
            if a is not None:
                a = np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (n, w)))
            arrs.append(a)
        P = lambda a: C.c_void_p(a.ctypes.data) if a is not None else None
        _lib.check(self.L.tsg_set_state_host(self.h, *[P(a) for a in arrs]))

    def get_records(self):
        rec = np.zeros((self.num_envs, _lib.STATE_STRIDE))
        _lib.check(self.L.tsg_get_records_host(self.h, C.c_void_p(rec.ctypes.data)))
        return rec

    def get_records_t(self):
        return self.torch.as_tensor(self.get_records(), device=self.device)

    def set_records(self, rec):
        rec = np.ascontiguousarray(rec, np.float64)
        assert rec.shape == (self.num_envs, _lib.STATE_STRIDE)
        _lib.check(self.L.tsg_set_records_host(self.h, C.c_void_p(rec.ctypes.data)))

    def get_heading(self):
        """heading rings (turn / aiming reward delay): records + heading rings = a checkpoint of the env state"""
        hd = np.zeros((self.num_envs, _lib.HEADING_SLOTS))
        _lib.check(self.L.tsg_get_heading_host(self.h, C.c_void_p(hd.ctypes.data)))
        return hd

    def set_heading(self, hd):
        hd = np.ascontiguousarray(hd, np.float64)
        assert hd.shape == (self.num_envs, _lib.HEADING_SLOTS)
        _lib.check(self.L.tsg_set_heading_host(self.h, C.c_void_p(hd.ctypes.data)))

    def get_draws(self):
        d = np.zeros((self.num_envs, _lib.NDRAW))
        _lib.check(self.L.tsg_get_draws_host(self.h, C.c_void_p(d.ctypes.data)))
        return d

    def pool_stats(self):
        """{done envs, ready slots, slots handed out} of the last auto reset (synchronises)."""
        c = (C.c_int * 3)()
        _lib.check(self.L.tsg_pool_stats_host(self.h, c))
        return {"done": c[0], "ready": c[1], "assigned": c[2]}

    @property
    def launches(self):
        return int(self.L.tsg_launches(self.h))

    def kernel_config(self):
        w, s, r = C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.L.tsg_kernel_config(self.h, C.byref(w), C.byref(s), C.byref(r)))
        # the C ABI packs (warps per CTA, lanes per env) into one int: w * 100 + lanes
        return {"warps_per_cta": w.value // 100, "lanes_per_env": w.value % 100, "envs_per_warp": 10,
                "smem_bytes_per_cta": s.value, "regs_per_thread": r.value}

    # SB3 VecEnv odds and ends
    def close(self):
        if getattr(self, "h", None):
            self.L.tsg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def seed(self, seed=None):
        if seed is not None:
            self.seed_value = int(seed)
        return [self.seed_value + i for i in range(self.num_envs)]

    def get_attr(self, name, indices=None):
        return [getattr(self, name)] * self.num_envs

    def set_attr(self, name, value, indices=None):
        setattr(self, name, value)

    def env_method(self, name, *args, indices=None, **kwargs):
        return [getattr(self, name)(*args, **kwargs)] * self.num_envs

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * self.num_envs

    def render(self, mode=None):
        return None
