"""Host logic: model compiler, asset consistency, C-ABI surface (no compute without a GPU)."""
import ctypes as C
import json
import os
import re
import sys

import numpy as np
import pytest

from tensegrity_rl_b200 import lib as tlib
from tensegrity_rl_b200 import model as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_derived_constants_flat():
    md = M.load_model("flat")
    assert md["body_mass"] == [4.0, 4.0, 4.0]
    assert md["body_inertia"][0] == pytest.approx([1.096411235833, 1.096411235833, 0.003773305], rel=1e-12)
    assert md["meaninertia"] == pytest.approx(2.36609930, rel=1e-8)
    assert md["body_invweight0"][0] == pytest.approx([0.25, 88.94793], rel=1e-6)
    assert md["friction"] == [1.0, 1.0, 0.005, 0.0001, 0.0001]
    assert md["act_gain"] == 6667 and md["act_bias"] == [3290, -6666, -133] and md["forcerange"] == [-267, 0]
    assert md["ctrlrange"] == [-0.45, 0.15] and md["act_dyntype"] == M.DYN_NONE
    # tendon lengths at qpos0 (SURVEY App. A, derived independently there)
    assert np.allclose([l[0] for l in md["ten_lengthspring"][:6]],
                       [0.573839166, 0.571737603, 0.571086264, 0.573616978, 0.571999808, 0.570004094], atol=1e-8)


def test_derived_constants_uneven():
    md = M.load_model("uneven")
    assert md["act_dyntype"] == M.DYN_FILTER and md["act_gain"] == 15000 and not md["forcelimited"]
    assert md["ten_stiffness"] == [10000.0] * 9 and md["ten_damping"] == [1000.0] * 9
    assert md["body_inertia"][0] == pytest.approx([1.095588735833, 1.095588735833, 0.002950805], rel=1e-12)
    hf = md["hfield"]
    assert (hf["nrow"], hf["ncol"]) == (100, 100) and hf["size"] == [50, 50, 1, 0.1]
    d = hf["data"]
    assert d.dtype == np.float32 and d.min() == 0 and d.max() == 1
    assert d[99, 0] == 1.0  # the lone 255 pixel at image [0,0] lands on the last row after the flip
    assert (d == 0).mean() == pytest.approx(0.5, abs=0.05)


def test_struct_mirrors_match_header(tmp_path):
    """ctypes mirrors vs include/tsg_model.h: sizes and field offsets as gcc lays them out."""
    import subprocess
    fields = {"TsgModel": [f[0] for f in M.TsgModel._fields_], "TsgEnvConfig": [f[0] for f in M.TsgEnvConfig._fields_]}
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "%s"' % os.path.join(ROOT, "include", "tsg_model.h"),
           "int main(void){"]
    for st, names in fields.items():
        src.append('printf("%s %%zu\\n", sizeof(%s));' % (st, st))
        for n in names:
            src.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (st, n, st, n))
    src.append("return 0;}")
    c = tmp_path / "off.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "off"
    subprocess.check_call(["gcc", "-o", str(exe), str(c)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)]).decode().splitlines())
    for st, cls in (("TsgModel", M.TsgModel), ("TsgEnvConfig", M.TsgEnvConfig)):
        assert int(out[st]) == C.sizeof(cls)
        for n in fields[st]:
            assert int(out["%s.%s" % (st, n)]) == getattr(cls, n).offset, (st, n)


def test_oracle_and_product_agree_on_struct_size(oracle):
    assert oracle.lib().tsgo_sizeof_model() == C.sizeof(M.TsgModel)


def test_library_exports_every_declared_symbol():
    L = tlib.load()
    hdr = open(os.path.join(ROOT, "include", "tsg.h")).read()
    declared = set(re.findall(r"\b(tsg_[a-z_]+)\s*\(", hdr))
    assert declared == set(tlib.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), s
    assert L.tsg_version() >= 1


def test_no_cpu_fallback():
    """without a CUDA device tsg_create must fail loudly (no CPU path, no oracle behind the product)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = tlib.load()
    md = M.load_model("flat")
    ms, _ = M.model_struct(md)
    cfg = M.env_config(md)
    h = C.c_void_p()
    rc = L.tsg_create(C.byref(ms), C.byref(cfg), 4, 0, 0, C.byref(h))
    assert rc != 0 and b"no CUDA device" in L.tsg_last_error()
    with pytest.raises(tlib.TsgError):
        from tensegrity_rl_b200 import TensegrityVecEnv
        TensegrityVecEnv(4)


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "tensegrity_rl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("oracle-only", "").lower() or f in ("__init__.py",) and "oracle" not in src, f


def test_env_config_defaults():
    md = M.load_model("flat")
    c = M.env_config(md, env_kind="tr_env", desired_action="tracking")
    assert (c.obs_dim, c.reward_delay_steps, c.frame_skip, c.npose) == (48, 1, 20, 6)
    assert c.ctrl_cost_weight == 0.01 and c.tendon_reset_mean == 0.15 and c.tendon_max_length == 0.15
    c = M.env_config(md, env_kind="tensegrity_env", desired_action="turn")
    assert (c.obs_dim, c.reward_delay_steps, c.npose) == (39, 25, 1)
    assert c.ctrl_cost_weight == 0.001 and c.tendon_reset_mean == -0.15 and c.tendon_max_length == -0.15
    assert M.env_config(md, use_cap_velocity=False).obs_dim == 27
    with pytest.raises(ValueError):
        M.env_config(md, env_kind="tensegrity_env", desired_action="tracking")


def test_policy_assets_and_actor_cpu():
    import torch
    from tensegrity_rl_b200.policy import SacActor, load_actor_arrays
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "last_obs.json")))
    for name, meta in g.items():
        a = load_actor_arrays(name)
        assert a["obs_dim"] == meta["obs_dim"] and a["W0"].shape == (256, meta["obs_dim"])
        assert a["action_low"][0] == pytest.approx(-0.45)
    act = SacActor("traj_track", device="cpu", seed=0)
    obs = torch.tensor(np.array(g["traj_track"]["last_obs"])[None])
    d = act(obs, deterministic=True)
    assert d.shape == (1, 6) and (d >= -0.45 - 1e-6).all() and (d <= 0.15 + 1e-6).all()
    # plain fp32 torch reference of the same MLP
    a = load_actor_arrays("traj_track")
    x = torch.relu(obs.float() @ torch.tensor(a["W0"]).t() + torch.tensor(a["b0"]))
    x = torch.relu(x @ torch.tensor(a["W1"]).t() + torch.tensor(a["b1"]))
    mu = x @ torch.tensor(a["Wmu"]).t() + torch.tensor(a["bmu"])
    ref = -0.45 + 0.5 * (torch.tanh(mu) + 1) * 0.6
    assert torch.allclose(d, ref, atol=1e-5)


def test_run_py_shims(monkeypatch):
    """shims/: the module names run.py imports (`mujoco`, `tr_env`, run.py:4,8,158), so that it runs unmodified with
    shims/ on PYTHONPATH.  gym is not installed here: a stub `gym.envs.registration` records the registrations."""
    import importlib
    import types
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    monkeypatch.syspath_prepend(os.path.join(root, "shims"))
    calls = []
    gym = types.ModuleType("gym"); envs = types.ModuleType("gym.envs"); reg = types.ModuleType("gym.envs.registration")
    reg.register = lambda **kw: calls.append(kw)
    gym.envs, envs.registration = envs, reg
    for name, mod in (("gym", gym), ("gym.envs", envs), ("gym.envs.registration", reg)):
        monkeypatch.setitem(sys.modules, name, mod)
    for name in ("mujoco", "tr_env", "tr_env.envs", "tensegrity_env", "tensegrity_env.envs"):
        monkeypatch.delitem(sys.modules, name, raising=False)
    mujoco = importlib.import_module("mujoco")
    tr = importlib.import_module("tr_env")
    te = importlib.import_module("tensegrity_env")
    assert {c["id"] for c in calls} == {"tr_env-v0", "tensegrity_env-v0"}
    assert all(c["max_episode_steps"] == 5000 for c in calls)
    assert [c["entry_point"] for c in calls if c["id"] == "tr_env-v0"] == ["tr_env.envs:tr_env"]
    from tensegrity_rl_b200 import envs as E
    assert importlib.import_module("tr_env.envs").tr_env is E.tr_env
    assert importlib.import_module("tensegrity_env.envs").tensegrity_env is E.tensegrity_env
    # mj_contactForce on the contact shim: the aggregated bar-bar force lands in forcetorque[0] (run.py:155-161)
    data = types.SimpleNamespace(contact=[E._Contact(1, 6, 12.5)])
    ft = np.zeros(6)
    mujoco.mj_contactForce(None, data, 0, ft)
    assert ft[0] == 12.5 and np.all(ft[1:] == 0)
    assert data.contact[0].geom1 != 0 and data.contact[0].geom2 != 0
