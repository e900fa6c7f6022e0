"""Per-env tendon and actuator parameters on the B200: the per-env kernels with nominal rows against the default
kernels (bit for bit), distinct rows against the oracle built from each row, the reset draws of the rows (against the
emulator's draws, across shards and through the reset pool), checkpoints and error paths."""
import ctypes as C

import numpy as np
import pytest

from tensegrity_rl_b200 import lib as tlib
from tensegrity_rl_b200 import model as M

pytestmark = pytest.mark.gpu

TOL = 1e-9
RANGES = {f: (0.8, 1.2) for f in tlib.PARAM}


def _vec(n, xml="flat", **kw):
    from tensegrity_rl_b200 import TensegrityVecEnv
    return TensegrityVecEnv(n, xml_file=xml, **kw)


def _rel(a, b):
    return np.abs(a - b).max() / max(1.0, np.abs(b).max())


def _random_rows(md, rng, n, lo=0.7, hi=1.3):
    s = rng.uniform(lo, hi, (n, M.NPARAM))
    s[:, 19:36:2] = s[:, 18:36:2]
    return M.nominal_params(md) * s


def _oracle_step(oracle, xml, row, st, e, ctrl):
    mj = oracle.MjLike(xml, **M.param_overrides(row))
    mj.qpos[:] = st["qpos"][e]; mj.qvel[:] = st["qvel"][e]; mj.act[:] = st["act"][e]
    mj.qacc_warmstart[:] = st["qacc_warmstart"][e]
    mj.ctrl[:] = ctrl
    mj.step(20)
    return mj


@pytest.mark.parametrize("n,precision", [(4096, "f64"), (4096, "f32"), (20011, "f64"), (20011, "f32")])
def test_nominal_rows_bit_identical_to_params_off(n, precision):
    """50 auto-resetting steps (episodes of 20 steps, reset_pool=0): obs, reward, done, info and records of the
    per-env kernels with nominal rows equal the default kernels'; then a reset and a forward pass"""
    import torch
    kw = dict(auto_reset=True, reset_pool=0, precision=precision, max_episode_steps=20)
    a, b = _vec(n, **kw), _vec(n, **kw)
    b.set_env_params(torch.as_tensor(np.tile(M.nominal_params(b.md), (n, 1))))
    assert np.array_equal(a.reset_tensor().cpu().numpy(), b.reset_tensor().cpu().numpy())
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    ndone = 0
    for st in range(50):
        ctrl = -0.45 + 0.6 * torch.rand(n, 6, generator=g, device="cuda", dtype=torch.float64)
        oa, ra, da = (t.cpu().numpy() for t in a.step_tensor(ctrl))
        ob, rb, db = (t.cpu().numpy() for t in b.step_tensor(ctrl))
        assert np.array_equal(oa, ob) and np.array_equal(ra, rb) and np.array_equal(da, db), st
        assert np.array_equal(a.info.cpu().numpy(), b.info.cpu().numpy()), st
        ndone += int(da.sum())
    assert ndone >= n        # every env went through at least one auto reset
    assert np.array_equal(a.get_records(), b.get_records())
    assert np.array_equal(a.get_heading(), b.get_heading())
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda"); mask[::3] = 1
    assert np.array_equal(a.reset_tensor(mask=mask, seed=9).cpu().numpy(), b.reset_tensor(mask=mask, seed=9).cpu().numpy())
    assert np.array_equal(a.forward_tensor().cpu().numpy(), b.forward_tensor().cpu().numpy())
    assert np.array_equal(a.info.cpu().numpy(), b.info.cpu().numpy())
    assert np.array_equal(a.get_records(), b.get_records())
    assert np.array_equal(b.get_env_params().cpu().numpy(), np.tile(M.nominal_params(b.md), (n, 1)))
    a.close(); b.close()


@pytest.mark.parametrize("xml", ["flat", "uneven"])
def test_distinct_rows_match_oracle(oracle, xml):
    """1024 envs, each with its own row (every field scaled in [0.7, 1.3]); on every 8th step 48 sampled envs against
    the oracle built from their rows, with the outlier budget of test_single_step_parity_random_ctrl"""
    import torch
    n = 1024
    v = _vec(n, xml, auto_reset=False, terminate_when_unhealthy=False, max_episode_steps=0)
    rows = _random_rows(v.md, np.random.default_rng(1), n)
    v.set_env_params(torch.as_tensor(rows))
    v.reset_tensor()
    assert np.array_equal(v.get_env_params().cpu().numpy(), rows)      # resets keep explicit rows without ranges
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    rng = np.random.default_rng(0)
    nbad = ncheck = overflow = 0
    worst = 0.0
    for step in range(40):
        a = -0.45 + 0.6 * torch.rand(n, 6, generator=g, device="cuda", dtype=torch.float64)
        check = step % 8 == 7
        if check:
            before = v.get_state()
        v.step_tensor(a)
        if not check:
            continue
        after, info = v.get_state(), v.info.cpu().numpy()
        overflow += int(info[:, 28].sum())
        for e in rng.choice(n, 48, replace=False):
            mj = _oracle_step(oracle, xml, rows[e], before, e, after["ctrl"][e])
            err = max(_rel(after["qpos"][e], mj.qpos), _rel(after["qvel"][e], mj.qvel), _rel(info[e, 8:17], mj.ten_length))
            ncheck += 1
            if err > TOL:
                nbad += 1
            else:
                worst = max(worst, err)
    print(xml, "checked", ncheck, "outliers", nbad, "worst", worst)
    assert nbad <= max(1, ncheck // 100), (nbad, ncheck)
    assert overflow == 0
    v.close()


def test_reset_rows_equal_emulator_draws_and_shards_reproduce():
    """rows after reset_tensor() are the emulator's draws bit for bit; two handles with env_id_base reproduce one
    unsharded handle through auto resets (reset_pool=0)"""
    import torch
    from emul import emul as E
    n, seed = 2048, 17
    kw = dict(seed=seed, reset_pool=0, max_episode_steps=8, param_ranges=RANGES)
    full = _vec(n, **kw)
    lo, hi = M.param_scale_ranges(RANGES)
    pr = np.stack([M.nominal_params(full.md), lo, hi])
    obs_full = [full.reset_tensor().cpu().numpy()]
    assert np.array_equal(full.get_env_params().cpu().numpy(), E.param_draws(pr, seed, 0, 0, n=n))
    shards = [_vec(n // 2, env_id_base=k * (n // 2), **kw) for k in range(2)]
    obs_sh = [np.concatenate([s.reset_tensor().cpu().numpy() for s in shards])]
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    for st in range(20):
        a = -0.45 + 0.6 * torch.rand(n, 6, generator=g, device="cuda", dtype=torch.float64)
        obs_full.append(full.step_tensor(a)[0].cpu().numpy())
        obs_sh.append(np.concatenate([s.step_tensor(a[k * (n // 2):(k + 1) * (n // 2)].contiguous())[0].cpu().numpy()
                                      for k, s in enumerate(shards)]))
    for x, y in zip(obs_full, obs_sh):
        assert np.array_equal(x, y)
    p_full = full.get_env_params().cpu().numpy()
    assert np.array_equal(p_full, np.concatenate([s.get_env_params().cpu().numpy() for s in shards]))
    nres = full.get_records()[:, 85].astype(int)
    assert nres.min() >= 2         # every env was redrawn at its auto resets
    for e in (0, 1, n - 1):
        assert np.array_equal(p_full[e], E.param_draws(pr, seed, e, nres[e] - 1)[0])
    for v in [full] + shards:
        v.close()


def test_pool_resets_hand_over_valid_draws(oracle):
    """with a reset pool every env that auto-reset holds a row a slot drew, and its next step matches the oracle
    built from that row"""
    import torch
    from emul import emul as E
    n, seed = 1024, 23
    v = _vec(n, seed=seed, reset_pool="auto", max_episode_steps=6, param_ranges=RANGES)
    lo, hi = M.param_scale_ranges(RANGES)
    pr = np.stack([M.nominal_params(v.md), lo, hi])
    v.reset_tensor()
    g = torch.Generator(device="cuda"); g.manual_seed(8)
    # a slot's draws, or (done envs that found no ready slot reset synchronously) the env's own
    drawn = {r.tobytes() for k in range(4) for r in E.param_draws(pr, seed, 1 << 40, k, n=v.reset_pool)}
    drawn |= {r.tobytes() for k in range(4) for r in E.param_draws(pr, seed, 0, k, n=n)}
    assigned, nbad, ncheck = 0, 0, 0
    for st in range(14):
        a = -0.45 + 0.6 * torch.rand(n, 6, generator=g, device="cuda", dtype=torch.float64)
        done = v.step_tensor(a)[2].cpu().numpy().astype(bool)
        assigned += v.pool_stats()["assigned"]
        if not done.any():
            continue
        rows = v.get_env_params().cpu().numpy()
        for e in np.flatnonzero(done):
            assert rows[e].tobytes() in drawn, (st, e)
        before = v.get_state()
        a2 = -0.45 + 0.6 * torch.rand(n, 6, generator=g, device="cuda", dtype=torch.float64)
        v.step_tensor(a2)
        after, info = v.get_state(), v.info.cpu().numpy()
        for e in np.flatnonzero(done)[:8]:
            mj = _oracle_step(oracle, "flat", rows[e], before, e, after["ctrl"][e])
            ncheck += 1
            nbad += max(_rel(after["qpos"][e], mj.qpos), _rel(after["qvel"][e], mj.qvel), _rel(info[e, 8:17], mj.ten_length)) > TOL
    assert assigned > 0 and ncheck > 0
    assert nbad <= max(1, ncheck // 100), (nbad, ncheck)
    v.close()


def test_checkpoint_records_heading_and_rows_continue_bit_for_bit():
    import torch
    n, seed = 4096, 31
    kw = dict(seed=seed, reset_pool=0, max_episode_steps=7, param_ranges=RANGES, desired_action="turn")
    a = _vec(n, **kw)
    a.reset_tensor()
    g = torch.Generator(device="cuda"); g.manual_seed(4)
    acts = [-0.45 + 0.6 * torch.rand(n, 6, generator=g, device="cuda", dtype=torch.float64) for _ in range(24)]
    for x in acts[:10]:
        a.step_tensor(x)
    rec, hd, rows = a.get_records(), a.get_heading(), a.get_env_params().clone()
    ref = [[t.cpu().numpy() for t in a.step_tensor(x)] for x in acts[10:]]
    b = _vec(n, **kw)
    b.set_records(rec); b.set_heading(hd); b.set_env_params(rows)
    for x, r in zip(acts[10:], ref):
        for u, w in zip(b.step_tensor(x), r):
            assert np.array_equal(u.cpu().numpy(), w)
    assert np.array_equal(a.get_env_params().cpu().numpy(), b.get_env_params().cpu().numpy())
    assert not np.array_equal(rows.cpu().numpy(), b.get_env_params().cpu().numpy())   # resets after the restore redrew
    a.close(); b.close()


def test_errors():
    import torch
    v = _vec(64, reset_pool=32)
    with pytest.raises(tlib.TsgError, match="reset pool"):
        v.set_env_params(torch.as_tensor(np.tile(M.nominal_params(v.md), (64, 1))))
    with pytest.raises(ValueError):
        v.set_param_ranges({"act_gain": (1.2, 0.8)})
    lo, hi = np.ones(41), np.ones(41)
    for bad_lo, bad_hi in ((np.full(41, -0.5), hi), (lo, np.full(41, 0.5)), (np.where(np.arange(41) == 40, 0.0, 1.0), hi),
                           (np.where(np.arange(41) == 18, 0.9, 1.0), hi), (np.full(41, np.nan), hi)):
        bl, bh = np.ascontiguousarray(bad_lo), np.ascontiguousarray(bad_hi)
        assert v.L.tsg_set_param_ranges(v.h, C.c_void_p(bl.ctypes.data), C.c_void_p(bh.ctypes.data)) != 0
        assert b"tsg_set_param_ranges" in v.L.tsg_last_error()
    assert v.L.tsg_set_param_ranges(v.h, C.c_void_p(lo.ctypes.data), None) != 0
    with pytest.raises(ValueError):
        v.set_env_params(torch.zeros(64, 40, dtype=torch.float64))
    v.set_param_ranges(RANGES)           # valid ranges on a pooled handle
    v.reset_tensor()
    rows = v.get_env_params().cpu().numpy()
    nom = M.nominal_params(v.md)
    assert ((rows >= np.minimum(0.8 * nom, 1.2 * nom)) & (rows <= np.maximum(0.8 * nom, 1.2 * nom))).all()
    v.close()
