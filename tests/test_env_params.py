"""Per-env tendon and actuator parameters on the CPU: the per-env variant of the CUDA source (run by the warp emulator)
against the default variant and against the oracle built from each env's row, the reset draws of the rows, and the
host-side conversion and validation of param_ranges."""
import ctypes as C

import numpy as np
import pytest

from emul import emul as E
from oracle import oracle as O
from oracle.envs import OracleEnv
from tensegrity_rl_b200 import lib as tlib
from tensegrity_rl_b200 import model as M


def _draws(rng, n):
    return np.concatenate([rng.uniform(0, 1, (n, 2)), rng.standard_normal((n, 6)), rng.uniform(0, 1, (n, 2))], 1)


def _random_rows(md, rng, n, lo=0.7, hi=1.3):
    """n rows with every field scaled by U(lo, hi); a tendon's lower and upper spring length share their scale"""
    s = rng.uniform(lo, hi, (n, M.NPARAM))
    s[:, 19:36:2] = s[:, 18:36:2]
    return M.nominal_params(md) * s


def _warp_pair(xml, n, **kw):
    """the default variant and the per-env variant with nominal rows"""
    rows = np.tile(E.nominal_params(M.load_model(xml)), (n, 1))
    return E.EmulWarp(xml, n, **kw), E.EmulWarp(xml, n, rows=rows, **kw)


def _oracle_env(xml, kind, row, **kw):
    """OracleEnv whose oracle model carries the parameter row"""
    oe = OracleEnv(xml, kind, **kw)
    oe.mj = O.MjLike(xml, **M.param_overrides(row))
    return oe


def _same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("xml,pre", [("flat", 0), ("uneven", 30)])
def test_nominal_rows_bit_identical_to_default_variant(xml, pre):
    """per-env variant with nominal rows == default variant (np.array_equal): a reset, 10 desynchronised envs for 50
    env steps, a forward pass and raw mj_step in fp64 and fp32"""
    n = 10
    a, b = _warp_pair(xml, n, warmup_steps=5)
    rng = np.random.default_rng(2)
    d = _draws(rng, n)
    _same([a.reset(d)], [b.reset(d)])
    assert np.array_equal(a.rec, b.rec)
    for st in range(50):
        act = rng.uniform(-0.45, 0.15, (n, 6))
        act[st % n] = 0.15      # a different env gets a different push every step
        _same(a.step(act), b.step(act))
        assert np.array_equal(a.rec, b.rec) and np.array_equal(a.heading, b.heading)
    _same(a.forward(), b.forward())
    ctrl = rng.uniform(-0.45, -0.15, (n, 6))
    for k in range(pre // 10 + 2):
        _same(a.mj_step(ctrl, 20), b.mj_step(ctrl, 20))
        assert np.array_equal(a.rec, b.rec)
    ra, rb = a.rec.copy(), b.rec.copy()
    _same(a.mj_step_f32(ctrl, 5), b.mj_step_f32(ctrl, 5))
    assert np.array_equal(a.rec, b.rec) and not np.array_equal(a.rec, ra) and np.array_equal(ra, rb)


@pytest.mark.parametrize("xml,pre", [("flat", 0), ("uneven", 30)])
def test_distinct_rows_single_step_match_oracle(oracle, xml, pre):
    """ten envs with ten different rows (every field scaled in [0.7, 1.3]): one env step from identical states agrees
    with the oracle built from each env's row to 1e-9"""
    n = 10
    rng = np.random.default_rng(4)
    rows = _random_rows(M.load_model(xml), rng, n)
    w = E.EmulWarp(xml, n, rows=rows)
    mjs = [oracle.MjLike(xml, **M.param_overrides(r)) for r in rows]
    for i, mj in enumerate(mjs):
        for _ in range(pre + i):
            mj.ctrl[:] = rng.uniform(-0.45, -0.15, 6)
            mj.step(20)
    worst = 0.0
    for st in range(8):
        ctrl = rng.uniform(-0.45, 0.15, (n, 6))
        for i, mj in enumerate(mjs):
            w.rec[i, 0:21] = mj.qpos; w.rec[i, 21:39] = mj.qvel; w.rec[i, 39:57] = mj.qacc_warmstart; w.rec[i, 63:69] = mj.act
            mj.ctrl[:] = ctrl[i]
            mj.step(20)
        ten, cfrc, stats = w.mj_step(ctrl, 20)
        for i, mj in enumerate(mjs):
            for x, y in ((w.rec[i, 0:21], mj.qpos), (w.rec[i, 21:39], mj.qvel), (ten[i], mj.ten_length)):
                worst = max(worst, np.abs(x - y).max() / max(1.0, np.abs(y).max()))
            assert stats[i, 4] == 0 and stats[i, 5] == 0
    print(xml, "worst single-step error with distinct rows: %.1e" % worst)
    assert worst < 1e-9
    # the rows matter: the nominal oracle disagrees
    mj0, mj1 = oracle.MjLike(xml), mjs[0]
    mj0.qpos[:] = mj1.qpos; mj0.qvel[:] = mj1.qvel; mj0.act[:] = mj1.act; mj0.qacc_warmstart[:] = mj1.qacc_warmstart
    mj0.ctrl[:] = mj1.ctrl
    mj0.step(20); mj1.step(20)
    assert np.abs(mj0.qpos - mj1.qpos).max() > 1e-6


@pytest.mark.parametrize("xml,kind,task", [("flat", "tr_env", "straight"), ("uneven", "tr_env", "tracking")])
def test_distinct_row_env_semantics_match_oracle_env(xml, kind, task):
    """reset + 12 env steps of one env with its own row against the oracle env whose model carries the row (param_overrides), with
    the tolerances of test_env_semantics_parity; the uneven tracking case has filter actuators (dynprm0) and stiffness
    on all nine tendons"""
    rng = np.random.default_rng(12)
    for trial in range(2):
        row = _random_rows(M.load_model(xml), rng, 1)[0]
        em = E.Emul(xml, row, env_kind=kind, desired_action=task)
        oe = _oracle_env(xml, kind, row, desired_action=task)
        d = _draws(rng, 1)[0]
        o1, o2 = oe.reset(d), em.reset(d)
        assert np.abs(o1 - o2).max() < 1e-7
        for st in range(12):
            a = rng.uniform(-0.45, 0.15, 6)
            ob1, r1, t1, tr1, i1 = oe.step(a)
            ob2, r2, d2, info = em.step(a)
            assert np.abs(ob1 - ob2).max() < 1e-7
            assert abs(r1 - r2) <= 1e-7 * max(1.0, abs(r1))
            assert (t1 or tr1) == d2
            assert info[3] == pytest.approx(i1["x_position"], abs=1e-8)
            assert info[5] == pytest.approx(i1["psi"], abs=1e-7)


def _prange(md, lo, hi):
    return np.stack([M.nominal_params(md), lo, hi])


def test_param_draws_keys_bounds_and_shared_lengthspring_draw():
    md = M.load_model("uneven")
    nom = M.nominal_params(md)
    lo, hi = M.param_scale_ranges({f: (0.8, 1.2) for f in tlib.PARAM})
    pr = _prange(md, lo, hi)
    a, b = E.param_draws(pr, 7, 3, 0), E.param_draws(pr, 7, 3, 0)
    assert np.array_equal(a, b)
    for other in (E.param_draws(pr, 8, 3, 0), E.param_draws(pr, 7, 4, 0), E.param_draws(pr, 7, 3, 1)):
        assert not np.array_equal(a, other)
    rows = E.param_draws(pr, 1, 0, 0, n=4000)
    assert np.array_equal(rows[5], E.param_draws(pr, 1, 5, 0)[0])
    lo_v, hi_v = np.minimum(nom * 0.8, nom * 1.2), np.maximum(nom * 0.8, nom * 1.2)
    assert ((rows >= lo_v) & (rows <= hi_v)).all()
    s = rows[:, nom != 0] / nom[nom != 0]
    assert abs(s.mean() - 1.0) < 0.01 and abs(s.std() - 0.4 / np.sqrt(12)) < 0.01
    ls = rows[:, 18:36].reshape(-1, 9, 2) / nom[18:36].reshape(9, 2)
    assert np.array_equal(ls[:, :, 0], ls[:, :, 1])                # one draw per tendon
    assert (rows[:, 18:36:2] <= rows[:, 19:36:2]).all()            # the deadband stays ordered
    assert not np.array_equal(ls[:, 0, 0], ls[:, 1, 0])            # ... and the tendons draw independently
    # lo == hi: exactly nominal * lo
    lo2 = np.full(41, 0.9); lo2[0] = 1.0
    assert np.array_equal(E.param_draws(_prange(md, lo2, lo2), 5, 9, 2, n=3), np.tile(nom * lo2, (3, 1)))


@pytest.mark.parametrize("noise", [False, True])
def test_reset_draws_rows_and_other_draws_unchanged(noise):
    """a reset with ranges on draws each env's row from Philox(seed, env id, reset count); the reset draws, reset noise
    and observation noise are those of ranges off; scale 1 reproduces the default variant bit for bit"""
    n, seed = 10, 21
    kw = dict(warmup_steps=3, reset_noise_scale=0.01 if noise else 0.0, use_obs_noise=noise)
    md = M.load_model("flat")
    nom = M.nominal_params(md)
    pr1 = _prange(md, np.ones(41), np.ones(41))
    a, b = E.EmulWarp("flat", n, **kw), E.EmulWarp("flat", n, rows=np.zeros((n, 41)), prange=pr1, **kw)
    rows = b.params
    if noise:
        a.set_noise(seed, 100); b.set_noise(seed, 100)
    _same([a.reset(seed=seed, env_id=100)], [b.reset(seed=seed, env_id=100)])
    assert np.array_equal(rows, np.tile(nom, (n, 1)))
    assert np.array_equal(a.draws, b.draws) and np.array_equal(a.rec, b.rec)
    if noise:
        assert np.array_equal(a.real_obs, b.real_obs)
    act = np.full((n, 6), 0.1)
    _same(a.step(act), b.step(act))
    # ranges on: new rows, the same reset draws
    lo, hi = M.param_scale_ranges({f: (0.8, 1.2) for f in tlib.PARAM})
    pr = _prange(a.md, lo, hi)
    c = E.EmulWarp("flat", n, rows=np.zeros((n, 41)), prange=pr, **kw)
    rows = c.params
    c.rec[:, 85] = 3          # reset count 3
    a.rec[:, 85] = 3
    c.reset(seed=seed, env_id=100); a.reset(seed=seed, env_id=100)
    assert np.array_equal(rows, E.param_draws(pr, seed, 100, 3, n=n))
    assert np.array_equal(a.draws, c.draws)
    d = np.zeros(10)
    E.lib().tbe_make_draws(E.P(d), C.c_ulonglong(seed), C.c_ulonglong(104), C.c_ulonglong(3))
    assert np.array_equal(c.draws[4], d)


def test_pool_slot_draws_its_row_at_phase_zero():
    n_envs, n_pool, seed = 2, 3, 5
    md = M.load_model("flat")
    lo, hi = M.param_scale_ranges({"ten_stiffness": (0.5, 1.5), "act_gain": (0.9, 1.1)})
    pr = _prange(md, lo, hi)
    w = E.EmulWarp("flat", n_envs, rows=np.tile(M.nominal_params(md), (n_envs + n_pool, 1)), prange=pr, warmup_steps=2)
    rows = w.params
    rec = np.zeros((n_envs + n_pool, 96)); rec[:, 0:21] = w.md["qpos0"]
    head = np.zeros((n_envs + n_pool, 32)); draws = np.zeros((n_envs + n_pool, 10))
    pool_obs = np.zeros((n_pool, w.cfg.obs_dim))
    w.pool(n_pool, rec, head, draws, pool_obs, seed)
    assert np.array_equal(rows[n_envs:], E.param_draws(pr, seed, 1 << 40, 0, n=n_pool))
    assert np.array_equal(rows[:n_envs], np.tile(M.nominal_params(w.md), (n_envs, 1)))
    before = rows.copy()
    w.pool(n_pool, rec, head, draws, pool_obs, seed)
    assert np.array_equal(rows, before)       # later phases keep the row
    assert (rec[n_envs:, 84] == 3).all()      # warmup_steps + 1: ready


def test_nominal_params_match_model_struct():
    for xml in ("flat", "uneven"):
        md = M.load_model(xml)
        row = M.nominal_params(md)
        assert np.array_equal(row, E.nominal_params(md))
        ov = M.param_overrides(row)
        for k, v in ov.items():
            assert np.array_equal(np.asarray(v, float).reshape(-1), np.asarray(md[k], float).reshape(-1)), k
        assert tlib.NPARAM == 41 and sum(s.stop - s.start for s in tlib.PARAM.values()) == 41
        assert np.array_equal(row[tlib.PARAM["ten_lengthspring"]], np.asarray(md["ten_lengthspring"], float).reshape(-1))


def test_param_ranges_conversion_and_validation():
    lo, hi = M.param_scale_ranges({"ten_stiffness": (0.8, np.linspace(1.0, 1.2, 9)), "act_bias": ([0.5, 0.6, 0.7], 1.0)})
    assert np.array_equal(lo[0:9], np.full(9, 0.8)) and np.array_equal(hi[0:9], np.linspace(1.0, 1.2, 9))
    assert np.array_equal(lo[37:40], [0.5, 0.6, 0.7]) and np.array_equal(hi[37:40], np.ones(3))
    assert np.array_equal(lo[9:37], np.ones(28)) and lo[40] == hi[40] == 1.0
    bad = [{"nope": (1, 1)}, {"ten_damping": (np.ones(3), 1)}, {"ten_damping": 1.0}, {"act_gain": (1.2, 0.8)},
           {"act_gain": (-0.1, 1.0)}, {"act_dynprm0": (0.0, 1.0)}, {"act_gain": (np.nan, 1.0)},
           {"act_gain": (1.0, np.inf)}, {"ten_lengthspring": (np.linspace(0.8, 0.9, 18), 1.0)}]
    for pr in bad:
        with pytest.raises(ValueError):
            M.param_scale_ranges(pr)
    with pytest.raises(ValueError):
        M.param_overrides(np.zeros(40))
