"""SAC learner (SURVEY 8(f) rank 3) on CPU tensors: replay-buffer semantics, the SB3 loss formulas against an
independent numpy restatement, target update, checkpoint layout, a toy learning run.  The GPU twin (CUDA graph,
real simulator) is tests/test_gpu_sac.py."""
import io
import math
import zipfile

import numpy as np
import pytest
import torch

from tensegrity_rl_b200.sac import ReplayBuffer, SACLearner
from tensegrity_rl_b200.spaces import Box


def test_replay_ring_and_sampling():
    b = ReplayBuffer(10, 3, 2, "cpu")
    mk = lambda n, v: (torch.full((n, 3), float(v)), torch.full((n, 3), v + 0.5), torch.full((n, 2), -float(v)),
                       torch.full((n,), float(v)), torch.zeros(n))
    b.add(*mk(4, 1)); b.add(*mk(4, 2))
    assert b.size == 8 and not b.full and int(b.size_t) == 8
    idx = b.sample_indices(1000)
    assert int(idx.min()) >= 0 and int(idx.max()) <= 7          # never an unwritten slot
    b.add(*mk(4, 3))                                               # wraps: slots 8, 9, 0, 1
    assert b.full and b.size == 10 and b.pos == 2
    assert b.rew.tolist() == [3, 3, 1, 1, 2, 2, 2, 2, 3, 3]
    o, a, no, d, r = b.gather(torch.tensor([0, 2, 9]))
    assert o[:, 0].tolist() == [3, 1, 3] and no[:, 0].tolist() == [3.5, 1.5, 3.5] and a[:, 0].tolist() == [-3, -1, -3]
    with pytest.raises(ValueError):
        b.add(*mk(11, 4))


def _mlp(sd, prefix, x, n):
    for k in range(n):
        x = x @ sd[f"{prefix}.{2 * k}.weight"].T + sd[f"{prefix}.{2 * k}.bias"]
        if k < n - 1 or prefix.endswith("latent_pi"):
            x = np.maximum(x, 0)
    return x


def test_losses_match_numpy_restatement_of_sb3():
    """SB3 2.2.1 SAC.train formulas (sac.py:197-264 of that package), written out with numpy on the same weights."""
    L = SACLearner(7, 3, action_low=-1.0, action_high=2.0, device="cpu", seed=3, gamma=0.97)
    with torch.no_grad():
        L.log_ent_coef.fill_(math.log(0.37))
    g = torch.Generator().manual_seed(0)
    B = 16
    obs, nobs = torch.randn(B, 7, generator=g), torch.randn(B, 7, generator=g)
    act = torch.rand(B, 3, generator=g) * 2 - 1
    rew, done = torch.randn(B, generator=g), (torch.rand(B, generator=g) < 0.3).float()
    e1, e2 = torch.randn(B, 3, generator=g), torch.randn(B, 3, generator=g)
    ent_l, crit_l, act_l, ent_coef = [float(x.detach()) for x in L.losses(obs, act, nobs, done, rew, e1, e2)]
    sd = {k: v.detach().numpy().astype(np.float64) for k, v in L.policy.state_dict().items()}

    def pi(o, eps):
        z = _mlp(sd, "actor.latent_pi", o, 2)
        mu = z @ sd["actor.mu.weight"].T + sd["actor.mu.bias"]
        ls = np.clip(z @ sd["actor.log_std.weight"].T + sd["actor.log_std.bias"], -20, 2)
        gs = mu + np.exp(ls) * eps
        a = np.tanh(gs)
        logp = (-0.5 * ((gs - mu) / np.exp(ls)) ** 2 - ls - 0.5 * np.log(2 * np.pi)).sum(1) - np.log(1 - a * a + 1e-6).sum(1)
        return a, logp

    q = lambda net, o, a: np.minimum(_mlp(sd, net + ".qf0", np.concatenate([o, a], 1), 3),
                                     _mlp(sd, net + ".qf1", np.concatenate([o, a], 1), 3))[:, 0]
    o, no, a_b, r, d = (x.numpy().astype(np.float64) for x in (obs, nobs, act, rew, done))
    a_pi, logp = pi(o, e1.numpy().astype(np.float64))
    a_n, logp_n = pi(no, e2.numpy().astype(np.float64))
    alpha = 0.37
    target = r + (1 - d) * 0.97 * (q("critic_target", no, a_n) - alpha * logp_n)
    x = np.concatenate([o, a_b], 1)
    c0, c1 = _mlp(sd, "critic.qf0", x, 3)[:, 0], _mlp(sd, "critic.qf1", x, 3)[:, 0]
    assert crit_l == pytest.approx(0.5 * (((c0 - target) ** 2).mean() + ((c1 - target) ** 2).mean()), rel=2e-5)
    assert act_l == pytest.approx((alpha * logp - q("critic", o, a_pi)).mean(), rel=2e-5, abs=1e-6)
    assert ent_l == pytest.approx(-(math.log(0.37) * (logp + (-3.0))).mean(), rel=2e-5)
    assert ent_coef == pytest.approx(0.37, rel=1e-6)
    assert L.target_entropy == -3.0


def test_update_order_and_polyak():
    L = SACLearner(4, 2, device="cpu", seed=0, batch_size=8, buffer_size=64, tau=0.25)
    L.buffer.add(torch.randn(32, 4), torch.randn(32, 4), torch.rand(32, 2) * 2 - 1, torch.randn(32), torch.zeros(32))
    before = {k: v.clone() for k, v in L.policy.state_dict().items()}
    alpha0 = float(L.log_ent_coef)
    L.update(1)
    after = L.policy.state_dict()
    for k in before:
        if k.startswith("critic_target."):
            src = k.replace("critic_target.", "critic.")
            assert torch.allclose(after[k], 0.75 * before[k] + 0.25 * after[src], atol=1e-7)   # Polyak on the NEW critic
        else:
            assert not torch.equal(after[k], before[k])                                       # actor and critic both stepped
    assert float(L.log_ent_coef) != alpha0 and L.n_updates == 1
    for p in L.policy.critic_target.parameters():
        assert not p.requires_grad


def test_checkpoint_layout_and_roundtrip(tmp_path):
    L = SACLearner(45, 6, device="cpu", seed=5, batch_size=8, buffer_size=64)
    L.buffer.add(torch.randn(16, 45), torch.randn(16, 45), torch.rand(16, 6) * 2 - 1, torch.randn(16), torch.zeros(16))
    L.update(2)
    L.num_timesteps = 16
    with pytest.warns(UserWarning, match="not resumed from an SB3 checkpoint"):   # the `data` entry is plain JSON then
        p = L.save(str(tmp_path / "SAC_16.zip"))
    names = set(zipfile.ZipFile(p).namelist())
    assert {"data", "policy.pth", "pytorch_variables.pth", "actor.optimizer.pth", "critic.optimizer.pth",
            "ent_coef_optimizer.pth", "_stable_baselines3_version"} <= names
    sd = torch.load(io.BytesIO(zipfile.ZipFile(p).read("policy.pth")), weights_only=True)
    assert sd["actor.latent_pi.0.weight"].shape == (256, 45) and sd["critic.qf1.4.weight"].shape == (1, 256)
    assert sd["critic_target.qf0.0.weight"].shape == (256, 51) and sd["actor.log_std.bias"].shape == (6,)
    L2 = SACLearner(45, 6, device="cpu", seed=9, batch_size=8, buffer_size=64).load_sb3_zip(p)
    o = torch.randn(50, 45)
    assert torch.equal(L.act(o, deterministic=True)[1], L2.act(o, deterministic=True)[1])
    assert (L2.num_timesteps, L2.n_updates) == (16, 2) and float(L2.log_ent_coef) == float(L.log_ent_coef)
    # the zip is also readable by the rollout-side actor loader (policy.py), i.e. by everything that reads SB3 zips here
    from tensegrity_rl_b200.policy import SacActor
    act = SacActor(p, device="cpu")
    assert torch.allclose(act(o, deterministic=True), L.act(o, deterministic=True)[1], atol=1e-6)
    # Adam state survives: the same next update on both
    torch.manual_seed(1); L.update(1)
    L2.buffer.add(L.buffer.obs[:16], L.buffer.next_obs[:16], L.buffer.act[:16], L.buffer.rew[:16], L.buffer.done[:16])
    torch.manual_seed(1); L2.update(1)
    for a, b in zip(L.policy.parameters(), L2.policy.parameters()):
        assert torch.allclose(a, b, atol=1e-6)


class _Bandit:
    """tensor-protocol toy env: every step terminates; reward peaks at ctrl = 0.05 on every tendon"""
    def __init__(self, n=32, obs_dim=4):
        self.num_envs, self.obs_dim, self.auto_reset = n, obs_dim, True
        self.action_space = Box(np.full(6, -0.45, np.float32), np.full(6, 0.15, np.float32), dtype=np.float32)
        self.info = torch.zeros(n, 32, dtype=torch.float64)
        self.term_obs = torch.zeros(n, obs_dim, dtype=torch.float64)
        self.obs = torch.zeros(n, obs_dim, dtype=torch.float64)

    def reset_tensor(self):
        self.obs.normal_()
        return self.obs

    def step_tensor(self, ctrl):
        r = -((ctrl.double() - 0.05) ** 2).sum(1) * 100
        self.term_obs.copy_(self.obs)
        self.obs.normal_()
        self.info[:, 17] = 1
        return self.obs, r, torch.ones(self.num_envs, dtype=torch.uint8)


def test_learn_loop_improves_a_bandit():
    torch.set_num_threads(2)
    env = _Bandit()
    L = SACLearner(env.obs_dim, 6, device="cpu", learning_starts=128, batch_size=64, buffer_size=5000, gradient_steps=2, seed=1)
    o = torch.randn(500, env.obs_dim)
    r0 = float(-((L.act(o, deterministic=True)[1] - 0.05) ** 2).sum(1).mean())
    L.learn(env, 32 * 120)
    assert L.num_timesteps == 32 * 120 and L.n_updates == 2 * (120 - 4) and L.buffer.size == 32 * 120
    assert float(L.buffer.done[:L.buffer.size].min()) == 1.0                      # terminations stored as done
    r1 = float(-((L.act(o, deterministic=True)[1] - 0.05) ** 2).sum(1).mean())
    assert r1 > r0 * 0.6 and torch.isfinite(L.last_losses).all()    # squared distance to the optimum shrinks
