"""not gpu: the host side of gSDE in the fused rollout — the launch plan of one collect_rollouts call (learning_starts, sde_sample_freq,
use_sde_at_warmup and the reference's reset_noise count) and the named reasons a gSDE model keeps the reference's collect_rollouts."""
import importlib
from types import SimpleNamespace

import pytest
import torch
import torch.nn as nn

rollout = importlib.import_module("pytorch-rl-enhancedstablebaselines_b200.rollout")


def reference_schedule(K, n_envs, num_timesteps, learning_starts, use_sde, sde_sample_freq, use_sde_at_warmup):
    """Step by step what the reference's collect_rollouts / _sample_action do (off_policy_algorithm.py): per step, whether the action is
    the uniform warm-up draw and how many reset_noise calls precede it."""
    out, t = [], num_timesteps
    for step in range(K):
        resets = int(use_sde and step == 0)  # reset_noise(env.num_envs) before the loop
        if use_sde and sde_sample_freq > 0 and step % sde_sample_freq == 0:
            resets += 1
        out.append((t < learning_starts and not (use_sde and use_sde_at_warmup), resets))
        t += n_envs
    return out


def expand(plan):
    steps = []
    for k, warm, resets in plan:
        assert k > 0
        steps += [(warm, resets)] + [(warm, 0)] * (k - 1)
    return steps


@pytest.mark.parametrize("K,n_envs,t0,learning_starts", [(10, 4, 0, 0), (10, 4, 0, 20), (7, 3, 9, 20), (16, 1, 0, 5), (1, 8, 0, 100)])
@pytest.mark.parametrize("freq", [None, -1, 0, 1, 3, 4, 16])
@pytest.mark.parametrize("at_warmup", [False, True])
def test_launch_plan_is_the_reference_schedule(K, n_envs, t0, learning_starts, freq, at_warmup):
    use_sde = freq is not None
    plan = rollout.launch_plan(K, n_envs, t0, learning_starts, freq, at_warmup and use_sde)
    assert expand(plan) == reference_schedule(K, n_envs, t0, learning_starts, use_sde, freq or 0, at_warmup)
    # no launch is split where the reference changes nothing: a launch starts only at the call start, at learning_starts or at a reset
    starts = [sum(k for k, _, _ in plan[:i]) for i in range(len(plan))]
    for s, (_, warm, resets) in zip(starts[1:], plan[1:]):
        prev_warm = expand(plan)[s - 1][0]
        assert resets or warm != prev_warm


def test_launch_plan_without_gsde_is_the_learning_starts_split():
    """What bind_offpolicy_rollout launched before gSDE existed: the whole call, split once where warm-up ends."""
    for K, n_envs, t0, ls in [(10, 4, 0, 20), (10, 4, 40, 20), (5, 16, 0, 17), (3, 2, 0, 0)]:
        want, remaining, t = [], K, t0
        while remaining > 0:
            warm = t < ls
            k = min(remaining, -(-(ls - t) // n_envs)) if warm else remaining
            want.append((k, warm, 0))
            remaining -= k
            t += n_envs * k
        assert rollout.launch_plan(K, n_envs, t0, ls) == want


class FlattenExtractor(nn.Module):  # matched by class name, as the reference's is
    pass


def _sde_actor(h=(64, 64), mu=None, log_std_shape=None, **flags):
    trunk = nn.Sequential(nn.Linear(4, h[0]), nn.ReLU(), nn.Linear(h[0], h[1]), nn.ReLU())
    mu = mu if mu is not None else nn.Sequential(nn.Linear(h[1], 2), nn.Hardtanh(-2.0, 2.0))
    log_std = nn.Parameter(torch.full(log_std_shape or (h[1], 2), -3.0))
    return SimpleNamespace(features_extractor=FlattenExtractor(), latent_pi=trunk, mu=mu, log_std=log_std, use_sde=True, use_expln=False,
                           full_std=True, **flags)


def test_gsde_guard_names_each_refused_option():
    why = rollout._actor_unsupported
    assert why(_sde_actor(), "fp32") is None
    assert why(_sde_actor(mu=nn.Linear(64, 2)), "fp32") is None  # clip_mean <= 0: no Hardtanh
    assert "Linear + Hardtanh" in why(_sde_actor(mu=nn.Sequential(nn.Linear(64, 2), nn.Tanh())), "fp32")
    assert "Linear + Hardtanh" in why(_sde_actor(mu=nn.Sequential(nn.Linear(64, 2), nn.Hardtanh(-1.0, 2.0))), "fp32")
    assert "(H2, 2) parameter" in why(_sde_actor(log_std_shape=(64, 1)), "fp32")
    assert "H1 <= 448" in why(_sde_actor(h=(512, 64)), "fp32")
    sde = rollout._sde_unsupported
    assert sde(_sde_actor(), "fp32", False) is None
    assert "use_expln=True" in sde(_sde_actor().__class__(**{**vars(_sde_actor()), "use_expln": True}), "fp32", False)
    assert "full_std=False" in sde(_sde_actor().__class__(**{**vars(_sde_actor()), "full_std": False}), "fp32", False)
    assert "actor_mode='tc'" in sde(_sde_actor(), "tc", False)
    assert "GpuVecNormalize" in sde(_sde_actor(), "fp32", True)
    # the model-level guard reaches the option reasons before it looks at the env
    model = SimpleNamespace(actor=_sde_actor(), use_sde=True, _vec_normalize_env=None)
    freq = SimpleNamespace(unit="step", frequency=4)
    assert "actor_mode='tc'" in rollout.fused_rollout_unsupported(model, None, None, freq, None, actor_mode="tc")


def test_sde_mean_head():
    lin = nn.Linear(8, 2)
    assert rollout.sde_mean_head(lin) == (lin, 0.0)
    assert rollout.sde_mean_head(nn.Sequential(lin, nn.Hardtanh(-2.0, 2.0))) == (lin, 2.0)
    assert rollout.sde_mean_head(nn.Sequential(lin, nn.ReLU())) is None
    assert rollout.sde_mean_head(nn.Sequential(lin)) is None
