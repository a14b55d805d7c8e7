"""SAC with gSDE on the fused update (cstr_sac_update, sde = 1) against the float64 autograd restatement tests/sac_sde_ref.py of the reference's
loop body: explicit exploration eps, three consecutive updates, every GEMM mode; a batch where the atanh clamp binds; graph replay against
launch by launch; two data-parallel ranks drawing the same exploration matrix; the Philox draw's moments; adopt_policy by parameter identity."""
import numpy as np
import pytest
import torch
import torch.nn as nn

import sac_sde_ref as R
import td3_util as U

pytestmark = pytest.mark.gpu
H, B = 64, 256


def _nets(rng, h=H):
    nets = U.random_sac_nets(rng, h, h)
    head = nets["actor"][4].reshape(-1).copy()
    head[2 * h:] = (-1.0 + 0.3 * rng.standard_normal(2 * h)).astype(np.float32)  # log_std (h, 2)
    nets["actor"][4] = head.reshape(4, h)
    nets["actor"][5] = np.concatenate([nets["actor"][5][:2], np.zeros(2, np.float32)])
    return nets


def _batch(rng, obs_scale=1.0):
    f = np.float32
    return (rng.uniform(-1, 1, (B, 4)).astype(f) * f(obs_scale), rng.uniform(-1, 1, (B, 2)).astype(f), rng.uniform(-1, 1, (B, 4)).astype(f),
            (rng.uniform(0, 1, (B, 1)) < 0.1).astype(f), rng.standard_normal((B, 1)).astype(f))


def _rel(got, want):
    return float(np.linalg.norm(np.asarray(got, np.float64) - want) / max(np.linalg.norm(want), 1e-30))


@pytest.mark.parametrize("gemm,tol", [("fp32", 2e-4), ("tensor", 2e-2), ("bf16", 5e-2)])
@pytest.mark.parametrize("obs_scale", [1.0, 60.0], ids=["plain", "clamp_binds"])
def test_three_updates_against_float64_reference(pkg, gemm, tol, obs_scale):
    rng = np.random.default_rng(3)
    nets = _nets(rng)
    eng = pkg.FusedSACUpdate([H, H], B, seed=1, gemm=gemm, sde=True, clip_mean=2.0)
    eng.load_nets(nets)
    ref = R.SACSDEReference(nets, H, clip_mean=2.0)
    clamped = 0.0
    for step in range(3):
        batch = _batch(rng, obs_scale)
        eps = rng.standard_normal((H, 2)).astype(np.float32)
        out = ref.step(*batch, eps)
        eng.update([torch.as_tensor(x, device="cuda") for x in batch], eps_pi=eps)
        clamped = max(clamped, float(np.mean(np.abs(out["a_pi"]) >= 1 - R.EPS32)))
        gw, gls, gb = eng.sde_views("grads")
        g_ls, g_w, g_b = out["grads"]
        errs = {"d log_std": _rel(gls.cpu().numpy(), g_ls), "d mu.weight": _rel(gw.cpu().numpy(), g_w), "d mu.bias": _rel(gb.cpu().numpy(), g_b)}
        print(f"sde update {gemm} {'clamp' if obs_scale > 1 else 'plain'} step {step}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
        assert max(errs.values()) < tol, errs
        assert torch.equal(eng.views("grads")["actor"][5][2:].cpu(), torch.zeros(2))  # the bias pad gets gradient 0
        w_mu, log_std, b_mu = ref.actor_head_params()
        pw, pls, pb = (x.cpu().numpy() for x in eng.sde_views("params"))
        lr = eng.learning_rate
        # Adam moves every weight by about lr per step: a weight whose gradient sign differs from float64 may be off by 2 lr
        for got, want in ((pls, log_std), (pw, w_mu), (pb, b_mu)):
            assert np.mean(np.abs(got - want) <= 1e-6 + (0.05 if gemm != "fp32" else 0.01) * lr) > 0.95
            assert np.abs(got - want).max() <= 2 * (step + 1) * lr + 1e-6
    if obs_scale > 1:
        assert clamped > 0.2  # the case is the one it claims: the clamp binds on many rows


def test_graph_replay_equals_launch_by_launch(pkg):
    rng = np.random.default_rng(8)
    nets = _nets(rng, 256)
    n_envs = 512
    buf = pkg.GpuReplayBuffer(32 * n_envs, n_envs=n_envs, index_mode="philox", seed=5)
    buf.records.uniform_(-1, 1)
    buf.records[..., 11:13] = 0
    buf.pos, buf.full = 0, True

    def run(graph):
        buf._draw = 0
        eng = pkg.FusedSACUpdate([256, 256], 256, seed=2, sde=True)
        eng.load_nets(nets)
        for steps in (5, 3):
            eng.train(steps, buf, 256, graph=graph)
        return eng

    a, b = run(False), run(True)
    assert a.n_updates == b.n_updates == 8 and b._graph is not None
    np.testing.assert_allclose(b.params.cpu().numpy(), a.params.cpu().numpy(), rtol=0, atol=3e-7)
    np.testing.assert_allclose(b.targets.cpu().numpy(), a.targets.cpu().numpy(), rtol=0, atol=3e-7)
    assert not np.array_equal(a.sde_views("params")[1].cpu().numpy(), nets["actor"][4].reshape(-1)[512:].reshape(256, 2))  # log_std moved


def _explore(eng, h):
    """The update's exploration matrix E (h, 2): the last 4 h floats of the workspace are [E | std^2]."""
    return eng._workspace[-4 * h:-2 * h].view(h, 2)


def test_ranks_draw_the_same_exploration_matrix(pkg):
    """dp_rank keys the other Philox streams, not gSDE's: two ranks with the same seed and batch draw the same E and compute the same
    update bit for bit (averaged gradients are then one process's gradient of the global batch)."""
    rng = np.random.default_rng(4)
    nets = _nets(rng)
    batch = [torch.as_tensor(x, device="cuda") for x in _batch(rng)]
    out = []
    for rank in (0, 1):
        eng = pkg.FusedSACUpdate([H, H], B, seed=7, sde=True, dp_rank=rank)
        eng.load_nets(nets)
        eng.update(batch)
        out.append((_explore(eng, H).cpu().numpy().copy(), eng.params.cpu().numpy().copy(), eng.grads.cpu().numpy().copy()))
    for x, y in zip(*out):
        assert np.array_equal(x, y)


def test_philox_exploration_eps_moments_and_updates_differ(pkg):
    """E / std of the per-update Philox draw: over 10^4 updates each entry's eps has mean and variance within 5 sigma of N(0, 1), and
    consecutive updates draw different matrices."""
    h, n = 8, 10_000
    rng = np.random.default_rng(5)
    nets = _nets(rng, h)
    eng = pkg.FusedSACUpdate([h, h], 4, seed=11, sde=True, learning_rate=0.0)
    eng.load_nets(nets)
    f = np.float32
    batch = [torch.as_tensor(x, device="cuda") for x in (rng.uniform(-1, 1, (4, 4)).astype(f), rng.uniform(-1, 1, (4, 2)).astype(f),
                                                         rng.uniform(-1, 1, (4, 4)).astype(f), np.zeros((4, 1), f), np.zeros((4, 1), f))]
    std = np.exp(eng.sde_views("params")[1].cpu().numpy().astype(np.float64))
    z = np.empty((n, h, 2))
    for k in range(n):
        eng.update(batch)
        z[k] = _explore(eng, h).cpu().numpy() / std
    assert np.allclose(std, np.exp(eng.sde_views("params")[1].cpu().numpy().astype(np.float64)))  # lr 0: log_std fixed
    z = z.reshape(n, -1)
    assert np.all(np.abs(z.mean(0)) < 5.0 / np.sqrt(n))
    assert np.all(np.abs(z.var(0) - 1.0) < 5.0 * np.sqrt(2.0 / n))
    assert np.mean(z[1:] == z[:-1]) < 1e-3


def test_adopt_policy_maps_log_std_and_mu_by_identity(pkg):
    torch.manual_seed(0)
    from types import SimpleNamespace as NS

    def mlp(i, o=None):
        return nn.Sequential(*([nn.Linear(i, H), nn.ReLU(), nn.Linear(H, H), nn.ReLU()] + ([nn.Linear(H, o)] if o else []))).cuda()

    class Actor(nn.Module):  # the reference Actor's registration order: log_std (a direct Parameter) first, then latent_pi, mu
        def __init__(self):
            super().__init__()
            self.log_std = nn.Parameter(torch.full((H, 2), -3.0, device="cuda"))
            self.latent_pi = mlp(4)
            self.mu = nn.Sequential(nn.Linear(H, 2), nn.Hardtanh(-2.0, 2.0)).cuda()

    actor = Actor()
    assert next(iter(actor.parameters())) is actor.log_std
    critic, critic_t = NS(q_networks=[mlp(6, 1), mlp(6, 1)]), NS(q_networks=[mlp(6, 1), mlp(6, 1)])
    opt = torch.optim.Adam(actor.parameters(), lr=3e-4)
    (actor.log_std.sum() + sum(p.sum() for p in actor.mu.parameters())).backward()
    opt.step()
    m_ls = opt.state[actor.log_std]["exp_avg"].clone()
    eng = pkg.FusedSACUpdate([H, H], B, sde=True)
    eng.adopt_policy(NS(actor=actor, critic=critic, critic_target=critic_t))
    copt = torch.optim.Adam([p for q in critic.q_networks for p in q.parameters()], lr=3e-4)
    eng.import_optimizer_state(opt, copt)
    w_mu, log_std, b_mu = eng.sde_views("params")
    assert actor.log_std.data_ptr() == log_std.data_ptr() and actor.mu[0].weight.data_ptr() == w_mu.data_ptr()
    assert actor.mu[0].bias.data_ptr() == b_mu.data_ptr()
    off = (log_std.data_ptr() - eng.params.data_ptr()) // 4
    assert torch.equal(eng.adam_m[off:off + 2 * H].view(H, 2), m_ls)
    eng.update([torch.as_tensor(x, device="cuda") for x in _batch(np.random.default_rng(0))])
    eng.export_optimizer_state(opt, copt)
    assert opt.state[actor.log_std]["exp_avg"].data_ptr() == eng.adam_m[off:off + 2 * H].data_ptr()
