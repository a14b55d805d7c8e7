"""Hand-over of torch modules and Adam state to the fused update engines and back, for TD3 (two critics and one), SAC, BCQ, MADDPG
and IDDPG.

Each case builds ``SimpleNamespace`` stand-ins for the reference policy at the attribute paths the engine's ``adopt_policy`` reads, and
``torch.optim.Adam`` optimisers that have taken a few steps on random gradients (different step counts per optimiser).  After
``adopt_policy`` and ``import_optimizer_state``:
  * every module parameter is a view of the engine's ``params`` block (``targets`` for the target nets; BCQ's target VAE shares the VAE),
  * the engine's moments at each parameter's offset equal the optimiser's ``exp_avg`` / ``exp_avg_sq`` bit for bit,
  * ``critic_step`` / ``actor_step`` follow the engine's mapping of optimisers to counters.
After one ``update()`` and ``export_optimizer_state`` the optimisers' state tensors are the engine's moment views and carry the step
counts of the engine's counters.
"""
from types import SimpleNamespace as NS

import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

B = 64


def _mlp(i, h1, h2, o=None, squash=False):
    layers = [nn.Linear(i, h1), nn.ReLU(), nn.Linear(h1, h2), nn.ReLU()] + ([nn.Linear(h2, o)] if o else []) + ([nn.Tanh()] if squash else [])
    return nn.Sequential(*layers).cuda()


def _adam(params, steps, gen):
    """torch Adam over ``params`` after ``steps`` steps on random gradients: non-zero moments and a known step count."""
    params = list(params)
    opt = torch.optim.Adam(params, lr=1e-3)
    for _ in range(steps):
        for p in params:
            p.grad = torch.randn(p.shape, generator=gen, device="cuda")
        opt.step()
    for p in params:
        p.grad = None
    return opt


def _copy(dst, src):
    dst.load_state_dict(src.state_dict())
    return dst


def _td3(pkg, gen, n_critics):
    h1, h2 = 64, 48
    actor = _mlp(4, h1, h2, 2, True)
    qs = [_mlp(6, h1, h2, 1) for _ in range(n_critics)]
    policy = NS(actor=NS(mu=actor), actor_target=NS(mu=_copy(_mlp(4, h1, h2, 2, True), actor)),
                critic=NS(q_networks=qs), critic_target=NS(q_networks=[_copy(_mlp(6, h1, h2, 1), q) for q in qs]))
    opts = (_adam(actor.parameters(), 1, gen), _adam([p for q in qs for p in q.parameters()], 2, gen))
    eng = pkg.FusedTD3Update([h1, h2], B, n_critics=n_critics)
    online = [actor] + qs
    targets = [policy.actor_target.mu] + policy.critic_target.q_networks
    # import: actor_step from the actor optimiser, critic_step from the critic optimiser; export hands each its own counter
    return dict(eng=eng, policy=policy, online=online, targets=targets, shared=[], opts=opts, steps=(2, 1),
                counters=lambda e: (e.actor_step, e.critic_step))


def _sac(pkg, gen):
    h = 64
    actor = NS(latent_pi=_mlp(4, h, h), mu=nn.Linear(h, 2).cuda(), log_std=nn.Linear(h, 2).cuda())
    qs = [_mlp(6, h, h, 1) for _ in range(2)]
    policy = NS(actor=actor, critic=NS(q_networks=qs), critic_target=NS(q_networks=[_copy(_mlp(6, h, h, 1), q) for q in qs]))
    eng = pkg.FusedSACUpdate([h, h], B, ent_coef_init=0.8)
    log_ent = eng.log_ent_coef.clone().requires_grad_(True)
    actor_params = list(actor.latent_pi.parameters()) + list(actor.mu.parameters()) + list(actor.log_std.parameters())
    opts = (_adam(actor_params, 2, gen), _adam([p for q in qs for p in q.parameters()], 2, gen), _adam([log_ent], 3, gen))
    eng.log_ent_coef.copy_(log_ent.detach())
    log_ent.data = eng.log_ent_coef  # what bind_sac_class does: the coefficient lives in the params block
    # one step count for all three optimisers: the largest found
    return dict(eng=eng, policy=policy, online=[actor.latent_pi, actor.mu, actor.log_std] + qs, targets=policy.critic_target.q_networks,
                shared=[], opts=opts, steps=(3, 3), counters=lambda e: (e.critic_step, e.critic_step, e.critic_step))


def _bcq(pkg, gen):
    L, hv, hp, h1, h2 = 8, 36, 20, 36, 20

    def vae():
        return NS(encoder=_mlp(6, hv, hv), mean=nn.Linear(hv, L).cuda(), log_std=nn.Linear(hv, L).cuda(), decoder=_mlp(4 + L, hv, hv, 2))

    def modules(v):
        return [v.encoder, v.mean, v.log_std, v.decoder]

    v, vt = vae(), vae()
    pert, pert_t = _mlp(6, hp, hp, 2), _mlp(6, hp, hp, 2)
    _copy(pert_t, pert)
    qs = [_mlp(6, h1, h2, 1) for _ in range(2)]
    policy = NS(actor=NS(vae=v, perturbation=NS(model=pert)), actor_target=NS(vae=vt, perturbation=NS(model=pert_t)),
                critic=NS(q_networks=qs), critic_target=NS(q_networks=[_copy(_mlp(6, h1, h2, 1), q) for q in qs]))
    opts = (_adam([p for m in modules(v) for p in m.parameters()], 3, gen), _adam(pert.parameters(), 1, gen),
            _adam([p for q in qs for p in q.parameters()], 2, gen))
    eng = pkg.FusedBCQUpdate(L, hv, hp, [h1, h2], B)
    # critic_step = max(vae, critic), actor_step = perturbation
    return dict(eng=eng, policy=policy, online=modules(v) + [pert] + qs, targets=[pert_t] + policy.critic_target.q_networks,
                shared=list(zip(modules(vt), modules(v))), opts=opts, steps=(3, 1),
                counters=lambda e: (e.critic_step, e.actor_step, e.critic_step))


def _ma(pkg, gen, centralised, n_critics):
    h1, h2, ci = 36, 20, 6 if centralised else 3
    mus = [_mlp(2, h1, h2, 1, True) for _ in range(2)]
    qs = [[_mlp(ci, h1, h2, 1) for _ in range(n_critics)] for _ in range(2)]
    policy = NS(actor=NS(mu_list=mus), actor_target=NS(mu_list=[_copy(_mlp(2, h1, h2, 1, True), m) for m in mus]),
                critic=NS(q_networks_list=qs), critic_target=NS(q_networks_list=[[_copy(_mlp(ci, h1, h2, 1), q) for q in qq] for qq in qs]))
    a_opts = [_adam(mus[0].parameters(), 1, gen), _adam(mus[1].parameters(), 2, gen)]
    c_opts = [_adam([p for q in qs[0] for p in q.parameters()], 3, gen), _adam([p for q in qs[1] for p in q.parameters()], 2, gen)]
    eng = pkg.FusedMultiAgentUpdate([h1, h2], B, centralised, n_critics=n_critics)
    # actor_step = the largest actor step, critic_step = the largest critic step
    return dict(eng=eng, policy=policy, online=mus + [q for qq in qs for q in qq],
                targets=policy.actor_target.mu_list + [q for qq in policy.critic_target.q_networks_list for q in qq], shared=[],
                opts=(a_opts, c_opts), flat_opts=a_opts + c_opts, steps=(3, 2),
                counters=lambda e: (e.actor_step, e.actor_step, e.critic_step, e.critic_step))


CASES = {
    "td3": lambda pkg, gen: _td3(pkg, gen, 2),
    "ddpg_one_critic": lambda pkg, gen: _td3(pkg, gen, 1),
    "sac": _sac,
    "bcq": _bcq,
    "maddpg": lambda pkg, gen: _ma(pkg, gen, True, 2),
    "iddpg": lambda pkg, gen: _ma(pkg, gen, False, 1),
}


def _inside(t, block):
    lo, n = block.data_ptr(), block.numel() * block.element_size()
    return lo <= t.data_ptr() and t.data_ptr() + t.numel() * t.element_size() <= lo + n


def _moment_views(eng, p):
    """The engine's (adam_m, adam_v) slices at the offset of adopted parameter ``p`` in the params block."""
    off = (p.data_ptr() - eng.params.data_ptr()) // 4
    n = p.numel()
    return eng.adam_m[off:off + n].view(p.shape), eng.adam_v[off:off + n].view(p.shape)


def _batch(rng):
    return (rng.uniform(-1, 1, (B, 4)).astype(np.float32), rng.uniform(-1, 1, (B, 2)).astype(np.float32), rng.uniform(-1, 1, (B, 4)).astype(np.float32),
            (rng.random((B, 1)) < 0.1).astype(np.float32), rng.normal(size=(B, 1)).astype(np.float32))


@pytest.mark.parametrize("case", list(CASES))
def test_adopt_import_update_export(pkg, case):
    torch.manual_seed(3)
    gen = torch.Generator(device="cuda").manual_seed(11)
    c = CASES[case](pkg, gen)
    eng = c["eng"]
    opts = c.get("flat_opts", list(c["opts"]))
    before = {id(p): (opt.state[p]["exp_avg"].clone(), opt.state[p]["exp_avg_sq"].clone()) for opt in opts for p in opt.param_groups[0]["params"]}
    weights = {id(p): p.detach().clone() for m in c["online"] + c["targets"] for p in m.parameters()}

    eng.adopt_policy(c["policy"])
    eng.import_optimizer_state(*c["opts"])

    for m in c["online"]:
        for p in m.parameters():
            assert _inside(p.data, eng.params) and torch.equal(p.detach(), weights[id(p)])
    for m in c["targets"]:
        for p in m.parameters():
            assert _inside(p.data, eng.targets) and torch.equal(p.detach(), weights[id(p)])
    for mt, m in c["shared"]:  # BCQ's target VAE is the VAE
        for pt, p in zip(mt.parameters(), m.parameters()):
            assert pt.data_ptr() == p.data_ptr() and pt.shape == p.shape
    for opt in opts:
        for p in opt.param_groups[0]["params"]:
            assert _inside(p.data, eng.params)
            m, v = _moment_views(eng, p)
            want_m, want_v = before[id(p)]
            assert torch.equal(m, want_m) and torch.equal(v, want_v)
    critic_step, actor_step = c["steps"]
    assert (eng.critic_step, eng.actor_step) == (critic_step, actor_step)

    eng.n_updates = 1  # the next update is a policy step for policy_delay / actor_delay 2
    eng.update(_batch(np.random.default_rng(5)))
    torch.cuda.synchronize()
    if case == "sac":
        assert eng.critic_step == eng.actor_step == critic_step + 1
    else:
        assert (eng.critic_step, eng.actor_step) == (critic_step + 1, actor_step + 1)

    eng.export_optimizer_state(*c["opts"])
    for opt, step in zip(opts, c["counters"](eng)):
        for p in opt.param_groups[0]["params"]:
            st = opt.state[p]
            m, v = _moment_views(eng, p)
            assert st["exp_avg"].data_ptr() == m.data_ptr() and st["exp_avg_sq"].data_ptr() == v.data_ptr()
            assert st["exp_avg"].shape == p.shape and st["exp_avg_sq"].shape == p.shape
            assert float(st["step"]) == step
