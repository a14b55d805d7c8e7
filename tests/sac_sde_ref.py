"""Float64 restatement of one gradient step of the reference's SAC with gSDE (core/sac/sac.py loop body, core/sac/policies.py Actor with
use_sde=True, core/common/distributions.py StateDependentNoiseDistribution with learn_features=True, full_std=True, use_expln=False), written
with torch autograd and torch.optim.Adam in float64, and the closed-form gradient of the gSDE head that csrc/cstr_td3.cu implements.

Semantics (SB3 2.x): reset_noise() once per gradient step with batch size 1, so ONE E = exp(log_std) * eps (an rsample) serves every row of
actions_pi, next_actions and the actor loss; mean = Hardtanh(mu(latent), +-clip_mean); sigma = sqrt(latent^2 @ std^2 + 1e-6); a = tanh(mean +
latent @ E); log_prob inverts the tanh: g = atanh(clamp(a, -1 + eps32, 1 - eps32)), sum_j Normal(mean_j, sigma_j).log_prob(g_j) - sum_j
log(1 - tanh(g_j)^2 + 1e-6).  a is rounded to float32 before the inversion, as the reference's float32 tensors are: that rounding, not
the float64 arithmetic, decides where the clamp binds and dominates the error of g near |a| = 1.
"""
import numpy as np
import torch

F64 = torch.float64
EPS32 = float(np.finfo(np.float32).eps)


class _Tanh32(torch.autograd.Function):
    """tanh rounded to float32, with the backward torch's float32 tanh has: grad * (1 - y^2) of the stored (rounded) output y."""

    @staticmethod
    def forward(ctx, u):
        y = torch.tanh(u).float().double()
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, grad):
        (y,) = ctx.saved_tensors
        return grad * (1 - y * y)


def mlp(params, x, relu_last=False):
    W1, b1, W2, b2 = params[:4]
    h = torch.relu(torch.relu(x @ W1.T + b1) @ W2.T + b2)
    return h


def sde_head(latent, w_mu, b_mu, log_std, E, clip_mean):
    """(a, log_prob) of the gSDE actor for latent rows and exploration matrix E."""
    mu = latent @ w_mu.T + b_mu
    mean = torch.clamp(mu, -clip_mean, clip_mean) if clip_mean > 0 else mu
    std = torch.exp(log_std)
    sigma = torch.sqrt((latent ** 2) @ (std ** 2) + 1e-6)
    a = _Tanh32.apply(mean + latent @ E)
    g = torch.atanh(torch.clamp(a, -1.0 + EPS32, 1.0 - EPS32))
    lp = torch.distributions.Normal(mean, sigma).log_prob(g).sum(1) - torch.log(1.0 - torch.tanh(g) ** 2 + 1e-6).sum(1)
    return a, lp


class SACSDEReference:
    """nets: dict of numpy arrays as FusedSACUpdate.nets() returns them (actor head slot = [mu.weight | log_std], bias [mu.bias | 0 0])."""

    def __init__(self, nets, h2, lr=3e-4, gamma=0.99, tau=0.005, target_entropy=-2.0, log_ent_coef=0.0, clip_mean=2.0):
        t = lambda a: torch.tensor(np.asarray(a, np.float64), dtype=F64, requires_grad=True)  # noqa: E731
        A = nets["actor"]
        self.h2, self.clip_mean = h2, clip_mean
        self.trunk = [t(A[i]) for i in range(4)]
        head = np.asarray(A[4], np.float64).reshape(-1)
        self.w_mu, self.log_std, self.b_mu = t(head[: 2 * h2].reshape(2, h2)), t(head[2 * h2:].reshape(h2, 2)), t(np.asarray(A[5])[:2])
        self.actor = [self.log_std] + self.trunk + [self.w_mu, self.b_mu]  # log_std is actor.parameters()[0] in the reference
        self.critics = [[t(x) for x in nets[f"critic{z}"]] for z in range(2)]
        self.critic_targets = [[torch.tensor(np.asarray(x, np.float64), dtype=F64) for x in nets.get(f"critic{z}_target", nets[f"critic{z}"])]
                               for z in range(2)]
        self.log_ent = torch.tensor([log_ent_coef], dtype=F64, requires_grad=True)
        self.opt_a = torch.optim.Adam(self.actor, lr=lr)
        self.opt_c = torch.optim.Adam([p for c in self.critics for p in c], lr=lr)
        self.opt_e = torch.optim.Adam([self.log_ent], lr=lr)
        self.gamma, self.tau, self.target_entropy = gamma, tau, target_entropy

    @staticmethod
    def q(c, x):
        W1, b1, W2, b2, W3, b3 = c
        return torch.relu(torch.relu(x @ W1.T + b1) @ W2.T + b2) @ W3.T + b3

    def head(self, obs, E):
        return sde_head(mlp(self.trunk, obs), self.w_mu, self.b_mu, self.log_std, E, self.clip_mean)

    def step(self, obs, act, next_obs, dones, rewards, eps):
        """One gradient step; eps (h2, 2) standard normal.  Returns the losses and the actor gradients (log_std, mu.weight, mu.bias)."""
        d = lambda x: torch.as_tensor(np.asarray(x, np.float64), dtype=F64)  # noqa: E731
        obs, act, next_obs, dones, rewards = map(d, (obs, act, next_obs, dones, rewards))
        dones, rewards = dones.reshape(-1, 1), rewards.reshape(-1, 1)
        E = torch.exp(self.log_std) * d(eps)  # reset_noise(): rsample, differentiable in log_std
        a_pi, lp = self.head(obs, E)
        lp = lp.reshape(-1, 1)
        ent_coef = torch.exp(self.log_ent.detach())
        ent_loss = -(self.log_ent * (lp + self.target_entropy).detach()).mean()
        self.opt_e.zero_grad()
        ent_loss.backward()
        self.opt_e.step()
        with torch.no_grad():
            na, nlp = self.head(next_obs, E)
            x = torch.cat([next_obs, na], 1)
            qn = torch.minimum(self.q(self.critic_targets[0], x), self.q(self.critic_targets[1], x)) - ent_coef * nlp.reshape(-1, 1)
            target = rewards + (1 - dones) * self.gamma * qn
        x = torch.cat([obs, act], 1)
        critic_loss = 0.5 * sum(torch.nn.functional.mse_loss(self.q(c, x), target) for c in self.critics)
        self.opt_c.zero_grad()
        critic_loss.backward()
        self.opt_c.step()
        xp = torch.cat([obs, a_pi], 1)
        qmin = torch.minimum(self.q(self.critics[0], xp), self.q(self.critics[1], xp))
        actor_loss = (ent_coef * lp - qmin).mean()
        self.opt_a.zero_grad()
        for c in self.critics:
            for p in c:
                p.grad = None
        actor_loss.backward()
        grads = [self.log_std.grad.clone(), self.w_mu.grad.clone(), self.b_mu.grad.clone()]
        self.opt_a.step()
        with torch.no_grad():
            for c, tc in zip(self.critics, self.critic_targets):
                for p, tp in zip(c, tc):
                    tp.mul_(1 - self.tau).add_(self.tau * p)
        return dict(critic_loss=critic_loss.item(), actor_loss=actor_loss.item(), ent_loss=ent_loss.item(), a_pi=a_pi.detach().numpy(),
                    log_prob=lp.detach().numpy().ravel(), grads=[g.numpy() for g in grads], E=E.detach().numpy())

    def actor_head_params(self):
        """(mu.weight, log_std, mu.bias) as numpy float64."""
        return self.w_mu.detach().numpy(), self.log_std.detach().numpy(), self.b_mu.detach().numpy()


def sde_head_grads_closed_form(latent, w_mu, b_mu, log_std, E, clip_mean, dL_da, c):
    """The gradient csrc/cstr_td3.cu's sac_sde_bwd_head_kernel / sac_sde_wgrad_kernel form, in float64 NumPy, for the loss
    L = sum_b (dL_da[b] . a[b]) + c * sum_b log_prob[b] with E held fixed apart from its own dependence on log_std (E = std * eps):
    returns d latent, d mu.weight, d mu.bias, d log_std."""
    std2 = np.exp(2 * log_std)
    mu = latent @ w_mu.T + b_mu
    inside = (np.abs(mu) < clip_mean) if clip_mean > 0 else np.ones_like(mu, bool)
    mean = np.clip(mu, -clip_mean, clip_mean) if clip_mean > 0 else mu
    sigma = np.sqrt(latent ** 2 @ std2 + 1e-6)
    a = np.tanh(mean + latent @ E).astype(np.float32).astype(np.float64)
    clamped = (a < -1 + EPS32) | (a > 1 - EPS32)
    g = np.arctanh(np.clip(a, -1 + EPS32, 1 - EPS32))
    d, t = g - mean, np.tanh(g)
    dlp_dg = np.where(clamped, 0.0, -d / sigma ** 2 + 2 * t * (1 - t * t) / (1 - t * t + 1e-6))
    du = dL_da * (1 - a * a) + c * dlp_dg
    dmu = np.where(inside, du + c * d / sigma ** 2, 0.0)
    dn = du
    dvar = c * (d * d / sigma ** 3 - 1 / sigma) / (2 * sigma)
    dlat = dmu @ w_mu + dn @ E.T + 2 * latent * (dvar @ std2.T)
    dw_mu, db_mu = dmu.T @ latent, dmu.sum(0)
    dlog_std = (latent.T @ dn) * E + 2 * std2 * ((latent ** 2).T @ dvar)
    return dlat, dw_mu, db_mu, dlog_std
