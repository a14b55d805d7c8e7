"""not gpu: the gSDE SAC update's float64 restatement (tests/sac_sde_ref.py) against torch autograd, and the update guard's reasons."""
import importlib
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn as nn

import sac_sde_ref as R

update = importlib.import_module("pytorch-rl-enhancedstablebaselines_b200.update")


def _head_case(B=64, H2=24, clip_mean=2.0, scale=1.0, seed=0):
    rng = np.random.default_rng(seed)
    lat = np.maximum(rng.standard_normal((B, H2)), 0.0) * scale
    w_mu, b_mu = 0.3 * rng.standard_normal((2, H2)), 0.3 * rng.standard_normal(2)
    log_std = -1.0 + 0.3 * rng.standard_normal((H2, 2))
    eps = rng.standard_normal((H2, 2))
    return lat, w_mu, b_mu, log_std, eps, clip_mean, rng.standard_normal((B, 2)) / B, 0.7 / B


def _autograd(lat, w_mu, b_mu, log_std, eps, clip_mean, dL_da, c):
    t = lambda a: torch.tensor(a, dtype=torch.float64, requires_grad=True)  # noqa: E731
    L, W, b, S = t(lat), t(w_mu), t(b_mu), t(log_std)
    E = torch.exp(S) * torch.as_tensor(eps)
    a, lp = R.sde_head(L, W, b, S, E, clip_mean)
    (torch.sum(torch.as_tensor(dL_da) * a) + c * lp.sum()).backward()
    return L.grad.numpy(), W.grad.numpy(), b.grad.numpy(), S.grad.numpy(), E.detach().numpy()


def test_closed_form_head_gradient_is_autograds():
    """The derivation the kernels implement (d latent, d mu, d log_std through sigma AND through E) equals autograd's, Hardtanh on and off."""
    for clip in (2.0, 0.0, 0.2):
        case = _head_case(clip_mean=clip)
        gl, gw, gb, gs, E = _autograd(*case)
        lat, w_mu, b_mu, log_std, eps, clip_mean, dL_da, c = case
        cl, cw, cb, cs = R.sde_head_grads_closed_form(lat, w_mu, b_mu, log_std, E, clip_mean, dL_da, c)
        for got, want in ((cl, gl), (cw, gw), (cb, gb), (cs, gs)):
            np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-9)


def test_clamp_binding_rows_get_no_log_prob_gradient_through_g():
    """|mean + noise| beyond ~8.3: tanh rounds to +-1 in float32, the atanh clamp binds and autograd's gradient through it is zero."""
    lat, w_mu, b_mu, log_std, eps, _, dL_da, c = _head_case(scale=40.0, seed=1)
    u = np.clip(lat @ w_mu.T + b_mu, -2, 2) + lat @ (np.exp(log_std) * eps)
    assert (np.abs(u) > 8.5).mean() > 0.5
    gl, gw, gb, gs, E = _autograd(lat, w_mu, b_mu, log_std, eps, 2.0, dL_da, c)
    cl, cw, cb, cs = R.sde_head_grads_closed_form(lat, w_mu, b_mu, log_std, E, 2.0, dL_da, c)
    for got, want in ((cl, gl), (cw, gw), (cb, gb), (cs, gs)):
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-9)


class FlattenExtractor(nn.Module):
    pass


def _actor(mu=None, shape=(64, 2), **flags):
    return SimpleNamespace(mu=mu if mu is not None else nn.Sequential(nn.Linear(64, 2), nn.Hardtanh(-2.0, 2.0)),
                           log_std=nn.Parameter(torch.zeros(shape)), use_sde=True, **{"use_expln": False, "full_std": True, **flags})


def test_update_guard_names_each_refused_gsde_option():
    why = update._sde_update_unsupported
    assert why(_actor()) is None and why(_actor(mu=nn.Linear(64, 2))) is None
    assert "use_expln=True" in why(_actor(use_expln=True))
    assert "full_std=False" in why(_actor(full_std=False, shape=(64, 1)))
    assert "Linear + Hardtanh" in why(_actor(mu=nn.Sequential(nn.Linear(64, 2), nn.Tanh())))
    assert "(H2, 2) parameter" in why(_actor(shape=(32, 2)))
    assert update._sde_clip_mean(_actor()) == 2.0 and update._sde_clip_mean(_actor(mu=nn.Linear(64, 2))) == 0.0
