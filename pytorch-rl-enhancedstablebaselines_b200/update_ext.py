"""BCQ and MADDPG / IDDPG gradient steps on the device (SURVEY §8f-1) behind the reference's ``BCQ.train`` / ``MADDPG.train`` /
``IDDPG.train`` surfaces.

``FusedBCQUpdate`` runs one iteration of the loop body of ``BCQ.train`` (``core/bcq/bcq.py:137-205``) per ``update()`` through
``cstr_bcq_update``: the VAE step, the candidate target (ten latent draws through the refreshed VAE and the target perturbation net, max over
the reference's ``(B, 10)`` reshape as written), the twin critics, and the delayed perturbation step with polyak.
``FusedMultiAgentUpdate`` runs one iteration of ``MADDPG.train`` / ``IDDPG.train`` (``core/maddpg/maddpg.py:127-185``,
``core/iddpg/iddpg.py:127-185``) through ``cstr_ma_update`` for the two-reactor agents of BASELINE config #5.

Both keep five flat float32 device blocks (``params, targets, grads, adam_m, adam_v``) like :class:`FusedTD3Update`; the plumbing
(workspace, module and Adam hand-over, CUDA-graph replay, the peer-memory gradient all-reduce) is ``update._FusedEngine``'s.
``bind_bcq_class`` / ``bind_multiagent_class`` return subclasses of the reference algorithms whose ``train()`` runs here and whose policy
modules share memory with the flat blocks.
"""
from __future__ import annotations

from ctypes import byref, c_int64
from typing import Any, Dict, List, Optional, Sequence

import numpy as np

from . import _lib
from .update import _GEMM_MODES, _FusedEngine, _dist_rank, _fallback_once, _not_plain_adam, _spaces_reason


class _FlatEngine(_FusedEngine):
    """BCQ and multi-agent engines: no host-side all-reduce hook, so ``train`` runs ``update`` without one."""

    def train(self, gradient_steps: int, buffer, batch_size: Optional[int] = None, env=None, allreduce=None, graph: bool = False) -> None:
        """sample + update, ``gradient_steps`` times; ``graph=True`` (Philox-index buffer, full ring) replays whole cycles of ``actor_delay`` /
        ``policy_delay`` updates from one captured CUDA graph.  Data-parallel training: ``enable_peer_allreduce()`` (the averaging is part of the
        Adam kernels); a host-side ``allreduce=`` hook is not offered for these engines."""
        if allreduce is not None:
            raise ValueError("data-parallel BCQ / multi-agent updates average their gradients through enable_peer_allreduce()")
        bs = int(batch_size or self._batch)
        done = self._train_graph(graph, gradient_steps, buffer, bs, env, None)
        for _ in range(gradient_steps - done):
            self.update(buffer.sample(bs, env=env))


class FusedBCQUpdate(_FlatEngine):
    NETS = ("vae_enc", "vae_dec", "pert", "critic0", "critic1")
    N_LOSS = 6

    def __init__(self, latent_dim: int = 32, vae_hidden: int = 64, pert_hidden: int = 64, critic_arch: Sequence[int] = (400, 300), batch_size: int = 256,
                 device: Any = "cuda", gamma: float = 0.99, tau: float = 0.005, learning_rate: float = 1e-3, max_perturbation: float = 0.05,
                 actor_delay: int = 2, n_candidates: int = 10, betas=(0.9, 0.999), eps: float = 1e-8, seed: int = 0, gemm: str = "fp32", dp_rank: int = 0):
        super().__init__(device, gamma, tau, learning_rate, actor_delay, betas, eps, seed, gemm, dp_rank)
        self._two_hidden(critic_arch)
        self.latent, self.vae_hidden, self.pert_hidden = int(latent_dim), int(vae_hidden), int(pert_hidden)
        self.max_perturbation, self.actor_delay, self.n_candidates = float(max_perturbation), int(actor_delay), int(n_candidates)
        offs = (c_int64 * 31)()
        rc = self._libc.cstr_bcq_layout(byref(self._config(1)), offs)
        if rc:
            msg = self._libc.cstr_last_error()
            raise ValueError(msg.decode() if msg else "bad BCQ configuration")
        self._allocate(offs, batch_size)
        self.vae_range = (0, self._offsets[("pert", "W1")])
        self.pert_range = (self._offsets[("pert", "W1")], self._offsets[("critic0", "W1")])
        self.critic_range = (self._offsets[("critic0", "W1")], self.param_count)

    def _dims(self, net: str):
        L, Hv, Hp = self.latent, self.vae_hidden, self.pert_hidden
        return {"vae_enc": (6, Hv, Hv, 2 * L), "vae_dec": (4 + L, Hv, Hv, 2), "pert": (6, Hp, Hp, 2), "critic0": (6, self.h1, self.h2, 1),
                "critic1": (6, self.h1, self.h2, 1)}[net]

    def _config(self, batch: int) -> "_lib.BcqConfig":
        return _lib.BcqConfig(latent=self.latent, vae_hidden=self.vae_hidden, pert_hidden=self.pert_hidden, h1=self.h1, h2=self.h2, batch=batch,
                              actor_delay=self.actor_delay, n_candidates=self.n_candidates, gamma=self.gamma, tau=self.tau, lr=self.learning_rate,
                              beta1=self.betas[0], beta2=self.betas[1], eps=self.eps, max_perturbation=self.max_perturbation, seed=self._keyed_seed(),
                              gemm_mode=_GEMM_MODES[self.gemm])

    def _workspace_bytes(self, batch: int) -> int:
        return int(self._libc.cstr_bcq_workspace_bytes(byref(self._config(batch))))

    def nets(self) -> Dict[str, List[np.ndarray]]:
        out = super().nets()
        out.update({net + "_target": out[net] for net in ("vae_enc", "vae_dec")})  # the target VAE is a copy of the VAE (bcq.py:158-159)
        return out

    def update(self, batch, eps_vae=None, z_next=None, z_actor=None) -> None:
        """One iteration of bcq.py:137-205.  ``eps_vae`` (B, L), ``z_next`` (n_candidates*B, L), ``z_actor`` (B, L): explicit standard-normal
        draws (unclamped) for parity tests; default = Philox inside the kernels."""
        obs, act, nobs, dones, rew = self._batch_f32(batch)
        L = self.latent
        draws = [None if d is None else self._f32(d, cols) for d, cols in ((eps_vae, L), (z_next, self.n_candidates * L), (z_actor, L))]
        self.n_updates += 1
        self.critic_step += 1
        actor_now = self.n_updates % self.actor_delay == 0
        if actor_now:
            self.actor_step += 1
        cfg, st = self._config(self._batch), self._state(counters=False)
        with self._torch.cuda.device(self.device):
            rc = self._libc.cstr_bcq_update(byref(cfg), byref(st), _lib.ptr(obs), _lib.ptr(act), _lib.ptr(nobs), _lib.ptr(dones), _lib.ptr(rew),
                                            _lib.ptr(draws[0]), _lib.ptr(draws[1]), _lib.ptr(draws[2]), self.n_updates, self.critic_step,
                                            self.actor_step, self._stream())
        _lib.check(rc, "cstr_bcq_update")
        self.launches += 92 if actor_now else 66

    def _graph_launch(self, batch_size: int, st, out, k: int, allreduce=None) -> None:
        cfg = self._config(batch_size)
        rc = self._libc.cstr_bcq_update(byref(cfg), byref(st), _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]), _lib.ptr(out[3]), _lib.ptr(out[4]),
                                        None, None, None, k, 1, 1, self._stream())
        _lib.check(rc, "cstr_bcq_update (graph capture)")

    # ---- the reference's BCQPolicy (core/bcq/policies.py:263-452) ---------------------------------------------------------------
    def adopt_policy(self, policy) -> None:
        """Copy the weights of the reference's ``BCQPolicy`` in and re-point its parameters at the flat blocks.  The target VAE's parameters
        are pointed at the VAE's own storage: the reference overwrites it with the VAE after every step (bcq.py:158-159, 198)."""
        v, t, L = self.views("params"), self.views("targets"), self.latent
        enc = v["vae_enc"]

        def vae_pairs(vae):
            return (list(zip(enc[:4], vae.encoder.parameters())) + [(enc[4][0:L], vae.mean.weight), (enc[4][L:2 * L], vae.log_std.weight),
                                                                   (enc[5][0:L], vae.mean.bias), (enc[5][L:2 * L], vae.log_std.bias)]
                    + list(zip(v["vae_dec"], vae.decoder.parameters())))

        online = vae_pairs(policy.actor.vae) + list(zip(v["pert"], policy.actor.perturbation.model.parameters()))
        targets = list(zip(t["pert"], policy.actor_target.perturbation.model.parameters()))
        for z, q in enumerate(policy.critic.q_networks):
            online += zip(v[f"critic{z}"], q.parameters())
        for z, q in enumerate(policy.critic_target.q_networks):
            targets += zip(t[f"critic{z}"], q.parameters())
        self._adopt(online, targets)
        for view, p in vae_pairs(policy.actor_target.vae):  # shared storage with the VAE
            p.data = view

    def import_optimizer_state(self, vae_optimizer, perturbation_optimizer, critic_optimizer) -> None:
        vae, pert, critic = (self._import_adam(opt) for opt in (vae_optimizer, perturbation_optimizer, critic_optimizer))
        self.critic_step, self.actor_step = max(vae, critic), pert

    def export_optimizer_state(self, vae_optimizer, perturbation_optimizer, critic_optimizer) -> None:
        self._export_adam(vae_optimizer, self.critic_step)
        self._export_adam(perturbation_optimizer, self.actor_step)
        self._export_adam(critic_optimizer, self.critic_step)


def bcq_update_unsupported(model) -> Optional[str]:
    """Why ``cstr_bcq_update`` can NOT stand in for ``model.train()`` — or None when it can."""
    import torch.nn as nn

    pol = model.policy
    why = _spaces_reason(model)
    if why:
        return why
    if getattr(pol, "activation_fn", nn.ReLU) is not nn.ReLU:
        return "activation_fn is not ReLU"
    arch = pol.actor_arch
    if arch["vae_latent_dim"] % 4 or not 4 <= arch["vae_latent_dim"] <= 64 or arch["vae_hidden_dim"] % 4 or arch["perturbation_hidden_dim"] % 4:
        return f"actor_net_arch {arch}: latent must be a multiple of 4 in [4, 64], hidden sizes multiples of 4"
    c = list(pol.critic_arch)
    if len(c) != 2 or any(int(h) % 4 for h in c) or len(pol.critic.q_networks) != 2:
        return f"critic_net_arch {c} / n_critics {len(pol.critic.q_networks)}: two hidden layers (multiples of 4) and two critics"
    if type(pol.actor.features_extractor).__name__ != "FlattenExtractor":
        return f"features extractor {type(pol.actor.features_extractor).__name__}"
    opt = _not_plain_adam((pol.actor.vae_optimizer, pol.actor.perturbation_optimizer, pol.critic.optimizer))
    if opt is not None:
        return f"optimizer {type(opt).__name__} is not plain Adam"
    return None


def bind_bcq_class(bcq_base: type) -> type:
    """Subclass of the reference's ``BCQ`` whose ``train()`` (core/bcq/bcq.py:129-213) runs on ``cstr_bcq_update``; dataset loading, ``learn()``,
    evaluation, saving and ``predict`` stay the reference's code, the policy modules share memory with the flat parameter blocks."""

    class FusedBCQ(bcq_base):  # type: ignore[misc, valid-type]
        _fused: Optional[FusedBCQUpdate] = None

        def train(self, gradient_steps: int, batch_size: int = 100) -> None:
            why = bcq_update_unsupported(self) if self._fused is None else None
            if why:
                _fallback_once(self, why)
                return super().train(gradient_steps, batch_size)
            self.policy.set_training_mode(True)
            self._update_learning_rate([self.actor.perturbation_optimizer, self.actor.vae_optimizer, self.critic.optimizer])
            if self._fused is None:
                arch = self.policy.actor_arch
                eng = FusedBCQUpdate(arch["vae_latent_dim"], arch["vae_hidden_dim"], arch["perturbation_hidden_dim"], list(self.policy.critic_arch), batch_size,
                                     self.device, self.gamma, self.tau, float(self.lr_schedule(self._current_progress_remaining)),
                                     float(arch["max_perturbation"]), int(self.actor_delay), 10, seed=int(self.seed or 0), dp_rank=_dist_rank())
                eng.adopt_policy(self.policy)
                eng.import_optimizer_state(self.actor.vae_optimizer, self.actor.perturbation_optimizer, self.critic.optimizer)
                eng.n_updates = int(self._n_updates)
                self._fused = eng
            eng = self._fused
            eng.learning_rate = float(self.lr_schedule(self._current_progress_remaining))
            eng.train(gradient_steps, self.replay_buffer, batch_size, env=self._vec_normalize_env, graph=bool(getattr(self.replay_buffer, "full", False)))
            self._n_updates = eng.n_updates
            vae_loss, critic_loss, actor_loss = eng.pop_losses()
            self.logger.record("train/n_updates", self._n_updates, exclude="tensorboard")
            if actor_loss is not None:
                self.logger.record("train/actor_loss", actor_loss)
            self.logger.record("train/critic_loss", critic_loss)
            self.logger.record("train/vae_loss", vae_loss)

        def _excluded_save_params(self):
            return super()._excluded_save_params() + ["_fused"]

        def save(self, *args, **kwargs):
            if self._fused is not None:
                self._fused.export_optimizer_state(self.actor.vae_optimizer, self.actor.perturbation_optimizer, self.critic.optimizer)
            return super().save(*args, **kwargs)

    FusedBCQ.__name__ = "BCQ"
    FusedBCQ.__qualname__ = "BCQ"
    return FusedBCQ


class FusedMultiAgentUpdate(_FlatEngine):
    """MADDPG (``centralised=True``) / IDDPG (``centralised=False``) for the two-reactor agents: observation slices [0,1] and [2,3], one
    action each.  ``actor_lrs`` / ``critic_lrs``: per-agent Adam learning rates as the reference APPLIES them — its
    ``_update_learning_rate([actor_opt_i, critic_opt_i])`` pairs list entry k with ``learning_rate_list[k]`` (base_class.py:1112-1136), so
    ``reference_lrs(learning_rate_list)`` gives every actor ``learning_rate_list[0]`` and every critic ``learning_rate_list[1]``."""

    N_LOSS = 8

    @staticmethod
    def reference_lrs(learning_rate_list: Sequence[float]):
        return [float(learning_rate_list[0])] * 2, [float(learning_rate_list[1])] * 2

    def __init__(self, net_arch: Sequence[int] = (400, 300), batch_size: int = 256, centralised: bool = True, device: Any = "cuda", gamma: float = 0.99,
                 tau: float = 0.005, actor_lrs: Sequence[float] = (1e-3, 1e-3), critic_lrs: Sequence[float] = (1e-3, 1e-3), policy_delay: int = 2,
                 target_policy_noise: float = 0.2, target_noise_clip: float = 0.5, n_critics: int = 2, betas=(0.9, 0.999), eps: float = 1e-8, seed: int = 0,
                 gemm: str = "fp32", dp_rank: int = 0):
        super().__init__(device, gamma, tau, actor_lrs[0], policy_delay, betas, eps, seed, gemm, dp_rank)
        self._two_hidden(net_arch)
        self.centralised, self.n_critics = bool(centralised), int(n_critics)
        self.actor_lrs, self.critic_lrs = [float(x) for x in actor_lrs], [float(x) for x in critic_lrs]
        self.target_policy_noise, self.target_noise_clip = float(target_policy_noise), float(target_noise_clip)
        self.NETS = tuple([f"actor{i}" for i in range(2)] + [f"critic{i}_{k}" for i in range(2) for k in range(self.n_critics)])
        offs = (c_int64 * (len(self.NETS) * 6 + 1))()
        rc = self._libc.cstr_ma_layout(byref(self._config(1)), offs)
        if rc:
            msg = self._libc.cstr_last_error()
            raise ValueError(msg.decode() if msg else "bad multi-agent configuration")
        self._allocate(offs, batch_size)

    def _dims(self, net: str):
        return (2 if net.startswith("actor") else (6 if self.centralised else 3), self.h1, self.h2, 1)

    def _config(self, batch: int) -> "_lib.MaConfig":
        cfg = _lib.MaConfig(centralised=int(self.centralised), h1=self.h1, h2=self.h2, batch=batch, policy_delay=self.policy_delay, n_critics=self.n_critics,
                            gamma=self.gamma, tau=self.tau, beta1=self.betas[0], beta2=self.betas[1], eps=self.eps, target_policy_noise=self.target_policy_noise,
                            target_noise_clip=self.target_noise_clip, seed=self._keyed_seed(), gemm_mode=_GEMM_MODES[self.gemm])
        for i in range(2):
            cfg.actor_lr[i], cfg.critic_lr[i] = self.actor_lrs[i], self.critic_lrs[i]
        return cfg

    def _workspace_bytes(self, batch: int) -> int:
        return int(self._libc.cstr_ma_workspace_bytes(byref(self._config(batch))))

    def update(self, batch, noise=None) -> None:
        """One iteration of maddpg.py / iddpg.py :127-185.  ``noise``: explicit N(0, target_policy_noise) draws, (2, B) agent-major (or a
        sequence of two (B, 1) arrays), for parity tests; default = Philox in the kernel."""
        obs, act, nobs, dones, rew = self._batch_f32(batch)
        B = self._batch
        nz = None
        if noise is not None:
            torch = self._torch
            if not isinstance(noise, torch.Tensor):
                noise = np.stack([np.asarray(n, np.float32).reshape(B) for n in noise], 0)
            nz = torch.as_tensor(noise, device=self.device).to(torch.float32).reshape(2, B).contiguous()
        self.n_updates += 1
        self.critic_step += 1
        if self.n_updates % self.policy_delay == 0:
            self.actor_step += 1
        cfg, st = self._config(B), self._state(counters=False)
        with self._torch.cuda.device(self.device):
            rc = self._libc.cstr_ma_update(byref(cfg), byref(st), _lib.ptr(obs), _lib.ptr(act), _lib.ptr(nobs), _lib.ptr(dones), _lib.ptr(rew), _lib.ptr(nz),
                                           self.n_updates, self.critic_step, self.actor_step, self._stream())
        _lib.check(rc, "cstr_ma_update")
        self.launches += 100 if self.n_updates % self.policy_delay == 0 else 46

    def _graph_launch(self, batch_size: int, st, out, k: int, allreduce=None) -> None:
        cfg = self._config(batch_size)
        rc = self._libc.cstr_ma_update(byref(cfg), byref(st), _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]), _lib.ptr(out[3]), _lib.ptr(out[4]),
                                       None, k, 1, 1, self._stream())
        _lib.check(rc, "cstr_ma_update (graph capture)")

    def _make_graph_key(self, buffer, batch_size, env, allreduce):
        return super()._make_graph_key(buffer, batch_size, env, allreduce) + (tuple(self.actor_lrs), tuple(self.critic_lrs))

    def pop_losses(self):
        """((critic_loss, actor_loss) of agent 0, (critic_loss, actor_loss) of agent 1) — means since the last call."""
        c0, a0, c1, a1 = super().pop_losses()
        return (c0, a0), (c1, a1)

    # ---- the reference's MADDPGPolicy / IDDPGPolicy (core/maddpg/policies.py:281-500) -------------------------------------------------
    def adopt_policy(self, policy) -> None:
        v, t = self.views("params"), self.views("targets")
        online, targets = [], []
        for i in range(2):
            online += zip(v[f"actor{i}"], policy.actor.mu_list[i].parameters())
            targets += zip(t[f"actor{i}"], policy.actor_target.mu_list[i].parameters())
            for k in range(self.n_critics):
                online += zip(v[f"critic{i}_{k}"], policy.critic.q_networks_list[i][k].parameters())
                targets += zip(t[f"critic{i}_{k}"], policy.critic_target.q_networks_list[i][k].parameters())
        self._adopt(online, targets)

    def import_optimizer_state(self, actor_optimizers, critic_optimizers) -> None:
        self.actor_step = max([self._import_adam(opt) for opt in actor_optimizers], default=0)
        self.critic_step = max([self._import_adam(opt) for opt in critic_optimizers], default=0)

    def export_optimizer_state(self, actor_optimizers, critic_optimizers) -> None:
        for opt in actor_optimizers:
            self._export_adam(opt, self.actor_step)
        for opt in critic_optimizers:
            self._export_adam(opt, self.critic_step)


def _ma_arch(policy):
    """[h1, h2] shared by every per-agent actor (2 -> h1 -> h2 -> 1) and q-network (3|6 -> h1 -> h2 -> 1) of a reference multi-agent policy —
    read off the modules themselves (``policy.net_arch`` is a per-agent list of lists or dicts) — or None when they do not fit the kernels."""
    import torch.nn as nn

    def dims(module):
        lin = [m for m in module.modules() if isinstance(m, nn.Linear)]
        acts = [m for m in module.modules() if isinstance(m, (nn.ReLU, nn.Tanh, nn.Sigmoid, nn.ELU, nn.LeakyReLU, nn.GELU, nn.SiLU))]
        if len(lin) != 3 or sum(isinstance(a, nn.ReLU) for a in acts) != 2:
            return None
        return (lin[0].in_features, lin[0].out_features, lin[1].out_features, lin[2].out_features)

    actors = [dims(m) for m in policy.actor.mu_list]
    critics = [dims(q) for qs in policy.critic.q_networks_list for q in qs]
    if any(d is None for d in actors + critics):
        return None
    h = {(d[1], d[2]) for d in actors + critics}
    if len(h) != 1 or any(d[0] != 2 or d[3] != 1 for d in actors) or len({d[0] for d in critics}) != 1 or critics[0][0] not in (3, 6):
        return None
    h1, h2 = next(iter(h))
    if h1 % 4 or h2 % 4 or h1 < 4 or h2 < 4:
        return None
    return [int(h1), int(h2)]


def multiagent_update_unsupported(model) -> Optional[str]:
    import torch.nn as nn

    pol = model.policy
    why = _spaces_reason(model)
    if why:
        return why
    if model.n_agents != 2 or [list(s) for s in model.observation_splits] != [[0, 1], [2, 3]] or [list(s) for s in model.action_splits] != [[0], [1]]:
        return "agents are not the two reactors (observation_splits [[0,1],[2,3]], action_splits [[0],[1]])"
    if getattr(pol, "activation_fn", nn.ReLU) is not nn.ReLU:
        return "activation_fn is not ReLU"
    arch = _ma_arch(pol)
    if arch is None:
        return "actors / critics are not two-hidden-layer ReLU MLPs of one common width pair (multiples of 4) with inputs 2 and 3 or 6"
    if not 1 <= pol.critic.n_critics <= 2:
        return f"n_critics={pol.critic.n_critics}"
    opt = _not_plain_adam(list(pol.actor.optimizer_list) + list(pol.critic.optimizer_list))
    if opt is not None:
        return f"optimizer {type(opt).__name__} is not plain Adam"
    for i in range(2):
        if sum(1 for _ in pol.actor.features_extractor_list[i].parameters()):
            return "features extractors with parameters"
    return None


def bind_multiagent_class(algo_base: type) -> type:
    """Subclass of the reference's ``MADDPG`` or ``IDDPG`` whose ``train()`` (core/maddpg/maddpg.py:117-191, core/iddpg/iddpg.py:117-191) runs on
    ``cstr_ma_update``.  Which of the two it is follows from the critic's input width (6: centralised, 3: independent)."""

    class FusedMultiAgent(algo_base):  # type: ignore[misc, valid-type]
        _fused: Optional[FusedMultiAgentUpdate] = None

        def train(self, gradient_steps: int, batch_size: int) -> None:
            why = multiagent_update_unsupported(self) if self._fused is None else None
            if why:
                _fallback_once(self, why)
                return super().train(gradient_steps, batch_size)
            self.policy.set_training_mode(True)
            for agent_id in range(self.n_agents):
                self._update_learning_rate([self.actor.optimizer_list[agent_id], self.critic.optimizer_list[agent_id]])
            if self._fused is None:
                arch = _ma_arch(self.policy)
                width = int(next(self.critic.q_networks_list[0][0].parameters()).shape[1])
                eng = FusedMultiAgentUpdate(arch, batch_size, width == 6, self.device, self.gamma, self.tau, policy_delay=self.policy_delay,
                                            target_policy_noise=self.target_policy_noise, target_noise_clip=self.target_noise_clip,
                                            n_critics=self.critic.n_critics, seed=int(self.seed or 0), dp_rank=_dist_rank())
                eng.adopt_policy(self.policy)
                eng.import_optimizer_state(self.actor.optimizer_list, self.critic.optimizer_list)
                eng.n_updates = int(self._n_updates)
                self._fused = eng
            eng = self._fused
            # the rates the reference's optimisers actually hold after _update_learning_rate (its pairing quirk included)
            eng.actor_lrs = [float(o.param_groups[0]["lr"]) for o in self.actor.optimizer_list]
            eng.critic_lrs = [float(o.param_groups[0]["lr"]) for o in self.critic.optimizer_list]
            eng.train(gradient_steps, self.replay_buffer, batch_size, env=self._vec_normalize_env, graph=bool(getattr(self.replay_buffer, "full", False)))
            self._n_updates = eng.n_updates
            losses = eng.pop_losses()
            self.logger.record("train/n_updates", self._n_updates, exclude="tensorboard")
            for agent_id, (critic_loss, actor_loss) in enumerate(losses):
                if actor_loss is not None:
                    self.logger.record(f"train/agent_{agent_id}_actor_loss", actor_loss)
                self.logger.record(f"train/agent_{agent_id}_critic_loss", critic_loss)

        def _excluded_save_params(self):
            return super()._excluded_save_params() + ["_fused"]

        def save(self, *args, **kwargs):
            if self._fused is not None:
                self._fused.export_optimizer_state(self.actor.optimizer_list, self.critic.optimizer_list)
            return super().save(*args, **kwargs)

    FusedMultiAgent.__name__ = algo_base.__name__
    FusedMultiAgent.__qualname__ = algo_base.__qualname__
    return FusedMultiAgent
