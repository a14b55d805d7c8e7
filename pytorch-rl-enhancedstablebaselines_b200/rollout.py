"""Fast-mode rollout driver: K env steps per launch of the fused kernel ``cstr_rollout_fused``
(actor MLP -> noise -> bounds -> CSTR step -> reward/done -> replay record), nothing leaves the GPU.

Semantics per step = the reference's ``collect_rollouts`` body for a deterministic-actor algorithm
(TD3/DDPG): ``_sample_action`` (off_policy_algorithm.py:364-411) + ``env.step`` (:564) +
``_store_transition`` (:445-508) + ``ReplayBuffer.add`` (buffers.py:247-283), without the O(n_envs)
Python loops of SURVEY.md H1.  ``train()`` of the unchanged algorithm then samples from the buffer.
"""
from __future__ import annotations

from ctypes import byref
from typing import Optional

from . import _lib
from .buffer import GpuReplayBuffer
from .env import _MATH, GpuCSTRVecEnv
from .normalize import GpuVecNormalize

# rollout_f32_kernel keeps h1 of its 128 reactors in shared memory: 128 * max(H1, 64) floats + 128 float4 <= 227 KB
FP32_MAX_H1 = 448


def actor_shape_error(H1: int, H2: int, actor_mode: str) -> Optional[str]:
    """Why the rollout kernel of ``actor_mode`` cannot run a 4 -> H1 -> H2 actor — or None when it can."""
    if H1 <= 0 or H2 <= 0 or H1 % 4:
        return f"H1={H1}, H2={H2}: the rollout kernels need positive widths and H1 a multiple of 4"
    if actor_mode != "tc":
        return None if H1 <= FP32_MAX_H1 else f"H1={H1}: the float32 actor keeps h1 in shared memory, H1 <= {FP32_MAX_H1}"
    if H1 % 16 or H1 > 1024:
        return f"H1={H1}: the tensor-core actor needs H1 a multiple of 16 and <= 1024"
    # the size query of the W2 packer reads the shape only (W2 need not point anywhere) and returns <= 0 for a shape it rejects
    probe = _lib.ActorF32(W1=None, b1=None, W2=1, b2=None, W3=None, b3=None, H1=H1, H2=H2, kind=_lib.ACTOR_TANH)
    if _lib.load().cstr_actor_pack_bf16(byref(probe), None, None) <= 0:
        return (f"H1={H1}, H2={H2}: the tensor-core actor needs H2 rounded up to 16 plus two layer-1 K-chunks within 512 TMEM columns "
                "(H2 <= 480) and its operand buffers within 227 KB of shared memory")
    return None


class ActorWeights:
    """fp32 weights of a 4 -> H1 -> H2 -> head actor on the device, torch Linear layout (out,in).

    ``kind="tanh"``     TD3/DDPG: ``tanh(W3 relu(W2 relu(W1 x + b1) + b2) + b3)`` — the ``mu`` Sequential of the TD3
                        ``Actor`` (core/td3/policies.py:20-83); W3 is (2,H2).
    ``kind="gaussian"`` SAC: ``tanh(mu + exp(clamp(log_std,-20,2)) * eps)`` on the trunk ``latent_pi`` with heads ``mu`` and
                        ``log_std`` (core/sac/policies.py:25-178); W3 is (4,H2) = rows [mu_0, mu_1, log_std_0, log_std_1].
    ``kind="sde"``      SAC with gSDE (``use_sde=True``): ``tanh(hardtanh(W3 latent + b3, clip_mean) + latent @ E_i)`` with reactor i's
                        exploration matrix ``E_i = exp(log_std) * N(0,1)`` (StateDependentNoiseDistribution, full_std, no expln,
                        core/common/distributions.py); W3 is ``mu``'s (2,H2), ``log_std`` the (H2,2) parameter the matrices are drawn
                        from (:meth:`FusedRollout.reset_noise`), ``clip_mean <= 0`` means no Hardtanh.
    """

    def __init__(self, W1, b1, W2, b2, W3, b3, device="cuda", kind: str = "tanh", log_std=None, clip_mean: float = 0.0):
        torch = _lib.require_cuda()
        dev = torch.device(device)
        if kind not in ("tanh", "gaussian", "sde"):
            raise ValueError("kind must be 'tanh', 'gaussian' or 'sde'")
        if (log_std is not None) != (kind == "sde"):
            raise ValueError("log_std (H2, 2) is given for kind='sde' and only for it")

        def put(x):
            return torch.as_tensor(x).detach().to(device=dev, dtype=torch.float32).contiguous()

        self.W1, self.b1, self.W2, self.b2, self.W3, self.b3 = (put(x) for x in (W1, b1, W2, b2, W3, b3))
        self.H1, self.H2 = int(self.W1.shape[0]), int(self.W2.shape[0])
        self.kind = kind
        self.log_std = put(log_std) if kind == "sde" else None
        self.clip_mean = float(clip_mean) if kind == "sde" else 0.0
        n_out = 4 if kind == "gaussian" else 2
        if (tuple(self.W1.shape) != (self.H1, 4) or tuple(self.W2.shape) != (self.H2, self.H1) or tuple(self.W3.shape) != (n_out, self.H2)
                or tuple(self.b3.shape) != (n_out,)):
            raise ValueError(f"actor must be 4 -> H1 -> H2 -> {n_out}")
        if self.log_std is not None and tuple(self.log_std.shape) != (self.H2, 2):
            raise ValueError(f"log_std must be (H2, 2) = ({self.H2}, 2), got {tuple(self.log_std.shape)}")
        if self.H1 % 4:
            raise ValueError("H1 must be a multiple of 4")
        self.device = dev
        self.packed_bf16 = None
        self._struct = _lib.ActorF32(W1=self.W1.data_ptr(), b1=self.b1.data_ptr(), W2=self.W2.data_ptr(), b2=self.b2.data_ptr(),
                                     W3=self.W3.data_ptr(), b3=self.b3.data_ptr(), H1=self.H1, H2=self.H2,
                                     kind={"tanh": _lib.ACTOR_TANH, "gaussian": _lib.ACTOR_GAUSSIAN, "sde": _lib.ACTOR_SDE}[kind],
                                     clip_mean=self.clip_mean)

    @staticmethod
    def _linears(module):
        return [m for m in module.modules() if hasattr(m, "weight") and getattr(m, "weight").dim() == 2]

    @classmethod
    def from_module(cls, mu_sequential, device="cuda") -> "ActorWeights":
        """From the reference TD3 actor's ``mu`` ``nn.Sequential`` (Linear, ReLU, Linear, ReLU, Linear, Tanh)."""
        lin = cls._linears(mu_sequential)
        if len(lin) != 3:
            raise ValueError("expected three Linear layers")
        return cls(lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, lin[2].weight, lin[2].bias, device=device)

    @classmethod
    def from_sac_actor(cls, latent_pi, mu, log_std, device="cuda") -> "ActorWeights":
        """From the reference SAC ``Actor``: ``actor.latent_pi`` (Linear, ReLU, Linear, ReLU), ``actor.mu``, ``actor.log_std``.  With
        gSDE (``use_sde=True``) ``log_std`` is the (H2,2) parameter and ``mu`` a Linear or ``Sequential(Linear, Hardtanh)``: the
        result is ``kind="sde"``."""
        torch = _lib.require_cuda()
        lin = cls._linears(latent_pi)
        if len(lin) != 2:
            raise ValueError("expected a two-layer trunk")
        if isinstance(log_std, torch.Tensor):
            head = sde_mean_head(mu)
            if head is None:
                raise ValueError("the gSDE actor's mu must be a Linear or Sequential(Linear, Hardtanh(-c, c))")
            return cls(lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, head[0].weight, head[0].bias, device=device, kind="sde",
                       log_std=log_std, clip_mean=head[1])
        W3 = torch.cat([mu.weight.detach(), log_std.weight.detach()], 0)
        b3 = torch.cat([mu.bias.detach(), log_std.bias.detach()], 0)
        return cls(lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, W3, b3, device=device, kind="gaussian")

    def _targets(self):
        return (self.W1, self.b1, self.W2, self.b2, self.W3, self.b3) + ((self.log_std,) if self.kind == "sde" else ())

    def _sources(self, *modules):
        torch = _lib.require_cuda()
        if self.kind == "tanh":
            lin = self._linears(modules[0])
            return [lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, lin[2].weight, lin[2].bias]
        latent_pi, mu, log_std = modules
        lin = self._linears(latent_pi)
        if self.kind == "sde":
            head = sde_mean_head(mu)[0]
            return [lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, head.weight, head.bias, log_std]
        return [lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, torch.cat([mu.weight.detach(), log_std.weight.detach()], 0),
                torch.cat([mu.bias.detach(), log_std.bias.detach()], 0)]

    def refresh_from_module(self, *modules) -> None:
        """Copy updated parameters in place (device-to-device) after an optimiser step: ``refresh_from_module(actor.mu)``
        for TD3, ``refresh_from_module(actor.latent_pi, actor.mu, actor.log_std)`` for SAC (with gSDE ``log_std`` too; exploration
        matrices already drawn keep the std they were drawn with, as the reference's do)."""
        for dst, src in zip(self._targets(), self._sources(*modules)):
            dst.copy_(src.detach(), non_blocking=True)
        if self.packed_bf16 is not None:
            self.pack_bf16()

    def refresh_from_tensors(self, tensors) -> None:
        """Same, from six tensors ``W1, b1, W2, b2, W3, b3`` — e.g. ``FusedTD3Update.views("params")["actor"]`` (for SAC the head is
        already the stacked [mu; log_std] matrix); a ``kind="sde"`` actor takes ``log_std`` as a seventh."""
        for dst, src in zip(self._targets(), tensors):
            dst.copy_(src.detach(), non_blocking=True)
        if self.packed_bf16 is not None:
            self.pack_bf16()

    def pack_bf16(self):
        """Build the bf16 UMMA image of W2 for the tensor-core path (cstr_actor_pack_bf16)."""
        torch = _lib.require_cuda()
        why = actor_shape_error(self.H1, self.H2, "tc")
        if why:
            raise ValueError(why)
        lib = _lib.load()
        with torch.cuda.device(self.device):
            nbytes = lib.cstr_actor_pack_bf16(byref(self._struct), None, None)
            if nbytes <= 0:
                _lib.check(-1, "cstr_actor_pack_bf16")
            if self.packed_bf16 is None or self.packed_bf16.numel() != nbytes:
                self.packed_bf16 = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            rc = lib.cstr_actor_pack_bf16(byref(self._struct), self.packed_bf16.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
            if rc < 0:
                _lib.check(int(rc), "cstr_actor_pack_bf16")
        return self.packed_bf16


def sde_mean_head(mu):
    """(Linear, clip_mean) of a gSDE actor's ``mu`` — a Linear (clip_mean 0: no Hardtanh) or ``Sequential(Linear, Hardtanh(-c, c))``
    (SAC ``Actor`` with ``clip_mean = c > 0``, core/sac/policies.py) — or None for any other module."""
    import torch.nn as nn

    if type(mu) is nn.Linear:
        return mu, 0.0
    if type(mu) is nn.Sequential and len(mu) == 2 and type(mu[0]) is nn.Linear and type(mu[1]) is nn.Hardtanh:
        lo, hi = float(mu[1].min_val), float(mu[1].max_val)
        if hi > 0.0 and lo == -hi:
            return mu[0], hi
    return None


class AgentActorWeights:
    """The per-agent actors of the reference's multi-agent policies (``core/maddpg/policies.py:21-121``: ``actor.mu_list[i]`` =
    ``create_mlp(2, 1, [H1, H2]) + Tanh`` on agent i's observation slice) for the two-reactor agents (observation_splits [[0,1],[2,3]],
    action_splits [[0],[1]]), each zero-padded to the single-agent shape ``4 -> H1 -> H2 -> 2`` the rollout kernel evaluates: ``W1`` (H1,4)
    with the other agent's observation columns zero, ``W3`` (2,H2) with row i the agent's head."""

    def __init__(self, agent_modules, device="cuda"):
        torch = _lib.require_cuda()
        self.device = torch.device(device)
        if len(agent_modules) != 2:
            raise ValueError("the multi-agent rollout is specialised to the two reactors as two agents")
        self.kind = "agents"
        self.packed_bf16 = None
        self._tensors = []
        for i, module in enumerate(agent_modules):
            lin = ActorWeights._linears(module)
            if len(lin) != 3 or tuple(lin[0].weight.shape)[1] != 2 or tuple(lin[2].weight.shape)[0] != 1:
                raise ValueError("expected per-agent actors 2 -> H1 -> H2 -> 1")
            H1, H2 = int(lin[0].weight.shape[0]), int(lin[1].weight.shape[0])
            z = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=self.device)  # noqa: E731
            self._tensors.append(dict(W1=z(H1, 4), b1=z(H1), W2=z(H2, H1), b2=z(H2), W3=z(2, H2), b3=z(2)))
            self.H1, self.H2 = H1, H2
        if self.H1 % 4:
            raise ValueError("H1 must be a multiple of 4")
        self._structs = (_lib.ActorF32 * 2)()
        for i, t in enumerate(self._tensors):
            self._structs[i] = _lib.ActorF32(W1=t["W1"].data_ptr(), b1=t["b1"].data_ptr(), W2=t["W2"].data_ptr(), b2=t["b2"].data_ptr(), W3=t["W3"].data_ptr(),
                                             b3=t["b3"].data_ptr(), H1=self.H1, H2=self.H2, kind=_lib.ACTOR_TANH)
        self.refresh_from_modules(agent_modules)

    def refresh_from_modules(self, agent_modules) -> None:
        """Copy the agents' current parameters into the padded images (device to device)."""
        for i, (module, t) in enumerate(zip(agent_modules, self._tensors)):
            lin = ActorWeights._linears(module)
            t["W1"][:, 2 * i:2 * i + 2].copy_(lin[0].weight.detach(), non_blocking=True)
            t["b1"].copy_(lin[0].bias.detach(), non_blocking=True)
            t["W2"].copy_(lin[1].weight.detach(), non_blocking=True)
            t["b2"].copy_(lin[1].bias.detach(), non_blocking=True)
            t["W3"][i].copy_(lin[2].weight.detach()[0], non_blocking=True)
            t["b3"][i:i + 1].copy_(lin[2].bias.detach(), non_blocking=True)


class EpisodeStats:
    """Device-side ``Monitor`` for the fused rollout (monitor.py:85-111): running return per reactor and a compact list of
    finished episodes ``(return, length)`` that ``pop()`` hands to the host — the feed of ``ep_info_buffer`` /
    ``rollout/ep_rew_mean`` (base_class.py:462-481, off_policy_algorithm.py:413-435) without any per-env Python."""

    def __init__(self, num_envs: int, device="cuda", capacity: int = 1 << 20):
        torch = _lib.require_cuda()
        self.device = torch.device(device)
        self.capacity = int(capacity)
        self.ep_return = torch.zeros(num_envs, dtype=torch.float64, device=self.device)
        self.finished = torch.zeros((self.capacity, 2), dtype=torch.float32, device=self.device)
        self.count = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.dropped = 0
        self._struct = _lib.EpisodeStatsStruct(ep_return=self.ep_return.data_ptr(), finished=self.finished.data_ptr(),
                                               count=self.count.data_ptr(), capacity=self.capacity, reserved=0)

    def pop(self):
        """(k,2) float32 NumPy array of the episodes finished since the last call: columns return, length."""
        k = int(self.count.item())
        kept = min(k, self.capacity)
        self.dropped += k - kept
        out = self.finished[:kept].cpu().numpy().copy()
        self.count.zero_()
        return out


class FusedRollout:
    """Collects transitions from ``env`` straight into ``buffer`` with the fused kernel.

    :param actor_mode: ``"fp32"`` (CUDA-core parity path) or ``"tc"`` (bf16 tcgen05 hidden layer).
    :param sigma: std of the Gaussian exploration noise (``NormalActionNoise``, noise.py:29-48); ignored for
        ``kind="gaussian"`` actors, whose only randomness is their own eps ~ N(0,1).
    :param vec_normalize: a :class:`GpuVecNormalize` wrapping ``env``: the actor then reads normalised observations and every step advances
        the wrapper's statistics and returns on the device (``cstr_rollout_fused_norm``, one kernel launch per step); the buffer keeps the
        original observations, as the reference's ``_store_transition`` does.

    A ``kind="sde"`` (gSDE) actor runs on ``actor_mode="fp32"`` without ``vec_normalize``.  Its per-reactor exploration matrices live in
    :attr:`explore`, ``(num_envs, H2, 2)`` float32 — 2 GiB at 1,048,576 reactors and H2 = 256, the same object the reference keeps as
    ``exploration_matrices`` — and stay fixed until the next :meth:`reset_noise`.
    """

    def __init__(self, env: GpuCSTRVecEnv, buffer: GpuReplayBuffer, actor: Optional[ActorWeights] = None, sigma: float = 0.1,
                 actor_mode: str = "fp32", vec_normalize: Optional[GpuVecNormalize] = None):
        if env.dtype != "fp32":
            raise ValueError("the fused rollout is fp32 (the actor and the replay records are float32)")
        if env.reset_rng != "philox":
            raise ValueError("the fused rollout needs reset_rng='philox'")
        if buffer.n_envs != env.num_envs:
            raise ValueError("buffer.n_envs must equal env.num_envs")
        if buffer.device != env.device:
            raise ValueError("env and buffer must live on the same device")
        if actor_mode not in ("fp32", "tc"):
            raise ValueError("actor_mode must be 'fp32' or 'tc'")
        self.env, self.buffer, self.actor, self.sigma = env, buffer, actor, float(sigma)
        if isinstance(actor, AgentActorWeights) and actor_mode != "fp32":
            raise ValueError("the multi-agent rollout runs the float32 actor (actor_mode='fp32')")
        why = actor_shape_error(actor.H1, actor.H2, actor_mode) if actor is not None else None
        if why:
            raise ValueError(why)
        self.actor_mode = actor_mode
        self.t = 0  # global step counter: the Philox counter of the noise / warm-up action streams
        self._lib = _lib.load()
        self.launches = 0
        self.vec_normalize = vec_normalize
        if vec_normalize is not None:
            if vec_normalize.venv is not env:
                raise ValueError("vec_normalize must wrap env")
            if isinstance(actor, AgentActorWeights):
                raise ValueError("the two-agent rollout has no VecNormalize variant")
            nbytes = self._lib.cstr_rollout_norm_workspace_bytes(env.num_envs, int(actor_mode == "tc"))
            if nbytes < 0:
                _lib.check(int(nbytes), "cstr_rollout_norm_workspace_bytes")
            self._norm_workspace = env._torch.zeros(nbytes, dtype=env._torch.uint8, device=env.device)  # zeroed once; calls leave it zeroed
        if getattr(actor, "kind", None) == "sde" and (actor_mode != "fp32" or vec_normalize is not None):
            raise ValueError("the gSDE actor runs on the float32 kernel (actor_mode='fp32') without vec_normalize")
        self.explore = None  # gSDE: (num_envs, H2, 2), allocated by the first reset_noise()
        self.sde_epoch = 0   # gSDE: Philox counter of the next reset_noise()
        if actor_mode == "tc" and actor is not None and actor.packed_bf16 is None:
            actor.pack_bf16()

    def reset_noise(self) -> None:
        """gSDE: draw every reactor's exploration matrix ``explore[i] = exp(log_std) * N(0,1)`` from the actor's current ``log_std``
        (``cstr_sde_sample``) and advance :attr:`sde_epoch` — the reference's ``actor.reset_noise(n_envs)``.  Row i depends on the env's
        seed, the reactor's global id and the epoch only, so a sharded run draws the rows a single-GPU run would."""
        env, actor = self.env, self.actor
        if getattr(actor, "kind", None) != "sde":
            raise ValueError("reset_noise draws the exploration matrices of a kind='sde' actor")
        torch = env._torch
        if self.explore is None:
            self.explore = torch.zeros((env.num_envs, actor.H2, 2), dtype=torch.float32, device=env.device)
        with torch.cuda.device(env.device):
            rc = self._lib.cstr_sde_sample(actor.log_std.data_ptr(), actor.H2, env.num_envs, env._params.env_offset, env._params.seed,
                                           self.sde_epoch & 0xFFFFFFFF, self.explore.data_ptr(), env._stream())
        _lib.check(rc, "cstr_sde_sample")
        self.sde_epoch += 1

    def collect(self, K: int, warmup: bool = False, noise=None, reward_sum=None, stats: Optional[EpisodeStats] = None) -> None:
        """K env steps for every reactor; K ring rows are appended to the buffer.

        :param warmup: uniform random actions instead of the actor (``learning_starts`` phase).
        :param noise: optional device tensor (K,N,2) float32 added instead of Philox noise (parity tests).
        :param reward_sum: optional device float64[1] accumulating the sum of rewards.
        :param stats: optional :class:`EpisodeStats` (device-side Monitor).
        """
        env, buf = self.env, self.buffer
        torch = env._torch
        if env._needs_reset:
            raise ValueError("Please call env.reset() to reset the env first!")
        if not warmup and self.actor is None:
            raise ValueError("an ActorWeights is required unless warmup=True")
        if noise is not None and (tuple(noise.shape) != (K, env.num_envs, 2) or noise.dtype != torch.float32 or not noise.is_contiguous()):
            raise ValueError("noise must be a contiguous float32 tensor of shape (K, N, 2)")
        if isinstance(self.actor, AgentActorWeights):  # the two reactors as two agents (cstr_rollout_fused_multi): no noise, no rescale (Q5)
            if noise is not None:
                raise ValueError("the reference's multi-agent _sample_action never adds noise (quirk Q5)")
            with torch.cuda.device(env.device):
                rc = self._lib.cstr_rollout_fused_multi(
                    byref(env._params), env.num_envs, K, _MATH[env.math], self.actor._structs, int(warmup), self.t & 0xFFFFFFFF, _lib.ptr(env.state),
                    _lib.ptr(env.step_count), _lib.ptr(env.episode), env._sb_ptr(), buf.buffer_size, buf.pos, _lib.ptr(buf.records),
                    _lib.ptr(reward_sum), byref(stats._struct) if stats is not None else None, env._stream())
            _lib.check(rc, "cstr_rollout_fused_multi")
            self.launches += 1
            self.t += K
            buf.advance(K)
            return
        if getattr(self.actor, "kind", None) == "sde" and not warmup:
            if self.explore is None:
                raise ValueError("call reset_noise() before the gSDE actor's first collect")
            self.actor._struct.explore = self.explore.data_ptr()
        packed = None
        if self.actor_mode == "tc" and not warmup:
            packed = self.actor.packed_bf16 if self.actor.packed_bf16 is not None else self.actor.pack_bf16()
        if self.vec_normalize is not None:
            self._collect_norm(K, warmup, noise, reward_sum, stats, packed)
            return
        with torch.cuda.device(env.device):
            rc = self._lib.cstr_rollout_fused(
                byref(env._params), env.num_envs, K, _MATH[env.math], int(self.actor_mode == "tc"),
                byref(self.actor._struct) if self.actor is not None else None, _lib.ptr(packed), self.sigma, _lib.ptr(noise), int(warmup),
                self.t & 0xFFFFFFFF, _lib.ptr(env.state), _lib.ptr(env.step_count), _lib.ptr(env.episode), env._sb_ptr(),
                buf.buffer_size, buf.pos, _lib.ptr(buf.records), _lib.ptr(reward_sum), byref(stats._struct) if stats is not None else None,
                env._stream())
        _lib.check(rc, "cstr_rollout_fused")
        self.launches += 1
        self.t += K
        buf.advance(K)

    def _collect_norm(self, K, warmup, noise, reward_sum, stats, packed) -> None:
        env, buf, vn = self.env, self.buffer, self.vec_normalize
        norm = _lib.RolloutNorm(stats=vn.stats.data_ptr(), returns=vn.returns_device.data_ptr(), workspace=self._norm_workspace.data_ptr(),
                                gamma=vn.gamma, epsilon=vn.epsilon, clip_obs=vn.clip_obs, training=int(vn.training), norm_obs=int(vn.norm_obs))
        with env._torch.cuda.device(env.device):
            rc = self._lib.cstr_rollout_fused_norm(
                byref(env._params), env.num_envs, K, _MATH[env.math], int(self.actor_mode == "tc"),
                byref(self.actor._struct) if self.actor is not None else None, _lib.ptr(packed), self.sigma, _lib.ptr(noise), int(warmup),
                self.t & 0xFFFFFFFF, _lib.ptr(env.state), _lib.ptr(env.step_count), _lib.ptr(env.episode), env._sb_ptr(),
                buf.buffer_size, buf.pos, _lib.ptr(buf.records), _lib.ptr(reward_sum), byref(stats._struct) if stats is not None else None,
                byref(norm), env._stream())
        _lib.check(rc, "cstr_rollout_fused_norm")
        self.launches += K + int(K > 0 and vn.training and vn.norm_obs)  # one launch per step, then the done rows' fix-up
        self.t += K
        buf.advance(K)


# ---------------------------------------------------------------------------------------------------------------------
# the fused rollout behind the reference's own learn()
# ---------------------------------------------------------------------------------------------------------------------
def _noise_sigma(action_noise):
    """sigma of a zero-mean ``NormalActionNoise`` (noise.py:29-48), possibly wrapped in ``VectorizedActionNoise``; None if the noise is
    something the kernel does not draw (Ornstein-Uhlenbeck, non-zero mean, per-dimension sigmas)."""
    import numpy as np

    if action_noise is None:
        return 0.0
    base = getattr(action_noise, "base_noise", action_noise)
    if type(base).__name__ != "NormalActionNoise":
        return None
    mu, sigma = np.asarray(base._mu, np.float64).ravel(), np.asarray(base._sigma, np.float64).ravel()
    if np.any(mu != 0.0) or np.any(sigma != sigma[0]):
        return None
    return float(sigma[0])


def _leaf_types(module):
    return [type(m) for m in module.modules() if not any(True for _ in m.children())]


def _actor_unsupported(actor, actor_mode: str) -> Optional[str]:
    """Why the rollout kernels cannot evaluate this actor (the kernels are ReLU, ReLU, then a tanh, squashed-Gaussian or gSDE head on a
    flat 4-value observation) — or None when they can."""
    import torch
    import torch.nn as nn

    relu_trunk = [nn.Linear, nn.ReLU, nn.Linear, nn.ReLU]
    if hasattr(actor, "mu_list"):  # MADDPG / IDDPG: per-agent 2 -> H1 -> H2 -> 1, run by the float32 kernel
        shapes = set()
        for i, mu in enumerate(actor.mu_list):
            if _leaf_types(mu) != relu_trunk + [nn.Linear, nn.Tanh]:
                return f"agent {i}'s actor is not Linear, ReLU, Linear, ReLU, Linear, Tanh: {[t.__name__ for t in _leaf_types(mu)]}"
            lin = [m for m in mu.modules() if type(m) is nn.Linear]
            if lin[0].in_features != 2 or lin[2].out_features != 1:
                return f"agent {i}'s actor is {lin[0].in_features} -> {lin[2].out_features}, not 2 -> 1"
            shapes.add((lin[0].out_features, lin[1].out_features))
        if len(shapes) != 1:
            return f"the agents' hidden widths differ: {sorted(shapes)}"
        return actor_shape_error(*shapes.pop(), "fp32")
    if type(getattr(actor, "features_extractor", None)).__name__ != "FlattenExtractor":
        return f"features extractor {type(getattr(actor, 'features_extractor', None)).__name__} (the kernels read the raw observation)"
    if hasattr(actor, "latent_pi") and getattr(actor, "use_sde", False):  # SAC with gSDE
        if _leaf_types(actor.latent_pi) != relu_trunk:
            return f"actor.latent_pi is not Linear, ReLU, Linear, ReLU: {[t.__name__ for t in _leaf_types(actor.latent_pi)]}"
        head = sde_mean_head(getattr(actor, "mu", None))
        if head is None:
            return f"use_sde with an actor.mu that is not Linear or Linear + Hardtanh(-c, c): {[t.__name__ for t in _leaf_types(actor.mu)]}"
        lin = [m for m in actor.latent_pi.modules() if type(m) is nn.Linear] + [head[0]]
        outs = (head[0].out_features,)
        log_std = getattr(actor, "log_std", None)
        if not isinstance(log_std, torch.Tensor) or tuple(log_std.shape) != (head[0].in_features, 2):
            return "use_sde with an actor.log_std that is not an (H2, 2) parameter"
    elif hasattr(actor, "latent_pi"):  # SAC
        if _leaf_types(actor.latent_pi) != relu_trunk:
            return f"actor.latent_pi is not Linear, ReLU, Linear, ReLU: {[t.__name__ for t in _leaf_types(actor.latent_pi)]}"
        if type(getattr(actor, "mu", None)) is not nn.Linear or type(getattr(actor, "log_std", None)) is not nn.Linear:
            return "actor.mu / actor.log_std are not single Linear layers"
        lin = [m for m in actor.latent_pi.modules() if type(m) is nn.Linear] + [actor.mu, actor.log_std]
        outs = (actor.mu.out_features, actor.log_std.out_features)
    else:  # TD3 / DDPG
        if _leaf_types(actor.mu) != relu_trunk + [nn.Linear, nn.Tanh]:
            return f"actor.mu is not Linear, ReLU, Linear, ReLU, Linear, Tanh: {[t.__name__ for t in _leaf_types(actor.mu)]}"
        lin = [m for m in actor.mu.modules() if type(m) is nn.Linear]
        outs = (lin[2].out_features,)
    H1, H2 = lin[0].out_features, lin[1].out_features
    if lin[0].in_features != 4 or any(o != 2 for o in outs) or lin[1].in_features != H1 or any(m.in_features != H2 for m in lin[2:]):
        return f"actor is {lin[0].in_features} -> {H1} -> {H2} -> {outs}, not 4 -> H1 -> H2 -> 2"
    return actor_shape_error(H1, H2, actor_mode)


def _sde_unsupported(actor, actor_mode: str, normalized: bool) -> Optional[str]:
    """Why the gSDE options of this model are not the ones the SDE kernel implements (StateDependentNoiseDistribution with
    full_std=True, use_expln=False, on the float32 actor without VecNormalize) — or None."""
    dist = getattr(actor, "action_dist", None)
    if getattr(actor, "use_expln", getattr(dist, "use_expln", False)):
        return "use_sde with use_expln=True (the kernel's std is exp(log_std))"
    if not getattr(actor, "full_std", getattr(dist, "full_std", True)):
        return "use_sde with full_std=False (the kernel draws one std per latent unit and action)"
    if actor_mode == "tc":
        return "use_sde with actor_mode='tc' (the gSDE actor runs on the float32 kernel)"
    if normalized:
        return "use_sde under GpuVecNormalize (the VecNormalize rollout has no gSDE actor)"
    return None


def fused_rollout_unsupported(model, env, replay_buffer, train_freq, action_noise, actor_mode: str = "fp32") -> Optional[str]:
    """Why ``cstr_rollout_fused`` can NOT stand in for this ``collect_rollouts`` call — or None when it can.  ``actor_mode`` is the
    kernel that would run the actor (``"fp32"`` or ``"tc"``; the two-agent actors always run on ``"fp32"``).  ``env`` may be a
    :class:`GpuVecNormalize` around the env when it is the model's own ``_vec_normalize_env``."""
    vec_normalize = getattr(model, "_vec_normalize_env", None)
    if getattr(model, "use_sde", False):
        why = _sde_unsupported(getattr(model, "actor", None), actor_mode, isinstance(env, GpuVecNormalize))
        if why:
            return why
    if isinstance(env, GpuVecNormalize):
        if vec_normalize is not env:
            return "the GpuVecNormalize the rollout steps through is not the model's _vec_normalize_env"
        actor = getattr(model, "actor", None)
        if actor is not None and hasattr(actor, "mu_list"):
            return "two agents under VecNormalize (the reference's multi-agent store path is not covered by the fused rollout)"
        env = env.venv
    elif vec_normalize is not None:
        return "VecNormalize wraps the env (the reference's host VecNormalize steps through the NumPy protocol; use GpuVecNormalize)"
    if not isinstance(env, GpuCSTRVecEnv):
        return f"env is a {type(env).__name__}, not a GpuCSTRVecEnv (wrappers step through the NumPy protocol)"
    if env.dtype != "fp32" or env.reset_rng != "philox":
        return "the fused rollout needs GpuCSTRVecEnv(dtype='fp32', reset_rng='philox')"
    if not isinstance(replay_buffer, GpuReplayBuffer) or replay_buffer.n_envs != env.num_envs or replay_buffer.device != env.device:
        return "replay buffer is not a GpuReplayBuffer on the env's device with n_envs == env.num_envs"
    if getattr(train_freq.unit, "value", train_freq.unit) != "step":
        return "train_freq counts episodes (one kernel launch collects a fixed number of steps)"
    actor = getattr(model, "actor", None)
    if actor is not None and hasattr(actor, "mu_list"):  # multi-agent (MADDPG / IDDPG): any noise object is ignored by the reference itself (Q5)
        splits = ([list(s) for s in getattr(model, "observation_splits", [])], [list(s) for s in getattr(model, "action_splits", [])])
        if len(actor.mu_list) != 2 or splits != ([[0, 1], [2, 3]], [[0], [1]]):
            return "agents are not the two reactors (observation_splits [[0,1],[2,3]], action_splits [[0],[1]])"
        return _actor_unsupported(actor, "fp32")
    if _noise_sigma(action_noise) is None:
        return f"action noise {action_noise!r} is not a zero-mean NormalActionNoise with one sigma"
    if actor is None or not (hasattr(actor, "mu") and (hasattr(actor.mu, "__len__") or hasattr(actor, "latent_pi"))):
        return "the policy has no TD3/DDPG `actor.mu` Sequential or SAC `actor.latent_pi/mu/log_std`"
    return _actor_unsupported(actor, actor_mode)


def launch_plan(K: int, n_envs: int, num_timesteps: int, learning_starts: int, sde_sample_freq: Optional[int] = None,
                use_sde_at_warmup: bool = False):
    """The kernel launches of one fused ``collect_rollouts`` call of ``K`` steps: a list of ``(steps, warmup, noise_resets)``.

    A launch ends where the reference changes what ``_sample_action`` does (off_policy_algorithm.py:364-411, collect_rollouts :510-605):
    at ``learning_starts`` (tested before every step) and, under gSDE (``sde_sample_freq`` not None), before every within-call step that
    is a multiple of ``sde_sample_freq > 0``.  ``noise_resets`` counts the reference's ``actor.reset_noise`` calls before the launch: one
    at the start of the call and one at every such multiple, step 0 included.  ``use_sde_at_warmup`` runs the actor during warm-up."""
    plan, s, t = [], 0, num_timesteps
    while s < K:
        warm = t < learning_starts and not use_sde_at_warmup
        k = min(K - s, -(-(learning_starts - t) // n_envs)) if warm else K - s
        resets = 0
        if sde_sample_freq is not None:
            resets = int(s == 0)
            if sde_sample_freq > 0:
                resets += int(s % sde_sample_freq == 0)
                k = min(k, sde_sample_freq - s % sde_sample_freq)
        plan.append((k, warm, resets))
        s += k
        t += n_envs * k
    return plan


def bind_offpolicy_rollout(algo_base: type, actor_mode: str = "fp32") -> type:
    """Return a subclass of a reference off-policy algorithm (``core.TD3 / DDPG / SAC``, or what ``bind_td3_class`` / ``bind_sac_class``
    returned) whose ``collect_rollouts`` (core/common/off_policy_algorithm.py:510-605) is ONE ``cstr_rollout_fused`` launch per call:
    ``train_freq.frequency`` steps of ``_sample_action`` (:364-411) + ``env.step`` (:564) + ``_store_transition`` (:445-508) +
    ``ReplayBuffer.add`` for every reactor, with the bookkeeping the rest of ``learn()`` (:309-355) relies on kept intact:

    * ``num_timesteps += n_envs`` per step, the warm-up switch at ``learning_starts`` (a launch that straddles it is split there),
    * gSDE (``use_sde=True``): ``reset_noise`` at the start of every call and, with ``sde_sample_freq > 0``, before every within-call
      step that is a multiple of it (launches are split there, see :func:`launch_plan`); ``use_sde_at_warmup`` runs the actor during
      warm-up;
      ``_update_current_progress_remaining``, ``_on_step``;
    * finished episodes come from the device-side Monitor (:class:`EpisodeStats`) into ``ep_info_buffer`` (``rollout/ep_rew_mean`` /
      ``ep_len_mean``), ``_episode_num`` advances by their number, ``_dump_logs`` runs when it crosses a multiple of ``log_interval``;
    * callbacks: ``on_rollout_start`` / ``on_step`` / ``on_rollout_end`` once per launch (``on_step`` sees ``num_timesteps`` advanced by
      the whole launch); a False from ``on_step`` stops training as in the reference.

    Under a :class:`GpuVecNormalize` (``bind_vec_normalize_class``) the launches are ``cstr_rollout_fused_norm``: normalised actor input,
    the wrapper's statistics and returns advanced every step, original observations stored; when ``learn()`` returns, ``_last_obs``
    (normalised), ``_last_original_obs`` and the wrapper's ``old_obs`` / ``old_reward`` hold what the reference loop leaves there.

    Nothing per-env runs in Python and nothing leaves the device except the finished-episode list.  Models the kernel does not cover
    (see :func:`fused_rollout_unsupported`) keep the reference's own ``collect_rollouts`` with a one-time warning.
    ``actor_mode``: ``"fp32"`` (exact float32 actor) or ``"tc"`` (bf16 tcgen05 hidden layer)."""
    if actor_mode not in ("fp32", "tc"):
        raise ValueError("actor_mode must be 'fp32' or 'tc'")
    import importlib
    import time
    import warnings

    RolloutReturn = None
    for klass in algo_base.__mro__:  # the reference package the algorithm comes from ("core", or upstream "stable_baselines3")
        if klass.__name__ in ("OffPolicyAlgorithm", "OffMultiAgentPolicyAlgorithm"):
            RolloutReturn = importlib.import_module(klass.__module__.split(".")[0] + ".common.type_aliases").RolloutReturn
            break
    if RolloutReturn is None:
        raise TypeError(f"{algo_base.__name__} is not an off-policy algorithm of the reference (no OffPolicyAlgorithm base)")

    class FusedRolloutAlgorithm(algo_base):  # type: ignore[misc, valid-type]
        _fused_roll: Optional[FusedRollout] = None
        _fused_stats: Optional[EpisodeStats] = None
        _fused_rollout_warned = False
        fused_rollout_launches = 0

        # _setup_learn wraps the noise in VectorizedActionNoise = one deepcopy per env (off_policy_algorithm.py:293-299): skip it when the
        # kernel draws the noise itself
        def _setup_learn(self, *args, **kwargs):
            noise = self.action_noise
            if (noise is not None and isinstance(self.env, (GpuCSTRVecEnv, GpuVecNormalize)) and _noise_sigma(noise) is not None
                    and self.env.num_envs > 1):
                self.action_noise = None
            try:
                return super()._setup_learn(*args, **kwargs)
            finally:
                self.action_noise = noise

        def _fused_actor_modules(self):
            a = self.actor
            if hasattr(a, "mu_list"):  # MADDPG / IDDPG: one actor per agent
                return "agents", (list(a.mu_list),)
            if hasattr(a, "latent_pi"):  # SAC
                return "gaussian", (a.latent_pi, a.mu, a.log_std)
            return "tanh", (a.mu,)

        def _fused_rollout_engine(self, env, replay_buffer, sigma: float) -> FusedRollout:
            kind, modules = self._fused_actor_modules()
            roll = self._fused_roll
            vec_normalize = env if isinstance(env, GpuVecNormalize) else None
            env = env.venv if vec_normalize is not None else env
            if roll is None or roll.env is not env or roll.buffer is not replay_buffer or roll.vec_normalize is not vec_normalize:
                actor = (AgentActorWeights(modules[0], device=env.device) if kind == "agents"
                         else ActorWeights.from_sac_actor(*modules, device=env.device) if kind == "gaussian"
                         else ActorWeights.from_module(modules[0], device=env.device))
                roll = FusedRollout(env, replay_buffer, actor, sigma=sigma, actor_mode="fp32" if kind == "agents" else actor_mode,
                                    vec_normalize=vec_normalize)
                roll.t = int(self.num_timesteps // max(env.num_envs, 1))
                self._fused_roll, self._fused_stats = roll, EpisodeStats(env.num_envs, device=env.device)
            roll.sigma = sigma
            return roll

        def collect_rollouts(self, env, callback, train_freq, replay_buffer, action_noise=None, learning_starts: int = 0, log_interval=None):
            noise = action_noise if action_noise is not None else self.action_noise
            why = fused_rollout_unsupported(self, env, replay_buffer, train_freq, noise, actor_mode=actor_mode)
            if why:
                if not self._fused_rollout_warned:
                    warnings.warn(f"fused rollout not used, the reference's collect_rollouts runs instead: {why}", RuntimeWarning, stacklevel=2)
                    self._fused_rollout_warned = True
                return super().collect_rollouts(env, callback, train_freq, replay_buffer, action_noise, learning_starts, log_interval)
            self.policy.set_training_mode(False)
            n_envs, K = env.num_envs, int(train_freq.frequency)
            roll = self._fused_rollout_engine(env, replay_buffer, _noise_sigma(noise) or 0.0)
            stats = self._fused_stats
            sde = bool(getattr(self, "use_sde", False))
            plan = launch_plan(K, n_envs, self.num_timesteps, learning_starts, int(getattr(self, "sde_sample_freq", -1)) if sde else None,
                               sde and bool(getattr(self, "use_sde_at_warmup", False)))
            callback.on_rollout_start()
            for k, warm, resets in plan:
                if not warm or resets:  # the optimiser moved the weights since the last launch: refresh the kernel's copy (device to device)
                    if isinstance(roll.actor, AgentActorWeights):
                        roll.actor.refresh_from_modules(self._fused_actor_modules()[1][0])
                    else:
                        roll.actor.refresh_from_module(*self._fused_actor_modules()[1])
                if resets:  # the first of two draws at the start of a call is never used: only its epoch is spent
                    roll.sde_epoch += resets - 1
                    roll.reset_noise()
                roll.collect(k, warmup=warm, stats=stats)
                self.fused_rollout_launches += 1
                self.num_timesteps += n_envs * k
            num_collected_steps = K
            callback.update_locals(locals())
            if not callback.on_step():
                return RolloutReturn(K * n_envs, 0, continue_training=False)
            finished = stats.pop()  # (k, 2): return, length of the episodes that ended in this launch
            num_collected_episodes = int(finished.shape[0])
            if num_collected_episodes:
                t = round(time.time() - getattr(self, "_fused_t0", time.time()), 6)
                keep = finished[-self.ep_info_buffer.maxlen:] if self.ep_info_buffer.maxlen else finished
                self.ep_info_buffer.extend({"r": float(r), "l": int(l), "t": t} for r, l in keep)
                before = self._episode_num
                self._episode_num += num_collected_episodes
                if log_interval is not None and before // log_interval != self._episode_num // log_interval:
                    self._dump_logs()
            self._update_current_progress_remaining(self.num_timesteps, self._total_timesteps)
            self._on_step()
            callback.on_rollout_end()
            return RolloutReturn(K * n_envs, num_collected_episodes, True)

        def learn(self, *args, **kwargs):
            self._fused_t0 = time.time()
            out = super().learn(*args, **kwargs)
            roll = self._fused_roll
            if roll is not None:  # `_last_obs` is the host copy the reference's own paths (predict, save) expect
                raw = roll.env.state.cpu().numpy()
                vn = roll.vec_normalize
                if vn is None:
                    self._last_obs = raw
                else:  # what the reference's last step_wait + collect_rollouts leave (vec_normalize.py:183-186, off_policy_algorithm.py:497-503)
                    buf = roll.buffer
                    vn.old_obs, vn.old_reward = raw, buf.records[(buf.pos - 1) % buf.buffer_size, :, 10].cpu().numpy()
                    self._last_original_obs, self._last_obs = raw, vn.normalize_obs(raw)
            return out

        def _excluded_save_params(self):
            return super()._excluded_save_params() + ["_fused_roll", "_fused_stats"]

    FusedRolloutAlgorithm.__name__ = algo_base.__name__
    FusedRolloutAlgorithm.__qualname__ = algo_base.__qualname__
    return FusedRolloutAlgorithm
