"""TD3 gradient steps on the device (SURVEY §8f-1) behind the reference's ``TD3.train`` surface.

``FusedTD3Update`` owns five flat float32 device blocks (``params, targets, grads, adam_m, adam_v``, layout from
``cstr_td3_layout``) and runs one iteration of the loop body of ``TD3.train`` (``core/td3/td3.py:162-206``) per
``update()`` call through ``cstr_td3_update`` — target smoothing, twin-min target, critic forward/MSE/backward, Adam,
delayed actor update, polyak — as hand-written float32 CUDA kernels.  No torch autograd, no cuBLAS.

``gemm="fp32"`` (default) keeps the reference's float32 FMA arithmetic; ``gemm="tensor"`` runs the three hidden-layer GEMM roles on
tcgen05 with every fp32 operand split into three bf16 planes (fp32-grade accuracy, see csrc/cstr_td3_tc.cuh); ``gemm="bf16"`` uses plain bf16
operands with fp32 accumulation (reduced precision, throughput mode; no per-step parity bar).

``adopt_policy`` re-points the parameters of the reference's ``TD3Policy`` modules at views of the flat blocks, so
``policy.predict``, ``model.save`` and the fused rollout keep seeing the live weights without copies.
``bind_td3_class(TD3)`` returns a subclass of the reference algorithm whose ``train()`` runs here.

Every engine (:class:`FusedTD3Update`, :class:`FusedSACUpdate` and the BCQ / multi-agent engines of ``update_ext``) is built on
:class:`_FusedEngine`, which owns that flat-block plumbing.
"""
from __future__ import annotations

import ctypes
from ctypes import byref, c_int64
from typing import Any, Callable, Dict, List, Optional, Sequence

import numpy as np

from . import _lib

NET_NAMES = ("actor", "critic0", "critic1")
_GEMM_MODES = {"fp32": 0, "tensor": 1, "bf16": 2}
_TENSORS = ("W1", "b1", "W2", "b2", "W3", "b3")


class _FusedEngine:
    """What every fused update engine shares: five flat float32 device blocks (``params, targets, grads, adam_m, adam_v``) in the layout
    the library reports, the workspace, the hand-over of torch modules and Adam state, CUDA-graph replay and the peer-memory gradient
    all-reduce.  An engine names its three-layer nets (``NETS``, ``_dims``) and the nets with a target block of their own
    (``TARGET_NETS``); its constructor calls this one, sets its own fields, then hands the library's layout to ``_allocate``."""

    NETS: Sequence[str] = ()
    TARGET_NETS: Optional[Sequence[str]] = None  # None: every net of NETS
    N_LOSS = 4

    def __init__(self, device, gamma: float, tau: float, learning_rate: float, policy_delay: int, betas, eps: float, seed: int, gemm: str,
                 dp_rank: int):
        torch = _lib.require_cuda()
        self._torch, self._libc = torch, _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.CstrLibraryError(f"{type(self).__name__} needs a CUDA device (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if gemm not in _GEMM_MODES:
            raise ValueError("gemm must be 'fp32' (FFMA tiles, the reference's arithmetic), 'tensor' (tcgen05 bf16x3 split, fp32-grade) or "
                             "'bf16' (tcgen05, plain bf16 operands: reduced precision)")
        self.gamma, self.tau, self.learning_rate = float(gamma), float(tau), float(learning_rate)
        self.policy_delay = int(policy_delay)  # updates per actor step, and per captured graph cycle
        self.betas, self.eps, self.seed, self.gemm = (float(betas[0]), float(betas[1])), float(eps), int(seed), gemm
        # data-parallel training: every rank holds the same `seed`, and the in-kernel noise is keyed by (seed, batch row, update), so
        # without the rank in the key row b of every shard would draw the same smoothing noise / eps (perfectly correlated global batch)
        self.dp_rank = int(dp_rank)
        self._graph = self._graph_key = self._graph_out = None
        self._peer = None  # cstr_peer_comm of enable_peer_allreduce()
        self._workspace = None
        self._batch = 0
        self._moments: Dict[int, Any] = {}  # id(adopted parameter) -> (adam_m view, adam_v view)
        self.n_updates = self.critic_step = self.actor_step = self.launches = 0

    def _two_hidden(self, arch: Sequence[int]) -> None:
        if len(arch) != 2:
            raise ValueError(f"{type(self).__name__} supports two-hidden-layer MLPs ([h1, h2]), got {list(arch)}")
        self.h1, self.h2 = int(arch[0]), int(arch[1])
        if self.h1 % 4 or self.h2 % 4:
            raise ValueError("hidden sizes must be multiples of 4")

    def _allocate(self, offs, batch_size: int) -> None:
        """Take the layout the library wrote into ``offs`` (six offsets per net of ``NETS``, the parameter count last) and allocate the
        five blocks, the losses, the graph-mode counters and the workspace."""
        torch = self._torch
        self.param_count = int(offs[len(offs) - 1])
        self._offsets = {(net, t): int(offs[n * 6 + k]) for n, net in enumerate(self.NETS) for k, t in enumerate(_TENSORS)}
        with torch.cuda.device(self.device):
            z = lambda: torch.zeros(self.param_count, dtype=torch.float32, device=self.device)  # noqa: E731
            self.params, self.targets, self.grads, self.adam_m, self.adam_v = z(), z(), z(), z(), z()
            self.loss_sums = torch.zeros(self.N_LOSS, dtype=torch.float32, device=self.device)
            self._counters = torch.zeros(4, dtype=torch.int64, device=self.device)  # graph mode: n_updates, critic_step, actor_step, sample_draw
        self._set_batch(int(batch_size))

    # ---- layout ---------------------------------------------------------------------------------------------------
    def _shape(self, net: str, tensor: str):
        i, h1, h2, o = self._dims(net)
        return {"W1": (h1, i), "b1": (h1,), "W2": (h2, h1), "b2": (h2,), "W3": (o, h2), "b3": (o,)}[tensor]

    def views(self, block: str = "params") -> Dict[str, List[Any]]:
        """``{net: [W1, b1, W2, b2, W3, b3]}`` as views of one flat block (``params|targets|grads|adam_m|adam_v``)."""
        flat = getattr(self, block)
        out = {}
        for net in self.NETS:
            out[net] = []
            for t in _TENSORS:
                shape, off = self._shape(net, t), self._offsets[(net, t)]
                out[net].append(flat[off:off + int(np.prod(shape))].view(shape))
        return out

    def _set_batch(self, batch: int) -> None:
        if batch == self._batch:
            return
        need = self._workspace_bytes(batch)
        if need < 0:
            msg = self._libc.cstr_last_error()
            raise ValueError(msg.decode() if msg else "bad configuration")
        with self._torch.cuda.device(self.device):
            self._workspace = self._torch.empty(need // 4, dtype=self._torch.float32, device=self.device)
        self._batch = batch

    def _keyed_seed(self) -> int:
        return (self.seed + 0x9E3779B97F4A7C15 * self.dp_rank) & (2**64 - 1)

    # ---- weights in / out -------------------------------------------------------------------------------------------
    def _trained_nets(self) -> Sequence[str]:
        return self.NETS

    def _target_nets(self) -> Sequence[str]:
        return self.NETS if self.TARGET_NETS is None else self.TARGET_NETS

    def load_nets(self, nets: Dict[str, Sequence[Any]]) -> None:
        """``nets`` maps every net the engine trains to six arrays/tensors in nn.Linear layout (a head of several modules stacked), and
        optionally ``<net>_target`` for the nets with a target block (default: a copy of the net)."""
        torch = self._torch
        v, t = self.views("params"), self.views("targets")
        for net in self._trained_nets():
            pairs = list(zip(v[net], nets[net]))
            if net in self._target_nets():
                pairs += zip(t[net], nets.get(net + "_target", nets[net]))
            for dst, s in pairs:
                dst.copy_(torch.as_tensor(np.asarray(s) if not isinstance(s, torch.Tensor) else s).to(self.device, torch.float32).reshape(dst.shape))

    def nets(self) -> Dict[str, List[np.ndarray]]:
        out = {net: [x.cpu().numpy() for x in ts] for net, ts in self.views("params").items()}
        targets = self._target_nets()
        out.update({net + "_target": [x.cpu().numpy() for x in ts] for net, ts in self.views("targets").items() if net in targets})
        return out

    def _adopt(self, online, targets) -> None:
        """Copy each module parameter of the ``(view, parameter)`` pairs into its view and re-point ``p.data`` at it (zero-copy sharing
        from then on).  ``online`` views lie in ``params``: their parameters' Adam moments are the same slices of ``adam_m`` / ``adam_v``."""
        online = list(online)
        for view, p in online + list(targets):
            if tuple(p.shape) != tuple(view.shape):
                raise ValueError(f"shape mismatch: module {tuple(p.shape)} vs layout {tuple(view.shape)}")
            view.copy_(p.data.to(self.device, self._torch.float32))
            p.data = view
        self._moments = {}
        for view, p in online:
            off, n = (view.data_ptr() - self.params.data_ptr()) // 4, view.numel()
            self._moments[id(p)] = (self.adam_m[off:off + n].view(view.shape), self.adam_v[off:off + n].view(view.shape))

    def _import_adam(self, opt) -> int:
        """Copy ``exp_avg`` / ``exp_avg_sq`` of every adopted parameter of the ``torch.optim.Adam`` ``opt`` into the moments and take its
        ``betas`` / ``eps``; returns the largest step count found (0 for an optimiser that has not stepped)."""
        group = opt.param_groups[0]
        self.betas, self.eps = (float(group["betas"][0]), float(group["betas"][1])), float(group["eps"])
        step = 0
        for p in group["params"]:
            st = opt.state.get(p)
            if st and id(p) in self._moments:
                m, v = self._moments[id(p)]
                m.copy_(st["exp_avg"])
                v.copy_(st["exp_avg_sq"])
                step = max(step, int(float(st["step"])))
        return step

    def _export_adam(self, opt, step: int) -> None:
        """Make the engine's moment views the Adam state of every adopted parameter of ``opt``, at ``step`` (skipped when it is 0), so that
        ``model.save`` and a later torch ``optimizer.step()`` continue from here."""
        if step == 0:
            return
        for p in opt.param_groups[0]["params"]:
            if id(p) in self._moments:
                m, v = self._moments[id(p)]
                opt.state[p] = {"step": self._torch.tensor(float(step)), "exp_avg": m, "exp_avg_sq": v}

    # ---- the gradient step ----------------------------------------------------------------------------------------------
    def _stream(self) -> int:
        return self._torch.cuda.current_stream(self.device).cuda_stream

    def _f32(self, t, cols):
        torch = self._torch
        if not isinstance(t, torch.Tensor):
            t = torch.as_tensor(np.ascontiguousarray(t), device=self.device)
        t = t.to(device=self.device, dtype=torch.float32).contiguous()
        if t.numel() != self._batch * cols:
            raise ValueError(f"batch tensor has {t.numel()} elements, expected {self._batch}x{cols}")
        return t

    def _batch_f32(self, batch):
        """(obs, actions, next_obs, dones, rewards) of a ``ReplayBufferSamples`` or 5-tuple as contiguous float32 device tensors; sets
        the batch size."""
        obs, act, nobs, dones, rew = batch
        self._set_batch(int(obs.shape[0]))
        return self._f32(obs, 4), self._f32(act, 2), self._f32(nobs, 4), self._f32(dones, 1), self._f32(rew, 1)

    def _state(self, counters: bool) -> "_lib.Td3State":
        return _lib.Td3State(params=self.params.data_ptr(), targets=self.targets.data_ptr(), grads=self.grads.data_ptr(), adam_m=self.adam_m.data_ptr(),
                             adam_v=self.adam_v.data_ptr(), workspace=self._workspace.data_ptr(), workspace_bytes=self._workspace.numel() * 4,
                             losses=self.loss_sums.data_ptr(), counters=self._counters.data_ptr() if counters else None,
                             peer=ctypes.addressof(self._peer) if self._peer is not None else None)

    def _phases(self, run: Callable[[int], None], allreduce, actor_due: bool) -> None:
        """``run(TD3_ALL)``; or, with a host-side ``allreduce`` hook, GRAD -> all-reduce of the critic gradients -> APPLY | ACTOR_GRAD ->
        all-reduce of the actor gradients (when the actor steps) -> ACTOR_APPLY."""
        if allreduce is None:
            run(_lib.TD3_ALL)
            return
        run(_lib.TD3_CRITIC_GRAD)
        allreduce(self.grads[self._reduced_critic[0]:self._reduced_critic[1]])
        run(_lib.TD3_CRITIC_APPLY | _lib.TD3_ACTOR_GRAD)
        if actor_due:
            allreduce(self.grads[self.actor_range[0]:self.actor_range[1]])
        run(_lib.TD3_ACTOR_APPLY)

    # ---- data-parallel training: the gradient all-reduce inside the Adam kernel (include/cstr_b200.h, cstr_peer_comm) ---------------
    def enable_peer_allreduce(self, group=None) -> bool:
        """Move the flat gradient block into memory every rank of ``group`` maps (CUDA IPC over NVLink/NVSwitch, one process per GPU on one
        node) so that the APPLY phases average the gradient over the ranks inside the Adam kernel — no collective launch at all, and the
        update stays capturable as one CUDA graph.  Every rank must then call ``update``/``train`` in lockstep (same number of updates, same
        policy steps).  Returns False (and changes nothing) for a single-process group."""
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return False
        torch, lib = self._torch, self._libc
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        if world > _lib.PEER_MAX_WORLD:
            raise ValueError(f"peer all-reduce spans one NVSwitch node: world size {world} > {_lib.PEER_MAX_WORLD}")
        grad_bytes = (self.param_count * 4 + 255) // 256 * 256
        total = grad_bytes + int(lib.cstr_peer_flag_bytes())
        base, handle = ctypes.c_void_p(), ctypes.create_string_buffer(64)
        with torch.cuda.device(self.device):
            _lib.check(lib.cstr_peer_alloc(total, byref(base), handle), "cstr_peer_alloc")
            handles = [None] * world
            dist.all_gather_object(handles, handle.raw, group=group)
            bases = []
            for r in range(world):
                if r == rank:
                    bases.append(base.value)
                else:
                    p = ctypes.c_void_p()
                    _lib.check(lib.cstr_peer_open(handles[r], byref(p)), f"cstr_peer_open(rank {r})")
                    bases.append(p.value)
            comm = _lib.PeerComm(world=world, rank=rank)
            for r in range(world):
                comm.grads[r], comm.flags[r] = bases[r], bases[r] + grad_bytes
            local = torch.as_tensor(_DeviceMemory(base.value, self.param_count), device=self.device)
            local.copy_(self.grads)
            torch.cuda.synchronize(self.device)
        self.grads, self._peer, self._peer_bases, self._peer_group = local, comm, bases, group
        self._graph = None
        dist.barrier(group)  # nobody starts an update before every rank has mapped every block
        return True

    def peer_error(self) -> int:
        """Non-zero after a rank waited in vain for a peer inside the fused all-reduce (the update of that step was skipped)."""
        if self._peer is None:
            return 0
        err = ctypes.c_uint32(0)
        with self._torch.cuda.device(self.device):
            _lib.check(self._libc.cstr_peer_error(byref(self._peer), byref(err), self._stream()), "cstr_peer_error")
        return int(err.value)

    def close_peer_allreduce(self) -> None:
        """Unmap the peers' blocks and free the local one (collective: every rank calls it)."""
        if self._peer is None:
            return
        import torch.distributed as dist

        torch = self._torch
        torch.cuda.synchronize(self.device)
        dist.barrier(self._peer_group)
        keep = torch.empty(self.param_count, dtype=torch.float32, device=self.device)
        keep.copy_(self.grads)
        rank = self._peer.rank
        self.grads, self._graph = keep, None
        torch.cuda.synchronize(self.device)
        for r, b in enumerate(self._peer_bases):
            if r != rank:
                self._libc.cstr_peer_close(b)
        dist.barrier(self._peer_group)  # a block is freed only after every peer has unmapped it
        self._libc.cstr_peer_free(self._peer_bases[rank])
        self._peer = None

    # ---- CUDA-graph path: one captured cycle of policy_delay x (sample + update), replayed ------------------------------------
    def _capture(self, buffer, batch_size: int, env, allreduce=None) -> None:
        torch = self._torch
        self._set_batch(batch_size)
        f32 = dict(dtype=torch.float32, device=self.device)
        out = (torch.empty((batch_size, 4), **f32), torch.empty((batch_size, 2), **f32), torch.empty((batch_size, 4), **f32),
               torch.empty((batch_size, 1), **f32), torch.empty((batch_size, 1), **f32))
        st = self._state(counters=True)
        draw = self._counters[3:4]

        def cycle():
            for k in range(1, self.policy_delay + 1):  # by-value counters only choose the launch structure: update k of the cycle
                buffer.sample_into(out, draw, env=env)
                self._graph_launch(batch_size, st, out, k, allreduce)

        snapshot = [t.clone() for t in (self.params, self.targets, self.adam_m, self.adam_v, self.loss_sums, self._counters)]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):  # warm-up outside capture (first-launch attribute calls, lazy module loading)
            cycle()
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        # thread_local: a collective inside the cycle keeps NCCL's watchdog thread polling events while this thread captures
        with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
            cycle()
        for dst, src in zip((self.params, self.targets, self.adam_m, self.adam_v, self.loss_sums, self._counters), snapshot):
            dst.copy_(src)  # the warm-up cycle was a real update: undo it
        self._graph, self._graph_out = graph, out
        self._graph_key = self._make_graph_key(buffer, batch_size, env, allreduce)

    def _make_graph_key(self, buffer, batch_size: int, env, allreduce):
        return (id(buffer), batch_size, buffer.size(), buffer.n_envs, id(env), self.policy_delay, self.learning_rate, self.params.data_ptr(),
                self._workspace.data_ptr() if self._workspace is not None else 0, self.grads.data_ptr(), id(allreduce) if allreduce is not None else 0)

    def _train_graph(self, graph: bool, gradient_steps: int, buffer, batch_size: int, env, allreduce=None) -> int:
        """With ``graph`` and a capturable set-up (Philox-index buffer with a full ring, device-side normalisation, no host hook unless
        ``_hook_capturable``), replays whole cycles while the update count is cycle-aligned.  Returns the number of gradient steps done."""
        # a captured cycle bakes the sampling range in: only worth capturing once the ring is full (its range is constant from then on)
        if not (graph and _hook_capturable(allreduce) and getattr(buffer, "index_mode", None) == "philox" and buffer.full and _graph_env_ok(env)):
            return 0
        if self.n_updates % self.policy_delay or gradient_steps < self.policy_delay:
            return 0
        key = self._make_graph_key(buffer, batch_size, env, allreduce)
        if self._graph is None or key != self._graph_key:
            self._capture(buffer, batch_size, env, allreduce)
        cycles = gradient_steps // self.policy_delay
        self._counters.copy_(self._torch.tensor([self.n_updates, self.critic_step, self.actor_step, buffer._draw], dtype=self._torch.int64),
                             non_blocking=True)
        with self._torch.cuda.device(self.device):
            for _ in range(cycles):
                self._graph.replay()
        done = cycles * self.policy_delay
        self.n_updates += done
        self.critic_step += done
        self.actor_step += done // self.policy_delay
        buffer._draw += done
        self.launches += cycles * (23 * (self.policy_delay - 1) + 44 + self.policy_delay)
        return done

    def pop_losses(self):
        """Means since the last call of the losses the kernels sum, ``None`` for one not computed since (the actor's between policy steps):
        TD3 (critic, actor), SAC (critic, actor, ent_coef_loss, ent_coef), BCQ (vae, critic, actor) — what the reference's train() logs."""
        s = self.loss_sums.cpu().numpy().astype(np.float64)
        self.loss_sums.zero_()
        return tuple(s[2 * i] / s[2 * i + 1] if s[2 * i + 1] else None for i in range(self.N_LOSS // 2))


class FusedTD3Update(_FusedEngine):
    NETS = NET_NAMES

    def __init__(self, net_arch: Sequence[int] = (400, 300), batch_size: int = 256, device: Any = "cuda", gamma: float = 0.99, tau: float = 0.005,
                 learning_rate: float = 1e-3, policy_delay: int = 2, target_policy_noise: float = 0.2, target_noise_clip: float = 0.5,
                 betas=(0.9, 0.999), eps: float = 1e-8, seed: int = 0, gemm: str = "fp32", n_critics: int = 2, dp_rank: int = 0):
        super().__init__(device, gamma, tau, learning_rate, policy_delay, betas, eps, seed, gemm, dp_rank)
        self._two_hidden(net_arch)
        self.target_policy_noise, self.target_noise_clip = float(target_policy_noise), float(target_noise_clip)
        if n_critics not in (1, 2):
            raise ValueError("n_critics must be 2 (TD3) or 1 (DDPG)")
        self.n_critics = int(n_critics)
        offs = (c_int64 * 19)()
        _lib.check(self._libc.cstr_td3_layout(self.h1, self.h2, offs), "cstr_td3_layout")
        self._allocate(offs, batch_size)
        self.actor_range = (0, self._offsets[("critic0", "W1")])
        self.critic_range = (self._offsets[("critic0", "W1")], self.param_count)
        self._reduced_critic = self.critic_range

    def _dims(self, net: str):
        return (4, self.h1, self.h2, 2) if net == "actor" else (6, self.h1, self.h2, 1)

    def _trained_nets(self) -> Sequence[str]:
        return NET_NAMES[:1 + self.n_critics]  # DDPG's layout keeps critic1's slots, unused

    def _workspace_bytes(self, batch: int) -> int:
        return int(self._libc.cstr_td3_workspace_bytes(byref(self._config(batch))))

    def _config(self, batch: int) -> "_lib.Td3Config":
        return _lib.Td3Config(h1=self.h1, h2=self.h2, batch=batch, policy_delay=self.policy_delay, gamma=self.gamma, tau=self.tau, lr=self.learning_rate,
                              beta1=self.betas[0], beta2=self.betas[1], eps=self.eps, target_policy_noise=self.target_policy_noise,
                              target_noise_clip=self.target_noise_clip, seed=self._keyed_seed(), gemm_mode=_GEMM_MODES[self.gemm],
                              n_critics=self.n_critics)

    # ---- weights in / out -------------------------------------------------------------------------------------------
    def adopt_modules(self, actor, critics: Sequence[Any], actor_target, critic_targets: Sequence[Any]) -> None:
        """Copy the weights of ``nn.Sequential(Linear, ReLU, Linear, ReLU, Linear[, Tanh])`` modules in and re-point their
        parameters at the flat blocks (zero-copy sharing from then on)."""
        if len(critics) != self.n_critics or len(critic_targets) != self.n_critics:
            raise ValueError(f"expected {self.n_critics} critic network(s)")
        v, t = self.views("params"), self.views("targets")
        online, targets = [], []
        for net, module, target in [("actor", actor, actor_target)] + [(f"critic{z}", critics[z], critic_targets[z]) for z in range(self.n_critics)]:
            ps, pts = list(module.parameters()), list(target.parameters())
            if len(ps) != 6 or len(pts) != 6:
                raise ValueError("expected a 3-layer MLP (6 parameter tensors)")
            online += zip(v[net], ps)
            targets += zip(t[net], pts)
        self._adopt(online, targets)

    def adopt_policy(self, policy) -> None:
        """The reference's ``TD3Policy`` (core/td3/policies.py:172-210): ``actor.mu``, ``critic.q_networks`` and the targets."""
        if len(policy.critic.q_networks) != self.n_critics:
            raise ValueError(f"this engine was built for n_critics={self.n_critics}, the policy has {len(policy.critic.q_networks)}")
        self.adopt_modules(policy.actor.mu, list(policy.critic.q_networks), policy.actor_target.mu, list(policy.critic_target.q_networks))

    def import_optimizer_state(self, actor_optimizer, critic_optimizer) -> None:
        """Take over Adam moments / step counts of ``torch.optim.Adam`` optimisers created over the adopted modules."""
        self.actor_step = self._import_adam(actor_optimizer)
        self.critic_step = self._import_adam(critic_optimizer)

    def export_optimizer_state(self, actor_optimizer, critic_optimizer) -> None:
        """Write moments / step counts back so ``model.save`` and a later torch ``optimizer.step()`` continue from here."""
        self._export_adam(actor_optimizer, self.actor_step)
        self._export_adam(critic_optimizer, self.critic_step)

    # ---- the gradient step ----------------------------------------------------------------------------------------------
    def _graph_launch(self, batch_size: int, st, out, k: int, allreduce=None) -> None:
        cfg = self._config(batch_size)

        def run(phases):
            rc = self._libc.cstr_td3_update(byref(cfg), byref(st), _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]), _lib.ptr(out[3]),
                                            _lib.ptr(out[4]), None, k, 1, 1, phases, self._stream())
            _lib.check(rc, "cstr_td3_update (graph capture)")

        self._phases(run, allreduce, k % self.policy_delay == 0)  # a hook is captured between the phases: GRAD -> all-reduce -> APPLY is ONE graph

    def update(self, batch, noise=None, allreduce: Optional[Callable[[Any], None]] = None) -> None:
        """One iteration of the loop body (td3.py:162-206) on ``batch`` (``ReplayBufferSamples`` or a 5-tuple in that order).
        ``noise``: explicit N(0, target_policy_noise) draws (B,2) for parity tests; default = Philox in the kernel.
        ``allreduce``: called on the flat gradient range between backward and Adam (data-parallel training)."""
        obs, act, nobs, dones, rew = self._batch_f32(batch)
        nz = None if noise is None else self._f32(noise, 2)
        self.n_updates += 1
        self.critic_step += 1
        policy_step = self.n_updates % self.policy_delay == 0
        if policy_step:
            self.actor_step += 1
        cfg = self._config(self._batch)
        st = self._state(counters=False)

        def run(phases):
            rc = self._libc.cstr_td3_update(byref(cfg), byref(st), _lib.ptr(obs), _lib.ptr(act), _lib.ptr(nobs), _lib.ptr(dones), _lib.ptr(rew),
                                            _lib.ptr(nz), self.n_updates, self.critic_step, max(self.actor_step, 0), phases, self._stream())
            _lib.check(rc, "cstr_td3_update")

        with self._torch.cuda.device(self.device):
            self._phases(run, allreduce if self._peer is None else None, policy_step)  # a peer communicator averages inside the APPLY kernels
        self.launches += 23 if not policy_step else 44  # without the split-K finish kernels of small batches

    def train(self, gradient_steps: int, buffer, batch_size: Optional[int] = None, env=None, allreduce=None, graph: bool = False) -> None:
        """``TD3.train(gradient_steps, batch_size)`` (td3.py:154-206): sample + update, ``gradient_steps`` times.
        ``graph=True`` (Philox-index buffer): whole cycles of ``policy_delay`` updates are replayed from ONE captured CUDA graph (24-45
        launches per update become one graph launch per cycle); the remainder runs launch by launch.  Data-parallel training is captured
        too when the averaging is part of the Adam kernels (``enable_peer_allreduce``): sample -> GRAD -> mean over ranks -> APPLY is one
        graph on every rank.  An ``allreduce=`` hook (``dist.all_reduce`` over NCCL) runs launch by launch between the phases unless
        ``CSTR_NCCL_GRAPH=1`` (see ``_hook_capturable``)."""
        bs = int(batch_size or self._batch)
        if self._peer is not None:
            allreduce = None
        done = self._train_graph(graph, gradient_steps, buffer, bs, env, allreduce)
        for _ in range(gradient_steps - done):
            self.update(buffer.sample(bs, env=env), allreduce=allreduce)


class _DeviceMemory:
    """``__cuda_array_interface__`` view of float32 device memory the library allocated (``cstr_peer_alloc``), for ``torch.as_tensor``."""

    def __init__(self, ptr: int, n_floats: int):
        self.__cuda_array_interface__ = {"shape": (int(n_floats),), "typestr": "<f4", "data": (int(ptr), False), "version": 2}


def _dist_rank() -> int:
    """Rank of this process in the default process group (0 when torch.distributed is not initialised)."""
    try:
        import torch.distributed as dist

        return int(dist.get_rank()) if dist.is_available() and dist.is_initialized() else 0
    except Exception:
        return 0


def _hook_capturable(allreduce) -> bool:
    """Whether ``train(graph=True)`` may capture the update.  With no host-side hook (single GPU, or the peer-memory all-reduce inside the Adam
    kernels) always.  A ``dist.all_reduce`` hook captured between the phases worked on 2 GPUs (tests, bench) but HUNG on 8 (ProcessGroupNCCL's
    watchdog stuck while eight ranks captured; profiles/r02_multi_gpu.log), so it is opt-in (``CSTR_NCCL_GRAPH=1``): by default a hook means
    launch by launch, as in round 1 — use ``enable_peer_allreduce()`` for a captured data-parallel update."""
    import os

    return allreduce is None or os.environ.get("CSTR_NCCL_GRAPH", "0") == "1"


def _graph_env_ok(env) -> bool:
    """A captured sample can only normalise on the device (``GpuVecNormalize.norm_params``); the reference's host-side ``VecNormalize``
    needs the launch-by-launch path, whose ``sample()`` round-trips through ``env.normalize_obs`` (buffer.py ``_finish``)."""
    return env is None or getattr(env, "norm_params", None) is not None


def fused_update_unsupported(model, max_critics: int = 2) -> Optional[str]:
    """Why the fused kernels can NOT stand in for ``model.train()`` — or None when they can.  The kernels are specialised to what the
    reference's TD3/DDPG/SAC build by default for the CSTR task (core/td3/policies.py:117-170, core/sac/policies.py:218-262): a flat
    4-value observation, a 2-value action, two ReLU hidden layers shared by actor and critics (multiples of 4), 1-2 critics and plain
    Adam.  Anything else keeps the reference's own torch ``train()``."""
    import torch.nn as nn

    pol = model.policy
    why = _spaces_reason(model)
    if why:
        return why
    if getattr(pol, "activation_fn", nn.ReLU) is not nn.ReLU:
        return f"activation_fn {pol.activation_fn.__name__} (kernels are ReLU)"
    arch = pol.net_arch
    if isinstance(arch, dict):
        if list(arch.get("pi", [])) != list(arch.get("qf", [])):
            return "different actor and critic net_arch"
        arch = arch["pi"]
    arch = list(arch)
    if len(arch) != 2 or any(int(h) < 4 or int(h) > 4096 or int(h) % 4 for h in arch):
        return f"net_arch {arch}: two hidden layers, multiples of 4 in [4, 4096]"
    n_critics = len(pol.critic.q_networks)
    if not 1 <= n_critics <= max_critics:
        return f"n_critics={n_critics}"
    if type(pol.actor.features_extractor).__name__ != "FlattenExtractor":
        return f"features extractor {type(pol.actor.features_extractor).__name__}"
    opt = _not_plain_adam((pol.actor.optimizer, pol.critic.optimizer))
    if opt is not None:
        g = opt.param_groups[0]
        return f"optimizer {type(opt).__name__} {({k: v for k, v in g.items() if k in ('weight_decay', 'amsgrad', 'maximize')})} (kernels are plain Adam)"
    return None


def _spaces_reason(model) -> Optional[str]:
    """Why the model's spaces are not the CSTR's flat (4,) observation and (2,) action that every fused kernel is built for, or None."""
    if tuple(model.observation_space.shape or ()) != (4,) or tuple(model.action_space.shape or ()) != (2,):
        return f"spaces {model.observation_space.shape} -> {model.action_space.shape} are not the CSTR's (4,) -> (2,)"
    return None


def _not_plain_adam(optimizers):
    """The first of ``optimizers`` the fused Adam kernels cannot stand in for (not ``torch.optim.Adam``, or with weight decay, amsgrad or
    maximize), or None."""
    import torch.optim as optim

    for opt in optimizers:
        g = opt.param_groups[0]
        if type(opt) is not optim.Adam or g.get("weight_decay", 0) or g.get("amsgrad", False) or g.get("maximize", False):
            return opt
    return None


def _fallback_once(model, why: str) -> None:
    if not getattr(model, "_fused_fallback_warned", False):
        import warnings
        warnings.warn(f"fused update not used, the reference's torch train() runs instead: {why}", RuntimeWarning, stacklevel=3)
        model._fused_fallback_warned = True


def bind_td3_class(td3_base: type) -> type:
    """Return a subclass of the reference's ``TD3`` (or of ``DDPG``, which is TD3 with one critic, core/ddpg/ddpg.py) whose ``train()``
    (core/td3/td3.py:154-211) runs on ``cstr_td3_update``.
    Rollout collection, logging, saving and ``predict`` stay the reference's code; the policy modules share memory with the
    flat parameter blocks."""

    class FusedTD3(td3_base):  # type: ignore[misc, valid-type]
        _fused: Optional[FusedTD3Update] = None

        def _fused_engine(self, batch_size: int) -> FusedTD3Update:
            if self._fused is None:
                arch = self.policy.net_arch if isinstance(self.policy.net_arch, (list, tuple)) else self.policy.net_arch["pi"]
                eng = FusedTD3Update(arch, batch_size, self.device, self.gamma, self.tau, float(self.lr_schedule(self._current_progress_remaining)),
                                     self.policy_delay, self.target_policy_noise, self.target_noise_clip, seed=int(self.seed or 0),
                                     n_critics=len(self.policy.critic.q_networks),  # DDPG (a TD3 subclass) has one
                                     dp_rank=_dist_rank())
                eng.adopt_policy(self.policy)
                eng.import_optimizer_state(self.actor.optimizer, self.critic.optimizer)
                eng.n_updates = int(self._n_updates)
                self._fused = eng
            return self._fused

        def train(self, gradient_steps: int, batch_size: int = 100) -> None:
            why = fused_update_unsupported(self) if self._fused is None else None
            if why:
                _fallback_once(self, why)
                return super().train(gradient_steps, batch_size)
            self.policy.set_training_mode(True)
            self._update_learning_rate([self.actor.optimizer, self.critic.optimizer])
            eng = self._fused_engine(batch_size)
            eng.learning_rate = float(self.lr_schedule(self._current_progress_remaining))
            # a full ring has a constant sampling range: cycles of policy_delay updates replay from one captured CUDA graph
            eng.train(gradient_steps, self.replay_buffer, batch_size, env=self._vec_normalize_env, graph=bool(getattr(self.replay_buffer, "full", False)))
            self._n_updates = eng.n_updates
            critic_loss, actor_loss = eng.pop_losses()
            self.logger.record("train/n_updates", self._n_updates, exclude="tensorboard")
            if actor_loss is not None:
                self.logger.record("train/actor_loss", actor_loss)
            self.logger.record("train/critic_loss", critic_loss)

        def _excluded_save_params(self):
            return super()._excluded_save_params() + ["_fused"]

        def save(self, *args, **kwargs):
            if self._fused is not None:
                self._fused.export_optimizer_state(self.actor.optimizer, self.critic.optimizer)
            return super().save(*args, **kwargs)

    FusedTD3.__name__ = "TD3"
    FusedTD3.__qualname__ = "TD3"
    return FusedTD3


class FusedSACUpdate(_FusedEngine):
    """SAC gradient steps on the device: one iteration of the loop body of ``SAC.train`` (``core/sac/sac.py:213-288``) per ``update()``
    through ``cstr_sac_update`` — squashed-Gaussian actor sample and log-prob, automatic entropy coefficient, soft twin-min target,
    critics, actor (backward through both critics and the tanh-Gaussian), polyak.  Same flat-block design as :class:`FusedTD3Update`;
    the actor head is ONE (4, h2) matrix [mu; log_std], ``log_ent_coef`` lives in a slot after the three nets.

    ``sde=True``: the gSDE actor (``use_sde=True`` with ``full_std=True``, ``use_expln=False``): the head slot holds ``[mu.weight (2, h2) |
    log_std (h2, 2)]`` (see :meth:`sde_views`), ``clip_mean`` is the Hardtanh bound of the mean (<= 0: none), and every update draws one
    exploration matrix ``exp(log_std) * eps`` from the un-rank-keyed ``seed``, so data-parallel ranks share it."""

    NETS = NET_NAMES
    TARGET_NETS = NET_NAMES[1:]  # SAC has no target actor
    N_LOSS = 8

    def __init__(self, net_arch: Sequence[int] = (256, 256), batch_size: int = 256, device: Any = "cuda", gamma: float = 0.99, tau: float = 0.005,
                 learning_rate: float = 3e-4, target_entropy: float = -2.0, ent_coef_init: float = 1.0, target_update_interval: int = 1,
                 betas=(0.9, 0.999), eps: float = 1e-8, seed: int = 0, gemm: str = "fp32", dp_rank: int = 0, sde: bool = False,
                 clip_mean: float = 2.0):
        super().__init__(device, gamma, tau, learning_rate, 1, betas, eps, seed, gemm, dp_rank)
        self._two_hidden(net_arch)
        self.sde, self.clip_mean = bool(sde), float(clip_mean)
        self.target_entropy, self.target_update_interval = float(target_entropy), int(target_update_interval)
        offs = (c_int64 * 20)()
        _lib.check(self._libc.cstr_sac_layout(self.h1, self.h2, offs), "cstr_sac_layout")
        self._ent_offset = int(offs[18])
        self._allocate(offs, batch_size)
        self.actor_range = (0, self._offsets[("critic0", "W1")])
        self.critic_range = (self._offsets[("critic0", "W1")], self._ent_offset)
        self._reduced_critic = (self.critic_range[0], self._ent_offset + 4)  # both critics and the log_ent_coef slot, contiguous
        self.params[self._ent_offset] = float(np.log(ent_coef_init))

    def _dims(self, net: str):
        return (4, self.h1, self.h2, 4) if net == "actor" else (6, self.h1, self.h2, 1)

    def sde_views(self, block: str = "params"):
        """gSDE: (mu.weight (2, h2), log_std (h2, 2), mu.bias (2,)) as views of ``block``'s actor head slots."""
        w, b = self.views(block)["actor"][4:6]
        return w[0:2], w[2:4].reshape(self.h2, 2), b[0:2]

    @property
    def log_ent_coef(self):
        return self.params[self._ent_offset:self._ent_offset + 1]

    def _sac_config(self, batch: int) -> "_lib.SacConfig":
        return _lib.SacConfig(h1=self.h1, h2=self.h2, batch=batch, target_update_interval=self.target_update_interval, gamma=self.gamma, tau=self.tau,
                              lr=self.learning_rate, beta1=self.betas[0], beta2=self.betas[1], eps=self.eps, target_entropy=self.target_entropy,
                              seed=self._keyed_seed(), gemm_mode=_GEMM_MODES[self.gemm], sde=int(self.sde), clip_mean=self.clip_mean,
                              sde_seed=self.seed & (2**64 - 1))

    def _workspace_bytes(self, batch: int) -> int:
        return int(self._libc.cstr_sac_workspace_bytes(byref(self._sac_config(batch))))

    def adopt_policy(self, policy) -> None:
        """The reference's ``SACPolicy`` (core/sac/policies.py): ``actor.latent_pi`` + ``actor.mu`` + ``actor.log_std``, twin critics.  With gSDE
        ``mu`` is a Linear or ``Sequential(Linear, Hardtanh)`` and ``log_std`` the (h2, 2) parameter (the first of ``actor.parameters()``):
        parameters are mapped to their slots by identity, so their Adam moments follow them whatever the optimiser's order."""
        a, v, t = policy.actor, self.views("params"), self.views("targets")
        head_w, head_b = v["actor"][4], v["actor"][5]
        if self.sde:
            from .rollout import sde_mean_head

            lin = sde_mean_head(a.mu)
            if lin is None or not isinstance(a.log_std, self._torch.Tensor):
                raise ValueError("the gSDE actor needs mu = Linear or Sequential(Linear, Hardtanh(-c, c)) and an (h2, 2) log_std parameter")
            w_mu, w_ls, b_mu = self.sde_views("params")
            online = list(zip(v["actor"][:4], a.latent_pi.parameters())) + [(w_mu, lin[0].weight), (w_ls, a.log_std), (b_mu, lin[0].bias)]
            head_b[2:4].zero_()
        else:
            online = list(zip(v["actor"][:4], a.latent_pi.parameters())) + [(head_w[0:2], a.mu.weight), (head_w[2:4], a.log_std.weight),
                                                                            (head_b[0:2], a.mu.bias), (head_b[2:4], a.log_std.bias)]
        targets = []
        for z, q in enumerate(policy.critic.q_networks):
            online += zip(v[f"critic{z}"], q.parameters())
        for z, q in enumerate(policy.critic_target.q_networks):
            targets += zip(t[f"critic{z}"], q.parameters())
        self._adopt(online, targets)

    def import_optimizer_state(self, actor_optimizer, critic_optimizer, ent_coef_optimizer=None) -> None:
        """Take over Adam moments / the step count of the reference's three optimisers (sac.py:187, policies.py:264-284) after ``adopt_policy``.
        One step count serves all three: the reference steps each exactly once per gradient step."""
        step = max(self._import_adam(actor_optimizer), self._import_adam(critic_optimizer))
        if ent_coef_optimizer is not None:
            for p in ent_coef_optimizer.param_groups[0]["params"]:
                st = ent_coef_optimizer.state.get(p)
                if st:
                    self.adam_m[self._ent_offset] = float(st["exp_avg"])
                    self.adam_v[self._ent_offset] = float(st["exp_avg_sq"])
                    step = max(step, int(float(st["step"])))
        self.critic_step = self.actor_step = step

    def export_optimizer_state(self, actor_optimizer, critic_optimizer, ent_coef_optimizer=None) -> None:
        """Write moments / step count back so ``model.save`` and a later torch ``optimizer.step()`` continue from here."""
        step = self.critic_step
        self._export_adam(actor_optimizer, step)
        self._export_adam(critic_optimizer, step)
        if ent_coef_optimizer is not None and step:
            e = self._ent_offset
            for p in ent_coef_optimizer.param_groups[0]["params"]:
                ent_coef_optimizer.state[p] = {"step": self._torch.tensor(float(step)), "exp_avg": self.adam_m[e:e + 1].reshape(p.shape),
                                               "exp_avg_sq": self.adam_v[e:e + 1].reshape(p.shape)}

    def update(self, batch, eps_pi=None, eps_next=None, allreduce: Optional[Callable[[Any], None]] = None,
               gradient_step: Optional[int] = None) -> None:
        """One iteration of sac.py:213-288.  ``eps_pi`` / ``eps_next``: explicit standard-normal draws (B,2) of the two rsample() calls
        (parity tests); default = Philox inside the kernel.  gSDE engines: ``eps_pi`` is the (h2, 2) standard-normal eps of the update's
        exploration matrix and ``eps_next`` stays None.  ``allreduce``: called on grads[critics .. log_ent_coef] and on grads[actor]
        between backward and Adam (data-parallel training: every rank ends with the gradient of the global batch).
        ``gradient_step``: the index of this step inside the current ``train()`` call — what the reference's target sync tests
        (``gradient_step % target_update_interval``, sac.py:284); None = the engine's own running count of updates."""
        obs, act, nobs, dones, rew = self._batch_f32(batch)
        if self.sde:
            if eps_next is not None:
                raise ValueError("a gSDE update draws one exploration matrix: pass its (h2, 2) eps as eps_pi, eps_next=None")
            e1 = None if eps_pi is None else self._torch.as_tensor(eps_pi).to(self.device, self._torch.float32).contiguous()
            if e1 is not None and tuple(e1.shape) != (self.h2, 2):
                raise ValueError(f"gSDE eps_pi must be ({self.h2}, 2)")
            e2 = None
        else:
            e1 = None if eps_pi is None else self._f32(eps_pi, 2)
            e2 = None if eps_next is None else self._f32(eps_next, 2)
        self.n_updates += 1
        self.critic_step += 1
        self.actor_step += 1
        cfg, st = self._sac_config(self._batch), self._state(counters=False)
        cfg.local_step = 0 if gradient_step is None else int(gradient_step) + 1

        def run(phases):
            rc = self._libc.cstr_sac_update(byref(cfg), byref(st), _lib.ptr(obs), _lib.ptr(act), _lib.ptr(nobs), _lib.ptr(dones), _lib.ptr(rew),
                                            _lib.ptr(e1), _lib.ptr(e2), self.n_updates, self.critic_step, phases, self._stream())
            _lib.check(rc, "cstr_sac_update")

        with self._torch.cuda.device(self.device):
            self._phases(run, allreduce if self._peer is None else None, True)
        self.launches += 50

    def _graph_launch(self, batch_size: int, st, out, k: int, allreduce=None) -> None:
        cfg = self._sac_config(batch_size)

        def run(phases):
            rc = self._libc.cstr_sac_update(byref(cfg), byref(st), _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]), _lib.ptr(out[3]),
                                            _lib.ptr(out[4]), None, None, 1, 1, phases, self._stream())
            _lib.check(rc, "cstr_sac_update (graph capture)")

        self._phases(run, allreduce, True)

    def train(self, gradient_steps: int, buffer, batch_size: Optional[int] = None, env=None, allreduce=None, graph: bool = False) -> None:
        """``graph=True`` (single GPU, Philox-index buffer, full ring, target_update_interval 1): every update replays one captured CUDA graph."""
        bs = int(batch_size or self._batch)
        if self._peer is not None:
            allreduce = None
        done = self._train_graph(graph and self.target_update_interval == 1, gradient_steps, buffer, bs, env, allreduce)
        for g in range(done, gradient_steps):  # g = the reference's loop index: the target sync tests `g % target_update_interval` (sac.py:284)
            self.update(buffer.sample(bs, env=env), allreduce=allreduce, gradient_step=g)


def _sde_update_unsupported(actor) -> Optional[str]:
    """Why ``cstr_sac_update``'s gSDE mode cannot train this actor — or None when it can."""
    from .rollout import _sde_unsupported, sde_mean_head

    why = _sde_unsupported(actor, "fp32", False)
    if why:
        return why
    head = sde_mean_head(getattr(actor, "mu", None))
    if head is None:
        return "use_sde with an actor.mu that is not Linear or Linear + Hardtanh(-c, c)"
    log_std = getattr(actor, "log_std", None)
    if getattr(log_std, "shape", None) is None or tuple(log_std.shape) != (head[0].in_features, 2):
        return "use_sde with an actor.log_std that is not an (H2, 2) parameter"
    return None


def _sde_clip_mean(actor) -> float:
    from .rollout import sde_mean_head

    return sde_mean_head(actor.mu)[1]


def bind_sac_class(sac_base: type) -> type:
    """Subclass of the reference's ``SAC`` (``ent_coef="auto"``; gSDE with ``full_std=True``, ``use_expln=False`` and ``mu`` a Linear or
    Linear + Hardtanh) whose ``train()`` (core/sac/sac.py:199-296) runs on ``cstr_sac_update``."""

    class FusedSAC(sac_base):  # type: ignore[misc, valid-type]
        _fused: Optional[FusedSACUpdate] = None

        def train(self, gradient_steps: int, batch_size: int = 64) -> None:
            why = None
            if self._fused is None:
                why = ("fixed ent_coef" if self.ent_coef_optimizer is None else (_sde_update_unsupported(self.actor) if self.use_sde else None) or
                       ("n_critics != 2" if len(self.policy.critic.q_networks) != 2 else fused_update_unsupported(self)))
            if why:  # the reference's torch path
                _fallback_once(self, why)
                return super().train(gradient_steps, batch_size)
            self.policy.set_training_mode(True)
            self._update_learning_rate([self.actor.optimizer, self.critic.optimizer, self.ent_coef_optimizer])
            if self._fused is None:
                arch = self.policy.net_arch if isinstance(self.policy.net_arch, (list, tuple)) else self.policy.net_arch["pi"]
                eng = FusedSACUpdate(arch, batch_size, self.device, self.gamma, self.tau, float(self.lr_schedule(self._current_progress_remaining)),
                                     float(self.target_entropy), float(self.log_ent_coef.detach().exp().item()), self.target_update_interval,
                                     seed=int(self.seed or 0), dp_rank=_dist_rank(), sde=bool(self.use_sde),
                                     clip_mean=_sde_clip_mean(self.actor) if self.use_sde else 2.0)
                eng.adopt_policy(self.policy)
                self.log_ent_coef.data = eng.log_ent_coef  # shared storage
                eng.import_optimizer_state(self.actor.optimizer, self.critic.optimizer, self.ent_coef_optimizer)
                eng.n_updates = int(self._n_updates)
                self._fused = eng
            eng = self._fused
            eng.learning_rate = float(self.lr_schedule(self._current_progress_remaining))
            eng.train(gradient_steps, self.replay_buffer, batch_size, env=self._vec_normalize_env, graph=bool(getattr(self.replay_buffer, "full", False)))
            self._n_updates += gradient_steps
            critic_loss, actor_loss, ent_loss, ent_coef = eng.pop_losses()
            self.logger.record("train/n_updates", self._n_updates, exclude="tensorboard")
            self.logger.record("train/ent_coef", ent_coef)
            self.logger.record("train/actor_loss", actor_loss)
            self.logger.record("train/critic_loss", critic_loss)
            self.logger.record("train/ent_coef_loss", ent_loss)

        def _excluded_save_params(self):
            return super()._excluded_save_params() + ["_fused"]

        def save(self, *args, **kwargs):
            if self._fused is not None:
                self._fused.export_optimizer_state(self.actor.optimizer, self.critic.optimizer, self.ent_coef_optimizer)
            return super().save(*args, **kwargs)

    FusedSAC.__name__ = "SAC"
    FusedSAC.__qualname__ = "SAC"
    return FusedSAC
