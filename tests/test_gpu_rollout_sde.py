"""gSDE (SAC ``use_sde=True``) in the fused float32 rollout.

* The SDE actor kind of ``rollout_f32_kernel`` against a float64 restatement of the reference's gSDE ``predict``
  (StateDependentNoiseDistribution with learn_features, full_std, no expln: ``tanh(hardtanh(mu(latent), clip_mean) + latent @ E_i)``, core/sac/
  policies.py, core/common/distributions.py), with the per-reactor float32 error bound of test_gpu_rollout_shapes.py, additive action noise on
  top, and the env step, resets and counters of the oracle composition.
* ``cstr_sde_sample``: the Philox normals restated in NumPy, rows of a two-shard run equal to a single run's bit for bit, the moments of
  E / std over 10^4 draws, and new matrices at every epoch.
* ``FusedRollout`` refuses what the SDE kernel does not cover, and ``reset_noise`` advances the epoch.
"""
import numpy as np
import pytest
import torch
import torch.nn as nn

import cstr_oracle as O
import refload
import test_gpu_rollout_shapes as S

gpu = pytest.mark.gpu

N, K = S.N, S.K


def _sde_weights(H1, H2, seed=0, log_std_init=-1.0, mu_bias=0.0):
    W = S._weights(H1, H2, "tanh", seed)  # W3 (2,H2), b3 (2): mu
    W["b3"] = (W["b3"] + np.float32(mu_bias)).astype(np.float32)
    rng = np.random.default_rng(seed + 5)
    log_std = (log_std_init + 0.3 * rng.standard_normal((H2, 2))).astype(np.float32)
    return W, log_std


def sde_actor_f64(state, W, explore, clip_mean):
    """The reference's gSDE action in float64 (mean = Hardtanh(mu(latent)) when clip_mean > 0, noise = latent @ E_i per reactor,
    a = tanh(mean + noise)) and the per-reactor bound of rollout_f32_kernel's float32 forward pass against it."""
    W1, b1, W2, b2, W3, b3 = S._w(W)
    A = np.abs
    s = np.asarray(state, np.float64)
    E = np.asarray(explore, np.float64)
    v1 = s @ W1.T + b1
    e1 = S._gamma(4, A(s) @ A(W1).T + A(b1))
    h1 = np.maximum(v1, 0.0)
    z = h1 @ W2.T + b2
    e2 = e1 @ A(W2).T + S._gamma(W2.shape[1] + 1, (h1 + e1) @ A(W2).T + A(b2))
    lat = np.maximum(z, 0.0)
    H2 = lat.shape[1]
    mu = lat @ W3.T + b3
    emu = e2 @ A(W3).T + S._gamma(H2 + 16, (lat + e2) @ A(W3).T + A(b3))  # per-warp fma chains, b3 + 16 partials
    noise = np.einsum("nk,nkj->nj", lat, E)
    enoise = np.einsum("nk,nkj->nj", e2, A(E)) + S._gamma(H2 + 16, np.einsum("nk,nkj->nj", lat + e2, A(E)))
    mean = np.clip(mu, -clip_mean, clip_mean) if clip_mean > 0 else mu  # clip is 1-Lipschitz
    z = mean + noise
    ez = emu + enoise
    ez = ez + S.U * (A(z) + ez)  # the float32 add
    a = np.tanh(z)
    return a, ez + S.F32_FUNC_ULPS * S.ULP * (A(a) + ez)


def _explore(H2, log_std, seed=3):
    eps = np.random.default_rng(seed).standard_normal((N, H2, 2))
    return (np.exp(log_std.astype(np.float64)) * eps).astype(np.float32)


def _sde_roll(pkg, env, W, log_std, clip_mean, sigma=0.0, buf_rows=None):
    buf = pkg.GpuReplayBuffer(buf_rows or (K + 1) * N, device="cuda", n_envs=N)
    actor = pkg.ActorWeights(**W, kind="sde", log_std=log_std, clip_mean=clip_mean)
    return pkg.FusedRollout(env, buf, actor, sigma=sigma, actor_mode="fp32"), buf


# (H1, H2, clip_mean, mu bias, math): Hardtanh off / binding on some rows / binding on every row, H2 below, at and above 12-row passes
SDE_SHAPES = [
    (64, 64, 2.0, 0.0, "strict"),
    (68, 193, 0.0, 0.0, "strict"),
    (256, 256, 2.0, 0.0, "strict"),     # the SAC default
    (256, 256, 2.0, 0.0, "fast"),
    (4, 1, 0.5, 3.0, "strict"),         # one latent unit; the Hardtanh binds on every row
    (60, 12, 0.3, 0.0, "strict"),
]


@gpu
@pytest.mark.parametrize("H1,H2,clip_mean,mu_bias,math", SDE_SHAPES, ids=[f"{a}x{b}-clip{c}-{m}" for a, b, c, _, m in SDE_SHAPES])
def test_sde_actor_within_float32_bound_of_reference_predict(pkg, H1, H2, clip_mean, mu_bias, math):
    W, log_std = _sde_weights(H1, H2, mu_bias=mu_bias)
    E = _explore(H2, log_std)
    env, st = S._start(pkg, math)
    roll, buf = _sde_roll(pkg, env, W, log_std, clip_mean, sigma=0.3)
    roll.reset_noise()
    roll.explore.copy_(torch.as_tensor(E))
    add = (0.2 * np.random.default_rng(11).standard_normal((K, N, 2))).astype(np.float32)  # NormalActionNoise on top of the gSDE action
    roll.collect(K, noise=torch.as_tensor(add, device="cuda"))
    torch.cuda.synchronize()
    rec = buf.records.cpu().numpy()[:K]
    worst, _ = S._check_launch(env, st, rec, lambda s, k: sde_actor_f64(s, W, E, clip_mean), lambda k: add[k])
    print(f"rollout sde {H1}x{H2} clip {clip_mean} {math}: max |error| / bound = {worst:.3g}")
    if mu_bias:  # the case is the one it claims: mu lies beyond the Hardtanh bound on every row, so the clamped mean is what acts
        W1, b1, W2, b2, W3, b3 = S._w(W)
        lat = np.maximum(np.maximum(rec[:, :, 0:4].reshape(-1, 4).astype(np.float64) @ W1.T + b1, 0.0) @ W2.T + b2, 0.0)
        assert np.all(lat @ W3.T + b3 > clip_mean)


@gpu
def test_sde_matrices_stay_fixed_across_steps_and_launches(pkg):
    """The stored matrices are read, not redrawn: two launches of K/2 steps give the records of one launch of K steps, and a zero matrix
    gives the deterministic action tanh(hardtanh(mu))."""
    W, log_std = _sde_weights(64, 64)
    E = torch.as_tensor(_explore(64, log_std), device="cuda")
    recs = []
    for split in ((K,), (K // 2, K - K // 2)):
        env, _ = S._start(pkg)
        roll, buf = _sde_roll(pkg, env, W, log_std, 2.0)
        roll.reset_noise()
        roll.explore.copy_(E)
        for k in split:
            roll.collect(k)
        recs.append(buf.records[:K].cpu().numpy())
    assert np.array_equal(recs[0], recs[1])
    env, st = S._start(pkg)
    roll, buf = _sde_roll(pkg, env, W, log_std, 2.0)
    roll.reset_noise()
    roll.explore.zero_()
    roll.collect(1)
    a, bound = sde_actor_f64(st[0], W, np.zeros((N, 64, 2)), 2.0)
    assert np.all(np.abs(buf.records[0, :, 8:10].cpu().numpy() - a) <= bound + S.MAPS)


# ---- cstr_sde_sample ------------------------------------------------------------------------------------------------------------------
def sde_normals_f64(n, h2, env_offset, seed, epoch):
    """The (n, h2, 2) standard normals of cstr_sde_sample restated: Philox4x32-10 on counter (global id lo, hi, epoch, 11 << 8 | t & 0xff |
    (t >> 8) << 16) with key = seed, one call per four consecutive values of the flattened (h2, 2) matrix, Box-Muller in float64."""
    per = (2 * h2 + 3) // 4
    env = np.repeat(np.arange(env_offset, env_offset + n, dtype=np.uint64), per)
    t = np.tile(np.arange(per, dtype=np.uint32), n)
    ctr = np.stack([(env & np.uint64(0xFFFFFFFF)).astype(np.uint32), (env >> np.uint64(32)).astype(np.uint32), np.full_like(t, epoch),
                    (np.uint32(11 << 8) | (t & np.uint32(0xFF)) | ((t >> np.uint32(8)) << np.uint32(16)))], axis=1)
    r = O.philox4x32(ctr, np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint32))
    u = [O.u32_to_unit_f32(r[:, j]).astype(np.float64) for j in range(4)]
    u1, u3 = u[0] + 2.0 ** -24, u[2] + 2.0 ** -24
    ra, rb = np.sqrt(-2.0 * np.log(u1)), np.sqrt(-2.0 * np.log(u3))
    z = np.stack([ra * np.cos(2 * np.pi * u[1]), ra * np.sin(2 * np.pi * u[1]), rb * np.cos(2 * np.pi * u[3]), rb * np.sin(2 * np.pi * u[3])], 1)
    return z.reshape(n, per * 4)[:, : 2 * h2].reshape(n, h2, 2)


def _sample(pkg, log_std, n, env_offset, seed, epoch):
    lib = pkg._lib.load()
    h2 = log_std.shape[0]
    out = torch.full((n, h2, 2), float("nan"), device="cuda")
    ls = torch.as_tensor(log_std, device="cuda").contiguous()
    rc = lib.cstr_sde_sample(ls.data_ptr(), h2, n, env_offset, seed, epoch, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    pkg._lib.check(rc, "cstr_sde_sample")
    return out.cpu().numpy()


@gpu
@pytest.mark.parametrize("h2", [1, 13, 256, 600])  # odd h2: the last Philox call half used; 600: call indices past 255
def test_sde_sample_is_the_philox_restatement_and_independent_of_sharding(pkg, h2):
    n, seed, epoch = 293, 0x1234_5678_9ABC, 7
    log_std = (-1.0 + 0.5 * np.random.default_rng(h2).standard_normal((h2, 2))).astype(np.float32)
    full = _sample(pkg, log_std, n, 0, seed, epoch)
    assert np.isfinite(full).all()
    want = np.exp(log_std.astype(np.float64)) * sde_normals_f64(n, h2, 0, seed, epoch)
    assert np.all(np.abs(full - want) <= 2e-6 * (1.0 + np.abs(want))), float(np.abs(full - want).max())
    lo, hi = _sample(pkg, log_std, 150, 0, seed, epoch), _sample(pkg, log_std, n - 150, 150, seed, epoch)
    assert np.array_equal(np.concatenate([lo, hi]), full)  # a 2-rank shard draws the single run's rows bit for bit
    assert not np.array_equal(_sample(pkg, log_std, n, 0, seed, epoch + 1), full)


@gpu
def test_sde_sample_moments_and_epochs(pkg):
    """E / std over 10^4 draws per entry position: mean and variance within 5 sigma of N(0,1); consecutive epochs differ everywhere."""
    h2, n = 8, 10_000
    log_std = np.full((h2, 2), -3.0, np.float32)  # the reference's log_std_init
    e0 = _sample(pkg, log_std, n, 0, 42, 0) / np.exp(np.float32(-3.0))
    z = e0.reshape(n, -1).astype(np.float64)
    assert np.all(np.abs(z.mean(0)) < 5.0 / np.sqrt(n))
    assert np.all(np.abs(z.var(0) - 1.0) < 5.0 * np.sqrt(2.0 / n))
    e1 = _sample(pkg, log_std, n, 0, 42, 1) / np.exp(np.float32(-3.0))
    assert np.mean(e0 == e1) < 1e-3


@gpu
def test_reset_noise_draws_from_the_current_log_std_and_advances_the_epoch(pkg):
    W, log_std = _sde_weights(64, 64)
    env, _ = S._start(pkg)
    roll, buf = _sde_roll(pkg, env, W, log_std, 2.0)
    with pytest.raises(ValueError, match="reset_noise"):
        roll.collect(1)
    roll.collect(1, warmup=True)  # warm-up needs no matrices
    assert roll.sde_epoch == 0
    roll.reset_noise()
    assert roll.sde_epoch == 1 and tuple(roll.explore.shape) == (N, 64, 2)
    seed = int(env._params.seed)
    e0 = roll.explore.cpu().numpy().copy()
    assert np.array_equal(e0, _sample(pkg, log_std, N, 0, seed, 0))
    roll.actor.log_std.add_(1.0)  # refresh_from_module's effect: the next draw uses the new std, the stored matrices keep the old one
    assert np.array_equal(roll.explore.cpu().numpy(), e0)
    roll.reset_noise()
    assert roll.sde_epoch == 2 and np.array_equal(roll.explore.cpu().numpy(), _sample(pkg, log_std + 1.0, N, 0, seed, 1))
    roll.collect(2)
    assert buf.pos == 3


@gpu
def test_sde_actor_refuses_what_the_kernel_does_not_cover(pkg):
    W, log_std = _sde_weights(64, 64)
    env, _ = S._start(pkg)
    buf = pkg.GpuReplayBuffer(2 * N, device="cuda", n_envs=N)
    actor = pkg.ActorWeights(**W, kind="sde", log_std=log_std, clip_mean=2.0)
    with pytest.raises(ValueError, match="float32 kernel"):
        pkg.FusedRollout(env, buf, actor, actor_mode="tc")
    with pytest.raises(ValueError, match="log_std"):
        pkg.ActorWeights(**W, kind="sde", log_std=log_std[:, :1])
    with pytest.raises(ValueError, match="log_std"):
        pkg.ActorWeights(**W, kind="tanh", log_std=log_std)
    # the library's own checks, reached around the Python ones: argument errors, nothing launched
    from ctypes import byref

    lib = pkg._lib.load()

    def launch(actor_mode):
        return lib.cstr_rollout_fused(byref(env._params), N, 1, 0, actor_mode, byref(actor._struct), None, 0.0, None, 0, 0, env.state.data_ptr(),
                                      env.step_count.data_ptr(), env.episode.data_ptr(), None, 2, 0, buf.records.data_ptr(), None, None, None)

    assert launch(0) != 0 and b"cstr_sde_sample" in lib.cstr_last_error()  # no matrices yet
    E = torch.zeros((N, 64, 2), device="cuda")
    actor._struct.explore = E.data_ptr()
    assert launch(1) != 0 and b"actor_mode 0" in lib.cstr_last_error()
    torch.cuda.synchronize()
    assert buf.pos == 0 and (env.step_count == S.SC0).all()


@gpu
def test_from_sac_actor_reads_the_gsde_actor(pkg):
    torch.manual_seed(0)
    trunk = nn.Sequential(nn.Linear(4, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU())
    mu = nn.Sequential(nn.Linear(64, 2), nn.Hardtanh(-2.0, 2.0))
    log_std = nn.Parameter(torch.full((64, 2), -3.0))
    a = pkg.ActorWeights.from_sac_actor(trunk, mu, log_std)
    assert a.kind == "sde" and a.clip_mean == 2.0 and tuple(a.W3.shape) == (2, 64) and torch.equal(a.log_std.cpu(), log_std.detach())
    with torch.no_grad():
        log_std.add_(0.5)
        mu[0].bias.add_(1.0)
    a.refresh_from_module(trunk, mu, log_std)
    torch.cuda.synchronize()
    assert torch.equal(a.log_std.cpu(), log_std.detach()) and torch.equal(a.b3.cpu(), mu[0].bias.detach())
    assert pkg.ActorWeights.from_sac_actor(trunk, mu[0], log_std).clip_mean == 0.0
    with pytest.raises(ValueError, match="Hardtanh"):
        pkg.ActorWeights.from_sac_actor(trunk, nn.Sequential(nn.Linear(64, 2), nn.Tanh()), log_std)


@gpu
@pytest.mark.skipif(not refload.available(), reason="reference tree not available")
def test_learn_with_gsde_runs_the_fused_rollout(pkg):
    """bind_offpolicy_rollout(bind_sac_class(core.SAC)) with use_sde=True, sde_sample_freq=4, every RuntimeWarning an error: the rollout
    and the update both run fused, the exploration epochs are the reference's reset_noise calls, and log_std moves."""
    import warnings

    refload.install_shims()
    core = refload.load_core()
    from core.common.buffers import ReplayBuffer
    from core.common.vec_env import VecEnv

    n = 16
    env = pkg.bind_vec_env_class(VecEnv)(num_envs=n, init_mode="random", reset_rng="philox", seed=3)
    model = pkg.bind_offpolicy_rollout(pkg.bind_sac_class(core.SAC))("MlpPolicy", env, use_sde=True, sde_sample_freq=4, device="cuda",
                                                 replay_buffer_class=pkg.bind_replay_buffer_class(ReplayBuffer), buffer_size=64 * n,
                                                 learning_starts=2 * n, train_freq=(6, "step"), gradient_steps=2, batch_size=32, seed=0, verbose=0)
    before = model.actor.log_std.detach().clone()
    with warnings.catch_warnings():
        warnings.simplefilter("error", RuntimeWarning)  # neither the rollout nor the update falls back
        model.learn(total_timesteps=18 * n, log_interval=None)
    assert model.fused_rollout_launches > 0 and model._fused_roll is not None and model._fused_roll.actor.kind == "sde"
    assert model._fused is not None and model._fused.sde
    assert model._fused_roll.sde_epoch == 3 * (1 + 2)  # three calls of 6 steps: the start, then steps 0 and 4
    assert not torch.equal(model.actor.log_std.detach(), before)
