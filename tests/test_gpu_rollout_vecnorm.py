"""-m gpu: the fused rollout under VecNormalize (``cstr_rollout_fused_norm``, ``FusedRollout(vec_normalize=...)``) against the float64
oracle (``oracle/cstr_oracle.py::VecNormalizeOracle(exact=True)``) and against the fixture-pinned protocol path
(``GpuVecNormalize.step_wait`` + the reference's store rule, ``oracle/make_golden.py::gen_vecnorm``).

Bars: actions as in test_gpu_rollout.py (fp32 3e-6, tc 5e-3); statistics rel 1e-11 (same float64 moments, other summation order),
returns rel 1e-12; the stored next_obs of a done row bit for bit at K = 1 (statistics read back after the call), within 2 float32 ulp of
the oracle's statistics otherwise.
"""
import copy
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn as nn

import build_oracle as B
import cstr_oracle as O
import refload

pytestmark = pytest.mark.gpu

N = 128 * 3 + 5


def _weights(golden):
    g = golden("td3_actor.npz")
    return g, [(g["W1"], g["b1"]), (g["W2"], g["b2"]), (g["W3"], g["b3"])]


def _env_action(b):
    f = np.float32
    return (f(-1.0) + (f(0.5) * (b + f(1.0)) * f(2.0))).astype(f)


def _stats12(vn):
    return vn.stats.cpu().numpy()[:12]


def _oracle12(o):
    return np.concatenate([o.obs_rms.mean, o.obs_rms.var, [o.obs_rms.count, o.ret_rms.mean, o.ret_rms.var, o.ret_rms.count]])


def _setup(pkg, golden, n=N, seed=7, actor_mode="fp32", start=None, math="strict", use=True, **vn_kw):
    g, _ = _weights(golden)
    env = pkg.GpuCSTRVecEnv(n, seed=seed, monitor=False, math=math)
    env.reset()
    # reactors truncate at different steps, several inside one call
    env.step_count.copy_(torch.as_tensor(start if start is not None else 395 + np.arange(n) % 5, dtype=torch.int32, device="cuda"))
    vn = pkg.GpuVecNormalize(env, **vn_kw) if use else None
    buf = pkg.GpuReplayBuffer(64 * n, device="cuda", n_envs=n)
    actor = pkg.ActorWeights(g["W1"], g["b1"], g["W2"], g["b2"], g["W3"], g["b3"])
    roll = pkg.FusedRollout(env, buf, actor, sigma=0.1, actor_mode=actor_mode, vec_normalize=vn)
    return env, vn, buf, roll


def _replay_oracle(rec, env_state_after, orc, K, w, noise, check_actions=None):
    """Feed the oracle the rollout's own trajectory; return per-step (S_k copies, max |action error| with S_k and with S_{k-1})."""
    errs, errs_prev, prev = [], [], None
    for k in range(K):
        obs = rec[k, :, 0:4]
        if check_actions is not None:
            for o, out in ((orc, errs), (prev, errs_prev)):
                if o is None:
                    continue
                mu = O.actor_forward(o.normalize_obs(obs), w).astype(np.float32)
                _, a_buf = O.sample_action_maps(mu, noise[k])
                out.append(float(np.abs(rec[k, :, 8:10] - a_buf).max()))
        nxt = rec[k + 1, :, 0:4] if k + 1 < K else env_state_after
        prev = copy.deepcopy(orc)
        orc.step(nxt, rec[k, :, 10], rec[k, :, 11] > 0)
    return errs, errs_prev


# ---- 1. the VecNormalize launches change nothing else ---------------------------------------------------------------------------------
@pytest.mark.parametrize("math", ["strict", "fast"])
@pytest.mark.parametrize("actor_mode", ["fp32", "tc"])
def test_identity_wrapper_is_bit_identical_to_the_plain_rollout(pkg, golden, math, actor_mode):
    n, K = 128 * 5 + 37, 23
    outs = []
    for use in (False, True):
        env, vn, buf, roll = _setup(pkg, golden, n=n, seed=4, actor_mode=actor_mode, math=math, start=np.full(n, 390), use=use,
                                    norm_obs=False, norm_reward=False, training=False)
        roll.t = 5
        stats = pkg.EpisodeStats(n)
        rs = torch.zeros(1, dtype=torch.float64, device="cuda")
        roll.collect(K, reward_sum=rs, stats=stats)
        torch.cuda.synchronize()
        fin = stats.pop()
        outs.append(dict(rec=buf.records.cpu().numpy()[:K], state=env.state.cpu().numpy(), sc=env.step_count.cpu().numpy(),
                         ep=env.episode.cpu().numpy(), ep_ret=stats.ep_return.cpu().numpy(), fin=fin[np.lexsort(fin.T[::-1])], rs=rs.item()))
        if use:
            assert roll.launches == K
            assert np.array_equal(vn.stats.cpu().numpy()[:12], np.array([0, 0, 0, 0, 1, 1, 1, 1, 1e-4, 0, 1, 1e-4]))
            assert np.all(vn.returns_device.cpu().numpy() == 0.0)
    a, b = outs
    for key in ("rec", "state", "sc", "ep", "ep_ret", "fin"):
        assert np.array_equal(a[key].view(np.uint8), b[key].view(np.uint8)), key
    assert (a["rec"][9, :, 11] == 1).all()  # 390 + 10 = 400: the window crosses the truncation
    # reward_sum: both paths atomicAdd per-warp partial sums, in no fixed order
    assert a["rs"] == pytest.approx(b["rs"], rel=1e-12)


# ---- 2 + 3. the actor reads normalize(obs_k; S_k); the statistics follow the oracle and are reproducible ------------------------------
@pytest.mark.parametrize("actor_mode,atol", [("fp32", 3e-6), ("tc", 5e-3)])
def test_actor_input_and_statistics_follow_the_oracle(pkg, golden, actor_mode, atol):
    _, w = _weights(golden)
    K, calls = 6, 2
    noise = (0.1 * np.random.default_rng(1).standard_normal((calls, K, N, 2))).astype(np.float32)
    runs = []
    for rep in range(2):
        env, vn, buf, roll = _setup(pkg, golden, actor_mode=actor_mode)  # fresh statistics: count 1e-4, the first steps move them a lot
        orc = O.VecNormalizeOracle(N, exact=True)
        st0 = env.state.cpu().numpy().copy()
        assert np.array_equal(st0, env.state.cpu().numpy())
        snaps = []
        for c in range(calls):
            roll.collect(K, noise=torch.as_tensor(noise[c], device="cuda"))
            rec = buf.records.cpu().numpy()[c * K:(c + 1) * K]
            snaps.append((rec.copy(), vn.stats.cpu().numpy().copy(), vn.returns_device.cpu().numpy().copy()))
            if rep == 0:
                errs, errs_prev = _replay_oracle(rec, env.state.cpu().numpy(), orc, K, w, noise[c], check_actions=True)
                print(f"{actor_mode} call {c}: max |action - oracle(S_k)| {max(errs):.3e}, with S_(k-1) {max(errs_prev) if errs_prev else 0:.3e}")
                assert max(errs) <= atol
                if c == 0:
                    assert max(errs_prev) > 10 * atol  # normalising with the statistics one step late misses the bar
                s, e = _stats12(vn), _oracle12(orc)
                print(f"{actor_mode} call {c}: stats max rel {np.max(np.abs(s - e) / np.abs(e)):.2e}")
                np.testing.assert_allclose(s, e, rtol=1e-11, atol=1e-13)
                np.testing.assert_allclose(vn.returns_device.cpu().numpy(), orc.returns, rtol=1e-12, atol=1e-12)
                if c == 0:
                    assert (rec[:, :, 11] > 0).any(axis=0).sum() == N  # every reactor auto-resets inside the first call
        runs.append(snaps)
    for (r0, s0, q0), (r1, s1, q1) in zip(*runs):  # same inputs, same bits: the merge has a fixed order
        assert np.array_equal(r0.view(np.uint32), r1.view(np.uint32))
        assert np.array_equal(s0.view(np.uint64), s1.view(np.uint64)) and np.array_equal(q0.view(np.uint64), q1.view(np.uint64))


# ---- 4. done rows store unnormalize(normalize(terminal; S_(k+1))) ---------------------------------------------------------------------
@pytest.mark.parametrize("actor_mode", ["fp32", "tc"])
def test_terminal_round_trip(pkg, golden, actor_mode):
    env, vn, buf, roll = _setup(pkg, golden, actor_mode=actor_mode, start=397 + np.arange(N) % 3, clip_obs=0.5)
    vn.reset()  # the reference's learn() starts with a reset: statistics of the initial observations
    env.step_count.copy_(torch.as_tensor(397 + np.arange(N) % 3, dtype=torch.int32, device="cuda"))
    orc = O.VecNormalizeOracle(N, exact=True, clip_obs=0.5)
    orc.reset(env.state.cpu().numpy())
    sc = env.step_count.cpu().numpy().copy()
    n_done = 0
    for k in range(4):  # K = 1 per call: the statistics read after the call are the ones the round trip used
        obs = env.state.cpu().numpy().copy()
        roll.collect(1)
        rec = buf.records.cpu().numpy()[k]
        term, _, tr, sc, _ = B.step_f32(obs, _env_action(rec[:, 8:10]), sc, exp_mode=B.EXP_SHARED, sq_mode=B.SQ_MUL)
        done = tr.astype(bool)
        sc[done] = 0  # the oracle step counts on; the env restarts the episode
        assert np.array_equal(rec[:, 0:4], obs) and np.array_equal(done, rec[:, 11] > 0)
        assert np.array_equal(rec[~done, 4:8], term[~done])  # non-done rows: raw next observation
        if done.any():
            want = np.asarray(vn.unnormalize_obs(vn.normalize_obs(term[done])), np.float32)
            assert np.array_equal(rec[done, 4:8].view(np.uint32), want.view(np.uint32))
            assert not np.array_equal(rec[done, 4:8], term[done])  # the clip binds: not the terminal observation
            n_done += int(done.sum())
        orc.step(env.state.cpu().numpy(), rec[:, 10], done)
    assert n_done == N
    # K > 1: rows finished in the middle of a call, against the oracle's S_(k+1)
    env.step_count.copy_(torch.as_tensor(396 + np.arange(N) % 4, dtype=torch.int32, device="cuda"))
    orc_sc = env.step_count.cpu().numpy().copy()
    K, row0 = 5, buf.pos
    roll.collect(K)
    rec = buf.records.cpu().numpy()[row0:row0 + K]
    worst = 0.0
    for k in range(K):
        term, _, tr, orc_sc, _ = B.step_f32(rec[k, :, 0:4], _env_action(rec[k, :, 8:10]), orc_sc, exp_mode=B.EXP_SHARED, sq_mode=B.SQ_MUL)
        done = tr.astype(bool)
        orc_sc[done] = 0
        nxt = rec[k + 1, :, 0:4] if k + 1 < K else env.state.cpu().numpy()
        orc.step(nxt, rec[k, :, 10], done)
        assert np.array_equal(rec[k, ~done, 4:8], term[~done])
        if done.any():
            want = (orc.normalize_obs(term[done]) * np.sqrt(orc.obs_rms.var + orc.epsilon) + orc.obs_rms.mean).astype(np.float32)
            u = np.abs(rec[k, done, 4:8].astype(np.float64) - want) / np.spacing(np.abs(want)).astype(np.float64)
            worst = max(worst, float(u.max()))
    print(f"{actor_mode}: round trip at K={K}, max {worst:.1f} float32 ulp from the oracle")
    assert worst <= 2.0


# ---- 5. same records and statistics as GpuVecNormalize.step_wait + the reference's store rule -----------------------------------------
def test_matches_the_protocol_path(pkg, golden):
    K = 7
    env, vn, buf, roll = _setup(pkg, golden)
    vn.reset()
    env.step_count.copy_(torch.as_tensor(395 + np.arange(N) % 5, dtype=torch.int32, device="cuda"))
    roll.collect(K)
    rec = buf.records.cpu().numpy()[:K]
    env2 = pkg.GpuCSTRVecEnv(N, seed=7, monitor=False)
    env2.reset()
    vn2 = pkg.GpuVecNormalize(env2)
    vn2.reset()
    assert np.array_equal(rec[0, :, 0:4], vn2.get_original_obs())
    env2.step_count.copy_(torch.as_tensor(395 + np.arange(N) % 5, dtype=torch.int32, device="cuda"))
    buf2 = pkg.GpuReplayBuffer(64 * N, device="cuda", n_envs=N)
    last_raw = vn2.get_original_obs()
    for k in range(K):  # off_policy_algorithm.py:468-494 (oracle/make_golden.py::gen_vecnorm)
        _, _, d, infos = vn2.step(_env_action(rec[k, :, 8:10]))
        raw_o, raw_r = vn2.get_original_obs(), vn2.get_original_reward()
        nxt = raw_o.copy()
        for i, info in infos.done_items():
            nxt[i] = vn2.unnormalize_obs(info["terminal_observation"])
        buf2.add(last_raw, nxt, rec[k, :, 8:10], raw_r, d, infos)
        last_raw = raw_o
    rec2 = buf2.records.cpu().numpy()[:K]
    assert np.array_equal(rec.view(np.uint32), rec2.view(np.uint32))
    assert (rec[:, :, 11] > 0).sum() == N
    np.testing.assert_allclose(_stats12(vn), _stats12(vn2), rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(vn.returns_device.cpu().numpy(), vn2.returns_device.cpu().numpy(), rtol=1e-12, atol=1e-12)


# ---- 6. switches -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["norm_obs_off", "norm_reward_off", "frozen", "warmup"])
def test_switches(pkg, golden, case):
    kw = dict(norm_obs=case != "norm_obs_off", norm_reward=case != "norm_reward_off", training=case != "frozen")
    env, vn, buf, roll = _setup(pkg, golden, **kw)
    init = _stats12(vn).copy()
    if case == "frozen":
        vn.returns_device.fill_(1.0)
    orc = O.VecNormalizeOracle(N, exact=True, **kw)
    orc.returns[:] = vn.returns_device.cpu().numpy()
    K = 3  # reactors starting at 397..399 finish inside the call, those at 395 and 396 do not
    roll.collect(K, warmup=case == "warmup")
    rec = buf.records.cpu().numpy()[:K]
    for k in range(K):
        orc.step(rec[k + 1, :, 0:4] if k + 1 < K else env.state.cpu().numpy(), rec[k, :, 10], rec[k, :, 11] > 0)
    s = _stats12(vn)
    np.testing.assert_allclose(s, _oracle12(orc), rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(vn.returns_device.cpu().numpy(), orc.returns, rtol=1e-12, atol=1e-12)
    if case == "norm_obs_off":
        assert np.array_equal(s[:9], init[:9]) and s[11] == pytest.approx(init[11] + K * N)
    elif case == "frozen":
        assert np.array_equal(s, init)
        ret = vn.returns_device.cpu().numpy()
        finished = (rec[:, :, 11] > 0).any(axis=0)
        assert finished.any() and not finished.all()
        assert np.all(ret[finished] == 0.0) and np.all(ret[~finished] == 1.0)
    else:
        assert s[8] == pytest.approx(init[8] + K * N) and s[11] == pytest.approx(init[11] + K * N)


# ---- 7. the host guard, with stand-in models -------------------------------------------------------------------------------------------
class FlattenExtractor(nn.Module):
    pass


def _mlp(sizes, head=nn.Tanh):
    layers = []
    for i, (a, b) in enumerate(zip(sizes[:-1], sizes[1:])):
        layers += [nn.Linear(a, b)] + ([nn.ReLU()] if i < len(sizes) - 2 else ([head()] if head else []))
    return nn.Sequential(*layers)


def test_guard_accepts_gpu_vec_normalize(pkg):
    env = pkg.GpuCSTRVecEnv(8, seed=0, monitor=False)
    vn = pkg.GpuVecNormalize(env)
    buf = pkg.GpuReplayBuffer(64, device="cuda", n_envs=8)
    freq = SimpleNamespace(unit="step", frequency=4)
    trunk = _mlp([4, 64, 64], head=None)
    trunk.append(nn.ReLU())
    td3 = SimpleNamespace(actor=SimpleNamespace(features_extractor=FlattenExtractor(), mu=_mlp([4, 64, 64, 2])), use_sde=False, _vec_normalize_env=vn)
    sac = SimpleNamespace(actor=SimpleNamespace(features_extractor=FlattenExtractor(), latent_pi=trunk, mu=nn.Linear(64, 2), log_std=nn.Linear(64, 2)),
                          use_sde=False, _vec_normalize_env=vn)
    agents = SimpleNamespace(actor=SimpleNamespace(mu_list=nn.ModuleList([_mlp([2, 60, 12, 1]) for _ in range(2)])), use_sde=False,
                             _vec_normalize_env=vn, observation_splits=[[0, 1], [2, 3]], action_splits=[[0], [1]])

    def why(model, e, mode="fp32"):
        return pkg.rollout.fused_rollout_unsupported(model, e, buf, freq, None, actor_mode=mode)

    for mode in ("fp32", "tc"):
        assert why(td3, vn, mode) is None and why(sac, vn, mode) is None
        assert "two agents" in why(agents, vn, mode)
    host_vn = SimpleNamespace(venv=env, num_envs=8)  # the reference's own VecNormalize: not a GpuVecNormalize
    td3.__dict__["_vec_normalize_env"] = host_vn
    assert "VecNormalize wraps the env" in why(td3, host_vn)
    assert "VecNormalize wraps the env" in why(td3, env)
    td3.__dict__["_vec_normalize_env"] = None
    assert "_vec_normalize_env" in why(td3, vn)  # a wrapper the model does not know about
    pcg = pkg.GpuVecNormalize(pkg.GpuCSTRVecEnv(8, seed=0, monitor=False, reset_rng="pcg64"))
    td3.__dict__["_vec_normalize_env"] = pcg
    assert "philox" in why(td3, pcg)
    f64 = pkg.GpuVecNormalize.__new__(pkg.GpuVecNormalize)  # the constructor refuses fp64; a stand-in with the same attributes
    f64.__dict__["venv"] = pkg.GpuCSTRVecEnv(8, seed=0, monitor=False, dtype="fp64")
    td3.__dict__["_vec_normalize_env"] = f64
    assert "dtype='fp32'" in why(td3, f64)
    with pytest.raises(ValueError, match="wrap env"):
        pkg.FusedRollout(pkg.GpuCSTRVecEnv(8, seed=0, monitor=False), buf, None, vec_normalize=vn)


# ---- 8. the reference's learn() with the bound classes ---------------------------------------------------------------------------------
@pytest.mark.skipif(not refload.available(), reason="reference tree not staged")
def test_reference_learn_under_vec_normalize_uses_the_fused_rollout(pkg):
    import warnings

    refload.install_shims()
    core = refload.load_core()
    from core.common.buffers import ReplayBuffer
    from core.common.vec_env import VecEnv, VecNormalize

    n = 256
    env = pkg.bind_vec_env_class(VecEnv)(num_envs=n, init_mode="random", reset_rng="philox", seed=3)
    venv = pkg.bind_vec_normalize_class(VecNormalize)(env)
    model = pkg.bind_offpolicy_rollout(pkg.bind_td3_class(core.TD3))("MlpPolicy", venv, device="cuda", replay_buffer_class=pkg.bind_replay_buffer_class(ReplayBuffer),
                                                                    buffer_size=64 * n, learning_starts=4 * n, batch_size=64, train_freq=(4, "step"),
                                                                    gradient_steps=1, seed=0, verbose=0)
    with warnings.catch_warnings():
        warnings.simplefilter("error", RuntimeWarning)
        model.learn(total_timesteps=16 * n, log_interval=None)
    assert model.fused_rollout_launches > 0
    rec = model.replay_buffer.records.cpu().numpy()[:16]
    cont = rec[:-1, :, 11] == 0  # original (raw) observations are stored: next_obs of a step is the obs of the next one
    assert np.array_equal(rec[1:, :, 0:4][cont], rec[:-1, :, 4:8][cont]) and np.abs(rec[:, :, 0:8]).max() <= 1.0
    raw = env.state.cpu().numpy()
    assert np.array_equal(model._last_original_obs, raw) and np.array_equal(venv.old_obs, raw)
    assert np.array_equal(model._last_obs, venv.normalize_obs(raw)) and not np.array_equal(model._last_obs, raw)
