"""Bit pins of the fast-math kernels that share step_fast_raw: the tape kernel (every output flag combination, HBM and Philox
actions, the bench shape and a ragged one), one VecEnv step and the fp32 fused rollout.

Each case hashes every output of a seeded run.  The digests below were produced on a B200 by the build of commit f73aeb7,
before step_fast_raw paired the two tanks on f32x2 instructions and dropped the state clamps that cannot bind: the
rewrite keeps every lane's operation, operands and order, so the outputs must stay identical byte for byte.
``python tests/test_gpu_tape_bits.py`` prints the digests of the current build.  (The device-side double reward sum is an
atomicAdd in warp order, so it is checked against the rewards instead of hashed.)
"""
import hashlib
import importlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

EXPECTED = {
    "tape_65536x400": "5a703391887d9d260e10b79550d2e54a47c91f3b2f91f11dc6a823ea1d63a858",
    "tape_65536x400_obs_sum": "4c597ddcdf07cc672aa0e948bf73056e4665b178a1d41fae89f77fc55e769eea",
    "tape_1000x13_ragged": "171f7f2b461c1fe8d4b54c229e743490cd2688df18208b693d2ee2ccf54f27af",
    "tape_1000x13_ragged_philox": "6b85becaf30fc35bfe87d1822c61e964e7be95e58102a3d9acd428016717f99e",
    "vec_step_fast": "a6d835d20f2af39d82e22126a6cd752a78f501dfcb549384821b4dc92aa71ccb",
    "rollout_fp32_fast": "13e2aeca09b626ba84e84ff00b7f813995a2e70acb0b1247cc9ab9acba9c390f",
}


def _digest(*arrays) -> str:
    h = hashlib.sha256()
    for a in arrays:
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _env(pkg, n, seed, rng, torch):
    env = pkg.GpuCSTRVecEnv(n, device="cuda:0", math="fast", seed=seed, monitor=False)
    env.reset()
    # spread the step counters so that episodes end (truncate + reset) inside the runs below
    env.step_count.copy_(torch.as_tensor(rng.integers(0, 400, n).astype(np.int32), device="cuda:0"))
    return env


def _state(env):
    return env.state, env.step_count, env.episode


def _check_sum(out):
    rs = float(out["reward_sum"].item())
    ref = float(out["rewards"].double().sum().item())
    assert abs(rs - ref) <= 1e-9 * max(1.0, abs(ref))


def run_cases():
    import torch

    pkg = importlib.import_module("pytorch-rl-enhancedstablebaselines_b200")
    got = {}
    rng = np.random.default_rng(20261020)

    # the bench shape: 65,536 reactors x 400 intervals, HBM actions in [-1, 1)
    n, T = 65536, 400
    env = _env(pkg, n, 7, rng, torch)
    acts = torch.as_tensor(rng.uniform(-1, 1, (T, n, 2)).astype(np.float32), device="cuda:0")
    out = env.tape(T, acts)
    got["tape_65536x400"] = _digest(out["rewards"], out["dones"], *_state(env))
    out = env.tape(T, acts, want_obs=True, reward_sum=True)
    _check_sum(out)
    got["tape_65536x400_obs_sum"] = _digest(out["rewards"], out["dones"], out["obs"], *_state(env))
    del acts, out

    # ragged: n not a multiple of 64, T not a multiple of 8; actions outside [-1, 1] and NaN (bad rows), a NaN state row,
    # and every combination of requested outputs
    n, T = 1000, 13
    env = _env(pkg, n, 11, rng, torch)
    st = env.state.clone()
    st[5] = float("nan")
    env.state.copy_(st)
    parts = []
    for flags in ((True, True, False, False), (False, False, True, True), (True, False, False, False), (False, True, False, True),
                  (True, True, True, False)):
        a = rng.uniform(-1.3, 1.3, (T, n, 2)).astype(np.float32)
        a[rng.random((T, n)) < 0.003] = np.nan
        out = env.tape(T, torch.as_tensor(a, device="cuda:0"), want_rewards=flags[0], want_dones=flags[1], want_obs=flags[2],
                       reward_sum=flags[3])
        parts += [out[k] for k in ("rewards", "dones", "obs") if out[k] is not None] + list(_state(env))
        if flags[3] and flags[0]:
            _check_sum(out)
    got["tape_1000x13_ragged"] = _digest(*parts)
    parts = []
    for t_base, flags in ((0, (True, True, False)), (13, (True, True, True)), (26, (False, True, False))):
        out = env.tape(T, None, t_base=t_base, want_rewards=flags[0], want_dones=flags[1], want_obs=flags[2])
        parts += [out[k] for k in ("rewards", "dones", "obs") if out[k] is not None] + list(_state(env))
    got["tape_1000x13_ragged_philox"] = _digest(*parts)

    # one VecEnv step at a time (cstr_vec_step_f32, fast), auto-reset on truncation, NaN actions and a NaN state row
    n = 4099
    env = _env(pkg, n, 13, rng, torch)
    st = env.state.clone()
    st[17] = float("nan")
    env.state.copy_(st)
    parts = []
    for _ in range(6):
        a = rng.uniform(-1.3, 1.3, (n, 2)).astype(np.float32)
        a[rng.random(n) < 0.01] = np.nan
        obs, rew, done, _ = env.step(a)
        parts += [obs, rew, done] + list(_state(env))
    got["vec_step_fast"] = _digest(*parts)

    # the fp32 fused rollout (actor forward + noise + fast step + replay record)
    n = 2053
    env = _env(pkg, n, 17, rng, torch)
    buf = pkg.GpuReplayBuffer(64 * n, device="cuda:0", n_envs=n)
    g = torch.Generator().manual_seed(3)
    W = [torch.randn(64, 4, generator=g) * 0.5, torch.randn(64, generator=g) * 0.1, torch.randn(48, 64, generator=g) * 0.2,
         torch.randn(48, generator=g) * 0.1, torch.randn(2, 48, generator=g) * 0.3, torch.randn(2, generator=g) * 0.1]
    roll = pkg.FusedRollout(env, buf, pkg.ActorWeights(*W, device="cuda:0"), sigma=0.3, actor_mode="fp32")
    roll.collect(24)
    torch.cuda.synchronize()
    got["rollout_fp32_fast"] = _digest(buf.records, *_state(env))
    return got


@pytest.mark.gpu
def test_fast_kernels_bit_identical_to_pinned_digests():
    got = run_cases()
    assert set(got) == set(EXPECTED)
    bad = {k: (got[k], EXPECTED[k]) for k in EXPECTED if got[k] != EXPECTED[k]}
    assert not bad, f"outputs changed (got, pinned): {bad}"


if __name__ == "__main__":
    print(json.dumps(run_cases(), indent=1))
