"""The fused rollout's actor at every shape the two rollout kernels accept, against float64 references with per-reactor error bounds.

* ``rollout_f32_kernel`` (actor_mode "fp32") against the exact actor in float64, bounded by the float32 forward error of its three layers.
* ``rollout_tc_kernel`` (actor_mode "tc") against a float64 emulation of the arithmetic ``csrc/cstr_rollout_tc.cu`` documents: layer 1
  from the split-bf16 operands with the W_lo * s_lo term dropped, h1 and W2 rounded to bf16, fp32 accumulation.  Everything the kernel
  rounds on purpose is reproduced, so the bound is only the accumulation error: a lost b_lo or W_lo term, or a K-group read from the
  wrong place, moves the action by ~1e-4 and fails it, where the 5e-3 bar against the exact actor cannot see it.
* Given the stored action the env step is bit-exact (strict: the C oracle; fast: the fast vec_step kernel), and the state, counters and
  static base after the launch are the oracle composition's, resets included.
* Shapes either kernel rejects come back as a ValueError before anything is launched, and ``fused_rollout_unsupported`` sends actors the
  kernels cannot evaluate to the reference's own ``collect_rollouts``.
"""
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn as nn

import build_oracle as B
import refload

gpu = pytest.mark.gpu

N, K, SC0 = 2 * 128 + 37, 12, 395  # a ragged last tile; step 5 of the launch truncates every reactor and resets it

# ---- error model ------------------------------------------------------------------------------------------------------------------
U = 2.0 ** -24    # unit roundoff of float32: one correctly rounded op errs by at most U * |result|
ULP = 2.0 ** -23  # ulp(x) <= ULP * |x| for a normal float32 x
# tensor-core accumulation: each bf16 x bf16 product is exact in fp32, and one K=16 MMA step adds at most one fp32 ulp of the running
# sum, whose magnitude is at most the sum of |products| so far -> steps * ULP * sum|w * x| per dot product (derived, not fitted)
MMA_ULPS_PER_STEP = 1
F32_FUNC_ULPS = 2  # tanhf, expf: maximum ulp error in the CUDA C Programming Guide
MAPS = 2.0 ** -21  # the float32 action maps (policies.py scale / unscale, + noise, clip): at most five roundings of values below 2


def _gamma(k, absdot):
    """Forward error bound of a float32 dot product of length k accumulated in any order: (k + 2) * U * sum|w * x|."""
    return (k + 2) * U * absdot


def _bf16(x):
    """float32 (float64 is rounded to float32 first, as the kernel's fp32 accumulator is) -> bfloat16, round to nearest even."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32).astype(np.float64)


def _split(x):
    """x = hi + lo, two bf16 values (the kernel's __float2bfloat16_rn(x) and __float2bfloat16_rn(x - hi); x - hi is exact in fp32)."""
    x32 = np.asarray(x, np.float32)
    hi = _bf16(x32)
    return hi, _bf16((x32.astype(np.float64) - hi).astype(np.float32))


def _head(pre, e, kind, eps):
    """The actor head in float64 and the bound of the kernel's float32 head (actor_head) on pre-activations known to within e."""
    if kind == "tanh":
        z, ez = pre[:, :2], e[:, :2]
    else:  # tanh(mu + exp(clip(log_std, -20, 2)) * eps): clip is 1-Lipschitz, exp is bounded over the clipped interval
        mu, emu = pre[:, :2], e[:, :2]
        c, ec = np.clip(pre[:, 2:], -20.0, 2.0), e[:, 2:]
        s = np.exp(c)
        s_hi = np.exp(np.minimum(c + ec, 2.0))
        es = np.maximum(s_hi - s, s - np.exp(np.maximum(c - ec, -20.0))) + F32_FUNC_ULPS * ULP * s_hi
        eps = np.asarray(eps, np.float64)
        z = mu + s * eps
        ez = emu + np.abs(eps) * es
        ez = ez + U * (np.abs(z) + ez)  # the fmaf
    a = np.tanh(z)
    return a, ez + F32_FUNC_ULPS * ULP * (np.abs(a) + ez)  # tanh is 1-Lipschitz, then tanhf's own error


def _w(W):
    return [np.asarray(W[k], np.float64) for k in ("W1", "b1", "W2", "b2", "W3", "b3")]


def actor_f64(state, W, kind="tanh", eps=None):
    """The exact actor in float64 and the per-reactor bound of rollout_f32_kernel's float32 forward pass against it."""
    W1, b1, W2, b2, W3, b3 = _w(W)
    A = np.abs
    s = np.asarray(state, np.float64)
    v1 = s @ W1.T + b1
    e1 = _gamma(4, A(s) @ A(W1).T + A(b1))  # b1 then four fmas
    h1 = np.maximum(v1, 0.0)
    z = h1 @ W2.T + b2
    e2 = e1 @ A(W2).T + _gamma(W2.shape[1] + 1, (h1 + e1) @ A(W2).T + A(b2))  # H1 fmas, + b2
    h2 = np.maximum(z, 0.0)
    pre = h2 @ W3.T + b3
    e3 = e2 @ A(W3).T + _gamma(W3.shape[1] + 16, (h2 + e2) @ A(W3).T + A(b3))  # per-warp fma chains, then b3 + 16 partial sums
    return _head(pre, e3, kind, eps)


def actor_tc_emulated(state, W, kind="tanh", eps=None):
    """rollout_tc_kernel's actor emulated exactly in float64, and the per-reactor bound of the kernel against it."""
    W1, b1, W2, b2, W3, b3 = _w(W)
    A = np.abs
    H1 = W1.shape[0]
    # layer 1: one K=16 MMA of [s_hi | s_lo][s_hi | 1 1 0 0] against [W_hi | W_hi][W_lo | b_hi b_lo 0 0]; W_lo * s_lo is dropped
    sh, sl = _split(state)
    Wh, Wl = _split(W1)
    bh, bl = _split(b1)
    v1 = sh @ Wh.T + sl @ Wh.T + sh @ Wl.T + bh + bl
    e1 = MMA_ULPS_PER_STEP * ULP * (A(sh) @ A(Wh).T + A(sl) @ A(Wh).T + A(sh) @ A(Wl).T + A(bh) + A(bl))
    # relu, then bf16: round-to-nearest is monotone, so the kernel's h1 lies between the roundings of the ends of [v1 - e1, v1 + e1];
    # it differs from the emulated h1 only where a rounding midpoint lies within e1 (the rounding-flip allowance)
    h1 = _bf16(np.maximum(v1, 0.0))
    flip = np.maximum(_bf16(np.maximum(v1 + e1, 0.0)) - h1, h1 - _bf16(np.maximum(v1 - e1, 0.0)))
    # layer 2: bf16 W2 on the tensor core, H1 / 16 MMA steps accumulating in TMEM; the epilogue adds b2 in fp32
    W2b = _bf16(W2)
    z = h1 @ W2b.T
    e2 = flip @ A(W2b).T + (H1 // 16) * MMA_ULPS_PER_STEP * ULP * ((h1 + flip) @ A(W2b).T)
    y = z + b2
    e2 = e2 + U * (A(y) + e2)
    h2 = np.maximum(y, 0.0)
    # layer 3 in fp32 on the CUDA cores: per-thread fma chains over half of the columns, the two partials, + b3
    pre = h2 @ W3.T + b3
    e3 = e2 @ A(W3).T + _gamma(W3.shape[1] + 16, (h2 + e2) @ A(W3).T + A(b3))
    return _head(pre, e3, kind, eps)


# ---- the tensor-core geometry (a mirror of make_geometry in csrc/cstr_rollout_tc.cu) -------------------------------------------------
TC_M, TC_PER, SMEM_MAX = 128, 2, 227 * 1024


def tc_geometry(H1, H2):
    """dict(KC, NKC, NP, N0, N1, tmem, smem, bytes), or a string naming the limit the shape breaks."""
    if H1 <= 0 or H2 <= 0 or H1 % 16 or H1 > 1024:
        return "H1"
    NP = (H2 + 15) & ~15
    if NP > 512:
        return "NP"
    KC = next(c for c in (80, 64, 48, 32, 16) if H1 % c == 0)
    N0 = NP if NP <= 256 else ((NP // 2) + 15) & ~15
    if NP + 2 * KC > 512:
        return "tmem"
    tmem = 32
    while tmem < NP + 2 * KC:
        tmem <<= 1

    def up(x):
        return (x + 127) & ~127

    a_chunk, w_chunk = (KC // 8) * TC_M * 16, (KC // 8) * NP * 16
    off_a1 = up(256 + 2 * H1 * 16)
    off_ep = up(off_a1 + 2 * TC_M * 16)
    off_part = up(off_ep + 5 * NP * 4)
    off_a = up(off_part + 2 * TC_PER * TC_M * 16)
    smem = up(up(off_a + 2 * a_chunk) + 3 * w_chunk)
    if smem > SMEM_MAX:
        return "smem"
    return dict(KC=KC, NKC=H1 // KC, NP=NP, N0=N0, N1=NP - N0, tmem=tmem, smem=smem, bytes=(H1 // KC) * w_chunk)


# (H1, H2, kind, math): every accepted branch of make_geometry
TC_SHAPES = [
    (16, 1, "tanh", "strict"),        # KC 16, NKC 1, NP 16, TMEM 64
    (32, 20, "tanh", "strict"),       # KC 32, NKC 1, TMEM 128
    (48, 33, "tanh", "strict"),       # KC 48, NKC 1, H2 padded 33 -> 48
    (64, 64, "tanh", "strict"),       # KC 64, NKC 1
    (64, 64, "gauss", "strict"),      # Gaussian head, unsplit width
    (80, 256, "tanh", "strict"),      # KC 80, NKC 1, NP 256: the last unsplit width
    (96, 257, "tanh", "strict"),      # NKC 2, first split width, N0/N1 = 144/128
    (96, 257, "gauss", "strict"),     # Gaussian head, split width
    (144, 128, "tanh", "strict"),     # KC 48, NKC 3 (odd)
    (144, 128, "tanh", "fast"),
    (112, 300, "tanh", "strict"),     # KC 16, NKC 7
    (16, 480, "tanh", "strict"),      # N0 = N1 = 240, NP + 2 KC = 512: all of TMEM
    (960, 200, "tanh", "strict"),     # KC 80, NKC 12
    (1024, 256, "tanh", "strict"),    # the largest H1, NKC 16
    (400, 300, "tanh", "strict"),     # the bench default
    (256, 256, "gauss", "strict"),    # the SAC default
]
FP32_SHAPES = [
    (4, 1, "tanh", "strict"),          # H1 < 64: the partial heads overlay is larger than h1; one warp gets a layer-2 pass
    (8, 13, "tanh", "strict"),         # H2 not a multiple of 12: the row clamp
    (60, 12, "tanh", "strict"),
    (60, 12, "tanh", "fast"),
    (64, 191, "tanh", "strict"),       # H2 < 192: warps without a layer-2 pass
    (68, 193, "tanh", "strict"),
    (400, 300, "tanh", "strict"),
    (400, 300, "tanh", "fast"),
    (448, 300, "tanh", "strict"),      # the shared-memory limit
    (256, 1000, "tanh", "strict"),     # a large H2
    (4, 1, "gauss_clamp", "strict"),   # log_std biases +5 and -25: both clamps bind
    (68, 193, "gauss_clamp", "strict"),
]
TC_REJECTED = [(100, 50, "H1"), (1040, 16, "H1"), (16, 496, "tmem"), (160, 352, "smem"), (16, 513, "NP")]


def _ids(shapes):
    return [f"{h1}x{h2}-{kind}-{math}" for h1, h2, kind, math in shapes]


def test_tc_sweep_reaches_every_geometry_branch(pkg):
    """The sweep's coverage claim, checked against the mirror, and the mirror checked against the library's own size query."""
    geo = [tc_geometry(h1, h2) for h1, h2, _, _ in TC_SHAPES]
    assert all(isinstance(g, dict) for g in geo)
    assert {g["KC"] for g in geo} == {16, 32, 48, 64, 80}
    nkc = {g["NKC"] for g in geo}
    assert 1 in nkc and 2 in nkc and any(k >= 3 and k % 2 for k in nkc) and any(k >= 4 and k % 2 == 0 for k in nkc)
    assert {g["N1"] > 0 for g in geo} == {False, True}
    assert {g["tmem"] for g in geo} == {64, 128, 256, 512}
    assert any(g["NP"] + 2 * g["KC"] == 512 for g in geo) and any(g["NP"] < 256 for g in geo)
    assert any(g["NP"] == 256 and g["N1"] == 0 for g in geo) and any(g["NP"] != h2 for g, (_, h2, _, _) in zip(geo, TC_SHAPES))
    assert [tc_geometry(h1, h2) for h1, h2, _ in TC_REJECTED] == [why for _, _, why in TC_REJECTED]
    # the mirror agrees with make_geometry: the size query returns the W2 image size of an accepted shape and <= 0 for a rejected one
    from ctypes import byref

    lib = pkg._lib.load()
    for h1 in list(range(16, 1041, 16)) + [4, 100]:
        for h2 in (1, 20, 33, 128, 256, 257, 300, 352, 353, 384, 432, 480, 496, 513):
            probe = pkg._lib.ActorF32(W2=1, H1=h1, H2=h2, kind=pkg._lib.ACTOR_TANH)
            got, g = lib.cstr_actor_pack_bf16(byref(probe), None, None), tc_geometry(h1, h2)
            assert (got == g["bytes"]) if isinstance(g, dict) else got <= 0, (h1, h2, got, g)
            assert (pkg.rollout.actor_shape_error(h1, h2, "tc") is None) == isinstance(g, dict)


# ---- running the kernels ----------------------------------------------------------------------------------------------------------
def _weights(H1, H2, kind, seed=0):
    """torch Linear's default init U(+-1/sqrt(fan_in)), float32; the Gaussian head's W3/b3 rows are [mu_0, mu_1, log_std_0, log_std_1]."""
    rng = np.random.default_rng(seed + 7919 * H1 + H2)
    n_out = 2 if kind == "tanh" else 4

    def lin(o, i):
        k = 1.0 / np.sqrt(i)
        return rng.uniform(-k, k, (o, i)).astype(np.float32), rng.uniform(-k, k, o).astype(np.float32)

    (W1, b1), (W2, b2), (W3, b3) = lin(H1, 4), lin(H2, H1), lin(n_out, H2)
    if kind == "gauss":
        b3[2:] -= 1.0
    elif kind == "gauss_clamp":
        b3[2], b3[3] = 5.0, -25.0
    return dict(W1=W1, b1=b1, W2=W2, b2=b2, W3=W3, b3=b3)


def _env_action(buffer_action):
    f = np.float32
    return (f(-1.0) + (f(0.5) * (buffer_action + f(1.0)) * f(2.0))).astype(f)


def _start(pkg, math="strict", init_mode="random", seed=7):
    env = pkg.GpuCSTRVecEnv(N, seed=seed, math=math, init_mode=init_mode, monitor=False)
    env.reset()
    env.step_count.fill_(SC0)
    return env, _host_state(env)


def _host_state(env):
    sb = None if env.static_base is None else env.static_base.cpu().numpy().copy()
    return [env.state.cpu().numpy().copy(), env.step_count.cpu().numpy().copy(), env.episode.cpu().numpy().copy(), sb]


def _oracle_step(st, rec_k, env):
    """(c) given the stored action, next_obs, reward and done of the record are the oracle's bit for bit; then the auto-reset of the
    truncated reactors (Philox stream of their episode; static mode drifts their base).  Returns the oracle state after the step."""
    s, sc, ep, sb = st
    a_env = _env_action(rec_k[:, 8:10]) if rec_k is not None else None
    if env.math == "strict":
        nxt, r, done, sc, _ = B.step_f32(s, a_env, sc, exp_mode=B.EXP_SHARED, sq_mode=B.SQ_MUL)
    else:  # the fast vec_step runs the same step_fast_f32 as the rollout kernels
        import gpu_util

        d = gpu_util.raw_step_f32(s, a_env, sc, mode=1)
        nxt, r, done, sc = d["state"], d["reward"], d["done"], d["step_count"]
    f = np.float32
    assert np.array_equal(rec_k[:, 4:8], nxt) and np.array_equal(rec_k[:, 10], r)
    assert np.array_equal(rec_k[:, 11], done.astype(f)) and np.array_equal(rec_k[:, 12], done.astype(f))
    if done.any():
        im = 1 if env.init_mode == "static" else 0
        nxt, sc, ep, sb2 = B.reset_f32(len(s), 0, int(env._params.seed), im, episode=ep, static_base=sb, mask=done, state=nxt, step_count=sc)
        sb = sb2 if sb is not None else None
    return [nxt, sc, ep, sb]


def _check_launch(env, st, rec, reference, add):
    """Per step: (a) the record's obs is the oracle state, (b) the stored action is within the per-reactor bound of `reference`,
    (c) the step given the stored action is the oracle's; (d) after the launch the state and counters equal the composition's.
    Returns the largest |error| / bound."""
    worst = 0.0
    for k in range(rec.shape[0]):
        assert np.array_equal(rec[k, :, 0:4], st[0]), k
        a, bound = reference(st[0], k)
        want = np.clip(a + add(k), -1.0, 1.0)
        ratio = np.abs(rec[k, :, 8:10] - want) / (bound + MAPS)
        worst = max(worst, float(ratio.max()))
        assert ratio.max() <= 1.0, (k, float(ratio.max()), np.unravel_index(ratio.argmax(), ratio.shape))
        st = _oracle_step(st, rec[k], env)
    got = _host_state(env)
    for name, g, w in zip(("state", "step_count", "episode", "static_base"), got, st):
        assert (g is None and w is None) or np.array_equal(g, w), name
    return worst, st


def _collect(pkg, env, W, kind, mode, noise):
    buf = pkg.GpuReplayBuffer((K + 1) * N, device="cuda", n_envs=N)
    actor = pkg.ActorWeights(**W, kind="tanh" if kind == "tanh" else "gaussian")
    pkg.FusedRollout(env, buf, actor, sigma=0.3, actor_mode=mode).collect(noise.shape[0], noise=torch.as_tensor(noise, device="cuda"))
    torch.cuda.synchronize()
    return buf.records.cpu().numpy()[: noise.shape[0]]


def _noise(kind, seed=1, steps=K):
    z = np.random.default_rng(seed).standard_normal((steps, N, 2))
    return (z if kind != "tanh" else 0.2 * z).astype(np.float32)  # Gaussian: the actor's own eps; TD3: the exploration noise


def _sweep(pkg, mode, H1, H2, kind, math):
    W = _weights(H1, H2, kind)
    head = "tanh" if kind == "tanh" else "gauss"
    env, st = _start(pkg, math)
    noise = _noise(kind)
    rec = _collect(pkg, env, W, kind, mode, noise)
    eps = (lambda k: noise[k]) if head == "gauss" else (lambda k: None)
    add = (lambda k: noise[k]) if head == "tanh" else (lambda k: 0.0)
    ref = actor_f64 if mode == "fp32" else actor_tc_emulated
    worst, _ = _check_launch(env, st, rec, lambda s, k: ref(s, W, head, eps(k)), add)
    if mode == "tc":  # and the documented bar against the exact actor still holds
        for k in range(K):
            a, _ = actor_f64(rec[k, :, 0:4], W, head, eps(k))
            assert np.abs(rec[k, :, 8:10] - np.clip(a + add(k), -1.0, 1.0)).max() < 5e-3
    print(f"rollout {mode} {H1}x{H2} {kind} {math}: max |error| / bound = {worst:.3g}")
    return worst


@gpu
@pytest.mark.parametrize("H1,H2,kind,math", FP32_SHAPES, ids=_ids(FP32_SHAPES))
def test_fp32_actor_within_float32_bound_of_exact_actor(pkg, H1, H2, kind, math):
    _sweep(pkg, "fp32", H1, H2, kind, math)


@gpu
@pytest.mark.parametrize("H1,H2,kind,math", TC_SHAPES, ids=_ids(TC_SHAPES))
def test_tc_actor_within_accumulation_bound_of_bf16_emulation(pkg, H1, H2, kind, math):
    _sweep(pkg, "tc", H1, H2, kind, math)


@gpu
@pytest.mark.parametrize("mode", ["fp32", "tc"])
def test_static_init_mode_through_the_rollout_kernels(pkg, mode):
    """init_mode="static": every reset drifts the reactor's base state in place (quirk Q2).  The tc kernel keeps a per-thread copy of the
    base and writes it back from one thread of each reactor at the end of the launch.  Two launches, each truncating every reactor once."""
    H1, H2 = (64, 48) if mode == "fp32" else (96, 257)
    W = _weights(H1, H2, "tanh")
    ref = actor_f64 if mode == "fp32" else actor_tc_emulated
    env, st = _start(pkg, init_mode="static", seed=11)
    base0 = st[3].copy()
    for launch in range(2):
        noise = _noise("tanh", seed=launch, steps=8)
        rec = _collect(pkg, env, W, "tanh", mode, noise)
        _, st = _check_launch(env, st, rec, lambda s, k: ref(s, W, "tanh"), lambda k: noise[k])
        env.step_count.fill_(SC0)
        st[1][:] = SC0
    assert not np.array_equal(env.static_base.cpu().numpy(), base0)


@gpu
@pytest.mark.parametrize("H1,H2", [(4, 13), (60, 12)])
def test_two_agent_rollout_small_shapes(pkg, H1, H2):
    """cstr_rollout_fused_multi: agent i's actor 2 -> H1 -> H2 -> 1 on its observation slice, predict()'s unscale and nothing else (Q5)."""
    torch.manual_seed(H1)
    agents = [nn.Sequential(nn.Linear(2, H1), nn.ReLU(), nn.Linear(H1, H2), nn.ReLU(), nn.Linear(H2, 1), nn.Tanh()).cuda() for _ in range(2)]
    padded = []
    for i, m in enumerate(agents):  # the zero-padded 4 -> H1 -> H2 -> 2 actor the kernel evaluates, output i
        lin = [l for l in m if isinstance(l, nn.Linear)]
        W = {k: np.zeros(s, np.float32) for k, s in (("W1", (H1, 4)), ("b1", H1), ("W2", (H2, H1)), ("b2", H2), ("W3", (2, H2)), ("b3", 2))}
        W["W1"][:, 2 * i:2 * i + 2] = lin[0].weight.detach().cpu().numpy()
        W["b1"][:], W["W2"][:], W["b2"][:] = (t.detach().cpu().numpy() for t in (lin[0].bias, lin[1].weight, lin[1].bias))
        W["W3"][i], W["b3"][i] = lin[2].weight.detach().cpu().numpy()[0], lin[2].bias.detach().cpu().numpy()[0]
        padded.append(W)

    def reference(s, k):
        (a0, e0), (a1, e1) = (actor_f64(s, W) for W in padded)
        return np.stack([a0[:, 0], a1[:, 1]], 1), np.stack([e0[:, 0], e1[:, 1]], 1)

    env, st = _start(pkg, seed=13)
    buf = pkg.GpuReplayBuffer((K + 1) * N, device="cuda", n_envs=N)
    pkg.FusedRollout(env, buf, pkg.AgentActorWeights(agents, device="cuda")).collect(K)
    rec = buf.records.cpu().numpy()[:K]
    worst, _ = _check_launch(env, st, rec, reference, lambda k: 0.0)
    print(f"rollout multi {H1}x{H2}: max |error| / bound = {worst:.3g}")


# ---- rejected shapes ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("H1,H2,why", TC_REJECTED, ids=[f"{a}x{b}-{w}" for a, b, w in TC_REJECTED])
def test_tc_rejects_shapes_before_launch(pkg, H1, H2, why):
    W = _weights(H1, H2, "tanh")
    env, _ = _start(pkg)
    buf = pkg.GpuReplayBuffer(2 * N, device="cuda", n_envs=N)
    actor = pkg.ActorWeights(**W)
    with pytest.raises(ValueError, match="TMEM" if why in ("tmem", "NP", "smem") else "multiple of 16 and <= 1024"):
        actor.pack_bf16()
    with pytest.raises(ValueError):
        pkg.FusedRollout(env, buf, actor, actor_mode="tc")
    torch.cuda.synchronize()
    assert actor.packed_bf16 is None and buf.pos == 0 and (env.step_count == SC0).all()


@gpu
def test_fp32_rejects_shapes_before_launch(pkg):
    env, _ = _start(pkg)
    buf = pkg.GpuReplayBuffer(2 * N, device="cuda", n_envs=N)
    with pytest.raises(ValueError, match="multiple of 4"):
        pkg.ActorWeights(**_weights(30, 20, "tanh"))
    actor = pkg.ActorWeights(**_weights(452, 20, "tanh"))
    with pytest.raises(ValueError, match="H1 <= 448"):
        pkg.FusedRollout(env, buf, actor, actor_mode="fp32")
    # the library's own check, reached around the Python one: an argument error, nothing launched
    from ctypes import byref

    lib = pkg._lib.load()
    rc = lib.cstr_rollout_fused(byref(env._params), N, 1, 0, 0, byref(actor._struct), None, 0.0, None, 0, 0, env.state.data_ptr(),
                                env.step_count.data_ptr(), env.episode.data_ptr(), None, 2, 0, buf.records.data_ptr(), None, None, None)
    assert rc != 0 and b"448" in lib.cstr_last_error()
    torch.cuda.synchronize()
    assert buf.pos == 0 and (env.step_count == SC0).all()


# ---- the host guard of bind_offpolicy_rollout ---------------------------------------------------------------------------------------
class FlattenExtractor(nn.Module):  # matched by class name, as the reference's is
    pass


class NatureCNN(nn.Module):
    pass


def _mlp(sizes, act=nn.ReLU, head=nn.Tanh):
    layers = []
    for i, (a, b) in enumerate(zip(sizes[:-1], sizes[1:])):
        layers += [nn.Linear(a, b)] + ([act()] if i < len(sizes) - 2 else ([head()] if head else []))
    return nn.Sequential(*layers)


def _td3_model(arch, act=nn.ReLU, extractor=FlattenExtractor, obs=4, out=2):
    actor = SimpleNamespace(features_extractor=extractor(), mu=_mlp([obs, *arch, out], act))
    return SimpleNamespace(actor=actor, use_sde=False, _vec_normalize_env=None)


def _sac_model(arch, act=nn.ReLU, mu=None):
    trunk = _mlp([4, *arch], act, head=None)
    trunk.append(act())
    actor = SimpleNamespace(features_extractor=FlattenExtractor(), latent_pi=trunk, mu=mu if mu is not None else nn.Linear(arch[-1], 2),
                            log_std=nn.Linear(arch[-1], 2))
    return SimpleNamespace(actor=actor, use_sde=False, _vec_normalize_env=None)


def _agents_model(archs, acts=(nn.ReLU, nn.ReLU)):
    actor = SimpleNamespace(mu_list=nn.ModuleList([_mlp([2, *a, 1], act) for a, act in zip(archs, acts)]))
    return SimpleNamespace(actor=actor, use_sde=False, _vec_normalize_env=None, observation_splits=[[0, 1], [2, 3]], action_splits=[[0], [1]])


@gpu
def test_guard_sends_unsupported_actors_to_the_reference(pkg):
    env = pkg.GpuCSTRVecEnv(8, seed=0, monitor=False)
    buf = pkg.GpuReplayBuffer(64, device="cuda", n_envs=8)
    freq = SimpleNamespace(unit="step", frequency=4)

    def why(model, mode="fp32"):
        return pkg.rollout.fused_rollout_unsupported(model, env, buf, freq, None, actor_mode=mode)

    for mode in ("fp32", "tc"):
        assert why(_td3_model([400, 300]), mode) is None
        assert why(_sac_model([256, 256]), mode) is None
        assert why(_agents_model([[60, 12], [60, 12]]), mode) is None  # the agents always run on the float32 kernel
        assert "Tanh" in why(_td3_model([64, 64], act=nn.Tanh), mode)  # would silently run a ReLU actor
        assert "Linear, ReLU" in why(_td3_model([64, 64, 64]), mode)
        assert "multiple of 4" in why(_td3_model([30, 20]), mode)
        assert "NatureCNN" in why(_td3_model([64, 64], extractor=NatureCNN), mode)
        assert "not 4 -> H1 -> H2 -> 2" in why(_td3_model([64, 64], obs=5), mode)
        assert "not 4 -> H1 -> H2 -> 2" in why(_td3_model([64, 64], out=3), mode)
        assert "latent_pi" in why(_sac_model([64, 64], act=nn.ELU), mode)
        assert "single Linear" in why(_sac_model([64, 64], mu=nn.Sequential(nn.Linear(64, 2))), mode)
        assert "agent 1" in why(_agents_model([[60, 12], [60, 12]], acts=(nn.ReLU, nn.Tanh)), mode)
        assert "differ" in why(_agents_model([[60, 12], [64, 12]]), mode)
        assert "H1 <= 448" in why(_agents_model([[452, 12], [452, 12]]), mode)
    assert why(_td3_model([448, 300])) is None and "H1 <= 448" in why(_td3_model([512, 512]))
    assert why(_td3_model([100, 52])) is None and "multiple of 16" in why(_td3_model([100, 52]), "tc")
    for h1, h2, _ in TC_REJECTED[1:]:
        assert why(_td3_model([h1, h2]), "tc") is not None
    assert why(_td3_model([1024, 256]), "tc") is None and why(_td3_model([16, 480]), "tc") is None


@gpu
@pytest.mark.skipif(not refload.available(), reason="reference tree not available")
def test_learn_with_a_tanh_actor_runs_the_reference_rollout(pkg):
    """bind_offpolicy_rollout(core.TD3) with activation_fn=nn.Tanh: the kernel's actor is ReLU, so learn() must warn and run the reference's
    own collect_rollouts, and the stored actions are that actor's."""
    refload.install_shims()
    core = refload.load_core()
    from core.common.buffers import ReplayBuffer
    from core.common.vec_env import VecEnv

    n = 16
    env = pkg.bind_vec_env_class(VecEnv)(num_envs=n, init_mode="random", reset_rng="philox", seed=3)
    model = pkg.bind_offpolicy_rollout(core.TD3)("MlpPolicy", env, policy_kwargs=dict(activation_fn=nn.Tanh), device="cuda",
                                                 replay_buffer_class=pkg.bind_replay_buffer_class(ReplayBuffer), buffer_size=64 * n,
                                                 learning_starts=0, train_freq=(2, "step"), gradient_steps=0, seed=0, verbose=0)
    with pytest.warns(RuntimeWarning, match="fused rollout not used.*Tanh"):
        model.learn(total_timesteps=4 * n, log_interval=None)
    assert model.fused_rollout_launches == 0
    rec = model.replay_buffer.records[:4].reshape(-1, model.replay_buffer.records.shape[-1])
    with torch.no_grad():
        mu = model.actor(rec[:, 0:4].to(model.device)).cpu().numpy()
    np.testing.assert_allclose(rec[:, 8:10].cpu().numpy(), mu, rtol=0, atol=3e-6)
