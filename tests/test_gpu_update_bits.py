"""Bit pins of the five fused update engines: TD3 (two critics and one), SAC, BCQ and MADDPG / IDDPG, in all three GEMM modes.

Each case loads seeded random nets, then runs
  * launch-by-launch ``update()`` calls that include critic-only and policy steps (Philox draws inside the kernels),
  * one ``update()`` with a no-op ``allreduce`` hook, which runs the split-phase path (TD3 and SAC; for SAC it takes
    ``sac_ent_coef_kernel``'s modes 1 and 2 instead of 3),
  * ``train(..., graph=True)`` on a full Philox-index buffer: captured cycles, ``td3_tick_kernel`` and the device scalars,
and hashes ``params``, ``targets``, ``grads``, ``adam_m``, ``adam_v``, the losses and the step counters.

The digests below were produced on a B200 by the build of commit 6722f69, before the host code that chains the update kernels was
folded into shared helpers.  That change keeps every launch, argument and summation order, so the outputs must stay identical byte
for byte.  The split-K and slab-count choices depend on the SM count, so the pins hold on a 148-SM device only.
``python tests/test_gpu_update_bits.py`` prints the digests of the current build.
"""
import hashlib
import importlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import td3_util as TU  # noqa: E402

MODES = ("fp32", "tensor", "bf16")
CASES = ("td3_400x300_b256", "td3_36x20_b37", "ddpg_400x300_b256", "sac_256x256_b256", "bcq_defaults_b256", "maddpg_nc2_b256", "iddpg_nc1_b256")

EXPECTED = {
    "td3_400x300_b256_fp32": "53fe3f18302277e0d8393ec7aafffb78733e1698f62ae2d36ec0a8419d31c602",
    "td3_400x300_b256_tensor": "b432be86156ceaa05cb6f014fba5ed9d1c9ca11e7391372dce8c61254b45b33e",
    "td3_400x300_b256_bf16": "67e9c01ce4e1a351f04c9aaff66bcb6e3e034cd32a4b55f8b1d28cde0d63f2a2",
    "td3_36x20_b37_fp32": "cae669c5d8122b64c6f72c5dc531766f74f57cf5c59c4924ff292755e37861ea",
    "td3_36x20_b37_tensor": "1b5cc416dcadb5a3b39061aafbc151161e7a0d4a0be322585d55077346dc0933",
    "td3_36x20_b37_bf16": "1aaba8e010069a7bce9abe53d52452bc2b1e3480b1f9f206246d78f92e75ab76",
    "ddpg_400x300_b256_fp32": "f336b1b95d70a696b64e40bbf99f9758f0f5f6359d394c0e6183c393436019ca",
    "ddpg_400x300_b256_tensor": "74b9d15ddaca064c3fdac55dd78a86b27e96ec4cf9e0002e12f8ef26e3ac9e18",
    "ddpg_400x300_b256_bf16": "e66979d1fb44f3a072c0ca7940410cdf4ea38c41dda2a4a24b8b477dfae634d3",
    "sac_256x256_b256_fp32": "2b234511862707744f289da24768d7077aa0addd2d6c72b9fcc31dd211e5020c",
    "sac_256x256_b256_tensor": "dad8f725b13e3da3fb472d1c56cd29925db2ea3ca1252f72482d34299dd2c2d4",
    "sac_256x256_b256_bf16": "c4e2d0ce959ccc1dd5cd4533e22df88d970b48afa0322fea1538c9e030340df6",
    "bcq_defaults_b256_fp32": "bf63f2fa94e03058f956fed1eab029cef2a7ed9c47097d0688eb1d6d422ef82c",
    "bcq_defaults_b256_tensor": "ec5892302efdf4da237f304c4cbdf3feb462a69e89b53308b4c597e7180f8644",
    "bcq_defaults_b256_bf16": "96b8f610342e13b2f6f3573b67bb3d25fb8fda308d58019c48023b75ac2d424a",
    "maddpg_nc2_b256_fp32": "bdcc2f8489ae8ead63577402844419161aab5faa716006242a6115bce46ec3e1",
    "maddpg_nc2_b256_tensor": "b2b8972d8309fe77b610635c70d108b1bb557e518285550a16483be2595f85df",
    "maddpg_nc2_b256_bf16": "af8d1f3a9d69b73b426a81904b122666483283df9ecb6eb728de525587ce741a",
    "iddpg_nc1_b256_fp32": "fdfe53525010c021d6bdcf4a07c89ed039b64ed02e5a0a1fc961ba0ed82a6675",
    "iddpg_nc1_b256_tensor": "286c1a1b2ae60fb200c6cb9e9c86cbcde6bf62c42ae94d7138fad6341189f531",
    "iddpg_nc1_b256_bf16": "f5285e17b021000bddd5cff2b40279ec4f1a5ffec08e57f91e22db66064613bc",
}


def _mlp(rng, i, h1, h2, o):
    out = []
    for fi, fo in ((i, h1), (h1, h2), (h2, o)):
        b = 1.0 / np.sqrt(fi)
        out += [rng.uniform(-b, b, (fo, fi)).astype(np.float32), rng.uniform(-b, b, fo).astype(np.float32)]
    return out


def _batch(rng, B):
    return (rng.uniform(-1, 1, (B, 4)).astype(np.float32), rng.uniform(-1, 1, (B, 2)).astype(np.float32), rng.uniform(-1, 1, (B, 4)).astype(np.float32),
            (rng.random((B, 1)) < 0.1).astype(np.float32), rng.normal(size=(B, 1)).astype(np.float32))


def _engine(pkg, case, mode, rng):
    """(engine, batch size, whether update() takes an allreduce hook)"""
    if case.startswith(("td3", "ddpg")):
        arch, B = ([36, 20], 37) if case == "td3_36x20_b37" else ([400, 300], 256)
        eng = pkg.FusedTD3Update(arch, B, gemm=mode, seed=5, n_critics=1 if case.startswith("ddpg") else 2)
        eng.load_nets(TU.random_nets(rng, *arch))
        return eng, B, True
    if case.startswith("sac"):
        eng = pkg.FusedSACUpdate([256, 256], 256, gemm=mode, seed=5, ent_coef_init=0.7)
        eng.load_nets(TU.random_sac_nets(rng, 256, 256))
        return eng, 256, True
    if case.startswith("bcq"):
        L, Hv, Hp = 32, 64, 64
        eng = pkg.FusedBCQUpdate(L, Hv, Hp, [400, 300], 256, gemm=mode, seed=5)
        eng.load_nets({"vae_enc": _mlp(rng, 6, Hv, Hv, 2 * L), "vae_dec": _mlp(rng, 4 + L, Hv, Hv, 2), "pert": _mlp(rng, 6, Hp, Hp, 2),
                       "critic0": _mlp(rng, 6, 400, 300, 1), "critic1": _mlp(rng, 6, 400, 300, 1)})
        return eng, 256, False
    centralised, nc = case.startswith("maddpg"), 2 if "nc2" in case else 1
    # unequal rates: each agent's optimisers read their own device scalar slots
    eng = pkg.FusedMultiAgentUpdate([400, 300], 256, centralised, gemm=mode, seed=5, n_critics=nc, actor_lrs=[1e-3, 4e-4], critic_lrs=[7e-4, 2e-4])
    ci = 6 if centralised else 3
    eng.load_nets({n: _mlp(rng, 2 if n.startswith("actor") else ci, 400, 300, 1) for n in eng.NETS})
    return eng, 256, False


def _losses(eng):
    out = []
    for x in eng.pop_losses():
        for y in (x if isinstance(x, (tuple, list)) else (x,)):
            out.append(np.nan if y is None else y)
    return np.asarray(out, np.float64)


def run_case(pkg, torch, case, mode, buf):
    rng = np.random.default_rng(CASES.index(case) * 10 + MODES.index(mode))
    eng, B, hook = _engine(pkg, case, mode, rng)
    for _ in range(3):  # updates 1-3: critic-only and policy steps (policy_delay / actor_delay 2)
        eng.update(_batch(rng, B))
    if hook:
        eng.update(_batch(rng, B), allreduce=lambda t: None)
    else:
        eng.update(_batch(rng, B))
    parts = [_losses(eng)]
    buf._draw = 0
    eng.train(4, buf, B, graph=True)
    assert eng._graph is not None
    torch.cuda.synchronize()
    parts += [eng.params, eng.targets, eng.grads, eng.adam_m, eng.adam_v, eng._counters, _losses(eng),
              np.asarray([eng.n_updates, eng.critic_step, eng.actor_step], np.int64)]
    h = hashlib.sha256()
    for a in parts:
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def run_cases():
    import torch

    pkg = importlib.import_module("pytorch-rl-enhancedstablebaselines_b200")
    n_envs = 512
    buf = pkg.GpuReplayBuffer(32 * n_envs, device="cuda:0", n_envs=n_envs, index_mode="philox", seed=5)
    g = torch.Generator(device="cuda:0").manual_seed(20261020)
    buf.records.uniform_(-1, 1, generator=g)
    buf.records[..., 11:13] = 0
    buf.pos, buf.full = 0, True
    return {f"{case}_{mode}": run_case(pkg, torch, case, mode, buf) for case in CASES for mode in MODES}


def _sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 0


@pytest.mark.gpu
def test_update_engines_bit_identical_to_pinned_digests():
    if _sms() != 148:
        pytest.skip("the pinned digests are of a 148-SM B200 (split-K and slab counts follow the SM count)")
    got = run_cases()
    assert set(got) == set(EXPECTED)
    bad = {k: (got[k], EXPECTED[k]) for k in EXPECTED if got[k] != EXPECTED[k]}
    assert not bad, f"outputs changed (got, pinned): {bad}"


if __name__ == "__main__":
    print(json.dumps(run_cases(), indent=1))
