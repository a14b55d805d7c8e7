"""The float32 fused rollout of the SAC actor 4-256-256 with gSDE (use_sde=True) against the plain squashed-Gaussian actor: K = 16 env steps
per collect(), 131,072 and 1,048,576 reactors.  "sde" times collect() alone on fixed exploration matrices; "sde_reset" adds the reset_noise()
that bind_offpolicy_rollout runs at the start of every collect_rollouts call (sde_sample_freq = -1, the reference's default).  The variants
alternate three times on the same env and buffer; the number per variant is the median of the three.  One collect() of each variant at the
largest size runs under torch.profiler to list its kernel launches.  Then the SAC update 4-256-256 (graph replay, batch 256 and 4096),
plain against gSDE, alternated three times: milliseconds per update, median of the three.
Usage: python profiles/run_sac_sde.py [--out FILE] [--sizes 131072,1048576] [--collects 4]"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

pkg = importlib.import_module("pytorch-rl-enhancedstablebaselines_b200")
K = 16


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60).stdout.strip().splitlines()[0]
        out["nvidia_smi"] = q
    except Exception as exc:  # the number still stands with the device name; say why the power limit is missing
        out["nvidia_smi_error"] = repr(exc)
    return out


def time_collects(roll, collects, reset=False):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(collects):
        if reset:
            roll.reset_noise()
        roll.collect(K)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / collects


def kernel_list(roll, reset=False):
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        if reset:
            roll.reset_noise()
        roll.collect(K)
        torch.cuda.synchronize()
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        if ev.count and t:
            rows.append({"kernel": ev.key[:120], "launches": ev.count, "device_us": round(t, 1)})
    return sorted(rows, key=lambda r: -r["device_us"])


def time_updates(steps=200):
    n_envs = 4096
    buf = pkg.GpuReplayBuffer(64 * n_envs, n_envs=n_envs, index_mode="philox", seed=5)
    buf.records.uniform_(-1, 1)
    buf.records[..., 11:13] = 0
    buf.pos, buf.full = 0, True
    rows = []
    for batch in (256, 4096):
        engs = {"plain": pkg.FusedSACUpdate([256, 256], batch, seed=2), "sde": pkg.FusedSACUpdate([256, 256], batch, seed=2, sde=True)}
        for e in engs.values():
            e.train(20, buf, batch, graph=True)  # capture + warm-up
        ms = {v: [] for v in engs}
        for _ in range(3):
            for v, e in engs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                e.train(steps, buf, batch, graph=True)
                e1.record()
                e1.synchronize()
                ms[v].append(e0.elapsed_time(e1) / steps)
        row = {"batch": batch, **{v: {"ms_per_update": [round(x, 4) for x in ms[v]], "median_ms": round(statistics.median(ms[v]), 4)} for v in engs}}
        row["sde_over_plain"] = round(row["sde"]["median_ms"] / row["plain"]["median_ms"], 3)
        print(json.dumps({"batch": batch, "sde_over_plain": row["sde_over_plain"], "plain": row["plain"]["median_ms"], "sde": row["sde"]["median_ms"]}),
              flush=True)
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="131072,1048576")
    ap.add_argument("--collects", type=int, default=4)
    args = ap.parse_args()
    torch.manual_seed(0)
    trunk = torch.nn.Sequential(torch.nn.Linear(4, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU())
    mu, log_std_head = torch.nn.Linear(256, 2), torch.nn.Linear(256, 2)
    gauss = pkg.ActorWeights.from_sac_actor(trunk, mu, log_std_head)
    sde = pkg.ActorWeights.from_sac_actor(trunk, torch.nn.Sequential(mu, torch.nn.Hardtanh(-2.0, 2.0)), torch.nn.Parameter(torch.full((256, 2), -3.0)))
    sizes = [int(s) for s in args.sizes.split(",")]
    result = {"card": card(), "K": K, "actor": "SAC 4-256-256, fp32 rollout kernel", "runs": []}
    for n in sizes:
        env = pkg.GpuCSTRVecEnv(n, seed=1, monitor=False)
        env.reset()
        buf = pkg.GpuReplayBuffer(2 * K * n, n_envs=n)
        rolls = {"plain": pkg.FusedRollout(env, buf, gauss, actor_mode="fp32"), "sde": pkg.FusedRollout(env, buf, sde, actor_mode="fp32")}
        rolls["sde"].reset_noise()
        variants = {"plain": (rolls["plain"], False), "sde": (rolls["sde"], False), "sde_reset": (rolls["sde"], True)}
        for r, reset in variants.values():  # warm-up: module load, smem attributes, first touch of the ring and of the matrices
            time_collects(r, 2, reset)
        ms = {v: [] for v in variants}
        for _ in range(3):
            for v, (r, reset) in variants.items():
                ms[v].append(time_collects(r, args.collects, reset))
        row = {"n": n}
        for v in variants:
            med = statistics.median(ms[v])
            row[v] = {"ms_per_collect": [round(x, 3) for x in ms[v]], "median_ms": round(med, 3), "transitions_per_s": n * K / (med * 1e-3)}
        for v in ("sde", "sde_reset"):
            row[v + "_over_plain"] = round(row[v]["transitions_per_s"] / row["plain"]["transitions_per_s"], 3)
        if n == max(sizes):
            row["kernels_one_collect"] = {v: kernel_list(r, reset) for v, (r, reset) in variants.items()}
        print(json.dumps({k: row[k] for k in ("n", "sde_over_plain", "sde_reset_over_plain")} | {v: row[v]["median_ms"] for v in variants}), flush=True)
        result["runs"].append(row)
        del env, buf, rolls, variants
        torch.cuda.empty_cache()
    result["update"] = time_updates()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
