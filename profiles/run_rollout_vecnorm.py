"""The fused rollout with and without GpuVecNormalize(training=True): TD3 actor 4-400-300-2, K = 16 env steps per collect() (the bench's
`rollout` section), tc and fp32 actors, 131,072 and 1,048,576 reactors.  The two variants alternate three times on the same env and buffer;
the number per variant is the median of the three.  One collect() of each variant runs under torch.profiler to list its kernel launches.
Usage: python profiles/run_rollout_vecnorm.py [--out FILE] [--sizes 131072,1048576] [--collects 4]"""
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


def time_collects(roll, collects):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(collects):
        roll.collect(K)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / collects


def kernel_list(roll):
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        roll.collect(K)
        torch.cuda.synchronize()
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        if ev.count and t:
            rows.append({"kernel": ev.key[:120], "launches": ev.count, "device_us": round(t, 1)})
    return sorted(rows, key=lambda r: -r["device_us"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="131072,1048576")
    ap.add_argument("--collects", type=int, default=4)
    args = ap.parse_args()
    torch.manual_seed(0)
    lin = [torch.nn.Linear(4, 400), torch.nn.Linear(400, 300), torch.nn.Linear(300, 2)]
    actor = pkg.ActorWeights(lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, lin[2].weight, lin[2].bias)
    result = {"card": card(), "K": K, "actor": "4-400-300-2", "runs": []}
    for n in (int(s) for s in args.sizes.split(",")):
        env = pkg.GpuCSTRVecEnv(n, seed=1, monitor=False)
        env.reset()
        vn = pkg.GpuVecNormalize(env, training=True)
        vn.reset()
        buf = pkg.GpuReplayBuffer(2 * K * n, n_envs=n)
        for mode in ("tc", "fp32"):
            rolls = {"plain": pkg.FusedRollout(env, buf, actor, sigma=0.1, actor_mode=mode),
                     "vecnorm": pkg.FusedRollout(env, buf, actor, sigma=0.1, actor_mode=mode, vec_normalize=vn)}
            for r in rolls.values():  # warm-up: module load, smem attributes, first touch of the ring
                r.collect(K)
                r.collect(K)
            ms = {v: [] for v in rolls}
            for _ in range(3):
                for v, r in rolls.items():
                    ms[v].append(time_collects(r, args.collects))
            row = {"n": n, "actor_mode": mode}
            for v in rolls:
                med = statistics.median(ms[v])
                row[v] = {"ms_per_collect": [round(x, 3) for x in ms[v]], "median_ms": round(med, 3), "transitions_per_s": n * K / (med * 1e-3)}
            row["vecnorm_over_plain"] = round(row["vecnorm"]["transitions_per_s"] / row["plain"]["transitions_per_s"], 3)
            if mode == "tc" and n == max(int(s) for s in args.sizes.split(",")):
                row["kernels_one_collect"] = {v: kernel_list(r) for v, r in rolls.items()}
            print(json.dumps({k: row[k] for k in ("n", "actor_mode", "vecnorm_over_plain")} | {v: row[v]["median_ms"] for v in rolls}), flush=True)
            result["runs"].append(row)
        del env, vn, buf, rolls
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
