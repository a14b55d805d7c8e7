#!/usr/bin/env python
"""bench.py — CSTR env-steps/s on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--math strict|fast] [--dump-outputs DIR]

Workload at N=1 = BASELINE.json configs[1]: "TwoSeriesCSTR step-only, 65,536 batched envs, random
actions, fp32", one *step* = one pass of the hot path over one batch = ONE launch of the tape kernel
integrating 400 control intervals (a full episode incl. the truncation/auto-reset row) for 65,536
reactors = 26,214,400 env-steps, actions streamed from a (400, 65536, 2) float32 tape resident in HBM
(210 MB > the 126 MB L2, so every step reads its inputs from DRAM; no L2 flush needed).
N>1: one process per GPU (torchrun), every rank owns its own 65,536-reactor shard (weak scaling, no
data-path collective — reactors are independent); time = max over ranks.

Keys beyond the base contract:
  roofline     dominant kernel (tape_f32) against the FP32 pipe peak MEASURED in this run by an FMA-chain
               probe (MEASURED_PEAKS.json has no non-tensor peak): achieved = 176 flop/env-step (SURVEY 8d)
               x env-steps per launch / CUDA-event duration.
  cpu_baseline the oracle's C port (oracle/cstr_oracle.c, OpenMP, all host cores) on a bounded sample.
  e2e          same metric through the C-ABI call with HOST (pinned) buffers: H2D of the action tape and
               state, the kernel, D2H of rewards/dones/state, all inside the timed region.
  rollout      the other half of BASELINE's metric, at every N: fused-rollout transitions/s (config #3, tcgen05 actor), 1,048,576
               reactors sharded over the N ranks (strong) and 131,072 per rank (weak).
  dp_update    the only collective of the path, at every N: the TD3 gradient step data-parallel over the ranks (ms per update, max over
               ranks) — gradient mean inside the Adam kernels over NVLink peer memory, replayed from one CUDA graph, beside eager NCCL.
  extras       other variants (strict math, fp64, in-kernel Philox actions, VecEnv.step loop, replay GB/s, fused rollout, TD3 / SAC /
               BCQ / MADDPG update timings) — reported, not the headline; N=1 only.
  config / run `config` is the workload and is the same dictionary in both arms; `run` holds what varies with the run (math flavour,
               per-rank times, host placement).

--dump-outputs DIR writes what the last timed step returned (rewards, dones, final state, step and episode counters) for a fixed, seeded
sample of 8,192 reactors over all ranks as DIR/<name>.npy: all inputs are seeded, so two builds can be compared output for output.

Order: headline -> e2e -> cpu_baseline -> [hard stop armed] rollout / dp_update -> extras -> the ONE JSON line.  The optional sections
run under a hard stop (CSTR_BENCH_SECTION_LIMIT_S, default 300 s): if one of them hangs, rank 0 prints the line it already has (plus
"sections_timeout_s") and every rank leaves with exit code 0 — a wedged collective must not cost the headline.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_ENVS = 65_536
T_STEPS = 400
FLOP_PER_ENV_STEP = 176  # SURVEY.md 8d: 172 add/mul/div/min/max/abs/cmp + 4 exp, no FMA credit
METRIC = "CSTR env-steps/sec (TwoSeriesCSTR step-only, 65,536 batched envs per GPU, random actions)"
UNIT = "env-steps/s"


def workload_config(n_gpus: int) -> dict:
    """The workload both arms run and report under ``config`` — identical dictionaries, so the driver's config comparison of the two
    arms compares like with like; everything that varies with the run (math flavour, per-rank times, the reference arm's bounded sample)
    is reported under ``run`` / ``cpu_baseline.sample`` instead."""
    return {"workload": "TwoSeriesCSTR step-only, 65,536 batched envs, random actions, fp32 (BASELINE.json configs[1])",
            "n_envs_per_gpu": N_ENVS, "control_intervals_per_step": T_STEPS, "env_steps_per_step_per_gpu": N_ENVS * T_STEPS,
            "actions": "U(-1,1) float32 tape (400,65536,2)", "outputs_per_interval": "reward f32 + done u8",
            "parallelism": f"env-shard x{n_gpus}"}


# ------------------------------------------------------------------------------------------------------
# host placement and the hard stop of the optional sections
# ------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(torch, local_rank: int) -> dict:
    """N>1: run this rank on the host cores of the NUMA node its GPU hangs off, BEFORE the pinned buffers of the e2e leg are allocated
    (first touch puts them on that node).  Round 1: every rank sat on node 0, the ranks of the far socket pulled their 211 MB action
    tape across the socket link, and e2e scaled at 0.24 on 8 GPUs.  Pure host placement; any failure leaves the process as it was."""
    info = {"bound": False}
    try:
        props = torch.cuda.get_device_properties(local_rank)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        info["gpu_pci"] = bdf
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as fh:
            node = int(fh.read().strip())
        info["numa_node"] = node
        if node < 0:
            info["note"] = "the platform reports no NUMA node for this GPU"
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            info["note"] = "none of the node's cores is in this process's affinity mask"
            return info
        os.sched_setaffinity(0, allowed)
        info.update(bound=True, cores=len(allowed))
    except Exception as exc:  # placement is an optimisation, never a failure
        info["note"] = f"not bound: {exc!r}"
    return info


FAILED_SECTIONS = []  # the exceptions of failed sections, kept until the process leaves (describe_error)


def describe_error(exc: BaseException) -> str:
    """repr(exc) plus the innermost frames, so that an error key in the JSON line says where it happened.  The exception is kept in
    FAILED_SECTIONS: its traceback holds the failed section's frames and with them its tensors.  Dropping it would free them, and after a
    device error that free can abort the process (a pinned host buffer used in a non_blocking copy records a CUDA event when it is freed;
    with the error pending the record throws inside a destructor) before the JSON line is printed.  run_ours leaves through os._exit once
    a section has failed, so they are never freed."""
    import traceback

    FAILED_SECTIONS.append(exc)
    frames = traceback.extract_tb(exc.__traceback__)[-3:]
    return repr(exc) + " @ " + " <- ".join(f"{os.path.basename(f.filename)}:{f.lineno}" for f in reversed(frames))


class HardStop:
    """The headline numbers are final before the optional sections (multi-rank rollout / data-parallel update, extras) start.  If those
    sections hang — a rank lost in a collective, a wedged kernel — every rank's timer fires after ``seconds``: rank 0 prints the line it
    already has (with ``sections_timeout_s``), and the process leaves with exit code 0 instead of holding the box until an outer limit
    kills the whole run and the headline with it."""

    def __init__(self, seconds: float, rank: int):
        self.seconds, self.rank, self.line, self.emitted, self.lock = seconds, rank, None, False, threading.Lock()
        self.timer = threading.Timer(seconds, self._fire)
        self.timer.daemon = True

    def start(self, line) -> None:
        self.line = line
        self.timer.start()

    def emit(self, line) -> None:
        with self.lock:
            if not self.emitted and self.rank == 0:
                print(json.dumps(line), flush=True)
            self.emitted = True

    def _fire(self) -> None:
        try:
            if self.line is not None:
                self.line["sections_timeout_s"] = self.seconds
                self.emit(self.line)
            sys.stdout.flush()
        finally:
            os._exit(0)

    def cancel(self) -> None:
        self.timer.cancel()


# ------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks DURING the timed region")
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index, self.rows, self.proc, self.thread = gpu_index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15 and len(r) >= 9] or [r for (_, r) in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "no samples"}
        sm = [float(r[1]) for r in rows]
        reasons = set()
        for r in rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        power = [float(r[3]) for r in rows if r[3].replace(".", "", 1).isdigit()]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons), "samples": len(rows),
                "power_w_max": max(power) if power else None}


# ------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle's C port on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_port_rate(n_envs: int, target_seconds: float, seed: int = 0):
    """env-steps/s of oracle/cstr_oracle.c (libm exp, powf: the faithful scalar port; OpenMP all cores)
    on a bounded sample of the workload: n_envs reactors x T_cpu control intervals."""
    import numpy as np

    import build_oracle as B

    B.use_all_cores()
    rng = np.random.default_rng(seed)
    st, sc, ep, _ = B.reset_f32(n_envs, 0, seed, 0)
    cal_T = 8
    acts = rng.uniform(-1, 1, (cal_T, n_envs, 2)).astype(np.float32)
    B.tape_f32(st, sc, ep, acts, 0, seed, 0, want_rewards=False, want_dones=False)  # warm-up (page-in, thread pool)
    t0 = time.perf_counter()
    B.tape_f32(st, sc, ep, acts, 0, seed, 0, want_rewards=True, want_dones=True)
    dt = time.perf_counter() - t0
    rate = cal_T * n_envs / dt
    T_cpu = int(max(16, min(T_STEPS, target_seconds * rate / n_envs)))
    acts = rng.uniform(-1, 1, (T_cpu, n_envs, 2)).astype(np.float32)
    passes, dt = 0, 0.0
    while dt < target_seconds and passes < 4096:  # repeat the T_cpu-interval pass until ~target_seconds of CPU work has been timed
        t0 = time.perf_counter()
        B.tape_f32(st, sc, ep, acts, 0, seed, 0, want_rewards=True, want_dones=True)
        dt += time.perf_counter() - t0
        passes += 1
    return passes * T_cpu * n_envs / dt, T_cpu * passes, B.num_threads(), dt


def reference_python_rates(budget_s: float = 24.0) -> dict:
    """The UNMODIFIED reference (pure Python) timed on this box's host cores, when its tree is available (oracle/refload.py: CSTR_REFERENCE_ROOT, or
    a git-ignored copy in oracle/_ref or baseline/_ref): BASELINE.md §3's C1 / C2 / C4 / C5.  Reported beside the C port, never
    as the arm's value: the port is the strongest CPU statement of the same arithmetic, the Python original is what a user of the reference
    actually runs.  Bounded to ~budget_s seconds in total."""
    import numpy as np

    import refload

    if not refload.available():
        return {"unavailable": "reference tree not available (CSTR_REFERENCE_ROOT, oracle/_ref or baseline/_ref)"}
    out = {"cpu_count": os.cpu_count(), "reference_root": "staged copy" if os.path.basename(refload.reference_root()) == "_ref" else "in place"}
    try:
        refload.install_shims()
        core = refload.load_core()
        env_mod = refload.load_env_module()
        from core.common.noise import NormalActionNoise
        from core.common.vec_env import DummyVecEnv, SubprocVecEnv

        import torch

        share = budget_s / 4.0
        torch.set_num_threads(max(1, min(os.cpu_count() or 1, 8)))
        out["torch_threads"] = torch.get_num_threads()

        def step_rate(venv, seconds):
            venv.reset()
            n = venv.num_envs
            acts = np.random.default_rng(0).uniform(-1, 1, (64, n, 2)).astype(np.float32)
            for t in range(3):
                venv.step(acts[t])
            t0, k = time.perf_counter(), 0
            while time.perf_counter() - t0 < seconds:
                venv.step(acts[k % 64])
                k += 1
            return k * n / (time.perf_counter() - t0)

        # C1: DummyVecEnv of 64 unmodified TwoSeriesCSTREnv, one core (dummy_vec_env.py:56-73)
        venv = DummyVecEnv([lambda: env_mod.TwoSeriesCSTREnv() for _ in range(64)])
        out["dummy_vec_env_64_envs_1_core_env_steps_per_s"] = step_rate(venv, share)
        venv.close()
        # C4: the reference's rollout loop (collect_rollouts + _store_transition + ReplayBuffer.add), TD3 actor on the CPU, 16 envs, no training
        venv = DummyVecEnv([lambda: env_mod.TwoSeriesCSTREnv() for _ in range(16)])
        noise = NormalActionNoise(mean=np.zeros(2), sigma=0.1 * np.ones(2))
        model = core.TD3("MlpPolicy", venv, action_noise=noise, learning_starts=0, train_freq=(1, "step"), gradient_steps=0, buffer_size=100_000,
                         device="cpu", seed=0, verbose=0)
        model.learn(total_timesteps=16 * 8)

        def best_window(fn, units, seconds, windows=3):  # the best of a few windows: host cores of a shared box are noisy, be fair to the reference
            best = 0.0
            for _ in range(windows):
                t0, k = time.perf_counter(), 0
                while time.perf_counter() - t0 < seconds / windows:
                    fn()
                    k += units
                best = max(best, k / (time.perf_counter() - t0))
            return best

        out["collect_rollouts_16_envs_transitions_per_s"] = best_window(lambda: model.learn(total_timesteps=16 * 40, reset_num_timesteps=False), 16 * 40, share)
        # C5: TD3.train on the CPU, batch 256 (td3.py:154-211)
        model.train(gradient_steps=2, batch_size=256)
        out["td3_train_batch_256_updates_per_s"] = best_window(lambda: model.train(gradient_steps=4, batch_size=256), 4, share)
        venv.close()
        # C2: SubprocVecEnv (subproc_vec_env.py:79-221), one env per worker process, one worker per host core (last: it forks)
        try:
            workers = max(2, min(os.cpu_count() or 2, 64))
            venv = SubprocVecEnv([lambda: env_mod.TwoSeriesCSTREnv() for _ in range(workers)], start_method="fork")
            out["subproc_vec_env_workers"] = workers
            out["subproc_vec_env_env_steps_per_s"] = step_rate(venv, share)
            venv.close()
        except Exception as exc:
            out["subproc_vec_env_env_steps_per_s"] = f"failed: {exc!r}"
    except Exception as exc:
        out["error"] = repr(exc)
    return out


def run_reference_arm(args) -> None:
    """--impl reference: the reference's CPU implementation of the path, timed on this box's host cores.
    The reference is pure Python — there is nothing to compile into oracle/_ref — so the arm's value is the oracle's C port of it
    (kind "port", all host threads), a far stronger baseline than the Python original; the original itself (DummyVecEnv, SubprocVecEnv,
    collect_rollouts, TD3.train) is timed beside it when the tree is staged (reference_python)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np

    import build_oracle as B

    ref_python = reference_python_rates() if not args.no_extras else None  # before the OpenMP pool of the C port exists (thread oversubscription)
    B.use_all_cores()  # torchrun sets OMP_NUM_THREADS=1; the reference arm uses every host core
    rng = np.random.default_rng(0)
    st, sc, ep, _ = B.reset_f32(N_ENVS, 0, 0, 0)
    # size one step to ~2 s of CPU work so that K+W steps finish within a few minutes
    cal = rng.uniform(-1, 1, (4, N_ENVS, 2)).astype(np.float32)
    B.tape_f32(st, sc, ep, cal, 0, 0, 0)
    t0 = time.perf_counter()
    B.tape_f32(st, sc, ep, cal, 0, 0, 0)
    rate = 4 * N_ENVS / (time.perf_counter() - t0)
    per_step_budget = min(2.0, 150.0 / max(1, args.steps + args.warmup))
    T_ref = int(max(4, min(T_STEPS, per_step_budget * rate / N_ENVS)))
    acts = rng.uniform(-1, 1, (T_ref, N_ENVS, 2)).astype(np.float32)
    state = dict(state=st, step_count=sc, episode=ep)

    def one():
        r = B.tape_f32(state["state"], state["step_count"], state["episode"], acts, 0, 0, 0, want_rewards=True, want_dones=True)
        state.update(state=r["state"], step_count=r["step_count"], episode=r["episode"])

    for _ in range(args.warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one()
    dt = time.perf_counter() - t0
    value = args.steps * T_ref * N_ENVS / dt
    sample = f"{N_ENVS} reactors x {T_ref} control intervals per step (of the arm's 400), float32, libm expf/powf, OpenMP"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "run": {"control_intervals_per_step_timed": T_ref,
                "note": "the reference is pure Python (nothing to compile into oracle/_ref); the arm's value is its C port (oracle/cstr_oracle.c, strict "
                        "float32 arithmetic with libm expf/powf as NumPy evaluates the reference, all host threads); a step is a bounded sample of the "
                        "workload when the host cannot finish 400 intervals in ~2 s; the unmodified Python original is timed beside it under "
                        "reference_python when its tree is staged"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": B.num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "reference_python": ref_python,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def measure_pipe_peaks(pkg, torch, device) -> dict:
    """FMA-chain probes (cstr_probe_pipe): fp32 FFMA, fp64 DFMA, fp32 FMUL+FADD pairs, MUFU.EX2."""
    lib = pkg._lib.load()
    info = [__import__("ctypes").c_int() for _ in range(4)]
    lib.cstr_device_info(*[__import__("ctypes").byref(x) for x in info])
    sms = info[0].value
    grid, block, iters = sms * 16, 256, 4096
    out = torch.empty(grid * block, dtype=torch.float32, device=device)
    res = {"sm_count": sms}
    stream = torch.cuda.current_stream(device).cuda_stream
    for kind, name, flop in ((0, "fp32_ffma_tflops", 2), (1, "fp64_dfma_tflops", 2), (2, "fp32_fmul_fadd_tflops", 2), (3, "mufu_ex2_tops", 1)):
        best, mhz = 0.0, None
        for rep in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pkg._lib.check(lib.cstr_probe_pipe(kind, iters, grid, block, out.data_ptr(), stream), "probe")
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            rate = grid * block * iters * 8 * flop / (ms * 1e-3) / 1e12
            if rep and rate > best:
                best, mhz = rate, float(out[0].item())  # out[0]: the SM clock block 0 ran at (clock64 / globaltimer)
        res[name] = best
        res[name.rsplit("_", 1)[0] + "_sm_mhz"] = mhz
    res["sm_clock_khz_max"] = info[1].value
    # the clock-derived FP32 peak (SURVEY 8d: SMs x 128 lanes x 2 flop x f_clk) at the device's maximum SM clock
    res["fp32_clock_derived_tflops"] = sms * 128 * 2 * info[1].value * 1e3 / 1e12
    return res


def time_launches(torch, fn, k: int):
    """Run fn() k times, one CUDA-event pair per launch on the current stream; returns (total_ms, [ms])."""
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(k + 1)]
    evs[0].record()
    for i in range(k):
        fn()
        evs[i + 1].record()
    evs[-1].synchronize()
    per = [evs[i].elapsed_time(evs[i + 1]) for i in range(k)]
    return evs[0].elapsed_time(evs[-1]), per


DUMP_REACTORS = 8192  # reactors sampled over ALL ranks: 8192 x (400 x (4 + 4) + 16 + 8 + 8) B = 26.5 MB per dump, whatever the rank count


def dump_columns(n: int, world: int):
    """The reactors of one rank's shard that --dump-outputs writes: sorted indices of default_rng(0).choice(n, k, replace=False) with
    k = min(n, DUMP_REACTORS // world), so that the ranks together write at most DUMP_REACTORS reactors."""
    import numpy as np

    return np.sort(np.random.default_rng(0).choice(n, size=min(n, max(1, DUMP_REACTORS // world)), replace=False))


def dump_outputs(out_dir: str, env, rewards, dones, rank: int, world: int) -> None:
    """--dump-outputs: what the caller of the timed step receives after the last timed launch, as float32 / float64 .npy files, for the
    reactors of dump_columns(): rewards / dones (T, k), state (k, 4), step_count and episode (k).  With more than one rank each writes
    its own shard's sample under a _rank<r> suffix."""
    import numpy as np
    import torch

    cols = dump_columns(rewards.shape[1], world)
    idx = torch.as_tensor(cols, device=rewards.device)
    arrays = {"rewards": rewards.index_select(1, idx).cpu().numpy(),
              "dones": dones.index_select(1, idx).to(torch.float32).cpu().numpy(),
              "state": env.state.index_select(0, idx).cpu().numpy(),
              "step_count": env.step_count.index_select(0, idx).cpu().numpy().astype(np.float64),
              "episode": env.episode.index_select(0, idx).cpu().numpy().astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def run_ours(args) -> None:
    import numpy as np
    import torch

    pkg = importlib.import_module("pytorch-rl-enhancedstablebaselines_b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank) if world > 1 else {"bound": False, "note": "single rank: left where the launcher put it"}
    dist = None
    if world > 1:
        import torch.distributed as dist

        backend = os.environ.get("CSTR_BENCH_BACKEND", "nccl")  # "gloo": the CPU dry run of this file's control flow (tests/test_bench_dryrun.py)
        dist.init_process_group(backend, **({"device_id": device} if backend == "nccl" else {}))
    lib = pkg._lib.load()
    from ctypes import byref

    def barrier():
        torch.cuda.synchronize(device)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(device)

    n, T = N_ENVS, T_STEPS
    seed = 20260101
    env = pkg.GpuCSTRVecEnv(n, device=device, math=args.math, seed=seed, env_offset=rank * n, monitor=False)
    env.reset()
    gen = torch.Generator(device=device).manual_seed(1234 + rank)
    tape = (torch.rand((T, n, 2), generator=gen, device=device, dtype=torch.float32) * 2 - 1).contiguous()  # 210 MB > L2
    rewards = torch.empty((T, n), dtype=torch.float32, device=device)
    dones = torch.empty((T, n), dtype=torch.uint8, device=device)
    stream = torch.cuda.current_stream(device).cuda_stream
    mode = {"strict": 0, "fast": 1}[args.math]

    def step():
        pkg._lib.check(lib.cstr_tape_f32(byref(env._params), n, T, mode, tape.data_ptr(), 0, env.state.data_ptr(), env.step_count.data_ptr(),
                                         env.episode.data_ptr(), None, rewards.data_ptr(), dones.data_ptr(), None, None, stream), "cstr_tape_f32")

    peaks = measure_pipe_peaks(pkg, torch, device) if rank == 0 else None
    # the other arithmetic flavour, same workload, timed outside the headline region (rank 0 reports it)
    other_mode = 1 - mode
    other_name = "strict" if other_mode == 0 else "fast"

    def step_other():
        pkg._lib.check(lib.cstr_tape_f32(byref(env._params), n, T, other_mode, tape.data_ptr(), 0, env.state.data_ptr(), env.step_count.data_ptr(),
                                         env.episode.data_ptr(), None, rewards.data_ptr(), dones.data_ptr(), None, None, stream), "cstr_tape_f32")

    for _ in range(3):
        step_other()
    _, per_other = time_launches(torch, step_other, 10)
    other_ms = statistics.mean(per_other)
    # clocks are sampled (100 ms period) from just before the warm-up until the end of the e2e loop: the timed region
    # itself lasts only milliseconds, so the window is the whole GPU-busy phase around it
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    t_wall0 = time.time()
    for _ in range(args.warmup):
        step()
    barrier()
    # the timed region: K launches back to back between ONE event pair (no per-launch host work beyond the C call, so a busy
    # host — N rank processes on one box — cannot starve the 0.1 ms kernels); per-launch durations are taken in a second pass
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    ev1.synchronize()
    total_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:  # before the per-launch pass below steps the reactors on
        dump_outputs(args.dump_outputs, env, rewards, dones, rank, world)
    barrier()
    _, per = time_launches(torch, step, args.steps)
    tmax = torch.tensor([total_ms], dtype=torch.float64, device=device)
    per_rank_ms = [total_ms]
    if dist is not None:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        gathered = [torch.zeros(1, dtype=torch.float64, device=device) for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([total_ms], dtype=torch.float64, device=device))
        per_rank_ms = [float(g.item()) for g in gathered]
    total_ms_max = float(tmax.item())
    value = world * args.steps * n * T / (total_ms_max * 1e-3)
    # sanity inside the bench: one truncation row per episode, rewards finite
    assert int(dones.sum().item()) == n and bool(torch.isfinite(rewards).all().item())

    # ---- e2e: the C-ABI call with HOST buffers (H2D tape + state, kernel, D2H rewards/dones/state) --------------
    h_tape = torch.empty((T, n, 2), dtype=torch.float32).pin_memory()
    h_tape.copy_(tape)
    h_state = torch.empty((n, 4), dtype=torch.float32).pin_memory()
    h_state.copy_(env.state)
    h_sc = torch.zeros(n, dtype=torch.int32).pin_memory()
    h_ep = torch.ones(n, dtype=torch.int32).pin_memory()
    h_rew = torch.empty((T, n), dtype=torch.float32).pin_memory()
    h_done = torch.empty((T, n), dtype=torch.uint8).pin_memory()

    def e2e_step():
        pkg._lib.check(lib.cstr_tape_f32_host(byref(env._params), n, T, mode, h_tape.data_ptr(), h_state.data_ptr(), h_sc.data_ptr(),
                                              h_ep.data_ptr(), h_rew.data_ptr(), h_done.data_ptr(), stream), "cstr_tape_f32_host")

    e2e_reps = max(3, min(args.steps, 10))
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_reps):
        e2e_step()  # synchronises internally: results are on the host when it returns
    torch.cuda.synchronize(device)
    e2e_local_s = time.perf_counter() - t0
    e2e_dt = torch.tensor([e2e_local_s], dtype=torch.float64, device=device)
    e2e_per_rank_s = [e2e_local_s]
    if dist is not None:
        gathered = [torch.zeros(1, dtype=torch.float64, device=device) for _ in range(world)]
        dist.all_gather(gathered, e2e_dt.clone())
        e2e_per_rank_s = [float(g.item()) for g in gathered]
        dist.all_reduce(e2e_dt, op=dist.ReduceOp.MAX)
    e2e_value = world * e2e_reps * n * T / float(e2e_dt.item())
    h2d = T * n * 8 + n * (16 + 4 + 4)
    d2h = T * n * (4 + 1) + n * (16 + 4 + 4)
    assert int(h_done.sum().item()) == n
    clocks = sampler.stop(t_wall0, time.time()) if rank == 0 else None

    # ---- CPU baseline on a bounded sample (N=1, rank 0; BEFORE the optional sections so that the line below is complete) -------
    cpu = None
    if world == 1:
        try:
            rate, T_cpu, cores, dt = cpu_port_rate(n, target_seconds=12.0)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{n} reactors x {T_cpu} control intervals (repeated 400-interval passes), float32, libm expf/powf, OpenMP ({dt:.1f} s of CPU work)"}
        except Exception as exc:  # the baseline must never take the bench down
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {exc}"}

    # ---- the line as it stands once the headline, e2e and the CPU baseline are measured --------------------------------------------
    line = None
    if rank == 0:
        kernel_ms = statistics.mean(per)
        achieved = FLOP_PER_ENV_STEP * n * T / (kernel_ms * 1e-3) / 1e12
        peak = peaks["fp32_ffma_tflops"]
        # dram__bytes_read + dram__bytes_write of one launch: STATIC, from the committed ncu --set full capture (ncu cannot run inside the bench)
        traffic, traffic_source = None, None
        for name in ("r02_traffic.json", "r01_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath):
                try:
                    tj = json.load(open(tpath))
                    key = "tape_f32_kernel<0, 0, 0, 0>" if args.math == "strict" else "tape_f32_kernel<1, 0, 0, 0>"
                    traffic = tj.get(key, {}).get("dram_bytes")
                    traffic_source = f"static: ncu --set full capture in profiles/{name} (commit {tj.get('_commit', 'unrecorded')}), not measured in this run"
                except Exception:
                    traffic = None
                if traffic is not None:
                    break
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "run": {"math": args.math, "actions": "streamed from HBM", "l2": "inputs larger than L2 (210 MB tape vs 126 MB): no flush needed",
                    "per_rank_ms_per_step": [round(t / args.steps, 5) for t in per_rank_ms], "host_placement": numa,
                    "parity": "fast: |dobs|<=2e-6 per step, <=1e-5 over 400 steps, |dreward|<=1e-5, dones equal vs the oracle "
                              "(tests/test_gpu_step.py::test_fast_tape_hbm_actions_rewards_dones_vs_oracle; |dreward|<=5e-5 over the trajectory); strict: bit-exact vs the oracle"},
            "roofline": {"bound": "fp32-pipe", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                         "traffic": traffic, "traffic_source": traffic_source, "kernel": f"tape_f32_kernel<{args.math}>", "kernel_ms": kernel_ms,
                         "frac_of_clock_derived_peak": achieved / peaks["fp32_clock_derived_tflops"],
                         "peak_note": "the FFMA probe (64 FFMA per loop branch, SASS-checked) runs at the SM clock it reports (fp32_ffma_sm_mhz) — "
                                      "the clock-derived figure assumes the nominal maximum clock",
                         "flop_per_env_step": FLOP_PER_ENV_STEP, "peak_source": "measured in this run: cstr_probe_pipe FFMA chains (2 flop/FMA)",
                         "other_peaks": peaks,
                         "hbm_algorithmic_gbs": n * T * (8 + 4 + 1) / (kernel_ms * 1e-3) / 1e9},
            "other_math": {"math": other_name, "value": world * n * T / (other_ms * 1e-3), "unit": UNIT, "kernel_ms": other_ms,
                           "roofline_frac": (FLOP_PER_ENV_STEP * n * T / (other_ms * 1e-3) / 1e12) / peak if peak else None,
                           "note": "strict = reference association, no FMA contraction, bit-exact vs the oracle; fast = throughput variant, |dobs| <= 2e-6/step"},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "call": "cstr_tape_f32_host (pinned host buffers -> H2D -> tape kernel -> D2H, synchronous)",
                    "per_rank_h2d_gbs": [round(e2e_reps * h2d / t / 1e9, 2) for t in e2e_per_rank_s],
                    "per_rank_d2h_gbs": [round(e2e_reps * d2h / t / 1e9, 2) for t in e2e_per_rank_s]},
            "gpu_launches": args.steps, "clocks": clocks, "rollout": None, "dp_update": None, "multi_rank_error": None, "extras": {},
        }

    # ---- optional sections under a hard stop: they may fail or hang, the line above may not be lost -------------------------------
    stop = HardStop(float(os.environ.get("CSTR_BENCH_SECTION_LIMIT_S", "300")), rank)
    stop.start(line)
    sticky = False
    if not args.no_extras:
        # the other half of the metric and the only collective, at EVERY N (all ranks take part)
        try:
            multi = run_multi_rank_sections(pkg, torch, device, dist, rank, world, args)
        except Exception as exc:  # must never take the headline down
            multi, sticky = {"error": describe_error(exc)}, True
        if rank == 0:
            with stop.lock:
                line.update(rollout=multi.get("rollout"), dp_update=multi.get("dp_update"), multi_rank_error=multi.get("error"))
        # extras (rank 0, N=1 only: variants that explain the headline)
        if rank == 0 and world == 1:
            args._ffma_peak = peaks.get("fp32_ffma_tflops") if peaks else None
            extras = run_extras(pkg, torch, device, lib, env, tape, rewards, dones, args)
            sticky = sticky or any(k.endswith("error") for k in extras) or any(k.endswith("error") for k in extras.get("td3_update", {}))
            with stop.lock:
                line["extras"] = extras
    sticky = sticky or bool(FAILED_SECTIONS)
    stop.emit(line)
    if sticky:  # a failed section may have left a sticky CUDA error or a rank out of step: no teardown that could abort or wait
        sys.stdout.flush()
        os._exit(0)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    stop.cancel()


def run_multi_rank_sections(pkg, torch, device, dist, rank, world, args) -> dict:
    """BASELINE metric, second half ("rollout transitions/sec at 1/2/4/8 B200") and SURVEY 8e's only collective, measured at every N:

    rollout   config #3: TD3 actor 4-400-300-2 on tcgen05 fused with noise, bounds, CSTR step, reward/done and the replay record
              (cstr_rollout_fused, 16 steps per launch, ring of 64 rows per GPU).  strong: 1,048,576 reactors sharded over the N
              ranks; weak: 131,072 reactors per rank.  No collective on this path.  value = transitions of ALL ranks / max-over-ranks time.
    dp_update TD3 [400,300] gradient step, data-parallel over the N ranks, per-rank batch 4096 and 256, replayed from ONE CUDA graph
              per policy_delay cycle (Philox sample -> GRAD -> gradient mean over ranks -> Adam/polyak): "peer" = the mean is taken
              inside the Adam kernels over NVLink peer memory (cstr_peer_comm), "nccl_eager" = the round-1 path (launch by launch,
              ncclAllReduce(avg) between the phases), "local" = the same graph without any exchange (what one GPU does alone).
              ms per update, max over ranks.  (ncclAllReduce captured INSIDE the graph ran on 2 GPUs — 0.556 ms at batch 4096, 0.162 at
              256, profiles/r02_bench_n2_sections.json — but hung on 8 and is therefore opt-in, CSTR_NCCL_GRAPH=1, and not timed here.)"""
    import numpy as np

    def max_over_ranks(ms: float) -> float:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize(device)
        if dist is not None:
            dist.barrier()

    def timed(fn, reps, warm=3):
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        return max_over_ranks(e0.elapsed_time(e1) / reps)

    out = {"rollout": {}, "dp_update": {}}
    torch.manual_seed(0)
    lin = [torch.nn.Linear(4, 400), torch.nn.Linear(400, 300), torch.nn.Linear(300, 2)]
    K, rows = 16, 64
    for name, n_total in (("strong_1048576_total", 1 << 20), ("weak_131072_per_gpu", (1 << 17) * world)):
        off, cnt = pkg.dist.shard_range(n_total, rank, world)
        er = pkg.GpuCSTRVecEnv(cnt, device=device, math="strict", seed=4, env_offset=off, monitor=False)
        er.reset()
        buf = pkg.GpuReplayBuffer(rows * cnt, device=device, n_envs=cnt, index_mode="philox", seed=rank)
        actor = pkg.ActorWeights(lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, lin[2].weight, lin[2].bias, device=device)
        roll = pkg.FusedRollout(er, buf, actor, sigma=0.1, actor_mode="tc")
        ms = timed(lambda: roll.collect(K), reps=8, warm=4)
        out["rollout"][name] = {"transitions_per_s": n_total * K / (ms * 1e-3), "ms_per_launch": ms, "steps_per_launch": K,
                                "reactors_total": n_total, "reactors_this_rank": cnt, "actor": "TD3 4-400-300-2, bf16 tcgen05 hidden layer",
                                "algorithmic_tflops_per_gpu": (244_400 + 176) * cnt * K / (ms * 1e-3) / 1e12}
        del roll, actor, buf, er
    out["rollout"]["scaling"] = {"strong_1048576_total": "strong", "weak_131072_per_gpu": "weak"}

    n_envs = 65536
    buf = pkg.GpuReplayBuffer(16 * n_envs, device=device, n_envs=n_envs, index_mode="philox", seed=1000 + rank)
    buf.records.uniform_(-1, 1)
    buf.records[..., 11:13] = 0
    buf.pos, buf.full = 0, True
    rng = np.random.default_rng(0)

    def nets():
        def mlp(i, o):
            t = []
            for fi, fo in ((i, 400), (400, 300), (300, o)):
                b = 1.0 / np.sqrt(fi)
                t += [rng.uniform(-b, b, (fo, fi)).astype(np.float32), rng.uniform(-b, b, fo).astype(np.float32)]
            return t
        return {"actor": mlp(4, 2), "critic0": mlp(6, 1), "critic1": mlp(6, 1)}

    weights = nets()
    hook = pkg.dist.allreduce_flat if world > 1 else None
    for B in (4096, 256):
        row = {"per_rank_batch": B, "global_batch": B * world, "net_arch": [400, 300], "gradient_bucket_bytes": None}
        reps = 50 if B == 4096 else 100
        for mode in ("local", "peer", "nccl_eager"):
            if world == 1 and mode != "local":
                continue
            eng = pkg.FusedTD3Update([400, 300], B, device=device, seed=7, dp_rank=rank)
            eng.load_nets(weights)
            row["gradient_bucket_bytes"] = eng.param_count * 4
            if mode == "peer":
                eng.enable_peer_allreduce()
            ar = hook if mode == "nccl_eager" else None
            graph = mode != "nccl_eager"
            ms = timed(lambda: eng.train(2, buf, B, graph=graph, allreduce=ar), reps=reps, warm=5) / 2
            row[f"{mode}_ms_per_update"] = ms
            if mode == "peer":
                row["peer_error_word"] = eng.peer_error()
            eng.close_peer_allreduce()
            del eng
        if world > 1:
            row["peer_over_local"] = row["peer_ms_per_update"] / row["local_ms_per_update"]
            row["nccl_eager_over_local"] = row["nccl_eager_ms_per_update"] / row["local_ms_per_update"]
        out["dp_update"][f"per_rank_batch_{B}"] = row
    out["dp_update"]["collective"] = ("gradient mean over ranks: critics' range every update, actor's range on policy steps (the actor loss needs the "
                                      "UPDATED critic, td3.py:189-191, so the two ranges cannot share one exchange)")
    return out


def run_extras(pkg, torch, device, lib, env, tape, rewards, dones, args) -> dict:
    """Variants that explain the headline; each timed with CUDA events after its own warm-up.  Every section runs under its own
    try/except (`<section>_error` in the result): a section that fails must not take the others — or the headline — down."""
    from ctypes import byref

    import numpy as np

    n, T = N_ENVS, T_STEPS
    stream = torch.cuda.current_stream(device).cuda_stream
    ex = {}

    def rate_of(fn, env_steps, reps=5):
        for _ in range(2):
            fn()
        # ONE event pair around the reps: an event between launches puts host gaps into the time of kernels shorter than a Python call
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        return env_steps / (e0.elapsed_time(e1) / reps * 1e-3)

    def section(name, fn):
        try:
            fn()
            torch.cuda.synchronize(device)
        except Exception as exc:
            ex[f"{name}_error"] = describe_error(exc)

    def tapes():
        for math, mode in (("strict", 0), ("fast", 1)):
            ex[f"tape_f32_{math}_hbm_actions"] = rate_of(lambda: lib.cstr_tape_f32(
                byref(env._params), n, T, mode, tape.data_ptr(), 0, env.state.data_ptr(), env.step_count.data_ptr(), env.episode.data_ptr(),
                None, rewards.data_ptr(), dones.data_ptr(), None, None, stream), n * T)
            ex[f"tape_f32_{math}_philox_actions"] = rate_of(lambda: lib.cstr_tape_f32(
                byref(env._params), n, T, mode, None, 0, env.state.data_ptr(), env.step_count.data_ptr(), env.episode.data_ptr(),
                None, rewards.data_ptr(), dones.data_ptr(), None, None, stream), n * T)

    def tape_f64():  # north_star: fp64 vs fp32
        e64 = pkg.GpuCSTRVecEnv(n, device=device, dtype="fp64", seed=1, monitor=False)
        e64.reset()
        r64 = torch.empty((T, n), dtype=torch.float64, device=device)
        ex["tape_f64_philox_actions"] = rate_of(lambda: lib.cstr_tape_f64(
            byref(e64._params), n, T, None, 0, e64.state.data_ptr(), e64.step_count.data_ptr(), e64.episode.data_ptr(), None, r64.data_ptr(),
            dones.data_ptr(), None, None, stream), n * T, reps=3)

    nb, Tb = 1 << 20, 100

    def tapes_1m():  # 1,048,576 reactors (config #3 batch) — the chip is full at this size
        eb = pkg.GpuCSTRVecEnv(nb, device=device, math=args.math, seed=2, monitor=False)
        eb.reset()
        rb = torch.empty((Tb, nb), dtype=torch.float32, device=device)
        db = torch.empty((Tb, nb), dtype=torch.uint8, device=device)
        for math, mode in (("strict", 0), ("fast", 1)):
            ex[f"tape_f32_{math}_philox_1M_envs"] = rate_of(lambda: lib.cstr_tape_f32(
                byref(eb._params), nb, Tb, mode, None, 0, eb.state.data_ptr(), eb.step_count.data_ptr(), eb.episode.data_ptr(), None,
                rb.data_ptr(), db.data_ptr(), None, None, stream), nb * Tb, reps=3)
        # single VecEnv step kernel at 1M envs: HBM-bound (70 B/env-step)
        ab = torch.rand((nb, 2), device=device) * 2 - 1
        r1 = rate_of(lambda: eb.step_tensor(ab), nb, reps=20)
        ex["vec_step_f32_1M_envs"] = r1
        ex["vec_step_f32_1M_envs_hbm_gbs"] = r1 * 70 / 1e9

    def numpy_protocol():  # VecEnv.step() through NumPy buffers (the reference-facing protocol call), 65,536 envs
        ev = pkg.GpuCSTRVecEnv(n, device=device, math=args.math, seed=3, monitor=False)
        ev.reset()
        a_np = np.random.default_rng(0).uniform(-1, 1, (n, 2)).astype(np.float32)
        for _ in range(3):
            ev.step(a_np)
        t0 = time.perf_counter()
        for _ in range(20):
            ev.step(a_np)
        ex["vecenv_step_numpy_protocol"] = 20 * n / (time.perf_counter() - t0)

    def replay_and_rollout():
        # replay buffer: add (52 B/transition algorithmic) and sample (116 B/sample algorithmic), HBM-bound
        rows, ne = 64, 1 << 20
        buf = pkg.GpuReplayBuffer(rows * ne, device=device, n_envs=ne, index_mode="philox")
        o = torch.rand((ne, 4), device=device)
        a2 = torch.rand((ne, 2), device=device)
        r2 = torch.rand(ne, device=device)
        d2 = torch.zeros(ne, dtype=torch.uint8, device=device)
        add_rate = rate_of(lambda: buf.add(o, o, a2, r2, d2, None, timeouts=d2), ne, reps=64)
        ex["replay_add_transitions_per_s"] = add_rate
        ex["replay_add_algorithmic_gbs"] = add_rate * 52 / 1e9
        B_ = 1 << 22
        smp = rate_of(lambda: buf.sample(B_), B_, reps=10)
        ex["replay_sample_philox_samples_per_s"] = smp
        ex["replay_sample_algorithmic_gbs"] = smp * 116 / 1e9
        # fused rollout (config #3 shape: TD3 actor 4-400-300-2, sigma 0.1), transitions/s
        torch.manual_seed(0)
        lin = [torch.nn.Linear(4, 400), torch.nn.Linear(400, 300), torch.nn.Linear(300, 2)]
        actor = pkg.ActorWeights(lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, lin[2].weight, lin[2].bias, device=device)
        er = pkg.GpuCSTRVecEnv(ne, device=device, math=args.math, seed=4, monitor=False)
        er.reset()
        for mode_name in ("fp32", "tc"):
            try:
                roll = pkg.FusedRollout(er, buf, actor, sigma=0.1, actor_mode=mode_name)
                Kr = 2 if mode_name == "fp32" else 16
                ex[f"fused_rollout_{mode_name}_transitions_per_s"] = rate_of(lambda: roll.collect(Kr), ne * Kr, reps=3)
            except Exception as exc:
                FAILED_SECTIONS.append(exc)  # kept, see describe_error
                ex[f"fused_rollout_{mode_name}_transitions_per_s"] = f"unavailable: {exc}"

    def updates():
        ex["td3_update"] = td3_update_extras(pkg, torch, device, peaks_tflops=args._ffma_peak)

    for name, fn in (("tapes", tapes), ("tape_f64", tape_f64), ("tapes_1M", tapes_1m), ("numpy_protocol", numpy_protocol),
                     ("replay_and_rollout", replay_and_rollout), ("updates", updates)):
        section(name, fn)
    try:
        torch.cuda.synchronize(device)
    except Exception as exc:
        ex["sync_error"] = repr(exc)
    return ex


def td3_update_extras(pkg, torch, device, peaks_tflops) -> dict:
    """SURVEY §8f-1: one TD3 gradient step (sample + cstr_td3_update), float32, [400,300] nets, at the reference's default
    batch (256) and at 4096; beside it the same update in eager torch on this GPU (what the unmodified reference's TD3.train
    executes on a CUDA device: autograd + cuBLAS sgemm + torch.optim.Adam) and the NumPy restatement on the host (cpu_baseline)."""
    import numpy as np

    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import run_td3 as R
    import td3_oracle as TO
    import td3_util as TU

    out = {"flop_per_sample": R.flops_per_sample(400, 300), "dtype": "f32", "net_arch": [400, 300]}
    n_envs = 65536
    buf = pkg.GpuReplayBuffer(16 * n_envs, device=device, n_envs=n_envs, index_mode="philox")
    buf.records.uniform_(-1, 1)
    buf.records[..., 11:13] = 0
    buf.pos, buf.full = 0, True
    torch.backends.cuda.matmul.allow_tf32 = False
    for B in (256, 4096):
        torch.manual_seed(0)
        eng = pkg.FusedTD3Update([400, 300], B, device=device)
        eng.adopt_modules(R.mlp(4, 2, True, device), [R.mlp(6, 1, False, device), R.mlp(6, 1, False, device)], R.mlp(4, 2, True, device),
                          [R.mlp(6, 1, False, device), R.mlp(6, 1, False, device)])
        ms = R.timed(lambda: eng.update(buf.sample(B)), 200)
        ref = R.TorchTD3(device)
        ms_t = R.timed(lambda: ref.update(buf.sample(B)), 100)
        tf = out["flop_per_sample"] * B / (ms * 1e-3) / 1e12
        row = {"updates_per_s": 1e3 / ms, "samples_per_s": B * 1e3 / ms, "ms_per_update": ms, "algorithmic_tflops": tf,
               "frac_of_ffma_peak": tf / peaks_tflops if peaks_tflops else None, "torch_eager_same_gpu_ms_per_update": ms_t}
        if B == 256:  # cpu_baseline: NumPy restatement of TD3.train on the host (multi-threaded BLAS), a few gradient steps
            rng = np.random.default_rng(0)
            nets = TU.random_nets(rng, 400, 300)
            o = TO.TD3UpdateOracle(nets["actor"], [nets["critic0"], nets["critic1"]])
            mk = lambda: (rng.uniform(-1, 1, (B, 4)).astype(np.float32), rng.uniform(-1, 1, (B, 2)).astype(np.float32),  # noqa: E731
                          rng.uniform(-1, 1, (B, 4)).astype(np.float32), np.zeros((B, 1), np.float32), rng.normal(size=(B, 1)).astype(np.float32),
                          rng.normal(0, 0.2, (B, 2)).astype(np.float32))
            o.step(*mk())
            t0 = time.perf_counter()
            k = 0
            while time.perf_counter() - t0 < 2.0:
                o.step(*mk())
                k += 1
            row["cpu_oracle_updates_per_s"] = k / (time.perf_counter() - t0)
        # the same update with the hidden-layer GEMMs on tcgen05 (3-plane bf16 split, fp32-grade; opt-in gemm="tensor")
        eng_tc = pkg.FusedTD3Update([400, 300], B, device=device, gemm="tensor")
        eng_tc.adopt_modules(R.mlp(4, 2, True, device), [R.mlp(6, 1, False, device), R.mlp(6, 1, False, device)], R.mlp(4, 2, True, device),
                             [R.mlp(6, 1, False, device), R.mlp(6, 1, False, device)])
        ms_tc = R.timed(lambda: eng_tc.update(buf.sample(B)), 200)
        row["cuda_graph_ms_per_update"] = R.timed(lambda: eng.train(2, buf, B, graph=True), 100) / 2
        row["tensor_gemm_cuda_graph_ms_per_update"] = R.timed(lambda: eng_tc.train(2, buf, B, graph=True), 100) / 2
        row["tensor_gemm_ms_per_update"] = ms_tc
        row["tensor_gemm_algorithmic_tflops"] = out["flop_per_sample"] * B / (ms_tc * 1e-3) / 1e12
        out[f"batch_{B}"] = row
        del eng, ref, eng_tc
    # SAC gradient step (cstr_sac_update), the reference's default [256, 256] nets
    for B in (256, 4096):
        sac = pkg.FusedSACUpdate([256, 256], B, device=device)
        sac.params[:sac._ent_offset].normal_(0, 0.05)
        sac.targets.copy_(sac.params)
        ms = R.timed(lambda: sac.update(buf.sample(B)), 200)
        out[f"sac_batch_{B}"] = {"ms_per_update": ms, "updates_per_s": 1e3 / ms, "samples_per_s": B * 1e3 / ms,
                                 "cuda_graph_ms_per_update": R.timed(lambda: sac.train(2, buf, B, graph=True), 100) / 2}
        del sac
    # BCQ gradient step (cstr_bcq_update): BCQPolicy's default sizes and the experiment script's, beside the same update in eager torch
    try:
        sys.path.insert(0, os.path.join(ROOT, "examples"))
        import bcq_offline as BO

        for tag, (L, hv, hp) in (("default_sizes", (32, 64, 64)), ("script_sizes", (12, 700, 400))):
            for B in (256, 4096):
                ref = BO.TorchBCQ(device, L, hv, hp)
                eng = pkg.FusedBCQUpdate(L, hv, hp, [400, 300], B, device=device)
                P = lambda m: [p.detach() for p in m.parameters()]  # noqa: E731
                eng.load_nets({"vae_enc": P(ref.enc), "vae_dec": P(ref.dec), "pert": P(ref.xi), "critic0": P(ref.critics[0]), "critic1": P(ref.critics[1])})
                out[f"bcq_{tag}_batch_{B}"] = {"ms_per_update": R.timed(lambda: eng.update(buf.sample(B)), 100),
                                               "cuda_graph_ms_per_update": R.timed(lambda: eng.train(2, buf, B, graph=True), 100) / 2,
                                               "torch_eager_same_gpu_ms_per_update": R.timed(lambda: ref.update(buf.sample(B)), 50)}
                del eng, ref
    except Exception as exc:  # the TD3 / SAC rows above must survive
        out["bcq_error"] = describe_error(exc)
    # MADDPG / IDDPG gradient step (cstr_ma_update), two agents, [400, 300] nets
    try:
        for name, central in (("maddpg", True), ("iddpg", False)):
            for B in (256, 4096):
                eng = pkg.FusedMultiAgentUpdate([400, 300], B, central, device=device)
                eng.params.normal_(0, 0.05)
                eng.targets.copy_(eng.params)
                out[f"{name}_batch_{B}"] = {"ms_per_update": R.timed(lambda: eng.update(buf.sample(B)), 100),
                                            "cuda_graph_ms_per_update": R.timed(lambda: eng.train(2, buf, B, graph=True), 100) / 2}
                del eng
    except Exception as exc:
        out["multi_agent_error"] = describe_error(exc)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--math", choices=["strict", "fast"], default="fast",
                    help="headline kernel: fast = the throughput variant (FMA contraction, MUFU; documented tolerance), strict = bit-exact vs the oracle; the other one is timed too and reported under \"other_math\"")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
