"""CPU dry run of bench.py's control flow (not gpu): the driver depends on the ONE JSON line and its keys, and the bench's Python —
section ordering, the hard stop, the dictionaries — must be exercisable without a device.  Everything that touches the GPU is replaced
by inert stand-ins here (a fake library whose tape call writes one truncation row, fake engines that count calls); what runs for real is
bench.py itself: argument handling, the timing scaffolding, the CPU baseline on a tiny sample, the assembly of the line.  No number in
the line means anything — only its shape is asserted."""
import ctypes
import importlib
import json
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch._dynamo  # noqa: F401  (loaded before torch.device is patched below: its modules annotate with `torch.device | None`)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "pytorch-rl-enhancedstablebaselines_b200"


class _FakeEvent:
    def __init__(self, enable_timing=False):
        pass

    def record(self, *a):
        pass

    def synchronize(self):
        pass

    def elapsed_time(self, other):
        return 1.0


class _FakeLib:
    """Every entry point returns 0; the tape calls leave finite rewards and exactly one truncation row, as the real kernels do."""

    def __getattr__(self, name):
        return lambda *a: 0

    @staticmethod
    def _fill(n, T, rewards, dones):
        if rewards:
            ctypes.memset(rewards, 0, n * T * 4)
        if dones:
            ctypes.memset(dones, 0, n * T)
            ctypes.memset(dones + (T - 1) * n, 1, n)

    def cstr_tape_f32(self, params, n, T, mode, actions, t_base, state, sc, ep, static_base, rewards, dones, obs, rsum, stream):
        self._fill(n, T, rewards, dones)
        return 0

    def cstr_tape_f32_host(self, params, n, T, mode, h_act, h_state, h_sc, h_ep, h_rew, h_done, stream):
        self._fill(n, T, h_rew, h_done)
        return 0

    def cstr_device_info(self, sms, clock_khz, cc_major, cc_minor):
        sms._obj.value, clock_khz._obj.value, cc_major._obj.value, cc_minor._obj.value = 148, 1_965_000, 10, 0
        return 0


class _FakeEnv:
    def __init__(self, n, device=None, **kw):
        self.n = n
        self._params = ctypes.c_int(0)
        self.state = torch.zeros((n, 4))
        self.step_count = torch.zeros(n, dtype=torch.int32)
        self.episode = torch.ones(n, dtype=torch.int32)

    def reset(self):
        return self.state.numpy().copy()

    def step_tensor(self, a):
        return None

    def step(self, a):
        return None


class _FakeBuffer:
    def __init__(self, size, device=None, n_envs=1, **kw):
        self.records = torch.zeros((2, 4, 16))
        self.pos, self.full, self.index_mode, self.n_envs = 0, False, "philox", n_envs

    def add(self, *a, **kw):
        pass

    def sample(self, B, env=None):
        S = types.SimpleNamespace(observations=torch.zeros(B, 4), actions=torch.zeros(B, 2), next_observations=torch.zeros(B, 4),
                                  dones=torch.zeros(B, 1), rewards=torch.zeros(B, 1))
        return S


class _FakeEngine:
    param_count = 369_704
    _ent_offset = 8

    def __init__(self, *a, **kw):
        self.params, self.targets = torch.zeros(16), torch.zeros(16)

    def __getattr__(self, name):  # load_nets, adopt_modules, update, train, enable/close_peer_allreduce ...
        return lambda *a, **kw: 0


def install_fakes(monkeypatch):
    """Replace everything that touches the device; returns the bench module.  Also used by the two-rank worker below."""
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    pkg = importlib.import_module(PKG)
    b = importlib.import_module("bench")
    real_device = torch.device
    torch.optim.Adam([torch.nn.Parameter(torch.zeros(1))]).step()  # torch's lazily imported submodules annotate with `torch.device | None`: load them first
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "Event", _FakeEvent)
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: False)  # torch.optim asks once is_available() says True
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a: types.SimpleNamespace(cuda_stream=0))
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda i: types.SimpleNamespace(pci_domain_id=0, pci_bus_id=0xfe, pci_device_id=0x1f))
    monkeypatch.setattr(torch, "device", lambda *a, **kw: real_device("cpu"))
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    monkeypatch.setattr(pkg._lib, "load", lambda *a, **kw: _FakeLib())
    for name, fake in (("GpuCSTRVecEnv", _FakeEnv), ("GpuReplayBuffer", _FakeBuffer), ("ActorWeights", _FakeEngine), ("FusedRollout", _FakeEngine),
                       ("FusedTD3Update", _FakeEngine), ("FusedSACUpdate", _FakeEngine), ("FusedBCQUpdate", _FakeEngine),
                       ("FusedMultiAgentUpdate", _FakeEngine)):
        monkeypatch.setattr(pkg, name, fake)
    monkeypatch.setattr(b, "N_ENVS", 256)
    monkeypatch.setattr(b, "T_STEPS", 8)
    real_rate = b.cpu_port_rate
    monkeypatch.setattr(b, "cpu_port_rate", lambda n, target_seconds, seed=0: real_rate(n, 0.05, seed))
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import run_td3

    def once(fn, steps):
        fn()
        return 1.0

    monkeypatch.setattr(run_td3, "timed", once)
    return b


@pytest.fixture()
def bench(monkeypatch):
    b = install_fakes(monkeypatch)

    def no_exit(code):
        raise AssertionError(f"bench.py left through os._exit({code}): a section reported an error")

    monkeypatch.setattr(os, "_exit", no_exit)
    return b


BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
             "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"}


def test_bench_line_shape_single_rank(bench, monkeypatch, capsys):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "4", "--warmup", "3"])
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("RANK", raising=False)
    bench.main()
    out = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(out) == 1, "exactly ONE JSON line"
    line = json.loads(out[0])
    assert BASE_KEYS <= set(line), BASE_KEYS - set(line)
    assert line["n_gpus"] == 1 and line["steps"] == 4 and line["warmup"] == 3 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["scaling"] == "weak" and line["dtype"] == "f32" and line["gpu_launches"] == 4
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"]) and line["cpu_baseline"]["kind"] == "port"
    assert line["cpu_baseline"]["value"] > 0 and line["cpu_baseline"]["cores"] >= 1
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert line["e2e"]["h2d_bytes_per_step"] == 8 * 256 * 8 + 256 * 24 and line["e2e"]["d2h_bytes_per_step"] == 8 * 256 * 5 + 256 * 24
    assert "workload" in line["config"] and not any(k.startswith("model") for k in line["config"])
    # the optional sections ran and none of them reported an error
    assert line["multi_rank_error"] is None and "sections_timeout_s" not in line
    assert set(line["rollout"]) == {"strong_1048576_total", "weak_131072_per_gpu", "scaling"}
    assert set(line["dp_update"]) == {"per_rank_batch_4096", "per_rank_batch_256", "collective"}
    assert "local_ms_per_update" in line["dp_update"]["per_rank_batch_256"] and "peer_ms_per_update" not in line["dp_update"]["per_rank_batch_256"]
    errors = [k for k in line["extras"] if k.endswith("error")] + [k for k in line["extras"].get("td3_update", {}) if k.endswith("error")]
    assert not errors, {k: line["extras"].get(k, line["extras"].get("td3_update", {}).get(k)) for k in errors}
    assert {"tape_f32_strict_hbm_actions", "tape_f64_philox_actions", "vec_step_f32_1M_envs", "replay_add_transitions_per_s",
            "fused_rollout_tc_transitions_per_s", "td3_update"} <= set(line["extras"])
    assert {"batch_256", "batch_4096", "sac_batch_256", "bcq_default_sizes_batch_256", "bcq_script_sizes_batch_4096", "maddpg_batch_256",
            "iddpg_batch_4096"} <= set(line["extras"]["td3_update"])


def test_both_arms_report_the_same_config(bench, monkeypatch, capsys):
    """The driver compares the two arms' `config`: it is the workload, identical in both; what varies with the run lives under `run`."""
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "3", "--warmup", "3", "--no-extras"])
    bench.main()
    ours = json.loads([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][0])
    monkeypatch.setattr(bench, "reference_python_rates", lambda *a, **kw: {"unavailable": "dry run"})
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "2", "--warmup", "1", "--no-extras"])
    bench.main()
    ref = json.loads([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][0])
    assert ref["impl"] == "reference" and ref["config"] == ours["config"]
    assert ref["metric"] == ours["metric"] and ref["unit"] == ours["unit"] and ref["higher_is_better"] == ours["higher_is_better"]
    assert ref["e2e"] == {"value": ref["value"], "unit": ref["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert ref["cpu_baseline"]["value"] == ref["value"] and ref["gpu_launches"] == 0
    assert ours["rollout"] is None and ours["extras"] == {}  # --no-extras


class _CountingLib(_FakeLib):
    """The tape call numbers its launches: every reward is 1000 x (launch number) + the reactor's index, every state row the index."""

    def __init__(self):
        self.launches = 0

    def cstr_tape_f32(self, params, n, T, mode, actions, t_base, state, sc, ep, static_base, rewards, dones, obs, rsum, stream):
        self.launches += 1
        self._fill(n, T, rewards, dones)
        np.ctypeslib.as_array((ctypes.c_float * (T * n)).from_address(rewards)).reshape(T, n)[:] = 1000 * self.launches + np.arange(n)
        np.ctypeslib.as_array((ctypes.c_float * (n * 4)).from_address(state)).reshape(n, 4)[:] = np.arange(n)[:, None]
        return 0


def test_dump_outputs_writes_what_the_last_timed_step_returned(bench, monkeypatch, capsys, tmp_path):
    """--dump-outputs DIR: the arrays the caller of the LAST TIMED tape launch receives (not those of the per-launch pass after it), for the
    seeded sample of reactors, float32 / float64 .npy; the JSON line is unchanged."""
    lib = _CountingLib()
    monkeypatch.setattr(importlib.import_module(PKG)._lib, "load", lambda *a, **kw: lib)
    monkeypatch.setattr(bench, "DUMP_REACTORS", 64)  # below the fake batch of 256: a real sample
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("RANK", raising=False)
    out_dir = tmp_path / "dump"
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "2", "--warmup", "3", "--no-extras", "--dump-outputs", str(out_dir)])
    bench.main()
    assert len([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]) == 1
    last_timed = 3 + 10 + 3 + 2  # the other math flavour (3 warm-up + 10 timed), the warm-up, the 2 timed steps
    assert lib.launches == last_timed + 2  # then the per-launch timing pass
    got = {f.stem: np.load(f) for f in out_dir.iterdir()}
    n, T = bench.N_ENVS, bench.T_STEPS
    cols = np.sort(np.random.default_rng(0).choice(n, size=64, replace=False))
    assert np.array_equal(bench.dump_columns(n, 1), cols)
    assert {k: v.shape for k, v in got.items()} == {"rewards": (T, 64), "dones": (T, 64), "state": (64, 4), "step_count": (64,), "episode": (64,)}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert np.array_equal(got["rewards"], np.broadcast_to(1000 * last_timed + cols, (T, 64)).astype(np.float32))
    assert np.array_equal(got["state"], np.broadcast_to(cols[:, None], (64, 4)).astype(np.float32))
    assert got["dones"][T - 1].all() and not got["dones"][: T - 1].any()  # the fake tape's one truncation row


def test_failed_section_keeps_its_objects_until_the_process_leaves(bench, monkeypatch, capsys):
    """A section that fails with a device error: the error is in the line, and what the failed section's frames held is not freed before
    bench.py leaves through os._exit(0) — after a device error such a free can abort the process before the line is printed."""
    freed, exits = [], []

    class Held:
        def __del__(self):
            freed.append(True)

    def failing(*a, **kw):
        held = Held()  # noqa: F841  (a tensor of the section in a real failure)
        raise RuntimeError("CUDA error: an illegal memory access was encountered")

    monkeypatch.setattr(bench, "td3_update_extras", failing)
    monkeypatch.setattr(bench, "FAILED_SECTIONS", [])
    monkeypatch.setattr(os, "_exit", lambda code: exits.append((code, list(freed))))
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "2", "--warmup", "3"])
    bench.main()
    out = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(out) == 1 and "illegal memory access" in json.loads(out[0])["extras"]["updates_error"]
    assert exits == [(0, [])]  # left through os._exit(0), nothing of the failed section freed before


def test_hard_stop_prints_the_line_and_leaves_with_zero(bench, monkeypatch, capsys):
    """A section that never returns: the timer prints the line already assembled (with sections_timeout_s) and exits 0."""
    left = []

    def fake_exit(code):
        left.append(code)

    monkeypatch.setattr(os, "_exit", fake_exit)
    stop = bench.HardStop(0.05, rank=0)
    line = {"metric": "m", "value": 1.0}
    stop.start(line)
    stop.timer.join(5.0)
    out = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert left == [0] and len(out) == 1 and json.loads(out[0]) == {"metric": "m", "value": 1.0, "sections_timeout_s": 0.05}
    stop.emit(line)  # the normal path afterwards must not print a second line
    assert not [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    # ranks other than 0 leave silently
    quiet = bench.HardStop(0.05, rank=3)
    quiet.start(None)
    quiet.timer.join(5.0)
    assert left == [0, 0] and not capsys.readouterr().out.strip()


def test_numa_binding_never_raises(bench, monkeypatch):
    """Host placement is an optimisation: on a box without the sysfs entries (or without a GPU) it reports why and changes nothing."""
    before = os.sched_getaffinity(0)
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda i: types.SimpleNamespace(pci_domain_id=0, pci_bus_id=0xfe, pci_device_id=0x1f))
    info = bench.bind_to_gpu_numa_node(torch, 0)
    assert info["bound"] is False and "note" in info and os.sched_getaffinity(0) == before
    np.testing.assert_equal(bench.workload_config(4)["parallelism"], "env-shard x4")


def test_two_ranks_one_line(tmp_path):
    """torchrun, two ranks (gloo stands in for NCCL through CSTR_BENCH_BACKEND): rank 0 prints the one line with per-rank entries and the
    data-parallel rows for every mode, rank 1 prints nothing, both exit 0."""
    import subprocess

    worker = tmp_path / "worker.py"
    worker.write_text(
        "import sys, pytest\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})\n"
        "import test_bench_dryrun as T\n"
        "b = T.install_fakes(pytest.MonkeyPatch())\n"
        "b.DUMP_REACTORS = 64\n"
        f"sys.argv = ['bench.py', '--gpus', '2', '--steps', '3', '--warmup', '3', '--dump-outputs', {str(tmp_path / 'dump')!r}]\n"
        "b.main()\n")
    env = dict(os.environ, CSTR_BENCH_BACKEND="gloo", OMP_NUM_THREADS="1")
    import socket

    with socket.socket() as sock:  # a port that is free right now
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), str(worker)], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    out = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(out) == 1, r.stdout[-2000:]
    line = json.loads(out[0])
    assert BASE_KEYS <= set(line) and line["n_gpus"] == 2 and line["cpu_baseline"] is None
    assert len(line["run"]["per_rank_ms_per_step"]) == 2 and len(line["e2e"]["per_rank_h2d_gbs"]) == 2
    assert line["run"]["host_placement"]["bound"] is False  # no such PCI device here: reported, not raised
    assert line["multi_rank_error"] is None and "sections_timeout_s" not in line and line["extras"] == {}
    assert line["rollout"]["strong_1048576_total"]["reactors_this_rank"] == 1 << 19
    row = line["dp_update"]["per_rank_batch_4096"]
    assert {"local_ms_per_update", "peer_ms_per_update", "nccl_eager_ms_per_update", "peer_over_local", "nccl_eager_over_local"} <= set(row)
    assert row["global_batch"] == 8192
    # --dump-outputs: each rank writes its own shard's sample, DUMP_REACTORS reactors over both ranks together
    dumped = {f.name: np.load(f) for f in (tmp_path / "dump").iterdir()}
    assert set(dumped) == {f"{k}_rank{r}.npy" for k in ("rewards", "dones", "state", "step_count", "episode") for r in (0, 1)}
    assert sum(dumped[f"state_rank{r}.npy"].shape[0] for r in (0, 1)) == 64 and dumped["rewards_rank1.npy"].shape == (8, 32)
