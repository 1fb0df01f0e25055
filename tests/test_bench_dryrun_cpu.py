"""Dry run of bench.py's own arm on the CPU: the real loop (warm-up, timed region, lanes, end-to-end host-buffer section,
JSON line) driven on the SIMT-emulated library with inert stand-ins for CUDA streams / events, at toy sizes.  It proves
nothing about speed; it keeps a typo in a rarely used branch of the measurement script from costing a GPU call."""
import contextlib
import json
import sys

import pytest
import torch

import simt_native


class _Stream:
    cuda_stream = 0

    def wait_stream(self, s):
        pass

    def wait_event(self, e):
        pass


class _Event:
    def __init__(self, enable_timing=False):
        pass

    def record(self, stream=None):
        pass

    def elapsed_time(self, other):
        return 1.0


def toy_configs(bench, setitem):
    """every bench config at a size the emulator affords"""
    for name, cfg in list(bench.CONFIGS.items()):
        toy = dict(cfg, N=16, lm_iter=2)
        if cfg["M"]:
            toy.update(M=8, I=2)
        setitem(bench.CONFIGS, name, toy)


def run_bench(monkeypatch, capsys, argv, **module_overrides):
    import bench
    simt_native.install(monkeypatch)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "Stream", lambda *a, **k: _Stream())
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: _Stream())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    monkeypatch.setattr(torch, "empty", (lambda f: (lambda *a, pin_memory=False, **k: f(*a, **k)))(torch.empty))
    monkeypatch.setenv("EPNP_BENCH_DEVICE", "cpu")
    monkeypatch.setenv("EPNP_NO_SAMPLER", "1")
    toy_configs(bench, monkeypatch.setitem)
    for k, v in dict(WARM_SECONDS=0.05, L2_BYTES=1.0, **module_overrides).items():
        monkeypatch.setattr(bench, k, v)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--batch", "2", "--steps", "3", "--warmup", "3", "--no-cpu-baseline"] + argv)
    bench.main()
    lines = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    return json.loads(lines[0])


CONTRACT = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "roofline", "clocks", "gpu_launches", "e2e")


@pytest.mark.parametrize("argv,overrides", [([], {}), (["--streams", "1"], {}), ([], {"E2E_LANES": 1, "E2E_CHUNKS": 0}),
                                            (["--no-e2e"], {}), (["--config", "lm_only"], {}), (["--config", "dense"], {}),
                                            (["--config", "train"], {})])
def test_bench_loop_runs_and_prints_the_contract_line(monkeypatch, capsys, argv, overrides):
    line = run_bench(monkeypatch, capsys, argv, **overrides)
    for k in CONTRACT:
        if k == "e2e" and "--no-e2e" in argv:
            continue
        assert k in line, k
    per_step = {"lm_only": 1, "train": 5}.get(argv[1] if "--config" in argv else "", 2)
    assert line["n_gpus"] == 1 and line["steps"] == 3 and line["gpu_launches"] == 3 * per_step and line["value"] > 0
    assert line["config"]["name"] == (argv[1] if "--config" in argv else "fused")
    assert line["config"]["batches_in_flight"] == (1 if "--streams" in argv else 2)
    assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    if "--no-e2e" not in argv:
        e = line["e2e"]
        assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] > 0
        assert e["calls_in_flight"] == overrides.get("E2E_LANES", 3)
        assert set(e["step_interval_ms"]) == {"min", "median", "max"}


def dump_outputs(monkeypatch, capsys, out_dir, argv, **module_overrides):
    import numpy as np
    run_bench(monkeypatch, capsys, argv + ["--dump-outputs", str(out_dir)], **module_overrides)
    return {p.stem: np.load(p) for p in sorted(out_dir.glob("*.npy"))}


@pytest.mark.parametrize("config", ["fused", "train"])
def test_dump_outputs_is_the_last_timed_step(monkeypatch, capsys, tmp_path, config):
    """--dump-outputs writes what the last timed step returned, in float32 / float64: the same arguments give the same
    arrays (seeded inputs, AMIS seed = step index), and one more timed step gives a different last step."""
    import numpy as np
    argv = ["--config", config, "--no-e2e"]
    a = dump_outputs(monkeypatch, capsys, tmp_path / "a", argv)
    b = dump_outputs(monkeypatch, capsys, tmp_path / "b", argv)
    c = dump_outputs(monkeypatch, capsys, tmp_path / "c", argv + ["--steps", "4"])
    grads = ("gx3d", "gx2d", "gw2d")
    assert set(a) == ({"loss", *grads} if config == "train" else {"pose_opt", "pose_cov", "cost", "pose_samples", "logw"})
    for name, arr in a.items():
        assert arr.dtype in (np.float32, np.float64) and np.isfinite(arr).all(), name
        assert np.array_equal(arr, b[name]), name
    for name in (grads if config == "train" else ("logw",)):
        assert np.abs(a[name]).max() > 0 and not np.array_equal(a[name], c[name]), name


def test_dump_outputs_samples_the_same_objects_of_every_array_above_the_cap(monkeypatch, capsys, tmp_path):
    import numpy as np
    argv = ["--batch", "8", "--no-e2e"]
    full = dump_outputs(monkeypatch, capsys, tmp_path / "full", argv)
    cap = sum(p.stat().st_size for p in (tmp_path / "full").glob("*.npy")) // 2
    part = dump_outputs(monkeypatch, capsys, tmp_path / "part", argv, DUMP_MAX_BYTES=cap)
    assert set(part) == set(full) and sum(p.stat().st_size for p in (tmp_path / "part").glob("*.npy")) <= cap
    keep = part["pose_opt"].shape[0]
    assert 0 < keep < 8
    idx = np.sort(np.random.default_rng(0).choice(8, size=keep, replace=False))
    for name, arr in part.items():
        assert np.array_equal(arr, full[name][idx]), name


def test_reference_arm_times_exactly_the_requested_steps(monkeypatch, capsys):
    """--impl reference runs K timed steps however large K is; only the length of a step's slice adapts."""
    import bench
    asked = []
    monkeypatch.setattr(bench, "cpu_reference_rates",
                        lambda cfg, steps, warmup, per_step: asked.append((steps, warmup)) or ([10.0] * steps, 8, "port", "stub"))
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "400", "--warmup", "3"])
    bench.main()
    line = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    assert asked == [(400, 3)] and line["steps"] == 400


@pytest.mark.parametrize("argv", [[], ["--config", "dense"], ["--streams", "1"]])
def test_both_arms_name_the_same_config(monkeypatch, capsys, argv):
    """`--impl reference` must report the workload of `--impl ours` word for word (the driver pairs the two lines by
    metric / unit / config); what is specific to the CPU arm's sampling lives in its cpu_baseline block."""
    import bench
    ours = run_bench(monkeypatch, capsys, ["--no-e2e"] + argv)
    monkeypatch.setattr(bench, "cpu_reference_rates", lambda cfg, steps, warmup, per_step: ([10.0] * steps, 8, "reference+shim", "stub"))
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--batch", "2", "--steps", "3", "--warmup", "3"] + argv)
    bench.main()
    ref = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    assert ref["impl"] == "reference" and ref["gpu_launches"] == 0
    for k in ("metric", "unit", "higher_is_better", "config", "scaling", "dtype", "data"):
        assert ref[k] == ours[k], k
    assert ref["cpu_baseline"]["kind"] == "reference+shim" and ref["e2e"]["value"] == ref["value"]


@pytest.mark.parametrize("flags", [["--gather", "nccl"], ["--gather", "push"], ["--gather", "push", "--streams", "1"]])
def test_two_rank_bench_loop_over_gloo(flags):
    """bench.py --gpus 2 as torchrun would start it, on the CPU: gloo instead of NCCL, shared-memory host tensors instead
    of CUDA IPC (tests/bench_dryrun_worker.py).  Rank 0 must print the one JSON line; every rank must exit 0."""
    import os
    import socket
    import subprocess
    simt_native.build_emulated(())
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    here = os.path.dirname(os.path.abspath(__file__))
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(here, "bench_dryrun_worker.py"), "--gpus", "2"] + flags,
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=300) for p in procs]
    for p, (out, err) in zip(procs, outs):
        assert p.returncode == 0, err[-3000:]
    lines = [l for l in outs[0][0].splitlines() if l.startswith("{")]
    assert len(lines) == 1 and not [l for l in outs[1][0].splitlines() if l.startswith("{")]
    line = json.loads(lines[0])
    assert line["n_gpus"] == 2 and line["config"]["global_batch"] == 4 and line["gpu_launches"] == 20
    assert flags[1] in line["config"]["parallelism"]


def test_bench_configs_script_runs_in_toy_mode(monkeypatch, capsys):
    """tools/bench_configs.py with every optional section switched on, at toy sizes on the emulated library."""
    import importlib.util
    import os
    simt_native.install(monkeypatch)
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    for k in ("EPNP_BENCH_CONFIGS_TOY", "EPNP_BENCH_RSLM", "EPNP_BENCH_GN_PLUS", "EPNP_BENCH_MC_EPILOGUE"):
        monkeypatch.setenv(k, "1")
    monkeypatch.setenv("EPNP_BENCH_DEVICE", "cpu")
    from epropnp import monte_carlo_pose_loss as mcl
    monkeypatch.setattr(mcl, "_use_native", lambda t: os.environ.get("EPNP_NATIVE_MC_EPILOGUE", "0") == "1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_configs_toy", os.path.join(root, "tools", "bench_configs.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.main()
    rows = [json.loads(l) for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    names = " | ".join(r["config"] for r in rows)
    for needle in ("#2 LM", "#3 LM", "#4 dense", "Det:", "training step", "evaluate_pnp cost", "RSLM init", "pose_opt_plus",
                   "MC pose loss"):
        assert needle in names, needle
    assert all(v > 0 for r in rows for k, v in r.items() if k.startswith("ms"))


def test_graft_entry_smoke_runs_on_the_emulated_library(monkeypatch, capsys):
    """__graft_entry__.smoke() (the driver's round-end check on cuda:0) executed unchanged, with the emulated library
    and `cuda:0` mapped to the host: its own assertions against the fp64 oracle must hold."""
    import __graft_entry__ as entry
    simt_native.install(monkeypatch)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    real_device = torch.device

    class _Dev:
        def __call__(self, *a, **k):
            return real_device("cpu") if a and str(a[0]).startswith("cuda") else real_device(*a, **k)

        def __instancecheck__(self, obj):
            return isinstance(obj, real_device)
    import torch as _t
    monkeypatch.setattr(_t, "device", _Dev())
    try:
        entry.smoke()
    finally:
        monkeypatch.undo()
    assert "smoke:" in capsys.readouterr().out
