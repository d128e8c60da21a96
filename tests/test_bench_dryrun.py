"""bench.py's control flow on CPU: the real run_b200() - argument handling, optimizer attach + fallback, graph / eager step,
device-timed and end-to-end (pipelined input copy) legs, roofline pass, JSON assembly - with the C-ABI calls answered by
tests/ops_emulator.py and torch.cuda's streams / events / graphs replaced by inert stand-ins. Nothing about speed is checked
here (the numbers are meaningless); the point is that an unverified edit to the bench cannot take the bench line down with a
NameError or a wrong keyword on the GPU box."""
import contextlib
import json
import os
import sys
import time

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class _Stream:
    def __init__(self, *a, **k):
        self.cuda_stream = 0

    def wait_stream(self, s):
        pass

    def wait_event(self, e):
        pass

    def synchronize(self):
        pass


class _Event:
    def __init__(self, enable_timing=False, **k):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)

    def synchronize(self):
        pass


class _Graph:
    def replay(self):
        pass


@contextlib.contextmanager
def _ctx(*a, **k):
    yield


@pytest.fixture
def bench_on_cpu(monkeypatch):
    """bench.py in this process, single rank, with torch.cuda's streams / events / graphs replaced by the inert stand-ins above
    and the device set to the CPU (the C-ABI calls are answered by ops_emulator.emulated_ops in each test)."""
    import bench
    cpu = torch.device("cpu")
    for name, val in (("Stream", _Stream), ("Event", _Event), ("CUDAGraph", _Graph), ("graph", _ctx), ("stream", _ctx),
                      ("current_stream", lambda *a: _Stream()), ("synchronize", lambda *a: None), ("set_device", lambda *a: None),
                      ("is_available", lambda: False)):
        monkeypatch.setattr(torch.cuda, name, val)
    monkeypatch.setattr(bench, "_device", lambda r: cpu)
    monkeypatch.setattr(bench, "_pin", lambda t: t)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    return bench


@pytest.mark.parametrize("flags", [["--graph", "1", "--size", "128"],
                                   ["--graph", "0", "--prefetch", "0", "--fused_loss", "1", "--recast_in_step", "1", "--clip_batching", "0",
                                    "--stem", "im2col", "--mn3d", "1", "--occ2", "2"]])
def test_bench_control_flow_on_cpu(bench_on_cpu, monkeypatch, capsys, flags):
    bench = bench_on_cpu
    from ops_emulator import emulated_ops
    argv = ["bench.py", "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", "2", "--n_clips", "2", "--n_frm", "1", "--size", "64",
            "--txt_len", "12", "--no_cpu", "1", "--overlap_wgrad", "0", "--opt_steps", "1"] + flags
    size = int(flags[flags.index("--size") + 1]) if "--size" in flags else 64
    monkeypatch.setattr(sys, "argv", argv)
    with emulated_ops(ignore_dropout=True) as calls:
        bench.main()
    out, err = capsys.readouterr()
    line = [l for l in out.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["unit"] == "clips/s" and d["config"]["clips_per_step_per_gpu"] == 4
    assert d["e2e"]["h2d_bytes_per_step"] == 2 * 2 * 3 * size * size + 2 * (2 * 12 * 8) + 2 * 8 and d["e2e"]["d2h_bytes_per_step"] == 4
    assert "error" not in d["roofline"], d["roofline"]
    assert d["roofline"]["launches_per_step"] == calls_per_step_expected(flags)
    # FusedAdamW is attached before the loop (its kernels are emulated too), unless the round-1 flow is asked for
    assert "could not be attached" not in err and "fused optimizer timing failed" not in err, err
    assert d["config"]["weight_recast"].startswith("inside every step" if "--recast_in_step" in flags else "in the optimizer step")
    assert d["fused_optimizer"]["params"] > 100e6
    assert ("pipelined input copy failed" not in err) and ("roofline pass failed" not in err), err
    assert d["e2e"]["input_copy"].startswith("copy stream" if "--prefetch" not in flags else "on the compute stream")
    assert calls["gemm"] > 0
    hb = d["roofline"]["hbm_bound_launch"]
    if size == 128 and "--clip_batching" not in flags:      # batched pass: 4 frames -> res2 rows = 4 * 32 * 32 = 4096: a candidate exists
        assert hb["bound"] == "hbm" and hb["algorithmic_bytes"] > 0 and hb["traffic"] is None and "error" not in hb, hb
    else:
        assert hb is None or "error" not in hb, hb


@pytest.mark.parametrize("config", ["c4", "c5"])
def test_bench_other_baseline_configs_on_cpu(bench_on_cpu, monkeypatch, capsys, config):
    """bench.py --config c4 (TGIF-QA multiple choice train step) and c5 (paragraph-retrieval inference: CNN once per video, one
    BERT pass over clips x captions) in miniature through the emulated ABI: the workload plumbing and the JSON line."""
    bench = bench_on_cpu
    from ops_emulator import emulated_ops
    small = {"c4": ["--batch", "2", "--n_ex", "3", "--txt_len", "12"], "c5": ["--n_clips", "3", "--n_ex", "2", "--txt_len", "70"]}[config]
    argv = ["bench.py", "--config", config, "--gpus", "1", "--steps", "2", "--warmup", "1", "--size", "64", "--no_cpu", "1", "--overlap_wgrad", "0",
            "--opt_steps", "1", "--graph", "0", "--prefetch", "0"] + small
    monkeypatch.setattr(sys, "argv", argv)
    with emulated_ops(ignore_dropout=True) as calls:
        bench.main()
    out, err = capsys.readouterr()
    d = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    assert d["config"]["name"] == config and d["unit"] == "clips/s" and d["value"] > 0
    assert "roofline pass failed" not in err and "error" not in d["roofline"], (err, d["roofline"])
    if config == "c4":
        assert "multiple choice" in d["metric"] and d["config"]["clips_per_step_per_gpu"] == 4 and d["fused_optimizer"] is not None
        assert calls["clip_lse_loss"] > 0
    else:
        assert "inference" in d["metric"] and d["config"]["clips_per_step_per_gpu"] == 3 and d["config"]["seq_len"] == 71
        assert d["fused_optimizer"] is None and calls["attention_bwd"] == 0 and calls["attention_fwd"] > 0


@pytest.mark.parametrize("graph", ["0", "1"])
def test_bench_dump_outputs_on_cpu(bench_on_cpu, monkeypatch, capsys, tmp_path, graph):
    """--dump-outputs DIR: after the timed steps the logits, loss and a seeded sample of the gradients of the last step land in
    DIR as float32 .npy files, under 64 MB, the loss is the one of those logits, and two runs with the same arguments write the
    same arrays. (The stand-in graph replays nothing, so this checks the plumbing; the GPU test below runs the real graph.)"""
    import types
    import numpy as np
    bench = bench_on_cpu
    from ops_emulator import emulated_ops
    runs = []
    for i in range(2):
        out = tmp_path / ("run%d" % i)
        monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", "2", "--n_clips", "2",
                                          "--n_frm", "1", "--size", "64", "--txt_len", "12", "--no_cpu", "1", "--overlap_wgrad", "0",
                                          "--opt_steps", "1", "--graph", graph, "--dump-outputs", str(out)])
        with emulated_ops(ignore_dropout=True):
            bench.main()
        capsys.readouterr()
        runs.append({f.name[:-4]: np.load(str(f)) for f in sorted(out.iterdir())})
    a, b = runs
    assert sorted(a) == ["grads", "logits", "loss"]
    assert a["logits"].shape == (2, 2, 2) and a["loss"].shape == (1,) and all(v.dtype == np.float32 for v in a.values())
    assert a["grads"].size > 100e6 / 32 and sum(v.nbytes for v in a.values()) <= 64 << 20     # 1/32 of > 100 M gradients
    assert np.isfinite(a["grads"]).all() and np.abs(a["grads"]).max() > 0
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    labels = bench.make_host_batch(types.SimpleNamespace(batch=2, n_clips=2, n_frm=1, size=64, n_ex=1, txt_len=12, head="retrieval"), 0)["labels"]
    assert abs(float(bench.lse_loss(torch.from_numpy(a["logits"]), labels)) - float(a["loss"][0])) < 1e-5


@pytest.mark.gpu
def test_bench_dump_outputs_with_the_cuda_graph_on_the_device(cuda, tmp_path):
    """bench.py --dump-outputs on the device, whole-step CUDA graph on: the graph is used, the dumped loss is the LSE loss of the
    dumped logits (both from one replay), and one more timed step changes what is written - dropout draws fresh masks at every
    replay - so the arrays come from the timed steps, not from the capture."""
    import subprocess
    import types
    import numpy as np
    import bench
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    runs = {}
    for steps in (3, 4):
        out = tmp_path / ("steps%d" % steps)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "2", "--batch", "4",
                            "--no_cpu", "1", "--opt_steps", "1", "--dump-outputs", str(out)], capture_output=True, text=True, env=env, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert d["steps"] == steps and d["config"]["cuda_graph"] is True and "capture failed" not in r.stderr, r.stderr[-3000:]
        runs[steps] = {f.name[:-4]: np.load(str(f)) for f in sorted(out.iterdir())}
    args = types.SimpleNamespace(batch=4, n_clips=2, n_frm=2, size=224, n_ex=1, txt_len=32, head="retrieval")
    labels = bench.make_host_batch(args, 0)["labels"]
    for a in runs.values():
        assert sorted(a) == ["grads", "logits", "loss"] and a["logits"].shape == (2, 4, 2)
        assert np.isfinite(a["grads"]).all() and np.abs(a["grads"]).max() > 0
        want = float(bench.lse_loss(torch.from_numpy(a["logits"]).double(), labels))
        assert abs(want - float(a["loss"][0])) < 1e-4 * max(1.0, abs(want)), (want, a["loss"])
    assert not np.array_equal(runs[3]["logits"], runs[4]["logits"]) and not np.array_equal(runs[3]["grads"], runs[4]["grads"])


@pytest.mark.parametrize("flags,steps,warmup",[(["--steps", "4", "--warmup", "0"], 4, 0), ([], 3, 1)])
def test_bench_reference_arm_times_the_steps_asked_for(bench_on_cpu, monkeypatch, capsys, flags, steps, warmup):
    """--impl reference (the CPU oracle) runs exactly --warmup untimed and --steps timed steps (defaults 1 and 3 there) and reports
    them; --dump-outputs, which writes the outputs of this repository's timed path, is refused with it."""
    bench = bench_on_cpu
    calls = []
    real = bench._cpu_step
    monkeypatch.setattr(bench, "_cpu_step", lambda *a: calls.append(1) or real(*a))
    base = ["bench.py", "--impl", "reference", "--cpu_batch", "1", "--n_clips", "1", "--n_frm", "1", "--size", "64", "--txt_len", "12"]
    monkeypatch.setattr(sys, "argv", base + flags)
    bench.main()
    d = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    assert d["impl"] == "reference" and d["steps"] == steps and d["warmup"] == warmup and len(calls) == steps + warmup
    monkeypatch.setattr(sys, "argv", base + ["--dump-outputs", "unused"])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2 and "--dump-outputs" in capsys.readouterr().err


def calls_per_step_expected(flags):
    # GEMM launches of one training step: CNN 53 convs forward + backward of res3-5 / grid_encoder, transformer 12 layers + heads;
    # the per-clip loop runs the whole thing once per clip
    per_pass = 291
    return per_pass * (2 if "--clip_batching" in flags else 1)


def _mg_worker(rank, world, port, flags, outdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    import bench
    from ops_emulator import emulated_ops
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // world))
    cpu = torch.device("cpu")
    for name, val in (("Stream", _Stream), ("Event", _Event), ("CUDAGraph", _Graph), ("graph", _ctx), ("stream", _ctx),
                      ("current_stream", lambda *a: _Stream()), ("synchronize", lambda *a: None), ("set_device", lambda *a: None),
                      ("is_available", lambda: False)):
        setattr(torch.cuda, name, val)
    bench._device, bench._pin = (lambda r: cpu), (lambda t: t)
    real_init = dist.init_process_group
    dist.init_process_group = lambda backend=None, **kw: real_init("gloo")        # NCCL -> gloo, no device_id
    # symmetric memory stand-ins for --exchange nvls: plain tensors, a handle whose "multicast pointer" is the local address,
    # barriers over gloo; ops_emulator.nvls_allreduce resolves the address back to the registered tensor
    import torch.distributed._symmetric_memory as symm
    import ops_emulator

    class _Handle:
        def __init__(self, t):
            self.multicast_ptr, self.rank, self.world_size = t.data_ptr(), rank, world
            ops_emulator.NVLS_BUFFERS[t.data_ptr()] = t

        def barrier(self, channel=0, timeout_ms=0):
            dist.barrier()
    symm.empty = lambda *size, dtype=None, device=None: torch.zeros(*size, dtype=dtype)
    symm.rendezvous = lambda t, group: _Handle(t)
    sys.argv = ["bench.py", "--gpus", str(world), "--steps", "2", "--warmup", "1", "--batch", "1", "--n_clips", "2", "--n_frm", "1",
                "--size", "64", "--txt_len", "12", "--overlap_wgrad", "0", "--graph", "0", "--optimizer", "0"] + flags
    sys.stdout = open(os.path.join(outdir, "rank%d.out" % rank), "w")
    sys.stderr = open(os.path.join(outdir, "rank%d.err" % rank), "w")
    with emulated_ops(ignore_dropout=True):
        bench.main()          # ends in os._exit(0) on every rank at world > 1


@pytest.mark.parametrize("flags", [["--exchange", "nccl", "--cnn_buckets", "0"], ["--fused_loss", "1"]])
def test_bench_control_flow_two_ranks_over_gloo(tmp_path, flags):
    """The N > 1 flow of bench.py (overlapped exchange hooks through the real engines, collectives in the timed region, rank 0
    reporting, every rank leaving through os._exit) with NCCL swapped for gloo, plus the mid-backward CNN bucket."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    port = 29500 + (os.getpid() + 733 + len(flags)) % 1000
    procs = [ctx.Process(target=_mg_worker, args=(r, 2, port, flags, str(tmp_path))) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0, (open(os.path.join(str(tmp_path), "rank0.err")).read()[-2000:], open(os.path.join(str(tmp_path), "rank1.err")).read()[-2000:])
    out0 = open(os.path.join(str(tmp_path), "rank0.out")).read()
    assert not open(os.path.join(str(tmp_path), "rank1.out")).read().strip()          # only rank 0 prints
    d = json.loads([l for l in out0.splitlines() if l.startswith("{")][-1])
    assert d["n_gpus"] == 2 and d["config"]["parallelism"] == "dp2" and d["config"]["clips_per_step_per_gpu"] == 2
    assert d["cpu_baseline"] is None and d["fused_optimizer"] is None
    # defaults at N > 1: this library's NVLS all-reduce where every rank has a multicast mapping (probed collectively; the stand-ins
    # here provide one), res5 + grid_encoder gradients exchanged mid-backward
    assert "error" not in d["roofline"] and d["config"]["cnn_buckets"] == ("--cnn_buckets" not in flags)
    assert d["config"]["exchange"] == ("nccl" if "nccl" in flags else "nvls")
