"""Host-side pieces of bench.py that can run without a GPU: the clock sampler's windowing (against a fake nvidia-smi), the
reference arm's JSON line (the CPU path timed beside the GPU arm), argument checks, the --dump-outputs row sample, and the
multi-rank exit path."""
import importlib.util
import json
import os
import stat
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture
def fake_nvidia_smi(tmp_path, monkeypatch):
    """A stand-in that needs 0.3 s to come up (like the real tool on an 8-GPU box) and then prints one CSV row per 100 ms."""
    exe = tmp_path / "nvidia-smi"
    exe.write_text("#!/bin/bash\nsleep 0.3\nwhile true; do echo '1695, 1965, 801.2, Not Active, Not Active, Not Active, Active'; sleep 0.1; done\n")
    exe.chmod(exe.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{tmp_path}:{os.environ['PATH']}")


def test_clock_sampler_uses_rows_of_the_timed_region(fake_nvidia_smi):
    b = _bench()
    with b.ClockSampler(0) as c:
        time.sleep(0.5)                     # "warm-up": the sampler is already streaming
        c.mark_start()
        time.sleep(0.55)
        c.mark_end()
    s = c.summary()
    assert s["window"] == "timed region" and 3 <= s["samples"] <= 7
    assert s["sm_mhz"] == 1695 and s["sm_max_mhz"] == 1965 and s["reasons"] == ["sw_power_cap"]


def test_clock_sampler_falls_back_to_the_warm_up_rows_for_a_short_timed_region(fake_nvidia_smi):
    b = _bench()
    with b.ClockSampler(0) as c:
        time.sleep(0.65)
        c.mark_start()
        time.sleep(0.005)                   # an N = 8 timed region can be shorter than one sample period
        c.mark_end()
    s = c.summary()
    assert s["samples"] >= 1 and s["window"].startswith("warm-up + timed region") and s["sm_mhz"] == 1695


def test_clock_sampler_without_nvidia_smi_reports_unavailable(tmp_path, monkeypatch):
    monkeypatch.setenv("PATH", str(tmp_path))            # no nvidia-smi anywhere
    b = _bench()
    with b.ClockSampler(0) as c:
        c.mark_start()
        c.mark_end()
    assert c.summary() == {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference`: the reference's CPU-runnable path (dense SDPA of one block per timed step) on the host cores;
    same metric / unit / config keys as the GPU arm, impl tag, cpu_baseline and a zero-copy e2e object."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "frames_per_sec_4step_81f" and line["unit"] == "frames/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["config"]["L"] == 32760 and line["config"]["heads"] == 12


@pytest.mark.parametrize("argv,message", [(["--steps", "0"], "--steps must be at least 1"),
                                          (["--impl", "reference", "--dump-outputs", "unused"], "--dump-outputs writes the output of")])
def test_bad_arguments_are_refused(argv, message):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert out.returncode == 2 and message in out.stderr


def test_output_sample_is_a_fixed_sorted_row_sample_within_the_budget(monkeypatch):
    import torch
    b = _bench()
    y = torch.arange(1000, dtype=torch.float32)[:, None].repeat(1, 8)     # every row holds its own index
    monkeypatch.setattr(b, "DUMP_BYTES", 100 * 8 * 4)
    s = b.output_sample(y, 1000, 0, 1)
    assert s.dtype == torch.float32 and s.shape == (100, 8) and torch.equal(s, y[s[:, 0].long()])
    assert (s[1:, 0] > s[:-1, 0]).all() and torch.equal(s, b.output_sample(y, 1000, 0, 1))
    monkeypatch.setattr(b, "DUMP_BYTES", 1 << 20)                          # an output within the budget is written whole
    assert torch.equal(b.output_sample(y, 1000, 0, 1), y)


_SAMPLE_SCRIPT = """
import importlib.util, os, sys
import torch, torch.distributed as dist
spec = importlib.util.spec_from_file_location("bench_module", sys.argv[1]); b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=2)
b.DUMP_BYTES = 100 * 8 * 4
y = torch.arange(1000, dtype=torch.float32)[:, None].repeat(1, 8)
row0, row1 = (0, 640) if dist.get_rank() == 0 else (640, 1000)
s = b.output_sample(y[row0:row1], 1000, row0, 2)
if dist.get_rank() == 0:
    print("SAMPLE", torch.equal(s, b.output_sample(y, 1000, 0, 1)), flush=True)
dist.destroy_process_group()
"""


def test_output_sample_reassembles_the_row_shards_of_two_ranks(tmp_path):
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "sample.py"
    script.write_text(_SAMPLE_SCRIPT)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), GLOO_SOCKET_IFNAME="lo")
        procs.append(subprocess.Popen([sys.executable, str(script), os.path.join(ROOT, "bench.py")], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=120) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-500:] for o in outs]
    assert "SAMPLE True" in outs[0][0]


_LEAVE_SCRIPT = """
import datetime, importlib.util, os, sys, time
import torch.distributed as dist
spec = importlib.util.spec_from_file_location("bench_module", sys.argv[1]); b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
g = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=60))
if dist.get_rank() == 0:
    time.sleep(0.5)
    print("LINE", flush=True)
b._leave(g)
print("NOT REACHED", flush=True)
"""


def test_multi_rank_exit_path_leaves_promptly(tmp_path):
    """bench._leave: flush, (GPU drain - absent here), gloo rendezvous, os._exit(0) without tearing communicators down."""
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "leave.py"
    script.write_text(_LEAVE_SCRIPT)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), GLOO_SOCKET_IFNAME="lo")
        procs.append(subprocess.Popen([sys.executable, str(script), os.path.join(ROOT, "bench.py")], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    t0 = time.time()
    outs = [p.communicate(timeout=120) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-500:] for o in outs]
    assert time.time() - t0 < 60 and "LINE" in outs[0][0] and all("NOT REACHED" not in o[0] for o in outs)
