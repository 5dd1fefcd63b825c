"""tools/benchkit.py and the benchmarks built on it: what needs no GPU (the kernel table on fake profiler events, the
gpu_info fallback, the JSON line, and every script's --help)."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import benchkit  # noqa: E402

SCRIPTS = ["bench_attributes", "bench_cap", "bench_clip", "bench_closest", "bench_components", "bench_decimate",
           "bench_dtypes", "bench_keep_components", "bench_raycast", "bench_section", "bench_smooth",
           "bench_stage1_paths", "stage2_kernels"]


def fake_profiler(monkeypatch, events, device_time):
    """torch.profiler.profile returning `events` (with device_time_total, or only the older cuda_time_total) and a
    torch.cuda.synchronize that does nothing"""
    import torch
    import torch.profiler

    class Profile:
        def __init__(self, activities):
            pass

        def __enter__(self):
            return self

        def __exit__(self, *exc):
            return False

        def key_averages(self):
            field = "device_time_total" if device_time else "cuda_time_total"
            return [SimpleNamespace(key=k, count=c, **{field: t}) for k, c, t in events]

    monkeypatch.setattr(torch.profiler, "profile", Profile)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda: None)


EVENTS = [("void (anonymous namespace)::k_cap_faces<double>(Grid<double>, int)", 3, 10.0),
          ("void (anonymous namespace)::k_flag_scan<unsigned char>(unsigned char const*, long)", 2, 7.0),
          ("void cub::CUB_200700_1000_NS::DeviceRadixSortOnesweepKernel<Policy, false>(unsigned long*)", 4, 9.0),
          ("Memcpy DtoH (Device -> Pageable)", 2, 5.0),
          ("Memset (Device)", 0, 1.5),
          ("void at::native::vectorized_elementwise_kernel<4>(int)", 5, 50.0),
          ("cudaLaunchKernel", 9, 0.0)]


@pytest.mark.parametrize("device_time", [True, False])
def test_kernel_table_filters_shortens_and_rounds(monkeypatch, device_time):
    fake_profiler(monkeypatch, EVENTS, device_time)
    log = []
    table = benchkit.kernel_table(lambda: log.append("call"), ("k_cap_", "k_flag_scan", "DeviceRadixSort", "Memcpy",
                                                               "Memset"), setup=lambda: log.append("setup"), reps=3)
    assert log == ["setup", "call", "call", "call"]
    assert table == {"k_cap_faces": dict(launches=3, us_per_launch=3.33),
                     "k_flag_scan": dict(launches=2, us_per_launch=3.5),
                     "DeviceRadixSortOnesweepKernel": dict(launches=4, us_per_launch=2.25),
                     "Memcpy DtoH (Device -> Pageable)": dict(launches=2, us_per_launch=2.5),
                     "Memset (Device)": dict(launches=0, us_per_launch=1.5)}


def test_kernel_table_key_function(monkeypatch):
    fake_profiler(monkeypatch, EVENTS, True)
    table = benchkit.kernel_table(lambda: None, ("k_cap_", "Memset"), key=lambda key, tag: (tag, key[:10]))
    assert table == {("k_cap_", "void (anon"): dict(launches=3, us_per_launch=3.33),
                     ("Memset", "Memset (De"): dict(launches=0, us_per_launch=1.5)}


def test_gpu_info_without_nvidia_smi(monkeypatch, tmp_path):
    monkeypatch.setenv("PATH", str(tmp_path))
    info = benchkit.gpu_info()
    assert info["name"] is None and info["power_limit"] is None and info["error"]


def test_gpu_info_reads_name_and_power_limit(monkeypatch):
    monkeypatch.setattr(subprocess, "run", lambda *a, **k: SimpleNamespace(stdout="NVIDIA B200, 1000.00 W\n"))
    assert benchkit.gpu_info() == dict(name="NVIDIA B200", power_limit="1000.00 W")


def test_emit_prints_and_writes_one_line(tmp_path, capsys):
    res = dict(tool="bench_x", gpu=dict(name=None), cases={"fp32": [0.25, 1]})
    out = tmp_path / "res.json"
    benchkit.emit(res, str(out))
    assert capsys.readouterr().out == json.dumps(res) + "\n"
    assert out.read_text() == json.dumps(res) + "\n"
    benchkit.emit(res, None)
    assert capsys.readouterr().out == json.dumps(res) + "\n"


@pytest.mark.parametrize("script", SCRIPTS)
def test_script_help(script):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", script + ".py"), "--help"], capture_output=True,
                       text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.startswith("usage: %s.py" % script)
