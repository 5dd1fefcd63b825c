"""tools/stage2_kernels.py: the per-kernel times it reads from a chrome trace (no GPU needed)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import stage2_kernels  # noqa: E402


def test_kernel_times_keeps_k_kernels_in_launch_order(tmp_path):
    ev = [{"cat": "kernel", "name": "void (anonymous namespace)::k_count_b<float>(Grid<float>, unsigned int)", "dur": 60.0},
          {"cat": "cpu_op", "name": "k_count_b", "dur": 5.0},
          {"cat": "kernel", "name": "void at::native::elementwise_kernel<128, 4>()", "dur": 3.0},
          {"cat": "kernel", "name": "void (anonymous namespace)::k_scan<float>(Grid<float>)", "dur": 20.0},
          {"cat": "kernel", "name": "void (anonymous namespace)::k_count_b<float>(Grid<float>, unsigned int)", "dur": 70.0}]
    p = tmp_path / "trace.json"
    p.write_text(json.dumps({"traceEvents": ev}))
    per = stage2_kernels.kernel_times(str(p))
    assert list(per) == ["k_count_b", "k_scan"]
    assert per["k_count_b"] == [60.0, 70.0] and per["k_scan"] == [20.0]
