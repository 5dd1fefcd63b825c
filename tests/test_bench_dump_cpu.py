"""bench.py --dump-outputs without a GPU: the sample of a large mesh is fixed, keeps verts and normals on the same rows,
stays under 64 MB at the row cap, and the arguments that cannot work are refused."""
import os
import subprocess
import sys
import types

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_sample_is_fixed_and_row_aligned(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_ROWS", 1000)
    V, T = 5000, 9000
    verts = np.arange(V * 3, dtype=np.float32).reshape(V, 3)
    mesh = {"verts": verts, "normals": -verts, "tris": np.arange(T * 3, dtype=np.int32).reshape(T, 3) % V}
    counts = types.SimpleNamespace(n_verts=V, n_tris=T)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), counts, mesh)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["counts.npy", "normals.npy", "tris.npy", "verts.npy"]
    for name in names:
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name))
    got = {name[:-4]: np.load(tmp_path / "a" / name) for name in names}
    assert got["counts"].dtype == np.float64 and got["counts"].tolist() == [V, T]
    assert got["verts"].dtype == np.float32 and got["verts"].shape == (1000, 3)
    assert np.array_equal(got["normals"], -got["verts"])
    rows = got["verts"][:, 0].astype(np.int64) // 3
    assert np.all(np.diff(rows) > 0)
    assert got["tris"].dtype == np.float64 and got["tris"].shape == (1000, 3)

def test_row_cap_keeps_the_dump_under_64_mb():
    # fp32 verts and normals (12 B a row), fp64 triangles (24 B a row), headers and counts
    assert bench.DUMP_ROWS * (12 + 12 + 24) + 4 * 128 + 16 <= 64e6


def test_all_rows_below_the_cap(tmp_path):
    mesh = {"verts": np.ones((7, 3), np.float32), "normals": None, "tris": np.zeros((4, 3), np.int32)}
    bench.dump_outputs(str(tmp_path), types.SimpleNamespace(n_verts=7, n_tris=4), mesh)
    assert sorted(os.listdir(tmp_path)) == ["counts.npy", "tris.npy", "verts.npy"]
    assert np.load(tmp_path / "verts.npy").shape == (7, 3) and np.load(tmp_path / "tris.npy").shape == (4, 3)


def test_arguments_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, capture_output=True,
                           text=True, timeout=120)
        assert p.returncode == 2 and "error" in p.stderr
