"""bench.py --dump-outputs: the files hold what the timed steps computed -- the counts of the JSON line and, row for row,
the mesh an engine run of the same field returns."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_mesh_of_the_timed_steps(engine, tmp_path):
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    n = 64
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--n", str(n),
                          "--no-e2e", "--no-c5", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3
    got = {name: np.load(os.path.join(tmp_path, name + ".npy")) for name in ("counts", "verts", "normals", "tris")}
    assert got["counts"].dtype == np.float64 and got["counts"].tolist() == [line["n_verts"], line["n_tris"]]
    # the bench's field and call (one GPU: the whole n^3 volume, fp32 geometry with normals)
    field = synthetic.ct_like(n, device="cuda")
    torch.cuda.synchronize()
    c = engine.mt3d_run(field.data_ptr(), 0.5, shape=tuple(field.shape), dtype=np.float32, flags=E.WANT_NORMALS)
    want = engine.mt3d_fetch()
    assert (c.n_verts, c.n_tris) == (line["n_verts"], line["n_tris"]) and c.n_tris > 0
    assert got["verts"].dtype == np.float32 and np.array_equal(got["verts"], want["verts"])
    assert got["normals"].dtype == np.float32 and np.array_equal(got["normals"], want["normals"])
    assert got["tris"].dtype == np.float64 and np.array_equal(got["tris"], want["tris"])
