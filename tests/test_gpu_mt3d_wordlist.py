"""GPU parity of stage 2's interesting-word list at its edges: rows whose word count is no multiple of 4 (the one-word
quick test of k_count_a), a row's last word when the row length is no multiple of 32, the last row and plane (absent
neighbour rows), slab runs, near-flagged words everywhere, more than 8192 tiles (the tile prefix in k_tile_scan3), and
a word list that overflows its first capacity."""
import numpy as np
import pytest

from test_gpu_mt3d import run_and_compare

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(17, 13, 70), (9, 21, 100), (11, 6, 120), (8, 10, 33), (7, 9, 161)],
                         ids=["W3", "W4_tail4", "W4_tail24", "W2", "W6_tail1"])
def test_row_lengths_and_borders(engine, shape):
    """W = 3, 4, 4, 2, 6 words per row, every row's last word partial; the surface reaches the last plane and the last
    row of every plane."""
    rng = np.random.default_rng(sum(shape) + 1)
    f = rng.standard_normal(shape)
    c, o, r = run_and_compare(engine, f, 0.1)
    assert c.n_tris > 0
    assert r["pos"][:, 0].max() == shape[0] - 1 and r["pos"][:, 1].max() == shape[1] - 1


@pytest.mark.parametrize("n2", [70, 124])
def test_near_flagged_words(engine, n2):
    """Integer samples at an integer isovalue: a third of the samples equal it, so nearly every word carries the near
    flag and k_count_b takes the exact paths and its own work-list slots."""
    rng = np.random.default_rng(n2)
    f = rng.integers(0, 3, size=(15, 22, n2)).astype(np.float64)
    run_and_compare(engine, f, 1.0)


@pytest.mark.parametrize("n2", [70, 96])
def test_slab_runs_match_single_run(engine, n2):
    """z-slabs with halo planes (i_lo / i_hi / plane_offset): the planes from i_hi on are listed for their vertex ids
    only; near-flagged words in every slab."""
    from contourist_b200 import engine as E
    rng = np.random.default_rng(n2 + 3)
    g = np.linspace(-1, 1, 41)
    X, Y, Z = np.meshgrid(g, g[:29], np.linspace(-1, 1, n2), indexing="ij")
    f = (np.sin(4 * X) * np.cos(3 * Y) + Z * Z + 0.05 * rng.standard_normal(X.shape)).astype(np.float32)
    f[:, :, ::7] = np.round(f[:, :, ::7] * 4) / 4       # samples equal to the isovalue: near-flagged words in every slab
    flags = E.WANT_KEYS | E.WANT_NORMALS | E.GEOM_F64
    engine.mt3d_run(f, 0.25, flags=flags)
    ref = engine.mt3d_fetch()
    n0 = f.shape[0]
    for nshard in (2, 5):
        bounds = [round(r * n0 / nshard) for r in range(nshard + 1)]
        keys, verts, tris, voff = [], [], [], 0
        for r in range(nshard):
            a, b = bounds[r], bounds[r + 1]
            lo, hi = max(a - 1, 0), min(b + 2, n0)
            c = engine.mt3d_run(np.ascontiguousarray(f[lo:hi]), 0.25, flags=flags, i_lo=a - lo, i_hi=b - lo, plane_offset=lo)
            o = engine.mt3d_fetch()
            keys.append(o["keys"]); verts.append(o["verts"])
            tris.append(o["tris"].astype(np.int64) + voff)
            voff += c.n_verts
        assert np.array_equal(np.concatenate(keys), ref["keys"])
        assert np.array_equal(np.concatenate(verts), ref["verts"])
        assert np.array_equal(np.concatenate(tris), ref["tris"].astype(np.int64))


@pytest.mark.parametrize("shape", [(30, 64, 300), (30, 40, 500)], ids=["W10", "W16"])
def test_word_list_overflows_first_capacity(engine, shape):
    """A fresh context guesses max(words / 4, 16384) list entries; in a noise field nearly every one of its ~19 K words
    is interesting, so the entries past the capacity are skipped and the run is redone with a larger list."""
    from contourist_b200 import engine as E
    rng = np.random.default_rng(shape[2])
    f = rng.standard_normal(shape)
    fresh = E.Engine(0)
    try:
        run_and_compare(fresh, f, 0.0)
    finally:
        fresh.close()


def test_more_than_8192_tiles_matches_slab_runs(engine):
    """640 x 512 x 864 samples = 8.8 M words = 8640 tiles of 1024 words: the tile prefix runs in k_tile_scan3.  Two slab
    runs of half the planes each (4320 tiles: the fused prefix) must give the same mesh."""
    import torch
    from contourist_b200 import engine as E
    n0, n1, n2 = 640, 512, 864
    dev = torch.device("cuda", 0)
    x = torch.linspace(-1, 1, n0, device=dev, dtype=torch.float32)[:, None, None]
    y = torch.linspace(-1, 1, n1, device=dev, dtype=torch.float32)[None, :, None]
    z = torch.linspace(-1, 1, n2, device=dev, dtype=torch.float32)[None, None, :]
    f = (x * x + y * y + z * z + 0.05 * torch.sin(9 * x) * torch.cos(7 * z)).contiguous()
    torch.cuda.synchronize()
    flags = E.WANT_KEYS | E.WANT_NORMALS | E.GEOM_F64
    c = engine.mt3d_run(f.data_ptr(), 0.6, shape=(n0, n1, n2), dtype=np.float32, flags=flags)
    ref = engine.mt3d_fetch()
    assert c.n_tris > 100000
    half = n0 // 2
    plane = n1 * n2
    c_a = engine.mt3d_run(f.data_ptr(), 0.6, shape=(half + 2, n1, n2), dtype=np.float32, flags=flags, i_lo=0, i_hi=half)
    o_a = engine.mt3d_fetch()
    c_b = engine.mt3d_run(f.data_ptr() + 4 * plane * (half - 1), 0.6, shape=(n0 - half + 1, n1, n2), dtype=np.float32,
                          flags=flags, i_lo=1, i_hi=n0 - half + 1, plane_offset=half - 1)
    o_b = engine.mt3d_fetch()
    assert (c_a.n_verts + c_b.n_verts, c_a.n_tris + c_b.n_tris) == (c.n_verts, c.n_tris)
    assert c_a.n_active_cells + c_b.n_active_cells == c.n_active_cells
    assert np.array_equal(np.concatenate([o_a["keys"], o_b["keys"]]), ref["keys"])
    assert np.array_equal(np.concatenate([o_a["verts"], o_b["verts"]]), ref["verts"])
    tris = np.concatenate([o_a["tris"].astype(np.int64), o_b["tris"].astype(np.int64) + c_a.n_verts])
    assert np.array_equal(tris, ref["tris"].astype(np.int64))
    del f
    torch.cuda.empty_cache()
