"""GPU: which pass on the device mesh of the last 3D run may follow which.  Every pass runs on a small full-volume run
after each editing pass, after orientation, after ctr_mt3d_offset_ids and on a slab run; each is accepted or refused
with its error code, and a refused pass leaves the mesh as it was."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

STATE, UNSUPPORTED = -5, -4
N = 17


def _E():
    from contourist_b200 import engine as E
    return E


def _field():
    g = np.linspace(-1.0, 1.0, N)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    return X * X + Y * Y + 1.3 * Z * Z


def _offset_ids(engine, base=7):
    engine._check(engine.lib.ctr_mt3d_offset_ids(engine.h, base), "ctr_mt3d_offset_ids")


def _keep_all(engine):
    _, tab = engine.mt3d_components()
    engine.mt3d_keep_components(np.ones(len(tab), bool))


SHAPE = np.array([N - 1] * 3)
PASSES = {
    "orient": lambda e, f: e.mt3d_orient_reference(),
    "components": lambda e, f: e.mt3d_components(),
    "smooth": lambda e, f: e.mt3d_smooth(2),
    "section": lambda e, f: e.mt3d_section((0.0, 0.0, 1.0), [8.0]),
    "decimate": lambda e, f: e.mt3d_decimate(2.0),
    "select": lambda e, f: e.mt3d_select_seeded(np.array([[8, 8, 3]], np.int32)),
    "clean": lambda e, f: e.mt3d_clean(SHAPE),
    "cap": lambda e, f: e.mt3d_cap("high"),
    "interpolate": lambda e, f: e.mt3d_interpolate(f),
    "offset_ids": lambda e, f: _offset_ids(e),
}
BEFORE = {
    "run": lambda e, f: None,
    "select": PASSES["select"],
    "clean": PASSES["clean"],
    "keep": lambda e, f: _keep_all(e),
    "smooth": PASSES["smooth"],
    "decimate": PASSES["decimate"],
    "cap": PASSES["cap"],
    "orient": PASSES["orient"],
    "offset_ids": PASSES["offset_ids"],
    "slab": lambda e, f: None,
}
# error code of each pass after each earlier step; a pass not listed is accepted
REFUSED = {
    "run": {},
    "select": {"select": STATE, "cap": STATE},
    "clean": {"select": STATE, "clean": STATE, "cap": STATE},
    "keep": {"select": STATE, "cap": STATE},
    "smooth": {"select": STATE, "clean": STATE},
    "decimate": {"select": STATE, "clean": STATE, "cap": STATE},
    "cap": {"select": STATE, "clean": STATE, "cap": STATE},
    "orient": {"cap": STATE},
    # the passes that build an edge table or clusters check the ids first
    "offset_ids": {"components": STATE, "smooth": STATE, "section": STATE, "decimate": STATE, "cap": STATE},
    "slab": {"components": STATE, "smooth": STATE, "section": STATE, "decimate": STATE, "select": UNSUPPORTED,
             "clean": UNSUPPORTED, "cap": STATE},
}
# orientation, selection and clean-up read the vertices through the triangle ids without checking them first: they are
# not run on ids that point past the vertices (after offset_ids, and a slab's halo ids)
SKIP = {"offset_ids": {"orient", "select", "clean"}, "slab": {"orient"}}


def _code(fn):
    E = _E()
    try:
        fn()
    except (E.EngineError, ValueError) as e:
        m = re.search(r"failed \((-?\d+)\)", str(e))
        return int(m.group(1)) if m else -1                 # ValueError: CTR_ERR_BAD_ARG
    return 0


@pytest.mark.parametrize("before", list(BEFORE))
def test_pass_order(engine, before):
    E = _E()
    field = _field()
    flags = E.WANT_KEYS | E.WANT_NORMALS
    for name, call in PASSES.items():
        if name in SKIP.get(before, ()):
            continue
        engine.mt3d_run(field, 0.5, flags=flags, i_hi=N // 2 if before == "slab" else None)
        BEFORE[before](engine, field)
        pre = engine.mt3d_fetch()
        want = REFUSED[before].get(name, 0)
        got = _code(lambda: call(engine, field))
        assert got == want, (before, name, got, engine.lib.ctr_last_error(engine.h).decode())
        if want:
            post = engine.mt3d_fetch()
            for k in pre:
                assert np.array_equal(pre[k], post[k]), (before, name, k)
