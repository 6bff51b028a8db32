"""Lattice build: single-pass vertex numbering and hash regions that are emptied by the build itself.

The build's hash scratch belongs to the context and is shared by every lattice built on it.  Each build empties the
slots it used instead of clearing the whole region first, so a context that builds lattices of different sizes and
feature dimensions, or a build that reports an error, must leave nothing behind that changes a later build.
"""
import numpy as np
import pytest

from util import assert_bit_exact, bits, tie_features

pytestmark = pytest.mark.gpu


def _cases():
    rng = np.random.default_rng(7)
    out = []
    # few vertices, rows of 10^4..10^5 entries (the appearance lattice of the SLAM workloads)
    out.append(("long_rows", (rng.random((60000, 2)) * 0.5).astype(np.float32)))
    # tens of thousands of vertices in one problem
    out.append(("many_vertices", (rng.random((100000, 2)) * 300.0).astype(np.float32)))
    # multi-level keys
    out.append(("d5", tie_features(rng, 20000, 5, 3.0)))
    # N mod 4 != 0: phantom lanes
    out.append(("small", tie_features(rng, 7, 2, 3.0)))
    out.append(("d7", tie_features(rng, 3001, 7, 2.0)))
    return out


def _run(pkg, ctx, f, x):
    lg = pkg.Lattice(ctx, f)
    off, bary, nbr = lg.export()
    y = lg.filter(x)
    V = lg.V
    lg.close()
    return V, off, bary, nbr, y


def _check(got, lo, yo, what):
    V, off, bary, nbr, y = got
    assert V == lo["V"], what
    assert np.array_equal(off, lo["offset"]), what
    assert np.array_equal(bits(bary), bits(lo["bary"])), what
    assert np.array_equal(nbr, lo["nbr"]), what
    assert_bit_exact(y, yo, what=what)


def test_one_context_large_small_large_matches_fresh_and_oracle(pkg, oracle):
    cases = _cases()
    rng = np.random.default_rng(8)
    xs = {name: (rng.random((f.shape[0], 2)) * 5 - 1).astype(np.float32) for name, f in cases}
    ref = {}
    for name, f in cases:
        lo = oracle.lattice(f)
        ref[name] = (lo, oracle.filter(lo, xs[name]))
    # large, small, multi-level, large again, with a failing build in between: one context throughout
    order = ["many_vertices", "small", "d5", "long_rows", "d7", "many_vertices", "small", "long_rows", "d5"]
    shared = pkg.Context(0)
    try:
        for i, name in enumerate(order):
            f = dict(cases)[name]
            if i == 4:
                with pytest.raises(pkg.LccrfError, match="short range"):
                    pkg.Lattice(shared, np.full((16, 2), 3.0e4, dtype=np.float32))
            lo, yo = ref[name]
            _check(_run(pkg, shared, f, xs[name]), lo, yo, "shared context, build %d (%s)" % (i, name))
            # every slot the build used (for d >= 4 also the earlier key levels) is empty again: a stale key would
            # change no output, only fill the table
            assert shared.build_scratch_in_use() == 0, (i, name)
    finally:
        shared.close()
    for name, f in cases:
        fresh = pkg.Context(0)
        try:
            lo, yo = ref[name]
            _check(_run(pkg, fresh, f, xs[name]), lo, yo, "fresh context (%s)" % name)
        finally:
            fresh.close()
    for lo, _ in ref.values():
        oracle.lattice_free(lo)


def test_rebuild_after_other_objects(pkg, oracle):
    """Rebuilding two lattices after a third (d = 6, multi-level keys) was built on the same context gives the same lattices."""
    rng = np.random.default_rng(9)
    fa = (rng.random((40000, 2)) * 0.5).astype(np.float32)
    fb = (rng.random((40000, 2)) * 200.0).astype(np.float32)
    c = pkg.Context(0)
    try:
        first = [_run(pkg, c, f, np.ones((f.shape[0], 1), np.float32)) for f in (fa, fb)]
        _run(pkg, c, tie_features(rng, 5000, 6, 2.0), np.ones((5000, 1), np.float32))
        assert c.build_scratch_in_use() == 0
        again = [_run(pkg, c, f, np.ones((f.shape[0], 1), np.float32)) for f in (fa, fb)]
    finally:
        c.close()
    for a, b in zip(first, again):
        assert a[0] == b[0]
        for u, v in zip(a[1:], b[1:]):
            assert np.array_equal(bits(u) if u.dtype == np.float32 else u, bits(v) if v.dtype == np.float32 else v)
