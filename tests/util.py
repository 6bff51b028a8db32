"""Shared helpers for the parity tests."""
import numpy as np

REL_TOL = 1e-4      # north_star: marginals within 1e-4 relative
NEAR_TIE = 1e-5     # north_star: MAP labels identical except at near-ties |dQ| < 1e-5


def rel_err(a, ref):
    """Element-wise relative error; exact zeros of the reference (fast_exp cut-off, densecrf3d.h:58)
    must be matched by exact zeros."""
    a = np.asarray(a, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    out = np.abs(a - ref) / np.maximum(np.abs(ref), 1e-300)
    out[(ref == 0) & (a == 0)] = 0.0
    return out


def assert_marginals(Q, Qref, tol=REL_TOL, what=""):
    r = rel_err(Q, Qref)
    assert np.isfinite(np.asarray(Q)).all(), f"{what}: non-finite marginals"
    assert r.max() <= tol, f"{what}: max relative marginal error {r.max():.3e} > {tol}"
    return float(r.max())


def assert_bit_exact(a, ref, what=""):
    """The CUDA path keeps the reference's operation order everywhere (splat rows in point order, blur and
    slice associations, fast_exp), so floating-point outputs are expected to be BIT-identical."""
    a, ref = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(ref, np.float32)
    assert a.shape == ref.shape, f"{what}: shape {a.shape} vs {ref.shape}"
    bad = int((a.view(np.int32) != ref.view(np.int32)).sum())
    assert bad == 0, f"{what}: {bad} of {a.size} values differ in bits (max rel {rel_err(a, ref).max():.3e})"


def assert_map(m, mref, Qref, what=""):
    """MAP labels identical except where the reference's top-2 marginals differ by < NEAR_TIE."""
    m, mref = np.asarray(m), np.asarray(mref)
    diff = np.nonzero(m != mref)[0]
    if diff.size == 0:
        return 0
    srt = np.sort(np.asarray(Qref)[diff], axis=1)
    gap = srt[:, -1] - srt[:, -2]
    assert (gap < NEAR_TIE).all(), f"{what}: {int((gap >= NEAR_TIE).sum())} MAP mismatches that are not near-ties"
    return int(diff.size)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def tie_features(rng, N, d, scale=3.0):
    """Random features with grid-aligned rows (rank ties / half-way rounding cases)."""
    f = rng.normal(0, scale, (N, d)).astype(np.float32)
    if N > 8:
        f[::7] = np.round(f[::7])
        f[::11] = np.round(f[::11] * 2) / 2
    return f


REF_SWEEP = "golden_ref_sweep.npz"  # in tests/golden/, written by tests/golden/make_golden_ref_sweep.py


def fingerprint(a):
    """sha256 of an array's dtype, shape and bits: how the larger reference outputs are stored"""
    import hashlib
    a = np.ascontiguousarray(a)
    return "sha256:" + hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()


class Reference:
    """What the reference DenseCRF headers return on the inputs of tests/test_oracle.py: computed live by
    oracle/_ref/libref.so where it was built (oracle/Makefile with the reference tree present), otherwise read from
    tests/golden/golden_ref_sweep.npz."""

    def __init__(self):
        import os
        from oracle.pyoracle import Ref
        self.live = Ref() if Ref.available() else None
        self.stored = {}
        if self.live is None:
            with np.load(os.path.join(os.path.dirname(__file__), "golden", REF_SWEEP)) as g:
                for key in g.files:
                    case, name = key.split("|")
                    self.stored.setdefault(case, {})[name] = g[key]

    def outputs(self, case, compute):
        """{name: array} of one case; compute(Ref) evaluates it live.  A stored array may be a fingerprint."""
        if self.live is not None:
            return compute(self.live)
        assert case in self.stored, "%s: no stored reference vectors (tests/golden/make_golden_ref_sweep.py)" % case
        return self.stored[case]

    def cases(self, prefix):
        """the stored cases whose names start with `prefix`, in order"""
        return sorted(c for c in self.stored if c.startswith(prefix))


def assert_same_as_reference(case, got, want):
    """every array of `got` (the oracle) bit for bit equal to the reference's array of the same name"""
    for name, a in got.items():
        a, w = np.asarray(a), np.asarray(want[name])
        if w.dtype.kind == "U":
            assert fingerprint(a) == str(w), "%s: %s differs from the reference" % (case, name)
        else:
            assert a.dtype == w.dtype and a.shape == w.shape, "%s: %s is %s%s, the reference's %s%s" % (
                case, name, a.dtype, a.shape, w.dtype, w.shape)
            u = np.dtype("u%d" % a.dtype.itemsize)
            bad = int((np.ascontiguousarray(a).reshape(-1).view(u) != np.ascontiguousarray(w).reshape(-1).view(u)).sum())
            assert bad == 0, "%s: %d of %d values of %s differ from the reference in bits" % (case, bad, a.size, name)


def golden_unary_case(name):
    """One case of tests/golden/golden_unary.npz (made by tests/golden/make_golden_unary.py with the real cv2.gemm):
    returns (MapSnapshot, observs, error, depth)."""
    import importlib
    import os
    synth = importlib.import_module("lc-crf-slam_b200.synth")
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_unary.npz"))
    keys = ("xyz", "obs_ptr", "obs_kf", "obs_uv", "kf_pose", "kf_intr", "kf_bounds", "kp2d")
    s = synth.MapSnapshot(*(g[name + "_" + k] for k in keys), np.zeros(g[name + "_xyz"].shape[0], bool))
    return s, g[name + "_observs"], g[name + "_error"], g[name + "_depth"]
