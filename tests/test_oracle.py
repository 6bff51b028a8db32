"""CPU tests: the oracle (oracle/lccrf_oracle.c) is pinned against
  (1) the reference's one golden vector (examples/res1_cpu.ppm -> tests/golden/golden_im1.npz),
  (2) outputs of the UNMODIFIED reference headers stored in tests/golden/golden_ref.npz,
  (3) the reference headers compiled in place (oracle/_ref/libref.so) on seeded sweeps -- live where that library was
      built, otherwise against the sweeps' reference outputs stored in tests/golden/golden_ref_sweep.npz.
"""
import importlib
import os

import numpy as np
import pytest

from util import assert_same_as_reference, bits, golden_unary_case, tie_features

GOLD = os.path.join(os.path.dirname(__file__), "golden")
synth = importlib.import_module("lc-crf-slam_b200.synth")
LATTICE_DIMS = (2, 3, 5)
SLAM_SIZES = (2999, 3000, 3001, 3002, 20000)


def test_golden_image_kat(oracle):
    """example_cpu.cpp:80-98 on im1/anno1: DenseCRFCPU<21>, Gaussian(3,3) + bilateral(10,60,20), 10 iterations."""
    g = np.load(os.path.join(GOLD, "golden_im1.npz"))
    W, H, M = int(g["W"]), int(g["H"]), 21
    en_u = -np.log(np.float64(np.float32(1.0) / np.float32(M)))  # ::log(double) in example_cpu.cpp's TU
    c = np.float32(0.5)
    en_n = -np.log(np.float64((np.float32(1.0) - c) / np.float32(M - 1)))
    en_p = -np.log(np.float64(c))
    unary = oracle.unary_from_label(g["label"], M, np.float32(en_u), np.full(M, en_n, np.float32), np.full(M, en_p, np.float32))
    f2 = oracle.features_image(W, H, 2, 3.0)
    f5 = oracle.features_image(W, H, 5, 60.0, g["im"], 20.0)
    Q, mp, V = oracle.meanfield(unary, [f2, f5], [3.0, 10.0], 10)
    assert np.array_equal(mp, g["map"]), "%d px differ from res1_cpu.ppm" % int((mp != g["map"]).sum())


def test_golden_reference_vectors(oracle):
    g = np.load(os.path.join(GOLD, "golden_ref.npz"))
    for d, N in ((2, 6), (2, 257), (3, 130), (5, 203)):
        k = "lat_d%d_n%d_" % (d, N)
        lat = oracle.lattice(g[k + "feat"])
        assert np.array_equal(lat["offset"], g[k + "offset"])
        assert np.array_equal(bits(lat["bary"]), bits(g[k + "bary"]))
        assert np.array_equal(lat["nbr"], g[k + "nbr"])
        assert np.array_equal(bits(oracle.filter(lat, g[k + "x"])), bits(g[k + "y"]))
        oracle.lattice_free(lat)
    from oracle.pyoracle import slam_params
    prm = slam_params(**synth.SLAM_PARAMS)
    Q, mp, V = oracle.slam_crf(g["slam_observs"], g["slam_error"], g["slam_kp2d"], g["slam_label"], g["slam_energies"], prm)
    assert np.array_equal(bits(Q), bits(g["slam_Q"]))
    assert np.array_equal(mp, g["slam_map"])


def lattice_outputs(impl, f, xs):
    """lattice of f and its filter of every x, by the oracle or the reference (the same API)"""
    lat = impl.lattice(f)
    out = {"V": np.array(lat["V"], np.int32), "offset": lat["offset"], "bary": lat["bary"], "nbr": lat["nbr"]}
    for x in xs:
        out["filter_L%d" % x.shape[1]] = impl.filter(lat, x)
    impl.lattice_free(lat)
    return out


@pytest.mark.parametrize("d", LATTICE_DIMS)
def test_lattice_vs_compiled_reference(oracle, ref, d):
    rng = np.random.default_rng(d)
    for N in (0, 1, 4, 5, 6, 7, 8, 257, 1000, 5003):
        f = tie_features(rng, N, d)
        xs = [rng.random((N, L)).astype(np.float32) for L in (1, 2, 5)]
        case = "lattice_d%d_n%d" % (d, N)
        assert_same_as_reference(case, lattice_outputs(oracle, f, xs), ref.outputs(case, lambda r: lattice_outputs(r, f, xs)))


def test_phantom_lanes(oracle):
    """SURVEY Appendix C: N in {4..8} points far from the origin, d=2 -> M_ = 3,6,6,6,3."""
    got = []
    for N in (4, 5, 6, 7, 8):
        f = np.array([[100 + 0.01 * i, 100] for i in range(N)], dtype=np.float32)
        lat = oracle.lattice(f)
        got.append(lat["V"])
        oracle.lattice_free(lat)
    assert got == [3, 6, 6, 6, 3]


@pytest.mark.parametrize("N", SLAM_SIZES)
def test_slam_crf_vs_compiled_reference(oracle, ref, N):
    from oracle.pyoracle import slam_params
    prm = slam_params(**synth.SLAM_PARAMS)
    fr = synth.slam_frame(N, seed=N)
    lab = oracle.rough_classify(fr.observs, fr.error, fr.depth, prm)
    assert 0 < lab.sum() < N
    case = "slam_n%d" % N
    want = ref.outputs(case, lambda r: dict(zip(("energies", "Q", "map"), (r.label_energies(2, prm.confidence),) +
                                                r.slam_crf(fr.observs, fr.error, fr.kp2d, lab, prm))))
    Qo, mo, _ = oracle.slam_crf(fr.observs, fr.error, fr.kp2d, lab, want["energies"], prm)
    assert_same_as_reference(case, {"Q": Qo, "map": mo}, want)
    assert 0 < mo.sum() < N  # non-trivial labelling


def test_generic_labels_and_relax_vs_compiled_reference(oracle, ref):
    rng = np.random.default_rng(5)
    N = 1500
    for L, dims in ((3, (2, 3)), (4, (5,)), (21, (2,))):
        feats = [tie_features(rng, N, d, 2.0) for d in dims]
        unary = rng.random((N, L)).astype(np.float32) * 3
        w = [3.0 + k for k in range(len(dims))]
        for relax in (1.0, 0.5):
            Qo, mo, _ = oracle.meanfield(unary, feats, w, 4, relax)
            case = "generic_L%d_relax%g" % (L, relax)
            want = ref.outputs(case, lambda r: dict(zip(("Q", "map"), r.crf3d(L, feats, w, 4, unary=unary, relax=relax))))
            assert_same_as_reference(case, {"Q": Qo, "map": mo}, want)


def test_fast_exp_properties(oracle):
    assert oracle.fast_exp(0.0) == 1.0
    assert oracle.fast_exp(-20.5) == 0.0          # densecrf3d.h:58 cut-off
    xs = np.linspace(-20, 0, 2001)
    ys = np.array([oracle.fast_exp(float(x)) for x in xs])
    assert np.all(np.diff(ys) >= -1e-12)
    assert np.max(np.abs(ys - np.exp(xs)) / np.exp(xs)) < 1e-4


def test_unary_restatement_properties(oracle):
    """Defining properties of the unary restatement (its arithmetic is pinned by test_unary_vs_opencv_golden)."""
    snap = synth.map_snapshot(400, 16, seed=9, ragged=True)
    ob, er, de = oracle.map_point_unary(snap)
    cnt = np.diff(snap.obs_ptr)
    assert np.array_equal(ob, cnt.astype(np.float32))
    # float64 re-evaluation
    P = snap.kf_pose.astype(np.float64).reshape(-1, 3, 4)
    pt = np.repeat(np.arange(snap.n), cnt)
    X = snap.xyz.astype(np.float64)[pt]
    Pk = P[snap.obs_kf]
    Xc = np.einsum("nij,nj->ni", Pk[:, :, :3], X) + Pk[:, :, 3]
    K = snap.kf_intr.astype(np.float64)[snap.obs_kf]
    B = snap.kf_bounds.astype(np.float64)[snap.obs_kf]
    u = K[:, 0] * Xc[:, 0] / Xc[:, 2] + K[:, 2]
    v = K[:, 1] * Xc[:, 1] / Xc[:, 2] + K[:, 3]
    ok = (1.0 / Xc[:, 2] >= 0) & (u >= B[:, 0]) & (u <= B[:, 1]) & (v >= B[:, 2]) & (v <= B[:, 3])
    assert 0.01 < 1 - ok.mean() < 0.3, "skip rules not exercised"
    e = np.hypot(u - snap.obs_uv[:, 0], v - snap.obs_uv[:, 1]) * ok
    err = np.bincount(pt, e, snap.n) / cnt
    dep = np.bincount(pt, Xc[:, 2] * ok, snap.n) / cnt
    # points whose projection sits within float rounding of an image bound may legitimately differ
    close = np.isclose(er, err, rtol=2e-4, atol=2e-4) & np.isclose(de, dep, rtol=2e-4, atol=2e-4)
    assert close.mean() > 0.99


# ------------------------------------------------------------------ frontend feeders (SURVEY 8f)
UNARY_CASES = ("ragged", "uniform64", "uniform70", "mixed_cameras")


@pytest.mark.parametrize("name", UNARY_CASES)
def test_unary_vs_opencv_golden(oracle, name):
    """Tracking::ComputeMapPointErrAndObserv restatement against a statement-by-statement evaluation whose matrix
    product is the real cv::gemm (tests/golden/make_golden_unary.py): bit-identical observs / error / depth."""
    s, ob, er, de = golden_unary_case(name)
    o_ob, o_er, o_de = oracle.map_point_unary(s)
    assert np.array_equal(o_ob, ob)
    assert np.array_equal(bits(o_er), bits(er)) and np.array_equal(bits(o_de), bits(de))
    assert (er > 0).any() and np.isfinite(er).all()


def test_unary_vs_opencv_live(oracle):
    """Where the cv2 wheel is importable (the build container) the cv::gemm-based evaluation of Tracking.cc:1803-1839
    runs live on fresh random snapshots, beyond the committed fixture."""
    pytest.importorskip("cv2")
    import sys
    sys.path.insert(0, GOLD)
    try:
        gen = importlib.import_module("make_golden_unary")
    finally:
        sys.path.remove(GOLD)
    for seed in range(6):
        s = synth.map_snapshot(40 + 13 * seed, 3 + 4 * seed, seed=500 + seed, n_kf=12 + 5 * seed, ragged=seed % 2 == 0)
        if seed >= 3:  # different cameras per keyframe
            s.kf_intr = s.kf_intr.copy()
            s.kf_intr[::2, :2] *= np.float32(1.0 + 0.01 * seed)
            s.kf_bounds = s.kf_bounds.copy()
            s.kf_bounds[1::3, 1] -= np.float32(11 * seed)
        ob, er, de = gen.unary_cv2(s)
        o_ob, o_er, o_de = oracle.map_point_unary(s)
        assert np.array_equal(o_ob, ob), seed
        assert np.array_equal(bits(o_er), bits(er)) and np.array_equal(bits(o_de), bits(de)), seed


def test_bf_match_vs_opencv_golden(oracle):
    """Tracking::BfMatch restatement against cv::BFMatcher.knnMatch(k=2) outputs captured from OpenCV itself
    (tests/golden/make_golden_frontend.py): nearest-two lists incl. tie order, and the 0.6 ratio test."""
    g = np.load(os.path.join(GOLD, "golden_frontend.npz"))
    for name in ("orb", "ties", "one_train_row", "two_train_rows", "ragged"):
        match, knn, n = oracle.bf_match(g[name + "_dq"], g[name + "_dt"], 0.6)
        assert np.array_equal(knn, g[name + "_knn"]), name
        assert np.array_equal(match, g[name + "_match"]), name
        assert n == int((g[name + "_match"] >= 0).sum())
    # empty train / query sets: no correspondences, no crash
    m, k, n = oracle.bf_match(g["orb_dq"][:5], np.zeros((0, 32), np.uint8))
    assert (m == -1).all() and n == 0
    m, k, n = oracle.bf_match(np.zeros((0, 32), np.uint8), g["orb_dt"])
    assert m.size == 0 and n == 0


def test_epipolar_prior_restatement(oracle):
    """symmetricEpipolarDistance + likelihood (fundamental_estimator.h:90-127, Tracking.cc:2043) against an independent
    numpy float64 evaluation of the same expressions (numpy rounds every operation, like the -O3 no-FMA build)."""
    synth = importlib.import_module("lc-crf-slam_b200.synth")
    x1, x2, F, out = synth.epipolar_matches(500, 3)
    dis, prob = oracle.epipolar_prior(x1, x2, F, 0.5, 1.1)
    a, b = x1.astype(np.float64), x2.astype(np.float64)
    f = F.reshape(3, 3)
    l1 = f[0, 0] * b[:, 0] + f[1, 0] * b[:, 1] + f[2, 0]
    l2 = f[0, 1] * b[:, 0] + f[1, 1] * b[:, 1] + f[2, 1]
    l3 = f[0, 2] * b[:, 0] + f[1, 2] * b[:, 1] + f[2, 2]
    t1 = f[0, 0] * a[:, 0] + f[0, 1] * a[:, 1] + f[0, 2]
    t2 = f[1, 0] * a[:, 0] + f[1, 1] * a[:, 1] + f[1, 2]
    t3 = f[2, 0] * a[:, 0] + f[2, 1] * a[:, 1] + f[2, 2]
    d1 = (l1 * a[:, 0] + l2 * a[:, 1] + l3) / np.sqrt(l1 * l1 + l2 * l2)
    d2 = (t1 * b[:, 0] + t2 * a[:, 1] + t3) / np.sqrt(t1 * t1 + t2 * t2)  # y1, as fundamental_estimator.h:121 has it
    want = np.abs(0.5 * (d1 + d2))
    assert np.array_equal(dis.view(np.int64), want.view(np.int64))
    den = np.float64(np.float32(2) * np.float32(1.1) * np.float32(1.1))
    wp = np.exp(-(want - np.float64(np.float32(0.5))) * (want - np.float64(np.float32(0.5))) / den)
    assert np.allclose(prob, wp, rtol=4e-16, atol=0)
    assert np.median(dis[~out]) < np.median(dis[out])  # displaced matches sit further from their epipolar lines


def test_label_partition_restatement(oracle):
    """Tracking.cc:1945-1955: the loop acts on exactly the label-0 points, in point order."""
    rng = np.random.default_rng(9)
    lab = (rng.random(1000) < 0.7).astype(np.int16)
    fid = rng.permutation(5000)[:1000].astype(np.int32)
    d, s = oracle.label_partition(lab)
    assert np.array_equal(d, np.nonzero(lab == 0)[0]) and np.array_equal(s, np.nonzero(lab != 0)[0])
    d, s = oracle.label_partition(lab, fid)
    assert np.array_equal(d, fid[lab == 0]) and np.array_equal(s, fid[lab != 0])
    d, s = oracle.label_partition(np.zeros(0, np.int16))
    assert d.size == 0 and s.size == 0


def random_crf_case(oracle, ref, p):
    """one case of the randomised sweep, p = [N, L, iters, relax, seed, conf (0: a random unary instead of labels), dims...]"""
    N, L, iters, rs = int(p[0]), int(p[1]), int(p[2]), int(p[4])
    relax, conf, dims = float(p[3]), float(p[5]), [int(d) for d in p[6:]]
    rng = np.random.default_rng(rs)
    feats = [tie_features(rng, N, d, float(rng.uniform(0.5, 8.0))) for d in dims]
    w = rng.uniform(0.5, 30.0, len(dims)).astype(np.float32)
    case = "random_%d_%d_%d_%s_%d_%s_%s" % (N, L, iters, relax, rs, conf, "-".join(map(str, dims)))
    if conf:
        lab = rng.integers(-1, L, N).astype(np.int16)
        want = ref.outputs(case, lambda r: dict(zip(("params", "energies", "Q", "map"), (p, r.label_energies(L, conf)) +
                                                    r.crf3d(L, feats, w, iters, label=lab, conf=conf, relax=relax))))
        en = want["energies"]
        unary = oracle.unary_from_label(lab, L, en[0], np.full(L, en[1], np.float32), np.full(L, en[2], np.float32))
    else:
        unary = (rng.random((N, L)) * 4).astype(np.float32)
        want = ref.outputs(case, lambda r: dict(zip(("params", "Q", "map"), (p,) + r.crf3d(L, feats, w, iters, unary=unary, relax=relax))))
    Qo, mo, _ = oracle.meanfield(unary, feats, w, iters, relax)
    assert_same_as_reference(case, {"Q": Qo, "map": mo}, want)


def test_random_crf_shapes_vs_compiled_reference(oracle, ref):
    """Randomised sweep (hypothesis, fixed seed): point counts incl. 0 and every N % 4 residue, labels, kernels,
    feature dimensions and scales, weights, iterations, relax, unary-from-label with unknown (-1) labels -- oracle
    marginals and MAP bit-identical to the unmodified reference headers compiled in place.  Without them, the cases
    this sweep drew when the reference outputs were stored are run against those outputs."""
    if ref.live is None:
        cases = ref.cases("random_")
        assert cases
        for case in cases:
            random_crf_case(oracle, ref, ref.outputs(case, None)["params"])
        return
    from hypothesis import given, settings, strategies as st, HealthCheck, seed

    @seed(20241)
    @settings(max_examples=40, deadline=None, suppress_health_check=list(HealthCheck), database=None)
    @given(st.data())
    def run(data):
        N = data.draw(st.one_of(st.integers(0, 9), st.integers(10, 700)), label="N")
        L = data.draw(st.sampled_from([2, 3, 4]), label="L")
        dims = data.draw(st.lists(st.sampled_from([2, 3, 5]), min_size=1, max_size=3), label="dims")
        iters = data.draw(st.integers(1, 4), label="iters")
        relax = data.draw(st.sampled_from([1.0, 0.5, 0.3]), label="relax")
        rs = data.draw(st.integers(0, 2 ** 31 - 1), label="seed")
        conf = float(data.draw(st.sampled_from([0.55, 0.7, 0.9]), label="conf")) if data.draw(st.booleans(), label="from_label") else 0.0
        random_crf_case(oracle, ref, np.array([N, L, iters, relax, rs, conf] + dims, np.float64))

    run()


def window_outputs(impl, f, x, L, io, oo, isz, osz):
    """the reference's windowed filter (PermutohedralLatticeCPU::compute) of x on the lattice of f"""
    lat = impl.lattice(f)
    y = impl.filter_window(lat, x, L, io, oo, isz, osz)
    impl.lattice_free(lat)
    return {"y": y}


def test_compute_window_is_zero_padding_plus_crop(oracle, ref):
    """PermutohedralLatticeCPU::compute's windowing arguments (permutohedral_cpu.h:634-637) on the compiled reference
    equal the full filter of a zero-padded input, cropped -- bit for bit, signed inputs included (a vertex sum starts
    at +0 and is unchanged by +-0 addends).  This is what lccrf_lattice_filter_window relies on."""
    rng = np.random.default_rng(12)
    N, d = 1501, 2
    f = rng.normal(0, 2.0, (N, d)).astype(np.float32)
    lo = oracle.lattice(f)
    for L, (io, oo, isz, osz) in ((1, (0, 0, -1, -1)), (2, (100, 0, 700, -1)), (3, (0, 37, -1, 900)), (21, (500, 1400, 1001, 101)),
                                  (2, (1500, 0, 1, 1)), (4, (0, 0, 0, -1))):
        n_in = N - io if isz == -1 else isz
        x = rng.normal(0, 1, (n_in, L)).astype(np.float32)
        full = np.zeros((N, L), np.float32)
        full[io:io + n_in] = x
        n_out = N - oo if osz == -1 else osz
        case = "window_L%d_%d_%d_%d_%d" % (L, io, oo, isz, osz)
        want = ref.outputs(case, lambda r: window_outputs(r, f, x, L, io, oo, isz, osz))
        assert_same_as_reference(case, {"y": oracle.filter(lo, full)[oo:oo + n_out]}, want)
    oracle.lattice_free(lo)
