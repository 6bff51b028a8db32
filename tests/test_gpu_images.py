"""GPU tests of the batched image CRF (lccrf_images, Images): every image of a batch is bit-identical to the per-object
DenseCRF path on the same inputs (which is bit-identical to the reference), whatever else shares the batch."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

from test_images_abi import build_images_batch
from util import REL_TOL, assert_bit_exact, assert_marginals

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
synth = importlib.import_module("lc-crf-slam_b200.synth")

C2_KERNELS = [(2, 3.0, 3.0, 0.0), (5, 10.0, 60.0, 20.0)]  # Gaussian (sigma 3) + bilateral (sigma 60 / 20), w = 3 / 10


def problems(sizes, seed=0, L=2):
    """(img [N,3] u8, label [N]) per image"""
    return [synth.image_problem(W, H, seed + i, n_labels=L) for i, (W, H) in enumerate(sizes)]


def per_object(pkg, ctx, W, H, L, kernels, img, lab=None, en=None, unary=None, T=10, relax=1.0):
    """the same image through lccrf_crf: (map, prob, [V per kernel])"""
    crf = pkg.DenseCRF(ctx, W * H, L)
    if unary is not None:
        crf.setUnaryEnergy(unary)
    else:
        crf.setUnaryEnergyFromLabel(lab, energies=en)
    for F, w, posdev, fd in kernels:
        if F == 2:
            crf.addPairwiseFromImage(W, H, w, posdev)
        else:
            crf.addPairwiseFromImage(W, H, w, posdev, img, fd)
    crf.inference(T, True, relax)
    out = crf.getMap(), crf.getProbability(), [crf.potts_vertices(k) for k in range(len(kernels))]
    crf.close()
    return out


def run_batch(pkg, ctx, sizes, L, kernels, probs, en, T=10, relax=1.0, C=3):
    im = pkg.Images(ctx, sizes, L, kernels, C=C)
    im.set_inputs([p[0] for p in probs] if C else None, label=[p[1] for p in probs], energies=en)
    im.run(T, relax)
    mp, pr, split = im.get_outputs()
    V = im.vertices()
    im.close()
    return mp, pr, split, V


def assert_same(a, b, what):
    assert np.array_equal(a[0], b[0]), "%s: MAP differs" % what
    assert_bit_exact(a[1], b[1], what=what)


def oracle_image(oracle, W, H, L, kernels, img, lab, en, T=10, relax=1.0):
    unary = oracle.unary_from_label(lab, L, en[0], np.full(L, en[1], np.float32), np.full(L, en[2], np.float32))
    feats = [oracle.features_image(W, H, F, posdev, img if F > 2 else None, fd) for F, _, posdev, fd in kernels]
    return oracle.meanfield(unary, feats, [w for _, w, _, _ in kernels], T, relax)


# ------------------------------------------------------------------ 1. golden image inside a batch
def test_golden_image_inside_a_batch(pkg, ctx, oracle):
    g = np.load(os.path.join(GOLD, "golden_im1.npz"))
    M = 21
    c = np.float32(0.5)  # GT_PROB of example_cpu.cpp
    en = np.array([-np.log(np.float64(np.float32(1.0) / np.float32(M))), -np.log(np.float64((np.float32(1.0) - c) / np.float32(M - 1))),
                   -np.log(np.float64(c))]).astype(np.float32)
    sizes = [(97, 61), (int(g["W"]), int(g["H"])), (200, 150)]  # 97 * 61 % 4 == 1: phantom lanes
    probs = problems(sizes, seed=31, L=M)
    probs[1] = (g["im"], g["label"])
    mp, pr, split, V = run_batch(pkg, ctx, sizes, M, C2_KERNELS, probs, en)
    assert np.array_equal(split[1][0], g["map"]), "%d px differ from res1_cpu.ppm" % int((split[1][0] != g["map"]).sum())
    for b, ((W, H), (img, lab)) in enumerate(zip(sizes, probs)):
        Qo, mo, Vo = oracle_image(oracle, W, H, M, C2_KERNELS, img, lab, en)
        assert_bit_exact(split[b][1], Qo, what="image %d marginals" % b)
        assert np.array_equal(split[b][0], mo)
        assert tuple(V[b]) == tuple(Vo), (b, V[b], Vo)


# ------------------------------------------------------------------ 2. C2 recipe, ragged batch, L = 2
def test_c2_ragged_batch(pkg, ctx, oracle):
    sizes = [(640, 480), (161, 121), (33, 17), (1, 1), (0, 0)]
    probs = problems(sizes, seed=40)
    en = pkg.label_energies(2, 0.7)
    mp, pr, split, V = run_batch(pkg, ctx, sizes, 2, C2_KERNELS, probs, en)
    assert mp.size == sum(W * H for W, H in sizes)
    for b, ((W, H), (img, lab)) in enumerate(zip(sizes, probs)):
        if W * H == 0:
            assert split[b][0].size == 0 and tuple(V[b]) == (0, 0)
            continue
        m, Q, Vp = per_object(pkg, ctx, W, H, 2, C2_KERNELS, img, lab, en)
        assert_same(split[b], (m, Q), "image %d (%dx%d) vs per-object" % (b, W, H))
        assert tuple(V[b]) == tuple(Vp)
        if W * H < 640 * 480:
            Qo, mo, _ = oracle_image(oracle, W, H, 2, C2_KERNELS, img, lab, en)
            assert_bit_exact(split[b][1], Qo, what="image %d vs oracle" % b)
            assert np.array_equal(split[b][0], mo)


def test_sixteen_full_size_images(pkg, ctx):
    """16 x 640x480: the lattices' CSR count tables would exceed 2^31 entries at the default sort chunk, so the batch
    sorts in coarser chunks; every image still equals the per-object path (checked on the first and the last)."""
    sizes = [(640, 480)] * 16
    probs = problems(sizes, seed=45)
    en = pkg.label_energies(2, 0.7)
    mp, pr, split, V = run_batch(pkg, ctx, sizes, 2, C2_KERNELS, probs, en)
    for b in (0, 15):
        m, Q, Vp = per_object(pkg, ctx, 640, 480, 2, C2_KERNELS, probs[b][0], probs[b][1], en)
        assert_same(split[b], (m, Q), "image %d of 16" % b)
        assert tuple(V[b]) == tuple(Vp)


# ------------------------------------------------------------------ 3. input modes
def test_input_modes(pkg, ctx, oracle):
    sizes = [(120, 90), (75, 41)]
    probs = problems(sizes, seed=50)
    en = pkg.label_energies(2, 0.6)
    imgs, labs = [p[0] for p in probs], [p[1] for p in probs]
    ref = run_batch(pkg, ctx, sizes, 2, C2_KERNELS, probs, en)
    # energies mode: the unary table setUnaryEnergyFromLabel would build
    unary = [oracle.unary_from_label(l, 2, en[0], np.full(2, en[1], np.float32), np.full(2, en[2], np.float32)) for l in labs]
    im = pkg.Images(ctx, sizes, 2, C2_KERNELS)
    im.set_inputs(imgs, unary=unary)
    im.run(10)
    assert_same(im.get_outputs()[:2], ref[:2], "energies mode vs label mode")
    # f32 image holding the same integer values
    im.set_inputs([i.astype(np.float32) for i in imgs], label=labs, energies=en)
    im.run(10)
    assert_same(im.get_outputs()[:2], ref[:2], "f32 image vs u8 image")
    # relax = 0.5
    im.set_inputs(imgs, label=labs, energies=en)
    im.run(10, 0.5)
    split = im.get_outputs()[2]
    for b, (W, H) in enumerate(sizes):
        assert_same(split[b], per_object(pkg, ctx, W, H, 2, C2_KERNELS, imgs[b], labs[b], en, relax=0.5)[:2], "relax 0.5 image %d" % b)
    im.close()
    # K = 1 (Gaussian only, no image) and K = 0 (unary only)
    for kernels in ([C2_KERNELS[0]], []):
        mp, pr, split, V = run_batch(pkg, ctx, sizes, 2, kernels, probs, en, C=0)
        for b, (W, H) in enumerate(sizes):
            m, Q, Vp = per_object(pkg, ctx, W, H, 2, kernels, None, labs[b], en)
            assert_same(split[b], (m, Q), "K=%d image %d" % (len(kernels), b))
            assert tuple(V[b]) == tuple(Vp)


# ------------------------------------------------------------------ 4. no cross-talk
def test_permuted_batch_and_single_image(pkg, ctx):
    sizes = [(150, 100), (64, 64), (99, 37), (180, 140)]
    probs = problems(sizes, seed=60)
    en = pkg.label_energies(2, 0.7)
    ref = run_batch(pkg, ctx, sizes, 2, C2_KERNELS, probs, en)
    perm = [2, 0, 3, 1]
    got = run_batch(pkg, ctx, [sizes[i] for i in perm], 2, C2_KERNELS, [probs[i] for i in perm], en)
    for j, i in enumerate(perm):
        assert_same(got[2][j], ref[2][i], "permuted batch, image %d" % i)
        assert tuple(got[3][j]) == tuple(ref[3][i])
    alone = run_batch(pkg, ctx, sizes[1:2], 2, C2_KERNELS, probs[1:2], en)
    assert_same(alone[2][0], ref[2][1], "B = 1 vs inside the batch")


# ------------------------------------------------------------------ 5. repeated runs (plain, capture, replays)
@pytest.mark.parametrize("graphs", [1, 0])
def test_repeated_runs_equal_fresh_objects(pkg, ctx, graphs):
    sizes = [(160, 120), (90, 70), (40, 30)]
    en = pkg.label_energies(2, 0.7)
    ctx.set_option("graphs", graphs)
    try:
        im = pkg.Images(ctx, sizes, 2, C2_KERNELS)
        for r, T in enumerate((10, 10, 10, 10, 5, 5, 5)):  # plain, capture, replay, replay; T changes: plain, capture, replay
            probs = problems(sizes, seed=100 + 10 * r)
            im.set_inputs([p[0] for p in probs], label=[p[1] for p in probs], energies=en)
            im.run(T)
            got = im.get_outputs()
            ref = run_batch(pkg, ctx, sizes, 2, C2_KERNELS, probs, en, T=T)
            assert_same(got[:2], ref[:2], "run %d (T = %d, graphs = %d)" % (r, T, graphs))
        im.close()
    finally:
        ctx.set_option("graphs", 1)


# ------------------------------------------------------------------ 6. one launch sequence per batch
def launches_of_one_run(pkg, ctx, sizes, en):
    probs = problems(sizes, seed=70)
    im = pkg.Images(ctx, sizes, 2, C2_KERNELS)
    im.set_inputs([p[0] for p in probs], label=[p[1] for p in probs], energies=en)
    l0 = ctx.kernel_launches
    im.run(10)
    n = ctx.kernel_launches - l0
    im.get_outputs()
    im.close()
    return n


def test_launches_do_not_grow_with_the_batch(pkg, ctx):
    en = pkg.label_energies(2, 0.7)
    # every launch count of a run depends on the image size only through the blur choice (fused for <= 32768 pixels:
    # one launch per filter call, else one per lattice dimension); images of one size take the same choice
    for W, H, B in ((64, 48, 8), (640, 480, 4)):
        one = launches_of_one_run(pkg, ctx, [(W, H)], en)
        many = launches_of_one_run(pkg, ctx, [(W, H)] * B, en)
        assert one == many, (W, H, B, one, many)


@pytest.mark.parametrize("W,H,fused", [(640, 480, False), (181, 181, True), (160, 120, True)])
def test_blur_choice_follows_the_image_size(pkg, ctx, W, H, fused):
    en = pkg.label_energies(2, 0.7)
    probs = problems([(W, H)] * 3, seed=80)
    im = pkg.Images(ctx, [(W, H)] * 3, 2, C2_KERNELS)
    im.set_inputs([p[0] for p in probs], label=[p[1] for p in probs], energies=en)
    ctx.set_option("profile", 1)
    try:
        ctx.profile_report()
        im.run(3)
        rep = ctx.profile_report()
    finally:
        ctx.set_option("profile", 0)
    im.close()
    assert ("k_blur_fused" in rep) == fused and ("k_blur" in rep) == (not fused), (W * H, sorted(rep))


# ------------------------------------------------------------------ 7. tolerance mode (tree splat)
def test_tree_splat_within_tolerance(pkg, ctx, oracle):
    sizes = [(160, 120)] * 3
    probs = problems(sizes, seed=90)
    en = pkg.label_energies(2, 0.7)
    ctx.set_option("ordered_splat", 0)
    try:
        mp, pr, split, V = run_batch(pkg, ctx, sizes, 2, C2_KERNELS, probs, en)
    finally:
        ctx.set_option("ordered_splat", 1)
    for b, (img, lab) in enumerate(probs):
        Qo, mo, _ = oracle_image(oracle, 160, 120, 2, C2_KERNELS, img, lab, en)
        assert_marginals(split[b][1], Qo, tol=REL_TOL, what="tree splat image %d" % b)
        assert np.array_equal(split[b][0], mo)


# ------------------------------------------------------------------ 8. errors
def create_rc(pkg, ctx, sizes, nch, L, kernels, K=None):
    wh = np.asarray(sizes, dtype=np.int32).reshape(-1, 2)
    W, H = np.ascontiguousarray(wh[:, 0]), np.ascontiguousarray(wh[:, 1])
    ks = (pkg.ImageKernel * max(len(kernels), 1))(*[pkg.ImageKernel(*k) for k in kernels])
    h = C.c_void_p()
    rc = ctx.lib.lccrf_images_create(ctx.h, wh.shape[0] if K != "B-1" else -1, W.ctypes.data, H.ctypes.data, nch, L,
                                     len(kernels) if K in (None, "B-1") else K, ks, C.byref(h))
    if rc == 0:
        ctx.lib.lccrf_images_destroy(h)
    return rc


def test_create_validation(pkg, ctx):
    ok = [(2, 3.0, 3.0, 0.0), (5, 10.0, 60.0, 20.0)]
    assert create_rc(pkg, ctx, [(8, 8)], 3, 2, ok) == 0
    assert create_rc(pkg, ctx, [], 3, 2, ok) == 0                                   # B = 0
    assert create_rc(pkg, ctx, [(8, 8)], 3, 2, ok, K="B-1") == -1                   # B < 0
    assert create_rc(pkg, ctx, [(-1, 8)], 3, 2, ok) == -1                           # W < 0
    assert create_rc(pkg, ctx, [(8, -1)], 3, 2, ok) == -1                           # H < 0
    assert create_rc(pkg, ctx, [(2048, 2048)], 3, 2, ok) == 0                       # 2^22 pixels
    assert create_rc(pkg, ctx, [(2048, 2049)], 3, 2, ok) == -1                      # more
    assert create_rc(pkg, ctx, [(8, 8)], 3, 0, ok) == -1                            # L = 0
    assert create_rc(pkg, ctx, [(8, 8)], 3, 65, ok) == -1                           # L > LCCRF_MAX_L
    assert create_rc(pkg, ctx, [(8, 8)], 3, 2, ok, K=-1) == -1                      # K < 0
    assert create_rc(pkg, ctx, [(8, 8)], 3, 2, ok * 5) == -1                        # K > LCCRF_MAX_K
    assert create_rc(pkg, ctx, [(8, 8)], 3, 2, [(4, 1.0, 1.0, 1.0)]) == -1          # F neither 2 nor C + 2
    assert create_rc(pkg, ctx, [(8, 8)], 6, 2, [(8, 1.0, 1.0, 1.0)]) == -1          # F > LCCRF_MAX_D
    assert create_rc(pkg, ctx, [(8, 8)], 0, 2, [(2, 1.0, 1.0, 1.0)]) == 0           # Gaussian only, no channels


def test_runtime_errors_leave_the_object_usable(pkg, ctx):
    sizes = [(70, 50), (33, 21)]
    probs = problems(sizes, seed=110)
    en = pkg.label_energies(2, 0.7)
    imgs, labs = [p[0] for p in probs], [p[1] for p in probs]
    ref = run_batch(pkg, ctx, sizes, 2, C2_KERNELS, probs, en)
    im = pkg.Images(ctx, sizes, 2, C2_KERNELS)
    with pytest.raises(pkg.LccrfError, match="error -3"):
        im.get_outputs()                                                     # before any run
    with pytest.raises(pkg.LccrfError, match="error -1"):
        im.set_inputs(None, label=labs, energies=en)                         # bilateral kernel without an image
    for bad in (2, -2):
        lab = [l.copy() for l in labs]
        lab[1][17] = bad
        im.set_inputs(imgs, label=lab, energies=en)
        im.run(10)
        with pytest.raises(pkg.LccrfError, match="error -1.*label"):
            im.get_outputs()
        im.set_inputs(imgs, label=labs, energies=en)
        im.run(10)
        assert_same(im.get_outputs()[:2], ref[:2], "after label %d" % bad)
    im.close()


# ------------------------------------------------------------------ 9. the C example
def test_images_batch_example_runs(pkg, tmp_path):
    exe = build_images_batch(tmp_path)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "image 2: lattices of" in r.stdout
