"""GPU tests (-m gpu): crafted observations through every instantiation of the map-point unary (k_map_point_unary),
compared bit for bit with the oracle (oracle.map_point_unary) on the equivalent flat snapshot.

Every crafted observation is made visible in the output.  A point has n observations, n a power of two; exactly one of
them is live, in a keyframe with R = I, t = 0 and the camera fx = fy = 1, cx = cy = 0 with wide image bounds, so that
(xc, yc, zc) are the point's own coordinates and u = xc / zc.  The other n - 1 observations use keyframes whose third
pose row is (0, 0, 0, -1): their zc is -1, they are skipped and add +0.  So error = er / n and depth = zc / n exactly.
Point coordinates stay finite (0 * x in a skipped keyframe's row would otherwise be NaN); non-finite zc (+-Inf, NaN)
comes from live keyframes whose third row is (0, 0, 0, t) with t non-finite.

Classes: zc at exponent fields 0, 1, 2, 126, 127, 252, 253, 254, at +-0, +-Inf, NaN and negative; u / v on each image
bound and one float ulp either side; a zero residual; residuals just inside and outside the (2^-60, 2^60) range of the
fast square root; residuals whose sqrt sits within +-2^14 double ulps of a float rounding midpoint (3-4-5 triangles, so
the midpoint itself is exact); 0 * Inf NaNs; and whole warps in which every observation is recomputed.  They sit in the
round layout (n = 16, n = 64), the chunk layout (n = 4 and ragged n in {1, 2, 4, 8}: full and tail steps), at lanes 0
and 31 of their warps and in a final partial warp.

The Frames routes feed the unary into the lattice build, so there only classes whose per-point error and depth stay
finite and whose error stays well inside the lattice's key range are used; their unary outputs are read through
get_debug().  ROUTES maps every route to the kernel instantiation it reaches (unary.cu: unary_map_points_packed /
_visible / _visible_multi); together they reach all 36."""
import importlib

import numpy as np
import pytest

from util import bits

pytestmark = pytest.mark.gpu
synth = importlib.import_module("lc-crf-slam_b200.synth")

F32 = np.float32
INF = F32(np.inf)
BX, BY = F32(2.0 ** 20), F32(786432.0)  # image bounds of the live keyframes: (-BX, BX, -BY, BY)
N_LIVE = 16   # live keyframe copies (distinct keyframes for the all-live points)
N_SKIP = 64   # skipped keyframe copies
LIVE, ZINF, ZNINF, ZNAN, SKIP = 0, N_LIVE, N_LIVE + 1, N_LIVE + 2, N_LIVE + 3
BLOCK_MIN = SKIP + N_SKIP   # keyframes of one block
SAFE_ERROR = 1000.0         # largest per-point error on the Frames routes (lattice keys are 16-bit)

# route -> (KFMODE, observation index type, VIS, MULTI) per keyframe set; UCAM follows the camera variant
ROUTES = {
    "ctx.map_point_unary":       {"small": (1, "int", 0, 0), "large": (0, "int", 0, 0)},
    "set_map_inputs int32":      {"small": (1, "int", 0, 0), "large": (0, "int", 0, 0), "large+kf_ptr": (2, "int", 0, 0)},
    "submit_map uint16":         {"small": (1, "ushort", 0, 0), "large": (0, "ushort", 0, 0), "large+kf_ptr": (2, "ushort", 0, 0)},
    "set_map_inputs_indexed int32": {"small": (1, "int2", 0, 0), "large": (0, "int2", 0, 0), "large+kf_ptr": (2, "int2", 0, 0)},
    "set_map_inputs_indexed uint16": {"small": (1, "ushort2", 0, 0), "large": (0, "ushort2", 0, 0), "large+kf_ptr": (2, "ushort2", 0, 0)},
    "set_visible pitched":       {"small": (1, "int", 1, 0), "large": (0, "int", 1, 0), "large+kf_ptr": (2, "int", 1, 0)},
    "set_visible moved":         {"small": (1, "int", 1, 0), "large": (0, "int", 1, 0), "large+kf_ptr": (2, "int", 1, 0)},
    "set_visible_maps":          {"small": (1, "int", 1, 1), "large": (0, "int", 1, 1), "large+kf_ptr": (2, "int", 1, 1)},
}


def fbits(b):
    return np.array([b], np.uint32).view(F32)[0]


def crafted_classes(rng):
    """[(x, y, z, live keyframe, keypoint u, keypoint v)] of the live observation of a point"""
    C = []

    def add(x, y, z, kind=LIVE, uv=(0.5, 0.25)):
        C.append((F32(x), F32(y), F32(z), kind, F32(uv[0]), F32(uv[1])))

    # zc at the reciprocal's edges (x, y scaled with z so that u, v stay normal where 1/z does)
    for field in (0, 1, 2, 126, 127, 252, 253, 254):
        for sign in (0, 1):
            z = fbits((sign << 31) | (field << 23) | int(rng.integers(1, 1 << 23)))
            add(z * F32(0.75), z * F32(-0.375), z)
    for zb in (0x00000001, 0x007fffff, 0x00800000, 0x7f7fffff, 0x3f800000, 0x7e800000, 0x7e7fffff):
        z = fbits(zb)
        add(z * F32(0.5), z * F32(0.25), z)
    add(1.0, 1.0, 0.0)                       # z = +0: u = +Inf, out of bounds
    add(1.0, 0.0, 0.0)                       # u = +Inf, v = 0 * Inf = NaN: out of bounds through u
    add(0.0, 0.0, 0.0)                       # 0 * Inf: u = v = NaN, kept, er NaN
    add(0.0, 0.0, -0.0)                      # z = -0: 1/z = -Inf, skipped
    add(1.0, 1.0, -2.0)                      # behind the camera
    add(0.5, 0.25, 1.0, ZINF)                # zc = +Inf: 1/z = +0, u = v = 0, kept, depth Inf
    add(0.5, 0.25, 1.0, ZNINF)               # zc = -Inf: 1/z = -0 is not < 0, kept, depth -Inf
    add(0.5, 0.25, 1.0, ZNAN)                # zc = NaN: kept, er and depth NaN
    # u / v on each image bound and one float ulp either side (z = 1: u = x, v = y)
    for b, axis in ((-BX, 0), (BX, 0), (-BY, 1), (BY, 1)):
        for to in (-INF, None, INF):
            w = b if to is None else np.nextafter(b, to)
            xy = (w, F32(3.0)) if axis == 0 else (F32(-3.0), w)
            add(xy[0], xy[1], 1.0, uv=(xy[0] - F32(0.5), xy[1] + F32(0.75)))
    # residuals (x = y = 0, z = 1, keypoint (-a, -b): du = a, dv = b, s = a^2 + b^2)
    for a, b in ((0.0, 0.0), (2.0 ** -30, 0.0), (float.fromhex("0x1.000002p-30"), 0.0), (float.fromhex("0x1.fffffep-31"), 0.0),
                 (2.0 ** -30, 2.0 ** -56), (2.0 ** -31, 2.0 ** -31), (2.0 ** 30, 0.0), (float.fromhex("0x1.fffffep29"), 0.0),
                 (float.fromhex("0x1.000002p30"), 0.0), (2.0 ** 29, 2.0 ** 29), (2.0 ** -149, 0.0)):
        add(0.0, 0.0, 1.0, uv=(-a, -b))
    add(0.0, 0.0, 1.0, uv=(0.0, 0.0))
    add(1.5, -2.25, 1.0, uv=(1.5, -2.25))    # zero residual away from the origin
    # sqrt(s) near a float midpoint: a = 3k, b = 4k (k odd, 5k in [2^24, 2^25): 5k is a midpoint), scaled by 2^-20;
    # v = y moves sqrt(s) by about 0.8 y, i.e. 0.8 y / 2^-48 double ulps
    for o in (0, 1, -1, 7, -7, 100, -100, 4096, -4096, 8191, -8191, 8192, -8192, 10240, -10240, 16383, -16383, 20000, -20000):
        k = 2 * int(rng.integers(3355444 // 2, 5592405 // 2)) + 1
        y = F32(o * 2.0 ** -48)
        add(0.0, y, 1.0, uv=(-3 * k * 2.0 ** -20, -4 * k * 2.0 ** -20))
    # ordinary observations
    for _ in range(8):
        add(rng.uniform(-2, 2), rng.uniform(-2, 2), rng.uniform(0.5, 5), uv=(rng.uniform(-1, 1), rng.uniform(-1, 1)))
    return C


def keyframe_block(size, mixed):
    """[LIVE x N_LIVE, ZINF, ZNINF, ZNAN, SKIP x (size - SKIP)]: poses, intrinsics, bounds.  mixed: the skipped keyframes
    have another camera (the UCAM = false path reads every keyframe's own)"""
    pose = np.zeros((size, 12), F32)
    pose[:, 0] = pose[:, 5] = 1.0
    pose[:LIVE + N_LIVE, 10] = 1.0
    pose[ZINF, 11], pose[ZNINF, 11], pose[ZNAN, 11] = INF, -INF, np.nan
    pose[SKIP:, 11] = -1.0
    intr = np.tile(np.array([1, 1, 0, 0], F32), (size, 1))
    bnd = np.tile(np.array([-BX, BX, -BY, BY], F32), (size, 1))
    if mixed:
        intr[SKIP:] = (535.4, 539.2, 320.1, 247.6)
        bnd[SKIP:] = (0, 640, 0, 480)
    return pose, intr, bnd


class Problem:
    """points with their observation lists (block-local keyframe ids) and keypoints; kf offset added on assembly"""

    def __init__(self):
        self.xyz, self.lists = [], []

    def point(self, xyz, obs):
        self.xyz.append(xyz)
        self.lists.append(obs)


def live_point(P, rng, c, n, pos):
    x, y, z, kind, ku, kv = c
    skips = SKIP + rng.permutation(N_SKIP)[:n - 1]
    obs = [(int(k), (F32(rng.uniform(0, 9)), F32(rng.uniform(0, 9)))) for k in skips]
    obs.insert(pos, (kind, (ku, kv)))
    P.point((x, y, z), obs)


def make_problem(rng, classes, all_live_z, partial):
    """groups aligned to 32-point warps: n = 16 (rounds), n = 64 (rounds), all-live warps (every observation recomputed:
    n = 16 rounds and n = 4 chunk), n = 4 (chunk), ragged n in {1, 2, 4, 8} (chunk, tail steps); lane 0 of warp w takes
    class w, lane 31 class w + 1; partial: a final warp of 17 points"""
    P = Problem()
    C = len(classes)
    for n, warps in ((16, C + 1), (64, C + 1), (4, C + 1), (None, C + 1)):
        for w in range(warps):
            for lane in range(32):
                c = classes[w % C] if lane == 0 else classes[(w + 1) % C] if lane == 31 else classes[int(rng.integers(C))]
                m = n if n else int(2 ** rng.integers(0, 4))
                pos = (0, m - 1, int(rng.integers(m)))[(w + lane) % 3]
                live_point(P, rng, c, m, pos)
    for n in (16, 4):   # every observation live and flagged (zc subnormal or at exponent field 253)
        for lane in range(32):
            z = all_live_z[lane % len(all_live_z)]
            obs = [(LIVE + j, (F32(rng.uniform(-1, 1)), F32(rng.uniform(-1, 1)))) for j in range(n)]
            P.point((z * F32(0.5), z * F32(-0.25), z), obs)
    if partial:
        for lane in range(17):
            live_point(P, rng, classes[(3 * lane) % C], 4 if lane % 2 else 8, int(rng.integers(4)))
    return P


def assemble(problems, blocks, block_of, mixed):
    """flat snapshot (MapSnapshot), kf_ptr of the blocks, per-observation feature index in its keyframe, stride"""
    poses, intrs, bnds, kf_first = [], [], [], [0]
    for size in blocks:
        p, i, b = keyframe_block(size, mixed)
        poses.append(p), intrs.append(i), bnds.append(b)
        kf_first.append(kf_first[-1] + size)
    xyz, ptr, kf, uv = [], [0], [], []
    for P, blk in zip(problems, block_of):
        for x, obs in zip(P.xyz, P.lists):
            xyz.append(x)
            for k, u in obs:
                kf.append(kf_first[blk] + k)
                uv.append(u)
            ptr.append(len(kf))
    kf = np.asarray(kf, np.int32)
    nkf = kf_first[-1]
    cnt = np.bincount(kf, minlength=nkf)
    stride = 1 << int(np.ceil(np.log2(max(cnt.max(), 2))))
    order = np.argsort(kf, kind="stable")
    fid = np.empty(kf.size, np.int32)
    start = np.concatenate([[0], np.cumsum(cnt)])
    fid[order] = np.arange(kf.size) - start[kf[order]]
    uv = np.asarray(uv, F32).reshape(-1, 2)
    table = np.zeros((nkf, stride, 2), F32)
    table[kf, fid] = uv
    n = len(xyz)
    snap = synth.MapSnapshot(np.asarray(xyz, F32).reshape(-1, 3), np.asarray(ptr, np.int32), kf, uv, np.concatenate(poses),
                             np.concatenate(intrs), np.concatenate(bnds),
                             np.zeros((n, 2), F32), np.zeros(n, bool))
    return snap, np.asarray(kf_first, np.int32), fid, table, stride


def same(got, want, what):
    """bit for bit; NaN positions compared as sets (CPU and GPU NaN payloads differ)"""
    got, want = np.asarray(got, F32), np.asarray(want, F32)
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), "%s: NaN at %s vs %s" % (what, np.nonzero(gn)[0][:8], np.nonzero(wn)[0][:8])
    bad = np.nonzero(~gn & (bits(got) != bits(want)))[0]
    assert bad.size == 0, "%s: %d differ, first at %d: %r vs %r" % (what, bad.size, bad[0], got[bad[0]], want[bad[0]])


def check(out, ref, what):
    for g, w, name in zip(out, ref, ("observs", "error", "depth")):
        same(g, w, "%s %s" % (what, name))


def class_is_safe(oracle, classes):
    """the class's live observation alone gives a finite error and depth, and an error that the lattice keys hold"""
    probs = [Problem()]
    for c in classes:
        probs[0].point(c[:3], [(c[3], (c[4], c[5]))])
    snap = assemble(probs, [BLOCK_MIN], [0], False)[0]
    _, er, de = oracle.map_point_unary(snap)
    return np.isfinite(er) & np.isfinite(de) & (np.abs(er) <= SAFE_ERROR)


@pytest.fixture(scope="module")
def crafted(oracle):
    """(all classes, the Frames-safe classes) and two problems of each"""
    rng = np.random.default_rng(2024)
    classes = crafted_classes(rng)
    safe = [c for c, ok in zip(classes, class_is_safe(oracle, classes)) if ok]
    assert 0 < len(safe) < len(classes)
    # all-live points: zc subnormal or at exponent field 253 (1/z subnormal); the latter sum to an infinite depth
    sub_z = [fbits(0x00345678), fbits(0x00654321)]
    probs = [make_problem(rng, classes, sub_z + [fbits(0x7e812345), fbits(0x7eff0000)], partial=p) for p in (False, True)]
    probs_safe = [make_problem(rng, safe, sub_z, partial=p) for p in (False, True)]
    return probs, probs_safe


def unary_of(F):
    d = F.get_debug()
    return d["observs"], d["error"], d["depth"]


@pytest.mark.parametrize("mixed", [False, True], ids=["ucam", "mixed_cameras"])
@pytest.mark.parametrize("kfset", ["small", "large"])
def test_unary_crafted_observations(pkg, ctx, oracle, crafted, kfset, mixed):
    probs, probs_safe = crafted
    # with UCAM on and off the routes reach 24 snapshot, 6 VIS and 6 MULTI instantiations
    reached = {(m, t, u, v, mu) for r in ROUTES.values() for m, t, v, mu in r.values() for u in (0, 1)}
    assert len(reached) == 36
    blocks, block_of = ([96], [0, 0]) if kfset == "small" else ([200, 200], [0, 1])
    cam = " mixed" if mixed else ""

    # ---- ctx.map_point_unary: every class
    snap, kf_first, fid, table, stride = assemble(probs, blocks, block_of, mixed)
    nkf = int(kf_first[-1])
    assert (nkf <= 384) == (kfset == "small")
    ref = oracle.map_point_unary(snap)
    n = np.diff(snap.obs_ptr)
    assert ((n & (n - 1)) == 0).all()    # powers of two: error = er / n keeps every bit of er
    assert np.isnan(ref[1]).any() and np.isinf(ref[2]).any() and (ref[1] == 0).any()
    check(ctx.map_point_unary(snap), ref, "ctx.map_point_unary " + kfset + cam)

    # ---- the Frames routes: the safe classes
    snap, kf_first, fid, table, stride = assemble(probs_safe, blocks, block_of, mixed)
    ref = oracle.map_point_unary(snap)
    assert np.isfinite(ref[1]).all() and np.isfinite(ref[2]).all()
    sizes = [len(P.xyz) for P in probs_safe]
    ids = np.arange(snap.n, dtype=np.int32)
    pairs = np.stack([snap.obs_kf, fid], 1).astype(np.int32)

    def load(ptr, ref_pairs):
        mp = pkg.Map(ctx, stride)
        mp.apply(kf_pose=snap.kf_pose, kf_intr=snap.kf_intr, kf_bounds=snap.kf_bounds, kf_keypoints=table, xyz=snap.xyz)
        mp.set_observations(ptr, ref_pairs)
        return mp

    mp = load(snap.obs_ptr, pairs)   # bulk-loaded: every list at a constant pitch
    # odd points are loaded without their last observation, which one delta appends: their (full) lists move
    cnt = np.diff(snap.obs_ptr)
    odd = (np.arange(snap.n) % 2 == 1) & (cnt > 1)
    last = snap.obs_ptr[1:] - 1
    drop = np.zeros(snap.nnz, bool)
    drop[last[odd]] = True
    mp2 = load(np.concatenate([[0], np.cumsum(cnt - odd)]).astype(np.int32), pairs[~drop])
    mp2.apply(add_pt=np.nonzero(odd)[0], add_kf=snap.obs_kf[last[odd]], add_fid=fid[last[odd]])
    assert mp2.sizes()["pool_used"] > mp.sizes()["pool_used"]

    F = pkg.Frames(ctx, sizes)
    F.set_keyframe_keypoints(table)
    for kf_ptr in ([None] if kfset == "small" else [None, kf_first]):
        tag = kfset + ("+kf_ptr" if kf_ptr is not None else "") + cam
        F.set_map_inputs(snap.xyz, snap.obs_ptr, snap.obs_kf, snap.obs_uv, snap.kf_pose, snap.kf_intr, snap.kf_bounds, snap.kp2d, kf_ptr)
        F.run()
        check(unary_of(F), ref, "set_map_inputs int32 " + tag)
        mo, po = np.zeros(snap.n, np.int16), np.zeros((snap.n, 2), F32)
        F.submit_map(0, snap.xyz, snap.obs_ptr, snap.obs_kf.astype(np.uint16), snap.obs_uv, snap.kf_pose, snap.kf_intr,
                     snap.kf_bounds, snap.kp2d, kf_ptr, mo, po)
        F.wait(0)
        check(unary_of(F), ref, "submit_map uint16 " + tag)
        for dt in (np.int32, np.uint16):
            F.set_map_inputs_indexed(snap.xyz, snap.obs_ptr, pairs.astype(dt), snap.kf_pose, snap.kf_intr, snap.kf_bounds,
                                     snap.kp2d, kf_ptr)
            F.run()
            check(unary_of(F), ref, "set_map_inputs_indexed %s %s" % (np.dtype(dt).name, tag))
        for m, what in ((mp, "pitched"), (mp2, "moved")):
            F.set_visible(m, ids, snap.kp2d, kf_ptr=kf_ptr)
            F.run()
            check(unary_of(F), ref, "set_visible %s %s" % (what, tag))
        # two maps.  Without kf_ptr one problem each; with kf_ptr one map serves both problems (slices [0, 200) and
        # [200, 400) of its keyframes) while the other serves none -- a map's last problem ends at its keyframe count
        if kf_ptr is None:
            F.set_visible_maps([mp, mp2], [0, 1, 2], ids, snap.kp2d)
            F.run()
            check(unary_of(F), ref, "set_visible_maps " + tag)
        else:
            for mprob in ([0, 2, 2], [0, 0, 2]):
                F.set_visible_maps([mp, mp2], mprob, ids, snap.kp2d, kf_ptr=kf_ptr)
                F.run()
                check(unary_of(F), ref, "set_visible_maps %s %s" % (mprob, tag))
    F.close()
    mp.close()
    mp2.close()
