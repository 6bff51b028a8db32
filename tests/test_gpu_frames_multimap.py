"""GPU tests (-m gpu) of frame batches against several resident maps (lccrf_frames_set_visible_maps /
submit_visible_maps).  Map m serves a contiguous segment of the batch's problems; every problem's labels, marginals and
debug vectors must be bit-identical to lccrf_frames_set_visible on that problem's map alone (a fresh frames object
per map, and a twin map that receives the same deltas)."""
import importlib

import numpy as np
import pytest

from util import assert_map, assert_marginals, bits

pytestmark = pytest.mark.gpu
synth = importlib.import_module("lc-crf-slam_b200.synth")


# ---------------------------------------------------------------- fixtures
def small_replay(seed, kind):
    """a SequenceReplay at test size: 4 frames per batch of 150..700 points (not multiples of 32), a keyframe every
    4 frames, culling beyond 6 alive keyframes"""
    return synth.SequenceReplay(seed=seed, kind=kind, n_points=4000, frames_per_batch=4, kf_interval=4, kf_window=6,
                                stride=1024, n_frame_points=(150, 700), kf0=8, kf_obs=900)


def load_map(pkg, ctx, gen, init, mixed=False):
    kfs, xyz, ptr, ref = init
    intr = kfs["intr"].copy()
    if mixed:   # every other keyframe with the other sequence's camera: the map takes the UCAM = false path
        intr[1::2] = np.asarray(synth.BONN_INTR if gen.kind == "tum" else synth.TUM_INTR, np.float32)
    mp = pkg.Map(ctx, gen.stride)
    mp.apply(kf_pose=kfs["pose"], kf_intr=intr, kf_bounds=kfs["bounds"], kf_keypoints=kfs["kp"], xyz=xyz)
    mp.set_observations(ptr, ref)
    return mp


class Seq:
    """one replayed sequence with two identical resident maps: `mp` for the multi-map batch, `twin` for the reference
    runs through set_visible"""

    def __init__(self, pkg, ctx, seed, kind, mixed=False):
        self.gen = small_replay(seed, kind)
        init = self.gen.initial_map()
        self.mp, self.twin = load_map(pkg, ctx, self.gen, init, mixed), load_map(pkg, ctx, self.gen, init, mixed)
        self.sizes = list(self.gen.sizes)

    def close(self):
        self.mp.close()
        self.twin.close()


@pytest.fixture
def seqs(pkg, ctx):
    """TUM, Bonn and a mixed-camera TUM sequence"""
    s = [Seq(pkg, ctx, 11, "tum"), Seq(pkg, ctx, 12, "bonn"), Seq(pkg, ctx, 13, "tum", mixed=True)]
    yield s
    for q in s:
        q.close()


def hand_map(pkg, ctx, rng, zones, n_pts, stride=64, intr=synth.TUM_INTR):
    """a map with many keyframes (more than the 384 the unary caches whole): random poses near the origin, points in
    front of them, 2..6 observations per point with random keypoints.  Zone z = keyframes [zones[z], zones[z+1]) and
    points [z * n_pts // Z, (z + 1) * n_pts // Z): a point is observed in keyframes of its zone only.  Returns (map, twin)."""
    n_kf, Z = zones[-1], len(zones) - 1
    pose = np.zeros((n_kf, 12), np.float32)
    for k in range(n_kf):
        R = synth._rot(*rng.normal(0, 0.03, 3))
        pose[k] = np.concatenate([R, rng.normal(0, 0.05, (3, 1))], axis=1).reshape(-1)
    kp = np.stack([rng.uniform(0, 640, (n_kf, stride)), rng.uniform(0, 480, (n_kf, stride))], axis=2).astype(np.float32)
    fx, fy, cx, cy = intr
    z = rng.uniform(1.5, 4.0, n_pts)
    xyz = np.stack([(rng.uniform(20, 620, n_pts) - cx) / fx * z, (rng.uniform(20, 460, n_pts) - cy) / fy * z, z], 1).astype(np.float32)
    cnt = rng.integers(2, 7, n_pts)
    ptr = np.zeros(n_pts + 1, np.int32)
    np.cumsum(cnt, out=ptr[1:])
    zone = np.arange(n_pts) * Z // n_pts
    ref = np.stack([np.concatenate([zones[z] + np.sort(rng.choice(zones[z + 1] - zones[z], c, replace=False)) for z, c in zip(zone, cnt)]),
                    rng.integers(0, stride, int(ptr[-1]))], 1)
    out = []
    for _ in range(2):
        mp = pkg.Map(ctx, stride)
        mp.apply(kf_pose=pose, kf_intr=np.tile(np.asarray(intr, np.float32), (n_kf, 1)),
                 kf_bounds=np.tile(np.array([0, 640, 0, 480], np.float32), (n_kf, 1)), kf_keypoints=kp, xyz=xyz)
        mp.set_observations(ptr, ref.astype(np.int32))
        out.append(mp)
    return out[0], out[1]


def frame_points(rng, n_pts, sizes):
    """problem j takes points of zone j (hand_map)"""
    Z = len(sizes)
    ids = np.concatenate([j * n_pts // Z + rng.choice((j + 1) * n_pts // Z - j * n_pts // Z, s, replace=False)
                          for j, s in enumerate(sizes)]).astype(np.int32)
    kp = np.stack([rng.uniform(0, 640, ids.size), rng.uniform(0, 480, ids.size)], 1).astype(np.float32)
    return ids, kp


def results(F):
    m, p = F.get_outputs()
    d = F.get_debug()
    return [m, bits(p), d["init_label"], bits(d["observs"]), bits(d["error"]), bits(d["depth"])]


def reference(pkg, ctx, mp, sizes, ids, kp, delta=None, kf_ptr=None):
    """set_visible on a fresh frames object for one map's problems"""
    F = pkg.Frames(ctx, sizes)
    F.set_visible(mp, ids, kp, delta=delta, kf_ptr=kf_ptr)
    F.run()
    r = results(F)
    F.close()
    return r


def assert_segments(got, refs, seg_pts):
    """got: results of the multi-map batch; refs[m]: of map m alone; seg_pts: point range of every segment"""
    for m, (a, b) in enumerate(seg_pts):
        for x, y in zip(got, refs[m]):
            assert np.array_equal(x[a:b], y), "segment %d" % m


def cat(xs, dt):
    return np.ascontiguousarray(np.concatenate(xs), dt)


# ---------------------------------------------------------------- tests
def test_multimap_matches_per_map_runs(pkg, ctx, oracle, seqs):
    """TUM + Bonn + mixed-camera maps, a map with no problem but a delta, and a zero-point problem: one batch, per
    problem bit-identical to set_visible; a few problems against the oracle on the generator's host model"""
    from oracle.pyoracle import slam_params
    rng = np.random.default_rng(3)
    idle = Seq(pkg, ctx, 14, "bonn")   # serves no problem but applies its delta
    batches = [q.gen.next_batch() for q in seqs]
    idle_b = idle.gen.next_batch()
    sizes = [list(q.sizes) for q in seqs]
    # a zero-point problem at the end of the first segment: its points are none of the frame's
    sizes[0] = sizes[0] + [0]
    maps = [seqs[0].mp, idle.mp, seqs[1].mp, seqs[2].mp]
    order = [batches[0], idle_b, batches[1], batches[2]]
    nprob = [len(sizes[0]), 0, len(sizes[1]), len(sizes[2])]
    map_prob = np.concatenate([[0], np.cumsum(nprob)])
    deltas = [pkg.MapDelta.make(**b["delta"]) for b in order]
    ids = cat([batches[0]["ids"], batches[1]["ids"], batches[2]["ids"]], np.int32)
    kp = cat([batches[0]["kp2d"], batches[1]["kp2d"], batches[2]["kp2d"]], np.float32)
    F = pkg.Frames(ctx, sizes[0] + sizes[1] + sizes[2])
    F.set_visible_maps(maps, map_prob, ids, kp, deltas=deltas)
    F.run()
    got = results(F)
    refs, seg_pts, a = [], [], 0
    for q, b, sz in zip(seqs, batches, sizes):
        refs.append(reference(pkg, ctx, q.twin, sz, b["ids"], b["kp2d"], delta=pkg.MapDelta.make(**b["delta"])))
        seg_pts.append((a, a + int(sum(sz))))
        a += int(sum(sz))
    idle.twin.apply(pkg.MapDelta.make(**idle_b["delta"]))
    assert_segments(got, refs, seg_pts)
    assert all(idle.mp.sizes()[k] == idle.twin.sizes()[k] for k in ("n_kf", "n_points", "n_obs"))
    # the oracle on the host model (which has seen the same keyframes, culls, bad points and BA updates)
    prm_o = slam_params(**synth.SLAM_PARAMS)
    dbg = F.get_debug()
    en = pkg.label_energies(2, pkg.SlamParams.make().confidence)
    mp_out, pr_out = F.get_outputs()
    for q, b, (s0, _) in zip(seqs[:2], batches[:2], seg_pts[:2]):
        j = int(rng.integers(0, len(q.sizes)))
        a0 = s0 + int(sum(q.sizes[:j]))
        a1 = a0 + q.sizes[j]
        snap = q.gen.snapshot(ids[a0:a1], kp[a0:a1])
        ob, er, de = oracle.map_point_unary(snap)
        assert np.array_equal(bits(er), bits(dbg["error"][a0:a1])) and np.array_equal(bits(de), bits(dbg["depth"][a0:a1]))
        Qo, mo, _ = oracle.slam_crf(ob, er, snap.kp2d, dbg["init_label"][a0:a1], en, prm_o)
        assert_marginals(pr_out[a0:a1], Qo, what="multi-map vs oracle")
        assert_map(mp_out[a0:a1], mo, Qo, what="multi-map vs oracle")
    F.close()
    idle.close()


def test_multimap_single_map_equals_set_visible(pkg, ctx, seqs):
    """n_maps = 1 is set_visible"""
    q = seqs[1]
    b = q.gen.next_batch()
    F = pkg.Frames(ctx, q.sizes)
    F.set_visible_maps([q.mp], [0, len(q.sizes)], b["ids"], b["kp2d"], deltas=[pkg.MapDelta.make(**b["delta"])])
    F.run()
    got = results(F)
    ref = reference(pkg, ctx, q.twin, q.sizes, b["ids"], b["kp2d"], delta=pkg.MapDelta.make(**b["delta"]))
    for x, y in zip(got, ref):
        assert np.array_equal(x, y)
    F.close()


def test_multimap_keyframe_slices(pkg, ctx):
    """maps of more than 384 keyframes with kf_ptr slices (the per-problem shared slice of the unary): per segment
    equal to set_visible with that map's own kf_ptr; n_maps = 1 equals set_visible with the same kf_ptr"""
    rng = np.random.default_rng(7)
    fa, fb = [0, 150, 300, 420], [0, 250, 500]   # problem j's slice = zone j of its map
    (a, a2), (b, b2) = hand_map(pkg, ctx, rng, fa, 3000), hand_map(pkg, ctx, rng, fb, 2500, intr=synth.BONN_INTR)
    sa, sb = [300, 513, 257], [1000, 33]
    ia, ka = frame_points(rng, 3000, sa)
    ib, kb = frame_points(rng, 2500, sb)
    ra = reference(pkg, ctx, a2, sa, ia, ka, kf_ptr=np.array(fa, np.int32))
    rb = reference(pkg, ctx, b2, sb, ib, kb, kf_ptr=np.array(fb, np.int32))
    F = pkg.Frames(ctx, sa + sb)
    kf_ptr = np.array(fa[:-1] + fb, np.int32)   # the last problem of a segment ends at its map's keyframe count
    F.set_visible_maps([a, b], [0, 3, 5], cat([ia, ib], np.int32), cat([ka, kb], np.float32), kf_ptr=kf_ptr)
    F.run()
    assert_segments(results(F), [ra, rb], [(0, sum(sa)), (sum(sa), sum(sa) + sum(sb))])
    F.close()
    F = pkg.Frames(ctx, sa)
    F.set_visible_maps([a], [0, 3], ia, ka, kf_ptr=np.array(fa, np.int32))
    F.run()
    for x, y in zip(results(F), ra):
        assert np.array_equal(x, y)
    # an observation outside its problem's slice is reported by wait (a slice of one keyframe)
    out = (np.zeros(sum(sa), np.int16), np.zeros((sum(sa), 2), np.float32))
    F.submit_visible_maps(0, [a], [0, 3], ia, ka, out[0], out[1], kf_ptr=np.array([0, 1, 2, 420], np.int32))
    with pytest.raises(pkg.LccrfError, match="outside its table"):
        F.wait(0)
    F.close()
    for m in (a, a2, b, b2):
        m.close()


def run_pipelined(pkg, ctx, seqs, steps):
    """steps x (one submit_visible_maps with per-map deltas); returns the per-step results and the references"""
    sizes = [s for q in seqs for s in q.sizes]
    map_prob = np.concatenate([[0], np.cumsum([len(q.sizes) for q in seqs])]).astype(np.int32)
    seg_pts = []
    a = 0
    for q in seqs:
        seg_pts.append((a, a + sum(q.sizes)))
        a += sum(q.sizes)
    F = pkg.Frames(ctx, sizes)
    outs = [(np.zeros(a, np.int16), np.zeros((a, 2), np.float32)) for _ in (0, 1)]
    keep, got, want = {}, {}, {}
    for s in range(steps):
        bs = [q.gen.next_batch() for q in seqs]
        deltas = [pkg.MapDelta.make(**b["delta"]) for b in bs]
        ids, kp = cat([b["ids"] for b in bs], np.int32), cat([b["kp2d"] for b in bs], np.float32)
        want[s] = [reference(pkg, ctx, q.twin, q.sizes, b["ids"], b["kp2d"], delta=pkg.MapDelta.make(**b["delta"]))[:2]
                   for q, b in zip(seqs, bs)]
        if s >= 2:
            F.wait(s & 1)
            got[s - 2] = (outs[s & 1][0].copy(), bits(outs[s & 1][1]).copy())
        keep[s & 1] = (ids, kp, deltas)
        F.submit_visible_maps(s & 1, [q.mp for q in seqs], map_prob, ids, kp, outs[s & 1][0], outs[s & 1][1], deltas=deltas)
    for s in (steps - 2, steps - 1):
        F.wait(s & 1)
        got[s] = (outs[s & 1][0].copy(), bits(outs[s & 1][1]).copy())
    for s in range(steps):
        assert_segments(list(got[s]), want[s], seg_pts)
    return F


def test_multimap_pipelined_with_deltas(pkg, ctx, seqs):
    """submit_visible_maps over several steps (keyframe insertion, culling, pool growth, graph capture and replay)
    against per-map set_visible runs of the same steps on twin maps"""
    pool0 = [q.mp.sizes()["pool_cap"] for q in seqs]
    F = run_pipelined(pkg, ctx, seqs, 7)
    for q, p0 in zip(seqs, pool0):
        sz, tw = q.mp.sizes(), q.twin.sizes()
        assert sz["n_kf"] == tw["n_kf"] and sz["n_obs"] == tw["n_obs"]
    assert any(q.mp.sizes()["n_kf"] > 8 for q in seqs)
    F.close()


def test_multimap_graph_keys(pkg, ctx, seqs):
    """the same key replays bit-identically; a new map list, map_prob or bucket drops the graph and gives a fresh
    object's results; set_visible and set_visible_maps may alternate on one object"""
    rng = np.random.default_rng(9)
    q0, q1 = seqs[0], seqs[1]
    n0, n1 = sum(q0.sizes), sum(q1.sizes)
    b0, b1 = q0.gen.next_batch(), q1.gen.next_batch()
    for q, b in ((q0, b0), (q1, b1)):   # both maps of each sequence take the step's delta once
        q.mp.apply(pkg.MapDelta.make(**b["delta"]))
        q.twin.apply(pkg.MapDelta.make(**b["delta"]))
    sizes = q0.sizes + q1.sizes
    ids, kp = cat([b0["ids"], b1["ids"]], np.int32), cat([b0["kp2d"], b1["kp2d"]], np.float32)

    def fresh(maps, map_prob, sz, ids_, kp_):
        G = pkg.Frames(ctx, sz)
        G.set_visible_maps(maps, map_prob, ids_, kp_)
        G.run()
        r = results(G)
        G.close()
        return r

    F = pkg.Frames(ctx, sizes)
    mp01 = [0, len(q0.sizes), len(sizes)]
    base = fresh([q0.mp, q1.mp], mp01, sizes, ids, kp)
    l0 = ctx.kernel_launches
    for _ in range(4):   # first run, capture run, two replays
        F.set_visible_maps([q0.mp, q1.mp], mp01, ids, kp)
        F.run()
        for x, y in zip(results(F), base):
            assert np.array_equal(x, y)
    assert ctx.kernel_launches - l0 > 0
    # the map list changes: the same problems, the second map's points re-read from its twin
    F.set_visible_maps([q0.mp, q1.twin], mp01, ids, kp)
    F.run()
    for x, y in zip(results(F), base):
        assert np.array_equal(x, y)
    # map_prob changes: all problems from the first map (the second sequence's frames named in the first map)
    ids0 = ids.copy()
    ids0[n0:] = rng.choice(np.nonzero(q0.gen.has.any(1) & ~q0.gen.bad)[0], n1)
    for mprob in ([0, len(sizes), len(sizes)], mp01):
        ii = ids0 if mprob[1] == len(sizes) else ids
        F.set_visible_maps([q0.mp, q1.mp], mprob, ii, kp)
        F.run()
        for x, y in zip(results(F), fresh([q0.mp, q1.mp], mprob, sizes, ii, kp)):
            assert np.array_equal(x, y)
    # a bucket changes: 130 keyframes in the second map (bucket 128 -> 256)
    nk = q1.mp.sizes()["n_kf"]
    add = 130 - nk
    kfd = dict(kf_first=nk, kf_pose=np.tile(q1.gen.kf_pose[-1], (add, 1)), kf_intr=np.tile(q1.gen.intr, (add, 1)),
               kf_bounds=np.tile(q1.gen.bounds, (add, 1)), kf_keypoints=np.zeros((add, q1.gen.stride, 2), np.float32))
    F.set_visible_maps([q0.mp, q1.mp], mp01, ids, kp, deltas=[None, pkg.MapDelta.make(**kfd)])
    F.run()
    q1.twin.apply(pkg.MapDelta.make(**kfd))
    assert q1.mp.sizes()["n_kf"] == 130
    for x, y in zip(results(F), fresh([q0.twin, q1.twin], mp01, sizes, ids, kp)):
        assert np.array_equal(x, y)
    # alternating with set_visible / submit_visible on the same object (a one-map batch of the same problems)
    G = pkg.Frames(ctx, sizes)
    out = (np.zeros(n0 + n1, np.int16), np.zeros((n0 + n1, 2), np.float32))
    ids00 = cat([b0["ids"], ids0[n0:]], np.int32)
    for _ in range(3):
        F.set_visible_maps([q0.mp, q1.mp], mp01, ids, kp)
        F.run()
        r1 = results(F)
        F.submit_visible(1, q0.mp, ids00, kp, out[0], out[1])
        F.wait(1)
        F.set_visible(q0.mp, ids00, kp)
        F.run()
        r2 = results(F)
        G.set_visible(q0.twin, ids00, kp)
        G.run()
        for x, y in zip(r1, fresh([q0.twin, q1.twin], mp01, sizes, ids, kp)):
            assert np.array_equal(x, y)
        for x, y in zip(r2, results(G)):
            assert np.array_equal(x, y)
        assert np.array_equal(out[0], r2[0]) and np.array_equal(bits(out[1]), r2[1])
    F.close()
    G.close()


def test_multimap_errors(pkg, ctx, seqs):
    q0, q1 = seqs[0], seqs[1]
    sizes = q0.sizes + q1.sizes
    NT = sum(sizes)
    rng = np.random.default_rng(4)
    live = [np.nonzero(q.gen.has.any(1) & ~q.gen.bad)[0] for q in (q0, q1)]
    ids = cat([rng.choice(live[0], sum(q0.sizes), replace=False), rng.choice(live[1], sum(q1.sizes), replace=False)], np.int32)
    kp = np.stack([rng.uniform(0, 640, NT), rng.uniform(0, 480, NT)], 1).astype(np.float32)
    F = pkg.Frames(ctx, sizes)
    mp01 = [0, len(q0.sizes), len(sizes)]
    lib = ctx.lib
    with pytest.raises(pkg.LccrfError, match="n_maps"):
        ctx._check(lib.lccrf_frames_set_visible_maps(F.h, 0, (pkg._vp * 1)(q0.mp.h), None, np.array([0], np.int32).ctypes.data,
                                                      ids.ctypes.data, kp.ctypes.data, None))
    with pytest.raises(pkg.LccrfError, match="NULL"):
        ctx._check(lib.lccrf_frames_set_visible_maps(F.h, 2, (pkg._vp * 2)(q0.mp.h, None), None,
                                                      np.array(mp01, np.int32).ctypes.data, ids.ctypes.data, kp.ctypes.data, None))
    ctx2 = pkg.Context(0)
    other = pkg.Map(ctx2, 64)
    with pytest.raises(pkg.LccrfError, match="different contexts"):
        F.set_visible_maps([q0.mp, other], mp01, ids, kp)
    other.close()
    ctx2.close()
    with pytest.raises(pkg.LccrfError, match="twice"):
        F.set_visible_maps([q0.mp, q0.mp], mp01, ids, kp)
    for bad in ([0, 2, len(sizes) - 1], [1, 2, len(sizes)], [0, len(sizes), 2]):
        with pytest.raises(pkg.LccrfError, match="map_prob"):
            F.set_visible_maps([q0.mp, q1.mp], bad, ids, kp)
    n0, n1 = q0.mp.sizes()["n_kf"], q1.mp.sizes()["n_kf"]
    P0, P1 = len(q0.sizes), len(q1.sizes)
    for bad in ([0] * P0 + [0] * P1 + [n1 + 1],               # kf_ptr[B] beyond the last map's keyframes
                [0, n0 + 1] + [n0] * (P0 - 2) + [0] * P1 + [n1],  # a slice beyond its map's keyframes
                [1] + [n0] * (P0 - 1) + [0] * P1 + [n1],          # a segment that does not start at 0
                [0] * P0 + [0, 2, 1] + [n1] * (P1 - 2)):          # decreasing
        with pytest.raises(pkg.LccrfError, match="kf_ptr"):
            F.set_visible_maps([q0.mp, q1.mp], mp01, ids, kp, kf_ptr=np.array(bad, np.int32))
    empty = pkg.Map(ctx, 64)
    with pytest.raises(pkg.LccrfError, match="no keyframes"):
        F.set_visible_maps([q0.mp, empty], mp01, ids, kp)
    F.set_visible_maps([q0.mp, empty, q1.mp], [0, P0, P0, len(sizes)], ids, kp)  # (serves no problem)
    empty.close()
    # the in-flight guard
    out = (np.zeros(NT, np.int16), np.zeros((NT, 2), np.float32))
    F.submit_visible_maps(0, [q0.mp, q1.mp], mp01, ids, kp, out[0], out[1])
    with pytest.raises(pkg.LccrfError, match="in flight"):
        F.set_visible_maps([q0.mp, q1.mp], mp01, ids, kp)
    with pytest.raises(pkg.LccrfError, match="in flight"):
        F.submit_visible_maps(0, [q0.mp, q1.mp], mp01, ids, kp, out[0], out[1])
    F.wait(0)
    F.close()
