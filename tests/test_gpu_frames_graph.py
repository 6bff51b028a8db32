"""GPU tests (-m gpu) of the CUDA graphs of lccrf_frames: a slot replays its captured graph only while every launch
argument the graph holds is unchanged, and a context option that changes the launch sequence makes every captured
graph stale.  Each run must give the bits of a fresh object that runs the same inputs without graphs."""
import importlib

import numpy as np
import pytest

from util import bits

pytestmark = pytest.mark.gpu
synth = importlib.import_module("lc-crf-slam_b200.synth")
STRIDE = 64


@pytest.fixture
def gctx(pkg):
    """a context of its own: these tests switch context options"""
    c = pkg.Context(0)
    yield c
    c.close()


def direct_inputs(sizes, seed):
    frames = [synth.slam_frame(n, seed=seed + i) for i, n in enumerate(sizes)]
    return [np.concatenate([getattr(f, k) for f in frames]) for k in ("observs", "error", "depth", "kp2d")]


def test_fused_toggle_recaptures(pkg, gctx):
    """Switching "fused" off after a capture must not replay the fused launch sequence."""
    sizes = [1500, 2200]
    inputs = direct_inputs(sizes, seed=70)

    def counted_run(F):
        l0 = gctx.kernel_launches
        F.run()
        n = gctx.kernel_launches - l0
        return n, F.get_outputs()

    gctx.set_option("graphs", 1)
    F = pkg.Frames(gctx, sizes)
    F.set_inputs(*inputs)
    for _ in range(3):  # plain, capture, replay
        F.run()
    gctx.set_option("fused", 0)
    n_toggled, (m1, p1) = counted_run(F)
    gctx.set_option("graphs", 0)
    G = pkg.Frames(gctx, sizes)
    G.set_inputs(*inputs)
    G.run()
    n_plain, (m2, p2) = counted_run(G)  # the second run: no first-use launches
    assert n_toggled == n_plain
    assert np.array_equal(m1, m2) and np.array_equal(bits(p1), bits(p2))
    F.close()
    G.close()


def make_inputs(pkg, ctx):
    snaps = [synth.map_snapshot(n, o, seed=80 + i, n_kf=40, ragged=True) for i, (n, o) in enumerate(((2100, 12), (1300, 20)))]
    cat = pkg.concat_frames(snaps)
    n_kf = cat["kf_pose"].shape[0]
    fid, table, uvc = synth.index_observations(cat["obs_kf"], cat["obs_uv"], n_kf, seed=3, stride=STRIDE)
    d = dict(cat, obs_uv=uvc, n_kf=n_kf, sizes=[s.n for s in snaps], table=table)
    NT = int(cat["xyz"].shape[0])
    d["observs"], d["error"], d["depth"], _ = direct_inputs(d["sizes"], seed=90)
    d["obs_kf16"] = cat["obs_kf"].astype(np.uint16)
    d["ref"] = np.ascontiguousarray(np.stack([cat["obs_kf"], fid], axis=1).astype(np.uint16))
    d["p4"] = np.random.default_rng(4).random(NT) * 0.9
    d["has"] = np.array([1, 0], np.uint8)
    d["ids"] = np.arange(NT, dtype=np.int32)
    mp = pkg.Map(ctx, STRIDE)
    mp.apply(kf_pose=cat["kf_pose"], kf_intr=cat["kf_intr"], kf_bounds=cat["kf_bounds"], kf_keypoints=table, xyz=cat["xyz"])
    mp.set_observations(cat["obs_ptr"], np.stack([cat["obs_kf"], fid], axis=1))
    d["map"] = mp
    return d


def submit(F, d, src, with_kf_ptr, prior):
    """one pipelined step of slot 0 from the given input source; returns (MAP labels, marginals)"""
    out = (np.empty(F.NT, np.int16), np.empty((F.NT, 2), np.float32))
    kf_ptr = d["kf_ptr"] if with_kf_ptr else None
    if prior:
        F.set_prior(0, d["p4"], d["has"])
    else:
        F.set_prior(0, None)
    if src == "direct":
        F.submit(0, d["observs"], d["error"], d["depth"], d["kp2d"], *out)
    elif src in ("snapshot32", "snapshot16"):
        obs_kf = d["obs_kf"] if src == "snapshot32" else d["obs_kf16"]
        F.submit_map(0, d["xyz"], d["obs_ptr"], obs_kf, d["obs_uv"], d["kf_pose"], d["kf_intr"], d["kf_bounds"], d["kp2d"],
                     kf_ptr, *out)
    elif src == "indexed":
        F.submit_map_indexed(0, d["xyz"], d["obs_ptr"], d["ref"], d["kf_pose"], d["kf_intr"], d["kf_bounds"], d["kp2d"],
                             kf_ptr, *out)
    else:
        F.submit_visible(0, d["map"], d["ids"], d["kp2d"], *out, kf_ptr=kf_ptr)
    F.wait(0)
    return out


def test_input_switching_matches_plain_runs(pkg, gctx):
    """One object switches between every input source, keyframe slices and the prior on and off, and grows its
    indexed keypoint table; every run (plain, capture, replay) gives the bits of a fresh object without graphs."""
    d = make_inputs(pkg, gctx)
    # the table grows (it moves) and its first rows change: a stale graph would read the old rows
    table2 = d["table"] + np.float32(0.75)
    grown = np.concatenate([table2, np.zeros((40, STRIDE, 2), np.float32)])
    steps = [("direct", False, False), ("snapshot32", True, False), ("snapshot16", True, True), ("indexed", True, False),
             ("visible", True, False), ("visible", False, True), ("indexed", False, True), ("snapshot32", False, False),
             ("direct", False, True), "insert", ("indexed", True, False), ("snapshot16", False, False),
             ("indexed", True, True), ("visible", True, False)]
    gctx.set_option("graphs", 0)
    want, table = {}, d["table"]
    for st in steps:
        if st == "insert":
            table = table2
            continue
        key = st + ((table is table2 and st[0] == "indexed"),)
        if key not in want:
            G = pkg.Frames(gctx, d["sizes"])
            G.set_keyframe_keypoints(table)
            want[key] = submit(G, d, *st)
            G.close()
    assert not np.array_equal(bits(want[("indexed", True, False, False)][1]), bits(want[("indexed", True, False, True)][1]))
    gctx.set_option("graphs", 1)
    F = pkg.Frames(gctx, d["sizes"])
    F.set_keyframe_keypoints(d["table"])
    inserted = False
    for st in steps:
        if st == "insert":
            F.set_keyframe_keypoints(grown)
            inserted = True
            continue
        m0, p0 = want[st + ((inserted and st[0] == "indexed"),)]
        for rep in range(3):  # plain, capture, replay
            m, p = submit(F, d, *st)
            assert np.array_equal(m, m0) and np.array_equal(bits(p), bits(p0)), (st, rep)
    F.close()
    d["map"].close()
