"""C5 two ways on one GPU, in one process, alternating: (a) one context, stream, map and host thread per sequence with
lccrf_frames_submit_visible (bench.py's C5 arm), (b) one context whose frame batch serves all sequences' maps with
lccrf_frames_submit_visible_maps.  The sequences are bench.py's: synth.SequenceReplay seeds 5000 + s, 4 TUM and 4 Bonn,
64 frames per batch.  Every timed step of (b) must reproduce (a)'s labels and marginals bit for bit.

    python scripts/multimap_bench.py OUT_DIR [--steps K] [--warmup W] [--round R] [--prefix P]

writes OUT_DIR/P_a.json and OUT_DIR/P_b.json (one JSON line each; P defaults to multimap)."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEQUENCES, FB = 8, 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--round", type=int, default=4, help="steps per mode before the other mode runs the same steps")
    ap.add_argument("--prefix", default="multimap")
    args = ap.parse_args()
    import torch
    pkg = importlib.import_module("lc-crf-slam_b200")
    synth = importlib.import_module("lc-crf-slam_b200.synth")
    W, K, R = args.warmup, args.steps, args.round
    assert W % R == 0 and K % R == 0, "warmup and steps must be multiples of --round"
    prm = pkg.SlamParams.make()
    pinned = []

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        pinned.append(t)
        return t.numpy()

    def build(s):
        gen = synth.SequenceReplay(seed=5000 + s, kind="tum" if s < SEQUENCES // 2 else "bonn", frames_per_batch=FB)
        init = gen.initial_map()
        return gen, init, [gen.next_batch() for _ in range(W + K)]

    with ThreadPoolExecutor(max_workers=SEQUENCES) as ex:
        built = list(ex.map(build, range(SEQUENCES)))

    def load(ctx, gen, init):
        kfs, xyz, ptr, ref = init
        mp = pkg.Map(ctx, gen.stride)
        mp.apply(kf_pose=kfs["pose"], kf_intr=kfs["intr"], kf_bounds=kfs["bounds"], kf_keypoints=kfs["kp"], xyz=xyz)
        mp.set_observations(ptr, ref)
        return mp

    NTs = [int(sum(g.sizes)) for g, _, _ in built]
    off = np.concatenate([[0], np.cumsum(NTs)])
    NT = int(off[-1])
    steps = []   # per step: per-sequence (ids, kp, delta) and the concatenation
    for i in range(W + K):
        per = [(pin(b[i]["ids"]), pin(b[i]["kp2d"]), pkg.MapDelta.make(pin=pin, **b[i]["delta"])) for _, _, b in built]
        steps.append(dict(per=per, ids=pin(np.concatenate([p[0] for p in per])), kp=pin(np.concatenate([p[1] for p in per]))))
    # (a) per-sequence contexts
    A = []
    for s, (gen, init, _) in enumerate(built):
        st = torch.cuda.Stream()
        ctx = pkg.Context(0, stream=st.cuda_stream)
        A.append(dict(ctx=ctx, stream=st, mp=load(ctx, gen, init), F=pkg.Frames(ctx, gen.sizes, prm),
                      outs=[(pin(np.zeros(NTs[s], np.int16)), pin(np.zeros((NTs[s], 2), np.float32))) for _ in range(R)]))
    # (b) one context, one batch over all maps
    sb = torch.cuda.Stream()
    ctxb = pkg.Context(0, stream=sb.cuda_stream)
    maps_b = [load(ctxb, gen, init) for gen, init, _ in built]
    sizes = [n for g, _, _ in built for n in g.sizes]
    map_prob = np.arange(SEQUENCES + 1, dtype=np.int32) * FB
    Fb = pkg.Frames(ctxb, sizes, prm)
    outs_b = [(pin(np.zeros(NT, np.int16)), pin(np.zeros((NT, 2), np.float32))) for _ in range(R)]
    pool = ThreadPoolExecutor(max_workers=SEQUENCES)

    def run_a(i0, i1):
        def seq(s):
            a = A[s]
            for i in range(i0, i1):
                ids, kp, d = steps[i]["per"][s]
                a["F"].wait(i & 1)
                o = a["outs"][i % R]
                a["F"].submit_visible(i & 1, a["mp"], ids, kp, o[0], o[1], delta=d)
            a["F"].wait(0)
            a["F"].wait(1)
        list(pool.map(seq, range(SEQUENCES)))

    def run_b(i0, i1):
        for i in range(i0, i1):
            Fb.wait(i & 1)
            o = outs_b[i % R]
            Fb.submit_visible_maps(i & 1, maps_b, map_prob, steps[i]["ids"], steps[i]["kp"], o[0], o[1],
                                   deltas=[p[2] for p in steps[i]["per"]])
        Fb.wait(0)
        Fb.wait(1)

    def timed(fn, i0, i1, ctxs):
        torch.cuda.synchronize()
        l0 = sum(c.kernel_launches for c in ctxs)
        t0 = time.perf_counter()
        fn(i0, i1)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, sum(c.kernel_launches for c in ctxs) - l0

    tot = {"a": [0.0, 0], "b": [0.0, 0]}
    checked = 0
    for r0 in range(0, W + K, R):
        ta, la = timed(run_a, r0, r0 + R, [a["ctx"] for a in A])
        tb, lb = timed(run_b, r0, r0 + R, [ctxb])
        for i in range(r0, r0 + R):
            for s in range(SEQUENCES):
                ma, pa = A[s]["outs"][i % R]
                mb, pb = outs_b[i % R]
                assert np.array_equal(ma, mb[off[s]:off[s + 1]]), "labels differ: step %d sequence %d" % (i, s)
                assert np.array_equal(pa.view(np.int32), pb[off[s]:off[s + 1]].view(np.int32)), "marginals differ: step %d sequence %d" % (i, s)
            checked += r0 >= W
        if r0 >= W:
            tot["a"][0] += ta
            tot["a"][1] += la
            tot["b"][0] += tb
            tot["b"][1] += lb
    # device rate: the last batch, inputs resident, K graph replays (as bench.py's value)
    last = W + K - 1
    for s, a in enumerate(A):
        a["F"].set_visible(a["mp"], steps[last]["per"][s][0], steps[last]["per"][s][1])
    Fb.set_visible_maps(maps_b, map_prob, steps[last]["ids"], steps[last]["kp"])
    dev = {}
    for mode in ("a", "b"):
        Fs = [a["F"] for a in A] if mode == "a" else [Fb]
        streams = [a["stream"] for a in A] if mode == "a" else [sb]
        for F in Fs:
            F.run()
            F.run()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record(streams[0])
        for _ in range(K):
            for F in Fs:
                F.run()
        ends = []
        for st in streams:
            e = torch.cuda.Event(enable_timing=True)
            e.record(st)
            ends.append(e)
        torch.cuda.synchronize()
        dev[mode] = max(e0.elapsed_time(e) for e in ends) / K
    gpu = card()
    os.makedirs(args.out_dir, exist_ok=True)
    what = {"a": "per-sequence contexts, streams and host threads, lccrf_frames_submit_visible",
            "b": "one context, one frame batch over the 8 maps per step, lccrf_frames_submit_visible_maps"}
    for mode in ("a", "b"):
        sec, launches = tot[mode]
        line = {"workload": "c5", "mode": mode, "arrangement": what[mode], "gpu": gpu, "steps": K, "warmup": W,
                "steps_per_alternation": R, "problems_per_step": SEQUENCES * FB, "points_per_step": NT,
                "device_problems_per_s": SEQUENCES * FB / (dev[mode] * 1e-3), "device_ms_per_step": dev[mode],
                "e2e_problems_per_s": SEQUENCES * FB * K / sec, "e2e_ms_per_step": 1e3 * sec / K,
                "kernel_launches_per_step": launches / K,
                "graphs": "option 'graphs' on: a slot whose launch key repeats replays its captured graph",
                "bit_identical_to_a": True, "steps_checked": checked}
        with open(os.path.join(args.out_dir, "%s_%s.json" % (args.prefix, mode)), "w") as f:
            f.write(json.dumps(line) + "\n")
        print(json.dumps(line), flush=True)
    pool.shutdown()


if __name__ == "__main__":
    main()
