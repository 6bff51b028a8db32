"""Batched image CRF (lccrf_images) against the per-object path (lccrf_crf, the loop of `bench.py --workload c2`) on the
same images, in one process on one GPU.  One JSON line per workload, to stdout and to --out.

Workloads (name: W x H, L, B; T = 10, Gaussian sigma 3 w 3 + bilateral sigma 60 / 20 w 10, labels 70 % unknown, the
`synth.image_problem` inputs of bench.py's c2 workload):
  c2_b1, c2_b4, c2_b16   640 x 480, L = 2   -- the C2 shape; 640 x 480 lies above the fused-blur threshold (32768 px)
  golden_b1, golden_b16  320 x 240, L = 21  -- the golden demo's shape (unfused slice / axpy / softmax chain)
  small_b64              160 x 120, L = 2   -- below the threshold: k_blur_fused, one CTA per image

Per workload: device images/s (CUDA events around lccrf_images_run on the context's stream, inputs resident),
end-to-end images/s (host clock around set_inputs + run + get_outputs from page-locked host arrays), kernel launches
per batch, per-kernel shares of one separate profiled run, and the per-object path over the same images (device and
end-to-end, as bench.py times it) with MAP labels asserted equal image by image.

    python scripts/images_bench.py --out DIR [--workloads c2_b16,small_b64] [--pkg-root DIR] [--tag NAME]
--pkg-root imports lc-crf-slam_b200 from another tree (a variant build of the library, scripts/images_blur_threshold.sh).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKLOADS = {
    "c2_b1": (640, 480, 2, 1), "c2_b4": (640, 480, 2, 4), "c2_b16": (640, 480, 2, 16),
    "golden_b1": (320, 240, 21, 1), "golden_b16": (320, 240, 21, 16),
    "small_b64": (160, 120, 2, 64),
}
KERNELS = [(2, 3.0, 3.0, 0.0), (5, 10.0, 60.0, 20.0)]
T = 10
CONF = 0.7          # bench.py C2["conf"]
L2_BYTES = 126e6


def gpu_info():
    """name and power limit of GPU 0 (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # the measurement stands without it, but says so
        return {"error": str(e)}


def pinned(torch, a):
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t.numpy()


def measure(pkg, torch, name, target_s):
    W, H, L, B = WORKLOADS[name]
    synth = pkg.synth
    probs = [synth.image_problem(W, H, 1000 + i, n_labels=L) for i in range(B)]  # bench.py c2 seeds
    en = pkg.label_energies(L, CONF)
    stream = torch.cuda.Stream()
    ctx = pkg.Context(0, stream=stream.cuda_stream)
    img = pinned(torch, np.concatenate([p[0] for p in probs]))
    lab = pinned(torch, np.concatenate([p[1] for p in probs]))
    N = W * H
    mp_out = pinned(torch, np.empty(N * B, np.int16))
    pr_out = pinned(torch, np.empty((N * B, L), np.float32))
    line = {"workload": name, "W": W, "H": H, "L": L, "B": B, "T": T, "kernels": KERNELS, "gpu": gpu_info()}
    with torch.cuda.stream(stream):
        im = pkg.Images(ctx, [(W, H)] * B, L, KERNELS)

        def e2e_step():
            im.set_inputs(img, label=lab, energies=en)
            im.run(T)
            return im.get_outputs(map_out=mp_out, prob_out=pr_out)

        for _ in range(3):  # plain run, capture, replay
            e2e_step()
        maps_batched = mp_out.copy()
        l0 = ctx.kernel_launches
        im.run(T)
        ctx.sync()
        line["launches_per_batch"] = ctx.kernel_launches - l0
        # device: replays of the captured run, inputs resident
        t0 = time.perf_counter()
        im.run(T)
        ctx.sync()
        one = time.perf_counter() - t0
        steps = max(5, int(target_s / max(one, 1e-4)))
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            im.run(T)
        ev1.record(stream)
        ev1.synchronize()
        ms = ev0.elapsed_time(ev1) / steps
        line["device"] = {"images_per_s": B / (ms * 1e-3), "ms_per_batch": ms, "batches": steps}
        # end to end: host clock around set_inputs + run + get_outputs (page-locked host arrays)
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_step()
        ms = 1e3 * (time.perf_counter() - t0) / steps
        line["e2e"] = {"images_per_s": B / (ms * 1e-3), "ms_per_batch": ms, "batches": steps,
                       "h2d_bytes_per_batch": int(img.nbytes + lab.nbytes), "d2h_bytes_per_batch": int(mp_out.nbytes + pr_out.nbytes)}
        assert np.array_equal(mp_out, maps_batched)
        V = im.vertices()
        # per-kernel shares: one separate profiled run (graphs and the second branch are off while profiling)
        ctx.set_option("profile", 1)
        ctx.profile_report()
        im.run(T)
        rep = ctx.profile_report()
        ctx.set_option("profile", 0)
        tot = sum(v[1] for v in rep.values()) or 1.0
        line["profile"] = {"kernel_ms_total": round(tot, 4),
                           "shares": {k: round(v[1] / tot, 4) for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1])},
                           "launches": {k: v[0] for k, v in rep.items()}}
        line["blur"] = "k_blur_fused" if "k_blur_fused" in rep else "element-parallel (k_blur)"
        im.close()

        # the per-object path over the same images: bench.py's c2 step loop
        def obj_step(maps):
            for i, (im_i, lab_i) in enumerate(probs):
                crf = pkg.DenseCRF(ctx, N, L)
                crf.setUnaryEnergyFromLabel(lab_i, energies=en)
                for F, w, posdev, fd in KERNELS:
                    if F == 2:
                        crf.addPairwiseFromImage(W, H, w, posdev)
                    else:
                        crf.addPairwiseFromImage(W, H, w, posdev, im_i, fd)
                crf.inference(T, True)
                maps[i] = crf.getMap().copy()
                crf.close()

        maps = [None] * B
        obj_step(maps)  # warm-up
        t0 = time.perf_counter()
        obj_step(maps)
        one = time.perf_counter() - t0
        osteps = max(2, int(target_s / max(one, 1e-4)))
        ev0.record(stream)
        t0 = time.perf_counter()
        for _ in range(osteps):
            obj_step(maps)
        ev1.record(stream)
        ev1.synchronize()
        wall = time.perf_counter() - t0
        ms = ev0.elapsed_time(ev1) / osteps
        line["per_object"] = {"images_per_s": B / (ms * 1e-3), "ms_per_batch": ms, "e2e_images_per_s": B * osteps / wall,
                              "passes": osteps, "launches_per_image": None}
        for i in range(B):
            assert np.array_equal(maps[i], maps_batched[i * N:(i + 1) * N]), "image %d: batched MAP differs from per-object" % i
        line["maps_equal_per_object"] = True
        l0 = ctx.kernel_launches
        obj_step(maps)
        line["per_object"]["launches_per_image"] = (ctx.kernel_launches - l0) / B
    line["ratio_device_batched_over_per_object"] = line["device"]["images_per_s"] / line["per_object"]["images_per_s"]
    line["ratio_e2e_batched_over_per_object"] = line["e2e"]["images_per_s"] / line["per_object"]["e2e_images_per_s"]
    # bytes one image keeps on the device: per (pixel, remainder) an offset, a barycentric weight and a sorted CSR entry
    # (16 B); per vertex D neighbour pairs and two blur buffers of L values; per pixel unary, marginals, next, tmp and
    # one norm per kernel
    lat_bytes = sum(N * (F + 1) * 16 + int(V[:, k].mean()) * ((F + 1) * 8 + 8 * L) for k, (F, _, _, _) in enumerate(KERNELS))
    lat_bytes += N * (16 * L + 4 * len(KERNELS))
    line["working_set"] = {"lattice_bytes_per_image_est": lat_bytes, "batch_bytes_est": lat_bytes * B,
                           "fits_126MB_L2": lat_bytes * B < L2_BYTES, "V_per_image": V[0].tolist(),
                           "note": "not flushed between timed runs: a batch that fits L2 is read from there after the first pass"}
    ctx.close()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory of the r03_images_<workload>[_<tag>].json files")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--tag", default="")
    ap.add_argument("--target-s", type=float, default=1.0, help="seconds per timed window")
    ap.add_argument("--pkg-root", default=ROOT)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.pkg_root))
    pkg = importlib.import_module("lc-crf-slam_b200")
    import torch
    if not torch.cuda.is_available():
        sys.exit("images_bench: no CUDA device (the measurement needs a B200)")
    os.makedirs(args.out, exist_ok=True)
    for name in args.workloads.split(","):
        line = measure(pkg, torch, name, args.target_s)
        line["build"] = "tree" if os.path.samefile(args.pkg_root, ROOT) else "variant " + os.path.basename(os.path.normpath(args.pkg_root))
        if args.tag:
            line["tag"] = args.tag
        txt = json.dumps(line)
        print(txt, flush=True)
        fn = "r03_images_%s%s.json" % (name, "_" + args.tag if args.tag else "")
        with open(os.path.join(args.out, fn), "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
