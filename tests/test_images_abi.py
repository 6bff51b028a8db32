"""CPU test of the batched image section of include/lccrf.h: tests/cpp/images_batch.c is valid C (gcc, no C++) and
links against liblccrf.so.  Without a B200 the program stops at lccrf_ctx_create with exit code 2 (no CPU fallback);
tests/test_gpu_images.py runs it for real."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "lc-crf-slam_b200")


def build_images_batch(tmp_path):
    exe = tmp_path / "images_batch"
    cmd = ["gcc", "-O1", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I" + os.path.join(ROOT, "include"),
           "-o", str(exe), os.path.join(ROOT, "tests", "cpp", "images_batch.c"), "-L" + LIBDIR, "-llccrf", "-lm",
           "-Wl,-rpath," + LIBDIR]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_images_batch_example_compiles_and_links(pkg, tmp_path):
    pkg.load_library()
    exe = build_images_batch(tmp_path)
    if pkg.load_library().lccrf_device_count() == 0:
        run = subprocess.run([str(exe)], capture_output=True, text=True)
        assert run.returncode == 2 and "no CPU fallback" in run.stderr
