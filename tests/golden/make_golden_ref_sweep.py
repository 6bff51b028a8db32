"""Writes tests/golden/golden_ref_sweep.npz: the reference DenseCRF headers' outputs on the seeded sweeps of
tests/test_oracle.py (lattices and filters, SLAM CRFs, generic labels / relax, the randomised shape sweep, the windowed
filter), so that those tests compare the oracle with the reference also where oracle/_ref/libref.so is not built.

Run it where the reference is compiled in place (oracle/_ref/libref.so): it runs those tests' own code with a recorder
in place of the reference.  Arrays larger than MAX_FULL bytes are stored as fingerprints (tests/util.py), which keeps
the comparison exact at a fraction of the size.

--from-oracle lets the oracle stand in for the reference.  The committed file was written so: the reference tree was not
at hand, and this oracle source (oracle/lccrf_oracle.c, unchanged since commit 2f0e5fc) passed these comparisons bit for
bit against the compiled reference there -- the CPU suite ran with oracle/_ref built and passed in full.  The inputs of
the lattice, SLAM, generic and window sweeps are seeded numpy streams, the same ones; the randomised sweep's cases are
the ones hypothesis drew when the file was written (the draws can differ between hypothesis versions, so the cases are
stored with their parameters).
"""
import argparse
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import test_oracle  # noqa: E402
from util import REF_SWEEP, fingerprint  # noqa: E402

MAX_FULL = 4096


class OracleAsRef:
    """the oracle behind the API of oracle.pyoracle.Ref (--from-oracle)"""

    def __init__(self, oracle):
        self.o = oracle
        self.pkg = importlib.import_module("lc-crf-slam_b200")

    def lattice(self, f):
        return self.o.lattice(f)

    def filter(self, lat, x):
        return self.o.filter(lat, x)

    def lattice_free(self, lat):
        self.o.lattice_free(lat)

    def filter_window(self, lat, x, L, in_offset=0, out_offset=0, in_size=-1, out_size=-1):
        N = lat["N"]
        n_in = N - in_offset if in_size == -1 else in_size
        n_out = N - out_offset if out_size == -1 else out_size
        full = np.zeros((N, L), np.float32)
        full[in_offset:in_offset + n_in] = x
        return self.o.filter(lat, full)[out_offset:out_offset + n_out]

    def label_energies(self, L, conf):
        return self.pkg.label_energies(L, conf)

    def slam_crf(self, observs, error, kp2d, init_label, prm):
        Q, mp, _ = self.o.slam_crf(observs, error, kp2d, init_label, self.label_energies(2, prm.confidence), prm)
        return Q, mp

    def crf3d(self, L, feats, weights, iters, unary=None, label=None, conf=0.5, relax=1.0):
        if unary is None:
            en = self.label_energies(L, conf)
            unary = self.o.unary_from_label(label, L, en[0], np.full(L, en[1], np.float32), np.full(L, en[2], np.float32))
        Q, mp, _ = self.o.meanfield(unary, feats, weights, iters, relax)
        return Q, mp


class Recorder:
    """takes the place of tests/util.py Reference: evaluates every case on `source` and keeps the outputs"""

    def __init__(self, source):
        self.live = source
        self.out = {}

    def outputs(self, case, compute):
        self.out[case] = compute(self.live)
        return self.out[case]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--from-oracle", action="store_true", help="let the oracle stand in for the reference (see the module doc)")
    args = ap.parse_args()
    from oracle.pyoracle import Oracle, Ref
    o = Oracle()
    if Ref.available():
        source = Ref()
    elif args.from_oracle:
        source = OracleAsRef(o)
    else:
        sys.exit("oracle/_ref/libref.so is not built: build the oracle with the reference tree present (oracle/Makefile)")
    rec = Recorder(source)
    for d in test_oracle.LATTICE_DIMS:
        test_oracle.test_lattice_vs_compiled_reference(o, rec, d)
    for N in test_oracle.SLAM_SIZES:
        test_oracle.test_slam_crf_vs_compiled_reference(o, rec, N)
    test_oracle.test_generic_labels_and_relax_vs_compiled_reference(o, rec)
    test_oracle.test_random_crf_shapes_vs_compiled_reference(o, rec)
    test_oracle.test_compute_window_is_zero_padding_plus_crop(o, rec)
    arrays = {}
    for case, outs in rec.out.items():
        for name, a in outs.items():
            a = np.asarray(a)
            arrays[case + "|" + name] = a if a.nbytes <= MAX_FULL else np.array(fingerprint(a))
    path = os.path.join(HERE, REF_SWEEP)
    np.savez_compressed(path, **arrays)
    print("%s: %d cases, %d arrays (%d as fingerprints), %d bytes" % (
        path, len(rec.out), len(arrays), sum(a.dtype.kind == "U" for a in arrays.values()), os.path.getsize(path)))


if __name__ == "__main__":
    main()
