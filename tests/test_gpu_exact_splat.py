"""Adversarial long-row tests of the ordered splat (-m gpu): every vertex value must be the reference's left-to-right
fp32 sum, bit for bit, also where the exact scan of csrc/filter.cu (integer ulp composites, predicted binades, crossing
windows, fallbacks) meets its edges.

The rows are built from clusters of identical feature vectors at positions whose barycentric row is a single 1: the
weight-1 vertex of a cluster then sums exactly the chosen inputs, in point order, and the cluster's other vertices sum
+-0 (or NaN for non-finite inputs).  The clusters' points are interleaved, so no row is contiguous in point order.  An
event meant for the O(1) chunk records sits in a chunk behind the row's head chunk (entry >= 2048).

Every case runs at L = 1, 2 and 3 (label l holds the label-0 inputs times 2^l; L = 3 is the two-label group plus a
masked one) and checks with lattice.debug_counters() that the path it aims at was taken."""
import numpy as np
import pytest

from util import assert_bit_exact

pytestmark = pytest.mark.gpu

f32 = np.float32
CH = 2048                                          # entries per chunk of a long row (engine.cuh: kScanChunk)
CENTERS = [(0.0, 12.0 * k) for k in range(-4, 5)]  # d = 2 positions whose barycentric row is one 1 and two 0


def at(chunk, rnd=0, lane=0, k=0):
    """entry index of a row: chunk, round of 256 entries, lane of 8 entries, entry of the lane"""
    return chunk * CH + rnd * 256 + lane * 8 + k


def row(n, events):
    """n products, zero except {entry: value}"""
    r = np.zeros(n, f32)
    for i, v in events.items():
        r[i] = f32(v)
    return r


def seq(r, s=0.0):
    """the reference's sum: ((s + r0) + r1) + ... in fp32"""
    s = f32(s)
    for c in r:
        s = f32(s + c)
    return s


def interleave(rows):
    """features and label-0 inputs: cluster k holds rows[k] in point order, the clusters' points interleaved"""
    K = len(rows)
    assert K <= len(CENTERS)
    keys = np.concatenate([(np.arange(len(r)) + (k + 1) / (K + 1)) / len(r) for k, r in enumerate(rows)])
    cl = np.concatenate([np.full(len(r), k) for k, r in enumerate(rows)])
    val = np.concatenate(rows).astype(f32)
    p = np.argsort(keys, kind="stable")
    return np.array(CENTERS, f32)[cl[p]], val[p], cl[p]


class Case:
    def __init__(self, rows, expect=(), sums=None, wrong=None, counts=None, absent=()):
        self.rows = rows
        self.counts = counts or {}    # {counter: value} of the lattice's row classification
        self.expect = expect          # counters that must grow in every call: rec_fast, rec_cross, rec_fallback, rec_zero
        self.absent = absent          # counters that must not grow
        self.sums = sums or {}        # {row: the sequential sum the case is built to reach}
        self.wrong = wrong or {}      # {row: inputs whose sum is the value a rounded lower bound accepted instead}


U1 = 2.0 ** -22                       # ulp of [2, 4)
BELOW2 = f32(2 - 2.0 ** -23)          # 1.9999999


def binade_bottom(where):
    """running sum 2 + k*u, then one product that lands the exact sum at 2 - t*u (t = 3/8, the tie 1/2 and the
    boundary 1/4, which rounds back to 2) for k = 0..2 (both parities of m).  The last row is the same layout with a
    negative product that stays inside the binade (k = 3, t = -2.625): its chunk 2 record must apply, which pins the
    record kind the layout gets (plain, or a crossing for cross_a / cross_b)."""
    rows, sums, wrong = [], {}, {}
    for k, t in [(k, t) for k in range(3) for t in (0.375, 0.5)] + [(1, 0.25), (3, -2.625)]:
        ev = {0: 2.0}
        if where == "plain":         # chunk 1: a record applied in O(1); chunk 2: the event; chunk 3: zeros
            ev[at(1, 0, 12)] = k * U1
            e = at(2, 4, 19, 3)
            n = 4 * CH
        elif where == "fallback":    # chunk 2 leaves the binade and comes back first: summed by row_sum_exact
            ev[at(1, 0, 12)] = k * U1
            ev[at(2, 0, 1, 2)] = -1.0
            ev[at(2, 0, 1, 6)] = 1.0
            e = at(2, 4, 19, 3)
            n = 3 * CH + 17
        elif where == "cross_a":     # chunk 2 is a kRecCross record (sp = 2 + k*u, total about 4 + 3u): the event in
            # composite A, the crossing 3 rounds later in the window
            ev[at(1, 0, 12)] = k * U1
            e = at(2, 1, 5, 1)
            ev[at(2, 4, 10, 3)] = 2.0 + 3 * U1
            n = 3 * CH
        else:                        # "cross_b": chunk 2 is a kRecCross record (sp = 2 + 2k*u, total about 4): the
            # crossing first, in the window on lanes 2-5 of round 0, the event in composite B at binade [4, 8)
            ev[at(1, 0, 12)] = 2 * k * U1   # running sum 4 + k*2u behind the crossing
            ev[at(2, 0, 3, 1)] = 2.0
            e = at(2, 3, 7, 1)
            n = 3 * CH
        scale = 2.0 if where == "cross_b" else 1.0
        ev[e] = -(k + t) * U1 * scale
        i = len(rows)
        rows.append(row(n, ev))
        if t < 0:
            continue
        if where == "cross_a":
            sums[i] = seq([BELOW2 if t > 0.25 else f32(2), f32(2.0 + 3 * U1)])
        elif where == "cross_b":
            sums[i] = f32(4 - 2.0 ** -22) if t > 0.25 else f32(4)
        else:
            sums[i] = BELOW2 if t > 0.25 else f32(2)
        if t > 0.25:   # what the old lower bound produced: the event as if it landed on 2^E
            w = dict(ev)
            w[e] = -k * U1 * scale
            wrong[i] = row(n, w)
    return rows, sums, wrong


def case_binade_bottom(where):
    rows, sums, wrong = binade_bottom(where)
    expect = ("rec_fast", "rec_fallback") + (("rec_zero",) if where == "plain" else ()) + \
        (("rec_cross",) if where.startswith("cross") else ())
    return rows, sums, wrong, expect


def case_binade_top():
    """exact sums in [2^24 - 1/2, 2^24) ulps of [2, 4), which round up to 4: from 4 - k*u, and from 3 inside a chunk"""
    rows, sums = [], {}
    for k, t in ((1, 0.5), (1, 0.75), (2, 1.5), (3, 2.625)):
        # from 4 - k*u: +t*u early in a chunk that ends near 3
        rows.append(row(2 * CH + 5, {0: 4 - k * U1, at(1, 0, 2, 5): t * U1, at(1, 6, 1): -1.0}))
        sums[len(rows) - 1] = f32(3.0)
        # from 3: +1 - k*u, then +t*u, then -1 again: a plain chunk whose upper bound must send it to real additions
        rows.append(row(2 * CH + 900, {0: 3.0, at(1, 2, 4): 1 - k * U1, at(1, 2, 20): t * U1, at(1, 5, 0): -1.0}))
        sums[len(rows) - 1] = f32(3.0)
    return rows, sums, ("rec_fallback",)


def case_crossings():
    rows = [
        # the predicted crossing hits lane 0 of a round (tw clamps to 0), the window applied
        row(3 * CH, {0: 2.0, at(1, 3, 0, 0): 1.999, at(1, 3, 0, 1): 0.5, at(2, 1, 3): 0.25}),
        # predicted to reach 4 (1 - 1e-4) but not 4 (1 - 2e-5): no crossing by the last round, window on its last lanes
        row(2 * CH + 3, {0: 2.0, at(1, 0, 5): 1.0, at(1, 7, 28, 2): 0.99971, at(1, 7, 30): 2.0 ** -20}),
        # two crossings in one chunk (2 -> 4 -> 8 and back under 8)
        row(2 * CH + 64, {0: 2.0, at(1, 1, 3): 2.0, at(1, 4, 7): 4.5, at(1, 6, 0): -3.0}),
        # a crossing is predicted but does not happen: chunk 1 cancels to 0.5 in order, but its unordered sum says 2.5
        # in front of chunk 2, whose +1.6 then predicts 4.1 while the true running sum only reaches 2.1
        row(3 * CH, {0: 2.0, at(1, 0, 0, 5): 1e8, at(1, 0, 1, 1): -1e8, at(1, 0, 6): 0.5, at(2, 2, 2): 1.6}),
        # a clean crossing (A, window, B all applied) and a clean plain chunk
        row(3 * CH, {0: 2.0, at(1, 0, 3): 0.75, at(1, 3, 17): 1.5, at(1, 6, 2): 0.125, at(2, 2, 2): 1.0}),
    ]
    return rows, {}, ("rec_fast", "rec_cross", "rec_fallback")


def signed_steps(rng, n, u):
    """n products of whole ulps, quarter ulps, ties (1/2) and 3/8 ulps, of either sign, at least one negative"""
    q = rng.choice([-3, -2, -1, -0.5, -0.375, 0.25, 0.5, 0.625, 1, 2, 3], n)
    q[0] = -1
    return (q * u).astype(f32)


def case_signed_records(rng):
    """signed chunks that stay inside their binade: every non-head chunk of the weight-1 rows has a negative product,
    so its record is a non-monotone composite, and every one of them must apply without a fallback.  The first row
    starts from an odd m with q = -1/2 + 2^-25, whose fraction q - floor(q) rounds to exactly 1/2 in fp32."""
    rows, sums, wrong = [], {}, {}
    half = -0.5 + 2.0 ** -25
    for a in range(2):
        r = np.zeros(3 * CH + 100, f32)
        r[0] = f32(3.0 + (1 - a) * U1)                     # m = 1.5 * 2^23 + 1 (odd), or even
        for c in (1, 2, 3):
            pos = np.sort(rng.choice(np.arange(at(c) + 1, min(at(c + 1), len(r))), 80, replace=False))
            r[pos] = signed_steps(rng, 80, U1)
        r[at(1)] = f32(half * U1)                          # the first product of chunk 1
        rows.append(r)
        if a == 0:
            w = r.copy()
            w[at(1)] = f32(-U1)                            # where a fraction read as a tie rounds to: m - 1
            wrong[len(rows) - 1] = w
    for a in range(2):
        # a crossing record from signed composites: A in [2, 4), the +1.5 in the window (round 3, lane 10), B in [4, 8)
        r = np.zeros(3 * CH, f32)
        r[0] = f32(3.0 + a * U1)
        pos = np.sort(rng.choice(np.arange(at(1) + 1, at(2)), 80, replace=False))
        r[pos] = signed_steps(rng, 80, U1)
        pos = np.sort(rng.choice(np.arange(at(2), at(2, 3)), 40, replace=False))
        r[pos] = signed_steps(rng, 40, U1)
        pos = np.sort(rng.choice(np.arange(at(2, 4), at(3)), 40, replace=False))
        r[pos] = signed_steps(rng, 40, 2 * U1)
        r[at(2, 3, 10, 2)] = f32(1.5)
        rows.append(r)
    return rows, sums, wrong


def case_exponent_range(rng):
    """running sums in binades -101, -100, 100, 101 (the scan's range is [-100, 100]), each with a signed tail and a
    binade-bottom event in a later chunk"""
    rows, sums = [], {}
    for E in (-101, -100, 100, 101):
        u = 2.0 ** (E - 23)
        r = np.zeros(3 * CH, f32)
        r[0] = f32(1.5 * 2.0 ** E)
        tail = rng.integers(-4, 5, 600)              # whole ulps: every prefix exact inside the binade
        r[CH + 7: CH + 7 + 3 * 600: 3] = (tail * u).astype(f32)
        r[at(2, 0, 0)] = f32(-(0.5 * 2.0 ** 23 + tail.sum()) * u)   # back to exactly 2^E in front of the event
        r[at(2, 1, 1)] = f32(-0.375 * u)
        rows.append(r)
        sums[len(rows) - 1] = f32(2.0 ** E - 2.0 ** (E - 24))
    return rows, sums, ("rec_fallback",)


def case_subnormal(rng):
    sub = f32(2.0 ** -140)
    rows = [
        # subnormal products, subnormal running sums (signed, with exact cancellations)
        (rng.integers(-40, 41, 3 * CH + 11) * sub).astype(f32),
        # a normal running sum near 2^-100 and subnormal products: ulps of 2^-123
        np.concatenate([[f32(2.0 ** -100)], (rng.integers(-9, 10, 3 * CH) * sub).astype(f32)]),
        # running sum 2^-126 (the smallest normal) falling into the subnormals and back
        np.concatenate([[f32(2.0 ** -126)], (rng.integers(-3, 4, 2 * CH + 700) * f32(2.0 ** -149)).astype(f32)]),
    ]
    rows[0][0] = f32(5 * sub)
    return rows, {}, ("rec_fallback",)


def case_cancel_to_zero(rng):
    """a row that cancels to exactly +0 in the middle (in the head, at a chunk boundary, inside a chunk) and goes on"""
    rows = []
    for z in (at(0, 5, 2), at(1, 0, 0), at(1, 3, 9, 4)):
        r = np.zeros(4 * CH + 100, f32)
        r[:z] = (rng.random(z) < 0.05) * rng.integers(1, 5, z) * f32(0.25)
        r[z] = -seq(r[:z])
        r[z + 1: z + 40] = -0.0
        r[at(3):] = (rng.random(len(r) - at(3)) * 0.01).astype(f32)
        r[at(2, 4):at(2, 4) + 30] = f32(-0.0)
        rows.append(r)
    return rows, {}, ("rec_fast", "rec_zero")


def case_nonfinite():
    big = f32(3e38)
    rows = [
        row(3 * CH, {0: 2.0, at(1, 2, 3): big, at(1, 2, 4): big, at(2, 0, 0): 1.0}),                     # overflow to +inf
        row(3 * CH, {0: 2.0, at(1, 2, 3): big, at(1, 2, 4): big, at(1, 6, 1): -np.inf, at(2, 3): 1.0}),  # inf - inf
        row(3 * CH, {0: 2.0, at(1, 4, 4): np.nan, at(2, 1): 0.5}),                                        # NaN input
        row(3 * CH, {0: 2.0, at(2, 1, 2): np.inf}),                                                       # inf input
        row(3 * CH, {0: 2.0, at(1, 0, 1): 0.5}),                                                          # finite beside them
    ]
    return rows, {}, ()


def case_row_lengths(rng):
    """long rows of every boundary length, short rows that start near the end of a 2048-entry tile"""
    rows = [(rng.normal(0, 1, n) * (rng.random(n) < 0.3)).astype(f32) for n in
            (1023, 1024, 1025, 2047, 2048, 2049, 4096, 4097)]
    for r in rows:
        r[0] = f32(2.0)
        r[-1] = f32(-0.375)        # the last entry of the row (the whole last chunk of the 2049 and 4097 rows)
    return rows, {}, ()


def case_short_tiles(rng):
    rows = [(rng.normal(0, 1, n)).astype(f32) for n in (1000, 1000, 1000, 1023, 1023, 1023, 1022, 700, 1021)]
    return rows, {}, ()


def make_case(name):
    rng = np.random.default_rng(sum(map(ord, name)))
    if name.startswith("bottom_"):
        rows, sums, wrong, expect = case_binade_bottom(name[len("bottom_"):])
        return Case(rows, expect, sums, wrong)
    if name == "signed_records":
        rows, sums, wrong = case_signed_records(rng)
        return Case(rows, ("rec_fast", "rec_cross"), sums, wrong, absent=("rec_fallback",))
    rows, sums, expect = {
        "top": case_binade_top, "crossings": case_crossings,
        "exponent_range": lambda: case_exponent_range(rng), "subnormal": lambda: case_subnormal(rng),
        "cancel_to_zero": lambda: case_cancel_to_zero(rng), "nonfinite": case_nonfinite,
        "row_lengths": lambda: case_row_lengths(rng), "short_tiles": lambda: case_short_tiles(rng),
    }[name]()
    counts = {}
    if name == "row_lengths":   # each cluster has three rows of its length: the weight-1 row and two rows of +-0
        counts = {"long_rows": 3 * 7, "chunks": 3 * (1 + 1 + 1 + 1 + 2 + 2 + 3)}
    return Case(rows, expect, sums, counts=counts)


def check_layout(lo, rows, cl):
    """each cluster's points have one weight-1 vertex, its row holds exactly the cluster's points in point order;
    returns {cluster: vertex}"""
    off, bary = lo["offset"], lo["bary"]
    assert ((bary == 1.0).sum(1) == 1).all() and ((bary == 0.0).sum(1) == 2).all()
    one = off[bary == 1.0]
    vert = {}
    for k, r in enumerate(rows):
        vs = np.unique(one[cl == k])
        assert vs.size == 1, k
        vert[k] = int(vs[0])
        assert int((off == vert[k]).sum()) == len(r), k
    return vert


def labels(x1, L):
    with np.errstate(over="ignore"):   # the non-finite case overflows on purpose
        return np.stack([x1 * f32(2.0 ** l) for l in range(L)], axis=1).astype(f32)


def assert_same(yg, yo, what):
    """finite values and infinities bit for bit, NaN as positions (x86 and the GPU make different NaN bits)"""
    ng, no = np.isnan(yg), np.isnan(yo)
    assert np.array_equal(ng, no), "%s: NaN positions differ (%d vs %d)" % (what, int(ng.sum()), int(no.sum()))
    assert_bit_exact(np.where(ng, 0, yg), np.where(no, 0, yo), what=what)


def prepare(oracle, case):
    """features, inputs, oracle lattice; asserts the layout, the sums the rows were built to reach, and that the filter
    output separates them from the value a rounded lower bound accepted"""
    f, x1, cl = interleave(case.rows)
    lo = oracle.lattice(f)
    check_layout(lo, case.rows, cl)
    for k, s in case.sums.items():
        assert seq(case.rows[k]).view(np.int32) == f32(s).view(np.int32), (k, seq(case.rows[k]), s)
    if case.wrong:
        y = oracle.filter(lo, x1[:, None])
        for k, w in case.wrong.items():
            rows = list(case.rows)
            rows[k] = w
            yw = oracle.filter(lo, interleave(rows)[1][:, None])
            assert (y[cl == k] != yw[cl == k]).all(), "row %d: the output does not see the one-ulp difference" % k
    return f, x1, cl, lo


CASES = ["bottom_plain", "bottom_fallback", "bottom_cross_a", "bottom_cross_b", "signed_records", "top", "crossings",
         "exponent_range", "subnormal", "cancel_to_zero", "nonfinite", "row_lengths", "short_tiles"]


@pytest.mark.parametrize("name", CASES)
def test_long_rows_adversarial(pkg, ctx, oracle, name):
    case = make_case(name)
    f, x1, cl, lo = prepare(oracle, case)
    lg = pkg.Lattice(ctx, f)
    assert lg.V == lo["V"]
    try:
        for L in (1, 2, 3):
            x = labels(x1, L)
            c0 = lg.debug_counters()
            yg, yo = lg.filter(x), oracle.filter(lo, x)
            c1 = lg.debug_counters()
            assert_same(yg, yo, "%s L=%d" % (name, L))
            for k, v in case.counts.items():
                assert c1[k] == v, "%s: %s = %d, not %d" % (name, k, c1[k], v)
            grown = {k: c1[k] - c0[k] for k in ("rec_fast", "rec_cross", "rec_fallback", "rec_zero")}
            for k in case.expect:
                assert grown[k] > 0, "%s L=%d: no %s (%s)" % (name, L, k, grown)
            for k in case.absent:
                assert grown[k] == 0, "%s L=%d: %s (%s)" % (name, L, k, grown)
    finally:
        oracle.lattice_free(lo)
        lg.close()


def test_short_rows_start_near_tile_ends(oracle):
    """the short-tile case really has short rows that start in the last entries of a 2048-entry tile"""
    case = make_case("short_tiles")
    f, x1, cl = interleave(case.rows)
    lo = oracle.lattice(f)
    cnt = np.bincount(lo["offset"].ravel(), minlength=lo["V"])
    start = np.concatenate([[0], np.cumsum(cnt)[:-1]])
    near = [(s, n) for s, n in zip(start, cnt) if 0 < n < 1024 and s % CH + n > CH]
    oracle.lattice_free(lo)
    assert len(near) >= 3, near


def test_one_lattice_many_calls(pkg, ctx, oracle):
    """one lattice, calls of L = 1, 3, 2, 21 with signed and unsigned inputs and filter windows: the compose kernel's
    published words and tags, and the chunk records, are reused across calls; every call must match a fresh lattice
    and the reference"""
    rng = np.random.default_rng(77)
    rows = [(rng.random(n) * (rng.random(n) < 0.5)).astype(f32) for n in (5000, 4097, 2049, 1500, 900)]
    f, x1, cl = interleave(rows)
    N = len(x1)
    lo = oracle.lattice(f)
    lg = pkg.Lattice(ctx, f)
    try:
        seen = {"rec_fast": 0, "rec_cross": 0, "rec_fallback": 0, "rec_zero": 0}
        for i, (L, signed) in enumerate([(1, False), (3, True), (2, False), (21, True), (1, True), (3, False),
                                         (2, True), (21, False), (2, True)]):
            x = rng.random((N, L)).astype(f32) * 3
            if signed:
                x -= f32(1.5)
            x[rng.random(N) < 0.3] = 0
            x[:, 0] *= (rng.random(N) < 0.9)
            c0 = lg.debug_counters()
            if i % 3 == 2:   # a window: only points [a, a + n) splatted, points [b, b + m) sliced
                a, n, b, m = 311, N // 2, 1000, N // 3
                got = lg.filter_window(x[a:a + n], L, a, b, n, m)
                fresh = pkg.Lattice(ctx, f)
                ref_fresh = fresh.filter_window(x[a:a + n], L, a, b, n, m)
                fresh.close()
                xp = np.zeros_like(x)
                xp[a:a + n] = x[a:a + n]
                want = oracle.filter(lo, xp)[b:b + m]
            else:
                got = lg.filter(x)
                fresh = pkg.Lattice(ctx, f)
                ref_fresh = fresh.filter(x)
                fresh.close()
                want = oracle.filter(lo, x)
            assert_bit_exact(got, ref_fresh, what="call %d (L=%d) vs a fresh lattice" % (i, L))
            assert_bit_exact(got, want, what="call %d (L=%d) vs the reference" % (i, L))
            c1 = lg.debug_counters()
            assert c1["long_rows"] == c0["long_rows"] and c1["chunks"] == c0["chunks"]
            for k in seen:
                seen[k] += c1[k] - c0[k]
        assert seen["rec_fast"] > 0 and seen["rec_fallback"] > 0, seen
    finally:
        oracle.lattice_free(lo)
        lg.close()
