"""CPU model of the exact ordered scan of long splat rows (csrc/filter.cu: split_ulps, row_sum_exact /
thread_composite, scan_combine, composite_append, apply_composite), restated in numpy float32 and Python integers,
against the sequential float32 sum it must reproduce.

A composite maps a running sum s = m*u of binade E (u its ulp, m in [2^23, 2^24)) to (m + a_parity(m))*u, and is only
applied when the safe range check m + lo >= 2^23 and m + hi < 2^24 passes.  The rule the kernels use must never accept
a result that differs from the sequential sum; the rule they used before (lo over the ROUNDED prefixes, fraction read
as q - floor(q)) accepts wrong results, which the last tests pin down."""
import itertools
import math

import numpy as np

f32 = np.float32
MLO, MHI = 1 << 23, 1 << 24


def split_new(q):
    """split_ulps: (floor(q), fraction > 1/2, fraction == 1/2), read from floor(2q)"""
    q = f32(q)
    if not abs(q) < f32(MHI):
        return (MHI if q > 0 else -MHI), False, False
    q2 = q * f32(2)
    i2 = math.floor(float(q2))
    n = i2 >> 1
    if i2 & 1:
        tie = f32(i2) == q2
        return n, not tie, tie
    return n, False, False


def split_old(q):
    """the fraction as the kernels read it before: fr = RN(q - floor(q))"""
    q = f32(q)
    if not abs(q) < f32(MHI):
        return (MHI if q > 0 else -MHI), False, False
    n = math.floor(float(q))
    fr = q - f32(n)
    return n, bool(fr > f32(0.5)), bool(fr == f32(0.5))


def combine(l, r):
    """scan_combine: apply l, then r"""
    return (l[0] + (r[1] if l[0] & 1 else r[0]), l[1] + (r[0] if l[1] & 1 else r[1]))


def thread_composite(qs, new=True):
    """(a0, a1, lo0, hi0, lo1, hi1) of the entries q (in ulps) for an even / odd start"""
    split = split_new if new else split_old
    a0 = a1 = lo0 = hi0 = lo1 = hi1 = 0
    for q in qs:
        n, up, tie = split(q)
        if new:  # floor of the exact prefix behind the entry
            lo0, lo1 = min(lo0, a0 + n), min(lo1, a1 + n)
        if not tie:
            a0, a1 = a0 + n + up, a1 + n + up
        else:
            a0, a1 = combine((a0, a1), (n + (n & 1), n + ((n + 1) & 1)))
        hi0, hi1 = max(hi0, a0), max(hi1, a1)
        if not new:  # the rounded prefix behind the entry
            lo0, lo1 = min(lo0, a0), min(lo1, a1)
    return a0, a1, lo0, hi0, lo1, hi1


def composite_append(R, C):
    """R followed by C"""
    a0, a1, lo0, hi0, lo1, hi1 = R
    return (a0 + (C[1] if a0 & 1 else C[0]), a1 + (C[0] if a1 & 1 else C[1]),
            min(lo0, a0 + (C[4] if a0 & 1 else C[2])), max(hi0, a0 + (C[5] if a0 & 1 else C[3])),
            min(lo1, a1 + (C[2] if a1 & 1 else C[4])), max(hi1, a1 + (C[3] if a1 & 1 else C[5])))


def apply_composite(s, E, C):
    """the new running sum, or None when the start is outside binade E or the safe range"""
    s = f32(s)
    if not (s > 0 and np.frexp(s)[1] - 1 == E):
        return None
    u = f32(2.0 ** (E - 23))
    m = int(s / u)
    a, lo, hi = (C[1], C[4], C[5]) if m & 1 else (C[0], C[2], C[3])
    if not (m + lo >= MLO and m + hi < MHI):
        return None
    return f32(f32(m + a) * u)


def sequential(s, cs):
    s = f32(s)
    for c in cs:
        s = f32(s + f32(c))
    return s


def model(s, E, qs, new=True, split_at=None):
    """apply one chunk's composite (optionally built as two thread composites appended) to s"""
    if split_at is None:
        C = thread_composite(qs, new)
    else:
        C = composite_append(thread_composite(qs[:split_at], new), thread_composite(qs[split_at:], new))
    return apply_composite(s, E, C)


E0 = 1                          # binade [2, 4): u = 2^-22
U0 = 2.0 ** (E0 - 23)
STARTS = [MLO + k for k in range(5)] + [MHI - k for k in range(1, 5)]   # m: both parities at both ends
QGRID = [k / 8 for k in range(-48, 49)]                                    # q on a 1/8 grid in [-6, 6]


def sweep(new):
    """(accepted, wrong) over the exhaustive grid: one or two entries, whole or as two appended thread composites"""
    acc = bad = 0
    for m in STARTS:
        s = f32(m * U0)
        seqs = [[q] for q in QGRID] + [list(p) for p in itertools.product(QGRID, QGRID)]
        for qs in seqs:
            want = sequential(s, [f32(q * U0) for q in qs])
            for split_at in ((None,) if len(qs) == 1 else (None, 1)):
                got = model(s, E0, qs, new, split_at)
                if got is not None:
                    acc += 1
                    bad += int(got.view(np.int32) != want.view(np.int32))
    return acc, bad


def test_exhaustive_grid_never_accepts_a_wrong_sum():
    acc, bad = sweep(new=True)
    assert bad == 0, "%d accepted results differ from the sequential sum" % bad
    assert acc > 20000, acc     # the check is not vacuous: most of the grid stays inside the binade


def test_random_signed_sequences():
    rng = np.random.default_rng(7)
    acc = 0
    for _ in range(3000):
        E = int(rng.integers(-100, 101))
        u = 2.0 ** (E - 23)
        m = int(rng.choice([MLO + int(rng.integers(0, 64)), MHI - 1 - int(rng.integers(0, 64)), int(rng.integers(MLO, MHI))]))
        s = f32(m * u)
        n = int(rng.integers(1, 40))
        kind = rng.integers(0, 4, n)
        q = np.where(kind == 0, rng.integers(-24, 25, n) / 8.0,                # grid values: ties and exact integers
            np.where(kind == 1, rng.normal(0, 3, n),                           # arbitrary fractions of either sign
            np.where(kind == 2, -0.5 + rng.integers(-2, 3, n) * 2.0 ** -25,    # next to -1/2
                     rng.normal(0, 1, n) * 2.0 ** -30)))                       # far below an ulp
        cs = [f32(v * u) for v in q]
        qs = [f32(c / f32(u)) for c in cs]
        want = sequential(s, cs)
        for split_at in (None, n // 2):
            got = model(s, E, qs, True, split_at)
            if got is not None:
                acc += 1
                assert got.view(np.int32) == want.view(np.int32), (E, m, q.tolist(), split_at, got, want)
    assert acc > 1000, acc


def test_binade_bottom_counterexample():
    """s = 2 and c = -0.375 * 2^-22: the exact sum 2 - 0.75 * 2^-23 lies below 2, where fp32 is twice as fine, and
    rounds to 1.9999999.  On the grid of [2, 4) it rounds to 2, which the old lower bound accepted."""
    s, c = f32(2.0), f32(-0.375 * 2.0 ** -22)
    assert sequential(s, [c]) == f32(1.9999999)
    q = [c / f32(U0)]
    assert model(s, E0, q, new=False) == f32(2.0)      # the old rule: accepted and wrong
    assert model(s, E0, q, new=True) is None           # the floor bound sends it to real additions
    s2, c2 = f32(2.0 + 2.0 ** -22), f32(-1.375 * 2.0 ** -22)
    assert model(s2, E0, [c2 / f32(U0)], new=False) == f32(2.0) != sequential(s2, [c2])
    assert model(s2, E0, [c2 / f32(U0)], new=True) is None
    acc, bad = sweep(new=False)
    assert bad > 0


def test_fraction_just_above_one_half():
    """q = -1/2 + 2^-25 from an odd m: q - floor(q) = 1/2 + 2^-25 rounds to 1/2 in fp32 and read as a tie, which rounds
    down to the even m - 1; the sequential sum stays at m.  The fraction read from floor(2q) is exact."""
    m = MLO + 1
    s = f32(m * U0)
    q = f32(-0.5 + 2.0 ** -25)
    c = f32(q * f32(U0))
    assert sequential(s, [c]) == s
    assert split_old(q) == (-1, False, True)
    assert split_new(q) == (-1, True, False)
    assert model(s, E0, [q], new=False) == f32((m - 1) * U0)
    assert model(s, E0, [q], new=True) == s
