"""CPU model checks (no GPU) of the arithmetic claim behind observe() in csrc/unary_obs.cuh.

The reference computes the inverse depth as `float invzc = 1.0 / z` (Tracking.cc:1821): a double division rounded to
float.  observe() uses the correctly rounded float reciprocal __frcp_rn instead, which is bit-identical only if the
double rounding RN32(RN64(1/z)) never differs from RN32(1/z).  numpy's float32 division is IEEE single division,
i.e. RN32(1/z) exactly, so the claim is checked here for every float in the binades where it can go wrong."""
import numpy as np
import pytest

MANT = np.arange(1 << 23, dtype=np.uint32)


def binade(field, sign=0):
    """all 2^23 floats with the given exponent field (0: the subnormals and +-0)"""
    return ((np.uint32(sign) << np.uint32(31)) | (np.uint32(field) << np.uint32(23)) | MANT).view(np.float32)


def assert_rcp_double_rounding(z):
    with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
        twice = (1.0 / z.astype(np.float64)).astype(np.float32)   # the reference: RN32(RN64(1/z))
        once = np.float32(1) / z                                    # IEEE single division: RN32(1/z)
    nan_t, nan_o = np.isnan(twice), np.isnan(once)
    assert np.array_equal(nan_t, nan_o)
    bad = np.nonzero(~nan_t & (twice.view(np.int32) != once.view(np.int32)))[0]
    assert bad.size == 0, "RN32(RN64(1/z)) != RN32(1/z) for %d floats, first z = %r (bits %#x)" % (
        bad.size, float(z[bad[0]]), int(z.view(np.uint32)[bad[0]]))


@pytest.mark.parametrize("sign", [0, 1])
def test_reciprocal_double_rounding_normal_binade(sign):
    """Exhaustive over [1, 2) (and (-2, -1]).  Scaling z by 2^k scales 1/z by 2^-k exactly in both formats as long as z
    and 1/z stay normal floats, and rounding commutes with that scaling, so this one binade stands for every binade
    whose reciprocal is a normal float (exponent fields 1..252); the edge binades are checked separately below."""
    assert_rcp_double_rounding(binade(127, sign))


@pytest.mark.parametrize("sign", [0, 1])
@pytest.mark.parametrize("field", [0, 1, 252, 253, 254])
def test_reciprocal_double_rounding_edge_binades(field, sign):
    """Exhaustive over the binades where z is subnormal (0: 1/z large or overflowing), 1/z is subnormal (253, 254) or
    their neighbours (1, 252): there the scaling argument does not hold and the rounding grid changes."""
    assert_rcp_double_rounding(binade(field, sign))


def test_reciprocal_double_rounding_specials():
    z = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan], np.float32)
    assert_rcp_double_rounding(z)
    with np.errstate(divide="ignore"):
        r = (1.0 / z[:4].astype(np.float64)).astype(np.float32)
    assert r.view(np.uint32).tolist() == np.array([np.inf, -np.inf, 0.0, -0.0], np.float32).view(np.uint32).tolist()


def test_edge_binades_reach_subnormal_and_overflow():
    """the edge binades above do contain the cases they are chosen for"""
    with np.errstate(divide="ignore", over="ignore"):
        r0 = np.float32(1) / binade(0)[1:]
        r254 = np.float32(1) / binade(254)
    assert np.isinf(r0).any() and np.isfinite(r0).any()
    assert (r254 < np.finfo(np.float32).tiny).all() and (r254 > 0).all()
