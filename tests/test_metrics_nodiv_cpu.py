"""The division-free delta-counts of metrics_sum_fast_kernel (metric_terms_nodiv, t3d_metrics_internal.cuh), restated in
numpy: for a >= b > 0 the kernel counts  a / b < T  by the sign bit of  fma(2^-24, b, fma(-T, b, a)).  Each FMA is
emulated as its exact result in float64 (every product and sum below needs at most 33 bits) followed by one rounding
to float32, subnormals and the sign of zero included.  The counts must equal numpy's (thresh < T, thresh the correctly
rounded fp32 quotient, utils/metrics.py:51-54) wherever the kernel takes that path: g and the scaled prediction in
[2^-120, 2^126).  Below 2^-120 the first FMA's result falls under the fp32 subnormal spacing and is rounded, which is
why the kernel sends smaller values to the literal formula.  The pair generator is shared with
test_metrics_edges_gpu.py, which puts the same pairs through every sum kernel."""
import numpy as np

THRESHOLDS = (1.25, 1.5625, 1.953125)       # 1.25, 1.25^2, 1.25^3: all exact in fp32, multiples of 2^-6
F32 = np.float32


def _bits_add(x, k):
    """x (positive fp32) moved by k ulp (through the bit pattern: crosses exponent boundaries)."""
    return (np.asarray(x, F32).view(np.uint32).astype(np.int64) + k).astype(np.uint32).view(F32)


def random_in_band(rng, lo_exp, hi_exp, n):
    """n positive fp32 values with an exponent uniform in [lo_exp, hi_exp) and a uniform random mantissa."""
    e = rng.integers(lo_exp, hi_exp, n)
    m = rng.integers(0, 1 << 23, n)
    return ((e + 127).astype(np.uint32) << 23 | m.astype(np.uint32)).view(F32)


def near_threshold_pairs(rng, lo_exp, hi_exp, n, T):
    """(a, b), a >= b > 0: for each of n random b (exponent in [lo_exp, hi_exp)), a = fl32(T b) + k ulp for
    k in -3..3, and the fp32 nearest to (T - 2^-24) b + k ulp for k in -1..1.  The quotient a / b can never equal the
    midpoint T - 2^-24 below T (2^24 T - 1 is odd and wider than 24 bits), so those last three are the pairs closest to
    a tie that fp32 admits.  Every a is finite as long as hi_exp <= 127."""
    b = random_in_band(rng, lo_exp, hi_exp, n)
    at = (np.float64(T) * b.astype(np.float64)).astype(F32)
    am = ((np.float64(T) - 2.0 ** -24) * b.astype(np.float64)).astype(F32)
    a = np.concatenate([_bits_add(at, k) for k in range(-3, 4)] + [_bits_add(am, k) for k in (-1, 0, 1)])
    return a, np.tile(b, 10)


def nodiv_counts(a, b, T):
    """metric_terms_nodiv's count of a / b < T: the sign bit of fma(2^-24, b, fma(-T, b, a))."""
    r = (a.astype(np.float64) - T * b.astype(np.float64)).astype(F32)             # fma(-T, b, a): exact, one rounding
    s = (r.astype(np.float64) + 2.0 ** -24 * b.astype(np.float64)).astype(F32)  # fma(2^-24, b, r)
    return np.signbit(s)


def numpy_counts(a, b, T):
    with np.errstate(all="ignore"):
        return np.maximum(a / b, b / a) < F32(T)


def test_agrees_with_numpy_from_2_to_the_minus_120():
    rng = np.random.default_rng(0)
    for T in THRESHOLDS:
        a, b = near_threshold_pairs(rng, -120, 126, 200_000, T)
        want = numpy_counts(a, b, T)
        assert 0.1 < want.mean() < 0.9                      # the pairs straddle the threshold
        bad = np.flatnonzero(nodiv_counts(a, b, T) != want)
        assert bad.size == 0, (T, [(hex(a[i:i + 1].view(np.uint32)[0]), hex(b[i:i + 1].view(np.uint32)[0])) for i in bad[:5]])


def test_disagrees_below_2_to_the_minus_120():
    rng = np.random.default_rng(1)
    for T in THRESHOLDS:
        a, b = near_threshold_pairs(rng, -126, -120, 100_000, T)
        assert (nodiv_counts(a, b, T) != numpy_counts(a, b, T)).any(), T
    # one mismatch per threshold, both directions (a = larger, b = smaller value)
    for T, a, b, counted in ((1.25, 0x017a11e2, 0x01480e4f, False), (1.5625, 0x00f377bd, 0x009bd1c1, False),
                             (1.953125, 0x017b1aed, 0x010090dc, True)):
        a, b = np.array([a], np.uint32).view(F32), np.array([b], np.uint32).view(F32)
        assert numpy_counts(a, b, T)[0] == counted and nodiv_counts(a, b, T)[0] != counted, T
