"""
Edge lists for the tests of the device edge-list writer (bin3c_b200/csrc/edgefmt.cuh, edgefmt.cu): weights of every
class the two float styles treat differently, and ids of every length.
"""
import numpy as np

from test_io import WEIGHTS

INT32_EDGES = [0, 9, 10, -1, 2 ** 31 - 1, -2 ** 31, 99999, 100000, -10]


def _ulp_neighbours(x, steps=(-2, -1, 0, 1, 2)):
    """x and the doubles 1 and 2 ulps either side of it (finite, same sign)"""
    b = np.asarray(x, dtype=np.float64).view(np.int64)
    out = [(b + d).view(np.float64) for d in steps]
    out = np.concatenate(out)
    return out[np.isfinite(out)]


def weights(rng, n_random):
    """
    WEIGHTS of tests/test_io.py; n_random random 64-bit patterns (every exponent, subnormals, NaN payloads, both
    signs); n_random uniform values in (0, 1] and log-uniform over 1e-12..1e20; every power of two and every
    float('1e%d' % k) with their +-1 and +-2 ulp neighbours; exact 12-digit ties with their +-1 ulp neighbours; decade
    carries at 12 digits; the layout switch points; 17-digit shortest cases.
    """
    parts = [np.array(WEIGHTS, dtype=np.float64)]
    parts.append(np.frombuffer(rng.bytes(8 * n_random), dtype=np.float64))
    parts.append(1.0 - rng.random(n_random // 2))
    parts.append(10.0 ** rng.uniform(-12, 20, n_random - n_random // 2))
    parts.append(_ulp_neighbours(np.ldexp(1.0, np.arange(-1074, 1024))))
    parts.append(_ulp_neighbours(np.array([float('1e%d' % k) for k in range(-323, 309)])))
    # exact ties at 12 digits: 13-digit integers ending in 5 (below 2^53 all are doubles) and
    # 12-digit integers plus one half
    ties = (rng.integers(10 ** 11, 10 ** 12, 20000) * 10 + 5).astype(np.float64)
    halves = rng.integers(10 ** 11, 10 ** 12, 20000).astype(np.float64) + 0.5          # 12 digits + .5 exactly
    scaled = np.ldexp(ties, rng.integers(-40, 1, len(ties)))                          # short binary expansions
    parts.append(_ulp_neighbours(np.concatenate([ties, halves, scaled]), steps=(-1, 0, 1)))
    # rounding into a new decade at 12 digits
    carries = np.array([999999999999.5, 9999999999995.0, 99999999999.95, 0.9999999999995, 9.9999999999995e-5,
                        9.9999999999995e100, 9.9999999999995e-300, 9.99999999999951e15, 9.9999999999996e307])
    parts.append(_ulp_neighbours(carries))
    switch = np.array([1e-4, 1e-5, 9.9999e-5, 1e12, 1e13, 999999999999.0, 9999999999999.0, 1e16, 1e17,
                       9999999999999998.0, 12345678901234567.0])
    parts.append(_ulp_neighbours(switch))
    parts.append(np.array([0.30000000000000004, 5e-324, 2.2250738585072014e-308, 2.225073858507201e-308,
                           1.7976931348623157e308, 0.1 + 0.2, 1 / 3, 2 / 3, 123456789012345680.0]))
    w = np.concatenate(parts)
    return np.concatenate([w, -w])


def special_edges():
    """
    (u, v, w), a few hundred edges in a fixed order: WEIGHTS and the decade carries, layout switch points and
    17-digit cases of weights() with their ulp neighbours, some exact 12-digit ties, powers of two and of ten at the
    ends of the exponent range, all in both signs; ids cycling through INT32_EDGES
    """
    fixed = np.concatenate([
        np.array(WEIGHTS, dtype=np.float64),
        _ulp_neighbours(np.array([999999999999.5, 9999999999995.0, 0.9999999999995, 9.9999999999995e-300,
                                  9.9999999999996e307, 1e-4, 1e-5, 1e12, 1e13, 1e16, 1e17, 9999999999999998.0])),
        _ulp_neighbours(np.array([1234567890125.0, 100000000000.5, 4503599627370495.5, 1e22, 1e23]), (-1, 0, 1)),
        _ulp_neighbours(np.array([5e-324, 2.2250738585072014e-308, 1e-323, 1e-300, 0.5, 2.0 ** 52, 2.0 ** 53,
                                  1e308, 1.7976931348623157e308, 0.30000000000000004])),
    ])
    w = np.concatenate([fixed, -fixed])
    ids = np.array(INT32_EDGES, dtype=np.int32)
    k = np.arange(len(w))
    return ids[k % len(ids)], ids[(k // len(ids)) % len(ids)], w


def edges(rng, n_random):
    """(u, v, w): the weights of weights(), ids mostly below 250 k with every special int32 mixed in"""
    w = weights(rng, n_random)
    n = len(w)
    u = rng.integers(0, 250000, n).astype(np.int32)
    v = rng.integers(-2 ** 31, 2 ** 31, n, dtype=np.int64).astype(np.int32)
    k = np.arange(n) % 7 == 0
    u[k] = rng.choice(INT32_EDGES, int(k.sum()))
    v[:len(INT32_EDGES)] = INT32_EDGES
    order = rng.permutation(n)
    return u[order], v[order], w[order]
