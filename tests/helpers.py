"""Shared input builders for the parity tests."""
import numpy as np


def f32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def make_unit(rng, n, kind):
    if kind == 0:  # pure null
        x = rng.normal(0, 0.2, n)
    elif kind == 1:  # a few steps
        x = rng.normal(0, 0.2, n)
        for _ in range(int(rng.integers(1, 4))):
            a = int(rng.integers(0, n))
            b = int(rng.integers(a, n + 1))
            x[a:b] += rng.choice([-0.4, 0.15, 0.3, 1.0])
    elif kind == 2:  # tie heavy: integers
        x = np.round(rng.normal(0, 1, n))
    elif kind == 3:  # outlier spikes
        x = rng.normal(0, 0.2, n)
        i = rng.integers(0, n, max(1, n // 100))
        x[i] += 3
    else:  # three-valued
        x = rng.integers(0, 3, n).astype(float)
    return f32(x)


def pack(units):
    off = np.concatenate([[0], np.cumsum([len(u) for u in units])]).astype(np.int64)
    vals = np.concatenate(units) if len(units) else np.zeros(0)
    return vals, off


def same_result(a_counts, a_len, a_means, b_counts, b_len, b_means):
    return (np.array_equal(a_counts, b_counts) and np.array_equal(a_len, b_len)
            and np.array_equal(a_means, b_means))


def equal_arrays(got, want):
    """np.array_equal, where `want` may also be a stored reference result known by its digest (tests/refgolden.py)."""
    from refgolden import Digest
    if isinstance(want, Digest):
        return want.matches(got)
    return np.array_equal(got, want)
