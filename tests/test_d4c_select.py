"""k_d4c's coarse-aperiodicity sums without a sort (world_analysis.cu, d4c_select_sums), transcribed to numpy and checked against
the sort + cumulative sums that WORLD's D4C uses: the sum of the m smallest of n non-negative band powers and the sum of all n."""
import numpy as np
import pytest


def select_sums(p, m):
    """8-bit radix select over the IEEE-754 bit patterns (non-negative doubles order like their uint64 patterns) for the m-th
    smallest value t, then sum(v < t) + (m - #{v < t}) * t.  Digit by digit, as the kernel does it."""
    keys = np.ascontiguousarray(p, dtype=np.float64).view(np.uint64)
    prefix, rank = 0, m - 1
    for k in range(8):
        shift = 56 - 8 * k
        cand = keys if k == 0 else keys[(keys >> np.uint64(shift + 8)) == np.uint64(prefix >> (shift + 8))]
        hist = np.bincount(((cand >> np.uint64(shift)) & np.uint64(255)).astype(np.int64), minlength=256)
        cum = np.cumsum(hist)
        digit = int(np.searchsorted(cum, rank, side='right'))
        below = int(cum[digit - 1]) if digit > 0 else 0
        prefix |= digit << shift
        rank -= below
    t = np.array([prefix], dtype=np.uint64).view(np.float64)[0]
    lt = keys < np.uint64(prefix)
    return float(p[lt].sum() + (m - int(lt.sum())) * t), float(p.sum()), t


def d4c_counts(fs=24000):
    fft = 2 ** (1 + int(np.log(4.0 * fs / 47.0 + 1) / np.log(2.0)))
    wl = int(3000.0 * fft / fs) * 2 + 1
    boundary = int(fft * 8.0 / wl + 0.5)
    return fft // 2 + 1, fft // 2 - boundary      # hb band powers, pa sums the smallest fft/2 - boundary


def _spectra():
    rng = np.random.default_rng(11)
    for fs in (16000, 24000, 48000):
        n, m = d4c_counts(fs)
        yield f'lognormal_{fs}', rng.lognormal(0.0, 6.0, n), m
        yield f'squared_{fs}', np.abs(rng.standard_normal(n) + 1j * rng.standard_normal(n)) ** 2 * 1e-9, m
    n, m = d4c_counts()
    v = rng.integers(0, 5, n).astype(np.float64) * 0.25                  # heavy exact ties, zeros included
    yield 'ties', v, m
    yield 'all_equal', np.full(n, 3.0e-7), m
    yield 'zeros', np.zeros(n), m
    v = rng.random(n)
    v[-(n - m):] = np.sort(v)[m - 1]                                     # ties straddle rank m, at the tail (the padding edge)
    yield 'ties_at_rank', v, m
    v = rng.random(n)
    v[-1] = 1e300; v[-2] = 5e-324                                          # extremes of the double range in the last slots
    yield 'extremes_at_tail', v, m
    yield 'rank_1', rng.random(n), 1
    yield 'rank_n', rng.random(n), n


@pytest.mark.parametrize('name,p,m', list(_spectra()), ids=lambda v: v if isinstance(v, str) else '')
def test_select_sums_match_sort_and_cumsum(name, p, m):
    s = np.sort(p)
    want_m, want_all = np.cumsum(s)[m - 1], np.cumsum(s)[-1]
    got_m, got_all, t = select_sums(p, m)
    assert t == s[m - 1]
    assert got_m == pytest.approx(want_m, rel=1e-12, abs=0)
    assert got_all == pytest.approx(want_all, rel=1e-12, abs=0)


def test_counts_at_24k():
    assert d4c_counts(24000) == (1025, 992)
