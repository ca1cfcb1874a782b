"""Harvest restatement (oracle/world_oracle.c, Harvest section; PARITY UNPINNED like the rest of the oracle): pinned against an
independent numpy / scipy writing of decimate() (scipy.signal.cheby1 + lfilter), against the f0 ground truth of synthetic harmonic
signals, against DIO + StoneMask on synthetic speech, and frozen as a golden fixture (tests/golden/harvest_f0.npz,
tests/golden/make_harvest_fixture.py)."""
from pathlib import Path

import numpy as np
import pytest
from scipy import signal

from oracle import world as ow
from realtime_yukarin_b200 import synthetic

GOLDEN = Path(__file__).resolve().parent / 'golden'


def _decimate_numpy(x, r):
    """matlabfunctions.cpp decimate() written with scipy: reflect 9 samples, cheby1(3, 0.05 dB, 0.8 / r) forwards and backwards."""
    b, a = signal.cheby1(3, 0.05, 0.8 / r)
    nf = 9
    head = 2 * x[0] - x[nf:0:-1]
    tail = 2 * x[-1] - x[-2:-nf - 2:-1]
    t = np.concatenate([head, x, tail])
    t = signal.lfilter(b, a, t)[::-1]
    t = signal.lfilter(b, a, t)[::-1]
    nout = (len(x) - 1) // r + 1
    nbeg = r - r * nout + len(x)
    idx = np.arange(nbeg, len(x) + nf, r) + nf - 1
    return t[idx][:nout]


@pytest.mark.parametrize('r', [2, 3, 4, 6, 11, 12])
def test_decimate_matches_scipy_transcription(r):
    rng = np.random.default_rng(r)
    x = rng.standard_normal(2000) + np.sin(np.arange(2000) * 0.01)
    got = ow.decimate(x, r)
    ref = _decimate_numpy(x, r)
    assert got.shape == ref.shape
    assert np.allclose(got, ref, rtol=0, atol=1e-11)


def _harmonic(f0_track, fs, seed=0):
    """Band-limited pulse-like harmonic signal following f0_track (Hz per sample) plus a little noise."""
    rng = np.random.default_rng(seed)
    phase = 2 * np.pi * np.cumsum(f0_track) / fs
    x = np.zeros_like(phase)
    for h in range(1, 9):
        x += np.where(h * f0_track < 0.45 * fs, np.cos(h * phase + 0.3 * h) / h, 0.0)
    return 0.2 * x + 1e-3 * rng.standard_normal(len(x))


@pytest.mark.parametrize('fs', [24000, 16000])
def test_harvest_tracks_a_known_f0_contour(fs):
    n = int(1.2 * fs)
    t = np.arange(n) / fs
    f0_true = 140.0 + 40.0 * np.sin(2 * np.pi * 1.5 * t)
    x = _harmonic(f0_true, fs)
    x[: int(0.15 * fs)] = 0.0                       # leading silence
    f0, tt = ow.harvest(x, fs)
    assert len(f0) == int(1000.0 * n / fs / 5.0) + 1
    assert np.allclose(tt, np.arange(len(f0)) * 0.005)
    assert np.all(f0[tt < 0.10] == 0.0)             # silence stays unvoiced
    inner = (tt > 0.25) & (tt < 1.1)
    assert np.all(f0[inner] > 0)
    truth = np.interp(tt[inner], t, f0_true)
    assert np.max(np.abs(f0[inner] - truth) / truth) < 0.02
    assert np.all((f0 == 0) | ((f0 >= 71.0) & (f0 <= 800.0)))


def test_harvest_agrees_with_dio_stonemask_on_synthetic_speech():
    x = synthetic.synthetic_speech(2.0, stream=1).astype(np.float64)
    f0h, t = ow.harvest(x, 24000)
    f0d, td = ow.dio(x, 24000)
    f0d = ow.stonemask(x, 24000, td, f0d)
    both = (f0h > 0) & (f0d > 0)
    assert both.sum() > 200
    rel = np.abs(f0h[both] - f0d[both]) / f0d[both]
    assert np.median(rel) < 0.01
    assert (f0h > 0).sum() >= 0.9 * (f0d > 0).sum()


def test_harvest_intermediates_are_consistent():
    x = synthetic.synthetic_speech(0.6, stream=4)[:7200].astype(np.float64)
    f0, t, d = ow.harvest(x, 24000, debug=True)
    ch, nf1, ylen, fft_size, maxc, ratio = ow.harvest_geometry(len(x), 24000)
    assert (ch, nf1, ylen, fft_size, maxc, ratio) == (152, 301, 2400, 4096, 105, 3)
    assert abs(d['y'].mean()) < 1e-12
    assert d['nc'] % 7 == 0 and 0 < d['nc'] <= maxc
    assert np.all(d['cand'][:, d['nc']:] == 0)
    assert np.all((d['score'] == 0) == (d['cand'] == 0))
    # the 5 ms output is the 1 ms contour sub-sampled
    assert np.array_equal(f0, d['basic'][np.minimum(nf1 - 1, np.arange(len(f0)) * 5)])
    # all-zero input: nothing voiced, no NaN
    f0z, _ = ow.harvest(np.zeros(7200), 24000)
    assert np.all(f0z == 0)


def test_harvest_golden_fixture():
    g = np.load(GOLDEN / 'harvest_f0.npz')
    x = synthetic.synthetic_speech(float(g['seconds']), stream=int(g['stream'])).astype(np.float64)
    f0, _ = ow.harvest(x, 24000)
    assert np.array_equal(f0 != 0, g['f0'] != 0)
    assert np.allclose(f0, g['f0'], rtol=1e-9, atol=0)


# the reference's own recording tests/data/audioA.wav: its first 4 s at 24 kHz (tests/golden/make_reference_fixtures.py)
AUDIO_A = Path(__file__).resolve().parent / 'golden' / 'audioA_24k_4s.wav'


def test_harvest_on_the_reference_recording():
    """Real speech (the reference's tests/data/audioA.wav at 24 kHz, 4 s): Harvest and DIO + StoneMask -- two different published
    extractors restated independently of each other -- agree on the pitch where both are voiced, Harvest's contour is the smoother
    one and covers more of the voiced speech, and every value is inside [f0_floor, f0_ceil]."""
    from realtime_yukarin_b200 import wave_io
    data, fs = wave_io.read_wav(AUDIO_A)
    x = data.astype(np.float64)
    if x.ndim > 1:
        x = x.mean(axis=1)
    x = signal.resample_poly(x, 24000, fs)[:24000 * 4]
    f0h, t = ow.harvest(x, 24000)
    f0d, td = ow.dio(x, 24000)
    f0d = ow.stonemask(x, 24000, td, f0d)
    both = (f0h > 0) & (f0d > 0)
    rel = np.abs(f0h[both] - f0d[both]) / f0d[both]
    print(f'audioA: harvest voiced {int((f0h > 0).sum())}, dio voiced {int((f0d > 0).sum())}, both {int(both.sum())}; '
          f'median |rel diff| {np.median(rel):.4f}, 90th percentile {np.percentile(rel, 90):.4f}')
    assert both.sum() > 150
    assert np.median(rel) < 0.01 and np.percentile(rel, 90) < 0.05
    assert (f0h > 0).sum() >= 0.9 * (f0d > 0).sum()
    assert np.all((f0h == 0) | ((f0h >= 71.0) & (f0h <= 800.0)))
    d2 = lambda f: np.abs(np.diff(f[both], 2)).mean()          # roughness of the contour on the common frames
    assert d2(f0h) <= d2(f0d)


def test_independent_numpy_writing_of_the_harvest_array_stages():
    """A second writing of Harvest's array stages in numpy / scipy (tests/independent_world.py: scipy's cheby1 + lfilter decimation,
    numpy FFT filter bank, vectorised zero-crossing trains, numpy rfft refinement, lfilter smoothing) against the C restatement's
    intermediate arrays (the sequential contour tracking has its own second writing below)."""
    from . import independent_world as iw
    x = synthetic.synthetic_speech(0.6, stream=4)[:7200].astype(np.float64)
    f0, t, d = ow.harvest(x, 24000, debug=True)
    s = iw.harvest_stages_np(x, 24000)
    assert np.allclose(s['y'], d['y'], rtol=0, atol=1e-11)
    assert np.array_equal(s['raw'] > 0, d['raw'] > 0)
    assert np.allclose(s['raw'], d['raw'], rtol=1e-8, atol=0)
    assert s['nc'] == d['nc']
    assert np.array_equal(s['cand'] > 0, d['cand'] > 0)
    assert np.allclose(s['cand'], d['cand'], rtol=1e-7, atol=0)
    assert np.allclose(s['score'], d['score'], rtol=1e-5, atol=0)
    assert np.allclose(s['smooth'](d['best']), d['basic'], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize('seconds,stream', [(0.6, 4), (2.0, 1), (1.5, 2)])
def test_independent_writing_of_the_contour_tracking(seconds, stream):
    """FixF0Contour (SearchF0Base, FixStep1..4) written a second time in numpy (tests/independent_world.py) on the C restatement's pruned
    candidates: the tracked contour must come out identical (the values are copies of candidates or linear bridges)."""
    from . import independent_world as iw
    x = synthetic.synthetic_speech(seconds, stream=stream).astype(np.float64)
    f0, t, d = ow.harvest(x, 24000, debug=True)
    best = iw.harvest_fix_contour_np(d['cand'], d['score'], d['nc'])
    assert np.array_equal(best > 0, d['best'] > 0)
    assert np.allclose(best, d['best'], rtol=1e-12, atol=0)
