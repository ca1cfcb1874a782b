"""D4C aperiodicity and StoneMask on the GPU against the CPU oracle.

k_d4c takes each band's pa / pb (sum of the fft/2 - boundary smallest band powers / of all of them) from a radix selection instead
of a sort, and packs two band transforms into one complex FFT: sums and transforms round differently from the oracle's, so ap is
held to the analysis tolerance (1e-4 relative, 1e-6 absolute), on the same f0 as the oracle.  The inputs include unvoiced frames,
voiced frames that the LoveTrain test rejects, and voiced frames whose LoveTrain ratio lies within 0.01 of the 0.85 threshold.
"""
from pathlib import Path

import numpy as np
import pytest

from oracle import pipeline as opipe
from oracle import world as oworld
from realtime_yukarin_b200 import synthetic
from realtime_yukarin_b200.wave_io import read_wav

pytestmark = pytest.mark.gpu

CFG = opipe.PathConfig()
AUDIO_A = Path(__file__).resolve().parent / 'golden' / 'audioA_24k_4s.wav'


def _noisy_speech():
    """1 s of synthetic speech plus > 4.5 kHz noise rising from silence: the LoveTrain ratio sweeps down through 0.85."""
    x = synthetic.synthetic_speech(1.0, stream=7).astype(np.float64)
    rng = np.random.default_rng(5)
    spec = np.fft.rfft(rng.standard_normal(len(x)))
    spec[np.fft.rfftfreq(len(x), 1.0 / CFG.fs) < 4500.0] = 0.0
    hp = np.fft.irfft(spec, len(x))
    return (x + 0.06 * np.linspace(0.0, 1.0, len(x)) * hp / np.std(hp)).astype(np.float32)


def _cases():
    xs = {f'speech_{s}s': synthetic.synthetic_speech(s, stream=i) for i, s in enumerate((0.1, 0.3, 1.0))}
    w, fs = read_wav(AUDIO_A)
    assert fs == CFG.fs
    xs['audioA_4s'] = np.asarray(w, np.float32)
    xs['speech_1s_rising_noise'] = _noisy_speech()
    return xs


def test_d4c_matches_oracle(engine):
    near, rejected, unvoiced = 0, 0, 0
    for name, x in _cases().items():
        ref = opipe.extract_features(x, CFG)
        f0 = ref['f0'].ravel().astype(np.float64)
        got = engine.world_analyze(x, CFG.fs, CFG.frame_period, CFG.f0_floor, CFG.f0_ceil, CFG.fft_length, CFG.order, CFG.alpha,
                                   f0=f0)
        assert np.allclose(got['ap'], ref['ap'], rtol=1e-4, atol=1e-6), (name, np.abs(got['ap'] - ref['ap']).max())
        t = np.arange(len(f0)) * CFG.frame_period / 1000.0
        _, ap0 = oworld.d4c(x.astype(np.float64), CFG.fs, t, f0, debug=True)
        v = f0 > 0
        near += int(np.sum(v & (np.abs(ap0 - 0.85) < 0.01)))
        rejected += int(np.sum(v & ~(ap0 > 0.85)))
        unvoiced += int(np.sum(~v))
    assert near > 0 and rejected > 0 and unvoiced > 0, (near, rejected, unvoiced)


def test_stonemask_shared_memory_guard(engine):
    """StoneMask's shared memory is sized from f0_floor.  An estimate below it whose FFT would not fit (here 45 Hz: 4096 points,
    against 2048 reserved for 71 Hz) comes back unrefined; the same estimates with a 40 Hz floor are refined like the oracle."""
    x = synthetic.synthetic_speech(1.0, stream=3)
    f0_ref, t = oworld.dio(x.astype(np.float64), CFG.fs, CFG.frame_period, CFG.f0_floor, CFG.f0_ceil)
    f0_in = f0_ref.copy()
    low = np.flatnonzero(f0_in > 0)[::5]
    f0_in[low] = 45.0
    want = oworld.stonemask(x.astype(np.float64), CFG.fs, t, f0_in)
    got71 = engine.debug_stonemask(x, CFG.fs, CFG.frame_period, 71.0, f0_in)
    got40 = engine.debug_stonemask(x, CFG.fs, CFG.frame_period, 40.0, f0_in)
    rest = np.setdiff1d(np.arange(len(f0_in)), low)
    assert np.array_equal(got71[low], f0_in[low])
    assert np.allclose(got71[rest], want[rest], rtol=1e-9, atol=0)
    assert np.allclose(got40, want, rtol=1e-9, atol=0)
