"""How far do DECIDE 10 (randn addressed by sample position) and DECIDE 11 (blocked phase sum) move the oracle's realtime
synthesizer from canonical WORLD (sequential randn consumption, one running phase sum)?  VERDICT r1 item 2.

Reference behaviour matched: realtime_voice_conversion/yukarin_wrapper/vocoder.py:89-120 (RealtimeVocoder.decode ->
world4py _AddParameters / _Synthesis2 = WORLD synthesisrealtime.cpp).  Parity stays UNPINNED (no WORLD binary here); this test
turns the self-inflicted part of the gap into numbers (quoted in DESIGN.md section 3):
  * pulse indices and voiced/unvoiced flags: identical between the modes on voiced speech and on a real recording;
  * waveform: the PERIODIC part is bit-identical wherever the pulses are; the difference is the noise realisation only
    (the position-addressed stream is WORLD's sequential stream shifted by the first pulse's index).
"""
from pathlib import Path

import numpy as np

from oracle import pipeline as opipe
from oracle import world as W
from realtime_yukarin_b200 import synthetic

CFG = opipe.PathConfig()
# the reference's own recording tests/data/audioA.wav: its first 4 s at 24 kHz (tests/golden/make_reference_fixtures.py)
AUDIO_A = Path(__file__).resolve().parent / 'golden' / 'audioA_24k_4s.wav'


def _resynth(feat, canonical, chunk=60, skip=0):
    s = W.RealtimeSynthesizer(CFG.fs, CFG.frame_period, W.cheaptrick_fft_size(CFG.fs), 1024, canonical=canonical)
    if skip:
        s.skip_randn(skip)
    ys = []
    for a in range(0, len(feat['f0']), chunk):
        sl = slice(a, a + chunk)
        ys.append(s.decode(feat['f0'][sl].ravel().astype(np.float64), feat['sp'][sl], feat['ap'][sl]))
    idx, tm, vuv = s.pulses()
    return np.concatenate(ys), idx, vuv


def _compare(x, label):
    feat = opipe.extract_features(x, CFG)
    y0, i0, v0 = _resynth(feat, 0)
    out = {}
    for mode, name in ((W.RealtimeSynthesizer.CANON_PHASE, 'running-sum phase'), (W.RealtimeSynthesizer.CANON_RANDN, 'sequential randn'),
                       (3, 'both (canonical WORLD)')):
        y, i, v = _resynth(feat, mode)
        assert len(y) == len(y0)
        same_pulses = len(i) == len(i0) and np.array_equal(i, i0) and np.array_equal(v, v0)
        moved = int((i != i0).sum()) if len(i) == len(i0) else -1
        rmse = float(np.sqrt(np.mean((y - y0) ** 2)))
        rms = float(np.sqrt(np.mean(y0 ** 2)))
        out[mode] = (same_pulses, moved, rmse, rms, len(i0))
        print(f'{label}: {name}: pulses {len(i0)}, identical {same_pulses} (moved {moved}), sample RMSE vs default mode {rmse:.3e} (signal RMS {rms:.3e})')
    # DECIDE 10 is a pure re-indexing: WORLD's sequential stream advanced by the first pulse's sample index IS the position-addressed
    # stream (noise_size = next index - index, never clamped for f0 >= 24 Hz), so the two waveforms agree to rounding
    q0 = max(int(i0[0]), 0) if len(i0) else 0
    ys, _, _ = _resynth(feat, W.RealtimeSynthesizer.CANON_RANDN, skip=q0)
    shift_rmse = float(np.sqrt(np.mean((ys - y0) ** 2)))
    print(f'{label}: sequential randn advanced by the first pulse index ({q0}): sample RMSE vs default mode {shift_rmse:.3e}')
    out['shifted'] = shift_rmse
    return out


def test_decide_10_11_on_synthetic_speech():
    x = synthetic.synthetic_speech(3.0, stream=5)
    r = _compare(x, 'synthetic speech 3 s')
    # DECIDE 11: the blocked sum may move a pulse by one sample only where the phase sits within rounding of a 2 pi multiple
    # (unvoiced 500 Hz default at 24 kHz); report, and require that voiced pulses are untouched
    same, moved, rmse, rms, n = r[W.RealtimeSynthesizer.CANON_PHASE]
    assert moved >= 0 and moved <= max(2, n // 50), (moved, n)
    # DECIDE 10 alone never touches pulse placement
    assert r[W.RealtimeSynthesizer.CANON_RANDN][0]
    # the waveform difference is a noise-realisation difference: bounded by the aperiodic energy, far below the signal
    assert r[3][2] < 0.5 * r[3][3]
    assert r['shifted'] < 1e-12 * max(1.0, r[3][3])


def test_decide_10_11_on_the_reference_recording():
    from realtime_yukarin_b200 import wave_io
    import scipy.signal
    data, fs = wave_io.read_wav(AUDIO_A)
    x = data.astype(np.float64)
    if x.ndim > 1:
        x = x.mean(axis=1)
    x = scipy.signal.resample_poly(x, 24000, fs).astype(np.float32)[:24000 * 4]
    r = _compare(x, 'audioA.wav @ 24 kHz, 4 s')
    assert r[W.RealtimeSynthesizer.CANON_RANDN][0]
    same, moved, rmse, rms, n = r[W.RealtimeSynthesizer.CANON_PHASE]
    assert moved >= 0 and moved <= max(2, n // 50), (moved, n)
    assert r['shifted'] < 1e-12 * max(1.0, rms)
    # analysis -> synthesis on the real recording: the resynthesis is a sane waveform (finite, comparable level)
    feat = opipe.extract_features(x, CFG)
    y, _, _ = _resynth(feat, 0)
    assert np.isfinite(y).all()
    assert 0.2 < np.sqrt(np.mean(y ** 2)) / np.sqrt(np.mean(x[:len(y)].astype(np.float64) ** 2)) < 5.0
