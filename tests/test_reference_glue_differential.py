"""The reference's REAL glue classes on top of this package's third-party replacements, against what they produced (CPU).

`realtime_voice_conversion/{stream,segment,worker,converter}/*.py`, `config.py`, `yukarin_wrapper/voice_changer.py` and
`yukarin_wrapper/acoustic_feature_wrapper.py` are pure Python over `yukarin` / `become_yukarin` / the vocoder.
tests/golden/make_reference_fixtures.py imported them from a checkout of the original project, with `yukarin`, `become_yukarin`
resolved by `dropin` and `yukarin_wrapper.vocoder` (the module that binds pyworld / world4py) replaced by ours, drove the
reference's EncodeStream -> ConvertStream(VoiceChanger) -> DecodeStream chain and its workers exactly as the helpers below do, and
stored what they produced in tests/golden/reference_glue.{json,npz}.  This package's own classes, driven the same way on the same
oracle-backed engine, must give the same.  The engine's U-Nets run on torch's CPU kernels, which are picked per CPU, so values
downstream of them (the converted spectrum and the decoded wave) are compared to a tolerance far below what any framing or indexing
difference would move them; the f0 contours, from the C WORLD analysis and the f0 statistics, must match exactly."""
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

GOLDEN = Path(__file__).resolve().parent / 'golden'
CHAIN_CASES = [(0.3, (0.0, 0.5, 0.0)), (0.1, (0.1, 0.2, 0.1))]
WORKER_T, WORKER_EXTRA = 0.3, (0.0, 0.5, 0.0)
RTOL = 1e-4
EXACT = (0, 1)             # per chain step: the encoded and the converted f0 (stored as digests); the sp (2) and the wave (3) as profiles
MODEL_KEYS = ('input_statistics_path', 'target_statistics_path', 'stage1_model_path', 'stage1_config_path', 'stage2_model_path',
              'stage2_config_path')


def digest(a) -> str:
    """dtype, shape and SHA-256 of the bytes: equal digests <=> equal arrays (NaNs included)."""
    a = np.ascontiguousarray(a)
    return f'{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()}'


def profile(a) -> np.ndarray:
    """What the fixture keeps of an output array: its values at 16 seeded positions and its sums over 32 consecutive blocks of the
    flattened array (a shifted window or a dropped or repeated frame moves both)."""
    a = np.asarray(a, np.float64).ravel()
    pos = np.random.default_rng(a.size).choice(a.size, size=min(a.size, 16), replace=False)
    return np.concatenate([a[pos], [b.sum() for b in np.array_split(a, min(a.size, 32))]])


def same_profile(want, got) -> bool:
    """Sampled values and block sums each within RTOL, relative to the largest of their own kind."""
    have = profile(got).astype(np.float32)
    parts = (slice(0, min(want.size, 16)), slice(min(want.size, 16), None))
    return all(np.allclose(have[p], want[p], rtol=RTOL, atol=RTOL * max(1e-3, float(np.nanmax(np.abs(want[p])))), equal_nan=True)
               for p in parts if want[p].size)


def plain(v):
    """A Config field as JSON stores it: enums by value, paths as strings."""
    return v.value if hasattr(v, 'value') else str(v) if isinstance(v, Path) else v


def golden():
    return json.loads((GOLDEN / 'reference_glue.json').read_text()), np.load(GOLDEN / 'reference_glue.npz')


def converters(models):
    """Oracle-backed engine and the converter objects both sides drive; the caller makes the engine the default one."""
    from realtime_yukarin_b200.models import AcousticConverter, F0Converter, SuperResolution
    from realtime_yukarin_b200.params import create_from_json, create_sr_from_json
    from tests.fake_engine import OracleEngine
    fake = OracleEngine(models['stage1_model_path'], models['stage2_model_path'])
    f0c = F0Converter(models['input_statistics_path'], models['target_statistics_path'])
    ac = AcousticConverter(create_from_json(models['stage1_config_path']), models['stage1_model_path'], f0_converter=f0c, engine=fake)
    sr = SuperResolution(create_sr_from_json(models['stage2_config_path']), models['stage2_model_path'], engine=fake)
    acp = create_from_json(models['stage1_config_path']).dataset.acoustic_param
    return fake, ac, sr, acp


def stream_chain(conv, T, extra, EncodeStream, ConvertStream, DecodeStream, StreamWrapper, VoiceChanger):
    """Encode -> convert -> decode of 1.5 s of synthetic speech in T-second pieces; per piece the encoded f0, the converted f0 / sp
    and the decoded wave.  `conv` = converters(...), its engine the default one."""
    from realtime_yukarin_b200 import synthetic
    from realtime_yukarin_b200.config import VocodeMode
    from realtime_yukarin_b200.vocoder import RealtimeVocoder
    _, ac, sr, acp = conv
    voc = RealtimeVocoder(acoustic_param=acp, out_sampling_rate=24000, extract_f0_mode=VocodeMode.WORLD)
    voc.create_synthesizer(buffer_size=1024, number_of_pointers=16)
    es, cs, ds = EncodeStream(vocoder=voc), ConvertStream(voice_changer=VoiceChanger(acoustic_converter=ac, super_resolution=sr, threshold=60)), DecodeStream(vocoder=voc)
    ws = [StreamWrapper(stream=es, extra_time=extra[0]), StreamWrapper(stream=cs, extra_time=extra[1]), StreamWrapper(stream=ds, extra_time=extra[2])]
    x = synthetic.synthetic_speech(1.5, 31)
    n = round(T * 24000)
    outs = []
    for k in range(len(x) // n):
        es.add(start_time=extra[0] + k * T, data=x[k * n:(k + 1) * n])
        f = ws[0].process_next(time_length=T)
        cs.add(start_time=extra[1] + k * T, data=f)
        c = ws[1].process_next(time_length=T)
        ds.add(start_time=extra[2] + k * T, data=c)
        y = ws[2].process_next(time_length=T)
        outs.append((np.asarray(f.f0).copy(), np.asarray(c.f0).copy(), np.asarray(c.sp).copy(), np.asarray(y.wave if hasattr(y, 'wave') else y).copy()))
    return outs


def librosa_stand_in():
    """`librosa.stft` / `librosa.core.power_to_db` for the reference's decode worker (decode_worker.py:56), written here in numpy
    (librosa 0.6/0.7 defaults: n_fft 2048, hop 512, periodic Hann, reflect-centred; ref 1, amin 1e-10, top_db 80).  Test harness only."""
    import types
    import scipy.signal as ss

    def stft(y, n_fft=2048, hop_length=None):
        hop = hop_length or n_fft // 4
        yp = np.pad(np.asarray(y, np.float64), n_fft // 2, mode='reflect')
        win = ss.get_window('hann', n_fft, fftbins=True)
        frames = 1 + len(y) // hop
        return np.stack([np.fft.rfft(yp[f * hop:f * hop + n_fft] * win) for f in range(frames)], 1)

    def power_to_db(S, ref=1.0, amin=1e-10, top_db=80.0):
        db = 10.0 * np.log10(np.maximum(amin, S)) - 10.0 * np.log10(np.maximum(amin, ref))
        return np.maximum(db, db.max() - top_db)

    lib = types.ModuleType('librosa'); lib.__path__ = []
    core = types.ModuleType('librosa.core')
    lib.stft, core.power_to_db, lib.core = stft, power_to_db, core
    return lib, core


def worker_setup(models, fake, acp):
    """Input, chunking and a Config whose output gate keeps some chunks and drops others: the powers of the ungated chunks through
    this package's RealtimePipeline, split at their widest gap.  -> (x, n, K, cfg, number of ungated chunks)."""
    from realtime_yukarin_b200 import synthetic
    from realtime_yukarin_b200.config import Config, VocodeMode
    from realtime_yukarin_b200.worker import Item, RealtimePipeline
    T, extra = WORKER_T, WORKER_EXTRA
    x = synthetic.synthetic_speech(3.0, stream=37)
    x[int(1.2 * 24000):int(2.1 * 24000)] *= 1e-4
    n = round(T * 24000)
    K = len(x) // n

    def make_cfg(out_thr):
        return Config(input_device_name=None, output_device_name=None, input_rate=24000, output_rate=24000, frame_period=5.0, buffer_time=T,
                      extract_f0_mode=VocodeMode.WORLD, vocoder_buffer_size=1024, input_scale=1.0, output_scale=1.0,
                      input_silent_threshold=60.0, output_silent_threshold=out_thr, encode_extra_time=extra[0],
                      convert_extra_time=extra[1], decode_extra_time=extra[2], **{k: models[k] for k in MODEL_KEYS})

    lib_probe, core_probe = librosa_stand_in()
    probe = RealtimePipeline(make_cfg(1e9), acoustic_param=acp, engine=fake, depth=1)
    powers = []
    for k in range(K):
        probe.put(Item(item=x[k * n:(k + 1) * n].copy(), index=k))
        it = probe.get()
        if it.item is not None:
            powers.append(float(core_probe.power_to_db(np.abs(lib_probe.stft(it.item)) ** 2).mean()))
    probe.close()
    ps = np.sort(np.asarray(powers))
    gi = int(np.argmax(np.diff(ps)))
    assert ps[gi + 1] - ps[gi] > 1e-3
    return x, n, K, make_cfg(-float(0.5 * (ps[gi] + ps[gi + 1]))), len(powers)


@pytest.mark.parametrize('T,extra', CHAIN_CASES)
def test_reference_streams_and_voice_changer_over_our_replacements(small_models, T, extra):
    from realtime_yukarin_b200 import engine as eng_mod
    from realtime_yukarin_b200 import stream as our_stream
    from realtime_yukarin_b200 import voice_changer as our_vc
    meta, arrays = golden()
    shapes = meta['chain'][f'{T:g}']
    conv = converters(small_models)
    eng_mod.set_default_engine(conv[0])
    try:
        got_ours = stream_chain(conv, T, extra, our_stream.EncodeStream, our_stream.ConvertStream, our_stream.DecodeStream,
                                our_stream.StreamWrapper, our_vc.VoiceChanger)
        assert len(shapes) == len(got_ours) > 0
        for k, (a, b) in enumerate(zip(shapes, got_ours)):
            assert a == [list(v.shape) for v in b], k
            for i, v in enumerate(b):
                if i in EXACT:
                    assert meta['chain_digests'][f'{T:g}'][k][str(i)] == digest(v), (k, i)
                else:
                    assert same_profile(arrays[f'chain_{T:g}_{k}_{i}'], v), (k, i)
    finally:
        eng_mod.set_default_engine(None)


def test_reference_workers_over_our_replacements_match_realtime_pipeline(small_models):
    """SURVEY 8(f) ranks 1 / 2 against the REAL worker code: the reference's encode_worker / convert_worker / decode_worker (worker/*.py,
    each in a thread with queue.Queue standing in for multiprocessing.Queue) over this package's replacements gave, per input chunk,
    the chunk played or None (not enough samples yet / gated as silent); worker.RealtimePipeline on the same engine must give the same
    Items in the same order."""
    from realtime_yukarin_b200 import engine as eng_mod
    from realtime_yukarin_b200.worker import Item, RealtimePipeline
    meta, arrays = golden()
    want = meta['workers']
    fake, _, _, acp = converters(small_models)
    eng_mod.set_default_engine(fake)
    try:
        x, n, K, cfg, n_ungated = worker_setup(small_models, fake, acp)
        assert abs(cfg.output_silent_threshold - want['output_silent_threshold']) < RTOL * abs(want['output_silent_threshold'])
        pipe = RealtimePipeline(cfg, acoustic_param=acp, engine=fake, depth=1)
        ours = []
        for k in range(K):
            pipe.put(Item(item=x[k * n:(k + 1) * n].copy(), index=k))
            ours.append(pipe.get())
        pipe.close()
        assert want['index'] == [it.index for it in ours] == list(range(K))
        played = 0
        for played_ref, b in zip(want['played'], ours):
            assert played_ref == (b.item is not None), b.index
            if played_ref:
                played += 1
                assert len(b.item) == cfg.out_audio_chunk
                assert same_profile(arrays[f'workers_{b.index}'], b.item), b.index
        assert 0 < played < n_ungated                     # the gate kept some chunks and dropped others, identically on both sides
    finally:
        eng_mod.set_default_engine(None)


def test_reference_converter_and_config_modules_over_our_replacements(small_models):
    """The reference's real converter/yukarin_converter.py and config.py: model loading through the reference's own call site
    (kwargs gpu=0, out_sampling_rate=24000, F0Converter(input_statistics=...)) landed in this package's classes, and its Config read
    these values from its config.yaml (stored as tests/golden/reference_config.yaml); ours must load the same classes and read the
    same values."""
    from realtime_yukarin_b200 import engine as eng_mod
    from realtime_yukarin_b200 import config as our_config
    from realtime_yukarin_b200.converter import YukarinConverter
    want = golden()[0]['converter_and_config']
    fake = converters(small_models)[0]
    eng_mod.set_default_engine(fake)
    try:
        conv = YukarinConverter.make_yukarin_converter(**{k: small_models[k] for k in MODEL_KEYS})
        for attr in ('acoustic_converter', 'super_resolution'):
            cls = type(getattr(conv, attr))
            assert f'{cls.__module__}.{cls.__qualname__}' == want['classes'][attr]
        assert fake.stats is not None
        b = our_config.Config.from_yaml(GOLDEN / 'reference_config.yaml')
        for name, va in want['fields'].items():
            assert va == plain(getattr(b, name)), name
        assert [b.in_audio_chunk, b.out_audio_chunk] == want['chunks']
    finally:
        eng_mod.set_default_engine(None)
