"""Host-side plugin API conformance (no GPU): the framing / indexing contract of the reference's
Stream + SegmentMethod layer, restated as known-answer tests, plus -- when the reference checkout is
present -- the reference's own mock-based unit tests executed unmodified against this package
through the drop-in import aliases.  Results of the reference's own code are stored under tests/golden/
(tests/golden/make_reference_fixtures.py)."""
import importlib.util
import json
import os
import unittest
from pathlib import Path

import numpy as np
import pytest

from realtime_yukarin_b200 import dropin
from realtime_yukarin_b200.feature import AcousticFeature, AcousticFeatureWrapper, Wave
from realtime_yukarin_b200.params import AcousticParam, Param
from realtime_yukarin_b200.segment import (BaseSegmentMethod, FeatureWrapperSegmentMethod, Segment, WaveSegmentMethod)
from realtime_yukarin_b200.stream import BaseStream, ConvertStream, EncodeStream, StreamWrapper


class TextMethod(BaseSegmentMethod):
    def length(self, data):
        return len(data)

    def pad(self, width):
        return ' ' * width

    def pick(self, data, first, last):
        return data[first:last]

    def concat(self, datas):
        return ''.join(datas)


class TextStream(BaseStream):
    def process(self, start_time, time_length, extra_time):
        return self.fetch(start_time, time_length, extra_time)


def make_text_stream(rate=10):
    s = TextStream(TextMethod(rate), TextMethod(rate))
    s.add(start_time=0, data='a' * rate)
    s.add(start_time=1, data='b' * rate)
    return s


def test_segment_record():
    m = TextMethod(4)
    seg = Segment(start_time=1, data='xxxxxxxx', method=m)
    assert (seg.start_time, seg.data, seg.method) == (1, 'xxxxxxxx', m)
    assert seg.length == 8 and seg.time_length == 2.0 and seg.end_time == 3.0 and seg.sampling_rate == 4
    assert tuple(seg) == (1, 'xxxxxxxx', m)


def test_fetch_known_answers():            # base_stream.py:32-79 via tests/test_base_stream.py:65-93
    s = make_text_stream()
    assert s.fetch(0, 1, 0) == 'a' * 10
    assert s.fetch(0.5, 1, 0) == 'a' * 5 + 'b' * 5
    assert s.fetch(-0.5, 1, 0) == ' ' * 5 + 'a' * 5
    assert s.fetch(1.5, 1, 0) == 'b' * 5 + ' ' * 5
    assert s.fetch(0, 1, 0.3) == ' ' * 3 + 'a' * 10 + 'b' * 3
    assert s.fetch(0, 2, 0.3) == ' ' * 3 + 'a' * 10 + 'b' * 10 + ' ' * 3


def test_remove_keeps_segments_ending_after():   # tests/test_base_stream.py:47-63
    s = make_text_stream()
    s.add(start_time=2, data='c' * 10)
    for end, left in ((0, 3), (1, 2), (2, 1), (3, 0)):
        s.remove(end_time=end)
        assert len(s.stream) == left


def test_fetch_gap_between_segments_is_padded():
    s = TextStream(TextMethod(10), TextMethod(10))
    s.add(start_time=0, data='a' * 10)
    s.add(start_time=2, data='c' * 10)
    assert s.fetch(0.5, 2, 0) == 'a' * 5 + ' ' * 10 + 'c' * 5


class VocoderMock:
    acoustic_param = AcousticParam()


def test_encode_stream_wave_fetch():       # tests/test_encode_stream.py:34-85
    st = EncodeStream(vocoder=VocoderMock())
    sr = VocoderMock.acoustic_param.sampling_rate
    one, two = np.ones(sr, np.float32), np.ones(sr, np.float32) * 2
    st.add(0, one)
    st.add(1, two)
    np.testing.assert_equal(st.fetch(0, 1, 0), one)
    np.testing.assert_equal(st.fetch(0.5, 1, 0), np.concatenate([one[:sr // 2], two[:sr // 2]]))
    np.testing.assert_equal(st.fetch(-0.5, 1, 0), np.concatenate([np.zeros(sr // 2, np.float32), one[:sr // 2]]))
    np.testing.assert_equal(st.fetch(0, 2, 0.3), np.concatenate([np.zeros(sr // 10 * 3), one, two, np.zeros(sr // 10 * 3)]))
    assert st.out_segment_method.sampling_rate == 200


class AttrDict(dict):
    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.__dict__ = self


def _wrapper(values, lengths, sr=16000, rate=200):
    return AcousticFeatureWrapper(
        wave=Wave(np.concatenate([np.ones(round(t * sr), np.float32) * v for v, t in zip(values, lengths)]), sr),
        f0=np.concatenate([np.ones((round(t * rate), 1), np.float32) * v for v, t in zip(values, lengths)]))


def test_convert_stream_feature_wrapper_fetch():   # tests/test_convert_stream.py:19-104
    vc = AttrDict(
        acoustic_converter=AttrDict(config=AttrDict(dataset=AttrDict(acoustic_param=AcousticParam(sampling_rate=16000)))),
        super_resolution=AttrDict(config=AttrDict(dataset=AttrDict(param=Param()))),
        output_sampling_rate=24000)
    st = ConvertStream(voice_changer=vc)
    st.in_segment_method._keys = ['f0']
    st.add(0, _wrapper([1], [1]))
    st.add(1, _wrapper([2], [1]))
    assert st.fetch(0, 1, 0) == _wrapper([1], [1])
    assert st.fetch(0.5, 1, 0) == _wrapper([1, 2], [0.5, 0.5])
    assert st.fetch(-0.5, 1, 0) == _wrapper([0, 1], [0.5, 0.5])
    assert st.fetch(1.5, 1, 0) == _wrapper([2, 0], [0.5, 0.5])
    assert st.fetch(0, 1, 0.3) == _wrapper([0, 1, 2], [0.3, 1, 0.3])
    assert st.fetch(0, 2, 0.3) == _wrapper([0, 1, 2, 0], [0.3, 1, 1, 0.3])


def test_feature_wrapper_segment_method():          # tests/test_feature_wrapper_segment_method.py:17-70
    m = FeatureWrapperSegmentMethod(sampling_rate=100, wave_sampling_rate=10000, order=5, frame_period=10)
    seg = lambda v, t: _wrapper(v, t, sr=10000, rate=100)
    pad = m.pad(width=100)
    assert pad == seg([0], [1])
    assert pad.wave.wave.dtype == np.float32 and pad.f0.shape == (100, 1) and pad.mc.shape == (100, 6)
    full = seg([1], [1])
    assert m.pick(full, 0, 50) == seg([1], [0.5])
    assert m.pick(full, 50, 100) == seg([1], [0.5])
    m._keys = ['f0']
    assert m.concat([seg([0], [1]), seg([1], [1])]) == seg([0, 1], [1, 1])


def test_acoustic_feature_helpers():
    sizes = AcousticFeature.get_sizes(sampling_rate=24000, order=8)
    assert sizes == dict(f0=1, sp=513, ap=513, coded_ap=3, mc=9, voiced=1)
    s = AcousticFeature.silent(4, sizes, keys=['f0', 'ap', 'mc', 'voiced'])
    assert s.f0.shape == (4, 1) and s.voiced.dtype == bool and not s.voiced.any() and (s.ap == 0).all()
    assert set(s.__dict__) == {'f0', 'sp', 'ap', 'coded_ap', 'mc', 'voiced'}
    rebuilt = AcousticFeature(**s.__dict__)                       # __dict__ round-trips through the constructor
    assert rebuilt.mc is s.mc
    p = s.pick(1, -1, keys=['f0', 'mc'])
    assert len(p.f0) == 2
    c = AcousticFeature.concatenate([s, s], keys=['f0'])
    assert len(c.f0) == 8
    idx = s.indexing(np.array([True, False, True, False]))
    assert len(idx.f0) == 2 and len(idx.mc) == 2


@pytest.mark.parametrize('rate,T,extra', [(24000, 0.3, 0.0), (24000, 0.3, 0.1), (200, 0.3, 0.5), (200, 0.1, 0.5), (200, 1.0, 0.5), (200, 0.3, 0.05)])
def test_worker_drive_window_identity(rate, T, extra):
    """SURVEY A.9a: driven like the workers (add at extra + k T, process_next(T)), step k's window is
    exactly round((T + 2 extra) rate) items long and item i is input item k n - 2 e + i (0 where negative)."""
    class Ident(BaseStream):
        def process(self, start_time, time_length, extra_time):
            return self.fetch(start_time, time_length, extra_time)
    st = Ident(WaveSegmentMethod(rate), WaveSegmentMethod(rate))
    w = StreamWrapper(st, extra_time=extra)
    n, e = round(T * rate), round(extra * rate)
    start = extra
    for k in range(400):
        st.add(start_time=start, data=np.arange(k * n, (k + 1) * n, dtype=np.float32) + 1)
        start += T
        win = w.process_next(T)
        assert len(win) == round((T + 2 * extra) * rate)
        idx = k * n - 2 * e + np.arange(len(win))
        np.testing.assert_array_equal(win, np.where(idx >= 0, idx + 1, 0).astype(np.float32))
        if k % 50 == 49:
            st.remove(end_time=start - 3 * T - 4 * extra)


GOLDEN = Path(__file__).resolve().parent / 'golden'
# a checkout of the original project: the tests that restate its own test modules then also run those modules
REF_ROOT = Path(os.environ['RYK_REFERENCE_CHECKOUT']) if os.environ.get('RYK_REFERENCE_CHECKOUT') else None


def reference_streams():
    return json.loads((GOLDEN / 'reference_streams.json').read_text())


REFERENCE_UNIT_TESTS = ['test_segment', 'test_base_stream', 'test_encode_stream', 'test_convert_stream', 'test_feature_wrapper_segment_method']


def compared_value(v):
    """An assertion operand as tests/golden/reference_unit_tests.json stores it (None for any other object)."""
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    from tests.test_reference_glue_differential import digest
    if isinstance(v, np.ndarray):
        return digest(v)
    if isinstance(v, AcousticFeatureWrapper):
        return dict(wave=digest(v.wave.wave), rate=v.wave.sampling_rate, f0=digest(v.f0))
    return None


def compared(kind, a, b=None):
    """One assertion as recorded: its kind and both operands (for other objects: whether they are the same object)."""
    if kind == 'assertTrue':
        return [kind, bool(a)]
    ra, rb = compared_value(a), compared_value(b)
    if (ra is None and a is not None) or (rb is None and b is not None):
        return [kind, dict(same_object=a is b)]
    return [kind, [ra, rb]]


def _unit_cases(name):
    """The cases of the reference's tests/<name>.py restated on this package: test method -> the assertions it makes, in order."""
    eq = lambda a, b: compared('assertEqual', a, b)
    npeq = lambda a, b: compared('assert_equal', a, b)
    if name == 'test_segment':
        m = TextMethod(1)
        seg = Segment(start_time=1, data='', method=m)
        return {'test': [eq(1, seg.start_time), eq('', seg.data), eq(m, seg.method)]}
    if name == 'test_base_stream':
        def three():
            s = make_text_stream()
            s.add(start_time=2, data='c' * 10)
            return s
        s = three()
        removed = [eq(len(s.stream), 3)]
        for end in (0, 1, 2, 3):
            s.remove(end_time=end)
            removed.append(eq(len(s.stream), 3 - end))
        f = make_text_stream().fetch
        return {'test_initialize': [], 'test_add': [eq(len(three().stream), 3)], 'test_remove': removed,
                'test_fetch': [eq(f(0, 1, 0), 'a' * 10), eq(f(0.5, 1, 0), 'a' * 5 + 'b' * 5)],
                'test_fetch_with_padding': [eq(f(-0.5, 1, 0), ' ' * 5 + 'a' * 5), eq(f(1.5, 1, 0), 'b' * 5 + ' ' * 5)],
                'test_fetch_with_extra': [eq(f(0, 1, 0.3), ' ' * 3 + 'a' * 10 + 'b' * 3),
                                          eq(f(0, 2, 0.3), ' ' * 3 + 'a' * 10 + 'b' * 10 + ' ' * 3)]}
    if name == 'test_encode_stream':
        sr = AcousticParam().sampling_rate
        ones = lambda v, n=sr: np.ones(n, dtype=np.float32) * v
        cat = lambda *parts: np.concatenate([ones(*p) for p in parts])
        st = EncodeStream(vocoder=VocoderMock())
        st.add(start_time=0, data=ones(1))
        st.add(start_time=1, data=ones(2))
        h, e = sr // 2, sr // 10 * 3
        return {'test_initialize': [],
                'test_fetch': [npeq(st.fetch(0, 1, 0), ones(1)), npeq(st.fetch(0.5, 1, 0), cat((1, h), (2, h)))],
                'test_fetch_with_padding': [npeq(st.fetch(-0.5, 1, 0), cat((0, h), (1, h))), npeq(st.fetch(1.5, 1, 0), cat((2, h), (0, h)))],
                'test_fetch_with_extra': [npeq(st.fetch(0, 1, 0.3), cat((0, e), (1,), (2, e))),
                                          npeq(st.fetch(0, 2, 0.3), cat((0, e), (1,), (2,), (0, e)))]}
    if name == 'test_convert_stream':
        vc = AttrDict(
            acoustic_converter=AttrDict(config=AttrDict(dataset=AttrDict(acoustic_param=AcousticParam(sampling_rate=16000)))),
            super_resolution=AttrDict(config=AttrDict(dataset=AttrDict(param=Param()))),
            output_sampling_rate=24000)
        st = ConvertStream(voice_changer=vc)
        st.in_segment_method._keys = ['f0']
        st.add(start_time=0, data=_wrapper([1], [1]))
        st.add(start_time=1, data=_wrapper([2], [1]))
        return {'test_initialize': [],
                'test_fetch': [eq(st.fetch(0, 1, 0), _wrapper([1], [1])), eq(st.fetch(0.5, 1, 0), _wrapper([1, 2], [0.5, 0.5]))],
                'test_fetch_with_padding': [eq(st.fetch(-0.5, 1, 0), _wrapper([0, 1], [0.5, 0.5])),
                                            eq(st.fetch(1.5, 1, 0), _wrapper([2, 0], [0.5, 0.5]))],
                'test_fetch_with_extra': [eq(st.fetch(0, 1, 0.3), _wrapper([0, 1, 2], [0.3, 1, 0.3])),
                                          eq(st.fetch(0, 2, 0.3), _wrapper([0, 1, 2, 0], [0.3, 1, 1, 0.3]))]}
    assert name == 'test_feature_wrapper_segment_method', name
    m = FeatureWrapperSegmentMethod(sampling_rate=100, wave_sampling_rate=10000, order=5, frame_period=10)
    seg = lambda v, t: _wrapper(v, t, sr=10000, rate=100)
    return {'test_pad': [eq(m.pad(width=100), seg([0], [1]))],
            'test_pick': [eq(m.pick(seg([1], [1]), first=0, last=50), seg([1], [0.5])),
                          eq(m.pick(seg([1], [1]), first=50, last=100), seg([1], [0.5]))],
            'test_concat': [eq(m.concat([seg([0], [1]), seg([1], [1])]), seg([0, 1], [1, 1]))]}


def _run_reference_module(path):
    dropin.install()
    spec = importlib.util.spec_from_file_location(f'_reference_{path.stem}', path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    suite = unittest.defaultTestLoader.loadTestsFromModule(mod)
    return unittest.TextTestRunner(verbosity=0).run(suite)


@pytest.mark.parametrize('name', REFERENCE_UNIT_TESTS)
def test_reference_unit_test_cases(name):
    """The reference's own mock-based unit-test module tests/<name>.py against this package.  Its source is not part of this
    repository, so every assertion it made -- run unmodified through the drop-in aliases -- is recorded in
    tests/golden/reference_unit_tests.json (tests/golden/make_reference_fixtures.py), and its cases, restated here, must make the
    same assertions with the same operands.  With RYK_REFERENCE_CHECKOUT naming a checkout, the module itself runs too."""
    want = json.loads((GOLDEN / 'reference_unit_tests.json').read_text())[name]
    assert _unit_cases(name) == want
    if REF_ROOT is not None:
        result = _run_reference_module(REF_ROOT / 'tests' / f'{name}.py')
        assert result.testsRun > 0 and result.wasSuccessful(), result.failures + result.errors


CHECK_PY_PIECES = 3


def check_py_input():
    from realtime_yukarin_b200 import synthetic
    return synthetic.synthetic_speech(CHECK_PY_PIECES + 0.4, stream=23)


def check_py_sample_positions(length):
    """The stored sample of check.py's output: 512 seeded positions (the whole wave would not fit a small fixture)."""
    return np.sort(np.random.default_rng(23).choice(length, size=min(length, 512), replace=False))


def check_py_flow(x, pieces, conv):
    """check.py's flow on this package: 1 s pieces of x through EncodeStream -> ConvertStream(VoiceChanger) -> DecodeStream, each
    stream fed every piece at start i and asked for every 1 s window with extras (0, 1, 0); the windows' waves concatenated as
    float32.  `conv` = converters(...) of tests/test_reference_glue_differential.py, its engine the default one."""
    from realtime_yukarin_b200 import stream as our_stream
    from realtime_yukarin_b200.config import VocodeMode
    from realtime_yukarin_b200.vocoder import RealtimeVocoder
    from realtime_yukarin_b200.voice_changer import VoiceChanger
    _, ac, sr_model, acp = conv
    rate = acp.sampling_rate
    voc = RealtimeVocoder(acoustic_param=acp, out_sampling_rate=24000, extract_f0_mode=VocodeMode.WORLD)
    voc.create_synthesizer(buffer_size=1024, number_of_pointers=16)
    vc = VoiceChanger(acoustic_converter=ac, super_resolution=sr_model, output_sampling_rate=24000)
    datas = [x[i * rate:(i + 1) * rate] for i in range(len(x) // rate)][:pieces]
    for st, extra in zip((our_stream.EncodeStream(vocoder=voc), our_stream.ConvertStream(voice_changer=vc), our_stream.DecodeStream(vocoder=voc)),
                         (0, 1, 0)):
        for i, d in enumerate(datas):
            st.add(start_time=i, data=d)
        datas = [st.process(start_time=i, time_length=1, extra_time=extra) for i in range(pieces)]
    return np.concatenate(datas).astype(np.float32)


def test_reference_check_py_flow_matches_its_output_and_the_oracle(small_models):
    """BASELINE config 1: the reference's own check.py -- wav in, EncodeStream / ConvertStream / DecodeStream over 1 s pieces with
    extras (0, 1, 0), wav out -- run unmodified through the drop-in aliases with the oracle-backed engine, wrote the wave sampled
    in tests/golden/reference_streams.json.  Its flow, restated on this package's classes (check_py_flow), must give that wave
    and must equal the same flow composed by hand from the oracle's functions.  Against the hand-built flow, computed in the same
    process, the tolerance is 1e-6 of the peak; against the stored sample it is RTOL of the peak, because the engine's U-Nets run
    on torch's CPU kernels, which are picked per CPU."""
    from oracle import nets as onets
    from oracle import pipeline as opipe
    from oracle import world as W
    from realtime_yukarin_b200 import engine as eng_mod
    from realtime_yukarin_b200.models import F0Converter
    from tests.test_reference_glue_differential import RTOL, converters
    g = reference_streams()['check_py']
    assert g['rate'] == 24000
    N = CHECK_PY_PIECES
    x = check_py_input()
    conv = converters(small_models)
    eng_mod.set_default_engine(conv[0])
    try:
        got = check_py_flow(x, N, conv)
    finally:
        eng_mod.set_default_engine(None)
    assert len(got) == g['length'] > 0
    pos = check_py_sample_positions(len(got))
    assert np.abs(got[pos] - np.asarray(g['values'], np.float32)).max() <= RTOL * g['abs_max']
    assert abs(float(np.abs(got).max()) - g['abs_max']) <= RTOL * g['abs_max']
    # the same flow by hand: per-piece analysis, convert windows of 1 + 1 + 1 s with silent padding outside the file, decode
    cfg = opipe.PathConfig()
    p1, p2 = onets.load_npz(small_models['stage1_model_path']), onets.load_npz(small_models['stage2_model_path'])
    stats = F0Converter(small_models['input_statistics_path'], small_models['target_statistics_path']).stats()
    pieces = [x[i * 24000:(i + 1) * 24000] for i in range(N)]
    feats = [opipe.extract_features(w, cfg) for w in pieces]
    cat = {k: np.concatenate([f[k] for f in feats]) for k in ('f0', 'ap', 'mc', 'voiced')}
    wave_all = np.concatenate(pieces)
    T = 200
    silent_mc = np.zeros((1, cfg.order + 1), np.float32)
    silent_mc[0, 0] = opipe.SILENT_MC0
    win = opipe.StreamOracle._window
    synth = W.RealtimeSynthesizer(24000, 5.0, 1024, 1024)
    outs = []
    for i in range(N):
        first = (i - 1) * T
        wfeat = dict(f0=win(cat['f0'], first, 3 * T, 0.0), ap=win(cat['ap'], first, 3 * T, 0.0), mc=win(cat['mc'], first, 3 * T, silent_mc),
                     voiced=win(cat['voiced'], first, 3 * T, False))
        wwave = win(wave_all, first * cfg.hop, 3 * T * cfg.hop, 0.0)
        conv = opipe.convert_window(wwave, wfeat, cfg, p1, p2, stats, backend='torch')
        y = synth.decode(conv['f0'][T:-T].ravel().astype(np.float64), conv['sp'][T:-T], conv['ap'][T:-T])
        outs.append(np.nan_to_num(y, nan=0.0))
    ref = np.concatenate(outs).astype(np.float32)
    assert len(got) == len(ref)
    assert np.abs(got - ref).max() < 1e-6 * max(1.0, float(np.abs(ref).max()))


def test_config_reads_the_reference_yaml():
    """Config.from_yaml (config.py:44-71) on the reference's own config.yaml: same fields, enum and derived chunk sizes."""
    from realtime_yukarin_b200.config import Config, VocodeMode
    c = Config.from_yaml(GOLDEN / 'reference_config.yaml')
    assert c.input_rate == 24000 and c.output_rate == 24000 and c.frame_period == 5 and c.buffer_time == 1
    assert c.extract_f0_mode is VocodeMode.WORLD and c.vocoder_buffer_size == 1024
    assert (c.encode_extra_time, c.convert_extra_time, c.decode_extra_time) == (0.0, 0.5, 0.0)
    assert c.input_silent_threshold == 80 and c.output_silent_threshold == 80
    assert c.in_audio_chunk == 24000 and c.out_audio_chunk == 24000          # config.py:37-43
    assert isinstance(c.stage1_model_path, Path) and c.stage2_config_path.name == 'config.json'


def test_make_yukarin_converter_loads_both_stages(small_models):
    """YukarinConverter.make_yukarin_converter (converter/yukarin_converter.py:22-60): statistics, stage-1 and stage-2 models land
    in the engine (here the oracle-backed stand-in) and the converter exposes the objects VoiceChanger needs."""
    from realtime_yukarin_b200 import engine as eng_mod
    from realtime_yukarin_b200.converter import YukarinConverter
    from realtime_yukarin_b200.voice_changer import VoiceChanger
    from tests.fake_engine import OracleEngine
    fake = OracleEngine(small_models['stage1_model_path'], small_models['stage2_model_path'])
    eng_mod.set_default_engine(fake)
    try:
        conv = YukarinConverter.make_yukarin_converter(**{k: small_models[k] for k in (
            'input_statistics_path', 'target_statistics_path', 'stage1_model_path', 'stage1_config_path', 'stage2_model_path',
            'stage2_config_path')})
        assert conv.acoustic_converter.config.dataset.acoustic_param.sampling_rate == 24000
        assert fake.stats is not None and len(fake.stats) == 4           # log-f0 statistics reached the engine
        vc = VoiceChanger(super_resolution=conv.super_resolution, acoustic_converter=conv.acoustic_converter, threshold=80)
        assert vc.threshold == 80
    finally:
        eng_mod.set_default_engine(None)


def fetch_case(case):
    """A stored fetch case, from 5 ms grid units to seconds: (rate, [(start, frames)], (start, length, extra), remove time or None)."""
    rate, layout, win, rm = case
    return rate, [(k * 0.005, frames) for k, frames in layout], tuple(k * 0.005 for k in win), None if rm is None else rm * 0.005


def short_digest(a) -> str:
    """dtype, shape and the first 64 bits of the SHA-256 of the bytes (see digest in tests/test_reference_glue_differential.py)."""
    from tests.test_reference_glue_differential import digest
    return digest(a)[:-48]


def fetch_case_segments(rate, layout):
    """(start_time, data) of one stored fetch case: consecutive ramps, so that every sample tells where it came from."""
    base = 1.0
    for start, n_frames in sorted(layout):
        n = round(n_frames * 0.005 * rate)
        yield start, (base + np.arange(n)).astype(np.float32)
        base += 100000.0


def test_fetch_and_remove_differential_against_the_reference_classes():
    """Rows a1-a3 against the REAL reference code: 300 seeded random segment layouts (gaps, overlaps, touching segments) with random
    fetch windows / remove times went through the reference's BaseStream + a wave segment method (stored in
    tests/golden/reference_streams.json); through this package's the segments kept and the fetched arrays must be identical
    element for element."""
    g = reference_streams()['fetch']
    assert len(g['cases']) == len(g['results']) == 300
    for case, want in zip(g['cases'], g['results']):
        rate, layout, win, rm = fetch_case(case)
        ours = BaseStream(in_segment_method=WaveSegmentMethod(sampling_rate=rate), out_segment_method=WaveSegmentMethod(sampling_rate=rate))
        for start, data in fetch_case_segments(rate, layout):
            ours.add(start_time=start, data=data)
        if rm is not None:
            ours.remove(end_time=rm)
            assert want['kept'] == [s.start_time for s in ours.stream]
        assert want['fetched'] == short_digest(ours.fetch(start_time=win[0], time_length=win[1], extra_time=win[2])), (rate, layout, win, rm)


def test_reference_integration_test_cases(tmp_path, small_models, monkeypatch):
    """The reference's own integration-test module tests/test_all_stream.py (encode / convert / decode streams over its audioA.wav
    recording with the oracle-backed engine).  Its source is not part of this repository, so its cases are restated here on the
    first 4 s of that recording (tests/golden/audioA_24k_4s.wav, read at 24 kHz): both models load; a 1 s piece is 24000 samples;
    the encode stream's output for a picked, a concatenated and a padded window equals encoding that window directly; the convert
    stream's output f0 equals converting directly; the three streams over ten 0.3 s pieces with extras (0, 1, 0) give a finite,
    non-silent wave.  With RYK_REFERENCE_CHECKOUT naming a checkout, the module itself runs too."""
    import scipy.signal
    from realtime_yukarin_b200 import engine as eng_mod
    from realtime_yukarin_b200 import stream as our_stream
    from realtime_yukarin_b200 import wave_io
    from realtime_yukarin_b200.config import VocodeMode
    from realtime_yukarin_b200.vocoder import RealtimeVocoder
    from realtime_yukarin_b200.voice_changer import VoiceChanger
    from tests.test_reference_glue_differential import converters
    fake, ac, sr_model, acp = converters(small_models)
    eng_mod.set_default_engine(fake)
    try:
        assert ac is not None and sr_model is not None
        data, fs = wave_io.read_wav(GOLDEN / 'audioA_24k_4s.wav')
        x = scipy.signal.resample_poly(data.astype(np.float64), 24000, fs).astype(np.float32)
        rate = acp.sampling_rate

        def pieces(t):
            n = round(t * rate)
            return [x[i * n:(i + 1) * n] for i in range(len(x) // n)]

        def new_vocoder():
            voc = RealtimeVocoder(acoustic_param=acp, out_sampling_rate=24000, extract_f0_mode=VocodeMode.WORLD)
            voc.create_synthesizer(buffer_size=1024, number_of_pointers=16)
            return voc

        voc = new_vocoder()
        vc = VoiceChanger(acoustic_converter=ac, super_resolution=sr_model, output_sampling_rate=24000)
        encode = lambda w: voc.encode(Wave(wave=w, sampling_rate=rate))
        waves = pieces(1)
        assert len(waves[0]) == rate == 24000

        es = our_stream.EncodeStream(vocoder=voc)
        es.add(start_time=0, data=waves[0])
        es.add(start_time=1, data=waves[1])
        k = rate * 3 // 10
        assert es.process(start_time=0, time_length=1, extra_time=0) == encode(waves[0])
        assert es.process(start_time=0.3, time_length=1, extra_time=0) == encode(np.concatenate([waves[0][k:], waves[1][:k]]))
        assert es.process(start_time=1.3, time_length=1, extra_time=0) == encode(np.concatenate([waves[1][k:], np.zeros(k)]))

        cs = our_stream.ConvertStream(voice_changer=vc)
        cs.add(start_time=0, data=encode(waves[0]))
        cs.add(start_time=1, data=encode(waves[1]))
        assert np.all(cs.process(start_time=0, time_length=1, extra_time=0).f0 == vc.convert_from_acoustic_feature(encode(waves[0])).f0)

        voc = new_vocoder()
        streams = (our_stream.EncodeStream(vocoder=voc), our_stream.ConvertStream(voice_changer=vc), our_stream.DecodeStream(vocoder=voc))
        T, N = 0.3, 10
        datas = pieces(T)[:N]
        for st, extra in zip(streams, (0, 1, 0)):
            for i, d in enumerate(datas):
                st.add(start_time=i * T, data=d)
            datas = [st.process(start_time=i * T, time_length=T, extra_time=extra) for i in range(N)]
        y = np.concatenate([d.wave if hasattr(d, 'wave') else d for d in datas]).astype(np.float32)
        assert len(y) > 24000 and np.isfinite(y).all() and np.abs(y).max() > 0
    finally:
        eng_mod.set_default_engine(None)
    if REF_ROOT is None:
        return
    from tests.fake_engine import OracleEngine
    work = tmp_path / 'work'
    (work / 'tests' / 'data').mkdir(parents=True)
    (work / 'tests' / 'data' / 'audioA.wav').symlink_to(REF_ROOT / 'tests' / 'data' / 'audioA.wav')      # read in place, never copied
    monkeypatch.chdir(work)                                   # the module reads tests/data/... and writes ../test_convert_extra05.wav
    for env, key in (('INPUT_STATISTICS', 'input_statistics_path'), ('TARGET_STATISTICS', 'target_statistics_path'),
                     ('ACOUSTIC_CONVERT_MODEL', 'stage1_model_path'), ('ACOUSTIC_CONVERT_CONFIG', 'stage1_config_path'),
                     ('SUPER_RESOLUTION_MODEL', 'stage2_model_path'), ('SUPER_RESOLUTION_CONFIG', 'stage2_config_path')):
        monkeypatch.setenv(env, str(small_models[key]))
    fake = OracleEngine(small_models['stage1_model_path'], small_models['stage2_model_path'])
    eng_mod.set_default_engine(fake)
    try:
        result = _run_reference_module(REF_ROOT / 'tests' / 'test_all_stream.py')
        assert result.testsRun >= 6 and result.wasSuccessful(), result.failures + result.errors
        y, sr = wave_io.read_wav(tmp_path / 'test_convert_extra05.wav')
        assert sr == 24000 and len(y) > 24000 and np.isfinite(y).all() and np.abs(y).max() > 0
    finally:
        eng_mod.set_default_engine(None)
