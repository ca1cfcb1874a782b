"""Regenerates the fixtures that pin this package to the original project (realtime-yukarin) it re-implements:

  python tests/golden/make_reference_fixtures.py <checkout of the original project>     (run from the repo root, CPU only)

  audioA_24k_4s.wav          the first 4 s of the original's tests/data/audioA.wav (44.1 kHz), resampled to 24 kHz, 16-bit PCM
  reference_config.yaml      the original's config.yaml, unchanged
  reference_glue.json/.npz   what the original's own pure-Python glue (streams, voice changer, workers, converter, config) produced
                             over this package's replacements, driven as tests/test_reference_glue_differential.py drives ours
                             (shapes, gate decisions and profiles of the arrays: see profile() there)
  reference_unit_tests.json  every assertion (kind and operands) the original's own unit-test modules made, run unmodified
                             against this package -- for tests/test_stream_api.py
  reference_streams.json     the original's BaseStream on seeded segment layouts / fetch windows / remove times, and what its
                             check.py wrote (seeded sample) -- for tests/test_stream_api.py

The original's modules are imported from the checkout (never copied): `yukarin` / `become_yukarin` resolve to this package through
`dropin`, and `yukarin_wrapper.vocoder` (the pyworld / world4py binding) is replaced by ours."""
import importlib
import importlib.util
import json
import os
import queue
import shutil
import sys
import tempfile
import threading
import types
import wave
from pathlib import Path

import numpy as np
import scipy.signal

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from realtime_yukarin_b200 import dropin, synthetic, wave_io  # noqa: E402
from realtime_yukarin_b200 import engine as eng_mod  # noqa: E402
from realtime_yukarin_b200 import vocoder  # noqa: E402
from tests import test_reference_glue_differential as glue  # noqa: E402
from tests import test_stream_api as sapi  # noqa: E402

OUT = Path(__file__).resolve().parent


class RealReferencePackage:
    """Context manager: `realtime_voice_conversion` resolves to the checkout (except yukarin_wrapper.vocoder = ours)."""

    def __init__(self, ref_root: Path):
        self.root = ref_root / 'realtime_voice_conversion'

    def __enter__(self):
        dropin.install()                                   # yukarin / become_yukarin / librosa aliases
        self.saved = {k: v for k, v in sys.modules.items() if k == 'realtime_voice_conversion' or k.startswith('realtime_voice_conversion.')}
        for k in self.saved:
            del sys.modules[k]
        pkg = types.ModuleType('realtime_voice_conversion')
        pkg.__path__ = [str(self.root)]                    # real files for every submodule ...
        sys.modules['realtime_voice_conversion'] = pkg
        yw = types.ModuleType('realtime_voice_conversion.yukarin_wrapper')
        yw.__path__ = [str(self.root / 'yukarin_wrapper')]
        sys.modules['realtime_voice_conversion.yukarin_wrapper'] = yw
        voc = types.ModuleType('realtime_voice_conversion.yukarin_wrapper.vocoder')    # ... except the pyworld / world4py binding
        voc.Vocoder, voc.RealtimeVocoder = vocoder.Vocoder, vocoder.RealtimeVocoder
        sys.modules['realtime_voice_conversion.yukarin_wrapper.vocoder'] = voc
        self.saved_aux = {k: sys.modules.get(k) for k in ('librosa', 'librosa.core', 'chainer')}
        lib, core = glue.librosa_stand_in()                # worker/__init__ imports librosa and chainer
        sys.modules['librosa'], sys.modules['librosa.core'] = lib, core
        self.chainer = types.ModuleType('chainer')
        self.chainer.global_config = types.SimpleNamespace(enable_backprop=True, train=True)
        sys.modules['chainer'] = self.chainer
        return self

    def load(self, name):
        mod = importlib.import_module(f'realtime_voice_conversion.{name}')
        assert Path(mod.__file__).is_relative_to(self.root), mod.__file__          # really the checkout's code
        return mod

    def __exit__(self, *exc):
        for k in [k for k in sys.modules if k == 'realtime_voice_conversion' or k.startswith('realtime_voice_conversion.')]:
            del sys.modules[k]
        sys.modules.update(self.saved)
        for k, v in self.saved_aux.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        return False


def write_audio(ref_root: Path):
    data, fs = wave_io.read_wav(ref_root / 'tests' / 'data' / 'audioA.wav')
    x = data.astype(np.float64)
    if x.ndim > 1:
        x = x.mean(axis=1)
    x = scipy.signal.resample_poly(x, 24000, fs)[:24000 * 4]
    pcm = np.clip(np.round(x * 32768.0), -32768, 32767).astype('<i2')
    with wave.open(str(OUT / 'audioA_24k_4s.wav'), 'wb') as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(24000)
        w.writeframes(pcm.tobytes())


def glue_fixture(ref_root: Path, models):
    out, arrays = {}, {}
    conv = glue.converters(models)
    eng_mod.set_default_engine(conv[0])
    try:
        out['chain'] = {}
        for T, extra in glue.CHAIN_CASES:
            with RealReferencePackage(ref_root) as ref:
                rs, rvc = ref.load('stream'), ref.load('yukarin_wrapper.voice_changer')
                got = glue.stream_chain(conv, T, extra, rs.EncodeStream, rs.ConvertStream, rs.DecodeStream, rs.StreamWrapper, rvc.VoiceChanger)
            out['chain'][f'{T:g}'] = [[list(v.shape) for v in step] for step in got]
            out.setdefault('chain_digests', {})[f'{T:g}'] = [{i: glue.digest(v) for i, v in enumerate(step) if i in glue.EXACT} for step in got]
            arrays.update({f'chain_{T:g}_{k}_{i}': glue.profile(v).astype(np.float32) for k, step in enumerate(got) for i, v in enumerate(step)
                           if i not in glue.EXACT})

        fake, _, _, acp = conv
        _, ac, sr, _ = conv
        x, n, K, cfg, _ = glue.worker_setup(models, fake, acp)
        T, extra = glue.WORKER_T, glue.WORKER_EXTRA
        with RealReferencePackage(ref_root) as ref:
            workers = ref.load('worker')
            item_cls = ref.load('worker.utility').Item
            q_in, q_feat, q_conv, q_out = queue.Queue(), queue.Queue(), queue.Queue(), queue.Queue()
            locks = [threading.Lock() for _ in range(3)]
            for lk in locks:
                lk.acquire()
            voc = vocoder.RealtimeVocoder(acoustic_param=acp, out_sampling_rate=24000, extract_f0_mode=cfg.extract_f0_mode)
            threads = [
                threading.Thread(target=workers.encode_worker, daemon=True, kwargs=dict(
                    realtime_vocoder=voc, time_length=T, extra_time=extra[0], queue_input=q_in, queue_output=q_feat, acquired_lock=locks[0])),
                threading.Thread(target=workers.convert_worker, daemon=True, kwargs=dict(
                    acoustic_converter=ac, super_resolution=sr, time_length=T, extra_time=extra[1], input_silent_threshold=cfg.input_silent_threshold,
                    queue_input=q_feat, queue_output=q_conv, acquired_lock=locks[1])),
                threading.Thread(target=workers.decode_worker, daemon=True, kwargs=dict(
                    realtime_vocoder=voc, time_length=T, extra_time=extra[2], vocoder_buffer_size=1024, out_audio_chunk=cfg.out_audio_chunk,
                    output_silent_threshold=cfg.output_silent_threshold, queue_input=q_conv, queue_output=q_out, acquired_lock=locks[2])),
            ]
            cwd = Path.cwd()
            work = Path(tempfile.mkdtemp())
            os.chdir(work)                                 # the original's init_logger writes ./log.txt
            try:
                for th in threads:
                    th.start()
                for lk in locks:                           # run.py:95-96: wait until every worker is ready
                    assert lk.acquire(timeout=30)
                items = []
                for k in range(K):
                    q_in.put(item_cls(item=x[k * n:(k + 1) * n].copy(), index=k))
                    items.append(q_out.get(timeout=120))
            finally:
                os.chdir(cwd)
                shutil.rmtree(work, ignore_errors=True)
            assert ref.chainer.global_config.train is False and ref.chainer.global_config.enable_backprop is False    # convert_worker.py:33-34 ran
        out['workers'] = dict(output_silent_threshold=cfg.output_silent_threshold, index=[it.index for it in items],
                              played=[it.item is not None for it in items])
        arrays.update({f'workers_{it.index}': glue.profile(it.item).astype(np.float32) for it in items if it.item is not None})

        with RealReferencePackage(ref_root) as ref:
            yc = ref.load('converter.yukarin_converter')
            c = yc.YukarinConverter.make_yukarin_converter(**{k: models[k] for k in glue.MODEL_KEYS})
            classes = {a: f'{type(getattr(c, a)).__module__}.{type(getattr(c, a)).__qualname__}' for a in ('acoustic_converter', 'super_resolution')}
            a = ref.load('config').Config.from_yaml(ref_root / 'config.yaml')
        out['converter_and_config'] = dict(classes=classes, fields={f: glue.plain(getattr(a, f)) for f in a._fields},
                                           chunks=[a.in_audio_chunk, a.out_audio_chunk])
    finally:
        eng_mod.set_default_engine(None)
    return out, arrays


def fetch_cases(n=300, seed=7):
    """Seeded [rate, layout, window, remove time] cases in 5 ms grid units (see fetch_case in tests/test_stream_api.py): up to 6
    segments (half of them starting exactly where the previous one ends), a fetch window that may reach outside them, and a
    remove time or None."""
    rng = np.random.default_rng(seed)
    cases = []
    for _ in range(n):
        rate = int(rng.choice([200, 1000, 24000]))
        layout, end = [], None
        for _ in range(int(rng.integers(0, 7))):
            start = end if end is not None and end <= 400 and rng.random() < 0.5 else int(rng.integers(0, 401))
            frames = int(rng.integers(1, 301))
            layout.append([start, frames])
            end = start + frames
        win = [int(rng.integers(-50, 401)), int(rng.integers(1, 201)), int(rng.integers(0, 101))]
        rm = int(rng.integers(0, 401)) if rng.random() < 0.5 else None
        cases.append([rate, layout, win, rm])
    return cases


def streams_fixture(ref_root: Path, models) -> dict:
    out = {}
    with RealReferencePackage(ref_root) as ref:
        seg_mod, bs_mod = ref.load('segment.segment'), ref.load('stream.base_stream')

        class RefWave(seg_mod.BaseSegmentMethod):      # wave_segment.py:8-19 restated on the original's own base class
            def length(self, data): return len(data)
            def pad(self, width): return np.zeros(width, dtype=np.float32)
            def pick(self, data, first, last): return data[first:last]
            def concat(self, datas): return np.concatenate(list(datas))

        cases = fetch_cases()
        results = []
        for case in cases:
            rate, layout, win, rm = sapi.fetch_case(case)
            s = bs_mod.BaseStream(in_segment_method=RefWave(rate), out_segment_method=RefWave(rate))
            for start, data in sapi.fetch_case_segments(rate, layout):
                s.add(start_time=start, data=data)
            kept = None
            if rm is not None:
                s.remove(end_time=rm)
                kept = [x.start_time for x in s.stream]
            results.append(dict(kept=kept, fetched=sapi.short_digest(s.fetch(start_time=win[0], time_length=win[1], extra_time=win[2]))))
        out['fetch'] = dict(cases=cases, results=results)

    eng_mod.set_default_engine(glue.converters(models)[0])
    try:
        spec = importlib.util.spec_from_file_location('_reference_check', ref_root / 'check.py')
        check = importlib.util.module_from_spec(spec)
        dropin.install()
        spec.loader.exec_module(check)
        with tempfile.TemporaryDirectory() as d:
            wave_io.write_wav(Path(d) / 'in.wav', sapi.check_py_input(), 24000)
            check.check(input_path=Path(d) / 'in.wav', input_time_length=sapi.CHECK_PY_PIECES, output_path=Path(d) / 'out.wav',
                        **{k: models[k] for k in glue.MODEL_KEYS})
            got, sr = wave_io.read_wav(Path(d) / 'out.wav')
    finally:
        eng_mod.set_default_engine(None)
    pos = sapi.check_py_sample_positions(len(got))
    out['check_py'] = dict(rate=sr, length=len(got), abs_max=float(np.abs(got).max()),
                           values=[float(str(v)) for v in got[pos]])         # shortest text that reads back as the same float32
    return out


def unit_tests_fixture(ref_root: Path) -> dict:
    """Runs each of the original's unit-test modules unmodified, recording every assertion it makes, test method by test method."""
    import unittest
    import numpy.testing
    out = {}
    current = []

    def recording(kind, f, method):
        def g(*a, **k):
            operands = a[1:3] if method else a[:2]
            current.append(sapi.compared(kind, *operands))
            return f(*a, **k)
        return g

    saved = {k: getattr(unittest.TestCase, k) for k in ('assertEqual', 'assertNotEqual', 'assertTrue')}
    saved_np = numpy.testing.assert_equal
    try:
        for k, f in saved.items():
            setattr(unittest.TestCase, k, recording(k, f, True))
        numpy.testing.assert_equal = recording('assert_equal', saved_np, False)
        dropin.install()
        for name in sapi.REFERENCE_UNIT_TESTS:
            spec = importlib.util.spec_from_file_location(f'_reference_{name}', ref_root / 'tests' / f'{name}.py')
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            out[name] = {}
            for case in unittest.defaultTestLoader.loadTestsFromModule(mod):
                for test in case:
                    current = out[name][test._testMethodName] = []
                    result = unittest.TestResult()
                    test.run(result)
                    assert result.wasSuccessful() and result.testsRun == 1, (name, result.failures, result.errors)
    finally:
        for k, f in saved.items():
            setattr(unittest.TestCase, k, f)
        numpy.testing.assert_equal = saved_np
    return out


def main():
    ref_root = Path(sys.argv[1]).resolve()
    write_audio(ref_root)
    shutil.copyfile(ref_root / 'config.yaml', OUT / 'reference_config.yaml')
    with tempfile.TemporaryDirectory() as d:
        models = synthetic.write_synthetic_models(d, seed=3, base1=16, base2=16)     # the `small_models` fixture of tests/conftest.py
        meta, arrays = glue_fixture(ref_root, models)
        (OUT / 'reference_glue.json').write_text(json.dumps(meta, indent=0) + '\n')
        np.savez_compressed(OUT / 'reference_glue.npz', **arrays)
        (OUT / 'reference_unit_tests.json').write_text(json.dumps(unit_tests_fixture(ref_root), separators=(',', ':')) + '\n')
        (OUT / 'reference_streams.json').write_text(json.dumps(streams_fixture(ref_root, models), separators=(',', ':')) + '\n')
    for f in ('audioA_24k_4s.wav', 'reference_config.yaml', 'reference_glue.json', 'reference_glue.npz', 'reference_unit_tests.json', 'reference_streams.json'):
        print(f, (OUT / f).stat().st_size, 'bytes')


if __name__ == '__main__':
    main()
