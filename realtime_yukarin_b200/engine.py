"""ctypes binding of libryk.so (include/ryk.h): the only door between the Python host layer and
the CUDA hot path.  There is NO CPU fallback: if the shared object is missing, cannot be loaded, or
no B200 is visible, every call raises.
"""
import os as _os

# must be in the environment before the CUDA context exists (see ryk_engine_create): many independent streams need their own hardware queues
_os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

import ctypes
import os
import threading
from pathlib import Path
from typing import Dict, List, Optional, Sequence

import numpy

from .world_consts import cheaptrick_fft_size, dio_num_frames  # noqa: F401  (re-exported)

_CSRC = Path(__file__).resolve().parent / 'csrc'
_LIB_PATH = Path(os.environ['RYK_LIB']) if os.environ.get('RYK_LIB') else _CSRC / 'libryk.so'     # RYK_LIB: diagnostics builds

c_int_p = ctypes.POINTER(ctypes.c_int)
c_float_p = ctypes.POINTER(ctypes.c_float)
c_double_p = ctypes.POINTER(ctypes.c_double)
c_u8_p = ctypes.POINTER(ctypes.c_uint8)


class RykError(RuntimeError):
    pass


class SessionConfig(ctypes.Structure):
    _fields_ = [
        ('fs', ctypes.c_int), ('frame_period_ms', ctypes.c_double), ('f0_floor', ctypes.c_double),
        ('f0_ceil', ctypes.c_double), ('fft_length', ctypes.c_int), ('order', ctypes.c_int),
        ('alpha', ctypes.c_double), ('buffer_time', ctypes.c_double), ('encode_extra_time', ctypes.c_double),
        ('convert_extra_time', ctypes.c_double), ('decode_extra_time', ctypes.c_double),
        ('threshold_db', ctypes.c_double), ('vocoder_buffer_size', ctypes.c_int),
    ]


_lib = None
_lib_lock = threading.Lock()

# every symbol include/ryk.h declares (tests check that the library exports all of them)
EXPORTED_SYMBOLS = [
    'ryk_abi_version', 'ryk_last_error', 'ryk_engine_create', 'ryk_engine_destroy', 'ryk_engine_set_precision',
    'ryk_engine_get_precision', 'ryk_engine_launch_count', 'ryk_engine_synchronize', 'ryk_world_analyze', 'ryk_world_f0',
    'ryk_world_num_frames', 'ryk_silence_mask', 'ryk_model_create', 'ryk_model_set_layer', 'ryk_model_layer_shape',
    'ryk_stage1_set_stats', 'ryk_f0_set_stats', 'ryk_stage1_convert', 'ryk_f0_convert', 'ryk_mc2sp',
    'ryk_stage2_convert', 'ryk_convert_window', 'ryk_synth_create', 'ryk_synth_destroy', 'ryk_synth_add_parameters',
    'ryk_synth_synthesis2', 'ryk_synth_decode', 'ryk_session_create', 'ryk_session_destroy', 'ryk_session_push',
    'ryk_session_push_device', 'ryk_session_submit', 'ryk_session_collect', 'ryk_group_create', 'ryk_group_destroy',
    'ryk_group_size', 'ryk_session_stage_times', 'ryk_group_submit', 'ryk_group_collect', 'ryk_group_push_device', 'ryk_test_conv_layer', 'ryk_debug_dio', 'ryk_debug_stonemask', 'ryk_debug_synth_pulses', 'ryk_debug_synth_timebase', 'ryk_engine_profile', 'ryk_engine_profile_read', 'ryk_engine_timer_start', 'ryk_engine_timer_stop',
    'ryk_world_synthesize_length', 'ryk_world_synthesize', 'ryk_output_gate', 'ryk_reblock_create', 'ryk_reblock_destroy',
    'ryk_reblock_push', 'ryk_reblock_push_device', 'ryk_reblock_collect', 'ryk_reblock_result_device', 'ryk_resample_length',
    'ryk_resample_poly', 'ryk_session_poll', 'ryk_reblock_poll', 'ryk_engine_profile_read2', 'ryk_engine_set_stage1_fused',
    'ryk_engine_set_f0_method', 'ryk_engine_get_f0_method', 'ryk_debug_harvest', 'ryk_debug_stage1_bench',
    'ryk_crepe_create', 'ryk_crepe_set_conv', 'ryk_crepe_set_dense', 'ryk_crepe_set_decoder_tables', 'ryk_crepe_num_frames', 'ryk_crepe_predict',
]


def load_library() -> ctypes.CDLL:
    """dlopen csrc/libryk.so (built by __graft_entry__.build() / csrc/build.sh)."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not _LIB_PATH.exists():
                raise RykError(f'{_LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                               f'(the hot path has no CPU fallback)')
            # RYK_LIB: a diagnostics build of the same library (e.g. -DRYK_TC_TIMELINE); never a different implementation
            lib = ctypes.CDLL(os.environ.get('RYK_LIB') or str(_LIB_PATH))
            lib.ryk_last_error.restype = ctypes.c_char_p
            lib.ryk_engine_launch_count.restype = ctypes.c_longlong
            _lib = lib
    return _lib


def _f32(a) -> numpy.ndarray:
    return numpy.ascontiguousarray(a, dtype=numpy.float32)


def _fp(a: numpy.ndarray):
    return a.ctypes.data_as(c_float_p)


def _dp(a: numpy.ndarray):
    return a.ctypes.data_as(c_double_p)


def _bp(a: numpy.ndarray):
    return a.ctypes.data_as(c_u8_p)


class Engine(object):
    """One per process per GPU (not thread-safe, like the reference's single-threaded stages)."""

    def __init__(self, device: Optional[int] = None):
        self.lib = load_library()
        if device is None:
            device = int(os.environ.get('LOCAL_RANK', '0'))
        self.device = device
        h = ctypes.c_void_p()
        self._check(self.lib.ryk_engine_create(ctypes.c_int(device), ctypes.byref(h)))
        self._h = h
        self._synth_block = {}
        self._reblock_chunk = {}           # re-blocker id -> out_audio_chunk

    # ---- plumbing ----
    def _check(self, rc: int):
        if rc < 0:
            raise RykError(self.lib.ryk_last_error().decode('utf-8', 'replace'))
        return rc

    def close(self):
        if getattr(self, '_h', None):
            self.lib.ryk_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_precision(self, mode: str):
        self._check(self.lib.ryk_engine_set_precision(self._h, {'fp32': 0, 'fp16': 1}[mode]))

    def set_stage1_fused(self, enable: bool) -> int:
        """Stage 1 as one cluster kernel (default) or as 16 layer launches; returns the cluster size (<= 0: unavailable)."""
        return int(self.lib.ryk_engine_set_stage1_fused(self._h, 1 if enable else 0))

    @property
    def precision(self) -> str:
        return ['fp32', 'fp16'][self.lib.ryk_engine_get_precision(self._h)]

    @property
    def launch_count(self) -> int:
        return int(self.lib.ryk_engine_launch_count(self._h))

    def timer_start(self):
        self._check(self.lib.ryk_engine_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = ctypes.c_float()
        self._check(self.lib.ryk_engine_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    def profile(self, enable: bool):
        self._check(self.lib.ryk_engine_profile(self._h, int(bool(enable))))

    def profile_read(self):
        ms, runs = ctypes.c_double(), ctypes.c_int()
        self._check(self.lib.ryk_engine_profile_read(self._h, ctypes.byref(ms), ctypes.byref(runs)))
        return ms.value, runs.value

    def profile_read2(self):
        """(sum of per-forward durations ms, union of the intervals ms, forwards) of the stage-2 k4 block since the last read."""
        tot, uni, runs = ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
        self._check(self.lib.ryk_engine_profile_read2(self._h, ctypes.byref(tot), ctypes.byref(uni), ctypes.byref(runs)))
        return tot.value, uni.value, runs.value

    def synchronize(self):
        self._check(self.lib.ryk_engine_synchronize(self._h))

    # ---- WORLD analysis ----
    def world_f0(self, x, fs, frame_period, f0_floor, f0_ceil):
        x = _f32(x)
        n = dio_num_frames(fs, len(x), frame_period)
        f0 = numpy.empty(n, dtype=numpy.float64)
        t = numpy.empty(n, dtype=numpy.float64)
        self._check(self.lib.ryk_world_f0(self._h, _fp(x), len(x), int(fs), ctypes.c_double(frame_period),
                                          ctypes.c_double(f0_floor), ctypes.c_double(f0_ceil), _dp(f0), _dp(t)))
        return f0, t

    def world_analyze(self, x, fs, frame_period, f0_floor, f0_ceil, fft_length, order, alpha, f0=None) -> Dict[str, numpy.ndarray]:
        x = _f32(x)
        hop = int(fs * frame_period / 1000)
        T = len(x) // hop
        nb = fft_length // 2 + 1
        out = dict(
            f0=numpy.zeros(T, dtype=numpy.float32), sp=numpy.zeros((T, nb), dtype=numpy.float32),
            ap=numpy.zeros((T, nb), dtype=numpy.float32), mc=numpy.zeros((T, order + 1), dtype=numpy.float32),
            voiced=numpy.zeros(T, dtype=numpy.uint8))
        f0_arg = None
        if f0 is not None:
            nw = dio_num_frames(fs, len(x), frame_period)
            f0_full = numpy.zeros(nw, dtype=numpy.float64)
            f0_full[:min(nw, len(f0))] = numpy.asarray(f0, dtype=numpy.float64).ravel()[:nw]
            f0_arg = _dp(f0_full)
        if T > 0:
            self._check(self.lib.ryk_world_analyze(
                self._h, _fp(x), len(x), int(fs), ctypes.c_double(frame_period), ctypes.c_double(f0_floor),
                ctypes.c_double(f0_ceil), int(fft_length), int(order), ctypes.c_double(alpha), f0_arg,
                _fp(out['f0']), _fp(out['sp']), _fp(out['ap']), _fp(out['mc']), _bp(out['voiced'])))
        out['voiced'] = out['voiced'].astype(bool)
        return out

    # ---- silence gate ----
    def silence_mask(self, wave, frame_length, hop, threshold_db, n_frames) -> numpy.ndarray:
        w = _f32(wave)
        mask = numpy.zeros(n_frames, dtype=numpy.uint8)
        thr = -1.0 if threshold_db is None else float(threshold_db)
        self._check(self.lib.ryk_silence_mask(self._h, _fp(w), len(w), int(frame_length), int(hop), ctypes.c_double(thr),
                                              int(n_frames), _bp(mask)))
        return mask.astype(bool)

    # ---- models ----
    def model_create(self, stage: int, in_channels: int, out_channels: int, base_channels: int):
        self._check(self.lib.ryk_model_create(self._h, stage, in_channels, out_channels, base_channels))

    def model_layer_shape(self, stage: int, layer: int):
        tr, cin, cout, k = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        self._check(self.lib.ryk_model_layer_shape(self._h, stage, layer, ctypes.byref(tr), ctypes.byref(cin),
                                                   ctypes.byref(cout), ctypes.byref(k)))
        return bool(tr.value), cin.value, cout.value, k.value

    def model_set_layer(self, stage: int, layer: int, W, scale, shift):
        W, scale, shift = _f32(W), _f32(scale), _f32(shift)
        self._check(self.lib.ryk_model_set_layer(self._h, stage, layer, _fp(W), _fp(scale), _fp(shift)))

    def stage1_set_stats(self, in_mean, in_std, out_mean, out_std):
        a, b, c, d = _f32(in_mean), _f32(in_std), _f32(out_mean), _f32(out_std)
        self._check(self.lib.ryk_stage1_set_stats(self._h, len(a), _fp(a), _fp(b), _fp(c), _fp(d)))

    def f0_set_stats(self, in_mean, in_std, target_mean, target_std):
        self._check(self.lib.ryk_f0_set_stats(self._h, ctypes.c_double(in_mean), ctypes.c_double(in_std),
                                              ctypes.c_double(target_mean), ctypes.c_double(target_std)))

    def stage1_convert(self, x) -> numpy.ndarray:
        x = _f32(x)
        y = numpy.empty_like(x)
        self._check(self.lib.ryk_stage1_convert(self._h, _fp(x), x.shape[0], _fp(y)))
        return y

    def f0_convert(self, f0, voiced) -> numpy.ndarray:
        f = _f32(numpy.asarray(f0).ravel())
        v = numpy.ascontiguousarray(numpy.asarray(voiced).ravel(), dtype=numpy.uint8)
        out = numpy.empty_like(f)
        self._check(self.lib.ryk_f0_convert(self._h, _fp(f), _bp(v), len(f), _fp(out)))
        return out

    def mc2sp(self, mc, alpha, fftlen) -> numpy.ndarray:
        mc = _f32(mc)
        sp = numpy.empty((mc.shape[0], fftlen // 2 + 1), dtype=numpy.float64)
        if mc.shape[0]:
            self._check(self.lib.ryk_mc2sp(self._h, _fp(mc), mc.shape[0], mc.shape[1] - 1, ctypes.c_double(alpha), int(fftlen), _dp(sp)))
        return sp

    def stage2_convert(self, sp) -> numpy.ndarray:
        sp = _f32(sp)
        out = numpy.empty_like(sp)
        self._check(self.lib.ryk_stage2_convert(self._h, _fp(sp), sp.shape[0], _fp(out)))
        return out

    def convert_window(self, wave, fs, frame_length, hop, threshold_db, f0, ap, mc, voiced, order, alpha, fftlen):
        wave, f0, ap, mc = _f32(wave), _f32(numpy.asarray(f0).ravel()), _f32(ap), _f32(mc)
        v = numpy.ascontiguousarray(numpy.asarray(voiced).ravel(), dtype=numpy.uint8)
        T, nb = len(f0), fftlen // 2 + 1
        out = dict(f0=numpy.empty(T, numpy.float32), ap=numpy.empty((T, nb), numpy.float32), sp=numpy.empty((T, nb), numpy.float32),
                   voiced=numpy.empty(T, numpy.uint8), mc=numpy.empty((T, order + 1), numpy.float32))
        thr = -1.0 if threshold_db is None else float(threshold_db)
        self._check(self.lib.ryk_convert_window(
            self._h, _fp(wave), len(wave), int(fs), int(frame_length), int(hop), ctypes.c_double(thr),
            _fp(f0), _fp(ap), _fp(mc), _bp(v), T, int(order), ctypes.c_double(alpha), int(fftlen),
            _fp(out['f0']), _fp(out['ap']), _fp(out['sp']), _bp(out['voiced']), _fp(out['mc'])))
        out['voiced'] = out['voiced'].astype(bool)
        return out

    # ---- synthesizer ----
    def synth_create(self, fs, frame_period, fft_size, buffer_size, number_of_pointers=16) -> int:
        sid = ctypes.c_int()
        self._check(self.lib.ryk_synth_create(self._h, int(fs), ctypes.c_double(frame_period), int(fft_size), int(buffer_size),
                                              int(number_of_pointers), ctypes.byref(sid)))
        self._synth_block[sid.value] = (int(buffer_size), int(fft_size), float(fs) * float(frame_period) / 1000.0)
        return sid.value

    def synth_destroy(self, sid: int):
        self._check(self.lib.ryk_synth_destroy(self._h, sid))

    def synth_add_parameters(self, sid, f0, sp, ap) -> int:
        f0 = numpy.ascontiguousarray(numpy.asarray(f0).ravel(), dtype=numpy.float64)
        sp, ap = _f32(sp), _f32(ap)
        return self._check(self.lib.ryk_synth_add_parameters(self._h, sid, _dp(f0), len(f0), _fp(sp), _fp(ap)))

    def synth_synthesis2(self, sid):
        B = self._synth_block[sid][0]
        buf = numpy.empty(B, dtype=numpy.float64)
        ok = self._check(self.lib.ryk_synth_synthesis2(self._h, sid, _dp(buf)))
        return buf if ok else None

    def synth_decode(self, sid, f0, sp, ap, max_blocks=None) -> numpy.ndarray:
        f0 = numpy.ascontiguousarray(numpy.asarray(f0).ravel(), dtype=numpy.float64)
        sp, ap = _f32(sp), _f32(ap)
        B = self._synth_block[sid][0]
        if max_blocks is None:
            # samples one call can add = frames * (fs * frame_period / 1000) of THIS synthesizer (not a fixed 240 per frame): the
            # reference loops `while _Synthesis2() != 0` until the synthesizer is empty (vocoder.py:103-116)
            max_blocks = max(4, int(len(f0) * self._synth_block[sid][2]) // B + 4)
        out = numpy.empty(max_blocks * B, dtype=numpy.float64)
        nblk = ctypes.c_int()
        self._check(self.lib.ryk_synth_decode(self._h, sid, _dp(f0), len(f0), _fp(sp), _fp(ap), _dp(out), int(max_blocks), ctypes.byref(nblk)))
        return out[:nblk.value * B].copy()

    # ---- offline synthesis (pyworld.synthesize) and the output silence gate / re-blocker ----
    def world_synthesize(self, f0, sp, ap, fs, frame_period, fft_size=None, return_pulses=False):
        """Vocoder.decode's pyworld.synthesize (vocoder.py:50-62): (T,) f0, (T, nb) sp / ap -> float64 wave."""
        f0 = numpy.ascontiguousarray(numpy.asarray(f0).ravel(), dtype=numpy.float64)
        sp, ap = _f32(sp), _f32(ap)
        if fft_size is None:
            fft_size = (sp.shape[1] - 1) * 2
        n = self.lib.ryk_world_synthesize_length(len(f0), ctypes.c_double(frame_period), int(fs))
        y = numpy.zeros(max(n, 1), dtype=numpy.float64)
        cap = max(n, 1) if return_pulses else 1
        idx = numpy.zeros(cap, numpy.int64); shift = numpy.zeros(cap); vuv = numpy.zeros(cap, numpy.int32)
        ny, npulse = ctypes.c_int(), ctypes.c_int()
        self._check(self.lib.ryk_world_synthesize(
            self._h, _dp(f0), len(f0), _fp(sp), _fp(ap), int(fs), ctypes.c_double(frame_period), int(fft_size), _dp(y), len(y), ctypes.byref(ny),
            idx.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), _dp(shift), vuv.ctypes.data_as(c_int_p), cap if return_pulses else 0,
            ctypes.byref(npulse)))
        y = y[:ny.value]
        if return_pulses:
            k = min(npulse.value, cap)
            return y, idx[:k], shift[:k], vuv[:k]
        return y

    def output_gate(self, wave, threshold_db, n_fft=2048, hop=512):
        """(mean STFT power in dB, keep?) of one output chunk (decode_worker.py:56-58)."""
        w = numpy.ascontiguousarray(numpy.asarray(wave).ravel(), dtype=numpy.float64)
        pw, ok = ctypes.c_double(), ctypes.c_int()
        self._check(self.lib.ryk_output_gate(self._h, _dp(w), len(w), int(n_fft), int(hop), ctypes.c_double(threshold_db), ctypes.byref(pw),
                                             ctypes.byref(ok)))
        return pw.value, bool(ok.value)

    def reblock_create(self, out_audio_chunk, max_in, threshold_db, n_fft=2048, hop=512) -> int:
        rid = ctypes.c_int()
        self._check(self.lib.ryk_reblock_create(self._h, int(out_audio_chunk), int(max_in), int(n_fft), int(hop), ctypes.c_double(threshold_db),
                                                ctypes.byref(rid)))
        self._reblock_chunk[rid.value] = int(out_audio_chunk)
        return rid.value

    def reblock_destroy(self, rid: int):
        self._check(self.lib.ryk_reblock_destroy(self._h, rid))

    def reblock_push(self, rid: int, wave):
        """Host samples in; returns (status, chunk or None, power_db): status 0 none, 1 chunk, 2 silent chunk (dropped)."""
        w = numpy.ascontiguousarray(numpy.asarray(wave).ravel(), dtype=numpy.float64)
        out = numpy.empty(self._reblock_chunk[rid], dtype=numpy.float64)
        st, pw = ctypes.c_int(), ctypes.c_double()
        self._check(self.lib.ryk_reblock_push(self._h, rid, _dp(w), len(w), _dp(out), ctypes.byref(st), ctypes.byref(pw)))
        return st.value, (out if st.value == 1 else None), pw.value

    def reblock_push_device(self, rid: int, session_id: int = -1, wave_dev_ptr: int = 0, n_dev_ptr: int = 0) -> int:
        ticket = ctypes.c_longlong()
        self._check(self.lib.ryk_reblock_push_device(self._h, rid, int(session_id), ctypes.c_void_p(wave_dev_ptr or None),
                                                     ctypes.c_void_p(n_dev_ptr or None), ctypes.byref(ticket)))
        return ticket.value

    def reblock_collect(self, rid: int, ticket: int):
        out = numpy.empty(self._reblock_chunk[rid], dtype=numpy.float64)
        st, pw = ctypes.c_int(), ctypes.c_double()
        self._check(self.lib.ryk_reblock_collect(self._h, rid, ctypes.c_longlong(ticket), _dp(out), ctypes.byref(st), ctypes.byref(pw)))
        return st.value, (out if st.value == 1 else None), pw.value

    def reblock_poll(self, rid: int, ticket: int) -> bool:
        done = ctypes.c_int()
        self._check(self.lib.ryk_reblock_poll(self._h, rid, ctypes.c_longlong(ticket), ctypes.byref(done)))
        return bool(done.value)

    def resample_poly(self, x, up: int, down: int, taps) -> numpy.ndarray:
        """scipy.signal.resample_poly's filtering step on the device (wave_io.resample designs `taps`)."""
        x = _f32(x)
        taps = numpy.ascontiguousarray(taps, dtype=numpy.float64)
        n = self.lib.ryk_resample_length(len(x), int(up), int(down))
        y = numpy.empty(max(n, 1), dtype=numpy.float32)
        no = ctypes.c_int()
        self._check(self.lib.ryk_resample_poly(self._h, _fp(x), len(x), int(up), int(down), _dp(taps), len(taps), _fp(y), len(y), ctypes.byref(no)))
        return y[:no.value]

    # ---- diagnostics ----
    def debug_synth_pulses(self, sid, first=0, count=None):
        st = numpy.zeros(7, numpy.int64)
        z = numpy.zeros(1, numpy.int64); zd = numpy.zeros(1); zi = numpy.zeros(1, numpy.int32)
        self._check(self.lib.ryk_debug_synth_pulses(self._h, sid, ctypes.c_longlong(0), 0, z.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)),
                                                    _dp(zd), zi.ctypes.data_as(c_int_p), st.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))))
        if count is None:
            count = int(st[0]) - first
        idx = numpy.zeros(max(count, 1), numpy.int64); tm = numpy.zeros(max(count, 1)); vuv = numpy.zeros(max(count, 1), numpy.int32)
        self._check(self.lib.ryk_debug_synth_pulses(self._h, sid, ctypes.c_longlong(first), count, idx.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)),
                                                    _dp(tm), vuv.ctypes.data_as(c_int_p), st.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))))
        return idx[:count], tm[:count], vuv[:count], st

    def debug_synth_timebase(self, sid, n):
        a, b, c = numpy.zeros(n), numpy.zeros(n), numpy.zeros(n)
        self._check(self.lib.ryk_debug_synth_timebase(self._h, sid, int(n), _dp(a), _dp(b), _dp(c)))
        return a, b, c

    F0_METHODS = {'dio': 0, 'harvest': 1}

    def set_f0_method(self, method: str):
        """f0 extractor of world_f0 / world_analyze / sessions created afterwards: 'dio' (pyworld.dio + stonemask, default) or
        'harvest' (pyworld.harvest + stonemask) -- yukarin's AcousticFeature.extract f0 hook (acoustic_feature_wrapper.py:28-33)."""
        self._check(self.lib.ryk_engine_set_f0_method(self._h, self.F0_METHODS[method]))

    @property
    def f0_method(self) -> str:
        return ['dio', 'harvest'][self.lib.ryk_engine_get_f0_method(self._h)]

    def debug_harvest(self, n, fs, frame_period, f0_floor, f0_ceil):
        """Intermediate arrays of the last Harvest analysis with this plan (see ryk_debug_harvest)."""
        import math
        ratio = int(fs / 8000.0 + 0.5)
        channels = 1 + int(math.log((f0_ceil * 1.1) / (f0_floor * 0.9)) / 0.69314718055994529 * 40.0)
        nf1 = int(1000.0 * n / fs) + 1
        ylen = -(-n // ratio)
        maxc = int(channels / 10.0 + 0.5) * 7
        info = numpy.zeros(7, numpy.int32)
        out = dict(y=numpy.zeros(ylen), raw=numpy.zeros((channels, nf1)), cand=numpy.zeros((nf1, maxc)), score=numpy.zeros((nf1, maxc)),
                   best=numpy.zeros(nf1), basic=numpy.zeros(nf1), f0_raw=numpy.zeros(dio_num_frames(fs, n, frame_period)))
        self._check(self.lib.ryk_debug_harvest(self._h, int(n), int(fs), ctypes.c_double(frame_period), ctypes.c_double(f0_floor),
                                               ctypes.c_double(f0_ceil), info.ctypes.data_as(c_int_p), _dp(out['y']), _dp(out['raw']),
                                               _dp(out['cand']), _dp(out['score']), _dp(out['best']), _dp(out['basic']), _dp(out['f0_raw'])))
        assert (info[0], info[1], info[2], info[4]) == (channels, nf1, ylen, maxc), info
        out['nc'] = int(info[6])
        return out

    def stage1_bench(self, Tp: int, iters: int = 50):
        """(ms per stand-alone stage-1 forward fused, layered, fused-kernel phase timeline in us)."""
        a, b = ctypes.c_float(), ctypes.c_float()
        tl = numpy.zeros(31)
        self._check(self.lib.ryk_debug_stage1_bench(self._h, int(Tp), int(iters), ctypes.byref(a), ctypes.byref(b), _dp(tl)))
        return float(a.value), float(b.value), tl

    def debug_dio(self, n, fs, frame_period, f0_floor, f0_ceil):
        nf = dio_num_frames(fs, n, frame_period)
        nbands = 1 + int(numpy.log(f0_ceil / f0_floor) / 0.69314718055994529 * 2.0)
        f0 = numpy.empty(nf); cand = numpy.empty((nbands, nf)); score = numpy.empty((nbands, nf)); counts = numpy.empty((nbands, 4), numpy.int32)
        self._check(self.lib.ryk_debug_dio(self._h, int(n), int(fs), ctypes.c_double(frame_period), ctypes.c_double(f0_floor),
                                           ctypes.c_double(f0_ceil), _dp(f0), _dp(cand), _dp(score), counts.ctypes.data_as(c_int_p)))
        return f0, cand, score, counts

    def debug_stonemask(self, x, fs, frame_period, f0_floor, f0_in):
        """StoneMask alone on the given f0 estimates (one per frame), shared memory sized from f0_floor as in analysis."""
        x = _f32(x)
        f0_in = numpy.ascontiguousarray(f0_in, dtype=numpy.float64)
        f0 = numpy.empty(len(f0_in))
        self._check(self.lib.ryk_debug_stonemask(self._h, _fp(x), len(x), int(fs), ctypes.c_double(frame_period),
                                                 ctypes.c_double(f0_floor), _dp(f0_in), len(f0_in), _dp(f0)))
        return f0

    def test_conv_layer(self, in0, in1, W, scale, shift, transposed, k, stride, pad, act, use_tc, repeat=0):
        """One conv layer in isolation; in0/in1 NHWC float32, W in the Chainer layout. Returns (out NHWC, ms per run)."""
        in0 = _f32(in0)
        B, H, Wd, C0 = in0.shape
        C1 = 0 if in1 is None else in1.shape[3]
        in1a = _f32(in1) if in1 is not None else numpy.zeros(1, numpy.float32)
        W, scale, shift = _f32(W), _f32(scale), _f32(shift)
        cout = W.shape[1] if transposed else W.shape[0]
        if H == 1:
            Ho = 1
        else:
            Ho = (H - 1) * stride + k - 2 * pad if transposed else (H + 2 * pad - k) // stride + 1
        Wo = (Wd - 1) * stride + k - 2 * pad if transposed else (Wd + 2 * pad - k) // stride + 1
        out = numpy.empty((B, Ho, Wo, cout), numpy.float32)
        ms = ctypes.c_float()
        self._check(self.lib.ryk_test_conv_layer(
            self._h, int(transposed), int(k), int(stride), int(pad), B, H, Wd, C0, C1, cout, _fp(in0), _fp(in1a), _fp(W),
            _fp(scale), _fp(shift), int(act), int(use_tc), int(repeat), _fp(out), ctypes.byref(ms)))
        return out, ms.value

    # ---- sessions ----
    def session_create(self, cfg: SessionConfig) -> int:
        sid = ctypes.c_int()
        self._check(self.lib.ryk_session_create(self._h, ctypes.byref(cfg), ctypes.byref(sid)))
        return sid.value

    def session_destroy(self, sid: int):
        self._check(self.lib.ryk_session_destroy(self._h, sid))

    def session_push(self, sid: int, wave, out: Optional[numpy.ndarray] = None) -> numpy.ndarray:
        w = _f32(wave)
        if out is None:
            out = numpy.empty(len(w) * 2 + 8192, dtype=numpy.float64)
        n_out = ctypes.c_int()
        self._check(self.lib.ryk_session_push(self._h, sid, _fp(w), len(w), _dp(out), len(out), ctypes.byref(n_out)))
        return out[:n_out.value]

    def session_submit(self, sid: int, wave) -> int:
        w = _f32(wave)
        ticket = ctypes.c_longlong()
        self._check(self.lib.ryk_session_submit(self._h, sid, _fp(w), len(w), ctypes.byref(ticket)))
        return ticket.value

    def session_collect(self, sid: int, ticket: int, out: numpy.ndarray) -> numpy.ndarray:
        n_out = ctypes.c_int()
        self._check(self.lib.ryk_session_collect(self._h, sid, ctypes.c_longlong(ticket), _dp(out), len(out), ctypes.byref(n_out)))
        return out[:n_out.value]

    def session_poll(self, sid: int, ticket: int) -> bool:
        """True when session_collect(ticket) would return without waiting (cudaEventQuery, never blocks)."""
        done = ctypes.c_int()
        self._check(self.lib.ryk_session_poll(self._h, sid, ctypes.c_longlong(ticket), ctypes.byref(done)))
        return bool(done.value)

    def session_push_device(self, sid: int, wave_dev_ptr: int, n: int, out_dev_ptr: int, out_capacity: int, n_out_dev_ptr: int):
        self._check(self.lib.ryk_session_push_device(self._h, sid, ctypes.c_void_p(wave_dev_ptr), int(n), ctypes.c_void_p(out_dev_ptr),
                                                     int(out_capacity), ctypes.c_void_p(n_out_dev_ptr)))

    def session_stage_times(self, sid: int):
        """(start, end) arrays of shape (steps, 5) in ms; see ryk_session_stage_times."""
        st, en = (ctypes.c_float * 40)(), (ctypes.c_float * 40)()
        n = self._check(self.lib.ryk_session_stage_times(self._h, sid, st, en))
        return numpy.array(st[:n * 5]).reshape(n, 5), numpy.array(en[:n * 5]).reshape(n, 5)

    # ---- groups (several streams per GPU, one batched stage-2 forward per step) ----
    def group_create(self, session_ids: Sequence[int]) -> int:
        ids = (ctypes.c_int * len(session_ids))(*[int(i) for i in session_ids])
        gid = ctypes.c_int()
        self._check(self.lib.ryk_group_create(self._h, ids, len(session_ids), ctypes.byref(gid)))
        return gid.value

    def group_destroy(self, gid: int):
        self._check(self.lib.ryk_group_destroy(self._h, gid))

    def group_size(self, gid: int) -> int:
        return self._check(self.lib.ryk_group_size(self._h, gid))

    def group_submit(self, gid: int, waves: Sequence) -> int:
        ws = [_f32(w) for w in waves]
        ptrs = (ctypes.POINTER(ctypes.c_float) * len(ws))(*[_fp(w) for w in ws])
        ticket = ctypes.c_longlong()
        self._check(self.lib.ryk_group_submit(self._h, gid, ptrs, len(ws[0]), ctypes.byref(ticket)))
        return ticket.value

    def group_collect(self, gid: int, ticket: int, outs: Sequence[numpy.ndarray]) -> List[numpy.ndarray]:
        ptrs = (ctypes.POINTER(ctypes.c_double) * len(outs))(*[_dp(o) for o in outs])
        n_outs = (ctypes.c_int * len(outs))()
        self._check(self.lib.ryk_group_collect(self._h, gid, ctypes.c_longlong(ticket), ptrs, min(len(o) for o in outs), n_outs))
        return [o[:n] for o, n in zip(outs, n_outs)]

    def group_push(self, gid: int, waves: Sequence) -> List[numpy.ndarray]:
        outs = [numpy.empty(len(waves[0]) * 2 + 8192, dtype=numpy.float64) for _ in waves]
        return self.group_collect(gid, self.group_submit(gid, waves), outs)

    def group_push_device(self, gid: int, wave_dev_ptrs: Sequence[int], n: int, out_dev_ptrs: Sequence[int], out_capacity: int,
                          n_out_dev_ptrs: Sequence[int]):
        B = len(wave_dev_ptrs)
        w = (ctypes.c_void_p * B)(*[int(p) for p in wave_dev_ptrs])
        o = (ctypes.c_void_p * B)(*[int(p) for p in out_dev_ptrs])
        c = (ctypes.c_void_p * B)(*[int(p) for p in n_out_dev_ptrs])
        self._check(self.lib.ryk_group_push_device(self._h, gid, w, int(n), o, int(out_capacity), c))



_default: Optional[Engine] = None


def default_engine() -> Engine:
    """Process-wide engine on cuda:LOCAL_RANK (created on first use)."""
    global _default
    if _default is None:
        _default = Engine()
    return _default


def set_default_engine(engine: Optional[Engine]):
    global _default
    _default = engine
