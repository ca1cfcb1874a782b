"""Stand-alone timing of the WORLD analysis kernels (k_stonemask, k_cheaptrick, k_d4c) on one 0.3 s chunk at 24 kHz, and a dump of
the analysis outputs on seeded inputs, so that two builds of libryk can be compared kernel for kernel and output for output.

usage:
  RYK_LIB=<lib> python tools/gpu_bench_analysis.py --reps 300 --json OUT.json [--dump OUT.npz]
      per-kernel mean device time (torch.profiler, CUDA activities) over --reps world_analyze calls; one process per library
  python tools/gpu_bench_analysis.py --compare A.npz B.npz
      f0 / voiced bit-for-bit, ap max relative difference
  RYK_LIB=<-DRYK_D4C_TIMELINE build> RYK_D4C_TIMELINE_FILE=F python tools/gpu_bench_analysis.py --timeline-runs 20
  python tools/gpu_bench_analysis.py --timeline-summary F
      median duration of each k_d4c phase over the voiced frames of every launch
"""
import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

KERNELS = ('k_stonemask', 'k_cheaptrick', 'k_d4c')
# what ends at each timeline slot of k_d4c (world_analysis.cu, D4C_TL)
SLOTS = {1: 'LoveTrain', 2: 'centroid 1', 3: 'centroid 2 + DC correction', 4: 'power spectrum + smoothing',
         5: 'group delay smoothings', 6: 'bands 0+1: window + complex FFT', 7: 'bands 2+3: window + complex FFT',
         8: 'band 4: window + FFT', 9: 'band power spectra', 10: 'radix select + sums', 11: 'coarse aperiodicity',
         15: 'output'}


def _inputs():
    from realtime_yukarin_b200 import synthetic
    from realtime_yukarin_b200.wave_io import read_wav
    xs = {f'speech_{s}s': synthetic.synthetic_speech(s, stream=i) for i, s in enumerate((0.1, 0.3, 1.0))}
    w, fs = read_wav(ROOT / 'tests' / 'golden' / 'audioA_24k_4s.wav')
    assert fs == 24000
    xs['audioA_4s'] = np.asarray(w, np.float32)
    return xs


def _gpu_info():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f'unavailable: {e}'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=300)
    ap.add_argument('--json')
    ap.add_argument('--dump')
    ap.add_argument('--compare', nargs=2)
    ap.add_argument('--timeline-runs', type=int, default=0)
    ap.add_argument('--timeline-summary')
    a = ap.parse_args()
    if a.compare:
        A, B = np.load(a.compare[0]), np.load(a.compare[1])
        res = {}
        for k in sorted({n.rsplit('/', 1)[0] for n in A.files}):
            ra, rb = A[k + '/ap'].astype(np.float64), B[k + '/ap'].astype(np.float64)
            res[k] = dict(f0_bit_identical=bool(np.array_equal(A[k + '/f0'], B[k + '/f0'])),
                          voiced_identical=bool(np.array_equal(A[k + '/voiced'], B[k + '/voiced'])),
                          ap_max_rel=float(np.max(np.abs(ra - rb) / np.maximum(np.abs(ra), 1e-30))),
                          ap_identical=bool(np.array_equal(ra, rb)))
        print(json.dumps(res, indent=1))
        return
    if a.timeline_summary:
        launches, cur = [], None
        for line in open(a.timeline_summary):
            if line.startswith('#'):
                cur = []
                launches.append(cur)
            elif line.strip():
                cur.append([int(v) for v in line.split()])
        rows = np.array([r for L in launches for r in L], dtype=np.float64)
        voiced = rows[(rows[:, 15] > 0) & (rows[:, 2] > 0)]
        cols = [c for c in range(16) if np.all(voiced[:, c] > 0)]
        d = np.diff(voiced[:, cols], axis=1) / 1000.0
        print(f'{len(launches)} launches, {len(rows)} frames, {len(voiced)} voiced (full path); median us per phase:')
        for a_, b_, v in zip(cols[:-1], cols[1:], np.median(d, axis=0)):
            print(f'  slot {a_:2d} -> {b_:2d}  {SLOTS.get(b_, ""):40s} {v:8.2f}')
        print(f'  {"total (voiced frame)":30s} {np.median((voiced[:, 15] - voiced[:, 0]) / 1000.0):8.2f}')
        unv = rows[(rows[:, 1] > 0) & (rows[:, 2] == 0)]
        if len(unv):
            print(f'  {"LoveTrain-only frame":30s} {np.median((unv[:, 1] - unv[:, 0]) / 1000.0):8.2f}  ({len(unv)} frames)')
        return

    import torch
    from oracle import pipeline as opipe
    from realtime_yukarin_b200.engine import default_engine
    cfg = opipe.PathConfig()
    eng = default_engine()
    xs = _inputs()

    def run(x):
        return eng.world_analyze(x, cfg.fs, cfg.frame_period, cfg.f0_floor, cfg.f0_ceil, cfg.fft_length, cfg.order, cfg.alpha)

    if a.timeline_runs:
        for _ in range(a.timeline_runs):
            run(xs['speech_0.3s'])
        run(xs['audioA_4s'])
        return
    if a.dump:
        out = {}
        for k, x in xs.items():
            r = run(x)
            out.update({f'{k}/f0': r['f0'], f'{k}/voiced': r['voiced'], f'{k}/ap': r['ap']})
        np.savez(a.dump, **out)
    x = xs['speech_0.3s']
    for _ in range(20):
        run(x)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.reps):
            run(x)
        torch.cuda.synchronize()
    times = {k: [] for k in KERNELS}
    for ev in prof.events():
        for k in KERNELS:
            if ev.device_type is not None and 'CUDA' in str(ev.device_type) and (k + '(') in ev.name:
                times[k].append(ev.device_time_total if hasattr(ev, 'device_time_total') else ev.cuda_time_total)
    res = dict(lib=os.environ.get('RYK_LIB', 'libryk.so'), gpu=_gpu_info(), reps=a.reps, chunk_s=0.3,
               frames=int(len(x) // cfg.hop),
               kernels={k: dict(launches=len(v), mean_us=float(np.mean(v)) if v else None,
                                median_us=float(np.median(v)) if v else None) for k, v in times.items()})
    if not all(times.values()):
        res['kernel_names_seen'] = sorted({ev.name for ev in prof.events()})[:50]
    print(json.dumps(res))
    if a.json:
        Path(a.json).write_text(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
