"""Layer-by-layer timing of the stage-2 k4 layers: per-tap kernel (RYK_TC3=0), the default choice, and the halo kernel with M = 128 / 256.
Usage (GPU box): python tools/gpu_bench_halo.py [TP=384] ; prints one table, no correctness check (tests do that)."""
import os, sys; sys.path.insert(0, '.')
import numpy as np
from realtime_yukarin_b200.engine import default_engine
eng = default_engine()
rng = np.random.default_rng(0)
Tp, base, B = int(os.environ.get('TP', 384)), 64, int(os.environ.get('BATCH', 1))
enc = [1, 2, 4, 8, 8, 8, 8, 8]; dec = [8, 8, 8, 8, 4, 2, 1]
layers = []
for i in range(1, 8):
    layers.append((f'c{i}', 0, Tp >> (i - 1), 512 >> (i - 1), base * enc[i - 1], 0, base * enc[i]))
for d in range(7):
    c0 = base * enc[7] if d == 0 else base * dec[d - 1]
    c1 = 0 if d == 0 else base * enc[7 - d]
    layers.append((f'd{d}', 1, Tp >> (7 - d), 512 >> (7 - d), c0, c1, base * dec[d]))
only = os.environ.get('LAYERS')
configs = [('per-tap', dict(RYK_TC3='0')), ('default', dict())]
for mt in (1, 2):
    configs.append((f'persist mt{mt}', dict(RYK_TC3='2', RYK_TC3_MT=str(mt))))
keys = ('RYK_TC3', 'RYK_TC3_MT', 'RYK_TC3_TW')
print('layer      GFLOP ' + ' '.join(f'{n:>13s}' for n, _ in configs))
tot = np.zeros(len(configs)); totf = 0.0
for name, tr, H, W, C0, C1, Cout in layers:
    if only and name not in only.split(','):
        continue
    in0 = rng.standard_normal((B, H, W, C0)).astype(np.float32)
    in1 = rng.standard_normal((B, H, W, C1)).astype(np.float32) if C1 else None
    Cin = C0 + C1
    shape = (Cin, Cout, 4, 4) if tr else (Cout, Cin, 4, 4)
    Wt = (rng.standard_normal(shape) / np.sqrt(Cin * 16 / (4 if tr else 1))).astype(np.float32)
    fl = 2.0 * 16 * Cin * Cout * B * (H * W if tr else H * W // 4)
    row = []
    ref = None
    for ci, (cname, env) in enumerate(configs):
        for k in keys:
            os.environ.pop(k, None)
        os.environ.update(env)
        try:
            out, ms = eng.test_conv_layer(in0, in1, Wt, np.ones(Cout, np.float32), np.zeros(Cout, np.float32), tr, 4, 2, 1, 1, use_tc=1, repeat=20)
            if ref is None:
                ref = out
            bad = float(np.abs(out - ref).max())
            row.append(f'{ms * 1e3:6.1f}us {fl / ms / 1e9:5.0f}' + ('!' if bad > 2e-2 else ' '))
            tot[ci] += ms
        except Exception as exc:
            row.append(f'{"ERR":>13s}')
            print('   ', cname, name, str(exc)[:150], file=sys.stderr)
    totf += fl
    print(f'{name:8s} {fl / 1e9:7.2f} ' + ' '.join(row), flush=True)
print('TOTAL us          ' + ' '.join(f'{t * 1e3:13.1f}' for t in tot))
print('TFLOP/s           ' + ' '.join(f'{(totf / t / 1e9 if t > 0 else 0):13.1f}' for t in tot))
