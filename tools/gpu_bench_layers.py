"""Times every k4 layer of the stage-2 U-Net (Tp = 384, base 64) through ryk_test_conv_layer (tcgen05 path)."""
import os, sys; sys.path.insert(0, '.')
import numpy as np
from realtime_yukarin_b200.engine import default_engine
eng = default_engine()
rng = np.random.default_rng(0)
Tp, base = int(os.environ.get('TP', 384)), 64
enc = [1, 2, 4, 8, 8, 8, 8, 8]; dec = [8, 8, 8, 8, 4, 2, 1]
layers = []
for i in range(1, 8):
    layers.append((f'c{i}', 0, Tp >> (i - 1), 512 >> (i - 1), base * enc[i - 1], 0, base * enc[i]))
for d in range(7):
    c0 = base * enc[7] if d == 0 else base * dec[d - 1]
    c1 = 0 if d == 0 else base * enc[7 - d]
    layers.append((f'd{d}', 1, Tp >> (7 - d), 512 >> (7 - d), c0, c1, base * dec[d]))
tot = 0.0; totf = 0.0
for name, tr, H, W, C0, C1, Cout in layers:
    in0 = rng.standard_normal((1, H, W, C0)).astype(np.float32)
    in1 = rng.standard_normal((1, H, W, C1)).astype(np.float32) if C1 else None
    Cin = C0 + C1
    shape = (Cin, Cout, 4, 4) if tr else (Cout, Cin, 4, 4)
    Wt = (rng.standard_normal(shape) / np.sqrt(Cin * 16 / (4 if tr else 1))).astype(np.float32)
    out, ms = eng.test_conv_layer(in0, in1, Wt, np.ones(Cout, np.float32), np.zeros(Cout, np.float32), tr, 4, 2, 1, 1, use_tc=1, repeat=20)
    Ho, Wo = (H * 2, W * 2) if tr else (H // 2, W // 2)
    fl = 2.0 * 16 * Cin * Cout * (H * W if tr else Ho * Wo)
    tot += ms; totf += fl
    print(f'{name}: in {H}x{W}x{Cin} -> {Cout}: {ms * 1e3:7.1f} us  {fl / ms / 1e9:7.1f} TFLOP/s')
print(f'TOTAL: {tot * 1e3:.1f} us, {totf / tot / 1e9:.1f} TFLOP/s')
# edge layers (3x3): c0 = 1 -> 64 (fp32 in, fp16 out), out = 64 + 64 -> 1 (fp16 in, fp32 out)
in0 = rng.standard_normal((1, Tp, 512, 1)).astype(np.float32)
Wt = rng.standard_normal((64, 1, 3, 3)).astype(np.float32) / 3
out, ms = eng.test_conv_layer(in0, None, Wt, np.ones(64, np.float32), np.zeros(64, np.float32), 0, 3, 1, 1, 1, use_tc=2, repeat=20)
print(f'c0 (cin1): {ms * 1e3:7.1f} us   {Tp * 512 * 64 * 2 / ms / 1e6:7.1f} GB/s written')
in0 = rng.standard_normal((1, Tp, 512, 64)).astype(np.float32); in1 = rng.standard_normal((1, Tp, 512, 64)).astype(np.float32)
Wt = rng.standard_normal((1, 128, 3, 3)).astype(np.float32) / 30
out, ms = eng.test_conv_layer(in0, in1, Wt, np.ones(1, np.float32), np.zeros(1, np.float32), 0, 3, 1, 1, 0, use_tc=2, repeat=20)
print(f'out (cout1): {ms * 1e3:7.1f} us   {Tp * 512 * 128 * 2 / ms / 1e6:7.1f} GB/s read')
