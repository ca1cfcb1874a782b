"""Unit parity of the two convolution kernels against torch's CPU conv on the same data:
FP32 CUDA-core kernel (conv_direct.cu) and FP16 tcgen05 kernel (conv_tc.cu, TMA + UMMA + TMEM)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ref(in0, in1, W, scale, shift, transposed, k, stride, pad, act):
    x = in0 if in1 is None else np.concatenate([in0, in1], axis=3)
    xt = torch.from_numpy(x).permute(0, 3, 1, 2).double()
    Wt = torch.from_numpy(W).double()
    st, pd = (stride, stride), (pad, pad)
    if x.shape[1] == 1:                       # 1-D layer: kernel (1, k), stride (1, s), padding (0, p)
        st, pd = (1, stride), (0, pad)
    y = F.conv_transpose2d(xt, Wt, stride=st, padding=pd) if transposed else F.conv2d(xt, Wt, stride=st, padding=pd)
    y = y * torch.from_numpy(scale).double()[None, :, None, None] + torch.from_numpy(shift).double()[None, :, None, None]
    if act == 1:
        y = torch.where(y > 0, y, 0.2 * y)
    elif act == 2:
        y = torch.relu(y)
    return y.permute(0, 2, 3, 1).float().numpy()


CASES = [
    # transposed, k, s, p, B, H, W, C0, C1, Cout, act
    (0, 3, 1, 1, 1, 16, 32, 1, 0, 16, 1),
    (0, 4, 2, 1, 1, 32, 64, 64, 0, 128, 1),
    (0, 4, 2, 1, 2, 16, 16, 128, 0, 256, 1),
    (0, 4, 2, 1, 1, 6, 8, 256, 0, 256, 1),
    (1, 4, 2, 1, 1, 3, 4, 256, 0, 256, 2),
    (1, 4, 2, 1, 1, 12, 16, 128, 128, 64, 2),
    (1, 4, 2, 1, 2, 24, 32, 64, 64, 128, 2),
    (0, 3, 1, 1, 1, 16, 32, 16, 16, 1, 0),
    (0, 3, 1, 1, 1, 16, 32, 64, 64, 1, 0),
    # 1-D (stage-1) layers: H == 1
    (0, 4, 2, 1, 1, 1, 384, 64, 0, 128, 1),
    (0, 4, 2, 1, 1, 1, 6, 512, 0, 512, 1),
    (1, 4, 2, 1, 1, 1, 3, 512, 0, 512, 2),
    (1, 4, 2, 1, 1, 1, 96, 256, 256, 128, 2),
    (0, 3, 1, 1, 1, 1, 256, 128, 0, 9, 0),
]


@pytest.mark.parametrize('case', CASES)
def test_conv_kernels(engine, case):
    tr, k, s, p, B, H, W, C0, C1, Cout, act = case
    rng = np.random.default_rng(hash(case) % (2 ** 31))
    in0 = rng.standard_normal((B, H, W, C0)).astype(np.float32)
    in1 = rng.standard_normal((B, H, W, C1)).astype(np.float32) if C1 else None
    Cin = C0 + C1
    kh = 1 if H == 1 else k
    shape = (Cin, Cout, kh, k) if tr else (Cout, Cin, kh, k)
    Wt = (rng.standard_normal(shape) / np.sqrt(Cin * kh * k / (4 if tr else 1))).astype(np.float32)
    scale = rng.uniform(0.8, 1.2, Cout).astype(np.float32)
    shift = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    ref = _ref(in0, in1, Wt, scale, shift, tr, k, s, p, act)
    got, _ = engine.test_conv_layer(in0, in1, Wt, scale, shift, tr, k, s, p, act, use_tc=0)
    err = np.abs(got - ref).max()
    print('direct', case, 'max err', err)
    assert err < 1e-4
    if k == 4 and C0 % 64 == 0 and C1 % 64 == 0 and Cout % 64 == 0:
        got16, ms = engine.test_conv_layer(in0, in1, Wt, scale, shift, tr, k, s, p, act, use_tc=1, repeat=3)
        err16 = np.abs(got16 - ref).max()
        print('tcgen05', case, 'max err', err16, 'ms', ms)
        assert err16 < 3e-2, err16


EDGE_CASES = [
    # the stage-2 edge layers as the fp16 plan runs them (mixed precision): B, H, W, Cin (1 -> 64) or (64 + 64 -> 1)
    (1, 16, 32, 1, 64), (2, 37, 75, 1, 64), (1, 128, 512, 1, 64), (1, 5, 40, 1, 16),
    (1, 16, 32, 128, 1), (2, 37, 75, 128, 1), (1, 128, 512, 128, 1), (1, 2, 9, 128, 1),
]


@pytest.mark.parametrize('case', EDGE_CASES)
def test_edge_layer_kernels(engine, case):
    """k_conv3x3_cin1 / k_conv3x3_cout1_h (conv_direct.cu) with ragged tile edges, against torch on fp16-rounded inputs."""
    B, H, W, Cin, Cout = case
    rng = np.random.default_rng(B * 1000 + H * 10 + W + Cin)
    C0 = 1 if Cin == 1 else 64
    C1 = Cin - C0
    in0 = rng.standard_normal((B, H, W, C0)).astype(np.float32)
    in1 = rng.standard_normal((B, H, W, C1)).astype(np.float32) if C1 else None
    Wt = (rng.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(Cin * 9)).astype(np.float32)
    scale = rng.uniform(0.8, 1.2, Cout).astype(np.float32)
    shift = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    act = 1 if Cin == 1 else 0
    if Cin > 1:   # the kernel reads fp16 activations: compare on the same rounded values
        r0, r1 = in0.astype(np.float16).astype(np.float32), in1.astype(np.float16).astype(np.float32)
    else:
        r0, r1 = in0, None
    ref = _ref(r0, r1, Wt, scale, shift, 0, 3, 1, 1, act)
    got, _ = engine.test_conv_layer(in0, in1, Wt, scale, shift, 0, 3, 1, 1, act, use_tc=2)
    err = np.abs(got - ref).max()
    print('edge', case, 'max err', err)
    assert err < (5e-3 if Cin == 1 else 1e-4), err     # Cin = 1 writes fp16 (|y| < 8 -> half ulp 2^-9 * 4)


@pytest.mark.parametrize('case', [(1, 384, 9), (2, 131, 9), (1, 40, 16)])
def test_stage1_last_layer_kernel(engine, case):
    """k_conv1d_k3_small (conv_direct.cu): the 1-D k3 output layer of the stage-1 net, fp16 inputs (64 + 64 channels) -> fp32."""
    B, W, Cout = case
    rng = np.random.default_rng(W + Cout)
    in0 = rng.standard_normal((B, 1, W, 64)).astype(np.float32)
    in1 = rng.standard_normal((B, 1, W, 64)).astype(np.float32)
    Wt = (rng.standard_normal((Cout, 128, 1, 3)) / np.sqrt(128 * 3)).astype(np.float32)
    scale = rng.uniform(0.8, 1.2, Cout).astype(np.float32)
    shift = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    r0, r1 = in0.astype(np.float16).astype(np.float32), in1.astype(np.float16).astype(np.float32)
    ref = _ref(r0, r1, Wt, scale, shift, 0, 3, 1, 1, 0)
    got, _ = engine.test_conv_layer(in0, in1, Wt, scale, shift, 0, 3, 1, 1, 0, use_tc=2)
    err = np.abs(got - ref).max()
    print('stage-1 last layer', case, 'max err', err)
    assert err < 1e-4, err


# The 14 k4 layers of the stage-2 U-Net exactly as the benchmarked forward runs them (base 64, Tp = 384 x 512 bins, batch 1):
# same tile geometry, same split-K factor (ksplit is a function of the layer shape and the SM count only), same skip-concat
# split of the decoder inputs.   name, transposed, H, W, C0, C1, Cout, act
PRODUCTION_LAYERS = [
    ('c1', 0, 384, 512, 64, 0, 128, 1), ('c2', 0, 192, 256, 128, 0, 256, 1), ('c3', 0, 96, 128, 256, 0, 512, 1),
    ('c4', 0, 48, 64, 512, 0, 512, 1), ('c5', 0, 24, 32, 512, 0, 512, 1), ('c6', 0, 12, 16, 512, 0, 512, 1), ('c7', 0, 6, 8, 512, 0, 512, 1),
    ('d0', 1, 3, 4, 512, 0, 512, 2), ('d1', 1, 6, 8, 512, 512, 512, 2), ('d2', 1, 12, 16, 512, 512, 512, 2),
    ('d3', 1, 24, 32, 512, 512, 512, 2), ('d4', 1, 48, 64, 512, 512, 256, 2), ('d5', 1, 96, 128, 256, 256, 128, 2),
    ('d6', 1, 192, 256, 128, 128, 64, 2),
    # the batch-8 / Tp = 512 grouped shape (BASELINE config 5) for the two layers whose tiling changes most with M
    ('c1_b2_512', 0, 512, 512, 64, 0, 128, 1), ('d6_512', 1, 256, 256, 128, 128, 64, 2),
]


def _ref32(in0, in1, W, scale, shift, transposed, act):
    """float32 torch-CPU reference (oneDNN) for the large shapes: a float64 conv of 13-26 GFLOP would take minutes"""
    x = in0 if in1 is None else np.concatenate([in0, in1], axis=3)
    xt = torch.from_numpy(x).permute(0, 3, 1, 2).contiguous()
    Wt = torch.from_numpy(W)
    y = F.conv_transpose2d(xt, Wt, stride=2, padding=1) if transposed else F.conv2d(xt, Wt, stride=2, padding=1)
    y = y * torch.from_numpy(scale)[None, :, None, None] + torch.from_numpy(shift)[None, :, None, None]
    if act == 1:
        y = torch.where(y > 0, y, 0.2 * y)
    elif act == 2:
        y = torch.relu(y)
    return y.permute(0, 2, 3, 1).contiguous().numpy()


@pytest.mark.parametrize('case', PRODUCTION_LAYERS, ids=[c[0] for c in PRODUCTION_LAYERS])
def test_production_layer_shapes(engine, case):
    """tcgen05 kernel (and, where the default RYK_TC3=1 rule picks it, the halo kernel) on the shapes bench.py runs; inputs are fp16-representable
    so that the only differences from the float32 reference are accumulation order and the fp16 output rounding."""
    name, tr, H, W, C0, C1, Cout, act = case
    B = 2 if name.endswith('_b2_512') else 1
    rng = np.random.default_rng(sum(name.encode()) * 7919)
    in0 = rng.standard_normal((B, H, W, C0)).astype(np.float16).astype(np.float32)
    in1 = rng.standard_normal((B, H, W, C1)).astype(np.float16).astype(np.float32) if C1 else None
    Cin = C0 + C1
    shape = (Cin, Cout, 4, 4) if tr else (Cout, Cin, 4, 4)
    Wt = (rng.standard_normal(shape) / np.sqrt(Cin * 16 / (4 if tr else 1))).astype(np.float16).astype(np.float32)
    scale = rng.uniform(0.8, 1.2, Cout).astype(np.float32)
    shift = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    ref = _ref32(in0, in1, Wt, scale, shift, tr, act)
    got, ms = engine.test_conv_layer(in0, in1, Wt, scale, shift, tr, 4, 2, 1, act, use_tc=1, repeat=5)
    err = np.abs(got - ref)
    flop = 2.0 * 16 * Cin * Cout * (B * H * W / 4 if not tr else B * H * W)
    print(f'production layer {name}: max err {err.max():.2e} rms {np.sqrt((err ** 2).mean()):.2e} (|ref| max {np.abs(ref).max():.2f}); '
          f'{ms * 1e3:.1f} us, {flop / (ms * 1e-3) / 1e12 if ms > 0 else 0:.0f} TFLOP/s')
    # fp16 output rounding of |y| < 8 is 2^-9 * 4 = 8e-3; accumulation-order noise is ~1e-5
    assert err.max() < 1.2e-2, err.max()
    assert np.sqrt((err ** 2).mean()) < 1.5e-3


HALO_CASES = [
    # halo kernel (conv_tc3.cu), forced with RYK_TC3=2: transposed, B, H, W, C0, C1, Cout, act, MT, tile_w
    (0, 1, 32, 64, 64, 0, 128, 1, 1, 8),        # conv: 16 x 32 outputs, one row of M tiles
    (0, 1, 64, 64, 64, 0, 128, 1, 2, 8),        # conv, M = 256 CTA tiles (32 x 32 outputs)
    (0, 2, 32, 32, 128, 0, 256, 1, 1, 16),      # conv, batch 2, two N tiles, 8 x 16 pixel tiles, two channel chunks
    (0, 1, 48, 80, 64, 64, 128, 1, 2, 8),       # conv, two sources, ragged CTA tiles (24 x 40 outputs: 24 rows in 32-row tiles)
    (0, 1, 80, 48, 64, 0, 128, 1, 1, 8),        # conv, 40 x 24 outputs: ragged 16-row tiles
    (1, 1, 16, 32, 128, 0, 128, 2, 1, 8),       # deconv, one class per tile (N = 128)
    (1, 2, 32, 16, 64, 64, 256, 2, 2, 8),       # deconv, batch 2, two sources, two N tiles, M = 256
    (1, 1, 24, 32, 128, 128, 128, 2, 1, 16),    # deconv, d3-like class grid 24 x 32 with 8 x 16 tiles
    (1, 1, 12, 24, 64, 0, 128, 2, 2, 8),        # deconv, ragged (12 rows in 32-row CTA tiles)
    (1, 1, 16, 32, 128, 128, 64, 2, 1, 8),      # deconv Cout = 64: fused column classes (d6 family)
    (1, 1, 32, 16, 64, 64, 64, 2, 2, 8),        # fused classes, M = 256
    (1, 2, 20, 24, 64, 0, 64, 2, 2, 8),         # fused classes, ragged rows, batch 2
    (1, 1, 16, 32, 64, 0, 64, 2, 1, 16),        # fused classes, 8 x 16 tiles
]


@pytest.mark.parametrize('case', HALO_CASES)
def test_halo_kernel(engine, case):
    """k_conv_halo: shared halo rows (two taps per A box), M = 128 / 256 per CTA, fused column classes, dynamic tile scheduler.
    Same tolerance as the per-tap tcgen05 kernel, and the result must agree with it (same fp16 operands, fp32 accumulation)."""
    import os
    tr, B, H, W, C0, C1, Cout, act, mt, tw = case
    rng = np.random.default_rng(sum(case) * 104729 + 7)
    in0 = rng.standard_normal((B, H, W, C0)).astype(np.float32)
    in1 = rng.standard_normal((B, H, W, C1)).astype(np.float32) if C1 else None
    Cin = C0 + C1
    shape = (Cin, Cout, 4, 4) if tr else (Cout, Cin, 4, 4)
    Wt = (rng.standard_normal(shape) / np.sqrt(Cin * 16 / (4 if tr else 1))).astype(np.float32)
    scale = rng.uniform(0.8, 1.2, Cout).astype(np.float32)
    shift = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    ref = _ref(in0, in1, Wt, scale, shift, tr, 4, 2, 1, act)
    keys = ('RYK_TC3', 'RYK_TC3_MT', 'RYK_TC3_TW')
    old = {k: os.environ.get(k) for k in keys}
    try:
        os.environ['RYK_TC3'] = '0'
        base, _ = engine.test_conv_layer(in0, in1, Wt, scale, shift, tr, 4, 2, 1, act, use_tc=1)
        os.environ.update(RYK_TC3='2', RYK_TC3_MT=str(mt), RYK_TC3_TW=str(tw))
        got, ms = engine.test_conv_layer(in0, in1, Wt, scale, shift, tr, 4, 2, 1, act, use_tc=1, repeat=3)
        err, err_base = np.abs(got - ref).max(), np.abs(base - ref).max()
        print('halo kernel', case, 'max err', err, '(per-tap kernel', err_base, ') ms', ms)
        assert err < 3e-2, err
        assert np.abs(got - base).max() < 2e-2
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
