// conv_tc.cu -- tcgen05 (5th-gen tensor core) implicit-GEMM convolution for the stage-2
// "Become-Yukarin" 2-D U-Net (SURVEY row a13, component I: > 99 % of the hot path's FLOPs).
//
//   D[pixels, Cout] = sum over taps t, channels c of  A_t[pixels, c] * W[t, c, Cout]
//
// * Operands are FP16, accumulation FP32 in TMEM (kind::f16, UMMA 128 x BLOCK_N x 16).
// * A tiles (128 output pixels x 64 input channels of ONE tap) are fetched by TMA straight from the
//   NHWC activation tensor: a 4-D box (64 ch, tile_w, tile_h, 1) whose W/H traversal stride is the
//   conv stride (elementStrides = 2 for the k4 s2 p1 encoder convs) and whose out-of-bounds part is
//   zero-filled by the TMA unit -- that IS the zero padding; no im2col buffer ever exists.
//   Transposed convs (decoder) are run per output-parity class, each a dense 2x2-tap conv.
// * The U-Net skip concat is "by pointer": the K loop walks the channels of tensor 0, then tensor 1.
// * B tiles (BLOCK_N output channels x 64 K) come from a K-major packed weight matrix, also by TMA.
// * Both tiles land in the canonical 128-byte-swizzled K-major layout that UMMA smem descriptors
//   address; a ring of kStages stages is handed between three warp roles through mbarriers:
//     warp 4 lane 0 : TMA producer        (waits empty[s], arms full[s] with expect_tx, issues 2 loads)
//     warp 5 lane 0 : MMA issuer          (waits full[s], 4 x tcgen05.mma, tcgen05.commit -> empty[s])
//     warps 0-3     : epilogue            (wait tmem_full, tcgen05.ld 32 lanes x 32 columns at a time,
//                                          folded BN scale/shift + LeakyReLU/ReLU, FP16 NHWC store)
// * Small-M bottleneck layers are weight-bandwidth bound: split-K over blockIdx.z spreads the weight
//   stream over all SMs; each split stores its FP32 partial tile into its own slice of a workspace,
//   and a reduce kernel sums the slices in a fixed order (deterministic) and applies the epilogue.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <stdlib.h>

#include <vector>
#include <stdio.h>
#include "conv.h"
#include "tc_ptx.cuh"

namespace ryk {

struct TcParams {
  int transposed, Cout;
  int tile_w, tile_h, tiles_w, tiles_h;
  int chunks0, chunks1;          // 64-channel chunks of source 0 / 1
  int taps_w, ntaps;             // taps per class: conv KH*KW (taps_w = KW); deconv (KH/SH)*(KW/SW)
  int sh, sw, ph, pw;            // conv stride / padding per dimension (1-D nets: sh = 1, ph = 0)
  int classes_w;                 // deconv output-parity classes along W (SW); along H it is SH
  int ksplit, chunks_per_split;
  int act;
  const float* scale; const float* shift;
  float* ws;                     // split-K workspace [ksplit][pixels][Cout] or nullptr
  int debug;                     // RYK_TC_DEBUG bit 1 (perf experiments only): skip the output stores
};

#ifdef RYK_TC_TIMELINE
// diagnostics build only (RYK_NVCC_EXTRA=-DRYK_TC_TIMELINE): per-CTA phase timestamps
constexpr int kTlMaxCtas = 8192, kTlSlots = 10;
__device__ unsigned long long g_tl[kTlMaxCtas * kTlSlots];
__device__ __forceinline__ unsigned long long tl_now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define TL(slot) do { int c_ = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z); if (c_ < kTlMaxCtas) g_tl[c_ * kTlSlots + (slot)] = tl_now(); } while (0)
#else
#define TL(slot) do {} while (0)
#endif
// Two co-resident CTAs per SM let one tile's epilogue overlap the other's main loop.
template <int BLOCK_N, int kStages>
__global__ void __launch_bounds__(kTcThreads, 2)
k_conv_tc(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
          const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmW,
          const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kABytes = kBlockM * kBlockK * 2;
  constexpr uint32_t kBBytes = BLOCK_N * kBlockK * 2;
  // carve: 1024-aligned stage buffers first, barriers after
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * kABytes;
  uint64_t* full_bar = (uint64_t*)(smem_b + kStages * kBBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;
  uint32_t* tmem_ptr_smem = (uint32_t*)(tmem_full_bar + 1);
  // per-channel scale / shift of this CTA's BLOCK_N output channels, staged once: the epilogue reads them as broadcast
  // LDS.128 (reading them with __ldg per element cost 128 LSU instructions per 32 columns and made the epilogue
  // longer than the MMA main loop)
  float* s_scale = (float*)(((uintptr_t)(tmem_ptr_smem + 4) + 15) & ~(uintptr_t)15);
  float* s_shift = s_scale + BLOCK_N;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
  if (threadIdx.x == 0) {
    TL(0);
#ifdef RYK_TC_TIMELINE
    { unsigned sm; asm volatile("mov.u32 %0, %smid;" : "=r"(sm)); int c_ = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z); if (c_ < kTlMaxCtas) g_tl[c_ * kTlSlots + 9] = sm; }
#endif
  }

  // tile coordinates
  int mt = blockIdx.x;
  const int tw = mt % p.tiles_w; mt /= p.tiles_w;
  const int th = mt % p.tiles_h; mt /= p.tiles_h;
  const int b = mt;
  const int n0 = blockIdx.y * BLOCK_N;
  const int cls = blockIdx.z / p.ksplit, split = blockIdx.z % p.ksplit;
  const int py = cls / p.classes_w, px = cls % p.classes_w;
  const int oy0 = th * p.tile_h, ox0 = tw * p.tile_w;       // class-local output origin of the tile
  const int chunks_per_tap = p.chunks0 + p.chunks1;
  const int total_chunks = p.ntaps * chunks_per_tap;
  const int kc_begin = split * p.chunks_per_split;
  const int kc_end = min(total_chunks, kc_begin + p.chunks_per_split);
  const int my_chunks = kc_end - kc_begin;

  if (threadIdx.x == 128) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA0) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    if (p.chunks1 > 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA1) : "memory");
    if (!p.ws) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmO) : "memory");
    else asm volatile("prefetch.tensormap [%0];" ::"l"(&tmW) : "memory");
  }
  if (threadIdx.x == 160) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp < 4 && !p.ws) {
    for (int i = threadIdx.x; i < BLOCK_N; i += 128) { s_scale[i] = __ldg(p.scale + n0 + i); s_shift[i] = __ldg(p.shift + n0 + i); }
  }
  if (warp == 4) {   // TMEM allocation (whole warp), BLOCK_N fp32 accumulator columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)BLOCK_N) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();                       // the previous layer's outputs (our A operand) are complete from here on
  if (threadIdx.x == 0) TL(1);

  if (warp == 4) {
    // ===== TMA producer (warp-uniform loop, one elected lane issues: see elect_one() in tc_ptx.cuh) =====
    for (int i = 0; i < my_chunks; ++i) {
      const int s = i % kStages;
      const uint32_t ph = (i / kStages) & 1;
      mbar_wait(&empty_bar[s], ph ^ 1);
      const int kc = kc_begin + i;
      const int tap = kc / chunks_per_tap;
      const int cc = kc - tap * chunks_per_tap;
      const int ty = tap / p.taps_w, tx = tap - ty * p.taps_w;
      int ix, iy;
      if (!p.transposed) { ix = ox0 * p.sw + tx - p.pw; iy = oy0 * p.sh + ty - p.ph; }
      else {   // k4 s2 p1 along a strided dimension: input = m + d - 1 + parity; k1 s1 p0 along the other: input = m
        ix = p.sw == 2 ? ox0 + tx - 1 + px : ox0;
        iy = p.sh == 2 ? oy0 + ty - 1 + py : oy0;
      }
      if (elect_one()) {
        mbar_expect_tx(&full_bar[s], kABytes + kBBytes);
        if (cc < p.chunks0) tma_load_4d(smem_a + s * kABytes, &tmA0, &full_bar[s], cc * kBlockK, ix, iy, b);
        else tma_load_4d(smem_a + s * kABytes, &tmA1, &full_bar[s], (cc - p.chunks0) * kBlockK, ix, iy, b);
        tma_load_2d(smem_b + s * kBBytes, &tmB, &full_bar[s], kc * kBlockK, cls * p.Cout + n0);
      }
    }
  } else if (warp == 5) {
    // ===== MMA issuer (warp-uniform loop, one elected lane issues) =====
    // instruction descriptor: D=F32, A=B=F16, both K-major, N = BLOCK_N, M = 128
    constexpr uint32_t idesc = (1u << 4) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);
    for (int i = 0; i < my_chunks; ++i) {
      const int s = i % kStages;
      const uint32_t ph = (i / kStages) & 1;
      mbar_wait(&full_bar[s], ph);
      if (i == 0 && lane == 0) TL(2);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint64_t adesc = make_sw128_desc(smem_u32(smem_a + s * kABytes));
      const uint64_t bdesc = make_sw128_desc(smem_u32(smem_b + s * kBBytes));
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < kBlockK / kUmmaK; ++k) {
          // advance 32 bytes (16 fp16) inside the swizzle atom: +2 in the (addr >> 4) field
          umma_f16(tmem_base, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (i > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty_bar[s]);
      }
    }
    if (elect_one()) umma_commit(tmem_full_bar);
    if (lane == 0) TL(3);
  } else if (warp < 4) {
    // ===== epilogue =====
    if (lane == 0) mbar_wait(tmem_full_bar, 0);        // one polling lane per warp
    __syncwarp();
    if (threadIdx.x == 0) TL(4);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int row = warp * 32 + lane;                 // accumulator row == TMEM lane == pixel of the tile
    // (out-of-range pixels of ragged tiles need no masking: both TMA stores below clip at the tensor-map bounds)
#pragma unroll 1
    for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
      uint32_t r[32];
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0;
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
            "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
            "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
            "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
          : "r"(taddr));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (p.ws) {
        // split-K partial tile (raw FP32 sums) -> swizzled staging, one [128 pixels][32 channels] block per iteration;
        // stored below by TMA into this split's slice of the workspace; k_splitk_reduce sums the slices
        uint8_t* blk = smem + (c0 >> 5) * (kBlockM * 128) + row * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<uint4*>(blk + ((j ^ (row & 7)) << 4)) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
      } else {
        // scale/shift/activation -> FP16 -> 128B-swizzled staging tile in the (now idle) pipeline stage buffers:
        // BLOCK_N / 64 blocks of [128 pixels][64 channels]; one TMA store per block writes full 128-byte rows
        uint8_t* blk = smem + (c0 >> 6) * (kBlockM * 128) + row * 128;
        const int cbase = (c0 & 32) >> 3;          // first 16-byte chunk of this 32-channel half inside the block: 0 or 4
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          const float4 sc0 = *reinterpret_cast<const float4*>(s_scale + c0 + j), sc1 = *reinterpret_cast<const float4*>(s_scale + c0 + j + 4);
          const float4 sh0 = *reinterpret_cast<const float4*>(s_shift + c0 + j), sh1 = *reinterpret_cast<const float4*>(s_shift + c0 + j + 4);
          const float sc[8] = {sc0.x, sc0.y, sc0.z, sc0.w, sc1.x, sc1.y, sc1.z, sc1.w};
          const float sh[8] = {sh0.x, sh0.y, sh0.z, sh0.w, sh1.x, sh1.y, sh1.z, sh1.w};
          uint32_t pk[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float v0 = fmaf(__uint_as_float(r[j + 2 * q]), sc[2 * q], sh[2 * q]);
            float v1 = fmaf(__uint_as_float(r[j + 2 * q + 1]), sc[2 * q + 1], sh[2 * q + 1]);
            if (p.act == ACT_LEAKY) { v0 = v0 > 0.f ? v0 : 0.2f * v0; v1 = v1 > 0.f ? v1 : 0.2f * v1; }
            else if (p.act == ACT_RELU) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
            __half2 h = __floats2half2_rn(v0, v1);
            pk[q] = *reinterpret_cast<uint32_t*>(&h);
          }
          const int chunk = cbase + (j >> 3);
          *reinterpret_cast<uint4*>(blk + ((chunk ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
    }
    if (!p.ws && my_chunks > 0) {
      // generic-proxy smem writes -> visible to the async proxy; one thread hands the tile to the TMA unit
      // (out-of-range pixels are clipped by the tensor map, so no masking is needed)
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (threadIdx.x == 0 && !(p.debug & 1)) {
        const int xs = p.transposed ? ox0 * p.sw + px : ox0;
        const int ys = p.transposed ? oy0 * p.sh + py : oy0;
#pragma unroll
        for (int jb = 0; jb < BLOCK_N / 64; ++jb) {
          asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                       ::"l"(&tmO), "r"(smem_u32(smem + jb * (kBlockM * 128))), "r"(n0 + jb * 64), "r"(xs), "r"(ys), "r"(b) : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
      }
    }
    if (p.ws && my_chunks > 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (threadIdx.x == 0 && !(p.debug & 1)) {
        const int xs = p.transposed ? ox0 * p.sw + px : ox0;
        const int ys = p.transposed ? oy0 * p.sh + py : oy0;
#pragma unroll
        for (int jb = 0; jb < BLOCK_N / 32; ++jb) {
          asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
                       ::"l"(&tmW), "r"(smem_u32(smem + jb * (kBlockM * 128))), "r"(n0 + jb * 32), "r"(xs), "r"(ys), "r"(b), "r"(split) : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
      }
    }
  }
  if (threadIdx.x == 0) TL(5);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 4) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)BLOCK_N) : "memory");
    if (lane == 0) TL(6);
  }
}

// split-K reduce + epilogue: out = act((sum over splits of ws[s]) * scale + shift) as fp16, 4 channels per thread.
// Block = G warps x 32 lanes: lane = one float4 of the output (512 contiguous bytes per warp load), warp g sums the
// slices g, g + G, g + 2G, ... ; the G partial sums are combined through shared memory in a fixed order, so the result
// is deterministic (same summation tree every run) while G x more loads are in flight than with one thread per output.
__global__ void __launch_bounds__(256) k_splitk_reduce(const float* __restrict__ ws, size_t total4, size_t slice_elems, int ksplit, int Cout,
                                const float* __restrict__ scale, const float* __restrict__ shift, int act, __half* __restrict__ out) {
  __shared__ float4 part[8][32];
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5, G = blockDim.x >> 5;
  const size_t i = (size_t)blockIdx.x * 32 + lane;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < total4) {
    const float4* p = reinterpret_cast<const float4*>(ws) + i;
    const size_t stride4 = slice_elems / 4;
#pragma unroll 4
    for (int s = g; s < ksplit; s += G) {
      const float4 b = __ldg(p + (size_t)s * stride4);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
  }
  part[g][lane] = a;
  __syncthreads();
  if (g != 0 || i >= total4) return;
  for (int k = 1; k < G; ++k) { const float4 b = part[k][lane]; a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
  const int n = (int)((i * 4) % Cout);
  const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + n)), sh = __ldg(reinterpret_cast<const float4*>(shift + n));
  float v[4] = {fmaf(a.x, sc.x, sh.x), fmaf(a.y, sc.y, sh.y), fmaf(a.z, sc.z, sh.z), fmaf(a.w, sc.w, sh.w)};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (act == ACT_LEAKY) v[j] = v[j] > 0.f ? v[j] : 0.2f * v[j]; else if (act == ACT_RELU) v[j] = fmaxf(v[j], 0.f);
  }
  __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
  reinterpret_cast<uint2*>(out)[i] = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
}

// few splits, large outputs (c3 / c4 / d3): one thread per float4 of the output, grid-stride, all slices summed in order
__global__ void __launch_bounds__(256) k_splitk_reduce_few(const float* __restrict__ ws, size_t total4, size_t slice_elems, int ksplit, int Cout,
                                    const float* __restrict__ scale, const float* __restrict__ shift, int act, __half* __restrict__ out) {
  const size_t stride4 = slice_elems / 4;
  pdl_trigger();
  pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total4; i += (size_t)gridDim.x * blockDim.x) {
    const float4* p = reinterpret_cast<const float4*>(ws) + i;
    float4 a = __ldg(p);
#pragma unroll 4
    for (int s = 1; s < ksplit; ++s) {
      const float4 b = __ldg(p + (size_t)s * stride4);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    const int n = (int)((i * 4) % Cout);
    const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + n)), sh = __ldg(reinterpret_cast<const float4*>(shift + n));
    float v[4] = {fmaf(a.x, sc.x, sh.x), fmaf(a.y, sc.y, sh.y), fmaf(a.z, sc.z, sh.z), fmaf(a.w, sc.w, sh.w)};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (act == ACT_LEAKY) v[j] = v[j] > 0.f ? v[j] : 0.2f * v[j]; else if (act == ACT_RELU) v[j] = fmaxf(v[j], 0.f);
    }
    __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
    reinterpret_cast<uint2*>(out)[i] = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
  }
}

// ------------------------------------------------------------------------------------ host side
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;

template <int BN, int ST> static constexpr size_t tc_smem_bytes() {
  return (size_t)ST * (kBlockM * kBlockK * 2 + BN * kBlockK * 2) + (2 * ST + 1) * 8 + 16 + 1024 + 2 * BN * 4 + 32;
}

int tc_init() {
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    RYK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    RYK_CHECK(qres == cudaDriverEntryPointSuccess && fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
    g_encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  }
  if (tc3_init()) return -1;
  RYK_CUDA(cudaFuncSetAttribute(k_conv_tc<128, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes<128, 3>()));
  RYK_CUDA(cudaFuncSetAttribute(k_conv_tc<64, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes<64, 4>()));
  return 0;
}

bool tc_layer_eligible(const ConvLayer& L) {
  const bool k2d = L.KH == 4 && L.KW == 4 && L.SH == 2 && L.SW == 2 && L.PH == 1 && L.PW == 1;
  const bool k1d = L.KH == 1 && L.KW == 4 && L.SH == 1 && L.SW == 2 && L.PH == 0 && L.PW == 1;
  if (!k2d && !k1d) return false;
  if (L.C0 % kBlockK != 0 || L.C1 % kBlockK != 0 || L.C0 == 0) return false;
  if (L.Cout % 64 != 0) return false;
  if (L.in_dtype != DT_F16 || L.out_dtype != DT_F16) return false;
  return true;
}

static int pow2_floor(int v) { int p = 1; while (p * 2 <= v) p *= 2; return p; }

static int make_act_map(CUtensorMap* m, const void* ptr, int C, int W, int H, int B, int box_w, int box_h, int stride_w, int stride_h) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)kBlockK, (cuuint32_t)(box_w * stride_w), (cuuint32_t)(box_h * stride_h), 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride_w, (cuuint32_t)stride_h, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(activation) failed: " + std::to_string((int)r)); return -1; }
  return 0;
}

// split-K workspace [ksplit][B][Hout][Wout][Cout] fp32 as a 5-D map: box = (32 channels, tile_w, tile_h, 1, 1) with the same
// W / H element strides as the output map (deconv parity classes write every other pixel)
static int make_ws_map(CUtensorMap* m, const void* ptr, int C, int W, int H, int B, int ksplit, int box_w, int box_h, int stride_w, int stride_h) {
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B, (cuuint64_t)ksplit};
  cuuint64_t strides[4] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4, (cuuint64_t)B * H * W * C * 4};
  cuuint32_t box[5] = {32, (cuuint32_t)(box_w * stride_w), (cuuint32_t)(box_h * stride_h), 1, 1};
  cuuint32_t estr[5] = {1, (cuuint32_t)stride_w, (cuuint32_t)stride_h, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(split-K workspace) failed: " + std::to_string((int)r)); return -1; }
  return 0;
}

static int make_weight_map(CUtensorMap* m, const void* ptr, size_t K, size_t rows, int block_n) {
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)block_n};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weights) failed: " + std::to_string((int)r)); return -1; }
  return 0;
}

constexpr int kMinChunksPerSplit = 8;                  // split-K: at least this many 64-channel K chunks per split

static void tc_geometry(const ConvLayer& L, int num_sms, int* tile_w, int* tile_h, int* block_n, int* ksplit) {
  int Wc = L.transposed ? L.Win : L.Wout;
  int Hc = L.transposed ? L.Hin : L.Hout;
  int tw = pow2_floor(Wc < kBlockM ? Wc : kBlockM);
  int th = kBlockM / tw;
  int bn = L.Cout >= 128 ? 128 : 64;                    // N <= 128: the epilogue's staging tile must fit the stage buffers
  int classes = L.transposed ? L.SH * L.SW : 1;
  int tiles = L.B * ((Wc + tw - 1) / tw) * ((Hc + th - 1) / th) * (L.Cout / bn) * classes;
  int ntaps = L.transposed ? (L.KH / L.SH) * (L.KW / L.SW) : L.KH * L.KW;
  int total_chunks = ntaps * (L.C0 + L.C1) / kBlockK;
  int ks = 1;
  const int slots = 2 * num_sms;                        // two co-resident CTAs per SM
  if (tiles < slots) {
    ks = slots / tiles;
    if (ks > total_chunks / kMinChunksPerSplit) ks = total_chunks / kMinChunksPerSplit;
    if (ks < 1) ks = 1;
    int cps = (total_chunks + ks - 1) / ks;
    ks = (total_chunks + cps - 1) / cps;                // every split owns at least one chunk
  }
  { int a_, b_, c_; if (tc3_layer_config(L, num_sms, &a_, &b_, &c_)) ks = 1; }     // halo kernel: no split-K
  *tile_w = tw; *tile_h = th; *block_n = bn; *ksplit = ks;
}

bool tc_layer_wants_counter(const ConvLayer& L, int num_sms) {
  int a_, b_, c_;
  return tc_layer_eligible(L) && tc3_layer_config(L, num_sms, &a_, &b_, &c_);
}

size_t tc_splitk_ws_bytes(const ConvLayer& L, int num_sms) {
  int tw, th, bn, ks;
  tc_geometry(L, num_sms, &tw, &th, &bn, &ks);
  return ks > 1 ? (size_t)ks * L.B * L.Hout * L.Wout * L.Cout * sizeof(float) : 0;
}

int tc_layer_prepare(ConvLayer& L, int num_sms) {
  RYK_CHECK(g_encode != nullptr, "tc_init() was not called");
  RYK_CHECK(tc_layer_eligible(L), "layer is not eligible for the tensor-core path");
  tc_geometry(L, num_sms, &L.tile_w, &L.tile_h, &L.block_n, &L.ksplit);
  int stw = L.transposed ? 1 : L.SW, sth = L.transposed ? 1 : L.SH;
  if (make_act_map(&L.tmA0, L.in0, L.C0, L.Win, L.Hin, L.B, L.tile_w, L.tile_h, stw, sth)) return -1;
  if (L.C1 > 0) { if (make_act_map(&L.tmA1, L.in1, L.C1, L.Win, L.Hin, L.B, L.tile_w, L.tile_h, stw, sth)) return -1; }
  else L.tmA1 = L.tmA0;
  int classes = L.transposed ? L.SH * L.SW : 1;
  int ntaps = L.transposed ? (L.KH / L.SH) * (L.KW / L.SW) : L.KH * L.KW;
  size_t K = (size_t)ntaps * (L.C0 + L.C1);
  size_t rows = (size_t)classes * L.Cout;
  if (make_weight_map(&L.tmB, L.w_tc, K, rows, L.block_n)) return -1;
  // output map for the TMA-store epilogue: deconv classes write every other pixel (element strides = conv strides)
  if (make_act_map(&L.tmO, L.out, L.Cout, L.Wout, L.Hout, L.B, L.tile_w, L.tile_h, L.transposed ? L.SW : 1, L.transposed ? L.SH : 1)) return -1;
  L.tc3 = tc3_layer_config(L, num_sms, &L.t3_tile_w, &L.t3_tile_h, &L.t3_mt);
  if (L.tc3 && tc3_layer_prepare(L, g_encode)) return -1;
  RYK_CHECK(L.ksplit == 1 || L.splitk_ws != nullptr, "split-K layer without a workspace");
  if (L.ksplit > 1) {
    if (make_ws_map(&L.tmW, L.splitk_ws, L.Cout, L.Wout, L.Hout, L.B, L.ksplit, L.tile_w, L.tile_h, L.transposed ? L.SW : 1, L.transposed ? L.SH : 1)) return -1;
  } else L.tmW = L.tmO;
  L.tc_ready = true;
  return 0;
}

// Launch with the programmatic-stream-serialization attribute (see pdl_trigger / pdl_wait); RYK_NO_PDL=1 falls back to
// plain stream order (the device-side instructions are then no-ops).
static int g_pdl_force = -1;                       // -1: environment decides; 0 / 1: forced (captures that must not carry programmatic edges)
void tc_force_pdl(int v) { g_pdl_force = v; }
static bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("RYK_NO_PDL"); v = (e && atoi(e) != 0) ? 0 : 1; }
  return g_pdl_force >= 0 ? g_pdl_force != 0 : v != 0;
}
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int conv_tc_run(const ConvLayer& L, cudaStream_t st) {
  RYK_CHECK(L.tc_ready, "tc layer not prepared");
  if (L.tc3) return conv_tc3_run(L, st, pdl_enabled());
  TcParams p;
  const int Hc = L.transposed ? L.Hin : L.Hout, Wc = L.transposed ? L.Win : L.Wout;    // class-local output grid
  p.transposed = L.transposed; p.Cout = L.Cout;
  p.tile_w = L.tile_w; p.tile_h = L.tile_h;
  p.tiles_w = (Wc + L.tile_w - 1) / L.tile_w; p.tiles_h = (Hc + L.tile_h - 1) / L.tile_h;
  p.chunks0 = L.C0 / kBlockK; p.chunks1 = L.C1 / kBlockK;
  p.taps_w = L.transposed ? L.KW / L.SW : L.KW;
  p.ntaps = L.transposed ? (L.KH / L.SH) * (L.KW / L.SW) : L.KH * L.KW;
  p.sh = L.SH; p.sw = L.SW; p.ph = L.PH; p.pw = L.PW;
  p.classes_w = L.transposed ? L.SW : 1;
  const int classes = L.transposed ? L.SH * L.SW : 1;
  p.ksplit = L.ksplit;
  int total_chunks = p.ntaps * (p.chunks0 + p.chunks1);
  p.chunks_per_split = (total_chunks + L.ksplit - 1) / L.ksplit;
  p.act = L.act; p.scale = L.scale; p.shift = L.shift;
  p.ws = L.ksplit > 1 ? L.splitk_ws : nullptr;
#ifdef RYK_DIAG
  { static int dbg = -1; if (dbg < 0) { const char* v = getenv("RYK_TC_DEBUG"); dbg = v ? atoi(v) : 0; } p.debug = dbg; }   // diagnostics builds only
#else
  p.debug = 0;
#endif
  size_t out_elems = (size_t)L.B * L.Hout * L.Wout * L.Cout;
  dim3 grid(L.B * p.tiles_w * p.tiles_h, L.Cout / L.block_n, classes * L.ksplit);
  if (L.block_n == 128) RYK_CUDA(launch_pdl(k_conv_tc<128, 3>, grid, dim3(kTcThreads), tc_smem_bytes<128, 3>(), st, L.tmA0, L.tmA1, L.tmB, L.tmO, L.tmW, p));
  else RYK_CUDA(launch_pdl(k_conv_tc<64, 4>, grid, dim3(kTcThreads), tc_smem_bytes<64, 4>(), st, L.tmA0, L.tmA1, L.tmB, L.tmO, L.tmW, p));
  RYK_CUDA(cudaGetLastError());
#ifdef RYK_TC_TIMELINE
  cudaStreamCaptureStatus cap_ = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cap_);
  if (const char* path = cap_ == cudaStreamCaptureStatusNone ? getenv("RYK_TC_TIMELINE_FILE") : nullptr) {
    cudaStreamSynchronize(st);
    static std::vector<unsigned long long> h(kTlMaxCtas * kTlSlots);
    cudaMemcpyFromSymbol(h.data(), g_tl, sizeof(unsigned long long) * h.size());
    int n = grid.x * grid.y * grid.z; if (n > kTlMaxCtas) n = kTlMaxCtas;
    if (FILE* f = fopen(path, "w")) {
      fprintf(f, "# grid %d %d %d block_n %d ksplit %d\n", grid.x, grid.y, grid.z, L.block_n, L.ksplit);
      for (int c = 0; c < n; ++c) { for (int k = 0; k < kTlSlots; ++k) fprintf(f, "%llu ", h[c * kTlSlots + k]); fprintf(f, "\n"); }
      fclose(f);
    }
  }
#endif
  if (p.ws) {
    size_t total4 = out_elems / 4;
    if (L.ksplit <= 4) {
      int blocks = (int)((total4 + 255) / 256); if (blocks > 2368) blocks = 2368;
      RYK_CUDA(launch_pdl(k_splitk_reduce_few, dim3(blocks), dim3(256), 0, st, (const float*)p.ws, total4, out_elems, L.ksplit, L.Cout, L.scale, L.shift, L.act, (__half*)L.out));
    } else {
      RYK_CUDA(launch_pdl(k_splitk_reduce, dim3((unsigned)((total4 + 31) / 32)), dim3(256), 0, st, (const float*)p.ws, total4, out_elems, L.ksplit, L.Cout, L.scale, L.shift, L.act, (__half*)L.out));
    }
    RYK_CUDA(cudaGetLastError());
  }
  return 0;
}

}  // namespace ryk
