// conv_tc3.cu -- "halo" tcgen05 kernel for the LARGE k4 s2 p1 layers of the stage-2 U-Net (c1-c3, d3-d6: 91 % of the FLOPs).
//
// Why: the per-tap kernel of conv_tc.cu stages 64 FLOP per byte fetched from L2 (128 x 128 x 64 tiles, one A tile per tap) and
// its big layers run AT the chip's L2 -> SM output cap (10-12 TB/s measured, profiles/r01c): the tensor pipe waits for operands.
// This kernel roughly halves the bytes per FLOP:
//   * HALO ROWS.  An output tile is tile_h x tile_w pixels with tile_w = 8 or 16, so one image row of the tile is a whole number of
//     8-row swizzle atoms (1024 B).  The two taps of a k4 s2 conv that share a column tap and a row parity (ky = 0 / 2 or 1 / 3)
//     read the SAME strided input rows shifted by one; the two row taps of a transposed-conv parity class likewise.  One TMA box
//     with tile_h + 1 rows therefore serves both taps: the second tap's UMMA descriptor simply starts tile_w * 128 B further
//     (1024-B aligned, so the 128B-swizzle phase is unchanged).  A bytes per tap pair: 17/32 (tile_w 8) of the per-tap kernel's.
//   * M = 256 PER CTA (MT = 2).  Two stacked M tiles (box of 2 * tile_h + 1 rows) share every weight tile.
//   * FUSED COLUMN CLASSES for Cout = 64 (d6): the two output-column parities of a transposed conv use 3 distinct input column
//     offsets for their 4 (class, dx) pairs and accumulate side by side in TMEM (2 x 64 columns): N = 128 per A view.
//   * PERSISTENT, DYNAMICALLY SCHEDULED.  One CTA per SM draws tiles from a global counter (the draw for tile i + 1 is issued
//     while tile i's loads are queued), accumulators are double-buffered in TMEM so the epilogue of tile i (tcgen05.ld -> BN
//     scale/shift + activation -> FP16 -> swizzled staging -> TMA store) overlaps the main loop of tile i + 1, and CTAs that
//     start late (SM busy with a co-running WORLD kernel) simply take fewer tiles.
//   * DECOUPLED RINGS.  A boxes (17-34 KB) and B tiles (8-16 KB) have separate mbarrier rings: a B slot is released after its
//     4 * MT MMAs, an A slot after its 2-4 taps.
// Roles: warp 4 lane 0 = tile scheduler + TMA producer, warp 5 lane 0 = MMA issuer, warps 0-3 = epilogue.
// Reference op: the Chainer Convolution2D / Deconvolution2D (k4 s2 p1) + BN + (Leaky)ReLU of become_yukarin's U-Net, reached
// through realtime_voice_conversion/yukarin_wrapper/voice_changer.py:41.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "conv.h"
#include "tc_ptx.cuh"

namespace ryk {

constexpr int kT3MaxGroups = 8;     // A boxes per channel chunk (conv: 4 column taps x 2 row parities)
constexpr int kT3MaxB = 4;          // weight tiles per A box
constexpr int kT3Sched = 4;         // tile-id ring

struct T3Group {
  int16_t ax, ay;                   // box origin relative to (ox0 * sx, oy0 * sy)
  int16_t nb;
  int16_t pad_;
  int32_t brow[kT3MaxB];            // weight-matrix row of the tile (class * Cout); the N-tile offset n0 is added at run time
  int16_t btap[kT3MaxB];            // tap index on the packed K axis (k = btap * Cin + channel)
  int16_t ashift[kT3MaxB];          // halo rows skipped by this tap (0 / 1)
  int16_t bcol[kT3MaxB];            // accumulator column offset (fused classes)
};
struct T3Program { int ngroups; T3Group g[kT3MaxGroups]; };
struct T3Block { int16_t chan, px, py, pad_; };     // one 64-channel output block: channel offset (relative to n0), output parity

struct Tc3Params {
  int B, Hc, Wc;                    // class-local output grid (conv: Hout x Wout, deconv: Hin x Win)
  int tile_w, tile_h;               // one M tile (tile_w * tile_h == 128); a CTA tile stacks MT of them along H
  int tiles_w, tiles_h, tiles_m;    // CTA tiles per image row / column, per variant and N tile (B * tiles_h * tiles_w)
  int n_tiles_n, n_variants, total_tiles;
  int sx, sy;                       // input step per class-grid pixel (conv 2, deconv 1)
  int osx, osy;                     // output step per class-grid pixel (conv 1, deconv 2)
  int chunks0, chunks1, cin_total;
  int bn;                           // UMMA N = weight-tile rows (128 or 64)
  int ncols;                        // accumulator columns per M tile (128)
  int nblk;                         // 64-channel output blocks per M tile
  int act;
  uint32_t a_bytes, b_bytes;
  const float* scale; const float* shift;
  int* tile_ctr;
  T3Block blk[4][2];                // [variant][block]
  T3Program prog[4];                // [variant]
};

#ifdef RYK_TC_TIMELINE
// diagnostics build only (RYK_NVCC_EXTRA=-DRYK_TC_TIMELINE): per-CTA event log (clock64 of the CTA's SM), dumped to RYK_TC_TIMELINE_FILE.
// roles: 0 producer (event = A box issued), 1 MMA thread (a_full satisfied / group issued), 2 epilogue thread 0 (block begin / store issued)
constexpr int kTl3Ctas = 160, kTl3Events = 192;
__device__ long long g_tl3[kTl3Ctas * 3 * kTl3Events];
__device__ int g_tl3_n[kTl3Ctas * 3];
__device__ __forceinline__ void tl3_log(int role, int tag) {
  if (blockIdx.x >= kTl3Ctas) return;
  const int slot = blockIdx.x * 3 + role;
  const int i = g_tl3_n[slot];
  if (i + 1 < kTl3Events) { g_tl3[(size_t)slot * kTl3Events + i] = ((long long)tag << 48) | (clock64() & 0xFFFFFFFFFFFFll); g_tl3_n[slot] = i + 1; }
}
#define TL3(role, tag) tl3_log(role, tag)
#else
#define TL3(role, tag) do {} while (0)
#endif

__device__ __forceinline__ void t3_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

constexpr int kT3Threads = 352;    // warps 0-7 epilogue, 8 = scheduler + A loader, 9 = B loader, 10 = MMA issuer

// One pipeline stage = one halo box (A) + the weight tiles of all taps that read it (B region, 32 KB) behind ONE full / empty
// barrier pair: the MMA thread waits once per 8-16 MMAs.  (A first version with separate A / B rings waited per weight tile; its
// timeline -- profiles/r02_halo_v1_timeline.txt -- showed the tensor pipe idling ~40 % of the time behind the issuing thread.)
template <int MT, int STAGES> struct T3Smem {
  static constexpr uint32_t kASlot = (MT * 128 + 16) * 128;      // worst case tile_w = 16: (MT * 8 + 1) rows of 16 pixels
  static constexpr uint32_t kBRegion = 2 * 128 * 128;            // two 128-row (or four 64-row) weight tiles of 64 K
  static constexpr uint32_t kStage = kASlot + kBRegion;
  static constexpr uint32_t kOut = 128 * 128;                    // one [128 pixels][64 channels] fp16 staging block
  static constexpr uint32_t kBars = 2 * STAGES + 4 + 2 * kT3Sched;
  static constexpr size_t bytes = (size_t)STAGES * kStage + kOut + kBars * 8 + kT3Sched * 4 + 16 + 2 * 128 * 4 + 1024 + 64;
};

template <int MT, int STAGES>
__global__ void __launch_bounds__(kT3Threads, 1)
k_conv_halo(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmO, const __grid_constant__ Tc3Params p) {
  using S = T3Smem<MT, STAGES>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_out = smem + STAGES * S::kStage;
  uint64_t* full = (uint64_t*)(smem + STAGES * S::kStage + S::kOut);   // [STAGES] count 2: A loader + B loader (each arrive.expect_tx its bytes)
  uint64_t* empty = full + STAGES;                    // [STAGES] count 1: tcgen05.commit after the stage's MMAs
  uint64_t* t_full = empty + STAGES;                  // [2] accumulator stage ready for the epilogue
  uint64_t* t_empty = t_full + 2;                     // [2] accumulator stage drained (8 epilogue warps)
  uint64_t* s_full = t_empty + 2;                     // [kT3Sched] tile id published
  uint64_t* s_empty = s_full + kT3Sched;              // [kT3Sched] tile id consumed by the B loader, the MMA thread and the 8 epilogue warps
  int* s_tile = (int*)(s_empty + kT3Sched);
  uint32_t* tmem_ptr_smem = (uint32_t*)(s_tile + kT3Sched);
  float* s_scale = (float*)(((uintptr_t)(tmem_ptr_smem + 2) + 15) & ~(uintptr_t)15);     // [nblk * 64]
  float* s_shift = s_scale + 128;
  constexpr uint32_t kTmemCols = MT == 2 ? 512 : 256;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
#ifdef RYK_TC_TIMELINE
  if (lane == 0 && (warp == 8 || warp == 10 || warp == 0) && blockIdx.x < kTl3Ctas) g_tl3_n[blockIdx.x * 3 + (warp == 8 ? 0 : (warp == 10 ? 1 : 2))] = 0;
  if (threadIdx.x == 256) TL3(0, 0);
#endif
  if (threadIdx.x == 256) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA0) : "memory");
    if (p.chunks1 > 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA1) : "memory");
  }
  if (threadIdx.x == 288) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  if (threadIdx.x == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmO) : "memory");
  if (threadIdx.x == 320) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 8); }
    for (int i = 0; i < kT3Sched; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], 10); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_ptr_smem;

  const int chunks = p.chunks0 + p.chunks1;
  const int cta_h = MT * p.tile_h;                       // output rows of one CTA tile
  const uint32_t shift_bytes = (uint32_t)p.tile_w * 128u; // one halo row

  auto decode = [&](int t, int& v, int& n0, int& b, int& oy0, int& ox0) {
    int m = t % p.tiles_m; t /= p.tiles_m;
    const int nt = t % p.n_tiles_n; v = t / p.n_tiles_n;
    n0 = nt * p.ncols;
    const int tw = m % p.tiles_w; m /= p.tiles_w;
    const int th = m % p.tiles_h; b = m / p.tiles_h;
    oy0 = th * cta_h; ox0 = tw * p.tile_w;
  };
  // consumers of the tile-id ring (B loader, MMA thread, epilogue warps)
  // (called warp-uniformly: every lane waits and reads the id, one elected lane arrives for the warp)
  auto next_tile = [&](int& iq) -> int {
    const int q = iq % kT3Sched;
    mbar_wait(&s_full[q], (iq / kT3Sched) & 1);
    const int t = s_tile[q];
    __syncwarp();
    if (elect_one()) t3_arrive(&s_empty[q]);
    ++iq;
    return t;
  };

  if (warp == 8) {
    // ===== tile scheduler + A loader (warp-uniform; one elected lane issues) =====
    // First tile = blockIdx.x (no atomic on the critical path of the launch); every further tile is gridDim.x + a draw from the
    // global counter.  Draws happen only after griddepcontrol.wait: a programmatically launched successor that shares the counter
    // (the same layer replayed back to back) must not draw while this launch is still running.
    int is = 0, iq = 0;
    if (lane == 0) TL3(0, 1);
    pdl_wait();                                          // activations of the previous layer are complete from here on
    if (lane == 0) TL3(0, 2);
    int tile = blockIdx.x;
    while (true) {
      {
        const int q = iq % kT3Sched;
        mbar_wait(&s_empty[q], ((iq / kT3Sched) & 1) ^ 1);
        if (elect_one()) { s_tile[q] = tile; t3_arrive(&s_full[q]); }
        ++iq;
      }
      if (tile >= p.total_tiles) break;
      int draw = 0;
      if (lane == 0) draw = atomicAdd(p.tile_ctr, 1);    // in flight while this tile's loads are issued
      int v, n0, b, oy0, ox0;
      decode(tile, v, n0, b, oy0, ox0);
      const T3Program& P = p.prog[v];
      const int bx = ox0 * p.sx, by = oy0 * p.sy;
      for (int c = 0; c < chunks; ++c) {
        for (int g = 0; g < P.ngroups; ++g, ++is) {
          const T3Group& G = P.g[g];
          const int s = is % STAGES;
          mbar_wait(&empty[s], ((is / STAGES) & 1) ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&full[s], p.a_bytes);
            if (c < p.chunks0) tma_load_4d(smem + s * S::kStage, &tmA0, &full[s], c * kBlockK, bx + G.ax, by + G.ay, b);
            else tma_load_4d(smem + s * S::kStage, &tmA1, &full[s], (c - p.chunks0) * kBlockK, bx + G.ax, by + G.ay, b);
          }
          if (lane == 0) TL3(0, 10);
        }
      }
      draw = __shfl_sync(0xffffffffu, draw, 0);
      // total_tiles draws happen per launch (one per processed tile); the one that returns total_tiles - 1 is the last: re-arm
      if (lane == 0 && draw == p.total_tiles - 1) atomicExch(p.tile_ctr, 0);
      tile = (int)gridDim.x + draw;
    }
  } else if (warp == 9) {
    // ===== B loader: the weight tiles of every stage (a second TMA issuer; tools/mma_rate_probe.cu) =====
    int is = 0, iq = 0;
    while (true) {
      const int tile = next_tile(iq);
      if (tile >= p.total_tiles) break;
      const int v = (tile / p.tiles_m) / p.n_tiles_n, n0 = ((tile / p.tiles_m) % p.n_tiles_n) * p.ncols;
      const T3Program& P = p.prog[v];
      for (int c = 0; c < chunks; ++c) {
        for (int g = 0; g < P.ngroups; ++g, ++is) {
          const T3Group& G = P.g[g];
          const int s = is % STAGES;
          mbar_wait(&empty[s], ((is / STAGES) & 1) ^ 1);
          uint8_t* dst = smem + s * S::kStage + S::kASlot;
          if (elect_one()) {
            mbar_expect_tx(&full[s], (uint32_t)G.nb * p.b_bytes);
            for (int j = 0; j < G.nb; ++j)
              tma_load_2d(dst + j * p.b_bytes, &tmB, &full[s], G.btap[j] * p.cin_total + c * kBlockK, G.brow[j] + n0);
          }
        }
      }
    }
  } else if (warp == 10) {
    // ===== MMA issuer (warp-uniform loop; one elected lane issues the tcgen05 instructions) =====
    const uint32_t idesc = (1u << 4) | ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);
    int is = 0, iq = 0, ti = 0;
    while (true) {
      const int tile = next_tile(iq);
      if (tile >= p.total_tiles) break;
      const int v = (tile / p.tiles_m) / p.n_tiles_n;
      const T3Program& P = p.prog[v];
      const int as = ti & 1;
      mbar_wait(&t_empty[as], ((ti >> 1) & 1) ^ 1);      // the epilogue has drained this accumulator stage
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      uint32_t touched = 0;                               // accumulator column groups (of 64) already written in this tile
      const int n_stages = chunks * P.ngroups;
      // The wait for stage i + 1 is taken BEFORE the last weight tile of stage i is issued: its latency (try_wait + fence, ~150 clocks)
      // then overlaps MMAs that are already queued instead of draining the tensor pipe between stages.
      if (lane == 0) TL3(1, 20);
      mbar_wait(&full[is % STAGES], (is / STAGES) & 1);
      if (lane == 0) TL3(1, 21);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      int g = 0;
      for (int i = 0; i < n_stages; ++i, ++is) {
        const T3Group& G = P.g[g];
        if (++g == P.ngroups) g = 0;
        const int s = is % STAGES;
        const uint32_t a_addr = smem_u32(smem + s * S::kStage);
        const uint32_t b_addr = a_addr + S::kASlot;
        for (int j = 0; j < G.nb; ++j) {
          if (j == G.nb - 1 && i + 1 < n_stages) {
            mbar_wait(&full[(is + 1) % STAGES], ((is + 1) / STAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
          const uint64_t bdesc = make_sw128_desc(b_addr + (uint32_t)j * p.b_bytes);
          const uint32_t bit = 1u << (G.bcol[j] >> 6);
          const uint32_t acc0 = (touched & bit) ? 1u : 0u;
          if (elect_one()) {
#pragma unroll
            for (int h = 0; h < MT; ++h) {
              const uint64_t adesc = make_sw128_desc(a_addr + (uint32_t)h * (kBlockM * 128) + (uint32_t)G.ashift[j] * shift_bytes);
              const uint32_t tmem_d = tmem_base + (uint32_t)((as * MT + h) * 128 + G.bcol[j]);
#pragma unroll
              for (int k = 0; k < kBlockK / kUmmaK; ++k)
                umma_f16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (acc0 | (uint32_t)(k > 0)));
            }
          }
          touched |= bit;
        }
        if (elect_one()) umma_commit(&empty[s]);
        if (lane == 0) TL3(1, 23);
      }
      if (elect_one()) umma_commit(&t_full[as]);
      if (lane == 0) TL3(1, 29);
      ++ti;
    }
  } else if (warp < 8) {
    // ===== epilogue: 8 warps; warp w reads TMEM lanes 32 (w % 4) .. +31 (its pixels) and the 32-column half w / 4 of each 64-channel block =====
    int iq = 0, ti = 0;
    const int wq = warp & 3, half = warp >> 2;
    const int row = wq * 32 + lane;
    while (true) {
      const int tile = next_tile(iq);
      if (tile >= p.total_tiles) break;
      int v, n0, b, oy0, ox0;
      decode(tile, v, n0, b, oy0, ox0);
      // scale / shift of this tile's output blocks (all warps are past the previous tile's reads of s_scale after this barrier)
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int i = threadIdx.x; i < p.nblk * 64; i += 256) {
        const int ch = n0 + p.blk[v][i >> 6].chan + (i & 63);
        s_scale[i] = __ldg(p.scale + ch); s_shift[i] = __ldg(p.shift + ch);
      }
      const int as = ti & 1;
      if (threadIdx.x == 0) TL3(2, 30);
      if (lane == 0) mbar_wait(&t_full[as], (ti >> 1) & 1);
      __syncwarp();
      if (threadIdx.x == 0) TL3(2, 31);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
      for (int h = 0; h < MT; ++h) {
#pragma unroll 1
        for (int kb = 0; kb < p.nblk; ++kb) {
          // the previous TMA store must have finished READING the staging block before it is overwritten
          if (threadIdx.x == 0) { TL3(2, 32); asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); TL3(2, 33); }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          const int c0 = half * 32;
          uint32_t r[32];
          const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)((as * MT + h) * 128 + kb * 64 + c0);
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
          if (h == MT - 1 && kb == p.nblk - 1) {             // accumulator stage fully read: hand it back before the stores
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) t3_arrive(&t_empty[as]);
          }
          uint8_t* blkp = smem_out + row * 128;
          const int cbase = c0 >> 3;                            // first 16-byte chunk of this 32-channel half: 0 or 4
          const float* sc_p = s_scale + kb * 64 + c0;
          const float* sh_p = s_shift + kb * 64 + c0;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            const float4 sc0 = *reinterpret_cast<const float4*>(sc_p + j), sc1 = *reinterpret_cast<const float4*>(sc_p + j + 4);
            const float4 sh0 = *reinterpret_cast<const float4*>(sh_p + j), sh1 = *reinterpret_cast<const float4*>(sh_p + j + 4);
            const float sc[8] = {sc0.x, sc0.y, sc0.z, sc0.w, sc1.x, sc1.y, sc1.z, sc1.w};
            const float sh[8] = {sh0.x, sh0.y, sh0.z, sh0.w, sh1.x, sh1.y, sh1.z, sh1.w};
            uint32_t pk[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float v0 = fmaf(__uint_as_float(r[j + 2 * q]), sc[2 * q], sh[2 * q]);
              float v1 = fmaf(__uint_as_float(r[j + 2 * q + 1]), sc[2 * q + 1], sh[2 * q + 1]);
              if (p.act == ACT_LEAKY) { v0 = v0 > 0.f ? v0 : 0.2f * v0; v1 = v1 > 0.f ? v1 : 0.2f * v1; }
              else if (p.act == ACT_RELU) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
              __half2 h2 = __floats2half2_rn(v0, v1);
              pk[q] = *reinterpret_cast<uint32_t*>(&h2);
            }
            const int chunk = cbase + (j >> 3);
            *reinterpret_cast<uint4*>(blkp + ((chunk ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
          // generic-proxy smem writes -> async proxy, then one thread hands the block to the TMA unit (rows beyond the image are
          // clipped by the tensor map: ragged tiles need no masking)
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (threadIdx.x == 0) {
            const T3Block& K = p.blk[v][kb];
            const int xs = ox0 * p.osx + K.px, ys = (oy0 + h * p.tile_h) * p.osy + K.py;
            asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                         ::"l"(&tmO), "r"(smem_u32(smem_out)), "r"(n0 + K.chan), "r"(xs), "r"(ys), "r"(b) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            TL3(2, 34);
          }
        }
      }
      ++ti;
    }
    if (threadIdx.x == 0) { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); TL3(2, 39); }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 8) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------ host side
static int t3_env(const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; }

constexpr int kT3Stages = 3;

int tc3_init() {
  RYK_CUDA(cudaFuncSetAttribute(k_conv_halo<1, kT3Stages>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T3Smem<1, kT3Stages>::bytes));
  RYK_CUDA(cudaFuncSetAttribute(k_conv_halo<2, kT3Stages>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T3Smem<2, kT3Stages>::bytes));
  return 0;
}

// geometry of one candidate tiling
struct T3Geom { int tile_w, tile_h, mt, tiles; double cost; };

static T3Geom t3_geom(const ConvLayer& L, int tile_w, int mt, int num_sms) {
  const int Wc = L.transposed ? L.Win : L.Wout, Hc = L.transposed ? L.Hin : L.Hout;
  const int tile_h = kBlockM / tile_w, cta_h = mt * tile_h;
  const bool fused = L.transposed && L.Cout == 64;
  const int variants = L.transposed ? (fused ? 2 : 4) : 1;
  const int n_tiles_n = fused ? 1 : L.Cout / 128;
  const int tiles_m = L.B * ((Hc + cta_h - 1) / cta_h) * ((Wc + tile_w - 1) / tile_w);
  T3Geom g; g.tile_w = tile_w; g.tile_h = tile_h; g.mt = mt; g.tiles = variants * n_tiles_n * tiles_m;
  // per CTA tile and channel chunk: A boxes and weight tiles, MMA clocks (128 x N x 16 takes N / 2 clocks)
  const int groups = L.transposed ? (fused ? 3 : 2) : 8;
  const int btiles = L.transposed ? (fused ? 8 : 4) : 16;
  const int bn = fused ? 64 : 128;
  const double chunks = (L.C0 + L.C1) / 64.0;
  const double bytes = chunks * (groups * (double)(cta_h + 1) * tile_w * 128 + btiles * bn * 128.0);
  const double mma_clk = chunks * btiles * mt * 4 * (bn / 2.0);
  const double rounds = (double)((g.tiles + num_sms - 1) / num_sms);
  const double t_mma = rounds * mma_clk;
  const double t_l2 = (double)g.tiles * bytes / 5800.0;                // the chip's L2 -> SM cap in bytes per clock (B300_MICROARCH: ~6300)
  g.cost = (t_mma > t_l2 ? t_mma : t_l2) + 3000.0;                     // + prologue / epilogue tail
  return g;
}

// RYK_TC3: 1 (default) = use the halo kernel where every CTA gets several tiles (batched / long windows), 0 = never, 2 = wherever the
// shape allows (unit tests).  Measured (profiles/r02_layer_bench_*.txt): the persistent kernel's main loop runs at ~107 clocks per
// 128x128x16 MMA against ~170 for the per-tap kernel, but a CTA pays ~13k clocks of un-overlapped prologue + last epilogue; with fewer
// than ~3 tiles per SM (batch 1, 384 x 512) the two-CTAs-per-SM per-tap kernel, which overlaps those phases, is faster.
// RYK_TC3_MT / RYK_TC3_TW force the M tiles per CTA / the tile width (unit tests).
constexpr int kT3MinTilesPerSm = 3;

bool tc3_layer_config(const ConvLayer& L, int num_sms, int* tile_w, int* tile_h, int* mt) {
  const int mode = t3_env("RYK_TC3", 1);
  if (mode == 0) return false;
  const bool k2d = L.KH == 4 && L.KW == 4 && L.SH == 2 && L.SW == 2 && L.PH == 1 && L.PW == 1;
  if (!k2d || L.C0 % kBlockK != 0 || L.C1 % kBlockK != 0 || L.C0 == 0) return false;
  if (L.in_dtype != DT_F16 || L.out_dtype != DT_F16) return false;
  if (!(L.Cout % 128 == 0 || (L.transposed && L.Cout == 64))) return false;
  const int Wc = L.transposed ? L.Win : L.Wout, Hc = L.transposed ? L.Hin : L.Hout;
  if (Wc % 8 != 0 || Hc < 8) return false;
  const int force_mt = t3_env("RYK_TC3_MT", 0), force_tw = t3_env("RYK_TC3_TW", 0);
  T3Geom best; best.cost = 1e30; best.tiles = 0;
  for (int tw = 8; tw <= 16; tw *= 2) {
    if (Wc % tw != 0 || (force_tw && tw != force_tw)) continue;
    for (int m = 1; m <= 2; ++m) {
      if (force_mt && m != force_mt) continue;
      if (Hc < m * (kBlockM / tw) / 2) continue;                        // more than half of the CTA tile would be padding
      T3Geom g = t3_geom(L, tw, m, num_sms);
      if (g.cost < best.cost) best = g;
    }
  }
  if (best.tiles == 0) return false;
  if (mode == 1 && best.tiles < kT3MinTilesPerSm * num_sms) return false;
  *tile_w = best.tile_w; *tile_h = best.tile_h; *mt = best.mt;
  return true;
}

static int t3_map_act(PFN_cuTensorMapEncodeTiled_v12000 encode, CUtensorMap* m, const void* ptr, int C, int W, int H, int B, int box_w, int box_h,
                      int stride_w, int stride_h) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)kBlockK, (cuuint32_t)(box_w * stride_w), (cuuint32_t)(box_h * stride_h), 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride_w, (cuuint32_t)stride_h, 1};
  CUresult r = encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(halo kernel activation) failed: " + std::to_string((int)r)); return -1; }
  return 0;
}

// needs L.t3_tile_w / t3_tile_h / t3_mt (tc3_layer_config) and L.t3_ctr (one zero-initialised int owned by the plan)
int tc3_layer_prepare(ConvLayer& L, PFN_cuTensorMapEncodeTiled_v12000 encode) {
  RYK_CHECK(L.t3_ctr != nullptr, "halo kernel: tile counter not allocated");
  const int sx = L.transposed ? 1 : 2, osx = L.transposed ? 2 : 1;
  const int box_h = L.t3_mt * L.t3_tile_h + 1;
  if (t3_map_act(encode, &L.t3A0, L.in0, L.C0, L.Win, L.Hin, L.B, L.t3_tile_w, box_h, sx, sx)) return -1;
  if (L.C1 > 0) { if (t3_map_act(encode, &L.t3A1, L.in1, L.C1, L.Win, L.Hin, L.B, L.t3_tile_w, box_h, sx, sx)) return -1; }
  else L.t3A1 = L.t3A0;
  if (t3_map_act(encode, &L.t3O, L.out, L.Cout, L.Wout, L.Hout, L.B, L.t3_tile_w, L.t3_tile_h, osx, osx)) return -1;
  const bool fused = L.transposed && L.Cout == 64;
  const int classes = L.transposed ? 4 : 1, ntaps = L.transposed ? 4 : 16;
  cuuint64_t dims[2] = {(cuuint64_t)ntaps * (L.C0 + L.C1), (cuuint64_t)classes * L.Cout};
  cuuint64_t strides[1] = {dims[0] * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)(fused ? 64 : 128)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(&L.t3B, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(L.w_tc), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(halo kernel weights) failed: " + std::to_string((int)r)); return -1; }
  return 0;
}

int conv_tc3_run(const ConvLayer& L, cudaStream_t st, bool pdl) {
  Tc3Params p;
  memset(&p, 0, sizeof(p));
  const bool fused = L.transposed && L.Cout == 64;
  p.B = L.B; p.Hc = L.transposed ? L.Hin : L.Hout; p.Wc = L.transposed ? L.Win : L.Wout;
  p.tile_w = L.t3_tile_w; p.tile_h = L.t3_tile_h;
  const int mt = L.t3_mt, cta_h = mt * p.tile_h;
  p.tiles_w = (p.Wc + p.tile_w - 1) / p.tile_w; p.tiles_h = (p.Hc + cta_h - 1) / cta_h;
  p.tiles_m = L.B * p.tiles_w * p.tiles_h;
  p.n_variants = L.transposed ? (fused ? 2 : 4) : 1;
  p.n_tiles_n = fused ? 1 : L.Cout / 128;
  p.total_tiles = p.n_variants * p.n_tiles_n * p.tiles_m;
  p.sx = p.sy = L.transposed ? 1 : 2;
  p.osx = p.osy = L.transposed ? 2 : 1;
  p.chunks0 = L.C0 / kBlockK; p.chunks1 = L.C1 / kBlockK; p.cin_total = L.C0 + L.C1;
  p.bn = fused ? 64 : 128; p.ncols = 128; p.nblk = 2;
  p.act = L.act; p.scale = L.scale; p.shift = L.shift; p.tile_ctr = L.t3_ctr;
  p.a_bytes = (uint32_t)(cta_h + 1) * p.tile_w * 128u;
  p.b_bytes = (uint32_t)p.bn * 128u;
  if (!L.transposed) {
    // k4 s2 p1 conv: input (2 oy + ky - 1, 2 ox + kx - 1).  Row taps ky = 0 / 2 read odd input rows 2 oy - 1 and 2 oy + 1 (the same
    // stride-2 row sequence shifted by one), ky = 1 / 3 read even rows 2 oy and 2 oy + 2; one box per (kx, row parity).
    T3Program& P = p.prog[0];
    P.ngroups = 8;
    for (int kx = 0; kx < 4; ++kx) for (int yp = 0; yp < 2; ++yp) {
      T3Group& G = P.g[kx * 2 + yp];
      G.ax = (int16_t)(kx - 1); G.ay = (int16_t)(yp == 0 ? -1 : 0); G.nb = 2;
      for (int j = 0; j < 2; ++j) {
        const int ky = (yp == 0 ? 0 : 1) + 2 * j;
        G.brow[j] = 0; G.btap[j] = (int16_t)(ky * 4 + kx); G.ashift[j] = (int16_t)j; G.bcol[j] = 0;
      }
    }
    for (int kb = 0; kb < 2; ++kb) { p.blk[0][kb].chan = (int16_t)(kb * 64); p.blk[0][kb].px = 0; p.blk[0][kb].py = 0; }
  } else if (!fused) {
    // transposed conv, one output-parity class (py, px) per tile: out(2 y + py, 2 x + px) = sum over dy, dx of
    // in(y + py - 1 + dy, x + px - 1 + dx) * W[class][tap dy * 2 + dx] (k_pack_tc's layout).  One box per dx, both dy from it.
    for (int cls = 0; cls < 4; ++cls) {
      const int py = cls >> 1, px = cls & 1;
      T3Program& P = p.prog[cls];
      P.ngroups = 2;
      for (int dx = 0; dx < 2; ++dx) {
        T3Group& G = P.g[dx];
        G.ax = (int16_t)(px - 1 + dx); G.ay = (int16_t)(py - 1); G.nb = 2;
        for (int dy = 0; dy < 2; ++dy) { G.brow[dy] = cls * L.Cout; G.btap[dy] = (int16_t)(dy * 2 + dx); G.ashift[dy] = (int16_t)dy; G.bcol[dy] = 0; }
      }
      for (int kb = 0; kb < 2; ++kb) { p.blk[cls][kb].chan = (int16_t)(kb * 64); p.blk[cls][kb].px = (int16_t)px; p.blk[cls][kb].py = (int16_t)py; }
    }
  } else {
    // Cout = 64: both column parities of one row parity per tile.  Input column offsets: class px = 0 reads x - 1, x; class px = 1
    // reads x, x + 1 -> three boxes (-1, 0, +1) for four (class, dx) pairs; the classes accumulate in columns [0, 64) and [64, 128).
    for (int py = 0; py < 2; ++py) {
      T3Program& P = p.prog[py];
      P.ngroups = 3;
      for (int gi = 0; gi < 3; ++gi) {
        T3Group& G = P.g[gi];
        G.ax = (int16_t)(gi - 1); G.ay = (int16_t)(py - 1); G.nb = 0;
        for (int px = 0; px < 2; ++px) for (int dx = 0; dx < 2; ++dx) {
          if (px - 1 + dx != gi - 1) continue;
          for (int dy = 0; dy < 2; ++dy) {
            const int j = G.nb++;
            G.brow[j] = (py * 2 + px) * L.Cout; G.btap[j] = (int16_t)(dy * 2 + dx); G.ashift[j] = (int16_t)dy; G.bcol[j] = (int16_t)(px * 64);
          }
        }
      }
      for (int kb = 0; kb < 2; ++kb) { p.blk[py][kb].chan = 0; p.blk[py][kb].px = (int16_t)kb; p.blk[py][kb].py = (int16_t)py; }
    }
  }
  int num_sms = 148;
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, 0);
  const int ctas = p.total_tiles < num_sms ? p.total_tiles : num_sms;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ctas); cfg.blockDim = dim3(kT3Threads); cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  if (mt == 1) {
    cfg.dynamicSmemBytes = T3Smem<1, kT3Stages>::bytes;
    RYK_CUDA(cudaLaunchKernelEx(&cfg, k_conv_halo<1, kT3Stages>, L.t3A0, L.t3A1, L.t3B, L.t3O, p));
  } else {
    cfg.dynamicSmemBytes = T3Smem<2, kT3Stages>::bytes;
    RYK_CUDA(cudaLaunchKernelEx(&cfg, k_conv_halo<2, kT3Stages>, L.t3A0, L.t3A1, L.t3B, L.t3O, p));
  }
  RYK_CUDA(cudaGetLastError());
#ifdef RYK_TC_TIMELINE
  cudaStreamCaptureStatus cap_ = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cap_);
  if (const char* path = cap_ == cudaStreamCaptureStatusNone ? getenv("RYK_TC_TIMELINE_FILE") : nullptr) {
    cudaStreamSynchronize(st);
    static long long h[kTl3Ctas * 3 * kTl3Events]; static int hn[kTl3Ctas * 3];
    cudaMemcpyFromSymbol(h, g_tl3, sizeof(h)); cudaMemcpyFromSymbol(hn, g_tl3_n, sizeof(hn));
    if (FILE* f = fopen(path, "w")) {
      fprintf(f, "# halo kernel ctas %d mt %d tile_w %d total_tiles %d chunks %d\n", ctas, mt, p.tile_w, p.total_tiles, p.chunks0 + p.chunks1);
      for (int c = 0; c < ctas && c < kTl3Ctas; ++c) for (int r = 0; r < 3; ++r) {
        fprintf(f, "%d %d", c, r);
        for (int i = 0; i < hn[c * 3 + r]; ++i) fprintf(f, " %lld:%lld", h[((size_t)c * 3 + r) * kTl3Events + i] >> 48, h[((size_t)c * 3 + r) * kTl3Events + i] & 0xFFFFFFFFFFFFll);
        fprintf(f, "\n");
      }
      fclose(f);
    }
  }
#endif
  return 0;
}

}  // namespace ryk
