// conv.h -- convolution layer descriptors shared by the FP32 CUDA-core path (conv_direct.cu), the
// FP16 tcgen05 tensor-core path (conv_tc.cu) and the U-Net scheduler (unet.cu).
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>

#include "common.cuh"

namespace ryk {

enum Act { ACT_NONE = 0, ACT_LEAKY = 1, ACT_RELU = 2 };
enum DType { DT_F32 = 0, DT_F16 = 1 };

// One conv / transposed-conv layer over NHWC activations (1-D nets use H = 1, KH = 1).
// The input is the channel-concatenation of up to two tensors (U-Net skip "concat by pointer").
struct ConvLayer {
  int transposed = 0;
  int B = 1, Hin = 1, Win = 1, Hout = 1, Wout = 1;
  int C0 = 0, C1 = 0, Cout = 0;           // Cin = C0 + C1
  int KH = 1, KW = 1, SH = 1, SW = 1, PH = 0, PW = 0;
  int act = ACT_NONE;
  // device pointers
  const void* in0 = nullptr; const void* in1 = nullptr; int in_dtype = DT_F32;
  void* out = nullptr; int out_dtype = DT_F32;
  const float* w_direct = nullptr;        // [KH][KW][Cin][Cout] fp32
  const float* scale = nullptr;           // [Cout] folded BN scale (1 when no BN)
  const float* shift = nullptr;           // [Cout] folded bias / BN shift
  bool host_scale_valid = false;          // Cout == 1 layers: scalar scale/shift mirrored on the host
  float host_scale = 1.f, host_shift = 0.f;
  // tensor-core path (filled by tc_layer_prepare)
  const __half* w_tc = nullptr;           // conv: [Cout][KH*KW*Cin]; deconv: [4 classes][Cout][4*Cin]
  const __half* w_frag = nullptr;         // 1-D k4 layers: mma.sync B-fragment order for the fused stage-1 kernel (s1_map.h)
  float* splitk_ws = nullptr;             // [pixels][Cout] fp32 when ksplit > 1
  int ksplit = 1;
  CUtensorMap tmA0, tmA1, tmB, tmO, tmW;     // inputs, weights, fp16 output, fp32 split-K workspace
  int tile_w = 0, tile_h = 0;             // pixel tile = tile_w x tile_h = 128
  int block_n = 0;
  bool tc_ready = false;
  // halo kernel (conv_tc3.cu): persistent, dynamically scheduled; tile = t3_mt stacked M tiles of t3_tile_w x t3_tile_h pixels
  bool tc3 = false; int t3_tile_w = 0, t3_tile_h = 0, t3_mt = 0;
  int* t3_ctr = nullptr;                   // tile counter (one zero-initialised int, owned by the plan; re-armed by the kernel itself)
  CUtensorMap t3A0, t3A1, t3B, t3O;
};

// Weight repacking from the Chainer layouts the model files use:
//   conv   W: (Cout, Cin, KH, KW)      deconv W: (Cin, Cout, KH, KW)
int pack_weights_direct(const float* d_w_chainer, int transposed, int Cin, int Cout, int KH, int KW, float* d_out, cudaStream_t st);
int pack_weights_tc(const float* d_w_chainer, int transposed, int Cin, int Cout, int KH, int KW, int SH, int SW, __half* d_out, cudaStream_t st);

int conv_direct_run(const ConvLayer& L, cudaStream_t st);

bool tc_layer_eligible(const ConvLayer& L);
int tc_init();                                           // resolves cuTensorMapEncodeTiled, sets smem attributes
int tc_layer_prepare(ConvLayer& L, int num_sms);         // builds tensor maps, picks tiles / split-K (needs final pointers)
int conv_tc_run(const ConvLayer& L, cudaStream_t st);
size_t tc_splitk_ws_bytes(const ConvLayer& L, int num_sms);
void tc_force_pdl(int v);                                // -1 environment default, 0 / 1 forced

// s1_fused.cu: the whole 1-D U-Net as one cluster kernel
int s1_pack_weights(const float* d_w_chainer, int transposed, int Cin, int Cout, __half* d_out, cudaStream_t st);
int s1_fused_init();
int s1_fused_cluster_size();                             // CTAs of the cluster the kernel runs on (<= 0: unavailable)

// conv_tc3.cu
int tc3_init();
bool tc3_layer_config(const ConvLayer& L, int num_sms, int* tile_w, int* tile_h, int* mt);
int tc3_layer_prepare(ConvLayer& L, PFN_cuTensorMapEncodeTiled_v12000 encode);     // needs L.t3_ctr
int conv_tc3_run(const ConvLayer& L, cudaStream_t st, bool pdl);
bool tc_layer_wants_counter(const ConvLayer& L, int num_sms);                         // true: allocate L.t3_ctr before tc_layer_prepare

}  // namespace ryk
