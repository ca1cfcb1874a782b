// unet.cu -- the two pix2pix-style U-Nets of the hot path as static layer schedules over
// device-resident weights and per-shape activation plans.
//   stage 1: yukarin acoustic-feature converter, 1-D (SURVEY a10 / App. A.6):  (T, 9) -> (T, 9)
//   stage 2: become-yukarin spectrogram super-resolution, 2-D (a13 / App. A.7): (T, 512) -> (T, 512)
// Topology (both): enc c0 = conv k3 s1 p1 + LeakyReLU(0.2); enc c1..c7 = conv k4 s2 p1 + BN + LeakyReLU;
// dec c0..c6 = deconv k4 s2 p1 + BN + ReLU with skip concat (by pointer) before c1..c7;
// dec c7 = conv k3 s1 p1.  BatchNorm (eval, eps 2e-5) and biases arrive folded into scale/shift.
#include <vector>

#include "conv.h"
#include "engine.h"
#include "unet.h"

namespace ryk {

static int level_channels(int base, int level) {   // encoder output channels at level 0..7
  static const int mult[8] = {1, 2, 4, 8, 8, 8, 8, 8};
  return base * mult[level];
}
static int dec_out_channels(int base, int i) {     // decoder c0..c6 output channels
  static const int mult[7] = {8, 8, 8, 8, 4, 2, 1};
  return base * mult[i];
}

UNet* unet_create(int ndim, int in_ch, int out_ch, int base) {
  UNet* n = new UNet();
  n->ndim = ndim; n->in_ch = in_ch; n->out_ch = out_ch; n->base = base;
  n->layers.resize(16);
  for (int i = 0; i < 16; ++i) {
    UNetLayerW& L = n->layers[i];
    if (i == 0) { L.transposed = 0; L.cin = in_ch; L.cout = base; L.k = 3; L.s = 1; L.p = 1; L.act = ACT_LEAKY; }
    else if (i < 8) { L.transposed = 0; L.cin = level_channels(base, i - 1); L.cout = level_channels(base, i); L.k = 4; L.s = 2; L.p = 1; L.act = ACT_LEAKY; }
    else if (i < 15) {
      int d = i - 8;
      L.transposed = 1; L.k = 4; L.s = 2; L.p = 1; L.act = ACT_RELU;
      L.cout = dec_out_channels(base, d);
      L.cin = d == 0 ? level_channels(base, 7) : dec_out_channels(base, d - 1) + level_channels(base, 7 - d);
    } else { L.transposed = 0; L.cin = 2 * base; L.cout = out_ch; L.k = 3; L.s = 1; L.p = 1; L.act = ACT_NONE; }
  }
  return n;
}

static void free_plan(UNetPlan* p) {
  for (void* q : p->buffers) cudaFree(q);
  delete p;
}

void unet_destroy(UNet* n) {
  if (!n) return;
  for (auto& L : n->layers) {
    if (L.d_w_direct) cudaFree(L.d_w_direct);
    if (L.d_w_tc) cudaFree(L.d_w_tc);
    if (L.d_w_frag) cudaFree(L.d_w_frag);
    if (L.d_scale) cudaFree(L.d_scale);
    if (L.d_shift) cudaFree(L.d_shift);
  }
  for (auto& kv : n->plans) free_plan(kv.second);
  delete n;
}

// Drop every plan a destroyed session / group owned (call with its streams idle).
void unet_release_owner(UNet* n, int owner) {
  if (!n || owner == 0) return;
  for (auto it = n->plans.begin(); it != n->plans.end();) {
    if (std::get<4>(it->first) == owner) { free_plan(it->second); it = n->plans.erase(it); }
    else ++it;
  }
}

// W in the model file's (Chainer) layout: conv (Cout, Cin, k[, k]), deconv (Cin, Cout, k[, k]); host pointers.
int unet_set_layer(Engine* e, UNet* n, int idx, const float* W, const float* scale, const float* shift) {
  RYK_CHECK(idx >= 0 && idx < 16, "layer index out of range");
  UNetLayerW& L = n->layers[idx];
  int KH = n->ndim == 2 ? L.k : 1, KW = L.k;
  size_t nw = (size_t)L.cin * L.cout * KH * KW;
  float* d_tmp = nullptr;
  RYK_CUDA(cudaMalloc(&d_tmp, nw * sizeof(float)));
  RYK_CUDA(cudaMemcpyAsync(d_tmp, W, nw * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  if (!L.d_w_direct) RYK_CUDA(cudaMalloc(&L.d_w_direct, nw * sizeof(float)));
  if (pack_weights_direct(d_tmp, L.transposed, L.cin, L.cout, KH, KW, L.d_w_direct, e->stream)) return -1;
  bool tc_shape = L.k == 4 && L.cin % 64 == 0 && L.cout % 64 == 0;
  if (tc_shape) {
    if (!L.d_w_tc) RYK_CUDA(cudaMalloc(&L.d_w_tc, nw * sizeof(__half)));
    if (pack_weights_tc(d_tmp, L.transposed, L.cin, L.cout, KH, KW, n->ndim == 2 ? L.s : 1, L.s, L.d_w_tc, e->stream)) return -1;
  }
  if (n->ndim == 1 && L.k == 4 && L.s == 2 && L.cin % 64 == 0 && L.cout % 16 == 0) {
    if (!L.d_w_frag) RYK_CUDA(cudaMalloc(&L.d_w_frag, nw * sizeof(__half)));
    if (s1_pack_weights(d_tmp, L.transposed, L.cin, L.cout, L.d_w_frag, e->stream)) return -1;
  }
  if (!L.d_scale) RYK_CUDA(cudaMalloc(&L.d_scale, L.cout * sizeof(float)));
  if (!L.d_shift) RYK_CUDA(cudaMalloc(&L.d_shift, L.cout * sizeof(float)));
  RYK_CUDA(cudaMemcpyAsync(L.d_scale, scale, L.cout * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  RYK_CUDA(cudaMemcpyAsync(L.d_shift, shift, L.cout * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  RYK_CUDA(cudaFree(d_tmp));
  L.h_scale0 = scale[0]; L.h_shift0 = shift[0];
  L.loaded = true;
  return 0;
}

// Plan for a (batch, H, W) input; H = 1 for 1-D nets. precision: 0 = FP32 everywhere, 1 = FP16 activations + tcgen05.
int unet_get_plan(Engine* e, UNet* n, int B, int H, int W, int precision, UNetPlan** out, int owner) {
  for (auto& L : n->layers) RYK_CHECK(L.loaded, "U-Net layer weights not loaded");
  auto key = std::make_tuple(B, H, W, precision, owner);
  auto it = n->plans.find(key);
  if (it != n->plans.end()) { *out = it->second; return 0; }
  RYK_CHECK(W % 128 == 0 && (n->ndim == 1 || H % 128 == 0), "U-Net input extent must be a multiple of 128");
  UNetPlan* p = new UNetPlan();
  p->B = B; p->H = H; p->W = W; p->precision = precision;
  int num_sms = 148;
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, e->device);
  const int act_dt = precision ? DT_F16 : DT_F32;
  const size_t esz = precision ? 2 : 4;
  auto lvlH = [&](int l) { return n->ndim == 2 ? H >> l : 1; };
  auto lvlW = [&](int l) { return W >> l; };
  auto alloc = [&](size_t bytes, void** ptr) -> int {
    RYK_CUDA(cudaMalloc(ptr, bytes));
    RYK_CUDA(cudaMemsetAsync(*ptr, 0, bytes, e->stream));
    p->buffers.push_back(*ptr);
    return 0;
  };
  void* enc[8]; void* dec[7];
  for (int l = 0; l < 8; ++l)
    if (alloc((size_t)B * lvlH(l) * lvlW(l) * level_channels(n->base, l) * esz, &enc[l])) return -1;
  for (int d = 0; d < 7; ++d)
    if (alloc((size_t)B * lvlH(6 - d) * lvlW(6 - d) * dec_out_channels(n->base, d) * esz, &dec[d])) return -1;
  if (alloc((size_t)B * H * W * n->in_ch * sizeof(float), &p->d_in)) return -1;
  if (alloc((size_t)B * H * W * n->out_ch * sizeof(float), &p->d_out)) return -1;
  p->layers.resize(16);
  for (int i = 0; i < 16; ++i) {
    const UNetLayerW& LW = n->layers[i];
    ConvLayer& L = p->layers[i];
    L.transposed = LW.transposed; L.B = B; L.Cout = LW.cout; L.act = LW.act;
    L.KH = n->ndim == 2 ? LW.k : 1; L.KW = LW.k;
    L.SH = n->ndim == 2 ? LW.s : 1; L.SW = LW.s;
    L.PH = n->ndim == 2 ? LW.p : 0; L.PW = LW.p;
    L.w_direct = LW.d_w_direct; L.w_tc = LW.d_w_tc; L.w_frag = LW.d_w_frag; L.scale = LW.d_scale; L.shift = LW.d_shift;
    L.host_scale_valid = true; L.host_scale = LW.h_scale0; L.host_shift = LW.h_shift0;
    L.in_dtype = act_dt; L.out_dtype = act_dt;
    if (i == 0) {
      L.Hin = lvlH(0); L.Win = lvlW(0); L.Hout = lvlH(0); L.Wout = lvlW(0);
      L.C0 = n->in_ch; L.C1 = 0; L.in0 = p->d_in; L.in_dtype = DT_F32; L.out = enc[0];
    } else if (i < 8) {
      L.Hin = lvlH(i - 1); L.Win = lvlW(i - 1); L.Hout = lvlH(i); L.Wout = lvlW(i);
      L.C0 = LW.cin; L.C1 = 0; L.in0 = enc[i - 1]; L.out = enc[i];
    } else if (i < 15) {
      int d = i - 8;
      L.Hin = lvlH(7 - d); L.Win = lvlW(7 - d); L.Hout = lvlH(6 - d); L.Wout = lvlW(6 - d);
      if (d == 0) { L.C0 = LW.cin; L.C1 = 0; L.in0 = enc[7]; }
      else { L.C0 = dec_out_channels(n->base, d - 1); L.C1 = level_channels(n->base, 7 - d); L.in0 = dec[d - 1]; L.in1 = enc[7 - d]; }
      L.out = dec[d];
    } else {
      L.Hin = lvlH(0); L.Win = lvlW(0); L.Hout = lvlH(0); L.Wout = lvlW(0);
      L.C0 = n->base; L.C1 = n->base; L.in0 = dec[6]; L.in1 = enc[0]; L.out = p->d_out; L.out_dtype = DT_F32;
    }
    L.tc_ready = false;
    if (precision == 1 && L.w_tc && tc_layer_eligible(L)) {
      size_t ws = tc_splitk_ws_bytes(L, num_sms);
      if (ws) { void* w = nullptr; if (alloc(ws, &w)) return -1; L.splitk_ws = (float*)w; }
      if (tc_layer_wants_counter(L, num_sms)) { void* c = nullptr; if (alloc(16, &c)) return -1; L.t3_ctr = (int*)c; }
      if (tc_layer_prepare(L, num_sms)) return -1;
    }
  }
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  p->fused = s1_fused_eligible(n, p);
  n->plans[key] = p;
  *out = p;
  return 0;
}

// d_in / d_out live in the plan (p->d_in, p->d_out); callers fill / read them stream-ordered.
int unet_forward(Engine* e, UNetPlan* p, cudaStream_t st, int first_layer, int last_layer) {
  if (p->fused && e->s1_fused && first_layer == 0 && last_layer == 15) return s1_fused_run(e, p, st);
  const bool prof = e->profile && p->H > 1;        // time the k4 layers (1..14) of the 2-D (stage-2) net
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  for (int i = first_layer; i <= last_layer; ++i) {
    const ConvLayer& L = p->layers[i];
    if (prof && i == 1) { RYK_CUDA(cudaEventCreate(&ev0)); RYK_CUDA(cudaEventCreate(&ev1)); RYK_CUDA(cudaEventRecord(ev0, st)); }
    int rc = L.tc_ready ? conv_tc_run(L, st) : conv_direct_run(L, st);
    if (rc) return rc;
    if (prof && i == 14 && ev0) { RYK_CUDA(cudaEventRecord(ev1, st)); e->prof_events.emplace_back(ev0, ev1); }
    e->launches += (L.tc_ready && L.ksplit > 1) ? 2 : 1;     // split-K: kernel + reduce
  }
  return 0;
}

}  // namespace ryk
