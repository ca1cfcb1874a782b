// api.cu -- the C ABI of libryk.so (include/ryk.h).  Host pointers in, host pointers out; every
// entry point uploads its arguments, runs the CUDA path on the engine's stream and downloads the
// result.  The device-resident streaming session lives in session.cu.
#include <math.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <algorithm>
#include <vector>

#include "../../include/ryk.h"
#include "conv.h"
#include "engine.h"
#include "fft.cuh"
#include "features.h"
#include "synth.h"
#include "unet.h"

namespace ryk {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }

void fft_fill_twiddles(double2* t) {
  for (int k = 0; k < kTwiddleN / 2; ++k) t[k] = make_double2(cos(2.0 * kPi * k / kTwiddleN), -sin(2.0 * kPi * k / kTwiddleN));
}

int engine_scratch(Engine* e, size_t bytes, void** out) {
  if (bytes > e->scratch_bytes) {
    RYK_CUDA(cudaStreamSynchronize(e->stream));
    if (e->d_scratch) RYK_CUDA(cudaFree(e->d_scratch));
    size_t cap = bytes + bytes / 4 + (1 << 20);
    RYK_CUDA(cudaMalloc(&e->d_scratch, cap));
    e->scratch_bytes = cap;
  }
  *out = e->d_scratch;
  return 0;
}

int engine_pinned(Engine* e, size_t bytes, void** out) {
  if (bytes > e->pinned_bytes) {
    RYK_CUDA(cudaStreamSynchronize(e->stream));
    if (e->h_pinned) RYK_CUDA(cudaFreeHost(e->h_pinned));
    size_t cap = bytes + bytes / 4 + (1 << 16);
    RYK_CUDA(cudaMallocHost(&e->h_pinned, cap));
    e->pinned_bytes = cap;
  }
  *out = e->h_pinned;
  return 0;
}

struct Arena {
  char* base; size_t off = 0;
  explicit Arena(void* b) : base((char*)b) {}
  template <typename T> T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = (T*)(base + off);
    off += count * sizeof(T);
    return p;
  }
};
static size_t arena_need(std::initializer_list<size_t> sizes) {
  size_t t = 0;
  for (size_t s : sizes) t = ((t + 255) & ~(size_t)255) + s;
  return t + 256;
}

int dio_get_plan(Engine* e, int n, int fs, double frame_period, double f0_floor, double f0_ceil, DioPlan** out) {
  // the f0 method is part of the key: switching it never reuses a plan built for the other extractor
  auto key = std::make_tuple(n, fs + 1000000 * e->f0_method, (int)lround(frame_period * 1000), (int)lround(f0_floor * 1000), (int)lround(f0_ceil * 1000));
  auto it = e->dio_plans.find(key);
  if (it != e->dio_plans.end()) { *out = it->second; return 0; }
  DioPlan* p = nullptr;
  if (dio_plan_create(e, n, fs, frame_period, f0_floor, f0_ceil, &p, e->f0_method)) return -1;
  e->dio_plans[key] = p;
  *out = p;
  return 0;
}

static UNet*& stage_net(Engine* e, int stage) { return stage == 1 ? e->stage1 : e->stage2; }

static int upload_vec(float** d, const float* h, int n) {
  if (*d) cudaFree(*d);
  RYK_CUDA(cudaMalloc(d, sizeof(float) * n));
  RYK_CUDA(cudaMemcpy(*d, h, sizeof(float) * n, cudaMemcpyHostToDevice));
  return 0;
}

static int ensure_stage1_stats(Engine* e, int C) {
  if (e->d_s1_in_mean && (int)e->s1_in_mean.size() == C) return 0;
  std::vector<float> zero(C, 0.f), one(C, 1.f);
  e->s1_in_mean = zero; e->s1_in_std = one; e->s1_out_mean = zero; e->s1_out_std = one;
  if (upload_vec(&e->d_s1_in_mean, zero.data(), C)) return -1;
  if (upload_vec(&e->d_s1_in_std, one.data(), C)) return -1;
  if (upload_vec(&e->d_s1_out_mean, zero.data(), C)) return -1;
  if (upload_vec(&e->d_s1_out_std, one.data(), C)) return -1;
  return 0;
}

__global__ void k_affine_rows(const float* __restrict__ y, int T, int C, const float* __restrict__ scale, const float* __restrict__ shift, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < T * C) out[i] = __fadd_rn(__fmul_rn(y[i], scale[i % C]), shift[i % C]);
}

__global__ void k_f32_to_f16(const float* __restrict__ a, __half* __restrict__ b, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) b[i] = __float2half_rn(a[i]);
}
__global__ void k_f16_to_f32(const __half* __restrict__ a, float* __restrict__ b, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) b[i] = __half2float(a[i]);
}

__global__ void k_f0_convert(const float* __restrict__ f0, const uint8_t* __restrict__ voiced, int T, double mu_i, double sd_i,
                             double mu_t, double sd_t, int has_stats, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  float v = 0.f;
  if (voiced[i]) v = has_stats ? (float)exp((log((double)f0[i]) - mu_i) / sd_i * sd_t + mu_t) : f0[i];
  out[i] = v;
}

// stage-1 forward on device buffers: x already normalised+padded in plan->d_in; returns plan
static int stage1_plan_for(Engine* e, int Tp, UNetPlan** plan) {
  RYK_CHECK(e->stage1 != nullptr, "stage-1 model not loaded");
  return unet_get_plan(e, e->stage1, 1, 1, Tp, e->precision, plan);
}
static int stage2_plan_for(Engine* e, int Tp, UNetPlan** plan) {
  RYK_CHECK(e->stage2 != nullptr, "stage-2 model not loaded");
  return unet_get_plan(e, e->stage2, 1, Tp, 512, e->precision, plan);
}

}  // namespace ryk

using namespace ryk;

struct ryk_engine { Engine impl; };
static Engine* E(ryk_engine* e) { return &e->impl; }

extern "C" {

int ryk_abi_version(void) { return 1; }
const char* ryk_last_error(void) { return g_err.c_str(); }

int ryk_engine_create(int device, ryk_engine** out) {
  RYK_CHECK(out != nullptr, "null out pointer");
  // A session drives 7 streams and a group of 8 sessions 57: with the default 8 hardware work queues independent streams share a queue
  // and a stream that waits on an event holds up its queue-mates (measured: the steps of a group of 8 ran strictly one after another,
  // 1280 chunks/s; with 32 queues they overlap, 1678; profiles/r02b_max_connections_groups.txt).  Read by the driver when the CUDA
  // context is created, so it only takes effect if nothing initialised CUDA earlier in this process; never overrides the user's value.
  setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
  int count = 0;
  RYK_CUDA(cudaGetDeviceCount(&count));
  RYK_CHECK(count > 0 && device < count, "no such CUDA device (libryk has no CPU fallback)");
  RYK_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  RYK_CUDA(cudaGetDeviceProperties(&prop, device));
  RYK_CHECK(prop.major == 10, "libryk is built for sm_100a (B200) only");
  ryk_engine* h = new ryk_engine();
  Engine* e = &h->impl;
  e->device = device;
  RYK_CUDA(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  std::vector<double2> tw(kTwiddleN / 2);
  fft_fill_twiddles(tw.data());
  RYK_CUDA(cudaMalloc(&e->d_twiddle, sizeof(double2) * tw.size()));
  RYK_CUDA(cudaMemcpy(e->d_twiddle, tw.data(), sizeof(double2) * tw.size(), cudaMemcpyHostToDevice));
  if (analysis_kernels_init()) return -1;
  if (tc_init()) return -1;
  if (s1_fused_init()) return -1;
  { const char* ev = getenv("RYK_S1_FUSED"); e->s1_fused = !(ev && atoi(ev) == 0); }
  RYK_CUDA(cudaMalloc(&e->d_colmin, sizeof(float) * 64 * 512));   // stage-2 prologue scratch (never allocated inside a graph capture)
  *out = h;
  return 0;
}

int ryk_engine_destroy(ryk_engine* h) {
  if (!h) return 0;
  Engine* e = E(h);
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  for (auto& kv : e->dio_plans) dio_plan_free(kv.second);
  unet_destroy(e->stage1); unet_destroy(e->stage2);
  crepe_destroy();
  for (Synth* s : e->synths) synth_destroy(s);
  session_destroy_all(e);
  void* ptrs[] = {e->d_colmin, e->d_twiddle, e->d_jump, e->d_G, e->d_H, e->d_s1_in_mean, e->d_s1_in_std, e->d_s1_out_mean, e->d_s1_out_std, e->d_scratch};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (e->h_pinned) cudaFreeHost(e->h_pinned);
  cudaStreamDestroy(e->stream);
  delete h;
  return 0;
}

int ryk_engine_set_precision(ryk_engine* h, int mode) {
  RYK_CHECK(mode == 0 || mode == 1, "precision mode must be 0 (fp32) or 1 (fp16 tensor core)");
  E(h)->precision = mode;
  return 0;
}
int ryk_engine_get_precision(ryk_engine* h) { return E(h)->precision; }
// Stage 1 as one cluster kernel (default) or as the 16-layer sequence; returns the cluster size in use (<= 0: kernel unavailable).
// Sessions capture their stage-1 graphs at creation: switch before creating them.
int ryk_engine_set_stage1_fused(ryk_engine* h, int enable) { E(h)->s1_fused = enable != 0; return s1_fused_cluster_size(); }
long long ryk_engine_launch_count(ryk_engine* h) { return E(h)->launches; }
int ryk_engine_synchronize(ryk_engine* h) { RYK_CUDA(cudaSetDevice(E(h)->device)); RYK_CUDA(cudaDeviceSynchronize()); return 0; }

int ryk_engine_profile(ryk_engine* h, int enable) { E(h)->profile = enable != 0; return 0; }
// Device time (ms) of the stage-2 k4 (tensor-core) layer block over all forwards since the last read:
//   *stage2_ms_total = sum of the per-forward durations (CUDA events on the stream each forward runs on),
//   *stage2_ms_union = length of the union of those intervals.  A single session alternates its forwards between two streams, so
//   consecutive forwards overlap: the sum then counts the shared time twice; the union is the time during which the block was running.
int ryk_engine_profile_read2(ryk_engine* h, double* stage2_ms_total, double* stage2_ms_union, int* stage2_runs) {
  Engine* e = E(h);
  RYK_CUDA(cudaDeviceSynchronize());
  double tot = 0.0, uni = 0.0;
  std::vector<std::pair<double, double>> iv;
  for (auto& pr : e->prof_events) {
    float ms = 0.f, off = 0.f;
    RYK_CUDA(cudaEventElapsedTime(&ms, pr.first, pr.second));
    RYK_CUDA(cudaEventElapsedTime(&off, e->prof_events.front().first, pr.first));
    tot += ms;
    iv.emplace_back((double)off, (double)off + (double)ms);
  }
  std::sort(iv.begin(), iv.end());
  double cur0 = 0.0, cur1 = -1.0;
  for (auto& x : iv) {
    if (cur1 < cur0 || x.first > cur1) { if (cur1 >= cur0) uni += cur1 - cur0; cur0 = x.first; cur1 = x.second; }
    else if (x.second > cur1) cur1 = x.second;
  }
  if (cur1 >= cur0 && !iv.empty()) uni += cur1 - cur0;
  for (auto& pr : e->prof_events) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
  if (stage2_ms_total) *stage2_ms_total = tot;
  if (stage2_ms_union) *stage2_ms_union = uni;
  if (stage2_runs) *stage2_runs = (int)e->prof_events.size();
  e->prof_events.clear();
  return 0;
}
int ryk_engine_profile_read(ryk_engine* h, double* stage2_ms_total, int* stage2_runs) {
  return ryk_engine_profile_read2(h, stage2_ms_total, nullptr, stage2_runs);
}

// device-side stopwatch on the engine's stream (bench.py brackets its timed region with it)
int ryk_engine_timer_start(ryk_engine* h) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  for (int i = 0; i < 2; ++i) if (!e->timer_ev[i]) RYK_CUDA(cudaEventCreate(&e->timer_ev[i]));
  RYK_CUDA(cudaDeviceSynchronize());
  RYK_CUDA(cudaEventRecord(e->timer_ev[0], e->stream));
  return session_streams_fork(e, e->timer_ev[0]);      // the pipelined sessions run on their own streams
}
int ryk_engine_timer_stop(ryk_engine* h, float* elapsed_ms) {
  Engine* e = E(h);
  RYK_CHECK(e->timer_ev[0] != nullptr, "timer was not started");
  if (session_streams_join(e)) return -1;
  RYK_CUDA(cudaEventRecord(e->timer_ev[1], e->stream));
  RYK_CUDA(cudaEventSynchronize(e->timer_ev[1]));
  RYK_CUDA(cudaEventElapsedTime(elapsed_ms, e->timer_ev[0], e->timer_ev[1]));
  return 0;
}

int ryk_world_num_frames(int n, int fs, double frame_period_ms) { return (int)(1000.0 * n / fs / frame_period_ms) + 1; }

int ryk_world_f0(ryk_engine* h, const float* wave, int n, int fs, double fp, double f0_floor, double f0_ceil, double* f0, double* t) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(n > 0, "empty wave");
  DioPlan* plan = nullptr;
  if (dio_get_plan(e, n, fs, fp, f0_floor, f0_ceil, &plan)) return -1;
  void* scratch = nullptr;
  if (engine_scratch(e, sizeof(float) * n + 256, &scratch)) return -1;
  float* d_x = (float*)scratch;
  RYK_CUDA(cudaMemcpyAsync(d_x, wave, sizeof(float) * n, cudaMemcpyHostToDevice, e->stream));
  if (dio_stonemask_run(e, plan, d_x, e->stream)) return -1;
  e->launches += 9;
  int nf = dio_plan_frames(plan);
  RYK_CUDA(cudaMemcpyAsync(f0, dio_plan_f0(plan), sizeof(double) * nf, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  if (t) for (int i = 0; i < nf; ++i) t[i] = i * fp / 1000.0;
  return 0;
}

int ryk_world_analyze(ryk_engine* h, const float* wave, int n, int fs, double fp, double f0_floor, double f0_ceil, int fft_length,
                      int order, double alpha, const double* f0_override, float* f0, float* sp, float* ap, float* mc, uint8_t* voiced) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  int hop = (int)(fs * fp / 1000.0);
  RYK_CHECK(hop > 0, "bad frame period");
  int n_out = n / hop;
  if (n_out <= 0) return 0;
  int nb = fft_length / 2 + 1;
  if (sptk_prepare(e, order, alpha, fft_length)) return -1;
  DioPlan* plan = nullptr;
  if (dio_get_plan(e, n, fs, fp, f0_floor, f0_ceil, &plan)) return -1;
  void* scratch = nullptr;
  size_t need = arena_need({sizeof(float) * n, sizeof(float) * n_out, sizeof(float) * n_out * nb, sizeof(float) * n_out * nb,
                            sizeof(float) * n_out * (order + 1), (size_t)n_out});
  if (engine_scratch(e, need, &scratch)) return -1;
  Arena A(scratch);
  float* d_x = A.take<float>(n);
  float* d_f0 = A.take<float>(n_out);
  float* d_sp = A.take<float>((size_t)n_out * nb);
  float* d_ap = A.take<float>((size_t)n_out * nb);
  float* d_mc = A.take<float>((size_t)n_out * (order + 1));
  uint8_t* d_v = A.take<uint8_t>(n_out);
  RYK_CUDA(cudaMemcpyAsync(d_x, wave, sizeof(float) * n, cudaMemcpyHostToDevice, e->stream));
  if (f0_override) {
    RYK_CUDA(cudaMemcpyAsync(dio_plan_f0_mut(plan), f0_override, sizeof(double) * dio_plan_frames(plan), cudaMemcpyHostToDevice, e->stream));
  } else {
    if (dio_stonemask_run(e, plan, d_x, e->stream)) return -1;
    e->launches += 9;
  }
  if (spectral_analysis_run(e, d_x, n, fs, fp, dio_plan_f0(plan), n_out, fft_length, order, d_sp, d_ap, d_mc, d_f0, d_v, e->stream)) return -1;
  e->launches += 3;
  if (f0) RYK_CUDA(cudaMemcpyAsync(f0, d_f0, sizeof(float) * n_out, cudaMemcpyDeviceToHost, e->stream));
  if (sp) RYK_CUDA(cudaMemcpyAsync(sp, d_sp, sizeof(float) * n_out * nb, cudaMemcpyDeviceToHost, e->stream));
  if (ap) RYK_CUDA(cudaMemcpyAsync(ap, d_ap, sizeof(float) * n_out * nb, cudaMemcpyDeviceToHost, e->stream));
  if (mc) RYK_CUDA(cudaMemcpyAsync(mc, d_mc, sizeof(float) * n_out * (order + 1), cudaMemcpyDeviceToHost, e->stream));
  if (voiced) RYK_CUDA(cudaMemcpyAsync(voiced, d_v, n_out, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

int ryk_silence_mask(ryk_engine* h, const float* wave, int n, int frame_length, int hop, double threshold_db, int n_frames, uint8_t* mask) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  if (n_frames <= 0) return 0;
  void* scratch = nullptr;
  size_t need = arena_need({sizeof(float) * (size_t)(n > 0 ? n : 1), sizeof(double) * n_frames, (size_t)n_frames, sizeof(int) * n_frames, sizeof(int) * 2});
  if (engine_scratch(e, need, &scratch)) return -1;
  Arena A(scratch);
  float* d_x = A.take<float>(n > 0 ? n : 1);
  double* d_mse = A.take<double>(n_frames);
  uint8_t* d_mask = A.take<uint8_t>(n_frames);
  int* d_index = A.take<int>(n_frames);
  int* d_count = A.take<int>(2);
  if (n > 0) RYK_CUDA(cudaMemcpyAsync(d_x, wave, sizeof(float) * n, cudaMemcpyHostToDevice, e->stream));
  if (gate_mask_run(e, d_x, n, frame_length, hop, threshold_db, n_frames, d_mse, d_mask, d_index, d_count, e->stream)) return -1;
  RYK_CUDA(cudaMemcpyAsync(mask, d_mask, n_frames, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

int ryk_model_create(ryk_engine* h, int stage, int in_ch, int out_ch, int base) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(stage == 1 || stage == 2, "stage must be 1 or 2");
  UNet*& net = stage_net(e, stage);
  if (net) { RYK_CUDA(cudaStreamSynchronize(e->stream)); unet_destroy(net); net = nullptr; }
  net = unet_create(stage == 1 ? 1 : 2, in_ch, out_ch, base);
  return 0;
}

int ryk_model_set_layer(ryk_engine* h, int stage, int layer, const float* W, const float* scale, const float* shift) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  UNet* net = stage_net(e, stage);
  RYK_CHECK(net != nullptr, "ryk_model_create was not called for this stage");
  return unet_set_layer(e, net, layer, W, scale, shift);
}

int ryk_model_layer_shape(ryk_engine* h, int stage, int layer, int* transposed, int* cin, int* cout, int* k) {
  UNet* net = stage_net(E(h), stage);
  RYK_CHECK(net != nullptr && layer >= 0 && layer < 16, "no such layer");
  const UNetLayerW& L = net->layers[layer];
  *transposed = L.transposed; *cin = L.cin; *cout = L.cout; *k = L.k;
  return 0;
}

int ryk_stage1_set_stats(ryk_engine* h, int C, const float* in_mean, const float* in_std, const float* out_mean, const float* out_std) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  e->s1_in_mean.assign(in_mean, in_mean + C); e->s1_in_std.assign(in_std, in_std + C);
  e->s1_out_mean.assign(out_mean, out_mean + C); e->s1_out_std.assign(out_std, out_std + C);
  if (upload_vec(&e->d_s1_in_mean, in_mean, C)) return -1;
  if (upload_vec(&e->d_s1_in_std, in_std, C)) return -1;
  if (upload_vec(&e->d_s1_out_mean, out_mean, C)) return -1;
  if (upload_vec(&e->d_s1_out_std, out_std, C)) return -1;
  return 0;
}

int ryk_f0_set_stats(ryk_engine* h, double in_mean, double in_std, double target_mean, double target_std) {
  Engine* e = E(h);
  e->f0_in_mean = in_mean; e->f0_in_std = in_std; e->f0_tgt_mean = target_mean; e->f0_tgt_std = target_std;
  e->has_f0_stats = true;
  return 0;
}

int ryk_stage1_convert(ryk_engine* h, const float* x, int T, float* y) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(e->stage1 != nullptr, "stage-1 model not loaded");
  RYK_CHECK(T > 0, "empty input");
  const int C = e->stage1->in_ch, Co = e->stage1->out_ch;
  if (ensure_stage1_stats(e, C)) return -1;
  const int Tp = T + (128 - T % 128);
  UNetPlan* plan = nullptr;
  if (stage1_plan_for(e, Tp, &plan)) return -1;
  void* scratch = nullptr;
  if (engine_scratch(e, arena_need({sizeof(float) * T * C, sizeof(float) * T * Co, sizeof(int) * 2}), &scratch)) return -1;
  Arena A(scratch);
  float* d_x = A.take<float>((size_t)T * C);
  float* d_y = A.take<float>((size_t)T * Co);
  int* d_count = A.take<int>(2);
  int cnt[2] = {T, Tp};
  RYK_CUDA(cudaMemcpyAsync(d_x, x, sizeof(float) * T * C, cudaMemcpyHostToDevice, e->stream));
  RYK_CUDA(cudaMemcpyAsync(d_count, cnt, sizeof(cnt), cudaMemcpyHostToDevice, e->stream));
  if (stage1_prologue_run(e, d_x, nullptr, d_count, C, (float*)plan->d_in, Tp, e->stream)) return -1;
  if (unet_forward(e, plan, e->stream)) return -1;
  k_affine_rows<<<(T * Co + 255) / 256, 256, 0, e->stream>>>((const float*)plan->d_out, T, Co, e->d_s1_out_std, e->d_s1_out_mean, d_y);
  e->launches++;
  RYK_CUDA(cudaMemcpyAsync(y, d_y, sizeof(float) * T * Co, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

int ryk_f0_convert(ryk_engine* h, const float* f0, const uint8_t* voiced, int T, float* out) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  if (T <= 0) return 0;
  void* scratch = nullptr;
  if (engine_scratch(e, arena_need({sizeof(float) * T, (size_t)T, sizeof(float) * T}), &scratch)) return -1;
  Arena A(scratch);
  float* d_f0 = A.take<float>(T); uint8_t* d_v = A.take<uint8_t>(T); float* d_o = A.take<float>(T);
  RYK_CUDA(cudaMemcpyAsync(d_f0, f0, sizeof(float) * T, cudaMemcpyHostToDevice, e->stream));
  RYK_CUDA(cudaMemcpyAsync(d_v, voiced, T, cudaMemcpyHostToDevice, e->stream));
  k_f0_convert<<<(T + 127) / 128, 128, 0, e->stream>>>(d_f0, d_v, T, e->f0_in_mean, e->f0_in_std, e->f0_tgt_mean, e->f0_tgt_std,
                                                      e->has_f0_stats ? 1 : 0, d_o);
  e->launches++;
  RYK_CUDA(cudaMemcpyAsync(out, d_o, sizeof(float) * T, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

int ryk_mc2sp(ryk_engine* h, const float* mc, int T, int order, double alpha, int fftlen, double* sp) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  if (T <= 0) return 0;
  if (sptk_prepare(e, order, alpha, fftlen)) return -1;
  int nb = fftlen / 2 + 1;
  void* scratch = nullptr;
  if (engine_scratch(e, arena_need({sizeof(float) * T * (order + 1), sizeof(double) * T * nb}), &scratch)) return -1;
  Arena A(scratch);
  float* d_mc = A.take<float>((size_t)T * (order + 1));
  double* d_sp = A.take<double>((size_t)T * nb);
  RYK_CUDA(cudaMemcpyAsync(d_mc, mc, sizeof(float) * T * (order + 1), cudaMemcpyHostToDevice, e->stream));
  if (mc2sp_run(e, d_mc, T, order, fftlen, 0.0, nullptr, d_sp, e->stream)) return -1;
  RYK_CUDA(cudaMemcpyAsync(sp, d_sp, sizeof(double) * T * nb, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

int ryk_stage2_convert(ryk_engine* h, const float* sp, int T, float* out) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(T > 0, "empty input");
  const int nb = 513;
  const int Tp = T + (128 - T % 128);
  UNetPlan* plan = nullptr;
  if (stage2_plan_for(e, Tp, &plan)) return -1;
  void* scratch = nullptr;
  if (engine_scratch(e, arena_need({sizeof(float) * T * nb, sizeof(float) * T * nb}), &scratch)) return -1;
  Arena A(scratch);
  float* d_sp = A.take<float>((size_t)T * nb);
  float* d_out = A.take<float>((size_t)T * nb);
  RYK_CUDA(cudaMemcpyAsync(d_sp, sp, sizeof(float) * T * nb, cudaMemcpyHostToDevice, e->stream));
  if (sr_prologue_run(e, d_sp, T, Tp, nb, (float*)plan->d_in, e->stream)) return -1;
  if (unet_forward(e, plan, e->stream)) return -1;
  if (sr_epilogue_run(e, (const float*)plan->d_out, T, nb, d_out, e->stream)) return -1;
  RYK_CUDA(cudaMemcpyAsync(out, d_out, sizeof(float) * T * nb, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

int ryk_convert_window(ryk_engine* h, const float* wave, int n_wave, int fs, int frame_length, int hop, double threshold_db,
                       const float* f0, const float* ap, const float* mc, const uint8_t* voiced, int T, int order, double alpha,
                       int fftlen, float* f0_out, float* ap_out, float* sp_out, uint8_t* voiced_out, float* mc_out) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(T > 0, "empty window");
  RYK_CHECK(e->stage1 && e->stage2, "models not loaded");
  const int nb = fftlen / 2 + 1, C = order + 1;
  RYK_CHECK(nb == 513, "stage 2 expects 513-bin spectra");
  RYK_CHECK(e->stage1->in_ch == C && e->stage1->out_ch == C, "stage-1 channel count does not match order + 1");
  if (sptk_prepare(e, order, alpha, fftlen)) return -1;
  if (ensure_stage1_stats(e, C)) return -1;
  ConvertBuffers cb;
  if (convert_buffers_get(e, T, n_wave, nb, C, &cb)) return -1;
  cudaStream_t st = e->stream;
  RYK_CUDA(cudaMemcpyAsync(cb.d_wave, wave, sizeof(float) * n_wave, cudaMemcpyHostToDevice, st));
  RYK_CUDA(cudaMemcpyAsync(cb.d_f0, f0, sizeof(float) * T, cudaMemcpyHostToDevice, st));
  RYK_CUDA(cudaMemcpyAsync(cb.d_ap, ap, sizeof(float) * T * nb, cudaMemcpyHostToDevice, st));
  RYK_CUDA(cudaMemcpyAsync(cb.d_mc, mc, sizeof(float) * T * C, cudaMemcpyHostToDevice, st));
  RYK_CUDA(cudaMemcpyAsync(cb.d_voiced, voiced, T, cudaMemcpyHostToDevice, st));
  if (convert_window_device(e, cb, T, n_wave, frame_length, hop, threshold_db, order, fftlen, st)) return -1;
  RYK_CUDA(cudaMemcpyAsync(f0_out, cb.d_f0_out, sizeof(float) * T, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaMemcpyAsync(ap_out, cb.d_ap_out, sizeof(float) * T * nb, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaMemcpyAsync(sp_out, cb.d_sp_out, sizeof(float) * T * nb, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaMemcpyAsync(voiced_out, cb.d_voiced_out, T, cudaMemcpyDeviceToHost, st));
  if (mc_out) RYK_CUDA(cudaMemcpyAsync(mc_out, cb.d_mc_out, sizeof(float) * T * C, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ---- synthesizer -------------------------------------------------------------------------------
static Synth* get_synth(Engine* e, int id) { return (id >= 0 && id < (int)e->synths.size()) ? e->synths[id] : nullptr; }

int ryk_synth_create(ryk_engine* h, int fs, double fp, int fft_size, int buffer_size, int number_of_pointers, int* synth_id) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  (void)number_of_pointers;     // world4py's pointer ring is replaced by a frame ring owned by the library
  Synth* s = nullptr;
  if (synth_create(e, fs, fp, fft_size, buffer_size, 4096, &s)) return -1;
  e->synths.push_back(s);
  *synth_id = (int)e->synths.size() - 1;
  return 0;
}

int ryk_synth_destroy(ryk_engine* h, int id) {
  Engine* e = E(h);
  Synth* s = get_synth(e, id);
  RYK_CHECK(s != nullptr, "no such synthesizer");
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  synth_destroy(s);
  e->synths[id] = nullptr;
  return 0;
}

static int synth_upload(Engine* e, Synth* s, const double* f0, int n, const float* sp, const float* ap, double** d_f0, float** d_sp, float** d_ap,
                        double** d_out, int max_blocks) {
  int nb = s->dev.fft_size / 2 + 1;
  void* scratch = nullptr;
  size_t need = arena_need({sizeof(double) * n, sizeof(float) * n * nb, sizeof(float) * n * nb, sizeof(double) * (size_t)max_blocks * s->dev.buffer_size});
  if (engine_scratch(e, need, &scratch)) return -1;
  Arena A(scratch);
  *d_f0 = A.take<double>(n); *d_sp = A.take<float>((size_t)n * nb); *d_ap = A.take<float>((size_t)n * nb);
  *d_out = A.take<double>((size_t)max_blocks * s->dev.buffer_size);
  if (n > 0) {
    RYK_CUDA(cudaMemcpyAsync(*d_f0, f0, sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
    RYK_CUDA(cudaMemcpyAsync(*d_sp, sp, sizeof(float) * n * nb, cudaMemcpyHostToDevice, e->stream));
    RYK_CUDA(cudaMemcpyAsync(*d_ap, ap, sizeof(float) * n * nb, cudaMemcpyHostToDevice, e->stream));
  }
  return 0;
}

int ryk_synth_add_parameters(ryk_engine* h, int id, const double* f0, int n, const float* sp, const float* ap) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  Synth* s = get_synth(e, id);
  RYK_CHECK(s != nullptr, "no such synthesizer");
  if (n <= 0) return 1;
  double* d_f0; float *d_sp, *d_ap; double* d_out;
  if (synth_upload(e, s, f0, n, sp, ap, &d_f0, &d_sp, &d_ap, &d_out, 1)) return -1;
  long long before = s->host_cum_frames;
  if (synth_add_async(e, s, d_f0, n, d_sp, d_ap, e->stream)) return -1;
  int status = 0;
  RYK_CUDA(cudaMemcpyAsync(&status, (char*)s->dev.state + offsetof(SynthState, last_add_status), sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  if (!status) s->host_cum_frames = before;
  return status;
}

int ryk_synth_synthesis2(ryk_engine* h, int id, double* buffer) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  Synth* s = get_synth(e, id);
  RYK_CHECK(s != nullptr, "no such synthesizer");
  void* scratch = nullptr;
  if (engine_scratch(e, sizeof(double) * s->dev.buffer_size + 256, &scratch)) return -1;
  double* d_out = (double*)scratch;
  if (synth_drain_async(e, s, d_out, 1, e->stream)) return -1;
  int blocks = 0;
  RYK_CUDA(cudaMemcpyAsync(&blocks, (char*)s->dev.state + offsetof(SynthState, blocks_out), sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaMemcpyAsync(buffer, d_out, sizeof(double) * s->dev.buffer_size, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return blocks > 0 ? 1 : 0;
}

int ryk_synth_decode(ryk_engine* h, int id, const double* f0, int n, const float* sp, const float* ap, double* out, int max_blocks, int* n_blocks) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  Synth* s = get_synth(e, id);
  RYK_CHECK(s != nullptr, "no such synthesizer");
  RYK_CHECK(max_blocks > 0, "max_blocks must be positive");
  double* d_f0; float *d_sp, *d_ap; double* d_out;
  if (synth_upload(e, s, f0, n, sp, ap, &d_f0, &d_sp, &d_ap, &d_out, max_blocks)) return -1;
  if (n > 0 && synth_add_async(e, s, d_f0, n, d_sp, d_ap, e->stream)) return -1;
  if (synth_drain_async(e, s, d_out, max_blocks, e->stream)) return -1;
  int blocks = 0;
  RYK_CUDA(cudaMemcpyAsync(&blocks, (char*)s->dev.state + offsetof(SynthState, blocks_out), sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  if (blocks > 0) {
    RYK_CUDA(cudaMemcpyAsync(out, d_out, sizeof(double) * (size_t)blocks * s->dev.buffer_size, cudaMemcpyDeviceToHost, e->stream));
    RYK_CUDA(cudaStreamSynchronize(e->stream));
  }
  *n_blocks = blocks;
  return 0;
}


// ---- offline synthesis (pyworld.synthesize; vocoder.py:50-62) and the output silence gate (decode_worker.py:53-59) ----
int ryk_world_synthesize_length(int n_frames, double frame_period_ms, int fs) {
  return (int)((double)n_frames * frame_period_ms * fs / 1000.0);
}

int ryk_world_synthesize(ryk_engine* h, const double* f0, int n_frames, const float* sp, const float* ap, int fs, double frame_period_ms,
                         int fft_size, double* y, int y_capacity, int* y_length, long long* pulse_index, double* pulse_shift, int* pulse_vuv,
                         int max_pulses, int* n_pulses) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(f0 && sp && ap && y && n_frames >= 1, "null or empty synthesis input");
  const int ny = ryk_world_synthesize_length(n_frames, frame_period_ms, fs);
  RYK_CHECK(ny <= y_capacity, "output buffer too small: ryk_world_synthesize_length samples are written");
  const int np = world_synthesize_run(e, f0, n_frames, sp, ap, fs, frame_period_ms, fft_size, y, ny, pulse_index, pulse_shift, pulse_vuv, max_pulses);
  if (np < 0) return -1;
  if (y_length) *y_length = ny;
  if (n_pulses) *n_pulses = np;
  return 0;
}

int ryk_output_gate(ryk_engine* h, const double* wave, int n, int n_fft, int hop, double threshold_db, double* power_db, int* pass) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(wave != nullptr && n > 0, "empty chunk");
  const size_t scratch = output_gate_scratch_doubles(n, n_fft, hop);
  void* buf = nullptr;
  if (engine_scratch(e, sizeof(double) * (n + scratch + 2) + 64, &buf)) return -1;
  double* d_wave = (double*)buf;
  double* d_scr = d_wave + n;
  double* d_power = d_scr + scratch;
  int* d_status = (int*)(d_power + 1);
  RYK_CUDA(cudaMemcpyAsync(d_wave, wave, sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
  if (output_gate_async(e, d_wave, nullptr, n, n_fft, hop, threshold_db, d_scr, d_power, d_status, e->stream)) return -1;
  double pw = 0.0; int st = 0;
  RYK_CUDA(cudaMemcpyAsync(&pw, d_power, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaMemcpyAsync(&st, d_status, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  if (power_db) *power_db = pw;
  if (pass) *pass = st == 1 ? 1 : 0;
  return 0;
}


int ryk_resample_length(int n, int up, int down) {
  if (n <= 0 || up <= 0 || down <= 0) return 0;
  const long long m = (long long)n * up;
  return (int)(m / down + (m % down != 0));
}

int ryk_resample_poly(ryk_engine* h, const float* x, int n, int up, int down, const double* taps, int n_taps, float* y, int y_capacity, int* n_out) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(x && taps && y && n > 0 && up > 0 && down > 0 && n_taps > 0 && (n_taps & 1), "bad resampler arguments (the filter must have an odd number of taps)");
  const int no = ryk_resample_length(n, up, down);
  RYK_CHECK(no <= y_capacity, "output buffer too small: ryk_resample_length samples are written");
  void* buf = nullptr;
  const size_t bx = ((sizeof(float) * (size_t)n + 255) / 256) * 256, bh = ((sizeof(double) * (size_t)n_taps + 255) / 256) * 256;
  if (engine_scratch(e, bx + bh + sizeof(float) * (size_t)no + 256, &buf)) return -1;
  float* d_x = (float*)buf; double* d_h = (double*)((char*)buf + bx); float* d_y = (float*)((char*)buf + bx + bh);
  RYK_CUDA(cudaMemcpyAsync(d_x, x, sizeof(float) * n, cudaMemcpyHostToDevice, e->stream));
  RYK_CUDA(cudaMemcpyAsync(d_h, taps, sizeof(double) * n_taps, cudaMemcpyHostToDevice, e->stream));
  if (resample_poly_run(e, d_x, n, up, down, d_h, n_taps, d_y, no, e->stream)) return -1;
  RYK_CUDA(cudaMemcpyAsync(y, d_y, sizeof(float) * no, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  if (n_out) *n_out = no;
  return 0;
}

// ---- diagnostics: the synthesizer's pulse ring (index, time, vuv) and scalar state
int ryk_debug_synth_pulses(ryk_engine* h, int id, long long first, int count, long long* index, double* time, int* vuv, long long* state7) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  Synth* s = get_synth(e, id);
  RYK_CHECK(s != nullptr, "no such synthesizer");
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  SynthState st;
  RYK_CUDA(cudaMemcpy(&st, s->dev.state, sizeof(st), cudaMemcpyDeviceToHost));
  state7[0] = st.n_pulses; state7[1] = st.next_pulse; state7[2] = st.last_location; state7[3] = st.synthesized_sample;
  state7[4] = st.cumulative_frame; state7[5] = st.rng_generated; state7[6] = st.blocks_out;
  for (int i = 0; i < count; ++i) {
    int slot = (int)((first + i) % s->dev.cap_pulses);
    RYK_CUDA(cudaMemcpy(index + i, s->dev.p_index + slot, sizeof(long long), cudaMemcpyDeviceToHost));
    RYK_CUDA(cudaMemcpy(time + i, s->dev.p_time + slot, sizeof(double), cudaMemcpyDeviceToHost));
    RYK_CUDA(cudaMemcpy(vuv + i, s->dev.p_vuv + slot, sizeof(int), cudaMemcpyDeviceToHost));
  }
  return 0;
}

int ryk_debug_synth_timebase(ryk_engine* h, int id, int n, double* if0, double* ivuv, double* tp) {
  Engine* e = E(h);
  Synth* s = get_synth(e, id);
  RYK_CHECK(s != nullptr, "no such synthesizer");
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  RYK_CUDA(cudaMemcpy(if0, s->dev.if0, sizeof(double) * n, cudaMemcpyDeviceToHost));
  RYK_CUDA(cudaMemcpy(ivuv, s->dev.ivuv, sizeof(double) * n, cudaMemcpyDeviceToHost));
  RYK_CUDA(cudaMemcpy(tp, s->dev.tp, sizeof(double) * n, cudaMemcpyDeviceToHost));
  return 0;
}

// ---- CREPE f0 front-end (acoustic_feature_wrapper.py:65-80): model upload and crepe.predict + predict_voicing on 16 kHz audio
int ryk_crepe_create(ryk_engine* h, int capacity_multiplier) { RYK_CUDA(cudaSetDevice(E(h)->device)); return crepe_create(E(h), capacity_multiplier); }
int ryk_crepe_set_conv(ryk_engine* h, int layer, const float* W, const float* bias, const float* gamma, const float* beta, const float* mean,
                       const float* var) {
  RYK_CUDA(cudaSetDevice(E(h)->device));
  return crepe_set_conv(E(h), layer, W, bias, gamma, beta, mean, var);
}
int ryk_crepe_set_dense(ryk_engine* h, const float* W, const float* bias) { RYK_CUDA(cudaSetDevice(E(h)->device)); return crepe_set_dense(E(h), W, bias); }
int ryk_crepe_set_decoder_tables(ryk_engine* h, const double* log_trans, const double* cents_mapping, double log_start, double log_emit_self,
                                 double log_emit_other) {
  RYK_CUDA(cudaSetDevice(E(h)->device));
  return crepe_set_tables(E(h), log_trans, cents_mapping, log_start, log_emit_self, log_emit_other);
}
int ryk_crepe_num_frames(int n16, double step_ms) { return crepe_num_frames(n16, step_ms); }
int ryk_crepe_predict(ryk_engine* h, const float* audio16k, int n, double step_ms, double* f0, float* confidence, int* voicing, float* activation,
                      int* path) {
  RYK_CUDA(cudaSetDevice(E(h)->device));
  return crepe_predict(E(h), audio16k, n, step_ms, f0, confidence, voicing, activation, path);
}

// f0 extractor behind ryk_world_f0 / ryk_world_analyze / new sessions: 0 = DIO + StoneMask (default), 1 = Harvest + StoneMask.
int ryk_engine_set_f0_method(ryk_engine* h, int method) {
  RYK_CHECK(method == 0 || method == 1, "f0 method must be 0 (DIO) or 1 (Harvest)");
  E(h)->f0_method = method;
  return 0;
}
int ryk_engine_get_f0_method(ryk_engine* h) { return E(h)->f0_method; }

// ---- diagnostics: Harvest internals of the last analysis that used this plan (engine in f0 method 1)
int ryk_debug_harvest(ryk_engine* h, int n, int fs, double fp, double f0_floor, double f0_ceil, int* info, double* y, double* raw,
                      double* cand, double* score, double* best, double* basic, double* f0_raw) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(e->f0_method == 1, "engine is not in Harvest mode");
  DioPlan* plan = nullptr;
  if (dio_get_plan(e, n, fs, fp, f0_floor, f0_ceil, &plan)) return -1;
  if (f0_raw) RYK_CUDA(cudaMemcpyAsync(f0_raw, dio_plan_f0_raw(plan), sizeof(double) * dio_plan_frames(plan), cudaMemcpyDeviceToHost, e->stream));
  return harvest_plan_debug_copy(dio_plan_harvest(plan), info, y, raw, cand, score, best, basic, e->stream);
}

// ---- diagnostics: stage-1 forward of padded length Tp as one cluster kernel vs 16 layer launches (ms per forward, stand-alone),
// and the fused kernel's phase timeline (31 values in us: start, after layer 0, {tasks done, barrier passed} x 14, end)
int ryk_debug_stage1_bench(ryk_engine* h, int Tp, int iters, float* ms_fused, float* ms_layered, double* timeline_us) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(e->precision == 1 && Tp > 0 && Tp % 128 == 0 && iters > 0, "needs FP16 mode and a padded length (multiple of 128)");
  UNetPlan* plan = nullptr;
  if (stage1_plan_for(e, Tp, &plan)) return -1;
  return s1_fused_bench(e, plan, iters, ms_fused, ms_layered, timeline_us);
}

// ---- diagnostics: DIO internals of the last ryk_world_f0 / ryk_world_analyze call with this (n, fs, ...) plan
int ryk_debug_dio(ryk_engine* h, int n, int fs, double fp, double f0_floor, double f0_ceil, double* f0_raw, double* cand, double* score, int* counts) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  DioPlan* plan = nullptr;
  if (dio_get_plan(e, n, fs, fp, f0_floor, f0_ceil, &plan)) return -1;
  return dio_plan_debug_copy(plan, f0_raw, cand, score, counts, e->stream);
}

int ryk_debug_stonemask(ryk_engine* h, const float* wave, int n, int fs, double fp, double f0_floor, const double* f0_in, int frames,
                        double* f0_out) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  RYK_CHECK(n > 0 && frames > 0, "empty input");
  void* scratch = nullptr;
  size_t need = arena_need({sizeof(float) * n, sizeof(double) * frames, sizeof(double) * frames});
  if (engine_scratch(e, need, &scratch)) return -1;
  Arena A(scratch);
  float* d_x = A.take<float>(n);
  double* d_in = A.take<double>(frames);
  double* d_out = A.take<double>(frames);
  RYK_CUDA(cudaMemcpyAsync(d_x, wave, sizeof(float) * n, cudaMemcpyHostToDevice, e->stream));
  RYK_CUDA(cudaMemcpyAsync(d_in, f0_in, sizeof(double) * frames, cudaMemcpyHostToDevice, e->stream));
  if (stonemask_run(e, d_x, n, fs, fp, f0_floor, d_in, d_out, frames, e->stream)) return -1;
  e->launches += 1;
  RYK_CUDA(cudaMemcpyAsync(f0_out, d_out, sizeof(double) * frames, cudaMemcpyDeviceToHost, e->stream));
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

// ---- diagnostics: one conv / transposed-conv layer in isolation (unit parity + profiling) -------
// in0/in1: host fp32 NHWC [B][Hin][Win][C0|C1]; W: Chainer layout; out: host fp32 NHWC [B][Hout][Wout][Cout].
// use_tc = 1 runs the FP16 tcgen05 kernel (activations rounded to fp16), 0 the FP32 CUDA-core kernel.
int ryk_test_conv_layer(ryk_engine* h, int transposed, int k, int stride, int pad, int B, int Hin, int Win, int C0, int C1, int Cout,
                        const float* in0, const float* in1, const float* W, const float* scale, const float* shift, int act,
                        int use_tc, int repeat, float* out, float* ms_per_run) {
  Engine* e = E(h);
  RYK_CUDA(cudaSetDevice(e->device));
  cudaStream_t st = e->stream;
  ConvLayer L;
  L.transposed = transposed; L.B = B; L.Hin = Hin; L.Win = Win; L.C0 = C0; L.C1 = C1; L.Cout = Cout;
  L.KH = L.KW = k; L.SH = L.SW = stride; L.PH = L.PW = pad; L.act = act;
  if (Hin == 1) { L.KH = 1; L.SH = 1; L.PH = 0; }      // 1-D layer (stage-1 nets): kernel (1 x k), stride (1, s), padding (0, p)
  if (transposed) { L.Hout = (Hin - 1) * L.SH + L.KH - 2 * L.PH; L.Wout = (Win - 1) * stride + k - 2 * pad; }
  else { L.Hout = (Hin + 2 * L.PH - L.KH) / L.SH + 1; L.Wout = (Win + 2 * pad - k) / stride + 1; }
  const int Cin = C0 + C1;
  size_t n0 = (size_t)B * Hin * Win * C0, n1 = (size_t)B * Hin * Win * C1, no = (size_t)B * L.Hout * L.Wout * Cout;
  size_t nw = (size_t)Cin * Cout * L.KH * k;
  std::vector<void*> frees;
  auto A = [&](size_t bytes) -> void* { void* p = nullptr; if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) return nullptr; frees.push_back(p); return p; };
  float* d_in0 = (float*)A(n0 * 4); float* d_in1 = (float*)A(n1 * 4); float* d_w = (float*)A(nw * 4);
  float* d_wd = (float*)A(nw * 4); __half* d_wt = (__half*)A(nw * 2);
  float* d_scale = (float*)A(Cout * 4); float* d_shift = (float*)A(Cout * 4);
  __half* d_h0 = (__half*)A(n0 * 2); __half* d_h1 = (__half*)A(n1 * 2); __half* d_ho = (__half*)A(no * 2); float* d_out = (float*)A(no * 4);
  RYK_CHECK(d_out != nullptr, "cudaMalloc failed in ryk_test_conv_layer");
  RYK_CUDA(cudaMemcpyAsync(d_in0, in0, n0 * 4, cudaMemcpyHostToDevice, st));
  if (n1) RYK_CUDA(cudaMemcpyAsync(d_in1, in1, n1 * 4, cudaMemcpyHostToDevice, st));
  RYK_CUDA(cudaMemcpyAsync(d_w, W, nw * 4, cudaMemcpyHostToDevice, st));
  RYK_CUDA(cudaMemcpyAsync(d_scale, scale, Cout * 4, cudaMemcpyHostToDevice, st));
  RYK_CUDA(cudaMemcpyAsync(d_shift, shift, Cout * 4, cudaMemcpyHostToDevice, st));
  if (pack_weights_direct(d_w, transposed, Cin, Cout, L.KH, k, d_wd, st)) return -1;
  L.w_direct = d_wd; L.scale = d_scale; L.shift = d_shift;
  int rc = 0;
  cudaEvent_t ev0, ev1;
  RYK_CUDA(cudaEventCreate(&ev0)); RYK_CUDA(cudaEventCreate(&ev1));
  // time `repeat` runs replayed from a CUDA graph (as the session runs them): no host launch overhead in the figure
  auto timed_graph = [&](auto&& run) -> int {
    cudaGraph_t graph = nullptr; cudaGraphExec_t exec = nullptr;
    int r = 0;
    RYK_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    for (int i = 0; i < repeat && !r; ++i) r = run();
    cudaError_t err = cudaStreamEndCapture(st, &graph);
    if (r) return r;
    RYK_CUDA(err);
    RYK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
    RYK_CUDA(cudaGraphLaunch(exec, st));
    RYK_CUDA(cudaEventRecord(ev0, st));
    RYK_CUDA(cudaGraphLaunch(exec, st));
    RYK_CUDA(cudaEventRecord(ev1, st));
    RYK_CUDA(cudaStreamSynchronize(st));
    cudaGraphExecDestroy(exec); cudaGraphDestroy(graph);
    return 0;
  };
  if (use_tc == 1) {
    if (pack_weights_tc(d_w, transposed, Cin, Cout, L.KH, k, L.SH, stride, d_wt, st)) return -1;
    k_f32_to_f16<<<1184, 256, 0, st>>>(d_in0, d_h0, n0);
    if (n1) k_f32_to_f16<<<1184, 256, 0, st>>>(d_in1, d_h1, n1);
    L.in0 = d_h0; L.in1 = n1 ? d_h1 : nullptr; L.in_dtype = DT_F16; L.out = d_ho; L.out_dtype = DT_F16; L.w_tc = d_wt;
    RYK_CHECK(tc_layer_eligible(L), "layer shape is not eligible for the tensor-core kernel");
    int num_sms = 148;
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, e->device);
    size_t ws = tc_splitk_ws_bytes(L, num_sms);
    if (ws) L.splitk_ws = (float*)A(ws);
    if (tc_layer_wants_counter(L, num_sms)) { L.t3_ctr = (int*)A(16); RYK_CUDA(cudaMemsetAsync(L.t3_ctr, 0, 16, st)); }
    if (tc_layer_prepare(L, num_sms)) return -1;
    rc = conv_tc_run(L, st);
    if (!rc && repeat > 0) rc = timed_graph([&]() { return conv_tc_run(L, st); });
    k_f16_to_f32<<<1184, 256, 0, st>>>(d_ho, d_out, no);
  } else if (use_tc == 2) {
    // mixed-precision edge layers as the fp16 U-Net plans run them: the first layer (Cin = 1) reads fp32 / writes fp16, the last
    // layers (stage 2: Cout = 1, stage 1: 1-D k3 to `order + 1` channels) read fp16 / write fp32
    const bool in_h = Cin > 1, out_h = Cin == 1;
    if (in_h) { k_f32_to_f16<<<1184, 256, 0, st>>>(d_in0, d_h0, n0); if (n1) k_f32_to_f16<<<1184, 256, 0, st>>>(d_in1, d_h1, n1); }
    L.in0 = in_h ? (const void*)d_h0 : (const void*)d_in0; L.in1 = n1 ? (in_h ? (const void*)d_h1 : (const void*)d_in1) : nullptr;
    L.in_dtype = in_h ? DT_F16 : DT_F32; L.out = out_h ? (void*)d_ho : (void*)d_out; L.out_dtype = out_h ? DT_F16 : DT_F32;
    if (Cout == 1) { L.host_scale_valid = true; L.host_scale = scale[0]; L.host_shift = shift[0]; }
    rc = conv_direct_run(L, st);
    if (!rc && repeat > 0) rc = timed_graph([&]() { return conv_direct_run(L, st); });
    if (out_h) k_f16_to_f32<<<1184, 256, 0, st>>>(d_ho, d_out, no);
  } else {
    L.in0 = d_in0; L.in1 = n1 ? d_in1 : nullptr; L.in_dtype = DT_F32; L.out = d_out; L.out_dtype = DT_F32;
    rc = conv_direct_run(L, st);
    if (!rc && repeat > 0) rc = timed_graph([&]() { return conv_direct_run(L, st); });
  }
  if (!rc) {
    cudaError_t err = cudaMemcpyAsync(out, d_out, no * 4, cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    if (err != cudaSuccess) { set_error(std::string("conv layer test failed: ") + cudaGetErrorString(err)); rc = -1; }
  }
  float ms = 0.f;
  if (!rc && repeat > 0) { cudaEventElapsedTime(&ms, ev0, ev1); ms /= repeat; }
  if (ms_per_run) *ms_per_run = ms;
  cudaEventDestroy(ev0); cudaEventDestroy(ev1);
  for (void* p : frees) cudaFree(p);
  return rc;
}

}  // extern "C"
