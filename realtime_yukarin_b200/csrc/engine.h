// engine.h -- internal state of one libryk engine (one per process / GPU).
#pragma once
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "unet.h"
#include "synth.h"

namespace ryk {

struct DioPlan;
struct HarvestPlan;
struct Session;
struct Group;
struct Reblock;

struct Engine {
  int device = 0;
  cudaStream_t stream = nullptr;
  int precision = 1;                 // 0: FP32 CUDA-core convs everywhere, 1: FP16 tcgen05 tensor-core convs where eligible
  int f0_method = 0;                 // 0: DIO + StoneMask, 1: Harvest + StoneMask (world_harvest.cu)
  bool s1_fused = true;              // FP16 mode: stage 1 as ONE cluster kernel (s1_fused.cu) instead of 16 layer launches
  // FFT twiddles
  double2* d_twiddle = nullptr;
  // xorshift128 jump-ahead matrices (synthesis noise stream)
  uint32_t* d_jump = nullptr;
  // SPTK matrices
  double* d_G = nullptr; int G_order = -1, G_fft = 0; double G_alpha = 0;     // sp2mc: (order+1) x nb
  double* d_H = nullptr; int H_order = -1, H_fft = 0; double H_alpha = 0;     // mc2sp: nb x (order+1)
  // DIO plans keyed by (n, fs, frame_period*1000, floor*1000, ceil*1000)
  std::map<std::tuple<int, int, int, int, int>, DioPlan*> dio_plans;
  // networks
  UNet* stage1 = nullptr;
  UNet* stage2 = nullptr;
  // stage-1 statistics
  std::vector<float> s1_in_mean, s1_in_std, s1_out_mean, s1_out_std;
  float *d_s1_in_mean = nullptr, *d_s1_in_std = nullptr, *d_s1_out_mean = nullptr, *d_s1_out_std = nullptr;
  double f0_in_mean = 0, f0_in_std = 1, f0_tgt_mean = 0, f0_tgt_std = 1;
  bool has_f0_stats = false;
  // synthesizers
  std::vector<Synth*> synths;
  std::vector<Session*> sessions;
  std::vector<Group*> groups;
  std::vector<Reblock*> reblocks;     // output re-blockers + silence gates (decode_worker.py:38-59)
  float* d_colmin = nullptr;         // stage-2 prologue column-minimum partials
  // scratch arena for the per-op host-pointer API (grown on demand)
  void* d_scratch = nullptr; size_t scratch_bytes = 0;
  void* h_pinned = nullptr; size_t pinned_bytes = 0;
  // counters
  long long launches = 0;
  // optional device-side timing of the stage-2 tensor-core layers (bench roofline): event pairs per forward
  bool profile = false;
  cudaEvent_t timer_ev[2] = {nullptr, nullptr};
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
};

int engine_scratch(Engine* e, size_t bytes, void** out);
int engine_pinned(Engine* e, size_t bytes, void** out);

// world_analysis.cu
int analysis_kernels_init();
int dio_plan_create(Engine* e, int n, int fs, double frame_period, double f0_floor, double f0_ceil, DioPlan** out, int f0_method = 0);
void dio_plan_free(DioPlan* p);
int dio_get_plan(Engine* e, int n, int fs, double frame_period, double f0_floor, double f0_ceil, DioPlan** out);
int dio_stonemask_run(Engine* e, DioPlan* p, const float* d_x, cudaStream_t st);
int stonemask_run(Engine* e, const float* d_x, int n, int fs, double frame_period, double f0_floor, const double* d_f0_in,
                  double* d_f0_out, int frames, cudaStream_t st);
const double* dio_plan_f0(DioPlan* p);      // refined f0 (double) after dio_stonemask_run
double* dio_plan_f0_mut(DioPlan* p);
int dio_plan_frames(DioPlan* p);
HarvestPlan* dio_plan_harvest(DioPlan* p);
const double* dio_plan_f0_raw(DioPlan* p);     // f0 contour before StoneMask
// world_harvest.cu
int harvest_plan_create(Engine* e, int n, int fs, double frame_period, double f0_floor, double f0_ceil, HarvestPlan** out);
void harvest_plan_free(HarvestPlan* p);
int harvest_run(Engine* e, HarvestPlan* p, const float* d_x, double* d_f0, cudaStream_t st);
int harvest_plan_debug_copy(HarvestPlan* p, int* info, double* y, double* raw, double* cand, double* score, double* best, double* basic,
                            cudaStream_t st);
// crepe.cu: CREPE f0 front-end (acoustic_feature_wrapper.py:65-80)
int crepe_create(Engine* e, int capacity_multiplier);
void crepe_destroy();
int crepe_set_conv(Engine* e, int layer, const float* W, const float* bias, const float* gamma, const float* beta, const float* mean, const float* var);
int crepe_set_dense(Engine* e, const float* W, const float* bias);
int crepe_set_tables(Engine* e, const double* log_trans, const double* cents_mapping, double log_start, double log_emit_self, double log_emit_other);
int crepe_num_frames(int n16, double step_ms);
int crepe_predict(Engine* e, const float* audio16k, int n, double step_ms, double* f0, float* confidence, int* voicing, float* activation, int* path_out);
// s1_fused.cu diagnostics
int s1_fused_bench(Engine* e, UNetPlan* p, int iters, float* ms_fused, float* ms_layered, double* timeline_us);
int dio_plan_debug_copy(DioPlan* p, double* f0_raw, double* cand, double* score, int* counts, cudaStream_t st);
int spectral_analysis_run(Engine* e, const float* d_x, int n, int fs, double frame_period, const double* d_f0, int n_out,
                          int fft_size, int order, float* d_sp, float* d_ap, float* d_mc, float* d_f0_out, uint8_t* d_voiced,
                          cudaStream_t st);

// world_synth.cu: offline Synthesis() (pyworld.synthesize) and the output silence gate
int world_synthesize_run(Engine* e, const double* f0, int n_frames, const float* sp, const float* ap, int fs, double frame_period_ms,
                         int fft_size, double* y, int y_length, long long* pulse_index, double* pulse_shift, int* pulse_vuv, int max_pulses);
int output_gate_async(Engine* e, const double* d_wave, const int* d_n_valid, int n, int n_fft, int hop, double threshold_db,
                      double* d_scratch, double* d_power, int* d_status, cudaStream_t st);
size_t output_gate_scratch_doubles(int n, int n_fft, int hop);

// sptk.cu
int sptk_prepare(Engine* e, int order, double alpha, int fft_size);                 // builds G and H on the device
int mc2sp_run(Engine* e, const float* d_mc, int T, int order, int fft_size, double add, float* d_sp_f32, double* d_sp_f64, cudaStream_t st);

// features.cu: polyphase resampler (wav I/O row)
int resample_poly_run(Engine* e, const float* d_x, int n, int up, int down, const double* d_h, int n_taps, float* d_y, int n_out, cudaStream_t st);

// gate.cu
int gate_mask_run(Engine* e, const float* d_wave, int n, int frame_length, int hop, double threshold_db, int n_frames,
                  double* d_mse_scratch, uint8_t* d_mask, int* d_index /*compacted frame ids*/, int* d_count, cudaStream_t st);

}  // namespace ryk
