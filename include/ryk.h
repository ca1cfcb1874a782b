/*
 * ryk.h -- C ABI of libryk.so: the B200-native per-chunk hot path of realtime-yukarin
 *          (encode -> stage 1 -> stage 2 -> vocode).  Plain pointers and sizes only.
 *
 * Every entry point replaces one call the reference makes into an un-vendored third-party library
 * (file:line are paths under the reference checkout, realtime_voice_conversion/ abbreviated rvc/):
 *
 *   ryk_world_analyze          <- yukarin.AcousticFeature.extract (pyworld dio/stonemask/cheaptrick/d4c + pysptk.sp2mc)
 *                                 rvc/yukarin_wrapper/vocoder.py:26-48, rvc/yukarin_wrapper/acoustic_feature_wrapper.py:28-33
 *   ryk_world_f0               <- yukarin.AcousticFeature.extract_f0 (override hook at acoustic_feature_wrapper.py:66-80)
 *   ryk_silence_mask           <- AcousticConverter.separate_effective (librosa _signal_to_frame_nonsilent)  rvc/yukarin_wrapper/voice_changer.py:27-31
 *   ryk_stage1_load/_convert   <- yukarin.AcousticConverter(...)/.convert (Chainer forward)                   voice_changer.py:33, converter/yukarin_converter.py:40-46
 *   ryk_mc2sp                  <- AcousticConverter.decode_spectrogram (pysptk.mc2sp)                           voice_changer.py:38
 *   ryk_stage2_load/_convert   <- become_yukarin.SuperResolution(...)/.convert (Chainer forward)               voice_changer.py:41, converter/yukarin_converter.py:50-55
 *   ryk_convert_window         <- VoiceChanger.convert_from_acoustic_feature, fused on device                   voice_changer.py:24-42
 *   ryk_synth_create           <- world4py apidefinitions._InitializeSynthesizer                                rvc/yukarin_wrapper/vocoder.py:79-87
 *   ryk_synth_add_parameters   <- world4py apidefinitions._AddParameters                                        vocoder.py:99
 *   ryk_synth_synthesis2       <- world4py apidefinitions._Synthesis2 (+ the per-sample buffer read-out)        vocoder.py:102-104
 *   ryk_synth_decode           <- RealtimeVocoder.decode as one call (add + drain)                              vocoder.py:89-120
 *   ryk_session_*              <- the encode/convert/decode StreamWrapper chain of one audio stream kept on
 *                                 device                                                                       rvc/worker/, rvc/stream/ (all modules)
 *   ryk_world_synthesize       <- pyworld.synthesize (Vocoder.decode, offline)                                  rvc/yukarin_wrapper/vocoder.py:50-62
 *   ryk_output_gate, ryk_reblock_* <- decode worker: wave_fragment re-blocking + librosa stft/power_to_db gate   rvc/worker/decode_worker.py:38-59
 *   ryk_resample_poly          <- librosa.load(path, sr=input_rate) resampling                                  check.py:80
 *
 * Conventions: all functions return 0 on success and a negative value on error unless stated otherwise
 * (ryk_last_error() describes the failure); "host" pointers are ordinary process memory, "dev"
 * pointers are CUDA device memory of the engine's GPU.  One engine per process per GPU; an engine is
 * NOT thread-safe (the reference drives each stage from a single thread as well).
 */
#ifndef RYK_H_
#define RYK_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ryk_engine ryk_engine;

int ryk_abi_version(void);
const char* ryk_last_error(void);

/* ---- engine ---------------------------------------------------------------------------- */
int ryk_engine_create(int device, ryk_engine** out);
int ryk_engine_destroy(ryk_engine* e);
/* 0: FP32 CUDA-core convolutions everywhere (bisecting / numerics reference)
 * 1: FP16 operands + FP32 accumulate on tcgen05 tensor cores for the stage-2 k4 layers (default) */
int ryk_engine_set_precision(ryk_engine* e, int mode);
int ryk_engine_get_precision(ryk_engine* e);
/* FP16 mode: run the stage-1 1-D U-Net (AcousticConverter.convert_from_feature, voice_changer.py:36) as ONE thread-block-cluster
 * kernel (default, s1_fused.cu) or as 16 layer launches (enable = 0).  Returns the cluster size in use, <= 0 when the kernel is
 * unavailable.  Sessions capture their stage-1 graphs at creation, so switch before ryk_session_create. */
int ryk_engine_set_stage1_fused(ryk_engine* e, int enable);
long long ryk_engine_launch_count(ryk_engine* e);        /* kernels launched by this engine so far */
int ryk_engine_synchronize(ryk_engine* e);
/* CUDA-event timing of the stage-2 k4-layer block (layers 1..14, the tcgen05 kernels) on the engine's stream */
int ryk_engine_timer_start(ryk_engine* e);                    /* cudaEventRecord on the engine's stream */
int ryk_engine_timer_stop(ryk_engine* e, float* elapsed_ms);  /* record + synchronize + elapsed */
int ryk_engine_profile(ryk_engine* e, int enable);
int ryk_engine_profile_read(ryk_engine* e, double* stage2_ms_total, int* stage2_runs);
/* as above plus the UNION of the per-forward intervals (a session alternates its stage-2 forwards between two streams, so they overlap) */
int ryk_engine_profile_read2(ryk_engine* e, double* stage2_ms_total, double* stage2_ms_union, int* stage2_runs);

/* ---- WORLD analysis (encode) -------------------------------------------------------------- */
/* wave_host: n float32 samples.  Outputs are n_frames = n / hop rows (hop = fs * frame_period / 1000):
 * f0 [n_frames], sp/ap [n_frames][fft_length/2+1], mc [n_frames][order+1], voiced [n_frames] (0/1).
 * f0_override (nullable, double[n_frames_world = n/hop + 1]) replaces DIO+StoneMask. Any output may be NULL. */
int ryk_world_analyze(ryk_engine* e, const float* wave_host, int n, int fs, double frame_period_ms,
                      double f0_floor, double f0_ceil, int fft_length, int order, double alpha,
                      const double* f0_override, float* f0, float* sp, float* ap, float* mc, uint8_t* voiced);
/* DIO + StoneMask only; f0/t are double[n / hop + 1] (WORLD's own frame count). */
int ryk_world_f0(ryk_engine* e, const float* wave_host, int n, int fs, double frame_period_ms,
                 double f0_floor, double f0_ceil, double* f0, double* t);
int ryk_world_num_frames(int n, int fs, double frame_period_ms);
/* f0 extractor behind ryk_world_f0 / ryk_world_analyze and sessions created afterwards -- the f0 hook of yukarin's
 * AcousticFeature.extract (acoustic_feature_wrapper.py:28-33; f0_estimating_method, SURVEY A.2 / A.7):
 *   0 = pyworld.dio + pyworld.stonemask (default), 1 = pyworld.harvest + pyworld.stonemask. */
int ryk_engine_set_f0_method(ryk_engine* e, int method);
int ryk_engine_get_f0_method(ryk_engine* e);

/* ---- CREPE f0 front-end (CrepeAcousticFeatureWrapper.extract_f0, acoustic_feature_wrapper.py:65-80) --------------------------
 * crepe.predict(x, fs, viterbi=True, model_capacity=..., step_size=frame_period) + crepe.predict_voicing on the device.  The caller
 * resamples to 16 kHz (ryk_resample_poly) and applies the reference's rule voiced = (voicing == 1) | (confidence > 0.1).
 * capacity_multiplier: 4 tiny, 8 small, 16 medium, 24 large, 32 full.  Conv weights W (cout, cin, k) for blocks 0..5 with widths
 * 512, 64 x 5 and filters m * {32, 4, 4, 4, 8, 16}; BatchNorm statistics per block (eps 1e-3); dense W (360, 64 m).
 * log_trans: the 360 x 360 log transition matrix of the pitch HMM, its start / emission log-probabilities and the bin -> cents table, computed by the host
 * mirror exactly as crepe.to_viterbi_cents does (shared tables make the Viterbi sums bit-identical to the CPU restatement). */
int ryk_crepe_create(ryk_engine* e, int capacity_multiplier);
int ryk_crepe_set_conv(ryk_engine* e, int block, const float* W, const float* bias, const float* bn_gamma, const float* bn_beta,
                       const float* bn_mean, const float* bn_var);
int ryk_crepe_set_dense(ryk_engine* e, const float* W, const float* bias);
int ryk_crepe_set_decoder_tables(ryk_engine* e, const double* log_trans, const double* cents_mapping /* [360] */, double log_start,
                                 double log_emit_self, double log_emit_other);
int ryk_crepe_num_frames(int n16, double step_ms);
/* f0 / confidence / voicing (HMM state) [frames], activation [frames][360], path [frames] (pitch-bin Viterbi path); any may be NULL */
int ryk_crepe_predict(ryk_engine* e, const float* audio16k, int n, double step_ms, double* f0, float* confidence, int* voicing,
                      float* activation, int* path);

/* ---- silence gate --------------------------------------------------------------------------- */
/* mask[n_frames] (0/1); threshold_db < 0 disables the gate (all frames effective). */
int ryk_silence_mask(ryk_engine* e, const float* wave_host, int n, int frame_length, int hop,
                     double threshold_db, int n_frames, uint8_t* mask);

/* ---- networks ------------------------------------------------------------------------------- */
/* stage: 1 (1-D, yukarin) or 2 (2-D, become-yukarin).  Layers 0..7 = encoder c0..c7, 8..15 = decoder c0..c7.
 * W is the model file's (Chainer) layout: conv (Cout, Cin, k[, k]), transposed conv (Cin, Cout, k[, k]);
 * scale/shift [Cout] are the bias and eval-mode BatchNorm folded together (y = conv(x) * scale + shift). */
int ryk_model_create(ryk_engine* e, int stage, int in_channels, int out_channels, int base_channels);
int ryk_model_set_layer(ryk_engine* e, int stage, int layer, const float* W, const float* scale, const float* shift);
int ryk_model_layer_shape(ryk_engine* e, int stage, int layer, int* transposed, int* cin, int* cout, int* k);
/* per-channel normalisation of the stage-1 input/output features and the log-f0 statistics */
int ryk_stage1_set_stats(ryk_engine* e, int channels, const float* in_mean, const float* in_std,
                         const float* out_mean, const float* out_std);
int ryk_f0_set_stats(ryk_engine* e, double in_mean, double in_std, double target_mean, double target_std);
/* x, y: [T][channels] float32 (T >= 1; internally padded to the next multiple of 128 with the per-channel minimum) */
int ryk_stage1_convert(ryk_engine* e, const float* x, int T, float* y);
/* f0_out[i] = voiced[i] ? exp((ln f0[i] - mu_in) / sd_in * sd_tgt + mu_tgt) : 0 */
int ryk_f0_convert(ryk_engine* e, const float* f0, const uint8_t* voiced, int T, float* f0_out);
/* mc [T][order+1] float32 -> sp [T][fftlen/2+1] float64 = exp(H mc) (pysptk.mc2sp) */
int ryk_mc2sp(ryk_engine* e, const float* mc, int T, int order, double alpha, int fftlen, double* sp);
/* sp, out: [T][513] float32 */
int ryk_stage2_convert(ryk_engine* e, const float* sp, int T, float* out);

/* The whole VoiceChanger.convert_from_acoustic_feature on device: one upload, one download.
 * in : wave [n_wave], f0 [T], ap [T][nb], mc [T][order+1], voiced [T]
 * out: f0 [T], ap [T][nb], sp [T][nb], voiced [T], mc [T][order+1] (nullable)      nb = fftlen/2+1 */
int ryk_convert_window(ryk_engine* e, const float* wave, int n_wave, int fs, int frame_length, int hop, double threshold_db,
                       const float* f0, const float* ap, const float* mc, const uint8_t* voiced, int T,
                       int order, double alpha, int fftlen,
                       float* f0_out, float* ap_out, float* sp_out, uint8_t* voiced_out, float* mc_out);

/* ---- WORLD realtime synthesizer (vocode) ------------------------------------------------------ */
int ryk_synth_create(ryk_engine* e, int fs, double frame_period_ms, int fft_size, int buffer_size,
                     int number_of_pointers, int* synth_id);
int ryk_synth_destroy(ryk_engine* e, int synth_id);
/* returns 1 when the frames were queued, 0 when the ring is full (world4py semantics), < 0 on error */
int ryk_synth_add_parameters(ryk_engine* e, int synth_id, const double* f0, int n, const float* sp, const float* ap);
/* returns 1 and writes buffer_size doubles when a block was produced, 0 when not enough pulses are queued */
int ryk_synth_synthesis2(ryk_engine* e, int synth_id, double* buffer);
/* add + drain in one call: out receives *n_blocks * buffer_size doubles (at most max_blocks blocks) */
int ryk_synth_decode(ryk_engine* e, int synth_id, const double* f0, int n, const float* sp, const float* ap,
                     double* out, int max_blocks, int* n_blocks);

/* ---- offline synthesis: Vocoder.decode = pyworld.synthesize (SURVEY 8(f) rank 3) ---------------------
 * Replaces realtime_voice_conversion/yukarin_wrapper/vocoder.py:50-62 (pyworld.synthesize -> WORLD Synthesis()):
 * whole-utterance time base, fractional pulse shift, Hanning dc-remover, overlap-add.  y receives
 * ryk_world_synthesize_length(n_frames, frame_period_ms, fs) = (int)(n_frames * frame_period_ms * fs / 1000) doubles.
 * pulse_index / pulse_shift / pulse_vuv (each may be NULL, max_pulses entries) expose the pulse plan for parity tests. */
int ryk_world_synthesize_length(int n_frames, double frame_period_ms, int fs);
int ryk_world_synthesize(ryk_engine* e, const double* f0, int n_frames, const float* sp, const float* ap, int fs,
                         double frame_period_ms, int fft_size, double* y, int y_capacity, int* y_length,
                         long long* pulse_index, double* pulse_shift, int* pulse_vuv, int max_pulses, int* n_pulses);

/* ---- output silence gate and re-blocking (SURVEY 8(f) rank 2) ------------------------------------------
 * Replaces realtime_voice_conversion/worker/decode_worker.py:38-59: the synthesizer's 1024-sample blocks are queued in a
 * fragment, one out_audio_chunk is cut off its front per step when enough samples are queued, and the chunk is dropped
 * when librosa.power_to_db(abs(librosa.stft(chunk)) ** 2).mean() < -output_silent_threshold
 * (n_fft 2048, hop 512, periodic Hann, reflect-centred, amin 1e-10, top_db 80).
 * ryk_output_gate: the gate alone on a host chunk; *pass = 1 keeps the chunk.
 * ryk_reblock_*: device-resident fragment + gate.  push_device is stream-ordered and never syncs the host: with
 * session_id >= 0 it is queued on that session's decode stream right behind its latest step (wave_dev == NULL consumes the
 * step's blocks and count in place); results go to ring slot ticket % 8.  collect: *status 0 = no chunk this step,
 * 1 = chunk copied to chunk_out, 2 = chunk was silent (the reference forwards None). */
int ryk_output_gate(ryk_engine* e, const double* wave, int n, int n_fft, int hop, double threshold_db, double* power_db, int* pass);
int ryk_reblock_create(ryk_engine* e, int out_audio_chunk, int max_in, int n_fft, int hop, double threshold_db, int* reblock_id);
int ryk_reblock_destroy(ryk_engine* e, int reblock_id);
int ryk_reblock_push(ryk_engine* e, int reblock_id, const double* wave, int n, double* chunk_out, int* status, double* power_db);
int ryk_reblock_push_device(ryk_engine* e, int reblock_id, int session_id, const double* wave_dev, const int* n_dev, long long* ticket);
int ryk_reblock_collect(ryk_engine* e, int reblock_id, long long ticket, double* chunk_out, int* status, double* power_db);
/* Non-blocking: *done = 1 when ryk_reblock_collect(ticket) would not wait (queue_output_wave.get_nowait, run.py:176-182).
 * collect fails (instead of dropping samples) when a step produced more than the fragment can hold: the reference's
 * wave_fragment is unbounded (decode_worker.py:47-52), the device fragment holds 2 * (out_audio_chunk + max_in) samples. */
int ryk_reblock_poll(ryk_engine* e, int reblock_id, long long ticket, int* done);
int ryk_reblock_result_device(ryk_engine* e, int reblock_id, long long ticket, const double** chunk_dev, const int** status_dev,
                              const double** power_dev);

/* ---- sample-rate conversion for wav input (SURVEY 8(f) rank 3; check.py:80 librosa.load(path, sr=input_rate)) --------
 * Polyphase FIR resampling, the upfirdn step of scipy.signal.resample_poly: up / down must be coprime, `taps` is the
 * odd-length low-pass filter already scaled by `up` (realtime_yukarin_b200/wave_io.py: resample_filter), edges are
 * zero-padded; y receives ryk_resample_length(n, up, down) = ceil(n * up / down) samples. */
int ryk_resample_length(int n, int up, int down);
int ryk_resample_poly(ryk_engine* e, const float* x, int n, int up, int down, const double* taps, int n_taps, float* y,
                      int y_capacity, int* n_out);

/* ---- device-resident streaming session (one audio stream) -------------------------------------- */
typedef struct {
  int fs;                       /* 24000 */
  double frame_period_ms;       /* 5 */
  double f0_floor, f0_ceil;     /* 71, 800 */
  int fft_length, order;        /* 1024, 8 */
  double alpha;                 /* 0.466 */
  double buffer_time;           /* seconds of audio per pushed chunk (0.3) */
  double encode_extra_time, convert_extra_time, decode_extra_time;   /* 0, 0.5, 0 */
  double threshold_db;          /* silence gate, < 0 disables */
  int vocoder_buffer_size;      /* 1024 */
} ryk_session_config;

int ryk_session_create(ryk_engine* e, const ryk_session_config* cfg, int* session_id);
int ryk_session_destroy(ryk_engine* e, int session_id);
/* One chunk through encode -> convert -> decode with host buffers (H2D + kernels + D2H inside).
 * wave: round(fs * buffer_time) float32 samples; out: up to out_capacity float64 samples; *n_out is a
 * multiple of vocoder_buffer_size (the remainder stays in the synthesizer, as in the reference). */
int ryk_session_push(ryk_engine* e, int session_id, const float* wave, int n, double* out, int out_capacity, int* n_out);
/* Pipelined host API: submit queues a chunk and returns at once (ticket = chunk number), collect waits for that
 * chunk's output.  Up to 5 chunks may be in flight; encode / convert / decode of consecutive chunks then overlap on
 * three CUDA streams, exactly like the reference's three worker processes (run.py:58-93).  push == submit + collect. */
int ryk_session_submit(ryk_engine* e, int session_id, const float* wave, int n, long long* ticket);
int ryk_session_collect(ryk_engine* e, int session_id, long long ticket, double* out, int out_capacity, int* n_out);
/* Non-blocking: *done = 1 when ryk_session_collect(ticket) would not wait (ticket among the last 8 steps). */
int ryk_session_poll(ryk_engine* e, int session_id, long long ticket, int* done);
/* Same chunk step with the input already resident in HBM and the output left there (throughput measurement);
 * asynchronous: returns when the work is queued, results are valid after ryk_engine_synchronize. */
int ryk_session_push_device(ryk_engine* e, int session_id, const float* wave_dev, int n, double* out_dev, int out_capacity,
                            int* n_out_dev);

/* Diagnostics: device timeline (ms) of the last <= 8 steps x 5 stages {gate, analysis, stage 1, stage 2, synthesis}; needs
 * RYK_STAGE_TIMES=1 in the environment at session creation.  start/end hold 40 floats; returns the number of steps. */
int ryk_session_stage_times(ryk_engine* e, int session_id, float* start, float* end);

/* ---- session groups: several streams of one GPU sharing one batched stage-2 forward -------------------
 * BASELINE config 5 / SURVEY 8(e) "per-GPU batch = streams resident on it": the reference would run one
 * SuperResolution.convert (voice_changer.py:41) per stream; a group stacks the members' padded log-spectrograms into
 * one (B, 1, Tp, 512) stage-2 input per step.  Analysis, gate, stage 1 and synthesis stay per stream (per-stream state,
 * data-dependent lengths).  Members are fresh sessions with the same window length; member i of every call is
 * session_ids[i].  Outputs per member are those of an ungrouped session up to the FP16 stage-2 rounding. */
int ryk_group_create(ryk_engine* e, const int* session_ids, int n_sessions, int* group_id);
int ryk_group_destroy(ryk_engine* e, int group_id);        /* members survive, ungrouped */
int ryk_group_size(ryk_engine* e, int group_id);
int ryk_group_submit(ryk_engine* e, int group_id, const float* const* waves, int n, long long* ticket);
int ryk_group_collect(ryk_engine* e, int group_id, long long ticket, double* const* outs, int out_capacity, int* n_outs);
int ryk_group_push_device(ryk_engine* e, int group_id, const float* const* waves_dev, int n, double* const* outs_dev,
                          int out_capacity, int* const* n_outs_dev);

/* ---- diagnostics -------------------------------------------------------------------------------------- */
/* Synthesizer pulse ring entries [first, first+count) and state {n_pulses, next_pulse, last_location, synthesized_sample,
 * cumulative_frame, rng_generated, blocks_out}. */
int ryk_debug_synth_pulses(ryk_engine* e, int synth_id, long long first, int count, long long* index, double* time, int* vuv, long long* state7);
/* Per-sample time base of the last AddParameters call (interpolated f0, vuv, total phase), first n samples. */
int ryk_debug_synth_timebase(ryk_engine* e, int synth_id, int n, double* if0, double* ivuv, double* tp);
/* DIO internals (raw contour before StoneMask, per-band candidates [bands][frames], normalised scores, event counts [bands][4])
 * of the most recent analysis that used the (n, fs, frame_period, f0_floor, f0_ceil) plan. */
int ryk_debug_dio(ryk_engine* e, int n, int fs, double frame_period_ms, double f0_floor, double f0_ceil,
                  double* f0_raw, double* cand, double* score, int* counts);
/* StoneMask alone on caller-given f0 estimates (frames values, frame i at i * frame_period_ms), shared memory sized from f0_floor
 * as in analysis: an estimate below f0_floor whose FFT would not fit is returned unrefined. */
int ryk_debug_stonemask(ryk_engine* e, const float* wave_host, int n, int fs, double frame_period_ms, double f0_floor,
                        const double* f0_in, int frames, double* f0_out);
/* Harvest internals of the most recent analysis with this plan (engine in f0 method 1): info = {channels, 1 ms frames, decimated
 * length, fft size, candidate columns, decimation ratio, used columns}; y [info[2]], raw [channels][frames], cand / score
 * [frames][columns] (after refinement and removal), best / basic [frames], f0_raw [n / hop + 1] (before StoneMask).  Any may be NULL. */
int ryk_debug_harvest(ryk_engine* e, int n, int fs, double frame_period_ms, double f0_floor, double f0_ceil, int* info, double* y,
                      double* raw, double* cand, double* score, double* best, double* basic, double* f0_raw);
/* Stage-1 forward of padded length Tp stand-alone: ms per forward as one cluster kernel / as 16 layer launches, and the fused
 * kernel's phase timeline (31 doubles, us). */
int ryk_debug_stage1_bench(ryk_engine* e, int Tp, int iters, float* ms_fused, float* ms_layered, double* timeline_us);
/* One conv (transposed = 0) or transposed-conv layer of the U-Nets in isolation, host fp32 NHWC tensors in and
 * out, weights in the Chainer layout; use_tc selects the FP16 tcgen05 kernel (1) or the FP32 CUDA-core kernel (0).
 * `repeat` extra timed runs report the mean device time per run (ms) -- used by the unit parity tests and ncu. */
int ryk_test_conv_layer(ryk_engine* e, int transposed, int k, int stride, int pad, int B, int Hin, int Win, int C0, int C1, int Cout,
                        const float* in0, const float* in1, const float* W, const float* scale, const float* shift, int act,
                        int use_tc, int repeat, float* out, float* ms_per_run);

#ifdef __cplusplus
}
#endif
#endif  /* RYK_H_ */
