// Internal launcher interface between the kernel translation units and the C-ABI (sed_capi.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace sed {

struct FrontendArgs {
  const void* wave;   // clip b = wave + b*clip_stride, L samples (f32 or i16)
  int wave_dtype;     // 0 = float32, 1 = int16 PCM (x = q / 32767)
  long clip_stride;   // samples between clip starts (== L for a dense batch)
  const long* clip_offset;  // optional [B] device table of clip starts (samples from `wave`); overrides clip_stride
  long total_len;     // samples readable from `wave`; beyond -> 0
  int B, L, T, n_fft, hop;
  const float* window;   // [n_fft]
  const float* twiddle;  // [n_fft][2]  exp(-2 pi i k / n_fft)
  const int* mel_lo;     // [n_mels] first non-zero frequency bin
  const int* mel_len;    // [n_mels] band length
  const int* mel_off;    // [n_mels] offset into mel_val
  const float* mel_val;  // banded mel weights
  int n_mels;
  float amin, db_offset;
  int is_log;
  const float* bn_scale;  // [n_mels] or null
  const float* bn_shift;
  float* out;
  int mode;  // 0 = log-mel [B,T,n_mels], 1 = power spectrogram [B,T,F]
};
int frontend_launch(const FrontendArgs& a, cudaStream_t stream);
// largest hop whose staging buffers fit in shared memory (0: n_fft or wave_dtype not built); n_mels 0 = power mode
int frontend_max_hop(int n_fft, int wave_dtype, int n_mels);
int logmel_rows_launch(const float* spec, long rows, int F, const int* mel_lo, const int* mel_len, const int* mel_off,
                       const float* mel_val, int n_mels, float amin, float db_offset, int is_log, float* out,
                       cudaStream_t stream);

// dtype: 0 = fp16, 1 = bf16 (16-bit activation / weight element type of the tensor-core path)
int conv_first_launch(const float* x, int NB, int H, int W, const float* w9, const float* scale, const float* shift,
                      void* out, int dtype, cudaStream_t stream);

// mode: 0 = store NHWC, 1 = 2x2 avg-pool, 2 = freq-mean (W must be 8); every layer runs on CTA pairs
int conv3x3_launch(const void* x, int NB, int H, int W, int cin, const void* wpacked, const float* scale,
                   const float* shift, int cout, int mode, void* out, void* out_f32, long out_sn, long out_sh,
                   int dtype, cudaStream_t stream);

int conv_block1_launch(const float* x, int NB, int H, int W, const float* w1s, const float* shift1, const void* w2packed,
                       const float* scale2, const float* shift2, void* out, int dtype, cudaStream_t stream);

int linear_launch(const void* a16, long M, int K, const void* w16, const float* bias, int N, int relu, float* out,
                  void* out16, int out_layout, int dtype, cudaStream_t stream, void* out_lo = nullptr, int lo_cols = 0);

size_t gru_workspace_bytes(int B);
int gru_launch(const float* gi, const void* whh_packed, const float* bhh, int B, int T, float* out, void* workspace,
               int dtype, cudaStream_t stream, long long* stamps = nullptr);

int window_merge_launch(const float* frames, int n_windows, int frames_per_window, int classes, int overlap_interval,
                        int sample_duration, int n_recordings, float* merged, cudaStream_t stream);

int events_launch(const float* frames, int n_clips, int n_frames, int classes, const double* high, const double* low,
                  const int* n_smooth, const int* n_salt, int max_events, int* events, int* counts,
                  cudaStream_t stream);

int live_ingest_launch(const void* src, int dtype, const long* table, int n_entries, long max_len, long ring_samples,
                       void* arena, cudaStream_t stream);
int live_merge_launch(const float* win, const int* table, int n_entries, int max_span, int frames_per_window,
                      int classes, int overlap_interval, int sample_duration, int ring_frames, float* acc, float* out,
                      cudaStream_t stream);
int live_events_launch(const float* frames, const int* table, int n_entries, int classes, const double* high,
                       const double* low, const int* n_smooth, const int* n_salt, void* state, int* events, int* counts,
                       cudaStream_t stream);

// sed_resample.cu: sample-rate conversion + downmix
int resample_launch(const void* src, int dtype, int channels, const long* table, int n_rows, long max_out,
                    const float* taps, int up, int down, int half, float* dst, cudaStream_t stream);
int live_resample_launch(const void* src, int dtype, int channels, const long* table, int n_entries, long max_len,
                         const float* taps, int up, int down, int half, long ring_samples, float* arena, float* hist,
                         int history_len, const long* history_table, int n_history, cudaStream_t stream);
int resample_filter_host(int in_rate, int out_rate, int* up, int* down, int* n_taps, float* taps);

int mha_core_launch(const float* qkv, int B, int T, long rs_t, long rs_b, void* out16, int dtype, cudaStream_t stream);

int mha_tc_launch(const void* qkv16, const void* qk_lo16, int B, int T, long Bp, void* ctx16, int dtype,
                  cudaStream_t stream);

int attpool_launch(const float* x, int B, int T, const float* w_att, const float* b_att, const float* w_cla,
                   const float* b_cla, int ratio, int frames_out, float* clip, float* frame, float* cla_t,
                   float* norm_att_t, cudaStream_t stream);

size_t attpool_blocks_scratch_bytes(int B, int T);
int attpool_blocks_launch(const float* x_blocks, int B, int T, const float* w_att, const float* b_att,
                          const float* w_cla, const float* b_cla, int ratio, int frames_out, void* scratch, float* clip,
                          float* frame, float* cla_t, float* norm_att_t, int stage, int clip0, int n,
                          cudaStream_t stream);

// sed_pack.cu: weight preparation
int fold_bn_launch(const float* w, const float* b, const float* mean, const float* var, int n, double eps, float* scale,
                   float* shift, cudaStream_t stream);
int pack_conv3x3_launch(const float* w, int cout, int cin, void* out, int dtype, cudaStream_t stream);
int pack_conv_first_launch(const float* w, const float* scale, float* out, cudaStream_t stream);
int pack_gru_whh_launch(const float* fwd, const float* bwd, void* out, int dtype, cudaStream_t stream);
int cast16_launch(const float* src, long n, void* dst, int dtype, cudaStream_t stream);
int count_saturated16_launch(const void* x, long n, int dtype, unsigned long long* count, cudaStream_t stream);
int frontend_twiddle_host(int n_fft, float* out);
int band_mel_host(const float* melW, int F, int M, int* lo, int* len, int* off, float* val, int cap, int* n_val);
int fcpool_launch(const float* x, int B, int T, const float* w, const float* b, int C, int ratio, int use_max,
                  float* clip, float* frame, cudaStream_t stream);

const char* last_error();
void set_error(const char* fmt, ...);

}  // namespace sed
