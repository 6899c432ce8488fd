// extern "C" boundary: see include/sed_b200.h for the contract of every entry.
#include "../../include/sed_b200.h"

#include <cuda.h>
#include <cuda_runtime.h>
#include <string.h>

#include "sed_kernels.h"

#define SED_ABI_VERSION 13

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

#define SED_REQUIRE(ptr)                                         \
  do {                                                           \
    if ((ptr) == nullptr) {                                      \
      sed::set_error("%s: null pointer argument " #ptr, __func__); \
      return SED_ERR_NULL;                                       \
    }                                                            \
  } while (0)

extern "C" {

int sed_abi_version(void) { return SED_ABI_VERSION; }

const char* sed_last_error_string(void) { return sed::last_error(); }

int sed_frontend_logmel(const void* wave, int wave_dtype, int B, int L, long clip_stride, const long* clip_offset,
                        long total_len, int n_fft, int hop, const float* window, const float* twiddle, const int* mel_lo, const int* mel_len,
                        const int* mel_off, const float* mel_val, int n_mels, float amin, float db_offset, int is_log,
                        const float* bn_scale, const float* bn_shift, float* out, void* stream) {
  SED_REQUIRE(wave); SED_REQUIRE(window); SED_REQUIRE(twiddle); SED_REQUIRE(mel_lo); SED_REQUIRE(mel_len);
  SED_REQUIRE(mel_off); SED_REQUIRE(mel_val); SED_REQUIRE(out);
  if ((bn_scale == nullptr) != (bn_shift == nullptr)) {
    sed::set_error("sed_frontend_logmel: bn_scale and bn_shift must both be set or both be NULL");
    return SED_ERR_NULL;
  }
  sed::FrontendArgs a{};
  a.wave = wave; a.wave_dtype = wave_dtype; a.clip_stride = clip_stride; a.clip_offset = clip_offset;
  a.total_len = total_len;
  a.B = B; a.L = L; a.n_fft = n_fft; a.hop = hop;
  a.T = (hop > 0) ? L / hop + 1 : 0;
  a.window = window; a.twiddle = twiddle;
  a.mel_lo = mel_lo; a.mel_len = mel_len; a.mel_off = mel_off; a.mel_val = mel_val; a.n_mels = n_mels;
  a.amin = amin; a.db_offset = db_offset; a.is_log = is_log;
  a.bn_scale = bn_scale; a.bn_shift = bn_shift; a.out = out; a.mode = 0;
  int rc = sed::frontend_launch(a, as_stream(stream));
  if (rc == SED_ERR_BAD_SHAPE)
    sed::set_error("sed_frontend_logmel: bad shape B=%d L=%d stride=%ld total=%ld n_fft=%d hop=%d", B, L, clip_stride,
                   total_len, n_fft, hop);
  if (rc == SED_ERR_UNSUPPORTED) {
    const int max_hop = sed::frontend_max_hop(n_fft, wave_dtype, n_mels);
    if (max_hop > 0 && hop > max_hop)
      sed::set_error("sed_frontend_logmel: hop=%d too large: the staging buffers of a work item do not fit in shared "
                     "memory (n_fft=%d, %s input, %d mel bands: hop <= %d)", hop, n_fft,
                     wave_dtype == 1 ? "int16" : "float32", n_mels, max_hop);
    else
      sed::set_error("sed_frontend_logmel: n_fft=%d (256/512/1024) or wave_dtype=%d (0/1) unsupported", n_fft,
                     wave_dtype);
  }
  if (rc == SED_ERR_CUDA) sed::set_error("sed_frontend_logmel: %s", cudaGetErrorString(cudaGetLastError()));
  return rc;
}

int sed_spectrogram_f32(const float* wave, int B, int L, int n_fft, int hop, const float* window,
                        const float* twiddle, float* out, void* stream) {
  SED_REQUIRE(wave); SED_REQUIRE(window); SED_REQUIRE(twiddle); SED_REQUIRE(out);
  sed::FrontendArgs a{};
  a.wave = wave; a.wave_dtype = 0; a.clip_stride = L; a.total_len = static_cast<long>(B) * L;
  a.B = B; a.L = L; a.n_fft = n_fft; a.hop = hop;
  a.T = (hop > 0) ? L / hop + 1 : 0;
  a.window = window; a.twiddle = twiddle;
  a.out = out; a.mode = 1;
  int rc = sed::frontend_launch(a, as_stream(stream));
  if (rc == SED_ERR_BAD_SHAPE) sed::set_error("sed_spectrogram_f32: bad shape B=%d L=%d n_fft=%d hop=%d", B, L, n_fft, hop);
  if (rc == SED_ERR_UNSUPPORTED) {
    const int max_hop = sed::frontend_max_hop(n_fft, 0, 0);
    if (max_hop > 0 && hop > max_hop)
      sed::set_error("sed_spectrogram_f32: hop=%d too large: the staging buffers of a work item do not fit in shared "
                     "memory (n_fft=%d: hop <= %d)", hop, n_fft, max_hop);
    else
      sed::set_error("sed_spectrogram_f32: n_fft=%d unsupported (256/512/1024)", n_fft);
  }
  if (rc == SED_ERR_CUDA) sed::set_error("sed_spectrogram_f32: %s", cudaGetErrorString(cudaGetLastError()));
  return rc;
}

int sed_window_merge_avg(const float* frames, int n_windows, int frames_per_window, int classes, int overlap_interval,
                         int sample_duration, int n_recordings, float* merged, void* stream) {
  SED_REQUIRE(frames); SED_REQUIRE(merged);
  return sed::window_merge_launch(frames, n_windows, frames_per_window, classes, overlap_interval, sample_duration,
                                  n_recordings, merged, as_stream(stream));
}

int sed_events(const float* frames, int n_clips, int n_frames, int classes, const double* high, const double* low,
               const int* n_smooth, const int* n_salt, int max_events, int* events, int* counts, void* stream) {
  SED_REQUIRE(frames); SED_REQUIRE(high); SED_REQUIRE(n_smooth); SED_REQUIRE(n_salt); SED_REQUIRE(events);
  SED_REQUIRE(counts);
  return sed::events_launch(frames, n_clips, n_frames, classes, high, low, n_smooth, n_salt, max_events, events, counts,
                            as_stream(stream));
}

int sed_live_ingest(const void* src, int dtype, const long* table, int n_entries, long max_len, long ring_samples,
                    void* arena, void* stream) {
  SED_REQUIRE(src); SED_REQUIRE(table); SED_REQUIRE(arena);
  return sed::live_ingest_launch(src, dtype, table, n_entries, max_len, ring_samples, arena, as_stream(stream));
}

int sed_live_merge(const float* window_frames, const int* table, int n_entries, int max_span, int frames_per_window,
                   int classes, int overlap_interval, int sample_duration, int ring_frames, float* acc, float* out,
                   void* stream) {
  SED_REQUIRE(window_frames); SED_REQUIRE(table); SED_REQUIRE(acc); SED_REQUIRE(out);
  return sed::live_merge_launch(window_frames, table, n_entries, max_span, frames_per_window, classes, overlap_interval,
                                sample_duration, ring_frames, acc, out, as_stream(stream));
}

int sed_live_events(const float* frames, const int* table, int n_entries, int classes, const double* high,
                    const double* low, const int* n_smooth, const int* n_salt, void* state, int* events, int* counts,
                    void* stream) {
  SED_REQUIRE(frames); SED_REQUIRE(table); SED_REQUIRE(high); SED_REQUIRE(n_smooth); SED_REQUIRE(n_salt);
  SED_REQUIRE(state); SED_REQUIRE(events); SED_REQUIRE(counts);
  return sed::live_events_launch(frames, table, n_entries, classes, high, low, n_smooth, n_salt, state, events, counts,
                                 as_stream(stream));
}

int sed_resample_filter(int in_rate, int out_rate, int* up, int* down, int* n_taps, float* taps_or_NULL) {
  SED_REQUIRE(up); SED_REQUIRE(down); SED_REQUIRE(n_taps);
  return sed::resample_filter_host(in_rate, out_rate, up, down, n_taps, taps_or_NULL);
}

int sed_resample(const void* src, int dtype, int channels, const long* table, int n_rows, long max_out,
                 const float* taps, int up, int down, int half, float* dst, void* stream) {
  SED_REQUIRE(src); SED_REQUIRE(table); SED_REQUIRE(taps); SED_REQUIRE(dst);
  return sed::resample_launch(src, dtype, channels, table, n_rows, max_out, taps, up, down, half, dst,
                              as_stream(stream));
}

int sed_live_resample(const void* src, int dtype, int channels, const long* table, int n_entries, long max_len,
                      const float* taps, int up, int down, int half, long ring_samples, float* arena, float* hist,
                      int history_len, const long* history_table, int n_history, void* stream) {
  SED_REQUIRE(src); SED_REQUIRE(taps); SED_REQUIRE(arena); SED_REQUIRE(hist);
  if (n_entries > 0) SED_REQUIRE(table);  // a push's last call may only update the history
  if (n_history > 0) SED_REQUIRE(history_table);
  return sed::live_resample_launch(src, dtype, channels, table, n_entries, max_len, taps, up, down, half, ring_samples,
                                   arena, hist, history_len, history_table, n_history, as_stream(stream));
}

int sed_logmel_rows_f32(const float* spec, long rows, int F, const int* mel_lo, const int* mel_len,
                        const int* mel_off, const float* mel_val, int n_mels, float amin, float db_offset,
                        int is_log, float* out, void* stream) {
  SED_REQUIRE(spec); SED_REQUIRE(mel_lo); SED_REQUIRE(mel_len); SED_REQUIRE(mel_off); SED_REQUIRE(mel_val);
  SED_REQUIRE(out);
  int rc = sed::logmel_rows_launch(spec, rows, F, mel_lo, mel_len, mel_off, mel_val, n_mels, amin, db_offset, is_log,
                                   out, as_stream(stream));
  if (rc == SED_ERR_BAD_SHAPE) sed::set_error("sed_logmel_rows_f32: bad shape rows=%ld", rows);
  return rc;
}

int sed_conv_first_f32(const float* x, int NB, int H, int W, const float* w9, const float* scale,
                       const float* shift, void* out, int dtype, void* stream) {
  SED_REQUIRE(x); SED_REQUIRE(w9); SED_REQUIRE(scale); SED_REQUIRE(shift); SED_REQUIRE(out);
  if (dtype != SED_DTYPE_F16 && dtype != SED_DTYPE_BF16) {
    sed::set_error("sed_conv_first_f32: dtype must be SED_DTYPE_F16 or SED_DTYPE_BF16");
    return SED_ERR_UNSUPPORTED;
  }
  return sed::conv_first_launch(x, NB, H, W, w9, scale, shift, out, dtype, as_stream(stream));
}

int sed_conv3x3_bn_relu(const void* x, int NB, int H, int W, int cin, const void* wpacked, const float* scale,
                        const float* shift, int cout, int mode, void* out, void* out_f32, long out_stride_n,
                        long out_stride_h, int dtype, void* stream) {
  SED_REQUIRE(x); SED_REQUIRE(wpacked); SED_REQUIRE(scale); SED_REQUIRE(shift); SED_REQUIRE(out);
  return sed::conv3x3_launch(x, NB, H, W, cin, wpacked, scale, shift, cout, mode, out, out_f32, out_stride_n,
                             out_stride_h, dtype, as_stream(stream));
}

int sed_conv_block1(const float* x, int NB, int H, int W, const float* w1_scaled, const float* shift1,
                    const void* w2packed, const float* scale2, const float* shift2, void* out, int dtype,
                    void* stream) {
  SED_REQUIRE(x); SED_REQUIRE(w1_scaled); SED_REQUIRE(shift1); SED_REQUIRE(w2packed); SED_REQUIRE(scale2);
  SED_REQUIRE(shift2); SED_REQUIRE(out);
  return sed::conv_block1_launch(x, NB, H, W, w1_scaled, shift1, w2packed, scale2, shift2, out, dtype,
                                 as_stream(stream));
}

int sed_linear(const void* a16, long M, int K, const void* w16, const float* bias, int N, int relu, float* out,
               void* out16, int out_layout, int dtype, void* stream) {
  SED_REQUIRE(a16); SED_REQUIRE(w16);
  if (out == nullptr) SED_REQUIRE(out16);
  return sed::linear_launch(a16, M, K, w16, bias, N, relu, out, out16, out_layout, dtype, as_stream(stream));
}

// ---- peer-memory result buffers (see sed_b200.h) ----
static int peer_fail(const char* what, cudaError_t e) {
  sed::set_error("%s: %s", what, cudaGetErrorString(e));
  cudaGetLastError();
  return SED_ERR_CUDA;
}

int sed_peer_alloc(long bytes, void** dev_ptr) {
  SED_REQUIRE(dev_ptr);
  if (bytes <= 0) {
    sed::set_error("sed_peer_alloc: bytes=%ld", bytes);
    return SED_ERR_BAD_SHAPE;
  }
  cudaError_t e = cudaMalloc(dev_ptr, static_cast<size_t>(bytes));
  return e == cudaSuccess ? SED_OK : peer_fail("sed_peer_alloc", e);
}

int sed_peer_free(void* dev_ptr) {
  SED_REQUIRE(dev_ptr);
  cudaError_t e = cudaFree(dev_ptr);
  return e == cudaSuccess ? SED_OK : peer_fail("sed_peer_free", e);
}

int sed_peer_export(const void* dev_ptr, unsigned char* handle64) {
  SED_REQUIRE(dev_ptr); SED_REQUIRE(handle64);
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, const_cast<void*>(dev_ptr));
  if (e != cudaSuccess) return peer_fail("sed_peer_export", e);
  memcpy(handle64, &h, 64);
  return SED_OK;
}

int sed_peer_open(const unsigned char* handle64, void** dev_ptr) {
  SED_REQUIRE(handle64); SED_REQUIRE(dev_ptr);
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  cudaError_t e = cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess);
  return e == cudaSuccess ? SED_OK : peer_fail("sed_peer_open", e);
}

int sed_peer_close(void* dev_ptr) {
  SED_REQUIRE(dev_ptr);
  cudaError_t e = cudaIpcCloseMemHandle(dev_ptr);
  return e == cudaSuccess ? SED_OK : peer_fail("sed_peer_close", e);
}

int sed_peer_copy(void* dst, const void* src, long bytes, void* stream) {
  SED_REQUIRE(dst); SED_REQUIRE(src);
  if (bytes <= 0) {
    sed::set_error("sed_peer_copy: bytes=%ld", bytes);
    return SED_ERR_BAD_SHAPE;
  }
  cudaError_t e = cudaMemcpyAsync(dst, src, static_cast<size_t>(bytes), cudaMemcpyDefault, as_stream(stream));
  return e == cudaSuccess ? SED_OK : peer_fail("sed_peer_copy", e);
}

// stream-ordered 32-bit flag write / wait (driver stream memory operations): no kernel, no SM
typedef CUresult (*StreamValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
static StreamValue32Fn stream_value_fn(const char* name) {
  void* fp = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint(name, &fp, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess)
    return nullptr;
  return reinterpret_cast<StreamValue32Fn>(fp);
}

int sed_stream_write32(void* dev_ptr, unsigned int value, void* stream) {
  SED_REQUIRE(dev_ptr);
  static StreamValue32Fn fn = stream_value_fn("cuStreamWriteValue32");
  if (!fn) {
    sed::set_error("sed_stream_write32: cuStreamWriteValue32 unavailable");
    return SED_ERR_DRIVER;
  }
  CUresult r = fn(reinterpret_cast<CUstream>(stream), reinterpret_cast<CUdeviceptr>(dev_ptr), value,
                  CU_STREAM_WRITE_VALUE_DEFAULT);
  if (r != CUDA_SUCCESS) {
    sed::set_error("sed_stream_write32: driver error %d", static_cast<int>(r));
    return SED_ERR_DRIVER;
  }
  return SED_OK;
}

int sed_stream_wait_geq32(void* dev_ptr, unsigned int value, void* stream) {
  SED_REQUIRE(dev_ptr);
  static StreamValue32Fn fn = stream_value_fn("cuStreamWaitValue32");
  if (!fn) {
    sed::set_error("sed_stream_wait_geq32: cuStreamWaitValue32 unavailable");
    return SED_ERR_DRIVER;
  }
  CUresult r = fn(reinterpret_cast<CUstream>(stream), reinterpret_cast<CUdeviceptr>(dev_ptr), value,
                  CU_STREAM_WAIT_VALUE_GEQ);
  if (r != CUDA_SUCCESS) {
    sed::set_error("sed_stream_wait_geq32: driver error %d", static_cast<int>(r));
    return SED_ERR_DRIVER;
  }
  return SED_OK;
}

long sed_bigru_workspace_bytes(int B) { return B > 0 ? static_cast<long>(sed::gru_workspace_bytes(B)) : 0; }

int sed_bigru(const float* gi, const void* whh_packed, const float* bhh, int B, int T, float* out, void* workspace,
              int dtype, void* stream) {
  SED_REQUIRE(gi); SED_REQUIRE(whh_packed); SED_REQUIRE(bhh); SED_REQUIRE(out);  // workspace: reserved, may be NULL
  return sed::gru_launch(gi, whh_packed, bhh, B, T, out, workspace, dtype, as_stream(stream));
}

#ifdef SED_PROFILE
int sed_bigru_profile(const float* gi, const void* whh_packed, const float* bhh, int B, int T, float* out,
                      void* workspace, int dtype, long long* stamps, void* stream) {
  SED_REQUIRE(gi); SED_REQUIRE(whh_packed); SED_REQUIRE(bhh); SED_REQUIRE(out); SED_REQUIRE(workspace); SED_REQUIRE(stamps);
  return sed::gru_launch(gi, whh_packed, bhh, B, T, out, workspace, dtype, as_stream(stream), stamps);
}
#endif

int sed_mha_attention(const void* qkv16, const void* qk_lo16, int B, int T, long Bp, void* ctx16, int dtype,
                      void* stream) {
  SED_REQUIRE(qkv16); SED_REQUIRE(ctx16);
  return sed::mha_tc_launch(qkv16, qk_lo16, B, T, Bp, ctx16, dtype, as_stream(stream));
}

int sed_linear_split16(const void* a16, long M, int K, const void* w16, const float* bias, int N, void* out_hi,
                       void* out_lo, int lo_cols, int dtype, void* stream) {
  SED_REQUIRE(a16); SED_REQUIRE(w16); SED_REQUIRE(out_hi); SED_REQUIRE(out_lo);
  return sed::linear_launch(a16, M, K, w16, bias, N, 0, nullptr, out_hi, 0, dtype, as_stream(stream), out_lo, lo_cols);
}

long sed_attpool_blocks_scratch_bytes(int B, int T) {
  return (B > 0 && T > 0) ? static_cast<long>(sed::attpool_blocks_scratch_bytes(B, T)) : 0;
}

int sed_attpool_blocks(const float* x_blocks, int B, int T, const float* w_att, const float* b_att, const float* w_cla,
                       const float* b_cla, int ratio, int frames_out, void* scratch, float* clip, float* frame,
                       float* cla_t, float* norm_att_t, int stage, int clip_begin, int n_clips, void* stream) {
  SED_REQUIRE(x_blocks); SED_REQUIRE(w_att); SED_REQUIRE(b_att); SED_REQUIRE(w_cla); SED_REQUIRE(b_cla);
  SED_REQUIRE(scratch); SED_REQUIRE(clip); SED_REQUIRE(frame);
  return sed::attpool_blocks_launch(x_blocks, B, T, w_att, b_att, w_cla, b_cla, ratio, frames_out, scratch, clip, frame,
                                    cla_t, norm_att_t, stage, clip_begin, n_clips, as_stream(stream));
}

int sed_fcpool(const float* x, int B, int T, const float* w, const float* b, int classes, int ratio, int use_max,
               float* clip, float* frame, void* stream) {
  SED_REQUIRE(x); SED_REQUIRE(w); SED_REQUIRE(b); SED_REQUIRE(clip); SED_REQUIRE(frame);
  return sed::fcpool_launch(x, B, T, w, b, classes, ratio, use_max, clip, frame, as_stream(stream));
}

int sed_mha_core(const float* qkv, int B, int T, long row_stride_t, long row_stride_b, void* out16, int dtype,
                 void* stream) {
  SED_REQUIRE(qkv); SED_REQUIRE(out16);
  return sed::mha_core_launch(qkv, B, T, row_stride_t, row_stride_b, out16, dtype, as_stream(stream));
}

int sed_attpool(const float* x, int B, int T, const float* w_att, const float* b_att, const float* w_cla,
                const float* b_cla, int ratio, int frames_out, float* clip, float* frame, float* cla_t,
                float* norm_att_t, void* stream) {
  SED_REQUIRE(x); SED_REQUIRE(w_att); SED_REQUIRE(b_att); SED_REQUIRE(w_cla); SED_REQUIRE(b_cla);
  SED_REQUIRE(clip); SED_REQUIRE(frame);
  return sed::attpool_launch(x, B, T, w_att, b_att, w_cla, b_cla, ratio, frames_out, clip, frame, cla_t, norm_att_t,
                             as_stream(stream));
}

int sed_fold_bn(const float* weight, const float* bias, const float* running_mean, const float* running_var,
                int channels, double eps, float* scale, float* shift, void* stream) {
  SED_REQUIRE(weight); SED_REQUIRE(bias); SED_REQUIRE(running_mean); SED_REQUIRE(running_var);
  SED_REQUIRE(scale); SED_REQUIRE(shift);
  return sed::fold_bn_launch(weight, bias, running_mean, running_var, channels, eps, scale, shift, as_stream(stream));
}

int sed_pack_conv3x3(const float* w_oihw, int cout, int cin, void* wpacked, int dtype, void* stream) {
  SED_REQUIRE(w_oihw); SED_REQUIRE(wpacked);
  return sed::pack_conv3x3_launch(w_oihw, cout, cin, wpacked, dtype, as_stream(stream));
}

int sed_pack_conv_first(const float* w1, const float* scale1, float* w1_scaled, void* stream) {
  SED_REQUIRE(w1); SED_REQUIRE(scale1); SED_REQUIRE(w1_scaled);
  return sed::pack_conv_first_launch(w1, scale1, w1_scaled, as_stream(stream));
}

int sed_pack_gru_whh(const float* whh_fwd, const float* whh_bwd, void* whh_packed, int dtype, void* stream) {
  SED_REQUIRE(whh_fwd); SED_REQUIRE(whh_bwd); SED_REQUIRE(whh_packed);
  return sed::pack_gru_whh_launch(whh_fwd, whh_bwd, whh_packed, dtype, as_stream(stream));
}

int sed_cast_16(const float* src, long n, void* dst, int dtype, void* stream) {
  SED_REQUIRE(src); SED_REQUIRE(dst);
  return sed::cast16_launch(src, n, dst, dtype, as_stream(stream));
}

int sed_count_saturated16(const void* x, long n, int dtype, unsigned long long* count, void* stream) {
  SED_REQUIRE(x); SED_REQUIRE(count);
  return sed::count_saturated16_launch(x, n, dtype, count, as_stream(stream));
}

int sed_frontend_twiddle(int n_fft, float* twiddle_host) {
  SED_REQUIRE(twiddle_host);
  return sed::frontend_twiddle_host(n_fft, twiddle_host);
}

int sed_band_mel(const float* melW_host, int F, int n_mels, int* mel_lo, int* mel_len, int* mel_off, float* mel_val,
                 int val_capacity, int* n_val) {
  SED_REQUIRE(melW_host); SED_REQUIRE(mel_lo); SED_REQUIRE(mel_len); SED_REQUIRE(mel_off); SED_REQUIRE(mel_val);
  SED_REQUIRE(n_val);
  return sed::band_mel_host(melW_host, F, n_mels, mel_lo, mel_len, mel_off, mel_val, val_capacity, n_val);
}

}  // extern "C"
