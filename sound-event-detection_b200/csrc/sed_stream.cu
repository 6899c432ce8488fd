// Streaming post-processing on the device: overlap-add of per-window framewise probabilities and the
// reference's block-wise averaging (utils/utilities.py:405-446 merge / avg_merge, driven by the window loop of
// pytorch/predict.py:297-349).  Pure data movement + one division per element; bit-exact with the numpy code:
// windows are accumulated in ascending order in float32 and divided by float32(num_overlaps).
#include "sed_common.cuh"
#include "sed_kernels.h"
#include "../../include/sed_b200.h"

#include <algorithm>

namespace sed {

__global__ void window_merge_kernel(const float* __restrict__ frames, int n_windows, int fpw, int classes, int oi,
                                    int sample_duration, int total_frames, float* __restrict__ merged) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long>(total_frames) * classes) return;
  frames += static_cast<size_t>(blockIdx.y) * n_windows * fpw * classes;   // recording blockIdx.y
  merged += static_cast<size_t>(blockIdx.y) * total_frames * classes;
  const int f = static_cast<int>(idx / classes);
  const int c = static_cast<int>(idx - static_cast<long>(f) * classes);
  // merge(): window k (0-based) occupies frames [k*oi, k*oi + fpw); later windows are added to the running sum
  int k_lo = (f - fpw + oi) / oi;  // smallest k with f - k*oi < fpw  (ceil((f - fpw + 1) / oi))
  if (f - fpw + 1 <= 0) k_lo = 0;
  int k_hi = f / oi;
  if (k_hi > n_windows - 1) k_hi = n_windows - 1;
  float acc = 0.0f;
  bool first = true;
  for (int k = k_lo; k <= k_hi; ++k) {
    const float v = frames[(static_cast<long>(k) * fpw + (f - k * oi)) * classes + c];
    acc = first ? v : acc + v;
    first = false;
  }
  // avg_merge(): blocks start at i = oi, 2*oi, ... < total - oi; the divisor depends on the block start i
  const int interval = sample_duration * 100 - oi;
  if (f >= oi) {
    const int i = (f / oi) * oi;
    if (i < total_frames - oi) {
      int div;
      if (i < interval) div = i / oi + 1;
      else if (i >= total_frames - interval) div = (total_frames - i) / oi + 1;
      else div = sample_duration;
      acc = acc / static_cast<float>(div);
    }
  }
  merged[idx] = acc;
}

int window_merge_launch(const float* frames, int n_windows, int frames_per_window, int classes, int overlap_interval,
                        int sample_duration, int n_recordings, float* merged, cudaStream_t stream) {
  if (n_recordings <= 0 || n_recordings > 65535 || n_windows <= 0 || frames_per_window <= 0 || classes <= 0 || overlap_interval <= 0 || sample_duration <= 0 ||
      overlap_interval > frames_per_window) {
    set_error("window_merge: bad shape n_windows=%d frames=%d classes=%d overlap_interval=%d duration=%d", n_windows,
              frames_per_window, classes, overlap_interval, sample_duration);
    return SED_ERR_BAD_SHAPE;
  }
  const int total = (n_windows - 1) * overlap_interval + frames_per_window;
  const long n = static_cast<long>(total) * classes;
  window_merge_kernel<<<dim3(static_cast<unsigned>((n + 255) / 256), n_recordings), 256, 0, stream>>>(
      frames, n_windows, frames_per_window, classes, overlap_interval, sample_duration, total, merged);
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}


// =================================================================================================
// Event extraction: double-threshold hysteresis + smoothing + salt removal per (clip, class).
// utils/vad.py:11-45 activity_detection and its helpers :108-199, as called by
// utils/utilities.py:82-153 / pytorch/predict.py:57-121 (frame_prediction_to_event_prediction*).
// One thread per (clip, class) runs the reference's four list passes as a chain of O(1)-state streaming stages:
//   runs of x > high  -> [bgn, fin] with the reference's asymmetric +1s (find_bgn_fin_pairs)
//   -> extension while x >= low (activity_detection_with_second_thres) -> smooth(1) -> smooth(n_smooth)
//   -> drop fin - bgn <= n_salt -> events[clip][class][0..count) = (bgn, fin) in frames.
// Comparisons are done in float64 like numpy does for float32 data against the float64 thresholds of the
// shipped opt_thresholds pickles.
// =================================================================================================
struct SmoothState {
  int has, mem_bgn, last_fin, n;
};

template <typename Emit>
__device__ __forceinline__ void smooth_push(SmoothState& st, int bgn, int fin, Emit emit) {
  if (st.has && (bgn - st.last_fin > st.n)) {
    emit(st.mem_bgn, st.last_fin);
    st.mem_bgn = bgn;
  } else if (!st.has) {
    st.has = 1;
    st.mem_bgn = bgn;
  }
  st.last_fin = fin;
}
template <typename Emit>
__device__ __forceinline__ void smooth_flush(SmoothState& st, Emit emit) {
  if (st.has) emit(st.mem_bgn, st.last_fin);
}

__global__ void events_kernel(const float* __restrict__ frames, int n_clips, int n_frames, int classes,
                              const double* __restrict__ high, const double* __restrict__ low, int use_low,
                              const int* __restrict__ n_smooth, const int* __restrict__ n_salt, int max_events,
                              int* __restrict__ events, int* __restrict__ counts) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_clips * classes) return;
  const int clip = idx / classes, c = idx - clip * classes;
  const float* x = frames + static_cast<size_t>(clip) * n_frames * classes + c;
  auto X = [&](int i) { return static_cast<double>(x[static_cast<size_t>(i) * classes]); };
  const double th = high[c], tl = use_low ? low[c] : 0.0;
  const int salt = n_salt[c];
  int* ev = events + static_cast<size_t>(idx) * max_events * 2;
  int count = 0;

  auto emit_final = [&](int bgn, int fin) {  // remove_salt_noise (vad.py:187-199)
    if (fin - bgn <= salt) return;
    if (count < max_events) {
      ev[2 * count] = bgn;
      ev[2 * count + 1] = fin;
    }
    ++count;
  };
  SmoothState s2{0, 0, 0, n_smooth[c]};  // smooth(n_smooth) in activity_detection (vad.py:38)
  auto emit_s2 = [&](int bgn, int fin) { smooth_push(s2, bgn, fin, emit_final); };
  SmoothState s1{0, 0, 0, 1};            // smooth(n_smooth=1) inside the second-threshold pass (vad.py:154)
  auto emit_s1 = [&](int bgn, int fin) { smooth_push(s1, bgn, fin, emit_s2); };
  auto emit_raw = [&](int bgn, int fin) {  // activity_detection_with_second_thres (vad.py:133-152)
    if (use_low) {
      while (bgn != -1) {
        if (bgn >= n_frames || X(bgn) < tl) break;  // (the reference would raise IndexError at bgn == len(x))
        --bgn;
      }
      while (fin != n_frames) {
        if (X(fin) < tl) break;
        ++fin;
      }
      emit_s1(bgn + 1, fin);
    } else {
      emit_s2(bgn, fin);
    }
  };

  // find_bgn_fin_pairs (vad.py:108-130) over locts = where(x > high)
  int run_start = -1, run_end = -1, runs = 0;
  for (int i = 0; i < n_frames; ++i) {
    if (X(i) > th) {
      if (run_start >= 0 && i - run_end > 1) {  // a gap: the pending run is not the last one
        emit_raw(run_start + (runs > 0 ? 1 : 0), run_end + 1);
        ++runs;
        run_start = i;
      } else if (run_start < 0) {
        run_start = i;
      }
      run_end = i;
    }
  }
  if (run_start >= 0) emit_raw(run_start + (runs > 0 ? 1 : 0), run_end);  // last pair: fin without the +1
  if (use_low) smooth_flush(s1, emit_s2);
  smooth_flush(s2, emit_final);
  counts[idx] = count;
}

int events_launch(const float* frames, int n_clips, int n_frames, int classes, const double* high, const double* low,
                  const int* n_smooth, const int* n_salt, int max_events, int* events, int* counts,
                  cudaStream_t stream) {
  if (n_clips <= 0 || n_frames <= 0 || classes <= 0 || max_events <= 0) {
    set_error("events: bad shape clips=%d frames=%d classes=%d max_events=%d", n_clips, n_frames, classes, max_events);
    return SED_ERR_BAD_SHAPE;
  }
  const int n = n_clips * classes;
  events_kernel<<<(n + 127) / 128, 128, 0, stream>>>(frames, n_clips, n_frames, classes, high, low, low != nullptr,
                                                     n_smooth, n_salt, max_events, events, counts);
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}


// =================================================================================================
// Live streaming: windows of many streams whose audio is still arriving (the rolling window of
// pytorch/predict.py:297-349 run incrementally), merged and turned into events as frames become final.
// Per slot: a mirrored audio ring of 2C samples, a merge accumulator ring of R frames, and one LiveEventState per
// class.  The host keeps the counters (samples, windows run, frames returned) and passes, per push, one table row
// per stream with work: LIVE_SLOT, LIVE_K0 ... (SED_LIVE_TABLE_COLS int32 columns, see sed_b200.h).
// =================================================================================================
enum { LIVE_SLOT, LIVE_K0, LIVE_M, LIVE_ROW0, LIVE_LO, LIVE_FINAL, LIVE_OUT_ROW, LIVE_EV_OFF, LIVE_EV_CAP, LIVE_CLOSING };

// Ingest: entry e = (slot, source offset or -1 for zeros, length, absolute write position) of a [n, 4] int64 table.
// Sample p of a slot goes to (p mod C) and (p mod C) + C of the slot's 2C-sample ring, so that every window -- W <= C
// consecutive samples -- is one contiguous run of the arena whatever its start.
template <typename T>
__global__ void live_ingest_kernel(const T* __restrict__ src, const long* __restrict__ table, int n_entries,
                                   long ring, T* __restrict__ arena) {
  for (int e = blockIdx.y; e < n_entries; e += gridDim.y) {
    const long slot = table[4 * e], off = table[4 * e + 1], len = table[4 * e + 2], pos = table[4 * e + 3];
    T* base = arena + slot * 2 * ring;
    for (long j = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; j < len;
         j += static_cast<long>(gridDim.x) * blockDim.x) {
      const T v = off >= 0 ? src[off + j] : T(0);
      const long q = (pos + j) % ring;
      base[q] = v;
      base[q + ring] = v;
    }
  }
}

int live_ingest_launch(const void* src, int dtype, const long* table, int n_entries, long max_len, long ring_samples,
                       void* arena, cudaStream_t stream) {
  if (n_entries < 0 || max_len < 0 || ring_samples <= 0 || (dtype != 0 && dtype != 1)) {
    set_error("live_ingest: bad shape n_entries=%d max_len=%ld ring=%ld dtype=%d", n_entries, max_len, ring_samples,
              dtype);
    return SED_ERR_BAD_SHAPE;
  }
  if (n_entries == 0 || max_len == 0) return SED_OK;
  const dim3 grid(static_cast<unsigned>(std::min<long>((max_len + 255) / 256, 64)),
                  static_cast<unsigned>(std::min(n_entries, 65535)));
  if (dtype == 0)
    live_ingest_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(src), table, n_entries, ring_samples,
                                                        static_cast<float*>(arena));
  else
    live_ingest_kernel<short><<<grid, 256, 0, stream>>>(static_cast<const short*>(src), table, n_entries, ring_samples,
                                                        static_cast<short*>(arena));
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}

// Incremental merge: entry e brings windows k0 .. k0+m-1 of its slot (rows row0 .. of `win`, ascending k) and
// finalizes frames [lo, n_final).  Frame f lives at acc[slot][f mod R] until it is final.  The arithmetic is
// window_merge_kernel's: the first window that covers f SETS it, later windows add in ascending k, and a final frame
// is divided by avg_merge's divisor for total = (k0+m-1)*oi + fpw.  That total is the real one at close; before
// close a frame is only final when its divisor is the same for every total the stream can still reach (the host's
// finality rule), so the divisor computed with the current total is its divisor.  Final frames are written packed to
// out[out_row + f - lo].
__global__ void live_merge_kernel(const float* __restrict__ win, const int* __restrict__ table, int n_entries, int fpw,
                                  int classes, int oi, int sample_duration, int ring, float* __restrict__ acc_all,
                                  float* __restrict__ out) {
  for (int e = blockIdx.y; e < n_entries; e += gridDim.y) {
    const int* t = table + static_cast<size_t>(e) * SED_LIVE_TABLE_COLS;
    const int slot = t[LIVE_SLOT], k0 = t[LIVE_K0], m = t[LIVE_M], row0 = t[LIVE_ROW0], lo = t[LIVE_LO];
    const int n_final = t[LIVE_FINAL], out_row = t[LIVE_OUT_ROW];
    const int k_last = k0 + m - 1;
    const int total = k_last * oi + fpw;
    const int hi = m > 0 ? total : n_final;
    const int touched = k0 >= 1 ? (k0 - 1) * oi + fpw : 0;  // frames some earlier window already covers
    float* acc = acc_all + static_cast<size_t>(slot) * ring * classes;
    const long n = static_cast<long>(hi - lo) * classes;
    for (long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < n;
         idx += static_cast<long>(gridDim.x) * blockDim.x) {
      const int f = lo + static_cast<int>(idx / classes);
      const int c = static_cast<int>(idx % classes);
      float* a = acc + static_cast<size_t>(f % ring) * classes + c;
      bool first = f >= touched;
      float v = first ? 0.0f : *a;
      int k_lo = (f - fpw + oi) / oi;
      if (f - fpw + 1 <= 0) k_lo = 0;
      const int k_hi = min(k_last, f / oi);
      for (int k = max(k0, k_lo); k <= k_hi; ++k) {
        const float w = win[(static_cast<long>(row0 + k - k0) * fpw + (f - k * oi)) * classes + c];
        v = first ? w : v + w;
        first = false;
      }
      if (f < n_final) {
        const int interval = sample_duration * 100 - oi;
        if (f >= oi) {
          const int i = (f / oi) * oi;
          if (i < total - oi) {
            int div;
            if (i < interval) div = i / oi + 1;
            else if (i >= total - interval) div = (total - i) / oi + 1;
            else div = sample_duration;
            v = v / static_cast<float>(div);
          }
        }
        out[static_cast<size_t>(out_row + f - lo) * classes + c] = v;
      } else {
        *a = v;
      }
    }
  }
}

int live_merge_launch(const float* win, const int* table, int n_entries, int max_span, int frames_per_window,
                      int classes, int overlap_interval, int sample_duration, int ring_frames, float* acc, float* out,
                      cudaStream_t stream) {
  if (n_entries < 0 || max_span < 0 || frames_per_window <= 0 || classes <= 0 || overlap_interval <= 0 ||
      overlap_interval > frames_per_window || sample_duration <= 0 || ring_frames < frames_per_window ||
      max_span > ring_frames) {
    set_error("live_merge: bad shape entries=%d span=%d frames=%d classes=%d overlap_interval=%d duration=%d ring=%d",
              n_entries, max_span, frames_per_window, classes, overlap_interval, sample_duration, ring_frames);
    return SED_ERR_BAD_SHAPE;
  }
  if (n_entries == 0 || max_span == 0) return SED_OK;
  const long n = static_cast<long>(max_span) * classes;
  const dim3 grid(static_cast<unsigned>((n + 255) / 256), static_cast<unsigned>(std::min(n_entries, 65535)));
  live_merge_kernel<<<grid, 256, 0, stream>>>(win, table, n_entries, frames_per_window, classes, overlap_interval,
                                              sample_duration, ring_frames, acc, out);
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}

// Streaming activity_detection: the chain of events_kernel (runs above `high` -> pairs -> low-threshold extension ->
// smooth(1) -> smooth(n_smooth) -> salt) with the two walks of the extension replaced by state:
//   extended onset  S = (last frame at or before bgn below `low`) + 1       -> last_below when frame bgn arrives
//   extended offset E = first frame at or after fin below `low` (or len)  -> fbr: first such frame after run_end
// Why one pending pair is enough: every raw pair whose bgn lies inside one stretch of frames >= low extends to the
// same [S, E] -- S is the stretch's first frame, and E is the first frame below `low` after the stretch, because the
// pair's fin (run_end or run_end + 1) lies in the stretch or just after it.  smooth(1) then collapses such pairs
// (bgn - previous fin < 0).  So when a new run starts before the previous pair's E is known (no frame below `low`
// since its run ended), that pair is parked in `q` for one frame: if the next frame (the new pair's bgn) is >= low,
// both pairs are the same and `q` is dropped; if it is below, it is q's E.  A pair is pushed as soon as its run is over
// and its E is known (when x[run_end] < low -- only possible with high < low -- E depends on whether the pair is the
// last one and waits for the next run or the close).  smooth(1) / smooth(n_smooth) emit a pending group early once
// no later pair can merge with it: no pair is pending, and every later pair starts at or after last_below + 1.
// Without a low threshold the pair of the current run stays open until the next run starts (fin = run_end + 1) or
// the close (the last pair's fin has no +1).  O(1) ints per (slot, class); comparisons in float64 like events_kernel.
struct LiveEventState {
  int run_end, p_has, p_b, p_s, p_sk, p_pushed, p_lowend, fbr, last_below, q_has, q_s;
  SmoothState s1, s2;
};
static_assert(sizeof(LiveEventState) == SED_LIVE_EVENT_STATE_INTS * sizeof(int), "LiveEventState layout");

__global__ void live_events_kernel(const float* __restrict__ frames, const int* __restrict__ table, int n_entries,
                                   int classes, const double* __restrict__ high, const double* __restrict__ low,
                                   int use_low, const int* __restrict__ n_smooth, const int* __restrict__ n_salt,
                                   LiveEventState* __restrict__ state, int* __restrict__ events,
                                   int* __restrict__ counts) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long>(n_entries) * classes) return;
  const int e = static_cast<int>(idx / classes), c = static_cast<int>(idx % classes);
  const int* t = table + static_cast<size_t>(e) * SED_LIVE_TABLE_COLS;
  const int slot = t[LIVE_SLOT], lo = t[LIVE_LO], n = t[LIVE_FINAL] - lo, out_row = t[LIVE_OUT_ROW];
  const int cap = t[LIVE_EV_CAP], closing = t[LIVE_CLOSING];
  int* ev = events + (static_cast<size_t>(t[LIVE_EV_OFF]) + static_cast<size_t>(c) * cap) * 2;
  const double th = high[c], tl = use_low ? low[c] : 0.0;
  const int salt = n_salt[c];
  LiveEventState st = state[static_cast<size_t>(slot) * classes + c];
  if (lo == 0) {  // first frames of the stream: whatever the slot held before is gone
    st = LiveEventState{-1, 0, 0, 0, 0, 0, 0, -1, -1, 0, 0, {0, 0, 0, 0}, {0, 0, 0, 0}};
  }
  st.s1.n = 1;
  st.s2.n = n_smooth[c];
  int count = 0;
  auto emit_final = [&](int bgn, int fin) {
    if (fin - bgn <= salt) return;
    if (count < cap) {
      ev[2 * count] = bgn;
      ev[2 * count + 1] = fin;
    }
    ++count;
  };
  auto emit_s2 = [&](int bgn, int fin) { smooth_push(st.s2, bgn, fin, emit_final); };
  auto emit_s1 = [&](int bgn, int fin) { smooth_push(st.s1, bgn, fin, emit_s2); };

  const float* x = frames + static_cast<size_t>(out_row) * classes + c;
  for (int j = 0; j < n; ++j) {
    const int i = lo + j;
    const double v = static_cast<double>(x[static_cast<size_t>(j) * classes]);
    if (!use_low) {
      if (v > th) {
        if (st.p_has && i - st.run_end > 1) {  // a gap: the pending pair is not the last one
          emit_s2(st.p_b, st.run_end + 1);
          st.p_b = i + 1;
        } else if (!st.p_has) {
          st.p_has = 1;
          st.p_b = i;
        }
        st.run_end = i;
      }
      continue;
    }
    const bool below = v < tl;
    if (v > th) {
      if (st.p_has && i - st.run_end > 1) {
        if (!st.p_pushed) {
          if (st.fbr >= 0) {
            emit_s1(st.p_s, st.fbr);
          } else {
            st.q_has = 1;
            st.q_s = st.p_s;
          }
        }
        st.p_b = i + 1; st.p_sk = 0; st.p_pushed = 0;
      } else if (!st.p_has) {
        st.p_has = 1; st.p_b = i; st.p_sk = 0; st.p_pushed = 0;
      }
      st.run_end = i; st.fbr = -1; st.p_lowend = below;
    }
    if (st.p_has && !st.p_sk && st.p_b == i) {
      st.p_s = below ? i + 1 : st.last_below + 1;
      st.p_sk = 1;
    }
    if (below) {
      if (st.q_has) {
        emit_s1(st.q_s, i);
        st.q_has = 0;
      }
      if (st.fbr < 0 && i > st.run_end) st.fbr = i;
      st.last_below = i;
    } else if (st.q_has && i == st.p_b) {
      st.q_has = 0;  // the new run's pair extends to the same [S, E]: smooth(1) would collapse the two
    }
    if (st.p_has && !st.p_pushed && !st.q_has && st.p_sk && !st.p_lowend && st.fbr >= 0) {
      emit_s1(st.p_s, st.fbr);
      st.p_pushed = 1;
    }
    if (!st.q_has && (!st.p_has || st.p_pushed)) {
      const int lb = st.last_below + 1;  // no later pair starts before this frame
      if (st.s1.has && lb - st.s1.last_fin > 1) {
        emit_s2(st.s1.mem_bgn, st.s1.last_fin);
        st.s1.has = 0;
      }
      if (st.s2.has && !st.s1.has && lb - st.s2.last_fin > st.s2.n) {
        emit_final(st.s2.mem_bgn, st.s2.last_fin);
        st.s2.has = 0;
      }
    }
    if (st.s2.has && st.s1.has && st.s1.mem_bgn - st.s2.last_fin > st.s2.n) {
      emit_final(st.s2.mem_bgn, st.s2.last_fin);
      st.s2.has = 0;
    }
  }
  if (closing) {
    const int len = lo + n;
    if (!use_low) {
      if (st.p_has) emit_s2(st.p_b, st.run_end);  // last pair: fin without the +1
    } else {
      if (st.q_has) emit_s1(st.q_s, len);
      if (st.p_has && !st.p_pushed) {
        const int s = st.p_sk ? st.p_s : len + 1;  // bgn == len: the reference's walk stops at once
        emit_s1(s, st.p_lowend ? st.run_end : (st.fbr >= 0 ? st.fbr : len));
      }
      smooth_flush(st.s1, emit_s2);
    }
    smooth_flush(st.s2, emit_final);
  }
  state[static_cast<size_t>(slot) * classes + c] = st;
  counts[idx] = count;
}

int live_events_launch(const float* frames, const int* table, int n_entries, int classes, const double* high,
                       const double* low, const int* n_smooth, const int* n_salt, void* state, int* events, int* counts,
                       cudaStream_t stream) {
  if (n_entries < 0 || classes <= 0) {
    set_error("live_events: bad shape entries=%d classes=%d", n_entries, classes);
    return SED_ERR_BAD_SHAPE;
  }
  if (n_entries == 0) return SED_OK;
  const long n = static_cast<long>(n_entries) * classes;
  live_events_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, stream>>>(
      frames, table, n_entries, classes, high, low, low != nullptr, n_smooth, n_salt,
      static_cast<LiveEventState*>(state), events, counts);
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}

}  // namespace sed
