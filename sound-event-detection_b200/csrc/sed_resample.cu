// Sample-rate conversion and downmix on the device: the `librosa.load(path, sr=sample_rate, mono=True)` step of the
// reference's caller path (pytorch/predict.py:288-295) for audio that is already decoded, offline (many recordings
// per launch) and live (chunks of many streams, with a per-slot history of input samples).
//
// Definition (scipy.signal.resample_poly(x, up, down, window=h), with hu = up * h the stored float32 taps):
//   y[j] = sum_i x[i] * hu[j*down + half - i*up]      0 <= j < ceil(n_in * up / down),  x[i] = 0 outside [0, n_in)
// summed over ascending i with float32 FMAs.  x is the downmix of C <= 8 interleaved channels, computed as numpy's
// x.astype(float32).mean(axis=1): channel sum in float32 (sequential for C < 8, numpy's pairwise tree for C == 8),
// then an IEEE division by C; int16 PCM is q / 32767 (load_sample, shared with the front-end).
//
// Output j reads the taps of one phase: with t = j*down + half, i_hi = floor(t / up) and r = t mod up, input i
// (i_lo <= i <= i_hi) meets tap r + (i_hi - i)*up.  The taps are used in their natural order -- element (s, r) of the
// [taps_per_phase][up] matrix is tap r + s*up -- so the threads of a warp, which sit on consecutive outputs and
// hence on different phases, read neighbouring words.  A block computes a tile of 256 consecutive outputs, one per
// thread; the input span the tile needs is downmixed once into shared memory (in chunks when it is long), and every
// thread continues its ascending-i sum across the chunks, so the chunking never changes the order of the FMAs.
#include "sed_common.cuh"
#include "sed_kernels.h"
#include "../../include/sed_b200.h"

#include <algorithm>
#include <cmath>

namespace sed {

constexpr int kResampleThreads = 256;   // outputs per tile
constexpr int kResampleChunk = 4096;    // input samples staged per pass (16 KB of shared memory)

template <typename T>
__device__ __forceinline__ float downmix(const T* p, int C) {
  if (C == 8) {  // numpy's pairwise_sum unrolls eight elements into this tree
    const float s = ((load_sample(p) + load_sample(p + 1)) + (load_sample(p + 2) + load_sample(p + 3))) +
                    ((load_sample(p + 4) + load_sample(p + 5)) + (load_sample(p + 6) + load_sample(p + 7)));
    return s / 8.0f;
  }
  float s = load_sample(p);
  for (int c = 1; c < C; ++c) s += load_sample(p + c);
  return s / static_cast<float>(C);
}

struct ResampleFilter {
  const float* taps;  // [2*half + 1] = up * h
  int up, down, half;
  __device__ __forceinline__ long i_hi(long j) const { return (j * down + half) / up; }
  __device__ __forceinline__ long i_lo(long j) const {
    const long t = j * down + half, hi = t / up;
    return hi - (2 * half - (t - hi * up)) / up;
  }
};

// Outputs [j0, min(j0 + kResampleThreads, j_end)) of one signal.  fetch(i) returns x[i] (any i, zeros included);
// store(j, y) writes output j.  Every output is the same FMA chain whatever the tile, chunk or caller: sed_resample and
// sed_live_resample produce identical bits for identical x.
template <typename Fetch, typename Store>
__device__ __forceinline__ void resample_tile(long j0, long j_end, const ResampleFilter& f, float* xs,
                                              const Fetch& fetch, const Store& store) {
  const long j = j0 + threadIdx.x;
  const bool active = j < j_end;
  const long a = f.i_lo(j0), b = f.i_hi(min(j0 + kResampleThreads, j_end) - 1);
  long lo = 0, hi = -1;
  int r = 0;
  if (active) {
    const long t = j * f.down + f.half;
    hi = t / f.up;
    r = static_cast<int>(t - hi * f.up);
    lo = hi - (2 * f.half - r) / f.up;
  }
  float acc = 0.0f;
  for (long c0 = a; c0 <= b; c0 += kResampleChunk) {
    const long c1 = min(c0 + kResampleChunk, b + 1);
    __syncthreads();  // the previous chunk has been consumed
    for (long i = c0 + threadIdx.x; i < c1; i += kResampleThreads) xs[i - c0] = fetch(i);
    __syncthreads();
    const long l = max(lo, c0), h = min(hi, c1 - 1);
    if (l <= h) {
      const float* xp = xs + (l - c0);
      const float* tp = f.taps + r + (hi - l) * f.up;
      const int n = static_cast<int>(h - l + 1), up = f.up;
#pragma unroll 4
      for (int k = 0; k < n; ++k) acc = fmaf(xp[k], __ldg(tp - k * up), acc);
    }
  }
  if (active) store(j, acc);
}

// ---------------------------------------------------------------- offline: many recordings, one launch
// table [n_rows, 4] i64 = (first frame in src, n_in frames, first sample in dst, n_out samples)
template <typename T>
__global__ void __launch_bounds__(kResampleThreads) resample_kernel(const T* __restrict__ src, int C,
                                                                  const long* __restrict__ table, int n_rows,
                                                                  ResampleFilter f, float* __restrict__ dst) {
  __shared__ float xs[kResampleChunk];
  for (int e = blockIdx.y; e < n_rows; e += gridDim.y) {
    const long off = table[4 * e], n_in = table[4 * e + 1], d0 = table[4 * e + 2], n_out = table[4 * e + 3];
    const T* x = src + off * C;
    float* y = dst + d0;
    auto fetch = [&](long i) { return (i >= 0 && i < n_in) ? downmix(x + i * C, C) : 0.0f; };
    auto store = [&](long j, float v) { y[j] = v; };
    for (long j0 = static_cast<long>(blockIdx.x) * kResampleThreads; j0 < n_out;
         j0 += static_cast<long>(gridDim.x) * kResampleThreads)
      resample_tile(j0, n_out, f, xs, fetch, store);
  }
}

static bool filter_ok(int up, int down, int half, int channels, int dtype) {
  return up >= 1 && down >= 1 && half >= 0 && channels >= 1 && channels <= 8 && (dtype == 0 || dtype == 1) &&
         static_cast<long>(half) * 2 < (1L << 30);
}

int resample_launch(const void* src, int dtype, int channels, const long* table, int n_rows, long max_out,
                    const float* taps, int up, int down, int half, float* dst, cudaStream_t stream) {
  if (n_rows < 0 || max_out < 0 || !filter_ok(up, down, half, channels, dtype)) {
    set_error("sed_resample: bad shape rows=%d max_out=%ld up=%d down=%d half=%d channels=%d dtype=%d", n_rows, max_out,
              up, down, half, channels, dtype);
    return SED_ERR_BAD_SHAPE;
  }
  if (n_rows == 0 || max_out == 0) return SED_OK;
  const ResampleFilter f{taps, up, down, half};
  const dim3 grid(static_cast<unsigned>(std::min<long>((max_out + kResampleThreads - 1) / kResampleThreads, 1L << 20)),
                  static_cast<unsigned>(std::min(n_rows, 65535)));
  if (dtype == 0)
    resample_kernel<float><<<grid, kResampleThreads, 0, stream>>>(static_cast<const float*>(src), channels, table,
                                                                  n_rows, f, dst);
  else
    resample_kernel<short><<<grid, kResampleThreads, 0, stream>>>(static_cast<const short*>(src), channels, table,
                                                                  n_rows, f, dst);
  if (cudaGetLastError() != cudaSuccess) {
    set_error("sed_resample: launch failed");
    return SED_ERR_CUDA;
  }
  return SED_OK;
}

// ---------------------------------------------------------------- live: chunks of many streams, per-slot history
// table [n_entries, 6] i64 = (slot, first output j0, outputs, first frame of the stream's chunk in src or -1 for zeros,
// n_prev = input frames before the push, n_end = input frames after it).  Input i of the stream reads the chunk for
// n_prev <= i < n_end, the slot's history ring (hist[slot*H + i mod H]) for 0 <= i < n_prev, zero otherwise; output j
// goes to arena[slot*2*ring + (j mod ring)] and [.. + ring], the layout sed_live_ingest writes.
template <typename T>
__global__ void __launch_bounds__(kResampleThreads) live_resample_kernel(const T* __restrict__ src, int C,
                                                                       const long* __restrict__ table, int n_entries,
                                                                       ResampleFilter f, long ring,
                                                                       float* __restrict__ arena,
                                                                       const float* __restrict__ hist, int H) {
  __shared__ float xs[kResampleChunk];
  for (int e = blockIdx.y; e < n_entries; e += gridDim.y) {
    const long* t = table + 6 * e;
    const long slot = t[0], j_begin = t[1], count = t[2], off = t[3], n_prev = t[4], n_end = t[5];
    float* base = arena + slot * 2 * ring;
    const float* hs = hist + slot * H;
    const T* x = src + (off - n_prev) * C;  // frame i of the stream, for n_prev <= i < n_end
    auto store = [&](long j, float v) {
      const long q = j % ring;
      base[q] = v;
      base[q + ring] = v;
    };
    for (long j0 = j_begin + static_cast<long>(blockIdx.x) * kResampleThreads; j0 < j_begin + count;
         j0 += static_cast<long>(gridDim.x) * kResampleThreads) {
      if (off < 0) {  // zero fill of the closing window 0 of a stream shorter than one window
        const long j = j0 + threadIdx.x;
        if (j < j_begin + count) store(j, 0.0f);
        continue;
      }
      auto fetch = [&](long i) {
        if (i < 0 || i >= n_end) return 0.0f;
        return i < n_prev ? hs[i % H] : downmix(x + i * C, C);
      };
      resample_tile(j0, j_begin + count, f, xs, fetch, store);
    }
  }
}

// history table [n, 4] i64 = (slot, first frame of the chunk in src, n_prev, frames in the chunk): the last
// min(frames, H) input samples of the chunk go to hist[slot*H + i mod H].
template <typename T>
__global__ void live_history_kernel(const T* __restrict__ src, int C, const long* __restrict__ table, int n,
                                    float* __restrict__ hist, int H) {
  for (int e = blockIdx.y; e < n; e += gridDim.y) {
    const long slot = table[4 * e], off = table[4 * e + 1], n_prev = table[4 * e + 2], len = table[4 * e + 3];
    const long keep = min(len, static_cast<long>(H));
    for (long k = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; k < keep;
         k += static_cast<long>(gridDim.x) * blockDim.x) {
      const long s = len - keep + k;
      hist[slot * H + (n_prev + s) % H] = downmix(src + (off + s) * C, C);
    }
  }
}

int live_resample_launch(const void* src, int dtype, int channels, const long* table, int n_entries, long max_len,
                         const float* taps, int up, int down, int half, long ring_samples, float* arena, float* hist,
                         int history_len, const long* history_table, int n_history, cudaStream_t stream) {
  if (n_entries < 0 || max_len < 0 || ring_samples <= 0 || history_len < 1 || n_history < 0 ||
      !filter_ok(up, down, half, channels, dtype)) {
    set_error("sed_live_resample: bad shape entries=%d max_len=%ld ring=%ld history=%d n_history=%d up=%d down=%d "
              "half=%d channels=%d dtype=%d", n_entries, max_len, ring_samples, history_len, n_history, up, down, half,
              channels, dtype);
    return SED_ERR_BAD_SHAPE;
  }
  const ResampleFilter f{taps, up, down, half};
  if (n_entries > 0 && max_len > 0) {
    const dim3 grid(static_cast<unsigned>((max_len + kResampleThreads - 1) / kResampleThreads),
                    static_cast<unsigned>(std::min(n_entries, 65535)));
    if (dtype == 0)
      live_resample_kernel<float><<<grid, kResampleThreads, 0, stream>>>(
          static_cast<const float*>(src), channels, table, n_entries, f, ring_samples, arena, hist, history_len);
    else
      live_resample_kernel<short><<<grid, kResampleThreads, 0, stream>>>(
          static_cast<const short*>(src), channels, table, n_entries, f, ring_samples, arena, hist, history_len);
  }
  if (n_history > 0) {  // after every read of this push's ticks: same stream, launched last
    const dim3 grid(static_cast<unsigned>((history_len + 255) / 256), static_cast<unsigned>(std::min(n_history, 65535)));
    if (dtype == 0)
      live_history_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(src), channels, history_table,
                                                           n_history, hist, history_len);
    else
      live_history_kernel<short><<<grid, 256, 0, stream>>>(static_cast<const short*>(src), channels, history_table,
                                                           n_history, hist, history_len);
  }
  if (cudaGetLastError() != cudaSuccess) {
    set_error("sed_live_resample: launch failed");
    return SED_ERR_CUDA;
  }
  return SED_OK;
}

// ---------------------------------------------------------------- filter design (host)
// resampy's kaiser_best parameters: 64 zero crossings, rolloff 0.9475937167399596, Kaiser beta 14.769656459379492.
static double bessel_i0(double x) {
  const double q = 0.25 * x * x;
  double term = 1.0, sum = 1.0;
  for (int k = 1; k < 500 && term > sum * 1e-18; ++k) {
    term *= q / (static_cast<double>(k) * k);
    sum += term;
  }
  return sum;
}

int resample_filter_host(int in_rate, int out_rate, int* up, int* down, int* n_taps, float* taps) {
  if (in_rate <= 0 || out_rate <= 0 || in_rate > 384000 || out_rate > 384000) {
    set_error("sed_resample_filter: rates %d -> %d (1 .. 384000)", in_rate, out_rate);
    return SED_ERR_BAD_SHAPE;
  }
  int a = in_rate, b = out_rate;
  while (b) {
    const int t = a % b;
    a = b;
    b = t;
  }
  const int u = out_rate / a, d = in_rate / a, mx = std::max(u, d);
  if (mx > 4096) {
    set_error("sed_resample_filter: %d -> %d needs up/down = %d/%d; max(up, down) <= 4096 is supported", in_rate,
              out_rate, u, d);
    return SED_ERR_UNSUPPORTED;
  }
  const int half = 64 * mx, n = 2 * half + 1;
  *up = u;
  *down = d;
  *n_taps = n;
  if (taps == nullptr) return SED_OK;
  // scipy.signal.firwin(n, cutoff, window=('kaiser', beta)) in float64: windowed sinc, DC gain scaled to 1
  const double cutoff = 0.9475937167399596 / mx, beta = 14.769656459379492, pi = 3.141592653589793;
  const double i0_beta = bessel_i0(beta), alpha = 0.5 * (n - 1);
  double* h = new double[n];
  double sum = 0.0;
  for (int k = 0; k < n; ++k) {
    const double m = k - alpha, x = cutoff * m;
    const double y = pi * x;
    const double sinc = (x == 0.0) ? 1.0 : std::sin(y) / y;
    const double z = (k - alpha) / alpha;
    const double w = bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - z * z))) / i0_beta;
    h[k] = cutoff * sinc * w;
    sum += h[k];
  }
  for (int k = 0; k < n; ++k) taps[k] = static_cast<float>(u * (h[k] / sum));
  delete[] h;
  return SED_OK;
}

}  // namespace sed
