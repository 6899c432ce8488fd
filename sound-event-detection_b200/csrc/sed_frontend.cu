// Fused audio front-end for sm_100a: reflect-pad -> frame -> window -> real DFT -> power -> mel
// projection -> clamped 10*log10 -> bn0 affine, one kernel, float32 end to end.
//
// Reference: STFT.forward pytorch/stft.py:223-247 (two Conv1d with the windowed DFT matrix),
// Spectrogram.forward :651-670, LogmelFilterBank.forward/power_to_db :698-734, bn0 models.py:642-644.
//
// The reference evaluates the DFT as a dense [n_fft x (n_fft/2+1)] contraction (0.53 GFLOP per 10 s
// clip at 16 kHz).  Here two consecutive real frames are packed as one complex sequence and pushed
// through an in-shared-memory FFT, 25x fewer flops, in float32 with float64-derived twiddles -- the
// accuracy class of the reference's float32 conv1d, which the 1e-4 log-mel tolerance needs (single-pass
// 16-bit tensor-core DFTs do not reach it).  The window is read from the loaded conv_real kernel (row 0),
// so a checkpoint's window is honoured; the host wrapper verifies that the loaded kernels are a windowed
// DFT before selecting this path.  The mel projection uses the loaded melW in banded form (first/last
// non-zero per mel bin), cut into equal segments per persistent block (build_mel_schedule).
//
// Two kernels share everything but the transform:
//   frontend_kernel   n_fft 256 / 512: three Stockham passes (4 x 8 x 8, 8 x 8 x 8) over a swizzled buffer, the
//                     last one left in registers; four blocks of four warps per SM
//   frontend2_kernel  n_fft 1024: 32 x 32 in two passes, twiddles applied by the producing lane, ONE trip through
//                     shared memory; two blocks of six warps per SM
// Both end with X[.] of a frame pair spread over the warp's registers, split the two real spectra with one shuffle
// per component, and run the same mel projection / dB conversion / bn0 epilogue.  DESIGN.md K1 has the measurements
// behind every choice; tests/test_frontend_schedule_model.py restates the index arithmetic on the CPU.
#include <atomic>
#include <cstdlib>

#include "sed_common.cuh"
#include "sed_kernels.h"

namespace sed {

// Block shapes (compile-time knobs of the A/B runs in profiles/r02_frontend_ab_block_shapes.log).  The warps of a block
// meet at one barrier per work item and therefore run in phase -- all load, then all compute; several SMALL blocks per SM
// interleave their phases.  Same warps per SM, ms per 148 clips of 10 s on one box: n_fft 512 2 x 8 warps 0.136 -> 4 x 4
// warps 0.129; n_fft 256 0.093 -> 0.089; n_fft 1024 (two-pass kernel) 1 x 12 warps 0.249 -> 2 x 6 warps 0.214.
#ifndef SED_FE_WARPS3
#define SED_FE_WARPS3 4   // three-pass kernel, n_fft 256 / 512: warps per block ...
#define SED_FE_BLOCKS3 4  // ... and blocks per SM
#endif
#ifndef SED_FE_WARPS2_1024
#define SED_FE_WARPS2_1024 6   // two-pass kernel, n_fft 1024: warps per block ...
#define SED_FE_BLOCKS2_1024 2  // ... and blocks per SM
#endif
#ifndef SED_FE_WARPS2
#define SED_FE_WARPS2 4   // two-pass kernel, n_fft 256 / 512 (not the default kernel for these sizes)
#define SED_FE_BLOCKS2 3
#endif

template <int NFFT>
struct FrontCfg {
  // 256 / 512: SED_FE_BLOCKS3 blocks of SED_FE_WARPS3 warps (16 warps per SM at 127 registers); 1024 (only where the
  // two-pass kernel's buffers do not fit): one block of 12 warps
  static constexpr int WARPS = (NFFT == 1024) ? 12 : SED_FE_WARPS3;
  // frames per work item (even: frames are transformed in pairs) for 4-byte samples: two pairs per warp; 2-byte PCM
  // takes twice as many in the same staging space (fpb()).  A persistent block loops over work items = (clip, chunk of
  // frames); the waveform segment of the next item arrives by bulk copy while the current one is transformed.
  static constexpr int FPB = (NFFT == 1024) ? 24 : 4 * SED_FE_WARPS3;
  template <typename TIn>
  static constexpr int fpb() { return FPB * (sizeof(TIn) == 2 ? 2 : 1); }
  static constexpr int MIN_BLOCKS = (NFFT == 1024) ? 1 : SED_FE_BLOCKS3;
  // Mel projection: every band is cut into segments of SEG consecutive bins, one lane per segment, 32 segments per
  // round (see build_mel_schedule).  SEG is odd, so the 64-bit power reads of neighbouring segments of a band fall
  // into different banks; the values below give the fewest rows (rounds * SEG) for the reference's three presets
  // (8 kHz: 9 rows for 219 non-zero weights, 16 kHz: 21 for 436, 32 kHz: 36 for 866).  Other mel matrices only change
  // the number of rounds; beyond SEGS_MAX segments the projection falls back to one lane per band.
  static constexpr int SEG = (NFFT == 256) ? 3 : (NFFT == 512) ? 7 : 9;
  // segment sums live behind the power spectrum in the warp's own buffer: (NFFT - F) float2 slots are free
  static constexpr int SEGS_MAX = (NFFT == 256) ? 96 : 160;
  // segments of one band summed without a loop (widest band of the presets: 8 / 20 / 47 bins = 3 / 3 / 6 segments)
  static constexpr int NP_UNROLL = (NFFT == 1024) ? 6 : 3;
  // rounds of the presets (91 / 94 / 127 segments); this count runs fully unrolled, any other in a loop
  static constexpr int ROUNDS_UNROLL = (NFFT == 1024) ? 4 : 3;
};

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// Shared-memory FFT buffers are XOR-swizzled (low four bits of the complex index ^= bits 3..6): the unit-stride reads of
// a Stockham pass stay conflict-free and its strided autosort writes spread over the banks.  Simulated 64-bit
// wavefronts per 512-point transform: 212 against 324 with one-in-eight padding (ideal 196); 1024: 612 vs 964.
__host__ __device__ constexpr int pidx(int i) { return i ^ ((i >> 3) & 15); }

// pidx is linear over XOR, and every index a pass touches is (a part that depends on the lane) + (a compile-time part)
// with disjoint bits: element (lanepart + c) lives at pidx(lanepart) ^ pidx(c).  `base` = byte address of
// pidx(lanepart) in a 128-byte aligned buffer; the low four index bits of pidx(c) are XORed in, the rest is an
// immediate offset -- one LOP3 (or nothing) per access instead of the shift / and / xor / scale chain.
__device__ __forceinline__ uint32_t eaddr(uint32_t base, int c) {
  const int p = pidx(c);
  return (base ^ static_cast<uint32_t>((p & 15) << 3)) + static_cast<uint32_t>((p & ~15) << 3);
}
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f2(uint32_t addr, float2 v) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}

// complex add / sub as ONE packed instruction (FADD2 on a 64-bit register pair, sm_100): same IEEE results as two FADD
__device__ __forceinline__ float2 cadd(float2 a, float2 b) {
  unsigned long long x, y, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(y) : "f"(b.x), "f"(b.y));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(x), "l"(y));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(d));
  return r;
}
__device__ __forceinline__ float2 csub(float2 a, float2 b) {
  unsigned long long x, y, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(y) : "f"(b.x), "f"(b.y));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(x), "l"(y));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(d));
  return r;
}

template <int R>
__device__ __forceinline__ void butterfly(float2 (&v)[R]);

template <>
__device__ __forceinline__ void butterfly<2>(float2 (&v)[2]) {
  const float2 a0 = v[0], a1 = v[1];
  v[0] = cadd(a0, a1);
  v[1] = csub(a0, a1);
}

template <>
__device__ __forceinline__ void butterfly<4>(float2 (&v)[4]) {
  const float2 a0 = cadd(v[0], v[2]);
  const float2 a1 = csub(v[0], v[2]);
  const float2 a2 = cadd(v[1], v[3]);
  const float2 a3 = csub(v[1], v[3]);
  v[0] = cadd(a0, a2);
  v[1] = make_float2(a1.x + a3.y, a1.y - a3.x);  // a1 - i*a3
  v[2] = csub(a0, a2);
  v[3] = make_float2(a1.x - a3.y, a1.y + a3.x);  // a1 + i*a3
}

template <>
__device__ __forceinline__ void butterfly<8>(float2 (&v)[8]) {
  constexpr float kS = 0.70710678118654752440f;
  float2 a[4], b[4];
#pragma unroll
  for (int n = 0; n < 4; ++n) {
    a[n] = cadd(v[n], v[n + 4]);
    b[n] = csub(v[n], v[n + 4]);
  }
  // b[n] *= W8^n  (W8 = exp(-2 pi i / 8))
  b[1] = make_float2((b[1].x + b[1].y) * kS, (b[1].y - b[1].x) * kS);
  b[2] = make_float2(b[2].y, -b[2].x);
  b[3] = make_float2((b[3].y - b[3].x) * kS, -(b[3].x + b[3].y) * kS);
  butterfly<4>(a);
  butterfly<4>(b);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    v[2 * k] = a[k];
    v[2 * k + 1] = b[k];
  }
}

template <>
__device__ __forceinline__ void butterfly<16>(float2 (&v)[16]) {
  // n = 4a + i, k = m + 4p:  X[m + 4p] = sum_i W4^{ip} W16^{im} sum_a x[4a + i] W4^{am}
  constexpr float kC1 = 0.92387953251128675613f, kS1 = 0.38268343236508977173f;  // cos, sin(pi / 8)
  constexpr float kS = 0.70710678118654752440f;
  float2 u[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t[4] = {v[i], v[i + 4], v[i + 8], v[i + 12]};
    butterfly<4>(t);
#pragma unroll
    for (int m = 0; m < 4; ++m) u[i][m] = t[m];
  }
  // u[i][m] *= W16^{i m},  W16 = exp(-2 pi i / 16)
  u[1][1] = cmul(u[1][1], make_float2(kC1, -kS1));
  u[1][2] = make_float2((u[1][2].x + u[1][2].y) * kS, (u[1][2].y - u[1][2].x) * kS);      // W16^2 = W8
  u[1][3] = cmul(u[1][3], make_float2(kS1, -kC1));
  u[2][1] = make_float2((u[2][1].x + u[2][1].y) * kS, (u[2][1].y - u[2][1].x) * kS);      // W16^2
  u[2][2] = make_float2(u[2][2].y, -u[2][2].x);                                            // W16^4 = -i
  u[2][3] = make_float2((u[2][3].y - u[2][3].x) * kS, -(u[2][3].x + u[2][3].y) * kS);     // W16^6
  u[3][1] = cmul(u[3][1], make_float2(kS1, -kC1));                                         // W16^3
  u[3][2] = make_float2((u[3][2].y - u[3][2].x) * kS, -(u[3][2].x + u[3][2].y) * kS);     // W16^6
  u[3][3] = cmul(u[3][3], make_float2(-kC1, kS1));                                         // W16^9 = -W16^1
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    float2 t[4] = {u[0][m], u[1][m], u[2][m], u[3][m]};
    butterfly<4>(t);
#pragma unroll
    for (int pq = 0; pq < 4; ++pq) v[m + 4 * pq] = t[pq];
  }
}

template <>
__device__ __forceinline__ void butterfly<32>(float2 (&v)[32]) {
  // decimation in frequency: a[n] = v[n] + v[n + 16], b[n] = (v[n] - v[n + 16]) W32^n; X[2k] = DFT16(a)[k],
  // X[2k + 1] = DFT16(b)[k]
  constexpr float kC[16] = {1.0f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                            0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f,
                            0.19509032201612826785f, 0.0f, -0.19509032201612826785f, -0.38268343236508977173f,
                            -0.55557023301960222474f, -0.70710678118654752440f, -0.83146961230254523708f,
                            -0.92387953251128675613f, -0.98078528040323044913f};  // cos(pi n / 16)
  constexpr float kSn[16] = {0.0f, 0.19509032201612826785f, 0.38268343236508977173f, 0.55557023301960222474f,
                             0.70710678118654752440f, 0.83146961230254523708f, 0.92387953251128675613f,
                             0.98078528040323044913f, 1.0f, 0.98078528040323044913f, 0.92387953251128675613f,
                             0.83146961230254523708f, 0.70710678118654752440f, 0.55557023301960222474f,
                             0.38268343236508977173f, 0.19509032201612826785f};  // sin(pi n / 16)
  constexpr float kS = 0.70710678118654752440f;
  float2 a[16], b[16];
#pragma unroll
  for (int n = 0; n < 16; ++n) {
    a[n] = cadd(v[n], v[n + 16]);
    b[n] = csub(v[n], v[n + 16]);
  }
#pragma unroll
  for (int n = 1; n < 16; ++n) {
    if (n == 4) {
      b[n] = make_float2((b[n].x + b[n].y) * kS, (b[n].y - b[n].x) * kS);        // W32^4 = W8
    } else if (n == 8) {
      b[n] = make_float2(b[n].y, -b[n].x);                                        // W32^8 = -i
    } else if (n == 12) {
      b[n] = make_float2((b[n].y - b[n].x) * kS, -(b[n].x + b[n].y) * kS);       // W32^12 = W8^3
    } else {
      b[n] = cmul(b[n], make_float2(kC[n], -kSn[n]));                             // W32^n = cos - i sin
    }
  }
  butterfly<16>(a);
  butterfly<16>(b);
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    v[2 * k] = a[k];
    v[2 * k + 1] = b[k];
  }
}

// Per-lane twiddles of one Stockham pass (radix R, stride Ns) of an N-point transform.  They depend only on the
// lane, not on the frame, so a persistent warp keeps them in registers; the widest case (N = 1024, Ns = 128) reads
// the shared-memory table instead.
template <int N, int R, int Ns>
struct PassTw {
  static constexpr int NB = N / R, BPL = NB / 32;
  static constexpr int NK = (Ns > 32) ? BPL : 1;  // distinct k = (lane + 32 q) % Ns over the lane's butterflies
  static constexpr bool IN_REGS = (Ns > 1) && (NK * (R - 1) <= 14);
  static constexpr int TSTRIDE = N / (Ns * R);
  float2 t[IN_REGS ? NK : 1][R - 1];
  __device__ __forceinline__ void init(const float2* __restrict__ tw, int lane) {
    if (IN_REGS) {
#pragma unroll
      for (int q = 0; q < NK; ++q) {
        const int k = (lane + 32 * q) % Ns;
#pragma unroll
        for (int r = 1; r < R; ++r) t[q][r - 1] = tw[r * k * TSTRIDE];
      }
    }
  }
};

// load_sample (int16 PCM as q / 32767, correctly rounded) lives in sed_common.cuh: sed_resample.cu shares it.
__device__ __forceinline__ float load_sample_global(const float* p) { return __ldg(p); }
__device__ __forceinline__ float load_sample_global(const short* p) { return static_cast<float>(__ldg(p)); }
__device__ __forceinline__ void store_raw(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_raw(short* p, float v) { *p = static_cast<short>(v); }

// 10*log10(max(x, amin)) - db_offset (stft.py:726-727) as one MUFU.LG2 and one FMA.  lg2.approx is accurate to 2^-22
// (absolute inside (0.5, 2), relative elsewhere): at most 2.4e-5 dB over the whole range, against a tolerance of
// 1e-4 * max(|dB|, 1).  Values at or below amin return `db_floor`, the float32 value of 10*log10(amin) - db_offset the
// host computed with the reference's own operations (digital silence is exactly -100 dB).
__device__ __forceinline__ float power_to_db(float x, float amin, float db_offset, float db_floor) {
  float l;
  asm("lg2.approx.f32 %0, %1;" : "=f"(l) : "f"(x));
  return x > amin ? fmaf(l, 3.010299956639812f, -db_offset) : db_floor;
}

// global -> shared bulk copy (one instruction for a whole segment; completes bytes on an mbarrier)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// One Stockham pass of radix R over N complex points, IN PLACE in the swizzled shared-memory buffer of one warp:
// every lane first pulls the inputs of all its butterflies into registers, the warp synchronises, then the
// autosorted outputs are written back.  Element indices, per lane (j = lane + 32 q is the butterfly, i = q + BPL r):
//   inputs   j + r * NB                      = lane + 32 i                     -> eaddr(ld_base, 32 i)
//   outputs  (j / Ns) Ns R + j % Ns + r Ns   = j0(lane) + (r Ns + 32 R q)      -> eaddr(st_base, r Ns + 32 R q)
// with ld_base / st_base the byte addresses of pidx(lane) / pidx(j0(lane)) (PassAddr).
// FIRST: inputs come from the windowed frame pair instead (re = frame a, im = frame b), staged as raw input samples.
// LAST (Ns >= 32): nothing is written back -- the outputs stay in registers as X[lane + 32 i] = v[i % BPL][i / BPL]
// for the power split.
template <int N, int R, int Ns, bool FIRST, bool LAST, typename TIn>
__device__ __forceinline__ void fft_pass(float2 (&v)[N / R / 32][R], uint32_t ld_base, uint32_t st_base,
                                         const PassTw<N, R, Ns>& tws, const float2* __restrict__ s_tw,
                                         const TIn* __restrict__ seg_a, const TIn* __restrict__ seg_b,
                                         const float* __restrict__ s_win, int lane) {
  constexpr int NB = N / R;
  constexpr int BPL = NB / 32;  // butterflies per lane
  static_assert(!LAST || Ns >= 32, "the last pass must leave X[lane + 32 i] in the lane");
  static_assert(LAST || Ns <= 32, "store addressing: j / Ns must split into lane / Ns + q * 32 / Ns");
#pragma unroll
  for (int q = 0; q < BPL; ++q) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = q + BPL * r;
      if (FIRST) {
        const int idx = lane + 32 * i;
        const float w = s_win[idx];
        v[q][r] = make_float2(w * load_sample(seg_a + idx), w * load_sample(seg_b + idx));
      } else {
        v[q][r] = lds_f2(eaddr(ld_base, 32 * i));
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int q = 0; q < BPL; ++q) {
    if (Ns > 1) {
      const int k = (lane + 32 * q) % Ns;
#pragma unroll
      for (int r = 1; r < R; ++r) {
        const float2 w = PassTw<N, R, Ns>::IN_REGS ? tws.t[PassTw<N, R, Ns>::NK == 1 ? 0 : q][r - 1]
                                                   : s_tw[r * k * PassTw<N, R, Ns>::TSTRIDE];
        v[q][r] = cmul(v[q][r], w);
      }
    }
    butterfly<R>(v[q]);
    if (!LAST) {
#pragma unroll
      for (int r = 0; r < R; ++r) sts_f2(eaddr(st_base, r * Ns + 32 * R * q), v[q][r]);
    }
  }
  if (!LAST) __syncwarp();
}

// byte address of pidx(j0(lane)) for the stores of a pass (see fft_pass); buf_addr is 128-byte aligned
template <int R, int Ns>
__device__ __forceinline__ uint32_t pass_store_base(uint32_t buf_addr, int lane) {
  const int j0 = (lane / Ns) * Ns * R + lane % Ns;
  return buf_addr + 8u * static_cast<uint32_t>(pidx(j0));
}

// Radix schedule of the N-point transform, three passes each: 256 = 4*8*8, 512 = 8*8*8, 1024 = 8*8*16 (the earlier
// 2*8*8*8 cost a fourth trip through shared memory for a radix-2 pass).
template <int N> struct Sched;
template <> struct Sched<256> { static constexpr int R0 = 4, R1 = 8, R2 = 8; };
template <> struct Sched<512> { static constexpr int R0 = 8, R1 = 8, R2 = 8; };
template <> struct Sched<1024> { static constexpr int R0 = 8, R1 = 8, R2 = 16; };

// Stage the raw waveform segment [q0, q0 + seg_len) of clip b (reflect padding at the clip ends, stft.py:236-237;
// zero beyond total_len, pad_truncate_sequence utils/utilities.py:66-70) into shared memory.  Interior, 16-byte
// aligned segments are ONE bulk copy issued by thread 0 (returns true: the consumer waits on `bar`); edge segments go
// through guarded loads of all threads (returns false: the block barrier in front of the consumer orders them).  The
// caller has passed a block barrier since the last generic-proxy access to `dst`.
template <int NFFT, int FPB, typename TIn>
__device__ __forceinline__ bool stage_segment(TIn* __restrict__ dst, uint64_t* bar, const TIn* __restrict__ wave,
                                              long clip_stride, const long* __restrict__ clip_offset, long total_len,
                                              int L, int hop, int seg_len, int item, int chunks, bool aligned) {
  const int b = item / chunks, c = item - b * chunks;
  const long clip_base = clip_offset ? clip_offset[b] : static_cast<long>(b) * clip_stride;
  aligned = aligned && ((clip_base * static_cast<long>(sizeof(TIn))) & 15) == 0;
  const long q0 = static_cast<long>(c) * FPB * hop - NFFT / 2;
  const TIn* w = wave + clip_base;
  if (aligned && q0 >= 0 && q0 + seg_len <= L && clip_base + q0 + seg_len <= total_len) {
    if (threadIdx.x == 0) {
      const uint32_t bytes = static_cast<uint32_t>(seg_len) * static_cast<uint32_t>(sizeof(TIn));
      fence_proxy_async_smem();  // the buffer's previous readers used the generic proxy
      mbar_expect_tx(bar, bytes);
      bulk_g2s(dst, w + q0, bytes, bar);
    }
    return true;
  }
  // edge segments (first / last chunk of a clip: 2 of ~32 items): four independent loads in flight per thread
  for (int s0 = threadIdx.x; s0 < seg_len; s0 += 4 * blockDim.x) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int s = s0 + u * blockDim.x;
      long i = q0 + s;
      if (i < 0) i = -i;
      if (i >= L) i = 2L * (L - 1) - i;
      v[u] = (s < seg_len && i >= 0 && i < L && clip_base + i < total_len) ? load_sample_global(w + i) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int s = s0 + u * blockDim.x;
      if (s < seg_len) store_raw(dst + s, v[u]);
    }
  }
  return false;
}

// Mel projection schedule, built once per persistent block from the banded matrix (stft.py:709 restricted to the
// non-zero weights).  Band m (bins lo_m .. lo_m + len_m) is cut into ceil(len_m / SEG) segments of SEG consecutive bins;
// segments are numbered band after band, segment s belongs to lane s % 32 of round s / 32.  Per segment: the first bin
// it reads (moved down where lo + SEG would pass the last bin F - 1; the weights move with it) and SEG weights, zero
// where the segment sticks out of its band -- every lane runs the same SEG multiply-adds per round, no divergence, and
// the wide high-frequency bands are spread over several lanes instead of serialising the warp.
//   s_band[m]  = first segment | segments << 16
//   s_seglo[s] = first bin read by segment s          (s < 32 * rounds; unused lanes read bin 0 with zero weights)
//   s_segw[(round * SEG + i) * 32 + lane] = weight of bin s_seglo[s] + i, times 1/4 (the power split of the log-mel
//                                            path leaves 4 |X|^2 in P2; the scale is exact)
// Returns the number of segments, or -1 when they do not fit (SEGS_MAX): the caller then projects one lane per band.
template <int NFFT>
__device__ __forceinline__ int build_mel_schedule(const int* __restrict__ mel_lo, const int* __restrict__ mel_len,
                                                  const int* __restrict__ mel_off, const float* __restrict__ mel_val,
                                                  int n_mels, int* __restrict__ s_band, int* __restrict__ s_seglo,
                                                  int* __restrict__ s_segmj, float* __restrict__ s_segw,
                                                  int* __restrict__ s_total) {
  constexpr int SEG = FrontCfg<NFFT>::SEG, SEGS_MAX = FrontCfg<NFFT>::SEGS_MAX, F = NFFT / 2 + 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {  // exclusive scan of the segment counts, 32 bands at a time
    int carry = 0;
    for (int m0 = 0; m0 < n_mels; m0 += 32) {
      const int m = m0 + lane;
      const int np = (m < n_mels) ? (max(mel_len[m], 0) + SEG - 1) / SEG : 0;
      int incl = np;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
      }
      if (m < n_mels) s_band[m] = (carry + incl - np) | (np << 16);
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) *s_total = carry;
  }
  __syncthreads();
  const int nseg = *s_total;
  if (nseg > SEGS_MAX || nseg >= 65536) return -1;
  const int slots = ((nseg + 31) / 32) * 32;
  for (int s = threadIdx.x; s < slots; s += blockDim.x) s_segmj[s] = -1;
  __syncthreads();
  for (int m = threadIdx.x; m < n_mels; m += blockDim.x) {
    const int first = s_band[m] & 0xffff, np = s_band[m] >> 16;
    for (int j = 0; j < np; ++j) s_segmj[first + j] = m | (j << 16);
  }
  __syncthreads();
  // First bin each segment reads.  A segment that is shorter than SEG may start anywhere between (its last bin + 1 -
  // SEG) and its first bin; the 64-bit reads of a half-warp are conflict-free when their starts differ mod 16, so
  // every lane that shares its residue with a lower lane of its half-warp moves down one bin at a time while it can
  // (the reference's 16 kHz matrix: 91 -> 63 wavefronts per frame pair, 42 without any conflict).
  for (int r = warp; r < slots / 32; r += blockDim.x >> 5) {
    const int s = 32 * r + lane;
    const int mj = s_segmj[s];
    int start = 0, lowest = 0;
    if (mj >= 0) {
      const int m = mj & 0xffff, j = mj >> 16;
      const int lo = mel_lo[m], len = mel_len[m];
      start = min(lo + j * SEG, F - SEG);
      lowest = max(lo + min((j + 1) * SEG, len) - SEG, 0);
    }
    for (int it = 0; it < SEG; ++it) {
      const unsigned peers = __match_any_sync(0xffffffffu, (start & 15) | (lane & 16) | (mj >= 0 ? 0 : 32 + lane));
      const int first = __ffs(peers) - 1;
      const int first_start = __shfl_sync(0xffffffffu, start, first);
      if (lane != first && start != first_start && start > lowest) --start;
    }
    const int anchor = __shfl_sync(0xffffffffu, start, lane & 16);  // unused lanes re-read a neighbour's address
    s_seglo[s] = (mj >= 0) ? start : anchor;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < slots * SEG; e += blockDim.x) {
    const int s = e / SEG, i = e - s * SEG;
    const int mj = s_segmj[s];
    float w = 0.0f;
    if (mj >= 0) {
      const int m = mj & 0xffff, j = mj >> 16;
      const int rel = s_seglo[s] + i - mel_lo[m];  // position of this bin inside the band
      if (rel >= j * SEG && rel < min((j + 1) * SEG, mel_len[m])) w = 0.25f * mel_val[mel_off[m] + rel];
    }
    s_segw[((s >> 5) * SEG + i) * 32 + (s & 31)] = w;
  }
  __syncthreads();
  return nseg;
}

// Bytes of the block's constant tables and FFT buffers (everything in front of the two staging buffers), counted from
// the 128-byte aligned start of the dynamic shared memory; a multiple of 16.
template <int NFFT>
__host__ __device__ constexpr int frontend_fixed_smem(int n_mels, int buf_elems = FrontCfg<NFFT>::WARPS * NFFT,
                                                      int tw_elems = NFFT) {
  return ((8 * (buf_elems + tw_elems) + 4 * NFFT + 4 * FrontCfg<NFFT>::SEGS_MAX * FrontCfg<NFFT>::SEG +
           8 * FrontCfg<NFFT>::SEGS_MAX + 4 * ((n_mels + 1) & ~1) + 8 * n_mels) + 15) & ~15;
}

// mode 0: out = log-mel (+ optional bn0 affine) [B, T, n_mels];  mode 1: out = power spectrogram [B, T, F]
// Clip b starts at wave + b * clip_stride (or wave + clip_offset[b] when a table is given) and is L samples long; samples at or beyond total_len (counted from
// `wave`) read as zero.  clip_stride < L gives overlapping windows of one long recording (predict.py:297-307)
// without materialising them.
template <int NFFT, typename TIn, int MODE>
__global__ void __launch_bounds__(FrontCfg<NFFT>::WARPS * 32, FrontCfg<NFFT>::MIN_BLOCKS)
frontend_kernel(const TIn* __restrict__ wave, long clip_stride, const long* __restrict__ clip_offset, long total_len,
                int B, int L, int T, int hop,
                const float* __restrict__ window, const float2* __restrict__ twiddle,
                const int* __restrict__ mel_lo, const int* __restrict__ mel_len, const int* __restrict__ mel_off,
                const float* __restrict__ mel_val, int n_mels, float amin, float db_offset, int is_log,
                const float* __restrict__ bn_scale, const float* __restrict__ bn_shift, float* __restrict__ out,
                int aligned, int* __restrict__ work_counter) {
  constexpr int WARPS = FrontCfg<NFFT>::WARPS;
  constexpr int FPB = FrontCfg<NFFT>::template fpb<TIn>();
  constexpr int SEG = FrontCfg<NFFT>::SEG, SEGS_MAX = FrontCfg<NFFT>::SEGS_MAX;
  constexpr int NP_UNROLL = FrontCfg<NFFT>::NP_UNROLL;
  constexpr int RU = FrontCfg<NFFT>::ROUNDS_UNROLL;
  constexpr int F = NFFT / 2 + 1;
  constexpr int NS = NFFT / 32, H = NS / 2;  // spectrum values per lane after the last pass; half of them
  const float db_floor = 10.0f * log10f(amin) - db_offset;  // once per thread: the value every clamped bin takes
  constexpr int R0 = Sched<NFFT>::R0, R1 = Sched<NFFT>::R1, R2 = Sched<NFFT>::R2;
  static_assert(R0 * R1 * R2 == NFFT, "radix schedule");
  constexpr int NS1 = R0, NS2 = R0 * R1;  // strides of the second and third pass
  constexpr int BPL2 = NFFT / R2 / 32;
  static_assert(F + SEGS_MAX <= NFFT, "segment sums must fit behind the power spectrum");
  extern __shared__ float4 smem_f4[];
  const int seg_len = (FPB - 1) * hop + NFFT;
  const int seg_bytes = ((seg_len * static_cast<int>(sizeof(TIn)) + 15) & ~15);
  uint8_t* sp = reinterpret_cast<uint8_t*>(smem_f4);
  sp += (128u - (smem_u32(sp) & 127u)) & 127u;                        // the swizzled addressing XORs address bits 3..6
  float2* s_buf = reinterpret_cast<float2*>(sp);                      // [WARPS][NFFT]
  float2* s_tw = s_buf + WARPS * NFFT;                                // [NFFT]
  float* s_win = reinterpret_cast<float*>(s_tw + NFFT);               // [NFFT]
  float* s_segw = s_win + NFFT;                                       // [SEGS_MAX / 32 * SEG][32] segment weights
  int* s_seglo = reinterpret_cast<int*>(s_segw + SEGS_MAX * SEG);     // [SEGS_MAX]
  int* s_segmj = s_seglo + SEGS_MAX;                                  // [SEGS_MAX] (band, piece) while building
  int* s_band = s_segmj + SEGS_MAX;                                   // [n_mels] first segment | segments << 16
  float2* s_bn = reinterpret_cast<float2*>(s_band + ((n_mels + 1) & ~1));  // [n_mels] bn0 (scale, shift)
  TIn* s_stage0 = reinterpret_cast<TIn*>(sp + frontend_fixed_smem<NFFT>(n_mels));  // 16-byte aligned (bulk copy)
  TIn* s_stage1 = reinterpret_cast<TIn*>(reinterpret_cast<uint8_t*>(s_stage0) + seg_bytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunks = (T + FPB - 1) / FPB;
  const int items = B * chunks;
  __shared__ int s_next[2];
  __shared__ int s_total;
  __shared__ __align__(8) uint64_t s_bar[2];  // one per staging buffer: bytes of the bulk copy in flight
  if (threadIdx.x == 0) {
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  int item = blockIdx.x;
  bool cur_bulk = false;  // block-uniform: this item's segment arrives through s_bar[sel]
  if (item < items)
    cur_bulk = stage_segment<NFFT, FPB, TIn>(s_stage0, &s_bar[0], wave, clip_stride, clip_offset, total_len, L, hop, seg_len,
                                        item, chunks, aligned != 0);
  for (int i = threadIdx.x; i < NFFT; i += blockDim.x) {
    s_win[i] = window[i];
    s_tw[i] = twiddle[i];
  }
  int nseg = -1;
  if (MODE == 0) {
    for (int i = threadIdx.x; i < n_mels; i += blockDim.x)
      s_bn[i] = bn_scale != nullptr ? make_float2(bn_scale[i], bn_shift[i]) : make_float2(1.0f, 0.0f);
    nseg = build_mel_schedule<NFFT>(mel_lo, mel_len, mel_off, mel_val, n_mels, s_band, s_seglo, s_segmj, s_segw,
                                    &s_total);
  }
  const int rounds = (nseg + 31) >> 5;  // 0 when the schedule does not fit: one lane per band, weights from global

  // per-lane constants of the transform, loaded once per persistent warp
  PassTw<NFFT, R0, 1> tw0;  // first pass: no twiddles
  PassTw<NFFT, R1, NS1> tw1;
  PassTw<NFFT, R2, NS2> tw2;
  tw1.init(twiddle, lane);
  tw2.init(twiddle, lane);

  float2* buf = s_buf + warp * NFFT;
  const uint32_t buf_addr = smem_u32(buf);
  const uint32_t ld_base = buf_addr + 8u * static_cast<uint32_t>(pidx(lane));
  const uint32_t st_base0 = pass_store_base<R0, 1>(buf_addr, lane);
  const uint32_t st_base1 = pass_store_base<R1, NS1>(buf_addr, lane);
  float2* P2 = buf;             // P2[k] = (|A_k|^2, |B_k|^2): both frames of the pair side by side, k < F
  float2* part = buf + F;       // segment sums of the mel projection
  const int src_lane = (32 - lane) & 31;

  // Work items are claimed dynamically (block b starts with item b, every further item comes from an atomic counter):
  // a block that starts late -- its SM was still busy with another stream's kernel -- simply claims fewer items, so
  // the launch ends when the work is done, not when the slowest static share is.
  int sel = 0;
  uint32_t phase = 0;  // bit s: parity of s_bar[s]'s next completion
  bool nxt_bulk = false;
  for (int nxt = 0; item < items; item = nxt, sel ^= 1, cur_bulk = nxt_bulk) {
    if (threadIdx.x == 0) s_next[sel] = static_cast<int>(gridDim.x) + atomicAdd(work_counter, 1);
    __syncthreads();  // the claimed item and an edge segment's stores are visible; every warp has finished the previous item
    nxt = s_next[sel];
    nxt_bulk = false;
    if (nxt < items)
      nxt_bulk = stage_segment<NFFT, FPB, TIn>(sel ? s_stage0 : s_stage1, &s_bar[sel ^ 1], wave, clip_stride, clip_offset,
                                          total_len, L, hop, seg_len, nxt, chunks, aligned != 0);
    if (cur_bulk) {
      mbar_wait(&s_bar[sel], (phase >> sel) & 1u);
      phase ^= 1u << sel;
    }
    const TIn* s_seg = sel ? s_stage1 : s_stage0;
    const int b = item / chunks;
    const int f_base = (item - b * chunks) * FPB;

    for (int pair = warp; pair < FPB / 2; pair += WARPS) {
      const int fa = f_base + 2 * pair;
      if (fa >= T) break;
      const TIn* seg_a = s_seg + (2 * pair) * hop;
      const TIn* seg_b = seg_a + hop;

      // ---- 2 real frames -> 1 complex FFT of size NFFT (Stockham autosort); the last pass stays in registers ----
      {
        float2 v0[NFFT / R0 / 32][R0];
        fft_pass<NFFT, R0, 1, true, false, TIn>(v0, ld_base, st_base0, tw0, s_tw, seg_a, seg_b, s_win, lane);
      }
      {
        float2 v1[NFFT / R1 / 32][R1];
        fft_pass<NFFT, R1, NS1, false, false, TIn>(v1, ld_base, st_base1, tw1, s_tw, seg_a, seg_b, s_win, lane);
      }
      float2 X[BPL2][R2];  // X[lane + 32 i] = X[i % BPL2][i / BPL2]
      fft_pass<NFFT, R2, NS2, false, true, TIn>(X, ld_base, 0u, tw2, s_tw, seg_a, seg_b, s_win, lane);

      // ---- split the two real spectra and take the power (stft.py:663).  Bin k = lane + 32 i (i < H) needs
      //      Z[N - k]: slot NS - 1 - i of lane 32 - lane (one shuffle per component); lane 0 pairs with itself
      //      (slot (NS - i) % NS).  The warp has passed the barrier behind the last pass's reads, so P2 can overwrite
      //      the buffer. ----
#pragma unroll
      for (int i = 0; i < H; ++i) {
        const float2 zk = X[i % BPL2][i / BPL2];
        const float2 up = X[(NS - 1 - i) % BPL2][(NS - 1 - i) / BPL2];
        float2 zn = make_float2(__shfl_sync(0xffffffffu, up.x, src_lane), __shfl_sync(0xffffffffu, up.y, src_lane));
        if (lane == 0) zn = X[((NS - i) % NS) % BPL2][((NS - i) % NS) / BPL2];
        // A = (zk + conj(zn)) / 2, B = (zk - conj(zn)) / 2i; the halves are folded into one exact scale by 1/4
        const float ar = zk.x + zn.x, ai = zk.y - zn.y;
        const float br = zk.y + zn.y, bi = zn.x - zk.x;
        // (the log-mel path keeps 4 |.|^2 and carries the 1/4 in its mel weights)
        constexpr float kQ = (MODE == 0) ? 1.0f : 0.25f;
        P2[lane + 32 * i] = make_float2(kQ * fmaf(ai, ai, ar * ar), kQ * fmaf(bi, bi, br * br));
      }
      if (lane == 0) {  // Nyquist bin N / 2 = 32 H: its own partner, so A = re, B = im
        constexpr float kN = (MODE == 0) ? 4.0f : 1.0f;
        const float2 z = X[H % BPL2][H / BPL2];
        P2[NFFT / 2] = make_float2(kN * z.x * z.x, kN * z.y * z.y);
      }
      __syncwarp();

      const bool has_b = fa + 1 < T;
      if (MODE == 1) {
        float* o = out + (static_cast<size_t>(b) * T + fa) * F;
        for (int k = lane; k < F; k += 32) {
          const float2 p = P2[k];
          o[k] = p.x;
          if (has_b) o[F + k] = p.y;
        }
      } else {
        float* o = out + (static_cast<size_t>(b) * T + fa) * n_mels;
        // ---- mel projection, one lane per segment: SEG multiply-adds per round for both frames of the pair ----
        if (rounds == RU) {  // the presets: every round unrolled, all loads in flight, RU independent chains per frame
          float a0[RU], b0[RU];
          const float2* Pm[RU];
#pragma unroll
          for (int r = 0; r < RU; ++r) {
            Pm[r] = P2 + s_seglo[32 * r + lane];
            a0[r] = 0.0f;
            b0[r] = 0.0f;
          }
#pragma unroll
          for (int i = 0; i < SEG; ++i) {
#pragma unroll
            for (int r = 0; r < RU; ++r) {
              const float2 p = Pm[r][i];
              const float w = s_segw[(r * SEG + i) * 32 + lane];
              a0[r] = fmaf(p.x, w, a0[r]);
              b0[r] = fmaf(p.y, w, b0[r]);
            }
          }
#pragma unroll
          for (int r = 0; r < RU; ++r) part[32 * r + lane] = make_float2(a0[r], b0[r]);
        } else {
          for (int r = 0; r < rounds; ++r) {
            const float2* Pm = P2 + s_seglo[32 * r + lane];
            const float* wr = s_segw + r * (SEG * 32) + lane;
            float a0 = 0.0f, b0 = 0.0f;
#pragma unroll
            for (int i = 0; i < SEG; ++i) {
              const float2 p = Pm[i];
              const float w = wr[32 * i];
              a0 = fmaf(p.x, w, a0);
              b0 = fmaf(p.y, w, b0);
            }
            part[32 * r + lane] = make_float2(a0, b0);
          }
        }
        __syncwarp();
        for (int m = lane; m < n_mels; m += 32) {
          float ya = 0.0f, yb = 0.0f;
          if (rounds > 0) {
            const int first = s_band[m] & 0xffff, np = s_band[m] >> 16;
            const float2* pm = part + first;
            // ascending segments: the summation order is fixed.  The first NP_UNROLL are predicated (no loop for the
            // reference's presets), wider bands continue in a loop.
#pragma unroll
            for (int j = 0; j < NP_UNROLL; ++j) {
              if (j < np) {
                const float2 t = pm[j];
                ya += t.x;
                yb += t.y;
              }
            }
            for (int j = NP_UNROLL; j < np; ++j) {
              const float2 t = pm[j];
              ya += t.x;
              yb += t.y;
            }
          } else {
            const float2* Pm = P2 + mel_lo[m];
            const float* mv = mel_val + mel_off[m];
            const int len = mel_len[m];
            for (int i = 0; i < len; ++i) {
              const float2 p = Pm[i];
              const float w = 0.25f * __ldg(mv + i);
              ya = fmaf(p.x, w, ya);
              yb = fmaf(p.y, w, yb);
            }
          }
          if (is_log) {  // stft.py:726-727
            ya = power_to_db(ya, amin, db_offset, db_floor);
            yb = power_to_db(yb, amin, db_offset, db_floor);
          }
          const float2 sc = s_bn[m];  // models.py:642-644 (identity when no bn0 is fused)
          ya = fmaf(ya, sc.x, sc.y);
          yb = fmaf(yb, sc.x, sc.y);
          o[m] = ya;
          if (has_b) o[n_mels + m] = yb;
        }
      }
      __syncwarp();
    }
  }
}

// =====================================================================================================================
// Two-pass kernel (serves n_fft 1024; generic over 256 / 512 / 1024, see SED_FE_TWO_PASS): ONE trip of the spectrum
// through shared memory instead of two.
//
// N = RA * 32 (RA = 8 / 16 / 32).  With n = n2 + 32 n1 and k = k1 + RA k2:
//     X[k1 + RA k2] = sum_n2 W32^(n2 k2) { W_N^(n2 k1) sum_n1 x[n2 + 32 n1] W_RA^(n1 k1) }
// Pass A: lane n2 takes the RA-point DFT over n1 (inputs lane + 32 n1: unit stride across the warp) and multiplies by its
// own twiddles W_N^(lane k1) (RA - 1 register pairs).  Pass B: a 32-point DFT over n2 without any twiddle -- one per
// (transform, k1), so a warp carries T = 32 / RA transforms (2 T real frames) at a time and lane f RA + k1 owns butterfly
// k1 of transform f.  In between, value (f, k1, n2) sits at element 32 (f RA + k1) + (n2 ^ ((f RA + k1) & 15)): row =
// the pass-B lane, the XOR makes both the stores of pass A (fixed row, 32 lanes) and the loads of pass B (fixed n2, 16
// rows per half-warp) conflict-free.  Pass B leaves X_f[k1 + RA k2], k2 = 0..31, in the lane; bin k <= N/2 needs
// Z[N - k] = slot 31 - k2 of lane (f, RA - k1) (k1 = 0: the lane itself, slot (32 - k2) % 32) -- one shuffle per
// component as in the three-pass kernel.  Per frame pair this costs 64 shared-memory wavefronts for the transform
// instead of 128, and the window taps and mel weights are loaded once for T transforms.
template <int NFFT>
struct Front2Cfg {
  static constexpr int RA = NFFT / 32;        // radix of pass A
  static constexpr int T = 32 / RA;           // transforms (frame pairs) per warp and iteration
  // 8 KB of buffer per warp.  1024: 2 blocks of 6 warps per SM, pass-A twiddles in registers (168 registers); 256 / 512:
  // the twiddles are read from a lane-major shared-memory table right before they are used (TW_SMEM), which keeps the
  // kernel inside a 128-register budget
  static constexpr int WARPS = (NFFT == 1024) ? SED_FE_WARPS2_1024 : SED_FE_WARPS2;
  static constexpr int MIN_BLOCKS = (NFFT == 1024) ? SED_FE_BLOCKS2_1024 : SED_FE_BLOCKS2;
  static constexpr bool TW_SMEM = (NFFT != 1024);
  static constexpr int BUF = 1024;            // complex elements per warp: T transforms of NFFT points
  static constexpr int GROUP = 2 * T;         // frames per warp and iteration
  template <typename TIn>
  static constexpr int fpb() { return WARPS * GROUP * (sizeof(TIn) == 2 ? 2 : 1); }
  // transform t keeps its power spectrum (and the segment sums behind it) in its own NFFT elements of the buffer; at
  // RA = 8 two transforms share a half-warp, so odd ones start 8 elements later (conflict-free P2 stores)
  static constexpr int p2_base(int t) { return t * NFFT + ((RA == 8) ? 8 * (t & 1) : 0); }
};

template <int NFFT, typename TIn, int MODE>
__global__ void __launch_bounds__(Front2Cfg<NFFT>::WARPS * 32, Front2Cfg<NFFT>::MIN_BLOCKS)
frontend2_kernel(const TIn* __restrict__ wave, long clip_stride, const long* __restrict__ clip_offset, long total_len,
                 int B, int L, int T, int hop,
                 const float* __restrict__ window, const float2* __restrict__ twiddle,
                 const int* __restrict__ mel_lo, const int* __restrict__ mel_len, const int* __restrict__ mel_off,
                 const float* __restrict__ mel_val, int n_mels, float amin, float db_offset, int is_log,
                 const float* __restrict__ bn_scale, const float* __restrict__ bn_shift, float* __restrict__ out,
                 int aligned, int* __restrict__ work_counter) {
  // Shared-memory carve-up, block start-up, work-item loop and the mel / dB / bn0 epilogue run parallel to
  // frontend_kernel line by line (there for one transform per warp, here for NT); only the transform differs.
  using C2 = Front2Cfg<NFFT>;
  constexpr int WARPS = C2::WARPS, RA = C2::RA, NT = C2::T, GROUP = C2::GROUP, BUF = C2::BUF;
  constexpr int FPB = C2::template fpb<TIn>();
  constexpr int SEG = FrontCfg<NFFT>::SEG, SEGS_MAX = FrontCfg<NFFT>::SEGS_MAX;
  constexpr int NP_UNROLL = FrontCfg<NFFT>::NP_UNROLL;
  constexpr int RU = FrontCfg<NFFT>::ROUNDS_UNROLL;
  constexpr int F = NFFT / 2 + 1;
  static_assert(RA * 32 == NFFT && NT * NFFT == BUF, "two-pass geometry");
  static_assert(C2::p2_base(NT - 1) + F + SEGS_MAX <= NT * NFFT, "power spectrum + segment sums fit the transform's part");
  const float db_floor = 10.0f * log10f(amin) - db_offset;
  extern __shared__ float4 smem_f4[];
  const int seg_len = (FPB - 1) * hop + NFFT;
  const int seg_bytes = ((seg_len * static_cast<int>(sizeof(TIn)) + 15) & ~15);
  uint8_t* sp = reinterpret_cast<uint8_t*>(smem_f4);
  sp += (128u - (smem_u32(sp) & 127u)) & 127u;
  float2* s_buf = reinterpret_cast<float2*>(sp);                      // [WARPS][BUF]
  constexpr int TW_ELEMS = C2::TW_SMEM ? NFFT : 0;                    // lane-major pass-A twiddles (TW_SMEM only)
  float2* s_tw = s_buf + WARPS * BUF;
  float* s_win = reinterpret_cast<float*>(s_tw + TW_ELEMS);           // [NFFT]
  float* s_segw = s_win + NFFT;
  int* s_seglo = reinterpret_cast<int*>(s_segw + SEGS_MAX * SEG);
  int* s_segmj = s_seglo + SEGS_MAX;
  int* s_band = s_segmj + SEGS_MAX;
  float2* s_bn = reinterpret_cast<float2*>(s_band + ((n_mels + 1) & ~1));
  TIn* s_stage0 = reinterpret_cast<TIn*>(sp + frontend_fixed_smem<NFFT>(n_mels, WARPS * BUF, TW_ELEMS));
  TIn* s_stage1 = reinterpret_cast<TIn*>(reinterpret_cast<uint8_t*>(s_stage0) + seg_bytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunks = (T + FPB - 1) / FPB;
  const int items = B * chunks;
  __shared__ int s_next[2];
  __shared__ int s_total;
  __shared__ __align__(8) uint64_t s_bar[2];
  if (threadIdx.x == 0) {
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  int item = blockIdx.x;
  bool cur_bulk = false;
  if (item < items)
    cur_bulk = stage_segment<NFFT, FPB, TIn>(s_stage0, &s_bar[0], wave, clip_stride, clip_offset, total_len, L, hop,
                                             seg_len, item, chunks, aligned != 0);
  for (int i = threadIdx.x; i < NFFT; i += blockDim.x) s_win[i] = window[i];
  int nseg = -1;
  if (MODE == 0) {
    for (int i = threadIdx.x; i < n_mels; i += blockDim.x)
      s_bn[i] = bn_scale != nullptr ? make_float2(bn_scale[i], bn_shift[i]) : make_float2(1.0f, 0.0f);
    nseg = build_mel_schedule<NFFT>(mel_lo, mel_len, mel_off, mel_val, n_mels, s_band, s_seglo, s_segmj, s_segw,
                                    &s_total);
  }
  const int rounds = (nseg + 31) >> 5;

  // pass-A twiddles of this lane: W_N^(lane k1), k1 = 1 .. RA - 1
  // (TW_SMEM: s_tw[(k1 - 1) * 32 + lane], filled here; otherwise registers)
  float2 twa[C2::TW_SMEM ? 1 : RA - 1];
  if (C2::TW_SMEM) {
    for (int i = threadIdx.x; i < (RA - 1) * 32; i += blockDim.x)
      s_tw[i] = twiddle[((i & 31) * ((i >> 5) + 1)) & (NFFT - 1)];
  } else {
#pragma unroll
    for (int k1 = 1; k1 < RA; ++k1) twa[k1 - 1] = twiddle[(lane * k1) & (NFFT - 1)];
  }

  float2* buf = s_buf + warp * BUF;
  const uint32_t buf_addr = smem_u32(buf);
  const uint32_t st_base = buf_addr + 8u * static_cast<uint32_t>(lane);                    // pass A: element n2 = lane of a row
  const uint32_t ld_base = buf_addr + 256u * static_cast<uint32_t>(lane) + 8u * static_cast<uint32_t>(lane & 15);  // pass B: own row
  const int k1b = lane & (RA - 1), tb = lane / RA;                                         // pass-B role of this lane
  const int src_lane = (lane & ~(RA - 1)) | ((RA - k1b) & (RA - 1));
  float2* P2own = buf + C2::p2_base(0) + tb * NFFT + ((RA == 8) ? 8 * (tb & 1) : 0) + k1b;  // + RA k2

  int sel = 0;
  uint32_t phase = 0;
  bool nxt_bulk = false;
  for (int nxt = 0; item < items; item = nxt, sel ^= 1, cur_bulk = nxt_bulk) {
    if (threadIdx.x == 0) s_next[sel] = static_cast<int>(gridDim.x) + atomicAdd(work_counter, 1);
    __syncthreads();
    nxt = s_next[sel];
    nxt_bulk = false;
    if (nxt < items)
      nxt_bulk = stage_segment<NFFT, FPB, TIn>(sel ? s_stage0 : s_stage1, &s_bar[sel ^ 1], wave, clip_stride,
                                               clip_offset, total_len, L, hop, seg_len, nxt, chunks, aligned != 0);
    if (cur_bulk) {
      mbar_wait(&s_bar[sel], (phase >> sel) & 1u);
      phase ^= 1u << sel;
    }
    const TIn* s_seg = sel ? s_stage1 : s_stage0;
    const int b = item / chunks;
    const int f_base = (item - b * chunks) * FPB;

    for (int grp = warp; grp < FPB / GROUP; grp += WARPS) {
      const int fa0 = f_base + GROUP * grp;  // first frame of this warp's 2 T frames
      if (fa0 >= T) break;

      // ---- pass A: per transform the RA-point DFT over n1 of the windowed frame pair, twiddle, store to row (t, k1) ----
      {
        float wv[RA];
#pragma unroll
        for (int n1 = 0; n1 < RA; ++n1) wv[n1] = s_win[lane + 32 * n1];
#pragma unroll
        for (int t = 0; t < NT; ++t) {
          const TIn* seg_a = s_seg + (GROUP * grp + 2 * t) * hop + lane;
          const TIn* seg_b = seg_a + hop;
          float2 v[RA];
#pragma unroll
          for (int n1 = 0; n1 < RA; ++n1)
            v[n1] = make_float2(wv[n1] * load_sample(seg_a + 32 * n1), wv[n1] * load_sample(seg_b + 32 * n1));
          butterfly<RA>(v);
#pragma unroll
          for (int k1 = 0; k1 < RA; ++k1) {
            const int row = t * RA + k1;
            const float2 y = (k1 == 0) ? v[0] : cmul(v[k1], C2::TW_SMEM ? s_tw[(k1 - 1) * 32 + lane] : twa[k1 - 1]);
            sts_f2((st_base ^ static_cast<uint32_t>(8 * (row & 15))) + static_cast<uint32_t>(256 * row), y);
          }
        }
      }
      __syncwarp();

      // ---- pass B: 32-point DFT over n2 of this lane's row ----
      float2 X[32];
#pragma unroll
      for (int n2 = 0; n2 < 32; ++n2)
        X[n2] = lds_f2((ld_base ^ static_cast<uint32_t>(8 * (n2 & 15))) + static_cast<uint32_t>(8 * (n2 & 16)));
      __syncwarp();  // every row has been read: the buffer can take the power spectra
      butterfly<32>(X);

      // ---- split the two real spectra and take the power (stft.py:663): bin k = k1 + RA k2, k2 < 16 ----
#pragma unroll
      for (int k2 = 0; k2 < 16; ++k2) {
        const float2 zk = X[k2];
        const float2 up = X[31 - k2];
        float2 zn = make_float2(__shfl_sync(0xffffffffu, up.x, src_lane), __shfl_sync(0xffffffffu, up.y, src_lane));
        if (k1b == 0) zn = X[(32 - k2) & 31];
        const float ar = zk.x + zn.x, ai = zk.y - zn.y;
        const float br = zk.y + zn.y, bi = zn.x - zk.x;
        constexpr float kQ = (MODE == 0) ? 1.0f : 0.25f;  // the log-mel path carries the 1/4 in its mel weights
        P2own[RA * k2] = make_float2(kQ * fmaf(ai, ai, ar * ar), kQ * fmaf(bi, bi, br * br));
      }
      if (k1b == 0) {  // Nyquist bin N / 2 = RA * 16
        constexpr float kN = (MODE == 0) ? 4.0f : 1.0f;
        const float2 z = X[16];
        P2own[RA * 16] = make_float2(kN * z.x * z.x, kN * z.y * z.y);
      }
      __syncwarp();

      if (MODE == 1) {
#pragma unroll
        for (int t = 0; t < NT; ++t) {
          const int fa = fa0 + 2 * t;
          if (fa >= T) break;
          const float2* P2 = buf + C2::p2_base(t);
          float* o = out + (static_cast<size_t>(b) * T + fa) * F;
          for (int k = lane; k < F; k += 32) {
            const float2 p = P2[k];
            o[k] = p.x;
            if (fa + 1 < T) o[F + k] = p.y;
          }
        }
      } else {
        // ---- mel projection, one lane per segment; seglo and weights are loaded once for the T transforms ----
        if (rounds == RU) {
          float a0[RU][NT], b0[RU][NT];
          int slo[RU];
#pragma unroll
          for (int r = 0; r < RU; ++r) {
            slo[r] = s_seglo[32 * r + lane];
#pragma unroll
            for (int t = 0; t < NT; ++t) a0[r][t] = b0[r][t] = 0.0f;
          }
#pragma unroll
          for (int i = 0; i < SEG; ++i) {
#pragma unroll
            for (int r = 0; r < RU; ++r) {
              const float w = s_segw[(r * SEG + i) * 32 + lane];
#pragma unroll
              for (int t = 0; t < NT; ++t) {
                const float2 p = buf[C2::p2_base(t) + slo[r] + i];
                a0[r][t] = fmaf(p.x, w, a0[r][t]);
                b0[r][t] = fmaf(p.y, w, b0[r][t]);
              }
            }
          }
#pragma unroll
          for (int r = 0; r < RU; ++r)
#pragma unroll
            for (int t = 0; t < NT; ++t) buf[C2::p2_base(t) + F + 32 * r + lane] = make_float2(a0[r][t], b0[r][t]);
        } else {
          for (int r = 0; r < rounds; ++r) {
            const int slo = s_seglo[32 * r + lane];
            const float* wr = s_segw + r * (SEG * 32) + lane;
            float a0[NT], b0[NT];
#pragma unroll
            for (int t = 0; t < NT; ++t) a0[t] = b0[t] = 0.0f;
#pragma unroll
            for (int i = 0; i < SEG; ++i) {
              const float w = wr[32 * i];
#pragma unroll
              for (int t = 0; t < NT; ++t) {
                const float2 p = buf[C2::p2_base(t) + slo + i];
                a0[t] = fmaf(p.x, w, a0[t]);
                b0[t] = fmaf(p.y, w, b0[t]);
              }
            }
#pragma unroll
            for (int t = 0; t < NT; ++t) buf[C2::p2_base(t) + F + 32 * r + lane] = make_float2(a0[t], b0[t]);
          }
        }
        __syncwarp();
        for (int m = lane; m < n_mels; m += 32) {
          int first = 0, np = 0;
          if (rounds > 0) {
            first = s_band[m] & 0xffff;
            np = s_band[m] >> 16;
          }
          const float2 sc = s_bn[m];  // models.py:642-644 (identity when no bn0 is fused)
#pragma unroll
          for (int t = 0; t < NT; ++t) {
            const int fa = fa0 + 2 * t;
            if (fa >= T) break;
            float ya = 0.0f, yb = 0.0f;
            if (rounds > 0) {
              const float2* pm = buf + C2::p2_base(t) + F + first;
              // ascending segments: the summation order is fixed
#pragma unroll
              for (int j = 0; j < NP_UNROLL; ++j) {
                if (j < np) {
                  const float2 s = pm[j];
                  ya += s.x;
                  yb += s.y;
                }
              }
              for (int j = NP_UNROLL; j < np; ++j) {
                const float2 s = pm[j];
                ya += s.x;
                yb += s.y;
              }
            } else {
              const float2* Pm = buf + C2::p2_base(t) + mel_lo[m];
              const float* mv = mel_val + mel_off[m];
              const int len = mel_len[m];
              for (int i = 0; i < len; ++i) {
                const float2 p = Pm[i];
                const float w = 0.25f * __ldg(mv + i);
                ya = fmaf(p.x, w, ya);
                yb = fmaf(p.y, w, yb);
              }
            }
            if (is_log) {  // stft.py:726-727
              ya = power_to_db(ya, amin, db_offset, db_floor);
              yb = power_to_db(yb, amin, db_offset, db_floor);
            }
            ya = fmaf(ya, sc.x, sc.y);
            yb = fmaf(yb, sc.x, sc.y);
            float* o = out + (static_cast<size_t>(b) * T + fa) * n_mels;
            o[m] = ya;
            if (fa + 1 < T) o[n_mels + m] = yb;
          }
        }
      }
      __syncwarp();
    }
  }
}

// Standalone LogmelFilterBank.forward (stft.py:698-718): rows [R, F] -> [R, n_mels]
__global__ void logmel_rows_kernel(const float* __restrict__ spec, long rows, int F, const int* __restrict__ mel_lo,
                                   const int* __restrict__ mel_len, const int* __restrict__ mel_off,
                                   const float* __restrict__ mel_val, int n_mels, float amin, float db_offset,
                                   int is_log, float* __restrict__ out) {
  const long gw = (static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= rows) return;
  const float* Pf = spec + gw * F;
  float* o = out + gw * n_mels;
  for (int m = lane; m < n_mels; m += 32) {
    const int lo = mel_lo[m], len = mel_len[m];
    const float* mv = mel_val + mel_off[m];
    float acc = 0.0f;
    for (int i = 0; i < len; ++i) acc = fmaf(__ldg(Pf + lo + i), __ldg(mv + i), acc);
    o[m] = is_log ? 10.0f * log10f(fmaxf(acc, amin)) - db_offset : acc;
  }
}

// claim counters of the launches in flight (one per launch, round robin; zeroed on the launch's stream)
__device__ int g_frontend_work_counters[64];
static std::atomic<unsigned> g_frontend_launch_seq{0};

// Which kernel serves an n_fft.  Measured on one box, ms per 148 clips of 10 s (profiles/r02_frontend_ab_*.log):
//   n_fft 1024: three-pass 0.291, two-pass 0.249 (both one block of 12 warps), two-pass 2 x 6 warps 0.214 -> two-pass
//   n_fft 512 : three-pass 0.134 (2 x 8 warps) / 0.129 (4 x 4 warps); two-pass 0.140 (1 x 12 warps, twiddles in
//               registers), 0.141 (1 x 16 warps, twiddles in shared memory), 0.129 (3 x 4 warps)    -> three-pass
//   n_fft 256 : three-pass 0.089, two-pass 0.087 (int16 0.088 / 0.100)                             -> three-pass
// At 512 the two-pass kernel executes 7 % fewer instructions and 19 % fewer shared-memory wavefronts than the
// three-pass one (profiles/r02_ncu_full_frontend_two_pass_512.json) and only draws level with it: at 12 warps per SM it
// has a quarter less latency hiding than the three-pass kernel's 16.
// The two-pass kernel needs 8 KB of buffer per warp; where its shared memory does not fit (large hop) the three-pass
// kernel takes over.  -DSED_FE_TWO_PASS(N)=1 builds a library that uses the two-pass kernel at every size.
#ifndef SED_FE_TWO_PASS
#define SED_FE_TWO_PASS(NFFT) ((NFFT) == 1024)
#endif
template <int NFFT, typename TIn, int MODE, bool TWO_PASS>
struct FrontKernel {
  static auto get() { return frontend_kernel<NFFT, TIn, MODE>; }
};
template <int NFFT, typename TIn, int MODE>
struct FrontKernel<NFFT, TIn, MODE, true> {
  static auto get() { return frontend2_kernel<NFFT, TIn, MODE>; }
};

template <int NFFT, typename TIn, int MODE, bool TWO_PASS>
static int launch_frontend_v(const FrontendArgs& a, cudaStream_t stream) {
  constexpr int WARPS = TWO_PASS ? Front2Cfg<NFFT>::WARPS : FrontCfg<NFFT>::WARPS;
  constexpr int FPB = TWO_PASS ? Front2Cfg<NFFT>::template fpb<TIn>() : FrontCfg<NFFT>::template fpb<TIn>();
  constexpr int BUF_ELEMS = TWO_PASS ? Front2Cfg<NFFT>::WARPS * Front2Cfg<NFFT>::BUF : FrontCfg<NFFT>::WARPS * NFFT;
  auto kernel = FrontKernel<NFFT, TIn, MODE, TWO_PASS>::get();
  const int seg_len = (FPB - 1) * a.hop + NFFT;
  const int seg_bytes = (seg_len * static_cast<int>(sizeof(TIn)) + 15) & ~15;
  constexpr int TW_ELEMS = (TWO_PASS && !Front2Cfg<NFFT>::TW_SMEM) ? 0 : NFFT;
  const size_t smem = 128 +
                      static_cast<size_t>(frontend_fixed_smem<NFFT>(a.n_mels > 0 ? a.n_mels : 0, BUF_ELEMS, TW_ELEMS)) +
                      2 * static_cast<size_t>(seg_bytes);
  if (smem > 227 * 1024) return SED_ERR_UNSUPPORTED;
  static int sm_count = 0;
  if (sm_count == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count <= 0)
      sm_count = 148;
  }
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return SED_ERR_CUDA;
  int per_sm = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, WARPS * 32, smem) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  const long items = static_cast<long>(a.B) * ((a.T + FPB - 1) / FPB);
  long blocks = static_cast<long>(sm_count) * per_sm;
  if (blocks > items) blocks = items;
  // bulk-copy staging needs 16-byte aligned interior segments
  const size_t es = sizeof(TIn);
  const int aligned = (reinterpret_cast<uintptr_t>(a.wave) % 16 == 0) &&
                      (a.clip_offset != nullptr || (a.clip_stride * es) % 16 == 0) &&
                      ((static_cast<size_t>(FPB) * a.hop * es) % 16 == 0) && ((NFFT / 2 * es) % 16 == 0) &&
                      ((seg_len * es) % 16 == 0);
  int* counters = nullptr;
  if (cudaGetSymbolAddress(reinterpret_cast<void**>(&counters), g_frontend_work_counters) != cudaSuccess)
    return SED_ERR_CUDA;
  int* counter = counters + (g_frontend_launch_seq.fetch_add(1) & 63u);
  if (cudaMemsetAsync(counter, 0, sizeof(int), stream) != cudaSuccess) return SED_ERR_CUDA;
  kernel<<<static_cast<unsigned>(blocks), WARPS * 32, smem, stream>>>(
      reinterpret_cast<const TIn*>(a.wave), a.clip_stride, a.clip_offset, a.total_len, a.B, a.L, a.T, a.hop, a.window,
      reinterpret_cast<const float2*>(a.twiddle), a.mel_lo, a.mel_len, a.mel_off, a.mel_val, a.n_mels, a.amin,
      a.db_offset, a.is_log, a.bn_scale, a.bn_shift, a.out, aligned, counter);
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}

template <int NFFT, typename TIn, int MODE>
static int launch_frontend_t(const FrontendArgs& a, cudaStream_t stream) {
  if (SED_FE_TWO_PASS(NFFT)) {
    const int rc = launch_frontend_v<NFFT, TIn, MODE, true>(a, stream);
    if (rc != SED_ERR_UNSUPPORTED) return rc;
  }
  return launch_frontend_v<NFFT, TIn, MODE, false>(a, stream);
}

template <int NFFT>
static int launch_frontend(const FrontendArgs& a, cudaStream_t stream) {
  if (a.mode == 1)
    return a.wave_dtype == 1 ? launch_frontend_t<NFFT, short, 1>(a, stream) : launch_frontend_t<NFFT, float, 1>(a, stream);
  return a.wave_dtype == 1 ? launch_frontend_t<NFFT, short, 0>(a, stream) : launch_frontend_t<NFFT, float, 0>(a, stream);
}

int frontend_launch(const FrontendArgs& a, cudaStream_t stream) {
  if (a.B <= 0 || a.L <= a.n_fft / 2 || a.hop <= 0 || a.clip_stride <= 0 || a.total_len <= 0) return SED_ERR_BAD_SHAPE;
  if (a.wave_dtype != 0 && a.wave_dtype != 1) return SED_ERR_UNSUPPORTED;
  switch (a.n_fft) {
    case 256: return launch_frontend<256>(a, stream);
    case 512: return launch_frontend<512>(a, stream);
    case 1024: return launch_frontend<1024>(a, stream);
    default: return SED_ERR_UNSUPPORTED;
  }
}

int logmel_rows_launch(const float* spec, long rows, int F, const int* mel_lo, const int* mel_len, const int* mel_off,
                       const float* mel_val, int n_mels, float amin, float db_offset, int is_log, float* out,
                       cudaStream_t stream) {
  if (rows <= 0) return SED_ERR_BAD_SHAPE;
  const int threads = 256;
  const long blocks = (rows * 32 + threads - 1) / threads;
  logmel_rows_kernel<<<(unsigned)blocks, threads, 0, stream>>>(spec, rows, F, mel_lo, mel_len, mel_off, mel_val, n_mels,
                                                               amin, db_offset, is_log, out);
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}

}  // namespace sed
