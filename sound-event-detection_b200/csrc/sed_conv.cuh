// tcgen05 implicit-GEMM 3x3 convolution (+ folded BatchNorm + ReLU + 2x2 avg-pool / freq-mean) and
// the plain GEMM ("linear") used by the temporal blocks, for sm_100a.
//
// Reference semantics: ConvBlock.forward  pytorch/models.py:125-141 (conv 3x3 s1 p1 no bias -> BN(eval)
// -> ReLU, twice, then avg_pool2d), freq-mean models.py:668, nn.Linear inside nn.GRU / MultiHead.
//
// Conv GEMM view: M = output pixels (one 16(H) x 8(W) spatial patch = 128 rows per tile), N = Cout slice,
// K = 9 taps x Cin.  Activations are NHWC 16-bit, weights are [Cout][tap][Cin] 16-bit (K-major).
//
//  * conv_umma2_kernel (the conv layers, CTA pairs): per 64-channel chunk ONE TMA box (64ch x 10w x 18h)
//    brings the haloed patch into a SWIZZLE_128B buffer (180 pixel rows of 128 B, zero-filled outside the
//    image = conv padding).  The nine taps are nine UMMA descriptors into that single buffer: start address
//    + (r*10+s)*128 B, 8-row group stride 1280 B.  A is therefore read from L2 once, not nine times.
//    B is either streamed per (chunk, tap) through a ring, or RESIDENT in shared memory for the whole
//    persistent CTA pair when the Cout slice of the weights fits (weight-stationary).
//  * conv_umma_kernel (the GEMM, single CTA): one (64ch x 128 rows) box of A and one of B per K chunk.
//  * NT (1|2) pixel / row tiles share every B block, accumulators live in TMEM (NT*BN columns per stage).
#pragma once
#include "sed_common.cuh"

namespace sed {

enum : int { EPI_STORE = 0, EPI_POOL = 1, EPI_FREQMEAN = 2, EPI_LINEAR = 3 };

struct ConvParams {
  int NB, H, W;            // images, rows, cols of the (same-size) convolution; W % 8 == 0
  int tiles_h, tiles_w;    // ceil(H/16), W/8
  uint32_t magic_img, magic_w;  // fast_div magics for tiles_h*tiles_w and tiles_w
  int num_tiles;           // conv: NB*tiles_h*tiles_w ; linear: ceil(M/128)
  int cout;                // total output channels (row stride of the output)
  int nslices;             // cout / BN
  const float* scale;      // [cout] folded BN scale   (linear: unused)
  const float* shift;      // [cout] folded BN shift   (linear: bias)
  void* out;               // EPI 0/1/2: 16-bit NHWC ; EPI 3: float [M, ldc]
  void* out2;              // EPI 3: optional 16-bit copy [M, ldc]; EPI 2: optional f32 copy [NB,H,cout] (may be null)
  int M, ldc, relu;        // linear only
  int tblock;              // linear only: 1 = store float32 output as 128-row transposed blocks [tile][ldc/4][128][4]
  void* out3;              // linear only, optional: 16-bit residual (value - its 16-bit rounding) of columns < lo_cols,
  int lo_cols;             //   [M, lo_cols]: hi + lo carry ~21 bits of the float32 result (split-precision operands)
  long out_sn, out_sh;     // EPI 2: output row of (image n, row h) = n*out_sn + h*out_sh (default H, 1)
  // conv_block1_tc_kernel: the A operand is computed in the kernel from the 1-channel input
  const float* x1;         // [NB, H, W] f32 (log-mel after bn0)
  const float* w1;         // [64][9] f32 conv_block1.conv1 weights with the bn1 scale folded in
  const float* shift1;     // [64] f32 folded bn1 shift
#ifdef SED_PROFILE
  int dbg;                 // -DSED_PROFILE builds only (SED_CONV_DBG): 1 = no stores, 2 = no drain, 4 = no MMA
#endif
};

// profiling switches compile to the constant 0 in the shipped library
#ifdef SED_PROFILE
#define SED_CONV_DBG(p, bit) ((p).dbg & (bit))
#else
#define SED_CONV_DBG(p, bit) 0
#endif

constexpr int kPatchBytes = 180 * 128;       // 18 x 10 pixels x 64 ch x 2 B
constexpr int kPatchStride = 23 * 1024;      // padded so every patch starts 1024-aligned
constexpr int kTileBytes = 128 * 128;        // 128 pixels x 64 ch x 2 B

template <int CIN, int BN, int NT, int SA, int SB>
struct ConvCfg {
  // 8 epilogue warps: two per TMEM lane quarter, each draining half of the BN accumulator columns
  static constexpr int EW = 8;
  static constexpr int THREADS = 64 + 32 * EW;
  static constexpr int CPW = BN / 2;                                  // accumulator columns per epilogue warp
  static constexpr int SS = 1536;                                     // cached bias entries (one column panel)
  static constexpr int NCHUNK = CIN / 64;
  static constexpr int A_STAGE = NT * kTileBytes;
  static constexpr int B_BLOCK = BN * 128;
  static constexpr int B_BYTES = SB * B_BLOCK;
  static constexpr int ACC_COLS = NT * BN;
  static constexpr int ACC_STAGES = (2 * ACC_COLS <= 512) ? 2 : 1;
  static constexpr int TMEM_COLS = (ACC_COLS * ACC_STAGES <= 32) ? 32 : (ACC_COLS * ACC_STAGES <= 64) ? 64
                                   : (ACC_COLS * ACC_STAGES <= 128) ? 128 : (ACC_COLS * ACC_STAGES <= 256) ? 256 : 512;
  static constexpr int SMEM_A = SA * A_STAGE;
  static constexpr int SMEM_MISC = 2 * SS * 4 + 256;
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + SMEM_A + B_BYTES + SMEM_MISC;
  static_assert(CIN % 64 == 0, "CIN must be a multiple of 64");
  static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "UMMA N");
  static_assert(ACC_COLS <= 512, "TMEM columns");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

// Drain one 128 x BN accumulator tile: this warp handles TMEM lane quarter (warp & 3) and column half
// `chalf`.  Applies y = max(acc * scale + shift, 0) and the layer's output transform (store / 2x2 avg-pool /
// mean over the 8 frequency columns / plain GEMM row store).
template <typename T, int BN, bool BRES, int EPI>
SED_DEVICE_INLINE void conv_epilogue_tile(const uint32_t taddr, const int chalf, const int warp, const int lane,
                                          const float* s_scale, const float* s_shift, const int ch0,
                                          const int tile, const bool tile_ok, const int n, const int h0, const int w0,
                                          const ConvParams& p, uint8_t* smem_stg, const CUtensorMap* tmO_ptr) {
  constexpr int CPW = BN / 2;
  constexpr int LDB = (CPW >= 64) ? 4 : CPW / 16;  // 16-column TMEM loads in flight per wait
  // TMA-store staging (EPI_STORE): with CPW >= 64 each column half owns a staging tile and a 128-thread
  // named barrier; with CPW == 32 all 8 warps fill one 64-channel tile together.
  constexpr bool kSplitStg = CPW >= 64;
  const int stg_group = kSplitStg ? chalf : 0;
  const int stg_threads = kSplitStg ? 128 : 256;
  const bool stg_leader = (lane == 0) && (warp == (kSplitStg ? 2 + 4 * chalf : 2));
  uint8_t* stg = smem_stg + stg_group * kTileBytes;
  const int m = (warp & 3) * 32 + lane;  // row of the 128-row tile
  const int hl = m >> 3, wl = m & 7;
  const int h = h0 + hl, w = w0 + wl;
  T* out16 = reinterpret_cast<T*>(p.out);
  (void)w; (void)out16; (void)stg; (void)stg_leader; (void)stg_threads;
        for (int cb = 0; cb < CPW / 16; cb += LDB) {
          uint32_t rr[LDB][16];
#pragma unroll
          for (int u = 0; u < LDB; ++u) tmem_ld16(taddr + (cb + u) * 16, rr[u]);
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < LDB; ++u) {
          const int cc = chalf * (CPW / 16) + cb + u;
          const uint32_t(&r)[16] = rr[u];
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int ch = (BRES ? 0 : ch0) + cc * 16 + j;
            float x = fmaf(__uint_as_float(r[j]), s_scale[ch], s_shift[ch]);
            if (EPI != EPI_LINEAR || p.relu) x = fmaxf(x, 0.0f);
            v[j] = x;
          }
          if (EPI == EPI_STORE) {
            // stage this row's 16 channels in the SWIZZLE_128B tile; one TMA store per 64-channel chunk
            if (u == 0) {
              if (stg_leader) bulk_wait_read0();          // previous store has finished reading the tile
              named_bar_sync(1 + stg_group, stg_threads);
            }
            uint4 q0, q1;
            q0.x = Elem16<T>::pack2(v[0], v[1]);   q0.y = Elem16<T>::pack2(v[2], v[3]);
            q0.z = Elem16<T>::pack2(v[4], v[5]);   q0.w = Elem16<T>::pack2(v[6], v[7]);
            q1.x = Elem16<T>::pack2(v[8], v[9]);   q1.y = Elem16<T>::pack2(v[10], v[11]);
            q1.z = Elem16<T>::pack2(v[12], v[13]); q1.w = Elem16<T>::pack2(v[14], v[15]);
            const int c16 = ((cc * 16) & 63) >> 3;         // 16-byte chunk of the 64-channel row
            uint8_t* rowp = stg + m * 128;
            *reinterpret_cast<uint4*>(rowp + ((c16 ^ (m & 7)) << 4)) = q0;
            *reinterpret_cast<uint4*>(rowp + (((c16 + 1) ^ (m & 7)) << 4)) = q1;
            if (u == LDB - 1) {
              fence_proxy_async_smem();
              named_bar_sync(1 + stg_group, stg_threads);
              if (stg_leader && tile_ok) {
                tma_store_4d(tmO_ptr, stg, ch0 + ((cc * 16) & ~63), w0, h0, n);
                bulk_commit();
              }
            }
          } else if (EPI == EPI_POOL) {
            // 2x2 average: partners are lane^1 (w) and lane^8 (h); recursive halving so each lane
            // finishes with 4 channels of one pooled pixel.
            float k8[8];
            const bool wodd = (wl & 1) != 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float send = wodd ? v[j] : v[8 + j];
              const float keep = wodd ? v[8 + j] : v[j];
              k8[j] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
            }
            float k4[4];
            const bool hodd = (hl & 1) != 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float send = hodd ? k8[j] : k8[4 + j];
              const float keep = hodd ? k8[4 + j] : k8[j];
              k4[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);  // the 1/4 of the average is folded into scale/shift
            }
            const int Hp = p.H >> 1, Wp = p.W >> 1;
            const int hp = h >> 1, wp = w >> 1;
            if (tile_ok && hp < Hp) {
              const int ch = ch0 + cc * 16 + (wodd ? 8 : 0) + (hodd ? 4 : 0);
              uint2 q;
              q.x = Elem16<T>::pack2(k4[0], k4[1]);
              q.y = Elem16<T>::pack2(k4[2], k4[3]);
              T* dst = out16 + ((static_cast<size_t>(n) * Hp + hp) * Wp + wp) * p.cout + ch;
              *reinterpret_cast<uint2*>(dst) = q;
            }
          } else if (EPI == EPI_FREQMEAN) {
            // mean over the 8 frequency columns of a row (W == 8): lanes ^1, ^2, ^4
            float k8[8];
            const bool b0 = (wl & 1) != 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float send = b0 ? v[j] : v[8 + j];
              const float keep = b0 ? v[8 + j] : v[j];
              k8[j] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
            }
            float k4[4];
            const bool b1 = (wl & 2) != 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float send = b1 ? k8[j] : k8[4 + j];
              const float keep = b1 ? k8[4 + j] : k8[j];
              k4[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
            }
            float k2[2];
            const bool b2 = (wl & 4) != 0;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const float send = b2 ? k4[j] : k4[2 + j];
              const float keep = b2 ? k4[2 + j] : k4[j];
              k2[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);  // the 1/8 of the mean is folded into scale/shift
            }
            if (tile_ok && h < p.H) {
              const int ch = ch0 + cc * 16 + (b0 ? 8 : 0) + (b1 ? 4 : 0) + (b2 ? 2 : 0);
              const size_t orow = static_cast<size_t>(n) * p.out_sn + static_cast<size_t>(h) * p.out_sh;
              T* dst = out16 + orow * p.cout + ch;
              *reinterpret_cast<uint32_t*>(dst) = Elem16<T>::pack2(k2[0], k2[1]);
              if (p.out2)  // optional float32 copy of the features (heads without a temporal block)
                *reinterpret_cast<float2*>(reinterpret_cast<float*>(p.out2) + orow * p.cout + ch) =
                    make_float2(k2[0], k2[1]);
            }
          } else {  // EPI_LINEAR
            const long row = static_cast<long>(tile) * 128 + m;
            if (tile_ok && row < p.M) {
              if (p.out == nullptr) {
                // 16-bit output only (the QKV projection feeding the tensor-core attention kernel)
              } else if (p.tblock) {
                // 128-row transposed blocks: float4 column c4 of row m of tile `tile` sits at
                // ((tile * ldc/4 + c4) * 128 + m): a warp (32 consecutive rows) writes 512 contiguous bytes
                float4* dst4 = reinterpret_cast<float4*>(p.out) +
                               (static_cast<size_t>(tile) * (p.ldc >> 2) + ((ch0 + cc * 16) >> 2)) * 128 + m;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                  dst4[j * 128] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
              } else {
              float* dst = reinterpret_cast<float*>(p.out) + row * p.ldc + ch0 + cc * 16;
#pragma unroll
              for (int j = 0; j < 4; ++j)
                reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
              }
              if (p.out2) {
                uint4 q0, q1;
                q0.x = Elem16<T>::pack2(v[0], v[1]);   q0.y = Elem16<T>::pack2(v[2], v[3]);
                q0.z = Elem16<T>::pack2(v[4], v[5]);   q0.w = Elem16<T>::pack2(v[6], v[7]);
                q1.x = Elem16<T>::pack2(v[8], v[9]);   q1.y = Elem16<T>::pack2(v[10], v[11]);
                q1.z = Elem16<T>::pack2(v[12], v[13]); q1.w = Elem16<T>::pack2(v[14], v[15]);
                T* d2 = reinterpret_cast<T*>(p.out2) + row * p.ldc + ch0 + cc * 16;
                reinterpret_cast<uint4*>(d2)[0] = q0;
                reinterpret_cast<uint4*>(d2)[1] = q1;
                if (p.out3 && ch0 + cc * 16 < p.lo_cols) {
                  const uint32_t hi[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
                  uint32_t lo[8];
#pragma unroll
                  for (int j = 0; j < 8; ++j)
                    lo[j] = Elem16<T>::pack2(v[2 * j] - Elem16<T>::to_float(static_cast<uint16_t>(hi[j] & 0xFFFFu)),
                                             v[2 * j + 1] - Elem16<T>::to_float(static_cast<uint16_t>(hi[j] >> 16)));
                  T* d3 = reinterpret_cast<T*>(p.out3) + row * p.lo_cols + ch0 + cc * 16;
                  reinterpret_cast<uint4*>(d3)[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                  reinterpret_cast<uint4*>(d3)[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
                }
              }
            }
          }
          }
        }
}

// UMMA shared-memory descriptor split into its constant high word and an address-carrying low word:
// consecutive operands differ only by a small addend on the low word (addresses are < 256 KB, so the
// 14-bit start-address field never carries), which keeps the single issuing thread at ~2 integer
// instructions per tcgen05.mma.
SED_DEVICE_INLINE constexpr uint32_t desc_hi_sw128(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29);
}
SED_DEVICE_INLINE uint32_t desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
SED_DEVICE_INLINE uint64_t desc_join(uint32_t lo, uint32_t hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}

// The plain GEMM out[M, N] = A[M, K] * B[N, K]^T (+ bias, ReLU) of the temporal blocks: one work item is NT row tiles
// of 128 rows against one BN-column slice, the slices of a row-tile group are consecutive items.  Warp roles:
// warp0 = TMA producer, warp1 = MMA issuer (+TMEM alloc), warps2-9 = epilogue.  tmO is not read (the epilogue stores
// from registers); it keeps the parameter block laid out as in conv_umma2_kernel.
template <typename T, int CIN, int BN, int NT, int SA, int SB>
__global__ void __launch_bounds__(ConvCfg<CIN, BN, NT, SA, SB>::THREADS, 1)
conv_umma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO, const ConvParams p) {
  using Cfg = ConvCfg<CIN, BN, NT, SA, SB>;
  constexpr int NCHUNK = Cfg::NCHUNK;
  constexpr int ACC_STAGES = Cfg::ACC_STAGES;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::SMEM_A;
  float* s_scale = reinterpret_cast<float*>(smem_b + Cfg::B_BYTES);
  float* s_shift = s_scale + Cfg::SS;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_shift + Cfg::SS);
  uint64_t* a_full = bars;             // [SA]
  uint64_t* a_empty = a_full + SA;     // [SA]
  uint64_t* b_full = a_empty + SA;     // [SB]
  uint64_t* b_empty = b_full + SB;     // [SB]
  uint64_t* t_full = b_empty + SB;     // [2]
  uint64_t* t_empty = t_full + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // ---- work decomposition -------------------------------------------------------------
  const int groups = (p.num_tiles + NT - 1) / NT;
  const int item_begin = blockIdx.x, item_stride = gridDim.x, item_end = groups * p.nslices;

  // ---- one-time setup -------------------------------------------------------------------
  // the epilogue's affine is 1 x acc + bias
  for (int i = threadIdx.x; i < Cfg::SS && i < p.cout; i += blockDim.x) {
    s_scale[i] = 1.0f;
    s_shift[i] = p.shift ? p.shift[i] : 0.0f;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < SA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < SB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], Cfg::EW); }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =============================== TMA producer ===========================================
    if (elect_one()) {
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0;
      for (int item = item_begin; item < item_end; item += item_stride) {
        const int g = item / p.nslices;
        const int slice = item - g * p.nslices;
        for (int c = 0; c < NCHUNK; ++c) {
          mbar_wait(&a_empty[sa], pa ^ 1);
          mbar_expect_tx(&a_full[sa], NT * kTileBytes);
#pragma unroll
          for (int t = 0; t < NT; ++t)
            tma_load_2d(smem_a + sa * Cfg::A_STAGE + t * kTileBytes, &tmA, &a_full[sa], c * 64, (g * NT + t) * 128);
          if (++sa == SA) { sa = 0; pa ^= 1; }
          mbar_wait(&b_empty[sb], pb ^ 1);
          mbar_expect_tx(&b_full[sb], Cfg::B_BLOCK);
          tma_load_2d(smem_b + sb * Cfg::B_BLOCK, &tmB, &b_full[sb], c * 64, slice * BN);
          if (++sb == SB) { sb = 0; pb ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer =============================================
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_f16(Elem16<T>::kFmt, 128, BN);
      constexpr uint32_t a_hi = desc_hi_sw128(1024);
      constexpr uint32_t b_hi = desc_hi_sw128(1024);
      constexpr uint32_t a_tile_step = kTileBytes >> 4;
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a));
      const uint32_t b_lo0 = desc_lo(smem_u32(smem_b));
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0, acc = 0, pacc = 0;
      for (int item = item_begin; item < item_end; item += item_stride) {
        mbar_wait(&t_empty[acc], pacc ^ 1);
        tc_fence_after();
        const uint32_t d_base = tmem_base + acc * Cfg::ACC_COLS;
        for (int c = 0; c < NCHUNK; ++c) {
          mbar_wait(&a_full[sa], pa);
          tc_fence_after();
          const uint32_t a_lo = a_lo0 + sa * (Cfg::A_STAGE >> 4);
          mbar_wait(&b_full[sb], pb);
          tc_fence_after();
          const uint32_t b_lo = b_lo0 + sb * (Cfg::B_BLOCK >> 4);
#pragma unroll
          for (int t = 0; t < NT; ++t) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if (!SED_CONV_DBG(p, 4))
                umma_f16(d_base + t * BN, desc_join(a_lo + t * a_tile_step + k * 2, a_hi),
                         desc_join(b_lo + k * 2, b_hi), idesc, (c | k) ? 1u : 0u);
            }
          }
          umma_commit(&a_empty[sa]);
          if (++sa == SA) { sa = 0; pa ^= 1; }
          umma_commit(&b_empty[sb]);
          if (++sb == SB) { sb = 0; pb ^= 1; }
        }
        umma_commit(&t_full[acc]);
        if (++acc == ACC_STAGES) { acc = 0; pacc ^= 1; }
      }
    }
  } else {
    // =============================== epilogue (EW warps) =====================================
    const int quarter = warp & 3;            // TMEM lane quarter this warp may access
    const int chalf = (warp - 2) >> 2;       // which half of the BN columns this warp drains
    constexpr int CPW = Cfg::CPW;            // columns per warp
    uint32_t acc = 0, pacc = 0;
    for (int item = item_begin; item < item_end; item += item_stride) {
      const int g = item / p.nslices;
      const int slice = item - g * p.nslices;
      const int ch0 = slice * BN;
      mbar_wait(&t_full[acc], pacc);
      tc_fence_after();
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        if (SED_CONV_DBG(p, 2)) break;
        const int tile = g * NT + t;
        const bool tile_ok = (tile < p.num_tiles) && !SED_CONV_DBG(p, 1);
        const uint32_t taddr = tmem_base + acc * Cfg::ACC_COLS + t * BN + chalf * CPW +
                               (static_cast<uint32_t>(quarter * 32) << 16);
        conv_epilogue_tile<T, BN, false, EPI_LINEAR>(taddr, chalf, warp, lane, s_scale, s_shift, ch0, tile, tile_ok, 0,
                                                     0, 0, p, nullptr, nullptr);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&t_empty[acc]);
      if (++acc == ACC_STAGES) { acc = 0; pacc ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// =================================================================================================
// The conv layers on CTA pairs (tcgen05 cta_group::2).
//
// With the accumulator N of a single-CTA MMA limited to the layer's Cout slice (64 or 128), each
// K=16 MMA step reads 4 KB of A plus N*32 B of B from shared memory in N/2 cycles -- more than the
// 128 B/clk the shared-memory pipe delivers, so a single CTA runs at half the tensor rate.  A CTA pair
// computes M = 256 pixels (one 16x8 tile per CTA) against the SAME N columns; each CTA keeps only half of
// the weight rows (N/2) resident and the hardware shares the halves, so the per-CTA shared-memory traffic
// per MMA drops to 4 KB + N*16 B and the weight-resident footprint halves as well.
//
// Roles per CTA: warp0 = TMA producer (own haloed patch; completion is signalled on the LEADER's mbarrier),
// warp1 = TMEM allocation (+ MMA issue on the leader only, commits multicast to both CTAs),
// warps2-9 = epilogue of the CTA's own 128 accumulator rows.
// =================================================================================================
template <int CIN, int BN, int EPI, int SA, int ACC, bool BRES, int NT, int SB>
struct Conv2Cfg {
  static constexpr int NCHUNK = CIN / 64;
  static constexpr int TAPS = 9;
  static constexpr int B_HALF = (BN / 2) * 128;                       // one (chunk, tap) block of this CTA's rows
  static constexpr int B_BYTES = BRES ? NCHUNK * TAPS * B_HALF : SB * B_HALF;
  static constexpr int A_STAGE = NT * kPatchStride;
  static constexpr int SMEM_A = SA * A_STAGE;
  static constexpr int CPW = BN / 2;
  static constexpr int NSTG = (EPI == EPI_STORE) ? (CPW >= 64 ? 2 : 1) : 0;
  static constexpr int SMEM_STG = NSTG * kTileBytes;
  static constexpr int SS = BRES ? BN : 512;
  static constexpr int SMEM_MISC = 2 * SS * 4 + 256;
  static constexpr int SMEM_BYTES = 1024 + SMEM_A + B_BYTES + SMEM_STG + SMEM_MISC;
  static constexpr int ACC_COLS = NT * BN;
  static constexpr int TMEM_COLS = (ACC * ACC_COLS <= 32) ? 32 : (ACC * ACC_COLS <= 64) ? 64
                                   : (ACC * ACC_COLS <= 128) ? 128 : (ACC * ACC_COLS <= 256) ? 256 : 512;
  static constexpr int THREADS = 64 + 32 * 8;
  static_assert(ACC * ACC_COLS <= 512, "TMEM columns");
  static_assert(BN % 32 == 0 && BN <= 256, "pair MMA: N multiple of 16 per CTA half");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

template <typename T, int CIN, int BN, int EPI, int SA, int ACC, bool BRES, int NT, int SB>
__global__ void __cluster_dims__(2, 1, 1)
__launch_bounds__(Conv2Cfg<CIN, BN, EPI, SA, ACC, BRES, NT, SB>::THREADS, 1)
conv_umma2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmO, const ConvParams p) {
  using Cfg = Conv2Cfg<CIN, BN, EPI, SA, ACC, BRES, NT, SB>;
  constexpr int TAPS = Cfg::TAPS;
  constexpr int NCHUNK = Cfg::NCHUNK;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::SMEM_A;
  uint8_t* smem_stg = smem_b + Cfg::B_BYTES;
  float* s_scale = reinterpret_cast<float*>(smem_stg + Cfg::SMEM_STG);
  float* s_shift = s_scale + Cfg::SS;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_shift + Cfg::SS);
  uint64_t* a_full = bars;            // [SA]  leader's copy is the live one
  uint64_t* a_empty = a_full + SA;    // [SA]  per CTA (multicast commit)
  uint64_t* b_full = a_empty + SA;    // [SB]  leader's copy (index 0 = "resident weights landed")
  uint64_t* b_empty = b_full + SB;    // [SB]  per CTA (multicast commit)
  uint64_t* t_full = b_empty + SB;    // [ACC] per CTA (multicast commit)
  uint64_t* t_empty = t_full + ACC;   // [ACC] leader's copy, 16 arrivals (8 warps x 2 CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + ACC);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  // ---- work decomposition: an item = 2*NT tiles (NT per CTA of the pair) of one Cout slice ----
  const int pr = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int items = (p.num_tiles + 2 * NT - 1) / (2 * NT);
  int work_begin, work_stride, work_end, fixed_slice = 0;
  if (BRES) {
    fixed_slice = pr % p.nslices;
    work_begin = pr / p.nslices;
    work_stride = npairs / p.nslices;
    work_end = items;
  } else {
    work_begin = pr;
    work_stride = npairs;
    work_end = items * p.nslices;
  }

  const int ss_base = BRES ? fixed_slice * BN : 0;
  for (int i = threadIdx.x; i < Cfg::SS && ss_base + i < p.cout; i += blockDim.x) {
    // the averaging factor of the pooling epilogues rides the BN affine: relu(k x) = k relu(x) for k > 0, and scaling
    // by a power of two is exact, so the result is bit-identical to averaging afterwards
    constexpr float kAvg = (EPI == EPI_POOL) ? 0.25f : (EPI == EPI_FREQMEAN) ? 0.125f : 1.0f;
    s_scale[i] = kAvg * p.scale[ss_base + i];
    s_shift[i] = kAvg * p.shift[ss_base + i];
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI == EPI_STORE) tma_prefetch_desc(&tmO);
    for (int i = 0; i < SA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < SB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < ACC; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 16); }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc2(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish2();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // peer barriers / TMEM are ready before any cross-CTA signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto tile_coords = [&](int tile, int& n, int& h0, int& w0) {
    const int per_img = p.tiles_h * p.tiles_w;
    n = fast_div(tile, p.magic_img);
    const int rem = tile - n * per_img;
    const int th = fast_div(rem, p.magic_w);
    h0 = th * 16;
    w0 = (rem - th * p.tiles_w) * 8;
  };

  if (warp == 0) {
    // =============================== TMA producer (both CTAs) ===============================
    if (elect_one()) {
      if (BRES) {
        const uint32_t bfull_leader = map_to_cta(&b_full[0], 0);
        if (leader) mbar_expect_tx(&b_full[0], 2 * Cfg::B_BYTES);
        for (int c = 0; c < NCHUNK; ++c)
          for (int tap = 0; tap < TAPS; ++tap)
            tma_load_2d_2sm(smem_b + (c * TAPS + tap) * Cfg::B_HALF, &tmB, bfull_leader, tap * CIN + c * 64,
                            fixed_slice * BN + rank * (BN / 2));
      }
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0;
      for (int w = work_begin; w < work_end; w += work_stride) {
        const int item = BRES ? w : w / p.nslices;
        const int slice = BRES ? fixed_slice : w - item * p.nslices;
        for (int c = 0; c < NCHUNK; ++c) {
          mbar_wait(&a_empty[sa], pa ^ 1);
          if (leader) mbar_expect_tx(&a_full[sa], 2 * NT * kPatchBytes);
          const uint32_t afull_leader = map_to_cta(&a_full[sa], 0);
#pragma unroll
          for (int t = 0; t < NT; ++t) {
            int n, h0, w0;
            tile_coords((item * 2 + rank) * NT + t, n, h0, w0);  // past-the-end tiles: n >= NB -> zeros
            tma_load_4d_2sm(smem_a + sa * Cfg::A_STAGE + t * kPatchStride, &tmA, afull_leader, c * 64, w0 - 1, h0 - 1,
                            n);
          }
          if (++sa == SA) { sa = 0; pa ^= 1; }
          if (!BRES) {
            for (int tap = 0; tap < TAPS; ++tap) {
              mbar_wait(&b_empty[sb], pb ^ 1);
              if (leader) mbar_expect_tx(&b_full[sb], 2 * Cfg::B_HALF);
              tma_load_2d_2sm(smem_b + sb * Cfg::B_HALF, &tmB, map_to_cta(&b_full[sb], 0), tap * CIN + c * 64,
                              slice * BN + rank * (BN / 2));
              if (++sb == SB) { sb = 0; pb ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (leader CTA only) ===========================
    if (leader && elect_one()) {
      constexpr uint32_t idesc = umma_idesc_f16(Elem16<T>::kFmt, 256, BN);
      constexpr uint32_t a_hi = desc_hi_sw128(1280);
      constexpr uint32_t b_hi = desc_hi_sw128(1024);
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a));
      const uint32_t b_lo0 = desc_lo(smem_u32(smem_b));
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0, acc = 0, pacc = 0;
      if (BRES) {
        mbar_wait(&b_full[0], 0);
        tc_fence_after();
      }
      for (int w = work_begin; w < work_end; w += work_stride) {
        mbar_wait(&t_empty[acc], pacc ^ 1);
        tc_fence_after();
        const uint32_t d_base = tmem_base + acc * Cfg::ACC_COLS;
        for (int c = 0; c < NCHUNK; ++c) {
          mbar_wait(&a_full[sa], pa);
          tc_fence_after();
          const uint32_t a_lo = a_lo0 + sa * (Cfg::A_STAGE >> 4);
#pragma unroll
          for (int tap = 0; tap < TAPS; ++tap) {
            uint32_t b_lo;
            if (BRES) {
              b_lo = b_lo0 + (c * TAPS + tap) * (Cfg::B_HALF >> 4);
            } else {
              mbar_wait(&b_full[sb], pb);
              tc_fence_after();
              b_lo = b_lo0 + sb * (Cfg::B_HALF >> 4);
            }
            const uint32_t tap_off = ((tap / 3) * 10 + (tap % 3)) * 8;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                if (!SED_CONV_DBG(p, 4))
                  umma_f16_2sm(d_base + t * BN, desc_join(a_lo + t * (kPatchStride >> 4) + tap_off + k * 2, a_hi),
                               desc_join(b_lo + k * 2, b_hi), idesc, (c | tap | k) ? 1u : 0u);
              }
            }
            if (!BRES) {
              umma_commit_2sm(&b_empty[sb], 3);
              if (++sb == SB) { sb = 0; pb ^= 1; }
            }
          }
          umma_commit_2sm(&a_empty[sa], 3);
          if (++sa == SA) { sa = 0; pa ^= 1; }
        }
        umma_commit_2sm(&t_full[acc], 3);
        if (++acc == ACC) { acc = 0; pacc ^= 1; }
      }
    }
  } else if (warp >= 2 && warp < 10) {
    // =============================== epilogue (8 warps, both CTAs) ==========================
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int chalf = (ew & 7) >> 2;
    constexpr int CPW = Cfg::CPW;
    const bool stg_leader = (lane == 0) && (warp == ((CPW >= 64) ? 2 + 4 * chalf : 2));
    uint32_t it = 0;
    for (int w = work_begin; w < work_end; w += work_stride, ++it) {
      const uint32_t acc = it % ACC, pacc = (it / ACC) & 1;
      const int item = BRES ? w : w / p.nslices;
      const int slice = BRES ? fixed_slice : w - item * p.nslices;
      const int ch0 = slice * BN;
      mbar_wait(&t_full[acc], pacc);
      tc_fence_after();
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        if (SED_CONV_DBG(p, 2)) break;
        const int tile = (item * 2 + rank) * NT + t;
        const bool tile_ok = (tile < p.num_tiles) && !SED_CONV_DBG(p, 1);
        int n, h0, w0;
        tile_coords(tile, n, h0, w0);
        const uint32_t taddr = tmem_base + acc * Cfg::ACC_COLS + t * BN + chalf * CPW +
                               (static_cast<uint32_t>(quarter * 32) << 16);
        conv_epilogue_tile<T, BN, BRES, EPI>(taddr, chalf, warp, lane, s_scale, s_shift, ch0, tile, tile_ok, n, h0, w0,
                                             p, smem_stg, &tmO);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_light(&t_empty[acc], 0);
    }
    if (EPI == EPI_STORE && stg_leader) bulk_wait_all0();
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the leader's MMAs read the peer's shared memory: nobody leaves early
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace sed
