// Host-side launchers for the conv stack and the tensor-core GEMM, plus the CUDA-core first layer.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "sed_conv.cuh"
#include "sed_kernels.h"

namespace sed {

// ---------------------------------------------------------------------------------------------
// error string (thread-local)
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
const char* last_error() { return g_err; }
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency,
// so the library loads on hosts without a driver for symbol checks)
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static int make_map(CUtensorMap* m, int dtype, int rank, void* base, const uint64_t* dims, const uint64_t* strides_b,
                    const uint32_t* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point unavailable");
    return SED_ERR_DRIVER;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstr[5];
  cuuint32_t bdim[5], estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
    if (i > 0) gstr[i - 1] = strides_b[i - 1];
  }
  CUresult r = enc(m, dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, base, gdim,
                   gstr, bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d), rank %d", (int)r, rank);
    return SED_ERR_DRIVER;
  }
  return SED_OK;
}

static int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// ---------------------------------------------------------------------------------------------
// conv_block1.conv1 (Cin = 1, K = 9 taps) + bn1 + ReLU.  pytorch/models.py:128 (first conv of block 1)
//
// Float32-grade accuracy on the tensor cores: the 3x3 neighbourhood of each output pixel (9 taps padded
// to K = 16) and the weights are split into fp16 hi + lo parts and three tcgen05.mma (hi*hi + lo*hi +
// hi*lo, M = 128 pixels, N = 64 channels, K = 16) accumulate in fp32 TMEM -- the dropped lo*lo term is
// ~2^-22 relative.  Each CTA loops over tiles of 2 rows x 64 mel bins: its 128 threads gather the taps
// straight from the log-mel tensor (L1/L2 resident), write the K-major SWIZZLE_32B operand rows, one thread
// issues the MMAs, then every thread drains its own TMEM lane (one pixel, 64 channels), applies the folded
// BatchNorm + ReLU and stores 128 contiguous bytes of NHWC output.  Two CTAs per SM overlap the phases.
// ---------------------------------------------------------------------------------------------
SED_DEVICE_INLINE constexpr uint32_t desc_hi_sw32(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (6u << 29);  // layout_type 6 = SWIZZLE_32B
}

template <typename T>
__global__ void __launch_bounds__(128, 4)
conv_first_umma_kernel(const __grid_constant__ CUtensorMap tmO, const float* __restrict__ x, int NB, int H,
                       const float* __restrict__ w9, const float* __restrict__ scale,
                       const float* __restrict__ shift) {
  constexpr int W = 64;
  __shared__ __align__(1024) uint8_t s_stg[128 * 128];   // output tile, SWIZZLE_128B, TMA-stored
  __shared__ __align__(1024) uint8_t s_a[2][128 * 32];   // A hi / lo: 128 pixel rows x 16 taps (32 B)
  __shared__ __align__(1024) uint8_t s_b[2][64 * 32];    // B hi / lo: 64 channel rows x 16 taps
  __shared__ float s_scale[64], s_shift[64];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ uint32_t s_tmem;

  const int tid = threadIdx.x, warp = tid >> 5;
  // ---- weights -> split fp16 operand rows (row = channel, 32 B, 16-byte chunk j stored at j ^ bit2(row)) ----
  if (tid < 64) {
    float wv[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) wv[t] = (t < 9) ? w9[tid * 9 + t] : 0.0f;
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const __half h0 = __float2half_rn(wv[2 * t]), h1 = __float2half_rn(wv[2 * t + 1]);
      const __half l0 = __float2half_rn(wv[2 * t] - __half2float(h0));
      const __half l1 = __float2half_rn(wv[2 * t + 1] - __half2float(h1));
      hi[t] = static_cast<uint32_t>(__half_as_ushort(h0)) | (static_cast<uint32_t>(__half_as_ushort(h1)) << 16);
      lo[t] = static_cast<uint32_t>(__half_as_ushort(l0)) | (static_cast<uint32_t>(__half_as_ushort(l1)) << 16);
    }
    const int sw = (tid >> 2) & 1;
    *reinterpret_cast<uint4*>(&s_b[0][tid * 32 + ((0 ^ sw) << 4)]) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(&s_b[0][tid * 32 + ((1 ^ sw) << 4)]) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    *reinterpret_cast<uint4*>(&s_b[1][tid * 32 + ((0 ^ sw) << 4)]) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *reinterpret_cast<uint4*>(&s_b[1][tid * 32 + ((1 ^ sw) << 4)]) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
    s_scale[tid] = scale[tid];
    s_shift[tid] = shift[tid];
  }
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(&s_tmem, 64);
    tmem_relinquish();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem;
  // only fp16 operands here: the fp32-grade split needs the 11-bit significand of fp16 in both parts
  constexpr uint32_t idesc = umma_idesc_f16(0, 128, 64);
  constexpr uint32_t d_hi = desc_hi_sw32(256);
  const uint32_t a_lo_hi = desc_lo(smem_u32(&s_a[0][0])), a_lo_lo = desc_lo(smem_u32(&s_a[1][0]));
  const uint32_t b_lo_hi = desc_lo(smem_u32(&s_b[0][0])), b_lo_lo = desc_lo(smem_u32(&s_b[1][0]));

  const int tiles_h = (H + 1) >> 1;
  const int num_tiles = NB * tiles_h;
  const int hl = tid >> 6, w = tid & 63;
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int n = tile / tiles_h;
    const int h = (tile - n * tiles_h) * 2 + hl;
    // ---- gather the 3x3 neighbourhood (zero outside the image: conv padding=1) ----
    float in[9];
    const float* xn = x + static_cast<size_t>(n) * H * W;
#pragma unroll
    for (int dr = 0; dr < 3; ++dr) {
      const int hh = h + dr - 1;
      const bool rok = hh >= 0 && hh < H;
#pragma unroll
      for (int dc = 0; dc < 3; ++dc) {
        const int ww = w + dc - 1;
        in[dr * 3 + dc] = (rok && ww >= 0 && ww < W) ? __ldg(xn + hh * W + ww) : 0.0f;
      }
    }
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const float v0 = (2 * t < 9) ? in[2 * t] : 0.0f;
      const float v1 = (2 * t + 1 < 9) ? in[2 * t + 1] : 0.0f;
      const __half h0 = __float2half_rn(v0), h1 = __float2half_rn(v1);
      const __half l0 = __float2half_rn(v0 - __half2float(h0)), l1 = __float2half_rn(v1 - __half2float(h1));
      hi[t] = static_cast<uint32_t>(__half_as_ushort(h0)) | (static_cast<uint32_t>(__half_as_ushort(h1)) << 16);
      lo[t] = static_cast<uint32_t>(__half_as_ushort(l0)) | (static_cast<uint32_t>(__half_as_ushort(l1)) << 16);
    }
    const int sw = (tid >> 2) & 1;
    *reinterpret_cast<uint4*>(&s_a[0][tid * 32 + ((0 ^ sw) << 4)]) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(&s_a[0][tid * 32 + ((1 ^ sw) << 4)]) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    *reinterpret_cast<uint4*>(&s_a[1][tid * 32 + ((0 ^ sw) << 4)]) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *reinterpret_cast<uint4*>(&s_a[1][tid * 32 + ((1 ^ sw) << 4)]) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
    fence_proxy_async_smem();
    tc_fence_before();
    if (tid == 0) bulk_wait_read0();  // the previous tile's TMA store has finished reading s_stg
    __syncthreads();  // operands written by all threads; previous tile's TMEM reads are complete
    if (tid == 0) {
      tc_fence_after();
      umma_f16(tmem_base, desc_join(a_lo_hi, d_hi), desc_join(b_lo_hi, d_hi), idesc, 0u);
      umma_f16(tmem_base, desc_join(a_lo_lo, d_hi), desc_join(b_lo_hi, d_hi), idesc, 1u);
      umma_f16(tmem_base, desc_join(a_lo_hi, d_hi), desc_join(b_lo_lo, d_hi), idesc, 1u);
      umma_commit(&s_bar);
    }
    mbar_wait(&s_bar, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- drain: thread = TMEM lane = pixel (hl, w); 64 channels ----
    uint32_t r[4][16];
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
#pragma unroll
    for (int u = 0; u < 4; ++u) tmem_ld16(taddr + u * 16, r[u]);
    tmem_ld_wait();
    {
      uint8_t* rowp = s_stg + tid * 128;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int c = u * 16 + 2 * j;
          const float v0 = fmaxf(fmaf(__uint_as_float(r[u][2 * j]), s_scale[c], s_shift[c]), 0.0f);
          const float v1 = fmaxf(fmaf(__uint_as_float(r[u][2 * j + 1]), s_scale[c + 1], s_shift[c + 1]), 0.0f);
          pk[j] = Elem16<T>::pack2(v0, v1);
        }
        *reinterpret_cast<uint4*>(rowp + (((2 * u) ^ (tid & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        *reinterpret_cast<uint4*>(rowp + (((2 * u + 1) ^ (tid & 7)) << 4)) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      }
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {  // rows past H (odd H) are clipped by the tensor map
      tma_store_4d(&tmO, s_stg, 0, 0, (tile - n * tiles_h) * 2, n);
      bulk_commit();
    }
  }
  if (tid == 0) bulk_wait_all0();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 64);
  }
}

int conv_first_launch(const float* x, int NB, int H, int W, const float* w9, const float* scale, const float* shift,
                      void* out, int dtype, cudaStream_t stream) {
  if (W != 64 || NB <= 0 || H <= 0) {
    set_error("conv_first: W must be 64 (got %d)", W);
    return SED_ERR_BAD_SHAPE;
  }
  CUtensorMap tmO;
  {
    const uint64_t dims[4] = {64, 64, (uint64_t)H, (uint64_t)NB};
    const uint64_t str[3] = {64 * 2, 64 * 64 * 2, (uint64_t)H * 64 * 64 * 2};
    const uint32_t box[4] = {64, 64, 2, 1};
    int rc = make_map(&tmO, dtype, 4, out, dims, str, box);
    if (rc) return rc;
  }
  const long tiles = static_cast<long>(NB) * ((H + 1) / 2);
  const int grid = static_cast<int>(tiles < 4L * num_sms() ? tiles : 4L * num_sms());
  if (dtype == 0)
    conv_first_umma_kernel<__half><<<grid, 128, 0, stream>>>(tmO, x, NB, H, w9, scale, shift);
  else
    conv_first_umma_kernel<__nv_bfloat16><<<grid, 128, 0, stream>>>(tmO, x, NB, H, w9, scale, shift);
  return cudaGetLastError() == cudaSuccess ? SED_OK : SED_ERR_CUDA;
}

// ---------------------------------------------------------------------------------------------
// conv_block1 as ONE tensor-core kernel (engine variant 4): conv1 (1 -> 64 channels) runs as a split-fp16 tcgen05 GEMM
// (K = 9 taps padded to 16, hi*hi + lo*hi + hi*lo, float32-grade like conv_first_umma_kernel) on the 18 x 10 pixel halo
// patch of every conv2 tile; its accumulators are drained from TMEM through bn1 + ReLU straight into the swizzled
// shared-memory patch that conv2's implicit-GEMM MMAs read -- the [NB, H, 64, 64] intermediate never exists in HBM.
// CTA pairs (cta_group::2) as in conv_umma2_kernel: M = 256 = one tile per CTA, each CTA holds half of the weight
// rows of both layers.  Warp roles: 0 weight TMA, 1 MMA issuer (leader CTA: conv1 of tile i+1, then conv2 of tile i),
// 2-3 idle (they complete the control warpgroup that gives its registers away), 4-11 conv2 pooling epilogue, 12-19 two
// groups of conv1 operand builders (im2col of the one-channel input, hi/lo split) + TMEM drainers on alternate tiles.
// ---------------------------------------------------------------------------------------------
namespace c1tc {
constexpr int SA = 5;                       // conv2 patch stages
constexpr int ACC = 4;                      // conv2 accumulator stages (64 columns each)
constexpr int A_BYTES = SA * kPatchStride;  // 117,760
constexpr int B2_HALF = 32 * 128;           // one tap block of this CTA's 32 conv2 weight rows
constexpr int B2_BYTES = 9 * B2_HALF;       // 36,864
constexpr int OP_STAGE = 2 * 256 * 32;      // conv1 A operand, hi + lo, 256 rows x 32 B
constexpr int OP_BYTES = 2 * OP_STAGE;      // two stages
constexpr int MISC = 4096;
constexpr int SMEM_BYTES = 1024 + A_BYTES + B2_BYTES + OP_BYTES + 2048 + MISC;
constexpr int PG = 2;                       // producer groups (4 warps each): group g builds / drains tiles j = g mod 2
// Warpgroup 0 = control (warp 0 weights TMA, warp 1 MMA issue, warps 2-3 idle), warpgroups 1-2 = pooling epilogue,
// warpgroups 3-4 = producers.  20 warps launch at 96 registers per thread; the control group hands most of its
// registers to the producer groups (setmaxnreg), which need ~118.
constexpr int EPI_WARP0 = 4, PROD_WARP0 = 12;
constexpr int THREADS = 128 + 256 + 128 * PG;
constexpr int REG_CTRL = 40, REG_PROD = 120;
constexpr int C1_COL0 = ACC * 64;           // conv1 accumulators: columns 256 + stage*128 + mtile*64
}  // namespace c1tc

#ifdef SED_C1_STAMPS
// Debug build only (make NVFLAGS+=-DSED_C1_STAMPS; tools/c1_stamps.py): clock64 of each role of CTA 0 at the pipeline's
// hand-over points, for local work items [kStampFirst, kStampFirst + 32).
__device__ long long g_c1_stamps[3][32][8];
constexpr int kStampFirst = 200;
#define C1_STAMP(role, item, k)                                                               \
  do {                                                                                        \
    if (blockIdx.x == 0 && (item) >= kStampFirst && (item) < kStampFirst + 32)                \
      g_c1_stamps[role][(item) - kStampFirst][k] = clock64();                                 \
  } while (0)
#else
#define C1_STAMP(role, item, k) do {} while (0)
#endif

template <typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(c1tc::THREADS, 1)
conv_block1_tc_kernel(const __grid_constant__ CUtensorMap tmB, const ConvParams p) {
  using namespace c1tc;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* smem_a = smem;                          // [SA] conv2 patches (SWIZZLE_128B, 180 pixel rows x 128 B)
  uint8_t* smem_b = smem_a + A_BYTES;              // conv2 weights, 9 taps x 32 rows x 128 B
  uint8_t* s_op = smem_b + B2_BYTES;               // [2 stages][hi | lo][256 rows x 32 B] (SWIZZLE_32B)
  uint8_t* s_b1 = s_op + OP_BYTES;                 // [hi | lo][32 rows x 32 B]
  float* s_scale = reinterpret_cast<float*>(s_b1 + 2048);
  float* s_shift = s_scale + 64;
  float* s_shift1 = s_shift + 64;
  float* s_win = s_shift1 + 64;                    // [2 stages][256] one-channel input windows (20 x 12 used)
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_win + 512);
  uint64_t* a_full = bars;              // [SA]  leader: 8 producer-warp arrivals (both CTAs)
  uint64_t* a_empty = a_full + SA;      // [SA]  per CTA (multicast commit)
  uint64_t* b_full = a_empty + SA;      // leader: conv2 weights landed
  uint64_t* t_full = b_full + 1;        // [ACC] per CTA (multicast commit)
  uint64_t* t_empty = t_full + ACC;     // [ACC] leader: 16 epilogue-warp arrivals
  uint64_t* op_full = t_empty + ACC;    // [2]   leader: 8 producer-warp arrivals
  uint64_t* op_empty = op_full + 2;     // [2]   per CTA (multicast commit)
  uint64_t* c1_full = op_empty + 2;     // [2]   per CTA (multicast commit)
  uint64_t* c1_empty = c1_full + 2;     // [2]   leader: 8 producer-warp arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(c1_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pr_cta = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int items = (p.num_tiles + 1) / 2;

  if (threadIdx.x < 64) {
    s_scale[threadIdx.x] = 0.25f * p.scale[threadIdx.x];  // the 1/4 of the 2x2 average rides the bn2 affine (exact)
    s_shift[threadIdx.x] = 0.25f * p.shift[threadIdx.x];
    s_shift1[threadIdx.x] = p.shift1[threadIdx.x];
  }
  if (threadIdx.x >= 64 && threadIdx.x < 96) {
    // conv1 weights (bn1 scale folded in) of channel rank*32 + r -> split fp16 operand row r (SWIZZLE_32B)
    const int r = threadIdx.x - 64, ch = static_cast<int>(rank) * 32 + r;
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      // K slot 9 carries the folded bn1 shift (the operand rows hold a constant 1 there): the bias rides the GEMM
      const float v0 = (2 * t < 9) ? p.w1[ch * 9 + 2 * t] : 0.0f;
      const float v1 = (2 * t + 1 < 9) ? p.w1[ch * 9 + 2 * t + 1] : (2 * t + 1 == 9 ? p.shift1[ch] : 0.0f);
      const __half h0 = __float2half_rn(v0), h1 = __float2half_rn(v1);
      const __half l0 = __float2half_rn(v0 - __half2float(h0)), l1 = __float2half_rn(v1 - __half2float(h1));
      hi[t] = static_cast<uint32_t>(__half_as_ushort(h0)) | (static_cast<uint32_t>(__half_as_ushort(h1)) << 16);
      lo[t] = static_cast<uint32_t>(__half_as_ushort(l0)) | (static_cast<uint32_t>(__half_as_ushort(l1)) << 16);
    }
    // The 29 products hi*w_hi (10), lo*w_hi (9: the bias slot's lo is 0) and hi*w_lo (10) are packed into TWO K=16 steps
    // (the operand rows use the matching slot order, see build()):
    //   step 1: A = [hi0..hi9 | lo0..lo5]        B = [wh0..wh9 | wh0..wh5]
    //   step 2: A = [lo6 lo7 lo8 0 | hi0..hi9 | 0 0]   B = [wh6 wh7 wh8 0 | wl0..wl9 | 0 0]
    const int sw = (r >> 2) & 1;
    *reinterpret_cast<uint4*>(s_b1 + r * 32 + ((0 ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(s_b1 + r * 32 + ((1 ^ sw) << 4)) = make_uint4(hi[4], hi[0], hi[1], hi[2]);
    *reinterpret_cast<uint4*>(s_b1 + 1024 + r * 32 + ((0 ^ sw) << 4)) = make_uint4(hi[3], hi[4] & 0xFFFFu, lo[0], lo[1]);
    *reinterpret_cast<uint4*>(s_b1 + 1024 + r * 32 + ((1 ^ sw) << 4)) = make_uint4(lo[2], lo[3], lo[4], 0u);
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < SA; ++i) { mbar_init(&a_full[i], 8); mbar_init(&a_empty[i], 1); }
    mbar_init(b_full, 1);
    for (int i = 0; i < ACC; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 16); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&op_full[i], 8); mbar_init(&op_empty[i], 1);
      mbar_init(&c1_full[i], 1); mbar_init(&c1_empty[i], 8);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc2(tmem_slot, 512);
    tmem_relinquish2();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
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

  if (warp < EPI_WARP0) setmaxnreg_dec<REG_CTRL>();
  if (warp >= PROD_WARP0) setmaxnreg_inc<REG_PROD>();

  if (warp == 0) {
    // =============================== conv2 weights (resident) ================================
    if (elect_one()) {
      const uint32_t bfull_leader = map_to_cta(b_full, 0);
      if (leader) mbar_expect_tx(b_full, 2 * B2_BYTES);
      for (int tap = 0; tap < 9; ++tap)
        tma_load_2d_2sm(smem_b + tap * B2_HALF, &tmB, bfull_leader, tap * 64, static_cast<int>(rank) * 32);
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (leader CTA only) ============================
    if (leader && elect_one()) {
      constexpr uint32_t idesc2 = umma_idesc_f16(Elem16<T>::kFmt, 256, 64);
      constexpr uint32_t idesc1 = umma_idesc_f16(0, 256, 64);  // conv1 operands are fp16 whatever T is
      constexpr uint32_t a_hi = desc_hi_sw128(1280), b_hi = desc_hi_sw128(1024), d32 = desc_hi_sw32(256);
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a)), b_lo0 = desc_lo(smem_u32(smem_b));
      const uint32_t op_lo0 = desc_lo(smem_u32(s_op)), b1_hi_lo = desc_lo(smem_u32(s_b1)),
                     b1_lo_lo = desc_lo(smem_u32(s_b1 + 1024));
      mbar_wait(b_full, 0);
      tc_fence_after();
      const int n_local = (items - pr_cta + npairs - 1) / npairs;  // work items of this pair
      auto conv1 = [&](int j) {
        const int st = j & 1, ph = (j >> 1) & 1;
        mbar_wait_cluster(&op_full[st], ph);  // (CTA-scope polling + one fence.acq_rel.cluster per wait measured 1.8x slower)
        C1_STAMP(0, j, 0);
        mbar_wait_cluster(&c1_empty[st], ph ^ 1);
        C1_STAMP(0, j, 1);
        tc_fence_after();
        const uint32_t a_h = op_lo0 + st * (OP_STAGE >> 4), a_l = a_h + (8192 >> 4);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const uint32_t d = tmem_base + C1_COL0 + st * 128 + mt * 64;
          const uint32_t mo = mt * (4096 >> 4);
          umma_f16_2sm(d, desc_join(a_h + mo, d32), desc_join(b1_hi_lo, d32), idesc1, 0u);  // K step 1
          umma_f16_2sm(d, desc_join(a_l + mo, d32), desc_join(b1_lo_lo, d32), idesc1, 1u);  // K step 2
        }
        umma_commit_2sm(&c1_full[st], 3);
        umma_commit_2sm(&op_empty[st], 3);
      };
      uint32_t sa = 0, pa = 0, acc = 0, pacc = 0;
      if (n_local > 0) conv1(0);
      for (int i = 0; i < n_local; ++i) {
        if (i + 1 < n_local) conv1(i + 1);
        mbar_wait(&t_empty[acc], pacc ^ 1);
        C1_STAMP(0, i, 2);
        mbar_wait_cluster(&a_full[sa], pa);
        C1_STAMP(0, i, 3);
        tc_fence_after();
        const uint32_t d_base = tmem_base + acc * 64;
        const uint32_t a_lo = a_lo0 + sa * (kPatchStride >> 4);
        // rolled over the taps on purpose: unrolled, the 36 descriptor pairs get hoisted out of the item loop and do
        // not fit the control group's register budget
#pragma unroll 1
        for (int tr = 0; tr < 3; ++tr) {
#pragma unroll 1
          for (int tc = 0; tc < 3; ++tc) {
            const uint32_t b_lo = b_lo0 + (tr * 3 + tc) * (B2_HALF >> 4);
            const uint32_t tap_off = (tr * 10 + tc) * 8;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16_2sm(d_base, desc_join(a_lo + tap_off + k * 2, a_hi), desc_join(b_lo + k * 2, b_hi), idesc2,
                           (tr | tc | k) ? 1u : 0u);
          }
        }
        umma_commit_2sm(&a_empty[sa], 3);
        umma_commit_2sm(&t_full[acc], 3);
        C1_STAMP(0, i, 4);
        if (++sa == SA) { sa = 0; pa ^= 1; }
        if (++acc == ACC) { acc = 0; pacc ^= 1; }
      }
    }
  } else if (warp < EPI_WARP0) {
    // idle warps of the control group
  } else if (warp < PROD_WARP0) {
    // =============================== conv2 epilogue (8 warps, both CTAs) ====================
    const int quarter = warp & 3;
    const int chalf = (warp - EPI_WARP0) >> 2;
    uint32_t acc = 0, pacc = 0;
    int li = 0;
    (void)li;
    for (int w = pr_cta; w < items; w += npairs, ++li) {
      mbar_wait(&t_full[acc], pacc);
      if (warp == EPI_WARP0 && lane == 0) C1_STAMP(1, li, 0);
      tc_fence_after();
      const int tile = w * 2 + static_cast<int>(rank);
      const bool tile_ok = tile < p.num_tiles;
      int n, h0, w0;
      tile_coords(tile, n, h0, w0);
      const uint32_t taddr = tmem_base + acc * 64 + chalf * 32 + (static_cast<uint32_t>(quarter * 32) << 16);
      conv_epilogue_tile<T, 64, true, EPI_POOL>(taddr, chalf, warp, lane, s_scale, s_shift, 0, tile, tile_ok, n, h0, w0,
                                                p, nullptr, nullptr);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_light(&t_empty[acc], 0);
      if (warp == EPI_WARP0 && lane == 0) C1_STAMP(1, li, 1);
      if (++acc == ACC) { acc = 0; pacc ^= 1; }
    }
  } else {
    // =============================== conv1 operand build + TMEM drain (4 warps) ==============
    const int m_tm = (warp & 3) * 32 + lane;  // TMEM lane this thread may read = its patch row within an M-tile
    // patch rows of this thread: pr = mt*128 + m_tm (mt = 0, 1; rows >= 180 do not exist)
    int prr[2], prc[2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const int pr = mt * 128 + m_tm;
      prr[mt] = pr / 10;
      prc[mt] = pr - prr[mt] * 10;
    }
    const int grp = (warp - PROD_WARP0) >> 2;                  // producer group: owns operand / accumulator stage `grp`
    const int ptid = ((warp - PROD_WARP0) & 3) * 32 + lane;    // 0..127 within the producer group
    // the tile's 20 x 12 one-channel input window (zero outside the image = conv1's padding): two values per thread
    auto gather = [&](int tile, float (&g)[2]) {
      int n, h0, w0;
      tile_coords(tile, n, h0, w0);
      const bool tv = tile < p.num_tiles;
      const float* xn = p.x1 + static_cast<size_t>(n) * p.H * p.W;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int e = ptid + 128 * k;
        const int er = e / 12, ec = e - er * 12;
        const int hh = h0 - 2 + er, ww = w0 - 2 + ec;
        g[k] = (tv && e < 240 && hh >= 0 && hh < p.H && ww >= 0 && ww < p.W) ? __ldg(xn + hh * p.W + ww) : 0.0f;
      }
    };
    auto build = [&](int j, int tile, const float (&g)[2]) {
      const int st = j & 1, ph = (j >> 1) & 1;
      float* win = s_win + st * 256;
      if (ptid == 0) C1_STAMP(2, j, 0);
      win[ptid] = g[0];
      if (ptid < 112) win[128 + ptid] = g[1];
      int n, h0, w0;
      tile_coords(tile, n, h0, w0);
      const bool tv = tile < p.num_tiles;
      if (grp == 0) named_bar_sync(2, 128); else named_bar_sync(3, 128);  // window complete (the group's own barrier)
      if (ptid == 0) C1_STAMP(2, j, 1);
      mbar_wait(&op_empty[st], ph ^ 1);
      if (ptid == 0) C1_STAMP(2, j, 2);
      uint8_t* hi_base = s_op + st * OP_STAGE;
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        const int row = mt * 128 + m_tm;
        // a patch pixel outside the image is conv2's ZERO padding: its whole operand row (bias slot included) is zero
        const int ph_ = h0 - 1 + prr[mt], pw_ = w0 - 1 + prc[mt];
        const bool rowv = tv && row < 180 && ph_ >= 0 && ph_ < p.H && pw_ >= 0 && pw_ < p.W;
        float in[10];
#pragma unroll
        for (int dr = 0; dr < 3; ++dr)
#pragma unroll
          for (int dc = 0; dc < 3; ++dc)
            in[dr * 3 + dc] = (rowv) ? win[(prr[mt] + dr) * 12 + prc[mt] + dc] : 0.0f;
        in[9] = rowv ? 1.0f : 0.0f;
        uint32_t hi[5], lo[5];
#pragma unroll
        for (int t = 0; t < 5; ++t) {  // packed conversions: hi = rn16(v), lo = rn16(v - hi)
          const __half2 h = __floats2half2_rn(in[2 * t], in[2 * t + 1]);
          const float2 hf = __half22float2(h);
          const __half2 l = __floats2half2_rn(in[2 * t] - hf.x, in[2 * t + 1] - hf.y);
          hi[t] = *reinterpret_cast<const uint32_t*>(&h);
          lo[t] = *reinterpret_cast<const uint32_t*>(&l);
        }
        // slot order of the two K steps (see the weight rows above); lo[4] = (lo8, lo of the constant 1) = (lo8, 0)
        const int sw = (row >> 2) & 1;
        uint8_t* rp = hi_base + row * 32;
        *reinterpret_cast<uint4*>(rp + ((0 ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(rp + ((1 ^ sw) << 4)) = make_uint4(hi[4], lo[0], lo[1], lo[2]);
        *reinterpret_cast<uint4*>(rp + 8192 + ((0 ^ sw) << 4)) = make_uint4(lo[3], lo[4], hi[0], hi[1]);
        *reinterpret_cast<uint4*>(rp + 8192 + ((1 ^ sw) << 4)) = make_uint4(hi[2], hi[3], hi[4], 0u);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_light(&op_full[st], 0);
      if (ptid == 0) C1_STAMP(2, j, 3);
    };
    auto drain = [&](int j, int tile) {
      const uint32_t sa = static_cast<uint32_t>(j) % SA, pa = (static_cast<uint32_t>(j) / SA) & 1;
      const int st = j & 1, ph = (j >> 1) & 1;
      (void)tile;
      if (ptid == 0) C1_STAMP(2, j, 4);
      mbar_wait(&c1_full[st], ph);
      if (ptid == 0) C1_STAMP(2, j, 5);
      mbar_wait(&a_empty[sa], pa ^ 1);
      if (ptid == 0) C1_STAMP(2, j, 6);
      tc_fence_after();
      uint8_t* patch = smem_a + sa * kPatchStride;
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        uint32_t r[4][16];
        const uint32_t taddr = tmem_base + C1_COL0 + st * 128 + mt * 64 + (static_cast<uint32_t>((warp & 3) * 32) << 16);
#pragma unroll
        for (int u = 0; u < 4; ++u) tmem_ld16(taddr + u * 16, r[u]);
        tmem_ld_wait();
        const int pr = mt * 128 + m_tm;
        if (pr < 180) {
          // accumulators already hold conv1 + folded bn1 shift (zero for padding pixels): cvt.rn.relu packs + clamps
          uint8_t* rowp = patch + pr * 128;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            uint32_t pk[8];
#pragma unroll
            for (int q = 0; q < 8; ++q)
              pk[q] = Elem16<T>::pack2_relu(__uint_as_float(r[u][2 * q]), __uint_as_float(r[u][2 * q + 1]));
            *reinterpret_cast<uint4*>(rowp + (((2 * u) ^ (pr & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            *reinterpret_cast<uint4*>(rowp + (((2 * u + 1) ^ (pr & 7)) << 4)) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          }
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_remote_light(&a_full[sa], 0);
        mbar_arrive_remote_light(&c1_empty[st], 0);
      }
      if (ptid == 0) C1_STAMP(2, j, 7);
    };
    // software pipeline per group (tiles j = grp, grp + PG, ...): the one-channel inputs of the group's tile after next
    // are in flight while its next tile is built and its current tile drained
    float nin[2];
    auto tile_of = [&](int jj) { return (pr_cta + jj * npairs) * 2 + static_cast<int>(rank); };
    auto has = [&](int jj) { return pr_cta + jj * npairs < items; };
    int j = grp;
    if (has(j)) {
      gather(tile_of(j), nin);
      build(j, tile_of(j), nin);
      if (has(j + PG)) gather(tile_of(j + PG), nin);
    }
    for (; has(j); j += PG) {
      // drain first: conv2(j) waits for it, while the group's next operand (conv1(j + PG), queued behind conv2(j - 1) in
      // the tensor pipe) has a whole conv2 of slack
      drain(j, tile_of(j));
      if (has(j + PG)) {
        build(j + PG, tile_of(j + PG), nin);
        if (has(j + 2 * PG)) gather(tile_of(j + 2 * PG), nin);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, 512);
  }
}


// ---------------------------------------------------------------------------------------------
// tcgen05 conv / linear launch
// ---------------------------------------------------------------------------------------------
template <typename T, int CIN, int BN, int NT, int SA, int SB>
static int launch_cfg(const CUtensorMap& tmA, const CUtensorMap& tmB, const ConvParams& p, cudaStream_t stream) {
  using Cfg = ConvCfg<CIN, BN, NT, SA, SB>;
  auto kern = conv_umma_kernel<T, CIN, BN, NT, SA, SB>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
    return SED_ERR_CUDA;
  }
  const long items = static_cast<long>((p.num_tiles + NT - 1) / NT) * p.nslices;
  const int grid = items < num_sms() ? static_cast<int>(items) : num_sms();
  kern<<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(tmA, tmB, tmA, p);  // the third map is not read
  e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("conv_umma launch: %s", cudaGetErrorString(e));
    return SED_ERR_CUDA;
  }
  return SED_OK;
}

template <typename T, int CIN, int BN, int EPI, int SA, int ACC, bool BRES, int NT, int SB>
static int launch_pair(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, const ConvParams& p,
                       cudaStream_t stream) {
  using Cfg = Conv2Cfg<CIN, BN, EPI, SA, ACC, BRES, NT, SB>;
  auto kern = conv_umma2_kernel<T, CIN, BN, EPI, SA, ACC, BRES, NT, SB>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(pair, smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
    return SED_ERR_CUDA;
  }
  const int items = (p.num_tiles + 2 * NT - 1) / (2 * NT);
  int grid;
  if (BRES) {
    int pairs_per_slice = (num_sms() / 2) / p.nslices;
    if (pairs_per_slice > items) pairs_per_slice = items;
    if (pairs_per_slice < 1) pairs_per_slice = 1;
    grid = 2 * pairs_per_slice * p.nslices;
  } else {
    const long work = static_cast<long>(items) * p.nslices;
    const int pairs = num_sms() / 2;
    grid = 2 * static_cast<int>(work < pairs ? work : pairs);
  }
  kern<<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(tmA, tmB, tmO, p);
  e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("conv_umma2 launch: %s", cudaGetErrorString(e));
    return SED_ERR_CUDA;
  }
  return SED_OK;
}

template <typename T>
static int conv3x3_dispatch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, ConvParams& p,
                            int cin, int cout, int mode, cudaStream_t stream) {
  // (cin, cout, mode) are the seven tensor-core layers of Cnn_9layers (SURVEY.md 8a, row a7), all on CTA pairs.
  // weights resident: each CTA of a pair holds half of the BN rows of its Cout slice
  if (cin == 64 && cout == 64 && mode == EPI_POOL) { p.nslices = 1; return launch_pair<T, 64, 64, EPI_POOL, 6, 4, true, 1, 1>(tmA, tmB, tmO, p, stream); }
  if (cin == 64 && cout == 128 && mode == EPI_STORE) { p.nslices = 1; return launch_pair<T, 64, 128, EPI_STORE, 4, 4, true, 1, 1>(tmA, tmB, tmO, p, stream); }
  if (cin == 128 && cout == 128 && mode == EPI_POOL) { p.nslices = 1; return launch_pair<T, 128, 128, EPI_POOL, 3, 2, true, 1, 1>(tmA, tmB, tmO, p, stream); }
  if (cin == 128 && cout == 256 && mode == EPI_STORE) { p.nslices = 2; return launch_pair<T, 128, 128, EPI_STORE, 2, 2, true, 1, 1>(tmA, tmB, tmO, p, stream); }
  // streamed weights: each CTA loads half of every 256-row weight block, two pixel tiles per CTA share it
  if (cin == 256 && cout == 256 && mode == EPI_POOL) { p.nslices = 2; return launch_pair<T, 256, 128, EPI_POOL, 2, 2, false, 2, 6>(tmA, tmB, tmO, p, stream); }
  if (cin == 256 && cout == 512 && mode == EPI_STORE) { p.nslices = 4; return launch_pair<T, 256, 128, EPI_STORE, 2, 2, false, 2, 6>(tmA, tmB, tmO, p, stream); }
  if (cin == 512 && cout == 512 && mode == EPI_FREQMEAN) { p.nslices = 4; return launch_pair<T, 512, 128, EPI_FREQMEAN, 2, 2, false, 2, 6>(tmA, tmB, tmO, p, stream); }  // + freq mean, models.py:668
  set_error("conv3x3: unsupported layer (cin=%d, cout=%d, mode=%d)", cin, cout, mode);
  return SED_ERR_UNSUPPORTED;
}

int conv3x3_launch(const void* x, int NB, int H, int W, int cin, const void* wpacked, const float* scale,
                   const float* shift, int cout, int mode, void* out, void* out_f32, long out_sn, long out_sh,
                   int dtype, cudaStream_t stream) {
  if (NB <= 0 || H <= 0 || W <= 0 || (W % 8) != 0 || (cin % 64) != 0) {
    set_error("conv3x3: bad shape NB=%d H=%d W=%d cin=%d", NB, H, W, cin);
    return SED_ERR_BAD_SHAPE;
  }
  if (mode == EPI_FREQMEAN && W != 8) {
    set_error("conv3x3: freq-mean epilogue needs W == 8 (got %d)", W);
    return SED_ERR_BAD_SHAPE;
  }
  if (mode == EPI_POOL && (W % 16) != 0) {
    set_error("conv3x3: pooling epilogue needs W %% 16 == 0 (got %d)", W);
    return SED_ERR_BAD_SHAPE;
  }
  CUtensorMap tmA, tmB;
  {
    const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)W, (uint64_t)H, (uint64_t)NB};
    const uint64_t str[3] = {(uint64_t)cin * 2, (uint64_t)W * cin * 2, (uint64_t)H * W * cin * 2};
    const uint32_t box[4] = {64, 10, 18, 1};  // one haloed 16 x 8 pixel tile
    int rc = make_map(&tmA, dtype, 4, const_cast<void*>(x), dims, str, box);
    if (rc) return rc;
  }
  {
    const uint64_t dims[2] = {(uint64_t)9 * cin, (uint64_t)cout};
    const uint64_t str[1] = {(uint64_t)9 * cin * 2};
    const uint32_t box[2] = {64, cout == 64 ? 32u : 64u};  // each CTA of a pair loads half of the BN = 64 | 128 rows
    int rc = make_map(&tmB, dtype, 2, const_cast<void*>(wpacked), dims, str, box);
    if (rc) return rc;
  }
  CUtensorMap tmO = tmA;  // only read by the EPI_STORE epilogue
  if (mode == EPI_STORE) {
    const uint64_t dims[4] = {(uint64_t)cout, (uint64_t)W, (uint64_t)H, (uint64_t)NB};
    const uint64_t str[3] = {(uint64_t)cout * 2, (uint64_t)W * cout * 2, (uint64_t)H * W * cout * 2};
    const uint32_t box[4] = {64, 8, 16, 1};
    int rc = make_map(&tmO, dtype, 4, out, dims, str, box);
    if (rc) return rc;
  }
  ConvParams p{};
  p.NB = NB; p.H = H; p.W = W;
  p.tiles_h = (H + 15) / 16;
  p.tiles_w = W / 8;
  p.num_tiles = NB * p.tiles_h * p.tiles_w;
  {
    const unsigned long long per_img = static_cast<unsigned long long>(p.tiles_h) * p.tiles_w;
    if (per_img * (static_cast<unsigned long long>(p.num_tiles) + 4096) >= (1ull << 32)) {
      set_error("conv3x3: too many tiles for the index arithmetic (NB=%d H=%d W=%d)", NB, H, W);
      return SED_ERR_BAD_SHAPE;
    }
    p.magic_img = per_img > 1 ? static_cast<uint32_t>(((1ull << 32) + per_img - 1) / per_img) : 0u;
    p.magic_w = p.tiles_w > 1 ? static_cast<uint32_t>(((1ull << 32) + p.tiles_w - 1) / p.tiles_w) : 0u;
  }
  p.cout = cout;
  p.scale = scale; p.shift = shift;
  p.out = out; p.out2 = (mode == EPI_FREQMEAN) ? out_f32 : nullptr;
  p.M = 0; p.ldc = 0; p.relu = 1; p.tblock = 0;
  p.out_sn = (mode == EPI_FREQMEAN && out_sn > 0) ? out_sn : H;
  p.out_sh = (mode == EPI_FREQMEAN && out_sh > 0) ? out_sh : 1;
#ifdef SED_PROFILE
  {
    const char* e = getenv("SED_CONV_DBG");
    p.dbg = e ? atoi(e) : 0;
  }
#endif
  if (dtype == 0) return conv3x3_dispatch<__half>(tmA, tmB, tmO, p, cin, cout, mode, stream);
  if (dtype == 1) return conv3x3_dispatch<__nv_bfloat16>(tmA, tmB, tmO, p, cin, cout, mode, stream);
  set_error("conv3x3: dtype must be 0 (fp16) or 1 (bf16)");
  return SED_ERR_UNSUPPORTED;
}

// conv_block1 as one kernel: conv1 (1 -> 64, split-fp16 tensor-core GEMM) feeds conv2's tensor-core operand through
// shared memory; the [NB, H, 64, 64] intermediate never exists in HBM.
int conv_block1_launch(const float* x, int NB, int H, int W, const float* w1s, const float* shift1, const void* w2packed,
                       const float* scale2, const float* shift2, void* out, int dtype, cudaStream_t stream) {
  if (NB <= 0 || H <= 0 || W <= 0 || (W % 16) != 0) {
    set_error("conv_block1: bad shape NB=%d H=%d W=%d (W %% 16 == 0)", NB, H, W);
    return SED_ERR_BAD_SHAPE;
  }
  CUtensorMap tmB;
  {
    const uint64_t dims[2] = {(uint64_t)9 * 64, (uint64_t)64};
    const uint64_t str[1] = {(uint64_t)9 * 64 * 2};
    const uint32_t box[2] = {64, 32};  // each CTA of a pair loads half of the 64 weight rows
    int rc = make_map(&tmB, dtype, 2, const_cast<void*>(w2packed), dims, str, box);
    if (rc) return rc;
  }
  ConvParams p{};
  p.NB = NB; p.H = H; p.W = W;
  p.tiles_h = (H + 15) / 16;
  p.tiles_w = W / 8;
  p.num_tiles = NB * p.tiles_h * p.tiles_w;
  {
    const unsigned long long per_img = static_cast<unsigned long long>(p.tiles_h) * p.tiles_w;
    if (per_img * (static_cast<unsigned long long>(p.num_tiles) + 4096) >= (1ull << 32)) {
      set_error("conv_block1: too many tiles for the index arithmetic (NB=%d H=%d W=%d)", NB, H, W);
      return SED_ERR_BAD_SHAPE;
    }
    p.magic_img = per_img > 1 ? static_cast<uint32_t>(((1ull << 32) + per_img - 1) / per_img) : 0u;
    p.magic_w = p.tiles_w > 1 ? static_cast<uint32_t>(((1ull << 32) + p.tiles_w - 1) / p.tiles_w) : 0u;
  }
  p.cout = 64; p.nslices = 1;
  p.scale = scale2; p.shift = shift2;
  p.out = out; p.out2 = nullptr;
  p.relu = 1;
  p.out_sn = H; p.out_sh = 1;
  p.x1 = x; p.w1 = w1s; p.shift1 = shift1;
#ifdef SED_PROFILE
  {
    const char* e = getenv("SED_CONV_DBG");
    p.dbg = e ? atoi(e) : 0;
  }
#endif
  if (dtype != 0 && dtype != 1) {
    set_error("conv_block1: dtype must be 0 (fp16) or 1 (bf16)");
    return SED_ERR_UNSUPPORTED;
  }
  int pairs = num_sms() / 2;
  const int items = (p.num_tiles + 1) / 2;
  if (pairs > items) pairs = items;
  cudaError_t e;
  if (dtype == 0) {
    e = cudaFuncSetAttribute(conv_block1_tc_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             c1tc::SMEM_BYTES);
    if (e == cudaSuccess)
      conv_block1_tc_kernel<__half><<<2 * pairs, c1tc::THREADS, c1tc::SMEM_BYTES, stream>>>(tmB, p);
  } else {
    e = cudaFuncSetAttribute(conv_block1_tc_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             c1tc::SMEM_BYTES);
    if (e == cudaSuccess)
      conv_block1_tc_kernel<__nv_bfloat16><<<2 * pairs, c1tc::THREADS, c1tc::SMEM_BYTES, stream>>>(tmB, p);
  }
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("conv_block1 launch: %s", cudaGetErrorString(e));
    return SED_ERR_CUDA;
  }
  return SED_OK;
}

#ifdef SED_C1_STAMPS
extern "C" int sed_debug_c1_stamps(long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, g_c1_stamps, sizeof(g_c1_stamps)) == cudaSuccess ? 0 : 1;
}
#endif

int linear_launch(const void* a16, long M, int K, const void* w16, const float* bias, int N, int relu, float* out,
                  void* out16, int out_layout, int dtype, cudaStream_t stream, void* out_lo, int lo_cols) {
  if (out_lo != nullptr && (out16 == nullptr || lo_cols <= 0 || lo_cols > N || (lo_cols % 128) != 0 || N > 1536)) {
    set_error("linear: the 16-bit residual output needs the 16-bit output, lo_cols a multiple of 128 <= N <= 1536");
    return SED_ERR_BAD_SHAPE;
  }
  if (out_layout != 0 && (out_layout != 1 || out16 != nullptr || (M % 128) != 0)) {
    set_error("linear: out_layout must be 0 (row-major) or 1 (128-row transposed blocks: M %% 128 == 0, no 16-bit copy)");
    return SED_ERR_UNSUPPORTED;
  }
  if (out == nullptr && (out16 == nullptr || out_layout != 0)) {
    set_error("linear: a NULL float32 output needs the 16-bit output and the row-major layout");
    return SED_ERR_NULL;
  }
  if (M <= 0 || (N % 128) != 0 || N > 512 * 8) {
    set_error("linear: bad shape M=%ld N=%d K=%d", M, N, K);
    return SED_ERR_BAD_SHAPE;
  }
  if (K != 512 && K != 256) {
    set_error("linear: K must be 256 or 512 (got %d)", K);
    return SED_ERR_UNSUPPORTED;
  }
  CUtensorMap tmA, tmB;
  {
    const uint64_t dims[2] = {(uint64_t)K, (uint64_t)M};
    const uint64_t str[1] = {(uint64_t)K * 2};
    const uint32_t box[2] = {64, 128};
    int rc = make_map(&tmA, dtype, 2, const_cast<void*>(a16), dims, str, box);
    if (rc) return rc;
  }
  {
    const uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
    const uint64_t str[1] = {(uint64_t)K * 2};
    const uint32_t box[2] = {64, 128};
    int rc = make_map(&tmB, dtype, 2, const_cast<void*>(w16), dims, str, box);
    if (rc) return rc;
  }
  // the epilogue caches the bias of at most 1536 columns: wider outputs run in column panels.  One launch for the GRU
  // input projection (N = 1536): the 12 column slices of an A tile are consecutive work items, so the tile comes from
  // HBM once instead of once per panel
  constexpr int kPanel = 1536;
  int rc = SED_OK;
  for (int n0 = 0; n0 < N && rc == SED_OK; n0 += kPanel) {
    const int npanel = (N - n0) < kPanel ? (N - n0) : kPanel;
    CUtensorMap tmBp = tmB;
    if (n0 != 0) {
      const uint64_t dims[2] = {(uint64_t)K, (uint64_t)npanel};
      const uint64_t str[1] = {(uint64_t)K * 2};
      const uint32_t box[2] = {64, 128};
      rc = make_map(&tmBp, dtype, 2, (char*)const_cast<void*>(w16) + (size_t)n0 * K * 2, dims, str, box);
      if (rc) return rc;
    }
    ConvParams p{};
    p.num_tiles = (int)((M + 127) / 128);
    p.cout = npanel;
    p.nslices = npanel / 128;
    p.scale = nullptr;
    p.shift = bias ? bias + n0 : nullptr;
    p.out = out == nullptr ? nullptr : out_layout ? out + (size_t)n0 * 128 : out + n0;  // transposed blocks: float4 column n0/4 = +n0/4*128*4 floats
    p.out2 = out16 ? (void*)((char*)out16 + (size_t)n0 * 2) : nullptr;
    p.M = (int)M; p.ldc = N; p.relu = relu; p.tblock = out_layout;
    p.out3 = out_lo; p.lo_cols = lo_cols;
    p.out_sn = 0; p.out_sh = 0;
    if (K == 512 && M >= 128 * 296) {
      // large M (the GRU input projection / QKV projection of a whole batch): the kernel is bound by L2 -> shared
      // memory operand traffic (A 128 KB + B 128 KB per 128 x 128 tile = 125 B/clk/SM); two row tiles per work item
      // share every B block (94 B/clk/SM)
      rc = dtype == 0 ? launch_cfg<__half, 512, 128, 2, 4, 4>(tmA, tmBp, p, stream)
                      : launch_cfg<__nv_bfloat16, 512, 128, 2, 4, 4>(tmA, tmBp, p, stream);
    } else if (K == 512) {
      rc = dtype == 0 ? launch_cfg<__half, 512, 128, 1, 4, 4>(tmA, tmBp, p, stream)
                      : launch_cfg<__nv_bfloat16, 512, 128, 1, 4, 4>(tmA, tmBp, p, stream);
    } else {
      rc = dtype == 0 ? launch_cfg<__half, 256, 128, 1, 4, 4>(tmA, tmBp, p, stream)
                      : launch_cfg<__nv_bfloat16, 256, 128, 1, 4, 4>(tmA, tmBp, p, stream);
    }
  }
  return rc;
}

}  // namespace sed
