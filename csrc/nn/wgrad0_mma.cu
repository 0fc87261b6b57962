// Layer-1 weight gradient from the POOLED gradient on the tensor cores (warp-level mma.sync): the gather of
// wgrad_gather.cu rewritten as four masked GEMMs.
//
// After ReLU + 2x2 max-pool the conv-grid gradient has one non-zero per window and channel, at the arg-max
// position code c = (dy, dx). Splitting the pooled gradient by code,
//     G_c[px, co] = g[px, co]  if unit (px, co) is active and its arg-max code is c,  else 0,
// turns the data-dependent gather into
//     dW[(r, q, ci), co] = sum_c sum_px  X[(2i + dy + r, 2j + dx + q), ci] * G_c[px, co],        px = (b, i, j)
// i.e. for each code a GEMM over the pooled pixels with an A operand that is a plain strided view of the input.
// With the s-packed layer-1 input (channels = pixels (x, x+1, x+2) x 3, nn_kernels.cu) the 16 channels of pixel
// (2j + dx) ARE the (q, ci) rows of filter row r, so M = 3 x 16, N = 32, K = 4 x pooled pixels: 0.125 warp
// instructions per (window, channel) against 2.6 for the FP32-pipe gather (profiles/ncu_summary.md prof_gather:
// 43 M warp instructions, issue-bound at 66 us). The masks are built once per strip with byte-wise SIMD compares
// (4 codes x 16 B per 8 channels) and never leave shared memory.
//
//   * one CTA walks a contiguous run of pooled rows ("strips"): consecutive strips of an image share two of
//     their four input rows, kept in a six-slot ring. One thread issues the copies of the next strip while the
//     current one is multiplied: each input row is one TMA tensor copy ([pixel pairs][2 x 16 ch], SWIZZLE_64B),
//     gradient and codes are plain bulk copies; all of them complete on one mbarrier per strip parity;
//   * both operands are read with ldmatrix.trans from "K rows, M/N contiguous" tiles whose 16-byte chunks are
//     XOR-swizzled so that every phase touches 8 distinct bank groups (A: the TMA swizzle, rows 64 B apart;
//     B: [pixel][32 co] rows at 64 B, written by the mask pass with the same pattern);
//   * the mask pass uses PRMT as an 8-entry table: the code bytes, nibble-duplicated by one multiply, are the
//     selector, the table is 0xFF at entry 4 + c, so one instruction yields the 16-bit masks of two channels;
//   * 8 warps = 8 x 16 pooled pixels of a strip; each keeps the full 48 x 32 fp32 tile (48 registers). At the end
//     every warp parks its tile in shared memory (no atomics: fp32 shared atomics are CAS loops on this part and
//     cost 29 % of the first version), the tiles are summed in warp order and each CTA stores its 28 x 32 partial
//     sums; wgrad0_sum_kernel adds them, in CTA order, to the split-K buffer the other weight-gradient kernels
//     use (same result on every run, unlike an fp32 RED per CTA). The bias gradient is the sum of the active g,
//     taken in the mask pass.
//
// (Why mma.sync and not tcgen05 here: the B operand is produced by the CUDA cores, M x N is 48 x 32 and the
// kernel is bound by the 116 MB it reads; the legacy tensor path needs no TMEM / descriptor round trip for that.)
// Reference semantics: Keras Conv2D/MaxPooling2D backward of the first block (FLPyfhelin.py:120-121).
#include <cuda_bf16.h>

#include <cstdlib>
#include <stdexcept>

#include "../he/kernels.h"
#include "launch.cuh"
#include "nn.h"
#include "tc_common.cuh"

namespace hefl {
namespace nn {

namespace {

using namespace hefl::tc;

constexpr int kT = 256;                 // 8 warps
constexpr int kPx = 128;                // pooled pixels per strip tile (Wp <= 128)
constexpr int kSlot = 8192;             // one input row: W <= 256 pixels x 32 B
constexpr int kRing = 6;
constexpr int kGst = kPx * 64;          // staged g of a strip      [px][32] bf16
constexpr int kCst = kPx * 32;          // staged codes of a strip  [px][32] u8
constexpr int kGs = kPx * 64;           // one masked tile
constexpr int kBarOff = kRing * kSlot + 2 * kGst + 2 * kCst + 4 * kGs;
constexpr int kSmem = kBarOff + 64;     // 104 KB -> 2 CTAs / SM
constexpr int kPartStride = 40;         // floats per row of a parked accumulator tile (bank spread)
constexpr int kOut = 28 * 32;           // useful gradient elements: 27 (r, q, ci) rows + the bias row, x 32 co

// dW32 row of partial-sum row ``row``: tap * CK + ci for the 27 weight rows, 9 * CK for the bias
__device__ __forceinline__ int wgrad0_out_row(int row) {
  if (row == 27) return 9 * 16;
  const int r = row / 9, m = row - r * 9, q = m / 3, ci = m - q * 3;
  return (r * 3 + q) * 16 + ci;
}
constexpr int kPart = 48 * kPartStride + 32;   // one warp's tile + its bias sums
static_assert(8 * kPart * 4 <= kBarOff, "parked tiles must fit in the operand buffers");

__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void ldsm4t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(kT, 2)
wgrad0_mma_kernel(const __grid_constant__ CUtensorMap tmX, const __nv_bfloat16* __restrict__ g,
                  const uint8_t* __restrict__ amax, float* __restrict__ part, int B, int H, int W, int Hp, int Wp) {
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* ring = sm;
  uint8_t* gst = ring + kRing * kSlot;
  uint8_t* cst = gst + 2 * kGst;
  uint8_t* Gs = cst + 2 * kCst;
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + kBarOff);      // [2]: everything strip s needs, by strip parity
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // stale / never-written shared memory is multiplied by zero masks: it has to be finite
  for (int i = tid; i < (kRing * kSlot) / 16; i += kT) reinterpret_cast<uint4*>(ring)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (tid == 0) {
    prefetch_tmap(&tmX);
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  fence_proxy_async();                 // the zeros (generic proxy) before the TMA writes (async proxy)
  __syncthreads();
  pdl_prologue();

  const long long S = (long long)B * Hp;
  const int s0 = (int)(S * blockIdx.x / gridDim.x), s1 = (int)(S * (blockIdx.x + 1) / gridDim.x);
  const uint32_t row_bytes = (uint32_t)W * 32u, g_bytes = (uint32_t)Wp * 64u, c_bytes = (uint32_t)Wp * 32u;
  const int pairs = W >> 1;

  float acc[3][4][4];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int n = 0; n < 4; ++n) acc[r][n][0] = acc[r][n][1] = acc[r][n][2] = acc[r][n][3] = 0.f;
  float bsum[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) bsum[e] = 0.f;

  // lane-constant pieces of the ldmatrix addresses
  const int mq = lane >> 3, li = lane & 7;
  const int j0 = warp * 16;
  // A (slot = [pixel pair j][dx][16 ch], 16-byte chunk index XOR (j >> 1) & 3): matrices (k-half 0, m-half 0),
  // (0, 1), (1, 0), (1, 1) = a0..a3 of m16n8k16
  const int ja = j0 + (mq >> 1) * 8 + li;
  const uint32_t a_off0 = ja * 64 + (((0 + (mq & 1)) ^ ((ja >> 1) & 3)) << 4);      // dx = 0
  const uint32_t a_off1 = ja * 64 + (((2 + (mq & 1)) ^ ((ja >> 1) & 3)) << 4);      // dx = 1
  // B: matrices (k-half 0, n-tile nb), (1, nb), (0, nb + 1), (1, nb + 1)
  const int pb = j0 + (mq & 1) * 8 + li;
  const uint32_t b_off0 = pb * 64 + ((((mq >> 1) + 0) ^ ((pb >> 1) & 3)) << 4);
  const uint32_t b_off2 = pb * 64 + ((((mq >> 1) + 2) ^ ((pb >> 1) & 3)) << 4);
  const uint32_t ring_u = smem_u32(ring), Gs_u = smem_u32(Gs);

  int head = 0;
  bool pref = false;                                         // strip s was requested during strip s - 1
  for (int s = s0; s < s1; ++s) {
    const int b = s / Hp, i = s - b * Hp;
    const int par = (s - s0) & 1;
    if (!pref) head = 0;
    const bool pref_next = (s + 1 < s1) && (i + 1 < Hp);
    if (tid == 0) {
      if (!pref) {                                           // first strip of the CTA or of an image: all of it, now
        mbar_expect_tx(&full[par], 4 * row_bytes + g_bytes + c_bytes);
#pragma unroll
        for (int r = 0; r < 4; ++r) tma_load_2d(ring + r * kSlot, &tmX, 0, (b * H + 2 * i + r) * pairs, &full[par]);
        bulk_load(smem_u32(gst + par * kGst), g + (size_t)s * Wp * 32, g_bytes, &full[par]);
        bulk_load(smem_u32(cst + par * kCst), amax + (size_t)s * Wp * 32, c_bytes, &full[par]);
      }
      if (pref_next) {                                       // the next strip: two new rows, its gradient and codes
        const int q = par ^ 1;
        int sl4 = head + 4, sl5 = head + 5;
        sl4 = sl4 >= kRing ? sl4 - kRing : sl4;
        sl5 = sl5 >= kRing ? sl5 - kRing : sl5;
        mbar_expect_tx(&full[q], 2 * row_bytes + g_bytes + c_bytes);
        tma_load_2d(ring + sl4 * kSlot, &tmX, 0, (b * H + 2 * i + 4) * pairs, &full[q]);
        tma_load_2d(ring + sl5 * kSlot, &tmX, 0, (b * H + 2 * i + 5) * pairs, &full[q]);
        bulk_load(smem_u32(gst + q * kGst), g + (size_t)(s + 1) * Wp * 32, g_bytes, &full[q]);
        bulk_load(smem_u32(cst + q * kCst), amax + (size_t)(s + 1) * Wp * 32, c_bytes, &full[q]);
      }
    }
    mbar_wait(&full[par], ((s - s0) >> 1) & 1);

    // masks: item = (pooled pixel, 8 channels)
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int item = tid + it * kT;
      const int px = item >> 2, ch = item & 3;
      uint4 gv = make_uint4(0u, 0u, 0u, 0u);
      uint2 cv = make_uint2(0u, 0u);
      if (px < Wp) {
        gv = *reinterpret_cast<const uint4*>(gst + par * kGst + px * 64 + ch * 16);
        cv = *reinterpret_cast<const uint2*>(cst + par * kCst + px * 32 + ch * 8);
      }
      const uint32_t dsto = px * 64 + ((ch ^ ((px >> 1) & 3)) << 4);
      // selector nibbles (code, code) per channel: PRMT looks the mask byte up in {0,0,0,0, table}
      const uint32_t u0 = (cv.x & 0x07070707u) * 0x11u, u1 = (cv.y & 0x07070707u) * 0x11u;
      const uint32_t u0h = u0 >> 16, u1h = u1 >> 16;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint32_t tbl = 0xFFu << (8 * c);               // entry 4 + c: active and arg-max at position c
        uint4 o;
        o.x = gv.x & __byte_perm(0u, tbl, u0);
        o.y = gv.y & __byte_perm(0u, tbl, u0h);
        o.z = gv.z & __byte_perm(0u, tbl, u1);
        o.w = gv.w & __byte_perm(0u, tbl, u1h);
        *reinterpret_cast<uint4*>(Gs + c * kGs + dsto) = o;
      }
      {   // bias gradient: every active unit, whatever its position (entries 4..7)
        const uint32_t w0 = gv.x & __byte_perm(0u, 0xFFFFFFFFu, u0), w1 = gv.y & __byte_perm(0u, 0xFFFFFFFFu, u0h);
        const uint32_t w2 = gv.z & __byte_perm(0u, 0xFFFFFFFFu, u1), w3 = gv.w & __byte_perm(0u, 0xFFFFFFFFu, u1h);
        bsum[0] += __uint_as_float(w0 << 16); bsum[1] += __uint_as_float(w0 & 0xFFFF0000u);
        bsum[2] += __uint_as_float(w1 << 16); bsum[3] += __uint_as_float(w1 & 0xFFFF0000u);
        bsum[4] += __uint_as_float(w2 << 16); bsum[5] += __uint_as_float(w2 & 0xFFFF0000u);
        bsum[6] += __uint_as_float(w3 << 16); bsum[7] += __uint_as_float(w3 & 0xFFFF0000u);
      }
    }
    __syncthreads();

    if (j0 < Wp) {                                           // warp-uniform
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int dy = c >> 1;
        uint32_t bq[2][4];
        ldsm4t(bq[0], Gs_u + c * kGs + b_off0);
        ldsm4t(bq[1], Gs_u + c * kGs + b_off2);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          int slot = head + dy + r;
          slot = slot >= kRing ? slot - kRing : slot;
          uint32_t a[4];
          ldsm4t(a, ring_u + slot * kSlot + ((c & 1) ? a_off1 : a_off0));
          mma16816(acc[r][0], a, bq[0][0], bq[0][1]);
          mma16816(acc[r][1], a, bq[0][2], bq[0][3]);
          mma16816(acc[r][2], a, bq[1][0], bq[1][1]);
          mma16816(acc[r][3], a, bq[1][2], bq[1][3]);
        }
      }
    }
    __syncthreads();                                         // ring slots / masked tiles / staging are free again
    head = head + 2 >= kRing ? head + 2 - kRing : head + 2;
    pref = pref_next;
  }

  // every warp parks its tile (all copies have landed: the last strip requests nothing), then a plain sum
  float* tiles = reinterpret_cast<float*>(sm);
  {
    float* mine = tiles + warp * kPart;
    const int gq = lane >> 2, tq = lane & 3;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        const int col = n * 8 + 2 * tq;
        *reinterpret_cast<float2*>(mine + (r * 16 + gq) * kPartStride + col) = make_float2(acc[r][n][0], acc[r][n][1]);
        *reinterpret_cast<float2*>(mine + (r * 16 + gq + 8) * kPartStride + col) = make_float2(acc[r][n][2], acc[r][n][3]);
      }
#pragma unroll
    for (int e = 0; e < 8; ++e) {                            // lanes with the same (lane & 3) hold the same 8 channels
      float v = bsum[e];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      if (lane < 4) mine[48 * kPartStride + lane * 8 + e] = v;
    }
  }
  __syncthreads();
  for (int idx = tid; idx < kOut; idx += kT) {
    const int row = idx >> 5, co = idx & 31;
    int src;
    if (row < 27) {
      const int r = row / 9, m = row - r * 9;
      src = (r * 16 + m) * kPartStride + co;
    } else {
      src = 48 * kPartStride + co;                           // bias sums
    }
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += tiles[w * kPart + src];
    part[(size_t)blockIdx.x * kOut + idx] = v;
  }
}

// dW[wgrad0_out_row(row)][co] += sum of the CTAs' partial sums, in CTA order (one block per row)
// (32 x kSumRows threads per row: few dependent L2 round trips per thread, on the tail of the training step)
constexpr int kSumRows = 32;
__global__ void __launch_bounds__(32 * kSumRows) wgrad0_sum_kernel(const float* __restrict__ part, int splits,
                                                                   float* __restrict__ dW) {
  __shared__ float col[kSumRows][32];
  pdl_prologue();
  const int idx = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
#pragma unroll 8
  for (int s = threadIdx.y; s < splits; s += kSumRows) acc += part[(size_t)s * kOut + idx];
  col[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0) {
    float v = col[0][threadIdx.x];
#pragma unroll
    for (int y = 1; y < kSumRows; ++y) v += col[y][threadIdx.x];
    dW[wgrad0_out_row(blockIdx.x) * 32 + threadIdx.x] += v;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// X viewed as [pixel pairs][2 x 16 channels]: one box = one image row, 64-byte swizzle
CUtensorMap make_row_map(const void* X, uint64_t pairs_total, uint32_t pairs_per_row) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p)
      throw std::runtime_error("cuTensorMapEncodeTiled not available");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  CUtensorMap m;
  cuuint64_t dims[2] = {32, pairs_total};
  cuuint64_t strides[1] = {64};
  cuuint32_t box[2] = {32, pairs_per_row};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(X), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled(wgrad0 rows) failed");
  return m;
}

}  // namespace

bool wgrad0_mma_supported(int W, int Wp, int CK, int Ci, int Co) {
  static const bool on = []() { const char* e = std::getenv("HEFL_WGRAD0_MMA"); return !(e && e[0] == '0'); }();
  return on && CK == 16 && Ci <= 3 && Co == 32 && W <= 256 && (W & 1) == 0 && Wp <= kPx && Wp >= 1;
}

static int wgrad0_mma_grid(int B, int Hp) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  return sms * 2 < B * Hp ? sms * 2 : B * Hp;
}

size_t wgrad0_mma_part_floats(int B, int Hp) { return (size_t)wgrad0_mma_grid(B, Hp) * kOut; }

void wgrad0_mma(const void* X, const void* g, const uint8_t* amax, float* dW, float* part, int B, int H, int W, int Hp,
                int Wp, cudaStream_t st) {
  static bool attrs = false;
  if (!attrs) {
    cudaFuncSetAttribute(wgrad0_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    cudaFuncSetAttribute(wgrad0_mma_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    attrs = true;
  }
  const CUtensorMap tmX = make_row_map(X, (uint64_t)B * H * (W / 2), (uint32_t)(W / 2));
  const int grid = wgrad0_mma_grid(B, Hp);
  launch_pdl(wgrad0_mma_kernel, dim3(grid), dim3(kT), kSmem, st, tmX, reinterpret_cast<const __nv_bfloat16*>(g), amax,
             part, B, H, W, Hp, Wp);
  hefl::cuda::note_launch();
  launch_pdl(wgrad0_sum_kernel, dim3(kOut / 32), dim3(32, kSumRows), 0, st, part, grid, dW);
  hefl::cuda::note_launch();
}

}  // namespace nn
}  // namespace hefl
