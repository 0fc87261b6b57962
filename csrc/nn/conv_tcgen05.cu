// tcgen05 / TMEM / TMA implicit-GEMM 3x3 convolution for sm_100a (SURVEY.md K13-K15).
//
// Activations are NHWC bf16 viewed as a 2-D matrix [P = B*H*W pixels, C channels]. A 3x3 valid
// convolution is then 9 "tap" GEMMs whose A operand is the SAME matrix shifted by
// r*W + s rows:   Y[m, :] = sum_{r,s} X[m + r*W + s, :] * W[r,s]^T   (m on the input grid; rows
// with h >= H-2 or w >= W-2 are garbage and masked). Each tap's A tile is therefore one plain
// 2-D TMA box — no im2col buffer, no gather.
//
//   conv_fwd_pool : per CTA tile = 2 image rows x 128 columns (two TMEM accumulators) so that the
//                   epilogue does bias + ReLU + 2x2 max-pool + argmax straight out of TMEM (vertical
//                   max in-thread across the two accumulators, horizontal max by one shuffle) and
//                   writes only the pooled tensor (4x less HBM traffic than the conv output).
//   conv_dgrad    : dX[m,:] = sum_taps dY[m - off, :] * W[r,s]   (same kernel, negative offsets,
//                   plain bf16 store).
//   conv_wgrad    : dW[r,s] = sum_m X[m+off,:]^T dY[m,:]. Both operands are consumed in their
//                   native [P, C] layout as MN-major UMMA operands (pixels = K), so no transposed
//                   copies exist; taps are stacked along M (128/C tap atoms per MMA group), split-K
//                   over pixels: per-CTA partial sums, added to a [9*C+1, Co] buffer in a fixed order
//                   (deterministic); the extra row is the bias gradient (an all-ones tap atom).
//
// Warp roles: epilogue warps first (TMEM -> registers -> global; 8 in the tap-GEMM kernel, 4 in wgrad),
// then the TMA producer warp, then the MMA issuer warp (+TMEM owner). The two single-thread roles get the highest
// warp ids because the issue arbiter favours high warp ids (B300_MICROARCH.md): polling epilogue
// warps must not starve them (measured: 1.8x on the layer-1 weight gradient). smem ring of halo tiles with full/empty
// mbarriers; two TMEM tile buffers so the epilogue of tile i overlaps the MMAs of tile i+1.
// Weights for all 9 taps stay resident in shared memory for the CTA's lifetime.
#include <cuda_bf16.h>

#include <cstdio>
#include <stdexcept>

#include "../he/kernels.h"
#include "nn.h"
#include "tc_common.cuh"
#include "launch.cuh"

namespace hefl {
namespace nn {

using namespace hefl::tc;

// ------------------------------------------------------------------------------------------
// host: tensor maps
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p)
      throw std::runtime_error("cuTensorMapEncodeTiled not available");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D bf16 tensor [outer rows][inner cols], row pitch in bytes; box = box_inner x box_outer.
static CUtensorMap make_map(const void* ptr, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                            uint32_t box_inner, uint32_t box_outer) {
  CUtensorMap m;
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  const uint32_t inner_bytes = box_inner * 2;
  CUtensorMapSwizzle sw = inner_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : inner_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                              : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box,
                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[256];
    snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed (%d): inner=%llu outer=%llu pitch=%llu box=%ux%u",
             (int)r, (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)pitch_bytes,
             box_inner, box_outer);
    throw std::runtime_error(buf);
  }
  return m;
}

static int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  }
  return n;
}

// ------------------------------------------------------------------------------------------
// G1: halo-tile tap-GEMM kernel (forward + pool epilogue, or dgrad with plain store)
//
// Measured on B200 (bench/probe_shift.py): a K-major swizzled tile written by TMA can be read by
// tcgen05.mma starting at ANY row (descriptor start address + rows*row_bytes, base_offset 0) —
// the swizzle is a function of absolute shared-memory address bits. So each input row segment
// is loaded ONCE per tile and all 9 taps address shifted windows of it:
//   forward : tile = 2 image rows x 128 columns; 4 halo segments (rows h..h+3) of 130 pixels;
//             accumulator j (row h+j), tap (r,s) reads segment j+r at row offset s.
//   dgrad   : tile = 128 consecutive pixels; 3 segments starting at m0 - r*W - 2; tap (r,s)
//             reads segment r at row offset 2 - s.
// L2->SM traffic drops from 9 tap tiles to ~2 (fwd) / ~3 (dgrad) tiles per output tile.
// ------------------------------------------------------------------------------------------
struct TapGemmArgs {
  int B, H, W;          // input grid of the A matrix
  int Hp, Wp;           // pooled output grid (POOL)
  int tiles_w;          // column tiles per row pair (POOL)
  int num_tiles;
  int P;                // B*H*W
  int co_total;         // output channels of the layer (CO per CTA column block = blockIdx.y)
#ifdef HEFL_CONV_DEBUG
  int dbg;              // bottleneck isolation, ONLY in -DHEFL_CONV_DEBUG builds: 1 = skip TMA data, 2 = skip MMAs, 4 = skip epilogue
#endif
  const float* bias;    // [CO] (POOL)
  __nv_bfloat16* out;   // POOL: [B,Hp,Wp,CO]; else [P,CO]
  uint8_t* argmax;      // POOL, may be null
  // dgrad with the un-pooling of the PREVIOUS layer fused into the epilogue: the gradient of pixel m of this
  // layer's input (= pooled output of the previous layer) is scattered straight to the arg-max position of its
  // 2x2 window on the previous layer's conv grid (up_W x up_W per image), zeros to the other three positions.
  const uint8_t* up_amax;   // [P, co_total] codes of the previous layer (bits 0-1 position, bit 2 active) or null
  int up_W;
  // tile -> (image, row pair, column tile) without integer division: q = umulhi(n, magic) is exact for
  // n, d < 2^16 with magic = ceil(2^32 / d) (the epilogue warps spent ~40 of their ~100 per-tile set-up
  // instructions in two software divisions)
  uint32_t magic_per_img, magic_tiles_w;
};

__device__ __forceinline__ int fast_div(int n, int d, uint32_t magic) {
  if (d == 1) return n;
  return magic ? (int)__umulhi((uint32_t)n, magic) : n / d;
}

// TS = filter taps along the image row that are separate GEMMs: 3 normally; 1 when the three horizontal taps
// are packed into the channel dimension by the producer of the input (layer 1: 3 channels x 3 taps = 9 of the
// 16 padded channels, written by preprocess_u8) — a third of the MMAs for the same bytes.
template <int CK, int CO, bool POOL, int TS = 3>
struct TapGemmCfg {
  static constexpr int NTAP = 3 * TS;
  static constexpr int KB = CK < 64 ? CK : 64;            // channels per k-block (one swizzle atom)
  static constexpr int NKB = CK / KB;
  static constexpr int ROW_BYTES = KB * 2;
  static constexpr int NSEG = POOL ? 4 : 3;
  static constexpr int NACC = POOL ? 2 : 1;
  static constexpr int SEG_ROWS = 136;                    // 130 used, multiple of 8
  static constexpr int SEG_BYTES = SEG_ROWS * ROW_BYTES;
  static constexpr int HALO = NKB * NSEG * SEG_BYTES;     // one tile's input
  static constexpr int W_SUB = CO * ROW_BYTES;
  static constexpr int W_TAP = W_SUB * NKB;
  static constexpr int W_BYTES = NTAP * W_TAP;
  static constexpr int BAR_BYTES = 384;
  static constexpr int BUDGET = 225 * 1024;
  static constexpr int NBUF_RAW = (BUDGET - W_BYTES - BAR_BYTES - 1024) / HALO;
  // ring depth beyond 3 and more than 2 TMEM tile buffers measured no gain; small footprints let a
  // wgrad CTA and a dgrad/forward CTA share an SM (the backward pass runs them on two streams)
  static constexpr int NBUF = NBUF_RAW > 2 ? 2 : NBUF_RAW;
  static constexpr int SMEM = W_BYTES + NBUF * HALO + BAR_BYTES + 1024;
  // TMEM tile buffers: the MMA -> epilogue -> MMA hand-off costs ~1500 cycles of mbarrier latency
  // (measured with all work disabled: 750 cycles/tile with 2 buffers), so small-channel layers use
  // up to 8 buffers to keep several tiles in flight.
  static constexpr int NT_RAW = 512 / (NACC * CO);
  static constexpr int NT = NT_RAW > 2 ? 2 : NT_RAW;
  static constexpr int ACC_COLS = NT * NACC * CO;
  static constexpr int TMEM_COLS = ACC_COLS <= 32 ? 32 : (ACC_COLS <= 64 ? 64 : (ACC_COLS <= 128 ? 128 : (ACC_COLS <= 256 ? 256 : 512)));
  static_assert(NT >= 2, "need at least two TMEM tile buffers");
  // two CTAs per SM when shared memory and TMEM allow: the kernels are latency-bound (issue, TMA,
  // mbarrier hand-offs), so more independent pipelines on the same SM fill the bubbles
  static constexpr int OCC = (3 * SMEM <= 226 * 1024 && 3 * TMEM_COLS <= 512) ? 3
                             : ((2 * SMEM <= 226 * 1024 && 2 * TMEM_COLS <= 512) ? 2 : 1);
  static_assert(NBUF >= 1, "halo tile does not fit in shared memory");
  static_assert(ACC_COLS <= 512, "accumulators exceed TMEM");
  static_assert(CO % 32 == 0 && CO <= 128, "CO must be 32, 64, 96 or 128");
};

template <int CK, int CO, bool POOL, int TS>
__global__ void __launch_bounds__(352, TapGemmCfg<CK, CO, POOL, TS>::OCC)
tap_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                const TapGemmArgs a) {
  using Cfg = TapGemmCfg<CK, CO, POOL, TS>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sW = smem;
  uint8_t* sA = smem + Cfg::W_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + Cfg::NBUF * Cfg::HALO);
  uint64_t* full = bars;                       // [NBUF]
  uint64_t* empty = bars + Cfg::NBUF;          // [NBUF]
  uint64_t* wfull = bars + 2 * Cfg::NBUF;      // [1]
  uint64_t* tfull = wfull + 1;                 // [NT]
  uint64_t* tempty = tfull + Cfg::NT;          // [NT]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + Cfg::NT);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 8 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW);
    // POOL: two MMA-issuing warps (one per accumulator) => 2 commits per buffer / tile
    for (int s = 0; s < Cfg::NBUF; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], Cfg::NACC); }
    mbar_init(wfull, 1);
    for (int i = 0; i < Cfg::NT; ++i) { mbar_init(&tfull[i], Cfg::NACC); mbar_init(&tempty[i], 8); }
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: the set-up above and the weight tile (written only by the re-layout kernel, which never triggers its
  // dependents early — launch.cuh) overlap the previous kernel's tail; activations only after the wait.
  pdl_trigger();
  if (warp == 8 && elect_one()) {
    mbar_expect_tx(wfull, Cfg::W_BYTES);
    for (int tap = 0; tap < Cfg::NTAP; ++tap)
      for (int kb = 0; kb < Cfg::NKB; ++kb)
        tma_load_2d(sW + tap * Cfg::W_TAP + kb * Cfg::W_SUB, &tmW, kb * Cfg::KB,
                    tap * a.co_total + blockIdx.y * CO, wfull);
  }
  pdl_wait();

  if (warp == 8) {
    // ===== TMA producer =====
    if (elect_one()) {
      int buf = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
        int base, seg_stride;
        if (POOL) {
          const int per_img = a.Hp * a.tiles_w;
          const int b = fast_div(t, per_img, a.magic_per_img);
          const int rem = t - b * per_img;
          const int hp = fast_div(rem, a.tiles_w, a.magic_tiles_w);
          const int tw = rem - hp * a.tiles_w;
          base = (b * a.H + 2 * hp) * a.W + tw * 128;
          seg_stride = a.W;                      // segment j = image row h + j
        } else {
          base = t * 128 - 2;
          seg_stride = -a.W;                     // segment r starts at m0 - r*W - 2
        }
        mbar_wait(&empty[buf], phase ^ 1);
#ifdef HEFL_CONV_DEBUG
        if (a.dbg & 1) {
          mbar_arrive(&full[buf]);
        } else
#endif
        {
          mbar_expect_tx(&full[buf], Cfg::HALO);
          uint8_t* dst = sA + buf * Cfg::HALO;
          for (int kb = 0; kb < Cfg::NKB; ++kb)
            for (int sg = 0; sg < Cfg::NSEG; ++sg)
              tma_load_2d(dst + (kb * Cfg::NSEG + sg) * Cfg::SEG_BYTES, &tmA, kb * Cfg::KB, base + sg * seg_stride,
                          &full[buf]);
        }
        if (++buf == Cfg::NBUF) { buf = 0; phase ^= 1; }
      }
    }
  } else if (warp == 9 || warp == 10) {
    // ===== MMA issuers: warp 9 owns accumulator 0, warp 10 accumulator 1 (the small-N MMAs of these
    // layers are bound by per-thread issue cost, not by the tensor core, so two issuers run in parallel)
    const int jme = warp - 9;
    if (jme >= Cfg::NACC) goto done_roles;
    constexpr uint32_t idesc = make_idesc_bf16(128, CO);
    mbar_wait(wfull, 0);
    tc_fence_after();
    int buf = 0;
    uint32_t phase = 0;
    int tb = 0;
    uint32_t tb_phase = 0;
    for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
      mbar_wait(&tempty[tb], tb_phase ^ 1);
      mbar_wait(&full[buf], phase);
      tc_fence_after();
      if (elect_one()) {
        // descriptor low words: base + compile-time offsets (pure 32-bit adds per MMA)
        const uint32_t a_lo = desc_lo(smem_u32(sA + buf * Cfg::HALO));
        const uint32_t w_lo = desc_lo(smem_u32(sW));
        constexpr uint32_t hi = desc_hi(8 * Cfg::ROW_BYTES, Cfg::ROW_BYTES);
#pragma unroll
        for (int j = 0; j < Cfg::NACC; ++j) {
#ifdef HEFL_CONV_DEBUG
          if (a.dbg & 2) continue;
#endif
          if (j != jme) continue;
          const uint32_t d_tmem = tmem_base + (tb * Cfg::NACC + j) * CO;
#pragma unroll
          for (int tap = 0; tap < Cfg::NTAP; ++tap) {
            const int r = tap / TS, s = tap % TS;
            const int seg = POOL ? (j + r) : r;
            const int shift = POOL ? s : (2 - s);
#pragma unroll
            for (int kb = 0; kb < Cfg::NKB; ++kb) {
#pragma unroll
              for (int k = 0; k < Cfg::KB / 16; ++k) {
                const uint32_t ao = ((kb * Cfg::NSEG + seg) * Cfg::SEG_BYTES + shift * Cfg::ROW_BYTES + k * 32) >> 4;
                const uint32_t wo = (tap * Cfg::W_TAP + kb * Cfg::W_SUB + k * 32) >> 4;
                umma_bf16_lh(d_tmem, a_lo + ao, hi, w_lo + wo, hi, idesc, (tap | kb | k) != 0 ? 1u : 0u);
              }
            }
          }
        }
        umma_commit(&empty[buf]);
        umma_commit(&tfull[tb]);
      }
      __syncwarp();
      if (++buf == Cfg::NBUF) { buf = 0; phase ^= 1; }
      if (++tb == Cfg::NT) { tb = 0; tb_phase ^= 1; }
    }
  } else {
    // ===== epilogue warps (0..7): quadrant = warp % 4, channel slice = warp / 4 (8 channels a time).
    // (16 epilogue warps measured no faster than 8; 8 keeps the CTA small enough for 2 CTAs per SM.)
    const int qd = warp & 3;                       // TMEM lane quadrant this warp may read
    const int grp = warp >> 2;
    const uint32_t lane_base = (uint32_t)(qd * 32) << 16;
    int tb = 0;
    uint32_t tb_phase = 0;
    for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
      mbar_wait(&tfull[tb], tb_phase);
      tc_fence_after();
      if (POOL) {
        const int per_img = a.Hp * a.tiles_w;
        const int b = fast_div(t, per_img, a.magic_per_img);
        const int rem = t - b * per_img;
        const int hp = fast_div(rem, a.tiles_w, a.magic_tiles_w);
        const int tw = rem - hp * a.tiles_w;
        const int col = tw * 128 + qd * 32 + lane;           // conv-output column of this thread
        const int wp = col >> 1;
        const bool writer = wp < a.Wp;
        const bool odd = (lane & 1) != 0;
#pragma unroll 1
#ifdef HEFL_CONV_DEBUG
        const int ch_end = (a.dbg & 4) ? 0 : CO / 8;
#else
        constexpr int ch_end = CO / 8;
#endif
        for (int ch = grp; ch < ch_end; ch += 2) {
          float v0[8], v1[8];
          tmem_ld8_nowait(tmem_base + lane_base + (tb * 2 + 0) * CO + ch * 8, v0);
          tmem_ld8_nowait(tmem_base + lane_base + (tb * 2 + 1) * CO + ch * 8, v1);
          // the two lanes of a window split the 8 channels: even lane -> 0..3, odd lane -> 4..7 (the epilogue is
          // issue-bound — ncu: 64 % issue active, 5 % tensor pipe — so no lane may do redundant work)
          const float4 bq = __ldg(reinterpret_cast<const float4*>(a.bias + ch * 8 + (odd ? 4 : 0)));
          const float bias4[4] = {bq.x, bq.y, bq.z, bq.w};
          tmem_ld_wait();
          // max over the two image rows on the raw accumulators (bias + ReLU commute with max)
          uint32_t vbits = 0;                                 // 1 = lower image row wins
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const bool lw = v1[c] > v0[c];
            v0[c] = lw ? v1[c] : v0[c];
            vbits |= lw ? (1u << c) : 0u;
          }
          const uint32_t pvbits = __shfl_xor_sync(0xffffffffu, vbits, 1);
          const uint32_t mb = (vbits >> (odd ? 4 : 0)) & 15u;   // row bits of my column, my 4 channels
          const uint32_t pb = (pvbits >> (odd ? 4 : 0)) & 15u;  // ... of the partner's column
          float x[4];
          uint32_t idx = 0u;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float keep = odd ? v0[4 + i] : v0[i];
            const float send = odd ? v0[i] : v0[4 + i];
            const float recv = __shfl_xor_sync(0xffffffffu, send, 1);
            const float left = odd ? recv : keep, right = odd ? keep : recv;
            const bool rw = right > left;                       // right column wins only if strictly greater
            const uint32_t rowbit = ((rw != odd) ? (pb >> i) : (mb >> i)) & 1u;
            const float y = (rw ? right : left) + bias4[i];
            // bits 0-1: arg-max position (row*2 + col) in the window, bit 2: unit active (ReLU mask)
            idx |= ((rowbit << 1) | (rw ? 1u : 0u) | (y > 0.f ? 4u : 0u)) << (i * 8);
            x[i] = y > 0.f ? y : 0.f;
          }
          if (writer) {
            const size_t o = ((size_t)(b * a.Hp + hp) * a.Wp + wp) * CO + ch * 8 + (odd ? 4 : 0);
            *reinterpret_cast<uint2*>(a.out + o) = make_uint2(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]));
            if (a.argmax) *reinterpret_cast<uint32_t*>(a.argmax + o) = idx;
          }
        }
      } else {
        const int m = t * 128 + qd * 32 + lane;
        size_t up_base = 0;                                   // pixel index of the window's top-left position
        if (a.up_amax && m < a.P) {
          const int hw = a.H * a.W;
          const int b = m / hw, rem = m - b * hw;
          const int y = rem / a.W, x = rem - y * a.W;
          up_base = ((size_t)b * a.up_W + 2 * y) * a.up_W + 2 * x;
        }
#pragma unroll 1
        for (int ch = grp; ch < CO / 8; ch += 2) {
          float v[8];
          tmem_ld8_nowait(tmem_base + lane_base + tb * CO + ch * 8, v);
          tmem_ld_wait();
          if (m < a.P) {
            const int c0 = blockIdx.y * CO + ch * 8;
            const uint32_t pk[4] = {pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                                    pack_bf16x2(v[6], v[7])};
            if (a.up_amax == nullptr) {
              *reinterpret_cast<uint4*>(a.out + (size_t)m * a.co_total + c0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            } else {
              const uint2 code = *reinterpret_cast<const uint2*>(a.up_amax + (size_t)m * a.co_total + c0);
              const uint32_t cw[2] = {code.x, code.y};
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                uint32_t o[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const uint32_t ca = (cw[i >> 1] >> ((i & 1) * 16)) & 0xFFu;          // channel 2i
                  const uint32_t cb = (cw[i >> 1] >> ((i & 1) * 16 + 8)) & 0xFFu;      // channel 2i+1
                  const uint32_t lo = (ca == (4u | q)) ? (pk[i] & 0xFFFFu) : 0u;
                  const uint32_t hi = (cb == (4u | q)) ? (pk[i] & 0xFFFF0000u) : 0u;
                  o[i] = lo | hi;
                }
                const size_t px = up_base + (size_t)(q >> 1) * a.up_W + (q & 1);
                *reinterpret_cast<uint4*>(a.out + px * a.co_total + c0) = make_uint4(o[0], o[1], o[2], o[3]);
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[tb]);
      if (++tb == Cfg::NT) { tb = 0; tb_phase ^= 1; }
    }
  }
done_roles:
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int CK, int CO, bool POOL, int TS = 3>
static void launch_tap_gemm(const __nv_bfloat16* A, const __nv_bfloat16* Wt, TapGemmArgs a, cudaStream_t st) {
  using Cfg = TapGemmCfg<CK, CO, POOL, TS>;
  const CUtensorMap tmA = make_map(A, CK, (uint64_t)a.P, (uint64_t)CK * 2, Cfg::KB, Cfg::SEG_ROWS);
  const CUtensorMap tmW = make_map(Wt, CK, (uint64_t)Cfg::NTAP * a.co_total, (uint64_t)CK * 2, Cfg::KB, CO);
  auto kern = tap_gemm_kernel<CK, CO, POOL, TS>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
  const int ny = a.co_total / CO;
  const int slots = num_sms() * Cfg::OCC / ny;
  int gx = a.num_tiles < slots ? a.num_tiles : slots;
  if (gx < 1) gx = 1;
  dim3 grid(gx, ny);
  launch_pdl(kern, grid, dim3(352), Cfg::SMEM, st, tmA, tmW, a);
  hefl::cuda::note_launch();
}

// The work-skipping switch exists only in -DHEFL_CONV_DEBUG builds (HEFL_NVCC_EXTRA); release kernels carry
// no such code and conv_set_debug refuses to arm it.
#ifdef HEFL_CONV_DEBUG
static int g_dbg = 0;
void conv_set_debug(int mask) { g_dbg = mask; }
#else
void conv_set_debug(int mask) {
  if (mask != 0) throw std::runtime_error("conv_set_debug: this build has no debug switch (rebuild with -DHEFL_CONV_DEBUG)");
}
#endif

void conv_fwd_pool(const void* X, const void* Wf, const float* bias, void* out, uint8_t* argmax, int B, int H,
                   int W, int CK, int CO, int spack, cudaStream_t st) {
  TapGemmArgs a{};
#ifdef HEFL_CONV_DEBUG
  a.dbg = g_dbg;
#endif
  a.B = B; a.H = H; a.W = W;
  a.Hp = (H - 2) / 2; a.Wp = (W - 2) / 2;
  a.tiles_w = (2 * a.Wp + 127) / 128;
  a.num_tiles = B * a.Hp * a.tiles_w;
  {
    const int per_img = a.Hp * a.tiles_w;
    const bool ok = a.num_tiles < 65536 && per_img > 1 && per_img < 65536;
    a.magic_per_img = ok ? (uint32_t)((0x100000000ull + per_img - 1) / per_img) : 0u;
    a.magic_tiles_w = (ok && a.tiles_w > 1) ? (uint32_t)((0x100000000ull + a.tiles_w - 1) / a.tiles_w) : 0u;
  }
  a.P = B * H * W;
  a.co_total = CO;
  a.bias = bias;
  a.out = reinterpret_cast<__nv_bfloat16*>(out);
  a.argmax = argmax;
  const auto* x = reinterpret_cast<const __nv_bfloat16*>(X);
  const auto* w = reinterpret_cast<const __nv_bfloat16*>(Wf);
  if (CK == 16 && CO == 32 && spack) launch_tap_gemm<16, 32, true, 1>(x, w, a, st);
  else if (CK == 16 && CO == 32) launch_tap_gemm<16, 32, true>(x, w, a, st);
  else if (CK == 32 && CO == 32) launch_tap_gemm<32, 32, true>(x, w, a, st);
  else if (CK == 32 && CO == 64) launch_tap_gemm<32, 64, true>(x, w, a, st);
  else if (CK == 64 && CO == 64) launch_tap_gemm<64, 64, true>(x, w, a, st);
  else if (CK == 64 && CO == 128) launch_tap_gemm<64, 128, true>(x, w, a, st);
  else throw std::runtime_error("conv_fwd_pool: unsupported (CK, CO)");
}

void conv_dgrad(const void* dY, const void* Wd, void* dX, int B, int H, int W, int CK, int CO, const uint8_t* up_amax,
                int up_W, cudaStream_t st) {
  TapGemmArgs a{};
  a.up_amax = up_amax;
  a.up_W = up_W;
  a.B = B; a.H = H; a.W = W;
  a.P = B * H * W;
  a.num_tiles = (a.P + 127) / 128;
  a.co_total = CO;
  a.out = reinterpret_cast<__nv_bfloat16*>(dX);
  const auto* x = reinterpret_cast<const __nv_bfloat16*>(dY);
  const auto* w = reinterpret_cast<const __nv_bfloat16*>(Wd);
  if (CK == 32 && CO == 32) launch_tap_gemm<32, 32, false>(x, w, a, st);
  else if (CK == 64 && CO == 32) launch_tap_gemm<64, 32, false>(x, w, a, st);
  else if (CK == 64 && CO == 64) launch_tap_gemm<64, 64, false>(x, w, a, st);
  else if (CK == 128 && CO == 64) launch_tap_gemm<128, 32, false>(x, w, a, st);   // two column blocks
  else throw std::runtime_error("conv_dgrad: unsupported (CK, CO)");
}

// ------------------------------------------------------------------------------------------
// G1b (layer 1 by default, HEFL_FWD_PAIR=0 / all to change): forward + pool with both columns of a pooling window in
// the SAME TMEM lane.
// Validated against G1 on hardware (tests/test_gpu_conv.py::test_conv_fwd_pool_pair_matches_plain_kernel: same
// pooled values and arg-max codes); 33.7 vs 40.4 us on layer 1 (B=32, 256x256), slower on the small layers.
//
// ncu on G1 (prof_fwd0_v4): the pool epilogue is the limiter of the forward kernels — 62 % issue-active,
// 6 % tensor pipe, ~33 instructions per pooled output — because a lane owns one conv COLUMN, so the 2x2 window
// needs a lane exchange (5 shuffles, 16 parity selects) per 8-channel chunk.
//
// Here the activation matrix [pixels, CK] is viewed as [pixel PAIRS, 2*CK] (same memory; needs an even image
// width so pairs never straddle rows). GEMM row j of accumulator (dy, dx) is window j of the pooled row:
//     acc(dy,dx)[j] = sum_{r,s} X[row 2hp+dy+r, column 2j+dx+s] . W[r,s]
// With e = dx + s, column 2j+e is pair-row j + (e >> 1), half e & 1: a row shift of the A descriptor plus a
// K byte offset of (e & 1) * CK * 2 inside the pair-row — both are things G1 already does (row-shifted starts,
// 32-byte K steps inside a swizzle atom). Four accumulators (2 rows x 2 column parities), M = 128 windows.
// The epilogue thread of window j then holds all four values of its window: max/arg-max in registers, no
// shuffles, every lane stores a full 16-byte pooled pixel chunk. Restricted to CK <= 32 (one swizzle atom per
// pair-row) and CO <= 64 (4 accumulators x 2 TMEM buffers).
// ------------------------------------------------------------------------------------------
template <int CK, int CO>
struct PairFwdCfg {
  static constexpr int ROW_BYTES = 2 * CK * 2;            // one pair-row: 2 pixels x CK channels, 64 or 128 B
  static constexpr int NSEG = 4;                          // image rows 2hp .. 2hp+3
  static constexpr int SEG_ROWS = 136;                    // 130 pair-rows used (128 windows + shift 1 + slack)
  static constexpr int SEG_BYTES = SEG_ROWS * ROW_BYTES;
  static constexpr int HALO = NSEG * SEG_BYTES;
  static constexpr int W_ROW = CK * 2;                    // weight rows: [tap][CO][CK], 32 or 64 B (as G1)
  static constexpr int W_TAP = CO * W_ROW;
  static constexpr int W_BYTES = 9 * W_TAP;
  static constexpr int BAR_BYTES = 384;
  static constexpr int NBUF = 2;
  static constexpr int SMEM = W_BYTES + NBUF * HALO + BAR_BYTES + 1024;
  static constexpr int NACC = 4;
  static constexpr int NT = 2;
  static constexpr int ACC_COLS = NT * NACC * CO;
  static constexpr int TMEM_COLS = ACC_COLS <= 256 ? 256 : 512;
  static constexpr int OCC = (2 * SMEM <= 226 * 1024 && 2 * TMEM_COLS <= 512) ? 2 : 1;
  static_assert(CK == 16 || CK == 32, "pair-row forward: one swizzle atom per pair-row");
  static_assert(CO == 32 || CO == 64, "pair-row forward: 4 accumulators x 2 buffers must fit TMEM");
  static_assert(SMEM <= 226 * 1024, "shared memory");
};

struct PairFwdArgs {
  int B, H, W;          // input grid (W even)
  int Hp, Wp;           // pooled grid
  int num_tiles;        // B * Hp (one pooled row per tile; Wp <= 128)
  const float* bias;
  __nv_bfloat16* out;   // [B,Hp,Wp,CO]
  uint8_t* argmax;      // may be null
};

// SP: s-packed layer-1 input (channels = pixels x, x+1, x+2): the three horizontal taps are already inside the 16
// channels, so only the three filter rows remain — 3 MMAs per accumulator, column parity = K byte offset.
template <int CK, int CO, bool SP>
__global__ void __launch_bounds__(352, PairFwdCfg<CK, CO>::OCC)
pair_fwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                const PairFwdArgs a) {
  using Cfg = PairFwdCfg<CK, CO>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sW = smem;
  uint8_t* sA = smem + Cfg::W_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + Cfg::NBUF * Cfg::HALO);
  uint64_t* full = bars;
  uint64_t* empty = bars + Cfg::NBUF;
  uint64_t* wfull = bars + 2 * Cfg::NBUF;
  uint64_t* tfull = wfull + 1;
  uint64_t* tempty = tfull + Cfg::NT;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + Cfg::NT);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 8 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW);
    for (int s = 0; s < Cfg::NBUF; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 2); }   // two MMA issuers
    mbar_init(wfull, 1);
    for (int i = 0; i < Cfg::NT; ++i) { mbar_init(&tfull[i], 2); mbar_init(&tempty[i], 8); }
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();
  if (warp == 8 && elect_one()) {
    constexpr int NTAPW = SP ? 3 : 9;
    mbar_expect_tx(wfull, NTAPW * Cfg::W_TAP);
    for (int tap = 0; tap < NTAPW; ++tap) tma_load_2d(sW + tap * Cfg::W_TAP, &tmW, 0, tap * CO, wfull);
  }
  pdl_wait();
  const int half_w = a.W >> 1;

  if (warp == 8) {
    // ===== TMA producer: 4 image rows of pair-rows per tile =====
    if (elect_one()) {
      int buf = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
        const int b = t / a.Hp, hp = t - b * a.Hp;
        const int q0 = (b * a.H + 2 * hp) * half_w;          // first pair-row of image row 2hp
        mbar_wait(&empty[buf], phase ^ 1);
        mbar_expect_tx(&full[buf], Cfg::HALO);
        uint8_t* dst = sA + buf * Cfg::HALO;
        for (int sg = 0; sg < Cfg::NSEG; ++sg) tma_load_2d(dst + sg * Cfg::SEG_BYTES, &tmA, 0, q0 + sg * half_w, &full[buf]);
        if (++buf == Cfg::NBUF) { buf = 0; phase ^= 1; }
      }
    }
  } else if (warp == 9 || warp == 10) {
    // ===== MMA issuers: warp 9 -> accumulators (dy=0, dx=0/1), warp 10 -> (dy=1, dx=0/1) =====
    const int dy = warp - 9;
    constexpr uint32_t idesc = make_idesc_bf16(128, CO);
    mbar_wait(wfull, 0);
    tc_fence_after();
    int buf = 0, tb = 0;
    uint32_t phase = 0, tb_phase = 0;
    for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
      mbar_wait(&tempty[tb], tb_phase ^ 1);
      mbar_wait(&full[buf], phase);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_lo = desc_lo(smem_u32(sA + buf * Cfg::HALO));
        const uint32_t w_lo = desc_lo(smem_u32(sW));
        constexpr uint32_t a_hi = desc_hi(8 * Cfg::ROW_BYTES, Cfg::ROW_BYTES);
        constexpr uint32_t w_hi = desc_hi(8 * Cfg::W_ROW, Cfg::W_ROW);
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const uint32_t d_tmem = tmem_base + (tb * Cfg::NACC + dy * 2 + dx) * CO;
          if constexpr (SP) {
#pragma unroll
            for (int r = 0; r < 3; ++r) {
              const uint32_t ao = ((dy + r) * Cfg::SEG_BYTES + dx * CK * 2) >> 4;
              const uint32_t wo = (r * Cfg::W_TAP) >> 4;
              umma_bf16_lh(d_tmem, a_lo + ao, a_hi, w_lo + wo, w_hi, idesc, r != 0 ? 1u : 0u);
            }
            continue;
          }
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            const int r = tap / 3, s = tap % 3;
            const int e = dx + s;
#pragma unroll
            for (int k = 0; k < CK / 16; ++k) {
              const uint32_t ao = ((dy + r) * Cfg::SEG_BYTES + (e >> 1) * Cfg::ROW_BYTES + (e & 1) * CK * 2 + k * 32) >> 4;
              const uint32_t wo = (tap * Cfg::W_TAP + k * 32) >> 4;
              umma_bf16_lh(d_tmem, a_lo + ao, a_hi, w_lo + wo, w_hi, idesc, (tap | k) != 0 ? 1u : 0u);
            }
          }
        }
        umma_commit(&empty[buf]);
        umma_commit(&tfull[tb]);
      }
      __syncwarp();
      if (++buf == Cfg::NBUF) { buf = 0; phase ^= 1; }
      if (++tb == Cfg::NT) { tb = 0; tb_phase ^= 1; }
    }
  } else {
    // ===== epilogue warps 0..7: lane = window (quadrant = warp % 4), channel chunks interleaved by warp / 4 =====
    const int qd = warp & 3;
    const int grp = warp >> 2;
    const uint32_t lane_base = (uint32_t)(qd * 32) << 16;
    const int j = qd * 32 + lane;                          // window index in the pooled row
    int tb = 0;
    uint32_t tb_phase = 0;
    for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
      mbar_wait(&tfull[tb], tb_phase);
      tc_fence_after();
      const size_t row_out = (size_t)t * a.Wp;             // t = b * Hp + hp
#pragma unroll 1
      for (int ch = grp; ch < CO / 8; ch += 2) {
        float v00[8], v01[8], v10[8], v11[8];
        const uint32_t tcol = tmem_base + lane_base + tb * Cfg::NACC * CO + ch * 8;
        tmem_ld8_nowait(tcol + 0 * CO, v00);
        tmem_ld8_nowait(tcol + 1 * CO, v01);
        tmem_ld8_nowait(tcol + 2 * CO, v10);
        tmem_ld8_nowait(tcol + 3 * CO, v11);
        const float4 bA = __ldg(reinterpret_cast<const float4*>(a.bias + ch * 8));
        const float4 bB = __ldg(reinterpret_cast<const float4*>(a.bias + ch * 8 + 4));
        const float bias8[8] = {bA.x, bA.y, bA.z, bA.w, bB.x, bB.y, bB.z, bB.w};
        tmem_ld_wait();
        uint32_t packed[4], idx[2] = {0u, 0u};
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
          float x[2];
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            // same tie-breaking as G1: lower row wins only if strictly greater, then right column likewise
            const bool l0 = v10[c + i] > v00[c + i];
            const bool l1 = v11[c + i] > v01[c + i];
            const float m0 = l0 ? v10[c + i] : v00[c + i];
            const float m1 = l1 ? v11[c + i] : v01[c + i];
            const bool rw = m1 > m0;
            const uint32_t rowbit = (rw ? l1 : l0) ? 1u : 0u;
            const float y = (rw ? m1 : m0) + bias8[c + i];
            idx[(c + i) >> 2] |= ((rowbit << 1) | (rw ? 1u : 0u) | (y > 0.f ? 4u : 0u)) << (((c + i) & 3) * 8);
            x[i] = y > 0.f ? y : 0.f;
          }
          packed[c >> 1] = pack_bf16x2(x[0], x[1]);
        }
        if (j < a.Wp) {
          const size_t o = (row_out + j) * CO + ch * 8;
          *reinterpret_cast<uint4*>(a.out + o) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
          if (a.argmax) *reinterpret_cast<uint2*>(a.argmax + o) = make_uint2(idx[0], idx[1]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[tb]);
      if (++tb == Cfg::NT) { tb = 0; tb_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int CK, int CO, bool SP = false>
static void launch_pair_fwd(const __nv_bfloat16* X, const __nv_bfloat16* Wt, PairFwdArgs a, cudaStream_t st) {
  using Cfg = PairFwdCfg<CK, CO>;
  const uint64_t pair_rows = ((uint64_t)a.B * a.H * a.W) / 2;
  const CUtensorMap tmA = make_map(X, 2 * CK, pair_rows, (uint64_t)Cfg::ROW_BYTES, 2 * CK, Cfg::SEG_ROWS);
  const CUtensorMap tmW = make_map(Wt, CK, (uint64_t)(SP ? 3 : 9) * CO, (uint64_t)CK * 2, CK, CO);
  auto kern = pair_fwd_kernel<CK, CO, SP>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
  int gx = num_sms() * Cfg::OCC;
  if (gx > a.num_tiles) gx = a.num_tiles;
  launch_pdl(kern, dim3(gx), dim3(352), Cfg::SMEM, st, tmA, tmW, a);
  hefl::cuda::note_launch();
}

bool conv_fwd_pool_pair_supported(int H, int W, int CK, int CO) {
  return H == W && (W % 2) == 0 && (W - 2) / 2 <= 128 && (CK == 16 || CK == 32) && (CO == 32 || CO == 64);
}

// Same contract as conv_fwd_pool (plain 9-tap weight layout [9][CO][CK], or [3][CO][16] with the s-packed input);
// see G1b above.
void conv_fwd_pool_pair(const void* X, const void* Wf, const float* bias, void* out, uint8_t* argmax, int B, int H,
                        int W, int CK, int CO, int spack, cudaStream_t st) {
  if (!conv_fwd_pool_pair_supported(H, W, CK, CO)) throw std::runtime_error("conv_fwd_pool_pair: unsupported shape");
  PairFwdArgs a{};
  a.B = B; a.H = H; a.W = W;
  a.Hp = (H - 2) / 2; a.Wp = (W - 2) / 2;
  a.num_tiles = B * a.Hp;
  a.bias = bias;
  a.out = reinterpret_cast<__nv_bfloat16*>(out);
  a.argmax = argmax;
  const auto* x = reinterpret_cast<const __nv_bfloat16*>(X);
  const auto* w = reinterpret_cast<const __nv_bfloat16*>(Wf);
  if (spack && !(CK == 16 && CO == 32)) throw std::runtime_error("conv_fwd_pool_pair: s-packed input is CK=16, CO=32 only");
  if (CK == 16 && CO == 32 && spack) launch_pair_fwd<16, 32, true>(x, w, a, st);
  else if (CK == 16 && CO == 32) launch_pair_fwd<16, 32>(x, w, a, st);
  else if (CK == 32 && CO == 32) launch_pair_fwd<32, 32>(x, w, a, st);
  else if (CK == 32 && CO == 64) launch_pair_fwd<32, 64>(x, w, a, st);
  else throw std::runtime_error("conv_fwd_pool_pair: unsupported (CK, CO)");
}

// ------------------------------------------------------------------------------------------
// G2: weight-gradient kernel.
//
// dW[r,s][ci][co] = sum_m X[m + r*W + s][ci] * dY[m][co]. Both operands are consumed in their
// native NHWC layout as MN-major UMMA operands (pixels = K), so no transposed copies exist.
// Work is organised by image rows: a CTA walks down a 64-column strip; at row h it needs the X
// row segments h, h+1, h+2 (72 pixels each) and the dY chunk of row h. Segments live in a ring
// of stages, so each X segment is fetched ONCE and serves filter rows r = 2, 1, 0 on three
// consecutive steps; the tap column s is a row offset of the MMA descriptor (LBO = one pixel).
// 3-D tensor maps (C, W, B*H) keep chunks inside an image row (out-of-range columns zero-fill).
// Split over (image, strip, row range). Every CTA stores its partial sums ([9*C+1, Co], the last row is the bias
// gradient: an all-ones A tile) to its own slice of a workspace; splitk_sum_kernel then adds the slices to dW32 in
// CTA order, so the result is the same on every run (fp32 RED of the partials rounded in arrival order).
// ------------------------------------------------------------------------------------------
#ifndef HEFL_WGRAD_OCC3
#define HEFL_WGRAD_OCC3 0     // 1: allow three wgrad CTAs per SM (validated build flag, see WgradCfg::OCC)
#endif

struct WgradArgs {
  int H, W, Ho;     // input grid height/width, valid output rows
  int strips;       // ceil((W-2) / 64)
  int rsplit;       // row ranges per (image, strip)
  int rows_per;     // rows per range
  int units;        // B * strips * rsplit
  int nchunks;      // FLAT: ceil(B*H*W / 64)
  int Co;           // total output channels (row pitch of dW32)
  float* part;      // [gridDim.x][9*CK + 1][Co] fp32: one partial sum per CTA
};

// FLAT = small feature maps (W <= 32): a 64-pixel chunk of one image row would be mostly padding, so
// chunks are 64 consecutive pixels of the flattened [B*H*W] axis and each stage carries its own
// three X segments (rows offset by W); no ring reuse, L2 traffic is irrelevant at these sizes.
template <int CK, int COT, bool FLAT = false>
struct WgradCfg {
  // CK = 16 (layer 1): 32-byte MN-major atoms make the tensor core read shared memory 32 bytes at
  // a time (measured ~128 cycles per MMA). Instead the X tensor map uses OVERLAPPING rows: row m is
  // the 128 bytes starting at pixel m (4 pixels x 16 channels, row stride 32 B), so one 128-byte
  // atom already holds the tap columns s = 0..3 and no pixel shift is needed.
  static constexpr bool PACK4 = CK == 16;
  static constexpr int ATOM_A = PACK4 ? 128 : CK * 2;          // bytes of one k-row of the A atom
  static constexpr int ATOM_B = COT * 2;
  static constexpr int TPG = PACK4 ? 4 : 128 / CK;             // tap columns covered by one MMA
  static constexpr int MMA_PER_R = CK == 64 ? 2 : 1;           // s = {0,1},{2,3} for CK=64; one MMA otherwise
  static constexpr int NACC = 3 * MMA_PER_R;
  static constexpr int XROWS = PACK4 ? 64 : 72;                // 64 + pixel shifts (none when packed)
  static constexpr int A_LBO = PACK4 ? 0 : CK * 2;             // next atom = next pixel (packed: rows 64.. unused)
  static constexpr int X_BYTES = XROWS * ATOM_A;
  static constexpr int X_SEG = ((X_BYTES + 1023) / 1024) * 1024;
  static constexpr int DY_BYTES = 64 * ATOM_B;
  static constexpr int DY_OFF = FLAT ? 3 * X_SEG : X_SEG;
  static constexpr int TX = (FLAT ? 3 : 1) * X_BYTES + DY_BYTES;
  static constexpr int STAGE_FULL = DY_OFF + ((DY_BYTES + 1023) / 1024) * 1024;
  static_assert(!(FLAT && PACK4), "layer 1 always uses the rolling-window path");
  static constexpr int ONES_BYTES = 16 * 1024;                 // [128 x 64] bf16 of 1.0
  // deep ring: stages are small (one X row segment + one dY chunk), so the number of bytes in
  // flight, not the MMA rate, bounds throughput (measured: 6 stages -> 204 us on layer 1)
  static constexpr int NSTAGE_RAW = (200 * 1024 - ONES_BYTES) / STAGE_FULL;
  static constexpr int NSTAGE = NSTAGE_RAW > 6 ? 6 : NSTAGE_RAW;
  static constexpr int SMEM = NSTAGE * STAGE_FULL + ONES_BYTES + 512 + 1024;
  static constexpr int COLS = (NACC + 1) * COT;                // + bias accumulator
  static_assert(NSTAGE >= 4, "ring needs 3 live stages + 1 in flight");
  static constexpr int TMEM_COLS = COLS <= 32 ? 32 : (COLS <= 64 ? 64 : (COLS <= 128 ? 128 : (COLS <= 256 ? 256 : 512)));
  static_assert(COLS <= 512, "accumulators exceed TMEM");
  // CTAs per SM. ncu (prof_wgrad1): 22 % tensor-pipe active, 7 % issue active, occupancy limit 3 by shared memory
  // while 2 were launched — the kernel is latency-bound, so take the third CTA when smem and TMEM allow it.
  static constexpr int OCC = (HEFL_WGRAD_OCC3 && 3 * SMEM <= 226 * 1024 && 3 * TMEM_COLS <= 512) ? 3
                             : ((2 * SMEM <= 226 * 1024 && 2 * TMEM_COLS <= 512) ? 2 : 1);
  static_assert(CK == 16 || CK == 32 || CK == 64, "CK must be one swizzle atom");
  static_assert(COT == 32 || COT == 64, "COT must be one swizzle atom");
};

template <int CK, int COT, bool FLAT>
__global__ void __launch_bounds__(192, WgradCfg<CK, COT, FLAT>::OCC)
wgrad_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDY,
             const WgradArgs a) {
  using Cfg = WgradCfg<CK, COT, FLAT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ones = smem + Cfg::NSTAGE * Cfg::STAGE_FULL;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ones + Cfg::ONES_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + Cfg::NSTAGE;
  uint64_t* done = bars + 2 * Cfg::NSTAGE;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int co0 = blockIdx.y * COT;

  for (int i = threadIdx.x; i < Cfg::ONES_BYTES / 4; i += blockDim.x)
    reinterpret_cast<uint32_t*>(ones)[i] = 0x3F803F80u;        // bf16 1.0 x2 (uniform => layout-agnostic)
  if (warp == 4 && lane == 0) {
    prefetch_tmap(&tmX);
    prefetch_tmap(&tmDY);
    for (int s = 0; s < Cfg::NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  fence_proxy_async();   // generic-proxy writes (ones tile) visible to the tensor-core async proxy
  if (warp == 5) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue();
  const int per_img = a.strips * a.rsplit;

  if (warp == 4) {
    if (FLAT) {
      if (elect_one()) {
        int slot = 0;
        uint32_t phase = 0;
        for (int c = blockIdx.x; c < a.nchunks; c += gridDim.x) {
          mbar_wait(&empty[slot], phase ^ 1u);
          uint8_t* st = smem + slot * Cfg::STAGE_FULL;
          mbar_expect_tx(&full[slot], Cfg::TX);
          for (int r = 0; r < 3; ++r) tma_load_2d(st + r * Cfg::X_SEG, &tmX, 0, c * 64 + r * a.W, &full[slot]);
          tma_load_2d(st + Cfg::DY_OFF, &tmDY, co0, c * 64, &full[slot]);
          if (++slot == Cfg::NSTAGE) { slot = 0; phase ^= 1; }
        }
      }
    } else if (elect_one()) {
      int slot = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < a.units; u += gridDim.x) {
        const int b = u / per_img;
        const int rem = u - b * per_img;
        const int strip = rem / a.rsplit;
        const int h0 = (rem - strip * a.rsplit) * a.rows_per;
        const int h1 = min(a.Ho, h0 + a.rows_per);
        if (h0 >= h1) continue;
        for (int i = h0 - 2; i < h1; ++i) {
          mbar_wait(&empty[slot], phase ^ 1u);
          uint8_t* st = smem + slot * Cfg::STAGE_FULL;
          mbar_expect_tx(&full[slot], Cfg::X_BYTES + (i >= h0 ? Cfg::DY_BYTES : 0));
          tma_load_3d(st, &tmX, 0, strip * 64, b * a.H + i + 2, &full[slot]);   // PACK4: 128-byte windows
          if (i >= h0) tma_load_3d(st + Cfg::DY_OFF, &tmDY, co0, strip * 64, b * a.H + i, &full[slot]);
          if (++slot == Cfg::NSTAGE) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 5) {
    constexpr uint32_t idesc = make_idesc_bf16(128, COT, 1, 1);
    constexpr uint32_t a_hi = desc_hi(8 * Cfg::ATOM_A, Cfg::ATOM_A);
    constexpr uint32_t b_hi = desc_hi(8 * Cfg::ATOM_B, Cfg::ATOM_B);
    constexpr uint32_t o_hi = desc_hi(8 * 128, 128);
    const uint32_t smem_lo = desc_lo(smem_u32(smem));                 // stage 0, as a descriptor low word
    const uint32_t ones_lo = desc_lo(smem_u32(ones), 64 * 128);
    constexpr uint32_t a_lbo = (uint32_t)(Cfg::A_LBO >> 4) << 16;
    constexpr uint32_t b_lbo = (uint32_t)(Cfg::DY_BYTES >> 4) << 16;
    constexpr uint32_t stage16 = Cfg::STAGE_FULL >> 4;
    int slot = 0;                                                     // ring position of the current stage
    uint32_t phase = 0;
    uint32_t first = 1;
    if (FLAT) {
      for (int c = blockIdx.x; c < a.nchunks; c += gridDim.x) {
        mbar_wait(&full[slot], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t st_lo = smem_lo + slot * stage16;
          const uint32_t dy_lo = st_lo + (Cfg::DY_OFF >> 4) + b_lbo;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t blo = dy_lo + ((k * 16 * Cfg::ATOM_B) >> 4);
            const uint32_t accum = k == 0 ? (first ^ 1u) : 1u;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
              for (int mm = 0; mm < Cfg::MMA_PER_R; ++mm)
                umma_bf16_lh(tmem_base + (r * Cfg::MMA_PER_R + mm) * COT,
                             st_lo + a_lbo + ((r * Cfg::X_SEG + (mm * Cfg::TPG + k * 16) * Cfg::ATOM_A) >> 4), a_hi,
                             blo, b_hi, idesc, accum);
            }
            umma_bf16_lh(tmem_base + Cfg::NACC * COT, ones_lo + ((k * 16 * 128) >> 4), o_hi, blo, b_hi, idesc, accum);
          }
          umma_commit(&empty[slot]);
        }
        __syncwarp();
        first = 0;
        if (++slot == Cfg::NSTAGE) { slot = 0; phase ^= 1; }
      }
    }
    for (int u = FLAT ? a.units : (int)blockIdx.x; u < a.units; u += gridDim.x) {
      const int b = u / per_img;
      const int rem = u - b * per_img;
      const int strip = rem / a.rsplit;
      const int h0 = (rem - strip * a.rsplit) * a.rows_per;
      const int h1 = min(a.Ho, h0 + a.rows_per);
      if (h0 >= h1) continue;
      (void)b;
      for (int i = h0 - 2; i < h1; ++i) {
        mbar_wait(&full[slot], phase);
        tc_fence_after();
        const int s1 = slot == 0 ? Cfg::NSTAGE - 1 : slot - 1;       // stage of X row h+1
        const int s0 = s1 == 0 ? Cfg::NSTAGE - 1 : s1 - 1;           // stage of X row h
        if (i >= h0 && elect_one()) {
          const uint32_t x_lo[3] = {smem_lo + s0 * stage16 + a_lbo, smem_lo + s1 * stage16 + a_lbo,
                                    smem_lo + slot * stage16 + a_lbo};
          const uint32_t dy_lo = smem_lo + slot * stage16 + (Cfg::DY_OFF >> 4) + b_lbo;
#pragma unroll
          for (int k = 0; k < 4; ++k) {                        // 4 x UMMA_K(16) pixels per 64-pixel chunk
            const uint32_t blo = dy_lo + ((k * 16 * Cfg::ATOM_B) >> 4);
            const uint32_t accum = k == 0 ? (first ^ 1u) : 1u;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
              for (int mm = 0; mm < Cfg::MMA_PER_R; ++mm)
                umma_bf16_lh(tmem_base + (r * Cfg::MMA_PER_R + mm) * COT,
                             x_lo[r] + (((mm * Cfg::TPG + k * 16) * Cfg::ATOM_A) >> 4), a_hi, blo, b_hi, idesc, accum);
            }
            umma_bf16_lh(tmem_base + Cfg::NACC * COT, ones_lo + ((k * 16 * 128) >> 4), o_hi, blo, b_hi, idesc, accum);
          }
          umma_commit(&empty[s0]);                              // stage of X row h is done
        }
        __syncwarp();
        if (i >= h0) first = 0;
        if (++slot == Cfg::NSTAGE) { slot = 0; phase ^= 1; }
      }
      if (elect_one()) {                                        // release the last two stages of the unit
        const int l1 = slot == 0 ? Cfg::NSTAGE - 1 : slot - 1;
        const int l0 = l1 == 0 ? Cfg::NSTAGE - 1 : l1 - 1;
        umma_commit(&empty[l0]);
        umma_commit(&empty[l1]);
      }
      __syncwarp();
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
    mbar_wait(done, 0);                 // this warp is idle now: it waits for the tensor core ...
    named_barrier_arrive(2, 160);       // ... and releases the epilogue warps, which block in hardware
  } else {
    const int qd = warp;
    const uint32_t lane_base = (uint32_t)(qd * 32) << 16;
    named_barrier_sync(2, 160);         // no polling while the main loop runs
    if ((int)blockIdx.x < (FLAT ? a.nchunks : a.units)) {
      tc_fence_after();
      const int row = qd * 32 + lane;                          // row inside an accumulator: s_local*CK + ci
#pragma unroll 1
      for (int acc = 0; acc <= Cfg::NACC; ++acc) {
        int R;                                                 // dW32 row: (r*3+s)*CK + ci, or 9*CK = bias
        bool valid;
        if (acc == Cfg::NACC) {
          R = 9 * CK;
          valid = row == 0;
        } else {
          const int r = acc / Cfg::MMA_PER_R, mm = acc % Cfg::MMA_PER_R;
          const int s = mm * Cfg::TPG + row / CK;
          R = (r * 3 + s) * CK + row % CK;
          valid = s < 3 && (!Cfg::PACK4 || row < 64);
        }
#pragma unroll 1
        for (int ch = 0; ch < COT / 32; ++ch) {
          float v[32];
          tmem_ld32(tmem_base + lane_base + acc * COT + ch * 32, v);
          if (valid) {
            float* dst = a.part + ((size_t)blockIdx.x * (9 * CK + 1) + R) * a.Co + co0 + ch * 32;
#pragma unroll
            for (int c = 0; c < 32; c += 4)
              *reinterpret_cast<float4*>(dst + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// 3-D bf16 tensor [rows][W][C] (C contiguous); box = {box_c, box_w, 1}.
static CUtensorMap make_map_3d(const void* ptr, uint64_t C, uint64_t W, uint64_t rows, uint32_t box_c,
                               uint32_t box_w) {
  CUtensorMap m;
  cuuint64_t dims[3] = {C, W, rows};
  cuuint64_t strides[2] = {C * 2, W * C * 2};
  cuuint32_t box[3] = {box_c, box_w, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const uint32_t inner_bytes = box_c * 2;
  CUtensorMapSwizzle sw = inner_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : inner_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                              : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box,
                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled(3d) failed");
  return m;
}

// Same, with explicit byte strides (overlapping rows: stride_w < C*2 is legal for TMA).
static CUtensorMap make_map_3d_strided(const void* ptr, uint64_t C, uint64_t W, uint64_t rows, uint64_t stride_w,
                                       uint64_t stride_row, uint32_t box_c, uint32_t box_w) {
  CUtensorMap m;
  cuuint64_t dims[3] = {C, W, rows};
  cuuint64_t strides[2] = {stride_w, stride_row};
  cuuint32_t box[3] = {box_c, box_w, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box,
                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled(3d, strided) failed");
  return m;
}

// dst[i] += part[0][i] + part[1][i] + ... + part[splits-1][i], summed in that order whatever the launch timing
// (32 x kSumRows threads per 32 elements: each thread sums every kSumRows-th partial, so at most a few dependent L2
// round trips per thread; the kSumRows column sums are then added in row order)
constexpr int kSumRows = 16;
__global__ void __launch_bounds__(32 * kSumRows) splitk_sum_kernel(const float* __restrict__ part, int splits, int n,
                                                                   float* __restrict__ dst) {
  __shared__ float col[kSumRows][32];
  pdl_prologue();
  const int i = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
  if (i < n)
#pragma unroll 8
    for (int s = threadIdx.y; s < splits; s += kSumRows) acc += part[(size_t)s * n + i];
  col[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && i < n) {
    float v = col[0][threadIdx.x];
#pragma unroll
    for (int y = 1; y < kSumRows; ++y) v += col[y][threadIdx.x];
    dst[i] += v;
  }
}

template <int CK, int COT, bool FLAT>
static WgradArgs wgrad_args(int B, int H, int W, int Co) {
  WgradArgs a{};
  a.H = H; a.W = W; a.Ho = H - 2;
  a.strips = (W - 2 + 63) / 64;
  // units of <= 16 image rows, dealt round-robin: load imbalance <= one unit, ring warm-up 2/16
  a.rows_per = a.Ho < 16 ? a.Ho : 16;
  a.rsplit = (a.Ho + a.rows_per - 1) / a.rows_per;
  a.units = B * a.strips * a.rsplit;
  a.nchunks = (B * H * W + 63) / 64;
  a.Co = Co;
  return a;
}

// number of CTAs along the pixel axis = number of partial sums
template <int CK, int COT, bool FLAT>
static int wgrad_splits(int B, int H, int W, int Co) {
  using Cfg = WgradCfg<CK, COT, FLAT>;
  const WgradArgs a = wgrad_args<CK, COT, FLAT>(B, H, W, Co);
  const int total_steps = FLAT ? a.nchunks : a.units * (a.rows_per + 2);
  // every CTA pays a fixed epilogue (the store of all accumulators): give each at least a few steps
  int gx = total_steps / (FLAT ? 6 : 24);
  if (gx > num_sms() * Cfg::OCC / (Co / COT)) gx = num_sms() * Cfg::OCC / (Co / COT);
  if (gx > (FLAT ? a.nchunks : a.units)) gx = FLAT ? a.nchunks : a.units;
  return gx < 1 ? 1 : gx;
}

template <int CK, int COT, bool FLAT>
static void launch_wgrad(const __nv_bfloat16* X, const __nv_bfloat16* DY, int B, int H, int W, int Co, float* dW32,
                         float* part, cudaStream_t st) {
  using Cfg = WgradCfg<CK, COT, FLAT>;
  WgradArgs a = wgrad_args<CK, COT, FLAT>(B, H, W, Co);
  a.part = part;
  const int P = B * H * W;
  CUtensorMap tmX, tmD;
  if (FLAT) {
    tmX = make_map(X, CK, (uint64_t)P, (uint64_t)CK * 2, CK, Cfg::XROWS);
    tmD = make_map(DY, Co, (uint64_t)P, (uint64_t)Co * 2, COT, 64);
  } else {
    tmX = Cfg::PACK4 ? make_map_3d_strided(X, 64, W, (uint64_t)B * H, 32, (uint64_t)W * 32, 64, Cfg::XROWS)
                     : make_map_3d(X, CK, W, (uint64_t)B * H, CK, Cfg::XROWS);
    tmD = make_map_3d(DY, Co, W, (uint64_t)B * H, COT, 64);
  }
  auto kern = wgrad_kernel<CK, COT, FLAT>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
  const int gx = wgrad_splits<CK, COT, FLAT>(B, H, W, Co);
  launch_pdl(kern, dim3(gx, Co / COT), dim3(192), Cfg::SMEM, st, tmX, tmD, a);
  hefl::cuda::note_launch();
  const int n = (9 * CK + 1) * Co;
  launch_pdl(splitk_sum_kernel, dim3((n + 31) / 32), dim3(32, kSumRows), 0, st, part, gx, n, dW32);
  hefl::cuda::note_launch();
}

template <int CK, int COT, bool FLAT>
struct WgradShape {
  static constexpr int ck = CK, cot = COT;
  static constexpr bool flat = FLAT;
};

// the (CK, Co) -> kernel instance table, shared by the launcher and the workspace query
template <class F>
static auto wgrad_dispatch(int CK, int Co, int W, F&& f) {
  const bool flat = W <= 32 && CK != 16;
  if (CK == 16 && Co == 32) return f(WgradShape<16, 32, false>{});
  if (CK == 32 && Co == 32) return flat ? f(WgradShape<32, 32, true>{}) : f(WgradShape<32, 32, false>{});
  if (CK == 32 && Co == 64) return flat ? f(WgradShape<32, 64, true>{}) : f(WgradShape<32, 64, false>{});
  if (CK == 64 && (Co == 64 || Co == 128)) return flat ? f(WgradShape<64, 64, true>{}) : f(WgradShape<64, 64, false>{});
  throw std::runtime_error("conv_wgrad: unsupported (CK, Co)");
}

size_t conv_wgrad_part_floats(int B, int H, int W, int CK, int Co) {
  const int splits = wgrad_dispatch(CK, Co, W, [&](auto s) {
    using S = decltype(s);
    return wgrad_splits<S::ck, S::cot, S::flat>(B, H, W, Co);
  });
  return (size_t)splits * (9 * CK + 1) * Co;
}

void conv_wgrad(const void* X, const void* DY, float* dW32, float* part, int B, int H, int W, int CK, int Co,
                cudaStream_t st) {
  const auto* x = reinterpret_cast<const __nv_bfloat16*>(X);
  const auto* d = reinterpret_cast<const __nv_bfloat16*>(DY);
  wgrad_dispatch(CK, Co, W, [&](auto s) {
    using S = decltype(s);
    launch_wgrad<S::ck, S::cot, S::flat>(x, d, B, H, W, Co, dW32, part, st);
    return 0;
  });
}

}  // namespace nn
}  // namespace hefl

// ------------------------------------------------------------------------------------------
// Probe: can a K-major swizzled A tile be consumed starting at an arbitrary ROW offset (with the
// descriptor's base_offset field carrying the swizzle phase)? Used to validate halo-tile reuse.
// ------------------------------------------------------------------------------------------
namespace hefl {
namespace nn {
using namespace hefl::tc;

template <int CK>
__global__ void __launch_bounds__(128, 1)
umma_shift_probe_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                        float* out, int shift_rows, int mode) {
  constexpr int RB = CK * 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                      // 144 rows
  uint8_t* sB = smem + 144 * 128;          // 32 rows
  uint64_t* bar = reinterpret_cast<uint64_t*>(sB + 32 * 128);
  uint64_t* done = bar + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_init(done, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc<32>(slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *slot;
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, 144 * RB + 32 * RB);
    tma_load_2d(sA, &tmA, 0, 0, bar);
    tma_load_2d(sB, &tmB, 0, 0, bar);
    mbar_wait(bar, 0);
    tc_fence_after();
    const uint32_t a0 = smem_u32(sA) + shift_rows * RB;
    for (int k = 0; k < CK / 16; ++k) {
      uint64_t ad = make_kmajor_desc(a0 + k * 32, RB);
      if (mode == 1) ad |= (uint64_t)((a0 >> 7) & 7) << 49;   // base_offset = row phase in the 1024-B pattern
      const uint64_t bd = make_kmajor_desc(smem_u32(sB) + k * 32, RB);
      umma_bf16(tmem, ad, bd, make_idesc_bf16(128, 32), k ? 1u : 0u);
    }
    umma_commit(done);
  }
  mbar_wait(done, 0);
  tc_fence_after();
  float v[32];
  tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16), v);
  for (int c = 0; c < 32; ++c) out[(warp * 32 + lane) * 32 + c] = v[c];
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc<32>(tmem); }
}

void umma_shift_probe(const void* A, const void* Bm, float* out, int CK, int shift_rows, int mode, cudaStream_t st) {
  const CUtensorMap tmA = make_map(A, CK, 144, (uint64_t)CK * 2, CK, 144);
  const CUtensorMap tmB = make_map(Bm, CK, 32, (uint64_t)CK * 2, CK, 32);
  const int smem = 144 * 128 + 32 * 128 + 64 + 1024;
  if (CK == 64) {
    cudaFuncSetAttribute(umma_shift_probe_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    umma_shift_probe_kernel<64><<<1, 128, smem, st>>>(tmA, tmB, out, shift_rows, mode);
  } else if (CK == 32) {
    cudaFuncSetAttribute(umma_shift_probe_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    umma_shift_probe_kernel<32><<<1, 128, smem, st>>>(tmA, tmB, out, shift_rows, mode);
  } else {
    cudaFuncSetAttribute(umma_shift_probe_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    umma_shift_probe_kernel<16><<<1, 128, smem, st>>>(tmA, tmB, out, shift_rows, mode);
  }
}

}  // namespace nn
}  // namespace hefl
