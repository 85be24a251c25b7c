// Implicit-GEMM convolution on DFXP integer mantissas for B200 (sm_100a): no im2col matrix ever touches HBM.
//
//   out[m, n] = 2^e * sum_{tap=(r,s)} sum_c src[pixel(m) + tap, c] * Wp[n, tap*C + c]   (+ bias[n])
//
// A operand: TMA *im2col mode* over the NHWC mantissa tensor (C, W, H, N): one bulk load fetches, for 128
// consecutive output pixels (wrapping rows and images in hardware, zero-filling TF 'SAME' padding) and one
// filter tap, a [128 x Cb] block of channels straight into shared memory in the tensor core's K-major layout.
// B operand: 2-D tiled TMA over the packed weights Wp[N, taps*C] (K-major).  tcgen05.mma.kind::i8 accumulates
// exactly in s32 in tensor memory; the epilogue applies the power-of-two rescale read from the range variables.
//
// Replaces tf.nn.conv2d (dynamic_fixed_point.py:291) and, run on the output-gradient map with the filter
// rotated by 180 degrees, tf.gradients(y, X, gradq) for stride-1 convolutions (dynamic_fixed_point.py:305).
//
// Channel chunk Cb = min(C, 128) in {16, 32, 64, 128} selects the shared-memory layout: 16-byte rows of
// interleaved 8x16B core matrices, or 32/64/128-byte swizzled rows; a pipeline stage always carries 128 bytes
// of K per row (128/Cb tap-blocks), i.e. four K=32 MMAs.  Same warp roles and mbarrier protocol as gemm_i8.cu.
#include "conv_classes.h"
#include "conv_internal.h"
#include "qsite.cuh"
#include "tcgen05.cuh"

namespace lbt {
namespace {

using namespace tc;

constexpr int kBlockM = 128;
constexpr int kStageK = 128;  // bytes of K per row per stage
constexpr int kThreads = 192;        // wgrad: producer, MMA issuer, 4 epilogue warps
constexpr int kEpiWarps = 8;         // fprop: two epilogue warps per TMEM lane quadrant (the fused epilogue is ALU-heavy)
constexpr int kThreadsF = 32 * (2 + kEpiWarps);

__device__ int g_conv_error = 0;

struct ConvParams {
  uint32_t M, N;                 // output pixels, output channels
  uint32_t OW, OHW;              // output width, OH*OW
  FastDiv d_OW, d_OHW;           // constant-divisor division for the producer's pixel decomposition
  int lower_w, lower_h;          // base-pixel offset of output (0,0): -pad_left, -pad_top
  int sw, sh;
  uint32_t kw;                   // filter width (tap -> (r, s))
  uint32_t taps, cchunks;        // kh*kw, C / Cb
  uint32_t ksteps;               // taps * cchunks (+1 padding step when Cb == 16 and odd)
  uint32_t ksteps_real;
  uint32_t cb;                   // channel chunk bytes
  uint32_t mode;                 // log2(cb / 16)
  uint32_t C;                    // source channels
  uint32_t m_tiles, n_tiles;
  const int32_t* ibA;
  const int32_t* ibB;
  int exp_const;
  const float* bias;
  const float* addend;           // optional fp32 [M, ldc] added to the fp32 result (F32 epilogue only)
  float* out;
  size_t ldc;
  uint32_t idesc;
  uint32_t idesc2;               // DUAL: the low plane's MMAs (A = u8)
  BnqParams bnq;                 // fused re-quantising epilogue (bnq.q.bits == 0: off)
  int remap;                     // fp32 rows go to out + img * rs_n + oh * rs_y + ow * rs_x (OutRemap) instead of row * ldc
  long long rs_n, rs_y, rs_x;
};

template <int BN>
struct Cfg {
  static constexpr int kStageA = kBlockM * kStageK;
  static constexpr int kStageB = BN * kStageK;
  static constexpr int kStageBytes = kStageA + kStageB;
  // Narrow tiles do little work per tile, so their time is a chain of latencies (TMA -> MMA -> tcgen05.ld ->
  // store).  Hide it with several CTAs per SM (small smem rings) and a deep ring of TMEM accumulators.
  static constexpr int kCtasPerSm = BN <= 16 ? 3 : (BN <= 128 ? 2 : 1);
  static constexpr int kStages = BN <= 64 ? 4 : (BN == 128 ? 3 : 4);
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;
  static constexpr int kAccStages = BN <= 64 ? 4 : 2;
  static constexpr int kTmemCols = (kAccStages * BN) < 32 ? 32 : (kAccStages * BN);
  static_assert(kCtasPerSm * kSmemBytes <= 227 * 1024, "shared memory budget");
  static_assert(kCtasPerSm * kTmemCols <= 512, "tensor memory budget");
};

inline int ctas_per_sm(int bn) { return bn <= 16 ? 3 : (bn <= 128 ? 2 : 1); }

// fprop configuration.  DUAL: the SOURCE is a 9..16-bit mantissa as two byte planes (k = 256 * hi + lo: a 16-bit gradient on its
// way to the input gradient, BASELINE config 5): both planes' im2col blocks ride in one ring slot and meet the same filter tile in
// two accumulators; the fp32 epilogue rounds 256 * acc_hi + acc_lo once.  One CTA per SM (it owns all of tensor memory).
template <int BN, bool DUAL>
struct FCfg {
  static constexpr int kStageA = Cfg<BN>::kStageA;
  static constexpr int kStageB = Cfg<BN>::kStageB;
  static constexpr int kStageBytes = (DUAL ? 2 : 1) * kStageA + kStageB;
  static constexpr int kCtasPerSm = DUAL ? 1 : Cfg<BN>::kCtasPerSm;
  static constexpr int kStages = DUAL ? ((226 * 1024) / kStageBytes > 4 ? 4 : (226 * 1024) / kStageBytes) : Cfg<BN>::kStages;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;
  static constexpr int kAccW = (DUAL ? 2 : 1) * BN;
  static constexpr int kAccStages = DUAL ? (512 / kAccW > 4 ? 4 : 512 / kAccW) : Cfg<BN>::kAccStages;
  static constexpr int kTmemCols = (kAccStages * kAccW) < 32 ? 32 : (kAccStages * kAccW);
  static_assert(kStages >= 2 && kAccStages >= 1, "fprop ring");
  static_assert(kCtasPerSm * kSmemBytes <= 227 * 1024, "shared memory budget");
  static_assert(kCtasPerSm * kTmemCols <= 512, "tensor memory budget");
};

// wgrad configuration.  DUAL: the gradient is a 9..16-bit mantissa as two byte planes (k = 256 * hi + lo, BASELINE config 5): both
// planes' blocks ride in one ring slot and are multiplied with the SAME input block into two accumulators, so the input
// operand is loaded once and every element costs ONE int64 atomic (256 * acc_hi + acc_lo) instead of two passes' two.
template <int BN, bool DUAL>
struct WCfg {
  static constexpr int kStageA = Cfg<BN>::kStageA;
  static constexpr int kStageB1 = Cfg<BN>::kStageB;                    // one plane
  static constexpr int kStageBytes = kStageA + (DUAL ? 2 : 1) * kStageB1;
  static constexpr int kCtasPerSm = Cfg<BN>::kCtasPerSm;
  static constexpr int kBudget = (227 * 1024) / kCtasPerSm - 1024;
  static constexpr int kStages = !DUAL ? Cfg<BN>::kStages : (kBudget / kStageBytes > 4 ? 4 : kBudget / kStageBytes);
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;
  static constexpr int kAccW = (DUAL ? 2 : 1) * BN;                     // tensor-memory columns of one accumulator stage
  static constexpr int kAccStages = !DUAL ? Cfg<BN>::kAccStages : ((512 / kCtasPerSm) / kAccW > 4 ? 4 : (512 / kCtasPerSm) / kAccW);
  static constexpr int kTmemCols = (kAccStages * kAccW) < 32 ? 32 : (kAccStages * kAccW);
  static_assert(kStages >= 2 && kAccStages >= 1, "wgrad ring");
  static_assert(kCtasPerSm * kSmemBytes <= 227 * 1024, "shared memory budget");
  static_assert(kCtasPerSm * kTmemCols <= 512, "tensor memory budget");
};

template <int BN, bool DUAL = false>
__global__ void __launch_bounds__(kThreadsF, FCfg<BN, DUAL>::kCtasPerSm)
conv_fprop_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB,
                  const ConvParams p) {
  using C = FCfg<BN, DUAL>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[C::kStages];
  __shared__ __align__(8) uint64_t empty_bar[C::kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[C::kAccStages];
  __shared__ __align__(8) uint64_t tmem_empty_bar[C::kAccStages];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_abort;
  __shared__ int s_stat[kEpiWarps][2 * BN];
  __shared__ unsigned long long s_tot[2 * BN];   // CTA totals of the fused statistics (last N tile of the CTA)              // per epilogue warp: partial sum k, sum k^2 (fused BN statistics)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < C::kAccStages; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], kEpiWarps);
    }
    s_abort = 0;
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    if (DUAL) tma_prefetch_desc(&tmA2);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, C::kTmemCols);
  for (uint32_t i = threadIdx.x; i < 2 * BN; i += kThreadsF) s_tot[i] = 0ull;
  pdl_trigger();
  fence_before();
  __syncthreads();
  fence_after();
  pdl_wait();   // everything above touched only shared / tensor memory and kernel parameters
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);
  volatile int* abort_flag = &s_abort;

  const uint32_t total_tiles = p.m_tiles * p.n_tiles;
  const uint32_t spb = kStageK / p.cb;                       // tap-blocks per stage
  const uint32_t a_block = kBlockM * p.cb, b_block = BN * p.cb;
  const uint32_t nstages_k = (p.ksteps + spb - 1) / spb;     // pipeline stages per tile

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      bool ok = true;
      for (uint32_t tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
        const uint32_t m_tile = tile % p.m_tiles, n_tile = tile / p.m_tiles;
        const uint32_t m0 = m_tile * kBlockM;
        const uint32_t img = fastdiv(m0, p.d_OHW), rem = m0 - img * p.OHW;
        const uint32_t ohu = fastdiv(rem, p.d_OW);
        const int oh = (int)ohu, ow = (int)(rem - ohu * p.OW);
        const int base_w = p.lower_w + ow * p.sw, base_h = p.lower_h + oh * p.sh;
        uint32_t cc = 0, r = 0, s = 0;   // running decomposition of the k-step: no integer divisions in this loop
        for (uint32_t ks = 0; ks < nstages_k; ++ks) {
          if (!(ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag, &g_conv_error))) break;
          uint8_t* sa = smem + stage * C::kStageBytes;
          uint8_t* sb = sa + (DUAL ? 2 : 1) * C::kStageA;
          const uint32_t k0 = ks * spb;
          const uint32_t nblk = min(spb, p.ksteps - k0);
          mbar_expect_tx(&full_bar[stage], nblk * ((DUAL ? 2u : 1u) * a_block + b_block));
          for (uint32_t j = 0; j < nblk; ++j) {
            const uint32_t kstep = k0 + j;
            const bool pad = kstep >= p.ksteps_real;        // Cb == 16 pairing pad: B is OOB-zero, A is any tap
            tma_load_im2col_4d(&tmA, &full_bar[stage], sa + j * a_block, pad ? 0 : (int)(cc * p.cb), base_w, base_h, (int)img,
                               (uint16_t)(pad ? 0u : s), (uint16_t)(pad ? 0u : r));
            if (DUAL)   // the low plane's block of the same tap / channel chunk
              tma_load_im2col_4d(&tmA2, &full_bar[stage], sa + C::kStageA + j * a_block, pad ? 0 : (int)(cc * p.cb), base_w, base_h,
                                 (int)img, (uint16_t)(pad ? 0u : s), (uint16_t)(pad ? 0u : r));
            tma_load_2d(&tmB, &full_bar[stage], sb + j * b_block, (int)(kstep * p.cb), (int)(n_tile * BN));
            if (++cc == p.cchunks) {
              cc = 0;
              if (++s == p.kw) {
                s = 0;
                ++r;
              }
            }
          }
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      bool ok = true;
      for (uint32_t tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
        if (!(ok = mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, abort_flag, &g_conv_error))) break;
        fence_after();
        const uint32_t d_tmem = tmem_base + acc * C::kAccW;
        uint32_t first = 1;
        for (uint32_t ks = 0; ks < nstages_k; ++ks) {
          if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag, &g_conv_error))) break;
          fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::kStageBytes);
          const uint32_t sb = sa + (DUAL ? 2 : 1) * C::kStageA;
          const uint32_t nblk = min(spb, p.ksteps - ks * spb);
          if (p.mode == 0) {
            // 16-byte rows: one K=32 instruction spans two consecutive tap-blocks (leading byte offset = block size)
            for (uint32_t j = 0; j < nblk; j += 2) {  // nblk is even: ksteps is padded to an even count
              const uint64_t db = make_desc_kmajor(sb + j * b_block, 0, b_block);
              umma_i8(d_tmem, make_desc_kmajor(sa + j * a_block, 0, a_block), db, p.idesc, first ? 0u : 1u);
              if (DUAL) umma_i8(d_tmem + BN, make_desc_kmajor(sa + C::kStageA + j * a_block, 0, a_block), db, p.idesc2, first ? 0u : 1u);
              first = 0;
            }
          } else {
            const uint32_t per_block = p.cb / 32;
            for (uint32_t j = 0; j < nblk; ++j)
              for (uint32_t kk = 0; kk < per_block; ++kk) {
                const uint64_t db = make_desc_kmajor(sb + j * b_block + kk * 32, (int)p.mode, 16);
                umma_i8(d_tmem, make_desc_kmajor(sa + j * a_block + kk * 32, (int)p.mode, 16), db, p.idesc, first ? 0u : 1u);
                if (DUAL)   // the low plane against the same filter tile, into the second accumulator
                  umma_i8(d_tmem + BN, make_desc_kmajor(sa + C::kStageA + j * a_block + kk * 32, (int)p.mode, 16), db, p.idesc2,
                          first ? 0u : 1u);
                first = 0;
              }
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (!ok) break;
        umma_commit(&tmem_full_bar[acc]);
        if (++acc == C::kAccStages) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    const uint32_t quad = warp & 3;
    const uint32_t half = (uint32_t)(warp - 2) >> 2;  // which of the quadrant's two warps: chunks half, half + 2, ...
    int e = p.exp_const;
    if (p.ibA) e += *p.ibA;
    if (p.ibB) e += *p.ibB;
    const float scale = exp2i(e);
    const bool fused = p.bnq.q.bits != 0;
    int* my_stat = s_stat[warp - 2];
    BnqState bst;
    bst.tiles = 0;
    uint32_t stat_ntile = 0;
    if (fused) {
      bst.init(p.bnq);
      for (int i = lane; i < 2 * BN; i += 32) my_stat[i] = 0;
      __syncwarp();
    }
    uint32_t acc = 0, acc_phase = 0;
    bool ok = true;
    for (uint32_t tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
      const uint32_t m_tile = tile % p.m_tiles, n_tile = tile / p.m_tiles;
      const uint32_t row = m_tile * kBlockM + quad * 32 + lane;
      const uint32_t pix = fused ? row % p.bnq.rows_per_image : 0u;
      const uint32_t col0 = n_tile * BN;
      if (fused) {   // this warp's noise lines of the tile: into L1 while the accumulator is still being computed
#pragma unroll 1
        for (int c = (BN > 16 ? 16 * (int)half : 0); c < BN; c += (BN > 16 ? 32 : 16))
          bnq_prefetch(p.bnq, pix, p.N, col0 + (uint32_t)c, row < p.M && col0 + (uint32_t)c < p.N && !(BN == 16 && half));
      }
      ok = mbar_wait(&tmem_full_bar[acc], acc_phase, abort_flag, &g_conv_error);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      fence_after();
      const uint32_t taddr = tmem_base + acc * C::kAccW + ((quad * 32u) << 16);
      if (fused && (n_tile != stat_ntile || bst.tiles >= (uint32_t)kBnqFlushTiles)) {
        bnq_flush(p.bnq, my_stat, stat_ntile * BN, BN, p.N, lane);
        stat_ntile = n_tile;
        bst.tiles = 0;
      }
#pragma unroll 1
      for (int c = (BN > 16 ? 16 * (int)half : 0); c < BN; c += (BN > 16 ? 32 : 16)) {
        if (BN == 16 && half) break;  // a single chunk: the second warp of the quadrant has nothing to do
        uint32_t v[16];
        float4 u4[4];   // fused: the chunk's noise, requested before the accumulator wait (bnq_load_noise)
        const bool fchunk = fused && col0 + c < p.N;   // warp-uniform
        if (BN > 16 && fchunk) bnq_load_noise(p.bnq, bst, pix, row < p.M, col0 + c, min(16u, p.N - (col0 + c)), p.N, u4);
        tmem_ld16(taddr + c, v);
        uint32_t w[DUAL ? 16 : 1];
        if constexpr (DUAL) tmem_ld16(taddr + BN + c, w);
        tmem_ld_wait();
        if (BN <= 16 && fchunk)   // the 16-column instantiation runs three CTAs per SM at 64 registers: no room for early loads
          bnq_load_noise(p.bnq, bst, pix, row < p.M, col0 + c, min(16u, p.N - (col0 + c)), p.N, u4);
        if (fused) {
          if (fchunk) {
            const uint32_t ncol = min(16u, p.N - (col0 + c));
            bnq_chunk(p.bnq, bst, v, u4, scale, p.bias ? p.bias + col0 + c : nullptr, row, row < p.M, col0 + c, ncol, p.N, my_stat, BN,
                      (uint32_t)c, lane);
          }
        } else if (row < p.M && col0 + c < p.N) {
          const uint32_t ncol = min(16u, p.N - (col0 + c));
          float* o;
          if (p.remap) {
            const uint32_t img = fastdiv(row, p.d_OHW), rem = row - img * p.OHW;
            const uint32_t oh = fastdiv(rem, p.d_OW), ow = rem - oh * p.OW;
            o = p.out + ((long long)img * p.rs_n + (long long)oh * p.rs_y + (long long)ow * p.rs_x) + col0 + c;
          } else {
            o = p.out + (size_t)row * p.ldc + col0 + c;
          }
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            if constexpr (DUAL) f[j] = __ll2float_rn((long long)(int)v[j] * 256ll + (long long)(int)w[j]) * scale;   // one rounding
            else f[j] = __int2float_rn((int)v[j]) * scale;
            if (p.bias && j < (int)ncol) f[j] = __fadd_rn(f[j], __ldg(p.bias + col0 + c + j));
          }
          if (p.addend) {   // + an fp32 tensor of the output's shape (the other branch of a gradient sum)
            const float* ad = p.addend + (o - p.out);
            if (ncol == 16 && ((reinterpret_cast<uintptr_t>(ad) & 15u) == 0)) {
              float4 a4[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) a4[j] = __ldcs(reinterpret_cast<const float4*>(ad) + j);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                f[4 * j + 0] = __fadd_rn(f[4 * j + 0], a4[j].x);
                f[4 * j + 1] = __fadd_rn(f[4 * j + 1], a4[j].y);
                f[4 * j + 2] = __fadd_rn(f[4 * j + 2], a4[j].z);
                f[4 * j + 3] = __fadd_rn(f[4 * j + 3], a4[j].w);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (j < (int)ncol) f[j] = __fadd_rn(f[j], __ldg(ad + j));
            }
          }
          if (ncol == 16 && ((reinterpret_cast<uintptr_t>(o) & 15u) == 0)) {
#pragma unroll
            for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < (int)ncol) o[j] = f[j];
          }
        }
      }
      ++bst.tiles;
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      if (++acc == C::kAccStages) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (fused && ok) {
      bnq_flush_cta(p.bnq, my_stat, s_tot, stat_ntile * BN, BN, p.N, lane, threadIdx.x - 64, 32 * kEpiWarps, 1);
      bnq_finish(p.bnq, bst, (unsigned long long)p.M * p.N, warp == 2, lane);
    }
  }

  fence_before();
  __syncthreads();
  fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, C::kTmemCols);
}

// ------------------------------------------------------------------------------------------------
// wgrad: dW[(r,s,c), co] = sum over output pixels m of  X[pixel(m) + (r,s), c] * G[m, co]
// The reduction runs over PIXELS, so both operands are MN-major: the very same "128 pixels x Cb channels"
// blocks the TMA produces are the tensor core's K x M (K x N) atoms — no transposes, no im2col matrix.
// M tile = 128 consecutive (tap, channel) rows = 128/Cb tap-blocks; one pipeline stage = one block of 128
// pixels (four K=32 MMAs).  Pixel blocks are split across CTAs; partial sums go to the int64 buffer with
// 64-bit atomics (exact, order-independent).
// ------------------------------------------------------------------------------------------------
struct WgradParams {
  uint32_t Mpix, N;              // output pixels (reduction length), output channels
  uint32_t OW, OHW;
  FastDiv d_OW, d_OHW;
  int lower_w, lower_h, sw, sh;
  uint32_t kw, cchunks, ksteps;  // filter width, C / Cb, taps * cchunks
  uint32_t cb, mode_a;           // channel chunk bytes of X, log2(cb/16)
  uint32_t cbn, mode_b, nchunks; // channel chunk bytes of G, log2(cbn/16), BN / cbn
  uint32_t m_tiles, n_tiles;     // over (tap, channel) rows / output channels
  uint32_t pix_blocks, blocks_per_split, k_splits;
  uint32_t Kf;                   // taps * C
  long long* acc64;
  int alpha;
  uint32_t idesc;
  uint32_t idesc2;               // DUAL: the low plane's MMAs (B = u8)
};

template <int BN, bool DUAL = false>
__global__ void __launch_bounds__(kThreads, Cfg<BN>::kCtasPerSm)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmG2,
                  const WgradParams p) {
  using C = WCfg<BN, DUAL>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[C::kStages];
  __shared__ __align__(8) uint64_t empty_bar[C::kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[C::kAccStages];
  __shared__ __align__(8) uint64_t tmem_empty_bar[C::kAccStages];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_abort;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < C::kAccStages; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], 4);
    }
    s_abort = 0;
    fence_barrier_init();
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmG);
    if (DUAL) tma_prefetch_desc(&tmG2);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, C::kTmemCols);
  pdl_trigger();
  fence_before();
  __syncthreads();
  fence_after();
  pdl_wait();   // everything above touched only shared / tensor memory and kernel parameters
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);
  volatile int* abort_flag = &s_abort;

  const uint32_t total_items = p.m_tiles * p.n_tiles * p.k_splits;
  const uint32_t spb = kStageK / p.cb;                 // tap-blocks per M tile
  const uint32_t a_block = kBlockM * p.cb;             // 128 pixels x cb
  const uint32_t b_block = kBlockM * p.cbn;            // 128 pixels x cbn

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      bool ok = true;
      for (uint32_t item = blockIdx.x; item < total_items && ok; item += gridDim.x) {
        const uint32_t m_tile = item % p.m_tiles, rest = item / p.m_tiles;
        const uint32_t n_tile = rest % p.n_tiles, ks = rest / p.n_tiles;
        const uint32_t pb0 = ks * p.blocks_per_split, pb1 = min(pb0 + p.blocks_per_split, p.pix_blocks);
        const uint32_t k0 = m_tile * spb;
        const uint32_t nblk = min(spb, p.ksteps - k0);
        // the (channel chunk, tap) of each of the item's <= 8 tap-blocks: decomposed once, not per pixel block
        int jc[8];
        uint16_t js[8], jr[8];
#pragma unroll
        for (uint32_t j = 0; j < 8; ++j) {
          const uint32_t kstep = k0 + (j < nblk ? j : 0);
          const uint32_t tap = kstep / p.cchunks;
          jc[j] = (int)((kstep - tap * p.cchunks) * p.cb);
          jr[j] = (uint16_t)(tap / p.kw);
          js[j] = (uint16_t)(tap - (uint32_t)jr[j] * p.kw);
        }
        for (uint32_t pb = pb0; pb < pb1; ++pb) {
          if (!(ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag, &g_conv_error))) break;
          uint8_t* sa = smem + stage * C::kStageBytes;
          uint8_t* sb = sa + C::kStageA;
          const uint32_t m0 = pb * kBlockM;
          const uint32_t img = fastdiv(m0, p.d_OHW), rem = m0 - img * p.OHW;
          const uint32_t ohu = fastdiv(rem, p.d_OW);
          const int oh = (int)ohu, ow = (int)(rem - ohu * p.OW);
          const int base_w = p.lower_w + ow * p.sw, base_h = p.lower_h + oh * p.sh;
          mbar_expect_tx(&full_bar[stage], nblk * a_block + (DUAL ? 2u : 1u) * p.nchunks * b_block);
#pragma unroll
          for (uint32_t j = 0; j < 8; ++j)
            if (j < nblk)
              tma_load_im2col_4d(&tmX, &full_bar[stage], sa + j * a_block, jc[j], base_w, base_h, (int)img, js[j], jr[j]);
          for (uint32_t j = 0; j < p.nchunks; ++j)
            tma_load_2d(&tmG, &full_bar[stage], sb + j * b_block, (int)(n_tile * BN + j * p.cbn), (int)m0);
          if (DUAL)
            for (uint32_t j = 0; j < p.nchunks; ++j)
              tma_load_2d(&tmG2, &full_bar[stage], sb + C::kStageB1 + j * b_block, (int)(n_tile * BN + j * p.cbn), (int)m0);
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      bool ok = true;
      for (uint32_t item = blockIdx.x; item < total_items && ok; item += gridDim.x) {
        const uint32_t ks = (item / p.m_tiles) / p.n_tiles;
        const uint32_t pb0 = ks * p.blocks_per_split, pb1 = min(pb0 + p.blocks_per_split, p.pix_blocks);
        if (!(ok = mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, abort_flag, &g_conv_error))) break;
        fence_after();
        const uint32_t d_tmem = tmem_base + acc * C::kAccW;
        for (uint32_t pb = pb0; pb < pb1; ++pb) {
          if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag, &g_conv_error))) break;
          fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::kStageBytes);
          const uint32_t sb = sa + C::kStageA;
#pragma unroll
          for (uint32_t kk = 0; kk < kBlockM / 32; ++kk) {
            // 32 pixels (K) per instruction: advance by 32 rows of the block
            const uint64_t da = make_desc_mnmajor(sa + kk * 32 * p.cb, (int)p.mode_a, a_block);
            umma_i8(d_tmem, da, make_desc_mnmajor(sb + kk * 32 * p.cbn, (int)p.mode_b, b_block), p.idesc, (pb > pb0 || kk > 0) ? 1u : 0u);
            if (DUAL)   // the low plane against the same input block, into the second accumulator
              umma_i8(d_tmem + BN, da, make_desc_mnmajor(sb + C::kStageB1 + kk * 32 * p.cbn, (int)p.mode_b, b_block), p.idesc2,
                      (pb > pb0 || kk > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (!ok) break;
        umma_commit(&tmem_full_bar[acc]);
        if (++acc == C::kAccStages) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    const uint32_t quad = warp & 3;
    uint32_t acc = 0, acc_phase = 0;
    bool ok = true;
    for (uint32_t item = blockIdx.x; item < total_items && ok; item += gridDim.x) {
      const uint32_t m_tile = item % p.m_tiles, rest = item / p.m_tiles;
      const uint32_t n_tile = rest % p.n_tiles;
      ok = mbar_wait(&tmem_full_bar[acc], acc_phase, abort_flag, &g_conv_error);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      fence_after();
      const uint32_t row = m_tile * kBlockM + quad * 32 + lane;   // (tap, channel) index kf
      const uint32_t col0 = n_tile * BN;
      const uint32_t taddr = tmem_base + acc * C::kAccW + ((quad * 32u) << 16);
#pragma unroll 1
      for (int c = 0; c < BN; c += 16) {
        uint32_t v[16], w[DUAL ? 16 : 1];
        tmem_ld16(taddr + c, v);
        if constexpr (DUAL) tmem_ld16(taddr + BN + c, w);
        tmem_ld_wait();
        if (row < p.Kf && col0 + c < p.N) {
          const uint32_t ncol = min(16u, p.N - (col0 + c));
          unsigned long long* o = reinterpret_cast<unsigned long long*>(p.acc64) + (size_t)row * p.N + col0 + c;
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (j < (int)ncol) {
              long long a = (long long)(int)v[j];
              if constexpr (DUAL) a = a * 256ll + (long long)(int)w[j];   // k = 256 * hi + lo
              a *= (long long)p.alpha;
              if (a != 0) atomicAdd(o + j, (unsigned long long)a);
            }
        }
      }
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      if (++acc == C::kAccStages) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  fence_before();
  __syncthreads();
  fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, C::kTmemCols);
}

// ---- host ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

void* driver_fn(const char* name) {
  void* f = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint(name, &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
  return f;
}

CUtensorMapSwizzle swizzle_of(uint32_t mode) {
  switch (mode) {
    case 0: return CU_TENSOR_MAP_SWIZZLE_NONE;
    case 1: return CU_TENSOR_MAP_SWIZZLE_32B;
    case 2: return CU_TENSOR_MAP_SWIZZLE_64B;
    default: return CU_TENSOR_MAP_SWIZZLE_128B;
  }
}

template <int BN, bool DUAL = false>
int launch(const CUtensorMap& ta, const CUtensorMap& ta2, const CUtensorMap& tb, const ConvParams& p, unsigned grid, cudaStream_t st) {
  static bool attr_done[16] = {};
  const int dev = device_info().device;
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv_fprop_kernel<BN, DUAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, FCfg<BN, DUAL>::kSmemBytes);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(conv_fprop_kernel)");
      return LBT_ECUDA;
    }
    attr_done[dev] = true;
  }
  launch_pdl(conv_fprop_kernel<BN, DUAL>, grid, kThreadsF, FCfg<BN, DUAL>::kSmemBytes, st, ta, ta2, tb, p);
  return check_launch(DUAL ? "lbt_conv_i8_fprop_dual" : "lbt_conv_i8_fprop");
}

}  // namespace
}  // namespace lbt

using namespace lbt;

extern "C" int lbt_conv_i8_fprop(const void* src, int src_kind, int N, int H, int W, int C, const void* wp, int w_kind,
                                 size_t ldw, int Cout, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH,
                                 int OW, const int32_t* ib_src, const int32_t* ib_w, int exp_const, const float* bias,
                                 float* out, size_t ldc, const lbt_qsite* q_out, int8_t* k_out, int64_t* sums,
                                 const float* addend, void* stream) {
  return conv_fprop_run(src, src_kind, N, H, W, C, wp, w_kind, ldw, Cout, kh, kw, sh, sw, pad_top, pad_left, OH, OW, ib_src, ib_w,
                        exp_const, bias, out, ldc, q_out, k_out, sums, addend, stream, nullptr, nullptr);
}

extern "C" int lbt_conv_i8_fprop_dual(const int8_t* src_hi, const uint8_t* src_lo, int N, int H, int W, int C, const void* wp, int w_kind,
                                      size_t ldw, int Cout, int kh, int kw, int pad_top, int pad_left, int OH, int OW,
                                      const int32_t* ib_src, const int32_t* ib_w, int exp_const, float* out, size_t ldc,
                                      const float* addend, void* stream) {
  if (!src_hi || !src_lo || !wp || !out) return LBT_EINVAL;
  if (ldc < (size_t)Cout) return LBT_EINVAL;
  return conv_fprop_run(src_hi, LBT_MANT_S8, N, H, W, C, wp, w_kind, ldw, Cout, kh, kw, 1, 1, pad_top, pad_left, OH, OW, ib_src, ib_w,
                        exp_const, nullptr, out, ldc, nullptr, nullptr, nullptr, addend, stream, nullptr, src_lo);
}

int lbt::conv_fprop_run(const void* src, int src_kind, int N, int H, int W, int C, const void* wp, int w_kind, size_t ldw, int Cout,
                        int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH, int OW, const int32_t* ib_src,
                        const int32_t* ib_w, int exp_const, const float* bias, float* out, size_t ldc, const lbt_qsite* q_out,
                        int8_t* k_out, int64_t* sums, const float* addend, void* stream, const OutRemap* remap, const void* src_lo) {
  const bool dual = src_lo != nullptr;   // src = high byte plane (s8), src_lo = low byte plane (u8) of a 16-bit source
  if (!src || !wp) return LBT_EINVAL;
  if (dual && (q_out || bias || !out || src_kind != LBT_MANT_S8 || (reinterpret_cast<uintptr_t>(src_lo) & 15))) return LBT_EUNSUPPORTED;
  if (q_out) {
    if (!k_out || !sums || !q_out->ib) return LBT_EINVAL;
    if (q_out->bits < 2 || q_out->bits > 8 || (Cout & 3)) return LBT_EUNSUPPORTED;
  } else if (!out) {
    return LBT_EINVAL;
  }
  if ((src_kind != LBT_MANT_S8 && src_kind != LBT_MANT_U8) || (w_kind != LBT_MANT_S8 && w_kind != LBT_MANT_U8)) return LBT_EINVAL;
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || Cout <= 0 || kh <= 0 || kw <= 0 || sh <= 0 || sw <= 0 || OH <= 0 || OW <= 0)
    return LBT_EINVAL;
  if (C % 16) return LBT_EUNSUPPORTED;
  // measured (benchmarks/gemm_bench.py --path 0|1): the cp.async gather wins for 16- and 32-byte pixel rows (3.1x / 1.1x),
  // the TMA im2col kernel for 64 bytes and more
  if (remap && q_out) return LBT_EINVAL;
  if (!dual && !remap && conv_ldg_enabled() && (C <= 32 || (C == 64 && conv_ldg_c64_halo() && conv_ldg_halo_applies(N, OH, OW, kh, kw, sh, sw, C))) &&
      conv_ldg_ok(C, Cout, kh, kw) && !(reinterpret_cast<uintptr_t>(src) & 15) &&
      !(reinterpret_cast<uintptr_t>(wp) & 15) && !(ldw & 15) && ldw >= (size_t)kh * kw * C && (q_out || ldc >= (size_t)Cout)) {
    LBT_REQUIRE_ARCH();   // narrow channels: the cp.async-gather kernel (conv_ldg.cu)
    return conv_ldg_run(src, src_kind, N, H, W, C, wp, w_kind, ldw, Cout, kh, kw, sh, sw, pad_top, pad_left, OH, OW, 0, ib_src,
                        ib_w, exp_const, bias, out, ldc, q_out, k_out, sums, addend, stream);
  }
  const uint32_t cb = C >= 128 ? 128u : (uint32_t)C;
  if (cb != 16 && cb != 32 && cb != 64 && cb != 128) return LBT_EUNSUPPORTED;
  if (C % cb) return LBT_EUNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(wp) & 15) || (ldw & 15)) return LBT_EUNSUPPORTED;
  if (!q_out && ldc < (size_t)Cout) return LBT_EINVAL;
  const size_t Ktot = (size_t)kh * kw * C;
  if (ldw < Ktot) return LBT_EINVAL;
  // stride-1 filters on 64- / 128-channel images that fill 8 x 16 patches: halo patches through the TMA engine (conv_halo.cu)
  if (conv_halo_applies(N, OH, OW, C, Cout, kh, kw, sh, sw)) {
    LBT_REQUIRE_ARCH();
    const int rc = conv_halo_run(src, src_kind, N, H, W, C, wp, w_kind, ldw, Cout, kh, kw, pad_top, pad_left, OH, OW, ib_src, ib_w,
                                 exp_const, bias, out, ldc, q_out, k_out, sums, addend, stream, remap, src_lo);
    if (!(dual && rc == LBT_EUNSUPPORTED)) return rc;   // two planes: the filter bank + two patches may not fit; im2col-TMA kernel below
  }
  // exactness bound of one s32 accumulator (two planes: the low plane is u8, so a u8 filter makes it u8 x u8)
  if (Ktot > max_products(dual ? LBT_MANT_U8 : src_kind, w_kind)) return LBT_EUNSUPPORTED;
  if (kh > 255 || kw > 255) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  const DeviceInfo& di = device_info();
  static EncodeTiledFn enc_tiled = reinterpret_cast<EncodeTiledFn>(driver_fn("cuTensorMapEncodeTiled"));
  static EncodeIm2colFn enc_im2col = reinterpret_cast<EncodeIm2colFn>(driver_fn("cuTensorMapEncodeIm2col"));
  if (!enc_tiled || !enc_im2col) return LBT_ECUDA;

  int bn = 256;
  for (int c : {16, 32, 64, 128, 256})
    if (c >= Cout) {
      bn = c;
      break;
    }
  if (dual && bn > 128) bn = 128;   // two accumulators of bn columns per stage
  if (dual && bn < 64) return LBT_EUNSUPPORTED;
  uint32_t mode = 0;
  while ((16u << mode) < cb) ++mode;

  ConvParams p{};
  p.M = (uint32_t)((size_t)N * OH * OW);
  p.N = (uint32_t)Cout;
  p.OW = (uint32_t)OW;
  p.OHW = (uint32_t)(OH * OW);
  p.d_OW = make_fastdiv(p.OW);
  p.d_OHW = make_fastdiv(p.OHW);
  if ((size_t)N * OH * OW >= (1ull << 31)) return LBT_EUNSUPPORTED;
  p.lower_w = -pad_left;
  p.lower_h = -pad_top;
  p.sw = sw;
  p.sh = sh;
  p.kw = (uint32_t)kw;
  p.taps = (uint32_t)(kh * kw);
  p.cchunks = (uint32_t)C / cb;
  p.ksteps_real = p.taps * p.cchunks;
  p.ksteps = p.ksteps_real + ((cb == 16 && (p.ksteps_real & 1)) ? 1 : 0);
  p.cb = cb;
  p.mode = mode;
  p.C = (uint32_t)C;
  p.m_tiles = (p.M + kBlockM - 1) / kBlockM;
  p.n_tiles = ((uint32_t)Cout + bn - 1) / bn;
  p.ibA = ib_src;
  p.ibB = ib_w;
  p.exp_const = exp_const;
  p.bias = bias;
  p.addend = q_out ? nullptr : addend;
  p.out = out;
  p.ldc = ldc;
  p.idesc = tc::make_idesc_i8(src_kind == LBT_MANT_S8, w_kind == LBT_MANT_S8, false, false, bn, kBlockM);
  p.idesc2 = tc::make_idesc_i8(false, w_kind == LBT_MANT_S8, false, false, bn, kBlockM);
  p.bnq.q = site_from_abi(q_out);
  p.bnq.k = k_out;
  p.bnq.sums = reinterpret_cast<long long*>(sums);
  p.bnq.rows_per_image = (uint32_t)(OH * OW);
  if (remap) {
    p.remap = 1;
    p.rs_n = remap->sn;
    p.rs_y = remap->sy;
    p.rs_x = remap->sx;
  }

  // A: im2col map over (C, W, H, N).  The bounding box of base pixels is [lower, dim + upper): with
  // lower = -pad_before and upper = pad_after - (k - 1) it has exactly (out - 1) * stride + 1 positions.
  CUtensorMap ta, ta2, tb;
  {
    cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t gstr[3] = {(cuuint64_t)C, (cuuint64_t)W * C, (cuuint64_t)H * W * C};
    // pad_after chosen so that the last output pixel's base position is inside the box
    const int upper_w = (OW - 1) * sw + 1 - W - pad_left;
    const int upper_h = (OH - 1) * sh + 1 - H - pad_top;
    int lower[2] = {-pad_left, -pad_top};
    int upper[2] = {upper_w, upper_h};
    cuuint32_t estr[4] = {1, (cuuint32_t)sw, (cuuint32_t)sh, 1};
    CUresult r = enc_im2col(&ta, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(src), gdim, gstr, lower, upper, cb, kBlockM,
                            estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(mode), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeIm2col");
      return LBT_ECUDA;
    }
    ta2 = ta;
    if (dual) {
      r = enc_im2col(&ta2, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(src_lo), gdim, gstr, lower, upper, cb, kBlockM,
                     estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(mode), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) {
        set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeIm2col(low plane)");
        return LBT_ECUDA;
      }
    }
  }
  {
    cuuint64_t gdim[2] = {(cuuint64_t)Ktot, (cuuint64_t)Cout};
    cuuint64_t gstr[1] = {(cuuint64_t)ldw};
    cuuint32_t box[2] = {cb, (cuuint32_t)bn};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc_tiled(&tb, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(wp), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(mode), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled(weights)");
      return LBT_ECUDA;
    }
  }
  const uint64_t tiles = (uint64_t)p.m_tiles * p.n_tiles;
  const uint64_t cap = (uint64_t)di.sm_count * (dual ? 1 : ctas_per_sm(bn));
  const unsigned grid = (unsigned)(tiles < cap ? tiles : cap);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dual) return bn == 64 ? launch<64, true>(ta, ta2, tb, p, grid, st) : launch<128, true>(ta, ta2, tb, p, grid, st);
  switch (bn) {
    case 16: return launch<16>(ta, ta2, tb, p, grid, st);
    case 32: return launch<32>(ta, ta2, tb, p, grid, st);
    case 64: return launch<64>(ta, ta2, tb, p, grid, st);
    case 128: return launch<128>(ta, ta2, tb, p, grid, st);
    default: return launch<256>(ta, ta2, tb, p, grid, st);
  }
}

namespace lbt {
namespace {
template <int BN, bool DUAL = false>
int launch_wgrad(const CUtensorMap& tx, const CUtensorMap& tg, const CUtensorMap& tg2, const WgradParams& p, unsigned grid, cudaStream_t st) {
  static bool attr_done[16] = {};
  const int dev = device_info().device;
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_kernel<BN, DUAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, WCfg<BN, DUAL>::kSmemBytes);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(conv_wgrad_kernel)");
      return LBT_ECUDA;
    }
    attr_done[dev] = true;
  }
  launch_pdl(conv_wgrad_kernel<BN, DUAL>, grid, kThreads, WCfg<BN, DUAL>::kSmemBytes, st, tx, tg, tg2, p);
  return check_launch(DUAL ? "lbt_conv_i8_wgrad_dual" : "lbt_conv_i8_wgrad");
}
}  // namespace
}  // namespace lbt

// g_lo != NULL: g is the high byte plane (s8) and g_lo the low one (u8) of a 16-bit gradient: one dual-accumulator launch
static int conv_wgrad_run(const void* src, int src_kind, int N, int H, int W, int C, const void* g, int g_kind, const void* g_lo, int Cout,
                          int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH, int OW, int64_t* acc64,
                          int alpha, int k_splits, void* stream) {
  const bool dual = g_lo != nullptr;
  if (!src || !g || !acc64) return LBT_EINVAL;
  if (dual && (g_kind != LBT_MANT_S8 || (reinterpret_cast<uintptr_t>(g_lo) & 15))) return LBT_EUNSUPPORTED;
  if ((src_kind != LBT_MANT_S8 && src_kind != LBT_MANT_U8) || (g_kind != LBT_MANT_S8 && g_kind != LBT_MANT_U8)) return LBT_EINVAL;
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || Cout <= 0 || kh <= 0 || kw <= 0 || sh <= 0 || sw <= 0 || OH <= 0 || OW <= 0)
    return LBT_EINVAL;
  const uint32_t cb = C >= 128 ? 128u : (uint32_t)C;
  const uint32_t cbn = Cout >= 128 ? 128u : (uint32_t)Cout;
  if ((cb != 16 && cb != 32 && cb != 64 && cb != 128) || (C % cb)) return LBT_EUNSUPPORTED;
  if ((cbn != 16 && cbn != 32 && cbn != 64 && cbn != 128) || (Cout % cbn)) return LBT_EUNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(g) & 15)) return LBT_EUNSUPPORTED;
  if (kh > 255 || kw > 255) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  // the gather wgrad only pays off for 16-byte pixel rows (elsewhere both kernels are bound by the int64 atomics)
  if (!dual && conv_ldg_enabled() && k_splits <= 0 && C == 16 && Cout <= 16 && conv_wgrad_ldg_ok(C, Cout, kh, kw)) {
    const int rc = conv_wgrad_ldg_run(src, src_kind, N, H, W, C, g, g_kind, Cout, kh, kw, sh, sw, pad_top, pad_left, OH, OW, acc64,
                                      alpha, stream);
    if (rc != LBT_EUNSUPPORTED) return rc;
  }
  const DeviceInfo& di = device_info();
  static EncodeTiledFn enc_tiled = reinterpret_cast<EncodeTiledFn>(driver_fn("cuTensorMapEncodeTiled"));
  static EncodeIm2colFn enc_im2col = reinterpret_cast<EncodeIm2colFn>(driver_fn("cuTensorMapEncodeIm2col"));
  if (!enc_tiled || !enc_im2col) return LBT_ECUDA;

  int bn = Cout >= 256 ? 256 : Cout;  // 16, 32, 64, 128 or 256 (Cout is a multiple of cbn)
  if (Cout > 128 && Cout % 256) bn = 128;
  if (dual && bn > 128) bn = 128;     // two accumulators of bn columns each per stage
  uint32_t mode_a = 0, mode_b = 0;
  while ((16u << mode_a) < cb) ++mode_a;
  while ((16u << mode_b) < cbn) ++mode_b;

  WgradParams p{};
  p.Mpix = (uint32_t)((size_t)N * OH * OW);
  p.N = (uint32_t)Cout;
  p.OW = (uint32_t)OW;
  p.OHW = (uint32_t)(OH * OW);
  p.d_OW = make_fastdiv(p.OW);
  p.d_OHW = make_fastdiv(p.OHW);
  if ((size_t)N * OH * OW >= (1ull << 31)) return LBT_EUNSUPPORTED;
  p.lower_w = -pad_left;
  p.lower_h = -pad_top;
  p.sw = sw;
  p.sh = sh;
  p.kw = (uint32_t)kw;
  p.cchunks = (uint32_t)C / cb;
  p.ksteps = (uint32_t)(kh * kw) * p.cchunks;
  p.cb = cb;
  p.mode_a = mode_a;
  p.cbn = cbn;
  p.mode_b = mode_b;
  p.nchunks = (uint32_t)bn / cbn;
  const uint32_t spb = kStageK / cb;
  p.m_tiles = (p.ksteps + spb - 1) / spb;
  p.n_tiles = ((uint32_t)Cout + bn - 1) / bn;
  p.pix_blocks = (p.Mpix + kBlockM - 1) / kBlockM;
  uint32_t splits = k_splits > 0 ? (uint32_t)k_splits : 0;
  if (!splits) {
    const uint32_t tiles = p.m_tiles * p.n_tiles;
    splits = (uint32_t)(di.sm_count * ctas_per_sm(bn)) / (tiles ? tiles : 1);
    // every split ends in Kf x Cout int64 atomics: give it at least 8 pixel blocks of work (measured optimum on the
    // ResNet-20 shapes, benchmarks/wgrad_sweep.py)
    if (splits > p.pix_blocks / 8) splits = p.pix_blocks / 8;
    if (splits < 1) splits = 1;
  }
  if (splits > p.pix_blocks) splits = p.pix_blocks;
  p.blocks_per_split = (p.pix_blocks + splits - 1) / splits;
  // s32 exactness bound per CTA; two planes: the low one is u8, so a u8 source makes it u8 x u8
  const uint32_t max_blocks = max_products(src_kind, dual ? LBT_MANT_U8 : g_kind) / kBlockM;
  if (p.blocks_per_split > max_blocks) p.blocks_per_split = max_blocks;
  p.k_splits = (p.pix_blocks + p.blocks_per_split - 1) / p.blocks_per_split;
  p.Kf = (uint32_t)(kh * kw * C);
  p.acc64 = reinterpret_cast<long long*>(acc64);
  p.alpha = alpha;
  p.idesc = tc::make_idesc_i8(src_kind == LBT_MANT_S8, g_kind == LBT_MANT_S8, true, true, bn, kBlockM);
  p.idesc2 = tc::make_idesc_i8(src_kind == LBT_MANT_S8, false, true, true, bn, kBlockM);

  CUtensorMap tx, tg, tg2;
  {
    cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t gstr[3] = {(cuuint64_t)C, (cuuint64_t)W * C, (cuuint64_t)H * W * C};
    int lower[2] = {-pad_left, -pad_top};
    int upper[2] = {(OW - 1) * sw + 1 - W - pad_left, (OH - 1) * sh + 1 - H - pad_top};
    cuuint32_t estr[4] = {1, (cuuint32_t)sw, (cuuint32_t)sh, 1};
    CUresult r = enc_im2col(&tx, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(src), gdim, gstr, lower, upper, cb, kBlockM,
                            estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(mode_a), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeIm2col(wgrad)");
      return LBT_ECUDA;
    }
  }
  {
    cuuint64_t gdim[2] = {(cuuint64_t)Cout, (cuuint64_t)p.Mpix};
    cuuint64_t gstr[1] = {(cuuint64_t)Cout};
    cuuint32_t box[2] = {cbn, (cuuint32_t)kBlockM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc_tiled(&tg, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(g), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(mode_b), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled(grad)");
      return LBT_ECUDA;
    }
    tg2 = tg;
    if (dual) {
      r = enc_tiled(&tg2, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(g_lo), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(mode_b), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) {
        set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled(grad, low plane)");
        return LBT_ECUDA;
      }
    }
  }
  const uint64_t items = (uint64_t)p.m_tiles * p.n_tiles * p.k_splits;
  const uint64_t cap = (uint64_t)di.sm_count * ctas_per_sm(bn);
  const unsigned grid = (unsigned)(items < cap ? items : cap);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dual) {
    switch (bn) {
      case 16: return launch_wgrad<16, true>(tx, tg, tg2, p, grid, st);
      case 32: return launch_wgrad<32, true>(tx, tg, tg2, p, grid, st);
      case 64: return launch_wgrad<64, true>(tx, tg, tg2, p, grid, st);
      default: return launch_wgrad<128, true>(tx, tg, tg2, p, grid, st);
    }
  }
  switch (bn) {
    case 16: return launch_wgrad<16>(tx, tg, tg2, p, grid, st);
    case 32: return launch_wgrad<32>(tx, tg, tg2, p, grid, st);
    case 64: return launch_wgrad<64>(tx, tg, tg2, p, grid, st);
    case 128: return launch_wgrad<128>(tx, tg, tg2, p, grid, st);
    default: return launch_wgrad<256>(tx, tg, tg2, p, grid, st);
  }
}

extern "C" int lbt_conv_i8_wgrad(const void* src, int src_kind, int N, int H, int W, int C, const void* g, int g_kind, int Cout,
                                 int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH, int OW, int64_t* acc64,
                                 int alpha, int k_splits, void* stream) {
  return conv_wgrad_run(src, src_kind, N, H, W, C, g, g_kind, nullptr, Cout, kh, kw, sh, sw, pad_top, pad_left, OH, OW, acc64, alpha,
                        k_splits, stream);
}

extern "C" int lbt_conv_i8_wgrad_dual(const void* src, int src_kind, int N, int H, int W, int C, const int8_t* g_hi, const uint8_t* g_lo,
                                      int Cout, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH, int OW,
                                      int64_t* acc64, int alpha, int k_splits, void* stream) {
  if (!g_lo) return LBT_EINVAL;
  return conv_wgrad_run(src, src_kind, N, H, W, C, g_hi, LBT_MANT_S8, g_lo, Cout, kh, kw, sh, sw, pad_top, pad_left, OH, OW, acc64,
                        alpha, k_splits, stream);
}

// ------------------------------------------------------------------------------------------------
// Input gradient of a downsampling block in ONE persistent launch (lbt_conv_i8_dgrad_block):
//
//   dX = dgrad_{kh x kw / s}(g, W2)  [+ dgrad_{1x1 / s}(g_short, W_short)]  [+ addend]
//
// The tile list runs over (parity class, M tile, N tile) of every class of lbt_conv_i8_dgrad_strided's decomposition, classes
// with the most K-steps first and each class's tiles together (its slice of g stays in L2).  Per class: its own im2col map of
// g (sub-filter extents and padding differ), the K column of its sub-filter in the class-ordered W2 and the (a::sh, b::sw)
// sub-lattice of dX it writes.  The 1x1/s shortcut samples exactly class (0, 0): its rows are g_short's rows in order, so its
// K-steps (plain 2-D tiles of g_short and W_short) go into a second accumulator at +BN columns of the same tile, and the
// epilogue writes RN(f_main + f_short) there — the rounding of the shortcut dgrad followed by the main dgrad with it as
// addend.  Classes no tap reaches (a 1x1/s main convolution) are tiles without K-steps: the epilogue writes the addend or 0.
// ------------------------------------------------------------------------------------------------
namespace lbt {
namespace {

constexpr int kBlkMaxClasses = 4;   // strides <= 2

struct BlkClass {
  uint32_t M, OW, OHW;       // pixels of the class, its grid width, Hc * Wc
  FastDiv d_OW, d_OHW;
  int lower_w, lower_h;      // -pad_left, -pad_top of the class's stride-1 sub-convolution
  uint32_t kw;               // sub-filter width
  uint32_t ksteps;           // main K-steps (taps * channel chunks; 0: no tap reaches the class)
  uint32_t kcol;             // first K column of the sub-filter in W2
  uint32_t shortcut;         // 1: the shortcut's pixels are this class's pixels
  uint32_t tile0, m_tiles;   // first tile of the class in the tile list, its M tiles
  long long out_off;         // element offset of the class's first pixel in dX
};

struct BlkParams {
  uint32_t nclasses;
  BlkClass cls[kBlkMaxClasses];
  uint32_t total_tiles, n_tiles, N;   // N: dX channels
  uint32_t cb, mode;                  // channel chunk bytes of g and g_short, log2(cb / 16)
  uint32_t cchunks_g;                 // Cout / cb
  uint32_t ks_short;                  // shortcut K-steps (0: no shortcut)
  const int32_t *ib_g, *ib_w, *ib_gs, *ib_ws;
  int exp_const, exp_short;
  const float* addend;
  float* out;
  long long rs_n, rs_y, rs_x;
  uint32_t idesc, idesc_s;
};

struct BlkMaps {
  CUtensorMap a[kBlkMaxClasses];   // im2col of g per class
  CUtensorMap b;                   // W2[Cin, kh*kw*Cout]
  CUtensorMap as, bs;              // g_short rows, W_short[Cin, Cout_s]
};

// Two accumulators (main, shortcut) per TMEM stage; two CTAs per SM share the 512 columns
template <int BN>
struct BCfg {
  static constexpr int kStageA = Cfg<BN>::kStageA;
  static constexpr int kStageB = Cfg<BN>::kStageB;
  static constexpr int kStageBytes = kStageA + kStageB;
  static constexpr int kCtasPerSm = 2;
  static constexpr int kStages = BN <= 64 ? 4 : 3;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;
  static constexpr int kAccW = 2 * BN;
  static constexpr int kAccStages = (512 / kCtasPerSm) / kAccW;
  static constexpr int kTmemCols = kAccStages * kAccW;
  static_assert(kAccStages >= 1, "block dgrad accumulators");
  static_assert(kCtasPerSm * kSmemBytes <= 227 * 1024, "shared memory budget");
  static_assert(kCtasPerSm * kTmemCols <= 512, "tensor memory budget");
};

__device__ __forceinline__ uint32_t blk_class_of(const BlkParams& p, uint32_t tile) {
  uint32_t c = 0;
  while (c + 1 < p.nclasses && tile >= p.cls[c + 1].tile0) ++c;
  return c;
}

template <int BN>
__global__ void __launch_bounds__(kThreadsF, BCfg<BN>::kCtasPerSm)
conv_dgrad_block_kernel(const __grid_constant__ BlkMaps maps, const __grid_constant__ BlkParams p) {
  using C = BCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[C::kStages];
  __shared__ __align__(8) uint64_t empty_bar[C::kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[C::kAccStages];
  __shared__ __align__(8) uint64_t tmem_empty_bar[C::kAccStages];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_abort;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < C::kAccStages; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], kEpiWarps);
    }
    s_abort = 0;
    fence_barrier_init();
    for (uint32_t c = 0; c < p.nclasses; ++c)
      if (p.cls[c].ksteps) tma_prefetch_desc(&maps.a[c]);
    tma_prefetch_desc(&maps.b);
    if (p.ks_short) {
      tma_prefetch_desc(&maps.as);
      tma_prefetch_desc(&maps.bs);
    }
  }
  if (warp == 1) tmem_alloc(&tmem_slot, C::kTmemCols);
  pdl_trigger();
  fence_before();
  __syncthreads();
  fence_after();
  pdl_wait();   // everything above touched only shared / tensor memory and kernel parameters
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);
  volatile int* abort_flag = &s_abort;

  const uint32_t spb = kStageK / p.cb;   // tap-blocks per stage
  const uint32_t a_block = kBlockM * p.cb, b_block = BN * p.cb;
  const uint32_t ss_short = (p.ks_short + spb - 1) / spb;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      bool ok = true;
      for (uint32_t tile = blockIdx.x; tile < p.total_tiles && ok; tile += gridDim.x) {
        const uint32_t ci = blk_class_of(p, tile);
        const BlkClass& k = p.cls[ci];
        const uint32_t ss_main = (k.ksteps + spb - 1) / spb, ss_sc = k.shortcut ? ss_short : 0u;
        if (ss_main + ss_sc == 0) continue;
        const uint32_t local = tile - k.tile0;
        const uint32_t m_tile = local % k.m_tiles, n_tile = local / k.m_tiles;
        const uint32_t m0 = m_tile * kBlockM;
        const uint32_t img = fastdiv(m0, k.d_OHW), rem = m0 - img * k.OHW;
        const uint32_t ohu = fastdiv(rem, k.d_OW);
        const int base_w = k.lower_w + (int)(rem - ohu * k.OW), base_h = k.lower_h + (int)ohu;
        uint32_t cc = 0, r = 0, s = 0;   // running decomposition of the main K-step into (channel chunk, tap)
        for (uint32_t ks = 0; ks < ss_main + ss_sc && ok; ++ks) {
          if (!(ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag, &g_conv_error))) break;
          uint8_t* sa = smem + stage * C::kStageBytes;
          uint8_t* sb = sa + C::kStageA;
          if (ks < ss_main) {
            const uint32_t k0 = ks * spb, nblk = min(spb, k.ksteps - k0);
            mbar_expect_tx(&full_bar[stage], nblk * (a_block + b_block));
            for (uint32_t j = 0; j < nblk; ++j) {
              tma_load_im2col_4d(&maps.a[ci], &full_bar[stage], sa + j * a_block, (int)(cc * p.cb), base_w, base_h, (int)img,
                                 (uint16_t)s, (uint16_t)r);
              tma_load_2d(&maps.b, &full_bar[stage], sb + j * b_block, (int)(k.kcol + (k0 + j) * p.cb), (int)(n_tile * BN));
              if (++cc == p.cchunks_g) {
                cc = 0;
                if (++s == k.kw) {
                  s = 0;
                  ++r;
                }
              }
            }
          } else {   // the shortcut: plain tiles of g_short's rows (the class's pixels in order) and of W_short
            const uint32_t k0 = (ks - ss_main) * spb, nblk = min(spb, p.ks_short - k0);
            mbar_expect_tx(&full_bar[stage], nblk * (a_block + b_block));
            for (uint32_t j = 0; j < nblk; ++j) {
              tma_load_2d(&maps.as, &full_bar[stage], sa + j * a_block, (int)((k0 + j) * p.cb), (int)m0);
              tma_load_2d(&maps.bs, &full_bar[stage], sb + j * b_block, (int)((k0 + j) * p.cb), (int)(n_tile * BN));
            }
          }
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      bool ok = true;
      for (uint32_t tile = blockIdx.x; tile < p.total_tiles && ok; tile += gridDim.x) {
        const BlkClass& k = p.cls[blk_class_of(p, tile)];
        const uint32_t ss_main = (k.ksteps + spb - 1) / spb, ss_sc = k.shortcut ? ss_short : 0u;
        if (ss_main + ss_sc == 0) continue;
        if (!(ok = mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, abort_flag, &g_conv_error))) break;
        fence_after();
        const uint32_t d_main = tmem_base + acc * C::kAccW;
        for (uint32_t ks = 0; ks < ss_main + ss_sc; ++ks) {
          if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag, &g_conv_error))) break;
          fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::kStageBytes);
          const uint32_t sb = sa + C::kStageA;
          const bool sc = ks >= ss_main;
          const uint32_t k0 = (sc ? ks - ss_main : ks) * spb;
          const uint32_t nblk = min(spb, (sc ? p.ks_short : k.ksteps) - k0);
          const uint32_t d = sc ? d_main + BN : d_main;
          const uint32_t idesc = sc ? p.idesc_s : p.idesc;
          const uint32_t per_block = p.cb / 32;
          for (uint32_t j = 0; j < nblk; ++j)
            for (uint32_t kk = 0; kk < per_block; ++kk) {
              const uint32_t accumulate = (k0 + j > 0 || kk > 0) ? 1u : 0u;   // each accumulator starts at its first K-step
              umma_i8(d, make_desc_kmajor(sa + j * a_block + kk * 32, (int)p.mode, 16),
                      make_desc_kmajor(sb + j * b_block + kk * 32, (int)p.mode, 16), idesc, accumulate);
            }
          umma_commit(&empty_bar[stage]);
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (!ok) break;
        umma_commit(&tmem_full_bar[acc]);
        if (++acc == C::kAccStages) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    const uint32_t quad = warp & 3;
    const uint32_t half = (uint32_t)(warp - 2) >> 2;   // which of the quadrant's two warps: chunks half, half + 2, ...
    const float scale = exp2i(p.exp_const + *p.ib_g + *p.ib_w);
    const float scale_s = p.ks_short ? exp2i(p.exp_short + *p.ib_gs + *p.ib_ws) : 0.f;
    uint32_t acc = 0, acc_phase = 0;
    bool ok = true;
    for (uint32_t tile = blockIdx.x; tile < p.total_tiles && ok; tile += gridDim.x) {
      const BlkClass& k = p.cls[blk_class_of(p, tile)];
      const bool has_m = k.ksteps != 0, has_s = k.shortcut && p.ks_short;   // warp-uniform
      const bool has_acc = has_m || has_s;
      const uint32_t local = tile - k.tile0;
      const uint32_t m_tile = local % k.m_tiles, n_tile = local / k.m_tiles;
      const uint32_t row = m_tile * kBlockM + quad * 32 + lane;
      const uint32_t col0 = n_tile * BN;
      if (has_acc) {
        ok = mbar_wait(&tmem_full_bar[acc], acc_phase, abort_flag, &g_conv_error);
        ok = __all_sync(0xffffffffu, ok);
        if (!ok) break;
        fence_after();
      }
      const uint32_t taddr = tmem_base + acc * C::kAccW + ((quad * 32u) << 16);
      float* orow = nullptr;
      if (row < k.M) {
        const uint32_t img = fastdiv(row, k.d_OHW), rem = row - img * k.OHW;
        const uint32_t oh = fastdiv(rem, k.d_OW), ow = rem - oh * k.OW;
        orow = p.out + (k.out_off + (long long)img * p.rs_n + (long long)oh * p.rs_y + (long long)ow * p.rs_x) + col0;
      }
#pragma unroll 1
      for (int c = 16 * (int)half; c < BN; c += 32) {
        uint32_t v[16], w[16];
        if (has_m) tmem_ld16(taddr + c, v);
        if (has_s) tmem_ld16(taddr + BN + c, w);
        if (has_acc) tmem_ld_wait();
        if (orow && col0 + c < p.N) {   // N is a multiple of BN: whole 16-column chunks
          float* o = orow + c;
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = has_m ? __int2float_rn((int)v[j]) * scale : 0.f;
          if (has_s) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float fs = __int2float_rn((int)w[j]) * scale_s;
              f[j] = has_m ? __fadd_rn(f[j], fs) : fs;
            }
          } else if (p.addend) {   // + an fp32 tensor of dX's shape (the other branch of a gradient sum)
            const float4* ad = reinterpret_cast<const float4*>(p.addend + (o - p.out));
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 a4 = __ldcs(ad + j);
              f[4 * j + 0] = has_m ? __fadd_rn(f[4 * j + 0], a4.x) : a4.x;
              f[4 * j + 1] = has_m ? __fadd_rn(f[4 * j + 1], a4.y) : a4.y;
              f[4 * j + 2] = has_m ? __fadd_rn(f[4 * j + 2], a4.z) : a4.z;
              f[4 * j + 3] = has_m ? __fadd_rn(f[4 * j + 3], a4.w) : a4.w;
            }
          }
#pragma unroll
          for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
        }
      }
      if (has_acc) {
        fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
        if (++acc == C::kAccStages) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  }

  fence_before();
  __syncthreads();
  fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, C::kTmemCols);
}

template <int BN>
int launch_block(const BlkMaps& maps, const BlkParams& p, unsigned grid, cudaStream_t st) {
  static bool attr_done[16] = {};
  const int dev = device_info().device;
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv_dgrad_block_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, BCfg<BN>::kSmemBytes);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(conv_dgrad_block_kernel)");
      return LBT_ECUDA;
    }
    attr_done[dev] = true;
  }
  launch_pdl(conv_dgrad_block_kernel<BN>, grid, kThreadsF, BCfg<BN>::kSmemBytes, st, maps, p);
  return check_launch("lbt_conv_i8_dgrad_block");
}

}  // namespace
}  // namespace lbt

// Arguments are validated by lbt_conv_i8_dgrad_block (conv_dgrad.cu); this builds the class table and the tensor maps.
int lbt::conv_dgrad_block_run(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* w2, int w_kind, size_t ldw, int Cin,
                              int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W, const int32_t* ib_g,
                              const int32_t* ib_w, int exp_const, const void* gs, int gs_kind, int Cout_s, const void* ws, int ws_kind,
                              size_t ldws, const int32_t* ib_gs, const int32_t* ib_ws, int exp_short, float* dx, size_t ldc,
                              const float* addend, void* stream) {
  const uint32_t cb = Cout >= 128 ? 128u : (uint32_t)Cout;
  uint32_t mode = 0;
  while ((16u << mode) < cb) ++mode;
  const int bn = Cin == 64 ? 64 : 128;
  LBT_REQUIRE_ARCH();
  const DeviceInfo& di = device_info();
  static EncodeTiledFn enc_tiled = reinterpret_cast<EncodeTiledFn>(driver_fn("cuTensorMapEncodeTiled"));
  static EncodeIm2colFn enc_im2col = reinterpret_cast<EncodeIm2colFn>(driver_fn("cuTensorMapEncodeIm2col"));
  if (!enc_tiled || !enc_im2col) return LBT_ECUDA;

  BlkParams p{};
  BlkMaps maps;
  memset(&maps, 0, sizeof(maps));
  p.n_tiles = (uint32_t)Cin / bn;
  p.N = (uint32_t)Cin;
  p.cb = cb;
  p.mode = mode;
  p.cchunks_g = (uint32_t)Cout / cb;
  p.ks_short = gs ? (uint32_t)Cout_s / cb : 0u;
  p.ib_g = ib_g;
  p.ib_w = ib_w;
  p.ib_gs = ib_gs;
  p.ib_ws = ib_ws;
  p.exp_const = exp_const;
  p.exp_short = exp_short;
  p.addend = addend;
  p.out = dx;
  p.rs_n = (long long)H * W * (long long)ldc;
  p.rs_y = (long long)sh * W * (long long)ldc;
  p.rs_x = (long long)sw * (long long)ldc;
  p.idesc = tc::make_idesc_i8(g_kind == LBT_MANT_S8, w_kind == LBT_MANT_S8, false, false, bn, kBlockM);
  p.idesc_s = tc::make_idesc_i8(gs_kind == LBT_MANT_S8, ws_kind == LBT_MANT_S8, false, false, bn, kBlockM);

  // classes with the most K-steps first (stable), each class's tiles together
  struct Cls {
    int a, b, work;
  } order[kBlkMaxClasses];
  int nc = 0;
  for (int a = 0; a < sh && a < H; ++a)
    for (int b = 0; b < sw && b < W; ++b) {
      const int r0 = (a + pad_top) % sh, s0 = (b + pad_left) % sw;
      const int work = class_count(r0, kh, sh) * class_count(s0, kw, sw) * (int)p.cchunks_g + (a == 0 && b == 0 ? (int)p.ks_short : 0);
      int i = nc++;
      while (i > 0 && order[i - 1].work < work) {
        order[i] = order[i - 1];
        --i;
      }
      order[i] = Cls{a, b, work};
    }
  p.nclasses = (uint32_t)nc;
  uint32_t tile0 = 0;
  for (int i = 0; i < nc; ++i) {
    const int a = order[i].a, b = order[i].b;
    const int Hc = (H - a + sh - 1) / sh, Wc = (W - b + sw - 1) / sw;
    const int r0 = (a + pad_top) % sh, s0 = (b + pad_left) % sw;
    const int nr = class_count(r0, kh, sh), ncol = class_count(s0, kw, sw);
    BlkClass& k = p.cls[i];
    k.M = (uint32_t)N * (uint32_t)(Hc * Wc);
    k.OW = (uint32_t)Wc;
    k.OHW = (uint32_t)(Hc * Wc);
    k.d_OW = make_fastdiv(k.OW);
    k.d_OHW = make_fastdiv(k.OHW);
    k.shortcut = (a == 0 && b == 0 && gs) ? 1u : 0u;
    k.m_tiles = (k.M + kBlockM - 1) / kBlockM;
    k.tile0 = tile0;
    tile0 += k.m_tiles * p.n_tiles;
    k.out_off = ((long long)a * W + b) * (long long)ldc;
    k.ksteps = (uint32_t)(nr * ncol) * p.cchunks_g;
    if (!k.ksteps) continue;
    const int pt2 = nr - 1 - (a + pad_top) / sh, pl2 = ncol - 1 - (b + pad_left) / sw;
    k.lower_w = -pl2;
    k.lower_h = -pt2;
    k.kw = (uint32_t)ncol;
    k.kcol = class_group_offset(r0, s0, kh, kw, sh, sw) * (uint32_t)Cout;
    // the class's stride-1 sub-convolution of g: box of base pixels [lower, OW + upper) with exactly Wc (Hc) positions
    cuuint64_t gdim[4] = {(cuuint64_t)Cout, (cuuint64_t)OW, (cuuint64_t)OH, (cuuint64_t)N};
    cuuint64_t gstr[3] = {(cuuint64_t)Cout, (cuuint64_t)OW * Cout, (cuuint64_t)OH * OW * Cout};
    int lower[2] = {-pl2, -pt2};
    int upper[2] = {Wc - OW - pl2, Hc - OH - pt2};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc_im2col(&maps.a[i], CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(g), gdim, gstr, lower, upper, cb, kBlockM,
                            estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(mode), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeIm2col(block dgrad)");
      return LBT_ECUDA;
    }
  }
  p.total_tiles = tile0;
  auto tiled = [&](CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch, uint32_t rows,
                   CUtensorMapL2promotion l2, const char* what) {
    cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    cuuint64_t gstr[1] = {(cuuint64_t)pitch};
    cuuint32_t box[2] = {cb, rows};
    cuuint32_t estr[2] = {1, 1};
    if (enc_tiled(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle_of(mode), l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
      set_cuda_error(cudaErrorInvalidValue, what);
      return false;
    }
    return true;
  };
  if (!tiled(&maps.b, w2, (uint64_t)kh * kw * Cout, (uint64_t)Cin, ldw, (uint32_t)bn, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             "cuTensorMapEncodeTiled(block dgrad weights)"))
    return LBT_ECUDA;
  if (gs) {
    const uint64_t rows_s = (uint64_t)N * ((H + sh - 1) / sh) * ((W + sw - 1) / sw);
    if (!tiled(&maps.as, gs, (uint64_t)Cout_s, rows_s, (uint64_t)Cout_s, (uint32_t)kBlockM, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               "cuTensorMapEncodeTiled(block dgrad shortcut gradient)") ||
        !tiled(&maps.bs, ws, (uint64_t)Cout_s, (uint64_t)Cin, ldws, (uint32_t)bn, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               "cuTensorMapEncodeTiled(block dgrad shortcut weights)"))
      return LBT_ECUDA;
  }
  const uint64_t cap = (uint64_t)di.sm_count * BCfg<64>::kCtasPerSm;
  const unsigned grid = (unsigned)(p.total_tiles < cap ? p.total_tiles : cap);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return bn == 64 ? launch_block<64>(maps, p, grid, st) : launch_block<128>(maps, p, grid, st);
}

extern "C" int lbt_conv_debug_error(void) {
  int v = 0, zero = 0;
  if (cudaMemcpyFromSymbol(&v, g_conv_error, sizeof(int)) != cudaSuccess) return -1;
  cudaMemcpyToSymbol(g_conv_error, &zero, sizeof(int));
  const int h = conv_halo_debug_error();
  if (h > 0) v |= h;
  const int st = conv_stem_debug_error();
  if (st > 0) v |= st;
  return v;
}
