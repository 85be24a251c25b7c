// Integer-mantissa GEMM on the 5th-gen tensor cores of B200 (sm_100a only):
//
//     D[M,N] (s32, in TMEM)  =  A[M,K] (u8|s8, K-major)  x  B[N,K]^T (u8|s8, K-major)
//
// TMA (cp.async.bulk.tensor, 128B swizzle) -> shared memory ring -> tcgen05.mma.kind::i8 (M128 x BN x K32,
// issued by one thread) -> s32 accumulators in tensor memory (double buffered) -> tcgen05.ld epilogue.
// Replaces the fp32 cuBLAS/cuDNN GEMMs the reference runs on fake-quantised floats
// (tf.matmul dynamic_fixed_point.py:388, tf.nn.conv2d :291 and their tf.gradients :302-305, :457-460):
// the products of DFXP mantissas are accumulated EXACTLY in int32, and the epilogue applies the
// power-of-two rescale 2^(ibA + ibB + const) read from the layers' range variables on the device.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (TMEM lane quadrant = warp % 4).  Persistent CTAs over (m-tile, n-tile, k-split).
//
// Epilogues:
//   LBT_EPI_F32   out[m, n] = fp32(acc) * 2^e (+ bias[n])            (fprop / dgrad / dense)
//   LBT_EPI_ACC64 acc64[m, n] += alpha * acc   (64-bit atomics)       (wgrad split-K: order-independent,
//                 bit-reproducible; per-split K <= 65536, or 32768 for u8 x u8, keeps the s32 partial exact, SURVEY.md H3)
#include <cuda.h>

#include "qsite.cuh"

namespace lbt {
namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 128;  // bytes == int8 elements == one 128B swizzle row
constexpr int kUmmaK = 32;    // kind::i8: 32 bytes of K per instruction
constexpr int kEpiWarps = 8;   // two warps per TMEM lane quadrant, interleaved over the 16-column chunks
constexpr int kThreads = 32 * (2 + kEpiWarps);
constexpr long long kWatchdogCycles = 4000000000ll;
#ifndef LBT_SUSPEND_HINT_NS
#define LBT_SUSPEND_HINT_NS 0
#endif
constexpr uint32_t kSuspendHintNs = LBT_SUSPEND_HINT_NS;   // see tcgen05.cuh

__device__ int g_gemm_error = 0;

struct GemmParams {
  uint32_t M, N, K;
  uint32_t m_tiles, n_tiles, k_blocks, k_blocks_per_split, k_splits;
  int epilogue;
  const int32_t* ibA;
  const int32_t* ibB;
  int exp_const;
  const float* bias;
  const float* addend;           // optional fp32 [M, ldc] added to the fp32 result (F32 epilogue only)
  float* out;
  size_t ldc;
  long long* acc64;
  int alpha;
  uint32_t idesc;
  uint32_t idesc2;   // DUAL: descriptor of the low-half MMAs (A = u8)
  BnqParams bnq;  // fused re-quantising epilogue (bnq.q.bits == 0: off)
};

// ---- PTX wrappers ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  if (kSuspendHintNs == 0) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
  }
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kSuspendHintNs)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as an error flag, never as a hung GPU.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, volatile int* abort_flag) {
  uint32_t spins = 0;
  long long t0 = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3f) == 0) {
      if (*abort_flag) return false;
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      if (now - t0 > kWatchdogCycles) {  // ~2 s: something is wrong with the pipeline protocol
        *abort_flag = 1;
        atomicExch(&g_gemm_error, 1);
        return false;
      }
    }
  }
  return true;
}

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::i8, s32 accumulate.
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// All previously issued MMAs of this thread arrive on `bar` when they complete.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor: K-major operand tile, 128-byte swizzle (rows of 128 B, 8-row
// atoms 1024 B apart).  Fields (PTX ISA "tcgen05 matrix descriptor"): [0,14) address>>4,
// [16,30) leading byte offset>>4 (unused for swizzled K-major: 1), [32,46) stride byte offset>>4
// (1024>>4), [46,48) version = 1, [61,64) layout = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// DUAL: the A operand is a 9..16-bit mantissa split k = 256 * hi + lo (hi s8, lo u8: the 16-bit gradients of BASELINE
// config 5).  Both halves are staged per K block next to ONE copy of B, two accumulators per tile live in tensor memory
// (hi . B and lo . B, each exact in s32), and the epilogue combines them 256 * acc_hi + acc_lo in 64-bit integers before the
// single rounding to fp32 — the result is RN_fp32(exact 16x8-bit dot * 2^e), with no int64 round trip through HBM.
template <int BN, bool DUAL = false>
struct Cfg {
  static constexpr int kStageA = kBlockM * kBlockK;
  static constexpr int kStageA2 = DUAL ? kStageA : 0;
  static constexpr int kStageB = BN * kBlockK;
  static constexpr int kStageBytes = kStageA + kStageA2 + kStageB;
  static constexpr int kStages = (200 * 1024 / kStageBytes) > 8 ? 8 : (200 * 1024 / kStageBytes);
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;  // + alignment slack
  static constexpr int kAccCols = (DUAL ? 2 : 1) * BN;             // tensor-memory columns of one accumulator stage
  static constexpr int kTmemCols = (2 * kAccCols) < 32 ? 32 : (2 * kAccCols);
  static_assert(kTmemCols <= 512, "two accumulator stages must fit the 512 tensor-memory columns");
};

template <int BN, bool DUAL>
__global__ void __launch_bounds__(kThreads, 1)
gemm_i8_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB,
               const GemmParams p) {
  using C = Cfg<BN, DUAL>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[C::kStages];
  __shared__ __align__(8) uint64_t empty_bar[C::kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_abort;
  __shared__ int s_stat[kEpiWarps][2 * BN];
  __shared__ unsigned long long s_tot[2 * BN];  // CTA totals of the fused statistics (last N tile of the CTA)  // per epilogue warp: partial sum k, sum k^2 (fused BN statistics)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], kEpiWarps);  // one arrive per epilogue warp
    }
    s_abort = 0;
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    if (DUAL) tma_prefetch_desc(&tmA2);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, C::kTmemCols);
  for (uint32_t i = threadIdx.x; i < 2 * BN; i += kThreads) s_tot[i] = 0ull;
  pdl_trigger();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();   // everything above touched only shared / tensor memory and kernel parameters
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);
  volatile int* abort_flag = &s_abort;

  const uint32_t total_items = p.m_tiles * p.n_tiles * p.k_splits;

  if (warp == 0) {
    // ===== TMA producer (one lane) =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      bool ok = true;
      for (uint32_t item = blockIdx.x; item < total_items && ok; item += gridDim.x) {
        const uint32_t m_tile = item % p.m_tiles, rest = item / p.m_tiles;
        const uint32_t n_tile = rest % p.n_tiles, ks = rest / p.n_tiles;
        const uint32_t kb0 = ks * p.k_blocks_per_split;
        const uint32_t kb1 = min(kb0 + p.k_blocks_per_split, p.k_blocks);
        for (uint32_t kb = kb0; kb < kb1; ++kb) {
          if (!(ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag))) break;
          uint8_t* sa = smem + stage * C::kStageBytes;
          mbar_expect_tx(&full_bar[stage], C::kStageBytes);
          tma_load_2d(&tmA, &full_bar[stage], sa, (int)(kb * kBlockK), (int)(m_tile * kBlockM));
          if (DUAL) tma_load_2d(&tmA2, &full_bar[stage], sa + C::kStageA, (int)(kb * kBlockK), (int)(m_tile * kBlockM));
          tma_load_2d(&tmB, &full_bar[stage], sa + C::kStageA + C::kStageA2, (int)(kb * kBlockK), (int)(n_tile * BN));
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one lane) =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      bool ok = true;
      for (uint32_t item = blockIdx.x; item < total_items && ok; item += gridDim.x) {
        const uint32_t ks = (item / p.m_tiles) / p.n_tiles;
        const uint32_t kb0 = ks * p.k_blocks_per_split;
        const uint32_t kb1 = min(kb0 + p.k_blocks_per_split, p.k_blocks);
        if (!(ok = mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, abort_flag))) break;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * C::kAccCols;
        for (uint32_t kb = kb0; kb < kb1; ++kb) {
          if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag))) break;
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::kStageBytes);
          const uint64_t da = make_desc_sw128(sa), db = make_desc_sw128(sa + C::kStageA + C::kStageA2);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) {
            // advance the descriptor start address by k*32 bytes inside the 128B swizzle row
            umma_i8(d_tmem, da + (uint64_t)(k * (kUmmaK >> 4)), db + (uint64_t)(k * (kUmmaK >> 4)), p.idesc,
                    (kb > kb0 || k > 0) ? 1u : 0u);
          }
          if (DUAL) {   // the low halves against the same B tile, into the second accumulator
            const uint64_t da2 = make_desc_sw128(sa + C::kStageA);
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma_i8(d_tmem + BN, da2 + (uint64_t)(k * (kUmmaK >> 4)), db + (uint64_t)(k * (kUmmaK >> 4)), p.idesc2,
                      (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // frees the smem slot when these MMAs have read it
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (!ok) break;
        umma_commit(&tmem_full_bar[acc]);  // accumulator complete -> epilogue
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // ===== epilogue warps 2..5: TMEM -> registers -> global =====
    const uint32_t quad = warp & 3;  // TMEM lanes [32*quad, 32*quad+32) are the only ones this warp may read
    const uint32_t half = (uint32_t)(warp - 2) >> 2;  // which of the quadrant's two warps: chunks half, half + 2, ...
    int e = p.exp_const;
    if (p.ibA) e += *p.ibA;
    if (p.ibB) e += *p.ibB;
    const float scale = exp2i(e);
    const bool fused = p.bnq.q.bits != 0;   // host guarantees LBT_EPI_F32 and k_splits == 1
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
    for (uint32_t item = blockIdx.x; item < total_items && ok; item += gridDim.x) {
      const uint32_t m_tile = item % p.m_tiles, rest = item / p.m_tiles;
      const uint32_t n_tile = rest % p.n_tiles;
      const uint32_t row = m_tile * kBlockM + quad * 32 + lane;
      const uint32_t pix = fused ? row % p.bnq.rows_per_image : 0u;
      const uint32_t col0 = n_tile * BN;
      if (fused) {   // this warp's noise lines of the tile: into L1 while the accumulator is still being computed
#pragma unroll 1
        for (int c = (BN > 16 ? 16 * (int)half : 0); c < BN; c += (BN > 16 ? 32 : 16))
          bnq_prefetch(p.bnq, pix, p.N, col0 + (uint32_t)c, row < p.M && col0 + (uint32_t)c < p.N && !(BN == 16 && half));
      }
      ok = mbar_wait(&tmem_full_bar[acc], acc_phase, abort_flag);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * C::kAccCols + ((quad * 32u) << 16);
      if (fused && (n_tile != stat_ntile || bst.tiles >= (uint32_t)kBnqFlushTiles)) {
        bnq_flush(p.bnq, my_stat, stat_ntile * BN, BN, p.N, lane);
        stat_ntile = n_tile;
        bst.tiles = 0;
      }
      ++bst.tiles;
#pragma unroll 1
      for (int c = (BN > 16 ? 16 * (int)half : 0); c < BN; c += (BN > 16 ? 32 : 16)) {
        if (BN == 16 && half) break;  // a single chunk: the second warp of the quadrant has nothing to do
        uint32_t v[16];
        float4 u4[4];   // fused: the chunk's noise, requested before the accumulator wait (bnq_load_noise; not in the 64-register BN = 16 build)
        const bool fchunk = !DUAL && BN > 16 && fused && col0 + c < p.N;   // warp-uniform
        if (fchunk) bnq_load_noise(p.bnq, bst, pix, row < p.M, col0 + c, min(16u, p.N - (col0 + c)), p.N, u4);
        tmem_ld16(taddr + c, v);
        if (DUAL) {   // host guarantees LBT_EPI_F32, no fused quantiser, k_splits == 1
          uint32_t w[16];
          tmem_ld16(taddr + BN + c, w);
          tmem_ld_wait();
          if (row < p.M && col0 + c < p.N) {
            const uint32_t ncol = min(16u, p.N - (col0 + c));
            float* o = p.out + (size_t)row * p.ldc + col0 + c;
            float f[16];
#pragma unroll
            for (int j = 0; j < 16; ++j)   // 256 * (hi . B) + (lo . B): exact in 64 bits, ONE rounding to fp32
              f[j] = __ll2float_rn((long long)(int)v[j] * 256ll + (long long)(int)w[j]) * scale;
            if (p.addend) {
              const float* ad = p.addend + (o - p.out);
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (j < (int)ncol) f[j] = __fadd_rn(f[j], __ldcs(ad + j));
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
          continue;
        }
        tmem_ld_wait();
        if (fused) {
          if (col0 + c < p.N) {  // warp-uniform
            const uint32_t ncol = min(16u, p.N - (col0 + c));
            if (fchunk)
              bnq_chunk(p.bnq, bst, v, u4, scale, p.bias ? p.bias + col0 + c : nullptr, row, row < p.M, col0 + c, ncol, p.N, my_stat, BN,
                        (uint32_t)c, lane);
            else
              bnq_chunk(p.bnq, bst, v, scale, p.bias ? p.bias + col0 + c : nullptr, row, pix, row < p.M, col0 + c, ncol, p.N, my_stat, BN,
                        (uint32_t)c, lane);
          }
        } else if (row < p.M && col0 + c < p.N) {
          const uint32_t ncol = min(16u, p.N - (col0 + c));
          if (p.epilogue == LBT_EPI_F32) {
            float* o = p.out + (size_t)row * p.ldc + col0 + c;
            float f[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              f[j] = __int2float_rn((int)v[j]) * scale;
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
          } else {
            unsigned long long* o = reinterpret_cast<unsigned long long*>(p.acc64) + (size_t)row * p.ldc + col0 + c;
            if (p.k_splits == 1 && ncol == 16 && ((reinterpret_cast<uintptr_t>(o) & 15u) == 0)) {
              // one CTA owns this output element (no K split): plain 128-bit read-modify-write instead of 16 atomics
              ulonglong2* o2 = reinterpret_cast<ulonglong2*>(o);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                ulonglong2 t = o2[j];
                t.x += (unsigned long long)((long long)(int)v[2 * j] * (long long)p.alpha);
                t.y += (unsigned long long)((long long)(int)v[2 * j + 1] * (long long)p.alpha);
                o2[j] = t;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (j < (int)ncol) {
                  const long long a = (long long)(int)v[j] * (long long)p.alpha;
                  if (a != 0) atomicAdd(o + j, (unsigned long long)a);
                }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (fused && ok) {
      bnq_flush_cta(p.bnq, my_stat, s_tot, stat_ntile * BN, BN, p.N, lane, threadIdx.x - 64, 32 * kEpiWarps, 1);
      bnq_finish(p.bnq, bst, (unsigned long long)p.M * p.N, warp == 2, lane);
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, C::kTmemCols);
}

// =====================================================================================================================
// CTA-pair variant (tcgen05 cta_group::2) for large fp32-epilogue GEMMs.  One 128x256 tile per SM asks the L2 for
// (128 + 256) * 128 B per 512 tensor-core clocks = 96 B/clk/SM, more than the ~43 B/clk/SM the L2 can deliver to 148 SMs at
// once (B300_MICROARCH.md: ~6300 B/clk chip-wide), so the single-CTA kernel tops out near half of the tensor peak.  A pair
// of SMs (a 2-CTA cluster on one TPC) computes a 256x256 tile: each CTA stages ITS 128 rows of A and ITS 128 rows of B, the
// leader's single thread issues M256 x N256 x K32 instructions that read both shared memories, and each CTA's tensor memory
// receives its 128 accumulator rows: 64 B/clk/SM for the same math.
//
//   full_bar   (leader only)  : tx-count barrier; BOTH CTAs' TMA loads complete on it (.cta_group::2 loads may signal the peer)
//   empty_bar  (both)         : tcgen05.commit multicast — the smem slot of BOTH CTAs is free when the pair's MMAs have read it
//   tmem_full  (both)         : tcgen05.commit multicast — accumulator stage complete
//   tmem_empty (leader only)  : 2 x 8 epilogue warps arrive (the peer's remotely) before the leader reuses the stage
constexpr int k2BN = 256;              // columns of the pair's tile
constexpr int k2StageA = kBlockM * kBlockK;
constexpr int k2StageB = (k2BN / 2) * kBlockK;
constexpr int k2StageBytes = k2StageA + k2StageB;
constexpr int k2Stages = 6;
constexpr int k2SmemBytes = k2Stages * k2StageBytes + 1024;
constexpr int k2TmemCols = 512;        // two 256-column accumulator stages

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nid_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory object in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint32_t bar_cluster_addr, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_i8_pair(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair when the issued MMAs complete
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}

// Tile order: groups of 8 row-pairs x all column tiles, rows fastest inside a group, so the ~74 tiles in flight cover an
// 8 x 9 patch (34 MB of operands at K = 8192) instead of a full column of A: the operands stay in L2 between waves.
__device__ __forceinline__ void pair_tile(uint32_t item, uint32_t m_pairs, uint32_t n_tiles, uint32_t& m_pair, uint32_t& n_tile) {
  constexpr uint32_t kGroup = 8;
  const uint32_t gsz = kGroup * n_tiles, group = item / gsz, first_m = group * kGroup;
  const uint32_t gm = min(kGroup, m_pairs - first_m), within = item - group * gsz;
  n_tile = within / gm;
  m_pair = first_m + (within - n_tile * gm);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
gemm_i8_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[k2Stages];
  __shared__ __align__(8) uint64_t empty_bar[k2Stages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_abort;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();

  if (threadIdx.x == 0) {
    for (int s = 0; s < k2Stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], 2 * kEpiWarps);  // the epilogue warps of BOTH CTAs (leader's copy is the live one)
    }
    s_abort = 0;
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc_pair(&tmem_slot, k2TmemCols);
  tc_fence_before();
  cluster_sync_all();   // barriers of both CTAs initialised, tensor memory allocated
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);
  volatile int* abort_flag = &s_abort;

  const uint32_t m_pairs = (p.m_tiles + 1) / 2;
  const uint32_t total_items = m_pairs * p.n_tiles;
  const uint32_t first = cluster_id_x(), stride = cluster_nid_x();

  if (warp == 0) {
    // ===== TMA producer (one lane per CTA): my 128 rows of A, my 128 rows of B; completion on the LEADER's barrier =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      bool ok = true;
      for (uint32_t item = first; item < total_items && ok; item += stride) {
        uint32_t m_pair, n_tile;
        pair_tile(item, m_pairs, p.n_tiles, m_pair, n_tile);
        for (uint32_t kb = 0; kb < p.k_blocks; ++kb) {
          if (!(ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag))) break;
          uint8_t* sa = smem + stage * k2StageBytes;
          if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * k2StageBytes);
          const uint32_t bar = mapa_u32(smem_u32(&full_bar[stage]), 0);
          tma_load_2d_pair(&tmA, bar, sa, (int)(kb * kBlockK), (int)(m_pair * 2 * kBlockM + rank * kBlockM));
          tma_load_2d_pair(&tmB, bar, sa + k2StageA, (int)(kb * kBlockK), (int)(n_tile * k2BN + rank * (k2BN / 2)));
          if (++stage == k2Stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: one lane of the LEADER CTA drives both tensor cores =====
    if (lane == 0 && rank == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      bool ok = true;
      for (uint32_t item = first; item < total_items && ok; item += stride) {
        if (!(ok = mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, abort_flag))) break;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * k2BN;
        for (uint32_t kb = 0; kb < p.k_blocks; ++kb) {
          if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag))) break;
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * k2StageBytes);
          const uint64_t da = make_desc_sw128(sa), db = make_desc_sw128(sa + k2StageA);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k)
            umma_i8_pair(d_tmem, da + (uint64_t)(k * (kUmmaK >> 4)), db + (uint64_t)(k * (kUmmaK >> 4)), p.idesc,
                         (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit_pair(&empty_bar[stage]);
          if (++stage == k2Stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (!ok) break;
        umma_commit_pair(&tmem_full_bar[acc]);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // ===== epilogue warps (both CTAs): my 128 accumulator rows -> fp32 =====
    const uint32_t quad = warp & 3;
    const uint32_t half = (uint32_t)(warp - 2) >> 2;
    int e = p.exp_const;
    if (p.ibA) e += *p.ibA;
    if (p.ibB) e += *p.ibB;
    const float scale = exp2i(e);
    uint32_t acc = 0, acc_phase = 0;
    bool ok = true;
    for (uint32_t item = first; item < total_items && ok; item += stride) {
      uint32_t m_pair, n_tile;
      pair_tile(item, m_pairs, p.n_tiles, m_pair, n_tile);
      ok = mbar_wait(&tmem_full_bar[acc], acc_phase, abort_flag);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      tc_fence_after();
      const uint32_t row = m_pair * 2 * kBlockM + rank * kBlockM + quad * 32 + lane;
      const uint32_t col0 = n_tile * k2BN;
      const uint32_t taddr = tmem_base + acc * k2BN + ((quad * 32u) << 16);
#pragma unroll 1
      for (int c = 16 * (int)half; c < k2BN; c += 32) {
        uint32_t v[16];
        tmem_ld16(taddr + c, v);
        tmem_ld_wait();
        if (row < p.M && col0 + c < p.N) {
          const uint32_t ncol = min(16u, p.N - (col0 + c));
          float* o = p.out + (size_t)row * p.ldc + col0 + c;
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            f[j] = __int2float_rn((int)v[j]) * scale;
            if (p.bias && j < (int)ncol) f[j] = __fadd_rn(f[j], __ldg(p.bias + col0 + c + j));
          }
          if (p.addend) {
            const float* ad = p.addend + (o - p.out);
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < (int)ncol) f[j] = __fadd_rn(f[j], __ldg(ad + j));
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
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tmem_empty_bar[acc]), 0));
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();   // nobody leaves (or frees tensor memory) while the peer may still signal into this CTA
  tc_fence_after();
  if (warp == 1) tmem_dealloc_pair(tmem_base, k2TmemCols);
}

std::atomic<int> g_gemm_pair{1};       // lbt_gemm_set_pair(): 0 = always the single-CTA kernel

int launch_pair(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, unsigned clusters, cudaStream_t st) {
  static bool attr_done[16] = {};
  const int dev = device_info().device;
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(gemm_i8_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, k2SmemBytes);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(gemm_i8_pair_kernel)");
      return LBT_ECUDA;
    }
    attr_done[dev] = true;
  }
  gemm_i8_pair_kernel<<<2 * clusters, kThreads, k2SmemBytes, st>>>(ta, tb, p);
  return check_launch("lbt_gemm_i8(pair)");
}

// out[i] = fp32(acc64[i]) * 2^e (+ add_scale * add[i])   — wgrad finalize: scale + weight-decay term
// (dynamic_fixed_point.py:302 `+ 2 * weight_decay * W`: a separate fp32 multiply then add).
__global__ void acc64_finalize_kernel(const long long* acc, size_t n, const int32_t* ibA, const int32_t* ibB, int exp_const,
                                      const float* add, float add_scale, float* out) {
  int e = exp_const;
  if (ibA) e += *ibA;
  if (ibB) e += *ibB;
  const float scale = exp2i(e);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float v = __ll2float_rn(acc[i]) * scale;
    if (add) v = __fadd_rn(v, __fmul_rn(add_scale, add[i]));
    out[i] = v;
  }
}

// ---- host side -------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}

// 2-D K-major operand [rows, K] of bytes, row pitch `ld`; box = 128 bytes of K x `box_rows` rows.
int make_operand_map(CUtensorMap* map, const void* base, size_t rows, size_t K, size_t ld, uint32_t box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return LBT_ECUDA;
  cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, box_rows};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstride, box, estride,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled");
    return LBT_ECUDA;
  }
  return LBT_OK;
}

template <int BN, bool DUAL = false>
int launch(const CUtensorMap& ta, const CUtensorMap& ta2, const CUtensorMap& tb, const GemmParams& p, unsigned grid, cudaStream_t st) {
  static bool attr_done[16] = {};
  const int dev = device_info().device;
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(gemm_i8_kernel<BN, DUAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<BN, DUAL>::kSmemBytes);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(gemm_i8_kernel)");
      return LBT_ECUDA;
    }
    attr_done[dev] = true;
  }
  launch_pdl(gemm_i8_kernel<BN, DUAL>, grid, kThreads, Cfg<BN, DUAL>::kSmemBytes, st, ta, ta2, tb, p);
  return check_launch(DUAL ? "lbt_gemm_i8_dual" : "lbt_gemm_i8");
}

}  // namespace
}  // namespace lbt

using namespace lbt;

extern "C" int lbt_gemm_i8(const void* A, int a_kind, size_t lda, const void* B, int b_kind, size_t ldb, size_t M, size_t N,
                           size_t K, int epilogue, const int32_t* ibA, const int32_t* ibB, int exp_const, const float* bias,
                           float* out_f32, int64_t* acc64, size_t ldc, int alpha, int k_splits, const lbt_qsite* q_out,
                           int8_t* k_out, int64_t* sums, size_t rows_per_image, const float* addend, void* stream) {
  if (!A || !B) return LBT_EINVAL;
  if (q_out) {
    if (epilogue != LBT_EPI_F32 || !k_out || !sums || !q_out->ib || rows_per_image == 0) return LBT_EINVAL;
    if (q_out->bits < 2 || q_out->bits > 8 || (N & 3) || rows_per_image > 0xffffffffull) return LBT_EUNSUPPORTED;
  }
  if ((a_kind != LBT_MANT_S8 && a_kind != LBT_MANT_U8) || (b_kind != LBT_MANT_S8 && b_kind != LBT_MANT_U8)) return LBT_EINVAL;
  if (epilogue == LBT_EPI_F32 ? (!out_f32 && !q_out) : (epilogue == LBT_EPI_ACC64 ? !acc64 : true)) return LBT_EINVAL;
  if (M == 0 || N == 0) return LBT_OK;
  if (K == 0) return LBT_EINVAL;
  if (!q_out && ldc < N) return LBT_EINVAL;
  if (lda < K || ldb < K || (lda & 15) || (ldb & 15)) return LBT_EUNSUPPORTED;  // TMA: 16-byte row pitch
  if ((reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(B) & 15)) return LBT_EUNSUPPORTED;
  if (M >= (1ull << 31) || N >= (1ull << 31) || K >= (1ull << 31)) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  const DeviceInfo& di = device_info();

  int bn = 256;
  for (int c : {16, 32, 64, 128, 256})
    if ((size_t)c >= N) {
      bn = c;
      break;
    }

  GemmParams p{};
  p.M = (uint32_t)M;
  p.N = (uint32_t)N;
  p.K = (uint32_t)K;
  p.m_tiles = (uint32_t)((M + kBlockM - 1) / kBlockM);
  p.n_tiles = (uint32_t)((N + bn - 1) / bn);
  p.k_blocks = (uint32_t)((K + kBlockK - 1) / kBlockK);
  uint32_t splits = k_splits < 1 ? 1u : (uint32_t)k_splits;
  if (epilogue == LBT_EPI_F32) splits = 1;
  if (splits > p.k_blocks) splits = p.k_blocks;
  p.k_blocks_per_split = (p.k_blocks + splits - 1) / splits;
  // s32 accumulator: one CTA may sum at most max_products(a_kind, b_kind) products exactly (32768 for u8 x u8)
  const uint32_t max_kb = max_products(a_kind, b_kind) / kBlockK;
  if (p.k_blocks_per_split > max_kb) {
    if (epilogue == LBT_EPI_F32) return LBT_EUNSUPPORTED;  // caller must use the split-K epilogue
    p.k_blocks_per_split = max_kb;
  }
  p.k_splits = (p.k_blocks + p.k_blocks_per_split - 1) / p.k_blocks_per_split;
  p.epilogue = epilogue;
  p.ibA = ibA;
  p.ibB = ibB;
  p.exp_const = exp_const;
  p.bias = bias;
  p.addend = (epilogue == LBT_EPI_F32 && !q_out) ? addend : nullptr;
  p.out = out_f32;
  p.ldc = ldc;
  p.acc64 = reinterpret_cast<long long*>(acc64);
  p.alpha = alpha;
  p.bnq.q = site_from_abi(q_out);
  p.bnq.k = k_out;
  p.bnq.sums = reinterpret_cast<long long*>(sums);
  p.bnq.rows_per_image = (uint32_t)rows_per_image;
  // instruction descriptor: c_format s32 (2) @4, a_format @7, b_format @10 (0 = u8, 1 = s8), K-major A and B,
  // N>>3 @17, M>>4 @24
  p.idesc = (2u << 4) | ((a_kind == LBT_MANT_S8 ? 1u : 0u) << 7) | ((b_kind == LBT_MANT_S8 ? 1u : 0u) << 10) |
            ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);

  CUtensorMap ta, tb;
  int rc = make_operand_map(&ta, A, M, K, lda, kBlockM);
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // large fp32-epilogue GEMMs: CTA pairs on 256x256 tiles (two thirds of the L2 -> shared-memory traffic per MAC)
  if (g_gemm_pair.load(std::memory_order_relaxed) && epilogue == LBT_EPI_F32 && !q_out && bn == 256 && M >= 256 &&
      (uint64_t)((p.m_tiles + 1) / 2) * p.n_tiles >= (uint64_t)(di.sm_count / 2)) {
    rc = make_operand_map(&tb, B, N, K, ldb, (uint32_t)(k2BN / 2));
    if (rc) return rc;
    p.idesc = (2u << 4) | ((a_kind == LBT_MANT_S8 ? 1u : 0u) << 7) | ((b_kind == LBT_MANT_S8 ? 1u : 0u) << 10) |
              ((uint32_t)(k2BN >> 3) << 17) | ((uint32_t)((2 * kBlockM) >> 4) << 24);
    const uint64_t pair_items = (uint64_t)((p.m_tiles + 1) / 2) * p.n_tiles;
    const uint64_t max_clusters = (uint64_t)(di.sm_count / 2);
    return launch_pair(ta, tb, p, (unsigned)(pair_items < max_clusters ? pair_items : max_clusters), st);
  }
  rc = make_operand_map(&tb, B, N, K, ldb, (uint32_t)bn);
  if (rc) return rc;

  const uint64_t items = (uint64_t)p.m_tiles * p.n_tiles * p.k_splits;
  const unsigned grid = (unsigned)(items < (uint64_t)di.sm_count ? items : (uint64_t)di.sm_count);
  switch (bn) {
    case 16: return launch<16>(ta, ta, tb, p, grid, st);
    case 32: return launch<32>(ta, ta, tb, p, grid, st);
    case 64: return launch<64>(ta, ta, tb, p, grid, st);
    case 128: return launch<128>(ta, ta, tb, p, grid, st);
    default: return launch<256>(ta, ta, tb, p, grid, st);
  }
}

// out[M, N] = fp32((256 * A_hi + A_lo)[M, K] . B[N, K]^T) * 2^(exp_const + ibA + ibB) (+ addend): the A operand is a 9..16-bit
// mantissa tensor given as its two byte planes k = 256 * hi + lo (hi s8, lo u8) with the same row pitch — the 16-bit
// gradients of BASELINE config 5 (dfxp:300, 305 with a 16-bit `gradq`).  One pass over B, two accumulators in tensor memory,
// combined exactly in the epilogue (gemm_i8_kernel<BN, true>).
extern "C" int lbt_gemm_i8_dual(const int8_t* A_hi, const uint8_t* A_lo, size_t lda, const void* B, int b_kind, size_t ldb, size_t M,
                                size_t N, size_t K, const int32_t* ibA, const int32_t* ibB, int exp_const, float* out_f32, size_t ldc,
                                const float* addend, void* stream) {
  if (!A_hi || !A_lo || !B || !out_f32) return LBT_EINVAL;
  if (b_kind != LBT_MANT_S8 && b_kind != LBT_MANT_U8) return LBT_EINVAL;
  if (M == 0 || N == 0) return LBT_OK;
  if (K == 0 || ldc < N) return LBT_EINVAL;
  if (lda < K || ldb < K || (lda & 15) || (ldb & 15)) return LBT_EUNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(A_hi) | reinterpret_cast<uintptr_t>(A_lo) | reinterpret_cast<uintptr_t>(B)) & 15) return LBT_EUNSUPPORTED;
  if (M >= (1ull << 31) || N >= (1ull << 31) || K >= (1ull << 31)) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  const DeviceInfo& di = device_info();
  int bn = 128;
  for (int c : {16, 32, 64, 128})
    if ((size_t)c >= N) {
      bn = c;
      break;
    }
  GemmParams p{};
  p.M = (uint32_t)M;
  p.N = (uint32_t)N;
  p.K = (uint32_t)K;
  p.m_tiles = (uint32_t)((M + kBlockM - 1) / kBlockM);
  p.n_tiles = (uint32_t)((N + bn - 1) / bn);
  p.k_blocks = (uint32_t)((K + kBlockK - 1) / kBlockK);
  p.k_blocks_per_split = p.k_blocks;
  p.k_splits = 1;
  // each s32 accumulator sums at most 65536 products, 32768 for the low plane (u8) x a u8 B
  if (p.k_blocks > max_products(LBT_MANT_U8, b_kind) / kBlockK) return LBT_EUNSUPPORTED;
  p.epilogue = LBT_EPI_F32;
  p.ibA = ibA;
  p.ibB = ibB;
  p.exp_const = exp_const;
  p.addend = addend;
  p.out = out_f32;
  p.ldc = ldc;
  const uint32_t common = (2u << 4) | ((b_kind == LBT_MANT_S8 ? 1u : 0u) << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);
  p.idesc = common | (1u << 7);    // hi: s8
  p.idesc2 = common;               // lo: u8
  CUtensorMap ta, ta2, tb;
  int rc = make_operand_map(&ta, A_hi, M, K, lda, kBlockM);
  if (rc) return rc;
  if ((rc = make_operand_map(&ta2, A_lo, M, K, lda, kBlockM))) return rc;
  if ((rc = make_operand_map(&tb, B, N, K, ldb, (uint32_t)bn))) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const uint64_t items = (uint64_t)p.m_tiles * p.n_tiles;
  const unsigned grid = (unsigned)(items < (uint64_t)di.sm_count ? items : (uint64_t)di.sm_count);
  switch (bn) {
    case 16: return launch<16, true>(ta, ta2, tb, p, grid, st);
    case 32: return launch<32, true>(ta, ta2, tb, p, grid, st);
    case 64: return launch<64, true>(ta, ta2, tb, p, grid, st);
    default: return launch<128, true>(ta, ta2, tb, p, grid, st);
  }
}

extern "C" int lbt_acc64_finalize(const int64_t* acc64, size_t n, const int32_t* ibA, const int32_t* ibB, int exp_const,
                                  const float* add, float add_scale, float* out, void* stream) {
  if (!acc64 || !out) return LBT_EINVAL;
  if (n == 0) return LBT_OK;
  LBT_REQUIRE_ARCH();
  const size_t blocks = (n + 255) / 256;
  const unsigned grid = (unsigned)(blocks < 4096 ? blocks : 4096);
  acc64_finalize_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const long long*>(acc64), n, ibA, ibB, exp_const, add, add_scale, out);
  return check_launch("lbt_acc64_finalize");
}

// Bench / test knob (not in lbt.h): 0 = never use the CTA-pair kernel, 1 (default) = use it for large fp32-epilogue GEMMs.
extern "C" int lbt_gemm_set_pair(int on) {
  g_gemm_pair.store(on ? 1 : 0, std::memory_order_relaxed);
  return LBT_OK;
}

// Test hook: 1 if any GEMM CTA hit the bounded-wait watchdog since the last call (synchronises).
extern "C" int lbt_gemm_debug_error(void) {
  int v = 0, zero = 0;
  if (cudaMemcpyFromSymbol(&v, g_gemm_error, sizeof(int)) != cudaSuccess) return -1;
  cudaMemcpyToSymbol(g_gemm_error, &zero, sizeof(int));
  return v;
}
