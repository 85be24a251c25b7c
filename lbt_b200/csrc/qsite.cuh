// Quantiser call sites shared by the fused kernels (bn.cu, conv_i8.cu, gemm_i8.cu): the arithmetic of
// stochastic_identity + overflow_rate (/root/reference/dynamic_fixed_point.py:32-38, 48-67) on one value, and
// the fused "quantise + per-channel statistics" epilogue of the tensor-core kernels (Normalization_q's input
// quantiser applied to the accumulators, dfxp:584-588).
#pragma once

#include "common.cuh"

namespace lbt {

struct QSite {
  int bits;
  const int32_t* ib;
  const float* noise;  // explicit noise [n_inner] or NULL -> Philox
  uint64_t seed, offset;
  const uint64_t* dev_step;
  unsigned long long* counters;
  int minmax;  // 1: min/max statistics (target_overflow_rate == 0)
};

struct QC {
  float m, inv_m, L, hi, half;
};

__device__ __forceinline__ QC make_qc(int bits, int ib) {
  QC c;
  int f = bits - ib - 1;
  f = max(-126, min(126, f));
  c.m = exp2i(f);
  c.inv_m = exp2i(-f);
  c.L = exp2i(bits - 1);
  c.hi = c.L - 1.0f;
  c.half = c.L * 0.5f;
  return c;
}

// stochastic_identity (dfxp:34-37) + overflow counters (dfxp:60-66); returns the integral mantissa as float
__device__ __forceinline__ float squant(float x, float u, const QC& c, uint32_t& n1, uint32_t& n2) {
  const float y = __fmul_rn(x, c.m);
  n1 += (uint32_t)(y >= c.L) + (uint32_t)(y < -c.L);
  n2 += (uint32_t)(y >= c.half) + (uint32_t)(y < -c.half);
  return floorf(fminf(fmaxf(__fadd_rn(y, u), -c.L), c.hi));
}

// min/max variant of the statistics (LBT_STATS_MINMAX): two FMNMX instead of four compares + adds
__device__ __forceinline__ float squant_mm(float x, float u, const QC& c, float& mx, float& mn) {
  const float y = __fmul_rn(x, c.m);
  mx = fmaxf(mx, y);
  mn = fminf(mn, y);
  return floorf(fminf(fmaxf(__fadd_rn(y, u), -c.L), c.hi));
}
__device__ __forceinline__ void mm_to_counts(const QC& c, float mx, float mn, uint32_t& n1, uint32_t& n2) {
  n1 = (mx >= c.L || mn < -c.L) ? 1u : 0u;
  n2 = (mx >= c.half || mn < -c.half) ? 1u : 0u;
}

// Conversion-free floor (the fused kernels are issue-bound and FRND / F2I / I2F run at quarter rate): for |t| < 2^22,
// tm = RD(t + 1.5 * 2^23) is ONE full-rate FADD.RM; floor(t) as an integer is bits(tm) - 0x4B400000, as a float tm - 1.5 * 2^23,
// and the low byte(s) of bits(tm) are the two's-complement mantissa byte(s).
constexpr float kFloorMagicF = 12582912.0f;

// a / b, correctly rounded (== __fdiv_rn), for MANY numerators over ONE denominator: r = frcp_rn(b) is computed once
// (per channel) and each quotient costs five FMA-class instructions instead of the ~12 + special-case branch of the
// generic IEEE division.  Markstein's scheme: q0 = RN(a*r); two residual corrections q += RN(a - b*q) * r with exact
// FMA residuals.  Valid while a/b and the residuals stay in the normal range (|a/b| in [2^-100, 2^100] or a == 0), which
// the batch-norm operands do (b = sqrt(var + eps) in [3e-3, 1e4]); checked against __fdiv_rn over 2^32 random and
// structured pairs by tests/test_quantize_gpu.py::test_fast_division_is_correctly_rounded (lbt_test_fdiv).
__device__ __forceinline__ float fdiv_by(float a, float b, float r) {
  const float q0 = __fmul_rn(a, r);
  float q = __fmaf_rn(__fmaf_rn(-b, q0, a), r, q0);
  q = __fmaf_rn(__fmaf_rn(-b, q, a), r, q);
  return a == 0.0f ? q0 : q;   // keeps the sign of a zero numerator
}

__device__ __forceinline__ float4 site_noise(const QSite& s, uint32_t v, uint64_t off) {
  if (s.noise) return __ldg(reinterpret_cast<const float4*>(s.noise) + v);
  return philox_noise4(v, s.seed, off);
}
__device__ __forceinline__ uint64_t site_offset(const QSite& s) {
  uint64_t off = s.offset;
  if (s.dev_step) off += (*s.dev_step) << 32;
  return off;
}


// ------------------------------------------------------------------------------------------------
// Fused "quantise + batch statistics" epilogue of the tensor-core kernels: BN forward pass 1
// (k = Q_norm(conv output), per-channel sum k and sum k^2; dfxp:584-588) applied to the accumulators while
// they are still in registers, so the fp32 convolution output never touches HBM.
// An epilogue thread owns one output row (pixel) and 16 consecutive channels per chunk.
// ------------------------------------------------------------------------------------------------
constexpr int kBnqFlushTiles = 2048;  // 32 rows * 2^14 per tile and channel: int32 partials stay exact

struct BnqParams {
  QSite q;                  // bits == 0: disabled
  int8_t* k;                // [M, N] mantissas, row pitch N
  long long* sums;          // [2*N]: sum k, sum k^2 per channel (caller-zeroed)
  uint32_t rows_per_image;  // OH*OW: noise index = (row % rows_per_image) * N + col  (noise is shared over the batch)
};

struct BnqState {
  QC qc;
  uint64_t off;
  uint32_t n1, n2;
  float mx, mn;
  uint32_t tiles;
  __device__ __forceinline__ void init(const BnqParams& b) {
    qc = make_qc(b.q.bits, __ldg(b.q.ib));
    off = site_offset(b.q);
    n1 = n2 = 0;
    mx = -INFINITY;
    mn = INFINITY;
    tiles = 0;
  }
};

// Per-channel sum k and sum k^2 of a warp's 32 rows x 16 channels from the PACKED mantissas (w[i] = channels 4i .. 4i+3 of
// this lane's row, two's-complement bytes), ~58 instructions instead of the ~140 of two 16-value butterflies:
//   1. a 4 x 4 byte transpose inside each lane quad (2 x {SHFL, PRMT} per word): the lane then holds ONE channel of FOUR rows,
//      channel 4i + 2 * (lane & 1) + ((lane >> 1) & 1);
//   2. IDP4A with 0x01010101 / with itself: the sum and the sum of squares of those four rows;
//   3. a reduce-scatter butterfly over the 8 quads (lane bits 4, 3, 2) of the 8 partials (7 SHFL).
// Afterwards every lane holds ONE total: kind = lane bit 4 (0: sum k, 1: sum k^2) of channel
// 4 * (2 * bit3 + bit2) + 2 * bit0 + bit1.  Returns the total; `chan` / `kind` tell the caller where it belongs.
__device__ __forceinline__ int warp_colstats_packed(const uint32_t (&w)[4], int lane, int& chan, int& kind) {
  const uint32_t sel1 = (lane & 1) ? 0x3726u : 0x5140u;   // even lane: [a0 b0 a1 b1]; odd lane: [a2 b2 a3 b3] (a = even lane's row)
  const uint32_t sel2 = (lane & 2) ? 0x3276u : 0x5410u;   // bit1 = 0: first channel of the pair x 4 rows; bit1 = 1: second
  int sv[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t r1 = __shfl_xor_sync(0xffffffffu, w[i], 1);
    const uint32_t t1 = __byte_perm(w[i], r1, sel1);
    const uint32_t r2 = __shfl_xor_sync(0xffffffffu, t1, 2);
    const uint32_t t2 = __byte_perm(t1, r2, sel2);
    sv[i] = __dp4a((int)t2, 0x01010101, 0);
    sv[4 + i] = __dp4a((int)t2, (int)t2, 0);
  }
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
  int a[4], b[2];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int send = b4 ? sv[j] : sv[j + 4];
    a[j] = (b4 ? sv[j + 4] : sv[j]) + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int send = b3 ? a[j] : a[j + 2];
    b[j] = (b3 ? a[j + 2] : a[j]) + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  const int send = b2 ? b[0] : b[1];
  const int tot = (b2 ? b[1] : b[0]) + __shfl_xor_sync(0xffffffffu, send, 4);
  kind = b4 ? 1 : 0;
  chan = 4 * (2 * (b3 ? 1 : 0) + (b2 ? 1 : 0)) + 2 * (lane & 1) + ((lane >> 1) & 1);
  return tot;
}

// The noise of a row's 16-channel chunk lives in the L2-resident noise arena; without help every chunk of the epilogue
// starts with a ~700-cycle L2 round trip that 8 - 16 epilogue warps per SM cannot hide (ncu: long_scoreboard is the top
// stall of the fused convolutions).  Called BEFORE the accumulator wait: pulls the line into L1 at no register cost.
__device__ __forceinline__ void bnq_prefetch(const BnqParams& b, uint32_t pix, uint32_t N, uint32_t col, bool ok) {
  if (b.q.noise && ok) asm volatile("prefetch.global.L1 [%0];" ::"l"(b.q.noise + (uint64_t)pix * N + col));
}

// One 16-channel chunk of one row, straight from the s32 accumulators `v`: x = RN(acc) * scale (+ bias) is the fp32 value the
// unfused path would have written (scale = 2^e), k = Q(x) the mantissa that is stored, sum k / sum k^2 the batch statistics.
// row_ok / ncol mask the tile tails (masked elements quantise the value 0: no counts, no sums).
// s_stat: this WARP's private [2][bn] int32 partial sums (bn = tile width); tcol = first column of the chunk inside the tile.
// pix = row % rows_per_image (the pixel inside its image; computed once per tile by the caller).
// ~13 instructions per element (ncu source view of the first version: ~24, a third of them tail masks and byte packing):
//   * FULL (warp-uniform: every row of the warp valid, 16 columns): no masks at all; else ONE select per element — a masked
//     element becomes the value 0, which quantises to mantissa 0 (u < 1), leaves min / max and the counts alone and adds nothing;
//   * without a bias the two power-of-two scalings fold into one multiply (exact while the exponents stay far from the
//     subnormal range — checked on the host side of the branch);
//   * the mantissa byte is the low byte of the magic-biased floor, packed with three PRMT per four elements;
//   * statistics from the packed bytes (warp_colstats_packed).
__device__ __forceinline__ uint32_t pack4_low_bytes(float t0, float t1, float t2, float t3) {
  const uint32_t p01 = __byte_perm(__float_as_uint(t0), __float_as_uint(t1), 0x0040);
  const uint32_t p23 = __byte_perm(__float_as_uint(t2), __float_as_uint(t3), 0x0040);
  return __byte_perm(p01, p23, 0x5410);
}

// The chunk's 16 noise values (four float4).  Split from bnq_chunk so that a caller can issue these loads BEFORE it waits for
// the accumulator (tcgen05.wait::ld): the L1 / L2 round trip then overlaps the wait instead of stalling the first addition
// (ncu source view of conv_halo_kernel: the four `y + u` FADDs held 28 % of all stall samples, long scoreboard).
__device__ __forceinline__ void bnq_load_noise(const BnqParams& b, const BnqState& st, uint32_t pix, bool row_ok, uint32_t col, uint32_t ncol,
                                               uint32_t N, float4 (&u)[4]) {
  const uint64_t inner = (uint64_t)pix * N + col;   // multiple of 4 (N % 4 == 0, col % 16 == 0)
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    if (b.q.noise) u[g] = (row_ok && 4u * g < ncol) ? __ldg(reinterpret_cast<const float4*>(b.q.noise + inner) + g) : make_float4(0.f, 0.f, 0.f, 0.f);
    else u[g] = philox_noise4((inner >> 2) + g, b.q.seed, st.off);
  }
}

// PRE: the noise comes in `u4` (bnq_load_noise, issued by the caller ahead of its accumulator wait); else it is fetched here,
// group by group between the arithmetic (what the register-bound gather kernels want; `pix` is only used then).
// FOLD: compile-time copy of the `fold` test below.  As a run-time flag inside the unrolled element loop it cost a BSSY / BRA /
// BSYNC triple per element (ncu source view of conv_halo_kernel: 3 of the ~18 per-element instructions) and, worse, a
// reconvergence barrier between consecutive elements that kept the compiler from interleaving their dependent chains.
// FOLD = 2: the test stays a run-time flag — the 16-epilogue-warp gather kernel of the 7x7/2 stem is paced by its cp.async
// loader warps and measurably loses (476 -> 506 us) when the epilogue warps issue in denser bursts.
template <bool FULL, bool MM, bool PRE, int FOLD>
__device__ __forceinline__ void bnq_chunk_impl(const BnqParams& b, BnqState& st, const uint32_t (&v)[16], const float4 (&u4)[4], float scale,
                                               const float* bias, uint32_t row, uint32_t pix, bool row_ok, uint32_t col, uint32_t ncol,
                                               uint32_t N, int* s_stat, uint32_t bn, uint32_t tcol, int lane) {
  const uint64_t inner = PRE ? 0ull : (uint64_t)pix * N + col;   // multiple of 4 (N % 4 == 0, col % 16 == 0)
  const QC& c = st.qc;
  // one multiply instead of two (decided by the caller, see bnq_chunk_sel)
  const bool fold = FOLD == 2 ? (bias == nullptr && fabsf(__log2f(scale)) < 60.0f && fabsf(__log2f(c.m)) < 60.0f) : (FOLD == 1);
  const float sm = scale * c.m;
  float tm[16];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float4 u;
    if (PRE) u = u4[g];
    else if (b.q.noise) u = (FULL || (row_ok && 4u * g < ncol)) ? __ldg(reinterpret_cast<const float4*>(b.q.noise + inner) + g) : make_float4(0.f, 0.f, 0.f, 0.f);
    else u = philox_noise4((inner >> 2) + g, b.q.seed, st.off);
    const float un[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int j = 4 * g + t;
      const float a = __int2float_rn((int)v[j]);
      float y;
      if (fold) {
        y = __fmul_rn(a, sm);
      } else {
        float x = __fmul_rn(a, scale);
        if (bias && (FULL || (uint32_t)j < ncol)) x = __fadd_rn(x, __ldg(bias + j));
        y = __fmul_rn(x, c.m);
      }
      if (!FULL) y = (row_ok && (uint32_t)j < ncol) ? y : 0.0f;
      if (MM) {
        st.mx = fmaxf(st.mx, y);
        st.mn = fminf(st.mn, y);
      } else {
        st.n1 += (uint32_t)(y >= c.L) + (uint32_t)(y < -c.L);
        st.n2 += (uint32_t)(y >= c.half) + (uint32_t)(y < -c.half);
      }
      tm[j] = __fadd_rd(fminf(fmaxf(__fadd_rn(y, un[t]), -c.L), c.hi), kFloorMagicF);   // bits = 0x4B400000 + k
    }
  }
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) w[i] = pack4_low_bytes(tm[4 * i], tm[4 * i + 1], tm[4 * i + 2], tm[4 * i + 3]);
  if (FULL || row_ok) {
    int8_t* o = b.k + (size_t)row * N + col;
    if ((FULL || ncol == 16) && ((reinterpret_cast<uintptr_t>(o) & 15u) == 0)) {
      *reinterpret_cast<uint4*>(o) = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if ((uint32_t)j < ncol) o[j] = (int8_t)(w[j >> 2] >> (8 * (j & 3)));
    }
  }
  int chan, kind;
  const int tot = warp_colstats_packed(w, lane, chan, kind);   // masked elements are 0: they add nothing
  s_stat[(kind ? bn : 0u) + tcol + (uint32_t)chan] += tot;
}

// `bias`: this chunk's 16 bias values (NULL: none); `u4`: the chunk's noise from bnq_load_noise.
template <bool PRE, bool UNSWITCH = true>
__device__ __forceinline__ void bnq_chunk_sel(const BnqParams& b, BnqState& st, const uint32_t (&v)[16], const float4 (&u4)[4], float scale,
                                              const float* bias, uint32_t row, uint32_t pix, bool row_ok, uint32_t col, uint32_t ncol, uint32_t N,
                                              int* s_stat, uint32_t bn, uint32_t tcol, int lane) {
  const bool full = ncol == 16 && __all_sync(0xffffffffu, row_ok);
  // one multiply when no bias sits between the two scalings and neither product can leave the normal range (warp-uniform)
  const bool fold = bias == nullptr && fabsf(__log2f(scale)) < 60.0f && fabsf(__log2f(st.qc.m)) < 60.0f;
#define LBT_BNQ_CHUNK(F, M, FO) bnq_chunk_impl<F, M, PRE, FO>(b, st, v, u4, scale, bias, row, pix, row_ok, col, ncol, N, s_stat, bn, tcol, lane)
  if constexpr (!UNSWITCH) {
    if (b.q.minmax) { if (full) LBT_BNQ_CHUNK(true, true, 2); else LBT_BNQ_CHUNK(false, true, 2); }
    else { if (full) LBT_BNQ_CHUNK(true, false, 2); else LBT_BNQ_CHUNK(false, false, 2); }
  } else if (b.q.minmax) {
    if (full) { if (fold) LBT_BNQ_CHUNK(true, true, 1); else LBT_BNQ_CHUNK(true, true, 0); }
    else { if (fold) LBT_BNQ_CHUNK(false, true, 1); else LBT_BNQ_CHUNK(false, true, 0); }
  } else {
    if (full) { if (fold) LBT_BNQ_CHUNK(true, false, 1); else LBT_BNQ_CHUNK(true, false, 0); }
    else { if (fold) LBT_BNQ_CHUNK(false, false, 1); else LBT_BNQ_CHUNK(false, false, 0); }
  }
#undef LBT_BNQ_CHUNK
}
__device__ __forceinline__ void bnq_chunk(const BnqParams& b, BnqState& st, const uint32_t (&v)[16], const float4 (&u4)[4], float scale,
                                          const float* bias, uint32_t row, bool row_ok, uint32_t col, uint32_t ncol, uint32_t N, int* s_stat,
                                          uint32_t bn, uint32_t tcol, int lane) {
  bnq_chunk_sel<true>(b, st, v, u4, scale, bias, row, 0u, row_ok, col, ncol, N, s_stat, bn, tcol, lane);
}
// Noise fetched inside the chunk, right before use.
template <bool UNSWITCH = true>
__device__ __forceinline__ void bnq_chunk(const BnqParams& b, BnqState& st, const uint32_t (&v)[16], float scale, const float* bias,
                                          uint32_t row, uint32_t pix, bool row_ok, uint32_t col, uint32_t ncol, uint32_t N, int* s_stat,
                                          uint32_t bn, uint32_t tcol, int lane) {
  float4 u4[4];   // not read
  bnq_chunk_sel<false, UNSWITCH>(b, st, v, u4, scale, bias, row, pix, row_ok, col, ncol, N, s_stat, bn, tcol, lane);
}

// Add the warp's partial sums for the tile columns [col0, col0 + bn) to the global int64 sums and clear them.
__device__ __forceinline__ void bnq_flush(const BnqParams& b, int* s_stat, uint32_t col0, uint32_t bn, uint32_t N, int lane) {
  __syncwarp();
  for (uint32_t i = lane; i < bn; i += 32) {
    const int v0 = s_stat[i], v1 = s_stat[bn + i];
    if (col0 + i < N) {
      if (v0) atomicAdd(reinterpret_cast<unsigned long long*>(b.sums) + col0 + i, (unsigned long long)(long long)v0);
      if (v1) atomicAdd(reinterpret_cast<unsigned long long*>(b.sums) + N + col0 + i, (unsigned long long)(long long)v1);
    }
    s_stat[i] = 0;
    s_stat[bn + i] = 0;
  }
  __syncwarp();
}

// Final flush of a CTA: the epilogue warps first combine their partials in shared memory (s_tot: [2][bn] 64-bit, zeroed
// at kernel start) and only then touch the global sums — one int64 atomic per channel per CTA instead of one per warp
// (the per-warp version put 8 x 296 CTAs deep contention on 2 x Cout addresses: ~10 us at the tail of every launch).
// Must be reached by ALL `nthreads` epilogue threads (named barrier `bar_id`); tid = index within the epilogue group.
__device__ __forceinline__ void bnq_flush_cta(const BnqParams& b, int* s_stat, unsigned long long* s_tot, uint32_t col0, uint32_t bn,
                                              uint32_t N, int lane, uint32_t tid, uint32_t nthreads, int bar_id) {
  __syncwarp();
  for (uint32_t i = lane; i < 2 * bn; i += 32) {
    const int v = s_stat[i];
    if (v) atomicAdd(s_tot + i, (unsigned long long)(long long)v);
    s_stat[i] = 0;
  }
  asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(nthreads) : "memory");
  for (uint32_t i = tid; i < 2 * bn; i += nthreads) {
    const uint32_t c = i < bn ? i : i - bn;
    const unsigned long long v = s_tot[i];
    if (v && col0 + c < N) atomicAdd(reinterpret_cast<unsigned long long*>(b.sums) + (i < bn ? 0 : N) + col0 + c, v);
  }
}

// End of the kernel: publish the overflow statistics; the `ticket` warp of CTA 0 adds the element count.
__device__ __forceinline__ void bnq_finish(const BnqParams& b, BnqState& st, unsigned long long numel, bool ticket, int lane) {
  if (b.q.minmax) mm_to_counts(st.qc, st.mx, st.mn, st.n1, st.n2);
  const uint32_t n1 = warp_sum(st.n1), n2 = warp_sum(st.n2);
  if (lane == 0 && b.q.counters) {
    if (n1) atomicAdd(b.q.counters + LBT_CNT_OVER, (unsigned long long)n1);
    if (n2) atomicAdd(b.q.counters + LBT_CNT_OVER_HALF, (unsigned long long)n2);
    if (ticket && blockIdx.x == 0) atomicAdd(b.q.counters + LBT_CNT_NUMEL, numel);   // fire-and-forget, no ticket
  }
}

// Host: lbt_qsite (C ABI) -> QSite; a NULL descriptor gives a disabled site (bits == 0).
inline QSite site_from_abi(const lbt_qsite* q) {
  QSite s{};
  if (!q) return s;
  s.bits = q->bits;
  s.ib = q->ib;
  s.noise = q->noise;
  s.seed = q->seed;
  s.offset = q->offset;
  s.dev_step = q->dev_step;
  s.counters = reinterpret_cast<unsigned long long*>(q->counters);
  s.minmax = q->stats_minmax;
  return s;
}

}  // namespace lbt
