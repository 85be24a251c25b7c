// Fused quantised batch-norm for B200 (sm_100a): Normalization_q + Rescale_q of
// /root/reference/dynamic_fixed_point.py:539-743 in two HBM-bound passes forward and two backward,
// instead of ~4 quantiser calls + ~25 TF elementwise/reduce kernels over activation-sized fp32 tensors.
//
//   fwd 1  lbt_bn_fwd_quant_stats : x (fp32) -> k1 = Q_norm(x) (s8) + exact per-channel sum(k1), sum(k1^2)
//   fwd 2  lbt_bn_fwd_apply       : k1 -> y1 = (xq - mean)/sqrt(var+eps) -> k2 = Q_rescale(y1) (s8)
//                                   -> out = relu?(xq2*gq + bq (+ add))   (fp32)
//   bwd 1  lbt_bn_bwd_quant_stats : g -> relu mask -> kg2 = Q(g) -> sums for dgamma/dbeta -> dx2 = gq2*gq
//                                   -> kg1 = Q(dx2) (s8) + sums for the batch-norm VJP (+ d_add)
//   bwd 2  lbt_bn_bwd_apply       : kg1, k1 -> dx = (gq1 - mean(gq1) - xhat*mean(gq1*xhat)) / sqrt(var+eps)
//
// Batch statistics are taken over the QUANTISED input (dfxp:588) and are computed exactly: integer
// sums of mantissas (int64), finished in fp64, rounded once to fp32.  Tensors are NHWC: [n_outer = N,
// n_inner = H*W*C]; the rounding noise is indexed by the inner position and shared over N (dfxp:36).
// A thread owns 4 consecutive channels of one inner position and walks down N, so its Philox draw and
// its per-channel partial sums live in registers.
#include <type_traits>

#include "qsite.cuh"

namespace lbt {
namespace {

// resident CTAs per SM the register allocation of the two heaviest kernels is bounded for (A/B builds: -DLBT_BN_BWD1_CTAS=3 ...)
#ifndef LBT_BN_BWD1_CTAS
#define LBT_BN_BWD1_CTAS 2
#endif
#ifndef LBT_BN_FWD2_CTAS
#define LBT_BN_FWD2_CTAS 3
#endif
constexpr int kThreads = 256;
constexpr int kRows = 4;  // rows (batch entries) in flight per thread

// bench aid (lbt_bn_set_debug): phase timestamps of CTA 0 / thread 0 (globaltimer ns)
__device__ unsigned long long* g_bn_dbg = nullptr;
__device__ __forceinline__ void bn_stamp(int slot) {
  if (g_bn_dbg && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    g_bn_dbg[slot] = t;
  }
}

struct Tiling {
  size_t n_outer, n_inner;
  int C;
  uint32_t n_vec, chunks, rows_per_group;
  uint64_t total_tiles;
  int fixed_channels;  // 1: a thread sees the same 4 channels in every tile (256 % (C/4) == 0)
};

__device__ __forceinline__ void publish_counters(unsigned long long* counters, uint32_t n1, uint32_t n2, size_t numel,
                                                 uint32_t* s_red) {
  // block reduce two u32 counters and add them to the site's statistics block; CTA 0 adds the element count.
  // Must be called by all threads.
  n1 = warp_sum(n1);
  n2 = warp_sum(n2);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) {
    s_red[w] = n1;
    s_red[8 + w] = n2;
  }
  __syncthreads();
  if (threadIdx.x == 0 && counters) {
    uint32_t b1 = 0, b2 = 0;
    for (int i = 0; i < kThreads / 32; ++i) {
      b1 += s_red[i];
      b2 += s_red[8 + i];
    }
    if (b1) atomicAdd(counters + LBT_CNT_OVER, (unsigned long long)b1);
    if (b2) atomicAdd(counters + LBT_CNT_OVER_HALF, (unsigned long long)b2);
    // the element count does not need a "last CTA": CTA 0 adds it (fire-and-forget reductions, no ticket round trip)
    if (blockIdx.x == 0) atomicAdd(counters + LBT_CNT_NUMEL, (unsigned long long)numel);
  }
}

// Per-channel partial sums: NS sums for each of the thread's 4 channels.  32-bit per thread (a thread sums at
// most a few 10^4 products of two 8-bit mantissas; the host rejects tensors where that could overflow),
// widened to 64 bits when the partials are combined.
template <int NS, typename T = int>
struct Acc {
  T s[NS][4];
  __device__ __forceinline__ void zero() {
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0;
  }
};

// Add the thread's partials for channels c0..c0+3 straight into the global sums (general path).
template <int NS, typename T>
__device__ __forceinline__ void flush_global(Acc<NS, T>& a, long long* sums, int C, int c0) {
#pragma unroll
  for (int i = 0; i < NS; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (a.s[i][j])
        atomicAdd(reinterpret_cast<unsigned long long*>(sums) + (size_t)i * C + c0 + j, (unsigned long long)(long long)a.s[i][j]);
  a.zero();
}

// Fixed-channel path: every thread kept the same channel group (c0 = 4 * (tid % (C/4))) for the whole
// kernel.  Reduce across the lanes of a warp that share a group, then across warps through shared memory,
// then one global atomic per (sum, channel) per CTA.
template <int NS, typename T>
__device__ __forceinline__ void flush_block(Acc<NS, T>& a32, long long* sums, int C, unsigned long long* s_acc) {
  const int groups = C >> 2;
  for (int i = threadIdx.x; i < NS * C; i += kThreads) s_acc[i] = 0ull;
  __syncthreads();
  long long v[NS][4];
#pragma unroll
  for (int i = 0; i < NS; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) v[i][j] = (long long)a32.s[i][j];
  if (groups < 32) {
    for (int o = 16; o >= groups; o >>= 1) {
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) v[i][j] += __shfl_xor_sync(0xffffffffu, v[i][j], o);
    }
  }
  const int lane = threadIdx.x & 31;
  if (groups >= 32 || lane < groups) {
    const int c0 = 4 * (threadIdx.x % groups);
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (v[i][j]) atomicAdd(s_acc + (size_t)i * C + c0 + j, (unsigned long long)v[i][j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NS * C; i += kThreads)
    if (s_acc[i]) atomicAdd(reinterpret_cast<unsigned long long*>(sums) + i, s_acc[i]);
}

// Pull the NEXT batch of rows towards the SM while the current one is being computed: the loop body then finds its
// operands in L1 instead of paying a DRAM round trip per iteration (the kernels run at ~14-30 resident warps per SM).
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

__device__ __forceinline__ void unpack4(uint32_t w, int (&k)[4]) {
  k[0] = (int)(int8_t)(w & 0xff);
  k[1] = (int)(int8_t)((w >> 8) & 0xff);
  k[2] = (int)(int8_t)((w >> 16) & 0xff);
  k[3] = (int)(int8_t)(w >> 24);
}
__device__ __forceinline__ uint32_t pack4(const float (&k)[4]) {
  const int i0 = __float2int_rn(k[0]), i1 = __float2int_rn(k[1]), i2 = __float2int_rn(k[2]), i3 = __float2int_rn(k[3]);
  return (uint32_t)(i0 & 0xff) | ((uint32_t)(i1 & 0xff) << 8) | ((uint32_t)(i2 & 0xff) << 16) | ((uint32_t)(i3 & 0xff) << 24);
}

// 16-bit gradient mantissas (BASELINE config 5: grad_bits = 16): four s16 values travel as one 8-byte word; a 16-bit
// mantissa handed to the tensor cores is stored as its two byte planes k = 256 * hi + lo (hi s8, lo u8).
__device__ __forceinline__ void unpack4_s16(uint2 w, int (&k)[4]) {
  k[0] = (int)(short)(w.x & 0xffff);
  k[1] = (int)(short)(w.x >> 16);
  k[2] = (int)(short)(w.y & 0xffff);
  k[3] = (int)(short)(w.y >> 16);
}
__device__ __forceinline__ uint2 pack4_s16(const float (&k)[4]) {
  const int i0 = __float2int_rn(k[0]), i1 = __float2int_rn(k[1]), i2 = __float2int_rn(k[2]), i3 = __float2int_rn(k[3]);
  return make_uint2((uint32_t)(i0 & 0xffff) | ((uint32_t)(i1 & 0xffff) << 16), (uint32_t)(i2 & 0xffff) | ((uint32_t)(i3 & 0xffff) << 16));
}
__device__ __forceinline__ void pack4_hilo(const float (&k)[4], uint32_t& hi, uint32_t& lo) {
  hi = lo = 0u;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int v = __float2int_rn(k[j]);
    hi |= (uint32_t)((v >> 8) & 0xff) << (8 * j);     // arithmetic shift: floor(v / 256) in [-128, 127]
    lo |= (uint32_t)(v & 0xff) << (8 * j);
  }
}

// ---- conversion-free arithmetic -------------------------------------------------------------------------------------
// The kernels below are issue-bound, and I2F / F2I / FRND run on the quarter-rate conversion pipe: five of them per element
// cost as much as ~40 FP32 instructions.  All of them are replaced by full-rate operations that give the SAME values:
//   floor(t) for |t| < 2^22 : tm = RD(t + 1.5*2^23) (one FADD.RM); the integer is bits(tm) - 0x4B400000, the float tm - 1.5*2^23,
//                             and the low byte(s) of bits(tm) are the two's-complement mantissa byte(s) to store;
//   int8 -> float           : PRMT builds bits 0x4B0000bb from the biased byte bb = k + 128, minus (2^23 + 128) (exact).
constexpr float kMagicF = 12582912.0f;   // 1.5 * 2^23
constexpr int kMagicI = 0x4B400000;

// stochastic_identity on an ALREADY SCALED value y = x * 2^f (dfxp:34-37) + overflow statistics (dfxp:60-66); returns the
// magic-biased floor tm (see above).  MM: min/max statistics (LBT_STATS_MINMAX) instead of the four compares + adds.
template <bool MM>
__device__ __forceinline__ float sq_scaled(float y, float u, const QC& c, float& mx, float& mn, uint32_t& n1, uint32_t& n2) {
  if (MM) {
    mx = fmaxf(mx, y);
    mn = fminf(mn, y);
  } else {
    n1 += (uint32_t)(y >= c.L) + (uint32_t)(y < -c.L);
    n2 += (uint32_t)(y >= c.half) + (uint32_t)(y < -c.half);
  }
  return __fadd_rd(fminf(fmaxf(__fadd_rn(y, u), -c.L), c.hi), kMagicF);
}
__device__ __forceinline__ int tm_int(float tm) { return __float_as_int(tm) - kMagicI; }
__device__ __forceinline__ float tm_float(float tm) { return __fsub_rn(tm, kMagicF); }
__device__ __forceinline__ uint32_t tm_pack4(const float (&tm)[4]) {   // four mantissas as s8 bytes
  const uint32_t a = __byte_perm(__float_as_uint(tm[0]), __float_as_uint(tm[1]), 0x0040);
  const uint32_t b = __byte_perm(__float_as_uint(tm[2]), __float_as_uint(tm[3]), 0x0040);
  return __byte_perm(a, b, 0x5410);
}
__device__ __forceinline__ uint2 tm_pack4_s16(const float (&tm)[4]) {   // four mantissas as s16
  return make_uint2(__byte_perm(__float_as_uint(tm[0]), __float_as_uint(tm[1]), 0x5410),
                    __byte_perm(__float_as_uint(tm[2]), __float_as_uint(tm[3]), 0x5410));
}
__device__ __forceinline__ void tm_pack4_hilo(const float (&tm)[4], uint32_t& hi, uint32_t& lo) {   // k = 256 * hi + lo byte planes
  lo = tm_pack4(tm);
  const uint32_t a = __byte_perm(__float_as_uint(tm[0]), __float_as_uint(tm[1]), 0x0051);
  const uint32_t b = __byte_perm(__float_as_uint(tm[2]), __float_as_uint(tm[3]), 0x0051);
  hi = __byte_perm(a, b, 0x5410);
}
__device__ __forceinline__ void dec4_f(uint32_t w, float (&f)[4]) {   // four s8 mantissas -> float, no I2F
  const uint32_t wb = w ^ 0x80808080u;
#pragma unroll
  for (int j = 0; j < 4; ++j) f[j] = __fsub_rn(__uint_as_float(__byte_perm(wb, 0x4B000000u, 0x7650u | (uint32_t)j)), 8388736.0f);
}
__device__ __forceinline__ void dec4_f_s16(uint2 w, float (&f)[4]) {  // four s16 mantissas -> float
  const uint32_t a = w.x ^ 0x80008000u, b = w.y ^ 0x80008000u;
  f[0] = __fsub_rn(__uint_as_float(__byte_perm(a, 0x4B000000u, 0x7610u)), 8421376.0f);   // 2^23 + 2^15
  f[1] = __fsub_rn(__uint_as_float(__byte_perm(a, 0x4B000000u, 0x7632u)), 8421376.0f);
  f[2] = __fsub_rn(__uint_as_float(__byte_perm(b, 0x4B000000u, 0x7610u)), 8421376.0f);
  f[3] = __fsub_rn(__uint_as_float(__byte_perm(b, 0x4B000000u, 0x7632u)), 8421376.0f);
}
// a / b for many a over one b, correctly rounded (see fdiv_by): without the select that only restores the sign of a zero
// numerator — the quotient of +-0 is +-0 either way and nothing downstream depends on the sign of a zero.
__device__ __forceinline__ float fdiv_fast(float a, float b, float r) {
  const float q0 = __fmul_rn(a, r);
  float q = __fmaf_rn(__fmaf_rn(-b, q0, a), r, q0);
  return __fmaf_rn(__fmaf_rn(-b, q, a), r, q);
}

// x / n for the per-channel element count n.  The fp64 division is a ~20-deep dependent chain on a chip with a token fp64
// pipe (it is most of the 1.8 us per-CTA prologue of the apply kernels); when n is a power of two — every CIFAR-shaped
// layer at a power-of-two batch — the quotient is the exact scaling x * 2^-k, bit-identical to the division.
struct DivN {
  double n, inv;
  bool pow2;
};
__device__ __forceinline__ DivN make_divn(unsigned long long nn) {
  DivN d;
  d.n = (double)nn;
  d.pow2 = nn != 0ull && (nn & (nn - 1ull)) == 0ull;
  d.inv = d.pow2 ? __longlong_as_double((long long)(1023 - (__ffsll((long long)nn) - 1)) << 52) : 0.0;
  return d;
}
__device__ __forceinline__ double div_n(double x, const DivN& d) { return d.pow2 ? x * d.inv : x / d.n; }

// Batch moments of the quantised input from the exact integer sums (dfxp:588, biased variance),
// finished in fp64 and rounded once: mean = 2^-f * S1/n, var = 2^-2f * (S2/n - (S1/n)^2).
__device__ __forceinline__ void moments(const long long* sums, int C, int c, const DivN& n, float inv_m, float& mean, float& var) {
  const double s1 = (double)sums[c], s2 = (double)sums[C + c];
  const double mu = div_n(s1, n);
  double v = div_n(s2, n) - mu * mu;
  if (v < 0.0) v = 0.0;
  mean = (float)(mu * (double)inv_m);
  var = (float)(v * (double)inv_m * (double)inv_m);
}

// ------------------------------------------------------------------------------------------------
// fwd 1
// ------------------------------------------------------------------------------------------------
struct Fwd1Params {
  Tiling t;
  const float* x;
  QSite q;
  int8_t* k1;
  long long* sums;  // [2*C]
};

__global__ void __launch_bounds__(kThreads) bn_fwd1_kernel(const Fwd1Params p) {
  extern __shared__ unsigned long long s_acc[];
  __shared__ uint32_t s_red[16];
  pdl_trigger();
  pdl_wait();
  const QC c = make_qc(p.q.bits, __ldg(p.q.ib));
  const uint64_t off = site_offset(p.q);
  uint32_t n1 = 0, n2 = 0;
  float mx = -INFINITY, mn = INFINITY;
  const bool mm = p.q.minmax != 0;
  Acc<2> acc;
  acc.zero();
  for (uint64_t tile = blockIdx.x; tile < p.t.total_tiles; tile += gridDim.x) {
    const uint32_t rg = (uint32_t)(tile / p.t.chunks), ch = (uint32_t)(tile % p.t.chunks);
    const uint32_t v = ch * kThreads + threadIdx.x;
    if (v < p.t.n_vec) {
      const float4 u = site_noise(p.q, v, off);
      const uint32_t r0 = rg * p.t.rows_per_group, r1 = min(r0 + p.t.rows_per_group, (uint32_t)p.t.n_outer);   // rows: 32-bit (make_tiling)
      for (uint32_t r = r0; r < r1; r += kRows) {
        float4 xv[kRows];
#pragma unroll
        for (int i = 0; i < kRows; ++i)
          if (r + i < r1) xv[i] = __ldcs(reinterpret_cast<const float4*>(p.x) + ((r + i) * p.t.n_vec + v));
#pragma unroll
        for (int i = 0; i < kRows; ++i)
          if (r + i < r1) {
            float k[4];
            if (mm) {
              k[0] = squant_mm(xv[i].x, u.x, c, mx, mn);
              k[1] = squant_mm(xv[i].y, u.y, c, mx, mn);
              k[2] = squant_mm(xv[i].z, u.z, c, mx, mn);
              k[3] = squant_mm(xv[i].w, u.w, c, mx, mn);
            } else {
              k[0] = squant(xv[i].x, u.x, c, n1, n2);
              k[1] = squant(xv[i].y, u.y, c, n1, n2);
              k[2] = squant(xv[i].z, u.z, c, n1, n2);
              k[3] = squant(xv[i].w, u.w, c, n1, n2);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int ki = __float2int_rn(k[j]);
              acc.s[0][j] += ki;
              acc.s[1][j] += ki * ki;
            }
            *reinterpret_cast<uint32_t*>(p.k1 + (r + i) * p.t.n_inner + 4 * (size_t)v) = pack4(k);
          }
      }
      if (!p.t.fixed_channels) flush_global(acc, p.sums, p.t.C, (int)((4ull * v) % (uint64_t)p.t.C));
    }
  }
  if (p.t.fixed_channels) flush_block(acc, p.sums, p.t.C, s_acc);
  if (mm) mm_to_counts(c, mx, mn, n1, n2);
  publish_counters(p.q.counters, n1, n2, p.t.n_outer * p.t.n_inner, s_red);
}

// ------------------------------------------------------------------------------------------------
// fwd 2
// ------------------------------------------------------------------------------------------------
struct Fwd2Params {
  Tiling t;
  const int8_t* k1;
  int bits1;
  const int32_t* ib1;
  const long long* sums;  // [2*C] from fwd 1 (RUN: unused)
  float eps;
  QSite q2;               // Rescale_q's X quantiser
  const float* gq;        // quantised gamma [C]
  const float* bq;        // quantised beta  [C]
  const float* add;       // optional shortcut tensor, same shape
  int relu;
  int8_t* k2;             // RUN: optional
  float* out;
  float* batch_mean;      // [C] optional
  float* batch_var;       // [C] optional
  float* run_mean;        // [C] optional, updated in place with `momentum` (dfxp:602-612); RUN: the (read-only) mean / var
  float* run_var;
  float momentum, one_minus_momentum;   // the reference's Python constants `momentum` and `(1-momentum)`, each rounded to fp32
  QSite q3;               // optional: the consuming layer's input quantiser (bits == 0: off)
  uint8_t* next_mant;     // its mantissas (u8 for a 9-bit non-negative tensor, s8 otherwise: same byte)
  QSite q4;               // optional: a SECOND consumer's input quantiser (a block's strided 1x1 shortcut convolution reads the
  uint8_t* next_mant2;    // same tensor as its first 3x3 through its own quantiser, dfxp:287 in both Conv2d_q)
};

// MM: every quantiser of the launch keeps min/max statistics (LBT_STATS_MINMAX).  Per element: ~28 full-rate instructions,
// no conversion-pipe instruction (see "conversion-free arithmetic" above); power-of-two scale factors are folded into the
// per-channel constants where that commutes with the roundings exactly (x * 2^f scalings commute with RN):
//   y1 * m2 = RN((xq - mean) / den) * m2 = RN((xq - mean) / (den / m2));   RN(xq2 * g) = RN(k2 * (g / m2)).
// Q4: the second-consumer instantiation (its own registers: only the HBM-bound add + out launches in front of a strided block use it)
// RUN: eval mode (dfxp:616 with the running statistics): mean / var are read from run_mean / run_var instead of being formed
// from the batch sums; no batch moments, no running-average update, k2 optional.  Only the per-channel prologue differs.
template <bool MM, bool Q4 = false, bool RUN = false>
__global__ void __launch_bounds__(kThreads, Q4 ? 2 : LBT_BN_FWD2_CTAS) bn_fwd2_kernel(const Fwd2Params p) {
  extern __shared__ float s_par[];  // [4*C]: mean, den / m2, gq / m2, bq
  __shared__ uint32_t s_red[16];
  pdl_trigger();
  pdl_wait();
  const int C = p.t.C;
  {  // start pulling this CTA's first rows while the (slow, fp64) per-channel prologue runs
    const uint64_t tile = blockIdx.x;
    const uint32_t rg = (uint32_t)(tile / p.t.chunks), v = (uint32_t)(tile % p.t.chunks) * kThreads + threadIdx.x;
    if (tile < p.t.total_tiles && v < p.t.n_vec) {
      const uint32_t r0 = rg * p.t.rows_per_group, r1 = min(r0 + p.t.rows_per_group, (uint32_t)p.t.n_outer);   // rows: 32-bit (make_tiling)
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r0 + i < r1) {
          const size_t idx = 4 * (size_t)((r0 + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          prefetch_l1(p.k1 + idx);
          if (p.add) prefetch_l1(p.add + idx);
        }
    }
  }
  const QC c1 = make_qc(p.bits1, __ldg(p.ib1));
  const QC c2 = make_qc(p.q2.bits, __ldg(p.q2.ib));
  const DivN n = make_divn((unsigned long long)(p.t.n_outer * (p.t.n_inner / C)));
  for (int ch = threadIdx.x; ch < C; ch += kThreads) {
    float mean, var;
    if (RUN) {
      mean = p.run_mean[ch];
      var = p.run_var[ch];
    } else {
      moments(p.sums, C, ch, n, c1.inv_m, mean, var);
    }
    s_par[ch] = mean;
    s_par[C + ch] = __fsqrt_rn(__fadd_rn(var, p.eps)) * c2.inv_m;  // (var + eps) ** 0.5 (dfxp:616), pre-divided by m2 (exact)
    s_par[2 * C + ch] = p.gq[ch] * c2.inv_m;                         // gq / m2 (exact)
    s_par[3 * C + ch] = p.bq[ch];
    if (!RUN && blockIdx.x == 0) {
      if (p.batch_mean) p.batch_mean[ch] = mean;
      if (p.batch_var) p.batch_var[ch] = var;
      if (p.run_mean) {  // momentum * average + (1 - momentum) * variable
        p.run_mean[ch] = __fadd_rn(__fmul_rn(p.momentum, p.run_mean[ch]), __fmul_rn(p.one_minus_momentum, mean));
        p.run_var[ch] = __fadd_rn(__fmul_rn(p.momentum, p.run_var[ch]), __fmul_rn(p.one_minus_momentum, var));
      }
    }
  }
  __syncthreads();
  const uint64_t off = site_offset(p.q2);
  uint32_t n1 = 0, n2 = 0;
  float mx = -INFINITY, mn = INFINITY;
  const bool nxt = p.q3.bits != 0;
  QC c3 = c2;
  uint64_t off3 = 0;
  if (nxt) {
    c3 = make_qc(p.q3.bits, __ldg(p.q3.ib));
    off3 = site_offset(p.q3);
  }
  uint32_t m1 = 0, m2 = 0;
  float mx3 = -INFINITY, mn3 = INFINITY;
  QC c4 = c2;
  uint64_t off4 = 0;
  if (Q4) {
    c4 = make_qc(p.q4.bits, __ldg(p.q4.ib));
    off4 = site_offset(p.q4);
  }
  uint32_t l1 = 0, l2 = 0;
  float mx4 = -INFINITY, mn4 = INFINITY;
  const bool has_add = p.add != nullptr, relu = p.relu != 0, has_out = p.out != nullptr;
  for (uint64_t tile = blockIdx.x; tile < p.t.total_tiles; tile += gridDim.x) {
    const uint32_t rg = (uint32_t)(tile / p.t.chunks), chk = (uint32_t)(tile % p.t.chunks);
    const uint32_t v = chk * kThreads + threadIdx.x;
    if (v >= p.t.n_vec) continue;
    const int c0 = (int)((4ull * v) % (uint64_t)C);
    const float4 u = site_noise(p.q2, v, off);
    const float un[4] = {u.x, u.y, u.z, u.w};
    float u3[4] = {0.f, 0.f, 0.f, 0.f};
    if (nxt) {
      const float4 t = site_noise(p.q3, v, off3);
      u3[0] = t.x; u3[1] = t.y; u3[2] = t.z; u3[3] = t.w;
    }
    float u4n[4] = {0.f, 0.f, 0.f, 0.f};
    if (Q4) {
      const float4 t = site_noise(p.q4, v, off4);
      u4n[0] = t.x; u4n[1] = t.y; u4n[2] = t.z; u4n[3] = t.w;
    }
    float nmean[4], den[4], rden[4], g[4], b[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      nmean[j] = -s_par[c0 + j];
      den[j] = s_par[C + c0 + j];
      rden[j] = __frcp_rn(den[j]);   // one reciprocal per channel: every quotient below is a correctly rounded division (5 FMAs)
      g[j] = s_par[2 * C + c0 + j];
      b[j] = s_par[3 * C + c0 + j];
    }
    const uint32_t r0 = rg * p.t.rows_per_group, r1 = min(r0 + p.t.rows_per_group, (uint32_t)p.t.n_outer);   // rows: 32-bit (make_tiling)
    for (uint32_t r = r0; r < r1; r += kRows) {
      uint32_t kw[kRows];
      float4 av[kRows];
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r + i < r1) {
          const size_t idx = 4 * (size_t)((r + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          kw[i] = __ldcs(reinterpret_cast<const uint32_t*>(p.k1 + idx));
          if (has_add) av[i] = __ldcs(reinterpret_cast<const float4*>(p.add + idx));
        }
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r + kRows + i < r1) {
          const size_t idx = 4 * (size_t)((r + kRows + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          prefetch_l1(p.k1 + idx);
          if (has_add) prefetch_l1(p.add + idx);
        }
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r + i < r1) {
          const size_t idx = 4 * (size_t)((r + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          float k1f[4];
          dec4_f(kw[i], k1f);
          const float a4[4] = {av[i].x, av[i].y, av[i].z, av[i].w};
          float t2[4], o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            // xq - mean in one rounding (k1 * 2^-f is exact), then y1 * m2 = (xq - mean) / (den / m2)      dfxp:616
            const float y1m = fdiv_fast(__fmaf_rn(k1f[j], c1.inv_m, nmean[j]), den[j], rden[j]);
            t2[j] = sq_scaled<MM>(y1m, un[j], c2, mx, mn, n1, n2);                    // dfxp:677
            float y2 = __fadd_rn(__fmul_rn(tm_float(t2[j]), g[j]), b[j]);               // dfxp:683 (xq2 * gq, then + bq)
            if (has_add) y2 = __fadd_rn(y2, a4[j]);                                     // residual sum, dfxp:862
            if (relu) y2 = fmaxf(0.0f, y2);                                             // tf.maximum(0.0, X), dfxp:986
            o[j] = y2;
          }
          if (!RUN || p.k2) *reinterpret_cast<uint32_t*>(p.k2 + idx) = tm_pack4(t2);
          if (has_out) *reinterpret_cast<float4*>(p.out + idx) = make_float4(o[0], o[1], o[2], o[3]);
          if (nxt) {                                                                    // the consumer's Xq, dfxp:287
            float t3[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) t3[j] = sq_scaled<MM>(__fmul_rn(o[j], c3.m), u3[j], c3, mx3, mn3, m1, m2);
            *reinterpret_cast<uint32_t*>(p.next_mant + idx) = tm_pack4(t3);
          }
          if (Q4) {                                                                     // the second consumer's Xq
            float t4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) t4[j] = sq_scaled<MM>(__fmul_rn(o[j], c4.m), u4n[j], c4, mx4, mn4, l1, l2);
            *reinterpret_cast<uint32_t*>(p.next_mant2 + idx) = tm_pack4(t4);
          }
        }
    }
  }
  if (MM) mm_to_counts(c2, mx, mn, n1, n2);
  publish_counters(p.q2.counters, n1, n2, p.t.n_outer * p.t.n_inner, s_red);
  if (nxt) {
    if (MM) mm_to_counts(c3, mx3, mn3, m1, m2);
    publish_counters(p.q3.counters, m1, m2, p.t.n_outer * p.t.n_inner, s_red);
  }
  if (Q4) {
    if (MM) mm_to_counts(c4, mx4, mn4, l1, l2);
    publish_counters(p.q4.counters, l1, l2, p.t.n_outer * p.t.n_inner, s_red);
  }
}

// ------------------------------------------------------------------------------------------------
// fwd 2 + stride-2 3x3 max-pool (the ImageNet stem: conv -> BN -> ReLU -> tf.nn.max_pool 3x3/2 'SAME', models.py / dfxp:993-1006)
//
// lbt_bn_fwd_apply followed by lbt_maxpool_fwd writes the fp32 module output (4 B per element) only for the pool to read it
// back: 1.6 GB of the 2.3 GB the two kernels move on ResNet-18's stem.  Here a CTA owns an 8 x 16 pixel tile of the image for a
// group of batch rows; a thread owns a 2 x 2 block of pixels x 4 channels (its noise and per-channel constants in registers,
// like the stand-alone kernel), applies fwd 2 to them with the SAME arithmetic, stores k2, and leaves the post-ReLU values in
// shared memory; the first 400 threads also evaluate one pixel each of the tile's one-pixel halo (row 8 / column 16: the
// windows of the last block row / column reach into the next tile; values only — statistics and k2 belong to the owning tile).
// After ONE barrier (two shared-memory buffers) every thread takes the 3 x 3 window whose top-left pixel is its block's:
// maximum and winning tap in lbt_maxpool_fwd's scan order, so pooled values and indices are bit-identical.  C == 64.
// ------------------------------------------------------------------------------------------------
constexpr int kPoolTH = 8, kPoolTW = 16, kPoolCG = 16, kPoolThreads = 512;
constexpr int kPoolHalo = (kPoolTH + 1) * (kPoolTW + 1) - kPoolTH * kPoolTW;   // 25 halo pixels per tile

struct Fwd2PoolParams {
  const int8_t* k1;
  int bits1;
  const int32_t* ib1;
  const long long* sums;
  float eps;
  QSite q2;
  const float* gq;
  const float* bq;
  int relu;
  int8_t* k2;
  float* run_mean;
  float* run_var;
  float momentum, one_minus_momentum;
  float* pooled;           // [N, POH, POW, 64]
  uint8_t* pidx;           // winning tap r * 3 + q
  QSite q3;                // optional: the input quantiser of the layer that consumes the POOLED tensor (bits == 0: off)
  uint8_t* next_mant;      // its mantissas [N, POH, POW, 64] (u8 for a 9-bit non-negative tensor, s8 otherwise: same byte)
  uint32_t N, H, W, POH, POW;
  uint32_t tiles_x, tiles_img, rows_per_group, total_tiles;
};

// RUN: eval mode, as in bn_fwd2_kernel (run_mean / run_var are the read-only source of mean / var, k2 optional)
template <bool MM, bool RUN = false>
__global__ void __launch_bounds__(kPoolThreads, 1) bn_fwd2_pool_kernel(const Fwd2PoolParams p) {
  extern __shared__ float4 s_y[];   // [2][kPoolTH + 1][kPoolTW + 1][kPoolCG]
  __shared__ float s_par[4 * 64];   // mean, den / m2, gq / m2, bq
  pdl_trigger();
  pdl_wait();
  constexpr int C = 64;
  const QC c1 = make_qc(p.bits1, __ldg(p.ib1));
  const QC c2 = make_qc(p.q2.bits, __ldg(p.q2.ib));
  const DivN n = make_divn((unsigned long long)p.N * p.H * p.W);
  if (threadIdx.x < C) {
    const int ch = threadIdx.x;
    float mean, var;
    if (RUN) {
      mean = p.run_mean[ch];
      var = p.run_var[ch];
    } else {
      moments(p.sums, C, ch, n, c1.inv_m, mean, var);
    }
    s_par[ch] = mean;
    s_par[C + ch] = __fsqrt_rn(__fadd_rn(var, p.eps)) * c2.inv_m;
    s_par[2 * C + ch] = p.gq[ch] * c2.inv_m;
    s_par[3 * C + ch] = p.bq[ch];
    if (!RUN && blockIdx.x == 0 && p.run_mean) {
      p.run_mean[ch] = __fadd_rn(__fmul_rn(p.momentum, p.run_mean[ch]), __fmul_rn(p.one_minus_momentum, mean));
      p.run_var[ch] = __fadd_rn(__fmul_rn(p.momentum, p.run_var[ch]), __fmul_rn(p.one_minus_momentum, var));
    }
  }
  __syncthreads();
  const uint64_t off = site_offset(p.q2);
  const uint32_t cg = threadIdx.x & (kPoolCG - 1), blk = threadIdx.x >> 4, by = blk >> 3, bx = blk & 7;
  float nmean[4], den[4], rden[4], g[4], b[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    nmean[j] = -s_par[4 * cg + j];
    den[j] = s_par[C + 4 * cg + j];
    rden[j] = __frcp_rn(den[j]);
    g[j] = s_par[2 * C + 4 * cg + j];
    b[j] = s_par[3 * C + 4 * cg + j];
  }
  const bool relu = p.relu != 0;
  // halo task of this thread: pixel hp of the tile's extra row (ly = 8, lx = 0..16) / extra column (lx = 16, ly = 0..7)
  const uint32_t hp = threadIdx.x >> 4;
  const bool halo_task = hp < (uint32_t)kPoolHalo;
  const uint32_t hly = hp <= (uint32_t)kPoolTW ? (uint32_t)kPoolTH : hp - (kPoolTW + 1), hlx = hp <= (uint32_t)kPoolTW ? hp : (uint32_t)kPoolTW;
  uint32_t n1 = 0, n2 = 0;
  float mx = -INFINITY, mn = INFINITY;
  const bool nxt = p.q3.bits != 0;
  QC c3 = c2;
  uint64_t off3 = 0;
  if (nxt) {
    c3 = make_qc(p.q3.bits, __ldg(p.q3.ib));
    off3 = site_offset(p.q3);
  }
  uint32_t m1 = 0, m2 = 0;
  float mx3 = -INFINITY, mn3 = INFINITY;
  const uint32_t HW = p.H * p.W, PHW = p.POH * p.POW;
  const uint32_t* const k1w = reinterpret_cast<const uint32_t*>(p.k1);
  uint32_t* const k2w = reinterpret_cast<uint32_t*>(p.k2);
  uint32_t buf = 0;
  auto apply4 = [&](uint32_t w, const float (&un)[4], float& smx, float& smn, uint32_t& s1, uint32_t& s2, float (&o)[4]) -> uint32_t {
    float k1f[4], t2[4];
    dec4_f(w, k1f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float y1m = fdiv_fast(__fmaf_rn(k1f[j], c1.inv_m, nmean[j]), den[j], rden[j]);   // dfxp:616
      t2[j] = sq_scaled<MM>(y1m, un[j], c2, smx, smn, s1, s2);                                // dfxp:677
      float y2 = __fadd_rn(__fmul_rn(tm_float(t2[j]), g[j]), b[j]);                           // dfxp:683
      if (relu) y2 = fmaxf(0.0f, y2);                                                          // dfxp:986
      o[j] = y2;
    }
    return tm_pack4(t2);
  };
  for (uint32_t tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const uint32_t rg = tile / p.tiles_img, tt = tile - rg * p.tiles_img;
    const uint32_t ty = tt / p.tiles_x, tx = tt - ty * p.tiles_x;
    const uint32_t y0 = ty * kPoolTH, x0 = tx * kPoolTW;
    // own 2 x 2 block
    uint32_t pw[4];     // word index of pixel (py, px) inside an image: (y * W + x) * 16 + cg
    bool pv[4];
    float un[4][4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t y = y0 + 2 * by + (q >> 1), x = x0 + 2 * bx + (q & 1);
      pv[q] = y < p.H && x < p.W;
      pw[q] = (y * p.W + x) * kPoolCG + cg;
      const float4 u = pv[q] ? site_noise(p.q2, pw[q], off) : make_float4(0.f, 0.f, 0.f, 0.f);
      un[q][0] = u.x; un[q][1] = u.y; un[q][2] = u.z; un[q][3] = u.w;
    }
    const uint32_t hy = y0 + hly, hx = x0 + hlx;
    const bool hv = halo_task && hy < p.H && hx < p.W;
    const uint32_t hw = (hy * p.W + hx) * kPoolCG + cg;
    float hun[4] = {0.f, 0.f, 0.f, 0.f};
    if (hv) {
      const float4 u = site_noise(p.q2, hw, off);
      hun[0] = u.x; hun[1] = u.y; hun[2] = u.z; hun[3] = u.w;
    }
    // the pooling window of this thread: output (a, b), top-left pixel = the block's
    const uint32_t pa = (y0 >> 1) + by, pb = (x0 >> 1) + bx;
    const bool wv = pa < p.POH && pb < p.POW;
    float u3[4] = {0.f, 0.f, 0.f, 0.f};
    if (nxt && wv) {
      const float4 t = site_noise(p.q3, (pa * p.POW + pb) * kPoolCG + cg, off3);
      u3[0] = t.x; u3[1] = t.y; u3[2] = t.z; u3[3] = t.w;
    }
    bool tok[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int q = 0; q < 3; ++q) tok[3 * r + q] = (y0 + 2 * by + r) < p.H && (x0 + 2 * bx + q) < p.W;
    const uint32_t r0 = rg * p.rows_per_group, r1 = min(r0 + p.rows_per_group, p.N);
    for (uint32_t r = r0; r < r1; ++r) {
      const uint32_t ibase = r * HW * kPoolCG;
      uint32_t w[4], wh = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (pv[q]) w[q] = __ldcs(k1w + ibase + pw[q]);
      if (hv) wh = __ldg(k1w + ibase + hw);   // the neighbouring tile reads this pixel too
      if (r + 1 < r1) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (pv[q]) prefetch_l1(k1w + ibase + HW * kPoolCG + pw[q]);
      }
      float4* sy = s_y + (size_t)buf * ((kPoolTH + 1) * (kPoolTW + 1) * kPoolCG);
      float own[4][4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (pv[q]) {
          const uint32_t k2p = apply4(w[q], un[q], mx, mn, n1, n2, own[q]);
          if (!RUN || k2w) k2w[ibase + pw[q]] = k2p;
          sy[((2 * by + (q >> 1)) * (kPoolTW + 1) + 2 * bx + (q & 1)) * kPoolCG + cg] = make_float4(own[q][0], own[q][1], own[q][2], own[q][3]);
        }
      if (hv) {
        float ho[4], dmx = 0.f, dmn = 0.f;
        uint32_t d1 = 0, d2 = 0;
        (void)apply4(wh, hun, dmx, dmn, d1, d2, ho);
        sy[(hly * (kPoolTW + 1) + hlx) * kPoolCG + cg] = make_float4(ho[0], ho[1], ho[2], ho[3]);
      }
      __syncthreads();
      if (wv) {
        float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
        uchar4 wt = make_uchar4(0, 0, 0, 0);
#pragma unroll
        for (int tq = 0; tq < 9; ++tq) {
          const int tr = tq / 3, tc = tq % 3;
          if (!tok[tq]) continue;
          float4 a;
          if (tr < 2 && tc < 2) a = make_float4(own[2 * tr + tc][0], own[2 * tr + tc][1], own[2 * tr + tc][2], own[2 * tr + tc][3]);
          else a = sy[((2 * by + tr) * (kPoolTW + 1) + 2 * bx + tc) * kPoolCG + cg];
          const unsigned char t8 = (unsigned char)tq;
          if (a.x > m.x || a.x != a.x) { m.x = a.x; wt.x = t8; }
          if (a.y > m.y || a.y != a.y) { m.y = a.y; wt.y = t8; }
          if (a.z > m.z || a.z != a.z) { m.z = a.z; wt.z = t8; }
          if (a.w > m.w || a.w != a.w) { m.w = a.w; wt.w = t8; }
        }
        const uint32_t o = (r * PHW + pa * p.POW + pb) * kPoolCG + cg;
        reinterpret_cast<float4*>(p.pooled)[o] = m;
        reinterpret_cast<uchar4*>(p.pidx)[o] = wt;
        if (nxt) {                                                                      // the consumer's Xq, dfxp:287
          const float mm4[4] = {m.x, m.y, m.z, m.w};
          float t3[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) t3[j] = sq_scaled<MM>(__fmul_rn(mm4[j], c3.m), u3[j], c3, mx3, mn3, m1, m2);
          reinterpret_cast<uint32_t*>(p.next_mant)[o] = tm_pack4(t3);
        }
      }
      buf ^= 1u;
    }
    __syncthreads();   // the next tile's first write may target the buffer another thread still reads
  }
  if (MM) mm_to_counts(c2, mx, mn, n1, n2);
  n1 = warp_sum(n1);
  n2 = warp_sum(n2);
  if ((threadIdx.x & 31) == 0 && p.q2.counters) {
    if (n1) atomicAdd(p.q2.counters + LBT_CNT_OVER, (unsigned long long)n1);
    if (n2) atomicAdd(p.q2.counters + LBT_CNT_OVER_HALF, (unsigned long long)n2);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && p.q2.counters)
    atomicAdd(p.q2.counters + LBT_CNT_NUMEL, (unsigned long long)p.N * p.H * p.W * C);
  if (nxt) {
    if (MM) mm_to_counts(c3, mx3, mn3, m1, m2);
    m1 = warp_sum(m1);
    m2 = warp_sum(m2);
    if ((threadIdx.x & 31) == 0 && p.q3.counters) {
      if (m1) atomicAdd(p.q3.counters + LBT_CNT_OVER, (unsigned long long)m1);
      if (m2) atomicAdd(p.q3.counters + LBT_CNT_OVER_HALF, (unsigned long long)m2);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && p.q3.counters)
      atomicAdd(p.q3.counters + LBT_CNT_NUMEL, (unsigned long long)p.N * p.POH * p.POW * C);
  }
}

// ------------------------------------------------------------------------------------------------
// bwd 1
// ------------------------------------------------------------------------------------------------
struct Bwd1Params {
  Tiling t;
  const float* g;       // gradient w.r.t. the module output
  const float* out;     // module output (needed for the ReLU mask when `add` was fused), or NULL
  int relu;             // 0 none, 1 mask recomputed from k2 (no add), 2 mask from `out`
  const int8_t* k2;
  const int8_t* k1;
  int bits2;
  const int32_t* ib2;
  const float* gq;
  const float* bq;
  QSite qg2;            // Rescale_q's gradient quantiser (dfxp:687)
  QSite qg1;            // Normalization_q's gradient quantiser (dfxp:621)
  float* d_add;         // optional: gradient w.r.t. the fused shortcut input (= masked g)
  void* kg1;            // s8, or s16 in the WIDE instantiation
  long long* sums;      // [4*C]: sum kg2, sum kg2*k2, sum kg1, sum kg1*k1
  // POOL instantiation: `g` is the gradient of a max-pool of the module output, [n_outer, pOH, pOW, C]; the pool's backward
  // (a gather over the <= 2 x 2 windows that cover a pixel, lbt_maxpool_bwd) runs in this kernel's load stage
  const uint8_t* pidx;  // winning tap of every pooled element
  int pW, pk, ps, ppt, ppl, pOH, pOW;
  FastDiv d_c4, d_pW, d_ps;
};

// WIDE: a gradient quantiser wider than 8 bits — kg1 is stored as s16 and the per-thread partial sums are 64-bit
// (a 16-bit mantissa times an 8-bit one, summed down 4096 rows, does not fit 32).  MM: min/max statistics for both sites.
// RELU: 0 none, 1 mask recomputed from k2, 2 mask from `out`.  ~31 full-rate instructions per element, no conversions;
// folded constants (exact, powers of two):  RN(xq2 * g) = RN(k2 * (g / m2));  dx2 * mg1 = RN(kg2 * (g * mg1 / mg2)).
template <bool WIDE, bool MM, int RELU, bool POOL = false>
__global__ void __launch_bounds__(kThreads, LBT_BN_BWD1_CTAS) bn_bwd1_kernel(const Bwd1Params p) {
  extern __shared__ unsigned long long s_acc[];
  __shared__ uint32_t s_red[16];
  pdl_trigger();
  pdl_wait();
  const int C = p.t.C;
  const QC c2 = make_qc(p.bits2, __ldg(p.ib2));
  const QC cg2 = make_qc(p.qg2.bits, __ldg(p.qg2.ib));
  const QC cg1 = make_qc(p.qg1.bits, __ldg(p.qg1.ib));
  const uint64_t off2 = site_offset(p.qg2), off1 = site_offset(p.qg1);
  uint32_t a1 = 0, a2 = 0, b1 = 0, b2 = 0;
  float amx = -INFINITY, amn = INFINITY, bmx = -INFINITY, bmn = INFINITY;
  using AccT = typename std::conditional<WIDE, long long, int>::type;
  Acc<4, AccT> acc;
  acc.zero();
  const float gscale = cg2.inv_m * cg1.m;   // kg2 -> dx2 (x 2^-fg2) -> scaled for the second quantiser (x 2^fg1): exact
  const bool has_dadd = p.d_add != nullptr;
  for (uint64_t tile = blockIdx.x; tile < p.t.total_tiles; tile += gridDim.x) {
    const uint32_t rg = (uint32_t)(tile / p.t.chunks), chk = (uint32_t)(tile % p.t.chunks);
    const uint32_t v = chk * kThreads + threadIdx.x;
    if (v < p.t.n_vec) {
      const int c0 = (int)((4ull * v) % (uint64_t)C);
      const float4 u2v = site_noise(p.qg2, v, off2), u1v = site_noise(p.qg1, v, off1);
      const float u2[4] = {u2v.x, u2v.y, u2v.z, u2v.w}, u1[4] = {u1v.x, u1v.y, u1v.z, u1v.w};
      float gk[4], b[4], gd[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float gq = __ldg(p.gq + c0 + j);
        gk[j] = gq * c2.inv_m;     // for the ReLU mask: xq2 * gq = k2 * (gq / m2)
        gd[j] = gq * gscale;       // dx2 * mg1 = kg2 * (gq * mg1 / mg2)
        b[j] = __ldg(p.bq + c0 + j);
      }
      const uint32_t r0 = rg * p.t.rows_per_group, r1 = min(r0 + p.t.rows_per_group, (uint32_t)p.t.n_outer);   // rows: 32-bit (make_tiling)
      // POOL: the <= 2 x 2 pooling windows over this thread's pixel — the same for every batch row (tf.nn.max_pool's
      // gradient, dfxp:993-1006: a pixel receives the gradient of each window it won; lbt_maxpool_bwd's gather and order)
      uint32_t poff[4] = {0u, 0u, 0u, 0u};
      uint32_t ptap[4] = {0u, 0u, 0u, 0u};
      bool pok[4] = {false, false, false, false};
      size_t pimg = 0;
      if (POOL) {
        const uint32_t pix = fastdiv(v, p.d_c4), cg = v - pix * p.d_c4.d;
        const uint32_t ih = fastdiv(pix, p.d_pW), iw = pix - ih * (uint32_t)p.pW;
        const int th = (int)ih + p.ppt, tw = (int)iw + p.ppl;
        const int oh_lo = th - p.pk + 1 <= 0 ? 0 : (int)fastdiv((uint32_t)(th - p.pk + p.ps), p.d_ps);
        const int ow_lo = tw - p.pk + 1 <= 0 ? 0 : (int)fastdiv((uint32_t)(tw - p.pk + p.ps), p.d_ps);
        const int oh_hi = min(p.pOH - 1, (int)fastdiv((uint32_t)th, p.d_ps)), ow_hi = min(p.pOW - 1, (int)fastdiv((uint32_t)tw, p.d_ps));
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b2 = 0; b2 < 2; ++b2) {
            const int oh = oh_lo + a, ow = ow_lo + b2;
            pok[2 * a + b2] = oh <= oh_hi && ow <= ow_hi;
            ptap[2 * a + b2] = (uint32_t)((th - oh * p.ps) * p.pk + (tw - ow * p.ps)) & 0xffu;
            poff[2 * a + b2] = pok[2 * a + b2] ? ((uint32_t)(oh * p.pOW + ow) * (uint32_t)C + 4u * cg) : 0u;
          }
        pimg = (size_t)p.pOH * p.pOW * C;
      }
      for (uint32_t r = r0; r < r1; r += kRows) {
        float4 gv[kRows], ov[kRows];
        uint32_t w2[kRows], w1[kRows];
#pragma unroll
        for (int i = 0; i < kRows; ++i)
          if (r + i < r1) {
            const size_t idx = 4 * (size_t)((r + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
            if (POOL) {
              const size_t base = (size_t)(r + i) * pimg;
              float4 gw[4];
              uint32_t iw4[4];
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (pok[q]) {
                  gw[q] = __ldg(reinterpret_cast<const float4*>(p.g + base + poff[q]));
                  iw4[q] = __ldg(reinterpret_cast<const uint32_t*>(p.pidx + base + poff[q]));
                }
              float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
              for (int q = 0; q < 4; ++q)       // (oh, ow) ascending: lbt_maxpool_bwd's order of additions
                if (pok[q]) {
                  if ((iw4[q] & 0xffu) == ptap[q]) a4.x += gw[q].x;
                  if (((iw4[q] >> 8) & 0xffu) == ptap[q]) a4.y += gw[q].y;
                  if (((iw4[q] >> 16) & 0xffu) == ptap[q]) a4.z += gw[q].z;
                  if ((iw4[q] >> 24) == ptap[q]) a4.w += gw[q].w;
                }
              gv[i] = a4;
            } else {
              gv[i] = __ldcs(reinterpret_cast<const float4*>(p.g + idx));
            }
            w2[i] = __ldcs(reinterpret_cast<const uint32_t*>(p.k2 + idx));
            w1[i] = __ldcs(reinterpret_cast<const uint32_t*>(p.k1 + idx));
            if (RELU == 2) ov[i] = __ldcs(reinterpret_cast<const float4*>(p.out + idx));
          }
#pragma unroll
        for (int i = 0; i < kRows; ++i)
          if (r + kRows + i < r1) {
            const size_t idx = 4 * (size_t)((r + kRows + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
            if (POOL) {
              const size_t base = (size_t)(r + kRows + i) * pimg;
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (pok[q]) {
                  prefetch_l1(p.g + base + poff[q]);
                  prefetch_l1(p.pidx + base + poff[q]);
                }
            } else {
              prefetch_l1(p.g + idx);
            }
            prefetch_l1(p.k2 + idx);
            prefetch_l1(p.k1 + idx);
            if (RELU == 2) prefetch_l1(p.out + idx);
          }
#pragma unroll
        for (int i = 0; i < kRows; ++i)
          if (r + i < r1) {
            const size_t idx = 4 * (size_t)((r + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
            int k2[4], k1[4];
            unpack4(w2[i], k2);
            unpack4(w1[i], k1);
            float k2f[4];
            if (RELU == 1) dec4_f(w2[i], k2f);
            const float gin[4] = {gv[i].x, gv[i].y, gv[i].z, gv[i].w};
            const float oin[4] = {ov[i].x, ov[i].y, ov[i].z, ov[i].w};
            float gm[4], t1[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float gj = gin[j];
              if (RELU == 1) {
                const float y2 = __fadd_rn(__fmul_rn(k2f[j], gk[j]), b[j]);
                if (!(y2 > 0.0f)) gj = 0.0f;
              } else if (RELU == 2) {
                if (!(oin[j] > 0.0f)) gj = 0.0f;
              }
              gm[j] = gj;
              const float tg2 = sq_scaled<MM>(__fmul_rn(gj, cg2.m), u2[j], cg2, amx, amn, a1, a2);   // dfxp:687
              const int kg2i = tm_int(tg2);
              acc.s[0][j] += kg2i;                                                 // dbeta  (dfxp:690)
              acc.s[1][j] += (AccT)kg2i * k2[j];                                   // dgamma (dfxp:689)
              // dx2 = gq2 * gamma_q (dfxp:691), scaled for the next quantiser (dfxp:621) in the same multiply
              t1[j] = sq_scaled<MM>(__fmul_rn(tm_float(tg2), gd[j]), u1[j], cg1, bmx, bmn, b1, b2);
              const int kg1i = tm_int(t1[j]);
              acc.s[2][j] += kg1i;
              acc.s[3][j] += (AccT)kg1i * k1[j];
            }
            if (has_dadd) *reinterpret_cast<float4*>(p.d_add + idx) = make_float4(gm[0], gm[1], gm[2], gm[3]);
            if (WIDE) *reinterpret_cast<uint2*>(reinterpret_cast<int16_t*>(p.kg1) + idx) = tm_pack4_s16(t1);
            else *reinterpret_cast<uint32_t*>(reinterpret_cast<int8_t*>(p.kg1) + idx) = tm_pack4(t1);
          }
      }
      if (!p.t.fixed_channels) flush_global(acc, p.sums, C, c0);
    }
  }
  if (p.t.fixed_channels) flush_block(acc, p.sums, C, s_acc);
  const size_t numel = p.t.n_outer * p.t.n_inner;
  if (MM) {
    mm_to_counts(cg2, amx, amn, a1, a2);
    mm_to_counts(cg1, bmx, bmn, b1, b2);
  }
  publish_counters(p.qg2.counters, a1, a2, numel, s_red);
  publish_counters(p.qg1.counters, b1, b2, numel, s_red);
}

// ------------------------------------------------------------------------------------------------
// bwd 2
// ------------------------------------------------------------------------------------------------
struct Bwd2Params {
  Tiling t;
  const void* kg1;         // s8, or s16 in the WIDE instantiation
  const int8_t* k1;
  int bits1;
  const int32_t* ib1;
  const long long* fsums;  // [2*C] forward sums
  float eps;
  int bitsg1;
  const int32_t* ibg1;
  const long long* bsums;  // [4*C] backward sums (uses [2C..4C))
  float* dx;               // may be NULL when qg is on
  QSite qg;                // optional: the producing convolution's gradient quantiser (bits == 0: off)
  int8_t* g_mant;          // its mantissas: s8, or the HIGH byte plane when qg.bits > 8 ...
  uint8_t* g_mant_lo;      // ... with the low byte plane here (k = 256 * hi + lo)
};

// WIDE: kg1 is s16.  MM: min/max statistics for the fused gradient quantiser.  ~27 full-rate instructions per element.
template <bool WIDE, bool MM>
__global__ void __launch_bounds__(kThreads) bn_bwd2_kernel(const Bwd2Params p) {
  extern __shared__ float s_par[];  // [4*C]: -mean, den, mean_g, mean_gxhat
  __shared__ uint32_t s_red[16];
  pdl_trigger();
  pdl_wait();
  bn_stamp(0);
  const int C = p.t.C;
  const bool gq_on = p.qg.bits != 0;
  QC cq = make_qc(8, 0);
  uint64_t offq = 0;
  if (gq_on) {
    cq = make_qc(p.qg.bits, __ldg(p.qg.ib));
    offq = site_offset(p.qg);
  }
  uint32_t n1 = 0, n2 = 0;
  float mx = -INFINITY, mn = INFINITY;
  {  // start pulling this CTA's first rows while the (slow, fp64) per-channel prologue runs
    const uint64_t tile = blockIdx.x;
    const uint32_t rg = (uint32_t)(tile / p.t.chunks), v = (uint32_t)(tile % p.t.chunks) * kThreads + threadIdx.x;
    if (tile < p.t.total_tiles && v < p.t.n_vec) {
      const uint32_t r0 = rg * p.t.rows_per_group, r1 = min(r0 + p.t.rows_per_group, (uint32_t)p.t.n_outer);   // rows: 32-bit (make_tiling)
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r0 + i < r1) {
          const size_t idx = 4 * (size_t)((r0 + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          prefetch_l1(reinterpret_cast<const int8_t*>(p.kg1) + (WIDE ? 2 : 1) * idx);
          prefetch_l1(p.k1 + idx);
        }
    }
  }
  const bool q16 = gq_on && p.qg.bits > 8;
  const bool has_dx = p.dx != nullptr;
  const QC c1 = make_qc(p.bits1, __ldg(p.ib1));
  const QC cg = make_qc(p.bitsg1, __ldg(p.ibg1));
  const DivN n = make_divn((unsigned long long)(p.t.n_outer * (p.t.n_inner / C)));
  for (int ch = threadIdx.x; ch < C; ch += kThreads) {
    float mean, var;
    moments(p.fsums, C, ch, n, c1.inv_m, mean, var);
    const float den = __fsqrt_rn(__fadd_rn(var, p.eps));
    // mean(gq) and mean(gq * xhat) from the exact integer sums, finished in fp64
    const double sg = (double)p.bsums[2 * C + ch] * (double)cg.inv_m;                       // sum gq
    const double sgx = (double)p.bsums[3 * C + ch] * (double)cg.inv_m * (double)c1.inv_m;   // sum gq*xq
    const double mg = div_n(sg, n);
    // mean(gq * xhat); every fp64 operation rounded on its own (no DFMA contraction) so the oracle can restate it
    const double mgx = div_n(__ddiv_rn(__dsub_rn(sgx, __dmul_rn((double)mean, sg)), (double)den), n);
    s_par[ch] = -mean;
    s_par[C + ch] = den;
    s_par[2 * C + ch] = (float)mg;
    s_par[3 * C + ch] = (float)mgx;
  }
  bn_stamp(1);
  __syncthreads();
  bn_stamp(2);
  const uint32_t nv = p.t.n_vec;   // words (4 elements) per row
  const uint32_t* const bkg = reinterpret_cast<const uint32_t*>(p.kg1);
  const uint32_t* const bk1 = reinterpret_cast<const uint32_t*>(p.k1);
  uint32_t* const bgm = reinterpret_cast<uint32_t*>(p.g_mant);
  uint32_t* const bgl = reinterpret_cast<uint32_t*>(p.g_mant_lo);
  float4* const bdx = reinterpret_cast<float4*>(p.dx);
  for (uint64_t tile = blockIdx.x; tile < p.t.total_tiles; tile += gridDim.x) {
    const uint32_t rg = (uint32_t)(tile / p.t.chunks), chk = (uint32_t)(tile % p.t.chunks);
    const uint32_t v = chk * kThreads + threadIdx.x;
    if (v >= p.t.n_vec) continue;
    const int c0 = (int)((4ull * v) % (uint64_t)C);
    float nmean[4], den[4], rden[4], mg[4], mgx[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      nmean[j] = s_par[c0 + j];
      den[j] = s_par[C + c0 + j];
      rden[j] = __frcp_rn(den[j]);
      mg[j] = s_par[2 * C + c0 + j];
      mgx[j] = s_par[3 * C + c0 + j];
    }
    float uq[4] = {0.f, 0.f, 0.f, 0.f};
    if (gq_on) {
      const float4 t = site_noise(p.qg, v, offq);
      uq[0] = t.x; uq[1] = t.y; uq[2] = t.z; uq[3] = t.w;
    }
    const uint32_t r0 = rg * p.t.rows_per_group, r1 = min(r0 + p.t.rows_per_group, (uint32_t)p.t.n_outer);   // rows: 32-bit (make_tiling)
    // One group of kRows rows.  FULL (all rows of the group exist — every group but a tile's last): no per-row predicates.
    // Every tensor is addressed as base + 4-element word index (32-bit, one IMAD.WIDE per access).
    auto group = [&](auto full_tag, const uint32_t r) {
      constexpr bool FULL = decltype(full_tag)::value;
      const uint32_t w0 = r * nv + v;
      uint2 wg[kRows];
      uint32_t w1[kRows];
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (FULL || r + i < r1) {
          const uint32_t w = w0 + (uint32_t)i * nv;
          if (WIDE) wg[i] = __ldcs(reinterpret_cast<const uint2*>(bkg) + w);
          else wg[i].x = __ldcs(bkg + w);
          w1[i] = __ldcs(bk1 + w);
        }
      if (r + 2 * kRows <= r1) {   // the next group, whole: into L1 while this one is computed
#pragma unroll
        for (int i = 0; i < kRows; ++i) {
          const uint32_t w = w0 + (uint32_t)(kRows + i) * nv;
          prefetch_l1(WIDE ? reinterpret_cast<const void*>(reinterpret_cast<const uint2*>(bkg) + w) : reinterpret_cast<const void*>(bkg + w));
          prefetch_l1(bk1 + w);
        }
      } else {
#pragma unroll
        for (int i = 0; i < kRows; ++i)
          if (r + kRows + i < r1) {
            const uint32_t w = w0 + (uint32_t)(kRows + i) * nv;
            prefetch_l1(WIDE ? reinterpret_cast<const void*>(reinterpret_cast<const uint2*>(bkg) + w) : reinterpret_cast<const void*>(bkg + w));
            prefetch_l1(bk1 + w);
          }
      }
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (FULL || r + i < r1) {
          const uint32_t w = w0 + (uint32_t)i * nv;
          float kgf[4], k1f[4];
          if (WIDE) dec4_f_s16(wg[i], kgf);
          else dec4_f(wg[i].x, kgf);
          dec4_f(w1[i], k1f);
          float o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float gq = __fmul_rn(kgf[j], cg.inv_m);
            const float xhat = fdiv_fast(__fmaf_rn(k1f[j], c1.inv_m, nmean[j]), den[j], rden[j]);
            // batch-norm VJP through mean and biased variance (tf.gradients of dfxp:616); one rounding per operation
            o[j] = fdiv_fast(__fsub_rn(__fsub_rn(gq, mg[j]), __fmul_rn(xhat, mgx[j])), den[j], rden[j]);
          }
          if (has_dx) bdx[w] = make_float4(o[0], o[1], o[2], o[3]);
          if (gq_on) {                                                        // the convolution's gradq, dfxp:300
            float tq[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) tq[j] = sq_scaled<MM>(__fmul_rn(o[j], cq.m), uq[j], cq, mx, mn, n1, n2);
            if (q16) {   // 9..16-bit gradient: the two byte planes the tensor cores consume (no separate split pass)
              uint32_t hi, lo;
              tm_pack4_hilo(tq, hi, lo);
              bgm[w] = hi;
              bgl[w] = lo;
            } else {
              bgm[w] = tm_pack4(tq);
            }
          }
        }
    };
    for (uint32_t r = r0; r < r1; r += kRows) {
      if (r + kRows <= r1) group(std::true_type{}, r);
      else group(std::false_type{}, r);
    }
  }
  bn_stamp(3);
  if (gq_on) {
    if (MM) mm_to_counts(cq, mx, mn, n1, n2);
    publish_counters(p.qg.counters, n1, n2, p.t.n_outer * p.t.n_inner, s_red);
  }
  bn_stamp(4);
}

// ------------------------------------------------------------------------------------------------
// bwd 1 + bwd 2 in ONE launch for tensors that fit one wave of resident CTAs (every tensor of a CIFAR-size step):
// pass 1 as above, but the mantissas the second pass needs (kg1, k1) stay in shared memory; the CTAs then meet at a
// grid-wide barrier (one int64 word from the step's zeroed arena: all CTAs are co-resident by construction) and run
// pass 2 from shared memory.  Saves a launch + dependent-launch gap, the kg1 round trip through HBM and a prologue.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxSavedRows = 16;

struct BwdFusedParams {
  Bwd1Params a;
  Bwd2Params b;               // b.kg1 / b.k1 unused (shared memory)
  unsigned long long* bar;    // grid barrier word, zero at launch
};

__device__ int g_bn_error = 0;

__global__ void __launch_bounds__(kThreads, 2) bn_bwd_fused_kernel(const BwdFusedParams q) {
  extern __shared__ unsigned long long s_dyn[];
  __shared__ uint32_t s_red[16];
  const Bwd1Params& p = q.a;
  const Bwd2Params& p2 = q.b;
  const int C = p.t.C;
  unsigned long long* s_acc = s_dyn;                                    // [4*C] (pass 1), then float s_par[4*C]
  uint2* s_save = reinterpret_cast<uint2*>(s_dyn + 4 * C);              // [rows_per_group][kThreads]: {kg1 word, k1 word}
  pdl_trigger();
  pdl_wait();
  const QC c2 = make_qc(p.bits2, __ldg(p.ib2));
  const QC cg2 = make_qc(p.qg2.bits, __ldg(p.qg2.ib));
  const QC cg1 = make_qc(p.qg1.bits, __ldg(p.qg1.ib));
  const QC c1 = make_qc(p2.bits1, __ldg(p2.ib1));
  const bool gq_on = p2.qg.bits != 0;
  QC cq = cg1;
  uint64_t offq = 0;
  if (gq_on) {
    cq = make_qc(p2.qg.bits, __ldg(p2.qg.ib));
    offq = site_offset(p2.qg);
  }
  const uint64_t off2 = site_offset(p.qg2), off1 = site_offset(p.qg1);
  uint32_t a1 = 0, a2 = 0, b1 = 0, b2 = 0;
  float amx = -INFINITY, amn = INFINITY, bmx = -INFINITY, bmn = INFINITY;
  const bool mm2 = p.qg2.minmax != 0, mm1 = p.qg1.minmax != 0;
  Acc<4> acc;
  acc.zero();
  const uint64_t tile = blockIdx.x;   // exactly one tile per CTA
  const uint32_t rg = (uint32_t)(tile / p.t.chunks), chk = (uint32_t)(tile % p.t.chunks);
  const uint32_t v = chk * kThreads + threadIdx.x;
  const bool active = v < p.t.n_vec;
  const int c0 = active ? (int)((4ull * v) % (uint64_t)C) : 0;
  const uint32_t r0 = rg * p.t.rows_per_group, r1 = min(r0 + p.t.rows_per_group, (uint32_t)p.t.n_outer);   // rows: 32-bit (make_tiling)
  if (active) {
    const float4 u2v = site_noise(p.qg2, v, off2), u1v = site_noise(p.qg1, v, off1);
    const float u2[4] = {u2v.x, u2v.y, u2v.z, u2v.w}, u1[4] = {u1v.x, u1v.y, u1v.z, u1v.w};
    float g[4], b[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      g[j] = __ldg(p.gq + c0 + j);
      b[j] = __ldg(p.bq + c0 + j);
    }
    for (uint32_t r = r0; r < r1; r += kRows) {
      float4 gv[kRows], ov[kRows];
      uint32_t w2[kRows], w1[kRows];
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r + i < r1) {
          const size_t idx = 4 * (size_t)((r + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          gv[i] = __ldcs(reinterpret_cast<const float4*>(p.g + idx));
          w2[i] = __ldcs(reinterpret_cast<const uint32_t*>(p.k2 + idx));
          w1[i] = __ldcs(reinterpret_cast<const uint32_t*>(p.k1 + idx));
          if (p.relu == 2) ov[i] = __ldcs(reinterpret_cast<const float4*>(p.out + idx));
        }
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r + kRows + i < r1) {
          const size_t idx = 4 * (size_t)((r + kRows + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          prefetch_l1(p.g + idx);
          prefetch_l1(p.k2 + idx);
          prefetch_l1(p.k1 + idx);
          if (p.relu == 2) prefetch_l1(p.out + idx);
        }
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        if (r + i < r1) {
          const size_t idx = 4 * (size_t)((r + i) * p.t.n_vec + v);   // element / 4 fits 32 bits
          int k2[4], k1[4];
          unpack4(w2[i], k2);
          unpack4(w1[i], k1);
          const float gin[4] = {gv[i].x, gv[i].y, gv[i].z, gv[i].w};
          const float oin[4] = {ov[i].x, ov[i].y, ov[i].z, ov[i].w};
          float gm[4], kq1[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float gj = gin[j];
            if (p.relu == 1) {
              const float y2 = __fadd_rn(__fmul_rn(__int2float_rn(k2[j]) * c2.inv_m, g[j]), b[j]);
              if (!(y2 > 0.0f)) gj = 0.0f;
            } else if (p.relu == 2) {
              if (!(oin[j] > 0.0f)) gj = 0.0f;
            }
            gm[j] = gj;
            const float kg2 = mm2 ? squant_mm(gj, u2[j], cg2, amx, amn) : squant(gj, u2[j], cg2, a1, a2);   // dfxp:687
            const int kg2i = __float2int_rn(kg2);
            acc.s[0][j] += kg2i;
            acc.s[1][j] += kg2i * k2[j];
            const float dx2 = __fmul_rn(kg2 * cg2.inv_m, g[j]);                  // dfxp:691
            kq1[j] = mm1 ? squant_mm(dx2, u1[j], cg1, bmx, bmn) : squant(dx2, u1[j], cg1, b1, b2);         // dfxp:621
            const int kg1i = __float2int_rn(kq1[j]);
            acc.s[2][j] += kg1i;
            acc.s[3][j] += kg1i * k1[j];
          }
          if (p.d_add) *reinterpret_cast<float4*>(p.d_add + idx) = make_float4(gm[0], gm[1], gm[2], gm[3]);
          s_save[(r + i - r0) * kThreads + threadIdx.x] = make_uint2(pack4(kq1), w1[i]);
        }
    }
  }
  flush_block(acc, p.sums, C, s_acc);
  const size_t numel = p.t.n_outer * p.t.n_inner;
  if (mm2) mm_to_counts(cg2, amx, amn, a1, a2);
  if (mm1) mm_to_counts(cg1, bmx, bmn, b1, b2);
  publish_counters(p.qg2.counters, a1, a2, numel, s_red);
  publish_counters(p.qg1.counters, b1, b2, numel, s_red);

  // ---- grid-wide barrier: every CTA's sums are in global memory before anyone reads them ----
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(q.bar, 1ull);
    long long t0 = 0;
    uint32_t spins = 0;
    while (*reinterpret_cast<volatile unsigned long long*>(q.bar) < (unsigned long long)gridDim.x) {
      if ((++spins & 0xff) == 0) {
        const long long now = clock64();
        if (t0 == 0) t0 = now;
        if (now - t0 > 4000000000ll) {  // ~2 s: never hang the GPU on a protocol bug
          atomicExch(&g_bn_error, 1);
          break;
        }
      }
    }
    __threadfence();
  }
  __syncthreads();

  // ---- pass 2 from shared memory ----
  float* s_par = reinterpret_cast<float*>(s_dyn);
  const DivN n = make_divn((unsigned long long)(p.t.n_outer * (p.t.n_inner / C)));
  for (int ch = threadIdx.x; ch < C; ch += kThreads) {
    float mean, var;
    moments(p2.fsums, C, ch, n, c1.inv_m, mean, var);
    const float den = __fsqrt_rn(__fadd_rn(var, p2.eps));
    const double sg = (double)__ldcg(p.sums + 2 * C + ch) * (double)cg1.inv_m;
    const double sgx = (double)__ldcg(p.sums + 3 * C + ch) * (double)cg1.inv_m * (double)c1.inv_m;
    const double mg = div_n(sg, n);
    const double mgx = div_n(__ddiv_rn(__dsub_rn(sgx, __dmul_rn((double)mean, sg)), (double)den), n);
    s_par[ch] = mean;
    s_par[C + ch] = den;
    s_par[2 * C + ch] = (float)mg;
    s_par[3 * C + ch] = (float)mgx;
  }
  __syncthreads();
  uint32_t n1 = 0, n2 = 0;
  float mx = -INFINITY, mn = INFINITY;
  const bool mmq = p2.qg.minmax != 0;
  if (active) {
    float mean[4], den[4], mg[4], mgx[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      mean[j] = s_par[c0 + j];
      den[j] = s_par[C + c0 + j];
      mg[j] = s_par[2 * C + c0 + j];
      mgx[j] = s_par[3 * C + c0 + j];
    }
    float rden[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) rden[j] = __frcp_rn(den[j]);
    float uq[4] = {0.f, 0.f, 0.f, 0.f};
    if (gq_on) {
      const float4 t = site_noise(p2.qg, v, offq);
      uq[0] = t.x; uq[1] = t.y; uq[2] = t.z; uq[3] = t.w;
    }
    for (size_t r = r0; r < r1; ++r) {
      const size_t idx = r * p.t.n_inner + 4 * (size_t)v;
      const uint2 sv = s_save[(r - r0) * kThreads + threadIdx.x];
      int kg[4], k1[4];
      unpack4(sv.x, kg);
      unpack4(sv.y, k1);
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float gqv = __int2float_rn(kg[j]) * cg1.inv_m;
        const float xhat = fdiv_by(__fsub_rn(__int2float_rn(k1[j]) * c1.inv_m, mean[j]), den[j], rden[j]);
        o[j] = fdiv_by(__fsub_rn(__fsub_rn(gqv, mg[j]), __fmul_rn(xhat, mgx[j])), den[j], rden[j]);
      }
      if (p2.dx) *reinterpret_cast<float4*>(p2.dx + idx) = make_float4(o[0], o[1], o[2], o[3]);
      if (gq_on) {
        float kq[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) kq[j] = mmq ? squant_mm(o[j], uq[j], cq, mx, mn) : squant(o[j], uq[j], cq, n1, n2);
        *reinterpret_cast<uint32_t*>(p2.g_mant + idx) = pack4(kq);
      }
    }
  }
  if (gq_on) {
    if (mmq) mm_to_counts(cq, mx, mn, n1, n2);
    publish_counters(p2.qg.counters, n1, n2, numel, s_red);
  }
}

// ---- host helpers ----------------------------------------------------------------------------
// Resident CTAs per SM of a kernel with `smem` dynamic bytes (cached per kernel and device).
template <typename K>
int ctas_per_sm(K kernel, size_t smem) {
  // keyed by the kernel's address: instantiations of one kernel template share their function-pointer TYPE
  struct Entry {
    const void* fn;
    int n;
  };
  static Entry cache[16][4] = {};
  const int dev = device_info().device;
  if (dev < 0 || dev >= 16) return 1;
  const void* key = reinterpret_cast<const void*>(kernel);
  for (Entry& e : cache[dev]) {
    if (e.fn == key) return e.n;
    if (e.fn == nullptr) {
      int n = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, kThreads, smem) != cudaSuccess || n < 1) n = 1;
      e.n = n;
      e.fn = key;
      return n;
    }
  }
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, kThreads, smem) != cudaSuccess || n < 1) n = 1;
  return n;
}

// Tiles = (256-float4 column chunks) x (groups of batch rows).  These tensors are small (a few MB): what matters is
// that the launch is ONE balanced wave of resident CTAs — a 1.15-wave grid costs two CTA latencies.  So the row
// groups are sized to give at most `occ * SMs` tiles; only tensors with more column chunks than that run a
// persistent multi-tile loop.
int make_tiling(Tiling& t, size_t n_outer, size_t n_inner, int C, unsigned& grid, int occ) {
  if (C <= 0 || (C & 3) || n_inner % (size_t)C) return LBT_EUNSUPPORTED;
  if (n_inner / 4 >= 0xffffffffull) return LBT_EUNSUPPORTED;
  if (n_outer * n_inner >= (1ull << 33)) return LBT_EUNSUPPORTED;  // keeps every thread's 32-bit partial sums exact
  const DeviceInfo& di = device_info();
  t.n_outer = n_outer;
  t.n_inner = n_inner;
  t.C = C;
  t.n_vec = (uint32_t)(n_inner / 4);
  t.chunks = (t.n_vec + kThreads - 1) / kThreads;
  const uint64_t cap = (uint64_t)di.sm_count * (uint64_t)(occ < 1 ? 1 : occ);
  // pick the number of row groups g that minimises (waves of resident CTAs) x (rows per CTA + fixed cost per wave)
  uint64_t best_g = 1, best_cost = ~0ull;
  const uint64_t gmax = n_outer < 4096 ? n_outer : 4096;
  for (uint64_t g = 1; g <= gmax; ++g) {
    const uint64_t rows = (n_outer + g - 1) / g;
    if (rows > 4096) continue;              // 32-bit per-thread partial sums: <= 4096 rows x 2^14 per tile visit
    const uint64_t gg = (n_outer + rows - 1) / rows;
    const uint64_t waves = (t.chunks * gg + cap - 1) / cap;
    const uint64_t cost = waves * (rows + 3);
    if (cost < best_cost) {
      best_cost = cost;
      best_g = gg;
    }
  }
  uint64_t rpg = (n_outer + best_g - 1) / best_g;
  const uint64_t groups = (n_outer + rpg - 1) / rpg;
  t.rows_per_group = (uint32_t)rpg;
  t.total_tiles = (uint64_t)t.chunks * groups;
  const int cgroups = C >> 2;
  t.fixed_channels = (cgroups <= kThreads && (kThreads % cgroups) == 0) ? 1 : 0;
  grid = (unsigned)(t.total_tiles < cap ? t.total_tiles : cap);
  return LBT_OK;
}

QSite make_site(int bits, const int32_t* ib, const float* noise, uint64_t seed, uint64_t offset, const uint64_t* dev_step,
                uint64_t* counters, int minmax = 0) {
  QSite s;
  s.minmax = minmax;
  s.bits = bits;
  s.ib = ib;
  s.noise = noise;
  s.seed = seed;
  s.offset = offset;
  s.dev_step = dev_step;
  s.counters = reinterpret_cast<unsigned long long*>(counters);
  return s;
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline bool al4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3) == 0; }

template <typename K>
int set_smem(K kernel, size_t bytes) {
  if (bytes > 40 * 1024) {   // the 48 KB default covers static + dynamic shared memory: opt in with some margin
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(bn)");
      return LBT_ECUDA;
    }
  }
  return LBT_OK;
}

}  // namespace
}  // namespace lbt

using namespace lbt;

extern "C" int lbt_bn_fwd_quant_stats(const float* x, size_t n_outer, size_t n_inner, int C, int bits, const int32_t* ib,
                                      const float* noise, uint64_t seed, uint64_t offset, const uint64_t* dev_step,
                                      int8_t* k1, int64_t* sums, uint64_t* counters, int stats_minmax, void* stream) {
  if (!x || !ib || !k1 || !sums) return LBT_EINVAL;
  if (bits < 2 || bits > 8) return LBT_EUNSUPPORTED;
  if (n_outer == 0 || n_inner == 0) return LBT_OK;
  if (!al16(x) || !al4(k1) || (noise && !al16(noise))) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  Fwd1Params p{};
  unsigned grid;
  int rc = make_tiling(p.t, n_outer, n_inner, C, grid, ctas_per_sm(bn_fwd1_kernel, (size_t)2 * C * 8));
  if (rc) return rc;
  p.x = x;
  p.q = make_site(bits, ib, noise, seed, offset, dev_step, counters, stats_minmax);
  p.k1 = k1;
  p.sums = reinterpret_cast<long long*>(sums);
  const size_t smem = (size_t)2 * C * 8;
  if ((rc = set_smem(bn_fwd1_kernel, smem))) return rc;
  launch_pdl(bn_fwd1_kernel, grid, kThreads, smem, reinterpret_cast<cudaStream_t>(stream), p);
  return check_launch("lbt_bn_fwd_quant_stats");
}

using Fwd2Kernel = void (*)(const Fwd2Params);
template <bool RUN>
Fwd2Kernel fwd2_kernel(bool mm, bool q4) {
  return q4 ? (mm ? bn_fwd2_kernel<true, true, RUN> : bn_fwd2_kernel<false, true, RUN>)
            : (mm ? bn_fwd2_kernel<true, false, RUN> : bn_fwd2_kernel<false, false, RUN>);
}

// running: eval mode — run_mean / run_var are the statistics (read only), `sums` and k2 are not used / optional
static int bn_fwd_apply_run(const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1, const int32_t* ib1,
                            const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                            uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                            const float* gamma_q, const float* beta_q, const float* add, int relu, int8_t* k2,
                            float* out, float* batch_mean, float* batch_var, float* run_mean, float* run_var,
                            double momentum, int stats_minmax, const lbt_qsite* q_next, void* next_mant, int next_kind,
                            const lbt_qsite* q_next2, void* next_mant2, int next_kind2, void* stream, bool running = false) {
  if (!k1 || !ib1 || !ib2 || !gamma_q || !beta_q) return LBT_EINVAL;
  if (running ? (!run_mean || !run_var || C <= 0 || (C & 3)) : (!sums || !k2)) return LBT_EINVAL;
  if (q_next2) {
    if (!q_next || !next_mant2 || !q_next2->ib || !al4(next_mant2) || (q_next2->noise && !al16(q_next2->noise))) return LBT_EINVAL;
    if (next_kind2 == LBT_MANT_U8 ? (q_next2->bits < 2 || q_next2->bits > 9 || !relu)
                                  : (next_kind2 != LBT_MANT_S8 || q_next2->bits < 2 || q_next2->bits > 8))
      return LBT_EUNSUPPORTED;
  }
  if (!out && !q_next) return LBT_EINVAL;
  if (bits1 < 2 || bits1 > 8 || bits2 < 2 || bits2 > 8) return LBT_EUNSUPPORTED;
  if (q_next) {
    if (!next_mant || !q_next->ib || !al4(next_mant) || (q_next->noise && !al16(q_next->noise))) return LBT_EINVAL;
    // u8 holds a 9-bit mantissa only when the tensor is non-negative, i.e. the ReLU is fused here
    if (next_kind == LBT_MANT_U8 ? (q_next->bits < 2 || q_next->bits > 9 || !relu)
                                 : (next_kind != LBT_MANT_S8 || q_next->bits < 2 || q_next->bits > 8))
      return LBT_EUNSUPPORTED;
  }
  if ((run_mean == nullptr) != (run_var == nullptr)) return LBT_EINVAL;
  if (n_outer == 0 || n_inner == 0) return LBT_OK;
  if (!al4(k1) || (k2 && !al4(k2)) || (out && !al16(out)) || (add && !al16(add)) || (noise2 && !al16(noise2))) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  Fwd2Params p{};
  unsigned grid;
  // one statistics flavour per launch: min/max only when EVERY site of the launch asked for it (exact counts are always valid)
  const bool mm = stats_minmax && (!q_next || q_next->stats_minmax) && (!q_next2 || q_next2->stats_minmax);
  const Fwd2Kernel kern = running ? fwd2_kernel<true>(mm, q_next2 != nullptr) : fwd2_kernel<false>(mm, q_next2 != nullptr);
  int rc = make_tiling(p.t, n_outer, n_inner, C, grid, ctas_per_sm(kern, (size_t)4 * C * 4));
  if (rc) return rc;
  p.k1 = k1;
  p.bits1 = bits1;
  p.ib1 = ib1;
  p.sums = reinterpret_cast<const long long*>(sums);
  p.eps = eps;
  p.q2 = make_site(bits2, ib2, noise2, seed, offset2, dev_step, counters2, stats_minmax);
  p.gq = gamma_q;
  p.bq = beta_q;
  p.add = add;
  p.relu = relu;
  p.k2 = k2;
  p.out = out;
  p.batch_mean = batch_mean;
  p.batch_var = batch_var;
  p.run_mean = run_mean;
  p.run_var = run_var;
  p.momentum = (float)momentum;
  p.one_minus_momentum = (float)(1.0 - momentum);   // dfxp:606: `(1-momentum)` is evaluated in Python (double), THEN becomes an fp32 constant
  p.q3 = site_from_abi(q_next);
  p.next_mant = reinterpret_cast<uint8_t*>(next_mant);
  p.q4 = site_from_abi(q_next2);
  p.next_mant2 = reinterpret_cast<uint8_t*>(next_mant2);
  const size_t smem = (size_t)4 * C * 4;
  if ((rc = set_smem(kern, smem))) return rc;
  launch_pdl(kern, grid, kThreads, smem, reinterpret_cast<cudaStream_t>(stream), p);
  return check_launch(running ? "lbt_bn_fwd_apply_running" : "lbt_bn_fwd_apply");
}

extern "C" int lbt_bn_fwd_apply(const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1, const int32_t* ib1,
                                const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                                uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                                const float* gamma_q, const float* beta_q, const float* add, int relu, int8_t* k2,
                                float* out, float* batch_mean, float* batch_var, float* run_mean, float* run_var,
                                double momentum, int stats_minmax, const lbt_qsite* q_next, void* next_mant, int next_kind,
                                void* stream) {
  return bn_fwd_apply_run(k1, n_outer, n_inner, C, bits1, ib1, sums, eps, bits2, ib2, noise2, seed, offset2, dev_step, counters2,
                          gamma_q, beta_q, add, relu, k2, out, batch_mean, batch_var, run_mean, run_var, momentum, stats_minmax,
                          q_next, next_mant, next_kind, nullptr, nullptr, 0, stream);
}

extern "C" int lbt_bn_fwd_apply2(const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1, const int32_t* ib1,
                                 const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                                 uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                                 const float* gamma_q, const float* beta_q, const float* add, int relu, int8_t* k2,
                                 float* out, float* batch_mean, float* batch_var, float* run_mean, float* run_var,
                                 double momentum, int stats_minmax, const lbt_qsite* q_next, void* next_mant, int next_kind,
                                 const lbt_qsite* q_next2, void* next_mant2, int next_kind2, void* stream) {
  if (!q_next2) return LBT_EINVAL;
  return bn_fwd_apply_run(k1, n_outer, n_inner, C, bits1, ib1, sums, eps, bits2, ib2, noise2, seed, offset2, dev_step, counters2,
                          gamma_q, beta_q, add, relu, k2, out, batch_mean, batch_var, run_mean, run_var, momentum, stats_minmax,
                          q_next, next_mant, next_kind, q_next2, next_mant2, next_kind2, stream);
}

extern "C" int lbt_bn_fwd_apply_running(const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1, const int32_t* ib1,
                                        const float* run_mean, const float* run_var, float eps, int bits2, const int32_t* ib2,
                                        const float* noise2, uint64_t seed, uint64_t offset2, const uint64_t* dev_step,
                                        uint64_t* counters2, const float* gamma_q, const float* beta_q, const float* add, int relu,
                                        int8_t* k2, float* out, int stats_minmax, const lbt_qsite* q_next, void* next_mant,
                                        int next_kind, const lbt_qsite* q_next2, void* next_mant2, int next_kind2, void* stream) {
  // the kernel only reads the running statistics (the Fwd2Params slots are shared with the training update)
  return bn_fwd_apply_run(k1, n_outer, n_inner, C, bits1, ib1, nullptr, eps, bits2, ib2, noise2, seed, offset2, dev_step, counters2,
                          gamma_q, beta_q, add, relu, k2, out, nullptr, nullptr, const_cast<float*>(run_mean),
                          const_cast<float*>(run_var), 0.0, stats_minmax, q_next, next_mant, next_kind, q_next2, next_mant2,
                          next_kind2, stream, true);
}

// running: eval mode, as in bn_fwd_apply_run
static int bn_fwd_apply_pooled_run(const int8_t* k1, size_t n_outer, int H, int W, int C, int bits1, const int32_t* ib1,
                                   const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                                   uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                                   const float* gamma_q, const float* beta_q, int relu, int8_t* k2, float* run_mean,
                                   float* run_var, double momentum, int stats_minmax, int k, int s, int pad_top, int pad_left,
                                   int POH, int POW, float* pooled, uint8_t* pidx, const lbt_qsite* q_next, void* next_mant,
                                   int next_kind, void* stream, bool running = false) {
  if (!k1 || !ib1 || !ib2 || !gamma_q || !beta_q || !pooled || !pidx) return LBT_EINVAL;
  if (running ? (!run_mean || !run_var || C <= 0 || (C & 3)) : (!sums || !k2)) return LBT_EINVAL;
  if (q_next) {
    if (!next_mant || !q_next->ib || !al4(next_mant) || (q_next->noise && !al16(q_next->noise))) return LBT_EINVAL;
    // u8 holds a 9-bit mantissa only when the tensor is non-negative, i.e. the ReLU is fused here
    if (next_kind == LBT_MANT_U8 ? (q_next->bits < 2 || q_next->bits > 9 || !relu)
                                 : (next_kind != LBT_MANT_S8 || q_next->bits < 2 || q_next->bits > 8))
      return LBT_EUNSUPPORTED;
  }
  if (H <= 0 || W <= 0 || C <= 0 || POH <= 0 || POW <= 0 || k <= 0 || s <= 0 || pad_top < 0 || pad_left < 0) return LBT_EINVAL;
  if ((run_mean == nullptr) != (run_var == nullptr)) return LBT_EINVAL;
  if (bits1 < 2 || bits1 > 8 || bits2 < 2 || bits2 > 8) return LBT_EUNSUPPORTED;
  // the ImageNet stem's shape class: 3x3 / 2 windows that start on the even pixels, 64 channels
  if (C != 64 || k != 3 || s != 2 || pad_top != 0 || pad_left != 0 || POH != (H + 1) / 2 || POW != (W + 1) / 2) return LBT_EUNSUPPORTED;
  if (n_outer == 0) return LBT_OK;
  if ((uint64_t)n_outer * H * W * 16 >= (1ull << 31)) return LBT_EUNSUPPORTED;   // 32-bit word indices
  if (!al4(k1) || (k2 && !al4(k2)) || !al16(pooled) || !al4(pidx) || (noise2 && !al16(noise2))) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  const DeviceInfo& di = device_info();
  Fwd2PoolParams p{};
  p.k1 = k1;
  p.bits1 = bits1;
  p.ib1 = ib1;
  p.sums = reinterpret_cast<const long long*>(sums);
  p.eps = eps;
  p.q2 = make_site(bits2, ib2, noise2, seed, offset2, dev_step, counters2, stats_minmax);
  p.gq = gamma_q;
  p.bq = beta_q;
  p.relu = relu;
  p.k2 = k2;
  p.run_mean = run_mean;
  p.run_var = run_var;
  p.momentum = (float)momentum;
  p.one_minus_momentum = (float)(1.0 - momentum);
  p.pooled = pooled;
  p.pidx = pidx;
  p.q3 = site_from_abi(q_next);
  p.next_mant = reinterpret_cast<uint8_t*>(next_mant);
  p.N = (uint32_t)n_outer;
  p.H = (uint32_t)H;
  p.W = (uint32_t)W;
  p.POH = (uint32_t)POH;
  p.POW = (uint32_t)POW;
  p.tiles_x = (uint32_t)((W + kPoolTW - 1) / kPoolTW);
  p.tiles_img = p.tiles_x * (uint32_t)((H + kPoolTH - 1) / kPoolTH);
  // row groups: about one wave of CTAs (one 512-thread CTA per SM), at least 4 rows per group
  uint64_t groups = ((uint64_t)di.sm_count * 2 + p.tiles_img / 2) / p.tiles_img;
  if (groups < 1) groups = 1;
  if (groups > (n_outer + 3) / 4) groups = (n_outer + 3) / 4;
  p.rows_per_group = (uint32_t)((n_outer + groups - 1) / groups);
  const uint64_t total = (uint64_t)p.tiles_img * ((n_outer + p.rows_per_group - 1) / p.rows_per_group);
  if (total >= (1ull << 31)) return LBT_EUNSUPPORTED;
  p.total_tiles = (uint32_t)total;
  const size_t smem = (size_t)2 * (kPoolTH + 1) * (kPoolTW + 1) * kPoolCG * sizeof(float4);
  const unsigned grid = (unsigned)total;
  // one statistics flavour per launch (exact counts are always valid)
  const bool mm = stats_minmax && (!q_next || q_next->stats_minmax);
  void (*kern)(const Fwd2PoolParams) = running ? (mm ? bn_fwd2_pool_kernel<true, true> : bn_fwd2_pool_kernel<false, true>)
                                               : (mm ? bn_fwd2_pool_kernel<true, false> : bn_fwd2_pool_kernel<false, false>);
  int rc;
  if ((rc = set_smem(kern, smem))) return rc;
  launch_pdl(kern, grid, kPoolThreads, smem, reinterpret_cast<cudaStream_t>(stream), p);
  return check_launch(running ? "lbt_bn_fwd_apply_running_pooled" : "lbt_bn_fwd_apply_pooled");
}

extern "C" int lbt_bn_fwd_apply_pooled(const int8_t* k1, size_t n_outer, int H, int W, int C, int bits1, const int32_t* ib1,
                                       const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                                       uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                                       const float* gamma_q, const float* beta_q, int relu, int8_t* k2, float* run_mean,
                                       float* run_var, double momentum, int stats_minmax, int k, int s, int pad_top, int pad_left,
                                       int POH, int POW, float* pooled, uint8_t* pidx, const lbt_qsite* q_next, void* next_mant,
                                       int next_kind, void* stream) {
  return bn_fwd_apply_pooled_run(k1, n_outer, H, W, C, bits1, ib1, sums, eps, bits2, ib2, noise2, seed, offset2, dev_step,
                                 counters2, gamma_q, beta_q, relu, k2, run_mean, run_var, momentum, stats_minmax, k, s, pad_top,
                                 pad_left, POH, POW, pooled, pidx, q_next, next_mant, next_kind, stream);
}

extern "C" int lbt_bn_fwd_apply_running_pooled(const int8_t* k1, size_t n_outer, int H, int W, int C, int bits1, const int32_t* ib1,
                                               const float* run_mean, const float* run_var, float eps, int bits2, const int32_t* ib2,
                                               const float* noise2, uint64_t seed, uint64_t offset2, const uint64_t* dev_step,
                                               uint64_t* counters2, const float* gamma_q, const float* beta_q, int relu, int8_t* k2,
                                               int stats_minmax, int k, int s, int pad_top, int pad_left, int POH, int POW,
                                               float* pooled, uint8_t* pidx, const lbt_qsite* q_next, void* next_mant, int next_kind,
                                               void* stream) {
  // the kernel only reads the running statistics (the Fwd2PoolParams slots are shared with the training update)
  return bn_fwd_apply_pooled_run(k1, n_outer, H, W, C, bits1, ib1, nullptr, eps, bits2, ib2, noise2, seed, offset2, dev_step,
                                 counters2, gamma_q, beta_q, relu, k2, const_cast<float*>(run_mean), const_cast<float*>(run_var),
                                 0.0, stats_minmax, k, s, pad_top, pad_left, POH, POW, pooled, pidx, q_next, next_mant, next_kind,
                                 stream, true);
}

static int bn_bwd1_run(const float* g, const float* out, int relu, const int8_t* k2, const int8_t* k1,
                       size_t n_outer, size_t n_inner, int C, int bits2, const int32_t* ib2,
                       const float* gamma_q, const float* beta_q, int bits_g2, const int32_t* ib_g2,
                       const float* noise_g2, uint64_t offset_g2, uint64_t* counters_g2, int bits_g1,
                       const int32_t* ib_g1, const float* noise_g1, uint64_t offset_g1,
                       uint64_t* counters_g1, uint64_t seed, const uint64_t* dev_step, float* d_add,
                       void* kg1, int64_t* sums, int stats_minmax, int kg1_kind, const lbt_pool_geom* pool, void* stream) {
  if (!g || !k2 || !k1 || !ib2 || !gamma_q || !beta_q || !ib_g2 || !ib_g1 || !kg1 || !sums) return LBT_EINVAL;
  if (pool) {
    if (!pool->idx || pool->H <= 0 || pool->W <= 0 || pool->k <= 0 || pool->s <= 0 || pool->OH <= 0 || pool->OW <= 0 ||
        pool->pad_top < 0 || pool->pad_left < 0)
      return LBT_EINVAL;
    // <= 2 x 2 windows per pixel, 4 channels per thread, no shortcut sum / saved-output mask in front of the pool
    if (pool->k > 2 * pool->s || pool->k > 15 || (C & 3) || relu == 2 || d_add) return LBT_EUNSUPPORTED;
    if (n_inner != (size_t)pool->H * pool->W * C) return LBT_EINVAL;
    if ((size_t)pool->OH * pool->OW * C >= (1ull << 31) || (reinterpret_cast<uintptr_t>(pool->idx) & 3)) return LBT_EUNSUPPORTED;
  }
  if (relu < 0 || relu > 2 || (relu == 2 && !out)) return LBT_EINVAL;
  if (kg1_kind != LBT_MANT_S8 && kg1_kind != LBT_MANT_S16) return LBT_EINVAL;
  const bool wide = kg1_kind == LBT_MANT_S16;
  const int gmax = wide ? 16 : 8;
  // the gradient quantisers take up to 16 bits with s16 storage; s8 storage needs BOTH <= 8 (32-bit partial sums)
  if (bits2 < 2 || bits2 > 8 || bits_g2 < 2 || bits_g2 > gmax || bits_g1 < 2 || bits_g1 > gmax) return LBT_EUNSUPPORTED;
  if (n_outer == 0 || n_inner == 0) return LBT_OK;
  if (!al16(g) || !al4(k2) || !al4(k1) || !(wide ? (reinterpret_cast<uintptr_t>(kg1) & 7) == 0 : al4(kg1)) || (out && !al16(out)) ||
      (d_add && !al16(d_add)) || (noise_g2 && !al16(noise_g2)) || (noise_g1 && !al16(noise_g1)))
    return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  Bwd1Params p{};
  unsigned grid;
  void (*kern)(const Bwd1Params) = nullptr;
  {
    const bool mm = stats_minmax != 0;
#define LBT_BWD1(W, M)                                                                                     \
  (relu == 0 ? bn_bwd1_kernel<W, M, 0> : (relu == 1 ? bn_bwd1_kernel<W, M, 1> : bn_bwd1_kernel<W, M, 2>))
#define LBT_BWD1P(W, M) (relu == 0 ? bn_bwd1_kernel<W, M, 0, true> : bn_bwd1_kernel<W, M, 1, true>)
    if (pool) kern = wide ? (mm ? LBT_BWD1P(true, true) : LBT_BWD1P(true, false)) : (mm ? LBT_BWD1P(false, true) : LBT_BWD1P(false, false));
    else kern = wide ? (mm ? LBT_BWD1(true, true) : LBT_BWD1(true, false)) : (mm ? LBT_BWD1(false, true) : LBT_BWD1(false, false));
#undef LBT_BWD1
#undef LBT_BWD1P
  }
  int rc = make_tiling(p.t, n_outer, n_inner, C, grid, ctas_per_sm(kern, (size_t)4 * C * 8));
  if (rc) return rc;
  p.g = g;
  p.out = out;
  p.relu = relu;
  p.k2 = k2;
  p.k1 = k1;
  p.bits2 = bits2;
  p.ib2 = ib2;
  p.gq = gamma_q;
  p.bq = beta_q;
  p.qg2 = make_site(bits_g2, ib_g2, noise_g2, seed, offset_g2, dev_step, counters_g2, stats_minmax);
  p.qg1 = make_site(bits_g1, ib_g1, noise_g1, seed, offset_g1, dev_step, counters_g1, stats_minmax);
  p.d_add = d_add;
  p.kg1 = kg1;
  p.sums = reinterpret_cast<long long*>(sums);
  if (pool) {
    p.pidx = pool->idx;
    p.pW = pool->W;
    p.pk = pool->k;
    p.ps = pool->s;
    p.ppt = pool->pad_top;
    p.ppl = pool->pad_left;
    p.pOH = pool->OH;
    p.pOW = pool->OW;
    p.d_c4 = make_fastdiv((uint32_t)C / 4);
    p.d_pW = make_fastdiv((uint32_t)pool->W);
    p.d_ps = make_fastdiv((uint32_t)pool->s);
  }
  const size_t smem = (size_t)4 * C * 8;
  if ((rc = set_smem(kern, smem))) return rc;
  launch_pdl(kern, grid, kThreads, smem, reinterpret_cast<cudaStream_t>(stream), p);
  return check_launch("lbt_bn_bwd_quant_stats");
}

extern "C" int lbt_bn_bwd_quant_stats(const float* g, const float* out, int relu, const int8_t* k2, const int8_t* k1,
                                      size_t n_outer, size_t n_inner, int C, int bits2, const int32_t* ib2,
                                      const float* gamma_q, const float* beta_q, int bits_g2, const int32_t* ib_g2,
                                      const float* noise_g2, uint64_t offset_g2, uint64_t* counters_g2, int bits_g1,
                                      const int32_t* ib_g1, const float* noise_g1, uint64_t offset_g1,
                                      uint64_t* counters_g1, uint64_t seed, const uint64_t* dev_step, float* d_add,
                                      void* kg1, int64_t* sums, int stats_minmax, int kg1_kind, void* stream) {
  return bn_bwd1_run(g, out, relu, k2, k1, n_outer, n_inner, C, bits2, ib2, gamma_q, beta_q, bits_g2, ib_g2, noise_g2, offset_g2,
                     counters_g2, bits_g1, ib_g1, noise_g1, offset_g1, counters_g1, seed, dev_step, d_add, kg1, sums, stats_minmax,
                     kg1_kind, nullptr, stream);
}

extern "C" int lbt_bn_bwd_quant_stats_pooled(const float* g_pooled, const lbt_pool_geom* pool, int relu, const int8_t* k2,
                                             const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits2, const int32_t* ib2,
                                             const float* gamma_q, const float* beta_q, int bits_g2, const int32_t* ib_g2,
                                             const float* noise_g2, uint64_t offset_g2, uint64_t* counters_g2, int bits_g1,
                                             const int32_t* ib_g1, const float* noise_g1, uint64_t offset_g1,
                                             uint64_t* counters_g1, uint64_t seed, const uint64_t* dev_step, void* kg1,
                                             int64_t* sums, int stats_minmax, int kg1_kind, void* stream) {
  if (!pool) return LBT_EINVAL;
  return bn_bwd1_run(g_pooled, nullptr, relu, k2, k1, n_outer, n_inner, C, bits2, ib2, gamma_q, beta_q, bits_g2, ib_g2, noise_g2,
                     offset_g2, counters_g2, bits_g1, ib_g1, noise_g1, offset_g1, counters_g1, seed, dev_step, nullptr, kg1, sums,
                     stats_minmax, kg1_kind, pool, stream);
}

extern "C" int lbt_bn_bwd_apply(const void* kg1, const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1,
                                const int32_t* ib1, const int64_t* fwd_sums, float eps, int bits_g1, const int32_t* ib_g1,
                                const int64_t* bwd_sums, float* dx, const lbt_qsite* q_grad, int8_t* g_mant, int kg1_kind,
                                uint8_t* g_mant_lo, void* stream) {
  if (!kg1 || !k1 || !ib1 || !fwd_sums || !ib_g1 || !bwd_sums) return LBT_EINVAL;
  if (!dx && !q_grad) return LBT_EINVAL;
  if (kg1_kind != LBT_MANT_S8 && kg1_kind != LBT_MANT_S16) return LBT_EINVAL;
  const bool wide = kg1_kind == LBT_MANT_S16;
  if (bits1 < 2 || bits1 > 8 || bits_g1 < 2 || bits_g1 > (wide ? 16 : 8)) return LBT_EUNSUPPORTED;
  if (q_grad) {
    if (!g_mant || !q_grad->ib || !al4(g_mant) || (q_grad->noise && !al16(q_grad->noise))) return LBT_EINVAL;
    if (q_grad->bits < 2 || q_grad->bits > 16) return LBT_EUNSUPPORTED;
    if (q_grad->bits > 8 && (!g_mant_lo || !al4(g_mant_lo))) return LBT_EINVAL;   // two byte planes: k = 256 * hi + lo
  }
  if (n_outer == 0 || n_inner == 0) return LBT_OK;
  if (!(wide ? (reinterpret_cast<uintptr_t>(kg1) & 7) == 0 : al4(kg1)) || !al4(k1) || (dx && !al16(dx))) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  Bwd2Params p{};
  unsigned grid;
  const bool mm = q_grad != nullptr && q_grad->stats_minmax != 0;
  void (*kern)(const Bwd2Params) = wide ? (mm ? bn_bwd2_kernel<true, true> : bn_bwd2_kernel<true, false>)
                                        : (mm ? bn_bwd2_kernel<false, true> : bn_bwd2_kernel<false, false>);
  int rc = make_tiling(p.t, n_outer, n_inner, C, grid, ctas_per_sm(kern, (size_t)4 * C * 4));
  if (rc) return rc;
  p.kg1 = kg1;
  p.k1 = k1;
  p.bits1 = bits1;
  p.ib1 = ib1;
  p.fsums = reinterpret_cast<const long long*>(fwd_sums);
  p.eps = eps;
  p.bitsg1 = bits_g1;
  p.ibg1 = ib_g1;
  p.bsums = reinterpret_cast<const long long*>(bwd_sums);
  p.dx = dx;
  p.qg = site_from_abi(q_grad);
  p.g_mant = g_mant;
  p.g_mant_lo = g_mant_lo;
  const size_t smem = (size_t)4 * C * 4;
  if ((rc = set_smem(kern, smem))) return rc;
  launch_pdl(kern, grid, kThreads, smem, reinterpret_cast<cudaStream_t>(stream), p);
  return check_launch("lbt_bn_bwd_apply");
}

extern "C" int lbt_bn_bwd_fused(const lbt_bn_bwd_args* a, void* stream) {
  if (!a || !a->g || !a->k2 || !a->k1 || !a->ib2 || !a->gamma_q || !a->beta_q || !a->q_g2.ib || !a->q_g1.ib || !a->bwd_sums ||
      !a->ib1 || !a->fwd_sums || !a->barrier)
    return LBT_EINVAL;
  if (a->relu < 0 || a->relu > 2 || (a->relu == 2 && !a->out)) return LBT_EINVAL;
  if (!a->dx && !a->has_q_grad) return LBT_EINVAL;
  if (a->has_q_grad && (!a->g_mant || !a->q_grad.ib || a->q_grad.bits < 2 || a->q_grad.bits > 8)) return LBT_EINVAL;
  for (int b : {a->bits2, a->q_g2.bits, a->q_g1.bits, a->bits1})
    if (b < 2 || b > 8) return LBT_EUNSUPPORTED;
  if (a->n_outer == 0 || a->n_inner == 0) return LBT_OK;
  if (!al16(a->g) || !al4(a->k2) || !al4(a->k1) || (a->out && !al16(a->out)) || (a->d_add && !al16(a->d_add)) ||
      (a->dx && !al16(a->dx)) || (a->g_mant && !al4(a->g_mant)))
    return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  const int C = a->C;
  BwdFusedParams q{};
  // occupancy with the largest row buffer; the tiling must then be ONE tile per resident CTA with <= kMaxSavedRows rows
  const size_t smem_max = (size_t)4 * C * 8 + (size_t)kMaxSavedRows * kThreads * sizeof(uint2);
  int rc = set_smem(bn_bwd_fused_kernel, smem_max);
  if (rc) return rc;
  unsigned grid;
  rc = make_tiling(q.a.t, a->n_outer, a->n_inner, C, grid, ctas_per_sm(bn_bwd_fused_kernel, smem_max));
  if (rc) return rc;
  if (!q.a.t.fixed_channels || q.a.t.total_tiles != grid || q.a.t.rows_per_group > (uint32_t)kMaxSavedRows) return LBT_EUNSUPPORTED;
  q.b.t = q.a.t;
  q.a.g = a->g;
  q.a.out = a->out;
  q.a.relu = a->relu;
  q.a.k2 = a->k2;
  q.a.k1 = a->k1;
  q.a.bits2 = a->bits2;
  q.a.ib2 = a->ib2;
  q.a.gq = a->gamma_q;
  q.a.bq = a->beta_q;
  q.a.qg2 = site_from_abi(&a->q_g2);
  q.a.qg1 = site_from_abi(&a->q_g1);
  q.a.d_add = a->d_add;
  q.a.kg1 = nullptr;
  q.a.sums = reinterpret_cast<long long*>(a->bwd_sums);
  q.b.bits1 = a->bits1;
  q.b.ib1 = a->ib1;
  q.b.fsums = reinterpret_cast<const long long*>(a->fwd_sums);
  q.b.eps = a->eps;
  q.b.bitsg1 = a->q_g1.bits;
  q.b.ibg1 = a->q_g1.ib;
  q.b.bsums = reinterpret_cast<const long long*>(a->bwd_sums);
  q.b.dx = a->dx;
  q.b.qg = site_from_abi(a->has_q_grad ? &a->q_grad : nullptr);
  q.b.g_mant = a->g_mant;
  q.bar = reinterpret_cast<unsigned long long*>(a->barrier);
  const size_t smem = (size_t)4 * C * 8 + (size_t)q.a.t.rows_per_group * kThreads * sizeof(uint2);
  launch_pdl(bn_bwd_fused_kernel, grid, kThreads, smem_max, reinterpret_cast<cudaStream_t>(stream), q);
  (void)smem;
  return check_launch("lbt_bn_bwd_fused");
}

// Non-zero once the grid barrier of lbt_bn_bwd_fused has timed out (synchronises the device; not in lbt.h).
extern "C" int lbt_bn_debug_error() {
  int v = 0;
  if (cudaMemcpyFromSymbol(&v, lbt::g_bn_error, sizeof(v)) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return v;
}

extern "C" int lbt_bn_set_debug(void* dev_u64) {
  unsigned long long* p = reinterpret_cast<unsigned long long*>(dev_u64);
  return cudaMemcpyToSymbol(lbt::g_bn_dbg, &p, sizeof(p)) == cudaSuccess ? LBT_OK : LBT_ECUDA;
}

// Test hook (not in lbt.h): counts the pairs where fdiv_by(a, b, frcp_rn(b)) differs from __fdiv_rn(a, b) bit for bit.
// Pairs are generated on the device: b over [2^-9, 2^14) (any mantissa), a as a small-integer multiple of a power of two
// (mantissa differences like the batch-norm numerators), as a full random mantissa, or exactly 0 / -0.
namespace lbt {
namespace {
__global__ void test_fdiv_kernel(unsigned long long n, uint64_t seed, unsigned long long* mismatches, float* first_bad) {
  unsigned long long bad = 0;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
    const uint4 rnd = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), 7u, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const int eb = (int)(rnd.x % 23u) - 9;                      // exponent of b
    const float b = __int_as_float(((eb + 127) << 23) | (rnd.y & 0x7fffffu));
    float a;
    const uint32_t kind = rnd.z & 3u;
    if (kind == 0) {
      a = (float)((int)(rnd.w % 513u) - 256) * exp2i((int)((rnd.z >> 2) % 24u) - 16);      // k * 2^-f
    } else if (kind == 1) {
      const float t = (float)((int)(rnd.w % 513u) - 256) * exp2i(-7);
      a = __fsub_rn(t, __int_as_float(0x3d000000u | (rnd.z >> 9)));                          // k*2^-f - mean
    } else if (kind == 2) {
      a = __int_as_float((rnd.w & 0x807fffffu) | ((((rnd.z >> 2) % 60u) + 97u) << 23));     // any mantissa, 2^-30 .. 2^29
    } else {
      a = (rnd.w & 1u) ? 0.0f : -0.0f;
    }
    const float want = __fdiv_rn(a, b), got = fdiv_by(a, b, __frcp_rn(b));
    if (__float_as_uint(want) != __float_as_uint(got)) {
      if (bad == 0 && first_bad) {
        first_bad[0] = a;
        first_bad[1] = b;
      }
      ++bad;
    }
  }
  if (bad) atomicAdd(mismatches, bad);
}
}  // namespace
}  // namespace lbt

extern "C" int lbt_test_fdiv(uint64_t n, uint64_t seed, uint64_t* mismatches_dev, float* first_bad_dev, void* stream) {
  if (!mismatches_dev) return LBT_EINVAL;
  LBT_REQUIRE_ARCH();
  lbt::test_fdiv_kernel<<<148 * 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      (unsigned long long)n, seed, reinterpret_cast<unsigned long long*>(mismatches_dev), first_bad_dev);
  return lbt::check_launch("lbt_test_fdiv");
}
