/*
 * lbt.h — C ABI of liblbt_b200.so: the B200 (sm_100a) kernels behind the dynamic-fixed-point
 * (DFXP) training hot path of freudh/lbt.
 *
 * The reference has no FFI layer (it is pure Python on TensorFlow 1.x); the "interface each entry
 * point replaces" is therefore the reference Python function / the TF op it dispatched to
 * (file:line under /root/reference).  Conventions:
 *   - plain C types only; every buffer is owned by the caller (device memory unless stated);
 *   - the library never allocates or frees device memory and never synchronises with the host:
 *     all scalar state (ranges, overflow counters, the step counter) lives on the device, so a
 *     whole training step is CUDA-graph capturable;
 *   - `stream` is a cudaStream_t passed as void*; NULL = the legacy default stream;
 *   - return 0 on success, a negative LBT_E* code otherwise (lbt_strerror() names it); nothing
 *     throws or aborts across the ABI;
 *   - 16-byte aligned base pointers take the vectorised paths; anything else falls back to a
 *     scalar kernel with identical results.
 */
#ifndef LBT_H_
#define LBT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LBT_VERSION 100 /* 0.1.0 */

enum lbt_status {
  LBT_OK = 0,
  LBT_EINVAL = -1,       /* bad argument (null pointer, bits out of range, ...) */
  LBT_EUNSUPPORTED = -2, /* shape / alignment / kind not supported by this build */
  LBT_EARCH = -3,        /* device is not sm_100 (B200) */
  LBT_ECUDA = -4,        /* a CUDA runtime / driver call failed (see lbt_last_cuda_error) */
  LBT_EWORKSPACE = -5    /* workspace too small */
};

/* Rounding of lbt_quantize. */
enum lbt_round_mode {
  LBT_ROUND_NEAREST = 0,           /* `identity`,            dynamic_fixed_point.py:25-30 */
  LBT_ROUND_STOCHASTIC_NOISE = 1,  /* `stochastic_identity`, dynamic_fixed_point.py:32-38, noise from `noise[n_inner]` */
  LBT_ROUND_STOCHASTIC_PHILOX = 2, /* same, noise generated in-kernel (identical to lbt_noise_fill) */
  /* OR-able flag: gather the overflow statistics by min/max tracking instead of exact counts.  The counters then
   * hold "number of threads that saw an overflow" — still > 0 iff any element overflowed, which is all the
   * controller tests when target_overflow_rate == 0 (the reference's only setting); ignored for a non-zero target. */
  LBT_STATS_MINMAX = 0x100
};

/* Integer mantissa output of lbt_quantize (mantissa k = q * 2^(bits-integer_bits-1)). */
enum lbt_mant_kind {
  LBT_MANT_NONE = 0,
  LBT_MANT_S8 = 1,  /* bits <= 8 */
  LBT_MANT_U8 = 2,  /* bits <= 9 and input known non-negative (post-ReLU conv activations, F7) */
  LBT_MANT_S16 = 3, /* bits <= 16 */
  /* 3-channel signed 9-bit input (the image fed to a first Conv2d_q, bits+1 = 9): every pixel becomes 16
   * s8 bytes {hi0,hi1,hi2, hi0,hi1,hi2, lo0,lo1,lo2, 0 x 7} with k = 2*hi + lo, i.e. a 16-channel s8 NHWC
   * tensor the implicit-GEMM kernels consume against weights packed {W, W, W, 0}.  n_inner % 3 == 0. */
  LBT_MANT_S9C3 = 4,
  /* OR-able flag on the FILTER kind of the convolution entry points: the packed filter was written at least two launches
   * before this call on the same stream (e.g. by lbt_param_prep at the start of the step), so the kernel may start copying
   * it before it waits for its immediate predecessor (programmatic dependent launch).  Never set it for a filter produced by
   * the launch right before the call. */
  LBT_MANT_PREPARED = 0x100
};

/* Per-quantiser overflow statistics block: uint64_t[4] on the device. */
#define LBT_CNT_OVER 0      /* #{x*m >= L} + #{x*m < -L}        dynamic_fixed_point.py:63-64 */
#define LBT_CNT_OVER_HALF 1 /* #{x*m >= L/2} + #{x*m < -L/2}    dynamic_fixed_point.py:65-66 */
#define LBT_CNT_NUMEL 2     /* elements seen (denominator of reduce_mean, :67) */
#define LBT_CNT_TICKET 3    /* internal: CTA arrival ticket, always 0 between launches */
#define LBT_CNT_WORDS 4

int lbt_version(void);
const char* lbt_strerror(int status);
/* Text of the last CUDA error seen by the calling thread ("" if none). */
const char* lbt_last_cuda_error(void);
/* Number of kernels this library has launched from the calling process (for bench accounting). */
uint64_t lbt_launch_count(void);

/*
 * Fused DFXP quantiser: replaces weight_quantization() + overflow_rate() + update_range()
 * (dynamic_fixed_point.py:4-45, 48-67, 70-94), i.e. ~25 TF elementwise/reduce launches, with ONE
 * pass over x.  x is viewed as [n_outer, n_inner] = [dim0, prod(rest)]; stochastic noise has
 * n_inner values and is shared by all n_outer rows (tf.random_uniform(X.shape[1:]), :36).
 *
 *   m = 2^(bits - *integer_bits - 1), L = 2^(bits-1)
 *   nearest:     k = rint (min(max(x*m,     -L), L-1))          (ties to even)
 *   stochastic:  k = floor(min(max(x*m + u, -L), L-1))
 *   out_fp32 = k / m   (may be -0.0);   out_mant = (mant_kind) k
 *   counters += {#over, #over_half, n} measured on x*m (un-noised, un-clipped)
 *   update_range != 0: the last CTA applies  ib <- min(bits-1, ib + delta)  and zeroes counters,
 *     delta = +1 if over/n > t, else -1 if over_half/n <= t, else 0  (read-then-update: every
 *     element of this launch is quantised with the value *integer_bits had at launch).
 *   update_range == 0: counters are left accumulated for lbt_update_ranges() (data-parallel:
 *     all-reduce them first).
 *
 * bits in [1, 31] (everything dfxp:21 accepts below the pass-through); bits == 32 must be handled by the caller
 * (pass-through, :22-23).  fp32 output for every width; packed mantissas up to 16 bits (17 unsigned).  For bits > 25 the
 * clip bound L-1 is not an fp32 number and rounds to L, exactly as the reference's fp32 constant does.
 * out_fp32 and out_mant may each be NULL; with both NULL and counters given the launch is a
 * statistics-only pass (overflow_rate / update_range on their own, dynamic_fixed_point.py:48,70).
 * counters may be NULL only when update_range == 0 (no statistics are gathered).  dev_step (device uint64, may be NULL) is added
 * to the high word of `offset` so a captured CUDA graph draws fresh noise every replay.
 * out_fp32 may alias x (in-place).
 */
int lbt_quantize(const float* x, size_t n_outer, size_t n_inner, int bits, int32_t* integer_bits,
                 float target_overflow_rate, int mode, const float* noise, uint64_t seed,
                 uint64_t offset, const uint64_t* dev_step, float* out_fp32, void* out_mant,
                 int mant_kind, uint64_t* counters, int update_range, void* stream);

/*
 * u[j] for j < n_inner of the Philox4x32-10 stream lbt_quantize(mode=2) uses:
 *   r = philox4x32_10(counter = {g_lo, g_hi, off_lo, off_hi}, key = {seed_lo, seed_hi}), g = j / 4
 *   u[j] = (r[j % 4] >> 8) * 2^-24,  off = offset + (dev_step ? *dev_step << 32 : 0)
 * Stands in for tf.random_uniform (dynamic_fixed_point.py:36) so a run stays checkable on the CPU.
 */
int lbt_noise_fill(float* u, size_t n_inner, uint64_t seed, uint64_t offset, const uint64_t* dev_step,
                   void* stream);

/*
 * The range controller (update_range, dynamic_fixed_point.py:84-94) for n quantisers at once:
 *   ranges[i] <- min(bits[i]-1, ranges[i] + delta(counters[i], target[i])); counters[i] <- 0.
 * All arrays on the device; counters is uint64_t[n][LBT_CNT_WORDS].  Replaces the reference's
 * host-scheduled tf.cond/tf.assign per quantiser (trainer.py:63,157).
 */
int lbt_update_ranges(int32_t* ranges, uint64_t* counters, const int32_t* bits, const float* target,
                      size_t n, void* stream);

/* *dev_step += 1 (one thread); keeps the step counter on the device for graph replay. */
int lbt_step_advance(uint64_t* dev_step, void* stream);

/*
 * One `weight_quantization(..., stochastic=True)` call site (dynamic_fixed_point.py:4-45) as the fused kernels
 * see it: the quantiser's width, its `*_range` variable, its noise (explicit tensor [n_inner], or NULL = the
 * in-kernel Philox stream keyed by (seed, offset + (*dev_step << 32)), identical to lbt_noise_fill) and its
 * statistics block.  Host struct, passed by pointer; every pointer inside is a device pointer.
 */
typedef struct lbt_qsite {
  int32_t bits;          /* total mantissa bits incl. sign */
  int32_t stats_minmax;  /* 1: LBT_STATS_MINMAX statistics (valid for target_overflow_rate == 0) */
  const int32_t* ib;     /* integer_bits (read only; the controller runs in lbt_update_ranges) */
  const float* noise;
  uint64_t seed, offset;
  const uint64_t* dev_step; /* may be NULL */
  uint64_t* counters;       /* uint64[LBT_CNT_WORDS], may be NULL */
} lbt_qsite;

/* Epilogue of lbt_gemm_i8. */
enum lbt_gemm_epilogue {
  LBT_EPI_F32 = 0,  /* out_f32[m*ldc+n] = fp32(acc) * 2^e (+ bias[n]),  e = exp_const + *ibA + *ibB */
  LBT_EPI_ACC64 = 1 /* acc64[m*ldc+n] += alpha * acc  (64-bit integer atomics; split-K, exact) */
};

/*
 * D[M,N] = A[M,K] * B[N,K]^T on DFXP integer mantissas with exact int32 accumulation in tensor memory
 * (tcgen05.mma.kind::i8, TMA-fed).  Replaces the fp32 GEMMs the reference runs on fake-quantised
 * floats: tf.matmul (dynamic_fixed_point.py:388), tf.nn.conv2d after im2col (:196, :291) and their
 * tf.gradients (:207-210, :302-305, :457-460).
 *   A, B: K-major byte matrices (row pitch lda/ldb bytes, multiples of 16; 16-byte aligned bases);
 *         a_kind/b_kind = LBT_MANT_S8 or LBT_MANT_U8.
 *   LBT_EPI_F32: the value of a mantissa with `bits` total bits is k * 2^-(bits-1-ib), so pass
 *         exp_const = -(bitsA-1) - (bitsB-1) and the two device range pointers (either may be NULL = 0).
 *         Result == RN_fp32(exact_dot * 2^e) bit for bit.  K <= 65536, or 32768 when both operands are unsigned
 *         (LBT_EUNSUPPORTED above).
 *   LBT_EPI_ACC64: K is cut into k_splits chunks (each <= 65536, or 32768 when both operands are unsigned; more
 *         chunks than k_splits if needed) spread over the SMs; partial sums are
 *         added to acc64 (caller zeroes it) scaled by the integer alpha.  Finish with lbt_acc64_finalize.
 *   q_out != NULL (LBT_EPI_F32 only, N % 4 == 0): the fused re-quantising epilogue.  Instead of storing the
 *         fp32 result v, the kernel stores k_out[m*N + n] = Q_site(v) (s8, stochastic) and adds the exact
 *         per-column sums[n] += k, sums[N + n] += k*k (int64, caller-zeroed) plus the site's overflow
 *         statistics: Normalization_q's input quantiser + batch moments (dfxp:584-588) folded into the GEMM
 *         that produces its input.  The noise index of element (m, n) is (m % rows_per_image) * N + n.
 *         out_f32 may be NULL.
 *   addend != NULL (LBT_EPI_F32 without q_out): out_f32 = result + addend[m*ldc + n] — the other branch of a gradient
 *         sum (residual shortcut) folded into the epilogue instead of a separate add over the tensor.
 */
int lbt_gemm_i8(const void* A, int a_kind, size_t lda, const void* B, int b_kind, size_t ldb, size_t M,
                size_t N, size_t K, int epilogue, const int32_t* ibA, const int32_t* ibB, int exp_const,
                const float* bias, float* out_f32, int64_t* acc64, size_t ldc, int alpha, int k_splits,
                const lbt_qsite* q_out, int8_t* k_out, int64_t* sums, size_t rows_per_image, const float* addend,
                void* stream);

/*
 * The same GEMM with a 9..16-bit A operand given as its two byte planes k = 256 * hi + lo (A_hi s8, A_lo u8, same pitch):
 *   out_f32[m*ldc + n] = RN_fp32((256 * A_hi + A_lo)[m, :] . B[n, :] * 2^(exp_const + *ibA + *ibB)) (+ addend[m*ldc + n]).
 * The input-gradient GEMM of dfxp:305 / :460 with a gradient quantiser wider than 8 bits (BASELINE config 5, 16-bit G): both
 * halves are staged per K block beside ONE copy of B, two s32 accumulators per tile live in tensor memory and the epilogue
 * combines them in 64-bit integers before the single rounding — no int64 accumulator in HBM, no second pass over B.
 * K <= 65536, or 32768 when B is unsigned (A_lo x B is then u8 x u8); N tiles of at most 128 columns (two accumulator pairs
 * fill the 512 tensor-memory columns).
 */
int lbt_gemm_i8_dual(const int8_t* A_hi, const uint8_t* A_lo, size_t lda, const void* B, int b_kind, size_t ldb, size_t M,
                     size_t N, size_t K, const int32_t* ibA, const int32_t* ibB, int exp_const, float* out_f32, size_t ldc,
                     const float* addend, void* stream);

/*
 * out[i] = fp32(acc64[i]) * 2^(exp_const + *ibA + *ibB) (+ add_scale * add[i]) — the wgrad tail
 * `tf.gradients(y, W, gradq) + 2 * weight_decay * W` (dynamic_fixed_point.py:207, 302, 457).
 */
int lbt_acc64_finalize(const int64_t* acc64, size_t n, const int32_t* ibA, const int32_t* ibB, int exp_const,
                       const float* add, float add_scale, float* out, void* stream);

/*
 * im2col gather of an NHWC mantissa tensor src[N,H,W,C] into the K-major GEMM operand
 * out[M = N*OH*OW, K = kh*kw*C] (row pitch ld bytes), k = (r*kw + s)*C + c — the A operand of the
 * implicit GEMMs behind tf.nn.conv2d / Conv2DBackpropInput (dynamic_fixed_point.py:291, 305).
 *   transposed == 0 (fprop): row (n,oh,ow) reads src[n, oh*sh - pad_top + r, ow*sw - pad_left + s, c]
 *   transposed == 1 (dgrad): src is the output-gradient map; row (n,oh,ow) iterates the conv INPUT
 *     grid and reads src[n, (oh + pad_top - r)/sh, (ow + pad_left - s)/sw, c] where divisible.
 * Out-of-range taps are 0 (TF 'SAME' zero padding).  src_kind S8/U8 copies bytes; S16 (signed
 * mantissas wider than 8 bits, e.g. the 9-bit first-layer activations) writes K*3 bytes per row:
 * [hi | hi | lo] with k = 2*hi + lo, to be multiplied against [W | W | W].
 */
int lbt_im2col_i8(const void* src, int src_kind, int N, int H, int W, int C, int OH, int OW, int kh, int kw,
                  int sh, int sw, int pad_top, int pad_left, int transposed, void* out, size_t ld,
                  void* stream);

/*
 * Implicit-GEMM convolution on mantissas (no im2col matrix in HBM): TMA im2col-mode loads of the NHWC
 * source + tcgen05.mma.kind::i8.  Replaces tf.nn.conv2d (dynamic_fixed_point.py:196, 291); run on the
 * output-gradient map with the 180-degree-rotated filter it is tf.gradients(y, X, gradq) of a stride-1
 * convolution (:210, :305).
 *   Narrow inputs (C in {16, 32, 64}, Cout <= 128) are gathered by cp.async loader warps with the filter bank
 *   resident in shared memory (the TMA engine retires only one pixel row per ~3 clocks per SM).
 *   src[N,H,W,C] s8|u8, C in {16, 32, 64} or a multiple of 128;  wp[Cout, kh*kw*C] packed K-major
 *   (k = (r*kw + s)*C + c, row pitch ldw bytes);  out[N*OH*OW, Cout] fp32 (row pitch ldc floats):
 *   out = fp32(acc) * 2^(exp_const + *ib_src + *ib_w) (+ bias[co]).  kh*kw*C <= 65536, or 32768 when both operands are
 *   unsigned.
 *   q_out != NULL (Cout % 4 == 0): fused re-quantising epilogue as in lbt_gemm_i8 — k_out[N*OH*OW, Cout] s8,
 *   sums[2*Cout], rows_per_image = OH*OW; `out` may then be NULL.  addend: as in lbt_gemm_i8 (fp32 [M, ldc]).
 */
int lbt_conv_i8_fprop(const void* src, int src_kind, int N, int H, int W, int C, const void* wp, int w_kind,
                      size_t ldw, int Cout, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH,
                      int OW, const int32_t* ib_src, const int32_t* ib_w, int exp_const, const float* bias,
                      float* out, size_t ldc, const lbt_qsite* q_out, int8_t* k_out, int64_t* sums, const float* addend,
                      void* stream);

/*
 * Stride-1 convolution of a 9..16-bit source given as its two byte planes k = 256 * hi + lo (hi s8, lo u8 — what
 * lbt_bn_bwd_apply emits for a 16-bit gradient quantiser, BASELINE config 5) with an 8-bit filter, as ONE implicit GEMM with two
 * accumulators in tensor memory: out[(n,oh,ow), co] = fp32(256 * (hi * W) + (lo * W)) * 2^e (+ addend), one rounding — the
 * arithmetic of lbt_gemm_i8_dual without the im2col matrices of the two planes.  With the rotated filter this is the stride-1
 * input gradient tf.gradients(y, X, gradq) (dynamic_fixed_point.py:305).  The TMA halo kernel (two patches per ring slot) where
 * its filter bank fits beside them (C == 64), the im2col-TMA kernel (both planes' blocks per ring slot) for C >= 64 otherwise;
 * LBT_EUNSUPPORTED for narrower sources or Cout < 64: lbt_im2col_i8 + lbt_gemm_i8_dual.  e = exp_const + *ib_src + *ib_w.
 * kh*kw*C <= 65536, or 32768 with an unsigned filter (lo * W is then u8 x u8).
 */
int lbt_conv_i8_fprop_dual(const int8_t* src_hi, const uint8_t* src_lo, int N, int H, int W, int C, const void* wp, int w_kind,
                           size_t ldw, int Cout, int kh, int kw, int pad_top, int pad_left, int OH, int OW,
                           const int32_t* ib_src, const int32_t* ib_w, int exp_const, float* out, size_t ldc,
                           const float* addend, void* stream);

/*
 * Input gradient of a convolution of ANY stride as an implicit GEMM (no im2col matrix in HBM), the transposed
 * gather of lbt_im2col_i8(transposed = 1) done by the kernel's loader warps: dx[(n,h,w), ci] = 2^e * sum over taps
 * (r,s) and co of g[n, (h + pad_top - r)/sh, (w + pad_left - s)/sw, co] * wp[ci, (r*kw + s)*Cout + co] where
 * divisible — tf.gradients(y, X, gradq) (dynamic_fixed_point.py:210, 305).  g[N,OH,OW,Cout] s8|u8 with
 * Cout in {16, 32, 64}; Cin <= 128; dx[N*H*W, Cin] fp32 (row pitch ldc floats); e = exp_const + *ib_g + *ib_w.
 */
int lbt_conv_i8_dgrad(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* wp, int w_kind,
                      size_t ldw, int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W,
                      const int32_t* ib_g, const int32_t* ib_w, int exp_const, float* dx, size_t ldc, const float* addend,
                      void* stream);

/*
 * Implicit-GEMM weight gradient: acc64[(r*kw+s)*C + c, co] += alpha * sum over output pixels m of
 * src[pixel(m) + (r,s), c] * g[m, co] — tf.gradients(y, W, gradq) (dynamic_fixed_point.py:207, 302) in HWIO
 * order, exact.  Both operands are consumed MN-major straight from TMA loads (no transposes); the pixel
 * dimension is split over the SMs (k_splits, 0 = auto; each CTA sums <= 65536 pixels in s32, or 32768 when both operands
 * are unsigned, which may add splits) and reduced
 * with 64-bit atomics.  src[N,H,W,C] and g[N*OH*OW, Cout] are s8|u8 with C, Cout in {16,32,64} or
 * multiples of 128.  Caller zeroes acc64[kh*kw*C, Cout]; finish with lbt_acc64_finalize.
 */
int lbt_conv_i8_wgrad(const void* src, int src_kind, int N, int H, int W, int C, const void* g, int g_kind, int Cout,
                      int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH, int OW, int64_t* acc64,
                      int alpha, int k_splits, void* stream);

/* lbt_conv_i8_wgrad for a 9..16-bit gradient given as its byte planes k = 256 * hi + lo (g_hi s8, g_lo u8; BASELINE config 5):
 * ONE launch with two accumulators in tensor memory — the input blocks are loaded once and every element costs one int64
 * atomic, acc64 += alpha * (256 * sum(src * hi) + sum(src * lo)) — instead of two lbt_conv_i8_wgrad passes (alpha = 256 | 1). */
int lbt_conv_i8_wgrad_dual(const void* src, int src_kind, int N, int H, int W, int C, const int8_t* g_hi, const uint8_t* g_lo,
                           int Cout, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int OH, int OW,
                           int64_t* acc64, int alpha, int k_splits, void* stream);

/*
 * Weight gradient of a FIRST convolution (3-channel 9-bit image, LBT_MANT_S9C3 pixels x16[N,H,W,16]) of stride 2 with
 * <= 8 x 8 taps and 64 output channels (the 7x7/2 ImageNet stem; tf.gradients(y, W, gradq), dynamic_fixed_point.py:207,
 * 302 for models.py's first Conv2d_q): the image is re-packed into work8 (lbt_stem_pack8_bytes(N, H, OW) bytes: 8-byte
 * pixels {hi0,hi1,hi2,0,lo0,lo1,lo2,0} with zero margins) and every filter row of a 128-pixel patch then arrives as ONE
 * tiled TMA load.  acc8[((r*8 + s)*8 + b), co] (int64[512, Cout], zeroed by the caller) += sum over pixels of byte b of
 * tap (r, s) times g, times alpha; the caller combines dW[r,s,c,co] = 2 * acc8[r,s,c,co] + acc8[r,s,4+c,co].
 * g[N*OH*OW, Cout] s8 | u8 (g_kind; the byte planes of a 16-bit gradient: alpha = 256 | 1, repack = 0 on the second call:
 * work8 still holds this step's image).  LBT_EUNSUPPORTED for other shapes (odd H, Cout != 64, ...): use
 * lbt_conv_i8_wgrad on the 16-byte pixels.
 */
size_t lbt_stem_pack8_bytes(int N, int H, int OW);
/* The re-pack alone (what lbt_conv_i8_wgrad_c3 does first when repack != 0): a caller that runs it during the forward pass,
 * beside the first convolution, takes it off the end of the step. */
int lbt_stem_pack8(const int8_t* x16, int N, int H, int W, int OW, int pad_left, int8_t* work8, void* stream);
int lbt_conv_i8_wgrad_c3(const int8_t* x16, int N, int H, int W, const void* g, int g_kind, int Cout, int kh, int kw,
                         int pad_top, int pad_left, int OH, int OW, int8_t* work8, int repack, int64_t* acc8, int alpha,
                         void* stream);

/*
 * Mantissas wider than 8 bits (the 16-bit gradients of BASELINE config 5) as two tensor-core operands:
 * k = 256 * hi + lo with hi = k >> 8 (s8) and lo = k & 255 (u8).  The GEMMs run once per half and add
 * alpha * acc into the int64 accumulator with alpha = 256 and 1 (exact).
 */
int lbt_split_s16(const int16_t* in, size_t n, int8_t* hi, uint8_t* lo, void* stream);

/* out[c*ld_out + r] = in[r*ld_in + c] for an R x C byte matrix (operand re-majoring for wgrad). */
int lbt_transpose_i8(const void* in, size_t R, size_t C, size_t ld_in, void* out, size_t ld_out,
                     void* stream);

/*
 * acc64[c] += sum_r in[r*C + c] over an R x C matrix of s8 / s16 mantissas (exact).  The bias gradient
 * tf.gradients(y, b, gradq) (dynamic_fixed_point.py:209, 304, 459); finish with lbt_acc64_finalize.
 */
int lbt_colsum_i(const void* in, int kind, size_t R, size_t C, int64_t* acc64, void* stream);

/*
 * One launch for every gradient of the step: out[k] = fp32(acc64[k]) * 2^(exp_const + *ibA + *ibB)
 * (+ add_scale * add[k]) for each job — the tails `tf.gradients(...) + 2*weight_decay*W` of every layer
 * (dynamic_fixed_point.py:207-209, 302-304, 457-459, 689-690).  The job table lives on the device;
 * `start` is the running sum of n over the preceding jobs and `total` the sum of all n.
 */
typedef struct lbt_finalize_job {
  const int64_t* acc64;
  uint64_t n;
  const int32_t* ibA; /* may be NULL */
  const int32_t* ibB; /* may be NULL */
  int32_t exp_const;
  float add_scale;
  const float* add; /* may be NULL */
  float* out;
  uint64_t start;
} lbt_finalize_job;
int lbt_finalize_multi(const lbt_finalize_job* jobs_dev, size_t njobs, uint64_t total, void* stream);

/*
 * One launch for the noise vectors of many quantiser sites: u[e] for e < n of each job = the Philox4x32-10 stream of
 * lbt_noise_fill with (seed, job.offset + (*dev_step << 32)).  `start` is the running sum of ceil(n/4) over the
 * preceding jobs and total_groups the sum over all jobs; every u is 16-byte aligned.  Feeds lbt_qsite.noise of the
 * fused tensor-core epilogues (their threads then load the noise instead of generating it).
 */
typedef struct lbt_noise_job {
  float* u;
  uint64_t n;
  uint64_t offset;
  uint64_t start;
} lbt_noise_job;
int lbt_noise_fill_multi(const lbt_noise_job* jobs_dev, size_t njobs, uint64_t total_groups, uint64_t seed,
                         const uint64_t* dev_step, void* stream);

/*
 * One launch for every PARAMETER quantiser of the step (weights dfxp:289, 386; biases :294, 391; BN gamma /
 * beta :679-682): stochastic DFXP quantisation with the in-kernel Philox stream (offset = quantiser id,
 * + *dev_step << 32), overflow counters, and the operands the tensor-core kernels consume:
 *   out_f32  fake-quantised fp32 copy (vectors), or NULL
 *   LBT_PREP_CONV  (x is HWIO [kh,kw,Cin,Cout]): out_a[Cout, (r,s,ci)] (fprop B, pitch ld_a; c3pad: 16
 *                  pseudo-channels {W,W,W,0} per tap for a 3-channel first layer), out_b[Cin, (r',s',co)]
 *                  (dgrad B, pitch ld_b; rot180: taps reversed for the stride-1 implicit dgrad)
 *   LBT_PREP_DENSE (x is [in = Cin, out = Cout]): out_a[out, in], out_b[in, out]
 * Each CTA handles `chunk_elems` consecutive elements of one job: block_job / block_chunk give the mapping.
 */
enum lbt_prep_layout { LBT_PREP_VECTOR = 0, LBT_PREP_CONV = 1, LBT_PREP_DENSE = 2 };
typedef struct lbt_prep_job {
  const float* x;
  uint64_t n_outer, n_inner;
  const int32_t* ib;
  uint64_t* counters;
  uint64_t offset;
  float* out_f32;
  int8_t* out_a;
  int8_t* out_b;
  uint64_t ld_a, ld_b;
  int32_t bits, layout;
  uint32_t kh, kw, Cin, Cout;
  int32_t c3pad, rot180;   /* rot180: 0 filter order, 1 rotated by 180 degrees (stride-1 dgrad), 2 parity-class order (strided dgrad) */
  int32_t sh, sw;          /* convolution strides (rot180 == 2) */
} lbt_prep_job;
int lbt_param_prep(const lbt_prep_job* jobs_dev, const uint32_t* block_job_dev, const uint32_t* block_chunk_dev,
                   size_t nblocks, uint32_t chunk_elems, uint64_t seed, const uint64_t* dev_step, void* stream);

/*
 * Momentum SGD on flat fp32 buffers (tf.train.MomentumOptimizer.apply_gradients, trainer.py:81-82,
 * non-Nesterov):  accum <- momentum*accum + grad_scale*grad ;  w <- w - lr*accum.
 * dev_lr (device float, may be NULL) overrides lr so a captured graph can follow an LR schedule;
 * grad_scale = 1/world_size turns the all-reduced gradient sum into the data-parallel mean.
 */
int lbt_sgd_momentum(float* w, float* accum, const float* grad, size_t n, float lr, const float* dev_lr,
                     float momentum, float grad_scale, void* stream);

/*
 * Fused quantised batch-norm = Normalization_q + Rescale_q (dynamic_fixed_point.py:539-743), training mode,
 * NHWC tensors viewed as [n_outer = N, n_inner = H*W*C] with C % 4 == 0, all quantisers <= 8 bits and
 * stochastic (noise pointer [n_inner] or NULL = in-kernel Philox keyed by (seed, offset_*, dev_step)).
 * Statistics are exact integer sums of mantissas: `sums` buffers are int64, zeroed by the caller.
 *
 * fwd 1: k1 = Q_norm(x) (dfxp:584) ; sums[0..C) = sum k1, sums[C..2C) = sum k1^2 over N,H,W ; counters += stats.
 */
int lbt_bn_fwd_quant_stats(const float* x, size_t n_outer, size_t n_inner, int C, int bits, const int32_t* ib,
                           const float* noise, uint64_t seed, uint64_t offset, const uint64_t* dev_step,
                           int8_t* k1, int64_t* sums, uint64_t* counters, int stats_minmax, void* stream);
/*
 * fwd 2: mean/var (biased, dfxp:588) from `sums`; y1 = (xq - mean) / sqrt(var + eps) (dfxp:616);
 * k2 = Q_rescale(y1) (dfxp:677); out = xq2 * gamma_q + beta_q (dfxp:683) [+ add] [ReLU, dfxp:986].
 * Optionally writes the batch moments and updates the running averages (momentum*avg + (1-momentum)*batch,
 * dfxp:602-612).  gamma_q / beta_q are the fake-quantised vectors (lbt_quantize, dfxp:679-682).
 * q_next != NULL: the module output is additionally quantised with the CONSUMING layer's input quantiser
 * (Conv2d_q's `Xq`, dfxp:287: bits+1, stochastic) and stored as mantissas next_mant (next_kind LBT_MANT_U8 for a
 * 9-bit non-negative tensor, LBT_MANT_S8 for <= 8 bits), with that site's overflow statistics; `out` may then
 * be NULL when no other consumer needs the fp32 tensor.
 */
int lbt_bn_fwd_apply(const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1, const int32_t* ib1,
                     const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                     uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                     const float* gamma_q, const float* beta_q, const float* add, int relu, int8_t* k2,
                     float* out, float* batch_mean, float* batch_var, float* run_mean, float* run_var,
                     double momentum, int stats_minmax, const lbt_qsite* q_next, void* next_mant, int next_kind,
                     void* stream);
/* lbt_bn_fwd_apply with a SECOND consumer quantiser on the module output: a residual block whose first convolution and whose
 * strided 1x1 shortcut convolution both read the block input quantises it twice (one Conv2d_q `Xq` each, dfxp:287); both run
 * in the producing kernel.  q_next2 / next_mant2 / next_kind2 as q_next / next_mant / next_kind (q_next must be set too). */
int lbt_bn_fwd_apply2(const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1, const int32_t* ib1,
                      const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                      uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                      const float* gamma_q, const float* beta_q, const float* add, int relu, int8_t* k2,
                      float* out, float* batch_mean, float* batch_var, float* run_mean, float* run_var,
                      double momentum, int stats_minmax, const lbt_qsite* q_next, void* next_mant, int next_kind,
                      const lbt_qsite* q_next2, void* next_mant2, int next_kind2, void* stream);
/*
 * fwd 2 with the stride-2 3x3 max-pool that consumes the module output folded in (the ImageNet stem: conv -> BN -> ReLU ->
 * tf.nn.max_pool 3x3/2 'SAME', dfxp:993-1006): k2 and the statistics / running averages exactly as lbt_bn_fwd_apply; instead
 * of the fp32 module output, pooled[n_outer, POH, POW, C] and idx (winning tap r*k + s of every pooled element) exactly as
 * lbt_maxpool_fwd would produce from it (first maximum in scan order) — the fp32 tensor never exists.  k1[n_outer, H, W, C].
 * q_next / next_mant / next_kind as in lbt_bn_fwd_apply, applied to the POOLED tensor (the input quantiser of its consumer).
 * Shapes: C == 64, k == 3, s == 2, pad_top == pad_left == 0; else LBT_EUNSUPPORTED (run the two kernels).
 */
int lbt_bn_fwd_apply_pooled(const int8_t* k1, size_t n_outer, int H, int W, int C, int bits1, const int32_t* ib1,
                            const int64_t* sums, float eps, int bits2, const int32_t* ib2, const float* noise2,
                            uint64_t seed, uint64_t offset2, const uint64_t* dev_step, uint64_t* counters2,
                            const float* gamma_q, const float* beta_q, int relu, int8_t* k2, float* run_mean,
                            float* run_var, double momentum, int stats_minmax, int k, int s, int pad_top, int pad_left,
                            int POH, int POW, float* pooled, uint8_t* pidx, const lbt_qsite* q_next, void* next_mant,
                            int next_kind, void* stream);
/*
 * fwd 2 in eval mode (dfxp:616 with the running statistics): lbt_bn_fwd_apply / lbt_bn_fwd_apply2 with mean = run_mean[c] and
 * var = run_var[c] in place of the batch moments of `sums` — y1 = (xq - run_mean) / (run_var + eps) ** 0.5, then the same
 * Rescale_q quantiser, affine, add, ReLU and consumer quantisers, bit-identical to the training kernel's arithmetic.  Nothing
 * is written but the outputs: no batch moments, no running-average update.  k2 may be NULL (nothing is saved for a backward
 * pass).  q_next2 may be NULL (one consumer quantiser) or set together with q_next.  NULL k1 / run_mean / run_var / gamma_q /
 * beta_q, or C % 4 != 0: LBT_EINVAL before any CUDA call.
 */
int lbt_bn_fwd_apply_running(const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1, const int32_t* ib1,
                             const float* run_mean, const float* run_var, float eps, int bits2, const int32_t* ib2,
                             const float* noise2, uint64_t seed, uint64_t offset2, const uint64_t* dev_step,
                             uint64_t* counters2, const float* gamma_q, const float* beta_q, const float* add, int relu,
                             int8_t* k2, float* out, int stats_minmax, const lbt_qsite* q_next, void* next_mant,
                             int next_kind, const lbt_qsite* q_next2, void* next_mant2, int next_kind2, void* stream);
/* lbt_bn_fwd_apply_pooled in eval mode: the running statistics as in lbt_bn_fwd_apply_running, the max-pool as in
 * lbt_bn_fwd_apply_pooled (same shape limits, else LBT_EUNSUPPORTED); k2 may be NULL. */
int lbt_bn_fwd_apply_running_pooled(const int8_t* k1, size_t n_outer, int H, int W, int C, int bits1, const int32_t* ib1,
                                    const float* run_mean, const float* run_var, float eps, int bits2, const int32_t* ib2,
                                    const float* noise2, uint64_t seed, uint64_t offset2, const uint64_t* dev_step,
                                    uint64_t* counters2, const float* gamma_q, const float* beta_q, int relu, int8_t* k2,
                                    int stats_minmax, int k, int s, int pad_top, int pad_left, int POH, int POW,
                                    float* pooled, uint8_t* pidx, const lbt_qsite* q_next, void* next_mant, int next_kind,
                                    void* stream);
/*
 * bwd 1: g (w.r.t. the module output) -> ReLU mask (relu: 0 none, 1 recomputed from k2, 2 from `out`)
 * [-> d_add = masked g] -> kg2 = Q(g) (dfxp:687) -> sums[0..C) = sum kg2 (dbeta, :690),
 * sums[C..2C) = sum kg2*k2 (dgamma, :689) -> dx2 = gq2 * gamma_q (:691) -> kg1 = Q(dx2) (dfxp:621)
 * -> sums[2C..3C) = sum kg1, sums[3C..4C) = sum kg1*k1.
 * kg1_kind: LBT_MANT_S8 (both gradient quantisers <= 8 bits) or LBT_MANT_S16 (up to 16 bits — BASELINE config 5's 16-bit
 * gradients: kg1 is then int16 [n_outer, n_inner] and the per-thread partial sums are 64-bit).
 */
int lbt_bn_bwd_quant_stats(const float* g, const float* out, int relu, const int8_t* k2, const int8_t* k1,
                           size_t n_outer, size_t n_inner, int C, int bits2, const int32_t* ib2,
                           const float* gamma_q, const float* beta_q, int bits_g2, const int32_t* ib_g2,
                           const float* noise_g2, uint64_t offset_g2, uint64_t* counters_g2, int bits_g1,
                           const int32_t* ib_g1, const float* noise_g1, uint64_t offset_g1,
                           uint64_t* counters_g1, uint64_t seed, const uint64_t* dev_step, float* d_add,
                           void* kg1, int64_t* sums, int stats_minmax, int kg1_kind, void* stream);
/*
 * bwd 1 behind a max-pool (the ImageNet stems: conv -> BN -> ReLU -> 3x3/2 max-pool, models.py layer lists with MaxPool_q,
 * dfxp:993-1006): `g_pooled` [n_outer, OH, OW, C] is the gradient w.r.t. the POOLED tensor and `pool->idx` the winning tap
 * lbt_maxpool_fwd recorded for every pooled element; the pool's backward (each pixel collects the gradient of every window
 * it won, windows visited in (oh, ow) order as lbt_maxpool_bwd does) runs in this kernel's load stage, so the dense fp32
 * gradient of the un-pooled tensor (4 B written + 4 B read per element) never exists.  Bit-identical to
 * lbt_maxpool_bwd followed by lbt_bn_bwd_quant_stats.  Windows with k <= 2 * s, C % 4 == 0, relu in {0, 1}.
 * n_inner = pool->H * pool->W * C.
 */
typedef struct lbt_pool_geom {
  const uint8_t* idx;                 /* [n_outer, OH, OW, C] winning tap (r * k + s) */
  int32_t H, W;                       /* un-pooled grid */
  int32_t k, s, pad_top, pad_left;    /* window, stride, TF 'SAME' padding before */
  int32_t OH, OW;                     /* pooled grid */
} lbt_pool_geom;
int lbt_bn_bwd_quant_stats_pooled(const float* g_pooled, const lbt_pool_geom* pool, int relu, const int8_t* k2,
                                  const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits2, const int32_t* ib2,
                                  const float* gamma_q, const float* beta_q, int bits_g2, const int32_t* ib_g2,
                                  const float* noise_g2, uint64_t offset_g2, uint64_t* counters_g2, int bits_g1,
                                  const int32_t* ib_g1, const float* noise_g1, uint64_t offset_g1,
                                  uint64_t* counters_g1, uint64_t seed, const uint64_t* dev_step, void* kg1,
                                  int64_t* sums, int stats_minmax, int kg1_kind, void* stream);
/*
 * bwd 2: dx = (gq1 - mean(gq1) - xhat * mean(gq1 * xhat)) / sqrt(var + eps), the batch-norm VJP that
 * tf.gradients(y, X, gradq) yields for dfxp:616 (dfxp:623), from kg1, k1 and the two sum buffers.
 * q_grad != NULL: dx is quantised on the spot with the PRODUCING convolution's gradient quantiser (`gradq`,
 * dfxp:300) into g_mant (s8) with that site's statistics; `dx` may then be NULL.  A q_grad of 9..16 bits writes the
 * mantissa as its two byte planes k = 256 * hi + lo — g_mant = hi (s8), g_mant_lo = lo (u8) — the operands of
 * lbt_gemm_i8_dual / the alpha = 256 | 1 passes of lbt_conv_i8_wgrad.  kg1_kind as in lbt_bn_bwd_quant_stats.
 */
int lbt_bn_bwd_apply(const void* kg1, const int8_t* k1, size_t n_outer, size_t n_inner, int C, int bits1,
                     const int32_t* ib1, const int64_t* fwd_sums, float eps, int bits_g1, const int32_t* ib_g1,
                     const int64_t* bwd_sums, float* dx, const lbt_qsite* q_grad, int8_t* g_mant, int kg1_kind,
                     uint8_t* g_mant_lo, void* stream);

/*
 * lbt_bn_bwd_quant_stats + lbt_bn_bwd_apply in ONE launch, for tensors small enough that the whole tensor is one wave of
 * resident CTAs (<= 16 batch rows per CTA): the mantissas the second pass needs stay in shared memory and the CTAs meet
 * at a grid-wide barrier (`barrier`: one zeroed uint64 on the device).  Same arithmetic, bit-identical results.  Returns
 * LBT_EUNSUPPORTED when the tensor does not fit that shape — the caller then runs the two passes as separate launches.
 */
typedef struct lbt_bn_bwd_args {
  const float* g;          /* gradient w.r.t. the module output [n_outer, n_inner] */
  const float* out;        /* module output (relu == 2), or NULL */
  const int8_t* k2;
  const int8_t* k1;
  uint64_t n_outer, n_inner;
  int32_t C, relu;
  int32_t bits2, bits1;    /* Rescale_q X bits / Normalization_q X bits */
  const int32_t* ib2;
  const int32_t* ib1;
  const float* gamma_q;
  const float* beta_q;
  lbt_qsite q_g2, q_g1;    /* Rescale_q / Normalization_q gradient quantisers */
  float* d_add;            /* optional */
  int64_t* bwd_sums;       /* [4*C], zeroed */
  const int64_t* fwd_sums; /* [2*C] */
  float eps;
  int32_t has_q_grad;
  lbt_qsite q_grad;        /* the producing convolution's gradient quantiser (has_q_grad != 0) */
  float* dx;               /* optional when has_q_grad */
  int8_t* g_mant;
  uint64_t* barrier;
} lbt_bn_bwd_args;
int lbt_bn_bwd_fused(const lbt_bn_bwd_args* args, void* stream);

/*
 * tf.nn.max_pool on an NHWC fp32 tensor (`MaxPool_q`, dynamic_fixed_point.py:993-1006): 'SAME' padding ignores
 * out-of-range taps (pad_top / pad_left = TF's pad_before), 'VALID' is pad 0.  C % 4 == 0.  idx[N,OH,OW,C] receives the
 * winning tap r*k + s (first maximum in scan order); lbt_maxpool_bwd routes g[N,OH,OW,C] back through it as a gather
 * over the windows covering each input pixel (no atomics; dx is written exactly once).
 */
int lbt_maxpool_fwd(const float* x, int N, int H, int W, int C, int k, int s, int pad_top, int pad_left, int OH, int OW,
                    float* out, uint8_t* idx, void* stream);
int lbt_maxpool_bwd(const float* g, const uint8_t* idx, int N, int H, int W, int C, int k, int s, int pad_top,
                    int pad_left, int OH, int OW, float* dx, void* stream);

/*
 * tf.nn.avg_pool 'VALID' on an NHWC fp32 tensor (`AvgPool_q`, dynamic_fixed_point.py:1009-1022): window sums in
 * (row, column) order divided by k*k, and the gradient (each input pixel gathers g / (k*k) from the windows covering it).
 */
int lbt_avgpool_fwd(const float* x, int N, int H, int W, int C, int k, int s, int OH, int OW, float* out, void* stream);
int lbt_avgpool_bwd(const float* g, int N, int H, int W, int C, int k, int s, int OH, int OW, float* dx, void* stream);

/*
 * Mean sparse softmax cross-entropy (models.py:30-32): probs[B,C] = softmax(logits), *loss = mean_b -log probs[b,label_b];
 * backward: dlogits = (probs - onehot(labels)) * (*grad_loss) / B  (grad_loss NULL = 1).
 */
int lbt_softmax_xent_fwd(const float* logits, const int64_t* labels, int B, int C, float* probs, float* loss, void* stream);
int lbt_softmax_xent_bwd(const float* probs, const int64_t* labels, const float* grad_loss, int B, int C, float* dlogits,
                         void* stream);

/*
 * ReLU_q (dynamic_fixed_point.py:983-990): g == NULL: out = max(0, x); g != NULL: out = g where x > 0, else 0 (x may be
 * the forward input or output).  Dropout_q (:1025-1040): out = x / keep_prob * floor(keep_prob + u), u an explicit
 * uniform tensor [n] or (NULL) the Philox stream of lbt_noise_fill with (seed, offset + (*dev_step << 32)); the gradient is
 * the same call on g (the mask is recomputed, not stored).
 */
int lbt_relu(const float* x, const float* g, float* out, size_t n, void* stream);
int lbt_dropout(const float* x, const float* u, float keep_prob, uint64_t seed, uint64_t offset, const uint64_t* dev_step,
                float* out, size_t n, void* stream);

/*
 * Data-parallel end of a step as ONE kernel over NVLink peer memory (SURVEY.md 8e; the reference, trainer.py:79-84 +
 * :157-160, is single-device): barrier, reduce-scatter of the replicas' flat gradients by peer loads (sum in rank order),
 * momentum SGD on the owned slice with grad_scale = 1/world (as lbt_sgd_momentum), all-gather of the UPDATED WEIGHTS by
 * peer stores, overflow counters summed over the replicas + the range controller (as lbt_update_ranges), barrier,
 * counters zeroed, *dev_step += 1 (as lbt_step_advance).  Replaces two all-reduces and three launches.
 *
 * lbt_dp_peers: for every replica r the peer-mapped addresses of its flat gradient [n], flat weights [n], counters
 * [n_sites][LBT_CNT_WORDS] and a zero-initialised uint32 pad[LBT_DP_PAD_WORDS] (flags written by the peers' kernels).
 * Entry `rank` is the caller's own memory.  shard = 0: every replica reduces and updates all n parameters itself (no weight
 * stores, w[r != rank] unused); shard = 1: replica r owns parameters [r*ceil(n/4/world)*4, ...) and `accum` is only
 * maintained there.  n % 4 == 0.  All replicas must launch the call once per step (it spins on the peers' flags; waits are
 * bounded: after 20 s pad[LBT_DP_PAD_ERROR] is set and the kernel carries on).
 */
#define LBT_DP_MAX_WORLD 8
#define LBT_DP_PAD_READY 0   /* [world] flags: replica r has finished its backward (epoch number) */
#define LBT_DP_PAD_DONE 8    /* [world] flags: replica r has finished reading / writing peer memory */
#define LBT_DP_PAD_EPOCH 16
#define LBT_DP_PAD_TICKET 17
#define LBT_DP_PAD_ERROR 18  /* != 0: a wait timed out */
#define LBT_DP_PAD_WORDS 32
#define LBT_DP_HANDLE_BYTES 64
typedef struct lbt_dp_peers {
  int32_t world, rank;
  const float* grad[LBT_DP_MAX_WORLD];
  float* w[LBT_DP_MAX_WORLD];
  const uint64_t* counters[LBT_DP_MAX_WORLD];
  uint32_t* pad[LBT_DP_MAX_WORLD];
} lbt_dp_peers;
int lbt_dp_step(const lbt_dp_peers* peers, float* accum, size_t n, float lr, const float* dev_lr, float momentum,
                int shard, int32_t* ranges, const int32_t* bits, const float* target, size_t n_sites, uint64_t* dev_step,
                void* stream);
/*
 * Peer mapping of caller-owned buffers between the replica processes (CUDA IPC): lbt_dp_export gives the handle
 * (LBT_DP_HANDLE_BYTES) of the allocation containing ptr and ptr's offset in it; the caller ships both to the peers over
 * its own control plane; lbt_dp_open maps the allocation there (*base + offset = the buffer); lbt_dp_close unmaps.
 */
int lbt_dp_export(const void* ptr, void* handle64, size_t* offset);
int lbt_dp_open(const void* handle64, void** base);
int lbt_dp_close(void* base);

/*
 * The input pipeline of one training batch on the device (main.py:71-75 normalisation; trainer.py:24-28 preprocess_image;
 * trainer.py:92-96 shuffle + batch).  For output sample b, with i = index[b] (NULL: i = b):
 *   img = (double(src[i]) - mean) / 128, rounded to fp32 once (numpy float64 arithmetic, fp32 feed);
 *   flipped left-right if do_flip && flip_b; padded by `pad` zeros on every side; cropped H x W at (oy_b, ox_b).
 * params int32 [B][3] = (flip, oy, ox) explicit, or NULL: drawn in-kernel from Philox4x32-10 with counter (b, 0, offset) and
 * key seed: flip = r0 & 1, oy = r1 % (2*pad+1), ox = r2 % (2*pad+1).  src uint8 [n, H, W, C]; mean float64 [H, W, C] or NULL;
 * out fp32 NHWC [B, H, W, C]; labels_out[b] = labels[i] when both are given.  pad = 0, do_flip = 0: plain normalised batch.
 */
int lbt_augment_batch(const uint8_t* src, const double* mean, const int64_t* index, int B, int H, int W, int C, int pad,
                      int do_flip, const int32_t* params, uint64_t seed, uint64_t offset, const int64_t* labels,
                      int64_t* labels_out, float* out, void* stream);

/*
 * GradientBuffer_q (dynamic_fixed_point.py:473-509), the error-feedback gradient quantiser, in one pass:
 *   total = pad(grad, to n_outer rows) + buffer ; q = Q(total) (rounding / noise / statistics as lbt_quantize) ;
 *   buffer <- total - q ; out[r] = q[r] for r < n_grad_rows.
 * grad, out: [n_grad_rows, n_inner] (n_grad_rows <= n_outer: a short last batch); buffer: [n_outer, n_inner] in/out.
 * counters accumulate over all n_outer * n_inner elements of `total`; the range moves in lbt_update_ranges.
 */
int lbt_quantize_residual(const float* grad, size_t n_grad_rows, float* buffer, size_t n_outer, size_t n_inner, int bits,
                          int32_t* integer_bits, int mode, const float* noise, uint64_t seed, uint64_t offset,
                          const uint64_t* dev_step, float* out, uint64_t* counters, void* stream);

/*
 * Stride-1 input gradient of a convolution whose INPUT was produced by a fused batch-norm unit, with that batch-norm's
 * backward pass 1 (lbt_bn_bwd_quant_stats) run in the epilogue: the fp32 gradient dX = conv(g, rot180(W)) is never written;
 * instead, per element, the ReLU mask is recomputed from k2 (relu = 1) or skipped (0), kg2 = Q_g2(dX) (dfxp:687),
 * dx2 = gq2 * gamma_q (:691), kg1 = Q_g1(dx2) (:621) is stored, and sums[0..C) += kg2, [C..2C) += kg2*k2, [2C..3C) += kg1,
 * [3C..4C) += kg1*k1 (C = Cout of this call = the batch-norm's channels; caller-zeroed).  Same quantiser ids, noise streams,
 * counters and arithmetic as the two separate launches: bit-identical.  g[N,H,W,C] gradient mantissas of the convolution's
 * output; wp: filter packed for the transposed convolution as for lbt_conv_i8_fprop; OH x OW: the convolution's input grid.
 * Narrow-channel shapes only (LBT_EUNSUPPORTED otherwise: run lbt_conv_i8_fprop + lbt_bn_bwd_quant_stats).
 */
typedef struct lbt_bn_bwd_link {
  lbt_qsite q_g2, q_g1;      /* Rescale_q / Normalization_q gradient quantisers */
  int32_t bits2, relu;       /* Rescale_q input quantiser bits; ReLU: 0 none, 1 recomputed from k2 */
  const int32_t* ib2;
  const float* gamma_q;      /* [C] fake-quantised gamma / beta (16-byte aligned) */
  const float* beta_q;
  const int8_t* k2;          /* [N*OH*OW, C] saved forward mantissas */
  const int8_t* k1;
  int8_t* kg1;               /* [N*OH*OW, C] out */
  int64_t* sums;             /* [4*C] out */
} lbt_bn_bwd_link;
int lbt_conv_i8_dgrad_bn(const void* g, int g_kind, int N, int H, int W, int C, const void* wp, int w_kind, size_t ldw, int Cout,
                         int kh, int kw, int pad_top, int pad_left, int OH, int OW, const int32_t* ib_g, const int32_t* ib_w,
                         int exp_const, const lbt_bn_bwd_link* link, void* stream);

/*
 * Input gradient of a STRIDED convolution whose gathered tensor (the output gradient g[N,OH,OW,Cout]) is wide
 * (tf.gradients(y, X, gradq), dfxp:305, for the 3x3/2 and 1x1/2 convolutions that open the ResNet stages): run as sh*sw
 * stride-1 sub-convolutions, one per parity class (h mod sh, w mod sw) of input pixels, each on the sub-filter of the taps
 * that reach that class and each writing its own sub-lattice of dX[N,H,W,Cin] (row pitch ldc) — no transposed im2col
 * matrix, no multiplication by the zeros of a dilated gradient.  w2[Cin, kh*kw*Cout] (row pitch ldw) holds the filter
 * with its taps in PARITY-CLASS ORDER (lbt_param_prep with rot180 = 2: taps grouped by (r mod sh, s mod sw), groups in
 * row-major order, reversed (r / sh, s / sw) order inside a group).  Classes no tap reaches get `addend` (or zeros).
 * dX = RN_fp32(exact * 2^(*ib_g + *ib_w + exp_const)) (+ addend), bit-identical to the im2col + GEMM formulation.
 * Cout % 16 == 0 (and a multiple of 128 above 64), Cin % 4 == 0, strides <= 4.  Each class sums at most 65536 products per
 * accumulator (sub-filter taps * Cout), or 32768 when both operands are unsigned.
 */
int lbt_conv_i8_dgrad_strided(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* w2, int w_kind, size_t ldw,
                              int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W,
                              const int32_t* ib_g, const int32_t* ib_w, int exp_const, float* dx, size_t ldc,
                              const float* addend, void* stream);
/*
 * The whole input gradient of a downsampling residual block in ONE launch:
 *   dX = dgrad_{kh x kw / (sh, sw)}(g, w2) [+ dgrad_{1x1 / (sh, sw)}(g_short, w_short)] [+ addend]
 * The main term is lbt_conv_i8_dgrad_strided's parity-class decomposition (same operands: g[N,OH,OW,Cout], w2 in parity-class
 * order, e = exp_const + *ib_g + *ib_w), all classes in one tile list.  g_short[N, OHs, OWs, Cout_s] (or NULL) is the output
 * gradient of a 1x1 shortcut convolution of stride (sh, sw) without padding over the same input, w_short[Cin, Cout_s] (row
 * pitch ldws) its filter, e_s = exp_short + *ib_gs + *ib_ws; it samples parity class (0, 0), so OHs x OWs must be
 * ceil(H / sh) x ceil(W / sw).  Where the shortcut lands dX = RN(RN(main * 2^e) + RN(short * 2^e_s)), elsewhere RN(main * 2^e):
 * bit-identical to lbt_conv_i8_dgrad_strided on the shortcut followed by lbt_conv_i8_dgrad_strided on the main convolution
 * with that result as addend.  addend (the layout of dX) only without a shortcut.  Null pointers, bad kinds or shapes:
 * LBT_EINVAL; Cin % 4 != 0, strides > 2, Cin neither 64 nor a multiple of 128, Cout (Cout_s) not 32, 64 or a multiple of 128
 * (with the same channel chunk), kh*kw*Cout or Cout_s above 65536 (32768 when both operands of that term are unsigned),
 * misalignment, a shortcut lattice that does not match or a shortcut together with addend:
 * LBT_EUNSUPPORTED — all before any CUDA call.  Run the two lbt_conv_i8_dgrad_strided calls then.
 */
int lbt_conv_i8_dgrad_block(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* w2, int w_kind, size_t ldw,
                            int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W,
                            const int32_t* ib_g, const int32_t* ib_w, int exp_const, const void* g_short, int gs_kind,
                            int OHs, int OWs, int Cout_s, const void* w_short, int ws_kind, size_t ldws,
                            const int32_t* ib_gs, const int32_t* ib_ws, int exp_short, float* dx, size_t ldc,
                            const float* addend, void* stream);
/* The same for a 9..16-bit gradient given as its byte planes k = 256 * hi + lo (g_hi s8, g_lo u8; BASELINE config 5): every class is
 * a dual-accumulator convolution (lbt_conv_i8_fprop_dual's kernels), one rounding.  Cin >= 64, Cout == 64 or a multiple of 128. */
int lbt_conv_i8_dgrad_strided_dual(const int8_t* g_hi, const uint8_t* g_lo, int N, int OH, int OW, int Cout, const void* w2,
                                   int w_kind, size_t ldw, int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left,
                                   int H, int W, const int32_t* ib_g, const int32_t* ib_w, int exp_const, float* dx, size_t ldc,
                                   const float* addend, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LBT_H_ */
