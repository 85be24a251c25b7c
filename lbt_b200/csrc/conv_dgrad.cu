// Input gradient of a STRIDED convolution with wide gathered channels (tf.gradients(y, X, gradq),
// /root/reference/dynamic_fixed_point.py:305; the 3x3/2 and 1x1/2 convolutions that open ResNet stages 2-4), as
// sh*sw stride-1 sub-convolutions instead of a transposed im2col matrix + GEMM:
//
//   dX[sh*i + a, sw*j + b] = sum_{taps of residue group ((a+pt) mod sh, (b+pl) mod sw)} g[i + qa - r/sh, j + qb - s/sw] * W[r, s]
//
// Each parity class (a, b) of input pixels is a stride-1 correlation of the gradient map g with a 2x2 / 2x1 / 1x2 / 1x1
// sub-filter (3x3, stride 2) that is a contiguous column range of the class-ordered operand W2 (conv_classes.h, packed by
// lbt_param_prep), run on the halo-patch or im2col TMA kernels with the output rows written through the (a::sh, b::sw)
// sub-lattice of dX.  The im2col path wrote and re-read kh*kw*Cout bytes per input pixel (925 MB for ResNet-18's first 3x3/2)
// and multiplied the zeros of the dilated gradient; here every MAC is a real one and g is read once per class.
// Classes without taps (1x1 stride 2: three of four) are filled with the `addend` (or zeros) by a small kernel.
#include "conv_classes.h"
#include "conv_internal.h"
#include "common.cuh"

namespace lbt {
namespace {

__global__ void __launch_bounds__(256) dgrad_fill_kernel(float* __restrict__ out, const float* __restrict__ addend, uint32_t Hc,
                                                          uint32_t Wc, uint32_t c4, long long sn, long long sy, long long sx,
                                                          size_t total) {
  pdl_trigger();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (size_t)gridDim.x * 256) {
    const uint32_t c = (uint32_t)(i % c4);
    size_t t = i / c4;
    const uint32_t x = (uint32_t)(t % Wc);
    t /= Wc;
    const uint32_t y = (uint32_t)(t % Hc), n = (uint32_t)(t / Hc);
    const long long o = (long long)n * sn + (long long)y * sy + (long long)x * sx + 4ll * c;
    const float4 v = addend ? __ldcs(reinterpret_cast<const float4*>(addend + o)) : make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(out + o) = v;
  }
}

}  // namespace
}  // namespace lbt

using namespace lbt;

// g_lo != NULL: g is the high byte plane (s8) and g_lo the low one (u8) of a 16-bit gradient (k = 256 * hi + lo): every class runs
// as a dual-accumulator convolution (lbt_conv_i8_fprop_dual's kernels, one rounding)
static int dgrad_strided_run(const void* g, int g_kind, const void* g_lo, int N, int OH, int OW, int Cout, const void* w2, int w_kind,
                             size_t ldw, int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W,
                             const int32_t* ib_g, const int32_t* ib_w, int exp_const, float* dx, size_t ldc,
                             const float* addend, void* stream) {
  if (!g || !w2 || !dx) return LBT_EINVAL;
  if ((g_kind != LBT_MANT_S8 && g_kind != LBT_MANT_U8)) return LBT_EINVAL;
  if (g_lo && (g_kind != LBT_MANT_S8 || Cin < 64 || (Cout != 64 && Cout % 128))) return LBT_EUNSUPPORTED;
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cout <= 0 || kh <= 0 || kw <= 0 || sh <= 0 || sw <= 0 || OH <= 0 || OW <= 0)
    return LBT_EINVAL;
  if (pad_top < 0 || pad_left < 0 || ldc < (size_t)Cin || ldw < (size_t)kh * kw * Cout) return LBT_EINVAL;
  if (sh > 4 || sw > 4 || (Cout & 15) || (Cin & 3) || (ldc & 3) || (reinterpret_cast<uintptr_t>(dx) & 15) ||
      (addend && (reinterpret_cast<uintptr_t>(addend) & 15)))
    return LBT_EUNSUPPORTED;
  // every class must be a correlation with non-negative padding (true for every 'SAME' / 'VALID' layer of the model zoo)
  for (int a = 0; a < sh; ++a) {
    const int r0 = (a + pad_top) % sh, nr = class_count(r0, kh, sh);
    if (nr && nr - 1 - (a + pad_top) / sh < 0) return LBT_EUNSUPPORTED;
  }
  for (int b = 0; b < sw; ++b) {
    const int s0 = (b + pad_left) % sw, nc = class_count(s0, kw, sw);
    if (nc && nc - 1 - (b + pad_left) / sw < 0) return LBT_EUNSUPPORTED;
  }
  LBT_REQUIRE_ARCH();
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  for (int a = 0; a < sh && a < H; ++a)
    for (int b = 0; b < sw && b < W; ++b) {
      const int Hc = (H - a + sh - 1) / sh, Wc = (W - b + sw - 1) / sw;   // pixels of this class
      const int r0 = (a + pad_top) % sh, s0 = (b + pad_left) % sw;
      const int nr = class_count(r0, kh, sh), nc = class_count(s0, kw, sw);
      OutRemap rm{(long long)H * W * (long long)ldc, (long long)sh * W * (long long)ldc, (long long)sw * (long long)ldc};
      float* out = dx + ((size_t)a * W + b) * ldc;
      const float* ad = addend ? addend + ((size_t)a * W + b) * ldc : nullptr;
      if (nr == 0 || nc == 0) {   // no tap reaches this class: dX = the other branch's gradient (or 0)
        const size_t total = (size_t)N * Hc * Wc * (Cin / 4);
        const size_t blocks = (total + 255) / 256, cap = (size_t)device_info().sm_count * 8;
        launch_pdl(dgrad_fill_kernel, (unsigned)(blocks < cap ? blocks : cap), 256, 0, st, out, ad, (uint32_t)Hc, (uint32_t)Wc,
                   (uint32_t)(Cin / 4), rm.sn, rm.sy, rm.sx, total);
        const int rc = check_launch("lbt_conv_i8_dgrad_strided (fill)");
        if (rc) return rc;
        continue;
      }
      const int pt2 = nr - 1 - (a + pad_top) / sh, pl2 = nc - 1 - (b + pad_left) / sw;
      const uint8_t* wp = reinterpret_cast<const uint8_t*>(w2) + (size_t)class_group_offset(r0, s0, kh, kw, sh, sw) * Cout;
      const int rc = conv_fprop_run(g, g_kind, N, OH, OW, Cout, wp, w_kind, ldw, Cin, nr, nc, 1, 1, pt2, pl2, Hc, Wc, ib_g, ib_w,
                                    exp_const, nullptr, out, ldc, nullptr, nullptr, nullptr, ad, stream, &rm, g_lo);
      if (rc) return rc;
    }
  return LBT_OK;
}

extern "C" int lbt_conv_i8_dgrad_strided(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* w2, int w_kind,
                                         size_t ldw, int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W,
                                         const int32_t* ib_g, const int32_t* ib_w, int exp_const, float* dx, size_t ldc,
                                         const float* addend, void* stream) {
  return dgrad_strided_run(g, g_kind, nullptr, N, OH, OW, Cout, w2, w_kind, ldw, Cin, kh, kw, sh, sw, pad_top, pad_left, H, W, ib_g, ib_w,
                           exp_const, dx, ldc, addend, stream);
}

// The whole input gradient of a downsampling block in one launch (conv_i8.cu, conv_dgrad_block_kernel): every parity class
// of the main convolution's dgrad and, in a second accumulator of the class it samples, the 1x1/s shortcut's dgrad.
extern "C" int lbt_conv_i8_dgrad_block(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* w2, int w_kind, size_t ldw,
                                       int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W,
                                       const int32_t* ib_g, const int32_t* ib_w, int exp_const, const void* g_short, int gs_kind,
                                       int OHs, int OWs, int Cout_s, const void* w_short, int ws_kind, size_t ldws,
                                       const int32_t* ib_gs, const int32_t* ib_ws, int exp_short, float* dx, size_t ldc,
                                       const float* addend, void* stream) {
  if (!g || !w2 || !dx || !ib_g || !ib_w) return LBT_EINVAL;
  if ((g_kind != LBT_MANT_S8 && g_kind != LBT_MANT_U8) || (w_kind != LBT_MANT_S8 && w_kind != LBT_MANT_U8)) return LBT_EINVAL;
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cout <= 0 || kh <= 0 || kw <= 0 || sh <= 0 || sw <= 0 || OH <= 0 || OW <= 0)
    return LBT_EINVAL;
  if (pad_top < 0 || pad_left < 0 || ldc < (size_t)Cin || ldw < (size_t)kh * kw * Cout) return LBT_EINVAL;
  if (g_short) {
    if (!w_short || !ib_gs || !ib_ws) return LBT_EINVAL;
    if ((gs_kind != LBT_MANT_S8 && gs_kind != LBT_MANT_U8) || (ws_kind != LBT_MANT_S8 && ws_kind != LBT_MANT_U8)) return LBT_EINVAL;
    if (OHs <= 0 || OWs <= 0 || Cout_s <= 0 || ldws < (size_t)Cout_s) return LBT_EINVAL;
    // the 1x1 / (sh, sw) shortcut without padding samples exactly parity class (0, 0), in g_short's row order
    if (OHs != (H + sh - 1) / sh || OWs != (W + sw - 1) / sw) return LBT_EUNSUPPORTED;
    if (addend) return LBT_EUNSUPPORTED;   // one sum per element: the shortcut term or an external addend
  }
  const int cb = Cout >= 128 ? 128 : Cout;
  if (Cin % 4) return LBT_EUNSUPPORTED;
  if (sh > 2 || sw > 2 || (cb != 32 && cb != 64 && cb != 128) || Cout % cb || (Cin != 64 && Cin % 128)) return LBT_EUNSUPPORTED;
  // exactness bound of one s32 accumulator, for the main term and for the shortcut's
  if (g_short && (Cout_s % cb || (uint32_t)Cout_s > max_products(gs_kind, ws_kind) || (Cout_s >= 128 ? 128 : Cout_s) != cb))
    return LBT_EUNSUPPORTED;
  if ((size_t)kh * kw * Cout > max_products(g_kind, w_kind) || kh > 255 || kw > 255) return LBT_EUNSUPPORTED;
  if ((size_t)N * H * W >= (1ull << 31)) return LBT_EUNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(g) & 15) || (reinterpret_cast<uintptr_t>(w2) & 15) || (ldw & 15) || (ldc & 3) ||
      (reinterpret_cast<uintptr_t>(dx) & 15) || (addend && (reinterpret_cast<uintptr_t>(addend) & 15)) ||
      (g_short && ((reinterpret_cast<uintptr_t>(g_short) & 15) || (reinterpret_cast<uintptr_t>(w_short) & 15) || (ldws & 15))))
    return LBT_EUNSUPPORTED;
  for (int a = 0; a < sh; ++a) {
    const int r0 = (a + pad_top) % sh, nr = class_count(r0, kh, sh);
    if (nr && nr - 1 - (a + pad_top) / sh < 0) return LBT_EUNSUPPORTED;
  }
  for (int b = 0; b < sw; ++b) {
    const int s0 = (b + pad_left) % sw, nc = class_count(s0, kw, sw);
    if (nc && nc - 1 - (b + pad_left) / sw < 0) return LBT_EUNSUPPORTED;
  }
  return conv_dgrad_block_run(g, g_kind, N, OH, OW, Cout, w2, w_kind, ldw, Cin, kh, kw, sh, sw, pad_top, pad_left, H, W, ib_g, ib_w,
                              exp_const, g_short, gs_kind, Cout_s, w_short, ws_kind, ldws, ib_gs, ib_ws, exp_short, dx, ldc, addend,
                              stream);
}

extern "C" int lbt_conv_i8_dgrad_strided_dual(const int8_t* g_hi, const uint8_t* g_lo, int N, int OH, int OW, int Cout, const void* w2,
                                              int w_kind, size_t ldw, int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left,
                                              int H, int W, const int32_t* ib_g, const int32_t* ib_w, int exp_const, float* dx, size_t ldc,
                                              const float* addend, void* stream) {
  if (!g_lo) return LBT_EINVAL;
  return dgrad_strided_run(g_hi, LBT_MANT_S8, g_lo, N, OH, OW, Cout, w2, w_kind, ldw, Cin, kh, kw, sh, sw, pad_top, pad_left, H, W, ib_g,
                           ib_w, exp_const, dx, ldc, addend, stream);
}
