// Internal (not part of the C ABI): the cp.async-gather implicit-GEMM kernel of conv_ldg.cu, shared by
// lbt_conv_i8_fprop and lbt_conv_i8_dgrad.
#pragma once

#include <stddef.h>
#include <stdint.h>

#include "../../include/lbt.h"

namespace lbt {

// Output rows of a convolution written through a strided (n, y, x) grid instead of `row * ldc`: the parity-class
// sub-convolutions of a strided input gradient (lbt_conv_i8_dgrad_strided) each fill one (a::sh, b::sw) sub-lattice of dX.
// Strides in ELEMENTS of the fp32 output (and of `addend`, which has the output's layout).
struct OutRemap {
  long long sn, sy, sx;
};

bool conv_ldg_ok(int C, int Cout, int kh, int kw);
bool conv_ldg_enabled();
bool conv_ldg_halo_applies(int N, int OH, int OW, int kh, int kw, int sh, int sw, int C);
int conv_ldg_c64_halo();   // 1: 64-channel inputs take the gather kernel when its halo loader applies
int conv_ldg_run(const void* src, int src_kind, int N, int SH, int SW, int C, const void* wp, int w_kind, size_t ldw, int Cout,
                 int kh, int kw, int sh, int sw, int pt, int pl, int OH, int OW, int gather, const int32_t* ibA,
                 const int32_t* ibB, int exp_const, const float* bias, float* out, size_t ldc, const lbt_qsite* q_out,
                 int8_t* k_out, int64_t* sums, const float* addend, void* stream);

// conv_halo.cu: stride-1 convolutions of 64- / 128-channel inputs, halo patches through the TMA engine, resident filter bank
bool conv_halo_applies(int N, int OH, int OW, int C, int Cout, int kh, int kw, int sh, int sw);
void conv_halo_enable(int mode);   // bit 0: on, bit 1: ignore the patch fill-ratio rule (tests)
int conv_halo_debug_error();
int conv_stem_debug_error();   // conv_stem.cu (first-layer weight gradient)
int conv_halo_run(const void* src, int src_kind, int N, int H, int W, int C, const void* wp, int w_kind, size_t ldw, int Cout, int kh,
                  int kw, int pt, int pl, int OH, int OW, const int32_t* ibA, const int32_t* ibB, int exp_const, const float* bias,
                  float* out, size_t ldc, const lbt_qsite* q_out, int8_t* k_out, int64_t* sums, const float* addend, void* stream,
                  const OutRemap* remap = nullptr, const void* src_lo = nullptr);   // src_lo: low byte plane (u8) of a 16-bit source
// lbt_conv_i8_fprop's body; remap != NULL: fp32 epilogue only, the im2col-TMA or halo kernels only
int conv_fprop_run(const void* src, int src_kind, int N, int H, int W, int C, const void* wp, int w_kind, size_t ldw, int Cout, int kh,
                   int kw, int sh, int sw, int pad_top, int pad_left, int OH, int OW, const int32_t* ib_src, const int32_t* ib_w,
                   int exp_const, const float* bias, float* out, size_t ldc, const lbt_qsite* q_out, int8_t* k_out, int64_t* sums,
                   const float* addend, void* stream, const OutRemap* remap, const void* src_lo = nullptr);   // src_lo: see conv_halo_run

// conv_i8.cu: lbt_conv_i8_dgrad_block's launch (arguments already validated by the entry point in conv_dgrad.cu)
int conv_dgrad_block_run(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* w2, int w_kind, size_t ldw, int Cin,
                         int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W, const int32_t* ib_g,
                         const int32_t* ib_w, int exp_const, const void* gs, int gs_kind, int Cout_s, const void* ws, int ws_kind,
                         size_t ldws, const int32_t* ib_gs, const int32_t* ib_ws, int exp_short, float* dx, size_t ldc,
                         const float* addend, void* stream);

bool conv_wgrad_ldg_ok(int C, int Cout, int kh, int kw);
int conv_wgrad_ldg_run(const void* src, int src_kind, int N, int H, int W, int C, const void* g, int g_kind, int Cout, int kh, int kw,
                       int sh, int sw, int pt, int pl, int OH, int OW, int64_t* acc64, int alpha, void* stream);

}  // namespace lbt
