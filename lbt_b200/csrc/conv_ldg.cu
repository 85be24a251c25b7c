// Implicit-GEMM convolution for NARROW channel counts (C in {16, 32, 64}, Cout <= 128) on B200 (sm_100a).
//
// Measured on B200 (benchmarks/tma_probe.cu): the TMA engine retires one [pixel x C] row every ~3 clocks per SM,
// im2col mode or tiled, whatever the row width — 5 B/clk/SM at C = 16, eight times below what the HBM-bound
// first-stage convolutions of the CIFAR / ImageNet ResNets need.  Here the A operand (the im2col rows) is gathered
// by four loader warps with 16-byte cp.async (512 B per warp instruction, zero-fill for the padding), straight into
// the tensor core's un-swizzled K-major layout; the whole filter bank stays resident in shared memory for the life
// of the persistent CTA; tcgen05.mma.kind::i8 accumulates in tensor memory and the epilogue is the same as the
// TMA-fed kernel's (fp32 rescale, or the fused re-quantise + batch statistics of qsite.cuh).
//
//   gather == 0  fprop:  row (n, oh, ow), tap (r, s) reads src[n, oh*sh - pt + r, ow*sw - pl + s, :]
//                         (tf.nn.conv2d, dynamic_fixed_point.py:291; with a rot180 filter also the stride-1 dgrad)
//   gather == 1  dgrad:  row (n, h, w) of dX, tap (r, s) reads g[n, (h + pt - r)/sh, (w + pl - s)/sw, :] where
//                         divisible (tf.gradients(y, X, gradq), dynamic_fixed_point.py:305, any stride) — the
//                         strided transposed convolution without an im2col matrix in HBM.
//
// Shared-memory layouts (SWIZZLE_NONE, "interleaved" 8x16B core matrices):
//   A stage : [8 K-chunks][128 rows][16 B]   chunk kc of the tile = (tap, 16-channel group), kc = tap * (C/16) + cc
//   B       : [KCp K-chunks][BN rows][16 B]  resident; KCp = chunk count rounded up to even (zero chunk)
// One K=32 MMA covers two consecutive chunks (leading byte offset = chunk stride).
#include <atomic>

#include "conv_internal.h"
#include "qsite.cuh"
#include "tcgen05.cuh"

namespace lbt {
namespace {

using namespace tc;

constexpr int kBlockM = 128;
constexpr int kLoaderWarps = 4;
constexpr int kEpiWarps = 8;  // two per TMEM lane quadrant, interleaved over the 16-column chunks
constexpr int kThreads = 32 * (kLoaderWarps + 1 + kEpiWarps);  // loaders, MMA issuer, epilogue
constexpr int kChunksPerStage = 8;
constexpr int kStageBytes = kChunksPerStage * kBlockM * 16;  // 16 KB
constexpr int kMaxStages = 8;
constexpr int kMaxAccStages = 4;
constexpr int kMaxKC = 256;   // 16-byte K chunks per tile (taps * C/16, padded to even)
constexpr int kMaxTaps = 64;  // per-row validity mask is one 64-bit word

__device__ int g_ldg_error = 0;

struct LdgParams {
  const uint8_t* src;            // NHWC mantissas of the gathered tensor
  const uint8_t* wp;             // packed filter [Cout, taps*C] K-major
  uint32_t ldw;
  uint32_t M, N;                 // output rows (pixels), output channels
  uint32_t SH, SW, C;            // gathered tensor: height, width, channels
  uint32_t OW, OHW;              // output grid width, height*width
  uint32_t ohw_mul, ohw_shr, ow_mul, ow_shr;   // n / d == __umulhi(n, mul) >> shr for n < 2^31 (d > 1)
  uint32_t cmask[4];             // filter columns s with s % sw == j (gather 1; all columns for gather 0, j = 0)
  unsigned long long rspread[4]; // sum over filter rows r with r % sh == j of 1 << (r * kw)
  int sh, sw, pt, pl;
  uint32_t kw, taps, cpp;        // filter width, kh*kw, C/16
  uint32_t KC, KCp;              // 16-byte K chunks (real, padded to even)
  uint32_t stages_per_tile;      // ceil(KCp / 8)
  uint32_t nstages;              // ring depth
  uint32_t m_tiles;
  int gather;                    // 0 fprop, 1 transposed (dgrad)
  const int32_t* ibA;
  const int32_t* ibB;
  int exp_const;
  const float* bias;
  const float* addend;           // optional fp32 [M, ldc] added to the fp32 result (F32 epilogue only)
  float* out;
  size_t ldc;
  uint32_t idesc;
  BnqParams bnq;
  unsigned long long* dbg;       // optional timeline of CTA 0 (globaltimer ns), see lbt_conv_ldg_set_debug
  // halo mode (stride-1 gather 0): an M tile is an 8-wide x 16-high patch of output pixels of ONE image
  uint32_t OH, n_img;
  uint32_t halo_w, halo_px;      // 8 + kw - 1, halo_w * (16 + kh - 1)
  uint32_t halo_plane;           // bytes of one 16-channel plane of the halo: halo_px * 16
  uint32_t stage_bytes;          // ring slot: kStageBytes (gather modes) / CPP planes + slack (halo mode)
  FastDiv d_tiles_img, d_tiles_x;
  // strided halo (sh = sw = 2, 16-byte pixels: the 7x7/2 ImageNet stem on the {hi,hi,lo,0} x 16 image layout): the patch is
  // stored as `sw` column-parity planes so that neighbouring OUTPUT pixels are 16 bytes apart for every filter tap
  uint32_t halo_hw2;             // columns of one parity plane: halo_w / sw
  uint32_t halo_par_plane;       // bytes of one parity plane: halo rows * halo_hw2 * 16
  uint32_t halo_mmas;            // MMA instructions per tile (stride 1: KCp / 2)
  FastDiv d_halo_w;
  int epi16;                     // host: launch the 16-epilogue-warp instantiation (one CTA per SM)
};

__device__ __forceinline__ void dbg_stamp(const LdgParams& p, int slot) {
  if (p.dbg && blockIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    p.dbg[slot] = t;
  }
}

__device__ __forceinline__ uint32_t fast_div(uint32_t n, uint32_t d, uint32_t mul, uint32_t shr) {
  return d == 1 ? n : (__umulhi(n, mul) >> shr);
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");   // .cg: L1 is kept for the epilogue's noise lines
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Shared-memory descriptor of a K-major, un-swizzled operand with explicit strides: `lbo` between the two 16-byte K chunks
// of an instruction, `sbo` between consecutive 8-row groups.
__device__ __forceinline__ uint64_t make_desc_k16(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
         (1ull << 46);
}

// HALO = true (stride-1 convolutions on images of at least ~8 x 16 output pixels): instead of gathering the im2col rows of a
// tile — every input pixel crosses L2 -> shared memory kh*kw times, which is what bounds the gather path — the loaders copy the
// (16 + kh - 1) x (8 + kw - 1) input patch under an 8 x 16 output patch ONCE ([C/16 planes][halo pixels][16 B]), and the MMA
// descriptors walk it: the 8 rows of a core matrix are 8 neighbouring pixels of an output row (16-byte pitch), consecutive
// 8-row groups are halo rows (stride halo_w * 16 B), and a filter tap is just a different start address.
// EPI epilogue warps: 8 with two CTAs per SM, or 16 in ONE CTA per SM when the resident filter bank is too big for two CTAs
// (the 7x7 ImageNet stem: 8 epilogue warps alone on an SM cannot keep up with the fused epilogue).
template <int BN, int CPP, bool HALO, int EPI = 8>   // CPP = C / 16: 16-byte chunks per pixel
__global__ void __launch_bounds__(32 * (kLoaderWarps + 1 + EPI), EPI == 8 ? 2 : 1) conv_ldg_kernel(const LdgParams p) {
  constexpr int kEpiWarps = EPI;
  constexpr int kThreads = 32 * (kLoaderWarps + 1 + EPI);
  constexpr int kSub = EPI / 4;   // epilogue warps per TMEM lane quadrant
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
  __shared__ __align__(8) uint64_t full_bar[kMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
  constexpr int kAccStages = (BN <= 64 || EPI == 16) ? 4 : 2;   // two CTAs per SM must fit the 512 TMEM columns
  __shared__ __align__(8) uint64_t tmem_full_bar[kMaxAccStages];
  __shared__ __align__(8) uint64_t tmem_empty_bar[kMaxAccStages];
  __shared__ __align__(8) uint64_t b_bar;   // the resident filter bank has landed
  __shared__ uint32_t tmem_slot;
  __shared__ int s_abort;
  constexpr int kStats = 2;                      // per-channel sums of the fused epilogue
  __shared__ int s_stat[kEpiWarps][kStats * BN];
  __shared__ unsigned long long s_tot[kStats * BN];   // CTA totals of the fused statistics
  __shared__ int2 s_tab[kMaxKC + 8];       // tap slot: {byte offset from the row's base pixel, tap code}
  __shared__ uint2 s_mma[HALO ? kMaxKC / 2 : 1];   // halo mode, MMA j: {A start offset in the stage, leading byte offset}
  __shared__ short s_kmap[HALO ? kMaxKC : 1];      // halo mode: filter chunk at each position of the resident bank

  constexpr int kTmemCols = (kAccStages * BN) < 32 ? 32 : (kAccStages * BN);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* sB = smem;                                        // KCp * BN * 16
  uint8_t* sA = smem + (((size_t)p.KCp * BN * 16 + 127) & ~(size_t)127);

  if (threadIdx.x == 0) {
    for (uint32_t s = 0; s < p.nstages; ++s) {
      mbar_init(&full_bar[s], HALO ? 32 : kLoaderWarps * 32);   // halo mode: one loader warp fills a slot
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], BN > 32 ? kEpiWarps : 4);   // narrow tiles: the two warps of a quadrant alternate TILES
    }
    mbar_init(&b_bar, kEpiWarps * 32);
    s_abort = 0;
    fence_barrier_init();
  }
  if (warp == kLoaderWarps) tmem_alloc(&tmem_slot, kTmemCols);
  for (uint32_t i = threadIdx.x; i < kStats * BN; i += kThreads) s_tot[i] = 0ull;
  // gather table, one entry per tap slot: source of (row, slot) = base(row) + x, valid iff bit y of the row's tap mask;
  // y == 255: zero chunk (K padding), y == 254: beyond the tile's chunks (nothing to copy)
  constexpr int TPS = kChunksPerStage / CPP;  // tap slots per pipeline stage
  for (uint32_t ts = threadIdx.x; !HALO && ts < p.stages_per_tile * TPS; ts += kThreads) {
    const int r = (int)(ts / p.kw), sx = (int)(ts % p.kw);
    int d;
    if (p.gather == 0) d = (r * (int)p.SW + sx) * (int)p.C;
    else d = -((r / p.sh) * (int)p.SW + (sx / p.sw)) * (int)p.C;
    const int code = ts < p.taps ? (int)ts : (ts * CPP < p.KCp ? 255 : 254);
    s_tab[ts] = make_int2(ts < p.taps ? d : 0, code);
  }
  if (HALO) {
    // MMA j of a tile: {A start offset inside the ring slot, leading byte offset}; s_kmap[kc] = the filter chunk (tap * CPP + cc)
    // that sits at position kc of the resident bank (-1: zero chunk)
    if (p.sw == 1) {
      for (uint32_t j = threadIdx.x; j < p.halo_mmas; j += kThreads) {
        const uint32_t kc = 2 * j, tap = kc / CPP;   // K chunk = tap * CPP + cc
        const uint32_t r = tap / p.kw, sx = tap - r * p.kw;
        uint32_t lbo = p.halo_plane;
        if (CPP == 1) {   // the instruction's second chunk is the NEXT tap (or, past the last one, anything: zero weights)
          const uint32_t t1 = tap + 1 < p.taps ? tap + 1 : tap, r1 = t1 / p.kw, s1 = t1 - r1 * p.kw;
          lbo = t1 > tap ? ((r1 * p.halo_w + s1) - (r * p.halo_w + sx)) * 16 : 16;
        }
        s_mma[j] = make_uint2((kc % CPP) * p.halo_plane + (r * p.halo_w + sx) * 16, lbo);
      }
      for (uint32_t kc = threadIdx.x; kc < p.KCp; kc += kThreads) s_kmap[kc] = kc < p.KC ? (short)kc : (short)-1;
    } else {
      // stride 2 (CPP == 1): an instruction covers taps (r, s) and (r, s + 2) — same column parity, neighbouring columns of
      // that parity plane (lbo = 16 B); per filter row: ceil(n0 / 2) + ceil(n1 / 2) instructions, n0 / n1 even / odd columns
      const uint32_t n0 = (p.kw + 1) / 2, n1 = p.kw / 2, p0 = (n0 + 1) / 2, per_row = p0 + (n1 + 1) / 2;
      for (uint32_t j = threadIdx.x; j < p.halo_mmas; j += kThreads) {
        const uint32_t r = j / per_row, jj = j - r * per_row;
        const uint32_t q = jj < p0 ? 0u : 1u, pi = jj - (q ? p0 : 0u);
        const uint32_t s0 = q + 4 * pi, s1 = s0 + 2;
        s_mma[j] = make_uint2(q * p.halo_par_plane + (r * p.halo_hw2 + (s0 >> 1)) * 16, 16u);
        s_kmap[2 * j] = (short)(r * p.kw + s0);
        s_kmap[2 * j + 1] = s1 < p.kw ? (short)(r * p.kw + s1) : (short)-1;
      }
    }
  }
  pdl_trigger();
  fence_before();
  __syncthreads();
  fence_after();
  // everything above touched only shared / tensor memory and kernel parameters
  pdl_wait();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);
  volatile int* abort_flag = &s_abort;
  if (threadIdx.x == 0) dbg_stamp(p, 1);

  if (HALO && warp < kLoaderWarps) {
    // ===== halo loaders: the input patch of a tile, each 16-byte chunk exactly once (zero-fill outside the image).  A loader
    // warp completes one ring slot per memory round trip (measured: ~0.8 us per tile whatever the copy count), so each of the
    // four warps loads WHOLE tiles, round robin: four patches are in flight per CTA =====
    bool ok = true;
    uint32_t seq = warp;                          // this warp's tiles: sequence numbers warp, warp + 4, ...
    for (uint32_t tile = blockIdx.x + warp * gridDim.x; tile < p.m_tiles && ok; tile += kLoaderWarps * gridDim.x, seq += kLoaderWarps) {
      const uint32_t stage = seq % p.nstages, phase = (seq / p.nstages) & 1u;
      const uint32_t img = fastdiv(tile, p.d_tiles_img), t2 = tile - img * p.d_tiles_img.d;
      const uint32_t ty = fastdiv(t2, p.d_tiles_x), tx = t2 - ty * p.d_tiles_x.d;
      const int y0 = (int)(ty * 16) * p.sh - p.pt, x0 = (int)(tx * 8) * p.sw - p.pl;
      const uint8_t* ibase = p.src + (size_t)img * p.SH * p.SW * p.C;
      ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag, &g_ldg_error);
      if (!ok) break;
      const uint32_t dst0 = smem_u32(sA + (size_t)stage * p.stage_bytes);
      for (uint32_t idx = lane; idx < p.halo_px * CPP; idx += 32) {
        const uint32_t hp = idx / CPP, cc = idx % CPP;
        const uint32_t hr = fastdiv(hp, p.d_halo_w), hc = hp - hr * p.halo_w;   // (row, column) of the halo pixel
        const int iy = y0 + (int)hr, ix = x0 + (int)hc;
        const bool v = iy >= 0 && iy < (int)p.SH && ix >= 0 && ix < (int)p.SW;
        // stride 1: pixel hp of plane cc; stride 2 (CPP == 1): column-parity plane hc & 1, column hc >> 1
        const uint32_t d = p.sw == 1 ? cc * p.halo_plane + hp * 16 : (hc & 1u) * p.halo_par_plane + (hr * p.halo_hw2 + (hc >> 1)) * 16;
        cp_async16(dst0 + d, v ? ibase + ((size_t)iy * p.SW + ix) * p.C + cc * 16 : p.src, v ? 16u : 0u);
      }
      cp_async_arrive_noinc(&full_bar[stage]);
      if (threadIdx.x == 0 && tile == blockIdx.x) dbg_stamp(p, 2);
      if (p.dbg && lane == 0 && seq < 10) dbg_stamp(p, 44 + seq);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else if (warp < kLoaderWarps) {
    // ===== loaders: one warp instruction copies 32/CPP consecutive pixels x C bytes (512 contiguous bytes when the
    // pixels are neighbours in memory); a thread serves CPP rows of the tile and always the same 16-byte chunk cc =====
    constexpr int RPI = 32 / CPP;  // rows per instruction
    const uint32_t cc = lane % CPP;
    const uint32_t rloc0 = warp * 32 + lane / CPP;  // + i * RPI
    const uint32_t kh = p.taps / p.kw;
    uint32_t stage = 0, phase = 0;
    bool ok = true;
    for (uint32_t tile = blockIdx.x; tile < p.m_tiles && ok; tile += gridDim.x) {
      unsigned long long mask[CPP];
      const uint8_t* base[CPP];
#pragma unroll
      for (int i = 0; i < CPP; ++i) {
        const uint32_t m = tile * kBlockM + rloc0 + i * RPI;
        const uint32_t img = fast_div(m, p.OHW, p.ohw_mul, p.ohw_shr), rem = m - img * p.OHW;
        const uint32_t oyu = fast_div(rem, p.OW, p.ow_mul, p.ow_shr);
        const int oy = (int)oyu, ox = (int)(rem - oyu * p.OW);
        // tap validity without loops: columns [lo, hi) x rows [rlo, rhi) of the filter (and, for the transposed
        // gather, the residue classes that land on a source pixel) -> mask bit r * kw + s
        int by, bx, lo, hi, rlo, rhi, rx = 0, ry = 0;
        if (p.gather == 0) {
          by = oy * p.sh - p.pt;
          bx = ox * p.sw - p.pl;
          lo = max(0, -bx);
          hi = min((int)p.kw, (int)p.SW - bx);
          rlo = max(0, -by);
          rhi = min((int)kh, (int)p.SH - by);
        } else {
          const int ty = oy + p.pt, tx = ox + p.pl;
          by = ty / p.sh;
          bx = tx / p.sw;
          ry = ty - by * p.sh;
          rx = tx - bx * p.sw;
          lo = max(0, bx - (int)p.SW + 1) * p.sw;
          hi = min((int)p.kw, (bx + 1) * p.sw);
          rlo = max(0, by - (int)p.SH + 1) * p.sh;
          rhi = min((int)kh, (by + 1) * p.sh);
        }
        const uint32_t colbits = hi > lo ? (((1u << hi) - (1u << lo)) & p.cmask[rx]) : 0u;
        unsigned long long mk = 0ull;
        if (rhi > rlo) {
          const int b0 = rlo * (int)p.kw, b1 = rhi * (int)p.kw;
          const unsigned long long range = (b1 >= 64 ? ~0ull : ((1ull << b1) - 1ull)) & ~((1ull << b0) - 1ull);
          mk = (unsigned long long)colbits * (p.rspread[ry] & range);
        }
        mask[i] = m < p.M ? mk : 0ull;   // rows beyond M and padding taps: zero-filled (no global access at size 0)
        base[i] = p.src + ((long long)img * p.SH * p.SW + (long long)by * (int)p.SW + bx) * (long long)p.C + cc * 16;
      }
      for (uint32_t st = 0; st < p.stages_per_tile; ++st) {
        ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag, &g_ldg_error);
        if (!ok) break;
        const uint32_t dst0 = smem_u32(sA + (size_t)stage * kStageBytes) + cc * (kBlockM * 16) + rloc0 * 16;
        int dl[TPS];
#pragma unroll
        for (int tl = 0; tl < TPS; ++tl) dl[tl] = s_tab[st * TPS + tl].x;
        // tap slot index == tap index: the stage's validity bits are a window of the row's mask (padding slots are 0)
        uint32_t bits[CPP];
#pragma unroll
        for (int i = 0; i < CPP; ++i) bits[i] = (uint32_t)(mask[i] >> (st * TPS));
#pragma unroll
        for (int tl = 0; tl < TPS; ++tl) {
          if ((st * TPS + tl) * CPP < p.KCp) {  // warp-uniform: slots beyond the tile's chunks copy nothing
#pragma unroll
            for (int i = 0; i < CPP; ++i)
              cp_async16(dst0 + tl * (CPP * kBlockM * 16) + i * (RPI * 16), base[i] + dl[tl], (bits[i] >> tl) & 1u ? 16u : 0u);
          }
        }
        cp_async_arrive_noinc(&full_bar[stage]);
        if (threadIdx.x == 0 && tile == blockIdx.x) dbg_stamp(p, 2 + (st < 5 ? st : 5));
        if (++stage == p.nstages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else if (warp == kLoaderWarps) {
    // ===== MMA issuer =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      bool ok = true;
      const uint32_t sb0 = smem_u32(sB);
      ok = mbar_wait(&b_bar, 0, abort_flag, &g_ldg_error);
      for (uint32_t tile = blockIdx.x; tile < p.m_tiles && ok; tile += gridDim.x) {
        if (!(ok = mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, abort_flag, &g_ldg_error))) break;
        fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        uint32_t first = 1;
        if (HALO) {
          if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag, &g_ldg_error))) break;
          fence_after();
          if (tile == blockIdx.x) dbg_stamp(p, 8);
          if (p.dbg && blockIdx.x == 0 && tile / gridDim.x < 10) dbg_stamp(p, 32 + tile / gridDim.x);
          const uint32_t sa = smem_u32(sA + (size_t)stage * p.stage_bytes);
          const uint32_t sbo = p.sw == 1 ? p.halo_w * 16 : p.sh * p.halo_hw2 * 16;   // next output row of the patch
          for (uint32_t j = 0; j < p.halo_mmas; ++j) {
            const uint2 t = s_mma[j];
            umma_i8(d_tmem, make_desc_k16(sa + t.x, t.y, sbo), make_desc_kmajor(sb0 + 2 * j * (BN * 16), 0, BN * 16), p.idesc,
                    first ? 0u : 1u);
            first = 0;
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == p.nstages) {
            stage = 0;
            phase ^= 1;
          }
        }
        for (uint32_t st = 0; !HALO && st < p.stages_per_tile; ++st) {
          if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag, &g_ldg_error))) break;
          fence_after();
          if (tile == blockIdx.x) dbg_stamp(p, 8 + (st < 5 ? st : 5));
          const uint32_t sa = smem_u32(sA + (size_t)stage * kStageBytes);
          const uint32_t kc0 = st * kChunksPerStage;
          const uint32_t n2 = min((uint32_t)kChunksPerStage, p.KCp - kc0) >> 1;
          for (uint32_t j = 0; j < n2; ++j) {
            umma_i8(d_tmem, make_desc_kmajor(sa + 2 * j * (kBlockM * 16), 0, kBlockM * 16),
                    make_desc_kmajor(sb0 + (kc0 + 2 * j) * (BN * 16), 0, BN * 16), p.idesc, first ? 0u : 1u);
            first = 0;
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == p.nstages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (!ok) break;
        umma_commit(&tmem_full_bar[acc]);
        if (tile == blockIdx.x) dbg_stamp(p, 14);
        if (++acc == kAccStages) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // ===== epilogue warps; first they fetch the resident filter bank (the loaders are already gathering tile 0):
    // chunk kc, output channel n -> 16 bytes (zeros beyond Cout / KC), all copies in flight at once =====
    for (uint32_t i = threadIdx.x - 32 * (kLoaderWarps + 1); i < p.KCp * BN; i += 32 * kEpiWarps) {
      const uint32_t kp = i / BN, n = i % BN;
      const int kc = HALO ? (int)s_kmap[kp] : (kp < p.KC ? (int)kp : -1);
      const bool v = kc >= 0 && n < p.N;
      cp_async16(smem_u32(sB + (size_t)i * 16), v ? p.wp + (size_t)n * p.ldw + (size_t)kc * 16 : p.wp, v ? 16u : 0u);
    }
    cp_async_arrive_noinc(&b_bar);
    // TMEM lane quadrant = warp % 4
    const uint32_t quad = warp & 3;
    const uint32_t half = (uint32_t)(warp - (kLoaderWarps + 1)) >> 2;  // which of the quadrant's kSub warps
    int e = p.exp_const;
    if (p.ibA) e += *p.ibA;
    if (p.ibB) e += *p.ibB;
    const float scale = exp2i(e);
    const bool fused = p.bnq.q.bits != 0;
    int* my_stat = s_stat[warp - (kLoaderWarps + 1)];
    BnqState bst;
    bst.tiles = 0;
    if (fused) {
      bst.init(p.bnq);
      for (int i = lane; i < kStats * BN; i += 32) my_stat[i] = 0;
      __syncwarp();
    }
    uint32_t acc = 0, acc_phase = 0, tcount = 0;
    bool ok = true;
    constexpr bool kByTile = BN <= 32;   // one 16/32-column group per tile: split the TILES between the quadrant's warps
    for (uint32_t tile = blockIdx.x; tile < p.m_tiles && ok; tile += gridDim.x, ++tcount) {
      if (kByTile && (tcount & 1u) != half) {   // the other warp of this quadrant drains this accumulator
        if (++acc == kAccStages) {
          acc = 0;
          acc_phase ^= 1;
        }
        continue;
      }
      uint32_t row, pix;
      bool rvalid;
      if (HALO) {   // accumulator row m = 8 * (row of the patch) + column of the patch
        const uint32_t m = quad * 32 + lane;
        const uint32_t img = fastdiv(tile, p.d_tiles_img), t2 = tile - img * p.d_tiles_img.d;
        const uint32_t ty = fastdiv(t2, p.d_tiles_x), tx = t2 - ty * p.d_tiles_x.d;
        const uint32_t oy = ty * 16 + (m >> 3), ox = tx * 8 + (m & 7);
        rvalid = oy < p.OH && ox < p.OW;
        pix = oy * p.OW + ox;
        row = img * p.OHW + pix;
      } else {
        row = tile * kBlockM + quad * 32 + lane;
        pix = fused ? row - fast_div(row, p.OHW, p.ohw_mul, p.ohw_shr) * p.OHW : 0u;   // row % (OH*OW)
        rvalid = row < p.M;
      }
      constexpr int G = BN >= 64 ? 16 : (BN < 32 ? BN : 32);  // columns fetched from tensor memory per wait (wide tiles: 16, register budget)
      constexpr bool kSplit = BN > G;       // wide tiles: both warps of a quadrant alternate the G-column groups
      if (fused) {   // this warp's noise lines of the tile: into L1 while the accumulator is still being computed
#pragma unroll 1
        for (int c0 = kSplit ? G * (int)half : 0; c0 < BN; c0 += kSplit ? kSub * G : G)
#pragma unroll
          for (int q = 0; q < G / 16; ++q) bnq_prefetch(p.bnq, pix, p.N, (uint32_t)(c0 + 16 * q), rvalid && (uint32_t)(c0 + 16 * q) < p.N);
      }
      ok = mbar_wait(&tmem_full_bar[acc], acc_phase, abort_flag, &g_ldg_error);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      fence_after();
      if (threadIdx.x == 32 * (kLoaderWarps + 1) && tile == blockIdx.x) dbg_stamp(p, 15);
      const uint32_t taddr = tmem_base + acc * BN + ((quad * 32u) << 16);
      if (fused && bst.tiles >= (uint32_t)kBnqFlushTiles) {
        bnq_flush(p.bnq, my_stat, 0, BN, p.N, lane);
        bst.tiles = 0;
      }
      ++bst.tiles;
#pragma unroll 1
      for (int c0 = kSplit ? G * (int)half : 0; c0 < BN; c0 += kSplit ? kSub * G : G) {
        uint32_t vv[G / 16][16];
#pragma unroll
        for (int q = 0; q < G / 16; ++q) tmem_ld16(taddr + c0 + 16 * q, vv[q]);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < G / 16; ++q) {
          const int c = c0 + 16 * q;
          if ((uint32_t)c >= p.N) continue;  // warp-uniform
          const uint32_t ncol = min(16u, p.N - (uint32_t)c);
          if (fused) {
            bnq_chunk<EPI != 16>(p.bnq, bst, vv[q], scale, p.bias ? p.bias + c : nullptr, row, pix, rvalid, (uint32_t)c, ncol, p.N, my_stat,
                                 BN, (uint32_t)c, lane);   // the loader-paced 16-warp instantiation keeps the run-time fold test (qsite.cuh)
            continue;
          }
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = __int2float_rn((int)vv[q][j]) * scale;
          if (p.bias) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < (int)ncol) f[j] = __fadd_rn(f[j], __ldg(p.bias + c + j));
          }
          if (rvalid) {
            float* o = p.out + (size_t)row * p.ldc + c;
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
      }
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      if (threadIdx.x == 32 * (kLoaderWarps + 1) && tile == blockIdx.x) dbg_stamp(p, 16);
      if (p.dbg && (warp & 3) == ((kLoaderWarps + 1) & 3) && lane == 0 && tcount < 10) dbg_stamp(p, 20 + tcount);
      if (++acc == kAccStages) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (fused && ok) {
      bnq_flush_cta(p.bnq, my_stat, s_tot, 0, BN, p.N, lane, threadIdx.x - 32 * (kLoaderWarps + 1), 32 * kEpiWarps, 1);
      bnq_finish(p.bnq, bst, (unsigned long long)p.M * p.N, warp == kLoaderWarps + 1, lane);
    }
  }

  fence_before();
  __syncthreads();
  fence_after();
  if (threadIdx.x == 0) dbg_stamp(p, 17);
  if (warp == kLoaderWarps) tmem_dealloc(tmem_base, kTmemCols);
  if (threadIdx.x == 32 * kLoaderWarps) dbg_stamp(p, 18);
}

template <int BN, int CPP, bool HALO, int EPI>
int launch_ldg3(const LdgParams& p, unsigned grid, size_t smem, cudaStream_t st) {
  static size_t attr_smem[16] = {};
  const int dev = device_info().device;
  if (attr_smem[dev] < smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_ldg_kernel<BN, CPP, HALO, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(conv_ldg_kernel)");
      return LBT_ECUDA;
    }
    attr_smem[dev] = smem;
  }
  launch_pdl(conv_ldg_kernel<BN, CPP, HALO, EPI>, grid, 32 * (kLoaderWarps + 1 + EPI), smem, st, p);
  return check_launch("lbt_conv_i8 (cp.async gather)");
}

// p.epi16: one CTA per SM (big filter bank) with a halo loader and a wide tile -> the 16-epilogue-warp instantiation
template <int BN, int CPP, bool HALO>
int launch_ldg2(const LdgParams& p, unsigned grid, size_t smem, cudaStream_t st) {
  if constexpr (HALO && BN >= 64) {
    if (p.epi16) return launch_ldg3<BN, CPP, HALO, 16>(p, grid, smem, st);
  }
  return launch_ldg3<BN, CPP, HALO, 8>(p, grid, smem, st);
}

template <int BN, bool HALO>
int launch_ldg1(const LdgParams& p, unsigned grid, size_t smem, cudaStream_t st) {
  switch (p.cpp) {
    case 1: return launch_ldg2<BN, 1, HALO>(p, grid, smem, st);
    case 2: return launch_ldg2<BN, 2, HALO>(p, grid, smem, st);
    default: return launch_ldg2<BN, 4, HALO>(p, grid, smem, st);
  }
}

template <int BN>
int launch_ldg(const LdgParams& p, unsigned grid, size_t smem, cudaStream_t st, bool halo) {
  return halo ? launch_ldg1<BN, true>(p, grid, smem, st) : launch_ldg1<BN, false>(p, grid, smem, st);
}

// ------------------------------------------------------------------------------------------------------------------
// Weight gradient for narrow channels: acc64[(tap, c), co] += alpha * sum over output pixels of X[pixel + tap, c] * G[pixel, co]
// (tf.gradients(y, W, gradq), dynamic_fixed_point.py:302).  The reduction runs over pixels, so a pipeline stage is one
// block of 128 output pixels: the loader warps gather every tap of X ([KC chunk planes][128 pixels][16 B]) and the
// gradient rows ([Cout/16 planes][128 pixels][16 B]) once, and the tensor core consumes both MN-major (planes = groups of
// 16 M/N indices, pixels = K): all MT = ceil(KC/8) M tiles accumulate in tensor memory across the CTA's pixel blocks, and
// one epilogue at the end adds the s32 partials into the int64 sums.  Unlike the TMA kernel (which re-reads X per M tile
// and pays the 3-clock-per-row TMA rate on 16-byte rows) every pixel block is loaded exactly once.
// ------------------------------------------------------------------------------------------------------------------
struct WgLdgParams {
  const uint8_t* x;
  const uint8_t* g;
  uint32_t Mpix, Cout;
  uint32_t SH, SW, C;
  uint32_t OW, OHW;
  uint32_t ohw_mul, ohw_shr, ow_mul, ow_shr;
  int sh, sw, pt, pl;
  uint32_t kw, taps, cpp, np;       // filter width, kh*kw, C/16, Cout/16
  uint32_t KC, MT;                  // chunk planes of X per stage, M tiles
  uint32_t a_planes;                // 8 * MT
  uint32_t stage_bytes, nstages;
  uint32_t pix_blocks;
  uint32_t Kf;
  unsigned long long rspread;       // sum over filter rows of 1 << (r * kw)
  long long* acc64;
  int alpha;
  uint32_t idesc;
  uint32_t tmem_cols;
};

template <int CPP>
__global__ void __launch_bounds__(32 * (kLoaderWarps + 1 + 4), 2) conv_wgrad_ldg_kernel(const WgLdgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
  __shared__ __align__(8) uint64_t full_bar[kMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
  __shared__ __align__(8) uint64_t done_bar;
  __shared__ uint32_t tmem_slot;
  __shared__ int s_abort;
  __shared__ int s_delta[kMaxTaps];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (uint32_t s = 0; s < p.nstages; ++s) {
      mbar_init(&full_bar[s], kLoaderWarps * 32);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&done_bar, 1);
    s_abort = 0;
    fence_barrier_init();
  }
  if (warp == kLoaderWarps) tmem_alloc(&tmem_slot, p.tmem_cols);
  for (uint32_t ts = threadIdx.x; ts < p.taps; ts += blockDim.x)
    s_delta[ts] = ((int)(ts / p.kw) * (int)p.SW + (int)(ts % p.kw)) * (int)p.C;
  pdl_trigger();
  fence_before();
  __syncthreads();
  fence_after();
  pdl_wait();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);
  volatile int* abort_flag = &s_abort;
  const uint32_t kh = p.taps / p.kw;
  const uint32_t b_off = p.a_planes * (kBlockM * 16);  // gradient planes follow the X planes inside a stage

  if (warp < kLoaderWarps) {
    constexpr int RPI = 32 / CPP;
    const uint32_t cc = lane % CPP;
    const uint32_t rloc0 = warp * 32 + lane / CPP;
    const uint32_t grow = threadIdx.x;  // the gradient row this thread copies
    uint32_t stage = 0, phase = 0;
    bool ok = true;
    for (uint32_t pb = blockIdx.x; pb < p.pix_blocks && ok; pb += gridDim.x) {
      unsigned long long mask[CPP];
      const uint8_t* base[CPP];
#pragma unroll
      for (int i = 0; i < CPP; ++i) {
        const uint32_t m = pb * kBlockM + rloc0 + i * RPI;
        const uint32_t img = fast_div(m, p.OHW, p.ohw_mul, p.ohw_shr), rem = m - img * p.OHW;
        const uint32_t oyu = fast_div(rem, p.OW, p.ow_mul, p.ow_shr);
        const int by = (int)oyu * p.sh - p.pt, bx = (int)(rem - oyu * p.OW) * p.sw - p.pl;
        const int lo = max(0, -bx), hi = min((int)p.kw, (int)p.SW - bx);
        const int rlo = max(0, -by), rhi = min((int)kh, (int)p.SH - by);
        const uint32_t colbits = hi > lo ? ((1u << hi) - (1u << lo)) : 0u;
        unsigned long long mk = 0ull;
        if (rhi > rlo) {
          const int b0 = rlo * (int)p.kw, b1 = rhi * (int)p.kw;
          const unsigned long long range = (b1 >= 64 ? ~0ull : ((1ull << b1) - 1ull)) & ~((1ull << b0) - 1ull);
          mk = (unsigned long long)colbits * (p.rspread & range);
        }
        mask[i] = m < p.Mpix ? mk : 0ull;
        base[i] = p.x + ((long long)img * p.SH * p.SW + (long long)by * (int)p.SW + bx) * (long long)p.C + cc * 16;
      }
      ok = mbar_wait(&empty_bar[stage], phase ^ 1, abort_flag, &g_ldg_error);
      if (!ok) break;
      const uint32_t st0 = smem_u32(smem + (size_t)stage * p.stage_bytes);
      const uint32_t dst0 = st0 + cc * (kBlockM * 16) + rloc0 * 16;
#pragma unroll 2
      for (uint32_t ts = 0; ts < p.taps; ++ts) {
        const int d = s_delta[ts];
#pragma unroll
        for (int i = 0; i < CPP; ++i)
          cp_async16(dst0 + ts * (CPP * kBlockM * 16) + i * (RPI * 16), base[i] + d, (mask[i] >> ts) & 1ull ? 16u : 0u);
      }
      {  // gradient rows: thread t copies the Cout bytes of pixel t into the np planes
        const uint32_t m = pb * kBlockM + grow;
        const bool v = m < p.Mpix;
        const uint8_t* src = p.g + (size_t)(v ? m : 0) * p.Cout;
        const uint32_t dstb = st0 + b_off + grow * 16;
        for (uint32_t j = 0; j < p.np; ++j) cp_async16(dstb + j * (kBlockM * 16), src + j * 16, v ? 16u : 0u);
      }
      cp_async_arrive_noinc(&full_bar[stage]);
      if (++stage == p.nstages) {
        stage = 0;
        phase ^= 1;
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else if (warp == kLoaderWarps) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      bool ok = true, first = true;
      for (uint32_t pb = blockIdx.x; pb < p.pix_blocks && ok; pb += gridDim.x) {
        if (!(ok = mbar_wait(&full_bar[stage], phase, abort_flag, &g_ldg_error))) break;
        fence_after();
        const uint32_t sa = smem_u32(smem + (size_t)stage * p.stage_bytes);
        const uint32_t sb = sa + b_off;
        for (uint32_t mt = 0; mt < p.MT; ++mt)
#pragma unroll
          for (uint32_t kk = 0; kk < kBlockM / 32; ++kk)
            umma_i8(tmem_base + mt * p.Cout, make_desc_mnmajor(sa + mt * 8 * (kBlockM * 16) + kk * 32 * 16, 0, kBlockM * 16),
                    make_desc_mnmajor(sb + kk * 32 * 16, 0, kBlockM * 16), p.idesc, (first && kk == 0) ? 0u : 1u);
        first = false;
        umma_commit(&empty_bar[stage]);
        if (++stage == p.nstages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (ok) umma_commit(&done_bar);
    }
  } else {
    // ===== epilogue (once): s32 partials -> int64 sums =====
    const uint32_t quad = warp & 3;
    const bool has_work = blockIdx.x < p.pix_blocks;
    bool ok = has_work && mbar_wait(&done_bar, 0, abort_flag, &g_ldg_error);
    ok = __all_sync(0xffffffffu, ok);
    if (ok) {
      fence_after();
      for (uint32_t mt = 0; mt < p.MT; ++mt) {
        const uint32_t kf = mt * kBlockM + quad * 32 + lane;
        for (uint32_t c = 0; c < p.Cout; c += 16) {
          uint32_t v[16];
          tmem_ld16(tmem_base + mt * p.Cout + c + ((quad * 32u) << 16), v);
          tmem_ld_wait();
          if (kf < p.Kf) {
            unsigned long long* o = reinterpret_cast<unsigned long long*>(p.acc64) + (size_t)kf * p.Cout + c;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const long long a = (long long)(int)v[j] * (long long)p.alpha;
              if (a != 0) atomicAdd(o + j, (unsigned long long)a);
            }
          }
        }
      }
    }
  }
  fence_before();
  __syncthreads();
  fence_after();
  if (warp == kLoaderWarps) tmem_dealloc(tmem_base, p.tmem_cols);
}

template <int CPP>
int launch_wgrad_ldg(const WgLdgParams& p, unsigned grid, size_t smem, cudaStream_t st) {
  static size_t attr_smem[16] = {};
  const int dev = device_info().device;
  if (attr_smem[dev] < smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_ldg_kernel<CPP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_cuda_error(e, "cudaFuncSetAttribute(conv_wgrad_ldg_kernel)");
      return LBT_ECUDA;
    }
    attr_smem[dev] = smem;
  }
  launch_pdl(conv_wgrad_ldg_kernel<CPP>, grid, 32 * (kLoaderWarps + 1 + 4), smem, st, p);
  return check_launch("lbt_conv_i8_wgrad (cp.async gather)");
}

}  // namespace


std::atomic<int> g_use_ldg{1};
std::atomic<int> g_use_halo{1};   // lbt_conv_set_halo(): 0 = gather the im2col rows even where the halo patch applies
std::atomic<unsigned long long*> g_dbg{nullptr};
bool conv_ldg_enabled() { return g_use_ldg.load(std::memory_order_relaxed) != 0; }
std::atomic<int> g_halo_any_fill{0};   // test knob: take the halo loader whatever fraction of the 8 x 16 patches lies outside the image
std::atomic<int> g_c64_halo{0};   // measured: ResNet-18's 64-channel layers lose 4 % in the step against the TMA kernel (the microbench gains 15 %)
int conv_ldg_c64_halo() { return g_c64_halo.load(std::memory_order_relaxed); }

// Shapes this kernel takes.
// Halo-patch loader: stride-1 gather of a filter up to 5x5 on images that fill 8 x 16 output patches reasonably (<= 35 % of
// the patch pixels outside the image).
bool conv_ldg_halo_applies(int N, int OH, int OW, int kh, int kw, int sh, int sw, int C) {
  if (!g_use_halo.load(std::memory_order_relaxed) || kh * kw <= 1) return false;
  const bool s1 = sh == 1 && sw == 1 && kh <= 5 && kw <= 5;
  const bool s2 = sh == 2 && sw == 2 && C == 16 && kh <= 8 && kw <= 8 && kh * kw <= kMaxTaps;   // the 7x7/2 stem on 16-byte pixels
  if (!s1 && !s2) return false;
  const uint64_t tx = (uint64_t)(OW + 7) / 8, ty = (uint64_t)(OH + 15) / 16;
  const bool fill_ok = g_halo_any_fill.load(std::memory_order_relaxed) || tx * 8 * ty * 16 * 100 <= (uint64_t)OH * OW * 135;
  return fill_ok && (uint64_t)N * tx * ty < (1ull << 31);
}

bool conv_ldg_ok(int C, int Cout, int kh, int kw) {
  if (C != 16 && C != 32 && C != 64) return false;
  if (Cout < 1 || Cout > 128) return false;
  const size_t kc = (size_t)kh * kw * (C / 16);
  const size_t kcp = (kc + 1) & ~(size_t)1;
  const int bn = Cout <= 16 ? 16 : (Cout <= 32 ? 32 : (Cout <= 64 ? 64 : 128));
  return kcp * bn * 16 + 2 * kStageBytes + 1024 <= 200 * 1024 && (size_t)kh * kw * C <= 65536 && kcp <= (size_t)kMaxKC &&
         kh * kw <= kMaxTaps && kw <= 16 && kh <= 16;
}

// Shapes the gather wgrad kernel takes: all M tiles of the filter must fit tensor memory next to each other.
bool conv_wgrad_ldg_ok(int C, int Cout, int kh, int kw) {
  if (C != 16 && C != 32 && C != 64) return false;
  if (Cout != 16 && Cout != 32 && Cout != 64 && Cout != 128) return false;
  if (kh * kw > kMaxTaps || kw > 16 || kh > 16) return false;
  const int kc = kh * kw * (C / 16), mt = (kc + 7) / 8;
  if (mt * Cout > 512) return false;
  const size_t stage = (size_t)(8 * mt + Cout / 16) * kBlockM * 16;
  return 2 * stage + 1024 <= 200 * 1024;
}

int conv_wgrad_ldg_run(const void* src, int src_kind, int N, int H, int W, int C, const void* g, int g_kind, int Cout, int kh, int kw,
                       int sh, int sw, int pt, int pl, int OH, int OW, int64_t* acc64, int alpha, void* stream) {
  const DeviceInfo& di = device_info();
  if ((size_t)N * OH * OW >= (1ull << 31)) return LBT_EUNSUPPORTED;
  WgLdgParams p{};
  p.x = reinterpret_cast<const uint8_t*>(src);
  p.g = reinterpret_cast<const uint8_t*>(g);
  p.Mpix = (uint32_t)((size_t)N * OH * OW);
  p.Cout = (uint32_t)Cout;
  p.SH = (uint32_t)H;
  p.SW = (uint32_t)W;
  p.C = (uint32_t)C;
  p.OW = (uint32_t)OW;
  p.OHW = (uint32_t)(OH * OW);
  auto magic = [](uint32_t d, uint32_t& mul, uint32_t& shr) {
    if (d <= 1) {
      mul = 0;
      shr = 0;
      return;
    }
    uint32_t lg = 0;
    while ((1ull << lg) < d) ++lg;
    const uint32_t pw = 31 + lg;
    mul = (uint32_t)(((1ull << pw) + d - 1) / d);
    shr = pw - 32;
  };
  magic(p.OHW, p.ohw_mul, p.ohw_shr);
  magic(p.OW, p.ow_mul, p.ow_shr);
  p.sh = sh;
  p.sw = sw;
  p.pt = pt;
  p.pl = pl;
  p.kw = (uint32_t)kw;
  p.taps = (uint32_t)(kh * kw);
  p.cpp = (uint32_t)C / 16;
  p.np = (uint32_t)Cout / 16;
  p.KC = p.taps * p.cpp;
  p.MT = (p.KC + 7) / 8;
  p.a_planes = 8 * p.MT;
  p.stage_bytes = (p.a_planes + p.np) * kBlockM * 16;
  p.pix_blocks = (p.Mpix + kBlockM - 1) / kBlockM;
  p.Kf = (uint32_t)(kh * kw * C);
  for (int r = 0; r < kh; ++r) p.rspread |= 1ull << (r * kw);
  p.acc64 = reinterpret_cast<long long*>(acc64);
  p.alpha = alpha;
  p.idesc = tc::make_idesc_i8(src_kind == LBT_MANT_S8, g_kind == LBT_MANT_S8, true, true, Cout, kBlockM);
  uint32_t cols = 32;
  while (cols < p.MT * p.Cout) cols <<= 1;
  p.tmem_cols = cols;
  const bool two = cols <= 256 && 2 * (size_t)p.stage_bytes + 1024 <= 100 * 1024;
  size_t budget = (two ? 108 * 1024 : 200 * 1024) - 1024;
  uint32_t nst = (uint32_t)(budget / p.stage_bytes);
  if (nst > (uint32_t)kMaxStages) nst = kMaxStages;
  if (nst < 2) return LBT_EUNSUPPORTED;
  p.nstages = nst;
  const size_t smem = (size_t)nst * p.stage_bytes + 256;
  const uint64_t cap = (uint64_t)di.sm_count * (two ? 2u : 1u);
  unsigned grid = (unsigned)(p.pix_blocks < cap ? p.pix_blocks : cap);
  // one CTA may sum at most max_products(src_kind, g_kind) products per s32 accumulator: 512 pixel blocks, 256 for u8 x u8
  if ((p.pix_blocks + grid - 1) / grid > max_products(src_kind, g_kind) / kBlockM) return LBT_EUNSUPPORTED;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (p.cpp) {
    case 1: return launch_wgrad_ldg<1>(p, grid, smem, st);
    case 2: return launch_wgrad_ldg<2>(p, grid, smem, st);
    default: return launch_wgrad_ldg<4>(p, grid, smem, st);
  }
}

// Shared by lbt_conv_i8_fprop (gather 0) and lbt_conv_i8_dgrad (gather 1).  (M rows) x (Cout columns); the gathered
// tensor is src[N, SH, SW, C]; the output grid is OH x OW per image.
int conv_ldg_run(const void* src, int src_kind, int N, int SH, int SW, int C, const void* wp, int w_kind, size_t ldw, int Cout,
                 int kh, int kw, int sh, int sw, int pt, int pl, int OH, int OW, int gather, const int32_t* ibA,
                 const int32_t* ibB, int exp_const, const float* bias, float* out, size_t ldc, const lbt_qsite* q_out,
                 int8_t* k_out, int64_t* sums, const float* addend, void* stream) {
  const DeviceInfo& di = device_info();
  const int bn = Cout <= 16 ? 16 : (Cout <= 32 ? 32 : (Cout <= 64 ? 64 : 128));
  if ((size_t)N * OH * OW >= (1ull << 31)) return LBT_EUNSUPPORTED;
  LdgParams p{};
  p.src = reinterpret_cast<const uint8_t*>(src);
  p.wp = reinterpret_cast<const uint8_t*>(wp);
  p.ldw = (uint32_t)ldw;
  p.M = (uint32_t)((size_t)N * OH * OW);
  p.N = (uint32_t)Cout;
  p.SH = (uint32_t)SH;
  p.SW = (uint32_t)SW;
  p.C = (uint32_t)C;
  p.OW = (uint32_t)OW;
  p.OHW = (uint32_t)(OH * OW);
  auto magic = [](uint32_t d, uint32_t& mul, uint32_t& shr) {   // CUTLASS FastDivmod: valid for n < 2^31
    if (d <= 1) {
      mul = 0;
      shr = 0;
      return;
    }
    uint32_t lg = 0;
    while ((1ull << lg) < d) ++lg;
    const uint32_t pw = 31 + lg;
    mul = (uint32_t)(((1ull << pw) + d - 1) / d);
    shr = pw - 32;
  };
  magic(p.OHW, p.ohw_mul, p.ohw_shr);
  magic(p.OW, p.ow_mul, p.ow_shr);
  for (int j = 0; j < 4; ++j) {
    p.cmask[j] = 0;
    p.rspread[j] = 0;
  }
  if (gather == 0) {
    p.cmask[0] = 0xffffffffu;
    for (int r = 0; r < kh; ++r) p.rspread[0] |= 1ull << (r * kw);
  } else {
    if (sh > 4 || sw > 4) return LBT_EUNSUPPORTED;
    for (int sx = 0; sx < kw; ++sx) p.cmask[sx % sw] |= 1u << sx;
    for (int r = 0; r < kh; ++r) p.rspread[r % sh] |= 1ull << (r * kw);
  }
  p.sh = sh;
  p.sw = sw;
  p.pt = pt;
  p.pl = pl;
  p.kw = (uint32_t)kw;
  p.taps = (uint32_t)(kh * kw);
  p.cpp = (uint32_t)C / 16;
  p.KC = p.taps * p.cpp;
  p.KCp = (p.KC + 1) & ~1u;
  p.stages_per_tile = (p.KCp + kChunksPerStage - 1) / kChunksPerStage;
  p.m_tiles = (p.M + kBlockM - 1) / kBlockM;
  p.gather = gather;
  p.ibA = ibA;
  p.ibB = ibB;
  p.exp_const = exp_const;
  p.bias = bias;
  p.addend = q_out ? nullptr : addend;
  p.out = out;
  p.ldc = ldc;
  p.idesc = tc::make_idesc_i8(src_kind == LBT_MANT_S8, w_kind == LBT_MANT_S8, false, false, bn, kBlockM);
  p.bnq.q = site_from_abi(q_out);
  p.bnq.k = k_out;
  p.bnq.sums = reinterpret_cast<long long*>(sums);
  p.bnq.rows_per_image = (uint32_t)(OH * OW);
  p.dbg = g_dbg.load(std::memory_order_relaxed);
  // halo mode: every input pixel is copied to shared memory ~1.4 times instead of kh * kw times
  p.OH = (uint32_t)OH;
  p.n_img = (uint32_t)N;
  p.stage_bytes = kStageBytes;
  bool halo = false;
  if (gather == 0 && conv_ldg_halo_applies(N, OH, OW, kh, kw, sh, sw, C)) {
    const uint32_t tx = (uint32_t)(OW + 7) / 8, ty = (uint32_t)(OH + 15) / 16;
    halo = true;
    const uint32_t halo_h = 15u * (uint32_t)sh + (uint32_t)kh;
    p.halo_w = 7u * (uint32_t)sw + (uint32_t)kw;
    p.halo_w = (p.halo_w + (uint32_t)sw - 1) / (uint32_t)sw * (uint32_t)sw;          // whole column-parity groups
    p.halo_px = p.halo_w * halo_h;
    p.halo_plane = p.halo_px * 16;
    p.halo_hw2 = p.halo_w / (uint32_t)sw;
    p.halo_par_plane = halo_h * p.halo_hw2 * 16;
    p.d_halo_w = make_fastdiv(p.halo_w);
    if (sw == 1) {
      p.halo_mmas = p.KCp >> 1;
    } else {   // taps (r, s), (r, s + 2) per instruction: see the kernel
      const uint32_t n0 = ((uint32_t)kw + 1) / 2, n1 = (uint32_t)kw / 2;
      p.halo_mmas = (uint32_t)kh * ((n0 + 1) / 2 + (n1 + 1) / 2);
      p.KCp = 2 * p.halo_mmas;
      if (p.KCp > (uint32_t)kMaxKC) return LBT_EUNSUPPORTED;
    }
    p.stage_bytes = ((p.cpp * p.halo_plane + 64) + 127) & ~127u;   // + slack: the padding chunk of an odd tap count
    p.d_tiles_img = make_fastdiv(tx * ty);
    p.d_tiles_x = make_fastdiv(tx);
    p.m_tiles = (uint32_t)N * tx * ty;
    p.stages_per_tile = 1;
  }
  const size_t b_bytes = (((size_t)p.KCp * bn * 16) + 127) & ~(size_t)127;
  // ring depth: two CTAs per SM when the filter bank is small, else one CTA with a deep ring
  const bool two = b_bytes <= 44 * 1024;
  size_t budget = (two ? 108 * 1024 : 200 * 1024) - b_bytes - 1024;
  uint32_t nst = (uint32_t)(budget / p.stage_bytes);
  if (nst > (uint32_t)kMaxStages) nst = kMaxStages;
  if (nst < 2) return LBT_EUNSUPPORTED;
  p.nstages = nst;
  size_t smem = b_bytes + (size_t)nst * p.stage_bytes + 256;
  const unsigned ctas_per_sm = two ? 2u : 1u;
  p.epi16 = (!two && halo && bn >= 64) ? 1 : 0;
  if (p.epi16 && smem < 120 * 1024) smem = 120 * 1024;   // that instantiation owns up to all 512 TMEM columns: never two per SM
  const uint64_t cap = (uint64_t)di.sm_count * ctas_per_sm;
  const unsigned grid = (unsigned)(p.m_tiles < cap ? p.m_tiles : cap);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (bn) {
    case 16: return launch_ldg<16>(p, grid, smem, st, halo);
    case 32: return launch_ldg<32>(p, grid, smem, st, halo);
    case 64: return launch_ldg<64>(p, grid, smem, st, halo);
    default: return launch_ldg<128>(p, grid, smem, st, halo);
  }
}

}  // namespace lbt

using namespace lbt;

extern "C" int lbt_conv_i8_dgrad(const void* g, int g_kind, int N, int OH, int OW, int Cout, const void* wp, int w_kind, size_t ldw,
                                 int Cin, int kh, int kw, int sh, int sw, int pad_top, int pad_left, int H, int W,
                                 const int32_t* ib_g, const int32_t* ib_w, int exp_const, float* dx, size_t ldc, const float* addend,
                                 void* stream) {
  if (!g || !wp || !dx) return LBT_EINVAL;
  if ((g_kind != LBT_MANT_S8 && g_kind != LBT_MANT_U8) || (w_kind != LBT_MANT_S8 && w_kind != LBT_MANT_U8)) return LBT_EINVAL;
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cout <= 0 || kh <= 0 || kw <= 0 || sh <= 0 || sw <= 0 || OH <= 0 || OW <= 0)
    return LBT_EINVAL;
  if (ldc < (size_t)Cin || ldw < (size_t)kh * kw * Cout) return LBT_EINVAL;
  if ((reinterpret_cast<uintptr_t>(g) & 15) || (reinterpret_cast<uintptr_t>(wp) & 15) || (ldw & 15)) return LBT_EUNSUPPORTED;
  if (!conv_ldg_ok(Cout, Cin, kh, kw)) return LBT_EUNSUPPORTED;
  LBT_REQUIRE_ARCH();
  // rows = input pixels (n, h, w); gathered tensor = g[N, OH, OW, Cout]; output channels = Cin
  return conv_ldg_run(g, g_kind, N, OH, OW, Cout, wp, w_kind, ldw, Cin, kh, kw, sh, sw, pad_top, pad_left, H, W, 1, ib_g, ib_w,
                      exp_const, nullptr, dx, ldc, nullptr, nullptr, nullptr, addend, stream);
}

// Test / bench knob (not in lbt.h): 0 routes every convolution through the TMA-im2col kernel, 1 (default) lets the
// narrow-channel shapes take the cp.async-gather kernel.
extern "C" int lbt_conv_set_path(int use_ldg) {
  g_use_ldg.store(use_ldg ? 1 : 0, std::memory_order_relaxed);
  return LBT_OK;
}

// Test / bench knob (not in lbt.h): bit 0 = use the halo-patch loader of the gather kernel where it applies; bit 1 = also
// route 64-channel inputs to it (otherwise they stay on the TMA im2col kernel).  Default 1.
extern "C" int lbt_conv_set_halo(int mask) {
  g_use_halo.store(mask & 1, std::memory_order_relaxed);
  g_c64_halo.store((mask >> 1) & 1, std::memory_order_relaxed);
  g_halo_any_fill.store((mask >> 2) & 1, std::memory_order_relaxed);   // bit 2: ignore the patch fill-ratio rule (tests)
  conv_halo_enable((((mask >> 3) & 1) ? 0 : 1) | (((mask >> 2) & 1) << 1));                                  // bit 3: 64- / 128-channel layers back on the im2col TMA kernel
  return LBT_OK;
}

// Bench knob (not in lbt.h): device buffer of >= 32 uint64 that receives CTA 0's phase timestamps (globaltimer, ns).
extern "C" int lbt_conv_ldg_set_debug(void* dev_u64) {
  g_dbg.store(reinterpret_cast<unsigned long long*>(dev_u64), std::memory_order_relaxed);
  return LBT_OK;
}

extern "C" int lbt_conv_ldg_debug_error(void) {
  int v = 0, zero = 0;
  if (cudaMemcpyFromSymbol(&v, g_ldg_error, sizeof(int)) != cudaSuccess) return -1;
  cudaMemcpyToSymbol(g_ldg_error, &zero, sizeof(int));
  return v;
}
