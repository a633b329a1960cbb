// conv_tcgen05.cu -- implicit-GEMM convolution on the 5th-generation tensor cores (sm_100a only).
//
// D[m][n] = sum_{tap, ci} A[m + delta(tap)][ci] * W[n][tap][ci]       (bf16 operands, fp32 accumulate in TMEM)
//
// "Shifted-view" formulation.  Every convolution of the U-Net is expressed over a VIRTUAL image addressed by a flat
// pixel index f = img * S + row * Wv + col in which each filter tap is a constant offset delta in f:
//
//   GEO_SAME  3x3 pad 1 : Wv = W+1, S = (H+1)*Wv; row 0 / col 0 of every image block are zero pads SHARED with the
//             (1x1 pad 0)  neighbouring row / image, delta = (ky-1)*Wv + (kx-1).  1x1: Wv = W, S = H*W, delta = 0.
//   GEO_DOWN  Conv k4 s2 p1 == 2x2 stride-1 conv over the shifted space-to-depth image: virtual pixel (u,v) holds the
//             2x2 input patch rows (2u-1, 2u) x cols (2v-1, 2v) as 4*C channels; Wv = W/2+1, delta = du*Wv + dv.
//   GEO_UP    ConvTranspose k4 s2 p1 == four sub-pixel phases (py,px); each phase is a 2x2 conv over the padded input
//             (layout of GEO_SAME 3x3) with its own 4 taps/weights; the phase is folded into the N-tile index.
//   GEO_INIT  7x7 pad 3 stem on the fp32 NCHW sampler state: the kx direction is packed into channels
//             (virtual channel = kx*Cin + ch, 7*Cin <= 32), 3 zero rows shared between images, delta = (ky-3)*W.
//
// A tile is 256 (or 128) consecutive flat positions x one N tile (two / one 128-row accumulators).  Its input window is
// loaded ONCE per 32-channel pass into shared memory; the operand of tap t is the same buffer with the start address advanced
// by delta rows: all taps of a k-step read one resident tile and nothing is re-fetched from L2.  Two operand feeds:
//   TMA (ATMA instantiations: the hot 128-column 3x3 / 1x1 / k4s2 / transposed convs): ONE cp.async.bulk.tensor im2col copy per
//     pass -- the tensor map's traversal order over (w, h, n) with the pad row / column inside its bounding box IS the flat padded
//     position order, out-of-tensor positions arrive as zeros -- into a SWIZZLE_64B tile [P rows][64 B]; tap t = start address
//     + delta * 64 B (the swizzle is keyed on absolute address bits, buffers are 1 KB aligned, so any row offset works).  The
//     GroupNorm prologue (GroupNorm-apply of the producing conv, SiLU, time-embedding add) transforms the landed tile in place.
//     Measured: 16-byte global -> shared transfers run at 16 B/clk/SM however they are issued, TMA rows of 64 B at 42 B/clk/SM
//     (tools/micro/), which is what had capped the engine.
//   cp.async (everything else: N tiles of 32 / 64, FiLM, residual / fold epilogues, the stem): the producer warps gather 16-byte
//     items into the UMMA K-major, no-swizzle canonical layout
//       A_smem[kchunk (8 channels = 16 B)][pixel]      (LBO = PA*16 B between k-chunks, SBO = 128 B between 8-row groups)
//     (tap t = start address + delta * 16 B) and apply the prologue to their own items one pass later.
// Weights are pre-blocked on the host into
// [n_tile][pass][tap][kchunk][n] 16-byte items and streamed with 1-D bulk async copies (cp.async.bulk -> UBLKCP, the TMA
// engine's non-tensor mode) through an mbarrier ring.
//
// PERSISTENT, warp-specialised CTA (one per SM, 576 threads; 832 in the 16-epilogue-warp instantiations), tiles assigned round-robin:
//   warps 0-7   operand producers (global -> prologue transform -> shared), run ahead across tiles (2 operand buffers)
//   warps 8-15  epilogue (TMEM -> registers -> +bias, +residual, GroupNorm statistics, bf16 -> global); two warps per TMEM
//               lane quarter, each taking half of the tile's columns
//   warp 16     weight loader (one lane), warp 17 TMEM allocator + single-thread MMA issuer
// The accumulators are double buffered in TMEM (2 x mt x NT <= 512 columns), so the epilogue of tile i overlaps the main
// loop of tile i+1 and the per-CTA setup is paid once per launch.
//
// The kernel is a template over <geometry, N tile, FiLM prologue, lean issue, rare epilogue terms, prologue mode, epilogue warps,
// swapped operand roles, TMA operand feed>:
// the engine is sensitive to the amount of code around its inner loops, so every launch picks the smallest instantiation that
// covers it (launch<>() below).  profiles/README.md and DESIGN.md record the alternatives that were measured and rejected (more
// producer warps, CTA-pair weight multicast, the block tail behind a grid barrier, ...); their code was removed, git history has it.
//
// Garbage rows: flat positions that fall on a pad column/row are computed and discarded (1 - HW/S of the MMA
// work for 3x3: 6 % at 32x32, 11 % at 16x16, 21 % at 8x8, 36 % at 4x4).
#include <cuda.h>     // CUtensorMap (type and enums only; the encoder is fetched through cudaGetDriverEntryPoint)
#include <array>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "ops.h"
#include "tc_ptx.cuh"

namespace dmn {
namespace tc {

enum { GEO_SAME = 0, GEO_DOWN = 1, GEO_UP = 2, GEO_INIT = 3 };

constexpr int kProdWarps = 8, kEpiWarps = 8;
constexpr int kProdThreads = kProdWarps * 32, kEpiThreads = kEpiWarps * 32;
constexpr int kLoaderWarp = kProdWarps + kEpiWarps, kMmaWarp = kLoaderWarp + 1;
constexpr int kThreads = (kMmaWarp + 1) * 32;     // 576
constexpr int kThreads16 = (kProdWarps + 16 + 2) * 32;   // 832: the 16-epilogue-warp instantiations (template parameter EW)
constexpr int kMTmax = 2;              // 128-row accumulators per tile: 2, or 1 when two would leave most SMs idle
constexpr int kMcta = 128 * kMTmax;    // table sizing
constexpr int kCk = 32;                // channels per pass (4 k-chunks of 8)
constexpr int kStagesMax = 8;          // weight-ring depth (chosen per launch to fit shared memory); one stage = G taps
constexpr int kABuf = 3;               // operand (A) buffers: the producers run up to kABuf passes ahead of the MMA issuer
constexpr int kABufMax = 6;            // barrier-array spacing / host sizing; the 1x1 instantiations use kABufOne buffers
constexpr int kABufPro = 5, kDepthPro = 2;   // GroupNorm-prologue instantiations (PRO = 1): ncu shows 13 % of producer time waiting for the
                                       // copies of the pass issued one iteration earlier; a deeper ring hides it at the price of shared memory
constexpr int kABufOne = 5, kDepthOne = kABufOne - 2;   // 1x1 convs: MMA work per pass is tiny, the producers are
                                       // bound by the global-load latency of the passes they keep in flight
constexpr int kABufPlain = 3, kDepthPlain = 1;   // plain (no prologue) swapped-role instantiations: operand ring and passes in flight
constexpr int kDepth = 1;              // passes a producer thread keeps in flight (cp.async groups) before it finishes the oldest;
                                       // kABuf >= kDepth + 2, else finishing pass c would wait for the MMAs of pass c-1
constexpr int kGS = 3;                 // items of a thread transformed side by side in one basic block (TMA prologue tiles)
// lean (unrolled) issue path: with fewer passes per tile the tile is epilogue-bound and the faster main loop only adds contention
// (level-0 convs 0.078 -> 0.084 ms); the GroupNorm-prologue 3x3 on the TMA feed measured the same threshold (level-0: 0.0843 ms
// looped, 0.0877 ms unrolled)
constexpr int kLeanMinPass = 8;
constexpr size_t kSmemLimit = (size_t)226 * 1024;   // dynamic shared memory per CTA (a CTA may opt in to 227 KB)
constexpr int kMaxItems = 7;           // 16-byte operand items per producer thread per pass (P <= 448)
constexpr int kNimgMax = 20;           // images a 256-position window may touch
constexpr int kGroupsMax = 32;         // GroupNorm groups of the prologue

struct Params {
  ConvP c;
  int geo;
  int S, Wv, pad, halo_lo, P, PA, mt, mcta;
  int H, W, HW;            // input image
  int ksize, ntap, NT, n_pass, tiles_per_phase, n_tiles_n, m_tiles, total_tiles;
  int abuf;                // operand buffers of the instantiation that will be launched (kABuf, or kABufOne for the 1x1 form)
  int n_big_tiles, big_rows, halo_hi;   // tiles [0, n_big_tiles) have 256 rows, the rest 128 rows starting at flat position big_rows
  long total_flat;
  uint32_t lbo_a, sbo_a, lbo_b, sbo_b;   // bytes
  uint32_t tmem_cols;
  int cpg_in, cpg_out, cpg_in_shift, cpg_out_shift, nstage, nt_shift;
  int G, stages_per_pass;  // taps per weight stage, ntap / G
  uint32_t stage_bytes;    // G * 4 * NT * 16
  int delta[64];           // [4 phases][16 taps] tap offsets in flat positions (constant bank => uniform registers in the issuer)
  uint32_t magic_S, magic_W;   // ceil(2^26 / S), ceil(2^24 / Wv): exact small-number division in vdecode_rel
  unsigned long long magic64_S;   // ceil(2^64 / S): f / S == umul64hi(f, magic64_S) for every 32-bit f (the per-tile decodes of the TMA path)
  float inv_cnt_in;
  long long* trace;        // debug timeline (null in production)
  int trace_cta;
  // GEO_INIT extras
  const float* cls_w;
  const int64_t* classes;
  int pad_class;
  // TMA operand path (ATMA instantiations): the window of a pass is ONE cp.async.bulk.tensor im2col copy of P pixels x 32 channels into
  // a SWIZZLE_64B tile [P rows][64 B]; tap offsets / descriptor strides below are then in that layout
  int swap;                // 1: launch a swapped-role (SWAP) instantiation
  int atma;                // 1: launch an ATMA instantiation
  uint32_t a_bytes;        // one operand buffer (both layouts)
  uint32_t a_half;         // 16-byte units between the two 128-row halves of a 256-row tile (128 | 512)
  alignas(64) CUtensorMap tm_a1, tm_a2;   // im2col views of src1 / src2
};

// debug timeline (DMN_TC_TRACE=1): CTA `trace_cta` records clock64 per role and tile: slot = 16*tile_iter + k
//   k: 0 producer tile start, 1 producer tables done, 2 producer last pass filled, 4 MMA got accumulators, 5 MMA first operand,
//      6 MMA tile issued, 8 epilogue tables done, 9 epilogue accumulators ready, 10 epilogue TMEM drained, 11 epilogue tile done,
//      12 / 13 clocks the MMA issuer waited for operands / weights, 14 / 15 clocks producer thread 0 waited for a free operand
//      buffer / for its own cp.async copies
__device__ long long g_trace[1024];
#ifndef DMN_TC_TRACE_PRODUCER
#define DMN_TC_TRACE_PRODUCER 0     // 1: also account the producers' wait clocks (slots 14 / 15); costs registers in the hot role
#endif
constexpr bool kTraceProducer = DMN_TC_TRACE_PRODUCER != 0;
#ifndef DMN_EXP_MMATRACE
#define DMN_EXP_MMATRACE 0          // 1: account the MMA issuer's wait clocks (slots 12 / 13); measured -1.3 % on the whole step
#endif
#ifndef DMN_TC_TRACE_BUILD
#define DMN_TC_TRACE_BUILD 0        // 1: compile the role timeline in (tools/trace_conv.py builds such a library); costs 1.5 % of the step
#endif
#define TRACE(it, k)                                                                                                             \
  do {                                                                                                                           \
    if (DMN_TC_TRACE_BUILD && p.trace && blockIdx.x == (unsigned)p.trace_cta && (it) < 60) p.trace[16 * (it) + (k)] = clock64(); \
  } while (0)

// flat virtual position -> (image, virtual row, virtual col); img < 0 when out of range.  32-bit arithmetic only
// (the host guarantees total_flat < 2^30).
struct VPos {
  int img, row, col;
};
__device__ __forceinline__ VPos vdecode(int f, const Params& p) {
  VPos r;
  r.img = -1;
  r.row = r.col = 0;
  if (f < 0 || f >= (int)p.total_flat) return r;
  const unsigned uf = (unsigned)f, uS = (unsigned)p.S, uW = (unsigned)p.Wv;
  const unsigned img = uf / uS;
  const unsigned rem = uf - img * uS;
  const unsigned row = rem / uW;
  r.img = (int)img;
  r.row = (int)row;
  r.col = (int)(rem - row * uW);
  return r;
}
// tile index -> (first flat position, 128-row accumulators, N tile).  Mixed tiling: whole rounds of 256-row tiles, then the
// remainder of the flat range in 128-row tiles so that the last round costs half (wave quantisation of one CTA per SM).
struct TileGeom {
  int m0, mt, n_tile;
};
__device__ __forceinline__ TileGeom tile_geom(int tile, const Params& p) {
  TileGeom g;
  const bool big = tile < p.n_big_tiles;
  const int k = big ? tile : tile - p.n_big_tiles;
  const int m = k / p.n_tiles_n;
  g.n_tile = k % p.n_tiles_n;
  g.mt = big ? 2 : 1;
  g.m0 = big ? m * 256 : p.big_rows + m * 128;
  return g;
}
// decode f = base_flat + n (0 <= n < 2^12 - ish) given the decoded base (img0, rem0 = base_flat - img0 * S): two multiply-shift
// divisions, exact for n + rem0 < 8192 and S <= 8192 (n * S < 2^26) and rem < S, Wv <= 128 (rem * Wv < 2^24)
__device__ __forceinline__ VPos vdecode_rel(int img0, int rem0, int n, const Params& p) {
  VPos r;
  const unsigned m = (unsigned)(rem0 + n);
  const unsigned k = (unsigned)(((unsigned long long)m * p.magic_S) >> 26);
  const unsigned rem = m - k * (unsigned)p.S;
  const unsigned row = (unsigned)(((unsigned long long)rem * p.magic_W) >> 24);
  r.img = img0 + (int)k;
  r.row = (int)row;
  r.col = (int)(rem - row * (unsigned)p.Wv);
  if ((long)r.img * p.S + rem >= p.total_flat) r.img = -1;
  return r;
}
// tap offset in flat positions (host: the table is passed in the kernel parameters = constant bank)
static int tap_delta(const Params& p, int geo, int t, int phase) {
  if (geo == GEO_SAME) {
    const int kh = p.ksize >> 1, ky = t / p.ksize, kx = t - ky * p.ksize;
    return (ky - kh) * p.Wv + (kx - kh);
  } else if (geo == GEO_DOWN) {
    return (t >> 1) * p.Wv + (t & 1);
  } else if (geo == GEO_UP) {
    const int py = phase >> 1, px = phase & 1, a = t >> 1, b = t & 1;
    const int dy = py ? (a ? 0 : 1) : (a ? -1 : 0);
    const int dx = px ? (b ? 0 : 1) : (b ? -1 : 0);
    return dy * p.Wv + dx;
  } else {
    return (t - 3) * p.Wv;
  }
}

// ---- packed fp32x2 arithmetic (FADD2 / FFMA2) ----
__device__ __forceinline__ unsigned long long pack2(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}

// Warp reduction of 8 per-row partials (4 group slots x {sum, sum of squares}) over the rows of ONE image and accumulation into
// the fixed-point statistics: halving butterfly (4 + 2 + 1 + 1 + 1 shuffles); afterwards every lane holds the total of value
// index lane >> 2, and lanes with (lane & 3) == 0 own one value each: slot = index >> 1, kind = index & 1.  The slots are
// RIGHT-ALIGNED: slot 3 is group g_last, slot 3 - i is group g_last - i; only the last `nslots` slots are valid.
__device__ __forceinline__ void reduce8_add(const float* v, int img, stat_t* ostats, int ogroups, int g_last, int nslots, int lane) {
  float a[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool hi = lane & 16;
    const float send = hi ? v[i] : v[i + 4], keep = hi ? v[i + 4] : v[i];
    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool hi = lane & 8;
    const float send = hi ? a[i] : a[i + 2], keep = hi ? a[i + 2] : a[i];
    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  {
    const bool hi = lane & 4;
    const float send = hi ? a[0] : a[1], keep = hi ? a[1] : a[0];
    a[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  a[0] += __shfl_xor_sync(0xffffffffu, a[0], 2);
  a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
  const int idx = lane >> 2, slot = idx >> 1, kind = idx & 1;
  if ((lane & 3) == 0 && slot >= 4 - nslots) {
    stat_t* dst = ostats + ((long)img * ogroups + g_last - 3 + slot) * 2 + kind;
    const float scale = kind ? kStatScaleSq : kStatScaleSum;
    atomicAdd(reinterpret_cast<unsigned long long*>(dst), (unsigned long long)__float2ll_rn(a[0] * scale));
  }
}
// rows of a warp are consecutive flat positions: usually one image (fast path), a few at low resolution (one pass per image)
__device__ __forceinline__ void stats_flush(const float* val, int key, bool valid, stat_t* ostats, int ogroups, int g_last, int nslots,
                                            int lane) {
  unsigned todo = __ballot_sync(0xffffffffu, valid);
  while (todo) {
    const int leader = __ffs(todo) - 1;
    const int k = __shfl_sync(0xffffffffu, key, leader);
    const unsigned mine = __ballot_sync(0xffffffffu, valid && key == k);
    todo &= ~mine;
    float m[8];
    const bool in = valid && key == k;
#pragma unroll
    for (int i = 0; i < 8; ++i) m[i] = in ? val[i] : 0.f;
    reduce8_add(m, k, ostats, ogroups, g_last, nslots, lane);
  }
}

// One weight stage (G taps x two k16 steps x 1|2 accumulators) of the MMA issuer.  Descriptor words are computed OUTSIDE the
// elected branch so that they are warp-uniform values (uniform registers); `didx` indexes the tap-offset table in the constant bank.
template <int G, bool TWO>
__device__ __forceinline__ void issue_stage(const Params& p, bool leader, uint32_t d0, uint32_t d1, uint32_t au, uint32_t bs, int didx, int t0,
                                            uint32_t acc0, uint32_t idesc, uint32_t hi_a, uint32_t hi_b, uint32_t lbo_a_f, uint32_t lbo_b_f,
                                            uint32_t a_k16, uint32_t b_k16, uint32_t b_tap_units, uint32_t a_half) {
  uint64_t ad[G][4], bd[G][2];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const uint32_t a0 = au + (uint32_t)p.delta[didx + g];
    const uint32_t b0 = bs + (uint32_t)g * b_tap_units;
    bd[g][0] = ((uint64_t)hi_b << 32) | ((b0 & 0x3FFFu) | lbo_b_f);
    bd[g][1] = ((uint64_t)hi_b << 32) | (((b0 + b_k16) & 0x3FFFu) | lbo_b_f);
    ad[g][0] = ((uint64_t)hi_a << 32) | ((a0 & 0x3FFFu) | lbo_a_f);
    ad[g][1] = ((uint64_t)hi_a << 32) | (((a0 + a_half) & 0x3FFFu) | lbo_a_f);
    ad[g][2] = ((uint64_t)hi_a << 32) | (((a0 + a_k16) & 0x3FFFu) | lbo_a_f);
    ad[g][3] = ((uint64_t)hi_a << 32) | (((a0 + a_k16 + a_half) & 0x3FFFu) | lbo_a_f);
  }
  if (leader) {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const uint32_t acc = (acc0 | (uint32_t)(t0 + g)) ? 1u : 0u;
      umma_bf16(d0, ad[g][0], bd[g][0], idesc, acc);
      if (TWO) umma_bf16(d1, ad[g][1], bd[g][0], idesc, acc);
      umma_bf16(d0, ad[g][2], bd[g][1], idesc, 1u);
      if (TWO) umma_bf16(d1, ad[g][3], bd[g][1], idesc, 1u);
    }
  }
}

// Lean issue path.  The issuing thread runs in near lock-step with the tensor pipe: what it executes between the last MMA of one
// tap and the first MMA of the next is hidden only while that last MMA (64 clk at N = 128) is still streaming its operands
// (tools/mma_rate2.cu: one extra mbarrier probe or an R2UR per tap costs its full latency).  So the per-tap preparation is cut
// to a handful of uniform adds: the tap offsets live in registers (loaded once), tap / stage indices are compile-time constants
// (fully unrolled pass), and the descriptor low words (start address | LBO field) are formed by plain additions -- shared memory
// is < 256 KB, so (address >> 4) never carries into the LBO field and no masking is needed.
template <bool TWO>
__device__ __forceinline__ void issue_tap(bool leader, uint32_t d0, uint32_t d1, uint32_t a_lo, uint32_t b_lo, uint32_t hi_a, uint32_t hi_b,
                                          uint32_t a_k16, uint32_t b_k16, uint32_t idesc, uint32_t acc, uint32_t a_half) {
  const uint64_t bd0 = ((uint64_t)hi_b << 32) | b_lo, bd1 = ((uint64_t)hi_b << 32) | (b_lo + b_k16);
  const uint64_t ad00 = ((uint64_t)hi_a << 32) | a_lo, ad10 = ((uint64_t)hi_a << 32) | (a_lo + a_k16);
  const uint64_t ad01 = ((uint64_t)hi_a << 32) | (a_lo + a_half), ad11 = ((uint64_t)hi_a << 32) | (a_lo + a_k16 + a_half);
  if (leader) {
    umma_bf16(d0, ad00, bd0, idesc, acc);
    if (TWO) umma_bf16(d1, ad01, bd0, idesc, acc);
    umma_bf16(d0, ad10, bd1, idesc, 1u);
    if (TWO) umma_bf16(d1, ad11, bd1, idesc, 1u);
  }
}
// One 32-channel pass = NTAP taps in stages of GG taps, fully unrolled.  `st` / `ph` walk the weight ring.
template <int NTAP, int GG, bool TWO>
__device__ __forceinline__ void issue_pass(bool leader, uint32_t d0, uint32_t d1, uint32_t au_lo, const int (&dl)[NTAP], uint32_t b_lo0,
                                           uint32_t b_stage_units, uint32_t b_tap_units, uint32_t hi_a, uint32_t hi_b, uint32_t a_k16,
                                           uint32_t b_k16, uint32_t idesc, uint32_t acc_first, uint64_t* full_b, uint64_t* empty_b, int nst,
                                           int& st, uint32_t& ph, uint32_t a_half) {
#pragma unroll
  for (int s = 0; s < NTAP / GG; ++s) {
    mbar_wait(smem_u32(&full_b[st]), ph);
    tc_fence_after();
    const uint32_t b_lo = b_lo0 + (uint32_t)st * b_stage_units;
#pragma unroll
    for (int g = 0; g < GG; ++g)
      issue_tap<TWO>(leader, d0, d1, au_lo + (uint32_t)dl[s * GG + g], b_lo + (uint32_t)g * b_tap_units, hi_a, hi_b, a_k16, b_k16, idesc,
                     (s | g) ? 1u : acc_first, a_half);
    if (leader) umma_commit(smem_u32(&empty_b[st]));     // frees the weight stage once these MMAs retire
    __syncwarp();
    if (++st == nst) { st = 0; ph ^= 1; }
  }
}

// Swapped operand roles: one MMA per k16 step (M = 128 output channels, N = 256 | 128 pixels).  `w_lo` / `x_lo` are the descriptor low
// words of the weight tap and of the shifted pixel view.
__device__ __forceinline__ void issue_tap_swap(bool leader, uint32_t d, uint32_t x_lo, uint32_t w_lo, uint32_t hi_x, uint32_t hi_w, uint32_t x_k16,
                                               uint32_t w_k16, uint32_t idesc, uint32_t acc) {
  const uint64_t wd0 = ((uint64_t)hi_w << 32) | w_lo, wd1 = ((uint64_t)hi_w << 32) | (w_lo + w_k16);
  const uint64_t xd0 = ((uint64_t)hi_x << 32) | x_lo, xd1 = ((uint64_t)hi_x << 32) | (x_lo + x_k16);
  if (leader) {
    umma_bf16(d, wd0, xd0, idesc, acc);
    umma_bf16(d, wd1, xd1, idesc, 1u);
  }
}
template <int NTAP, int GG>
__device__ __forceinline__ void issue_pass_swap(bool leader, uint32_t d, uint32_t au_lo, const int (&dl)[NTAP], uint32_t b_lo0, uint32_t b_stage_units,
                                                uint32_t b_tap_units, uint32_t hi_a, uint32_t hi_b, uint32_t a_k16, uint32_t b_k16, uint32_t idesc,
                                                uint32_t acc_first, uint64_t* full_b, uint64_t* empty_b, int nst, int& st, uint32_t& ph) {
#pragma unroll
  for (int s = 0; s < NTAP / GG; ++s) {
    mbar_wait(smem_u32(&full_b[st]), ph);
    tc_fence_after();
    const uint32_t b_lo = b_lo0 + (uint32_t)st * b_stage_units;
#pragma unroll
    for (int g = 0; g < GG; ++g)
      issue_tap_swap(leader, d, au_lo + (uint32_t)dl[s * GG + g], b_lo + (uint32_t)g * b_tap_units, hi_a, hi_b, a_k16, b_k16, idesc,
                     (s | g) ? 1u : acc_first);
    if (leader) umma_commit(smem_u32(&empty_b[st]));
    __syncwarp();
    if (++st == nst) { st = 0; ph ^= 1; }
  }
}

// ---------------------------------------------------------------------------------------------------
// kernel
// ---------------------------------------------------------------------------------------------------
// NT (the N tile: 32 / 64 / 128 output channels) is a template parameter so that the epilogue's geometry (columns per warp, staging
// swizzle, store pattern) folds to constants and its loops unroll
// FILM selects the FiLM signal prologue (LeakyReLU(0.2) + positional encoding, no GroupNorm; parts/film.py:22,58) at compile time so
// that the GroupNorm + SiLU prologue of the ResnetBlocks keeps its code unchanged
// LEAN selects the unrolled MMA issue path (a separate instantiation, so that the looped path keeps its own code generation)
// EXTRA keeps the rarely used epilogue terms (residual add, folded-GroupNorm affine); the hot instantiations drop them: the engine is
// measurably sensitive to the size of the code in its inner loops (compiling the debug timeline out alone gave +1.5 %)
// PRO: 0 = no fused prologue compiled in, 1 = the prologue is always on (GroupNorm convs), 2 = decided at run time (generic instantiations),
//      3 = 1x1 convolution without prologue: no halo and no padding, so the operand source of window pixel i is simply flat position
//          m0 + i and the per-tile tables (two producer barriers, a decode per pixel) are skipped
// EW: epilogue warps, 8 or 16.  The 16-warp form (832 threads, 72 registers per thread at launch) is for the epilogue-bound tiles
//     whose producers only issue copies: the producer warps hand registers back (setmaxnreg.dec 40) and the epilogue warps take
//     them (setmaxnreg.inc 88), so twice as many epilogue chains are in flight at the register budget the epilogue code needs.
// SWAP: operand roles exchanged -- the weights are the M operand (128 output channels on the TMEM lanes) and the tile's pixels the N
//     operand, so a 256-pixel tile is ONE M128 x N256 instruction per k-step instead of two M128 x N128: the tensor core then reads
//     12 KB of shared memory per 128 clk instead of 16 KB (the N = 128 form saturates the 128 B/clk shared-memory port, which is what
//     slows the operand producers and the epilogue staging down), and the single issuing thread has half as many instructions to feed.
//     The epilogue becomes channel-per-lane: bias and GroupNorm statistics are per-thread scalars / serial sums, the bf16 output is
//     transposed through a small per-warp staging tile (2 x 2 register transposes with one shuffle per pixel pair).
template <int GEO, int NT, bool FILM = false, bool LEAN = false, bool EXTRA = true, int PRO = 2, int EW = kEpiWarps, bool SWAP = false,
          bool ATMA = false>
__global__ void __launch_bounds__((kProdWarps + EW + 2) * 32, 1) conv_tcgen05_kernel(const __grid_constant__ Params p) {
  static_assert(!ATMA || (NT == 128 && !FILM && !EXTRA && (PRO == 0 || PRO == 1 || PRO == 3) && GEO != GEO_INIT),
                "TMA operand path: the hot 128-column instantiations");
  static_assert(!SWAP || (NT == 128 && !EXTRA && !FILM && GEO != GEO_INIT), "swapped operand roles: hot 128-channel instantiations only");
  constexpr int kLoaderW = kProdWarps + EW, kMmaW = kLoaderW + 1, kEpiT = EW * 32;
  constexpr int AB = (PRO == 3 && GEO == GEO_SAME) ? kABufOne : ((PRO == 1 && GEO == GEO_SAME) ? kABufPro : ((PRO == 0 && SWAP) ? kABufPlain : kABuf));
  constexpr int DEPTH = (PRO == 3 && GEO == GEO_SAME) ? kDepthOne : ((PRO == 1 && GEO == GEO_SAME) ? kDepthPro : ((PRO == 0 && SWAP) ? kDepthPlain : kDepth));
  static_assert(AB <= kABufMax && DEPTH >= 1 && DEPTH <= 3 && AB >= DEPTH + 2, "operand ring geometry");
  static_assert(EW == 8 || (EW == 16 && NT == 128 && (PRO == 0 || PRO == 3)), "16 epilogue warps: 128-column tiles without prologue");
  static_assert(!(LEAN && PRO == 3), "the lean issue path is for 9- and 4-tap convolutions");
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x;
  if (DMN_TC_TRACE_BUILD && p.trace && blockIdx.x == (unsigned)p.trace_cta && tid == 0) p.trace[1000] = clock64();     // kernel entry
  // broadcast => ptxas knows the role branches below are warp-uniform and may use the uniform datapath inside them
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int nst = p.nstage;

  // ---- shared memory carve-up ----
  const uint32_t a_bytes = p.a_bytes;                 // one A buffer (4 k-chunks x PA rows x 16 B, or P rows x 64 B rounded to 1 KB)
  const uint32_t tap_bytes = 4u * NT * 16u;           // weights of one tap of one pass
  const uint32_t b_bytes = p.stage_bytes;             // one B stage (G taps)
  uint8_t* sA = smem;
  uint8_t* sB = sA + AB * a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + nst * b_bytes);
  uint64_t* full_b = bars;
  uint64_t* empty_b = bars + kStagesMax;
  uint64_t* full_a = bars + 2 * kStagesMax;
  uint64_t* empty_a = full_a + kABufMax;
  uint64_t* raw_a = empty_a + kABufMax;               // ATMA with prologue: "the TMA copy of this buffer has landed"
  uint64_t* acc_full = raw_a + kABufMax;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float2* s_gn = reinterpret_cast<float2*>(tmem_slot + 2);                                  // [kNimgMax][kGroupsMax] (mean, rstd)
  int* s_pix = reinterpret_cast<int*>(s_gn + kNimgMax * kGroupsMax);                        // [P] operand source or -1
  int* s_pimg = s_pix + p.P;                                                                // [P] image - img_lo
  // epilogue, private per warp: bf16 output staging [32 rows][ncol] (16-byte chunks XOR-swizzled) + bias [ncol]
  // prologue coefficients per input channel, staged once per CTA: gamma | beta | time embedding (shared-row mode)
  float* s_coef = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(s_pimg + p.P) + 15) & ~(uintptr_t)15);
  const int ncoef = (p.c.pro != PRO_NONE) ? p.c.C1 : 0;
  uint8_t* s_stage = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(s_coef + 3 * ncoef) + 127) & ~(uintptr_t)127);

  // ---- one-time setup ----
  if (warp == kLoaderW) {          // one lane per barrier
    if (lane < nst) { mbar_init(smem_u32(&full_b[lane]), 1); mbar_init(smem_u32(&empty_b[lane]), 1); }
    if (lane >= 16 && lane < 16 + AB) {
      mbar_init(smem_u32(&full_a[lane - 16]), (ATMA && PRO != 1) ? 1 : kProdWarps);     // one arrival per producer WARP (see finish())
      mbar_init(smem_u32(&empty_a[lane - 16]), 1);
      mbar_init(smem_u32(&raw_a[lane - 16]), 1);
    }
    if (lane >= 24 && lane < 26) { mbar_init(smem_u32(&acc_full[lane - 24]), 1); mbar_init(smem_u32(&acc_empty[lane - 24]), kEpiT); }
    fence_barrier_init();
  }
  if (ATMA && tid == 0 && (smem_u32(sA) & 1023u)) __trap();      // SWIZZLE_64B tiles: the XOR pattern is keyed on absolute address bits 7-8
  if (warp == kMmaW) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();        // the next kernel may start its prologue; it waits for this grid's completion before reading our output

  if (warp < kProdWarps) {
    // =============================== operand producers ===============================
    if (EW == 16) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    // Each thread owns up to kMaxItems 16-byte items (pixel, k-chunk) of every pass.  A pass is ISSUED as cp.async (LDGSTS)
    // copies straight into the operand buffer (padding is stored as zeros), and FINISHED kDepth passes later: wait for the
    // thread's own copies, apply the fused prologue in place (GroupNorm-apply, SiLU, time-embedding add), make the writes
    // visible to the tensor core (async proxy) and arrive on the buffer's barrier.  Global latency is thereby covered by
    // kDepth passes in flight without staging the raw data in registers.
    pdl_wait();                                       // activations / statistics of the previous kernel are complete
    const int pc = tid & 3, px0 = tid >> 2;          // 16-byte chunk position in the row / k-chunk plane, first window pixel (step 64)
    // ATMA: the SWIZZLE_64B tile holds k-chunk (pc ^ ((row >> 1) & 3)) at chunk position pc of a row; the thread's rows are px0 + 64 j,
    // so that is one k-chunk for all of its items
    const int kc = ATMA ? (pc ^ ((px0 >> 1) & 3)) : pc;
    const bf16* src1 = (const bf16*)p.c.src1;
    const bf16* src2 = (const bf16*)p.c.src2;
    const float* temb_base = nullptr;
    if (GEO == GEO_SAME && (p.c.pro & PRO_TEMB)) temb_base = p.c.temb + (p.c.d_row ? (long)(*p.c.d_row) * p.c.temb_rstride : 0);
    const bool has_pro = PRO == 2 ? (GEO == GEO_SAME && p.c.pro != PRO_NONE) : (PRO == 1 && GEO == GEO_SAME);
    constexpr bool kOneTap = PRO == 3 && GEO == GEO_SAME;
    const bool temb_shared = (p.c.pro & PRO_TEMB) && p.c.temb_bstride == 0;
    if (has_pro) {                      // visible to all producers after the first tile's table barrier
      for (int i = tid; i < ncoef; i += kProdThreads) {
        s_coef[i] = FILM ? 1.f : p.c.pgamma[i];
        s_coef[ncoef + i] = FILM ? 0.f : p.c.pbeta[i];
        s_coef[2 * ncoef + i] = temb_shared ? temb_base[i] : 0.f;
      }
    }
    const uint32_t sA_u = smem_u32(sA);
    // ATMA: one im2col copy per pass.  (w, h, n) = tensor coordinates of the window's first position (decoded per tile)
    int tw = 0, th = 0, tn = 0;
    auto tma_window = [&](int c, int buf, uint64_t* bars_) {
      int cb = c * kCk;
      uint16_t ow = 0, oh = 0;
      const void* map = &p.tm_a1;
      if (GEO == GEO_DOWN) {
        const int sub = cb / p.c.C1;
        cb -= sub * p.c.C1;
        oh = (uint16_t)(sub >> 1);
        ow = (uint16_t)(sub & 1);
      } else if (cb >= p.c.C1) {
        cb -= p.c.C1;
        map = &p.tm_a2;
      }
      const uint32_t bar = smem_u32(&bars_[buf]);
      mbar_arrive_expect_tx(bar, (uint32_t)p.P * 64u);
      tma_load_im2col_4d(sA_u + (uint32_t)buf * a_bytes, map, cb, tw, th, tn, bar, ow, oh);
    };
    auto tma_tile_coords = [&](int m0) {
      const int f = m0 - p.halo_lo;
      tn = f >= 0 ? (int)__umul64hi((unsigned long long)(unsigned)f, p.magic64_S) : -1;     // halo_lo < S: a negative start lies in "image -1" (all zeros)
      const int rem = f - tn * p.S;
      const int row = (int)(((unsigned long long)(unsigned)rem * p.magic_W) >> 24), col = rem - row * p.Wv;
      if (GEO == GEO_DOWN) { tw = 2 * col - 1; th = 2 * row - 1; }
      else { tw = col - p.pad; th = row - p.pad; }
    };
    if constexpr (ATMA && PRO != 1) {
      // plain operands: nothing to transform -- one thread feeds the ring, the tensor core consumes the tiles as the copies land
      if (tid == 0) {
        int ibuf = 0;
        uint32_t iph = 1;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
          tma_tile_coords(tile_geom(tile, p).m0);
          for (int c = 0; c < p.n_pass; ++c) {
            mbar_wait_relaxed(smem_u32(&empty_a[ibuf]), iph);
            tma_window(c, ibuf, full_a);
            if (++ibuf == AB) { ibuf = 0; iph ^= 1; }
          }
        }
      }
    } else {
    int ibuf = 0, fbuf = 0;
    uint32_t rph = 0;                                  // ATMA: parity of the "copy has landed" wait
    uint32_t iph = 1;                                  // parity of the "buffer is free" wait; flips when the ring wraps
    int pit = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++pit) {
      if (tid == 0) TRACE(pit, 0);
      const TileGeom tg = tile_geom(tile, p);
      const int m0 = tg.m0;
      if constexpr (ATMA) tma_tile_coords(m0);
      const int Pt = tg.mt * 128 + p.halo_lo + p.halo_hi;       // window of THIS tile
      int f_lo = m0 - p.halo_lo;
      if (f_lo < 0) f_lo = 0;
      const int img_lo = f_lo / p.S;
      if (GEO == GEO_INIT) {
        // one pass: virtual channel vc = kx*Cin + ch  (7*Cin <= 32); source is the fp32 NCHW sampler state
        const float* x = (const float*)p.c.src1;
        const int Cin = p.c.C1;
        // this thread's 8 virtual channels (fixed k-chunk): source offset and kx shift, decoded once per tile instead of per element
        int koff[8], kxs[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int vc = kc * 8 + e;
          const int kx = vc / Cin, ch = vc - kx * Cin;
          kxs[e] = kx < 7 ? kx - 3 : (1 << 20);            // unused virtual channels never pass the range check below
          koff[e] = ch * p.HW + kx - 3;
        }
        const int ibase = m0 - p.halo_lo > 0 ? m0 - p.halo_lo : 0;
        const int iimg0 = ibase / p.S, irem0 = ibase - iimg0 * p.S;
        mbar_wait_relaxed(smem_u32(&empty_a[ibuf]), iph);
        for (int pixel = px0; pixel < Pt; pixel += kProdThreads / 4) {
          VPos v;
          v.img = -1; v.row = v.col = 0;
          if (m0 - p.halo_lo + pixel >= 0) v = vdecode_rel(iimg0, irem0, m0 - p.halo_lo + pixel - ibase, p);
          float f[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = 0.f;
          if (v.img >= 0 && v.row >= 3) {              // rows 0..2 of every block are the shared zero rows
            const float* xp = x + ((long)v.img * Cin * p.HW + (v.row - 3) * p.W + v.col);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const unsigned ix = (unsigned)(v.col + kxs[e]);
              if (ix < (unsigned)p.W) f[e] = __ldg(xp + koff[e]);
            }
          }
          *reinterpret_cast<uint4*>(sA + ibuf * a_bytes + (uint32_t)kc * p.lbo_a + pixel * 16) = pack8(f);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&full_a[ibuf]));
        if (++ibuf == AB) { ibuf = 0; iph ^= 1; }
        fbuf = ibuf;
        continue;
      }
      int goff[kMaxItems];      // SAME/UP: img*HW + pix (or -1 = padding); DOWN: packed (img, u, v) (or -1); -2 = outside the window
      int imgl[kMaxItems];
      if constexpr (kOneTap) {
#pragma unroll
        for (int j = 0; j < kMaxItems; ++j) {
          const int pixel = px0 + (kProdThreads / 4) * j;
          imgl[j] = 0;
          goff[j] = (pixel < Pt && m0 + pixel < (int)p.total_flat) ? m0 + pixel : -2;
        }
      } else {
      // ---- per-tile tables: operand source per window pixel, GroupNorm (mean, rstd) per touched image ----
      if (DMN_TC_TRACE_BUILD && p.trace && tid == 0 && pit == 2 && blockIdx.x == (unsigned)p.trace_cta) p.trace[900] = clock64();
      bar_sync_named(2, kProdThreads);                 // everyone is done with the previous tile's tables
      if (DMN_TC_TRACE_BUILD && p.trace && tid == 0 && pit == 2 && blockIdx.x == (unsigned)p.trace_cta) p.trace[901] = clock64();
      const int pbase = m0 - p.halo_lo > 0 ? m0 - p.halo_lo : 0;            // uniform: decode base of the window
      const int pimg0 = pbase / p.S, prem0 = pbase - pimg0 * p.S;
      for (int pixel = tid; pixel < Pt; pixel += kProdThreads) {
        VPos v;
        v.img = -1; v.row = v.col = 0;
        if (m0 - p.halo_lo + pixel >= 0) v = vdecode_rel(pimg0, prem0, m0 - p.halo_lo + pixel - pbase, p);
        int g = -1, il = 0;
        if (v.img >= 0) {
          if (GEO == GEO_DOWN) {
            g = (v.img << 14) | (v.row << 7) | v.col;
          } else if (v.row >= p.pad && v.col >= p.pad) {
            g = v.img * p.HW + (v.row - p.pad) * p.W + (v.col - p.pad);
            il = v.img - img_lo;
          }
        }
        s_pix[pixel] = g;
        s_pimg[pixel] = il;
      }
      if (DMN_TC_TRACE_BUILD && p.trace && tid == 0 && pit == 2 && blockIdx.x == (unsigned)p.trace_cta) p.trace[902] = clock64();
      if (GEO == GEO_SAME && (p.c.pro & PRO_GN)) {
        for (int i = tid; i < kNimgMax * p.c.pgroups; i += kProdThreads) {
          const int il = i / p.c.pgroups, g = i - il * p.c.pgroups;
          const int img = img_lo + il;
          float mean = 0.f, rstd = 0.f;
          if (img < p.c.B) gn_mean_rstd(p.c.pstats + ((long)img * p.c.pgroups + g) * 2, p.inv_cnt_in, kGnEps, mean, rstd);
          s_gn[il * kGroupsMax + g] = make_float2(mean, rstd);
        }
      }
      if (DMN_TC_TRACE_BUILD && p.trace && tid == 0 && pit == 2 && blockIdx.x == (unsigned)p.trace_cta) p.trace[903] = clock64();
      bar_sync_named(2, kProdThreads);
      if (tid == 0) TRACE(pit, 1);
#pragma unroll
      for (int j = 0; j < kMaxItems; ++j) {
        const int pixel = px0 + (kProdThreads / 4) * j;
        goff[j] = -2;
        imgl[j] = 0;
        if (pixel < Pt) {
          goff[j] = s_pix[pixel];
          imgl[j] = s_pimg[pixel];
        }
      }
      }

      // finish pass c (in buffer fbuf): prologue in place on this thread's own items, publish to the tensor core
      auto finish = [&](int c) {
        const bool fst = DMN_TC_TRACE_BUILD && p.trace && tid == 0 && pit == 2 && c == 1 && blockIdx.x == (unsigned)p.trace_cta;
        if (fst) p.trace[910] = clock64();
        if constexpr (ATMA) mbar_wait(smem_u32(&raw_a[fbuf]), rph);      // the window of this pass has landed
        if (fst) p.trace[911] = clock64();
        if (has_pro) {
          const int cb = c * kCk + kc * 8;
          float ga[8], be[8], te[8];
          {
            // (explicit shared-space loads: through the integer-cast pointer these compiled to generic LD.E.128)
            const uint32_t cu = smem_u32(s_coef) + (uint32_t)cb * 4u, nb = (uint32_t)ncoef * 4u;
            auto ldf4 = [](uint32_t a) { const uint4 u = lds128(a); return make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w)); };
            const float4 g0 = ldf4(cu), g1 = ldf4(cu + 16u);
            const float4 b0 = ldf4(cu + nb), b1 = ldf4(cu + nb + 16u);
            const float4 t0 = ldf4(cu + 2u * nb), t1 = ldf4(cu + 2u * nb + 16u);
            ga[0] = g0.x; ga[1] = g0.y; ga[2] = g0.z; ga[3] = g0.w; ga[4] = g1.x; ga[5] = g1.y; ga[6] = g1.z; ga[7] = g1.w;
            be[0] = b0.x; be[1] = b0.y; be[2] = b0.z; be[3] = b0.w; be[4] = b1.x; be[5] = b1.y; be[6] = b1.z; be[7] = b1.w;
            te[0] = t0.x; te[1] = t0.y; te[2] = t0.z; te[3] = t0.w; te[4] = t1.x; te[5] = t1.y; te[6] = t1.z; te[7] = t1.w;
          }
          const int g = cb >> p.cpg_in_shift;
          uint8_t* base = ATMA ? sA + fbuf * a_bytes + (uint32_t)pc * 16u : sA + fbuf * a_bytes + (uint32_t)kc * p.lbo_a;
          // packed fp32x2 arithmetic (FFMA2 / FADD2).  hx = t / 2 with t = GroupNorm affine: the halving is folded into gamma / beta
          // (exact: a power of two), SiLU(t) = hx * tanh(hx) + hx is one MUFU per element
          unsigned long long gah2[4], beh2[4], te2[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            gah2[e] = pack2(0.5f * ga[2 * e], 0.5f * ga[2 * e + 1]);
            beh2[e] = pack2(0.5f * be[2 * e], 0.5f * be[2 * e + 1]);
            te2[e] = pack2(te[2 * e], te[2 * e + 1]);
          }
          // one item = one independent chain (LDS -> FFMA2 -> MUFU -> FFMA2 -> STS), behind a per-item branch so that padding and slots
          // outside the window cost nothing.  (Transforming the slots that are always inside the window without the branch, as one
          // basic block, measured SLOWER on every conv of the step, including those without a prologue (+0.002..0.004 ms each): the
          // extra unrolled copies grow the kernel, and the engine is sensitive to code size.)
          auto do_item = [&](int j) {
            if (goff[j] < 0) return;
            uint4* slot = reinterpret_cast<uint4*>(base + (px0 + (kProdThreads / 4) * j) * (ATMA ? 64 : 16));
            const float2 mr = FILM ? make_float2(0.f, 1.f) : s_gn[imgl[j] * kGroupsMax + g];
            if ((p.c.pro & PRO_TEMB) && !temb_shared) {
              const float* tp = temb_base + (long)(img_lo + imgl[j]) * p.c.temb_bstride + cb;
              const float4 t0 = *reinterpret_cast<const float4*>(tp), t1 = *reinterpret_cast<const float4*>(tp + 4);
              te2[0] = pack2(t0.x, t0.y); te2[1] = pack2(t0.z, t0.w); te2[2] = pack2(t1.x, t1.y); te2[3] = pack2(t1.z, t1.w);
            }
            float v[8];
            unpack8(*slot, v);
            if (FILM) {                                 // LeakyReLU(0.2) + positional encoding (parts/film.py:22,58)
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const unsigned long long y2 = add2(pack2(fmaxf(v[2 * e], 0.2f * v[2 * e]), fmaxf(v[2 * e + 1], 0.2f * v[2 * e + 1])), te2[e]);
                unpack2(y2, v[2 * e], v[2 * e + 1]);
              }
            } else {
              const float sc = mr.y, sh = -mr.x * mr.y;
              const unsigned long long sc2 = pack2(sc, sc), sh2 = pack2(sh, sh);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                unsigned long long x2 = fma2(pack2(v[2 * e], v[2 * e + 1]), sc2, sh2);
                x2 = fma2(x2, gah2[e], beh2[e]);                       // hx
                unsigned long long y2;
                if (p.c.pro & PRO_SILU) {
                  float h0, h1, t0, t1;
                  unpack2(x2, h0, h1);
                  asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
                  asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
                  y2 = fma2(x2, pack2(t0, t1), x2);
                } else {
                  y2 = add2(x2, x2);
                }
                y2 = add2(y2, te2[e]);
                unpack2(y2, v[2 * e], v[2 * e + 1]);
              }
            }
            *slot = pack8(v);
          };
          // TMA tiles: groups of three items as ONE basic block -- all loads first (an item slot outside the window reads the thread's
          // first slot instead), then the three arithmetic chains side by side, then stores predicated in the instruction itself
          // (padding stays zero).  With a per-item `if` ptxas skips the whole chain of a padding item, which makes every item its own
          // branch region and serialises LDS -> FFMA2 -> MUFU -> STS item after item (SASS of the round-2 build)
          auto do_group = [&](auto j0_tag, auto silu_tag) {
            constexpr int J0 = decltype(j0_tag)::value;
            constexpr bool SILU = decltype(silu_tag)::value;
            constexpr int N = (kMaxItems - J0) < kGS ? (kMaxItems - J0) : kGS;
            const uint32_t base_u = smem_u32(base);
            uint4 raw[N];
            float2 mr[N];
#pragma unroll
            for (int i = 0; i < N; ++i) {
              const int j = J0 + i;
              const int px = goff[j] >= -1 ? px0 + (kProdThreads / 4) * j : px0;
              raw[i] = lds128(base_u + (uint32_t)px * 64u);
              mr[i] = s_gn[imgl[j] * kGroupsMax + g];
            }
#pragma unroll
            for (int i = 0; i < N; ++i) {
              float v[8];
              unpack8(raw[i], v);
              const float sc = mr[i].y, sh = -mr[i].x * mr[i].y;
              const unsigned long long sc2 = pack2(sc, sc), sh2 = pack2(sh, sh);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                unsigned long long x2 = fma2(pack2(v[2 * e], v[2 * e + 1]), sc2, sh2);
                x2 = fma2(x2, gah2[e], beh2[e]);                       // hx
                unsigned long long y2;
                if (SILU) {
                  float h0, h1, t0, t1;
                  unpack2(x2, h0, h1);
                  asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
                  asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
                  y2 = fma2(x2, pack2(t0, t1), x2);
                } else {
                  y2 = add2(x2, x2);
                }
                y2 = add2(y2, te2[e]);
                unpack2(y2, v[2 * e], v[2 * e + 1]);
              }
              raw[i] = pack8(v);
            }
#pragma unroll
            for (int i = 0; i < N; ++i) {
              const int j = J0 + i;
              asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %5, 0;\n\t@p st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n\t}" ::"r"(
                               base_u + (uint32_t)(px0 + (kProdThreads / 4) * j) * 64u),
                           "r"(raw[i].x), "r"(raw[i].y), "r"(raw[i].z), "r"(raw[i].w), "r"((uint32_t)(goff[j] >= 0))
                           : "memory");
            }
          };
          if (fst) p.trace[912] = clock64();
          if (ATMA && !FILM && !((p.c.pro & PRO_TEMB) && !temb_shared)) {
            const int n_it = (Pt + kProdThreads / 4 - 1) / (kProdThreads / 4);     // item slots that reach into the window (uniform)
            auto all_groups = [&](auto silu_tag) {
              do_group(std::integral_constant<int, 0>(), silu_tag);
              if (kMaxItems > kGS && n_it > kGS) do_group(std::integral_constant<int, (kMaxItems > kGS ? kGS : 0)>(), silu_tag);
              if (kMaxItems > 2 * kGS && n_it > 2 * kGS) do_group(std::integral_constant<int, (kMaxItems > 2 * kGS ? 2 * kGS : 0)>(), silu_tag);
              if (kMaxItems > 3 * kGS && n_it > 3 * kGS) do_group(std::integral_constant<int, (kMaxItems > 3 * kGS ? 3 * kGS : 0)>(), silu_tag);
            };
            if (p.c.pro & PRO_SILU) all_groups(std::true_type());
            else all_groups(std::false_type());
          } else {
#pragma unroll
            for (int j = 0; j < kMaxItems; ++j) do_item(j);
          }
        }
        // every writer fences its own stores towards the async proxy, then ONE lane per warp arrives: 256 / 512 arrivals on one
        // mbarrier serialise (measured: a pass that only loads and stores its items took 1.6k clk with per-thread arrivals)
        if (fst) p.trace[913] = clock64();
        fence_proxy_async();
        if (fst) p.trace[914] = clock64();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&full_a[fbuf]));
        if (fst) p.trace[915] = clock64();
        if (++fbuf == AB) { fbuf = 0; rph ^= 1; }
      };

      int inflight = 0;
      const bool ptracing = kTraceProducer && p.trace && tid == 0 && blockIdx.x == (unsigned)p.trace_cta && pit < 60;
      long long wait_e = 0, wait_g = 0, t_issue = 0, t_fin = 0;
      for (int c = 0; c < p.n_pass; ++c) {
        long long w0 = ptracing ? clock64() : 0;
        if constexpr (ATMA) {
          // one thread waits for the free buffer and issues the window copy; everybody meets the data at the raw_a barrier in finish()
          if (tid == 0) {
            mbar_wait_relaxed(smem_u32(&empty_a[ibuf]), iph);
            if (ptracing) wait_e += clock64() - w0;
            tma_window(c, ibuf, raw_a);
          }
        } else {
        mbar_wait_relaxed(smem_u32(&empty_a[ibuf]), iph);
        if (ptracing) wait_e += clock64() - w0;
        const long long wi0 = ptracing ? clock64() : 0;
        int cb = c * kCk + kc * 8;        // first (virtual) channel of this thread's k-chunk
        int sy = 0, sx = 0;
        if (GEO == GEO_DOWN) {            // virtual channel = sub * C + ci, sub = sy*2 + sx
          const int sub = cb / p.c.C1;
          cb -= sub * p.c.C1;
          sy = sub >> 1;
          sx = sub & 1;
        }
        const bf16* src;
        int Cs, cofs;
        if (cb < p.c.C1) { src = src1; Cs = p.c.C1; cofs = cb; }
        else { src = src2; Cs = p.c.C2; cofs = cb - p.c.C1; }
        const uint32_t dst0 = sA_u + ibuf * a_bytes + (uint32_t)kc * p.lbo_a + (uint32_t)px0 * 16u;
        // measured: the predicated zero-fill form wins when the fused prologue follows (-0.003 ms on the level-0 GroupNorm convs)
        // and loses for plain copies (+0.004 ms), so plain operands keep the branchy issue
        if (GEO == GEO_DOWN || !has_pro) {
#pragma unroll
          for (int j = 0; j < kMaxItems; ++j) {
            if (goff[j] < -1) continue;                  // outside the window
            const uint32_t dst = dst0 + (uint32_t)((kProdThreads / 4) * j) * 16u;
            const bf16* sp = nullptr;
            if (goff[j] >= 0) {
              if (GEO == GEO_DOWN) {
                const int img = goff[j] >> 14, iy = 2 * ((goff[j] >> 7) & 127) - 1 + sy, ix = 2 * (goff[j] & 127) - 1 + sx;
                if (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W) sp = src + ((long)img * p.HW + iy * p.W + ix) * Cs + cofs;
              } else {
                sp = src + (long)goff[j] * Cs + cofs;
              }
            }
            if (sp) cp_async16(dst, sp);
            else asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(dst), "r"(0) : "memory");   // padding -> zeros
          }
        } else {
          // straight-line issue: one predicated LDGSTS per item; padding positions copy 0 bytes and zero-fill the 16 (src-size
          // operand), items outside the window are predicated off.  32-bit byte offsets (the host checks the tensor is < 4 GB)
          const uint8_t* sbase = reinterpret_cast<const uint8_t*>(src + cofs);
          const uint32_t row_bytes = (uint32_t)Cs * 2u;
#pragma unroll
          for (int j = 0; j < kMaxItems; ++j) {
            const bool ok = goff[j] >= 0;
            const uint8_t* sp = sbase + (size_t)((uint32_t)(ok ? goff[j] : 0) * row_bytes);
            cp_async16_zfill_pred(dst0 + (uint32_t)((kProdThreads / 4) * j) * 16u, sp, ok ? 16u : 0u, goff[j] >= -1);
          }
        }
        cp_async_commit();
        if (ptracing) t_issue += clock64() - wi0;
        }   // !ATMA
        if (++ibuf == AB) { ibuf = 0; iph ^= 1; }
        if (++inflight > DEPTH) {
          w0 = ptracing ? clock64() : 0;
          if constexpr (!ATMA) cp_async_wait<DEPTH>();
          if (ptracing) wait_g += clock64() - w0;
          const long long wf0 = ptracing ? clock64() : 0;
          finish(c - DEPTH);
          if (ptracing) t_fin += clock64() - wf0;
          --inflight;
        }
      }
      if (ptracing) { p.trace[16 * pit + 14] = wait_e; p.trace[16 * pit + 15] = wait_g; p.trace[16 * pit + 3] = t_issue; p.trace[16 * pit + 7] = t_fin; }
      // drain: the last passes of the tile
      if (DEPTH >= 3 && inflight == 3) {
        if constexpr (!ATMA) cp_async_wait<2>();
        finish(p.n_pass - 3);
        --inflight;
      }
      if (DEPTH >= 2 && inflight == 2) {
        if constexpr (!ATMA) cp_async_wait<1>();
        finish(p.n_pass - 2);
        --inflight;
      }
      if (inflight == 1) {
        if constexpr (!ATMA) cp_async_wait<0>();
        finish(p.n_pass - 1);
      }
      if (tid == 0) TRACE(pit, 2);
    }
    }   // !(ATMA && PRO != 1)
  } else if (warp < kLoaderW) {
    // =============================== epilogue ===============================
    // register pool of the CTA: the 8 producer warps release 8 x 32 x (72 - 40) = 8192 registers, exactly what 16 epilogue warps need to
    // grow from 72 to 88 (setmaxnreg only moves registers inside the CTA's launch allocation; asking for 96 here deadlocks)
    if (EW == 16) asm volatile("setmaxnreg.inc.sync.aligned.u32 88;");
    // Warps are independent: no shared tables and no block barriers.  Each thread decodes its own accumulator rows
    // (flat position -> output pixel / image), reads 32-column chunks from TMEM, adds bias (+ class embedding, + residual),
    // stores bf16 and accumulates the GroupNorm statistics of its rows; a warp then reduces 8 partials at a time with a
    // halving butterfly (9 shuffles) and the owning lanes add them to the (image, group) slots with fixed-point integer
    // atomics (order independent => deterministic).
    pdl_wait();                                       // output / residual / statistics buffers are free to touch
    const int ew = warp - kProdWarps;                 // 0 .. EW-1
    const int quarter = ew & 3, part = ew >> 2;       // TMEM lane quarter, column part (half / quarter) of the tile
    if constexpr (SWAP) {
      // ---- swapped roles: TMEM lane = output channel, column = pixel of the tile ----
      bf16* out = (bf16*)p.c.out;
      constexpr int NPART = EW / 4;                     // the tile's pixel columns are split over NPART warps per lane quarter
      const bool do_stats = GEO == GEO_SAME && p.c.ostats != nullptr;
      const bool has_bias = p.c.bias != nullptr;
      // per-warp shared memory: [32 pixels][32 channels] bf16 staging (2 KB) + output pixel index of each of the warp's columns
      uint8_t* my_base = s_stage + ew * (EW == 8 ? 4608 : 2304);
      const uint32_t my_stage = smem_u32(my_base);
      int* s_opix = reinterpret_cast<int*>(my_base + 2048);
      float* s_ball = reinterpret_cast<float*>(s_stage + 8 * 4608);
      {
        const int et = tid - kProdThreads;
        if (has_bias)
          for (int i = et; i < p.c.Cout; i += kEpiT) s_ball[i] = p.c.bias[i];
        bar_sync_named(3, kEpiT);
      }
      const int sh = p.cpg_out_shift;
      const int red_lanes = p.cpg_out >= 32 ? 32 : p.cpg_out;     // lanes of this warp that share a statistics group (16 or 32)
      const int prow = lane >> 2, pchunk = lane & 3;              // store phase: pixel row within an instruction, 16-byte chunk of its 64 bytes
      int it = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
        const TileGeom tg = tile_geom(tile, p);
        const int n_tile = tg.n_tile, m0 = tg.m0, tmt = tg.mt;
        const int phase = (GEO == GEO_UP) ? n_tile / p.tiles_per_phase : 0;
        const int n0 = (GEO == GEO_UP ? n_tile % p.tiles_per_phase : n_tile) * NT;
        const int ncols = tmt * 128 / NPART;                      // pixel columns of this warp: 128 | 64 | 32
        const int col_base = part * ncols;
        const int eimg0 = m0 / p.S, erem0 = m0 - eimg0 * p.S;     // uniform
        // ---- decode this warp's columns once: output pixel (or -1), validity masks (uniform after the ballots) ----
        uint32_t vmask[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (i * 32 < ncols) {
            const VPos v = vdecode_rel(eimg0, erem0, col_base + i * 32 + lane, p);
            bool valid = v.img >= 0;
            int opix = -1;
            if (valid) {
              if (GEO == GEO_SAME) {
                valid = v.row >= p.pad && v.col >= p.pad;
                opix = v.img * p.HW + (v.row - p.pad) * p.W + (v.col - p.pad);
              } else if (GEO == GEO_DOWN) {
                valid = v.row < (p.H >> 1) && v.col < (p.W >> 1);
                opix = v.img * (p.HW >> 2) + v.row * (p.W >> 1) + v.col;
              } else {
                valid = v.row >= 1 && v.col >= 1;
                opix = v.img * (p.HW << 2) + (2 * (v.row - 1) + (phase >> 1)) * (2 * p.W) + 2 * (v.col - 1) + (phase & 1);
              }
            }
            s_opix[i * 32 + lane] = valid ? opix : -1;
            vmask[i] = __ballot_sync(0xffffffffu, valid);
          }
        }
        __syncwarp();
        const int my_c = n0 + quarter * 32 + lane;                // this thread's output channel
        const float bias = has_bias ? s_ball[my_c] : 0.f;
        // statistics bookkeeping (uniform): image of the current column, columns left in it
        int cur_img = eimg0 + (erem0 + col_base) / p.S;
        int to_boundary = p.S - (erem0 + col_base) % p.S;
        // Running (sum, sum of squares) of this channel over the current image in FIXED POINT: every 16-column chunk (an absolute
        // 16-position block of the flat index space, whatever the tiling) is summed in fp32 in a fixed order, converted, and added as an
        // integer -- so the statistics do not depend on how tiles align with images (batch-slice invariance, graph == plain launches)
        long long rs = 0, rq = 0;
        auto flush = [&]() {
          // integer reduction over the lanes of the group, then the group leader adds the partials
          long long a = rs, b = rq;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1)
            if (o < red_lanes) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
          if ((lane & (red_lanes - 1)) == 0 && cur_img < p.c.B) stat_add_fixed(p.c.ostats + ((long)cur_img * p.c.ogroups + (my_c >> sh)) * 2, a, b);
          rs = rq = 0;
        };

        const int as = it & 1;
        if (ew == 0 && lane == 0) TRACE(it, 8);
        mbar_wait_relaxed(smem_u32(&acc_full[as]), (it >> 1) & 1);
        tc_fence_after();
        if (ew == 0 && lane == 0) TRACE(it, 9);
        const uint32_t tlane = tmem_base + (uint32_t)(as * 2 * NT) + ((uint32_t)(quarter * 32) << 16) + (uint32_t)col_base;
        const int rounds = ncols >> 5;                            // 32 columns per staging round
        uint32_t rb[2][16];
        tmem_ld16_nowait(tlane, rb[0]);
#pragma unroll 1
        for (int rd = 0; rd < rounds; ++rd) {
          const uint32_t vm = rd == 0 ? vmask[0] : (rd == 1 ? vmask[1] : (rd == 2 ? vmask[2] : vmask[3]));
#pragma unroll
          for (int hc = 0; hc < 2; ++hc) {                        // two 16-column chunks per round
            tmem_ld_wait();
            const int cnext = rd * 32 + (hc + 1) * 16;
            if (cnext < ncols) {
              tmem_ld16_nowait(tlane + (uint32_t)cnext, rb[hc ^ 1]);
            } else {
              tc_fence_before();                                  // last TMEM read of this tile: hand the accumulators back
              mbar_arrive(smem_u32(&acc_empty[as]));
              if (ew == 0 && lane == 0) TRACE(it, 10);
            }
            const uint32_t* r = rb[hc];
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]) + bias;
            if (do_stats) {
              const uint32_t m16 = (vm >> (hc * 16)) & 0xffffu;
              if (to_boundary > 16) {                             // (uniform) the whole chunk belongs to the current image
                float s0 = 0.f, q0 = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  const float x = (m16 >> j) & 1u ? v[j] : 0.f;
                  s0 += x;
                  q0 = fmaf(x, x, q0);
                }
                rs += __float2ll_rn(s0 * kStatScaleSum);
                rq += __float2ll_rn(q0 * kStatScaleSq);
                to_boundary -= 16;
              } else {
                // columns [0, tb) close the current image, [tb, 16) open the next one (S >= 16: at most one boundary per chunk)
                const int tb = to_boundary;
                float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  const float x = (m16 >> j) & 1u ? v[j] : 0.f;
                  if (j < tb) { s0 += x; q0 = fmaf(x, x, q0); }
                  else { s1 += x; q1 = fmaf(x, x, q1); }
                }
                rs += __float2ll_rn(s0 * kStatScaleSum);
                rq += __float2ll_rn(q0 * kStatScaleSq);
                flush();
                ++cur_img;
                rs = __float2ll_rn(s1 * kStatScaleSum);
                rq = __float2ll_rn(q1 * kStatScaleSq);
                to_boundary = p.S - (16 - tb);
              }
            }
            // 2 x 2 transposes: after the exchange an even lane holds channels (lane, lane + 1) of pixel 2i, an odd lane channels
            // (lane - 1, lane) of pixel 2i + 1; one 32-bit store per pixel pair, conflict-free
            const bool odd = lane & 1;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float send = odd ? v[2 * i] : v[2 * i + 1];
              const float got = __shfl_xor_sync(0xffffffffu, send, 1);
              const uint32_t w = odd ? pack_bf16x2(got, v[2 * i + 1]) : pack_bf16x2(v[2 * i], got);
              const int px = hc * 16 + 2 * i + (odd ? 1 : 0);
              asm volatile("st.shared.b32 [%0], %1;" ::"r"(my_stage + (uint32_t)(px * 64 + (lane >> 1) * 4)), "r"(w) : "memory");
            }
          }
          __syncwarp();
          // store phase: 32 pixel rows x 64 bytes; one instruction covers 8 rows (4 lanes x 16 bytes each)
#pragma unroll
          for (int i0 = 0; i0 < 32; i0 += 8) {
            const int row = i0 + prow;
            const int opix = s_opix[rd * 32 + row];
            const uint4 o = lds128(my_stage + (uint32_t)(row * 64 + pchunk * 16));
            if (opix >= 0) *reinterpret_cast<uint4*>(out + (long)opix * p.c.Cout + n0 + quarter * 32 + pchunk * 8) = o;
          }
          __syncwarp();
        }
        if (do_stats) flush();
        if (ew == 0 && lane == 0) TRACE(it, 11);
      }
    } else {
    bf16* out = (bf16*)p.c.out;
    constexpr bool kExtra = EXTRA && GEO == GEO_SAME;      // fill_params rejects residual / fold for the other geometries
    const bf16* res = kExtra ? (const bf16*)p.c.res : nullptr;
    // columns owned by this warp: half of the tile; with NT = 32 only the first warp of each lane quarter works
    constexpr int NCOL = NT >= 64 ? NT / (EW / 4) : NT;      // 64 | 32 | 32 (8 warps), 32 (16 warps)
    constexpr int PPM = NCOL / 16;                    // 16-column pieces per 128-row accumulator (even)
    constexpr int ROWB = NCOL * 2, LPR = NCOL / 8, RPI = 32 / LPR;   // staging row bytes, lanes per row, rows per store instruction
    constexpr int SWS = ROWB == 64 ? 1 : 0, SWM = ROWB == 64 ? 3 : 7;
    const bool active = NT >= 64 || part == 0;
    const int col0 = NT >= 64 ? part * NCOL : 0;
    const int sh = p.cpg_out_shift;
    const bool do_stats = GEO == GEO_SAME && p.c.ostats != nullptr;     // fill_params rejects output statistics for the other geometries
    const bool has_bias = p.c.bias != nullptr;
    const bool has_fold = kExtra && p.c.fold_s1 != nullptr;     // GroupNorm(1) of the input folded into an epilogue affine (to_qkv)
    const uint32_t my_stage = smem_u32(s_stage) + (uint32_t)(ew * (32 * ROWB + NCOL * 8));   // shared-space addresses
    // bias (or the folded-GroupNorm vectors s1 | s2) of ALL output channels and, for the fold, (rstd, -mean * rstd) of every image are
    // staged ONCE per CTA: with several N tiles per M tile the N tile changes on every tile of a CTA, and re-staging from global
    // memory (plus a double-precision mean / rstd per accumulator row) was 30 % of the to_qkv epilogue
    float* s_ball = reinterpret_cast<float*>(s_stage + EW * (32 * ROWB + NCOL * 8));
    float2* s_rst = reinterpret_cast<float2*>(s_ball + 2 * p.c.Cout);
    {
      const int et = tid - kProdThreads;
      if (has_bias || has_fold)
        for (int i = et; i < p.c.Cout; i += kEpiT) {
          s_ball[i] = has_fold ? p.c.fold_s1[i] : p.c.bias[i];
          s_ball[p.c.Cout + i] = has_fold ? p.c.fold_s2[i] : 0.f;
        }
      if (has_fold)
        for (int i = et; i < p.c.B; i += kEpiT) {
          float mean, rstd;
          gn_mean_rstd(p.c.pstats + (long)i * 2, p.inv_cnt_in, kGnEps, mean, rstd);
          s_rst[i] = make_float2(rstd, -mean * rstd);
        }
      bar_sync_named(3, kEpiT);
    }
    const uint32_t s_ball_u = smem_u32(s_ball);
    const int my_swz = (lane >> SWS) & SWM;
    const int lrow = lane / LPR, lcol = lane % LPR;   // this lane's (row within a store instruction, 16-byte chunk)
    const uint32_t my_wr = my_stage + (uint32_t)(lane * ROWB);   // this lane's staging row
    int it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const TileGeom tg = tile_geom(tile, p);
      const int n_tile = tg.n_tile, m0 = tg.m0, tmt = tg.mt;
      const int phase = (GEO == GEO_UP) ? n_tile / p.tiles_per_phase : 0;
      const int n0 = (GEO == GEO_UP ? n_tile % p.tiles_per_phase : n_tile) * NT;
      // ---- this thread's rows ----
      const int eimg0 = m0 / p.S, erem0 = m0 - eimg0 * p.S;     // uniform
      int opixv[kMTmax], keyv[kMTmax];
#pragma unroll
      for (int mt = 0; mt < kMTmax; ++mt) {
        opixv[mt] = -1;
        keyv[mt] = -1;
        if (mt < tmt) {
          const VPos v = vdecode_rel(eimg0, erem0, mt * 128 + quarter * 32 + lane, p);
          bool valid = v.img >= 0;
          int opix = -1;
          if (valid) {
            if (GEO == GEO_SAME) {
              valid = v.row >= p.pad && v.col >= p.pad;
              opix = v.img * p.HW + (v.row - p.pad) * p.W + (v.col - p.pad);
            } else if (GEO == GEO_DOWN) {
              valid = v.row < (p.H >> 1) && v.col < (p.W >> 1);
              opix = v.img * (p.HW >> 2) + v.row * (p.W >> 1) + v.col;
            } else if (GEO == GEO_UP) {
              valid = v.row >= 1 && v.col >= 1;
              opix = v.img * (p.HW << 2) + (2 * (v.row - 1) + (phase >> 1)) * (2 * p.W) + 2 * (v.col - 1) + (phase & 1);
            } else {
              valid = v.row >= 3;
              opix = v.img * p.HW + (v.row - 3) * p.W + v.col;
            }
          }
          if (valid) { opixv[mt] = opix; keyv[mt] = v.img; }
        }
      }
      const uint32_t my_bias = s_ball_u + 4u * (uint32_t)(n0 + col0);      // this warp's columns of the staged vectors
      if (ew == 0 && lane == 0) TRACE(it, 8);

      const int as = it & 1;
      mbar_wait_relaxed(smem_u32(&acc_full[as]), (it >> 1) & 1);
      tc_fence_after();
      if (ew == 0 && lane == 0) TRACE(it, 9);
      const uint32_t tacc = tmem_base + (uint32_t)(as * 2 * NT);
      if (!active) {
        tc_fence_before();
        mbar_arrive(smem_u32(&acc_empty[as]));
        continue;
      }
      // software pipeline over 16-column pieces: the TMEM load of the next piece is in flight while this one is processed
      const uint32_t tlane = tacc + ((uint32_t)(quarter * 32) << 16) + (uint32_t)col0;
      bf16* const out_col = out + n0 + col0 + lcol * 8;       // store phase: + row * Cout
      uint32_t rb[2][16];
      tmem_ld16_nowait(tlane, rb[0]);
      float val[8];                                           // statistics shift register: 4 group slots x {sum, sumsq}
#pragma unroll
      for (int i = 0; i < 8; ++i) val[i] = 0.f;
      float cs = 0.f, cq = 0.f;                               // current group accumulator (this row)
      int nslots = 0;
#pragma unroll 1
      for (int mt = 0; mt < tmt; ++mt) {
        const int opix = mt == 0 ? opixv[0] : opixv[kMTmax - 1];
        const int key = mt == 0 ? keyv[0] : keyv[kMTmax - 1];
        const bool valid = opix >= 0;
        unsigned long long fa2 = 0ull, fc2 = 0ull;            // fold: (rstd, rstd), (-mean*rstd, -mean*rstd) of this row's image
        if (has_fold && valid) {
          const float2 rs = s_rst[key];
          fa2 = pack2(rs.x, rs.x);
          fc2 = pack2(rs.y, rs.y);
        }
#pragma unroll
        for (int pc = 0; pc < PPM; ++pc) {
          const int u = pc & 1;                               // static double-buffer index (PPM is even)
          tmem_ld_wait();
          if (pc + 1 < PPM) {
            tmem_ld16_nowait(tlane + (uint32_t)(mt * NT + (pc + 1) * 16), rb[u ^ 1]);
          } else if (mt + 1 < tmt) {
            tmem_ld16_nowait(tlane + (uint32_t)((mt + 1) * NT), rb[u ^ 1]);
          } else {
            tc_fence_before();                                // last TMEM read of this tile is complete: hand the accumulators back
            mbar_arrive(smem_u32(&acc_empty[as]));
            if (ew == 0 && lane == 0) TRACE(it, 10);
          }
          const uint32_t* r = rb[u];
          unsigned long long v2[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v2[j] = pack2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
          if (has_fold) {
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const uint4 s1 = lds128(my_bias + (uint32_t)(pc * 64 + q4 * 16));
              const uint4 s2 = lds128(my_bias + (uint32_t)(p.c.Cout * 4 + pc * 64 + q4 * 16));
              v2[2 * q4] = fma2(v2[2 * q4], fa2, fma2(fc2, ((unsigned long long)s1.y << 32) | s1.x, ((unsigned long long)s2.y << 32) | s2.x));
              v2[2 * q4 + 1] = fma2(v2[2 * q4 + 1], fa2, fma2(fc2, ((unsigned long long)s1.w << 32) | s1.z, ((unsigned long long)s2.w << 32) | s2.z));
            }
          } else if (has_bias) {
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const uint4 bq = lds128(my_bias + (uint32_t)(pc * 64 + q4 * 16));     // broadcast LDS.128
              v2[2 * q4] = add2(v2[2 * q4], ((unsigned long long)bq.y << 32) | bq.x);
              v2[2 * q4 + 1] = add2(v2[2 * q4 + 1], ((unsigned long long)bq.w << 32) | bq.z);
            }
          }
          if (GEO == GEO_INIT && p.cls_w && valid) {
            const float* cls_row = p.cls_w + (long)(p.classes ? (int)p.classes[key] : p.pad_class) * p.c.Cout + n0 + col0 + pc * 16;
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const float4 bq = __ldg(reinterpret_cast<const float4*>(cls_row) + q4);
              v2[2 * q4] = add2(v2[2 * q4], pack2(bq.x, bq.y));
              v2[2 * q4 + 1] = add2(v2[2 * q4 + 1], pack2(bq.z, bq.w));
            }
          }
          if (res && valid) {
            const bf16* rrow = res + (long)opix * p.c.Cout + n0 + col0 + pc * 16;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const uint4 rr = *reinterpret_cast<const uint4*>(rrow + q * 8);
              float rf[8];
              unpack8(rr, rf);
#pragma unroll
              for (int e = 0; e < 4; ++e) v2[q * 4 + e] = add2(v2[q * 4 + e], pack2(rf[2 * e], rf[2 * e + 1]));
            }
          }
          // bf16 -> this warp's staging tile, row = lane, 16-byte chunk index XOR-swizzled (conflict-free both ways)
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            uint4 o;
            float a0, a1;
            unpack2(v2[q * 4 + 0], a0, a1); o.x = pack_bf16x2(a0, a1);
            unpack2(v2[q * 4 + 1], a0, a1); o.y = pack_bf16x2(a0, a1);
            unpack2(v2[q * 4 + 2], a0, a1); o.z = pack_bf16x2(a0, a1);
            unpack2(v2[q * 4 + 3], a0, a1); o.w = pack_bf16x2(a0, a1);
            sts128(my_wr + (uint32_t)(((pc * 2 + q) ^ my_swz) << 4), o);
          }
          if (do_stats) {
            // (sum, sum of squares) of this row's 16 columns: two independent packed chains each
            unsigned long long s0 = 0ull, q0 = 0ull, s1 = 0ull, q1 = 0ull;
            if (valid) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                s0 = add2(s0, v2[j]);
                q0 = fma2(v2[j], v2[j], q0);
                s1 = add2(s1, v2[4 + j]);
                q1 = fma2(v2[4 + j], v2[4 + j], q1);
              }
            }
            float sa0, sb0, qa0, qb0, sa1, sb1, qa1, qb1;
            unpack2(s0, sa0, sb0); unpack2(q0, qa0, qb0); unpack2(s1, sa1, sb1); unpack2(q1, qa1, qb1);
            cs += (sa0 + sb0) + (sa1 + sb1);
            cq += (qa0 + qb0) + (qa1 + qb1);
            // group bookkeeping (uniform): does the group end with this piece?
            const int cbase = n0 + col0 + pc * 16;
            const int g = cbase >> sh;
            const bool last_of_mt = pc == PPM - 1;
            if (last_of_mt || ((cbase + 16) >> sh) != g) {
#pragma unroll
              for (int i = 0; i < 6; ++i) val[i] = val[i + 2];
              val[6] = cs; val[7] = cq;
              cs = cq = 0.f;
              if (++nslots == 4 || last_of_mt) {
                stats_flush(val, key, valid, p.c.ostats, p.c.ogroups, g, nslots, lane);
                nslots = 0;
              }
            }
          }
        }
        // the warp's 32 x NCOL block is staged: coalesced 16-byte stores, LPR consecutive lanes cover one output row.  Batches
        // of 4 store instructions: all row lookups (SHFL) and staging reads (LDS) first, then the predicated stores
        __syncwarp();
#pragma unroll
        for (int i0 = 0; i0 < 32; i0 += 4 * RPI) {
          int ropix[4];
          uint4 o[4];
#pragma unroll
          for (int ii = 0; ii < 4; ++ii) {
            const int rrow = i0 + ii * RPI + lrow;            // < 32 by construction (32 / RPI = LPR is a multiple of 4)
            ropix[ii] = __shfl_sync(0xffffffffu, opix, rrow);
            o[ii] = lds128(my_stage + (uint32_t)(rrow * ROWB + ((lcol ^ ((rrow >> SWS) & SWM)) << 4)));
          }
#pragma unroll
          for (int ii = 0; ii < 4; ++ii)
            if (ropix[ii] >= 0) *reinterpret_cast<uint4*>(out_col + (long)ropix[ii] * p.c.Cout) = o[ii];
        }
        __syncwarp();
      }
      if (ew == 0 && lane == 0) TRACE(it, 11);
    }
    }
  } else if (warp == kLoaderW) {
    // =============================== weight loader ===============================
    // warp-uniform loop, one elected lane issues: one bulk copy (UBLKCP) of G taps (stage_bytes, contiguous in the blocked
    // weight image) per stage.  Copies of >= 16 KB are needed to reach the L2 -> shared streaming rate the MMAs consume.
    const bool leader = elect_one();
    int st = 0;
    uint32_t ph = 1;
    const int per_tile = p.n_pass * p.stages_per_pass;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const int n_tile = tile_geom(tile, p).n_tile;
      const uint8_t* wsrc = (const uint8_t*)p.c.w + (size_t)n_tile * per_tile * b_bytes;
      for (int s = 0; s < per_tile; ++s) {
        mbar_wait_relaxed(smem_u32(&empty_b[st]), ph);
        if (leader) {
          mbar_arrive_expect_tx(smem_u32(&full_b[st]), b_bytes);
          bulk_g2s(smem_u32(sB + st * b_bytes), wsrc + (size_t)s * b_bytes, b_bytes, smem_u32(&full_b[st]));
        }
        __syncwarp();
        if (++st == nst) { st = 0; ph ^= 1; }
      }
    }
  } else {
    // =============================== MMA issuer ===============================
    // The whole warp runs the loop (waits included) and ONE elected lane issues tcgen05.mma / tcgen05.commit: with a
    // warp-uniform loop every descriptor word is computed in uniform registers (UIADD3/UMOV feeding UTCHMMA directly).  An
    // `if (lane == 0)` loop instead makes ptxas wrap every MMA in an R2UR + vote loop (~160 clk per MMA issued, measured),
    // which alone caps the tensor pipe at ~40 %; see tools/mma_rate2.cu.
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc(128, NT);
    const uint32_t idesc_s2 = make_idesc(128, 256), idesc_s1 = make_idesc(128, 128);     // SWAP: N = pixels of the tile
    // ATMA: the operand tile is [P rows][64 B] SWIZZLE_64B (layout type 4 in descriptor bits 61-63, SBO = 512 B between 8-row groups,
    // LBO unused); a k16 step is 32 B inside the row, a tap offset of d rows is d * 64 B.  The swizzle is a function of the absolute
    // shared-memory address (buffers are 1 KB aligned), so the shifted views need no base-offset field (tools/micro/im2col_umma_test.cu)
    const uint32_t hi_a = ATMA ? ((512u >> 4) | (1u << 14) | (4u << 29)) : ((p.sbo_a >> 4) | (1u << 14)), hi_b = (p.sbo_b >> 4) | (1u << 14);
    const uint32_t lbo_a_f = ATMA ? (1u << 16) : (((p.lbo_a >> 4) & 0x3FFFu) << 16), lbo_b_f = ((p.lbo_b >> 4) & 0x3FFFu) << 16;
    const uint32_t a_units0 = (smem_u32(sA) >> 4) + (uint32_t)p.halo_lo * (ATMA ? 4u : 1u);          // 16-byte units
    const uint32_t a_buf_units = a_bytes >> 4;
    const uint32_t a_k16 = ATMA ? 2u : 2u * (p.lbo_a >> 4);
    const uint32_t a_half = p.a_half;
    const uint32_t b_units0 = smem_u32(sB) >> 4, b_stage_units = b_bytes >> 4, b_tap_units = tap_bytes >> 4, b_k16 = 2u * (p.lbo_b >> 4);
    const int G = p.G;
    int st = 0, cbuf = 0, it = 0;
    uint32_t ph = 0, cph = 0;
    // lean, fully unrolled issue paths: 3x3 (9 taps in stages of 3) and the 2x2 forms (4 taps in stages of 2)
    constexpr bool lean9 = LEAN && GEO == GEO_SAME;                     // the host launches LEAN only for 9 taps in stages of 3 ...
    constexpr bool lean4 = LEAN && (GEO == GEO_DOWN || GEO == GEO_UP);  // ... or 4 taps in stages of 2 (lean_ok below)
    const uint32_t b_lo0 = b_units0 | lbo_b_f;
    int dl9[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) dl9[t] = lean9 ? p.delta[t] : 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const TileGeom tg = tile_geom(tile, p);
      const int n_tile = tg.n_tile;
      const bool two = tg.mt == 2;
      const int phase = (GEO == GEO_UP) ? n_tile / p.tiles_per_phase : 0;
      const int as = it & 1;
      mbar_wait(smem_u32(&acc_empty[as]), ((it >> 1) & 1) ^ 1);      // epilogue has drained this accumulator set
      tc_fence_after();
      if (leader) TRACE(it, 4);
      const uint32_t d0 = tmem_base + (uint32_t)(as * 2 * NT), d1 = d0 + (uint32_t)NT;
      const bool tracing = DMN_EXP_MMATRACE && p.trace && blockIdx.x == (unsigned)p.trace_cta && it < 60;
      long long wait_a = 0, wait_b = 0;
      for (int c = 0; c < p.n_pass; ++c) {
        long long w0 = tracing ? clock64() : 0;
        mbar_wait(smem_u32(&full_a[cbuf]), cph);
        if (tracing) wait_a += clock64() - w0;
        tc_fence_after();
        if (c == 0 && leader) TRACE(it, 5);
        const uint32_t au = a_units0 + (uint32_t)cbuf * a_buf_units;
        if constexpr (SWAP && (lean9 || lean4)) {
          const uint32_t au_lo = au | lbo_a_f, acc0 = c ? 1u : 0u;
          const uint32_t ids = two ? idesc_s2 : idesc_s1;
          if constexpr (lean9) {
            issue_pass_swap<9, 3>(leader, d0, au_lo, dl9, b_lo0, b_stage_units, b_tap_units, hi_a, hi_b, a_k16, b_k16, ids, acc0, full_b, empty_b, nst, st, ph);
          } else {
            int dl4[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) dl4[t] = p.delta[phase * 16 + t];
            issue_pass_swap<4, 2>(leader, d0, au_lo, dl4, b_lo0, b_stage_units, b_tap_units, hi_a, hi_b, a_k16, b_k16, ids, acc0, full_b, empty_b, nst, st, ph);
          }
        } else if constexpr (lean9 || lean4) {
          const uint32_t au_lo = au | lbo_a_f, acc0 = c ? 1u : 0u;
          if constexpr (lean9) {
            if (two) issue_pass<9, 3, true>(leader, d0, d1, au_lo, dl9, b_lo0, b_stage_units, b_tap_units, hi_a, hi_b, a_k16, b_k16, idesc, acc0, full_b, empty_b, nst, st, ph, a_half);
            else issue_pass<9, 3, false>(leader, d0, d1, au_lo, dl9, b_lo0, b_stage_units, b_tap_units, hi_a, hi_b, a_k16, b_k16, idesc, acc0, full_b, empty_b, nst, st, ph, a_half);
          } else {
            int dl4[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) dl4[t] = p.delta[phase * 16 + t];
            if (two) issue_pass<4, 2, true>(leader, d0, d1, au_lo, dl4, b_lo0, b_stage_units, b_tap_units, hi_a, hi_b, a_k16, b_k16, idesc, acc0, full_b, empty_b, nst, st, ph, a_half);
            else issue_pass<4, 2, false>(leader, d0, d1, au_lo, dl4, b_lo0, b_stage_units, b_tap_units, hi_a, hi_b, a_k16, b_k16, idesc, acc0, full_b, empty_b, nst, st, ph, a_half);
          }
        } else
        for (int s = 0; s < p.stages_per_pass; ++s) {
          const int t0 = s * G;
          w0 = tracing ? clock64() : 0;
          mbar_wait(smem_u32(&full_b[st]), ph);
          if (tracing) wait_b += clock64() - w0;
          tc_fence_after();
          const uint32_t bs = b_units0 + (uint32_t)st * b_stage_units;
          const uint32_t acc0 = c ? 1u : 0u;
          if constexpr (SWAP) {
            const uint32_t ids = two ? idesc_s2 : idesc_s1;
            for (int g = 0; g < G; ++g) {
              const int t = t0 + g;
              const uint32_t a0 = au + (uint32_t)p.delta[phase * 16 + t];
              const uint32_t b0 = bs + (uint32_t)g * b_tap_units;
              issue_tap_swap(leader, d0, (a0 & 0x3FFFu) | lbo_a_f, (b0 & 0x3FFFu) | lbo_b_f, hi_a, hi_b, a_k16, b_k16, ids, (c | t) ? 1u : 0u);
            }
          } else if (two) {
            // 256-row tiles: per-tap issue (4 MMAs = 256 clk of tensor work cover the ~20 uniform instructions of the next tap);
            // batching a whole stage's descriptors first measured slower here (the MMA queue drains during the longer prologue)
            for (int g = 0; g < G; ++g) {
              const int t = t0 + g;
              const uint32_t a0 = au + (uint32_t)p.delta[phase * 16 + t];
              const uint32_t b0 = bs + (uint32_t)g * b_tap_units;
              const uint32_t acc = (c | t) ? 1u : 0u;
              const uint64_t bd0 = ((uint64_t)hi_b << 32) | ((b0 & 0x3FFFu) | lbo_b_f);
              const uint64_t bd1 = ((uint64_t)hi_b << 32) | (((b0 + b_k16) & 0x3FFFu) | lbo_b_f);
              const uint64_t ad00 = ((uint64_t)hi_a << 32) | ((a0 & 0x3FFFu) | lbo_a_f);
              const uint64_t ad01 = ((uint64_t)hi_a << 32) | (((a0 + a_half) & 0x3FFFu) | lbo_a_f);
              const uint64_t ad10 = ((uint64_t)hi_a << 32) | (((a0 + a_k16) & 0x3FFFu) | lbo_a_f);
              const uint64_t ad11 = ((uint64_t)hi_a << 32) | (((a0 + a_k16 + a_half) & 0x3FFFu) | lbo_a_f);
              if (leader) {
                umma_bf16(d0, ad00, bd0, idesc, acc);
                umma_bf16(d1, ad01, bd0, idesc, acc);
                umma_bf16(d0, ad10, bd1, idesc, 1u);
                umma_bf16(d1, ad11, bd1, idesc, 1u);
              }
            }
          } else {
            if (G == 3) issue_stage<3, false>(p, leader, d0, d1, au, bs, phase * 16 + t0, t0, acc0, idesc, hi_a, hi_b, lbo_a_f, lbo_b_f, a_k16, b_k16, b_tap_units, a_half);
            else if (G == 2) issue_stage<2, false>(p, leader, d0, d1, au, bs, phase * 16 + t0, t0, acc0, idesc, hi_a, hi_b, lbo_a_f, lbo_b_f, a_k16, b_k16, b_tap_units, a_half);
            else issue_stage<1, false>(p, leader, d0, d1, au, bs, phase * 16 + t0, t0, acc0, idesc, hi_a, hi_b, lbo_a_f, lbo_b_f, a_k16, b_k16, b_tap_units, a_half);
          }
          if (leader) umma_commit(smem_u32(&empty_b[st]));     // frees the weight stage once these MMAs retire
          __syncwarp();
          if (++st == nst) { st = 0; ph ^= 1; }
        }
        if (leader) umma_commit(smem_u32(&empty_a[cbuf]));      // frees the operand buffer
        __syncwarp();
        if (++cbuf == AB) { cbuf = 0; cph ^= 1; }
      }
      if (leader) {
        umma_commit(smem_u32(&acc_full[as]));        // accumulators of this tile complete -> epilogue
        TRACE(it, 6);
        if (tracing) { p.trace[16 * it + 12] = wait_a; p.trace[16 * it + 13] = wait_b; }
      }
      __syncwarp();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaW) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
  if (DMN_TC_TRACE_BUILD && p.trace && blockIdx.x == (unsigned)p.trace_cta && tid == 0) p.trace[1001] = clock64();     // kernel exit
}

static size_t smem_fixed_bytes(const Params& p) {
  const int ncol = p.NT >= 64 ? p.NT / 2 : p.NT;
  return (size_t)p.abuf * p.a_bytes + (2 * kStagesMax + 3 * kABufMax + 4) * 8 + 16 + (size_t)kNimgMax * kGroupsMax * 8 +
         2 * (size_t)p.P * 4 + 128 + (p.c.pro != PRO_NONE ? 3 * (size_t)p.c.C1 * 4 + 16 : 0) + (size_t)kEpiWarps * (32 * ncol * 2 + ncol * 8) + 128 +
         2 * (size_t)p.c.Cout * 4 + (p.c.fold_s1 ? (size_t)p.c.B * 8 : 0) + 32;
}
static size_t smem_bytes(const Params& p) { return smem_fixed_bytes(p) + (size_t)p.nstage * p.stage_bytes; }
// taps per weight stage: a whole filter row for 3x3, a tap pair for the 2x2 forms; bulk copies of 16-24 KB stream well
static bool pick_stages(Params& p) {
  const size_t fixed = smem_fixed_bytes(p);
  for (int G = (p.ntap % 3 == 0 ? 3 : (p.ntap % 2 == 0 ? 2 : 1)); G >= 1; G = (G == 3 ? 1 : G - 1)) {
    const size_t stage = (size_t)G * 4 * p.NT * 16;
    if (fixed + 3 * stage > kSmemLimit) continue;
    int n = (int)((kSmemLimit - fixed) / stage);
    p.G = G;
    p.stages_per_pass = p.ntap / G;
    p.stage_bytes = (uint32_t)stage;
    p.nstage = n > kStagesMax ? kStagesMax : n;
    return true;
  }
  return false;
}

static int pick_nt(int cout) { return cout % 128 == 0 ? 128 : (cout % 64 == 0 ? 64 : (cout % 32 == 0 ? 32 : 0)); }

static int num_sms() { return current_device_sms(); }

// Swapped operand roles (weights on the TMEM lanes, ONE M128 x N256 instruction per k-step of a 256-position tile: the tensor core reads
// 12 KB instead of 16 KB of shared memory per 128 clk).  DMN_CONV_SWAP = 1: every eligible conv, 0: none, unset: the measured rule in
// fill_params (maps of at least 64 positions per image with >= 8 passes, or plain 3x3) -- on the TMA operand feed the form
// is 4-9 % faster there and slower for single-round 4x4 maps and the 4-pass GroupNorm-prologue / transposed convs (profiles/README.md)
static int swap_mode() {
  static const int m = [] {
    const char* e = getenv("DMN_CONV_SWAP");
    return !e ? 2 : (e[0] == '1' ? 1 : (e[0] == '0' ? 0 : 2));
  }();
  return m;
}

// ---- TMA operand path ----
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const int*, const int*, cuuint32_t,
                                   cuuint32_t, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeIm2colFn im2col_encoder() {
  static const EncodeIm2colFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
    return (EncodeIm2colFn)f;
  }();
  return fn;
}
static bool atma_enabled() {
  static const bool on = [] {
    const char* e = getenv("DMN_CONV_TMA");
    return !(e && e[0] == '0') && im2col_encoder() != nullptr;      // DMN_CONV_TMA=0: the cp.async operand producers (A/B comparison)
  }();
  return on;
}
// im2col view of one NHWC bf16 source whose traversal order IS the engine's flat padded position order: the bounding box adds the pad
// column / row in front (lower corner -1; nothing behind: upper corner 0), stride-2 traversal for the k4s2 form; positions outside the
// tensor (pads, images < 0 or >= B) arrive as zeros.  One copy = P positions x 32 channels, SWIZZLE_64B rows of 64 bytes
static bool encode_window_map(CUtensorMap* m, const void* src, int C, int B, int H, int W, int geo, int pad, int P) {
  EncodeIm2colFn fn = im2col_encoder();
  if (!fn || !src || (reinterpret_cast<uintptr_t>(src) & 15)) return false;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  const int lo = geo == GEO_DOWN ? -1 : -pad;
  int lower[2] = {lo, lo}, upper[2] = {0, 0};
  const cuuint32_t step = geo == GEO_DOWN ? 2 : 1;
  cuuint32_t estr[4] = {1, step, step, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(src), dims, strides, lower, upper, (cuuint32_t)kCk, (cuuint32_t)P, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static bool fill_params(const ConvP& c, int geo, Params& p) {
  p = Params();
  p.c = c;
  p.geo = geo;
  p.NT = pick_nt(c.Cout);
  if (!p.NT) return false;
  p.H = c.Hin; p.W = c.Win; p.HW = c.Hin * c.Win;
  p.ksize = c.ksize;
  p.tiles_per_phase = c.Cout / p.NT;
  p.n_tiles_n = (geo == GEO_UP ? 4 : 1) * p.tiles_per_phase;
  p.nt_shift = p.NT == 128 ? 7 : (p.NT == 64 ? 6 : 5);
  int halo_hi = 0;
  if (geo == GEO_SAME) {
    if (c.ksize != 1 && c.ksize != 3) return false;
    if (c.C1 <= 0 || c.C1 % kCk || c.C2 % kCk) return false;
    p.ntap = c.ksize * c.ksize;
    p.pad = c.ksize == 3 ? 1 : 0;
    p.Wv = c.Win + p.pad;
    p.S = (c.Hin + p.pad) * p.Wv;
    p.halo_lo = halo_hi = c.ksize == 3 ? p.Wv + 1 : 0;
    p.n_pass = (c.C1 + c.C2) / kCk;
  } else if (geo == GEO_DOWN) {
    if (c.C2 != 0 || c.C1 % kCk || (c.Hin & 1) || (c.Win & 1) || c.pro != PRO_NONE || c.ostats || c.res) return false;
    if (c.Hin / 2 + 1 > 127 || c.B >= (1 << 17)) return false;
    p.ntap = 4;
    p.pad = 0;
    p.Wv = c.Win / 2 + 1;
    p.S = (c.Hin / 2 + 1) * p.Wv;
    p.halo_lo = 0;
    halo_hi = p.Wv + 1;
    p.n_pass = 4 * c.C1 / kCk;
  } else if (geo == GEO_UP) {
    if (c.C2 != 0 || c.C1 % kCk || c.pro != PRO_NONE || c.ostats || c.res) return false;
    p.ntap = 4;
    p.pad = 1;
    p.Wv = c.Win + 1;
    p.S = (c.Hin + 1) * p.Wv;
    p.halo_lo = halo_hi = p.Wv + 1;
    p.n_pass = c.C1 / kCk;
  } else {
    if (7 * c.C1 > kCk || c.C2 != 0) return false;
    p.ntap = 7;
    p.pad = 0;
    p.Wv = c.Win;
    p.S = (c.Hin + 3) * p.Wv;
    p.halo_lo = halo_hi = 3 * p.Wv;
    p.n_pass = 1;
  }
  p.total_flat = (long)c.B * p.S;
  if (p.total_flat + 4096 >= (1L << 30) || (long)c.B * 4 * p.HW >= (1L << 30)) return false;   // 32-bit index arithmetic
  if (geo != GEO_INIT && (long)c.B * p.HW * (c.C1 > c.C2 ? c.C1 : c.C2) * 2 >= (1L << 32)) return false;   // 32-bit operand byte offsets
  {
    // two accumulators (256 rows) per tile halve the weight traffic per FLOP; with few tiles one accumulator keeps more SMs busy
    const long tiles2 = (p.total_flat + 255) / 256 * p.n_tiles_n;
    p.mt = tiles2 >= num_sms() ? 2 : 1;
    p.mcta = 128 * p.mt;
  }
  p.halo_hi = halo_hi;
  {
    // mixed tiling: whole rounds of 256-row tiles, the remainder in 128-row tiles (the last round then costs half)
    const long nsm = num_sms();
    const long m2 = (p.total_flat + 255) / 256, t2 = m2 * p.n_tiles_n;
    if (p.mt == 2) {
      long big_m = m2;
      if (t2 % nsm != 0) big_m = (t2 / nsm) * nsm / p.n_tiles_n;       // m-tiles inside the whole rounds
      long rem = p.total_flat - big_m * 256;
      long small_m = rem > 0 ? (rem + 127) / 128 : 0;
      // a 128-row tile costs ~0.6 of a 256-row tile (it streams the same weights): mix only when the estimate is lower
      const double cost_uniform = (double)((t2 + nsm - 1) / nsm);
      const double cost_mixed = (double)(t2 / nsm) + 0.6 * (double)((small_m * p.n_tiles_n + nsm - 1) / nsm);
      if (cost_mixed >= cost_uniform - 0.05) {
        big_m = m2;
        rem = 0;
        small_m = 0;
      }
      p.n_big_tiles = (int)(big_m * p.n_tiles_n);
      p.big_rows = (int)(big_m * 256);
      p.total_tiles = p.n_big_tiles + (int)(small_m * p.n_tiles_n);
    } else {
      p.n_big_tiles = 0;
      p.big_rows = 0;
      p.total_tiles = (int)((p.total_flat + 127) / 128) * p.n_tiles_n;
    }
    p.m_tiles = p.total_tiles / p.n_tiles_n;
  }
  p.P = p.mcta + p.halo_lo + halo_hi;
  p.PA = p.P;
  while (p.PA % 8 != 2) ++p.PA;
  if (geo != GEO_INIT && (4 * p.P + kProdThreads - 1) / kProdThreads > kMaxItems) return false;
  if (kMcta / p.S + 3 > kNimgMax || p.S < 16) return false;
  p.lbo_a = (uint32_t)p.PA * 16u;
  p.sbo_a = 128u;
  p.a_bytes = 4u * (uint32_t)p.PA * 16u;
  p.a_half = 128u;
  p.atma = 0;
  p.lbo_b = (uint32_t)p.NT * 16u;
  p.sbo_b = 128u;
  p.tmem_cols = 32;
  while (p.tmem_cols < (uint32_t)(2 * 2 * p.NT)) p.tmem_cols <<= 1;    // double-buffered pairs of accumulators, power of two
  p.cpg_in = 1;
  p.cpg_in_shift = p.cpg_out_shift = 0;
  p.inv_cnt_in = 0.f;
  if (c.Cout > 2048 || (c.fold_s1 && c.B > 4096)) return false;      // per-CTA staging of the bias / fold vectors and image statistics
  if (c.fold_s1) {
    if (geo != GEO_SAME || c.ksize != 1 || c.pro != PRO_NONE || !c.fold_s2 || !c.pstats || c.pgroups != 1 || c.C2 != 0) return false;
    p.inv_cnt_in = 1.f / (float)(p.HW * c.C1);
  }
  if (c.pro & PRO_GN) {
    if (geo != GEO_SAME || c.C2 != 0 || c.pgroups <= 0 || c.pgroups > kGroupsMax || c.C1 % c.pgroups) return false;
    p.cpg_in = c.C1 / c.pgroups;
    if (p.cpg_in % 8 || (p.cpg_in & (p.cpg_in - 1))) return false;
    while ((1 << p.cpg_in_shift) < p.cpg_in) ++p.cpg_in_shift;
    p.inv_cnt_in = 1.f / (float)(p.HW * p.cpg_in);
  } else if (c.pro != PRO_NONE) {
    // without the GroupNorm apply only the FiLM signal prologue exists: LeakyReLU (+ per-sample / per-step encoding)
    if (geo != GEO_SAME || c.C2 != 0 || !(c.pro & PRO_LRELU) || (c.pro & ~(PRO_LRELU | PRO_TEMB))) return false;
  }
  p.cpg_out = 1;
  if (c.ogroups > 0) {
    if (c.Cout % c.ogroups) return false;
    p.cpg_out = c.Cout / c.ogroups;
    if (p.cpg_out % 16 || (p.cpg_out & (p.cpg_out - 1))) return false;
    while ((1 << p.cpg_out_shift) < p.cpg_out) ++p.cpg_out_shift;
    if (p.NT < 64) return false;     // each epilogue warp must own whole 16-channel pairs
  }
  if (p.S > 8192 - 1024 || p.Wv > 128) return false;     // vdecode_rel exactness
  p.magic_S = (uint32_t)(((1ull << 26) + p.S - 1) / p.S);
  p.magic_W = (uint32_t)(((1ull << 24) + p.Wv - 1) / p.Wv);
  p.magic64_S = ~0ull / (unsigned long long)p.S + 1ull;
  for (int ph = 0; ph < 4; ++ph)
    for (int t = 0; t < 16; ++t) p.delta[ph * 16 + t] = t < p.ntap ? tap_delta(p, geo, t, ph) : 0;
  p.abuf = (geo == GEO_SAME && p.NT == 128 && p.ntap == 1 && c.pro == PRO_NONE) ? kABufOne : kABuf;
  // plain swapped-role instantiations (launch<>: hot path without prologue)
  {
    const bool eligible = geo != GEO_INIT && p.NT == 128 && !(c.pro & PRO_LRELU) && !c.res && !c.fold_s1 && (geo != GEO_SAME || p.ntap == 9);
    // the rule depends on the per-image geometry only, never on the batch: the two forms sum the GroupNorm statistics in different
    // fp32 orders, so a sample must meet the same form whatever batch it is part of (batch-slice invariance)
    const bool rule = atma_enabled() && p.S >= 64 && (p.n_pass >= 8 || (geo == GEO_SAME && c.pro == PRO_NONE));
    p.swap = eligible && (swap_mode() == 1 || (swap_mode() == 2 && rule));
  }
  if (p.swap && c.pro == PRO_NONE) p.abuf = kABufPlain;
  // the GroupNorm-prologue instantiation (PRO = 1) is launched for 128-column tiles without residual / fold / FiLM (launch<>)
  if (geo == GEO_SAME && p.NT == 128 && c.pro != PRO_NONE && !(c.pro & PRO_LRELU) && !c.res && !c.fold_s1) p.abuf = kABufPro;
  // TMA operand path: the hot instantiations (launch<>: 128-column tiles, 3x3 / k4s2 / transposed k4s2, no FiLM / residual / fold terms)
  const bool hot = geo != GEO_INIT && p.NT == 128 && !(c.pro & PRO_LRELU) && !c.res && !c.fold_s1 &&
                   ((geo == GEO_SAME && (p.ntap == 9 || (p.ntap == 1 && c.pro == PRO_NONE))) || geo == GEO_DOWN || geo == GEO_UP);
  // (prologue form: power-of-two group count <= 16, at most one (mean, rstd) table entry per producer thread)
  const bool pro_ok = c.pro == PRO_NONE || ((c.pro & PRO_GN) && kNimgMax * c.pgroups <= kProdThreads && c.pgroups <= 16 && (c.pgroups & (c.pgroups - 1)) == 0);
  if (hot && pro_ok && atma_enabled() && p.P <= 1024 && p.halo_lo < p.S) {
    Params q = p;
    q.atma = 1;
    q.a_bytes = ((uint32_t)q.P * 64u + 1023u) & ~1023u;
    q.a_half = 512u;
    for (int i = 0; i < 64; ++i) q.delta[i] *= 4;               // tap offsets in 16-byte units: one row of the tile is 64 bytes
    bool ok = pick_stages(q);
    if (ok && c.src1) {          // (shape queries come without pointers)
      ok = encode_window_map(&q.tm_a1, c.src1, c.C1, c.B, c.Hin, c.Win, geo, q.pad, q.P);
      if (ok && c.C2 > 0) ok = encode_window_map(&q.tm_a2, c.src2, c.C2, c.B, c.Hin, c.Win, geo, q.pad, q.P);
    }
    if (ok) {
      p = q;
      return true;
    }
  }
  return pick_stages(p);
}

static int geo_of(const ConvP& c) { return c.mode == CONV_SAME ? GEO_SAME : (c.mode == CONV_DOWN ? GEO_DOWN : GEO_UP); }

// > 48 KB of dynamic shared memory is a per-kernel, per-device opt-in
static cudaError_t ensure_smem_attr(const void* fn) {
  static std::vector<std::pair<int, const void*>> done;
  int dev = 0;
  cudaGetDevice(&dev);
  for (auto& d : done)
    if (d.first == dev && d.second == fn) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit);
  if (e == cudaSuccess) done.emplace_back(dev, fn);
  return e;
}
// launch log (dmn_debug_conv_log): one record of kLogInts int32 per launch, written on the host when the launch is enqueued (a replayed
// graph records nothing).  Tests read it to show which instantiation and tiling regime a convolution ran.  Off until first read.
//   [0, 1] kernel function pointer (low, high 32 bits), [2] geo, [3] ksize, [4] C1, [5] C2, [6] Cout, [7] H (input), [8] B, [9] pro,
//   [10] pgroups, [11] ogroups, [12] swap, [13] atma, [14] mt, [15] n_big_tiles, [16] total_tiles, [17] grid, [18] threads,
//   [19] n_tiles_n, [20] big_rows, [21] total_flat, [22] n_pass, [23] reserved; [24, 64) kernel name (cudaFuncGetName), NUL-terminated
constexpr int kLogInts = 64, kLogNameAt = 24, kLogMax = 1 << 16;
static std::mutex g_log_mu;
static std::vector<std::array<int32_t, kLogInts>> g_log;
static std::atomic<bool> g_log_on{false};
static void log_launch(const void* fn, int grid, int threads, const Params& p) {
  if (!g_log_on.load(std::memory_order_relaxed)) return;
  std::array<int32_t, kLogInts> r{};
  const uint64_t f = (uint64_t)(uintptr_t)fn;
  const int32_t v[kLogNameAt] = {(int32_t)(uint32_t)f, (int32_t)(uint32_t)(f >> 32), p.geo, p.ksize, p.c.C1, p.c.C2, p.c.Cout, p.H, p.c.B,
                                 p.c.pro, p.c.pgroups, p.c.ogroups, p.swap, p.atma, p.mt, p.n_big_tiles, p.total_tiles, grid, threads,
                                 p.n_tiles_n, p.big_rows, (int32_t)p.total_flat, p.n_pass, 0};
  std::memcpy(r.data(), v, sizeof(v));
  const char* name = nullptr;
  if (cudaFuncGetName(&name, fn) == cudaSuccess && name)
    std::strncpy(reinterpret_cast<char*>(r.data() + kLogNameAt), name, (kLogInts - kLogNameAt) * 4 - 1);
  else
    cudaGetLastError();
  std::lock_guard<std::mutex> g(g_log_mu);
  if (g_log.size() < (size_t)kLogMax) g_log.push_back(r);
}

typedef void (*ConvKernel)(Params);

static cudaError_t launch_kernel(ConvKernel kern, int grid, int threads, const Params& p, cudaStream_t st) {
  const cudaError_t e = ensure_smem_attr((const void*)kern);
  if (e != cudaSuccess) return e;
  log_launch((const void*)kern, grid, threads, p);
  return launch_pdl(kern, dim3(grid), dim3(threads), smem_bytes(p), st, p);
}

// The hot instantiations: 128-column tiles without FiLM, residual or fold terms, on the operand feed ATMA with operand roles SWAP.
// Sets `ew16` when it picks a 16-epilogue-warp form.
template <int GEO, bool SWAP, bool ATMA>
static ConvKernel hot_kernel(bool pro, bool lean, bool lean_shape, bool& ew16) {
  if constexpr (GEO == GEO_SAME) {
    if (pro) return lean ? conv_tcgen05_kernel<GEO, 128, false, true, false, 1, 8, SWAP, ATMA> : conv_tcgen05_kernel<GEO, 128, false, false, false, 1, 8, SWAP, ATMA>;
    if (lean) return conv_tcgen05_kernel<GEO, 128, false, true, false, 0, 8, SWAP, ATMA>;
    // epilogue-bound plain 3x3 tiles (fewer than kLeanMinPass passes): 16 epilogue warps; ncu then shows the epilogue waiting for the
    // accumulators 24 % of the time, so these tiles take the lean issue path as well
    ew16 = true;
    return lean_shape ? conv_tcgen05_kernel<GEO, 128, false, true, false, 0, 16, SWAP, ATMA> : conv_tcgen05_kernel<GEO, 128, false, false, false, 0, 16, SWAP, ATMA>;
  } else {
    return lean ? conv_tcgen05_kernel<GEO, 128, false, true, false, 0, 8, SWAP, ATMA> : conv_tcgen05_kernel<GEO, 128, false, false, false, 0, 8, SWAP, ATMA>;
  }
}

template <int GEO>
static int launch(Params p, cudaStream_t st) {
  static const bool trace_on = [] {
    const char* e = getenv("DMN_TC_TRACE");
    return e && e[0] == '1';
  }();
  if (trace_on) {
    void* sym = nullptr;
    DMN_CUDA_CHECK(cudaGetSymbolAddress(&sym, g_trace));
    DMN_CUDA_CHECK(cudaMemsetAsync(sym, 0, sizeof(long long) * 1024, st));
    p.trace = (long long*)sym;
    p.trace_cta = 3;
  }
  const int grid = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
  const bool film = (p.c.pro & PRO_LRELU) != 0;
  const bool extra = p.c.res != nullptr || p.c.fold_s1 != nullptr;
  ConvKernel kern = nullptr;
  bool ew16 = false;
  if (GEO == GEO_SAME && p.NT == 128 && p.ntap == 1 && p.c.pro == PRO_NONE) {
    // 1x1 convolutions (to_qkv with the folded GroupNorm, to_out, res_conv): table-free producers, 16 epilogue warps
    ew16 = true;
    if (p.atma) kern = conv_tcgen05_kernel<GEO_SAME, 128, false, false, false, 3, 16, false, true>;
    else if (extra) kern = conv_tcgen05_kernel<GEO_SAME, 128, false, false, true, 3, 16>;
    else kern = conv_tcgen05_kernel<GEO_SAME, 128, false, false, false, 3, 16>;
  } else if (GEO != GEO_INIT && p.NT == 128 && !film && !extra) {
    if constexpr (GEO != GEO_INIT) {
      const bool pro = GEO == GEO_SAME && p.c.pro != PRO_NONE;
      // lean (unrolled) issue path: 9 taps in stages of 3, or 4 in stages of 2, with at least kLeanMinPass passes.  The 2x2 forms on
      // the TMA feed with plain roles take it whatever the pass count (transposed 16x16 -> 32x32 conv 0.0392 -> 0.0299 ms)
      const bool lean_shape = (GEO == GEO_SAME && p.ntap == 9 && p.G == 3) || (GEO != GEO_SAME && p.ntap == 4 && p.G == 2);
      const bool lean = lean_shape && (p.n_pass >= kLeanMinPass || (GEO != GEO_SAME && p.atma && !p.swap));
      const auto pick = p.swap ? (p.atma ? hot_kernel<GEO, true, true> : hot_kernel<GEO, true, false>)
                               : (p.atma ? hot_kernel<GEO, false, true> : hot_kernel<GEO, false, false>);
      kern = pick(pro, lean, lean_shape, ew16);
    }
  } else if (GEO == GEO_SAME && film) {
    kern = p.NT == 128 ? conv_tcgen05_kernel<GEO_SAME, 128, true> : (p.NT == 64 ? conv_tcgen05_kernel<GEO_SAME, 64, true> : conv_tcgen05_kernel<GEO_SAME, 32, true>);
  } else {
    kern = p.NT == 128 ? conv_tcgen05_kernel<GEO, 128> : (p.NT == 64 ? conv_tcgen05_kernel<GEO, 64> : conv_tcgen05_kernel<GEO, 32>);
  }
  DMN_CUDA_CHECK(launch_kernel(kern, grid, ew16 ? kThreads16 : kThreads, p, st));
  count_launch();
  DMN_LAUNCH_CHECK("conv_tcgen05");
  return 0;
}

}  // namespace tc

bool conv_tcgen05_supported(const ConvP& c) {
  tc::Params p;
  return tc::fill_params(c, tc::geo_of(c), p);
}
bool init_conv_tcgen05_supported(int Cin, int S, int Cout, int B) {
  ConvP c;
  c.C1 = Cin; c.Hin = c.Win = S; c.Cout = Cout; c.B = B;
  tc::Params p;
  return tc::fill_params(c, tc::GEO_INIT, p);
}

size_t conv_tcgen05_weight_bytes(int mode, int ksize, int cin, int cout) {
  const int taps = (mode == CONV_SAME) ? ksize * ksize : 16;
  return (size_t)cout * cin * taps * 2;
}
size_t init_conv_tcgen05_weight_bytes(int cout) { return (size_t)cout * 7 * tc::kCk * 2; }

// blocked bf16 weight image [n_tile][pass][tap][kchunk 0..3][n 0..NT-1][8 channels]
void conv_tcgen05_pack_weights(int mode, int ksize, int cin, int cout, const float* w, void* dst_host) {
  const int NT = tc::pick_nt(cout);
  bf16* dst = (bf16*)dst_host;
  size_t o = 0;
  if (mode == CONV_SAME) {
    const int taps = ksize * ksize;
    for (int nt = 0; nt < cout / NT; ++nt)
      for (int c = 0; c < cin / tc::kCk; ++c)
        for (int t = 0; t < taps; ++t)
          for (int kc = 0; kc < 4; ++kc)
            for (int n = 0; n < NT; ++n)
              for (int e = 0; e < 8; ++e) {
                const int co = nt * NT + n, ci = c * tc::kCk + kc * 8 + e;
                dst[o++] = __float2bfloat16_rn(w[((long)co * cin + ci) * taps + t]);
              }
  } else if (mode == CONV_DOWN) {
    // Conv2d weight [co][ci][ky][kx], k4 s2 p1.  virtual channel = sub*C + ci, sub = sy*2+sx; tap t = du*2+dv;
    // ky = 2*du + sy, kx = 2*dv + sx
    for (int nt = 0; nt < cout / NT; ++nt)
      for (int c = 0; c < 4 * cin / tc::kCk; ++c)
        for (int t = 0; t < 4; ++t)
          for (int kc = 0; kc < 4; ++kc)
            for (int n = 0; n < NT; ++n)
              for (int e = 0; e < 8; ++e) {
                const int vc = c * tc::kCk + kc * 8 + e, sub = vc / cin, ci = vc % cin;
                const int ky = 2 * (t >> 1) + (sub >> 1), kx = 2 * (t & 1) + (sub & 1);
                const int co = nt * NT + n;
                dst[o++] = __float2bfloat16_rn(w[(((long)co * cin + ci) * 4 + ky) * 4 + kx]);
              }
  } else {
    // ConvTranspose2d weight [ci][co][ky][kx], k4 s2 p1.  n_tile = phase*(cout/NT) + ct, phase = py*2+px;
    // tap t = a*2+b: dy = py ? (a ? 0 : +1) : (a ? -1 : 0) (dx likewise); ky = py + 1 - 2*dy
    for (int ph = 0; ph < 4; ++ph)
      for (int ct = 0; ct < cout / NT; ++ct)
        for (int c = 0; c < cin / tc::kCk; ++c)
          for (int t = 0; t < 4; ++t) {
            const int py = ph >> 1, px = ph & 1, a = t >> 1, b = t & 1;
            const int dy = py ? (a ? 0 : 1) : (a ? -1 : 0), dx = px ? (b ? 0 : 1) : (b ? -1 : 0);
            const int ky = py + 1 - 2 * dy, kx = px + 1 - 2 * dx;
            for (int kc = 0; kc < 4; ++kc)
              for (int n = 0; n < NT; ++n)
                for (int e = 0; e < 8; ++e) {
                  const int ci = c * tc::kCk + kc * 8 + e, co = ct * NT + n;
                  dst[o++] = __float2bfloat16_rn(w[(((long)ci * cout + co) * 4 + ky) * 4 + kx]);
                }
          }
  }
}

// init conv weight [co][ch][7][7] -> [n_tile][tap ky][kchunk][n][8], virtual channel vc = kx*Cin + ch
void init_conv_tcgen05_pack_weights(int cin, int cout, const float* w, void* dst_host) {
  const int NT = tc::pick_nt(cout);
  bf16* dst = (bf16*)dst_host;
  size_t o = 0;
  for (int nt = 0; nt < cout / NT; ++nt)
    for (int ky = 0; ky < 7; ++ky)
      for (int kc = 0; kc < 4; ++kc)
        for (int n = 0; n < NT; ++n)
          for (int e = 0; e < 8; ++e) {
            const int vc = kc * 8 + e, kx = vc / cin, ch = vc % cin, co = nt * NT + n;
            dst[o++] = __float2bfloat16_rn(kx < 7 ? w[(((long)co * cin + ch) * 7 + ky) * 7 + kx] : 0.f);
          }
}

int conv_tcgen05_read_trace(long long* out, int n) {
  if (n > 1024) n = 1024;
  DMN_CUDA_CHECK(cudaDeviceSynchronize());
  DMN_CUDA_CHECK(cudaMemcpyFromSymbol(out, tc::g_trace, (size_t)n * sizeof(long long)));
  return 0;
}

int conv_tcgen05_read_log(int32_t* out, int cap) {
  std::lock_guard<std::mutex> g(tc::g_log_mu);
  tc::g_log_on.store(true);
  const int n = (int)tc::g_log.size();
  for (int i = 0; i < n && i < cap && out; ++i) std::memcpy(out + (size_t)i * tc::kLogInts, tc::g_log[i].data(), sizeof(int32_t) * tc::kLogInts);
  tc::g_log.clear();
  return n;
}

int conv_tcgen05(const ConvP& c, cudaStream_t st) {
  tc::Params p;
  const int geo = tc::geo_of(c);
  if (!tc::fill_params(c, geo, p)) return fail(-2, "conv_tcgen05: unsupported convolution shape");
  if (geo == tc::GEO_SAME) return tc::launch<tc::GEO_SAME>(p, st);
  if (geo == tc::GEO_DOWN) return tc::launch<tc::GEO_DOWN>(p, st);
  return tc::launch<tc::GEO_UP>(p, st);
}

int init_conv_tcgen05(const InitConvP& q, cudaStream_t st) {
  ConvP c;
  c.src1 = q.x; c.C1 = q.Cin; c.B = q.B; c.Hin = c.Win = q.S; c.Hout = c.Wout = q.S; c.Cout = q.Cout;
  c.w = q.w; c.bias = q.bias; c.out = q.out;
  tc::Params p;
  if (!tc::fill_params(c, tc::GEO_INIT, p)) return fail(-2, "init_conv_tcgen05: unsupported shape");
  p.cls_w = q.cls_w;
  p.classes = q.classes;
  p.pad_class = q.pad_class;
  return tc::launch<tc::GEO_INIT>(p, st);
}

}  // namespace dmn
