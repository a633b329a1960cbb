// attn_fused.cu -- Residual(PreNorm(dim, LinearAttention(dim))) as ONE kernel on the 5th-generation tensor cores (sm_100a only).
//
//   reference: utils.py:68-93 (Residual, PreNorm = GroupNorm(1, dim)), parts/mha.py:33-59 (LinearAttention: to_qkv 1x1 without bias,
//   q = softmax_d(q) * scale, k = softmax_n(k), ctx = k v^T, out = ctx^T q, to_out = Conv1x1 + GroupNorm(1, dim)), result + x.
//
// Images with fewer than 128 tokens (8x8, 4x4 maps) take one tile each: the TMA box only brings the image's N rows, the rest of the tile
// stays zero, the padded token columns are masked out of the k softmax and the padded rows are neither counted nor stored.
// One persistent CTA per SM walks whole images; per image (N tokens, C channels, heads 4 x dim_head 32):
//   phase A, per 128-token tile   GEMM1  [k | v]^T[256 ch x 128 tok] = W_kv[256 x C] . X[128 tok x C]^T        (lane = channel)
//                                 epilogue: PreNorm fold affine, ONLINE column softmax of k (running max / sum per channel, the
//                                 context accumulator in TMEM is rescaled when the max moves), P = exp(k - max) and v as bf16 operands
//                                 GEMM2  ctx[(h,d) x (h',e)] += P[128 x 128 tok] . V[128 x 128 tok]^T            (diagonal blocks used)
//   phase B, per 128-token tile   GEMM3  q[128 tok x 128] = X . W_q^T ; epilogue: fold affine, softmax over the 32 head channels
//                                 GEMM4  o[128 tok x 128] = softmax(q) . (ctx * scale / colsum)                  (block-diagonal B operand)
//                                 GEMM5  y[128 tok x C] = o . W_o^T ; epilogue: + bias, statistics of GroupNorm(1), raw bf16 y -> out
//   phase C                       out = GroupNorm(1)(y) * gamma + beta + x, in place over the image (y and x come back from L2)
// The q / k / v tensors never exist in global memory: x is read (HBM once, L2 twice more), out is written.
//
// Operands that come from global memory (x tiles, weight slabs of 128 rows x 64 channels) are loaded by TMA tensor copies
// (cp.async.bulk.tensor.2d, 128-byte swizzle) into mbarrier rings; operands produced by the epilogues (P, V, softmax(q), o, ctx) are
// written to shared memory in the UMMA K-major no-swizzle canonical layout [k-chunk of 8][row][8] that the convolution engine uses.
// Weight slabs stay resident in their ring slot while the slab sequence repeats (C = 128: the whole phase), see Loader::w().
//
// Warp roles (320 threads): warps 0-7 epilogues (two per TMEM lane quarter), warp 8 TMA loader, warp 9 TMEM allocator + MMA issuer.
#include <cuda.h>      // CUtensorMap and its enums only: the encoder is fetched through cudaGetDriverEntryPoint (no libcuda link dependency)

#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "ops.h"
#include "tc_ptx.cuh"

namespace dmn {
namespace fa {

using namespace tc;

// ---------------------------------------------------------------------------------------------------------------------
// tensor maps
// ---------------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}
// row-major bf16 [rows][cols], box = 64 columns (128 bytes) x box_rows rows, 128-byte swizzle; out-of-range rows read as zero
static int make_map(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(-3, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(-3, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
  return 0;
}

__device__ __forceinline__ void tma_load(uint32_t dst, const CUtensorMap* map, int col, int row, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(col), "r"(row)
               : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
      "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void sts16(uint32_t addr, unsigned short v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory"); }
__device__ __forceinline__ uint4 ldcg128(const void* p) {
  uint4 v;
  asm volatile("ld.global.cg.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ unsigned short bf16_bits(float v) {
  const bf16 b = __float2bfloat16_rn(v);
  return *reinterpret_cast<const unsigned short*>(&b);
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float kLog2e = 1.4426950408889634f;

constexpr uint32_t kSlab = 128u * 128u;        // one TMA slab: 128 rows x 64 bf16 (128-byte rows, 8-row swizzle atoms of 1 KB)
constexpr uint32_t kOpBytes = 16u * 128u * 16u;   // one epilogue-written operand: 16 k-chunks x 128 rows x 16 bytes = 32 KB
constexpr uint32_t kOpLbo = 128u * 16u, kOpSbo = 128u;   // no-swizzle K-major: k-chunk stride, 8-row group stride
constexpr uint32_t kOpK16 = 2u * kOpLbo;       // one MMA k-step = 2 k-chunks
// per-head context operand of GEMM4: B[N = 32 (e)][K = 32 (d)] no-swizzle K-major = [4 k-chunks][32 rows][16 B] = 2 KB per head
constexpr uint32_t kCtxHead = 4u * 32u * 16u, kCtxLbo = 32u * 16u;

// =====================================================================================================================
// self-test of the TMA / 128-byte-swizzle plumbing: D[M][N] (fp32) = A[M][K] . B[N][K]^T, one CTA per 128 x 128 output tile
// =====================================================================================================================
struct SelfTestP {
  CUtensorMap ma, mb;
  float* d;
  int M, N, K;
};
__global__ void __launch_bounds__(128, 1) sw128_gemm_selftest_kernel(const __grid_constant__ SelfTestP p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base0 = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (base0 & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * kSlab);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 4);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  if (tid == 0) {
    mbar_init(smem_u32(&bars[0]), 1);
    mbar_init(smem_u32(&bars[1]), 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t sa = smem_u32(smem), sb = sa + kSlab;
  const uint32_t idesc = make_idesc(128, 128);
  const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 128;
  if (warp == 0) {
    const bool leader = elect_one();
    uint32_t ph = 0;
    for (int kc = 0; kc < p.K / 64; ++kc) {
      if (leader) {
        mbar_arrive_expect_tx(smem_u32(&bars[0]), 2 * kSlab);
        tma_load(sa, &p.ma, kc * 64, m0, smem_u32(&bars[0]));
        tma_load(sb, &p.mb, kc * 64, n0, smem_u32(&bars[0]));
      }
      __syncwarp();
      mbar_wait(smem_u32(&bars[0]), ph);
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int j = 0; j < 4; ++j) umma_bf16(tmem, make_desc_sw128(sa + j * 32), make_desc_sw128(sb + j * 32), idesc, (kc | j) ? 1u : 0u);
        umma_commit(smem_u32(&bars[1]));
      }
      __syncwarp();
      mbar_wait(smem_u32(&bars[1]), ph);      // the slabs are free again (single-buffered: this is a plumbing test, not a fast GEMM)
      ph ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t r[32];
  for (int c = 0; c < 128; c += 32) {
    tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c, r);
    const int m = m0 + warp * 32 + lane;
    if (m < p.M)
      for (int i = 0; i < 32; ++i)
        if (n0 + c + i < p.N) p.d[(long)m * p.N + n0 + c + i] = __uint_as_float(r[i]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 128);
  }
}

// =====================================================================================================================
// fused LinearAttention block, N % 128 == 0 (an image is a whole number of 128-token tiles)
// =====================================================================================================================
constexpr int kEpiThreads = 256, kLoaderWarp = 8, kMmaWarp = 9, kThreads = 320;
constexpr int kXS = 3, kWS = 4;                // ring depths in slabs

struct Params {
  CUtensorMap mx, mw, mo;        // x [B*N][C],  W_qkv (PreNorm gamma folded in) [384][C],  W_o [C][128]
  const bf16* x;
  bf16* out;
  const stat_t* pstats;          // [B][2] fixed-point {sum, sum of squares} of x over the image (PreNorm GroupNorm(1))
  const float* s1;               // [384] fold vectors (ops.h: ConvP::fold_s1 / fold_s2)
  const float* s2;
  const float* bo;               // [C] to_out.0.bias
  const float* go;               // [C] to_out.1.weight (GroupNorm(1) gamma)
  const float* beo;              // [C] to_out.1.bias
  int B, N, C;
  float inv_cnt;                 // 1 / (N * C)
  long long* trace;              // debug timeline of CTA 0 (DMN_FA_TRACE=1), else null
};
__device__ long long g_fa_trace[64];
#define FA_TRACE(k) do { if (p.trace && blockIdx.x == 0 && tid == 0) p.trace[(k)] = clock64(); } while (0)

// barrier indices
enum { B_FULLX = 0, B_EMPTYX = B_FULLX + kXS, B_FULLW = B_EMPTYX + kXS, B_EMPTYW = B_FULLW + kWS, B_KV = B_EMPTYW + kWS, B_PV, B_CTX, B_Q, B_QS,
       B_OUT, B_OUTS, B_Y, B_COUNT };

__global__ void __launch_bounds__(kThreads, 1) linattn_fused_kernel(const __grid_constant__ Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base0 = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (base0 & 1023u)) & 1023u);
  uint8_t* s_x = smem;                                   // kXS slabs
  uint8_t* s_w = s_x + kXS * kSlab;                      // kWS slabs
  uint8_t* s_opa = s_w + kWS * kSlab;                    // P (phase A) | softmax(q) (phase B)        A operand
  uint8_t* s_opb = s_opa + kOpBytes;                     // V (phase A, B operand) | o (phase B, A operand)
  uint8_t* s_ctx = s_opb + kOpBytes;                     // per-head context operands of GEMM4 (4 x 2 KB)
  float* s_tq = reinterpret_cast<float*>(s_ctx + 4 * kCtxHead);   // [128] per-image additive term of the q fold (log2 domain)
  float* s_bo = s_tq + 128;                              // [C]
  float* s_go = s_bo + 256;                              // [C]
  float* s_beo = s_go + 256;                             // [C]
  float* s_red = s_beo + 256;                            // [8][2] statistics partials
  float* s_kx = s_red + 16;                              // [2][128] k softmax exchange between the two warps of a lane quarter: tile maxima
  float* s_ks = s_kx + 256;                              // [2][128] ... column sums
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_ks + 256);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + B_COUNT);

  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int C = p.C, N = p.N, KC = C >> 6, RH = C >> 7;
  const int T = N >= 128 ? (N >> 7) : 1;         // 128-token tiles per image
  const int NV = N >= 128 ? 128 : N;             // valid tokens of a tile (N < 128: one zero-padded tile per image)
  const uint32_t xbytes = (uint32_t)NV * 128u;   // bytes one x slab copy delivers
  auto bar = [&](int i) { return smem_u32(&bars[i]); };

  if (warp == kLoaderWarp) {
    if (lane < B_COUNT) {
      uint32_t cnt = 1;
      if (lane == B_PV || lane == B_QS || lane == B_OUTS) cnt = kEpiThreads;
      mbar_init(bar(lane), cnt);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(smem_u32(tslot), 512);
  if (warp < 8) {
    if (NV < 128)      // the TMA box only writes the first NV rows of a slab: the padded rows are zero for the whole launch
      for (uint32_t i = tid; i < kXS * kSlab / 16; i += kEpiThreads) sts128(smem_u32(s_x) + i * 16, make_uint4(0, 0, 0, 0));
    for (int i = tid; i < C; i += kEpiThreads) {
      s_bo[i] = p.bo[i];
      s_go[i] = p.go[i];
      s_beo[i] = p.beo[i];
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t tDk = tmem, tDv = tmem + 128, tDctx = tmem + 256;      // phase A
  const uint32_t tDq = tmem, tDo = tmem + 128, tDy = tmem + 256;        // phase B (aliases)

  if (warp == kLoaderWarp) {
    // =============================================== TMA loader ===============================================
    const bool leader = elect_one();
    int xs = 0, ws = 0;
    uint32_t xph = 1, wph = 1;                 // parity of the "slot is free" waits
    int wtag[kWS];
#pragma unroll
    for (int i = 0; i < kWS; ++i) wtag[i] = -1;
    auto load_x = [&](int row0, int kc) {
      mbar_wait_relaxed(bar(B_EMPTYX + xs), xph);
      if (leader) {
        mbar_arrive_expect_tx(bar(B_FULLX + xs), xbytes);
        tma_load(smem_u32(s_x) + xs * kSlab, &p.mx, kc * 64, row0, bar(B_FULLX + xs));
      }
      __syncwarp();
      if (++xs == kXS) { xs = 0; xph ^= 1; }
    };
    // weight slab `id`; a slot that already holds the wanted slab (the slab sequence of a phase repeats with a period that
    // divides the ring depth when C = 128) is handed over without a copy
    auto load_w = [&](const CUtensorMap* map, int id, int col, int row) {
      mbar_wait_relaxed(bar(B_EMPTYW + ws), wph);
      bool hit = false;
#pragma unroll
      for (int i = 0; i < kWS; ++i)
        if (i == ws) { hit = wtag[i] == id; wtag[i] = id; }
      if (leader) {
        if (hit) {
          mbar_arrive(bar(B_FULLW + ws));
        } else {
          mbar_arrive_expect_tx(bar(B_FULLW + ws), kSlab);
          tma_load(smem_u32(s_w) + ws * kSlab, map, col, row, bar(B_FULLW + ws));
        }
      }
      __syncwarp();
      if (++ws == kWS) { ws = 0; wph ^= 1; }
    };
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      const int row_img = b * N;
      for (int t = 0; t < T; ++t)
        for (int kc = 0; kc < KC; ++kc) {
          load_x(row_img + t * 128, kc);
          load_w(&p.mw, 8 + kc, kc * 64, 128);       // W_k rows [128, 256)
          load_w(&p.mw, 16 + kc, kc * 64, 256);      // W_v rows [256, 384)
        }
      // phase B in the order the MMA issuer consumes: q(0); then per tile q(t + 1), W_o(t)
      auto q_tile = [&](int t) {
        for (int kc = 0; kc < KC; ++kc) {
          load_x(row_img + t * 128, kc);
          load_w(&p.mw, kc, kc * 64, 0);             // W_q rows [0, 128)
        }
      };
      q_tile(0);
      for (int t = 0; t < T; ++t) {
        if (t + 1 < T) q_tile(t + 1);
        for (int kc2 = 0; kc2 < 2; ++kc2)
          for (int rh = 0; rh < RH; ++rh) load_w(&p.mo, 32 + kc2 * 2 + rh, kc2 * 64, rh * 128);
      }
    }
  } else if (warp == kMmaWarp) {
    // =============================================== MMA issuer ===============================================
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc(128, 128), idesc32 = make_idesc(128, 32);
    int xs = 0, ws = 0;
    uint32_t xph = 0, wph = 0;
    uint32_t ph_pv = 0, ph_qs = 0, ph_outs = 0;
    const uint32_t opa = smem_u32(s_opa), opb = smem_u32(s_opb), ctxb = smem_u32(s_ctx);
    auto wait_x = [&]() -> uint32_t {
      mbar_wait(bar(B_FULLX + xs), xph);
      return smem_u32(s_x) + xs * kSlab;
    };
    auto wait_w = [&]() -> uint32_t {          // the current weight slot (not advanced)
      mbar_wait(bar(B_FULLW + ws), wph);
      return smem_u32(s_w) + ws * kSlab;
    };
    auto adv_w = [&]() -> int {                // returns the slot that was current
      const int s0 = ws;
      if (++ws == kWS) { ws = 0; wph ^= 1; }
      return s0;
    };
    auto free_x = [&]() {                      // the slot is released once the MMAs issued so far have retired
      if (leader) umma_commit(bar(B_EMPTYX + xs));
      __syncwarp();
      if (++xs == kXS) { xs = 0; xph ^= 1; }
    };
    auto free_w_slot = [&](int slot) {
      if (leader) umma_commit(bar(B_EMPTYW + slot));
      __syncwarp();
    };
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      // ---------------- phase A ----------------
      for (int t = 0; t < T; ++t) {
        for (int kc = 0; kc < KC; ++kc) {
          const uint32_t ax = wait_x();
          const uint32_t wk = wait_w();
          const int slot_k = adv_w();
          const uint32_t wv = wait_w();
          const int slot_v = adv_w();
          tc_fence_after();
          if (leader) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t acc = (kc | j) ? 1u : 0u;
              const uint64_t xd = make_desc_sw128(ax + j * 32);
              umma_bf16(tDk, make_desc_sw128(wk + j * 32), xd, idesc, acc);
              umma_bf16(tDv, make_desc_sw128(wv + j * 32), xd, idesc, acc);
            }
          }
          __syncwarp();
          free_w_slot(slot_k);
          free_w_slot(slot_v);
          free_x();
        }
        if (leader) umma_commit(bar(B_KV));
        __syncwarp();
        mbar_wait(bar(B_PV), ph_pv);
        ph_pv ^= 1;
        tc_fence_after();
        if (leader) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            umma_bf16(tDctx, make_desc(opa + j * kOpK16, kOpLbo, kOpSbo), make_desc(opb + j * kOpK16, kOpLbo, kOpSbo), idesc, (t | j) ? 1u : 0u);
          if (t == T - 1) umma_commit(bar(B_CTX));
        }
        __syncwarp();
      }
      // ---------------- phase B (software pipelined: GEMM3 of tile t + 1 is issued before GEMM5 of tile t) ----------------
      auto gemm3 = [&]() {
        for (int kc = 0; kc < KC; ++kc) {
          const uint32_t ax = wait_x();
          const uint32_t wq = wait_w();
          tc_fence_after();
          if (leader) {
#pragma unroll
            for (int j = 0; j < 4; ++j) umma_bf16(tDq, make_desc_sw128(ax + j * 32), make_desc_sw128(wq + j * 32), idesc, (kc | j) ? 1u : 0u);
          }
          __syncwarp();
          free_w_slot(adv_w());
          free_x();
        }
        if (leader) umma_commit(bar(B_Q));
        __syncwarp();
      };
      gemm3();
      for (int t = 0; t < T; ++t) {
        mbar_wait(bar(B_QS), ph_qs);
        ph_qs ^= 1;
        tc_fence_after();
        if (leader) {
          // o[:, head h] = softmax(q)[:, head h] . ctx_h: four M128 x N32 x K32 products
#pragma unroll
          for (int h = 0; h < 4; ++h)
#pragma unroll
            for (int j = 0; j < 2; ++j)
              umma_bf16(tDo + h * 32, make_desc(opa + (h * 2 + j) * kOpK16, kOpLbo, kOpSbo),
                        make_desc(ctxb + h * kCtxHead + j * 2 * kCtxLbo, kCtxLbo, kOpSbo), idesc32, j ? 1u : 0u);
          umma_commit(bar(B_OUT));
        }
        __syncwarp();
        if (t + 1 < T) gemm3();                 // early: the epilogue of this tile's o / y overlaps the next tile's q product
        mbar_wait(bar(B_OUTS), ph_outs);
        ph_outs ^= 1;
        tc_fence_after();
        for (int kc2 = 0; kc2 < 2; ++kc2)
          for (int rh = 0; rh < RH; ++rh) {
            const uint32_t wo = wait_w();
            tc_fence_after();
            if (leader) {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                umma_bf16(tDy + rh * 128, make_desc(opb + (kc2 * 4 + j) * kOpK16, kOpLbo, kOpSbo), make_desc_sw128(wo + j * 32), idesc,
                          (kc2 | j) ? 1u : 0u);
            }
            __syncwarp();
            free_w_slot(adv_w());
          }
        if (leader) umma_commit(bar(B_Y));
        __syncwarp();
      }
    }
  } else {
    // =============================================== epilogues ===============================================
    const int q4 = warp & 3, half = warp >> 2;                 // TMEM lane quarter of this warp; column half
    const uint32_t lane_base = (uint32_t)(q4 * 32) << 16;
    const int ch = q4 * 32 + lane;                             // phase A: the channel of this thread (lane = channel)
    const uint32_t opa = smem_u32(s_opa), opb = smem_u32(s_opb), ctxb = smem_u32(s_ctx);
    // phase A: both warps of a lane quarter work on k AND v of the quarter's 32 channels, each on one half of the tile's tokens
    const float s1k = p.s1[128 + ch], s2k = p.s2[128 + ch], s1v = p.s1[256 + ch], s2v = p.s2[256 + ch];
    uint32_t ph_kv = 0, ph_ctx = 0, ph_q = 0, ph_out = 0, ph_y = 0;
    const float qscale = rsqrtf(32.f);
    const int tcol0 = half * 64;                               // phase A: this thread's token columns [tcol0, tcol0 + 64)
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      float mean_x, rstd_x;
      gn_mean_rstd(p.pstats + (long)b * 2, p.inv_cnt, kGnEps, mean_x, rstd_x);
      const float fa = rstd_x, fc = -mean_x * rstd_x;          // x_hat = fa * x + fc (gamma / beta live in the weights and s1 / s2)
      const float fa2 = fa * kLog2e;                           // softmax arguments are kept in the log2 domain (one ex2 per element)
      if (tid < 128) s_tq[tid] = (fc * p.s1[tid] + p.s2[tid]) * kLog2e;
      const float ck2 = (fc * s1k + s2k) * kLog2e, cv = fc * s1v + s2v;
      float run_max = -INFINITY, run_sum = 0.f;                // run_sum: this thread's half of the columns
      float sy = 0.f, sq = 0.f;
      const int tb = (b == (int)blockIdx.x) ? 0 : 8;
      FA_TRACE(tb + 0);
      // ---------------- phase A ----------------
      for (int t = 0; t < T; ++t) {
        mbar_wait_relaxed(bar(B_KV), ph_kv);
        ph_kv ^= 1;
        tc_fence_after();
        uint32_t r[32];
        // ---- k: online column softmax over the tokens; pass 1 = maximum of this thread's 64 columns ----
        float tmax = -INFINITY;
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
          tmem_ld32(tDk + lane_base + tcol0 + c0, r);
          const int nvalid = NV - (tcol0 + c0);                 // token columns >= NV are padding
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < nvalid) tmax = fmaxf(tmax, fmaf(fa2, __uint_as_float(r[i]), ck2));
        }
        s_kx[half * 128 + ch] = tmax;
        bar_sync_named(1, kEpiThreads);
        const float new_max = fmaxf(run_max, fmaxf(tmax, s_kx[(half ^ 1) * 128 + ch]));
        const float f = ex2(run_max - new_max);                // 0 on the first tile (run_max = -inf)
        float psum = 0.f;
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
          tmem_ld32(tDk + lane_base + tcol0 + c0, r);
          const int nvalid = NV - (tcol0 + c0);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int i0 = g * 8 + 2 * e;
              const bf16 p0 = __float2bfloat16_rn(i0 < nvalid ? ex2(fmaf(fa2, __uint_as_float(r[i0]), ck2) - new_max) : 0.f);
              const bf16 p1 = __float2bfloat16_rn(i0 + 1 < nvalid ? ex2(fmaf(fa2, __uint_as_float(r[i0 + 1]), ck2) - new_max) : 0.f);
              psum += __bfloat162float(p0) + __bfloat162float(p1);     // sums of the ROUNDED values: numerator and denominator agree
              w[e] = (uint32_t)(*reinterpret_cast<const unsigned short*>(&p0)) | ((uint32_t)(*reinterpret_cast<const unsigned short*>(&p1)) << 16);
            }
            sts128(opa + (uint32_t)(((((tcol0 + c0) >> 3) + g) * 128 + ch) * 16), make_uint4(w[0], w[1], w[2], w[3]));
          }
        }
        run_sum = run_sum * f + psum;
        run_max = new_max;
        // rescale this channel's row of the context accumulator (its head's diagonal block) when the max moved
        if (half == 0 && t > 0 && __any_sync(0xffffffffu, f != 1.f)) {
          tmem_ld32(tDctx + lane_base + (uint32_t)(q4 * 32), r);
#pragma unroll
          for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * f);
          tmem_st32(tDctx + lane_base + (uint32_t)(q4 * 32), r);
          tmem_st_wait();
        }
        // ---- v ----
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
          tmem_ld32(tDv + lane_base + tcol0 + c0, r);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e)
              w[e] = pack_bf16x2(fmaf(fa, __uint_as_float(r[g * 8 + 2 * e]), cv), fmaf(fa, __uint_as_float(r[g * 8 + 2 * e + 1]), cv));
            sts128(opb + (uint32_t)(((((tcol0 + c0) >> 3) + g) * 128 + ch) * 16), make_uint4(w[0], w[1], w[2], w[3]));
          }
        }
        fence_proxy_async();
        tc_fence_before();
        mbar_arrive(bar(B_PV));
      }
      FA_TRACE(tb + 1);
      // ---- context: ctx[d][e] * scale / colsum[d] -> per-head B operands of GEMM4, element (row e, k d) ----
      s_ks[half * 128 + ch] = run_sum;
      mbar_wait_relaxed(bar(B_CTX), ph_ctx);
      ph_ctx ^= 1;
      tc_fence_after();
      bar_sync_named(1, kEpiThreads);            // both halves of the column sums, and s_tq, are visible
      if (half == 0) {
        uint32_t r[32];
        tmem_ld32(tDctx + lane_base + (uint32_t)(q4 * 32), r);
        const float sc = qscale / (run_sum + s_ks[128 + ch]);
        const uint32_t dst = ctxb + (uint32_t)(q4 * kCtxHead + (lane >> 3) * kCtxLbo + (lane & 7) * 2);
#pragma unroll
        for (int e = 0; e < 32; ++e) sts16(dst + e * 16, bf16_bits(__uint_as_float(r[e]) * sc));
      }
      // ---------------- phase B ----------------
      // q: fold affine, softmax over the 32 channels of each head (the scale lives in the context operand) -> A operand of GEMM4
      auto epi_q = [&]() {
        uint32_t r[32];
        mbar_wait_relaxed(bar(B_Q), ph_q);
        ph_q ^= 1;
        tc_fence_after();
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int col0 = (half * 2 + hh) * 32;
          tmem_ld32(tDq + lane_base + col0, r);
          float v[32];
          float mx = -INFINITY;
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 tq = *reinterpret_cast<const float4*>(s_tq + col0 + i);
            v[i] = fmaf(fa2, __uint_as_float(r[i]), tq.x);
            v[i + 1] = fmaf(fa2, __uint_as_float(r[i + 1]), tq.y);
            v[i + 2] = fmaf(fa2, __uint_as_float(r[i + 2]), tq.z);
            v[i + 3] = fmaf(fa2, __uint_as_float(r[i + 3]), tq.w);
            mx = fmaxf(fmaxf(mx, fmaxf(v[i], v[i + 1])), fmaxf(v[i + 2], v[i + 3]));
          }
          float sum = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) { v[i] = ex2(v[i] - mx); sum += v[i]; }
          const float inv = 1.f / sum;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint4 o;
            o.x = pack_bf16x2(v[g * 8] * inv, v[g * 8 + 1] * inv);
            o.y = pack_bf16x2(v[g * 8 + 2] * inv, v[g * 8 + 3] * inv);
            o.z = pack_bf16x2(v[g * 8 + 4] * inv, v[g * 8 + 5] * inv);
            o.w = pack_bf16x2(v[g * 8 + 6] * inv, v[g * 8 + 7] * inv);
            sts128(opa + (uint32_t)((((col0 >> 3) + g) * 128 + q4 * 32 + lane) * 16), o);
          }
        }
        fence_proxy_async();
        tc_fence_before();
        mbar_arrive(bar(B_QS));
      };
      FA_TRACE(tb + 2);
      epi_q();                                   // (the B_QS arrival also publishes the context operands written above)
      for (int t = 0; t < T; ++t) {
        const int tok = t * 128 + q4 * 32 + lane;              // phase B: lane = token
        uint32_t r[32];
        // ---- o = softmax(q) . ctx: TMEM -> bf16 A operand of GEMM5 ----
        mbar_wait_relaxed(bar(B_OUT), ph_out);
        ph_out ^= 1;
        tc_fence_after();
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int col0 = (half * 2 + hh) * 32;
          tmem_ld32(tDo + lane_base + col0, r);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint4 o;
            o.x = pack_bf16x2(__uint_as_float(r[g * 8]), __uint_as_float(r[g * 8 + 1]));
            o.y = pack_bf16x2(__uint_as_float(r[g * 8 + 2]), __uint_as_float(r[g * 8 + 3]));
            o.z = pack_bf16x2(__uint_as_float(r[g * 8 + 4]), __uint_as_float(r[g * 8 + 5]));
            o.w = pack_bf16x2(__uint_as_float(r[g * 8 + 6]), __uint_as_float(r[g * 8 + 7]));
            sts128(opb + (uint32_t)((((col0 >> 3) + g) * 128 + q4 * 32 + lane) * 16), o);
          }
        }
        fence_proxy_async();
        tc_fence_before();
        mbar_arrive(bar(B_OUTS));
        if (t + 1 < T) epi_q();                  // the next tile's q while the tensor core computes this tile's y
        // ---- y = o . W_o^T + bias: statistics of GroupNorm(1), raw bf16 y parked in the output buffer ----
        mbar_wait_relaxed(bar(B_Y), ph_y);
        ph_y ^= 1;
        tc_fence_after();
        const int ncol = C >> 1;                               // columns of this warp: [half * ncol, (half + 1) * ncol)
        const bool row_ok = q4 * 32 + lane < NV;               // padded token rows are neither counted nor stored
        bf16* yrow = p.out + ((long)b * N + tok) * C + half * ncol;
#pragma unroll 1
        for (int c0 = 0; c0 < ncol; c0 += 32) {
          tmem_ld32(tDy + lane_base + (uint32_t)(half * ncol + c0), r);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float y[8];
#pragma unroll
            for (int e = 0; e < 8; e += 4) {
              const float4 bb = *reinterpret_cast<const float4*>(s_bo + half * ncol + c0 + g * 8 + e);
              y[e] = __uint_as_float(r[g * 8 + e]) + bb.x;
              y[e + 1] = __uint_as_float(r[g * 8 + e + 1]) + bb.y;
              y[e + 2] = __uint_as_float(r[g * 8 + e + 2]) + bb.z;
              y[e + 3] = __uint_as_float(r[g * 8 + e + 3]) + bb.w;
            }
            if (row_ok) {
#pragma unroll
              for (int e = 0; e < 8; ++e) { sy += y[e]; sq = fmaf(y[e], y[e], sq); }
              *reinterpret_cast<uint4*>(yrow + c0 + g * 8) = pack8(y);     // (finishing single-tile images straight from TMEM measured slower:
                                                                           //  per-row residual loads are uncoalesced, the coalesced pass below wins)
            }
          }
        }
        tc_fence_before();
      }
      FA_TRACE(tb + 3);
      // ---------------- phase C: out = GroupNorm(1)(y) * gamma + beta + x ----------------
      sy = warp_sum(sy);
      sq = warp_sum(sq);
      if (lane == 0) { s_red[warp * 2] = sy; s_red[warp * 2 + 1] = sq; }
      bar_sync_named(1, kEpiThreads);            // also orders this CTA's global y stores before the reads below
      float ts = 0.f, tq2 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { ts += s_red[2 * i]; tq2 += s_red[2 * i + 1]; }
      const float mean_y = ts * p.inv_cnt;
      float var_y = tq2 * p.inv_cnt - mean_y * mean_y;
      var_y = var_y < 0.f ? 0.f : var_y;
      const float rstd_y = rsqrtf(var_y + kGnEps);
      {
        const int per_row = C >> 3;                            // 16-byte items per token row (16 or 32: divides 256)
        const int c8 = (tid % per_row) * 8;
        float gsc[8], gsh[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          gsc[e] = rstd_y * s_go[c8 + e];
          gsh[e] = s_beo[c8 + e] - mean_y * gsc[e];
        }
        const long base = (long)b * N * C;
        const int items = N * per_row;
        constexpr int U = 8;                                   // independent 16-byte items in flight per thread
        for (int i0 = tid; i0 < items; i0 += U * kEpiThreads) {
          uint4 yv[U], xv[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int i = i0 + u * kEpiThreads;
            if (i < items) {
              yv[u] = ldcg128(p.out + base + (long)i * 8);
              xv[u] = ldcg128(p.x + base + (long)i * 8);
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int i = i0 + u * kEpiThreads;
            if (i < items) {
              float y[8], xx[8];
              unpack8(yv[u], y);
              unpack8(xv[u], xx);
#pragma unroll
              for (int e = 0; e < 8; ++e) y[e] = fmaf(y[e], gsc[e], gsh[e]) + xx[e];
              *reinterpret_cast<uint4*>(p.out + base + (long)i * 8) = pack8(y);
            }
          }
        }
      }
      FA_TRACE(tb + 4);
      bar_sync_named(1, kEpiThreads);            // s_red / s_tq / s_ks are rewritten by the next image
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

constexpr size_t kSmemFused = 1024 + (size_t)(kXS + kWS) * kSlab + 2 * (size_t)kOpBytes + 4 * kCtxHead + (128 + 3 * 256 + 16 + 512) * 4 + (B_COUNT + 2) * 8 + 64;

// =====================================================================================================================
// fused softmax Attention block (the U-Net bottleneck): Residual(PreNorm(dim, Attention(dim)))   (reference parts/mha.py:8-30)
//   out = to_out(softmax_j(scale * q_i . k_j) v_j) + x,  heads 4 x dim_head 32, at most 64 tokens per image (one zero-padded tile)
// Per image:  GEMM  q[tok x 128] = X W_q^T,  k^T | v^T [128 ch x tok] = W_k | W_v . X^T          (TMA operands, as above)
//             epilogue: fold affine; q * scale (log2 domain), k as the B operand [tok_j][(h,d)], v as the B operand [(h,e)][tok_j]
//             GEMM  S_h[tok_i x tok_j] = q_h k_h^T  (4 heads, N = padded token count)   ->   row softmax  ->  P_h as A operand
//             GEMM  o_h[tok_i x 32] = P_h v_h       ->  A operand of   GEMM  y = o W_o^T   ->   + bias + x, stored
// =====================================================================================================================
enum { S_FULLX = 0, S_EMPTYX = S_FULLX + kXS, S_FULLW = S_EMPTYX + kXS, S_EMPTYW = S_FULLW + kWS, S_QKV = S_EMPTYW + kWS, S_OPS, S_S, S_P, S_OUT,
       S_OUTS, S_Y, S_FREE, S_COUNT };

__global__ void __launch_bounds__(kThreads, 1) attn_softmax_fused_kernel(const __grid_constant__ Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base0 = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (base0 & 1023u)) & 1023u);
  uint8_t* s_x = smem;
  uint8_t* s_w = s_x + kXS * kSlab;
  uint8_t* s_opa = s_w + kWS * kSlab;                    // q operand (A of the S products); with s_kop it later holds P (A of the o products)
  uint8_t* s_kop = s_opa + kOpBytes;                     // k operand (B of the S products)
  uint8_t* s_opb = s_kop + kOpBytes;                     // v operand (B of the o products), then o (A of the to_out product)
  float* s_tq = reinterpret_cast<float*>(s_opb + kOpBytes);   // [128] additive fold term of q, already times scale * log2(e)
  float* s_bo = s_tq + 128;                              // [C]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_bo + 256);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + S_COUNT);

  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int C = p.C, N = p.N, KC = C >> 6, RH = C >> 7;
  const int NV = N;                                      // valid tokens (<= 64)
  const int NVp = (NV + 15) & ~15;                       // token count padded to the MMA granularity
  const uint32_t xbytes = (uint32_t)NV * 128u;
  auto bar = [&](int i) { return smem_u32(&bars[i]); };

  if (warp == kLoaderWarp) {
    if (lane < S_COUNT) {
      uint32_t cnt = 1;
      if (lane == S_OPS || lane == S_P || lane == S_OUTS || lane == S_FREE) cnt = kEpiThreads;
      mbar_init(bar(lane), cnt);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(smem_u32(tslot), 512);
  if (warp < 8) {
    for (uint32_t i = tid; i < kXS * kSlab / 16; i += kEpiThreads) sts128(smem_u32(s_x) + i * 16, make_uint4(0, 0, 0, 0));
    // the k operand's rows beyond the image (tok_j >= NV, up to NVp) must be finite: zero the buffer once
    for (uint32_t i = tid; i < kOpBytes / 16; i += kEpiThreads) sts128(smem_u32(s_kop) + i * 16, make_uint4(0, 0, 0, 0));
    for (int i = tid; i < C; i += kEpiThreads) s_bo[i] = p.bo[i];
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t tDk = tmem, tDv = tmem + 128, tDq = tmem + 256, tDo = tmem + 384;
  const uint32_t tS = tmem, tDy = tmem;                  // aliases of the k^T | v^T columns (dead once their operands are in shared memory)
  const uint32_t pHead = (uint32_t)(NVp >> 3) * kOpLbo;  // bytes of one head's P operand: NVp / 8 k-chunks

  if (warp == kLoaderWarp) {
    const bool leader = elect_one();
    int xs = 0, ws = 0;
    uint32_t xph = 1, wph = 1;
    auto load_x = [&](int row0, int kc) {
      mbar_wait_relaxed(bar(S_EMPTYX + xs), xph);
      if (leader) {
        mbar_arrive_expect_tx(bar(S_FULLX + xs), xbytes);
        tma_load(smem_u32(s_x) + xs * kSlab, &p.mx, kc * 64, row0, bar(S_FULLX + xs));
      }
      __syncwarp();
      if (++xs == kXS) { xs = 0; xph ^= 1; }
    };
    auto load_w = [&](const CUtensorMap* map, int col, int row) {
      mbar_wait_relaxed(bar(S_EMPTYW + ws), wph);
      if (leader) {
        mbar_arrive_expect_tx(bar(S_FULLW + ws), kSlab);
        tma_load(smem_u32(s_w) + ws * kSlab, map, col, row, bar(S_FULLW + ws));
      }
      __syncwarp();
      if (++ws == kWS) { ws = 0; wph ^= 1; }
    };
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      for (int kc = 0; kc < KC; ++kc) {
        load_x(b * N, kc);
        load_w(&p.mw, kc * 64, 0);
        load_w(&p.mw, kc * 64, 128);
        load_w(&p.mw, kc * 64, 256);
      }
      for (int kc2 = 0; kc2 < 2; ++kc2)
        for (int rh = 0; rh < RH; ++rh) load_w(&p.mo, kc2 * 64, rh * 128);
    }
  } else if (warp == kMmaWarp) {
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc(128, 128), idesc32 = make_idesc(128, 32), idescS = make_idesc(128, NVp);
    int xs = 0, ws = 0;
    uint32_t xph = 0, wph = 0, ph_ops = 0, ph_p = 0, ph_outs = 0, ph_free = 1;
    const uint32_t opa = smem_u32(s_opa), kop = smem_u32(s_kop), opb = smem_u32(s_opb);
    auto wait_w = [&]() -> uint32_t {
      mbar_wait(bar(S_FULLW + ws), wph);
      tc_fence_after();
      return smem_u32(s_w) + ws * kSlab;
    };
    auto free_w = [&]() {
      if (leader) umma_commit(bar(S_EMPTYW + ws));
      __syncwarp();
      if (++ws == kWS) { ws = 0; wph ^= 1; }
    };
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      mbar_wait(bar(S_FREE), ph_free);                   // the previous image's y has been read out of the aliased columns
      ph_free ^= 1;
      tc_fence_after();
      for (int kc = 0; kc < KC; ++kc) {
        mbar_wait(bar(S_FULLX + xs), xph);
        tc_fence_after();
        const uint32_t ax = smem_u32(s_x) + xs * kSlab;
        const uint32_t wq = wait_w();
        if (leader) {
#pragma unroll
          for (int j = 0; j < 4; ++j) umma_bf16(tDq, make_desc_sw128(ax + j * 32), make_desc_sw128(wq + j * 32), idesc, (kc | j) ? 1u : 0u);
        }
        __syncwarp();
        free_w();
        const uint32_t wk = wait_w();
        if (leader) {
#pragma unroll
          for (int j = 0; j < 4; ++j) umma_bf16(tDk, make_desc_sw128(wk + j * 32), make_desc_sw128(ax + j * 32), idesc, (kc | j) ? 1u : 0u);
        }
        __syncwarp();
        free_w();
        const uint32_t wv = wait_w();
        if (leader) {
#pragma unroll
          for (int j = 0; j < 4; ++j) umma_bf16(tDv, make_desc_sw128(wv + j * 32), make_desc_sw128(ax + j * 32), idesc, (kc | j) ? 1u : 0u);
        }
        __syncwarp();
        free_w();
        if (leader) umma_commit(bar(S_EMPTYX + xs));
        __syncwarp();
        if (++xs == kXS) { xs = 0; xph ^= 1; }
      }
      if (leader) umma_commit(bar(S_QKV));
      __syncwarp();
      // S_h = q_h k_h^T : M128 x N(NVp) x K32 per head
      mbar_wait(bar(S_OPS), ph_ops);
      ph_ops ^= 1;
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int h = 0; h < 4; ++h)
#pragma unroll
          for (int j = 0; j < 2; ++j)
            umma_bf16(tS + h * NVp, make_desc(opa + (h * 2 + j) * kOpK16, kOpLbo, kOpSbo), make_desc(kop + (h * 2 + j) * kOpK16, kOpLbo, kOpSbo),
                      idescS, j ? 1u : 0u);
        umma_commit(bar(S_S));
      }
      __syncwarp();
      // o_h = P_h v_h : M128 x N32 x K(NVp) per head
      mbar_wait(bar(S_P), ph_p);
      ph_p ^= 1;
      tc_fence_after();
      if (leader) {
        for (int h = 0; h < 4; ++h)
          for (int j = 0; j < (NVp >> 4); ++j)
            umma_bf16(tDo + h * 32, make_desc(opa + h * pHead + j * kOpK16, kOpLbo, kOpSbo),
                      make_desc(opb + (uint32_t)(h * 32) * 16u + j * kOpK16, kOpLbo, kOpSbo), idesc32, j ? 1u : 0u);
        umma_commit(bar(S_OUT));
      }
      __syncwarp();
      mbar_wait(bar(S_OUTS), ph_outs);
      ph_outs ^= 1;
      tc_fence_after();
      for (int kc2 = 0; kc2 < 2; ++kc2)
        for (int rh = 0; rh < RH; ++rh) {
          const uint32_t wo = wait_w();
          if (leader) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              umma_bf16(tDy + rh * 128, make_desc(opb + (kc2 * 4 + j) * kOpK16, kOpLbo, kOpSbo), make_desc_sw128(wo + j * 32), idesc, (kc2 | j) ? 1u : 0u);
          }
          __syncwarp();
          free_w();
        }
      if (leader) umma_commit(bar(S_Y));
      __syncwarp();
    }
  } else {
    const int q4 = warp & 3, half = warp >> 2;
    const uint32_t lane_base = (uint32_t)(q4 * 32) << 16;
    const int ch = q4 * 32 + lane;
    const uint32_t opa = smem_u32(s_opa), kop = smem_u32(s_kop), opb = smem_u32(s_opb);
    const float s1k = p.s1[128 + ch], s2k = p.s2[128 + ch], s1v = p.s1[256 + ch], s2v = p.s2[256 + ch];
    const float qs = rsqrtf(32.f) * kLog2e;                    // q * scale, softmax in the log2 domain
    uint32_t ph_qkv = 0, ph_s = 0, ph_out = 0, ph_y = 0;
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      float mean_x, rstd_x;
      gn_mean_rstd(p.pstats + (long)b * 2, p.inv_cnt, kGnEps, mean_x, rstd_x);
      const float fa = rstd_x, fc = -mean_x * rstd_x;
      if (tid < 128) s_tq[tid] = (fc * p.s1[tid] + p.s2[tid]) * qs;
      const float ck = fc * s1k + s2k, cv = fc * s1v + s2v;
      bar_sync_named(1, kEpiThreads);
      mbar_wait_relaxed(bar(S_QKV), ph_qkv);
      ph_qkv ^= 1;
      tc_fence_after();
      uint32_t r[32];
      // ---- q operand: [tok_i][(h,d)] (lane = token), two heads per warp ----
      const float faq = fa * qs;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int col0 = (half * 2 + hh) * 32;
        tmem_ld32(tDq + lane_base + col0, r);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float v[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = fmaf(faq, __uint_as_float(r[g * 8 + e]), s_tq[col0 + g * 8 + e]);
          sts128(opa + (uint32_t)((((col0 >> 3) + g) * 128 + q4 * 32 + lane) * 16), pack8(v));
        }
      }
      // ---- k operand [tok_j][(h,d)] (warps 0-3) / v operand [(h,e)][tok_j] (warps 4-7): lane = channel ----
      for (int c0 = 0; c0 < NVp; c0 += 32) {
        tmem_ld32((half ? tDv : tDk) + lane_base + c0, r);
        if (half == 0) {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (c0 + i < NV) sts16(kop + (uint32_t)(((ch >> 3) * 128 + c0 + i) * 16 + (ch & 7) * 2), bf16_bits(fmaf(fa, __uint_as_float(r[i]), ck)));
        } else {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            if (c0 + g * 8 < NVp) {
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) v[e] = fmaf(fa, __uint_as_float(r[g * 8 + e]), cv);
              sts128(opb + (uint32_t)((((c0 >> 3) + g) * 128 + ch) * 16), pack8(v));
            }
          }
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(bar(S_OPS));
      // ---- row softmax of S_h over the image's tokens -> P_h [tok_i][tok_j] (A operand; overwrites the q / k operands) ----
      mbar_wait_relaxed(bar(S_S), ph_s);
      ph_s ^= 1;
      tc_fence_after();
#pragma unroll 1
      for (int hh = 0; hh < 2; ++hh) {
        const int h = half * 2 + hh;
        float mx = -INFINITY, sum = 0.f;
        float e[64];
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
          if (c0 < NVp) {
            tmem_ld32(tS + lane_base + (uint32_t)(h * NVp + c0), r);      // (columns beyond NVp belong to the next head: masked below)
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              e[c0 + i] = c0 + i < NV ? __uint_as_float(r[i]) : -INFINITY;
              mx = fmaxf(mx, e[c0 + i]);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) e[c0 + i] = -INFINITY;
          }
        }
#pragma unroll
        for (int i = 0; i < 64; ++i) { e[i] = ex2(e[i] - mx); sum += e[i]; }
        const float inv = 1.f / sum;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          if (g * 8 < NVp) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = e[g * 8 + i] * inv;
            sts128(opa + h * pHead + (uint32_t)((g * 128 + q4 * 32 + lane) * 16), pack8(v));
          }
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(bar(S_P));
      // ---- o -> A operand of the to_out product (overwrites the v operand) ----
      mbar_wait_relaxed(bar(S_OUT), ph_out);
      ph_out ^= 1;
      tc_fence_after();
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int col0 = (half * 2 + hh) * 32;
        tmem_ld32(tDo + lane_base + col0, r);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[g * 8 + i]);
          sts128(opb + (uint32_t)((((col0 >> 3) + g) * 128 + q4 * 32 + lane) * 16), pack8(v));
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(bar(S_OUTS));
      // ---- y = o W_o^T + bias + x ----
      mbar_wait_relaxed(bar(S_Y), ph_y);
      ph_y ^= 1;
      tc_fence_after();
      {
        const int ncol = C >> 1;
        const bool row_ok = q4 * 32 + lane < NV;
        const long roff = ((long)b * N + q4 * 32 + lane) * C + half * ncol;
#pragma unroll 1
        for (int c0 = 0; c0 < ncol; c0 += 32) {
          tmem_ld32(tDy + lane_base + (uint32_t)(half * ncol + c0), r);
          if (row_ok) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float xx[8], y[8];
              unpack8(ldcg128(p.x + roff + c0 + g * 8), xx);
#pragma unroll
              for (int i = 0; i < 8; ++i) y[i] = __uint_as_float(r[g * 8 + i]) + s_bo[half * ncol + c0 + g * 8 + i] + xx[i];
              *reinterpret_cast<uint4*>(p.out + roff + c0 + g * 8) = pack8(y);
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar(S_FREE));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

constexpr size_t kSmemSoftmax = 1024 + (size_t)(kXS + kWS) * kSlab + 3 * (size_t)kOpBytes + (128 + 256) * 4 + (S_COUNT + 2) * 8 + 64;

// =====================================================================================================================
// softmax Attention core for bottlenecks of more than 64 tokens (16x16 maps at 128x128 images): flash attention on the tensor cores
//   o[b][i][(h,e)] = sum_j softmax_j(scale * q_i . k_j) v_j[e]      (reference parts/mha.py:18-29, between to_qkv and to_out)
// qkv bf16 [B][N][384] (channel = which * 128 + head * 32 + d, as to_qkv writes it), o bf16 [B][N][128].
// One CTA per work item (image, 128-query tile, head); work items of an image are adjacent, so its k / v tiles are read from L2.
// The rank-3 tensor map [B][N][384] gives each image its own bounds: rows past N arrive as zeros and never come from the next
// image.  Per 128-key tile j (ring of kFlStages tiles brought by TMA, 128 rows x 32 channels, SWIZZLE_64B):
//   MMA       S = q k_j^T                       M128 x N128 x K32 (two k16 steps), fp32 in TMEM columns [0, 128)
//   epilogue  lane = query row: running max m and sum l in the log2 domain; padded key columns (j*128 + c >= N) get zero weight;
//             when m moves, the O accumulator row is rescaled in TMEM; P = bf16(ex2(s * scale * log2 e - m)) -> shared memory
//             (UMMA K-major no-swizzle layout), l sums the ROUNDED P so numerator and denominator agree; v_j is transposed into
//             the K-major B operand v^T [32 e][128 keys]
//   MMA       O += P v_j                        M128 x N32 x K128 (eight k16 steps), fp32 in TMEM columns [128, 160)
// Finally o = O / l, stored as bf16 for the tile's real query rows only.
// Warp roles (192 threads): warps 0-3 epilogue (warp w reads TMEM lanes [32w, 32w + 32)), warp 4 TMA, warp 5 TMEM + MMA issuer.
// 256 TMEM columns and ~98 KB of shared memory per CTA: two CTAs per SM overlap one's softmax with the other's products.
// =====================================================================================================================
constexpr int kFlThreads = 192, kFlTmaWarp = 4, kFlMmaWarp = 5, kFlStages = 3;
constexpr uint32_t kFlTile = 128u * 64u;                 // 128 tokens x 32 channels bf16 (64-byte rows, SWIZZLE_64B)
constexpr uint32_t kFlVtLbo = 32u * 16u;                 // v^T operand [16 k-chunks][32 rows][16 B]: k-chunk stride
enum { F_FULLQ = 0, F_FULL, F_EMPTY = F_FULL + kFlStages, F_S = F_EMPTY + kFlStages, F_P, F_O, F_COUNT };

struct FlashP {
  CUtensorMap m;                 // qkv as [B][N][384], box 32 channels x 128 tokens x 1 image
  bf16* o;
  int N, QT;                     // tokens per image, 128-token tiles per image
};

// rank-3 bf16 map [d2][d1][d0], box = 32 x 128 x 1, 64-byte swizzle; out-of-range rows read as zero
static int make_map3_sw64(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(-3, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {d0 * 2, d0 * d1 * 2};
  cuuint32_t box[3] = {32, 128, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(-3, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
  return 0;
}
__device__ __forceinline__ void tma_load3(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// K-major SWIZZLE_64B descriptor: rows of 64 B, 8-row groups 512 B apart (SBO), LBO unused (1), layout type 4 (as the conv engine)
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(512u >> 4) << 32) | (1ull << 46) | (4ull << 61);
}

__global__ void __launch_bounds__(kFlThreads, 2) attn_flash_kernel(const __grid_constant__ FlashP p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base0 = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (base0 & 1023u)) & 1023u);
  uint8_t* s_q = smem;                                   // q tile
  uint8_t* s_k = s_q + kFlTile;                          // kFlStages k tiles
  uint8_t* s_v = s_k + kFlStages * kFlTile;              // kFlStages v tiles (token-major, as TMA brings them)
  uint8_t* s_vt = s_v + kFlStages * kFlTile;             // v^T: B operand of the P v product
  uint8_t* s_p = s_vt + kFlTile;                         // P: A operand of the P v product (kOpBytes)
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_p + kOpBytes);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + F_COUNT);

  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int N = p.N, T = p.QT;
  const int h = blockIdx.x & 3, qt = (blockIdx.x >> 2) % T, b = (blockIdx.x >> 2) / T;
  const int q0 = qt * 128;
  auto bar = [&](int i) { return smem_u32(&bars[i]); };

  if (warp == kFlTmaWarp) {
    if (lane < F_COUNT) mbar_init(bar(lane), lane == F_P ? 128u : 1u);
    fence_barrier_init();
  }
  if (warp == kFlMmaWarp) tmem_alloc(smem_u32(tslot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t tS = tmem, tO = tmem + 128;

  if (warp == kFlTmaWarp) {
    // =============================================== TMA ===============================================
    const bool leader = elect_one();
    if (leader) {
      mbar_arrive_expect_tx(bar(F_FULLQ), kFlTile);
      tma_load3(smem_u32(s_q), &p.m, h * 32, q0, b, bar(F_FULLQ));
    }
    __syncwarp();
    for (int j = 0; j < T; ++j) {
      const int st = j % kFlStages;
      mbar_wait_relaxed(bar(F_EMPTY + st), ((j / kFlStages) & 1) ^ 1);
      if (leader) {
        mbar_arrive_expect_tx(bar(F_FULL + st), 2 * kFlTile);
        tma_load3(smem_u32(s_k) + st * kFlTile, &p.m, 128 + h * 32, j * 128, b, bar(F_FULL + st));
        tma_load3(smem_u32(s_v) + st * kFlTile, &p.m, 256 + h * 32, j * 128, b, bar(F_FULL + st));
      }
      __syncwarp();
    }
  } else if (warp == kFlMmaWarp) {
    // =============================================== MMA issuer ===============================================
    const bool leader = elect_one();
    const uint32_t idescS = make_idesc(128, 128), idescO = make_idesc(128, 32);
    const uint32_t sq = smem_u32(s_q), sp = smem_u32(s_p), svt = smem_u32(s_vt);
    mbar_wait(bar(F_FULLQ), 0);
    for (int j = 0; j < T; ++j) {
      const int st = j % kFlStages;
      mbar_wait(bar(F_FULL + st), (j / kFlStages) & 1);   // (S of the previous tile was read out before its F_P arrival)
      tc_fence_after();
      const uint32_t sk = smem_u32(s_k) + st * kFlTile;
      if (leader) {
#pragma unroll
        for (int k = 0; k < 2; ++k) umma_bf16(tS, make_desc_sw64(sq + k * 32), make_desc_sw64(sk + k * 32), idescS, k ? 1u : 0u);
        umma_commit(bar(F_S));
      }
      __syncwarp();
      mbar_wait(bar(F_P), j & 1);
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int k = 0; k < 8; ++k)
          umma_bf16(tO, make_desc(sp + k * kOpK16, kOpLbo, kOpSbo), make_desc(svt + k * 2 * kFlVtLbo, kFlVtLbo, kOpSbo), idescO,
                    (j | k) ? 1u : 0u);
        umma_commit(bar(F_O));                 // P, v^T and the accumulator are free again once these retire
        umma_commit(bar(F_EMPTY + st));
      }
      __syncwarp();
    }
  } else {
    // =============================================== epilogue: online softmax ===============================================
    const int row = warp * 32 + lane;                      // query row of the tile = TMEM lane
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    const float c2 = rsqrtf(32.f) * kLog2e;                // scale, in the log2 domain
    const uint32_t sp = smem_u32(s_p), svt = smem_u32(s_vt);
    float m_run = -INFINITY, l_run = 0.f;
    uint32_t r[32];
    for (int j = 0; j < T; ++j) {
      const int nvalid = N - j * 128;                      // key columns >= nvalid are padding
      mbar_wait_relaxed(bar(F_S), j & 1);
      tc_fence_after();
      float tmax = -INFINITY;
#pragma unroll
      for (int c0 = 0; c0 < 128; c0 += 32) {
        tmem_ld32(tS + lane_base + c0, r);
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c0 + i < nvalid) tmax = fmaxf(tmax, __uint_as_float(r[i]));
      }
      const float m_new = fmaxf(m_run, tmax * c2);
      const float corr = ex2(m_run - m_new);              // 0 on the first tile (m_run = -inf)
      if (j > 0) {                                         // the previous P v product has retired: P, v^T and O may be touched
        mbar_wait_relaxed(bar(F_O), (j - 1) & 1);
        tc_fence_after();
        if (__any_sync(0xffffffffu, corr != 1.f)) {
          tmem_ld32(tO + lane_base, r);
#pragma unroll
          for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * corr);
          tmem_st32(tO + lane_base, r);
          tmem_st_wait();
        }
      }
      float psum = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < 128; c0 += 32) {
        tmem_ld32(tS + lane_base + c0, r);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t w[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int i0 = g * 8 + 2 * e;
            const bf16 p0 = __float2bfloat16_rn(c0 + i0 < nvalid ? ex2(fmaf(__uint_as_float(r[i0]), c2, -m_new)) : 0.f);
            const bf16 p1 = __float2bfloat16_rn(c0 + i0 + 1 < nvalid ? ex2(fmaf(__uint_as_float(r[i0 + 1]), c2, -m_new)) : 0.f);
            psum += __bfloat162float(p0) + __bfloat162float(p1);
            w[e] = (uint32_t)(*reinterpret_cast<const unsigned short*>(&p0)) | ((uint32_t)(*reinterpret_cast<const unsigned short*>(&p1)) << 16);
          }
          sts128(sp + (uint32_t)((((c0 >> 3) + g) * 128 + row) * 16), make_uint4(w[0], w[1], w[2], w[3]));
        }
      }
      l_run = l_run * corr + psum;
      m_run = m_new;
      // v^T: this thread's key row (SWIZZLE_64B: logical 16-byte chunk c of row t sits at chunk c ^ ((t >> 1) & 3))
      const int st = j % kFlStages;
      mbar_wait_relaxed(bar(F_FULL + st), (j / kFlStages) & 1);
      const uint32_t vrow = smem_u32(s_v) + st * kFlTile + (uint32_t)row * 64u;
      const uint32_t vdst = svt + (uint32_t)(row >> 3) * kFlVtLbo + (uint32_t)(row & 7) * 2u;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint4 v = lds128(vrow + (uint32_t)((c ^ ((row >> 1) & 3)) * 16));
        const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          sts16(vdst + (uint32_t)(c * 8 + 2 * e) * 16u, (unsigned short)(u[e] & 0xffffu));
          sts16(vdst + (uint32_t)(c * 8 + 2 * e + 1) * 16u, (unsigned short)(u[e] >> 16));
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(bar(F_P));
    }
    mbar_wait_relaxed(bar(F_O), (T - 1) & 1);
    tc_fence_after();
    tmem_ld32(tO + lane_base, r);
    if (q0 + row < N) {
      const float inv = 1.f / l_run;
      bf16* dst = p.o + ((long)b * N + q0 + row) * 128 + h * 32;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float y[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) y[e] = __uint_as_float(r[g * 8 + e]) * inv;
        *reinterpret_cast<uint4*>(dst + g * 8) = pack8(y);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kFlMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem, 256);
  }
}

constexpr size_t kSmemFlash = 1024 + (size_t)(2 + 2 * kFlStages) * kFlTile + kOpBytes + (F_COUNT + 2) * 8 + 64;

}  // namespace fa

bool linattn_fused_supported(int B, int N, int C) {
  const bool n_ok = (N >= 128 && N % 128 == 0) || (N >= 16 && N < 128 && N % 8 == 0);
  return B >= 1 && n_ok && (C == 128 || C == 256) && (long)B * N < (1L << 30);
}

int linattn_fused(const LinAttnFusedP& q, cudaStream_t st) {
  if (!linattn_fused_supported(q.B, q.N, q.C)) return fail(-2, "linattn_fused: unsupported shape");
  fa::Params p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = fa::make_map(&p.mx, q.x, (uint64_t)q.B * q.N, (uint64_t)q.C, q.N >= 128 ? 128 : q.N))) return rc;
  if ((rc = fa::make_map(&p.mw, q.wqkv, 384, (uint64_t)q.C, 128))) return rc;
  if ((rc = fa::make_map(&p.mo, q.wo, (uint64_t)q.C, 128, 128))) return rc;
  p.x = (const bf16*)q.x;
  p.out = (bf16*)q.out;
  p.pstats = q.pstats;
  p.s1 = q.s1; p.s2 = q.s2; p.bo = q.bo; p.go = q.go; p.beo = q.beo;
  p.B = q.B; p.N = q.N; p.C = q.C;
  p.inv_cnt = 1.f / ((float)q.N * (float)q.C);
  static const bool trace_on = [] { const char* e = getenv("DMN_FA_TRACE"); return e && e[0] == '1'; }();
  if (trace_on) {
    void* sym = nullptr;
    DMN_CUDA_CHECK(cudaGetSymbolAddress(&sym, fa::g_fa_trace));
    p.trace = (long long*)sym;
  }
  static DeviceOnce attr;
  if (attr.first()) DMN_CUDA_CHECK(cudaFuncSetAttribute(fa::linattn_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fa::kSmemFused));
  const int grid = q.B < current_device_sms() ? q.B : current_device_sms();
  DMN_CUDA_CHECK(launch_pdl(fa::linattn_fused_kernel, dim3(grid), dim3(fa::kThreads), fa::kSmemFused, st, p));
  count_launch();
  DMN_LAUNCH_CHECK("linattn_fused");
  return 0;
}

bool attn_softmax_fused_supported(int B, int N, int C) {
  return B >= 1 && N >= 16 && N <= 64 && N % 8 == 0 && (C == 128 || C == 256) && (long)B * N < (1L << 30);
}

// Residual(PreNorm(Attention)): same parameter block as the linear form; go / beo are unused (to_out is a bare 1x1 here)
int attn_softmax_fused(const LinAttnFusedP& q, cudaStream_t st) {
  if (!attn_softmax_fused_supported(q.B, q.N, q.C)) return fail(-2, "attn_softmax_fused: unsupported shape");
  fa::Params p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = fa::make_map(&p.mx, q.x, (uint64_t)q.B * q.N, (uint64_t)q.C, q.N))) return rc;
  if ((rc = fa::make_map(&p.mw, q.wqkv, 384, (uint64_t)q.C, 128))) return rc;
  if ((rc = fa::make_map(&p.mo, q.wo, (uint64_t)q.C, 128, 128))) return rc;
  p.x = (const bf16*)q.x;
  p.out = (bf16*)q.out;
  p.pstats = q.pstats;
  p.s1 = q.s1; p.s2 = q.s2; p.bo = q.bo; p.go = q.go; p.beo = q.beo;
  p.B = q.B; p.N = q.N; p.C = q.C;
  p.inv_cnt = 1.f / ((float)q.N * (float)q.C);
  static DeviceOnce attr;
  if (attr.first()) DMN_CUDA_CHECK(cudaFuncSetAttribute(fa::attn_softmax_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fa::kSmemSoftmax));
  const int grid = q.B < current_device_sms() ? q.B : current_device_sms();
  DMN_CUDA_CHECK(launch_pdl(fa::attn_softmax_fused_kernel, dim3(grid), dim3(fa::kThreads), fa::kSmemSoftmax, st, p));
  count_launch();
  DMN_LAUNCH_CHECK("attn_softmax_fused");
  return 0;
}

int attn_flash(const void* qkv, void* out, int B, int heads, int N, cudaStream_t st) {
  DMN_REQUIRE(heads == 4, "attn_flash: heads must be 4 (384 qkv channels)");
  DMN_REQUIRE(B >= 1 && N > 64, "attn_flash: needs more than 64 tokens");
  fa::FlashP p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = fa::make_map3_sw64(&p.m, qkv, 384, (uint64_t)N, (uint64_t)B))) return rc;
  p.o = (bf16*)out;
  p.N = N;
  p.QT = (N + 127) / 128;
  const long grid = (long)B * p.QT * 4;
  DMN_REQUIRE(grid < (1L << 31), "attn_flash: too many work items");
  static DeviceOnce attr;
  if (attr.first()) DMN_CUDA_CHECK(cudaFuncSetAttribute(fa::attn_flash_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fa::kSmemFlash));
  DMN_CUDA_CHECK(launch_pdl(fa::attn_flash_kernel, dim3((unsigned)grid), dim3(fa::kFlThreads), fa::kSmemFlash, st, p));
  count_launch();
  DMN_LAUNCH_CHECK("attn_flash");
  return 0;
}

int fa_read_trace(long long* out, int n) {
  if (n > 64) n = 64;
  DMN_CUDA_CHECK(cudaDeviceSynchronize());
  DMN_CUDA_CHECK(cudaMemcpyFromSymbol(out, fa::g_fa_trace, (size_t)n * sizeof(long long)));
  return 0;
}

int selftest_tma_sw128_gemm(const void* a_bf16, const void* b_bf16, float* d, int M, int N, int K, cudaStream_t st) {
  DMN_REQUIRE(M > 0 && N > 0 && K > 0 && K % 64 == 0, "selftest_tma_sw128_gemm: K must be a multiple of 64");
  fa::SelfTestP p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = fa::make_map(&p.ma, a_bf16, (uint64_t)M, (uint64_t)K, 128))) return rc;
  if ((rc = fa::make_map(&p.mb, b_bf16, (uint64_t)N, (uint64_t)K, 128))) return rc;
  p.d = d; p.M = M; p.N = N; p.K = K;
  const size_t smem = 1024 + 2 * fa::kSlab + 64;
  static DeviceOnce attr;
  if (attr.first()) DMN_CUDA_CHECK(cudaFuncSetAttribute(fa::sw128_gemm_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fa::sw128_gemm_selftest_kernel<<<dim3((M + 127) / 128, (N + 127) / 128), 128, smem, st>>>(p);
  DMN_LAUNCH_CHECK("sw128_gemm_selftest");
  return 0;
}

}  // namespace dmn
