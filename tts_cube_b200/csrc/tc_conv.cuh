// tcgen05 (5th-gen tensor core) implicit-GEMM convolution for sm_100a: the dense layers of the ClariNet
// residual stack (gated dilated causal conv + conditioning 1x1; res/skip 1x1) as
//     D[M = 128 time steps, N = 256 output channels] += A[M, K] * B[N, K]^T
// with error-compensated split-fp16 arithmetic: every fp32 value x is carried as (hi, lo) fp16 with
// hi = fp16(x), lo = fp16(x - hi)  (22 significant bits), and the product is accumulated in fp32 as
//     a*w ~= a_hi*w_hi + a_hi*w_lo + a_lo*w_hi          (3 tcgen05.mma per K-step, |err| ~ 2^-22)
// which keeps the waveform within the 1e-3 budget where single-pass TF32/BF16/FP16 does not
// (SURVEY hard-part 2).
//
// Data layout: activations are CHANNELS-LAST fp16 planes [2(hi,lo)][B][T][C]; a K-major A tile
// (128 time rows x 64 channels = 128 B per row) is then ONE TMA box, the conv taps are the same box
// at row offset -tap*dilation, and the causal / "same" zero padding is TMA's out-of-bounds fill.
// Weights are pre-split, pre-scaled (power-of-two per output row, undone in the epilogue) and stored
// as ready-made 128B-swizzled smem images, fetched with 1-D bulk copies (no tensor map).
//
// Roles (576 threads): warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner, warps 2-17 =
// epilogue (TMEM -> registers -> global; four warps per TMEM lane quarter, a quarter of the columns each).  Persistent CTAs, 2-stage smem ring of 96 KB stages,
// double-buffered 2 x 256-column fp32 accumulators in TMEM.
#pragma once
#include <cuda_fp8.h>
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cube {
namespace tc {

constexpr int BM = 128;          // time steps per tile (UMMA M)
constexpr int BN = 256;          // output channels per tile (UMMA N)
#ifndef CUBE_TC_BK
#define CUBE_TC_BK 32
#endif
constexpr int BK = CUBE_TC_BK;   // channels per K chunk = one swizzle span of fp16 (64 -> SWIZZLE_128B, 32 -> SWIZZLE_64B)
constexpr int STAGES = (BK == 64) ? 2 : 4;       // 2 x 96 KB or 4 x 48 KB: same smem, deeper prefetch with BK=32
constexpr int ROW_BYTES = BK * 2;                // bytes per tile row = swizzle span
constexpr int SBO_BYTES = 8 * ROW_BYTES;         // 8-row core-matrix group stride
static_assert(BK == 64 || BK == 32, "BK must be 64 (SW128) or 32 (SW64)");
constexpr int A_TILE_BYTES = BM * BK * 2;        // 16 / 8 KB per plane
constexpr int B_TILE_BYTES = BN * BK * 2;        // 32 / 16 KB per plane
constexpr int STAGE_BYTES = 2 * A_TILE_BYTES + 2 * B_TILE_BYTES;  // 96 / 48 KB

// position (in fp16 elements) of element (row r, k) inside a swizzled [rows][BK] K-major tile image
__host__ __device__ constexpr int swz_off(int r, int k) {
  return (BK == 64) ? (r / 8) * 512 + (r % 8) * 64 + (((k / 8) ^ (r % 8)) * 8) + (k % 8)
                    : r * 32 + (((k / 8) ^ ((r >> 1) & 3)) * 8) + (k % 8);
}
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + BN * 8 /*scale,bias*/;
// per-N-tile-width variants (HiFi-GAN stages have 256/128/64/32 output channels)
// MS > 0 overrides the number of 128-row sub-tiles per scheduled tile: <128, false, 2> is the WIDE variant of the 128- and
// 256-channel HiFi-GAN stages (the latter as two 128-column tiles).  With one sub-tile those convs re-stream the whole weight
// set (k * C * 2C * 2 B: 0.7 MB at C = 128, k = 11) from L2 for every 128 rows, 45-53 B/clk per SM at the tensor core's pace -
// the L2 -> SM fabric, not the tensor core, bounded them; two sub-tiles share every staged weight image.
template <int TN, bool CG2 = false, int MS = 0> struct Cfg {
  static_assert(TN == 256 || TN == 128 || TN == 64 || TN == 32, "tile N");
  // CG2: a CTA pair computes a 256-row x TN tile with tcgen05.mma.cta_group::2; each CTA stages its own
  // 128 rows of A and HALF of the weight tile (the pair's tensor cores exchange the halves)
  static constexpr int B_BYTES = (CG2 ? TN / 2 : TN) * BK * 2;
  // narrow tiles are overhead-bound at 128 rows (a 128x32 tile is only 16 KB of output): a scheduled tile
  // then covers MSUB 128-row sub-tiles that share the staged weight chunk, the barriers and the tile setup
  static constexpr int MSUB = MS > 0 ? MS : (TN == 32 ? 4 : (TN == 64 ? 2 : 1));
  static constexpr int A_BYTES = MSUB * A_TILE_BYTES;           // per plane
  static constexpr int STAGE = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr int NSTAGE = (190 * 1024 / STAGE) > 8 ? 8 : (190 * 1024 / STAGE);
  static constexpr int SMEM = NSTAGE * STAGE + 1024 + 256 + TN * 8;
  // CAT (tiles narrower than 256 columns, single CTA): the hi*hi and hi*lo passes are ONE MMA of N = 2 TN on the weight
  // image [w_hi rows | w_lo rows] - one fetch of a_hi for two products (shared memory feeds the tensor core at ~64 B/clk,
  // which is what bounds these MMAs) - into separate column halves that the epilogue adds; lo*hi follows with N = TN
  // ... as long as the double-buffered accumulators of all sub-tiles still fit the 512 TMEM columns
  static constexpr bool CAT = TN < 256 && !CG2 && 2 * MSUB * 2 * TN <= 512;
  static constexpr int ACC_COLS = CAT ? 2 * TN : TN;           // accumulator columns per 128-row sub-tile
  static constexpr int TMEM_COLS = 2 * MSUB * ACC_COLS;        // 256 or 512: double-buffered accumulators
};
// Window mode: the taps of a dilated conv are overlapping row windows of the SAME tensor, so the A operand of a
// channel chunk is staged ONCE as a window of CTA_ROWS + (taps-1)*dil rows and every tap's MMA reads it through a
// row-offset smem descriptor (the 64B/128B swizzles are functions of the absolute shared-memory address, so a
// descriptor may start at any row).  L2->smem traffic for A drops by ~taps (11x for the k=11 HiFi-GAN convs).
// Two rings: A windows (big, few) and per-(chunk, tap) weight images (small, many).
template <int TN, int MS = 0> struct WinCfg {
  static constexpr int MSUB = Cfg<TN, false, MS>::MSUB;
  static constexpr int NBOX = MSUB + 1;                         // boxes per plane in an A slot (span <= 128 rows)
  static constexpr int A_SLOT = 2 * NBOX * A_TILE_BYTES;        // hi boxes, then lo boxes
  static constexpr int B_SLOT = 2 * TN * BK * 2;                // hi image, lo image
  static constexpr int SA = (TN == 128 && MSUB == 1) ? 3 : 2;
  static constexpr int SB_ = (190 * 1024 - SA * A_SLOT) / B_SLOT;
  static constexpr int SB = SB_ > 8 ? 8 : SB_;
  static constexpr int SMEM = SA * A_SLOT + SB * B_SLOT + 1024 + 256 + TN * 8;
  static_assert(SB >= 2, "weight ring too shallow");
};
constexpr int NUM_EPI_WARPS = 16;
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;   // TMA warp + MMA warp + epilogue warps

enum { TC_EPI_GATE = 0, TC_EPI_RESSKIP = 1, TC_EPI_FINAL = 2, TC_EPI_CONV = 3 };
enum { TC_ACC_NONE = 0, TC_ACC_SET = 1, TC_ACC_ADD = 2, TC_ACC_ADD_DIV = 3 };

struct TcSeg {
  int taps, dil, off0;   // source row of output row t, tap j: t + off0 + j*dil
  int nchunks;           // K chunks (of BK channels) per tap
  int last_ksteps;       // K steps (of 16 channels) that hold real data in the last chunk (1..BK/16)
  int src;               // which tensor map (tmA[src]) this segment reads
  int wchunk0;           // index of this segment's first weight image; image of (tap, cc) = wchunk0 + tap*nchunks + cc
  int nbox;              // window mode: 128-row TMA boxes that cover rows [t0+off0, t0+off0+CTA_ROWS+(taps-1)*dil)
};
constexpr int MAX_SEG = 4;

struct TcParams {
  CUtensorMap tmA[2];       // per segment: fp16 [2B][T][C] channels-last, box {64, 128, 1}, SWIZZLE_128B
  const __half* Wimg;       // [n_tiles][nchunks_total][2 planes][BN*BK] swizzled images
  const float* inv_scale;   // [N] per-output-row power-of-two de-scale
  const float* bias;        // [N]
  TcSeg seg[MAX_SEG];
  int nseg, nchunks_total;
  int B, T, n_tiles, t_tiles;
  const int* lens;          // [B] valid length (rows >= len are written as 0) or null
  int epi;
  // TC_EPI_GATE: o = tanh(f)*sigmoid(g) -> fp16 planes [2][B][T][outC], tile covers outC/n_tiles channels
  __half* out16; int outC;
  // TC_EPI_RESSKIP: cols [0,128): h = (h + v)*scale in place (fp16 planes [2][B][T][hC]);
  //                 cols [128,256): skip[b][c][t] (=|+=) v   (fp32 channel-first)
  __half* h16; int hC;
  float* skip; int skip_set;
  float scale;
  __half* skip16;           // RESSKIP, last block of a flow: relu(skip total) as fp16 planes [2][B][T][128]
                            // (the A operand of the flow's final 1x1) instead of the fp32 store
  // TC_EPI_FINAL: cols [0,128) = final_conv.1 output y1; fused relu -> final_conv.3 (128->2) -> IAF:
  //   z_out[t+1] = z_in[t+1]*exp(logs[t]) + mu[t], z_out[0] = 0
  const float* w3;          // [2][128] + bias [2]
  const float* z_in; float* z_out;   // [B][T]
  // TC_EPI_CONV (HiFi-GAN convs; every A-operand tensor holds leaky-ReLU'd values a = lrelu(x)):
  //   v = acc*inv_scale + bias (+ x_res, x_res = inverse-lrelu of res16 at the same row/col)
  //   out16 (if set)  <- lrelu(v, out_slope) as fp16 planes [2][B][L_out][outC]
  //   acc32 (if set)  : fp32 [B][outC][L_out] channel-first; SET: =v, ADD: +=v,
  //                     ADD_DIV: y=(acc+v)/acc_div -> acc32 (if acc_store) and out16b <- lrelu(y, out_slope)
  int nphase;               // transposed conv: output phases (weights per phase), else 1
  long long w_phase_stride; // fp16 elements between phase weight sets
  int ostride, ooff[8];     // output row of tile row q, phase r: q*ostride + ooff[r]
  int L_out;                // output rows per batch item; T = rows of q per batch item
  const __half* res16; float res_inv_slope;   // residual source planes [2][B][L_out][outC], 1/slope it was stored with
  float out_slope;
  float a_inv_scale;        // 1/S of the A-operand planes (folded into the per-column de-scale); 1 when unscaled
  float plane_scale;        // S: power-of-two scale of stored activation planes (keeps the fp16 `lo` part out of
                            // the subnormal range for small activations); residual planes are read back with 1/S
  float* acc32; int acc_mode; float acc_div; int acc_store;
  __half* out16b;
  int lean;                 // window mode: 1 = the MMA thread's short instruction stream ("lean issue" in the kernel)
  int row0, nrows;          // scheduled rows [row0, row0 + nrows) of q (nrows = 0: all T); the same for every batch item
};

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// non-blocking probe: try_wait may SUSPEND the thread up to a system-dependent time limit when the phase is not complete -
// a thread that polls two barriers in turn must use test_wait, or it sleeps on the one while the other completes
__device__ __forceinline__ uint32_t mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// shared -> global tile store (bulk async group of the issuing thread)
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(reinterpret_cast<uint64_t>(tm)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// the same loads with the completion mbarrier given as a raw 32-bit shared::cluster address (e.g. the LEADER CTA's barrier
// of a CTA pair, obtained with mapa_u32): the bytes land in this CTA's shared memory, the complete_tx goes to that barrier
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tma_load_3d_bar(void* dst, const CUtensorMap* tm, uint32_t bar_addr, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void bulk_load_bar(void* dst, const void* src, uint32_t bytes, uint32_t bar_addr) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar_addr)
               : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, fp16 inputs, fp32 accumulate, single CTA
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all MMAs issued so far by this thread -> one arrival on the mbarrier
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// one lane of a converged warp (elect.sync): the lane that issues the warp's MMAs and commits in the lean issue loops
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// ---- 2-CTA (cta_group::2) variants ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_2(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs -> one arrival on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_2(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, swizzled operand tile (rows of ROW_BYTES, 8-row groups SBO_BYTES apart), sm_100 descriptor
// (cute/arch/mma_sm100_desc.hpp: start>>4 [0,14), LBO [16,30), SBO [32,46), version=1 [46,48),
//  layout [61,64): SWIZZLE_128B=2, SWIZZLE_64B=4).
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                 // LBO (unused for swizzled K-major)
  d |= (uint64_t)(SBO_BYTES >> 4) << 32;  // SBO between 8-row groups
  d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
  d |= (uint64_t)(BK == 64 ? 2 : 4) << 61;
  return d;
}

// descriptor of the tile `byte_off` bytes further on (byte_off a multiple of 16, the sum still inside shared memory): only the
// 14-bit start-address field changes, and it cannot carry out of the low word.  ONE integer add - which matters: a single thread
// issues every MMA, and building each descriptor from its address (shift, mask, ors, 64-bit pack) costs ~75 cycles per MMA
// (tools/umma_microbench.cu: 74.9 cycles with per-MMA descriptor arithmetic, 50.9 with descriptors ready, for MMAs whose math is
// 16-64 cycles) - the narrow HiFi-GAN MMAs were issue-bound by exactly that.
__device__ __forceinline__ uint64_t desc_add(uint64_t d, uint32_t byte_off) {
  return (d & 0xFFFFFFFF00000000ull) | (uint64_t)((uint32_t)d + (byte_off >> 4));
}

// instruction descriptor: D=f32, A=B=f16, both K-major, M=128, N=n
__host__ __device__ constexpr uint32_t make_idesc(int n, int m = BM) {
  return (1u << 4) | (0u << 7) | (0u << 10) | (0u << 15) | (0u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---- 8-bit correction passes (tc_block_kernel<.., Q8 = true>): a_hi*w_lo and a_lo*w_hi carry a 2^-11 weight, so their
// operands may be e4m3 / e5m2 (kind::f8f6f4, K = 32 per instruction: twice the fp16 rate); see
// profiles/r1_split_precision_study.md.  Tiles are [rows][32 bytes] K-major, SWIZZLE_32B.
// byte offset of (row r, byte k) inside such a tile
__host__ __device__ constexpr int swz32_off(int r, int k) { return r * 32 + ((((k >> 4) & 1) ^ ((r >> 2) & 1)) << 4) + (k & 15); }
__device__ __forceinline__ uint64_t make_desc32(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                 // LBO (unused for swizzled K-major)
  d |= (uint64_t)((8 * 32) >> 4) << 32;   // SBO between 8-row groups of 32-byte rows
  d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
  d |= (uint64_t)6 << 61;                 // SWIZZLE_32B
  return d;
}
// instruction descriptor for kind::f8f6f4: D = f32, B = e4m3, A = e4m3 (a_e5m2 = 0) or e5m2 (1), both K-major
__host__ __device__ constexpr uint32_t make_idesc_f8(int n, int m, int a_e5m2) {
  return (1u << 4) | ((uint32_t)a_e5m2 << 7) | (0u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the two 8-bit planes of an activation stored as fp16 (hi, lo): e4m3(hi) and e5m2(16 * lo); two values per call
__device__ __forceinline__ void q8_pair(uint32_t hi2, uint32_t lo2, uint32_t& q_hi, uint32_t& q_lo) {
  const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi2));
  const float2 l = __half22float2(*reinterpret_cast<const __half2*>(&lo2));
  q_hi = __nv_cvt_float2_to_fp8x2(h, __NV_SATFINITE, __NV_E4M3);                                   // low byte = .x
  q_lo = __nv_cvt_float2_to_fp8x2(make_float2(l.x * 16.f, l.y * 16.f), __NV_SATFINITE, __NV_E5M2);
}

__device__ __forceinline__ __half f2h_sat(float x) {
  unsigned short r;
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(r) : "f"(x));
  return __ushort_as_half(r);
}
__device__ __forceinline__ void split16(float x, __half& hi, __half& lo) {
  hi = f2h_sat(x);
  lo = f2h_sat(x - __half2float(hi));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// (x0, x1) -> packed fp16 pair {x1 : x0} with saturation, and the residual pair
__device__ __forceinline__ uint32_t pack_h2_sat(float x0, float x1) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(x1), "f"(x0));
  return r;
}
__device__ __forceinline__ void split16x2(float x0, float x1, uint32_t& hi2, uint32_t& lo2) {
  hi2 = pack_h2_sat(x0, x1);
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi2));
  lo2 = pack_h2_sat(x0 - hf.x, x1 - hf.y);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t v) { return __half22float2(*reinterpret_cast<const __half2*>(&v)); }

// gate non-linearities on the SFU: ex2.approx + rcp.approx, abs error ~1e-6 (budget 1e-3)
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) { return 1.f - __fdividef(2.f, 1.f + __expf(2.f * x)); }

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
template <int TN, bool CG2 = false, bool WIN = false, int MS = 0>
__global__ void __launch_bounds__(NUM_THREADS, 1) tc_conv_kernel(const __grid_constant__ TcParams p) {
  static_assert(!(CG2 && WIN), "window mode is single-CTA");
  static_assert(!(CG2 && MS > 0), "the sub-tile override is single-CTA");
  constexpr int SA = WinCfg<TN, MS>::SA, SB = WinCfg<TN, MS>::SB;       // window mode rings
  constexpr int A_SLOT = WinCfg<TN, MS>::A_SLOT, B_SLOT = WinCfg<TN, MS>::B_SLOT;
  constexpr int A_LO_OFF = WinCfg<TN, MS>::NBOX * A_TILE_BYTES;     // lo plane inside an A slot
  constexpr int STAGES = WIN ? (SA + SB + 1) / 2 : Cfg<TN, CG2, MS>::NSTAGE;    // barrier-array stride only, in window mode
  constexpr int STAGE_BYTES = WIN ? (SA * A_SLOT + SB * B_SLOT + STAGES - 1) / STAGES : Cfg<TN, CG2, MS>::STAGE;
  constexpr int B_TILE_BYTES = Cfg<TN, CG2, MS>::B_BYTES;
  constexpr int BN = TN;
  constexpr bool CAT = Cfg<TN, CG2, MS>::CAT;
  constexpr int ACCW = Cfg<TN, CG2, MS>::ACC_COLS;
  constexpr int MSUB = Cfg<TN, CG2, MS>::MSUB;
  constexpr int A_BYTES = Cfg<TN, CG2, MS>::A_BYTES;
  constexpr int CTA_ROWS = MSUB * BM;               // rows this CTA owns in a scheduled tile
  constexpr int TILE_ROWS = CG2 ? 2 * CTA_ROWS : CTA_ROWS;   // rows of one scheduled tile (p.t_tiles counts these)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int DATA_BYTES = WIN ? SA * A_SLOT + SB * B_SLOT : STAGES * STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + DATA_BYTES);
  uint64_t* full = bars;                 // [STAGES]            (window mode: fullA[SA], emptyA[SA], fullB[SB], emptyB[SB])
  uint64_t* empty = bars + STAGES;       // [STAGES]
  uint64_t* pfull = bars + 2 * STAGES;   // [STAGES] (CG2, leader CTA): the peer CTA's stage is full
  uint64_t* fullA = bars, *emptyA = bars + SA, *fullB = bars + 2 * SA, *emptyB = bars + 2 * SA + SB;
  constexpr int NB_RING = WIN ? 2 * SA + 2 * SB : 3 * STAGES;
  uint64_t* tfull = bars + NB_RING;      // [2]
  uint64_t* tempty = bars + NB_RING + 2; // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + NB_RING + 4);
  static_assert((NB_RING + 4) * 8 + 4 <= 256, "barrier block");
  const uint32_t crank = CG2 ? cluster_ctarank() : 0u;      // 0 = leader (issues the pair's MMAs)
  const int tile0 = CG2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = CG2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  float2* s_sb = reinterpret_cast<float2*>(smem + DATA_BYTES + 256);   // [BN] (inv_scale, bias) of this tile

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nphase = p.nphase > 0 ? p.nphase : 1;
  const int total_tiles = p.n_tiles * p.t_tiles * p.B * nphase;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmA[0]);
    if (p.nseg > 1) prefetch_tmap(&p.tmA[1]);
    if constexpr (WIN) {
      for (int s = 0; s < SA; ++s) { mbar_init(&fullA[s], 1); mbar_init(&emptyA[s], 1); }
      for (int s = 0; s < SB; ++s) { mbar_init(&fullB[s], 1); mbar_init(&emptyB[s], 1); }
    } else {
      for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); mbar_init(&pfull[s], 1); }
    }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], CG2 ? 2 * NUM_EPI_WARPS : NUM_EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == 1) {
    if constexpr (CG2) tmem_alloc2(tmem_slot, Cfg<TN, CG2, MS>::TMEM_COLS); else tmem_alloc(tmem_slot, Cfg<TN, CG2, MS>::TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG2) cluster_sync_all();     // both CTAs' barriers are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (lane == 0 && WIN) {
      uint32_t ia = 0, ib = 0;
      for (int tile = tile0; tile < total_tiles; tile += tile_step) {
        const int nt = tile % p.n_tiles;
        int rest = tile / p.n_tiles;
        const int ph = rest % nphase; rest /= nphase;
        const int tt = rest % p.t_tiles, b = rest / p.t_tiles;
        const int t0 = p.row0 + tt * TILE_ROWS;
        const __half* wt = p.Wimg + (size_t)ph * p.w_phase_stride + (size_t)nt * p.nchunks_total * 2 * (BN * BK);
        for (int s = 0; s < p.nseg; ++s) {
          const TcSeg sg = p.seg[s];
          const CUtensorMap* tm = &p.tmA[sg.src];
          for (int cc = 0; cc < sg.nchunks; ++cc, ++ia) {
            {  // the A window of this channel chunk: nbox boxes of 128 rows, hi and lo planes
              const int sa = ia % SA;
              mbar_wait(&emptyA[sa], ((ia / SA) & 1) ^ 1);
              uint8_t* as = smem + sa * A_SLOT;
              mbar_expect_tx(&fullA[sa], 2 * sg.nbox * A_TILE_BYTES);
              for (int bx = 0; bx < sg.nbox; ++bx) {
                tma_load_3d(as + bx * A_TILE_BYTES, tm, &fullA[sa], cc * BK, t0 + sg.off0 + bx * BM, b);
                tma_load_3d(as + A_LO_OFF + bx * A_TILE_BYTES, tm, &fullA[sa], cc * BK, t0 + sg.off0 + bx * BM, p.B + b);
              }
            }
            for (int tap = 0; tap < sg.taps; ++tap, ++ib) {   // the weight image of every tap of this chunk
              const int sbi = ib % SB;
              mbar_wait(&emptyB[sbi], ((ib / SB) & 1) ^ 1);
              uint8_t* bs = smem + SA * A_SLOT + sbi * B_SLOT;
              const __half* wc = wt + (size_t)(sg.wchunk0 + tap * sg.nchunks + cc) * 2 * (BN * BK);
              mbar_expect_tx(&fullB[sbi], B_SLOT);
              bulk_load(bs, wc, B_SLOT / 2, &fullB[sbi]);
              bulk_load(bs + B_SLOT / 2, wc + BN * BK, B_SLOT / 2, &fullB[sbi]);
            }
          }
        }
      }
    }
    if (lane == 0 && !WIN) {
      uint32_t it = 0;
      for (int tile = tile0; tile < total_tiles; tile += tile_step) {
        const int nt = tile % p.n_tiles;
        int rest = tile / p.n_tiles;
        const int ph = rest % nphase; rest /= nphase;
        const int tt = rest % p.t_tiles, b = rest / p.t_tiles;
        const int t0 = p.row0 + tt * TILE_ROWS + (int)crank * CTA_ROWS;
        const __half* wt = p.Wimg + (size_t)ph * p.w_phase_stride + (size_t)nt * p.nchunks_total * 2 * (BN * BK);
        int chunk = 0;
        for (int s = 0; s < p.nseg; ++s) {
          const TcSeg sg = p.seg[s];
          for (int tap = 0; tap < sg.taps; ++tap) {
            const int row = t0 + sg.off0 + tap * sg.dil;
            for (int cc = 0; cc < sg.nchunks; ++cc, ++chunk, ++it) {
              const int st = it % STAGES;
              const uint32_t par = (it / STAGES) & 1;
              mbar_wait(&empty[st], par ^ 1);
              uint8_t* sb = smem + st * STAGE_BYTES;
              mbar_expect_tx(&full[st], STAGE_BYTES);
#pragma unroll
              for (int ms = 0; ms < MSUB; ++ms) {
                tma_load_3d(sb + ms * A_TILE_BYTES, &p.tmA[s], &full[st], cc * BK, row + ms * BM, b);
                tma_load_3d(sb + A_BYTES + ms * A_TILE_BYTES, &p.tmA[s], &full[st], cc * BK, row + ms * BM, p.B + b);
              }
              // weight tile rows [crank*BN/2, +BN/2) when the pair splits it, else all BN rows
              const __half* wc = wt + (size_t)chunk * 2 * (BN * BK) + (CG2 ? (size_t)crank * (BN / 2) * BK : 0);
              bulk_load(sb + 2 * A_BYTES, wc, B_TILE_BYTES, &full[st]);
              bulk_load(sb + 2 * A_BYTES + B_TILE_BYTES, wc + BN * BK, B_TILE_BYTES, &full[st]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    if (WIN && p.lean) {
      // Lean issue (see tc_block.cuh): the issuing thread's instruction stream, not the tensor core, paced the window-mode convs -
      // ncu on the 128-channel HiFi-GAN stage: tensor pipe 49 % active, the issuing warp never waiting, ~32 instructions per MMA
      // (ring indices modulo 5, a run-time K-step loop, descriptors per tap, the per-thread-to-uniform hand-over in front of every
      // MMA).  Here the WHOLE warp runs the loop (waits and counters are warp-uniform -> offsets and descriptors on the uniform
      // datapath, the MMAs of a (chunk, tap) issue back to back) and one elected lane issues the MMAs and commits; one descriptor
      // for the start of shared memory + byte offsets, K steps unrolled, ring slots / phases as counters.  Same MMAs, same order,
      // same barriers as the generic loop below.
      constexpr uint32_t idesc = make_idesc(TN, BM);
      constexpr uint32_t idesc_cat = make_idesc(CAT ? 2 * TN : TN, BM);
      (void)idesc_cat;
      const uint64_t D16 = make_desc(smem_u32(smem));
      const bool leader = elect_one();
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      uint32_t sa = 0, pha = 0, sbi = 0, phb = 0, titer = 0;
      // the MMAs of K step ks of one (chunk, tap): every sub-tile against the staged weight image
      auto kstep = [&](uint32_t d_tmem, uint32_t ao, uint32_t bo, int ks, uint32_t acc) {
        const uint32_t ko = ks * 32;
#pragma unroll
        for (int ms = 0; ms < MSUB; ++ms) {
          const uint32_t a = ao + ms * A_TILE_BYTES + ko;
          const uint32_t d = d_tmem + ms * ACCW;
          if constexpr (CAT) {     // [w_hi | w_lo] is one K-major tile of 2 TN rows (the lo image follows the hi image)
            umma_f16(d, desc_add(D16, a), desc_add(D16, bo + ko), idesc_cat, acc);
            umma_f16(d, desc_add(D16, a + A_LO_OFF), desc_add(D16, bo + ko), idesc, 1);
          } else {
            umma_f16(d, desc_add(D16, a), desc_add(D16, bo + ko), idesc, acc);
            umma_f16(d, desc_add(D16, a), desc_add(D16, bo + B_SLOT / 2 + ko), idesc, 1);
            umma_f16(d, desc_add(D16, a + A_LO_OFF), desc_add(D16, bo + ko), idesc, 1);
          }
        }
      };
      for (int tile = tile0; tile < total_tiles; tile += tile_step, ++titer) {
        const uint32_t acc = titer & 1, aph = (titer >> 1) & 1;
        mbar_wait(&tempty[acc], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + acc * (MSUB * ACCW);
        uint32_t accumulate = 0;
        for (int s = 0; s < p.nseg; ++s) {
          const int taps = p.seg[s].taps, nchunks = p.seg[s].nchunks, last_ksteps = p.seg[s].last_ksteps;
          const uint32_t tap_bytes = (uint32_t)p.seg[s].dil * ROW_BYTES;
          for (int cc = 0; cc < nchunks; ++cc) {
            mbar_wait(&fullA[sa], pha);
            const int ksteps = cc != nchunks - 1 ? BK / 16 : last_ksteps;
            uint32_t ao = sa * A_SLOT;                          // tap 0; every tap starts `dil` rows further into the window
            for (int tap = 0; tap < taps; ++tap, ao += tap_bytes) {
              mbar_wait(&fullB[sbi], phb);
              tc_fence_after();
              const uint32_t bo = SA * A_SLOT + sbi * B_SLOT;
              if (leader) {
#pragma unroll
                for (int ks = 0; ks < BK / 16; ++ks)
                  if (ks < ksteps) kstep(d_tmem, ao, bo, ks, ks ? 1u : accumulate);
                umma_commit(&emptyB[sbi]);
              }
              accumulate = 1;
              if (++sbi == SB) { sbi = 0; phb ^= 1; }
            }
            if (leader) umma_commit(&emptyA[sa]);
            if (++sa == SA) { sa = 0; pha ^= 1; }
          }
        }
        if (leader) umma_commit(&tfull[acc]);
      }
    } else if (lane == 0) {
      if (CG2 && crank != 0) {
        // peer CTA of a pair: it issues no MMA; this thread relays "my stage is full" to the leader
        uint32_t it = 0;
        for (int tile = tile0; tile < total_tiles; tile += tile_step) {
          for (int s = 0; s < p.nseg; ++s) {
            const TcSeg sg = p.seg[s];
            for (int n = sg.taps * sg.nchunks; n > 0; --n, ++it) {
              const int st = it % STAGES;
              mbar_wait(&full[st], (it / STAGES) & 1);
              mbar_arrive_remote(&pfull[st], 0);
            }
          }
        }
      } else if (WIN) {
        constexpr uint32_t idesc = make_idesc(TN, BM);
        constexpr uint32_t idesc_cat = make_idesc(CAT ? 2 * TN : TN, BM);
        uint32_t ia = 0, ib = 0, titer = 0;
        for (int tile = tile0; tile < total_tiles; tile += tile_step, ++titer) {
          const uint32_t acc = titer & 1, aph = (titer >> 1) & 1;
          mbar_wait(&tempty[acc], aph ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * (MSUB * ACCW);
          uint32_t accumulate = 0;
          for (int s = 0; s < p.nseg; ++s) {
            const TcSeg sg = p.seg[s];
            for (int cc = 0; cc < sg.nchunks; ++cc, ++ia) {
              const int sa = ia % SA;
              mbar_wait(&fullA[sa], (ia / SA) & 1);
              const uint32_t a_base = smem_u32(smem + sa * A_SLOT);
              const int ksteps = (cc == sg.nchunks - 1) ? sg.last_ksteps : (BK / 16);
              for (int tap = 0; tap < sg.taps; ++tap, ++ib) {
                const int sbi = ib % SB;
                mbar_wait(&fullB[sbi], (ib / SB) & 1);
                tc_fence_after();
                const uint32_t b_hi = smem_u32(smem + SA * A_SLOT + sbi * B_SLOT);
                const uint32_t a_tap = a_base + (uint32_t)(tap * sg.dil) * ROW_BYTES;   // row offset of this tap in the window
                // descriptors once per (chunk, tap); every MMA below adds a compile-time offset (desc_add)
                const uint64_t dah = make_desc(a_tap), dal = make_desc(a_tap + A_LO_OFF), dbh = make_desc(b_hi), dbl = make_desc(b_hi + B_SLOT / 2);
                for (int ks = 0; ks < ksteps; ++ks) {
                  const uint32_t ko = ks * 32;
#pragma unroll
                  for (int ms = 0; ms < MSUB; ++ms) {
                    const uint32_t ao = ms * A_TILE_BYTES + ko;
                    const uint32_t d = d_tmem + ms * ACCW;
                    if constexpr (CAT) {     // [w_hi | w_lo] is one K-major tile of 2 TN rows (the lo image follows the hi image)
                      umma_f16(d, desc_add(dah, ao), desc_add(dbh, ko), idesc_cat, accumulate);
                      umma_f16(d, desc_add(dal, ao), desc_add(dbh, ko), idesc, 1);
                    } else {
                      umma_f16(d, desc_add(dah, ao), desc_add(dbh, ko), idesc, accumulate);
                      umma_f16(d, desc_add(dah, ao), desc_add(dbl, ko), idesc, 1);
                      umma_f16(d, desc_add(dal, ao), desc_add(dbh, ko), idesc, 1);
                    }
                  }
                  accumulate = 1;
                }
                umma_commit(&emptyB[sbi]);
              }
              umma_commit(&emptyA[sa]);
            }
          }
          umma_commit(&tfull[acc]);
        }
      } else {
        constexpr uint32_t idesc = make_idesc(TN, CG2 ? 2 * BM : BM);
        constexpr uint32_t idesc_cat = make_idesc(CAT ? 2 * TN : TN, BM);
        uint32_t it = 0, titer = 0;
        for (int tile = tile0; tile < total_tiles; tile += tile_step, ++titer) {
          const uint32_t acc = titer & 1, aph = (titer >> 1) & 1;
          mbar_wait(&tempty[acc], aph ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * (MSUB * ACCW);
          uint32_t accumulate = 0;
          for (int s = 0; s < p.nseg; ++s) {
            const TcSeg sg = p.seg[s];
            for (int tap = 0; tap < sg.taps; ++tap) {
              for (int cc = 0; cc < sg.nchunks; ++cc, ++it) {
                const int st = it % STAGES;
                const uint32_t par = (it / STAGES) & 1;
                mbar_wait(&full[st], par);
                if constexpr (CG2) mbar_wait(&pfull[st], par);
                tc_fence_after();
                const uint32_t a_hi0 = smem_u32(smem + st * STAGE_BYTES);
                const uint32_t b_hi = a_hi0 + 2 * A_BYTES;
                const uint32_t b_lo = b_hi + B_TILE_BYTES;
                const int ksteps = (cc == sg.nchunks - 1) ? sg.last_ksteps : (BK / 16);
                for (int ks = 0; ks < ksteps; ++ks) {
                  const uint32_t ko = ks * 32;  // 16 fp16 = 32 bytes along K inside the swizzle span
#pragma unroll
                  for (int ms = 0; ms < MSUB; ++ms) {
                    const uint32_t a_hi = a_hi0 + ms * A_TILE_BYTES, a_lo = a_hi + A_BYTES;
                    const uint32_t d = d_tmem + ms * ACCW;
                    if constexpr (CAT) {
                      umma_f16(d, make_desc(a_hi + ko), make_desc(b_hi + ko), idesc_cat, accumulate);
                      umma_f16(d, make_desc(a_lo + ko), make_desc(b_hi + ko), idesc, 1);
                    } else if constexpr (CG2) {
                      umma_f16_2(d, make_desc(a_hi + ko), make_desc(b_hi + ko), idesc, accumulate);
                      umma_f16_2(d, make_desc(a_hi + ko), make_desc(b_lo + ko), idesc, 1);
                      umma_f16_2(d, make_desc(a_lo + ko), make_desc(b_hi + ko), idesc, 1);
                    } else {
                      umma_f16(d, make_desc(a_hi + ko), make_desc(b_hi + ko), idesc, accumulate);
                      umma_f16(d, make_desc(a_hi + ko), make_desc(b_lo + ko), idesc, 1);
                      umma_f16(d, make_desc(a_lo + ko), make_desc(b_hi + ko), idesc, 1);
                    }
                  }
                  accumulate = 1;
                }
                // frees the smem stage (in both CTAs of a pair) when these MMAs have read it
                if constexpr (CG2) umma_commit_2(&empty[st]); else umma_commit(&empty[st]);
              }
            }
          }
          // accumulator complete -> epilogue (of both CTAs of a pair)
          if constexpr (CG2) umma_commit_2(&tfull[acc]); else umma_commit(&tfull[acc]);
        }
      }
    }
  } else {
    // =========================== epilogue (warps 2..17) ===========================
    constexpr float LOG2E = 1.4426950408889634f;
    const int q = warp & 3;                 // TMEM lane quarter this warp may access
    const int grp = (warp - 2) >> 2;        // 0..3: warp group (one warp per TMEM lane quarter each)
    const int msub = grp % MSUB;            // 128-row sub-tile this warp reads
    const int sub = grp / MSUB;             // which slice of that sub-tile's columns (4/MSUB slices)
    const int row = q * 32 + lane;          // tile row = time step within the tile
    const int etid = threadIdx.x - 64;      // 0..511
    uint32_t titer = 0;
    int sb_nt = -1;                         // column tile whose (de-scale, bias) pairs are in s_sb
    for (int tile = tile0; tile < total_tiles; tile += tile_step, ++titer) {
      const int nt = tile % p.n_tiles;
      int rest = tile / p.n_tiles;
      const int ph = rest % nphase; rest /= nphase;
      const int tt = rest % p.t_tiles, b = rest / p.t_tiles;
      const int t = p.row0 + tt * TILE_ROWS + (int)crank * CTA_ROWS + msub * BM + row;
      const uint32_t acc = titer & 1, aph = (titer >> 1) & 1;
      // per-column (de-scale, bias) of this tile -> smem.  For the gate the exp2 pre-factors are
      // folded in: filter columns carry 2*log2(e) (-> 2^a = e^{2f}), gate columns -log2(e) (-> e^{-g}).
      if (nt != sb_nt) {   // (re)load only when the column tile changes: with an even grid it never does after the first tile
        asm volatile("bar.sync 1, 512;" ::: "memory");   // previous tile's readers are done
        if (etid < BN) {
          float sc = __ldg(p.inv_scale + nt * BN + etid) * p.a_inv_scale, bi = __ldg(p.bias + nt * BN + etid);
          if (p.epi == TC_EPI_GATE) {
            const float k = etid < BN / 2 ? 2.f * LOG2E : -LOG2E;
            sc *= k; bi *= k;
          }
          s_sb[etid] = make_float2(sc, bi);
        }
        asm volatile("bar.sync 1, 512;" ::: "memory");
        sb_nt = nt;
      }
      const uint32_t taddr = tmem_base + (acc * MSUB + msub) * ACCW + ((uint32_t)(q * 32) << 16);
      const int len = p.lens ? min(p.lens[b], p.T) : p.T;
      const bool in_range = t < p.T;
      const bool valid = t < len;
      // The epilogue's GLOBAL operands (residual planes, skip accumulator) do not depend on the MMAs: pull
      // them into L2 now, so that the loads issued after the accumulator wait pay L2 latency, not DRAM
      // latency (a register prefetch of the same data spilled: 64 extra live registers at 96/thread).
      if (in_range) {
        if (p.epi == TC_EPI_CONV) {
          if (p.res16) {
            const int t_out = t * p.ostride + p.ooff[ph];
            if (t_out >= 0 && t_out < p.L_out) {
              const __half* r0 = p.res16 + ((size_t)b * p.L_out + t_out) * p.outC + nt * BN + sub * (BN * MSUB / 4);
              prefetch_l2(r0);
              prefetch_l2(r0 + (size_t)p.B * p.L_out * p.outC);
            }
          }
        } else if (p.epi == TC_EPI_RESSKIP) {
          if (sub < 2) {
            const __half* h0 = p.h16 + ((size_t)b * p.T + t) * p.hC + sub * 64;   // 128 B per plane
            prefetch_l2(h0);
            prefetch_l2(h0 + (size_t)p.B * p.T * p.hC);
          } else if (!p.skip_set && (lane & 7) == 0) {   // 8 floats = one 32 B sector per prefetch
            const float* s0 = p.skip + ((size_t)b * (BN / 2) + (sub - 2) * 64) * p.T + t;
#pragma unroll 8
            for (int j = 0; j < 64; ++j) prefetch_l2(s0 + (size_t)j * p.T);
          }
        }
      }
      mbar_wait(&tfull[acc], aph);
      tc_fence_after();
      if (p.epi == TC_EPI_CONV) {
        // ---- HiFi-GAN convolution epilogue: bias, residual, leaky-ReLU, ResBlock averaging ----
        constexpr int CPS = BN * MSUB / 4;                // columns per epilogue warp
        constexpr int CW = CPS < 16 ? CPS : 16;           // columns per TMEM load
        const int t_out = t * p.ostride + p.ooff[ph];
        const int olen = p.lens ? min(p.lens[b], p.L_out) : p.L_out;
        const bool o_in = in_range && t_out >= 0 && t_out < p.L_out;
        const bool o_valid = o_in && t_out < olen;
        const size_t rowoff = ((size_t)b * p.L_out + (o_in ? t_out : 0)) * p.outC + nt * BN;
        const size_t plane = (size_t)p.B * p.L_out * p.outC;
#pragma unroll
        for (int cc = sub * CPS; cc < sub * CPS + CPS; cc += CW) {
          uint32_t r[CW];
          if constexpr (CW == 16) tmem_ld16(taddr + cc, r); else tmem_ld8(taddr + cc, r);
          uint32_t r2[CAT ? CW : 1];                       // CAT: the a_hi*w_lo products, TN columns further on
          if constexpr (CAT) { if constexpr (CW == 16) tmem_ld16(taddr + BN + cc, r2); else tmem_ld8(taddr + BN + cc, r2); }
          uint32_t rh[CW / 2], rl[CW / 2];
          float old[CW];
          if (p.res16 && o_in) {
#pragma unroll
            for (int v = 0; v < CW / 8; ++v) {
              const uint4 a = reinterpret_cast<const uint4*>(p.res16 + rowoff + cc)[v];
              const uint4 c = reinterpret_cast<const uint4*>(p.res16 + plane + rowoff + cc)[v];
              rh[4 * v] = a.x; rh[4 * v + 1] = a.y; rh[4 * v + 2] = a.z; rh[4 * v + 3] = a.w;
              rl[4 * v] = c.x; rl[4 * v + 1] = c.y; rl[4 * v + 2] = c.z; rl[4 * v + 3] = c.w;
            }
          } else {
#pragma unroll
            for (int v = 0; v < CW / 2; ++v) rh[v] = rl[v] = 0u;
          }
          if (p.acc32 && p.acc_mode >= TC_ACC_ADD && o_in) {
#pragma unroll
            for (int j = 0; j < CW; ++j) old[j] = __ldcs(p.acc32 + ((size_t)b * p.outC + nt * BN + cc + j) * p.L_out + t_out);
          } else {
#pragma unroll
            for (int j = 0; j < CW; ++j) old[j] = 0.f;
          }
          tmem_ld_wait();
          if constexpr (CAT) {
#pragma unroll
            for (int j = 0; j < CW; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
          }
          float v[CW];
#pragma unroll
          for (int j = 0; j < CW; j += 2) {
            const float2 s0 = s_sb[cc + j], s1 = s_sb[cc + j + 1];
            const float2 ah = unpack_h2(rh[j >> 1]), al = unpack_h2(rl[j >> 1]);
            float a0 = (ah.x + al.x) * p.a_inv_scale, a1 = (ah.y + al.y) * p.a_inv_scale;   // a = lrelu(x_res): invert
            a0 = a0 < 0.f ? a0 * p.res_inv_slope : a0;
            a1 = a1 < 0.f ? a1 * p.res_inv_slope : a1;
            v[j] = o_valid ? fmaf(__uint_as_float(r[j]), s0.x, s0.y) + a0 : 0.f;
            v[j + 1] = o_valid ? fmaf(__uint_as_float(r[j + 1]), s1.x, s1.y) + a1 : 0.f;
          }
          if (p.out16 && o_in) {
            uint32_t hi2[CW / 2], lo2[CW / 2];
#pragma unroll
            for (int j = 0; j < CW; j += 2) {
              const float y0 = v[j] < 0.f ? v[j] * p.out_slope : v[j], y1 = v[j + 1] < 0.f ? v[j + 1] * p.out_slope : v[j + 1];
              split16x2(y0 * p.plane_scale, y1 * p.plane_scale, hi2[j >> 1], lo2[j >> 1]);
            }
#pragma unroll
            for (int q4 = 0; q4 < CW / 8; ++q4) {
              reinterpret_cast<uint4*>(p.out16 + rowoff + cc)[q4] = make_uint4(hi2[4 * q4], hi2[4 * q4 + 1], hi2[4 * q4 + 2], hi2[4 * q4 + 3]);
              reinterpret_cast<uint4*>(p.out16 + plane + rowoff + cc)[q4] = make_uint4(lo2[4 * q4], lo2[4 * q4 + 1], lo2[4 * q4 + 2], lo2[4 * q4 + 3]);
            }
          }
          if (p.acc32 && o_in) {
            if (p.acc_mode == TC_ACC_ADD_DIV) {
#pragma unroll
              for (int j = 0; j < CW; ++j) v[j] = o_valid ? (old[j] + v[j]) / p.acc_div : 0.f;
              if (p.acc_store) {
#pragma unroll
                for (int j = 0; j < CW; ++j) __stcs(p.acc32 + ((size_t)b * p.outC + nt * BN + cc + j) * p.L_out + t_out, v[j]);
              }
              if (p.out16b) {
                uint32_t hi2[CW / 2], lo2[CW / 2];
#pragma unroll
                for (int j = 0; j < CW; j += 2) {
                  const float y0 = v[j] < 0.f ? v[j] * p.out_slope : v[j], y1 = v[j + 1] < 0.f ? v[j + 1] * p.out_slope : v[j + 1];
                  split16x2(y0 * p.plane_scale, y1 * p.plane_scale, hi2[j >> 1], lo2[j >> 1]);
                }
#pragma unroll
                for (int q4 = 0; q4 < CW / 8; ++q4) {
                  reinterpret_cast<uint4*>(p.out16b + rowoff + cc)[q4] = make_uint4(hi2[4 * q4], hi2[4 * q4 + 1], hi2[4 * q4 + 2], hi2[4 * q4 + 3]);
                  reinterpret_cast<uint4*>(p.out16b + plane + rowoff + cc)[q4] = make_uint4(lo2[4 * q4], lo2[4 * q4 + 1], lo2[4 * q4 + 2], lo2[4 * q4 + 3]);
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < CW; ++j) __stcs(p.acc32 + ((size_t)b * p.outC + nt * BN + cc + j) * p.L_out + t_out, old[j] + v[j]);
            }
          }
        }
      }
      if constexpr (TN == 256) {
      if (p.epi == TC_EPI_GATE) {
        // cols [0,128) filter, [128,256) gate of output channels nt*128 + c; this warp: c in [32*sub, +32)
        //   o = tanh(f)*sigmoid(g) = (E1 - 1) / ((E1 + 1)(1 + E2)),  E1 = e^{2f}, E2 = e^{-g}: 2 ex2 + 1 rcp
        const size_t plane = (size_t)p.B * p.T * p.outC;
        __half* orow = p.out16 + ((size_t)b * p.T + t) * p.outC + nt * (BN / 2);
#pragma unroll
        for (int cc = sub * 32; cc < sub * 32 + 32; cc += 16) {
          uint32_t f[16], g[16];
          tmem_ld16(taddr + cc, f);
          tmem_ld16(taddr + BN / 2 + cc, g);
          tmem_ld_wait();
          uint32_t hi2[8], lo2[8];
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            float o[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const float2 sf = s_sb[cc + j + u], sg = s_sb[BN / 2 + cc + j + u];
              const float a = fminf(fmaxf(fmaf(__uint_as_float(f[j + u]), sf.x, sf.y), -40.f), 40.f);
              const float e = fminf(fmaf(__uint_as_float(g[j + u]), sg.x, sg.y), 60.f);
              const float E1 = ex2_fast(a), E2 = ex2_fast(e);
              o[u] = valid ? (E1 - 1.f) * rcp_fast((E1 + 1.f) * (1.f + E2)) : 0.f;
            }
            split16x2(o[0], o[1], hi2[j >> 1], lo2[j >> 1]);
          }
          if (in_range) {
#pragma unroll
            for (int v = 0; v < 2; ++v) {
              reinterpret_cast<uint4*>(orow + cc)[v] = make_uint4(hi2[4 * v], hi2[4 * v + 1], hi2[4 * v + 2], hi2[4 * v + 3]);
              reinterpret_cast<uint4*>(orow + plane + cc)[v] = make_uint4(lo2[4 * v], lo2[4 * v + 1], lo2[4 * v + 2], lo2[4 * v + 3]);
            }
          }
        }
      } else if (p.epi == TC_EPI_FINAL) {
        if (sub == 0) {
          // y1 = cols [0,128); (mu, logs) = W3 . relu(y1) + b3; IAF affine on sample t+1
          float mu = __ldg(p.w3 + 2 * (BN / 2)), logs = __ldg(p.w3 + 2 * (BN / 2) + 1);
#pragma unroll 1
          for (int c0 = 0; c0 < BN / 2; c0 += 16) {
            uint32_t r[16];
            tmem_ld16(taddr + c0, r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float2 sb = s_sb[c0 + j];
              const float y = fmaxf(fmaf(__uint_as_float(r[j]), sb.x, sb.y), 0.f);
              mu = fmaf(y, __ldg(p.w3 + c0 + j), mu);
              logs = fmaf(y, __ldg(p.w3 + (BN / 2) + c0 + j), logs);
            }
          }
          if (in_range) {
            float* zo = p.z_out + (size_t)b * p.T;
            if (t == 0) zo[0] = 0.f;
            if (t + 1 < p.T) zo[t + 1] = (t + 1 < len) ? fmaf(p.z_in[(size_t)b * p.T + t + 1], expf(logs), mu) : 0.f;
          }
        }
      } else if (p.epi == TC_EPI_RESSKIP && sub < 2) {
        // cols [0,128): residual stream, updated in place (fp16 planes); this warp: c in [64*sub, +64)
        const size_t plane = (size_t)p.B * p.T * p.hC;
        __half* hrow = p.h16 + ((size_t)b * p.T + t) * p.hC;
#pragma unroll
        for (int cc = sub * 64; cc < sub * 64 + 64; cc += 16) {
          uint32_t r[16];
          tmem_ld16(taddr + cc, r);
          uint4 hv[2], lv[2];
          if (in_range) {
#pragma unroll
            for (int v = 0; v < 2; ++v) {
              hv[v] = reinterpret_cast<const uint4*>(hrow + cc)[v];
              lv[v] = reinterpret_cast<const uint4*>(hrow + plane + cc)[v];
            }
          } else {
            hv[0] = hv[1] = lv[0] = lv[1] = make_uint4(0, 0, 0, 0);
          }
          tmem_ld_wait();
          const uint32_t* hp = reinterpret_cast<const uint32_t*>(hv);
          const uint32_t* lp = reinterpret_cast<const uint32_t*>(lv);
          uint32_t hi2[8], lo2[8];
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const float2 s0 = s_sb[cc + j], s1 = s_sb[cc + j + 1];
            const float2 oh = unpack_h2(hp[j >> 1]), ol = unpack_h2(lp[j >> 1]);
            const float v0 = fmaf(__uint_as_float(r[j]), s0.x, s0.y), v1 = fmaf(__uint_as_float(r[j + 1]), s1.x, s1.y);
            const float n0 = valid ? ((oh.x + ol.x) + v0) * p.scale : 0.f;
            const float n1 = valid ? ((oh.y + ol.y) + v1) * p.scale : 0.f;
            split16x2(n0, n1, hi2[j >> 1], lo2[j >> 1]);
          }
          if (in_range) {
#pragma unroll
            for (int v = 0; v < 2; ++v) {
              reinterpret_cast<uint4*>(hrow + cc)[v] = make_uint4(hi2[4 * v], hi2[4 * v + 1], hi2[4 * v + 2], hi2[4 * v + 3]);
              reinterpret_cast<uint4*>(hrow + plane + cc)[v] = make_uint4(lo2[4 * v], lo2[4 * v + 1], lo2[4 * v + 2], lo2[4 * v + 3]);
            }
          }
        }
      } else if (p.epi == TC_EPI_RESSKIP) {
        // cols [128,256): skip accumulator, fp32 [B][128][T]; lanes -> consecutive t: coalesced.
        // this warp: skip channels [64*(sub-2), +64).  All loads of a chunk are issued before the
        // first use (the compiler may not hoist them over the previous column's store by itself).
        float* sp0 = p.skip + (size_t)b * (BN / 2) * p.T + t;
#pragma unroll
        for (int cc = (sub - 2) * 64; cc < (sub - 2) * 64 + 64; cc += 16) {
          uint32_t r[16];
          float old[16];
          tmem_ld16(taddr + BN / 2 + cc, r);
          if (in_range && !p.skip_set) {
#pragma unroll
            for (int j = 0; j < 16; ++j) old[j] = __ldcs(sp0 + (size_t)(cc + j) * p.T);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) old[j] = 0.f;
          }
          tmem_ld_wait();
          if (p.skip16) {
            uint32_t hi2[8], lo2[8];
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              const float2 s0 = s_sb[BN / 2 + cc + j], s1 = s_sb[BN / 2 + cc + j + 1];
              const float y0 = old[j] + fmaf(__uint_as_float(r[j]), s0.x, s0.y);
              const float y1 = old[j + 1] + fmaf(__uint_as_float(r[j + 1]), s1.x, s1.y);
              split16x2(valid ? fmaxf(y0, 0.f) : 0.f, valid ? fmaxf(y1, 0.f) : 0.f, hi2[j >> 1], lo2[j >> 1]);
            }
            if (in_range) {
              __half* srow = p.skip16 + ((size_t)b * p.T + t) * (BN / 2) + cc;
              const size_t splane = (size_t)p.B * p.T * (BN / 2);
#pragma unroll
              for (int v = 0; v < 2; ++v) {
                reinterpret_cast<uint4*>(srow)[v] = make_uint4(hi2[4 * v], hi2[4 * v + 1], hi2[4 * v + 2], hi2[4 * v + 3]);
                reinterpret_cast<uint4*>(srow + splane)[v] = make_uint4(lo2[4 * v], lo2[4 * v + 1], lo2[4 * v + 2], lo2[4 * v + 3]);
              }
            }
          } else if (in_range) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float2 sb = s_sb[BN / 2 + cc + j];
              const float y = old[j] + fmaf(__uint_as_float(r[j]), sb.x, sb.y);
              __stcs(sp0 + (size_t)(cc + j) * p.T, valid ? y : 0.f);
            }
          }
        }
      }
      }  // TN == 256 (ClariNet epilogues)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG2 && crank != 0) mbar_arrive_remote(&tempty[acc], 0);   // the leader's MMA thread owns the accumulators' reuse
        else mbar_arrive(&tempty[acc]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG2) cluster_sync_all();     // no CTA of the pair exits while the other may still signal it
  if (warp == 1) {
    tc_fence_after();
    if constexpr (CG2) tmem_dealloc2(tmem_base, Cfg<TN, CG2, MS>::TMEM_COLS); else tmem_dealloc(tmem_base, Cfg<TN, CG2, MS>::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// fp32 [B][C][T] (channel-first) -> fp16 hi/lo planes [2][B][T][C] (channels-last); tiled transpose
// through shared memory so both sides are coalesced.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) to_hl16_kernel(const float* __restrict__ src, __half* __restrict__ dst, int B, int C, int T,
                                                      const int* __restrict__ lens = nullptr, float scale = 1.f,
                                                      int row0 = 0) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, t0 = row0 + blockIdx.x * 32;   // grid.x covers the rows wanted from row0
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, t = t0 + tx;
    const int tl = lens ? min(lens[blockIdx.z], T) : T;   // rows past the valid length read as zero
    tile[i][tx] = (c < C && t < tl) ? src[((size_t)b * C + c) * T + t] : 0.f;
  }
  __syncthreads();
  const size_t plane = (size_t)B * T * C;
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + i, c = c0 + tx;
    if (t < T && c < C) {
      __half hi, lo;
      split16(tile[tx][i] * scale, hi, lo);
      const size_t o = ((size_t)b * T + t) * C + c;
      dst[o] = hi;
      dst[plane + o] = lo;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Causal taps of a 1-channel signal as channels: z fp32 [B][T] -> fp16 hi/lo planes [2][B][T][K],
// plane element (b, t, j) = z[b][t - (K-1) + j] (zero before the start).  Turns the ClariNet front conv
// (Conv1d 1 -> 128, k = 32, causal) into a K-channel 1x1 GEMM for the tensor-core path.  A thread writes one
// 16-byte piece (8 taps) of a row per plane: consecutive threads = consecutive pieces, fully coalesced.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) taps_to_hl16_kernel(const float* __restrict__ z, __half* __restrict__ dst, int B, int T, int K) {
  const int ppr = K / 8;                                    // pieces per row
  const long long total = (long long)B * T * ppr;
  const size_t plane = (size_t)B * T * K;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int piece = (int)(i % ppr);
    const long long row = i / ppr;                          // b * T + t
    const int t = (int)(row % T);
    const float* zb = z + (row - t);
    const int t0 = t - (K - 1) + piece * 8;
    uint32_t hi2[4], lo2[4];
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      const float a = (t0 + j >= 0) ? __ldg(zb + t0 + j) : 0.f;
      const float b = (t0 + j + 1 >= 0) ? __ldg(zb + t0 + j + 1) : 0.f;
      split16x2(a, b, hi2[j >> 1], lo2[j >> 1]);
    }
    reinterpret_cast<uint4*>(dst)[i] = make_uint4(hi2[0], hi2[1], hi2[2], hi2[3]);
    reinterpret_cast<uint4*>(dst + plane)[i] = make_uint4(lo2[0], lo2[1], lo2[2], lo2[3]);
  }
}

// fp16 (hi, lo) planes [2][n] -> 8-bit planes [2][n]: e4m3(hi), e5m2(16 lo); 8 elements per thread and step
__global__ void __launch_bounds__(256) hl16_to_q8_kernel(const __half* __restrict__ src, uint8_t* __restrict__ dst, long long n) {
  const long long n8 = n / 8;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n8; i += (long long)gridDim.x * 256) {
    const uint4 h = reinterpret_cast<const uint4*>(src)[i];
    const uint4 l = reinterpret_cast<const uint4*>(src + n)[i];
    uint32_t a0, a1, a2, a3, b0, b1, b2, b3;
    q8_pair(h.x, l.x, a0, b0); q8_pair(h.y, l.y, a1, b1); q8_pair(h.z, l.z, a2, b2); q8_pair(h.w, l.w, a3, b3);
    reinterpret_cast<uint2*>(dst)[i] = make_uint2(a0 | (a1 << 16), a2 | (a3 << 16));
    reinterpret_cast<uint2*>(dst + n)[i] = make_uint2(b0 | (b1 << 16), b2 | (b3 << 16));
  }
}

}  // namespace tc
}  // namespace cube
