// One HiFi-GAN ResBlock1 step in ONE tcgen05 kernel (sm_100a), for the narrow stages (C = 32, 64 channels):
//     y1 = conv1_{k, dil}(lrelu(x)) + b1                  GEMM1, K = k * C          (hifigan/models.py:37-39)
//     a1 = lrelu(y1)                                       stays ON CHIP (TMEM -> registers -> swizzled smem A tiles)
//     y2 = conv2_{k, 1}(a1) + b2                           GEMM2, K = k * C          (hifigan/models.py:40-41)
//     x' = y2 + x                                          (:42)
// The unfused pair (two tc_conv_kernel launches) round-trips a1 through HBM as 4-byte hi/lo planes and re-reads x as the
// residual: 5 plane passes per step where the algorithm needs 2 (read x, write x').  These stages are HBM-bound on the
// tensor cores (24-176 FLOP/B, DESIGN.md), so the passes are the time.  Here a CTA stages ONE window of x per tile
// (rows [t0 - h2 - h1, ...), h1 = dil (k-1)/2, h2 = (k-1)/2), runs conv1 on NSUB*128 rows (the h2 halo rows of a1 that conv2
// needs are recomputed: 2 h2 of NSUB*128 rows, 2-4 %), writes a1 as K-major SWIZZLE_64B tiles into shared memory, and
// conv2's taps read them through row-offset descriptors (window mode of tc_conv.cuh).  Tile = NSUB*128 - 2 h2 output rows.
//
// Every A-operand tensor holds leaky-ReLU'd values (slope 0.1) as split-fp16 (hi, lo) planes, channels-last
// [2][B][L][C], exactly as tc_conv_kernel's TC_EPI_CONV leaves them; arithmetic is the same error-compensated
// a_hi*w_hi + a_hi*w_lo + a_lo*w_hi with fp32 accumulation in TMEM.
//
// Roles (608 threads): warp 0 = TMA producer (x window, weight ring), warps 1 and 18 = MMA issuers (half of the sub-tiles
// each), warps 2-17 = epilogue.  Software pipeline over the tiles of a CTA (it = tile counter):
//     producer :  X(it)  W1(it)  W2(it-1)
//     MMA      :  M1(it)         M2(it-1)          (conv1 of the next tile is issued BEFORE conv2 of this one, so the
//     epilogue :  E1(it)         E2(it-1)           tensor pipe runs M1(it) while E1(it-1)'s a1 tiles are being written)
// A run-time order (whichever of M1(it+1) / M2(it) is ready first; one weight ring per conv; issuer B following issuer A's
// decision log, because two issuers taking different orders deadlock on the shared weight rings) was built and measured in
// round 2: parity-green and 16 % MORE cycles (half-depth weight rings, polling), so the fixed order stays (git history).
// What a narrow MMA costs (tools/umma_microbench.cu, profiles/r2_umma_microbench_*.txt): the tensor core needs 40 / 48 / 65 / 129
// cycles for N = 32 / 64 / 128 / 256 (operand fetch at 128 B/clk, then math), but ONE issuing thread needs 51 cycles per MMA with
// its descriptors ready and 75 when it builds them per MMA.  Hence: descriptors once per (tap, chunk) + one integer add per MMA
// (desc_add), a warp-uniform TMEM base, two issuing warps, and the hi*hi and hi*lo passes as ONE MMA: the weight image
// [w_hi rows | w_lo rows] is a single B tile of N = 2C, its two products land in separate column halves of the accumulator (the
// epilogue adds them), and lo*hi follows with N = C into the first half - 2 MMAs per K step instead of 3.
// TMEM: [acc1: NSUB*2C | acc2: NSUB*2C] columns = 512, single-buffered: the interleaved schedule leaves E1(it) a whole
// M2(it-1) to drain acc1 before M1(it+1) needs it, and E2(it-1) a whole M1(it+1) to drain acc2 before M2(it).
#pragma once
#include "tc_conv.cuh"

namespace cube {
namespace tc {

template <int C, int NSUB> struct RbCfg {
  static_assert(C == 32 || C == 64, "narrow stages only");
  static constexpr int NCH = C / BK;                               // K chunks (of 32 channels) per tap
  static_assert(NSUB * NCH == 4, "16 epilogue warps = 4 lane quarters x (NSUB sub-tiles x NCH column chunks)");
  static constexpr int NBOX = NSUB + 1;                            // 128-row boxes of the x window (2 h1 <= 128)
  static constexpr int XPLANE = NBOX * A_TILE_BYTES;               // one (chunk, plane) of the window
  static constexpr int XWIN = NCH * 2 * XPLANE;
  static constexpr int MPLANE = NSUB * A_TILE_BYTES;               // one (chunk, plane) of a1
  static constexpr int MID = NCH * 2 * MPLANE + 1024;              // + slack: the last tap of the last sub-tile reads 2 h2 rows past the end
  static constexpr int WIMG = 2 * C * BK * 2;                      // (hi, lo) image of one (tap, chunk): C rows x 32 ch
  static constexpr int WS_ = (222 * 1024 - XWIN - MID - 1024) / WIMG;
  static constexpr int WS = WS_ > 12 ? 12 : WS_;                   // weight ring depth
  static constexpr int BAR_BYTES = 512;
  static constexpr int SMEM = 1024 + XWIN + MID + WS * WIMG + BAR_BYTES + 2 * C * 8;
  static constexpr int ACC = NSUB * 2 * C;                         // columns of one accumulator: per sub-tile [hi*hi + lo*hi | hi*lo]
  static_assert(2 * ACC == 512, "TMEM budget");
  static_assert(WS >= 4, "weight ring too shallow");
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
};

struct RbParams {
  CUtensorMap tmX;            // input planes lrelu(x): fp16 [2B][L][C] channels-last, box {32 ch, 128 rows, 1}, SWIZZLE_64B
  const __half* W1;           // conv1 images [k taps][NCH][2 planes][C x 32] (pack_tc_conv1d)
  const __half* W2;           // conv2 images, same layout
  const float* inv1; const float* bias1;   // [C] power-of-two de-scale and bias of conv1
  const float* inv2; const float* bias2;
  int k, dil;                 // conv1: k taps at dilation dil; conv2: k taps at dilation 1; "same" padding
  int B, L, t_tiles;          // L rows per batch item; t_tiles = ceil(nrows / (NSUB*128 - (k-1)))
  int row0, nrows;            // output rows [row0, row0 + nrows) are scheduled (nrows = 0: all L); the same for every item
  const int* lens;            // [B] valid rows (rows >= len are written as zero) or null
  const __half* x16;          // the same input planes, for the residual (x = inverse leaky-ReLU of the stored value)
  float slope, inv_slope;     // 0.1, 10
  __half* out16;              // lrelu(x') planes [2][B][L][C] (next step's input), or null on a ResBlock's last step
  // last step of a ResBlock: the stage's running sum, fp32 [B][C][L] channel-first (TC_ACC_* of tc_conv.cuh)
  float* acc32; int acc_mode; float acc_div; int acc_store;
  __half* out16b;             // TC_ACC_ADD_DIV: lrelu((acc + x') / acc_div) planes = the next stage's input
};

// 19 warps: TMA producer, MMA issuer A, 16 epilogue warps, MMA issuer B.  TWO issuing warps, each with half of the sub-tiles:
// a narrow MMA occupies the tensor core for 40-50 cycles (tools/umma_microbench.cu) but costs its issuing thread 50-75 (descriptor
// adds, the ELECT / UTCHMMA / branch sequence, a barrier wait and a commit per tap), so one thread cannot keep the pipe fed.
constexpr int RB_THREADS = NUM_THREADS + 32;
constexpr int RB_ISSUERS = 2;

// packed fp32 helpers of the PK epilogue (sm_100 FADD2 / FMUL2 / FFMA2: two IEEE round-to-nearest operations per instruction, so
// every value is bit-identical to the scalar epilogue's)
__device__ __forceinline__ float2 rb_f2(uint32_t a, uint32_t b) { return make_float2(__uint_as_float(a), __uint_as_float(b)); }
// leaky ReLU with 0 < slope < 1 as max(v, slope v); its inverse (factor > 1) as min(a, factor a)
__device__ __forceinline__ float2 rb_lrelu2(float2 v, float2 slope2) {
  const float2 t = __fmul2_rn(v, slope2);
  return make_float2(fmaxf(v.x, t.x), fmaxf(v.y, t.y));
}
__device__ __forceinline__ float2 rb_unlrelu2(float2 a, float2 inv2) {
  const float2 t = __fmul2_rn(a, inv2);
  return make_float2(fminf(a.x, t.x), fminf(a.y, t.y));
}
__device__ __forceinline__ void rb_split2(float2 v, uint32_t& hi2, uint32_t& lo2) {
  hi2 = pack_h2_sat(v.x, v.y);
  const float2 d = __ffma2_rn(unpack_h2(hi2), make_float2(-1.f, -1.f), v);   // v - fp16(v), one rounding as in split16x2
  lo2 = pack_h2_sat(d.x, d.y);
}

// PK: the epilogue's fp32 arithmetic on channel PAIRS (packed instructions), masks as branches around the stores instead of a
// select per value.  The 16 epilogue warps execute ~1100 instructions per tile each, and at k = 3 that - not the tensor pipe -
// sets the tile period (profiles/r2_ncu_hot_rbstep32.txt); the packed form needs about a quarter fewer.
template <int C, int NSUB, bool PK = false>
__global__ void __launch_bounds__(RB_THREADS, 1) tc_rbstep_kernel(const __grid_constant__ RbParams p) {
  using Cfg = RbCfg<C, NSUB>;
  constexpr int NCH = Cfg::NCH, NBOX = Cfg::NBOX, WS = Cfg::WS, ACC = Cfg::ACC;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* xwin = smem;                                   // [NCH][hi, lo][NBOX boxes]
  uint8_t* mid = xwin + Cfg::XWIN;                        // [NCH][hi, lo][NSUB tiles] (+ slack)
  uint8_t* wring = mid + Cfg::MID;                        // [WS][hi image | lo image]
  uint64_t* bars = reinterpret_cast<uint64_t*>(wring + WS * Cfg::WIMG);
  uint64_t* xfull = bars;                // [1]
  uint64_t* xempty = bars + 1;           // [1]
  uint64_t* wfull = bars + 2;            // [WS]
  uint64_t* wempty = wfull + WS;         // [WS]
  uint64_t* a1full = wempty + WS;        // [1]  MMA -> epilogue
  uint64_t* a1free = a1full + 1;         // [1]  epilogue (16 warps) -> MMA
  uint64_t* a2full = a1free + 1;         // [1]
  uint64_t* a2free = a2full + 1;         // [1]
  uint64_t* midfull = a2free + 1;        // [1]  epilogue (16 warps) -> MMA
  uint64_t* midfree = midfull + 1;       // [1]  MMA -> epilogue
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(midfree + 1);
  static_assert((2 + 2 * WS + 6) * 8 + 8 <= Cfg::BAR_BYTES, "barrier block");
  float2* sb1 = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(bars) + Cfg::BAR_BYTES);   // [C] (de-scale, bias) of conv1
  float2* sb2 = sb1 + C;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h2 = (p.k - 1) / 2, h1 = p.dil * h2;
  const int R_OUT = NSUB * BM - 2 * h2;                   // output rows of a tile
  const int total_tiles = p.t_tiles * p.B;
  int my_tiles = 0;
  if ((int)blockIdx.x < total_tiles) my_tiles = (total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmX);
    mbar_init(xfull, 1); mbar_init(xempty, RB_ISSUERS);                 // every issuer commits what IT issued
    for (int s = 0; s < WS; ++s) { mbar_init(&wfull[s], 1); mbar_init(&wempty[s], RB_ISSUERS); }
    mbar_init(a1full, RB_ISSUERS); mbar_init(a1free, NUM_EPI_WARPS);
    mbar_init(a2full, RB_ISSUERS); mbar_init(a2free, NUM_EPI_WARPS);
    mbar_init(midfull, NUM_EPI_WARPS); mbar_init(midfree, RB_ISSUERS);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  for (int i = threadIdx.x; i < C; i += RB_THREADS) {
    if constexpr (PK) {   // per channel pair {inv_j, inv_j+1, bias_j, bias_j+1}: one 16-byte read feeds a packed FFMA
      const int pr = i >> 1, hf = i & 1;
      reinterpret_cast<float*>(sb1)[pr * 4 + hf] = __ldg(p.inv1 + i); reinterpret_cast<float*>(sb1)[pr * 4 + 2 + hf] = __ldg(p.bias1 + i);
      reinterpret_cast<float*>(sb2)[pr * 4 + hf] = __ldg(p.inv2 + i); reinterpret_cast<float*>(sb2)[pr * 4 + 2 + hf] = __ldg(p.bias2 + i);
    } else {
      sb1[i] = make_float2(__ldg(p.inv1 + i), __ldg(p.bias1 + i));
      sb2[i] = make_float2(__ldg(p.inv2 + i), __ldg(p.bias2 + i));
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (lane == 0) {
      uint32_t iw = 0;
      int x_next = 0;                                         // next tile whose x window has not been requested yet
      // the x window of tile x_next may be loaded as soon as conv1 of tile x_next-1 has read the buffer; that moment falls
      // in the middle of this thread's weight streaming (which is paced by the MMAs), so every wait polls for it
      auto try_x = [&](bool block) {
        if (x_next >= my_tiles) return;
        const uint32_t par = (x_next & 1) ^ 1;
        if (block) mbar_wait(xempty, par);
        else if (!mbar_test_wait(xempty, par)) return;      // a probe, never a sleep: this thread is also feeding the weight ring
        const int tile = (int)blockIdx.x + x_next * (int)gridDim.x;
        const int tt = tile % p.t_tiles, b = tile / p.t_tiles;
        const int r0 = p.row0 + tt * R_OUT - h2 - h1;                 // first row of the x window
        mbar_expect_tx(xfull, Cfg::XWIN);
        for (int cc = 0; cc < NCH; ++cc)
          for (int bx = 0; bx < NBOX; ++bx) {
            tma_load_3d(xwin + (cc * 2 + 0) * Cfg::XPLANE + bx * A_TILE_BYTES, &p.tmX, xfull, cc * BK, r0 + bx * BM, b);
            tma_load_3d(xwin + (cc * 2 + 1) * Cfg::XPLANE + bx * A_TILE_BYTES, &p.tmX, xfull, cc * BK, r0 + bx * BM, p.B + b);
          }
        ++x_next;
      };
      auto weights = [&](const __half* W) {                 // the k * NCH images of one conv, in the MMA thread's order
        for (int img = 0; img < p.k * NCH; ++img, ++iw) {
          const int s = iw % WS;
          while (!mbar_test_wait(&wempty[s], ((iw / WS) & 1) ^ 1)) try_x(false);
          mbar_expect_tx(&wfull[s], Cfg::WIMG);
          bulk_load(wring + s * Cfg::WIMG, W + (size_t)img * (Cfg::WIMG / 2), Cfg::WIMG, &wfull[s]);
        }
      };
      for (int it = 0; it <= my_tiles; ++it) {
        if (it < my_tiles) {
          if (x_next <= it) try_x(true);                      // X(it), unless it went out early
          weights(p.W1);
        }
        if (it > 0) weights(p.W2);
      }
    }
  } else if (warp == 1 || warp == NUM_THREADS / 32) {
    // =========================== MMA issuers ===========================
    // the TMEM base as a warp-uniform value: UTCHMMA takes its operands from uniform registers, and a per-thread register
    // costs an ELECT / R2UR.BROADCAST / branch "waterfall" in front of every MMA
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    constexpr int MS_PER = NSUB / RB_ISSUERS;                  // sub-tiles per issuer
    static_assert(NSUB % RB_ISSUERS == 0, "sub-tiles split evenly over the issuers");
    const int ms0 = (warp == 1 ? 0 : 1) * MS_PER;
    if (lane == 0) {
      constexpr uint32_t idesc_cat = make_idesc(2 * C, BM);     // a_hi x [w_hi | w_lo]
      constexpr uint32_t idesc_one = make_idesc(C, BM);         // a_lo x w_hi
      uint32_t iw = 0;
      // one conv over the NSUB sub-tiles: A planes at a_base (+ cc*2*plane_bytes), tap j starts `tap_rows * j` rows in
      auto conv = [&](uint32_t d_tmem, uint32_t a_base, uint32_t plane_bytes, int tap_rows) {
        uint32_t accumulate = 0;
        for (int tap = 0; tap < p.k; ++tap)
          for (int cc = 0; cc < NCH; ++cc, ++iw) {
            const int s = iw % WS;
            mbar_wait(&wfull[s], (iw / WS) & 1);
            tc_fence_after();
            const uint32_t b_hi = smem_u32(wring + s * Cfg::WIMG);      // [w_hi: C rows][w_lo: C rows], one K-major tile of 2C rows
            const uint32_t a_hi0 = a_base + (uint32_t)(cc * 2) * plane_bytes + (uint32_t)(tap * tap_rows) * ROW_BYTES;
            const uint32_t a_lo0 = a_hi0 + plane_bytes;
            // three descriptors per (tap, chunk); every MMA below adds a compile-time offset: the issuing thread's instruction
            // stream, not the tensor core, bounded these narrow MMAs (tc_conv.cuh: desc_add)
            const uint64_t dah = make_desc(a_hi0 + ms0 * A_TILE_BYTES), dal = make_desc(a_lo0 + ms0 * A_TILE_BYTES), dbh = make_desc(b_hi);
#pragma unroll
            for (int ks = 0; ks < BK / 16; ++ks) {
#pragma unroll
              for (int mi = 0; mi < MS_PER; ++mi) {
                const uint32_t ao = mi * A_TILE_BYTES + ks * 32;
                const uint32_t d = d_tmem + mi * 2 * C;
                umma_f16(d, desc_add(dah, ao), desc_add(dbh, ks * 32), idesc_cat, ks == 0 ? accumulate : 1u);
                umma_f16(d, desc_add(dal, ao), desc_add(dbh, ks * 32), idesc_one, 1);
              }
            }
            accumulate = 1;
            umma_commit(&wempty[s]);
          }
      };
      for (int it = 0; it <= my_tiles; ++it) {
        if (it < my_tiles) {                                   // M1(it): conv1 of tile it
          mbar_wait(a1free, (it & 1) ^ 1);                     // E1(it-1) has drained acc1
          mbar_wait(xfull, it & 1);
          tc_fence_after();
          conv(tmem_u + ms0 * 2 * C, smem_u32(xwin), Cfg::XPLANE, p.dil);
          umma_commit(xempty);
          umma_commit(a1full);
        }
        if (it > 0) {                                          // M2(it-1): conv2 of the previous tile
          const int jt = it - 1;
          mbar_wait(a2free, (jt & 1) ^ 1);                     // E2(jt-1) has drained acc2
          mbar_wait(midfull, jt & 1);
          tc_fence_after();
          conv(tmem_u + ACC + ms0 * 2 * C, smem_u32(mid), Cfg::MPLANE, 1);
          umma_commit(midfree);
          umma_commit(a2full);
        }
      }
    }
  } else {
    // =========================== epilogue (warps 2..17) ===========================
    const int q = warp & 3;                 // TMEM lane quarter
    const int grp = (warp - 2) >> 2;        // 0..3
    const int ms = grp % NSUB;              // 128-row sub-tile
    const int cc = grp / NSUB;              // 32-column chunk
    const int row = q * 32 + lane;          // row inside the sub-tile
    const int m = ms * BM + row;            // row inside the tile's NSUB*128 rows
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    for (int it = 0; it <= my_tiles; ++it) {
      if (it < my_tiles) {
        // ---------------- E1(it): a1 = lrelu(conv1 + b1) -> shared-memory A tiles of conv2 ----------------
        const int tile = (int)blockIdx.x + it * (int)gridDim.x;
        const int tt = tile % p.t_tiles, b = tile / p.t_tiles;
        const int t = p.row0 + tt * R_OUT - h2 + m;                     // time step of this a1 row
        const int len = p.lens ? min(p.lens[b], p.L) : p.L;
        const bool valid = t >= 0 && t < len;                  // outside the utterance a1 is the conv's ZERO padding
        mbar_wait(a1full, it & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ms * 2 * C + cc * 32 + lane_addr;
        uint32_t hi2[16], lo2[16];
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          uint32_t r[16], rb[16];
          tmem_ld16(taddr + ci * 16, r);                       // a_hi*w_hi + a_lo*w_hi
          tmem_ld16(taddr + C + ci * 16, rb);                  // a_hi*w_lo
          tmem_ld_wait();
          if constexpr (PK) {
            const float2 slope2 = make_float2(p.slope, p.slope);
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              const float4 s = reinterpret_cast<const float4*>(sb1)[(cc * 32 + ci * 16 + j) >> 1];
              const float2 v = __ffma2_rn(__fadd2_rn(rb_f2(r[j], r[j + 1]), rb_f2(rb[j], rb[j + 1])), make_float2(s.x, s.y), make_float2(s.z, s.w));
              rb_split2(rb_lrelu2(v, slope2), hi2[ci * 8 + (j >> 1)], lo2[ci * 8 + (j >> 1)]);   // rows outside the utterance: masked at the store
            }
          } else {
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const float2 s0 = sb1[cc * 32 + ci * 16 + j], s1 = sb1[cc * 32 + ci * 16 + j + 1];
            float v0 = fmaf(__uint_as_float(r[j]) + __uint_as_float(rb[j]), s0.x, s0.y);
            float v1 = fmaf(__uint_as_float(r[j + 1]) + __uint_as_float(rb[j + 1]), s1.x, s1.y);
            v0 = v0 < 0.f ? v0 * p.slope : v0;
            v1 = v1 < 0.f ? v1 * p.slope : v1;
            split16x2(valid ? v0 : 0.f, valid ? v1 : 0.f, hi2[ci * 8 + (j >> 1)], lo2[ci * 8 + (j >> 1)]);
          }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(a1free);                    // accumulator drained
        mbar_wait(midfree, (it & 1) ^ 1);                      // conv2 of the previous tile has read the a1 tiles
        // K-major SWIZZLE_64B tile [128 rows][32 ch]: 16-byte piece c16 of row r lives at piece c16 ^ ((r >> 1) & 3)
        uint8_t* mt = mid + (cc * 2) * Cfg::MPLANE + ms * A_TILE_BYTES;
        if (PK && !valid) {                                    // a1 outside the utterance is conv2's zero padding
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16) {
            const uint32_t off = row * 64 + ((c16 ^ ((row >> 1) & 3)) << 4);
            *reinterpret_cast<uint4*>(mt + off) = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(mt + Cfg::MPLANE + off) = make_uint4(0u, 0u, 0u, 0u);
          }
        } else {
#pragma unroll
        for (int c16 = 0; c16 < 4; ++c16) {
          const uint32_t off = row * 64 + ((c16 ^ ((row >> 1) & 3)) << 4);
          *reinterpret_cast<uint4*>(mt + off) = make_uint4(hi2[4 * c16], hi2[4 * c16 + 1], hi2[4 * c16 + 2], hi2[4 * c16 + 3]);
          *reinterpret_cast<uint4*>(mt + Cfg::MPLANE + off) = make_uint4(lo2[4 * c16], lo2[4 * c16 + 1], lo2[4 * c16 + 2], lo2[4 * c16 + 3]);
        }
        }
        fence_proxy_async();                                   // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) mbar_arrive(midfull);
      }
      if (it > 0) {
        // ---------------- E2(it-1): x' = conv2 + b2 + x -> global ----------------
        const int jt = it - 1;
        const int tile = (int)blockIdx.x + jt * (int)gridDim.x;
        const int tt = tile % p.t_tiles, b = tile / p.t_tiles;
        const int t = p.row0 + tt * R_OUT + m;
        const int len = p.lens ? min(p.lens[b], p.L) : p.L;
        const bool o_in = m < R_OUT && t < p.L;                // rows this tile owns
        const bool o_valid = o_in && t < len;
        const size_t rowoff = ((size_t)b * p.L + (o_in ? t : 0)) * C + cc * 32;
        const size_t plane = (size_t)p.B * p.L * C;
        if (o_in) {                                            // residual rows: in L2 since the window load of this tile
          prefetch_l2(p.x16 + rowoff);
          prefetch_l2(p.x16 + plane + rowoff);
        }
        mbar_wait(a2full, jt & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ACC + ms * 2 * C + cc * 32 + lane_addr;
        if (PK && !p.acc32) {
          // packed form of the steps that only hand x' to the next step (two launches in three): no running sum, no select per value
          const float2 inv2 = make_float2(p.inv_slope, p.inv_slope), slope2 = make_float2(p.slope, p.slope);
#pragma unroll
          for (int ci = 0; ci < 2; ++ci) {
            const int c0 = ci * 16;
            uint32_t r[16], rb[16];
            tmem_ld16(taddr + c0, r);
            tmem_ld16(taddr + C + c0, rb);
            uint32_t rh[8], rl[8];
            if (o_in) {
#pragma unroll
              for (int v = 0; v < 2; ++v) {
                const uint4 a = reinterpret_cast<const uint4*>(p.x16 + rowoff + c0)[v];
                const uint4 c = reinterpret_cast<const uint4*>(p.x16 + plane + rowoff + c0)[v];
                rh[4 * v] = a.x; rh[4 * v + 1] = a.y; rh[4 * v + 2] = a.z; rh[4 * v + 3] = a.w;
                rl[4 * v] = c.x; rl[4 * v + 1] = c.y; rl[4 * v + 2] = c.z; rl[4 * v + 3] = c.w;
              }
            } else {
#pragma unroll
              for (int v = 0; v < 8; ++v) rh[v] = rl[v] = 0u;
            }
            tmem_ld_wait();
            if (ci == 1) {                                     // last TMEM read of this warp
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(a2free);
            }
            if (p.out16 && o_in) {
              uint4* oh = reinterpret_cast<uint4*>(p.out16 + rowoff + c0);
              uint4* ol = reinterpret_cast<uint4*>(p.out16 + plane + rowoff + c0);
              if (o_valid) {
                uint32_t h2_[8], l2_[8];
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                  const float4 s = reinterpret_cast<const float4*>(sb2)[(cc * 32 + c0 + j) >> 1];
                  const float2 a = rb_unlrelu2(__fadd2_rn(unpack_h2(rh[j >> 1]), unpack_h2(rl[j >> 1])), inv2);   // stored lrelu(x): invert
                  const float2 w = __fadd2_rn(__ffma2_rn(__fadd2_rn(rb_f2(r[j], r[j + 1]), rb_f2(rb[j], rb[j + 1])), make_float2(s.x, s.y), make_float2(s.z, s.w)), a);
                  rb_split2(rb_lrelu2(w, slope2), h2_[j >> 1], l2_[j >> 1]);
                }
#pragma unroll
                for (int q4 = 0; q4 < 2; ++q4) {
                  oh[q4] = make_uint4(h2_[4 * q4], h2_[4 * q4 + 1], h2_[4 * q4 + 2], h2_[4 * q4 + 3]);
                  ol[q4] = make_uint4(l2_[4 * q4], l2_[4 * q4 + 1], l2_[4 * q4 + 2], l2_[4 * q4 + 3]);
                }
              } else {                                         // rows past the utterance's end are written as zero
                oh[0] = make_uint4(0u, 0u, 0u, 0u); oh[1] = make_uint4(0u, 0u, 0u, 0u);
                ol[0] = make_uint4(0u, 0u, 0u, 0u); ol[1] = make_uint4(0u, 0u, 0u, 0u);
              }
            }
          }
        } else {
        // (de-scale, bias) of channel c in either layout of sb2
        auto sb2s = [&](int c) -> float2 {
          if constexpr (PK) { const float* f = reinterpret_cast<const float*>(sb2) + (c >> 1) * 4 + (c & 1); return make_float2(f[0], f[2]); }
          else return sb2[c];
        };
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const int c0 = ci * 16;
          uint32_t r[16], rb[16];
          tmem_ld16(taddr + c0, r);
          tmem_ld16(taddr + C + c0, rb);
          uint32_t rh[8], rl[8];
          float old[16];
          if (o_in) {
#pragma unroll
            for (int v = 0; v < 2; ++v) {
              const uint4 a = reinterpret_cast<const uint4*>(p.x16 + rowoff + c0)[v];
              const uint4 c = reinterpret_cast<const uint4*>(p.x16 + plane + rowoff + c0)[v];
              rh[4 * v] = a.x; rh[4 * v + 1] = a.y; rh[4 * v + 2] = a.z; rh[4 * v + 3] = a.w;
              rl[4 * v] = c.x; rl[4 * v + 1] = c.y; rl[4 * v + 2] = c.z; rl[4 * v + 3] = c.w;
            }
          } else {
#pragma unroll
            for (int v = 0; v < 8; ++v) rh[v] = rl[v] = 0u;
          }
          if (p.acc32 && p.acc_mode >= TC_ACC_ADD && o_in) {
#pragma unroll
            for (int j = 0; j < 16; ++j) old[j] = __ldcs(p.acc32 + ((size_t)b * C + cc * 32 + c0 + j) * p.L + t);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) old[j] = 0.f;
          }
          tmem_ld_wait();
          if (ci == 1) {                                       // last TMEM read of this warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(a2free);
          }
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const float2 s0 = sb2s(cc * 32 + c0 + j), s1 = sb2s(cc * 32 + c0 + j + 1);
            const float2 ah = unpack_h2(rh[j >> 1]), al = unpack_h2(rl[j >> 1]);
            float a0 = ah.x + al.x, a1 = ah.y + al.y;          // stored lrelu(x): invert
            a0 = a0 < 0.f ? a0 * p.inv_slope : a0;
            a1 = a1 < 0.f ? a1 * p.inv_slope : a1;
            v[j] = o_valid ? fmaf(__uint_as_float(r[j]) + __uint_as_float(rb[j]), s0.x, s0.y) + a0 : 0.f;
            v[j + 1] = o_valid ? fmaf(__uint_as_float(r[j + 1]) + __uint_as_float(rb[j + 1]), s1.x, s1.y) + a1 : 0.f;
          }
          if (p.out16 && o_in) {
            uint32_t h2_[8], l2_[8];
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              const float y0 = v[j] < 0.f ? v[j] * p.slope : v[j], y1 = v[j + 1] < 0.f ? v[j + 1] * p.slope : v[j + 1];
              split16x2(y0, y1, h2_[j >> 1], l2_[j >> 1]);
            }
#pragma unroll
            for (int q4 = 0; q4 < 2; ++q4) {
              reinterpret_cast<uint4*>(p.out16 + rowoff + c0)[q4] = make_uint4(h2_[4 * q4], h2_[4 * q4 + 1], h2_[4 * q4 + 2], h2_[4 * q4 + 3]);
              reinterpret_cast<uint4*>(p.out16 + plane + rowoff + c0)[q4] = make_uint4(l2_[4 * q4], l2_[4 * q4 + 1], l2_[4 * q4 + 2], l2_[4 * q4 + 3]);
            }
          }
          if (p.acc32 && o_in) {
            if (p.acc_mode == TC_ACC_ADD_DIV) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = o_valid ? (old[j] + v[j]) / p.acc_div : 0.f;
              if (p.acc_store) {
#pragma unroll
                for (int j = 0; j < 16; ++j) __stcs(p.acc32 + ((size_t)b * C + cc * 32 + c0 + j) * p.L + t, v[j]);
              }
              if (p.out16b) {
                uint32_t h2_[8], l2_[8];
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                  const float y0 = v[j] < 0.f ? v[j] * p.slope : v[j], y1 = v[j + 1] < 0.f ? v[j + 1] * p.slope : v[j + 1];
                  split16x2(y0, y1, h2_[j >> 1], l2_[j >> 1]);
                }
#pragma unroll
                for (int q4 = 0; q4 < 2; ++q4) {
                  reinterpret_cast<uint4*>(p.out16b + rowoff + c0)[q4] = make_uint4(h2_[4 * q4], h2_[4 * q4 + 1], h2_[4 * q4 + 2], h2_[4 * q4 + 3]);
                  reinterpret_cast<uint4*>(p.out16b + plane + rowoff + c0)[q4] = make_uint4(l2_[4 * q4], l2_[4 * q4 + 1], l2_[4 * q4 + 2], l2_[4 * q4 + 3]);
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) __stcs(p.acc32 + ((size_t)b * C + cc * 32 + c0 + j) * p.L + t, old[j] + v[j]);
            }
          }
        }
        }   // generic (scalar) form
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace tc
}  // namespace cube
