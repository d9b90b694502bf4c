// fp32 SIMT implicit-GEMM convolution kernels (sm_100a).
//
// One tiled kernel covers every dense layer of both vocoders:
//   HiFi-GAN  conv_pre / ResBlock convs (fused leaky-ReLU pre-activation, bias, residual add,
//             3-way ResBlock average) / ConvTranspose1d (phase-decomposed)   hifigan/models.py:35-42,100-114
//   ClariNet  front conv, gated dilated causal conv + conditioning 1x1 (tanh*sigmoid fused),
//             res/skip 1x1 (residual*sqrt(.5) and skip accumulation fused), final 1x1
// Layout: activations [B, C, L] fp32 (time contiguous -> lanes run along time, every global access
// is a coalesced 128 B line); weights repacked on the host to [K][M] (output channel contiguous).
// Tile: CTA = 256 threads, BM x BN outputs; a thread owns TM output channels x TN time steps
// strided by 32 (so dilated taps never cause shared-memory bank conflicts: lanes always read 32
// consecutive floats, weights are warp-broadcast float4 loads).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cube {

enum { PRE_NONE = 0, PRE_LRELU = 1, PRE_RELU = 2 };
enum { EPI_LINEAR = 0, EPI_RESADD = 1, EPI_GATE = 2, EPI_RESSKIP = 3 };
enum { POST_NONE = 0, POST_RELU = 1, POST_TANH = 2 };
enum { ACC_NONE = 0, ACC_SET = 1, ACC_ADD = 2, ACC_ADD_DIV = 3 };

struct Seg {                 // one K-segment of the implicit GEMM: `taps` shifted views of one tensor
  const float* src;          // [B, C, L]
  long long bstride;         // elements between batch items
  const int* lens;           // [B] valid source length (positions >= lens[b] read as 0) or null
  int C, L;                  // channels, row pitch (= allocated length)
  int taps, dil, off0;       // source index of output q, tap j:  q + off0 + j*dil
  int preact;                // PRE_*
  float slope;
  int ci_chunk;              // channels staged per shared-memory pass
};

struct ConvP {
  Seg seg[2];
  int nseg;
  const float* W;            // [nphase][Ktot][Mpad]
  const float* bias;         // [Mpad]
  long long w_phase_stride;
  int M, Mpad;
  int Q;                     // output positions (q) per batch item and phase
  int nphase, ostride;       // t_out = q*ostride + ooff[phase]
  int ooff[8];
  int L_out;                 // output row pitch
  const int* out_lens;       // [B] valid output length (outputs past it are written as 0) or null
  float* out;  long long out_bstride;
  const float* res; long long res_bstride;
  float* acc;  long long acc_bstride;
  int acc_mode; float acc_div;
  int epi, post;
  int Mh; float scale;       // EPI_RESSKIP: rows < Mh -> residual path, rows >= Mh -> skip path
  float* skip; long long skip_bstride; int skip_set;
};

__device__ __forceinline__ float apply_pre(float v, int mode, float slope) {
  if (mode == PRE_LRELU) return v > 0.f ? v : v * slope;
  if (mode == PRE_RELU) return fmaxf(v, 0.f);
  return v;
}

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.f / (1.f + expf(-x)); }

template <int TM, int WM, int TN, int WN>
__global__ void __launch_bounds__(256, (TM >= 16 ? 1 : 2)) conv_tile_kernel(const ConvP p) {
  constexpr int BM = TM * WM, BN = 32 * TN * WN;
  static_assert(WM * WN == 8, "8 warps");
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp % WM, wn = warp / WM;
  const int q0 = blockIdx.x * BN;
  const int m0 = blockIdx.y * BM;
  const int b = blockIdx.z / p.nphase, ph = blockIdx.z - b * p.nphase;
  const float* __restrict__ Wph = p.W + (long long)ph * p.w_phase_stride;

  // accumulators as (even row, odd row) pairs: the inner product runs on packed fma.rn.f32x2
  // (FFMA2) - on sm_100 a 3-register FFMA issues every other cycle per SMSP, FFMA2 restores the
  // full 128 FMA/clk/SM rate.
  float2 acc2[TM / 2][TN];
#pragma unroll
  for (int i = 0; i < TM / 2; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc2[i][j] = make_float2(0.f, 0.f);

  int kbase = 0;
  for (int s = 0; s < p.nseg; ++s) {
    const Seg& sg = p.seg[s];
    const int span = (sg.taps - 1) * sg.dil;
    const bool contig = span <= BN;
    const int XW = contig ? BN + span : sg.taps * BN;
    const int XP = (XW + 3) & ~3;
    const int tapstride = contig ? sg.dil : BN;
    const int cic = sg.ci_chunk;
    float* Xs = smem;
    float* Ws = smem + cic * XP;
    const float* __restrict__ srcb = sg.src + (long long)b * sg.bstride;
    const int slen = sg.lens ? min(sg.lens[b], sg.L) : sg.L;
    const int taps = sg.taps, dil = sg.dil;
    const int pos0 = q0 + sg.off0;
    for (int c0 = 0; c0 < sg.C; c0 += cic) {
      const int cn = min(cic, sg.C - c0);
      __syncthreads();
      // ---- stage the input window (pre-activation applied once, here) ----
      for (int ci = warp; ci < cn; ci += 8) {
        const float* __restrict__ row = srcb + (long long)(c0 + ci) * sg.L;
        float* xs = Xs + ci * XP;
        if (contig) {
          for (int sx = lane; sx < XW; sx += 32) {
            const int pos = pos0 + sx;
            float v = 0.f;
            if (pos >= 0 && pos < slen) v = apply_pre(__ldg(row + pos), sg.preact, sg.slope);
            xs[sx] = v;
          }
        } else {
          for (int sx = lane; sx < XW; sx += 32) {
            const int pos = pos0 + (sx / BN) * dil + (sx % BN);
            float v = 0.f;
            if (pos >= 0 && pos < slen) v = apply_pre(__ldg(row + pos), sg.preact, sg.slope);
            xs[sx] = v;
          }
        }
      }
      // ---- stage the weight slab [cn*taps][BM] ----
      const int nk = cn * taps;
      const float* __restrict__ wsrc = Wph + (long long)(kbase + c0 * taps) * p.Mpad + m0;
      for (int idx = tid; idx < nk * (BM / 4); idx += 256) {
        const int kk = idx / (BM / 4), v4 = idx - kk * (BM / 4);
        const float4 w = __ldg(reinterpret_cast<const float4*>(wsrc + (long long)kk * p.Mpad) + v4);
        reinterpret_cast<float4*>(Ws + kk * BM)[v4] = w;
      }
      __syncthreads();
      // ---- register-tiled FMA ----
      const float* xbase = Xs + wn * (32 * TN) + lane;
      const float* wbase = Ws + wm * TM;
      for (int ci = 0; ci < cn; ++ci) {
        const float* xrow = xbase + ci * XP;
        const float* wrow = wbase + ci * taps * BM;
        for (int t = 0; t < taps; ++t) {
          float2 w2[TM / 2];
          float x[TN];
#pragma unroll
          for (int i = 0; i < TM; i += 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(wrow + t * BM + i);
            w2[i / 2] = make_float2(w4.x, w4.y);
            w2[i / 2 + 1] = make_float2(w4.z, w4.w);
          }
#pragma unroll
          for (int j = 0; j < TN; ++j) x[j] = xrow[t * tapstride + 32 * j];
#pragma unroll
          for (int j = 0; j < TN; ++j) {
            const float2 xx = make_float2(x[j], x[j]);
#pragma unroll
            for (int i = 0; i < TM / 2; ++i) acc2[i][j] = __ffma2_rn(w2[i], xx, acc2[i][j]);
          }
        }
      }
    }
    kbase += sg.C * sg.taps;
  }

  // ---------------------------------- epilogue ----------------------------------
#define ACC(i, j) (((i) & 1) ? acc2[(i) >> 1][j].y : acc2[(i) >> 1][j].x)
  const int olen = p.out_lens ? min(p.out_lens[b], p.L_out) : p.L_out;
  const int ooff = p.ooff[ph];
  const int mbase = m0 + wm * TM;
#pragma unroll
  for (int j = 0; j < TN; ++j) {
    const int q = q0 + wn * (32 * TN) + lane + 32 * j;
    if (q >= p.Q) continue;
    const int t = q * p.ostride + ooff;
    if (t < 0 || t >= p.L_out) continue;
    const bool valid = t < olen;
    if (p.epi == EPI_LINEAR) {
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        const int m = mbase + i;
        if (m >= p.M) break;
        float y = ACC(i, j) + __ldg(p.bias + m);
        if (p.post == POST_RELU) y = fmaxf(y, 0.f);
        else if (p.post == POST_TANH) y = tanhf(y);
        p.out[(long long)b * p.out_bstride + (long long)m * p.L_out + t] = valid ? y : 0.f;
      }
    } else if (p.epi == EPI_RESADD) {
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        const int m = mbase + i;
        if (m >= p.M) break;
        const long long off = (long long)m * p.L_out + t;
        float y = ACC(i, j) + __ldg(p.bias + m) + p.res[(long long)b * p.res_bstride + off];
        if (!valid) y = 0.f;
        if (p.out) p.out[(long long)b * p.out_bstride + off] = y;
        if (p.acc_mode != ACC_NONE) {
          float* a = p.acc + (long long)b * p.acc_bstride + off;
          if (p.acc_mode == ACC_SET) *a = y;
          else if (p.acc_mode == ACC_ADD) *a = *a + y;
          else *a = valid ? (*a + y) / p.acc_div : 0.f;
        }
      }
    } else if (p.epi == EPI_GATE) {
#pragma unroll
      for (int i = 0; i < TM; i += 2) {
        const int m = mbase + i;
        if (m >= p.M) break;
        const float f = acc2[i >> 1][j].x + __ldg(p.bias + m);
        const float g = acc2[i >> 1][j].y + __ldg(p.bias + m + 1);
        const float y = tanhf(f) * sigmoid_acc(g);
        p.out[(long long)b * p.out_bstride + (long long)(m >> 1) * p.L_out + t] = valid ? y : 0.f;
      }
    } else {  // EPI_RESSKIP
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        const int m = mbase + i;
        if (m >= p.M) break;
        const float v = ACC(i, j) + __ldg(p.bias + m);
        if (m < p.Mh) {
          const long long off = (long long)m * p.L_out + t;
          const float y = (p.res[(long long)b * p.res_bstride + off] + v) * p.scale;
          p.out[(long long)b * p.out_bstride + off] = valid ? y : 0.f;
        } else {
          float* sp = p.skip + (long long)b * p.skip_bstride + (long long)(m - p.Mh) * p.L_out + t;
          const float y = p.skip_set ? v : (*sp + v);
          *sp = valid ? y : 0.f;
        }
      }
    }
  }
#undef ACC
}

// ------------------------------------------------------------------------------------------
// Convolutions with 1 or 2 output channels (HiFi-GAN conv_post + tanh, ClariNet final 1x1 +
// IAF affine).  HBM-bound: each input element is read once into shared memory.
// ------------------------------------------------------------------------------------------
enum { SEPI_TANH = 0, SEPI_IAF = 1, SEPI_LINEAR = 2 };

struct SmallP {
  const float* src; long long bstride; int C, L;
  int taps, dil, off0, preact; float slope;
  const float* W;     // [C*taps][MO]
  const float* bias;  // [MO]
  const int* out_lens;
  int L_out;
  float* out; long long out_bstride;     // TANH/LINEAR: [B, MO, L_out]; IAF: z_new [B, 1, L_out]
  int16_t* out_i16;                      // optional fused int16 (TANH only) [B, L_out]
  const float* z; long long z_bstride;   // IAF: z_old
  int ci_chunk;
  int epi;
  int row0, nrows;                       // output steps [row0, row0 + nrows) are computed (nrows = 0: all L_out)
  const int* out_rng;                    // [B][2] device: store only steps [rng[2b], rng[2b+1]) of item b, or null
};

template <int MO, int TPT>  // TPT = time steps per thread
__global__ void __launch_bounds__(256) conv_small_kernel(const SmallP p) {
  constexpr int BN = 256 * TPT;
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x;
  const int q0 = p.row0 + blockIdx.x * BN;
  const int b = blockIdx.y;
  const int span = (p.taps - 1) * p.dil;
  const int XW = BN + span;
  const int XP = XW | 1;
  float* Ws = smem;                            // [C*taps*MO]
  float* Xs = smem + ((p.C * p.taps * MO + 3) & ~3);
  for (int i = tid; i < p.C * p.taps * MO; i += 256) Ws[i] = __ldg(p.W + i);
  const float* __restrict__ srcb = p.src + (long long)b * p.bstride;
  float acc[MO][TPT];
#pragma unroll
  for (int m = 0; m < MO; ++m)
#pragma unroll
    for (int j = 0; j < TPT; ++j) acc[m][j] = 0.f;
  for (int c0 = 0; c0 < p.C; c0 += p.ci_chunk) {
    const int cn = min(p.ci_chunk, p.C - c0);
    __syncthreads();
    // 128-bit loads when the rows allow it (HBM-bound layer: bytes in flight per thread matter): the window
    // start is rounded down to a multiple of 4 samples and each lane moves one aligned float4 per step
    const int wstart = q0 + p.off0;
    const int astart = wstart & ~3;                         // floor to 4 (two's complement: fine for negatives)
    const bool vec_ok = ((p.L & 3) == 0) && ((reinterpret_cast<uintptr_t>(srcb) & 15) == 0);
    for (int ci = tid >> 5; ci < cn; ci += 8) {
      const float* __restrict__ row = srcb + (long long)(c0 + ci) * p.L;
      if (vec_ok) {
        const int nvec = (wstart + XW - astart + 3) >> 2;
        for (int v4 = tid & 31; v4 < nvec; v4 += 32) {
          const int pos = astart + 4 * v4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (pos >= 0 && pos + 3 < p.L) {
            v = __ldg(reinterpret_cast<const float4*>(row + pos));
          } else {
            if (pos >= 0 && pos < p.L) v.x = __ldg(row + pos);
            if (pos + 1 >= 0 && pos + 1 < p.L) v.y = __ldg(row + pos + 1);
            if (pos + 2 >= 0 && pos + 2 < p.L) v.z = __ldg(row + pos + 2);
            if (pos + 3 >= 0 && pos + 3 < p.L) v.w = __ldg(row + pos + 3);
          }
          const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int sx = pos + k - wstart;
            if (sx >= 0 && sx < XW) Xs[ci * XP + sx] = apply_pre(e[k], p.preact, p.slope);
          }
        }
      } else {
        for (int sx = tid & 31; sx < XW; sx += 32) {
          const int pos = wstart + sx;
          float v = 0.f;
          if (pos >= 0 && pos < p.L) v = apply_pre(__ldg(row + pos), p.preact, p.slope);
          Xs[ci * XP + sx] = v;
        }
      }
    }
    __syncthreads();
    for (int ci = 0; ci < cn; ++ci) {
      for (int t = 0; t < p.taps; ++t) {
        float w[MO];
#pragma unroll
        for (int m = 0; m < MO; ++m) w[m] = Ws[((c0 + ci) * p.taps + t) * MO + m];
#pragma unroll
        for (int j = 0; j < TPT; ++j) {
          const float x = Xs[ci * XP + t * p.dil + tid + 256 * j];
#pragma unroll
          for (int m = 0; m < MO; ++m) acc[m][j] = fmaf(w[m], x, acc[m][j]);
        }
      }
    }
  }
  const int olen = p.out_lens ? min(p.out_lens[b], p.L_out) : p.L_out;
#pragma unroll
  for (int j = 0; j < TPT; ++j) {
    const int t = q0 + tid + 256 * j;
    if (t >= p.L_out) continue;
    if (p.out_rng && (t < p.out_rng[2 * b] || t >= p.out_rng[2 * b + 1])) continue;
    if (p.epi == SEPI_IAF) {
      // (mu, logs) at t drive sample t+1:  z'[t+1] = z[t+1]*exp(logs[t]) + mu[t],  z'[0] = 0
      if (MO >= 2) {
        const float mu = acc[0][j] + __ldg(p.bias + 0);
        const float logs = acc[MO - 1][j] + __ldg(p.bias + MO - 1);
        if (t == 0) p.out[(long long)b * p.out_bstride] = 0.f;
        if (t + 1 < p.L_out) {
          const float zo = p.z[(long long)b * p.z_bstride + t + 1];
          p.out[(long long)b * p.out_bstride + t + 1] = (t + 1 < olen) ? zo * expf(logs) + mu : 0.f;
        }
      }
    } else {
#pragma unroll
      for (int m = 0; m < MO; ++m) {
        float y = acc[m][j] + __ldg(p.bias + m);
        if (p.epi == SEPI_TANH) y = tanhf(y);
        if (t >= olen) y = 0.f;
        p.out[(long long)b * p.out_bstride + (long long)m * p.L_out + t] = y;
        if (p.out_i16 && m == 0) p.out_i16[(long long)b * p.L_out + t] = (int16_t)(y * 32767.f);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// UpsampleNet2 layer: ConvTranspose2d(1,1,(3,2s),stride=(1,s),padding=(1,s/2)) + LeakyReLU(0.4)
// over the mel "image" [B, 80, L] -> [B, 80, L*s]   (cube/networks/modules.py:357-375)
// 6 MACs per output: pure bandwidth.
// ------------------------------------------------------------------------------------------
struct Up2dP {
  const float* src; float* out;
  const int* src_lens;   // valid input frames (positions past it read as 0) or null
  int nf, L_in, L_out, s, pad;
  float w[3 * 64];       // [3][2s], s <= 32
  float bias, slope;
  int lens_scale;        // src_lens[b] * lens_scale = valid source length at this layer
};

__global__ void __launch_bounds__(256) upsample2d_kernel(const Up2dP p) {
  // the tap index depends on t mod s, i.e. differs between lanes: a per-lane index into the kernel-parameter
  // (constant) bank is replayed once per distinct address, so the taps go through shared memory first
  __shared__ float sw[3 * 64];
  if (threadIdx.x < 3 * 64) sw[threadIdx.x] = p.w[threadIdx.x];
  __syncthreads();
  const int t = blockIdx.x * 256 + threadIdx.x;
  const int f = blockIdx.y, b = blockIdx.z;
  if (t >= p.L_out) return;
  const int slen = p.src_lens ? min(p.src_lens[b] * p.lens_scale, p.L_in) : p.L_in;
  const int tp = t + p.pad;
  const int s_hi = tp / p.s;
  const int k_hi = tp - s_hi * p.s;
  const float* __restrict__ sb = p.src + ((long long)b * p.nf) * p.L_in;
  float a = p.bias;
#pragma unroll
  for (int kf = 0; kf < 3; ++kf) {
    const int fi = f + 1 - kf;
    if (fi < 0 || fi >= p.nf) continue;
    const float* __restrict__ row = sb + (long long)fi * p.L_in;
    if (s_hi < slen) a = fmaf(sw[kf * 2 * p.s + k_hi], __ldg(row + s_hi), a);
    if (s_hi - 1 >= 0 && s_hi - 1 < slen) a = fmaf(sw[kf * 2 * p.s + k_hi + p.s], __ldg(row + s_hi - 1), a);
  }
  a = a > 0.f ? a : a * p.slope;
  if (t >= slen * p.s) a = 0.f;
  p.out[((long long)b * p.nf + f) * p.L_out + t] = a;
}

// Same layer, four consecutive outputs per thread (s, pad and L_out multiples of 4: the four share their two source
// columns, so 6 loads feed 24 FMAs and one 16-byte store).  Grid: (ceil(L_out/4/256), nf, B).
__global__ void __launch_bounds__(256) upsample2d_x4_kernel(const Up2dP p) {
  __shared__ float sw[3 * 64];
  if (threadIdx.x < 3 * 64) sw[threadIdx.x] = p.w[threadIdx.x];
  __syncthreads();
  const int t = (blockIdx.x * 256 + threadIdx.x) * 4;
  const int f = blockIdx.y, b = blockIdx.z;
  if (t >= p.L_out) return;
  const int slen = p.src_lens ? min(p.src_lens[b] * p.lens_scale, p.L_in) : p.L_in;
  const int tp = t + p.pad;
  const int s_hi = tp / p.s;
  const int k_hi = tp - s_hi * p.s;          // multiple of 4, k_hi + 3 < s
  const float* __restrict__ sb = p.src + ((long long)b * p.nf) * p.L_in;
  float a[4] = {p.bias, p.bias, p.bias, p.bias};
#pragma unroll
  for (int kf = 0; kf < 3; ++kf) {
    const int fi = f + 1 - kf;
    if (fi < 0 || fi >= p.nf) continue;
    const float* __restrict__ row = sb + (long long)fi * p.L_in;
    const float x0 = (s_hi < slen) ? __ldg(row + s_hi) : 0.f;
    const float x1 = (s_hi - 1 >= 0 && s_hi - 1 < slen) ? __ldg(row + s_hi - 1) : 0.f;
    const float4 w0 = *reinterpret_cast<const float4*>(sw + kf * 2 * p.s + k_hi);
    const float4 w1 = *reinterpret_cast<const float4*>(sw + kf * 2 * p.s + k_hi + p.s);
    a[0] = fmaf(w0.x, x0, a[0]); a[1] = fmaf(w0.y, x0, a[1]); a[2] = fmaf(w0.z, x0, a[2]); a[3] = fmaf(w0.w, x0, a[3]);
    a[0] = fmaf(w1.x, x1, a[0]); a[1] = fmaf(w1.y, x1, a[1]); a[2] = fmaf(w1.z, x1, a[2]); a[3] = fmaf(w1.w, x1, a[3]);
  }
  const int tend = slen * p.s;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    a[j] = a[j] > 0.f ? a[j] : a[j] * p.slope;
    if (t + j >= tend) a[j] = 0.f;
  }
  *reinterpret_cast<float4*>(p.out + ((long long)b * p.nf + f) * p.L_out + t) = make_float4(a[0], a[1], a[2], a[3]);
}

}  // namespace cube
