// libcube_vocoder.so - engine + C ABI (include/cube_vocoder.h).
//
// The engine owns: the folded / repacked weights on the device, a grow-only device workspace, and
// the launch plan of one forward pass.  Host code is plain C++; all compute is in the kernels of
// conv_simt.cuh / heads.cuh / tc_conv.cuh.  There is no CPU compute path.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/cube_vocoder.h"
#include "conv_simt.cuh"
#include "heads.cuh"
#include "tc_conv.cuh"
#include "tc_block.cuh"
#include "tc_rbstep.cuh"
#include "wavernn.cuh"
#include "melspec.cuh"

#define CUBE_VERSION "0.1.0"
#ifndef CUBE_FUSED_DEFAULT
#define CUBE_FUSED_DEFAULT true
#endif

namespace cube {

static thread_local char g_err[1024] = "";

static int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}

#define CU_TRY(expr)                                                                       \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

struct HostTensor {
  std::vector<int64_t> shape;
  std::vector<float> data;
  int64_t numel() const { int64_t n = 1; for (auto s : shape) n *= s; return n; }
};

struct DevBuf {
  float* p = nullptr;
  size_t bytes = 0;
};

// One dense layer in kernel form.
struct PackedConv {
  float* W = nullptr;      // device [nphase][Ktot][Mpad]
  float* bias = nullptr;   // device [Mpad]
  int M = 0, Mpad = 0, Ktot = 0, nphase = 1;
};

struct ProfRec { std::string name; cudaEvent_t a, b; };

// One dense layer in tcgen05 form (tc_conv.cuh): swizzled split-fp16 weight images.
struct TcPacked {
  __half* Wimg = nullptr;
  uint8_t* Wimg8 = nullptr;   // CUBE_TC_FP8 variant of the gate images (see pack_tc_q8)
  float* inv_scale = nullptr;
  float* bias = nullptr;
  int N = 0, n_tiles = 0, nchunks_total = 0, nseg = 0;
  int bn = 256, nphase = 1;
  long long w_phase_stride = 0;
  tc::TcSeg seg[2];   // logical segments (a window-mode launch may split them, see launch_tc_t)
};

}  // namespace cube

using namespace cube;

struct cube_voc {
  cube_voc_config cfg;
  int device = 0;
  bool finalized = false;
  std::map<std::string, HostTensor> host_w;
  std::vector<void*> dev_allocs;           // weights
  // workspace (grow-only)
  std::map<std::string, DevBuf> ws;
  int* d_lens = nullptr; size_t lens_cap = 0;
  std::vector<int> h_lens;                  // pageable on purpose: the runtime stages small
                                            // pageable H2D copies before returning, so the vector
                                            // can be rewritten by the next (still queued) forward
  // staging for forward_host
  void* hs_in = nullptr; size_t hs_in_cap = 0;
  float* d_mel = nullptr; size_t d_mel_cap = 0;
  float* d_noise = nullptr; size_t d_noise_cap = 0;
  float* d_wav = nullptr; size_t d_wav_cap = 0;
  int16_t* d_wav16 = nullptr; size_t d_wav16_cap = 0;
  cudaStream_t own_stream = nullptr;
  int64_t launches = 0;
  // CUDA graphs of the host-buffer call (cube_voc_forward_host): one per (B, Fmax, noise?, int16?).  The launch plan
  // depends only on that key (n_frames only changes the masks, uploaded from a pinned buffer the graph's memcpy node
  // reads at replay time); every device buffer the plan touches is owned by the handle, and `alloc_gen` counts their
  // (re)allocations - a graph captured under an older generation is discarded.
  struct GraphEntry { cudaGraphExec_t exec = nullptr; uint64_t gen = 0; int64_t launches = 0; int seen = 0; };
  std::map<std::vector<int64_t>, GraphEntry> graphs;
  uint64_t alloc_gen = 0;
  int* h_lens_pin = nullptr; size_t h_lens_pin_cap = 0;
  bool lens_from_pinned = false;            // set while capturing / replaying a graph
  int sm_count = 148;
  // profiling
  bool profile = false;
  std::vector<ProfRec> prof;
  // HiFi-GAN packed layers
  PackedConv conv_pre, conv_post_w;
  std::vector<PackedConv> ups;
  std::vector<std::vector<PackedConv>> rb_c1, rb_c2;  // [resblock idx][dilation idx]
  TcPacked tc_conv_pre;
  std::vector<TcPacked> tc_ups;
  std::vector<std::vector<TcPacked>> tc_c1, tc_c2;
  // ClariNet packed layers
  struct Flow {
    PackedConv front, final1, final3;
    std::vector<PackedConv> gate, resskip;
    std::vector<TcPacked> tc_gate, tc_resskip;
    TcPacked tc_final1;
    TcPacked tc_front;     // front conv as a [128 x front_kernel] GEMM over the taps-as-channels planes (empty: SIMT front)
    bool has_tc_front = false;
    float* w3 = nullptr;   // final_conv.3: [2][S] weights + [2] bias (fp32), for the fused FINAL epilogue
  };
  std::vector<Flow> flows;
  struct Up2 { float w[192]; float bias; int s; };
  std::vector<Up2> up2;
  // WaveRNN (Path W)
  struct Wrnn {
    PackedConv lowres[3], gx;
    float *w_last = nullptr, *whh1 = nullptr, *bhh1 = nullptr, *wih2 = nullptr, *bih2 = nullptr, *whh2 = nullptr, *bhh2 = nullptr;
    float *wpre = nullptr, *bpre = nullptr, *wout = nullptr, *bout = nullptr;
    int S = 0, ic = 0;
  } wr;
  // UpsampleNet (cube/networks/modules.py:317-343)
  struct UpNet { PackedConv conv[3]; std::vector<PackedConv> up; std::vector<int> J; } upnet;
  // last-forward geometry (for get_cond)
  int last_B = 0; int64_t last_T = 0;
  std::vector<int> h_rng;                   // cube_voc_forward_range: [B][2] sample ranges (pageable, as h_lens)
};

namespace cube {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
static int dev_upload(cube_voc* h, const std::vector<float>& v, float** out) {
  float* d = nullptr;
  CU_TRY(cudaMalloc(&d, std::max<size_t>(v.size(), 1) * sizeof(float)));
  CU_TRY(cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  h->dev_allocs.push_back(d);
  *out = d;
  return 0;
}

static int ws_get(cube_voc* h, const char* name, size_t n_floats, float** out) {
  DevBuf& b = h->ws[name];
  const size_t need = n_floats * sizeof(float);
  if (b.bytes < need) {
    if (b.p) CU_TRY(cudaFree(b.p));
    b.p = nullptr; b.bytes = 0;
    ++h->alloc_gen;
    CU_TRY(cudaMalloc(&b.p, need));
    b.bytes = need;
  }
  *out = b.p;
  return 0;
}

// weight-norm fold: w = g * v / ||v||_2 over every dim but 0  (torch.nn.utils.weight_norm, dim=0;
// hifigan/models.py:118-125).  Norm accumulated in double, result rounded to float.
static int get_weight(cube_voc* h, const std::string& base, HostTensor* out) {
  auto it = h->host_w.find(base + ".weight");
  if (it != h->host_w.end()) { *out = it->second; return 0; }
  auto ig = h->host_w.find(base + ".weight_g"), iv = h->host_w.find(base + ".weight_v");
  if (ig == h->host_w.end() || iv == h->host_w.end()) return fail("missing weight '%s.weight[_g/_v]'", base.c_str());
  const HostTensor& g = ig->second; const HostTensor& v = iv->second;
  const int64_t n0 = v.shape[0], inner = v.numel() / n0;
  if (g.numel() != n0) return fail("weight_g of '%s' has %lld elements, expected %lld", base.c_str(), (long long)g.numel(), (long long)n0);
  out->shape = v.shape;
  out->data.resize(v.data.size());
  for (int64_t i = 0; i < n0; ++i) {
    double ss = 0;
    for (int64_t j = 0; j < inner; ++j) { double x = v.data[i * inner + j]; ss += x * x; }
    const float scale = (float)((double)g.data[i] / sqrt(ss));
    for (int64_t j = 0; j < inner; ++j) out->data[i * inner + j] = v.data[i * inner + j] * scale;
  }
  return 0;
}

static int get_bias(cube_voc* h, const std::string& base, int64_t n, const HostTensor** out) {
  auto it = h->host_w.find(base + ".bias");
  if (it == h->host_w.end()) return fail("missing '%s.bias'", base.c_str());
  if (it->second.numel() != n) return fail("'%s.bias' has %lld elements, expected %lld", base.c_str(), (long long)it->second.numel(), (long long)n);
  *out = &it->second;
  return 0;
}

static int expect_shape(const std::string& name, const HostTensor& t, std::initializer_list<int64_t> s) {
  std::vector<int64_t> e(s);
  if (t.shape != e) {
    std::string got, exp;
    for (auto x : t.shape) got += std::to_string(x) + ",";
    for (auto x : e) exp += std::to_string(x) + ",";
    return fail("weight '%s' has shape [%s], expected [%s]", name.c_str(), got.c_str(), exp.c_str());
  }
  return 0;
}

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Conv1d weight [M][C][K] -> packed [C*K][Mpad]
static int pack_conv1d(cube_voc* h, const std::string& base, int M, int C, int K, PackedConv* pc) {
  HostTensor w; const HostTensor* b;
  if (get_weight(h, base, &w)) return 1;
  if (expect_shape(base, w, {M, C, K})) return 1;
  if (get_bias(h, base, M, &b)) return 1;
  pc->M = M; pc->Mpad = round_up(M, 128); pc->Ktot = C * K; pc->nphase = 1;
  std::vector<float> P((size_t)pc->Ktot * pc->Mpad, 0.f), B(pc->Mpad, 0.f);
  for (int m = 0; m < M; ++m) {
    B[m] = b->data[m];
    for (int c = 0; c < C; ++c)
      for (int k = 0; k < K; ++k) P[(size_t)(c * K + k) * pc->Mpad + m] = w.data[((size_t)m * C + c) * K + k];
  }
  if (dev_upload(h, P, &pc->W)) return 1;
  return dev_upload(h, B, &pc->bias);
}

// ConvTranspose1d weight [C][M][K], stride u -> per output phase r a (J-tap, dilation 1) correlation:
//   out[t = q*u + r - p] = sum_c sum_jj Wr[c*J + jj][m] * x[c][q - (J-1) + jj],  k = r + (J-1-jj)*u
static int pack_convT(cube_voc* h, const std::string& base, int C, int M, int K, int u, PackedConv* pc, int* J_out) {
  HostTensor w; const HostTensor* b;
  if (get_weight(h, base, &w)) return 1;
  if (expect_shape(base, w, {C, M, K})) return 1;
  if (get_bias(h, base, M, &b)) return 1;
  const int J = (K + u - 1) / u;
  pc->M = M; pc->Mpad = round_up(M, 128); pc->Ktot = C * J; pc->nphase = u;
  std::vector<float> P((size_t)u * pc->Ktot * pc->Mpad, 0.f), B(pc->Mpad, 0.f);
  for (int m = 0; m < M; ++m) B[m] = b->data[m];
  for (int r = 0; r < u; ++r)
    for (int c = 0; c < C; ++c)
      for (int jj = 0; jj < J; ++jj) {
        const int k = r + (J - 1 - jj) * u;
        if (k >= K) continue;
        for (int m = 0; m < M; ++m)
          P[((size_t)r * pc->Ktot + (size_t)c * J + jj) * pc->Mpad + m] = w.data[((size_t)c * M + m) * K + k];
      }
  *J_out = J;
  if (dev_upload(h, P, &pc->W)) return 1;
  return dev_upload(h, B, &pc->bias);
}

// Small conv (M <= 2): [M][C][K] -> [C*K][M]
static int pack_small(cube_voc* h, const std::string& base, int M, int C, int K, PackedConv* pc) {
  HostTensor w; const HostTensor* b;
  if (get_weight(h, base, &w)) return 1;
  if (expect_shape(base, w, {M, C, K})) return 1;
  if (get_bias(h, base, M, &b)) return 1;
  pc->M = M; pc->Mpad = M; pc->Ktot = C * K;
  std::vector<float> P((size_t)C * K * M), B(M);
  for (int m = 0; m < M; ++m) {
    B[m] = b->data[m];
    for (int c = 0; c < C; ++c)
      for (int k = 0; k < K; ++k) P[(size_t)(c * K + k) * M + m] = w.data[((size_t)m * C + c) * K + k];
  }
  if (dev_upload(h, P, &pc->W)) return 1;
  return dev_upload(h, B, &pc->bias);
}

// ------------------------------------------------------------------------------------------------
// tcgen05 weight packing: dense [N][nchunks*64] (chunk order = the kernel's K order, zero padded) ->
// per-row power-of-two scaling, fp16 hi/lo split, 128B-swizzled [BN x 64] smem images.
// ------------------------------------------------------------------------------------------------
static int dev_upload_bytes(cube_voc* h, const void* src, size_t bytes, void** out) {
  void* d = nullptr;
  CU_TRY(cudaMalloc(&d, std::max<size_t>(bytes, 16)));
  CU_TRY(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
  h->dev_allocs.push_back(d);
  *out = d;
  return 0;
}

static bool use_win(const cube_voc* h);
static bool use_cg2();
static bool use_wide();

static int pack_tc_multi(cube_voc* h, const std::vector<std::vector<float>>& dense, const std::vector<float>& bias, int N,
                         int nchunks, int bn, TcPacked* out) {
  using namespace tc;
  if (N % bn) return fail("tensor-core path needs N %% %d == 0 (got %d)", bn, N);
  const int Kp = nchunks * BK, nph = (int)dense.size();
  out->N = N; out->bn = bn; out->n_tiles = N / bn; out->nchunks_total = nchunks; out->nphase = nph;
  out->w_phase_stride = (long long)out->n_tiles * nchunks * 2 * bn * BK;
  std::vector<__half> img((size_t)nph * out->w_phase_stride);
  std::vector<float> inv(N);
  for (int n = 0; n < N; ++n) {
    float mx = 0.f;
    for (int ph = 0; ph < nph; ++ph)
      for (int k = 0; k < Kp; ++k) mx = std::max(mx, fabsf(dense[ph][(size_t)n * Kp + k]));
    int e = 0;
    if (mx > 0.f) { int ex; frexpf(mx, &ex); e = 12 - ex; }   // mx*2^e in [2^11, 2^12)
    const float sc = ldexpf(1.f, e);
    inv[n] = ldexpf(1.f, -e);
    const int nt = n / bn, r = n % bn;
    for (int ph = 0; ph < nph; ++ph)
      for (int ch = 0; ch < nchunks; ++ch)
        for (int kk = 0; kk < BK; ++kk) {
          const float w = dense[ph][(size_t)n * Kp + ch * BK + kk] * sc;
          const __half hi = __float2half_rn(w);
          const __half lo = __float2half_rn(w - __half2float(hi));
          const size_t off = (size_t)swz_off(r, kk);
          const size_t base = (size_t)ph * out->w_phase_stride + ((size_t)(nt * nchunks + ch) * 2) * (bn * BK);
          img[base + off] = hi;
          img[base + (size_t)bn * BK + off] = lo;
        }
  }
  void* d;
  if (dev_upload_bytes(h, img.data(), img.size() * sizeof(__half), &d)) return 1;
  out->Wimg = (__half*)d;
  if (dev_upload(h, inv, &out->inv_scale)) return 1;
  return dev_upload(h, bias, &out->bias);
}

// GEMM1's two correction passes of the fused block kernel on 8-bit operands (kind::f8f6f4): default on for the student
// (2.7e-5 max-abs on the shipped weights against the 1e-3 budget, profiles/r1_split_precision_study.md); CUBE_TC_FP8=0
// selects the three-fp16-pass arithmetic (6.9e-6)
static bool use_fp8() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_TC_FP8"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

// Gate images for the 8-bit correction passes (tc_block_kernel<.., Q8>): per (n-tile, K chunk) 32 KB =
//   [w_hi fp16, 256 rows x 64 B, SWIZZLE_64B | e4m3(w_lo), 256 x 32 B, SWIZZLE_32B | e4m3(w_hi / 16), 256 x 32 B, SWIZZLE_32B]
// with the same per-row power-of-two scale as pack_tc_multi (so inv_scale / bias of `out` stay valid).
static int pack_tc_q8(cube_voc* h, const std::vector<float>& dense, int N, int nchunks, TcPacked* out) {
  using namespace tc;
  const int bn = BN, Kp = nchunks * BK;
  if (N % bn || BK != 32) return fail("8-bit gate images need N %% 256 == 0 and 32-channel chunks");
  const size_t chunk_bytes = (size_t)2 * bn * BK * 2;     // 32 KB
  std::vector<uint8_t> img((size_t)(N / bn) * nchunks * chunk_bytes, 0);
  for (int n = 0; n < N; ++n) {
    float mx = 0.f;
    for (int k = 0; k < Kp; ++k) mx = std::max(mx, fabsf(dense[(size_t)n * Kp + k]));
    int e = 0;
    if (mx > 0.f) { int ex; frexpf(mx, &ex); e = 12 - ex; }
    const float sc = ldexpf(1.f, e);
    const int nt = n / bn, r = n % bn;
    for (int ch = 0; ch < nchunks; ++ch) {
      uint8_t* base = img.data() + ((size_t)nt * nchunks + ch) * chunk_bytes;
      __half* hi16 = reinterpret_cast<__half*>(base);
      uint8_t* lo8 = base + (size_t)bn * BK * 2;
      uint8_t* hi8 = lo8 + (size_t)bn * BK;
      for (int kk = 0; kk < BK; ++kk) {
        const float w = dense[(size_t)n * Kp + ch * BK + kk] * sc;
        const __half hi = __float2half_rn(w);
        const float hif = __half2float(hi);
        const float lof = __half2float(__float2half_rn(w - hif));
        hi16[swz_off(r, kk)] = hi;
        lo8[swz32_off(r, kk)] = (uint8_t)__nv_cvt_float_to_fp8(lof, __NV_SATFINITE, __NV_E4M3);
        hi8[swz32_off(r, kk)] = (uint8_t)__nv_cvt_float_to_fp8(hif * 0.0625f, __NV_SATFINITE, __NV_E4M3);
      }
    }
  }
  void* d;
  if (dev_upload_bytes(h, img.data(), img.size(), &d)) return 1;
  out->Wimg8 = (uint8_t*)d;
  return 0;
}

static int pack_tc(cube_voc* h, const std::vector<float>& dense, const std::vector<float>& bias, int N, int nchunks,
                   TcPacked* out) {
  std::vector<std::vector<float>> d1(1, dense);
  return pack_tc_multi(h, d1, bias, N, nchunks, tc::BN, out);
}

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// fp16 planes [2][B][T][C] channels-last -> 3-D tensor map (C, T, 2B), box (64, 128, 1), 128B swizzle,
// out-of-bounds rows/channels read as zero (that IS the conv zero padding).
static int make_tmap_hl16(CUtensorMap* tm, const __half* base, int B, int T, int C, int box_rows = tc::BM) {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    CU_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (!p || q != cudaDriverEntryPointSuccess) return fail("cuTensorMapEncodeTiled not available from the driver");
    fn = (PFN_tmapEncodeTiled)p;
  }
  if (C % 8) return fail("channels-last fp16 tensor needs C %% 8 == 0 (got %d)", C);
  cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)T, (cuuint64_t)(2 * B)};
  cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)T * C * 2};
  cuuint32_t box[3] = {(cuuint32_t)tc::BK, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  tc::BK == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed (%d) for [2*%d][%d][%d]", (int)r, B, T, C);
  return 0;
}

// uint8 planes [2][B][T][C] channels-last -> 3-D tensor map (C, T, 2B), box (32 bytes, 128 rows, 1), 32B swizzle
static int make_tmap_q8(CUtensorMap* tm, const uint8_t* base, int B, int T, int C) {
  CUtensorMap probe;
  if (make_tmap_hl16(&probe, (const __half*)base, B, T, 16)) return 1;     // resolves the driver entry point once
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  CU_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
  PFN_tmapEncodeTiled fn = (PFN_tmapEncodeTiled)p;
  if (C % 16) return fail("8-bit channels-last tensor needs C %% 16 == 0 (got %d)", C);
  cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)T, (cuuint64_t)(2 * B)};
  cuuint64_t strides[2] = {(cuuint64_t)C, (cuuint64_t)T * C};
  cuuint32_t box[3] = {32, (cuuint32_t)tc::BM, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (uint8) failed (%d) for [2*%d][%d][%d]", (int)r, B, T, C);
  return 0;
}

// Conv1d weight [M][C][K] -> tcgen05 images; K order = tap-major, channels padded to BK per tap
static int pack_tc_conv1d(cube_voc* h, const std::string& base, int M, int C, int K, TcPacked* out, int bn_cap = 256) {
  using namespace tc;
  HostTensor w; const HostTensor* b;
  if (get_weight(h, base, &w) || expect_shape(base, w, {M, C, K}) || get_bias(h, base, M, &b)) return 1;
  const int cpt = (C + BK - 1) / BK, Cp = cpt * BK, nch = K * cpt, Kp = nch * BK;
  std::vector<std::vector<float>> D(1, std::vector<float>((size_t)M * Kp, 0.f));
  for (int m = 0; m < M; ++m)
    for (int c = 0; c < C; ++c)
      for (int k = 0; k < K; ++k) D[0][(size_t)m * Kp + (size_t)k * Cp + c] = w.data[((size_t)m * C + c) * K + k];
  if (pack_tc_multi(h, D, b->data, M, nch, std::min(bn_cap, M), out)) return 1;
  out->nseg = 1;
  out->seg[0] = {K, 1, 0, cpt, ((C - (cpt - 1) * BK) + 15) / 16};
  return 0;
}

// ConvTranspose1d weight [C][M][K], stride u: phase r uses taps k = r + (J-1-jj)*u at source row q-(J-1)+jj
static int pack_tc_convT(cube_voc* h, const std::string& base, int C, int M, int K, int u, TcPacked* out) {
  using namespace tc;
  HostTensor w; const HostTensor* b;
  if (get_weight(h, base, &w) || expect_shape(base, w, {C, M, K}) || get_bias(h, base, M, &b)) return 1;
  if (C % BK) return fail("tensor-core transposed conv needs C %% %d == 0", BK);
  const int J = (K + u - 1) / u, cpt = C / BK, nch = J * cpt, Kp = nch * BK;
  std::vector<std::vector<float>> D(u, std::vector<float>((size_t)M * Kp, 0.f));
  for (int r = 0; r < u; ++r)
    for (int jj = 0; jj < J; ++jj) {
      const int k = r + (J - 1 - jj) * u;
      if (k >= K) continue;
      for (int m = 0; m < M; ++m)
        for (int c = 0; c < C; ++c) D[r][(size_t)m * Kp + (size_t)jj * C + c] = w.data[((size_t)c * M + m) * K + k];
    }
  if (pack_tc_multi(h, D, b->data, M, nch, std::min(256, M), out)) return 1;
  out->nseg = 1;
  out->seg[0] = {J, 1, -(J - 1), cpt, BK / 16};
  return 0;
}

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------
struct Launcher {
  cube_voc* h;
  cudaStream_t st;
  int err = 0;
  const char* cur = "";

  void begin(const char* name) {
    cur = name;
    if (h->profile) {
      ProfRec r; r.name = name;
      cudaEventCreate(&r.a); cudaEventCreate(&r.b);
      cudaEventRecord(r.a, st);
      h->prof.push_back(r);
    }
  }
  void end() {
    if (h->profile) cudaEventRecord(h->prof.back().b, st);
  }

  static int pick_chunk(const Seg& s, int BM, int BN, size_t budget) {
    const int span = (s.taps - 1) * s.dil;
    const int XW = span <= BN ? BN + span : s.taps * BN;
    const size_t per = (size_t)(((XW + 3) & ~3) + s.taps * BM) * sizeof(float);
    int c = (int)(budget / per);
    if (c < 1) c = 1;
    if (c > s.C) c = s.C;
    if (c > 32) c = 32;
    return c;
  }
  static size_t smem_of(const Seg& s, int BM, int BN) {
    const int span = (s.taps - 1) * s.dil;
    const int XW = span <= BN ? BN + span : s.taps * BN;
    return (size_t)s.ci_chunk * (((XW + 3) & ~3) + s.taps * BM) * sizeof(float);
  }

  template <int TM, int WM, int TN, int WN>
  void launch_tile(ConvP& p, int B) {
    constexpr int BM = TM * WM, BN = 32 * TN * WN;
    size_t smem = 0;
    for (int s = 0; s < p.nseg; ++s) {
      p.seg[s].ci_chunk = pick_chunk(p.seg[s], BM, BN, 56 * 1024);
      smem = std::max(smem, smem_of(p.seg[s], BM, BN));
    }
    static bool attr_set[64] = {false};
    const int dv = h->device & 63;
    if (!attr_set[dv]) {
      cudaFuncSetAttribute(conv_tile_kernel<TM, WM, TN, WN>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
      attr_set[dv] = true;
    }
    dim3 grid((p.Q + BN - 1) / BN, (p.M + BM - 1) / BM, B * p.nphase);
    conv_tile_kernel<TM, WM, TN, WN><<<grid, 256, smem, st>>>(p);
    check();
  }

  // choose the tile by output-channel count
  void conv(ConvP& p, int B) {
    if (err) return;
    if (p.M <= 32) launch_tile<8, 4, 8, 2>(p, B);       // 32 x 512
    else launch_tile<8, 8, 8, 1>(p, B);                  // 64 x 256
  }

  void small(SmallP& p, int B, int MO) {
    if (err) return;
    constexpr int TPT = 4, BN = 256 * TPT;
    const int span = (p.taps - 1) * p.dil;
    const int XP = (BN + span) | 1;
    int cic = (int)((60 * 1024 - (size_t)(p.C * p.taps * MO + 4) * 4) / ((size_t)XP * 4));
    if (cic > p.C) cic = p.C;
    if (cic < 1) cic = 1;
    p.ci_chunk = cic;
    const size_t smem = ((size_t)((p.C * p.taps * MO + 3) & ~3) + (size_t)cic * XP) * sizeof(float);
    dim3 grid(((p.nrows > 0 ? p.nrows : p.L_out) + BN - 1) / BN, B);
    static bool a1[64] = {false}, a2[64] = {false};
    const int dv = h->device & 63;
    if (MO == 1) {
      if (!a1[dv]) { cudaFuncSetAttribute(conv_small_kernel<1, TPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024); a1[dv] = true; }
      conv_small_kernel<1, TPT><<<grid, 256, smem, st>>>(p);
    } else {
      if (!a2[dv]) { cudaFuncSetAttribute(conv_small_kernel<2, TPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024); a2[dv] = true; }
      conv_small_kernel<2, TPT><<<grid, 256, smem, st>>>(p);
    }
    check();
  }

  void check() {
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess && !err) err = fail("kernel launch failed in '%s': %s", cur, cudaGetErrorString(e));
  }
};

static Seg make_seg(const float* src, long long bstride, int C, int L, int taps, int dil, int off0,
                    int preact, float slope, const int* lens = nullptr) {
  Seg s;
  memset(&s, 0, sizeof(s));
  s.src = src; s.bstride = bstride; s.C = C; s.L = L; s.taps = taps; s.dil = dil; s.off0 = off0;
  s.preact = preact; s.slope = slope; s.lens = lens; s.ci_chunk = 1;
  return s;
}

static ConvP make_conv(const PackedConv& pc) {
  ConvP p;
  memset(&p, 0, sizeof(p));
  p.W = pc.W; p.bias = pc.bias; p.M = pc.M; p.Mpad = pc.Mpad; p.nphase = 1; p.ostride = 1;
  p.w_phase_stride = (long long)pc.Ktot * pc.Mpad;
  p.epi = EPI_LINEAR; p.post = POST_NONE; p.acc_mode = ACC_NONE; p.acc_div = 1.f; p.scale = 1.f;
  return p;
}

// ------------------------------------------------------------------------------------------------
// finalize: strict weight check, fold, repack, upload
// ------------------------------------------------------------------------------------------------
static int finalize_hifigan(cube_voc* h) {
  const cube_voc_config& c = h->cfg;
  const int C0 = c.upsample_initial_channel;
  if (pack_conv1d(h, "conv_pre", C0, c.num_mels, 7, &h->conv_pre)) return 1;
  int ch = C0;
  h->ups.resize(c.n_ups);
  const int nk = c.n_resblock_kernels;
  h->rb_c1.assign(c.n_ups * nk, {});
  h->rb_c2.assign(c.n_ups * nk, {});
  for (int i = 0; i < c.n_ups; ++i) {
    int J;
    if (pack_convT(h, "ups." + std::to_string(i), ch, ch / 2, c.upsample_kernel_sizes[i], c.upsample_rates[i], &h->ups[i], &J)) return 1;
    ch /= 2;
    for (int j = 0; j < nk; ++j) {
      const int idx = i * nk + j, k = c.resblock_kernel_sizes[j], nd = c.n_dilations[j];
      h->rb_c1[idx].resize(nd);
      h->rb_c2[idx].resize(c.resblock_type == 1 ? nd : 0);
      for (int m = 0; m < nd; ++m) {
        const std::string rb = "resblocks." + std::to_string(idx);
        if (c.resblock_type == 1) {
          if (pack_conv1d(h, rb + ".convs1." + std::to_string(m), ch, ch, k, &h->rb_c1[idx][m])) return 1;
          if (pack_conv1d(h, rb + ".convs2." + std::to_string(m), ch, ch, k, &h->rb_c2[idx][m])) return 1;
        } else {
          if (pack_conv1d(h, rb + ".convs." + std::to_string(m), ch, ch, k, &h->rb_c1[idx][m])) return 1;
        }
      }
    }
  }
  if (pack_small(h, "conv_post", 1, ch, 7, &h->conv_post_w)) return 1;
  if (c.math == CUBE_MATH_TC_SPLIT16) {
    if (c.resblock_type != 1) return fail("tensor-core HiFi-GAN path supports resblock '1' only (use CUBE_MATH_FP32_SIMT)");
    auto okc = [](int n) { return n == 32 || n == 64 || n == 128 || n == 256 || n == 512; };
    if (!okc(C0) || (C0 >> c.n_ups) < 32) return fail("tensor-core HiFi-GAN path needs channels in {32..512} (C0=%d)", C0);
    if (c.num_mels % 8) return fail("tensor-core path needs num_mels %% 8 == 0");
    if (pack_tc_conv1d(h, "conv_pre", C0, c.num_mels, 7, &h->tc_conv_pre)) return 1;
    h->tc_ups.resize(c.n_ups);
    h->tc_c1.assign(c.n_ups * nk, {});
    h->tc_c2.assign(c.n_ups * nk, {});
    // The 256-channel stage keeps its 256-column tiles: as two 128-column tiles with two sub-tiles each it measured 25-30 %
    // SLOWER (profiles/r2n_*: 226 / 451 / 663 us against 184 / 347 / 506 for k = 3 / 7 / 11) - its MMAs are already 81 % of the
    // tensor pipe's time; the two-sub-tile variant is for the stage whose natural tile is 128 columns (launch_tc_bn)
    const int rb_bn = 256;
    int cc = C0;
    for (int i = 0; i < c.n_ups; ++i) {
      if (pack_tc_convT(h, "ups." + std::to_string(i), cc, cc / 2, c.upsample_kernel_sizes[i], c.upsample_rates[i], &h->tc_ups[i])) return 1;
      cc /= 2;
      for (int j = 0; j < nk; ++j) {
        const int idx = i * nk + j, k = c.resblock_kernel_sizes[j], nd = c.n_dilations[j];
        h->tc_c1[idx].resize(nd); h->tc_c2[idx].resize(nd);
        for (int m = 0; m < nd; ++m) {
          const std::string rb = "resblocks." + std::to_string(idx);
          if (pack_tc_conv1d(h, rb + ".convs1." + std::to_string(m), cc, cc, k, &h->tc_c1[idx][m], rb_bn)) return 1;
          if (pack_tc_conv1d(h, rb + ".convs2." + std::to_string(m), cc, cc, k, &h->tc_c2[idx][m], rb_bn)) return 1;
        }
      }
    }
  }
  return 0;
}

static int finalize_student(cube_voc* h) {
  const cube_voc_config& c = h->cfg;
  const int R = c.res_channels, G = c.gate_channels, S = c.skip_channels, CI = c.num_mels, K = c.kernel_size;
  if (R != S) return fail("res_channels must equal skip_channels (got %d, %d)", R, S);
  h->flows.resize(c.n_flows);
  for (int f = 0; f < c.n_flows; ++f) {
    cube_voc::Flow& fl = h->flows[f];
    const std::string fp = "iafs." + std::to_string(f) + ".";
    if (pack_conv1d(h, fp + "front_conv.0.conv", R, 1, c.front_kernel, &fl.front)) return 1;
    if (c.math == CUBE_MATH_TC_SPLIT16 && R == 128 && c.front_kernel % tc::BK == 0) {
      // Conv1d(1 -> R, k, causal) == 1x1 conv over k "channels" holding the k causal taps (tc::taps_to_hl16_kernel):
      // weight [R][1][k] read as [R][k]
      HostTensor wf0; const HostTensor* bf0;
      if (get_weight(h, fp + "front_conv.0.conv", &wf0) || expect_shape(fp + "front_conv.0.conv", wf0, {R, 1, c.front_kernel}) ||
          get_bias(h, fp + "front_conv.0.conv", R, &bf0)) return 1;
      const int nchf = c.front_kernel / tc::BK;
      std::vector<std::vector<float>> Df(1, std::vector<float>(wf0.data.begin(), wf0.data.begin() + (size_t)R * c.front_kernel));
      if (pack_tc_multi(h, Df, bf0->data, R, nchf, R, &fl.tc_front)) return 1;
      fl.tc_front.nseg = 1;
      fl.tc_front.seg[0] = {1, 1, 0, nchf, tc::BK / 16};
      fl.has_tc_front = true;
    }
    const int nb = c.flow_blocks[f];
    fl.gate.resize(nb); fl.resskip.resize(nb);
    for (int i = 0; i < nb; ++i) {
      const std::string bp = fp + "res_blocks." + std::to_string(i) + ".";
      HostTensor wf, wg, wfc, wgc, wr, ws;
      const HostTensor *bf, *bg, *bfc, *bgc, *br, *bs;
      if (get_weight(h, bp + "filter_conv.conv", &wf) || expect_shape(bp + "filter_conv.conv", wf, {G, R, K})) return 1;
      if (get_weight(h, bp + "gate_conv.conv", &wg) || expect_shape(bp + "gate_conv.conv", wg, {G, R, K})) return 1;
      if (get_weight(h, bp + "filter_conv_c", &wfc) || expect_shape(bp + "filter_conv_c", wfc, {G, CI, 1})) return 1;
      if (get_weight(h, bp + "gate_conv_c", &wgc) || expect_shape(bp + "gate_conv_c", wgc, {G, CI, 1})) return 1;
      if (get_weight(h, bp + "res_conv", &wr) || expect_shape(bp + "res_conv", wr, {R, G, 1})) return 1;
      if (get_weight(h, bp + "skip_conv", &ws) || expect_shape(bp + "skip_conv", ws, {S, G, 1})) return 1;
      if (get_bias(h, bp + "filter_conv.conv", G, &bf) || get_bias(h, bp + "gate_conv.conv", G, &bg) ||
          get_bias(h, bp + "filter_conv_c", G, &bfc) || get_bias(h, bp + "gate_conv_c", G, &bgc) ||
          get_bias(h, bp + "res_conv", R, &br) || get_bias(h, bp + "skip_conv", S, &bs)) return 1;
      // gate GEMM: rows interleaved (2j = filter j, 2j+1 = gate j); K = [h: c*K + k][cond: c]
      PackedConv& pg = fl.gate[i];
      pg.M = 2 * G; pg.Mpad = round_up(2 * G, 128); pg.Ktot = R * K + CI; pg.nphase = 1;
      std::vector<float> P((size_t)pg.Ktot * pg.Mpad, 0.f), Bv(pg.Mpad, 0.f);
      for (int j = 0; j < G; ++j) {
        Bv[2 * j] = bf->data[j] + bfc->data[j];
        Bv[2 * j + 1] = bg->data[j] + bgc->data[j];
        for (int cc = 0; cc < R; ++cc)
          for (int k = 0; k < K; ++k) {
            P[(size_t)(cc * K + k) * pg.Mpad + 2 * j] = wf.data[((size_t)j * R + cc) * K + k];
            P[(size_t)(cc * K + k) * pg.Mpad + 2 * j + 1] = wg.data[((size_t)j * R + cc) * K + k];
          }
        for (int cc = 0; cc < CI; ++cc) {
          P[(size_t)(R * K + cc) * pg.Mpad + 2 * j] = wfc.data[(size_t)j * CI + cc];
          P[(size_t)(R * K + cc) * pg.Mpad + 2 * j + 1] = wgc.data[(size_t)j * CI + cc];
        }
      }
      if (dev_upload(h, P, &pg.W) || dev_upload(h, Bv, &pg.bias)) return 1;
      // res/skip GEMM: rows [0,R) res_conv, [R,R+S) skip_conv; K = G
      PackedConv& pr = fl.resskip[i];
      pr.M = R + S; pr.Mpad = round_up(R + S, 128); pr.Ktot = G; pr.nphase = 1;
      std::vector<float> P2((size_t)G * pr.Mpad, 0.f), B2(pr.Mpad, 0.f);
      for (int m = 0; m < R; ++m) {
        B2[m] = br->data[m];
        for (int cc = 0; cc < G; ++cc) P2[(size_t)cc * pr.Mpad + m] = wr.data[(size_t)m * G + cc];
      }
      for (int m = 0; m < S; ++m) {
        B2[R + m] = bs->data[m];
        for (int cc = 0; cc < G; ++cc) P2[(size_t)cc * pr.Mpad + R + m] = ws.data[(size_t)m * G + cc];
      }
      if (dev_upload(h, P2, &pr.W) || dev_upload(h, B2, &pr.bias)) return 1;
      if (c.math == CUBE_MATH_TC_SPLIT16) {
        using namespace tc;
        if (R != 128 || S != 128 || G % 128 || K < 1) return fail("tensor-core path supports res=skip=128, gate %% 128 == 0 (got %d,%d,%d)", R, S, G);
        if (fl.tc_gate.empty()) { fl.tc_gate.resize(nb); fl.tc_resskip.resize(nb); }
        // ---- gate: N = 2G in tiles of 256 = [128 filter | 128 gate] of the same 128 channels;
        //      K chunks: taps 0..K-1 of h (R/64 chunks each), then the conditioning (ceil(CI/64) chunks)
        const int hch = R / BK, cch = (CI + BK - 1) / BK;
        const int nch = K * hch + cch, Kp = nch * BK, N = 2 * G;
        std::vector<float> D((size_t)N * Kp, 0.f), Bb(N, 0.f);
        for (int n = 0; n < N; ++n) {
          const int nt = n / BN, r = n % BN;
          const bool is_gate = r >= BN / 2;
          const int j = nt * (BN / 2) + (r % (BN / 2));
          const HostTensor& wk = is_gate ? wg : wf;
          const HostTensor& wc = is_gate ? wgc : wfc;
          Bb[n] = is_gate ? (bg->data[j] + bgc->data[j]) : (bf->data[j] + bfc->data[j]);
          for (int tap = 0; tap < K; ++tap)
            for (int cc = 0; cc < R; ++cc) D[(size_t)n * Kp + (size_t)tap * R + cc] = wk.data[((size_t)j * R + cc) * K + tap];
          for (int cc = 0; cc < CI; ++cc) D[(size_t)n * Kp + (size_t)K * R + cc] = wc.data[(size_t)j * CI + cc];
        }
        TcPacked& tg = fl.tc_gate[i];
        if (pack_tc(h, D, Bb, N, nch, &tg)) return 1;
        tg.nseg = 2;
        tg.seg[0] = {K, 0, 0, hch, BK / 16};
        tg.seg[1] = {1, 1, 0, cch, ((CI - (cch - 1) * BK) + 15) / 16};
        if (use_fp8() && N == 2 * BN && pack_tc_q8(h, D, N, nch, &tg)) return 1;
        // ---- res/skip: N = 256 = [128 res | 128 skip], K = G
        const int och = G / BK;
        std::vector<float> D2((size_t)(R + S) * G, 0.f), Bb2(R + S, 0.f);
        for (int m = 0; m < R; ++m) { Bb2[m] = br->data[m]; for (int cc = 0; cc < G; ++cc) D2[(size_t)m * G + cc] = wr.data[(size_t)m * G + cc]; }
        for (int m = 0; m < S; ++m) { Bb2[R + m] = bs->data[m]; for (int cc = 0; cc < G; ++cc) D2[(size_t)(R + m) * G + cc] = ws.data[(size_t)m * G + cc]; }
        TcPacked& tr = fl.tc_resskip[i];
        if (pack_tc(h, D2, Bb2, R + S, och, &tr)) return 1;
        tr.nseg = 1;
        tr.seg[0] = {1, 1, 0, och, BK / 16};
      }
    }
    if (pack_conv1d(h, fp + "final_conv.1.conv", S, S, 1, &fl.final1)) return 1;
    if (pack_small(h, fp + "final_conv.3.conv", 2, S, 1, &fl.final3)) return 1;
    if (c.math == CUBE_MATH_TC_SPLIT16) {
      using namespace tc;
      HostTensor w1, w3; const HostTensor *b1, *b3;
      if (get_weight(h, fp + "final_conv.1.conv", &w1) || get_bias(h, fp + "final_conv.1.conv", S, &b1)) return 1;
      if (get_weight(h, fp + "final_conv.3.conv", &w3) || get_bias(h, fp + "final_conv.3.conv", 2, &b3)) return 1;
      // final_conv.1 as a [256 x S] GEMM (rows >= S are zero padding of the 256-column tile)
      std::vector<float> D((size_t)BN * S, 0.f), Bb(BN, 0.f);
      for (int m = 0; m < S; ++m) { Bb[m] = b1->data[m]; for (int cc = 0; cc < S; ++cc) D[(size_t)m * S + cc] = w1.data[(size_t)m * S + cc]; }
      if (pack_tc(h, D, Bb, BN, S / BK, &fl.tc_final1)) return 1;
      fl.tc_final1.nseg = 1;
      fl.tc_final1.seg[0] = {1, 1, 0, S / BK, BK / 16};
      std::vector<float> W3(2 * S + 2);
      for (int cc = 0; cc < S; ++cc) { W3[cc] = w3.data[cc]; W3[S + cc] = w3.data[S + cc]; }
      W3[2 * S] = b3->data[0]; W3[2 * S + 1] = b3->data[1];
      if (dev_upload(h, W3, &fl.w3)) return 1;
    }
  }
  // UpsampleNet2 (teacher's upsample_conv.{0,2}): [1,1,3,2s]
  h->up2.resize(c.n_upsample);
  for (int n = 0; n < c.n_upsample; ++n) {
    const int s = c.upsample_scales[n];
    if (s > 32) return fail("upsample scale %d > 32 unsupported", s);
    const std::string base = "upsample_conv." + std::to_string(2 * n);
    HostTensor w; const HostTensor* b;
    if (get_weight(h, base, &w) || expect_shape(base, w, {1, 1, 3, 2 * s})) return 1;
    if (get_bias(h, base, 1, &b)) return 1;
    memset(h->up2[n].w, 0, sizeof(h->up2[n].w));
    for (int i = 0; i < 3 * 2 * s; ++i) h->up2[n].w[i] = w.data[i];
    h->up2[n].bias = b->data[0];
    h->up2[n].s = s;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// forward: HiFi-GAN
// ------------------------------------------------------------------------------------------------
static int64_t hifigan_len(const cube_voc_config& c, int64_t L, int upto) {
  for (int i = 0; i < upto; ++i) {
    const int u = c.upsample_rates[i], k = c.upsample_kernel_sizes[i];
    L = (L - 1) * u - 2 * ((k - u) / 2) + k;
  }
  return L;
}

// ------------------------------------------------------------------------------------------------
// streaming geometry: the rows of every layer that output samples [s0, s1) depend on
// ------------------------------------------------------------------------------------------------
struct RowRange { int64_t a, b; };   // rows [a, b)

struct HifiganPlan {
  RowRange mel, pre, post;                                // mel frames, conv_pre output rows, conv_post samples
  std::vector<RowRange> ups;                              // [stage]: ConvTranspose1d output rows its ResBlocks read
  std::vector<std::vector<std::vector<RowRange>>> step;   // [stage][resblock][m]: output rows of ResBlock step m
};

static inline int64_t fdiv(int64_t a, int64_t b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// ResBlock step m of kernel k: rows of its input that one output row reaches, left and right
static void step_halo(const cube_voc_config& c, int k, int d, int64_t* hl, int64_t* hr) {
  const int64_t l1 = (int64_t)(k * d - d) / 2, r1 = (int64_t)(k - 1) * d - l1;   // conv1 (or ResBlock2's only conv), "same" pad
  const int64_t l2 = (k - 1) / 2, r2 = (k - 1) - l2;                            // ResBlock1's conv2, dilation 1
  *hl = c.resblock_type == 1 ? l1 + l2 : l1;
  *hr = c.resblock_type == 1 ? r1 + r2 : r1;
}

// Per-phase rows q of ups[i] whose outputs t = q*u + r - pad (r < u) meet output rows [a, b)
static RowRange ups_phase_rows(const cube_voc_config& c, int i, RowRange t) {
  const int u = c.upsample_rates[i], pad = (c.upsample_kernel_sizes[i] - u) / 2;
  return {fdiv(t.a + pad, u), fdiv(t.b - 1 + pad, u) + 1};
}

// Walks the generator backward from output samples [s0, s1).  Every level's range is clipped below at 0 (rows before the
// start are the convs' zero padding and depend on nothing) and, if lens is given, above at lens[l] (l = 0: frames,
// l = n_ups: samples).  phase_reads: the ConvTranspose1d input is what the per-phase kernels read (J = ceil(K/u) taps per
// phase; where K % u != 0 the taps past K hold zero weights but their rows are still multiplied), else the rows with a
// non-zero weight: input i reaches outputs i*u - pad + j, j < K.
static void hifigan_plan(const cube_voc_config& c, int64_t s0, int64_t s1, const int64_t* lens, bool phase_reads,
                         HifiganPlan* P) {
  const int nU = c.n_ups, nk = c.n_resblock_kernels;
  auto clip = [&](RowRange r, int l) {
    r.a = std::max<int64_t>(r.a, 0);
    if (lens) r.b = std::min<int64_t>(r.b, lens[l]);
    if (r.b < r.a) r.b = r.a;
    return r;
  };
  P->ups.assign(nU, {0, 0});
  P->step.assign(nU, std::vector<std::vector<RowRange>>(nk));
  RowRange x = clip({s0, s1}, nU);
  P->post = x;
  x = clip({x.a - 3, x.b + 3}, nU);                        // conv_post: k = 7, pad 3
  for (int i = nU - 1; i >= 0; --i) {                      // x = rows of stage i's output (the ResBlock average)
    RowRange un{INT64_MAX, INT64_MIN};
    for (int j = 0; j < nk; ++j) {
      const int k = c.resblock_kernel_sizes[j], nd = c.n_dilations[j];
      P->step[i][j].assign(nd, {0, 0});
      RowRange r = x;                                      // every ResBlock's last step covers the stage output range
      for (int m = nd - 1; m >= 0; --m) {
        P->step[i][j][m] = r;
        int64_t hl, hr;
        step_halo(c, k, c.resblock_dilations[j][m], &hl, &hr);
        r = clip({r.a - hl, r.b + hr}, i + 1);
      }
      un.a = std::min(un.a, r.a); un.b = std::max(un.b, r.b);
    }
    P->ups[i] = un;                                        // the three ResBlocks share the ups output: the widest need
    const int u = c.upsample_rates[i], K = c.upsample_kernel_sizes[i], pad = (K - u) / 2;
    if (phase_reads) {
      const RowRange q = ups_phase_rows(c, i, un);
      const int J = (K + u - 1) / u;
      x = clip({q.a - (J - 1), q.b}, i);
    } else {
      x = clip({fdiv(un.a + pad - K + 1 + u - 1, u), fdiv(un.b - 1 + pad, u) + 1}, i);
    }
  }
  P->pre = x;
  P->mel = clip({x.a - 3, x.b + 3}, 0);                   // conv_pre: k = 7, pad 3
}

// what cube_voc_forward_range asks of the HiFi-GAN forward: samples [s0, s1) of the batch (the union of the items'
// ranges) and the per-item ranges the conv_post stores are masked to
struct RangeReq { int64_t s0, s1; const int* d_rng; };

// valid length of every utterance at every level of the network -> h->h_lens [nlevels][B] (host only)
static int fill_lens(cube_voc* h, const int32_t* n_frames, int B, int64_t Fmax, int nlevels) {
  const size_t need = (size_t)nlevels * B;
  h->h_lens.resize(need);
  for (int b = 0; b < B; ++b) {
    int64_t f = n_frames ? n_frames[b] : Fmax;
    if (f < 0 || f > Fmax) return fail("n_frames[%d]=%lld outside [0, %lld]", b, (long long)f, (long long)Fmax);
    for (int l = 0; l < nlevels; ++l) {
      int64_t L;
      if (h->cfg.arch == CUBE_VOC_HIFIGAN) L = f > 0 ? hifigan_len(h->cfg, f, l) : 0;
      else { L = f; for (int i = 0; i < l; ++i) L *= h->cfg.upsample_scales[i]; }
      h->h_lens[(size_t)l * B + b] = (int)L;
    }
  }
  return 0;
}

static int lens_levels(const cube_voc* h) {
  return h->cfg.arch == CUBE_VOC_HIFIGAN ? h->cfg.n_ups + 1 : h->cfg.n_upsample + 1;
}

// graph path: the masks travel through a pinned host buffer whose address is baked into the graph's memcpy node
static int stage_lens_pinned(cube_voc* h, const int32_t* n_frames, int B, int64_t Fmax) {
  const int nlevels = lens_levels(h);
  if (fill_lens(h, n_frames, B, Fmax, nlevels)) return 1;
  const size_t need = (size_t)nlevels * B;
  if (h->h_lens_pin_cap < need) {
    if (h->h_lens_pin) CU_TRY(cudaFreeHost(h->h_lens_pin));
    h->h_lens_pin = nullptr; h->h_lens_pin_cap = 0;
    ++h->alloc_gen;
    CU_TRY(cudaMallocHost((void**)&h->h_lens_pin, std::max<size_t>(need, 256) * sizeof(int)));
    h->h_lens_pin_cap = std::max<size_t>(need, 256);
  }
  memcpy(h->h_lens_pin, h->h_lens.data(), need * sizeof(int));
  return 0;
}

static int upload_lens(cube_voc* h, const int32_t* n_frames, int B, int64_t Fmax, int nlevels, cudaStream_t st) {
  const size_t need = (size_t)nlevels * B;
  if (h->lens_cap < need) {
    if (h->d_lens) CU_TRY(cudaFree(h->d_lens));
    ++h->alloc_gen;
    CU_TRY(cudaMalloc(&h->d_lens, need * sizeof(int)));
    h->lens_cap = need;
  }
  if (h->lens_from_pinned) {     // graph capture / replay: stage_lens_pinned() has filled the pinned buffer
    CU_TRY(cudaMemcpyAsync(h->d_lens, h->h_lens_pin, need * sizeof(int), cudaMemcpyHostToDevice, st));
    return 0;
  }
  if (fill_lens(h, n_frames, B, Fmax, nlevels)) return 1;
  CU_TRY(cudaMemcpyAsync(h->d_lens, h->h_lens.data(), need * sizeof(int), cudaMemcpyHostToDevice, st));
  return 0;
}

static int forward_hifigan_tc(cube_voc* h, const float* mel, const int32_t* n_frames, float* wav, int16_t* wav16,
                              int B, int64_t Fmax, cudaStream_t st, const RangeReq* rq);

// rq: cube_voc_forward_range.  The fp32 path computes the whole window and only crops and masks conv_post
static int forward_hifigan(cube_voc* h, const float* mel, const int32_t* n_frames, float* wav, int16_t* wav16,
                           int B, int64_t Fmax, cudaStream_t st, const RangeReq* rq = nullptr) {
  const cube_voc_config& c = h->cfg;
  if (c.math == CUBE_MATH_TC_SPLIT16) return forward_hifigan_tc(h, mel, n_frames, wav, wav16, B, Fmax, st, rq);
  const int nU = c.n_ups, nk = c.n_resblock_kernels;
  std::vector<int64_t> L(nU + 1);
  for (int i = 0; i <= nU; ++i) L[i] = hifigan_len(c, Fmax, i);
  if (L[nU] > 0x7fffffffLL / 2) return fail("utterance too long");
  if (upload_lens(h, n_frames, B, Fmax, nU + 1, st)) return 1;
  const int C0 = c.upsample_initial_channel;
  size_t stage_max = (size_t)C0 * L[0];
  for (int i = 0; i < nU; ++i) stage_max = std::max(stage_max, (size_t)(C0 >> (i + 1)) * L[i + 1]);
  float *bufA, *bufB, *bufC, *bufD;
  if (ws_get(h, "hA", stage_max * B, &bufA) || ws_get(h, "hB", stage_max * B, &bufB) ||
      ws_get(h, "hC", stage_max * B, &bufC) || ws_get(h, "hD", stage_max * B, &bufD)) return 1;
  Launcher lx{h, st};
  const float LR = 0.1f;  // hifigan/models.py:8

  // conv_pre: mel [B,80,F] -> D [B,C0,F]   (hifigan/models.py:101)
  {
    lx.begin("conv_pre");
    ConvP p = make_conv(h->conv_pre);
    p.nseg = 1;
    p.seg[0] = make_seg(mel, (long long)c.num_mels * Fmax, c.num_mels, (int)Fmax, 7, 1, -3, PRE_NONE, 0.f, h->d_lens);
    p.Q = (int)L[0]; p.L_out = (int)L[0]; p.out_lens = h->d_lens;
    p.out = bufD; p.out_bstride = (long long)C0 * L[0];
    lx.conv(p, B);
    lx.end();
  }
  int ch = C0;
  float* stage_in = bufD;
  for (int i = 0; i < nU; ++i) {
    const int u = c.upsample_rates[i], K = c.upsample_kernel_sizes[i], pad = (K - u) / 2;
    const int J = (K + u - 1) / u;
    const int Lin = (int)L[i], Lo = (int)L[i + 1];
    const int cho = ch / 2;
    const int* lens_in = h->d_lens + (size_t)i * B;
    const int* lens_out = h->d_lens + (size_t)(i + 1) * B;
    float *xu = bufA, *xt = bufB, *xr = bufC, *xs = bufD;
    {  // x = ups[i](leaky_relu(x, 0.1))   (hifigan/models.py:103-104)
      lx.begin("ups");
      ConvP p = make_conv(h->ups[i]);
      p.nseg = 1;
      p.seg[0] = make_seg(stage_in, (long long)ch * Lin, ch, Lin, J, 1, -(J - 1), PRE_LRELU, LR, lens_in);
      p.nphase = u; p.ostride = u;
      for (int r = 0; r < u; ++r) p.ooff[r] = r - pad;
      p.Q = (Lo - 1 + pad) / u + 1;
      p.L_out = Lo; p.out_lens = lens_out;
      p.out = xu; p.out_bstride = (long long)cho * Lo;
      lx.conv(p, B);
      lx.end();
    }
    ch = cho;
    const long long bs = (long long)ch * Lo;
    for (int j = 0; j < nk; ++j) {
      const int idx = i * nk + j, k = c.resblock_kernel_sizes[j], nd = c.n_dilations[j];
      const int accm = (j == 0) ? ACC_SET : (j == nk - 1 ? ACC_ADD_DIV : ACC_ADD);
      const float* xcur = xu;
      if (c.resblock_type == 1) {
        for (int m = 0; m < nd; ++m) {  // hifigan/models.py:35-42
          const int d = c.resblock_dilations[j][m];
          lx.begin("rb_conv1");
          ConvP p1 = make_conv(h->rb_c1[idx][m]);
          p1.nseg = 1;
          p1.seg[0] = make_seg(xcur, bs, ch, Lo, k, d, -((k * d - d) / 2), PRE_LRELU, LR);
          p1.Q = Lo; p1.L_out = Lo; p1.out_lens = lens_out; p1.out = xt; p1.out_bstride = bs;
          lx.conv(p1, B);
          lx.end();
          lx.begin("rb_conv2");
          ConvP p2 = make_conv(h->rb_c2[idx][m]);
          p2.nseg = 1;
          p2.seg[0] = make_seg(xt, bs, ch, Lo, k, 1, -((k - 1) / 2), PRE_LRELU, LR);
          p2.Q = Lo; p2.L_out = Lo; p2.out_lens = lens_out;
          p2.epi = EPI_RESADD; p2.res = xcur; p2.res_bstride = bs;
          const bool last = (m == nd - 1);
          p2.out = last ? nullptr : xr; p2.out_bstride = bs;
          if (last) { p2.acc = xs; p2.acc_bstride = bs; p2.acc_mode = accm; p2.acc_div = (float)nk; }
          if (last && nk == 1) { p2.acc_mode = ACC_SET; }
          lx.conv(p2, B);
          lx.end();
          xcur = xr;
        }
      } else {  // ResBlock2: x = conv(lrelu(x)) + x   (hifigan/models.py:63-68); ping-pong xt/xr
        float* pp[2] = {xt, xr};
        for (int m = 0; m < nd; ++m) {
          const int d = c.resblock_dilations[j][m];
          lx.begin("rb2_conv");
          ConvP p1 = make_conv(h->rb_c1[idx][m]);
          p1.nseg = 1;
          p1.seg[0] = make_seg(xcur, bs, ch, Lo, k, d, -((k * d - d) / 2), PRE_LRELU, LR);
          p1.Q = Lo; p1.L_out = Lo; p1.out_lens = lens_out;
          p1.epi = EPI_RESADD; p1.res = xcur; p1.res_bstride = bs;
          const bool last = (m == nd - 1);
          p1.out = last ? nullptr : pp[m & 1]; p1.out_bstride = bs;
          if (last) { p1.acc = xs; p1.acc_bstride = bs; p1.acc_mode = (nk == 1) ? ACC_SET : accm; p1.acc_div = (float)nk; }
          lx.conv(p1, B);
          lx.end();
          xcur = pp[m & 1];
        }
      }
    }
    stage_in = xs;
  }
  {  // x = tanh(conv_post(leaky_relu(x)))  - default slope 0.01   (hifigan/models.py:112-114)
    lx.begin("conv_post");
    const int Lo = (int)L[nU];
    SmallP p;
    memset(&p, 0, sizeof(p));
    p.src = stage_in; p.bstride = (long long)ch * Lo; p.C = ch; p.L = Lo;
    p.taps = 7; p.dil = 1; p.off0 = -3; p.preact = PRE_LRELU; p.slope = 0.01f;
    p.W = h->conv_post_w.W; p.bias = h->conv_post_w.bias;
    p.out_lens = h->d_lens + (size_t)nU * B; p.L_out = Lo;
    p.out = wav; p.out_bstride = Lo; p.out_i16 = wav16; p.epi = SEPI_TANH;
    if (rq) { p.row0 = (int)rq->s0; p.nrows = (int)(rq->s1 - rq->s0); p.out_rng = rq->d_rng; }
    lx.small(p, B, 1);
    lx.end();
  }
  return lx.err;
}

// ------------------------------------------------------------------------------------------------
// forward: HiFi-GAN on tensor cores.  Every MMA-input tensor is stored leaky-ReLU'd (slope 0.1) as
// fp16 hi/lo planes, channels-last; the residual stream is recovered from it by the inverse map.
// ------------------------------------------------------------------------------------------------
// window mode (tc_conv.cuh): measured +4 % on the HiFi-GAN generator (its k=7/11 taps re-read the same rows), -12 % on
// the student (3 taps only, and the window ring leaves a shallower weight ring) -> default on for HiFi-GAN only;
// CUBE_TC_WIN=0/1 overrides for experiments
static bool use_win(const cube_voc* h) {
  static int v = -2;
  if (v == -2) { const char* e = getenv("CUBE_TC_WIN"); v = e ? (e[0] == '1' ? 1 : 0) : -1; }
  if (v >= 0) return v == 1;
  return h->cfg.arch == CUBE_VOC_HIFIGAN;
}

// CUBE_BLOCK_STATS=1: run the instrumented fused block kernel and print CTA 0's wait cycles after each forward
static bool block_stats_on() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_BLOCK_STATS"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}
static unsigned long long* block_stats_buf() {
  static unsigned long long* buf = nullptr;
  if (!buf) { cudaMalloc(&buf, 32 * sizeof(unsigned long long)); cudaMemset(buf, 0, 32 * sizeof(unsigned long long)); }
  return buf;
}
static void block_stats_dump(cudaStream_t st) {
  if (!block_stats_on()) return;
  unsigned long long v[32];
  cudaStreamSynchronize(st);
  cudaMemcpy(v, block_stats_buf(), sizeof(v), cudaMemcpyDeviceToHost);
  cudaMemset(block_stats_buf(), 0, sizeof(v));
  static const char* names[27] = {"prod.wait_empty_g1", "prod.wait_empty_g2", "prod.total",
    "mma.wait_accfree_g1a", "mma.wait_accfree_g1b", "mma.wait_full_g1", "mma.wait_accfree_g2", "mma.wait_ofull_kh0", "mma.wait_ofull_kh1",
    "mma.wait_full_g2", "mma.total",
    "epiR.wait_accfull_nt0", "epiR.wait_accfull_nt1", "epiR.wait_ofree_nt0", "epiR.wait_ofree_nt1", "epiR.wait_accfull_rs", "epiR.gate_math",
    "epiR.resskip", "epiR.-",
    "epiS.wait_accfull_nt0", "epiS.wait_accfull_nt1", "epiS.wait_ofree_nt0", "epiS.wait_ofree_nt1", "epiS.wait_accfull_rs", "epiS.gate_math",
    "epiS.resskip", "epiS.-"};
  fprintf(stderr, "[cube block stats] CTA 0, cycles summed over the forward:\n");
  for (int i = 0; i < 27; ++i) fprintf(stderr, "  %-24s %14llu  (%.1f %% of mma.total)\n", names[i], v[i], 100.0 * (double)v[i] / (double)(v[10] ? v[10] : 1));
}

// fused residual-block kernel (tc_block.cuh) for the student: CUBE_TC_FUSED=0/1 overrides the default
static bool use_fused() {
  static int v = -2;
  if (v == -2) { const char* e = getenv("CUBE_TC_FUSED"); v = e ? (e[0] == '1' ? 1 : 0) : -1; }
  return v < 0 ? CUBE_FUSED_DEFAULT : v == 1;
}

// lean issue loops of the tcgen05 kernels (tc_block.cuh, tc_conv.cuh window mode): CUBE_TC_LEAN=0/1 overrides the default
#ifndef CUBE_LEAN_DEFAULT
#define CUBE_LEAN_DEFAULT 1   // B200 suite green with it (profiles/r2p_pytest_lean.log); student -6 % cycles per block launch, HiFi-GAN wide stages -8 %
#endif
static bool use_lean() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_TC_LEAN"); v = e ? (e[0] == '1' ? 1 : 0) : CUBE_LEAN_DEFAULT; }
  return v == 1;
}

static bool use_cg2() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_TC_CG2"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}

// fused ResBlock-step kernel (tc_rbstep.cuh) for the 32- and 64-channel HiFi-GAN stages: CUBE_TC_RBFUSE=0 falls back to
// the conv1 / conv2 pair of tc_conv_kernel launches
static bool use_rbstep() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_TC_RBFUSE"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

// packed-fp32 epilogue of the fused step kernel (tc_rbstep.cuh, PK): CUBE_RB_PK=0/1 overrides the default
#ifndef CUBE_RB_PK_DEFAULT
#define CUBE_RB_PK_DEFAULT 0   // parity green and bit-identical on a B200 (profiles/r2n_*), but no measurable gain (31.5 vs 32.1 ms): opt-in
#endif
static bool use_rb_pk() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_RB_PK"); v = e ? (e[0] == '1' ? 1 : 0) : CUBE_RB_PK_DEFAULT; }
  return v == 1;
}

template <int C, int NSUB, bool PK>
static int launch_rbstep_v(cube_voc* h, tc::RbParams& rp, cudaStream_t st) {
  using Cfg = tc::RbCfg<C, NSUB>;
  static bool attr[64] = {false};
  if (!attr[h->device & 63]) {
    CU_TRY(cudaFuncSetAttribute(tc::tc_rbstep_kernel<C, NSUB, PK>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
    attr[h->device & 63] = true;
  }
  const int r_out = NSUB * tc::BM - (rp.k - 1);
  rp.t_tiles = ((rp.nrows > 0 ? rp.nrows : rp.L) + r_out - 1) / r_out;
  const long long tiles = (long long)rp.t_tiles * rp.B;
  const int grid = (int)std::min<long long>(tiles, h->sm_count);
  tc::tc_rbstep_kernel<C, NSUB, PK><<<grid, tc::RB_THREADS, Cfg::SMEM, st>>>(rp);
  return 0;
}
template <int C, int NSUB>
static int launch_rbstep(cube_voc* h, tc::RbParams& rp, cudaStream_t st) {
  return use_rb_pk() ? launch_rbstep_v<C, NSUB, true>(h, rp, st) : launch_rbstep_v<C, NSUB, false>(h, rp, st);
}

// WIDE variant of the 128-column tile (tc_conv.cuh, Cfg<.., MS>): two 128-row sub-tiles share every staged weight image.
// For HiFi-GAN's 128-channel stage (-10 % per conv, profiles/r2n_*); CUBE_TC_WIDE=0 / 1 / 2 overrides the default
#ifndef CUBE_WIDE_DEFAULT
#define CUBE_WIDE_DEFAULT 1   // B200 parity green (profiles/r2n_pytest_variants.log, r2p_pytest_lean.log); 128-channel stage -10 % per conv
#endif
// 0 = never, 1 = where it pays (wide_pays), 2 = always (the parity suite forces it: its inputs are too small for the heuristic)
static int wide_mode() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_TC_WIDE"); v = e ? (e[0] == '2' ? 2 : (e[0] == '1' ? 1 : 0)) : CUBE_WIDE_DEFAULT; }
  return v;
}
static bool use_wide() { return wide_mode() > 0; }

// tp.T = rows per batch item, of which tp.nrows from tp.row0 are scheduled (0: all); fills t_tiles for the chosen variant
// and launches
template <int TN, int MS = 0>
static void launch_tc_t(cube_voc* h, tc::TcParams& tp, cudaStream_t st) {
  const int nph = tp.nphase > 0 ? tp.nphase : 1;
  const int rows = tp.nrows > 0 ? tp.nrows : tp.T;
  if (MS == 0 && use_cg2()) {
    static bool attr2[64] = {false};
    if (!attr2[h->device & 63]) {
      cudaFuncSetAttribute(tc::tc_conv_kernel<TN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Cfg<TN, true>::SMEM);
      attr2[h->device & 63] = true;
    }
    constexpr int rows2 = 2 * tc::BM * tc::Cfg<TN, true>::MSUB;
    tp.t_tiles = (rows + rows2 - 1) / rows2;
    const long long tiles = (long long)tp.n_tiles * tp.t_tiles * tp.B * nph;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(2 * (unsigned)std::min<long long>(tiles, h->sm_count / 2));
    cfg.blockDim = dim3(tc::NUM_THREADS);
    cfg.dynamicSmemBytes = tc::Cfg<TN, true>::SMEM;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, tc::tc_conv_kernel<TN, true>, tp);
    return;
  }
  constexpr int rows1 = tc::BM * tc::Cfg<TN, false, MS>::MSUB;
  tp.t_tiles = (rows + rows1 - 1) / rows1;
  const long long tiles = (long long)tp.n_tiles * tp.t_tiles * tp.B * nph;
  const int grid = (int)std::min<long long>(tiles, h->sm_count);
  if (use_win(h)) {
    // window mode: one staged A window per channel chunk serves all taps whose span fits one extra box;
    // wider dilations (ClariNet d = 81, 243) become single-tap segments
    tc::TcParams wp = tp;
    wp.nseg = 0;
    wp.lean = use_lean() ? 1 : 0;
    int base = 0;
    bool ok = true;
    for (int s_ = 0; s_ < tp.nseg && ok; ++s_) {
      const tc::TcSeg sg = tp.seg[s_];
      const int span = (sg.taps - 1) * sg.dil;
      if (span <= tc::BM) {
        if (wp.nseg >= tc::MAX_SEG) { ok = false; break; }
        tc::TcSeg n = sg;
        n.src = s_; n.wchunk0 = base; n.nbox = (rows1 + span + tc::BM - 1) / tc::BM;
        wp.seg[wp.nseg++] = n;
      } else {
        for (int j = 0; j < sg.taps; ++j) {
          if (wp.nseg >= tc::MAX_SEG) { ok = false; break; }
          tc::TcSeg n = sg;
          n.taps = 1; n.off0 = sg.off0 + j * sg.dil; n.src = s_; n.wchunk0 = base + j * sg.nchunks; n.nbox = rows1 / tc::BM;
          wp.seg[wp.nseg++] = n;
        }
      }
      base += sg.taps * sg.nchunks;
    }
    if (ok) {
      static bool attrw[64] = {false};
      if (!attrw[h->device & 63]) {
        cudaFuncSetAttribute(tc::tc_conv_kernel<TN, false, true, MS>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::WinCfg<TN, MS>::SMEM);
        attrw[h->device & 63] = true;
      }
      tc::tc_conv_kernel<TN, false, true, MS><<<grid, tc::NUM_THREADS, tc::WinCfg<TN, MS>::SMEM, st>>>(wp);
      return;
    }
  }
  static bool attr[64] = {false};
  if (!attr[h->device & 63]) {
    cudaFuncSetAttribute(tc::tc_conv_kernel<TN, false, false, MS>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Cfg<TN, false, MS>::SMEM);
    attr[h->device & 63] = true;
  }
  tc::tc_conv_kernel<TN, false, false, MS><<<grid, tc::NUM_THREADS, tc::Cfg<TN, false, MS>::SMEM, st>>>(tp);
}

// Two sub-tiles per scheduled tile halve the number of tiles: worth it only while 128-row tiles would fill the SMs more than
// twice over.  Decided from the whole tensor (tp.T), never from a cropped row range: the two-sub-tile variant accumulates
// a_hi*w_hi, a_hi*w_lo and a_lo*w_hi in one accumulator while the 128-column tile sums a_hi*w_lo separately (CAT in
// tc_conv.cuh), so the variants differ in the last bits and cube_voc_forward_range must pick what cube_voc_forward picks.  At batch 1 the 128-channel stage of a 10-s utterance has 108 such tiles for 148 SMs - as 54 double tiles every
// conv of the stage would take twice as long (the latency the `api1` workload measures).
static bool wide_pays(const cube_voc* h, const tc::TcParams& tp) {
  const long long nph = tp.nphase > 0 ? tp.nphase : 1;
  const long long tiles128 = (long long)tp.n_tiles * ((tp.T + tc::BM - 1) / tc::BM) * tp.B * nph;
  return wide_mode() == 2 || tiles128 >= 2LL * h->sm_count;
}

static void launch_tc_bn(cube_voc* h, int bn, tc::TcParams& tp, cudaStream_t st) {
  if (bn == 256) launch_tc_t<256>(h, tp, st);
  else if (bn == 128 && use_wide() && use_win(h) && !use_cg2() && wide_pays(h, tp)) launch_tc_t<128, 2>(h, tp, st);
  else if (bn == 128) launch_tc_t<128>(h, tp, st);
  else if (bn == 64) launch_tc_t<64>(h, tp, st);
  else launch_tc_t<32>(h, tp, st);
}

// rq (cube_voc_forward_range): every launch schedules only the rows its consumers read (hifigan_plan over the buffer
// lengths, never an item's valid length: rows between the two are written as zero and read as the next conv's padding)
static int forward_hifigan_tc(cube_voc* h, const float* mel, const int32_t* n_frames, float* wav, int16_t* wav16,
                              int B, int64_t Fmax, cudaStream_t st, const RangeReq* rq) {
  const cube_voc_config& c = h->cfg;
  const int nU = c.n_ups, nk = c.n_resblock_kernels;
  std::vector<int64_t> L(nU + 1);
  for (int i = 0; i <= nU; ++i) L[i] = hifigan_len(c, Fmax, i);
  if (L[nU] > 0x7fffffffLL / 2) return fail("utterance too long");
  HifiganPlan plan;
  if (rq) hifigan_plan(c, rq->s0, rq->s1, L.data(), true, &plan);
  auto crop = [&](auto& prm, RowRange r) {    // TcParams / RbParams: schedule rows [r.a, r.b) only
    if (!rq) return;
    prm.row0 = (int)r.a; prm.nrows = (int)std::max<int64_t>(r.b - r.a, 1);
  };
  if (upload_lens(h, n_frames, B, Fmax, nU + 1, st)) return 1;
  const int C0 = c.upsample_initial_channel;
  size_t stage_max = (size_t)C0 * L[0];
  for (int i = 0; i < nU; ++i) stage_max = std::max(stage_max, (size_t)(C0 >> (i + 1)) * L[i + 1]);
  float *p0, *p1, *p2, *p3, *xs, *m16;
  // four fp16-plane buffers (2 planes x 2 B = 4 B/element, i.e. one fp32 tensor each) + the fp32 ResBlock sum
  if (ws_get(h, "gP0", stage_max * B, &p0) || ws_get(h, "gP1", stage_max * B, &p1) || ws_get(h, "gP2", stage_max * B, &p2) ||
      ws_get(h, "gP3", stage_max * B, &p3) || ws_get(h, "gXS", stage_max * B, &xs) ||
      ws_get(h, "gMel16", (size_t)B * Fmax * c.num_mels, &m16)) return 1;
  __half *P0 = (__half*)p0, *P1 = (__half*)p1, *P2 = (__half*)p2, *P3 = (__half*)p3, *M16 = (__half*)m16;
  Launcher lx{h, st};
  const float LR = 0.1f;
  // power-of-two scale of the stored activation planes.  Measured (round 1): S=16 changes the waveform error
  // by < 2 % (7.5e-5 vs 7.6e-5 on the trained generator) - the error is set by the 22-bit products, not by
  // subnormal `lo` halves - so planes are stored unscaled, which keeps the full fp16 range (|a| < 65504;
  // the trained generator peaks near 1e3).
  const float PS = 1.f;
  auto base_params = [&](const TcPacked& pk, const __half* A, int La, int Ca, int Q, int Lout, int Cout, const int* lens,
                         tc::TcParams& tp) -> int {
    memset(&tp, 0, sizeof(tp));
    if (make_tmap_hl16(&tp.tmA[0], A, B, La, Ca)) return 1;
    tp.tmA[1] = tp.tmA[0];
    tp.Wimg = pk.Wimg; tp.inv_scale = pk.inv_scale; tp.bias = pk.bias;
    tp.nseg = 1; tp.seg[0] = pk.seg[0]; tp.nchunks_total = pk.nchunks_total;
    tp.B = B; tp.T = Q; tp.n_tiles = pk.n_tiles; tp.t_tiles = (Q + tc::BM - 1) / tc::BM;
    tp.lens = lens; tp.epi = tc::TC_EPI_CONV; tp.outC = Cout; tp.L_out = Lout;
    tp.nphase = pk.nphase; tp.w_phase_stride = pk.w_phase_stride; tp.ostride = 1;
    tp.out_slope = LR; tp.res_inv_slope = 1.f / LR; tp.acc_div = 1.f;
    tp.a_inv_scale = 1.f / PS; tp.plane_scale = PS;
    return 0;
  };
  {  // mel -> fp16 planes (pad frames masked), then conv_pre; its output is stored lrelu'd for ups[0]
    lx.begin("to_hl16");
    const RowRange mr = rq ? plan.mel : RowRange{0, Fmax};
    tc::to_hl16_kernel<<<dim3((int)(mr.b - mr.a + 31) / 32, (c.num_mels + 31) / 32, B), 256, 0, st>>>(mel, M16, B, c.num_mels, (int)Fmax,
                                                                                                     h->d_lens, PS, (int)mr.a);
    lx.check();
    lx.end();
    lx.begin("conv_pre");
    tc::TcParams tp;
    if (base_params(h->tc_conv_pre, M16, (int)L[0], c.num_mels, (int)L[0], (int)L[0], C0, h->d_lens, tp)) return 1;
    tp.seg[0].dil = 1; tp.seg[0].off0 = -3;
    tp.out16 = P0;
    crop(tp, plan.pre);
    launch_tc_bn(h, h->tc_conv_pre.bn, tp, st);
    lx.check();
    lx.end();
  }
  int ch = C0;
  for (int i = 0; i < nU; ++i) {
    const int u = c.upsample_rates[i], K = c.upsample_kernel_sizes[i], pad = (K - u) / 2;
    const int Lin = (int)L[i], Lo = (int)L[i + 1], cho = ch / 2;
    const int* lens_out = h->d_lens + (size_t)(i + 1) * B;
    __half *IN = P0, *U = P1, *T1 = P2, *R = P3, *NX = P0;
    {  // U = lrelu(ups[i](IN))   (IN already holds lrelu(x))
      lx.begin("ups");
      tc::TcParams tp;
      if (base_params(h->tc_ups[i], IN, Lin, ch, (Lo - 1 + pad) / u + 1, Lo, cho, lens_out, tp)) return 1;
      tp.ostride = u;
      for (int r = 0; r < u; ++r) tp.ooff[r] = r - pad;
      tp.out16 = U;
      if (rq) {   // per-phase rows q (output t = q*u + r - pad) of the ResBlocks' widest need
        const RowRange q = ups_phase_rows(c, i, plan.ups[i]);
        crop(tp, RowRange{std::max<int64_t>(q.a, 0), std::min<int64_t>(q.b, tp.T)});
      }
      launch_tc_bn(h, h->tc_ups[i].bn, tp, st);
      lx.check();
      lx.end();
    }
    ch = cho;
    const bool last_stage = (i == nU - 1);
    if (nk == 1) CU_TRY(cudaMemsetAsync(xs, 0, (size_t)B * ch * Lo * sizeof(float), st));   // (0 + v)/1
    for (int j = 0; j < nk; ++j) {
      const int idx = i * nk + j, k = c.resblock_kernel_sizes[j], nd = c.n_dilations[j];
      const int accm = (nk == 1) ? tc::TC_ACC_ADD_DIV : (j == 0 ? tc::TC_ACC_SET : (j == nk - 1 ? tc::TC_ACC_ADD_DIV : tc::TC_ACC_ADD));
      const __half* xcur = U;
      // narrow stages: the whole step (conv1 -> lrelu -> conv2 -> + x) in one launch, a1 never leaves the SM.  The step
      // reads x through halo windows of OTHER tiles, so it cannot run in place: outputs ping-pong between R and T1.
      const bool fuse_rb = use_rbstep() && (ch == 32 || ch == 64) && k >= 1 && k <= 17 && (k & 1);
      for (int m = 0; m < nd && fuse_rb; ++m) {
        const int d = c.resblock_dilations[j][m];
        if (d * (k - 1) > tc::BM) return fail("fused ResBlock step: dilation %d x kernel %d exceeds the staged window", d, k);
        lx.begin("rb_fused");
        tc::RbParams rp;
        memset(&rp, 0, sizeof(rp));
        if (make_tmap_hl16(&rp.tmX, xcur, B, Lo, ch)) return 1;
        const TcPacked &w1 = h->tc_c1[idx][m], &w2 = h->tc_c2[idx][m];
        rp.W1 = w1.Wimg; rp.inv1 = w1.inv_scale; rp.bias1 = w1.bias;
        rp.W2 = w2.Wimg; rp.inv2 = w2.inv_scale; rp.bias2 = w2.bias;
        rp.k = k; rp.dil = d; rp.B = B; rp.L = Lo; rp.lens = lens_out;
        rp.x16 = xcur; rp.slope = LR; rp.inv_slope = 1.f / LR;
        if (rq) crop(rp, plan.step[i][j][m]);
        const bool last = (m == nd - 1);
        __half* outp = (m & 1) ? T1 : R;
        if (!last) {
          rp.out16 = outp;
        } else {
          rp.acc32 = xs; rp.acc_mode = accm; rp.acc_div = (float)nk;
          if (accm == tc::TC_ACC_ADD_DIV) {
            rp.acc_store = last_stage ? 1 : 0;
            rp.out16b = last_stage ? nullptr : NX;
          }
        }
        if (ch == 32) { if (launch_rbstep<32, 4>(h, rp, st)) return 1; }
        else { if (launch_rbstep<64, 2>(h, rp, st)) return 1; }
        lx.check();
        lx.end();
        xcur = outp;
      }
      for (int m = 0; m < nd && !fuse_rb; ++m) {
        const int d = c.resblock_dilations[j][m];
        {
          lx.begin("rb_conv1");
          tc::TcParams tp;
          if (base_params(h->tc_c1[idx][m], xcur, Lo, ch, Lo, Lo, ch, lens_out, tp)) return 1;
          tp.seg[0].dil = d; tp.seg[0].off0 = -((k * d - d) / 2);
          tp.out16 = T1;
          if (rq) {   // conv2's input: the step's rows and conv2's halo
            const RowRange s = plan.step[i][j][m];
            crop(tp, RowRange{std::max<int64_t>(s.a - (k - 1) / 2, 0), std::min<int64_t>(s.b + (k - 1) - (k - 1) / 2, Lo)});
          }
          launch_tc_bn(h, h->tc_c1[idx][m].bn, tp, st);
          lx.check();
          lx.end();
        }
        {
          lx.begin("rb_conv2");
          tc::TcParams tp;
          if (base_params(h->tc_c2[idx][m], T1, Lo, ch, Lo, Lo, ch, lens_out, tp)) return 1;
          tp.seg[0].dil = 1; tp.seg[0].off0 = -((k - 1) / 2);
          tp.res16 = xcur;
          if (rq) crop(tp, plan.step[i][j][m]);
          const bool last = (m == nd - 1);
          if (!last) {
            tp.out16 = R;
          } else {
            tp.acc32 = xs; tp.acc_mode = accm; tp.acc_div = (float)nk;
            if (accm == tc::TC_ACC_ADD_DIV) {
              if (nk == 1) tp.acc_mode = tc::TC_ACC_ADD_DIV;   // (0 + v)/1
              tp.acc_store = last_stage ? 1 : 0;               // conv_post reads the fp32 sum
              tp.out16b = last_stage ? nullptr : NX;           // next ups reads lrelu(x) planes
            }
          }
          launch_tc_bn(h, h->tc_c2[idx][m].bn, tp, st);
          lx.check();
          lx.end();
          xcur = R;
        }
      }
    }
  }
  {  // x = tanh(conv_post(leaky_relu(x)))  - default slope 0.01   (hifigan/models.py:112-114)
    lx.begin("conv_post");
    const int Lo = (int)L[nU];
    SmallP p;
    memset(&p, 0, sizeof(p));
    p.src = xs; p.bstride = (long long)ch * Lo; p.C = ch; p.L = Lo;
    p.taps = 7; p.dil = 1; p.off0 = -3; p.preact = PRE_LRELU; p.slope = 0.01f;
    p.W = h->conv_post_w.W; p.bias = h->conv_post_w.bias;
    p.out_lens = h->d_lens + (size_t)nU * B; p.L_out = Lo;
    p.out = wav; p.out_bstride = Lo; p.out_i16 = wav16; p.epi = SEPI_TANH;
    if (rq) { p.row0 = (int)plan.post.a; p.nrows = (int)(plan.post.b - plan.post.a); p.out_rng = rq->d_rng; }
    lx.small(p, B, 1);
    lx.end();
  }
  return lx.err;
}

// ------------------------------------------------------------------------------------------------
// forward: ClariNet IAF student
// ------------------------------------------------------------------------------------------------
static int dilation_of(const cube_voc_config& c, int i) {
  int d = 1;
  for (int k = 0; k < i % c.dilation_cycle; ++k) d *= c.dilation_base;
  return d;
}

static int forward_student(cube_voc* h, const float* mel, const int32_t* n_frames, const float* noise,
                           float* wav, int16_t* wav16, int B, int64_t Fmax, cudaStream_t st) {
  const cube_voc_config& c = h->cfg;
  if (!noise) return fail("the IAF student needs `noise` (z ~ N(0,1), [B,1,T])");
  int64_t T64 = Fmax;
  for (int n = 0; n < c.n_upsample; ++n) T64 *= c.upsample_scales[n];
  if (T64 > 0x7fffffffLL / 2) return fail("utterance too long");
  const int T = (int)T64;
  const int R = c.res_channels, G = c.gate_channels, S = c.skip_channels, CI = c.num_mels, K = c.kernel_size;
  if (upload_lens(h, n_frames, B, Fmax, c.n_upsample + 1, st)) return 1;
  const int* lens_T = h->d_lens + (size_t)c.n_upsample * B;
  float *cmid, *cmid2 = nullptr, *cup, *hb, *ob, *sk, *y1, *za, *zb;
  // intermediate stages of the upsampler ping-pong between two buffers (a stage never reads and writes the same one)
  if (c.n_upsample > 2 && ws_get(h, "c_mid2", (size_t)B * CI * (T / c.upsample_scales[c.n_upsample - 1] + 1), &cmid2)) return 1;
  if (ws_get(h, "c_up", (size_t)B * CI * T, &cup) || ws_get(h, "c_mid", (size_t)B * CI * (T / c.upsample_scales[c.n_upsample - 1] + 1), &cmid) ||
      ws_get(h, "h", c.math == CUBE_MATH_TC_SPLIT16 ? 16 : (size_t)B * R * T, &hb) ||
      ws_get(h, "o", c.math == CUBE_MATH_TC_SPLIT16 ? 16 : (size_t)B * G * T, &ob) ||
      ws_get(h, "skip", (size_t)B * S * T, &sk) || ws_get(h, "y1", (size_t)B * S * T, &y1) ||
      ws_get(h, "za", (size_t)B * T, &za) || ws_get(h, "zb", (size_t)B * T, &zb)) return 1;
  Launcher lx{h, st};
  // ---- conditioning: UpsampleNet2 (cube/networks/modules.py:357-375) ----
  {
    const float* src = mel;
    int Lin = (int)Fmax, scale = 1;
    for (int n = 0; n < c.n_upsample; ++n) {
      lx.begin("upsample2d");
      Up2dP p;
      memset(&p, 0, sizeof(p));
      const int s = h->up2[n].s;
      p.src = src; p.out = (n == c.n_upsample - 1) ? cup : ((n & 1) ? cmid2 : cmid);
      p.src_lens = h->d_lens; p.lens_scale = scale;
      p.nf = CI; p.L_in = Lin; p.L_out = Lin * s; p.s = s; p.pad = s / 2;
      memcpy(p.w, h->up2[n].w, sizeof(p.w));
      p.bias = h->up2[n].bias; p.slope = 0.4f;
      if (s % 4 == 0 && p.pad % 4 == 0 && p.L_out % 4 == 0 && ((uintptr_t)p.out & 15) == 0) {
        dim3 grid((p.L_out / 4 + 255) / 256, CI, B);
        upsample2d_x4_kernel<<<grid, 256, 0, st>>>(p);
      } else {
        dim3 grid((p.L_out + 255) / 256, CI, B);
        upsample2d_kernel<<<grid, 256, 0, st>>>(p);
      }
      lx.check();
      lx.end();
      src = p.out; Lin = p.L_out; scale *= s;
    }
    if (c.n_upsample == 0) return fail("n_upsample must be >= 1");
  }
  h->last_B = B; h->last_T = T;
  const float* zin = noise;
  const float rs = sqrtf(0.5f);
  const bool use_tc = (c.math == CUBE_MATH_TC_SPLIT16);
  __half *h16 = nullptr, *h16b = nullptr, *o16 = nullptr, *c16 = nullptr, *s16 = nullptr, *zc16 = nullptr;
  uint8_t *h8 = nullptr, *h8b = nullptr, *c8 = nullptr;     // CUBE_TC_FP8: 8-bit planes of h (ping-pong) and c
  CUtensorMap tm_h, tm_hb, tm_o, tm_c, tm_s, tm_h32, tm_hb32, tm_z, tm_h8, tm_h8b, tm_c8;
  const bool fp8 = use_tc && use_fused() && use_fp8();
  if (use_tc) {
    float *t1, *t2, *t3, *t4;
    if (ws_get(h, "s16", (size_t)B * T * S, &t4)) return 1;
    s16 = (__half*)t4;
    if (make_tmap_hl16(&tm_s, s16, B, T, S)) return 1;
    if (use_fused()) {   // the fused block kernel ping-pongs the residual stream between two buffers
      float* t5;
      if (ws_get(h, "h16b", (size_t)B * T * R, &t5)) return 1;
      h16b = (__half*)t5;
      if (make_tmap_hl16(&tm_hb, h16b, B, T, R) || make_tmap_hl16(&tm_hb32, h16b, B, T, R, 32)) return 1;
    }
    // fp16 (hi, lo) planes, channels-last: 2*2 bytes per element = the footprint of one fp32 tensor
    if (ws_get(h, "h16", (size_t)B * T * R, &t1) || ws_get(h, "o16", (size_t)B * T * G, &t2) ||
        ws_get(h, "c16", (size_t)B * T * CI, &t3)) return 1;
    h16 = (__half*)t1; o16 = (__half*)t2; c16 = (__half*)t3;
    if (make_tmap_hl16(&tm_h, h16, B, T, R) || make_tmap_hl16(&tm_o, o16, B, T, G) || make_tmap_hl16(&tm_c, c16, B, T, CI)) return 1;
    if (use_fused() && make_tmap_hl16(&tm_h32, h16, B, T, R, 32)) return 1;
    if (c.front_kernel % tc::BK == 0) {   // taps-as-channels planes of z for the tensor-core front conv
      float* t6;
      if (ws_get(h, "zc16", (size_t)B * T * c.front_kernel, &t6)) return 1;
      zc16 = (__half*)t6;
      if (make_tmap_hl16(&tm_z, zc16, B, T, c.front_kernel)) return 1;
    }
    lx.begin("to_hl16");
    tc::to_hl16_kernel<<<dim3((T + 31) / 32, (CI + 31) / 32, B), 256, 0, st>>>(cup, c16, B, CI, T);
    lx.check();
    lx.end();
    if (fp8) {
      float *u1, *u2, *u3;
      if (ws_get(h, "h8", (size_t)B * T * R / 2, &u1) || ws_get(h, "h8b", (size_t)B * T * R / 2, &u2) ||
          ws_get(h, "c8", (size_t)B * T * CI / 2, &u3)) return 1;
      h8 = (uint8_t*)u1; h8b = (uint8_t*)u2; c8 = (uint8_t*)u3;
      if (make_tmap_q8(&tm_h8, h8, B, T, R) || make_tmap_q8(&tm_h8b, h8b, B, T, R) || make_tmap_q8(&tm_c8, c8, B, T, CI)) return 1;
      lx.begin("to_q8");
      tc::hl16_to_q8_kernel<<<h->sm_count * 8, 256, 0, st>>>(c16, c8, (long long)B * T * CI);
      lx.check();
      lx.end();
    }
  }
  auto launch_tc = [&](const TcPacked& pk, tc::TcParams& tp) {
    tp.Wimg = pk.Wimg; tp.inv_scale = pk.inv_scale; tp.bias = pk.bias;
    tp.nseg = pk.nseg; tp.nchunks_total = pk.nchunks_total;
    tp.B = B; tp.T = T; tp.n_tiles = pk.n_tiles;
    tp.lens = lens_T;
    tp.nphase = 1; tp.a_inv_scale = 1.f; tp.plane_scale = 1.f;
    launch_tc_t<256>(h, tp, st);
    lx.check();
  };
  for (int f = 0; f < c.n_flows; ++f) {
    cube_voc::Flow& fl = h->flows[f];
    const bool last_flow = (f == c.n_flows - 1);
    float* zout = last_flow ? wav : ((f & 1) ? zb : za);
    if (use_tc && fl.has_tc_front) {
      // h = relu(front_conv(z)) on the tensor cores: the k causal taps of z become k channels (fp16 planes), the conv a
      // [T x k] x [k x 128] GEMM whose epilogue (bias, ReLU = leaky-ReLU with slope 0) writes the residual-stream planes
      // directly - no fp32 [B][128][T] round trip and no transpose pass
      lx.begin("front_tc");
      tc::taps_to_hl16_kernel<<<h->sm_count * 8, 256, 0, st>>>(zin, zc16, B, T, c.front_kernel);
      lx.check();
      tc::TcParams tp;
      memset(&tp, 0, sizeof(tp));
      tp.tmA[0] = tm_z; tp.tmA[1] = tm_z;
      tp.Wimg = fl.tc_front.Wimg; tp.inv_scale = fl.tc_front.inv_scale; tp.bias = fl.tc_front.bias;
      tp.nseg = 1; tp.seg[0] = fl.tc_front.seg[0]; tp.nchunks_total = fl.tc_front.nchunks_total;
      tp.B = B; tp.T = T; tp.n_tiles = fl.tc_front.n_tiles;
      tp.lens = lens_T; tp.epi = tc::TC_EPI_CONV; tp.out16 = h16; tp.outC = R; tp.L_out = T;
      tp.nphase = 1; tp.ostride = 1; tp.out_slope = 0.f; tp.res_inv_slope = 1.f; tp.acc_div = 1.f;
      tp.a_inv_scale = 1.f; tp.plane_scale = 1.f;
      launch_tc_t<128>(h, tp, st);
      lx.check();
      lx.end();
      if (fp8) {
        lx.begin("to_q8");
        tc::hl16_to_q8_kernel<<<h->sm_count * 8, 256, 0, st>>>(h16, h8, (long long)B * T * R);
        lx.check();
        lx.end();
      }
    } else {  // h = relu(front_conv(z)) : causal k=32
      lx.begin("front");
      ConvP p = make_conv(fl.front);
      p.nseg = 1;
      p.seg[0] = make_seg(zin, T, 1, T, c.front_kernel, 1, -(c.front_kernel - 1), PRE_NONE, 0.f, lens_T);
      p.Q = T; p.L_out = T; p.out_lens = lens_T; p.post = POST_RELU;
      p.out = use_tc ? y1 : hb; p.out_bstride = (long long)R * T;
      lx.conv(p, B);
      lx.end();
      if (use_tc) {
        lx.begin("to_hl16");
        tc::to_hl16_kernel<<<dim3((T + 31) / 32, (R + 31) / 32, B), 256, 0, st>>>(y1, h16, B, R, T);
        lx.check();
        lx.end();
      }
    }
    const int nb = c.flow_blocks[f];
    for (int i = 0; i < nb; ++i) {
      const int d = dilation_of(c, i);
      if (use_tc && use_fused() && K * (R / tc::BK) + (CI + tc::BK - 1) / tc::BK == fl.tc_gate[i].nchunks_total && G == 256 && T % 4 == 0) {
        // whole residual block in one kernel: o stays on chip (tc_block.cuh)
        lx.begin("block_fused");
        tc::BlockParams bp;
        memset(&bp, 0, sizeof(bp));
        bp.tmH = tm_h; bp.tmC = tm_c;
        bp.tmHin32 = tm_h32; bp.tmHout32 = tm_hb32;
        bp.h_in16 = h16; bp.h_out16 = h16b;
        bp.W1 = fl.tc_gate[i].Wimg; bp.inv1 = fl.tc_gate[i].inv_scale; bp.bias1 = fl.tc_gate[i].bias;
        bp.W2 = fl.tc_resskip[i].Wimg; bp.inv2 = fl.tc_resskip[i].inv_scale; bp.bias2 = fl.tc_resskip[i].bias;
        bp.taps = K; bp.dil = d; bp.off0 = -(K - 1) * d;
        bp.h_chunks = R / tc::BK; bp.c_chunks = (CI + tc::BK - 1) / tc::BK;
        bp.c_last_ksteps = ((CI - (bp.c_chunks - 1) * tc::BK) + 15) / 16;
        bp.B = B; bp.T = T; bp.t_tiles = (T + tc::BM - 1) / tc::BM;
        bp.lens = lens_T; bp.skip = sk; bp.skip_set = (i == 0); bp.scale = rs;
        bp.skip16 = (i == nb - 1) ? s16 : nullptr;
        const bool q8 = fp8 && fl.has_tc_front && fl.tc_gate[i].Wimg8;
        if (q8) { bp.tmH8 = tm_h8; bp.tmC8 = tm_c8; bp.W1q = fl.tc_gate[i].Wimg8; bp.h8_out = h8b; bp.h8_in = h8; bp.c8_in = c8; }
        static int pfn = -1;        // L2 prefetch of the next tile's A rows by the epilogue warps; CUBE_TC_PREFETCH=0/1
        if (pfn < 0) { const char* e = getenv("CUBE_TC_PREFETCH"); pfn = (e && e[0] == '1') ? 1 : 0; }
        bp.prefetch_next = pfn; bp.c_in16 = c16; bp.c_ch = CI;
        bp.lean = use_lean() ? 1 : 0;
        static int pairv = -1;      // CTA-pair (cta_group::2) tiling of the block kernel; CUBE_TC_PAIR=0: one CTA per tile
        if (pairv < 0) { const char* e = getenv("CUBE_TC_PAIR"); pairv = (e && e[0] == '0') ? 0 : 1; }
        const bool stats = block_stats_on();                             // instrumented build: wait cycles of CTA 0
        if (stats) bp.stats = block_stats_buf();
        // the PAIR x Q8 x STATS instantiations of the one kernel template
        static int aonce = -1;      // pair tiling with the A chunk staged once for both n-tiles (tc_block.cuh, AONCE); CUBE_TC_AONCE=0/1
        if (aonce < 0) { const char* e = getenv("CUBE_TC_AONCE"); aonce = (e && e[0] == '1') ? 1 : 0; }
        const bool use_aonce = pairv == 1 && aonce == 1 && !stats;
        auto launch = [&](auto kernel, bool pair) -> int {
          const size_t smem = use_aonce ? tc::AONCE_SMEM : (pair ? tc::PAIR_SMEM : tc::BLK_SMEM);
          static std::map<std::pair<const void*, int>, bool> attr_done;
          const auto key = std::make_pair((const void*)kernel, h->device);
          if (!attr_done[key]) {
            CU_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_done[key] = true;
          }
          cudaLaunchConfig_t cfg;
          memset(&cfg, 0, sizeof(cfg));
          cudaLaunchAttribute at[1];
          if (pair) {
            bp.t_tiles = (T + 2 * tc::BM - 1) / (2 * tc::BM);           // a pair's tile is 256 rows
            const long long ptiles = (long long)bp.t_tiles * B;
            cfg.gridDim = dim3(2 * (unsigned)std::min<long long>(ptiles, h->sm_count / 2));
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
          } else {
            const long long tiles = (long long)bp.t_tiles * B;
            cfg.gridDim = dim3((unsigned)std::min<long long>(tiles, h->sm_count));
          }
          cfg.blockDim = dim3(tc::NUM_THREADS);
          cfg.dynamicSmemBytes = smem;
          cfg.stream = st;
          CU_TRY(cudaLaunchKernelEx(&cfg, kernel, bp));
          return 0;
        };
        int lrc;
        if (use_aonce) {
          lrc = q8 ? launch(tc::tc_block_kernel<true, true, false, true>, true) : launch(tc::tc_block_kernel<true, false, false, true>, true);
        } else if (pairv == 1) {
          if (stats) lrc = q8 ? launch(tc::tc_block_kernel<true, true, true>, true) : launch(tc::tc_block_kernel<true, false, true>, true);
          else lrc = q8 ? launch(tc::tc_block_kernel<true, true, false>, true) : launch(tc::tc_block_kernel<true, false, false>, true);
        } else {
          if (stats) lrc = q8 ? launch(tc::tc_block_kernel<false, true, true>, false) : launch(tc::tc_block_kernel<false, false, true>, false);
          else lrc = q8 ? launch(tc::tc_block_kernel<false, true, false>, false) : launch(tc::tc_block_kernel<false, false, false>, false);
        }
        if (lrc) return 1;
        lx.check();
        lx.end();
        std::swap(h16, h16b);          // the block's output is the next block's input
        std::swap(tm_h, tm_hb);
        std::swap(tm_h32, tm_hb32);
        if (fp8) { std::swap(h8, h8b); std::swap(tm_h8, tm_h8b); }
        continue;
      }
      if (use_tc) {
        {  // o = tanh(filter(h) + filter_c(c)) * sigmoid(gate(h) + gate_c(c))   [tcgen05]
          lx.begin("gate");
          tc::TcParams tp;
          memset(&tp, 0, sizeof(tp));
          tp.tmA[0] = tm_h; tp.tmA[1] = tm_c;
          tp.seg[0] = fl.tc_gate[i].seg[0]; tp.seg[1] = fl.tc_gate[i].seg[1];
          tp.seg[0].dil = d; tp.seg[0].off0 = -(K - 1) * d;
          tp.epi = tc::TC_EPI_GATE; tp.out16 = o16; tp.outC = G;
          launch_tc(fl.tc_gate[i], tp);
          lx.end();
        }
        {  // h = (h + res(o)) * sqrt(.5);  skip += skip_conv(o)               [tcgen05]
          lx.begin("resskip");
          tc::TcParams tp;
          memset(&tp, 0, sizeof(tp));
          tp.tmA[0] = tm_o; tp.tmA[1] = tm_o;
          tp.seg[0] = fl.tc_resskip[i].seg[0];
          tp.epi = tc::TC_EPI_RESSKIP; tp.h16 = h16; tp.hC = R; tp.skip = sk; tp.skip_set = (i == 0); tp.scale = rs;
          tp.skip16 = (i == nb - 1) ? s16 : nullptr;   // last block: relu(skip) straight into the final GEMM's A planes
          launch_tc(fl.tc_resskip[i], tp);
          lx.end();
        }
        continue;
      }
      {  // o = tanh(filter(h) + filter_c(c)) * sigmoid(gate(h) + gate_c(c))
        lx.begin("gate");
        ConvP p = make_conv(fl.gate[i]);
        p.nseg = 2;
        p.seg[0] = make_seg(hb, (long long)R * T, R, T, K, d, -(K - 1) * d, PRE_NONE, 0.f);
        p.seg[1] = make_seg(cup, (long long)CI * T, CI, T, 1, 1, 0, PRE_NONE, 0.f);
        p.Q = T; p.L_out = T; p.out_lens = lens_T; p.epi = EPI_GATE;
        p.out = ob; p.out_bstride = (long long)G * T;
        lx.conv(p, B);
        lx.end();
      }
      {  // h = (h + res(o)) * sqrt(.5);  skip += skip_conv(o)
        lx.begin("resskip");
        ConvP p = make_conv(fl.resskip[i]);
        p.nseg = 1;
        p.seg[0] = make_seg(ob, (long long)G * T, G, T, 1, 1, 0, PRE_NONE, 0.f);
        p.Q = T; p.L_out = T; p.out_lens = lens_T; p.epi = EPI_RESSKIP;
        p.Mh = R; p.scale = rs;
        p.res = hb; p.res_bstride = (long long)R * T; p.out = hb; p.out_bstride = (long long)R * T;
        p.skip = sk; p.skip_bstride = (long long)S * T; p.skip_set = (i == 0);
        lx.conv(p, B);
        lx.end();
      }
    }
    if (use_tc) {  // final_conv.1 on tensor cores with relu -> final_conv.3 -> IAF affine fused in the epilogue
      lx.begin("final_iaf_tc");
      tc::TcParams tp;
      memset(&tp, 0, sizeof(tp));
      tp.tmA[0] = tm_s; tp.tmA[1] = tm_s;
      tp.seg[0] = fl.tc_final1.seg[0];
      tp.epi = tc::TC_EPI_FINAL; tp.w3 = fl.w3; tp.z_in = zin; tp.z_out = zout;
      launch_tc(fl.tc_final1, tp);
      lx.end();
      zin = zout;
      continue;
    }
    {  // y1 = conv1x1(relu(skip))
      lx.begin("final1");
      ConvP p = make_conv(fl.final1);
      p.nseg = 1;
      p.seg[0] = make_seg(sk, (long long)S * T, S, T, 1, 1, 0, PRE_RELU, 0.f);
      p.Q = T; p.L_out = T; p.out_lens = lens_T;
      p.out = y1; p.out_bstride = (long long)S * T;
      lx.conv(p, B);
      lx.end();
    }
    {  // (mu, logs) = conv1x1(relu(y1));  z'[t+1] = z[t+1]*exp(logs[t]) + mu[t], z'[0] = 0
      lx.begin("final3_iaf");
      SmallP p;
      memset(&p, 0, sizeof(p));
      p.src = y1; p.bstride = (long long)S * T; p.C = S; p.L = T;
      p.taps = 1; p.dil = 1; p.off0 = 0; p.preact = PRE_RELU;
      p.W = fl.final3.W; p.bias = fl.final3.bias;
      p.out_lens = lens_T; p.L_out = T; p.out = zout; p.out_bstride = T;
      p.z = zin; p.z_bstride = T; p.epi = SEPI_IAF;
      lx.small(p, B, 2);
      lx.end();
    }
    zin = zout;
  }
  if (wav16 && !lx.err) {
    lx.begin("to_int16");
    const long long n = (long long)B * T;
    wav_to_int16_kernel<<<(int)std::min<long long>((n + 255) / 256, 148 * 16), 256, 0, st>>>(wav, wav16, n);
    lx.check();
    lx.end();
  }
  block_stats_dump(st);
  return lx.err;
}

// ------------------------------------------------------------------------------------------------
// WaveRNN (Path W): finalize + forward
// ------------------------------------------------------------------------------------------------
static int get_tensor(cube_voc* h, const std::string& name, std::initializer_list<int64_t> shape, const HostTensor** out) {
  auto it = h->host_w.find(name);
  if (it == h->host_w.end()) return fail("missing '%s'", name.c_str());
  if (expect_shape(name, it->second, shape)) return 1;
  *out = &it->second;
  return 0;
}

static int wrnn_head_size(int head) { return head == CUBE_HEAD_MOL ? 30 : (head == CUBE_HEAD_GM ? 2 : 256); }

static int finalize_wavernn(cube_voc* h) {
  const cube_voc_config& c = h->cfg;
  const int H = c.wrnn_size, L = c.wrnn_layers, nm = c.num_mels;
  const int ic = nm + 1 + (c.wrnn_use_lowres ? 21 : 0);
  const int S = wrnn_head_size(c.wrnn_head);
  h->wr.S = S; h->wr.ic = ic;
  if (c.wrnn_use_lowres) {
    int ci = 1;
    for (int i = 0; i < 3; ++i) {
      if (pack_conv1d(h, "_lowres_conv." + std::to_string(i) + ".conv", 20, ci, 7, &h->wr.lowres[i])) return 1;
      ci = 20;
    }
  }
  const HostTensor *wih, *whh, *bih, *bhh;
  if (get_tensor(h, "_rnns.0.weight_ih_l0", {3 * H, ic}, &wih) || get_tensor(h, "_rnns.0.weight_hh_l0", {3 * H, H}, &whh) ||
      get_tensor(h, "_rnns.0.bias_ih_l0", {3 * H}, &bih) || get_tensor(h, "_rnns.0.bias_hh_l0", {3 * H}, &bhh)) return 1;
  {  // input product for the ic-1 conditioning channels as a 1x1 conv: packed [C][Mpad]
    PackedConv& pc = h->wr.gx;
    pc.M = 3 * H; pc.Mpad = round_up(3 * H, 128); pc.Ktot = ic - 1; pc.nphase = 1;
    std::vector<float> P((size_t)pc.Ktot * pc.Mpad, 0.f), Bv(pc.Mpad, 0.f), wl(3 * H);
    for (int m = 0; m < 3 * H; ++m) {
      Bv[m] = bih->data[m];
      for (int k = 0; k < ic - 1; ++k) P[(size_t)k * pc.Mpad + m] = wih->data[(size_t)m * ic + k];
      wl[m] = wih->data[(size_t)m * ic + ic - 1];
    }
    if (dev_upload(h, P, &pc.W) || dev_upload(h, Bv, &pc.bias) || dev_upload(h, wl, &h->wr.w_last)) return 1;
  }
  if (dev_upload(h, whh->data, &h->wr.whh1) || dev_upload(h, bhh->data, &h->wr.bhh1)) return 1;
  if (L == 2) {
    const HostTensor *a, *b2, *c2, *d2;
    if (get_tensor(h, "_rnns.1.weight_ih_l0", {3 * H, H}, &a) || get_tensor(h, "_rnns.1.weight_hh_l0", {3 * H, H}, &b2) ||
        get_tensor(h, "_rnns.1.bias_ih_l0", {3 * H}, &c2) || get_tensor(h, "_rnns.1.bias_hh_l0", {3 * H}, &d2)) return 1;
    if (dev_upload(h, a->data, &h->wr.wih2) || dev_upload(h, b2->data, &h->wr.whh2) || dev_upload(h, c2->data, &h->wr.bih2) ||
        dev_upload(h, d2->data, &h->wr.bhh2)) return 1;
  }
  const HostTensor *wp, *bp, *wo, *bo;
  if (get_tensor(h, "_preoutput.linear_layer.weight", {wrnn::PRE, H}, &wp) || get_tensor(h, "_preoutput.linear_layer.bias", {wrnn::PRE}, &bp) ||
      get_tensor(h, "_output.linear_layer.weight", {S, wrnn::PRE}, &wo) || get_tensor(h, "_output.linear_layer.bias", {S}, &bo)) return 1;
  if (dev_upload(h, wp->data, &h->wr.wpre) || dev_upload(h, bp->data, &h->wr.bpre) || dev_upload(h, wo->data, &h->wr.wout) ||
      dev_upload(h, bo->data, &h->wr.bout)) return 1;
  return 0;
}

struct WrnnGeom { int G, U, P, SO, DG; size_t smem; };

static WrnnGeom wrnn_geom(const cube_voc* h, int B) {
  const cube_voc_config& c = h->cfg;
  const int H = c.wrnn_size, L = c.wrnn_layers, S = h->wr.S;
  WrnnGeom g;
  g.U = (H + h->sm_count - 1) / h->sm_count;
  g.G = (H + g.U - 1) / g.U;
  g.P = (wrnn::PRE + g.G - 1) / g.G;
  g.SO = S <= 32 ? S : (S + g.G - 1) / g.G;
  using wrnn::al4;
  g.DG = std::max(6 * g.U, std::max(g.P, S <= 32 ? 0 : g.SO));
  size_t f = (size_t)3 * g.U * H + 2 * al4(3 * g.U);
  if (L == 2) f += (size_t)6 * g.U * H + 2 * al4(3 * g.U);
  f += (size_t)g.P * H + al4(g.P) + (size_t)g.SO * wrnn::PRE + al4(g.SO);
  f += (size_t)al4(B * H) * (L == 2 ? 2 : 1) + al4(B * wrnn::PRE) + al4(B * std::max(S, 1)) + al4(B);
  f += (size_t)al4(g.DG * B) + wrnn::THREADS;
  g.smem = f * sizeof(float) + 64;
  return g;
}

static int forward_wavernn(cube_voc* h, const float* mel, const float* x_low, const float* draws, float* x, int B, int64_t F,
                           int64_t Tl, cudaStream_t st) {
  const cube_voc_config& c = h->cfg;
  const int H = c.wrnn_size, L = c.wrnn_layers, S = h->wr.S, nm = c.num_mels, ic = h->wr.ic;
  if (c.wrnn_use_lowres && !x_low) return fail("x_low is required when use_lowres = 1");
  int64_t T64 = F * c.wrnn_upsample;
  if (c.wrnn_use_lowres) T64 = std::min<int64_t>(T64, Tl * c.wrnn_upsample_low);
  if (T64 < 1 || T64 > 0x3fffffff) return fail("bad length");
  const int T = (int)T64;
  const WrnnGeom g = wrnn_geom(h, B);
  if (g.smem > 227 * 1024) return fail("batch %d needs %zu B of shared memory per CTA (max 232448): split it (cube_wavernn_max_batch)", B, g.smem);
  Launcher lx{h, st};
  float *lowA = nullptr, *lowB = nullptr, *cond, *gx, *hbuf, *prebuf, *logits;
  const int C = ic - 1;
  if (ws_get(h, "w_cond", (size_t)B * C * T, &cond) || ws_get(h, "w_gx", (size_t)B * 3 * H * T, &gx) ||
      ws_get(h, "w_h", (size_t)2 * L * B * H, &hbuf) || ws_get(h, "w_pre", (size_t)B * wrnn::PRE, &prebuf) ||
      ws_get(h, "w_lg", (size_t)B * std::max(S, 1), &logits)) return 1;
  if (c.wrnn_use_lowres) {
    if (ws_get(h, "w_lowA", (size_t)B * 20 * Tl, &lowA) || ws_get(h, "w_lowB", (size_t)B * 20 * Tl, &lowB)) return 1;
    // hidden = tanh(conv_k7(hidden)) x3 on the low-rate waveform (cube/networks/modules.py:459-461)
    const float* src = x_low; int ci = 1; float* dst = lowA;
    for (int i = 0; i < 3; ++i) {
      lx.begin("wrnn_lowres");
      ConvP p = make_conv(h->wr.lowres[i]);
      p.nseg = 1;
      p.seg[0] = make_seg(src, (long long)ci * Tl, ci, (int)Tl, 7, 1, -3, PRE_NONE, 0.f);
      p.Q = (int)Tl; p.L_out = (int)Tl; p.post = POST_TANH;
      p.out = dst; p.out_bstride = (long long)20 * Tl;
      lx.conv(p, B);
      lx.end();
      src = dst; dst = (dst == lowA) ? lowB : lowA; ci = 20;
    }
    lowA = const_cast<float*>(src);   // final features
  }
  {
    lx.begin("wrnn_cond");
    wrnn::wavernn_cond_kernel<<<dim3((T + 255) / 256, C, B), 256, 0, st>>>(mel, lowA, x_low, cond, B, (int)F, nm, (int)std::max<int64_t>(Tl, 1),
                                                                              c.wrnn_upsample, std::max(1, c.wrnn_upsample_low), T, C);
    lx.check();
    lx.end();
  }
  {  // gx[b][3H][t] = W_ih1[:, :ic-1] . cond[b][:, t] + b_ih1
    lx.begin("wrnn_gx");
    ConvP p = make_conv(h->wr.gx);
    p.nseg = 1;
    p.seg[0] = make_seg(cond, (long long)C * T, C, T, 1, 1, 0, PRE_NONE, 0.f);
    p.Q = T; p.L_out = T; p.out = gx; p.out_bstride = (long long)3 * H * T;
    lx.conv(p, B);
    lx.end();
  }
  CU_TRY(cudaMemsetAsync(hbuf, 0, (size_t)2 * L * B * H * sizeof(float), st));
  lx.begin("wrnn_loop");
  wrnn::WrnnParams wp;
  memset(&wp, 0, sizeof(wp));
  wp.H = H; wp.L = L; wp.B = B; wp.T = T; wp.S = S; wp.head = c.wrnn_head; wp.U = g.U; wp.P = g.P; wp.DG = g.DG;
  wp.gx = gx; wp.w_last = h->wr.w_last; wp.whh1 = h->wr.whh1; wp.bhh1 = h->wr.bhh1;
  wp.wih2 = h->wr.wih2; wp.bih2 = h->wr.bih2; wp.whh2 = h->wr.whh2; wp.bhh2 = h->wr.bhh2;
  wp.wpre = h->wr.wpre; wp.bpre = h->wr.bpre; wp.wout = h->wr.wout; wp.bout = h->wr.bout;
  wp.hbuf = hbuf; wp.prebuf = prebuf; wp.logits = logits; wp.draws = draws; wp.x_out = x;
  wp.log_scale_min = logf(1e-14f);
  static bool attr[64] = {false};
  if (!attr[h->device & 63]) {
    CU_TRY(cudaFuncSetAttribute(wrnn::wavernn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr[h->device & 63] = true;
  }
  void* args[] = {&wp};
  CU_TRY(cudaLaunchCooperativeKernel((void*)wrnn::wavernn_kernel, dim3(g.G), dim3(wrnn::THREADS), args, g.smem, st));
  h->launches++;
  lx.end();
  return lx.err;
}

// ------------------------------------------------------------------------------------------------
// UpsampleNet (cube/networks/modules.py:317-343): finalize + forward on the fp32 kernels
// ------------------------------------------------------------------------------------------------
static int finalize_upsamplenet(cube_voc* h) {
  const cube_voc_config& c = h->cfg;
  const int Cin = c.num_mels, Co = c.res_channels, K = c.kernel_size;
  int ic = Cin;
  for (int i = 0; i < 3; ++i) {       // ModuleList [Conv1d, Tanh] x 3: the convs sit at indices 0, 2, 4
    if (pack_conv1d(h, "_conv." + std::to_string(2 * i), Co, ic, K, &h->upnet.conv[i])) return 1;
    ic = Co;
  }
  h->upnet.up.resize(c.n_upsample);
  h->upnet.J.resize(c.n_upsample);
  for (int n = 0; n < c.n_upsample; ++n) {
    const int s_ = c.upsample_scales[n];
    if (pack_convT(h, "_upsample_conv." + std::to_string(2 * n), Co, Co, 2 * s_, s_, &h->upnet.up[n], &h->upnet.J[n])) return 1;
  }
  return 0;
}

static int forward_upsamplenet(cube_voc* h, const float* mel, const int32_t* n_frames, float* out, int B, int64_t Fmax, cudaStream_t st) {
  const cube_voc_config& c = h->cfg;
  const int Cin = c.num_mels, Co = c.res_channels, K = c.kernel_size;
  int64_t T64 = Fmax;
  for (int n = 0; n < c.n_upsample; ++n) T64 *= c.upsample_scales[n];
  if (T64 > 0x7fffffffLL / 2) return fail("utterance too long");
  if (upload_lens(h, n_frames, B, Fmax, c.n_upsample + 1, st)) return 1;
  float *a, *b2;
  const size_t big = (size_t)B * Co * (size_t)std::max<int64_t>(Fmax, T64 / c.upsample_scales[c.n_upsample - 1]);
  if (ws_get(h, "un_a", big, &a) || ws_get(h, "un_b", big, &b2)) return 1;
  Launcher lx{h, st};
  const float* src = mel;
  int ic = Cin;
  const int F = (int)Fmax;
  float* pp[2] = {a, b2};
  for (int i = 0; i < 3; ++i) {       // c = tanh(conv_k(c)), "same" padding k/2
    lx.begin("upnet_conv");
    ConvP p = make_conv(h->upnet.conv[i]);
    p.nseg = 1;
    p.seg[0] = make_seg(src, (long long)ic * F, ic, F, K, 1, -(K / 2), PRE_NONE, 0.f, h->d_lens);
    p.Q = F; p.L_out = F; p.out_lens = h->d_lens; p.post = POST_TANH;
    p.out = pp[i & 1]; p.out_bstride = (long long)Co * F;
    lx.conv(p, B);
    lx.end();
    src = pp[i & 1]; ic = Co;
  }
  int Lin = F, which = 1;             // the last conv wrote pp[0] (i = 2): the next output goes to pp[1]
  for (int n = 0; n < c.n_upsample; ++n) {   // c = tanh(convT_{2s, stride s, padding s/2}(c))
    const int s_ = c.upsample_scales[n], pad = s_ / 2, J = h->upnet.J[n], Lo = Lin * s_;
    const bool last = n == c.n_upsample - 1;
    lx.begin("upnet_up");
    ConvP p = make_conv(h->upnet.up[n]);
    p.nseg = 1;
    p.seg[0] = make_seg(src, (long long)Co * Lin, Co, Lin, J, 1, -(J - 1), PRE_NONE, 0.f, h->d_lens + (size_t)n * B);
    p.nphase = s_; p.ostride = s_;
    for (int r = 0; r < s_; ++r) p.ooff[r] = r - pad;
    p.Q = (Lo - 1 + pad) / s_ + 1;
    p.L_out = Lo; p.out_lens = h->d_lens + (size_t)(n + 1) * B; p.post = POST_TANH;
    p.out = last ? out : pp[which]; p.out_bstride = (long long)Co * Lo;
    lx.conv(p, B);
    lx.end();
    src = pp[which]; which ^= 1; Lin = Lo;
  }
  return lx.err;
}

static int ensure_device(cube_voc* h) {
  CU_TRY(cudaSetDevice(h->device));
  return 0;
}

template <typename T>
static int grow(T** p, size_t* cap, size_t need_bytes, uint64_t* gen = nullptr) {
  if (*cap >= need_bytes) return 0;
  if (*p) CU_TRY(cudaFree(*p));
  *p = nullptr; *cap = 0;
  if (gen) ++*gen;
  CU_TRY(cudaMalloc((void**)p, need_bytes));
  *cap = need_bytes;
  return 0;
}

static int head_grid(int64_t n) {
  int64_t g = (n + 255) / 256;
  if (g > 148 * 32) g = 148 * 32;
  if (g < 1) g = 1;
  return (int)g;
}

static int tables_ready() {
  static int dev_done[64] = {0};
  int dev = 0;
  CU_TRY(cudaGetDevice(&dev));
  if (dev < 64 && dev_done[dev]) return 0;
  CU_TRY(upload_mulaw_tables());
  if (dev < 64) dev_done[dev] = 1;
  return 0;
}

}  // namespace cube

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char* cube_voc_last_error(void) { return cube::g_err; }

#define CUBE_STR2(x) #x
#define CUBE_STR(x) CUBE_STR2(x)
const char* cube_voc_build_info(void) {
  return "libcube_vocoder " CUBE_VERSION " sm_100a (nvcc " CUBE_STR(__CUDACC_VER_MAJOR__) "." CUBE_STR(__CUDACC_VER_MINOR__) ")";
}

int cube_voc_create(cube_voc_t** out, const cube_voc_config* cfg, int device) {
  if (!out || !cfg) return fail("null argument");
  if (cfg->struct_size != sizeof(cube_voc_config))
    return fail("cube_voc_config.struct_size = %u but this library's struct is %zu bytes: the binding does not match include/cube_vocoder.h",
                cfg->struct_size, sizeof(cube_voc_config));
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail("no CUDA device: libcube_vocoder has no CPU path (%s)", e != cudaSuccess ? cudaGetErrorString(e) : "0 devices");
  if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
  if (cfg->arch != CUBE_VOC_HIFIGAN && cfg->arch != CUBE_VOC_PWN_STUDENT && cfg->arch != CUBE_VOC_WAVERNN && cfg->arch != CUBE_VOC_UPSAMPLENET)
    return fail("unknown arch %d", cfg->arch);
  if (cfg->arch == CUBE_VOC_HIFIGAN) {
    if (cfg->n_ups < 1 || cfg->n_ups > CUBE_MAX_UPS) return fail("n_ups %d out of range", cfg->n_ups);
    if (cfg->n_resblock_kernels < 1 || cfg->n_resblock_kernels > CUBE_MAX_RBK) return fail("n_resblock_kernels out of range");
    if (cfg->resblock_type != 1 && cfg->resblock_type != 2) return fail("resblock must be 1 or 2");
    if (cfg->upsample_initial_channel >> cfg->n_ups < 1) return fail("upsample_initial_channel too small");
    for (int i = 0; i < cfg->n_ups; ++i) {
      if (cfg->upsample_rates[i] < 1 || cfg->upsample_rates[i] > 8) return fail("upsample rate %d unsupported (1..8)", cfg->upsample_rates[i]);
      if (cfg->upsample_kernel_sizes[i] < cfg->upsample_rates[i]) return fail("upsample kernel smaller than rate");
    }
    for (int j = 0; j < cfg->n_resblock_kernels; ++j) {
      if (cfg->resblock_kernel_sizes[j] % 2 != 1) return fail("resblock kernel sizes must be odd");
      if (cfg->n_dilations[j] < 1 || cfg->n_dilations[j] > CUBE_MAX_DIL) return fail("n_dilations out of range");
    }
  } else if (cfg->arch == CUBE_VOC_WAVERNN) {
    if (cfg->wrnn_layers < 1 || cfg->wrnn_layers > 2) return fail("WaveRNN num_layers must be 1 or 2");
    if (cfg->wrnn_size < 8 || cfg->wrnn_size > 1024 || cfg->wrnn_size % 4) return fail("WaveRNN layer_size must be a multiple of 4 in [8, 1024]");
    if (cfg->wrnn_upsample < 1 || (cfg->wrnn_use_lowres && cfg->wrnn_upsample_low < 1)) return fail("bad upsample");
    if (cfg->wrnn_head < 0 || cfg->wrnn_head > 3) return fail("unknown head");
  } else if (cfg->arch == CUBE_VOC_UPSAMPLENET) {
    if (cfg->n_upsample < 1 || cfg->n_upsample > 4) return fail("n_upsample out of range");
    if (cfg->num_mels < 1 || cfg->res_channels < 1) return fail("UpsampleNet needs num_mels (in_channels) and res_channels (out_channels)");
    if (cfg->kernel_size < 1 || cfg->kernel_size % 2 != 1 || cfg->kernel_size > 31) return fail("UpsampleNet kernel_size must be odd (got %d)", cfg->kernel_size);
    for (int i = 0; i < cfg->n_upsample; ++i)
      if (cfg->upsample_scales[i] < 2 || cfg->upsample_scales[i] > 8 || cfg->upsample_scales[i] % 2)
        return fail("UpsampleNet scales must be even and in [2, 8] (got %d): odd scales change the length law", cfg->upsample_scales[i]);
  } else {
    if (cfg->n_flows < 1 || cfg->n_flows > CUBE_MAX_FLOWS) return fail("n_flows out of range");
    if (cfg->n_upsample < 1 || cfg->n_upsample > 4) return fail("n_upsample out of range");
    if (cfg->gate_channels % 4) return fail("gate_channels must be a multiple of 4");
  }
  cube_voc* h = new cube_voc();
  h->cfg = *cfg;
  h->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete h; return fail("cudaSetDevice(%d) failed", device); }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
    h->sm_count = prop.multiProcessorCount;
    if (prop.major != 10) { delete h; return fail("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); }
  }
  *out = h;
  return 0;
}

int cube_voc_load_weight(cube_voc_t* h, const char* name, const float* data, const int64_t* shape, int ndim) {
  if (!h || !name || !data || (ndim > 0 && !shape)) return fail("null argument");
  if (h->finalized) return fail("load_weight after finalize");
  std::string n(name);
  for (const char* pre : {"_generator.", "generator.", "module."})
    if (n.rfind(pre, 0) == 0) n = n.substr(strlen(pre));
  HostTensor t;
  t.shape.assign(shape, shape + ndim);
  const int64_t ne = t.numel();
  if (ne < 0 || ne > (1LL << 31)) return fail("bad shape for '%s'", name);
  t.data.assign(data, data + ne);
  h->host_w[n] = std::move(t);
  return 0;
}

int cube_voc_finalize(cube_voc_t* h) {
  if (!h) return fail("null handle");
  if (h->finalized) return 0;
  if (ensure_device(h)) return 1;
  if (tables_ready()) return 1;
  int rc = h->cfg.arch == CUBE_VOC_HIFIGAN ? finalize_hifigan(h)
         : h->cfg.arch == CUBE_VOC_WAVERNN ? finalize_wavernn(h)
         : h->cfg.arch == CUBE_VOC_UPSAMPLENET ? finalize_upsamplenet(h) : finalize_student(h);
  if (rc) return rc;
  h->host_w.clear();
  CU_TRY(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  h->finalized = true;
  return 0;
}

int64_t cube_voc_out_len(const cube_voc_t* h, int64_t n_frames) {
  if (!h || n_frames < 0) { fail("bad argument"); return -1; }
  if (h->cfg.arch == CUBE_VOC_HIFIGAN) return n_frames == 0 ? 0 : hifigan_len(h->cfg, n_frames, h->cfg.n_ups);
  int64_t T = n_frames;
  for (int i = 0; i < h->cfg.n_upsample; ++i) T *= h->cfg.upsample_scales[i];
  return T;
}

int cube_voc_forward(cube_voc_t* h, const float* mel, const int32_t* n_frames, const float* noise, float* wav,
                     int16_t* wav_i16, int B, int64_t Fmax, cube_stream_t stream) {
  if (!h) return fail("null handle");
  if (!h->finalized) return fail("forward before finalize");
  if (!mel || !wav) return fail("null mel/wav");
  if (B < 1 || Fmax < 1) return fail("empty batch (B=%d, Fmax=%lld)", B, (long long)Fmax);
  if (ensure_device(h)) return 1;
  h->launches = 0;
  for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  h->prof.clear();
  cudaStream_t st = (cudaStream_t)stream;
  if (h->cfg.arch == CUBE_VOC_WAVERNN) return fail("use cube_wavernn_forward for a WaveRNN handle");
  if (h->cfg.arch == CUBE_VOC_HIFIGAN) return forward_hifigan(h, mel, n_frames, wav, wav_i16, B, Fmax, st);
  if (h->cfg.arch == CUBE_VOC_UPSAMPLENET) {
    if (wav_i16) return fail("UpsampleNet has no int16 output");
    return forward_upsamplenet(h, mel, n_frames, wav, B, Fmax, st);
  }
  return forward_student(h, mel, n_frames, noise, wav, wav_i16, B, Fmax, st);
}

int cube_voc_hifigan_support(const cube_voc_config* cfg, int64_t s0, int64_t s1, int64_t* f0, int64_t* f1) {
  if (!cfg || !f0 || !f1) return fail("null argument");
  if (cfg->struct_size != sizeof(cube_voc_config))
    return fail("cube_voc_config.struct_size = %u but this library's struct is %zu bytes", cfg->struct_size, sizeof(cube_voc_config));
  if (cfg->arch != CUBE_VOC_HIFIGAN) return fail("sample support is defined for HiFi-GAN configs only");
  if (cfg->n_ups < 1 || cfg->n_ups > CUBE_MAX_UPS || cfg->n_resblock_kernels < 1 || cfg->n_resblock_kernels > CUBE_MAX_RBK)
    return fail("bad HiFi-GAN config (n_ups=%d, n_resblock_kernels=%d)", cfg->n_ups, cfg->n_resblock_kernels);
  for (int i = 0; i < cfg->n_ups; ++i)
    if (cfg->upsample_rates[i] < 1 || cfg->upsample_kernel_sizes[i] < cfg->upsample_rates[i])
      return fail("bad upsample stage %d (rate %d, kernel %d)", i, cfg->upsample_rates[i], cfg->upsample_kernel_sizes[i]);
  for (int j = 0; j < cfg->n_resblock_kernels; ++j)
    if (cfg->resblock_kernel_sizes[j] < 1 || cfg->n_dilations[j] < 1 || cfg->n_dilations[j] > CUBE_MAX_DIL)
      return fail("bad ResBlock %d", j);
  if (s0 < 0 || s0 >= s1) return fail("empty or negative sample range [%lld, %lld)", (long long)s0, (long long)s1);
  HifiganPlan P;
  hifigan_plan(*cfg, s0, s1, nullptr, false, &P);
  *f0 = P.mel.a; *f1 = P.mel.b;
  return 0;
}

int cube_voc_forward_range(cube_voc_t* h, const float* mel, const int32_t* n_frames, const int64_t* out_begin,
                           const int64_t* out_end, float* wav, int16_t* wav_i16, int B, int64_t Fmax, cube_stream_t stream) {
  if (!h) return fail("null handle");
  if (h->cfg.arch != CUBE_VOC_HIFIGAN) return fail("the sample-range forward is defined for HiFi-GAN handles only");
  if (!h->finalized) return fail("forward before finalize");
  if (!mel || !wav || !out_begin || !out_end) return fail("null mel/wav/out_begin/out_end");
  if (B < 1 || Fmax < 1) return fail("empty batch (B=%d, Fmax=%lld)", B, (long long)Fmax);
  int64_t s0 = INT64_MAX, s1 = 0;
  h->h_rng.resize((size_t)2 * B);
  for (int b = 0; b < B; ++b) {
    const int64_t f = n_frames ? n_frames[b] : Fmax;
    if (f < 0 || f > Fmax) return fail("n_frames[%d]=%lld outside [0, %lld]", b, (long long)f, (long long)Fmax);
    const int64_t T = f == 0 ? 0 : hifigan_len(h->cfg, f, h->cfg.n_ups);
    if (out_begin[b] < 0 || out_begin[b] >= out_end[b] || out_end[b] > T)
      return fail("sample range [%lld, %lld) of item %d is empty or outside [0, %lld)", (long long)out_begin[b],
                  (long long)out_end[b], b, (long long)T);
    s0 = std::min(s0, out_begin[b]); s1 = std::max(s1, out_end[b]);
    h->h_rng[2 * b] = (int)out_begin[b]; h->h_rng[2 * b + 1] = (int)out_end[b];
  }
  if (hifigan_len(h->cfg, Fmax, h->cfg.n_ups) > 0x7fffffffLL / 2) return fail("utterance too long");
  if (ensure_device(h)) return 1;
  h->launches = 0;
  for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  h->prof.clear();
  cudaStream_t st = (cudaStream_t)stream;
  float* d_rng;
  if (ws_get(h, "rng", (size_t)2 * B, &d_rng)) return 1;   // int32 in a float-sized buffer
  CU_TRY(cudaMemcpyAsync(d_rng, h->h_rng.data(), (size_t)2 * B * sizeof(int), cudaMemcpyHostToDevice, st));
  const RangeReq rq{s0, s1, (const int*)d_rng};
  return forward_hifigan(h, mel, n_frames, wav, wav_i16, B, Fmax, st, &rq);
}

// CUBE_GRAPH=0 disables the CUDA-graph replay of the host-buffer call
static bool graphs_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUBE_GRAPH"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

int cube_voc_forward_host(cube_voc_t* h, const float* mel, const int32_t* n_frames, const float* noise, float* wav,
                          int16_t* wav_i16, int B, int64_t Fmax) {
  if (!h) return fail("null handle");
  if (!h->finalized) return fail("forward before finalize");
  if (!mel || (!wav && !wav_i16)) return fail("null mel / no output buffer");
  if (B < 1 || Fmax < 1) return fail("empty batch");
  if (h->cfg.arch == CUBE_VOC_WAVERNN) return fail("use cube_wavernn_forward for a WaveRNN handle");
  if (h->cfg.arch == CUBE_VOC_UPSAMPLENET) return fail("the host-buffer call is defined for the waveform vocoders; use cube_voc_forward for UpsampleNet");
  if (h->cfg.arch == CUBE_VOC_PWN_STUDENT && !noise) return fail("the IAF student needs `noise` (z ~ N(0,1), [B,1,T])");
  if (ensure_device(h)) return 1;
  const int64_t T = cube_voc_out_len(h, Fmax);
  const size_t mel_b = (size_t)B * h->cfg.num_mels * Fmax * sizeof(float);
  const size_t wav_n = (size_t)B * T;
  if (grow(&h->d_mel, &h->d_mel_cap, mel_b, &h->alloc_gen) || grow(&h->d_wav, &h->d_wav_cap, wav_n * sizeof(float), &h->alloc_gen)) return 1;
  if (wav_i16 && grow(&h->d_wav16, &h->d_wav16_cap, wav_n * sizeof(int16_t), &h->alloc_gen)) return 1;
  if (noise && grow(&h->d_noise, &h->d_noise_cap, wav_n * sizeof(float), &h->alloc_gen)) return 1;
  cudaStream_t st = h->own_stream;
  CU_TRY(cudaMemcpyAsync(h->d_mel, mel, mel_b, cudaMemcpyHostToDevice, st));
  if (noise) CU_TRY(cudaMemcpyAsync(h->d_noise, noise, wav_n * sizeof(float), cudaMemcpyHostToDevice, st));

  // ---- the forward itself: replay a captured graph when one exists for this geometry, capture one on the second call
  // with a geometry (the first call runs eagerly and sizes the workspace), else launch kernel by kernel ----
  bool done = false;
  if (graphs_enabled() && !h->profile && !block_stats_on()) {
    const std::vector<int64_t> key = {B, Fmax, noise ? 1 : 0, wav_i16 ? 1 : 0};
    cube_voc::GraphEntry& ge = h->graphs[key];
    if (ge.exec && ge.gen != h->alloc_gen) { cudaGraphExecDestroy(ge.exec); ge.exec = nullptr; }
    if (ge.exec || ge.seen >= 1) {
      if (stage_lens_pinned(h, n_frames, B, Fmax)) return 1;        // validates n_frames, fills the pinned mask buffer
      if (ge.exec && ge.gen != h->alloc_gen) { cudaGraphExecDestroy(ge.exec); ge.exec = nullptr; }   // the pinned buffer moved
    }
    if (!ge.exec && ge.seen >= 1) {
      const uint64_t gen0 = h->alloc_gen;
      cudaGraph_t graph = nullptr;
      h->lens_from_pinned = true;
      cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
      int rc = 1;
      if (e == cudaSuccess) {
        rc = cube_voc_forward(h, h->d_mel, n_frames, noise ? h->d_noise : nullptr, h->d_wav, wav_i16 ? h->d_wav16 : nullptr, B, Fmax, st);
        e = cudaStreamEndCapture(st, &graph);
      }
      h->lens_from_pinned = false;
      if (e == cudaSuccess && rc == 0 && graph && gen0 == h->alloc_gen) {
        cudaGraphExec_t ex = nullptr;
        if (cudaGraphInstantiate(&ex, graph, 0) == cudaSuccess) { ge.exec = ex; ge.gen = h->alloc_gen; ge.launches = h->launches; }
      }
      if (graph) cudaGraphDestroy(graph);
      if (!ge.exec) {
        cudaGetLastError();                                         // a failed capture must not poison the eager path
        if (rc) return rc;
      }
    }
    if (ge.exec) {
      CU_TRY(cudaGraphLaunch(ge.exec, st));
      h->launches = ge.launches;
      done = true;
    }
    ++ge.seen;
  }
  if (!done && cube_voc_forward(h, h->d_mel, n_frames, noise ? h->d_noise : nullptr, h->d_wav, wav_i16 ? h->d_wav16 : nullptr, B, Fmax, st)) return 1;
  if (wav) CU_TRY(cudaMemcpyAsync(wav, h->d_wav, wav_n * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (wav_i16) CU_TRY(cudaMemcpyAsync(wav_i16, h->d_wav16, wav_n * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  return 0;
}

int64_t cube_wavernn_out_len(const cube_voc_t* h, int64_t n_frames, int64_t n_low) {
  if (!h || h->cfg.arch != CUBE_VOC_WAVERNN || n_frames < 0) { fail("bad argument"); return -1; }
  int64_t T = n_frames * h->cfg.wrnn_upsample;
  if (h->cfg.wrnn_use_lowres) T = std::min<int64_t>(T, n_low * h->cfg.wrnn_upsample_low);
  return T;
}

int cube_wavernn_max_batch(const cube_voc_t* h) {
  if (!h || h->cfg.arch != CUBE_VOC_WAVERNN || !h->finalized) { fail("bad handle"); return -1; }
  int b = 1;
  while (b < 1024 && wrnn_geom(h, b + 1).smem <= 227 * 1024) ++b;
  return b;
}

int cube_wavernn_forward(cube_voc_t* h, const float* mel, const float* x_low, const float* draws, float* x, int B, int64_t F,
                         int64_t Tl, cube_stream_t stream) {
  if (!h) return fail("null handle");
  if (h->cfg.arch != CUBE_VOC_WAVERNN) return fail("not a WaveRNN handle");
  if (!h->finalized) return fail("forward before finalize");
  if (!mel || !draws || !x) return fail("null argument");
  if (B < 1 || F < 1) return fail("empty batch");
  if (ensure_device(h)) return 1;
  h->launches = 0;
  for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  h->prof.clear();
  return forward_wavernn(h, mel, x_low, draws, x, B, F, Tl, (cudaStream_t)stream);
}

int cube_voc_get_cond(cube_voc_t* h, float* c_up, int B, int64_t Tmax, cube_stream_t stream) {
  if (!h || !c_up) return fail("null argument");
  if (h->cfg.arch != CUBE_VOC_PWN_STUDENT) return fail("get_cond is only defined for the IAF student");
  if (B != h->last_B || Tmax != h->last_T) return fail("geometry differs from the last forward");
  auto it = h->ws.find("c_up");
  if (it == h->ws.end()) return fail("no forward has run");
  CU_TRY(cudaMemcpyAsync(c_up, it->second.p, (size_t)B * h->cfg.num_mels * Tmax * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int64_t cube_voc_last_launches(const cube_voc_t* h) { return h ? h->launches : -1; }

int64_t cube_voc_workspace_bytes(const cube_voc_t* h) {
  if (!h) return -1;
  int64_t n = 0;
  for (auto& kv : h->ws) n += (int64_t)kv.second.bytes;
  return n;
}

int cube_voc_set_profile(cube_voc_t* h, int on) {
  if (!h) return fail("null handle");
  h->profile = on != 0;
  return 0;
}

int cube_voc_get_profile(cube_voc_t* h, char* names, float* ms, int cap) {
  if (!h || !names || !ms) { fail("null argument"); return -1; }
  std::map<std::string, float> agg;
  std::vector<std::string> order;
  for (auto& r : h->prof) {
    if (cudaEventSynchronize(r.b) != cudaSuccess) { fail("profile event sync failed"); return -1; }
    float t = 0.f;
    cudaEventElapsedTime(&t, r.a, r.b);
    if (!agg.count(r.name)) order.push_back(r.name);
    agg[r.name] += t;
  }
  int n = 0;
  for (auto& k : order) {
    if (n >= cap) break;
    snprintf(names + (size_t)n * 64, 64, "%s", k.c_str());
    ms[n] = agg[k];
    ++n;
  }
  return n;
}

void cube_voc_destroy(cube_voc_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (void* p : h->dev_allocs) cudaFree(p);
  for (auto& kv : h->ws) if (kv.second.p) cudaFree(kv.second.p);
  if (h->d_lens) cudaFree(h->d_lens);
  if (h->d_mel) cudaFree(h->d_mel);
  if (h->d_noise) cudaFree(h->d_noise);
  if (h->d_wav) cudaFree(h->d_wav);
  if (h->d_wav16) cudaFree(h->d_wav16);
  for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto& kv : h->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  if (h->h_lens_pin) cudaFreeHost(h->h_lens_pin);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

// ---- heads ----
#define HEAD_PROLOGUE(n)                        \
  if ((n) < 0) return fail("negative length");  \
  if ((n) == 0) return 0;                       \
  if (tables_ready()) return 1;

int cube_mulaw_encode(const float* x, int64_t* q, int64_t n, cube_stream_t s) {
  HEAD_PROLOGUE(n);
  if (!x || !q) return fail("null argument");
  mulaw_encode_kernel<<<head_grid(n), 256, 0, (cudaStream_t)s>>>(x, (long long*)q, n);
  CU_TRY(cudaGetLastError());
  return 0;
}
int cube_mulaw_decode(const int64_t* q, float* x, int64_t n, cube_stream_t s) {
  HEAD_PROLOGUE(n);
  if (!x || !q) return fail("null argument");
  mulaw_decode_kernel<<<head_grid(n), 256, 0, (cudaStream_t)s>>>((const long long*)q, x, n);
  CU_TRY(cudaGetLastError());
  return 0;
}
int cube_raw_encode(const float* x, int64_t* q, int64_t n, cube_stream_t s) {
  HEAD_PROLOGUE(n);
  if (!x || !q) return fail("null argument");
  raw_encode_kernel<<<head_grid(n), 256, 0, (cudaStream_t)s>>>(x, (long long*)q, n);
  CU_TRY(cudaGetLastError());
  return 0;
}
int cube_raw_decode(const int64_t* q, float* x, int64_t n, cube_stream_t s) {
  HEAD_PROLOGUE(n);
  if (!x || !q) return fail("null argument");
  raw_decode_kernel<<<head_grid(n), 256, 0, (cudaStream_t)s>>>((const long long*)q, x, n);
  CU_TRY(cudaGetLastError());
  return 0;
}
int cube_mol_sample(const float* y, const float* u_mix, const float* u_x, float* x, int64_t n, int nr_mix,
                    float log_scale_min, float temperature, cube_stream_t s) {
  HEAD_PROLOGUE(n);
  if (!y || !u_mix || !u_x || !x) return fail("null argument");
  if (nr_mix < 1) return fail("nr_mix < 1");
  mol_sample_kernel<<<head_grid(n), 256, 0, (cudaStream_t)s>>>(y, u_mix, u_x, x, n, nr_mix, log_scale_min, temperature);
  CU_TRY(cudaGetLastError());
  return 0;
}
int cube_gaussian_sample(const float* y, const float* eps, float* x, int64_t n, cube_stream_t s) {
  HEAD_PROLOGUE(n);
  if (!y || !eps || !x) return fail("null argument");
  gaussian_sample_kernel<<<head_grid(n), 256, 0, (cudaStream_t)s>>>(y, eps, x, n);
  CU_TRY(cudaGetLastError());
  return 0;
}
int cube_categorical_sample(const float* logits, const float* u, int64_t* idx, int64_t n, int C, cube_stream_t s) {
  HEAD_PROLOGUE(n);
  if (!logits || !u || !idx) return fail("null argument");
  if (C < 1) return fail("C < 1");
  categorical_sample_kernel<<<head_grid(n * 32), 256, 0, (cudaStream_t)s>>>(logits, u, (long long*)idx, n, C);
  CU_TRY(cudaGetLastError());
  return 0;
}
int cube_wav_to_int16(const float* wav, int16_t* out, int64_t n, cube_stream_t s) {
  if (n < 0) return fail("negative length");
  if (n == 0) return 0;
  if (!wav || !out) return fail("null argument");
  wav_to_int16_kernel<<<head_grid(n), 256, 0, (cudaStream_t)s>>>(wav, out, n);
  CU_TRY(cudaGetLastError());
  return 0;
}

// ---- log-mel spectrogram ----
struct cube_mel {
  cube_mel_config cfg;
  int device = 0, n_bins = 0, KB = 0;
  float *cosT = nullptr, *sinT = nullptr, *basis = nullptr;
  int *k_lo = nullptr, *k_hi = nullptr, *d_len = nullptr;
  int len_cap = 0;
  size_t smem = 0;
};

int cube_mel_create(cube_mel_t** out, const cube_mel_config* cfg, const float* window, const float* mel_basis, int device) {
  using namespace cube;
  if (!out || !cfg || !mel_basis) return fail("null argument");
  if (cfg->struct_size != sizeof(cube_mel_config))
    return fail("cube_mel_config.struct_size = %u but this library's struct is %zu bytes: the binding does not match include/cube_vocoder.h",
                cfg->struct_size, sizeof(cube_mel_config));
  const cube_mel_config& c = *cfg;
  if (c.n_fft < 16 || c.n_fft > 4096 || c.n_fft % 4) return fail("n_fft must be a multiple of 4 in [16, 4096] (got %d)", c.n_fft);
  if (c.hop_size < 4 || c.hop_size % 4) return fail("hop_size must be a positive multiple of 4 (got %d)", c.hop_size);
  if (c.win_size < 1 || c.win_size > c.n_fft) return fail("win_size must be in [1, n_fft] (got %d)", c.win_size);
  if (c.n_mels < 1 || c.n_mels > 512) return fail("n_mels out of range (%d)", c.n_mels);
  if (c.pad_left < 0 || c.pad_right < 0) return fail("negative padding");
  if (c.layout != 0 && c.layout != 1) return fail("layout must be 0 ([B,M,F]) or 1 ([B,F,M])");
  if (c.pad_mode != 0 && c.pad_mode != 1) return fail("pad_mode must be 0 (reflect) or 1 (constant zeros)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("no CUDA device: libcube_vocoder has no CPU fallback");
  if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
  CU_TRY(cudaSetDevice(device));
  cube_mel* h = new cube_mel();
  h->cfg = c; h->device = device;
  h->n_bins = c.n_fft / 2 + 1;
  h->KB = (h->n_bins + mel::BT - 1) / mel::BT * mel::BT;
  h->smem = mel::smem_bytes(c.n_fft, c.hop_size, h->KB);
  if (h->smem > 220 * 1024) { delete h; return fail("n_fft/hop too large for one CTA's shared memory (%zu bytes)", h->smem); }
  // window (centred in n_fft like torch.stft) folded into the DFT tables, all in double on the host
  const double PI = 3.14159265358979323846;
  std::vector<double> w(c.n_fft, 0.0);
  const int wl = (c.n_fft - c.win_size) / 2;
  for (int i = 0; i < c.win_size; ++i) w[wl + i] = window ? (double)window[i] : 0.5 - 0.5 * cos(2.0 * PI * i / c.win_size);
  std::vector<float> ct((size_t)c.n_fft * h->KB, 0.f), st((size_t)c.n_fft * h->KB, 0.f);
  for (int n = 0; n < c.n_fft; ++n)
    for (int k = 0; k < h->n_bins; ++k) {
      const long long r = ((long long)k * n) % c.n_fft;      // exact argument reduction
      const double a = 2.0 * PI * (double)r / c.n_fft;
      ct[(size_t)n * h->KB + k] = (float)(w[n] * cos(a));
      st[(size_t)n * h->KB + k] = (float)(-w[n] * sin(a));
    }
  std::vector<int> lo(c.n_mels), hi(c.n_mels);
  for (int m = 0; m < c.n_mels; ++m) {
    int a = h->n_bins, b = 0;
    for (int k = 0; k < h->n_bins; ++k)
      if (mel_basis[(size_t)m * h->n_bins + k] != 0.f) { a = std::min(a, k); b = std::max(b, k + 1); }
    lo[m] = std::min(a, b); hi[m] = b;
  }
  auto up = [&](const void* src, size_t bytes, void** dst) -> int {
    CU_TRY(cudaMalloc(dst, bytes));
    CU_TRY(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return 0;
  };
  if (up(ct.data(), ct.size() * 4, (void**)&h->cosT) || up(st.data(), st.size() * 4, (void**)&h->sinT) ||
      up(mel_basis, (size_t)c.n_mels * h->n_bins * 4, (void**)&h->basis) || up(lo.data(), lo.size() * 4, (void**)&h->k_lo) ||
      up(hi.data(), hi.size() * 4, (void**)&h->k_hi)) {
    cube_mel_destroy(h);
    return 1;
  }
  *out = h;
  return 0;
}

int64_t cube_mel_out_frames(const cube_mel_t* h, int64_t n_samples) {
  if (!h || n_samples < 0 || n_samples > INT32_MAX) return -1;
  return cube::mel::n_frames_of((int)n_samples, h->cfg.n_fft, h->cfg.hop_size, h->cfg.pad_left, h->cfg.pad_right, h->cfg.pad_mode);
}

int cube_mel_forward(cube_mel_t* h, const float* wav, const int32_t* n_samples, float* out, int B, int64_t Tmax, int64_t Fmax,
                     cube_stream_t stream) {
  using namespace cube;
  if (!h || !wav || !out) return fail("null argument");
  if (B <= 0 || Tmax <= 0 || Fmax <= 0 || Tmax > INT32_MAX || Fmax > INT32_MAX) return fail("bad shape B=%d Tmax=%lld Fmax=%lld", B, (long long)Tmax, (long long)Fmax);
  CU_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  int longest = (int)Tmax;
  if (n_samples) {
    longest = 0;
    for (int b = 0; b < B; ++b) {
      if (n_samples[b] < 0 || n_samples[b] > Tmax) return fail("n_samples[%d]=%d outside [0, Tmax=%lld]", b, n_samples[b], (long long)Tmax);
      longest = std::max(longest, (int)n_samples[b]);
    }
    if (h->len_cap < B) {
      if (h->d_len) CU_TRY(cudaFree(h->d_len));
      CU_TRY(cudaMalloc(&h->d_len, (size_t)B * sizeof(int)));
      h->len_cap = B;
    }
    CU_TRY(cudaMemcpyAsync(h->d_len, n_samples, (size_t)B * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  if (cube_mel_out_frames(h, longest) > Fmax) return fail("Fmax=%lld is smaller than the %lld frames of the longest utterance", (long long)Fmax, (long long)cube_mel_out_frames(h, longest));
  mel::MelParams p;
  p.wav = wav; p.n_samples = n_samples ? h->d_len : nullptr;
  p.cosT = h->cosT; p.sinT = h->sinT; p.basis = h->basis; p.k_lo = h->k_lo; p.k_hi = h->k_hi; p.out = out;
  p.B = B; p.Tmax = (int)Tmax; p.Fmax = (int)Fmax;
  p.n_fft = h->cfg.n_fft; p.hop = h->cfg.hop_size; p.n_bins = h->n_bins; p.KB = h->KB; p.n_mels = h->cfg.n_mels;
  p.pad_left = h->cfg.pad_left; p.pad_right = h->cfg.pad_right; p.layout = h->cfg.layout; p.log10_out = h->cfg.log10_out; p.pad_mode = h->cfg.pad_mode;
  p.mag_eps = h->cfg.mag_eps; p.floor_val = h->cfg.floor_val; p.pad_value = h->cfg.pad_value; p.preemph = h->cfg.preemph;
  {  // the opt-in shared-memory limit is per kernel and device, not per handle: only ever raise it
    static size_t granted[64] = {0};
    if (h->smem > granted[h->device & 63]) {
      CU_TRY(cudaFuncSetAttribute(mel::melspec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem));
      granted[h->device & 63] = h->smem;
    }
  }
  dim3 grid((unsigned)((Fmax + mel::FT - 1) / mel::FT), (unsigned)B);
  mel::melspec_kernel<<<grid, mel::THREADS, h->smem, st>>>(p);
  CU_TRY(cudaGetLastError());
  return 0;
}

void cube_mel_destroy(cube_mel_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (void* q : {(void*)h->cosT, (void*)h->sinT, (void*)h->basis, (void*)h->k_lo, (void*)h->k_hi, (void*)h->d_len})
    if (q) cudaFree(q);
  delete h;
}

}  // extern "C"
