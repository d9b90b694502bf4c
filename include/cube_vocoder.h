/*
 * cube_vocoder.h - C ABI of libcube_vocoder.so, the B200 (sm_100a) vocoder hot path of TTS-Cube.
 *
 * The reference has no FFI: its boundary is one Python call, `wav = self._generator(cond)`
 * (reference cube/networks/cubegan.py:83, cube/io_utils/runtime.py:78) on a module built by
 * `Generator(h)` + `load_state_dict` (+ `remove_weight_norm`) (cube/networks/cubegan.py:41-43,
 * cube/io_utils/runtime.py:51-54).  The entry points below are what a ctypes binding for that
 * call needs; each cites the reference interface it replaces.  INTEGRATION.md shows the binding.
 *
 * Conventions: every function returns 0 on success, non-zero on error (message via
 * cube_voc_last_error(), thread-local).  Device pointers are borrowed, never freed by the library.
 * Work is enqueued on the given cudaStream_t (pass torch.cuda.current_stream().cuda_stream) and is
 * asynchronous unless stated.  One handle per device; a handle is not thread-safe.
 * All tensors are float32, contiguous, channel-first ([B, C, L]) unless stated.
 * There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef CUBE_VOCODER_H_
#define CUBE_VOCODER_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cube_voc cube_voc_t;
typedef void* cube_stream_t; /* cudaStream_t */

enum cube_voc_arch {
  CUBE_VOC_HIFIGAN = 0,     /* hifigan/models.py:Generator (Path H)                               */
  CUBE_VOC_PWN_STUDENT = 1, /* ClariNet IAF student + UpsampleNet2 (Path C), weights-only in ref  */
  CUBE_VOC_WAVERNN = 2,     /* cube/networks/modules.py:WaveRNN (Path W), autoregressive          */
  CUBE_VOC_UPSAMPLENET = 3  /* cube/networks/modules.py:317-343 UpsampleNet: 3 x (Conv1d k + tanh), then per scale s a
                             * weight-normed ConvTranspose1d(2s, stride s, padding s/2) + tanh.  Config: num_mels = in_channels,
                             * res_channels = out_channels, kernel_size (odd), n_upsample / upsample_scales (even scales).
                             * cube_voc_forward(mel [B, in, F]) writes `wav` as [B, out_channels, F * prod(scales)];
                             * cube_voc_out_len = F * prod(scales) */
};

/* 'beta' (cube/networks/loss.py:69-106, selectable at modules.py:436-437) is NOT supported: its sample() draws from
 * torch.distributions.Beta (rejection sampling inside torch), which cannot be replayed from injected draws; the Python
 * layer raises CubeVocError for output='beta' */
enum cube_wavernn_head { CUBE_HEAD_MOL = 0, CUBE_HEAD_GM = 1, CUBE_HEAD_MULAW = 2, CUBE_HEAD_RAW = 3 };

enum cube_voc_math {
  CUBE_MATH_FP32_SIMT = 0,  /* fp32 FFMA everywhere                                                */
  CUBE_MATH_TC_SPLIT16 = 1  /* tcgen05 tensor cores, error-compensated split-fp16 x3, fp32 accum   */
};

#define CUBE_MAX_UPS 8
#define CUBE_MAX_RBK 8
#define CUBE_MAX_DIL 8
#define CUBE_MAX_FLOWS 8

/* Mirrors the keys of hifigan/config_v*.json that Generator.__init__ reads
 * (hifigan/models.py:72-98) and, for Path C, the module tree of the shipped checkpoints
 * (SURVEY Appendix C). */
typedef struct cube_voc_config {
  uint32_t struct_size; /* = sizeof(cube_voc_config) of the header the caller was built against: cube_voc_create rejects
                         * any other value, so a binding whose struct has drifted from this header (a missing or extra
                         * field) fails loudly instead of having the library read past the caller's struct */
  int32_t arch;  /* enum cube_voc_arch */
  int32_t math;  /* enum cube_voc_math */
  int32_t num_mels; /* 80 */
  /* ---- HiFi-GAN ---- */
  int32_t upsample_initial_channel;
  int32_t n_ups;
  int32_t upsample_rates[CUBE_MAX_UPS];
  int32_t upsample_kernel_sizes[CUBE_MAX_UPS];
  int32_t resblock_type; /* 1 or 2 */
  int32_t n_resblock_kernels;
  int32_t resblock_kernel_sizes[CUBE_MAX_RBK];
  int32_t n_dilations[CUBE_MAX_RBK];
  int32_t resblock_dilations[CUBE_MAX_RBK][CUBE_MAX_DIL];
  /* ---- ClariNet student ---- */
  int32_t n_flows;
  int32_t flow_blocks[CUBE_MAX_FLOWS];
  int32_t res_channels, gate_channels, skip_channels; /* 128, 256, 128 */
  int32_t kernel_size, front_kernel;                  /* 3, 32 */
  int32_t dilation_base, dilation_cycle;              /* 3, 6 : d_i = base^(i mod cycle) */
  int32_t n_upsample;
  int32_t upsample_scales[4];                         /* 16, 16 */
  /* ---- WaveRNN (cube/networks/modules.py:393-446 constructor arguments) ---- */
  int32_t wrnn_layers, wrnn_size;                     /* num_layers (1|2), layer_size */
  int32_t wrnn_upsample, wrnn_upsample_low;           /* upsample, upsample_low */
  int32_t wrnn_use_lowres;                            /* use_lowres */
  int32_t wrnn_head;                                  /* enum cube_wavernn_head ('mol','gm','mulaw','raw') */
} cube_voc_config;

/* Generator(h) / Wavenet_Student(...) constructor.  device = CUDA ordinal.  cfg->struct_size must equal
 * sizeof(cube_voc_config). */
int cube_voc_create(cube_voc_t** out, const cube_voc_config* cfg, int device);

/* load_state_dict(): one call per state_dict entry, `name` is the reference's key
 * (e.g. "ups.0.weight_g", "resblocks.3.convs1.0.weight_v", "conv_post.bias",
 * "iafs.2.res_blocks.5.filter_conv.conv.weight_v", "upsample_conv.0.weight_v").
 * `data` is a HOST pointer to float32; weight-norm (weight_g, weight_v) pairs or folded
 * `weight` are both accepted.  A leading "_generator." / "generator." prefix is stripped
 * (cube/networks/cubegan.py:317-319). */
int cube_voc_load_weight(cube_voc_t* h, const char* name, const float* data, const int64_t* shape, int ndim);

/* remove_weight_norm() + repack to the kernels' layouts + upload (hifigan/models.py:118-125).
 * Fails if a key the architecture needs is missing or has the wrong shape (strict). */
int cube_voc_finalize(cube_voc_t* h);

/* T = f(F): ConvTranspose1d length law (hifigan/models.py:84-88) or F * prod(scales). <0 on error */
int64_t cube_voc_out_len(const cube_voc_t* h, int64_t n_frames);

/* generator(cond) - the hot call (hifigan/models.py:100-116; cubegan.py:83).
 *   mel      device [B, num_mels, Fmax]
 *   n_frames HOST   [B] valid frames per utterance, or NULL (= all Fmax).  Utterance b is computed
 *            exactly as if run alone at its own length; samples past its end are written as 0.
 *   noise    device [B, 1, Tmax] z ~ N(0,1) for the IAF student (required there), NULL for HiFi-GAN
 *   wav      device [B, 1, Tmax], Tmax = cube_voc_out_len(h, Fmax)
 *   wav_i16  device [B, Tmax] int16 or NULL: fused `audio*32767 -> int16` (cube/api.py:65)
 */
int cube_voc_forward(cube_voc_t* h, const float* mel, const int32_t* n_frames, const float* noise,
                     float* wav, int16_t* wav_i16, int B, int64_t Fmax, cube_stream_t stream);

/* Streaming geometry of a HiFi-GAN config (no handle, no device): the mel frames [*f0, *f1) that output samples [s0, s1)
 * depend on, by exact interval propagation through conv_pre, every ConvTranspose1d (input i reaches outputs i*u - pad + j,
 * j < K) and ResBlock step, and conv_post.  *f0 is clipped at 0 (earlier rows are zero padding); *f1 is not clipped above,
 * so a caller holding N frames may emit [s0, s1) once *f1 <= N.  Fails for other archs and for s0 < 0 or s0 >= s1. */
int cube_voc_hifigan_support(const cube_voc_config* cfg, int64_t s0, int64_t s1, int64_t* f0, int64_t* f1);

/* cube_voc_forward for HiFi-GAN handles that writes only samples [out_begin[b], out_end[b]) of item b (HOST arrays [B]);
 * every other element of wav / wav_i16 is left untouched.  Same arguments and layout as cube_voc_forward.  The requested
 * samples are bit-identical to what cube_voc_forward computes for the same mel: every launch schedules only the rows its
 * consumers read (tensor-core path), and no row's arithmetic depends on the tile it falls in.  Fails for other archs and
 * for a range that is empty or outside [0, cube_voc_out_len(n_frames[b])). */
int cube_voc_forward_range(cube_voc_t* h, const float* mel, const int32_t* n_frames, const int64_t* out_begin,
                           const int64_t* out_end, float* wav, int16_t* wav_i16, int B, int64_t Fmax, cube_stream_t stream);

/* Same call with HOST buffers (pinned or pageable): H2D of mel/noise, forward, D2H of the audio;
 * synchronous.  This is the end-to-end form of `cube(text)`'s vocoder leg
 * (cube/api.py:60-65: .to(device) ... .detach().cpu().numpy(), *32767 -> int16).
 * Exactly one of wav / wav_i16 may be NULL. */
int cube_voc_forward_host(cube_voc_t* h, const float* mel, const int32_t* n_frames, const float* noise,
                          float* wav, int16_t* wav_i16, int B, int64_t Fmax);

/* WaveRNN._inference (cube/networks/modules.py:453-503): the autoregressive sample loop as one persistent
 * cooperative kernel.  Handle created with arch = CUBE_VOC_WAVERNN; weights by the reference's state_dict keys
 * ("_rnns.0.weight_ih_l0", "_lowres_conv.1.conv.weight", "_preoutput.linear_layer.bias", ...).
 *   mel    device [B, F, 80]  (time-major, as WaveRNN takes it)
 *   x_low  device [B, Tl] low-rate waveform, or NULL when use_lowres = 0
 *   draws  device [T][B][K]: the sampling head's random numbers, K = nr_mix+1 uniforms in (1e-5, 1-1e-5)
 *          (MOL: mixture pick then logistic), 1 normal (GM), or sample_size uniforms (MULAW/RAW, Gumbel-max)
 *   x      device [B, T], T = cube_wavernn_out_len(h, F, Tl) = min(F*upsample, Tl*upsample_low)
 * B is limited by shared memory (20 at layer_size 512); the Python layer splits larger batches. */
int64_t cube_wavernn_out_len(const cube_voc_t* h, int64_t n_frames, int64_t n_low);
int cube_wavernn_forward(cube_voc_t* h, const float* mel, const float* x_low, const float* draws, float* x,
                         int B, int64_t F, int64_t Tl, cube_stream_t stream);
int cube_wavernn_max_batch(const cube_voc_t* h);

/* Debug/validation tap for Path C: upsampled conditioning c_up [B, 80, Tmax] of the last forward
 * (UpsampleNet2, cube/networks/modules.py:357-375).  Copies to a device buffer. */
int cube_voc_get_cond(cube_voc_t* h, float* c_up, int B, int64_t Tmax, cube_stream_t stream);

/* Kernel launches issued by the last cube_voc_forward on this handle; bytes of workspace held. */
int64_t cube_voc_last_launches(const cube_voc_t* h);
int64_t cube_voc_workspace_bytes(const cube_voc_t* h);
/* Device time (ms, CUDA events on the forward's stream) of each layer class of the last forward
 * when profiling is enabled with cube_voc_set_profile(h, 1): fills up to `cap` (name[64], ms) pairs
 * and returns how many were written (>= 0), or -1 on error. */
int cube_voc_set_profile(cube_voc_t* h, int on);
int cube_voc_get_profile(cube_voc_t* h, char* names /*cap*64*/, float* ms, int cap);

void cube_voc_destroy(cube_voc_t* h);
const char* cube_voc_last_error(void);
/* "sm_100a" and library version; never fails */
const char* cube_voc_build_info(void);

/* ---- output heads (cube/networks/loss.py) : element-wise, device pointers ---- */
/* MULAWOutput.encode (loss.py:236-254): float32 -> int64 codes 0..255, BIT-EXACT with the
 * reference's float32 torch path (bin-edge table derived from it). */
int cube_mulaw_encode(const float* x, int64_t* q, int64_t n, cube_stream_t stream);
/* MULAWOutput.decode (loss.py:256-269): int64 codes -> float32 (table of the reference's values) */
int cube_mulaw_decode(const int64_t* q, float* x, int64_t n, cube_stream_t stream);
/* RAWOutput.encode/decode (loss.py:293-299) */
int cube_raw_encode(const float* x, int64_t* q, int64_t n, cube_stream_t stream);
int cube_raw_decode(const int64_t* q, float* x, int64_t n, cube_stream_t stream);
/* MOLOutput.sample (loss.py:163-201) with injected uniforms: y [N, 3*nr_mix], u_mix [N, nr_mix],
 * u_x [N] in U(1e-5, 1-1e-5) -> x [N] in [-1, 1] */
int cube_mol_sample(const float* y, const float* u_mix, const float* u_x, float* x, int64_t n,
                    int nr_mix, float log_scale_min, float temperature, cube_stream_t stream);
/* GaussianOutput.sample (loss.py:50-52) with injected normals: y [N,2], eps [N] -> x [N] */
int cube_gaussian_sample(const float* y, const float* eps, float* x, int64_t n, cube_stream_t stream);
/* Categorical(logits).sample() for MULAW/RAW (loss.py:227-229, 288-290) in Gumbel-max form with
 * injected uniforms: logits [N, C], u [N, C] in [0, 1) -> idx [N] int64 = argmax(logits - log(-log u)).
 * DISTRIBUTION-equivalent to the reference's sampler (chi-square tested against softmax(logits) and against
 * torch's Categorical), not replayable draw for draw: torch consumes its generator differently.  Feed full-range
 * uniforms - a truncated range such as (1e-5, 1 - 1e-5) caps the Gumbel noise and starves the rare classes. */
int cube_categorical_sample(const float* logits, const float* u, int64_t* idx, int64_t n, int C,
                            cube_stream_t stream);
/* cube/api.py:65: int16(audio * 32767), truncation toward zero */
int cube_wav_to_int16(const float* wav, int16_t* out, int64_t n, cube_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Log-mel spectrogram on the device (SURVEY 8(f)3): the feature front-end of the "gold mel" callers.
 * Replaces hifigan/meldataset.py:50-74 mel_spectrogram() (hifigan/inference.py:26, cube/networks/cubegan.py:137)
 * and cube/io_utils/vocoder.py:54-62 MelVocoder.melspectrogram() (cube/io_utils/io_vocoder.py:56).
 * The mel filter bank is an input (the reference gets it from librosa.filters.mel on the host).
 * ------------------------------------------------------------------------------------------- */
typedef struct cube_mel cube_mel_t;

typedef struct cube_mel_config {
  uint32_t struct_size; /* = sizeof(cube_mel_config); checked by cube_mel_create like cube_voc_config.struct_size */
  int32_t n_fft;      /* 1024; multiple of 4 */
  int32_t win_size;   /* <= n_fft (centred zero padding like torch.stft) */
  int32_t hop_size;   /* 240 / 256; multiple of 4 */
  int32_t n_mels;     /* 80 */
  int32_t pad_left;   /* reflect padding: (n_fft-hop)/2 for meldataset.py:62, n_fft/2 for librosa center=True */
  int32_t pad_right;
  int32_t log10_out;  /* 0: ln (meldataset.py:19-20)   1: log10 (io_utils/vocoder.py:96-98) */
  int32_t layout;     /* 0: [B, n_mels, F] (HiFi-GAN)  1: [B, F, n_mels] (MelVocoder / WaveRNN, time-major) */
  int32_t pad_mode;   /* 0: reflect (meldataset.py:62; librosa < 0.10 stft default)  1: constant zeros (librosa >= 0.10 stft
                       * default pad_mode; the reference does not pin librosa, cube/io_utils/vocoder.py:71-73) */
  float mag_eps;      /* sqrt(re^2 + im^2 + eps): 1e-9 in meldataset.py:70, 0 for np.abs */
  float floor_val;    /* clamp before the log: 1e-5 */
  float pad_value;    /* written to frames beyond an utterance's own frame count in a ragged batch */
  float preemph;      /* 0, or 0.97 = MelVocoder._preemphasis (io_utils/vocoder.py:64-65) */
} cube_mel_config;

/* window: host [win_size] or NULL = periodic Hann (torch.hann_window / scipy 'hann', fftbins=True);
 * mel_basis: host [n_mels][n_fft/2 + 1], row-major. */
int cube_mel_create(cube_mel_t** out, const cube_mel_config* cfg, const float* window, const float* mel_basis, int device);
/* frames of an utterance of n_samples samples (0 when reflect padding is impossible: n_samples <= pad) */
int64_t cube_mel_out_frames(const cube_mel_t* h, int64_t n_samples);
/* wav: device [B, Tmax]; n_samples: HOST [B] or NULL (= Tmax each); mel: device, Fmax frames per utterance
 * (Fmax >= cube_mel_out_frames(max n_samples)); rows beyond an utterance's frame count hold pad_value. */
int cube_mel_forward(cube_mel_t* h, const float* wav, const int32_t* n_samples, float* mel, int B, int64_t Tmax,
                     int64_t Fmax, cube_stream_t stream);
void cube_mel_destroy(cube_mel_t* h);

#ifdef __cplusplus
}
#endif
#endif /* CUBE_VOCODER_H_ */
