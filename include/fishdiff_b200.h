/* fishdiff_b200.h -- C ABI of the B200-native fish-diffusion hot path (libfishdiff_b200.so).
 *
 * The reference (fishaudio/fish-diffusion @ 8e8f8cd) contains no native code (SURVEY.md section 2.1): its
 * hot path is PyTorch library dispatch.  This library is what a maintainer binds (ctypes, see
 * INTEGRATION.md) behind the reference's own Python classes; each entry point cites the reference
 * computation it replaces.  Conventions:
 *   - plain pointers + sizes, no torch types; all pointers are DEVICE pointers unless named host_*;
 *   - the caller owns every buffer including workspaces; functions never allocate and never synchronise;
 *   - every function is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return 0 on success, negative on error; fd_last_error() returns the message (thread-local);
 *   - activations are channels-last "split planes" (fd_common.cuh): uint16 planes[2][B][T][C],
 *     value = hi + lo, `prec` = FD_PREC_F16 (22-bit mantissa) or FD_PREC_BF16 (16-bit mantissa);
 *   - `backend`: FD_BACKEND_TC = tcgen05/TMEM/TMA tensor-core kernel (sm_100a),
 *                FD_BACKEND_SIMT = fp32 CUDA-core twin (device-side checker / uncovered shapes).
 *     There is no CPU path in this library.
 */
#ifndef FISHDIFF_B200_H
#define FISHDIFF_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FD_PREC_F16 0
#define FD_PREC_BF16 1
/* or-ed into the `prec` of a GEMM entry point (fd_wavenet_block_fwd*, fd_conv_cl_fwd, fd_gemm_cl_fwd,
 * fd_stft_mag_fwd): multiply the hi planes only -- one tensor-core product per k-step instead of three, i.e. plain
 * half-precision operands (11-bit / 8-bit mantissa) with fp32 accumulation.  Storage stays two planes. */
#define FD_PREC_SINGLE 0x10
#define FD_BACKEND_TC 0
#define FD_BACKEND_SIMT 1
#define FD_ABI_VERSION 2

/* ------------------------------------------------------------------------------------------- misc */
int fd_abi_version(void);
const char* fd_last_error(void);
/* Device the caller's buffers live on (thread-local; -1 = "whatever is current", the default).  Every entry point
 * makes it the current CUDA device for the duration of the call and restores the caller's device afterwards, so a
 * module on cuda:N works without torch.cuda.set_device (the reference relies on PyTorch's per-tensor device
 * dispatch for the same thing, e.g. `model.to(device)` in tools/diffusion/inference.py:57-60).  Per-device state
 * (SM count, dynamic shared-memory attributes) is cached per device. */
void fd_set_device(int device);
/* number of kernel launches issued by this library since process start (bench.py "gpu_launches") */
long long fd_launch_count(void);
/* per-launch device timing of the tap-GEMM kernels (CUDA events on the launching stream), used by bench.py for
 * the roofline entry: kind = epilogue*2 + (backend==SIMT); epilogue 0 linear, 1 gate (WaveNet GEMM1),
 * 2 res/skip (WaveNet GEMM2), 3 DFT magnitude; kind 8 = gate backward fused into the dz GEMM; kinds 12..15 = fused ResBlock pair kernel at C = 128/64/32/16.  fd_prof_collect synchronises the device, fills ms_sum[k]/count[k]
 * for k < nkinds, resets the log and returns 1 if the log overflowed (65536 launches), 0 otherwise, <0 on error. */
void fd_prof_enable(int on);
int fd_prof_collect(double* ms_sum, long long* count, int nkinds);
/* 1 if tensor-core instantiation exists for the given linear tap-GEMM shape */
int fd_tc_supported_linear(int n_total, int k_seg, int num_seg);

/* ------------------------------------------------------------------------------ layout / packing */
/* fp32 [B,C,T] (reference NCW layout, wavenet.py:194 `x: [B, M, T]`) -> split planes [2][B][T][C];
 * rows with mask[b,t]!=0 are zeroed (wavenet.py:217-221 masked_fill). mask may be NULL. */
int fd_split_ncw(const float* src, const uint8_t* mask, uint16_t* planes, int B, int C, int T, int prec,
                 void* stream);
/* fp32 [B,T,C] channels-last -> split planes; value*scale; optional row mask */
int fd_split_nwc(const float* src, const uint8_t* mask, uint16_t* planes, int B, int T, int C, float scale,
                 int prec, void* stream);
/* Multi-receptive-field average + LeakyReLU in front of the next upsampling stage / conv_post (models.py:420,426-434):
 *   out planes [2][n] = split( lrelu( (sum_{i<num} x_i) * scale, out_slope ) ),  x_i = inverse-lrelu(in_i planes, in_slope)
 * in[i]: planes [2][n] holding lrelu(x_i, in_slope) (the outputs of the last fused pair of each ResBlock), num <= 4. */
int fd_mrf_finish(const uint16_t* const* in, int num, uint16_t* out, long long n, float in_slope, float scale,
                  float out_slope, int prec, void* stream);
/* fp32 [B,T,C] -> fp32 [B,C,T] and back (boundary transposes of the drop-in WaveNet.forward) */
int fd_transpose_nwc_to_ncw(const float* src, float* dst, int B, int T, int C, void* stream);
int fd_transpose_ncw_to_nwc(const float* src, float* dst, int B, int C, int T, void* stream);
/* fp32 weight matrix [N][K] -> split planes [2][N][K] of (w*scale) */
int fd_pack_weight(const float* w, uint16_t* planes, long long n_elems, float scale, int prec, void* stream);

/* All residual layers of a WaveNet packed in two launches from the raw parameters (device pointer tables of L entries:
 * conv weight [2C][C][3], conditioner weight [2C][E], output-projection weight [2C][C]; modules/wavenet.py:88-104).
 *   w1p_f32 [L][2C][3C+E]   fp32, rows in gate/filter-interleaved order (tile = 2*gate_half), K = tap0|tap1|tap2|cond
 *   w1 [L][2][2C][3C+E], w2 [L][2][2C][C]                     forward packs, scaled by scales[l] / scales[L+l]
 *   w1t [L][2][C][6C], wct [L][2][E][2C], w2t [L][2][C][2C]   transposed packs of the data-gradient GEMMs (all three or
 *                                                             all NULL); the residual half of w2t carries 1/sqrt2 */
int fd_wavenet_pack_layers(const float* const* conv_w, const float* const* cond_w, const float* const* out_w,
                           const float* scales, float* w1p_f32, uint16_t* w1, uint16_t* w2, uint16_t* w1t, uint16_t* wct,
                           uint16_t* w2t, int L, int C, int E, int gate_half, int prec, void* stream);

/* ------------------------------------------------------------------------- WaveNet denoiser (a10-a12) */
/* DiffusionEmbedding + mlp (wavenet.py:13-27,170-174,214-215): steps[Bs] (float; int steps are cast by
 * the caller exactly like `x[:, None] * emb`) -> s[Bs][C].
 * w0 [4C][C], b0 [4C] (may be NULL), w1 [C][4C], b1 [C] (may be NULL); ws: workspace Bs*5C floats. */
int fd_wavenet_step_mlp(const float* steps, const float* w0, const float* b0, const float* w1, const float* b1,
                        float* s_out, float* ws, int Bs, int C, void* stream);
/* Per-layer diffusion_projection (wavenet.py:107) folded into the gate bias of the fused block:
 *   d_l = Wd[l] s + bd[l];  full = bias_sum[l] + sum_tap W1p[l][:, tap*C:(tap+1)*C] d_l ; lo/hi = tap 0 / tap 2 term.
 * wd [L][C][C], bd [L][C] or NULL, w1p fp32 packed [L][2C][KT] (KT = 3C+E), bias_sum [L][2C] packed order.
 * outputs gb_full/gb_lo/gb_hi [L][Bs][2C]; ws: L*Bs*C floats. */
int fd_wavenet_gate_bias(const float* s, const float* wd, const float* bd, const float* w1p, const float* bias_sum,
                         float* gb_full, float* gb_lo, float* gb_hi, float* ws, int L, int Bs, int C, int KT,
                         void* stream);
/* One complete WaveNet.forward (wavenet.py:194-236) on channels-last split planes as ONE native call: step MLP,
 * gate-bias tables, input projection, L residual blocks, skip / output projections -- the launches of
 * fd_wavenet_step_mlp, fd_wavenet_gate_bias, fd_conv_cl_fwd and L x fd_wavenet_block_fwd issued back to back on
 * `stream` (capturable into a CUDA graph: nothing here synchronises or allocates).  Replaces the per-layer Python loop of
 * the reference (`for layer in self.residual_layers`, wavenet.py:223-226) and its ~245 kernel launches per call.
 * Host arrays: w1_inv / w2_inv / dilation [L].  w1 / w2 / b2 are [L] stacks with the given element strides. */
typedef struct fd_wavenet_fwd_desc {
  const uint16_t* x_planes;     /* [2][B][T][M] */
  const uint16_t* cond_planes;  /* [2][B][T][E] */
  const float* cond_term;       /* NULL, or the conditioner projections of fd_wavenet_cond_term [L][B][T][2C]: each GEMM1
                                   then multiplies only the three conv taps (K = 3C) and adds its layer's slice */
  const float* steps;           /* [Bs] diffusion steps (float), Bs = 1 or B */
  const uint8_t* x_mask;        /* [B][T] or NULL (wavenet.py:217-218, 233-234) */
  float* out;                   /* eps fp32 [B][T][M] */
  /* packed weights (WaveNet._packed) */
  const uint16_t* w_in; const float* b_in; float w_in_inv;
  const float* mlp_w0; const float* mlp_b0; const float* mlp_w1; const float* mlp_b1;
  const float* wd; const float* bd; const float* w1p_f32; const float* bias_sum;
  const uint16_t* w1; long long w1_lstride;
  const uint16_t* w2; long long w2_lstride;
  const float* b2; long long b2_lstride;
  const uint16_t* w_skip; const float* b_skip; float w_skip_inv;
  const uint16_t* w_out; const float* b_out; float w_out_inv;
  float w1_inv[64], w2_inv[64];
  int dilation[64];
  /* workspace (caller-owned, see WaveNet._workspace) */
  uint16_t* xr; uint16_t* z; uint16_t* skip_planes; float* skip_f32;
  float* s; float* mlp_ws; float* gb; float* gb_ws;
  int B, T, M, C, E, L, Bs;
  int gate_tile, prec, backend;
} fd_wavenet_fwd_desc;
int fd_wavenet_fwd(const fd_wavenet_fwd_desc* d, void* stream);

/* Conditioner projection of every residual layer, computed once for all evaluations of a sampler call (cond does not
 * change between them):  cond_term[l][b][t][n] = sum_e W1[l][n][3C + e] * cond[b][t][e] * w1_inv[l]  (fp32, the packed
 * gate/filter column order of w1, no bias: the conditioner bias is part of the gate-bias table).  One linear tap-GEMM
 * per layer over the conditioner columns of the same packed w1 [L][2][2C][3C+E] that fd_wavenet_fwd reads.
 * w1_inv: host array [L].  Rows that were zeroed in cond_planes give zeros. */
int fd_wavenet_cond_term(const uint16_t* cond_planes, const uint16_t* w1, long long w1_lstride, const float* w1_inv,
                         float* cond_term, int L, int B, int T, int C, int E, int prec, int backend, void* stream);

/* One ResidualBlock.forward (wavenet.py:106-120), fused as two tap-GEMM launches:
 *   GEMM1  y = [W_conv(3 taps) | W_cond] . [x(t-d), x(t), x(t+d), cond(t)] + gate bias ; z = sigmoid(y_g)*tanh(y_f)
 *   GEMM2  o = W_out z + b ;  x <- (x + o_res)/sqrt(2) (in place) ;  skip_acc (+)= o_skip
 * x_planes [2][B][T][C] in/out, cond_planes [2][B][T][E], z_planes workspace [2][B][T][C],
 * w1 planes [2][2C][3C+E] (gate/filter rows interleaved per `gate_tile`), w2 planes [2][2C][C],
 * gb_* [Bs][2C] for this layer (gb_bstride = 2C if per-item steps else 0), b2 [2C],
 * skip_f32 [B][T][C] accumulator; flags bit0 = first layer (skip written, not accumulated),
 * bit1 = last layer (skip_planes <- split((skip_f32 + o_skip) * skip_scale), x not updated). */
int fd_wavenet_block_fwd(uint16_t* x_planes, const uint16_t* cond_planes, uint16_t* z_planes,
                         const uint16_t* w1, const uint16_t* w2, const float* gb_full, const float* gb_lo,
                         const float* gb_hi, int gb_bstride, const float* b2, float* skip_f32,
                         uint16_t* skip_planes, float skip_scale, int B, int T, int C, int E, int dilation,
                         int gate_tile, float w1_inv_scale, float w2_inv_scale, int flags, int prec, int backend,
                         void* stream);

/* --------------------------------------------------------------- generic channels-last conv / linear */
/* out[b,t,n] = post( sum_j sum_c in[b, t + shifts[j], c] * w[n, j*Cin + c] * w_inv_scale + bias[n]
 *                    + addend[b,t,n] + res ) ; see FdTapGemm in csrc/fd_common.cuh for the exact epilogue.
 * Used for: WaveNet input/skip/output projections (wavenet.py:211-212,229-231), NSF-HiFiGAN conv_pre,
 * ResBlock1 convs (models.py:103-110), polyphase ConvTranspose1d (models.py:421), mel filterbank. */
typedef struct fd_conv_desc {
  const uint16_t* in_planes; /* [2][B][T][Cin] */
  const uint16_t* w_planes;  /* [2][N][ntaps*Cin] */
  const float* bias;         /* [N] or NULL */
  const float* addend;       /* fp32 [B][T][N] or NULL */
  const float* res_f32;      /* fp32 [B][T][N] or NULL */
  const uint16_t* res_planes;/* [2][B][T][N] or NULL */
  const uint8_t* row_mask;   /* [B][T] or NULL */
  float* out_f32;            /* [B][T][N] or NULL */
  uint16_t* out_planes;      /* [2][B][T][N] or NULL */
  int B, T, Cin, N;
  int ntaps;
  int shifts[16];
  float w_inv_scale, post_scale, planes_scale, act_slope;
  int out_accum;             /* out_f32 += */
  int act;                   /* 0 none, 1 relu, 2 leaky-relu(act_slope): applied to the planes output only */
  int prec, backend;
} fd_conv_desc;
int fd_conv_cl_fwd(const fd_conv_desc* d, void* stream);

/* One iteration of ResBlock1.forward (models.py:103-110), fused into ONE kernel:
 *     x' = x + c2( lrelu( c1( lrelu(x) ) , 0.1) )
 * c1: Conv1d(C->C, k1 taps, dilation d1, 'same'), c2: Conv1d(C->C, k2 taps, dilation 1, 'same').
 * in_planes holds lrelu(x, in_slope) as split planes [2][B][T][C]; the residual x is recovered in the kernel by
 * inverting the LeakyReLU (in_slope > 0), so no fp32 master of the residual stream exists in HBM.
 * out_planes [2][B][T][C] = split( lrelu(x', out_slope) * planes_scale )  (input of the next pair / of fd_mrf_finish).
 * w1/w2: packed weights [2][C][k*C] (tap-major K, as fd_pack_weight makes them), b1/b2 fp32 [C].
 * The c1 output lives only in shared memory; HBM traffic is 4 B/element in + 4 B/element out.
 * C in {16,32,64,128}; (k1-1)*d1 <= 56; k2 <= 17 (fd_respair_supported).  Out of place only. */
typedef struct fd_respair_desc {
  const uint16_t* in_planes;
  const uint16_t* w1;
  const uint16_t* w2;
  const float* b1;
  const float* b2;
  uint16_t* out_planes;
  int B, T, C;
  int k1, d1, k2;
  float w1_inv_scale, w2_inv_scale;
  float in_slope, out_slope, planes_scale;
  int prec;
  /* optional block-sparsity hint (0 = dense): bit tap*(C/16) + s set <=> the 16 input channels [16s, 16s+16) of that
   * tap hold a non-zero weight.  Slices without a bit are neither loaded (whole weight units) nor multiplied; used by
   * the time-folded C = 16 stage, whose folded kernels are block-sparse.  Ignored when k*(C/16) > 64. */
  unsigned long long kmask1, kmask2;
} fd_respair_desc;
int fd_respair_supported(int C, int k1, int d1, int k2);
int fd_respair_fwd(const fd_respair_desc* d, void* stream);

/* ------------------------------------------------------------------------- sampler (a5-a9, K10-K12) */
/* NaiveNoisePredictor.forward (noise_predictor.py:73-104):
 *   x0 = c_recip*x - c_recipm1*eps ; clamp ; mean = c1*x0 + c2*x ; x' = mean + sigma*noise
 * sigma = [t>0]*exp(0.5*logvar_t) computed by the caller from the bit-exact tables.
 * noise: injected N(0,1) tensor or NULL -> in-kernel Philox4x32-10: elements 4i..4i+3 are the normal4 draw of
 *   (seed, subsequence subseq0 + i, offset).  subseq0 = index of the first element / 4 inside the GLOBAL batch, so a
 *   batch sharded over ranks (or split into calls) draws exactly the noise of the unsharded run.
 * writes x_out (fp32, may alias x) and optionally split planes of x' for the next denoiser call. */
int fd_ddpm_step(const float* x, const float* eps, const float* noise, float* x_out, uint16_t* x_planes,
                 long long n, float c_recip, float c_recipm1, float c1, float c2, float sigma, float clip_min,
                 float clip_max, unsigned long long seed, unsigned long long offset, unsigned long long subseq0,
                 int prec, void* stream);
/* out = sum_i coef[i] * in[i]  (PLMS noise_predictor.py:118-148, UniPC uni_pc.py:664-680 updates);
 * nterms <= 6; optionally also writes split planes. in[i] may alias out. */
int fd_lincomb(float* out, uint16_t* out_planes, const float* const* host_in_ptrs, const float* host_coefs,
               int nterms, long long n, int prec, void* stream);
/* y = x*scale[c] + shift[c] over channels-last [rows][C] (norm_spec/denorm_spec diffusion.py:315-319);
 * scale/shift have length C or 1 (nparam). */
int fd_affine_cl(const float* x, float* y, const float* scale, const float* shift, int nparam, long long rows,
                 int C, void* stream);
/* q_sample (diffusion.py:120-127): y = a[b]*x + s[b]*noise, a/s per batch item (device arrays [B]) */
int fd_q_sample(const float* x, const float* noise, const float* a, const float* s, float* y, int B,
                long long per_item, void* stream);
/* fill with N(0,1) from Philox4x32-10 (same indexing as fd_ddpm_step) */
int fd_randn(float* out, long long n, unsigned long long seed, unsigned long long offset, unsigned long long subseq0,
             void* stream);

/* --------------------------------------------------------------- NSF-HiFiGAN source module (a15) */
/* Generator.forward f0 upsample + SourceModuleHnNSF (models.py:411-415, 201-294, 337-350):
 * f0 [B][T] frames -> har [B][T*hop] (fp32).  9 harmonics, phase accumulated exactly (64-bit fixed
 * point scan), sine_amp 0.1, noise_std 0.003.  lin_w[H], lin_b[1] = m_source.l_linear.
 * rand_ini [B][H] (rand_ini[:,0] must be 0) ; noise [B][S][H] injected N(0,1) or NULL -> Philox.
 * ws: workspace, fd_sinegen_ws_bytes(B, T*hop) bytes. */
size_t fd_sinegen_ws_bytes(int B, long long S);
int fd_sinegen_fwd(const float* f0, const float* lin_w, const float* lin_b, const float* rand_ini,
                   const float* noise, float* har, void* ws, int B, int T, int hop, int H, float sampling_rate,
                   float sine_amp, float noise_std, unsigned long long seed, void* stream);
/* noise_convs[i] (models.py:380-393,422): Conv1d(1 -> C, kernel k, stride s, padding p) over har [B][S]
 * -> fp32 channels-last [B][S_out][C],  S_out = (S + 2p - k)/s + 1 */
int fd_source_conv_fwd(const float* har, const float* w /*[C][k]*/, const float* bias /*[C]*/, float* out,
                       int B, long long S, int C, int k, int s, int p, void* stream);
/* conv_post + tanh (models.py:434-436): in planes [2][B][S][C] (already leaky-relu'd by the producer)
 * -> wav [B][S];  w [k][C], bias[1] */
int fd_conv_post_fwd(const uint16_t* in_planes, const float* w, const float* bias, float* wav, int B,
                     long long S, int C, int k, int prec, void* stream);

/* ------------------------------------------------------------------------ mel front end (a19-a20) */
/* reflect-pad + split: wav [B][N] -> planes [2][B][Np] with Np = N + 2*pad (pitch_adjustable_mel.py:61-69) */
int fd_reflect_pad_split(const float* wav, uint16_t* planes, int B, long long N, int pad, int prec, void* stream);
/* framed DFT magnitude as a tap-GEMM over overlapping frames (pitch_adjustable_mel.py:71-83):
 * padded planes [2][B][Np], frames = (Np - n_fft)/hop + 1, dft_w planes [2][2*NB][n_fft] (window folded in,
 * rows interleaved re/im per 256-column tile, NB = padded bin count, multiple of 128)
 * -> mag planes [2][B][frames][NB] of sqrt(re^2+im^2+1e-9)*mag_scale */
int fd_stft_mag_fwd(const uint16_t* padded, const uint16_t* dft_w, uint16_t* mag_planes, int B, long long Np,
                    int n_fft, int hop, int frames, int NB, float w_inv_scale, float mag_scale, int prec,
                    int backend, void* stream);
/* same with an explicit epsilon inside the square root: 0 for torchaudio's Spectrogram(power=1) used by
 * utils/audio.py:31-109 (get_mel_transform / get_mel_from_audio), 1e-9 for pitch_adjustable_mel.py:85 */
int fd_stft_mag_eps_fwd(const uint16_t* padded, const uint16_t* dft_w, uint16_t* mag_planes, int B, long long Np,
                    int n_fft, int hop, int frames, int NB, float w_inv_scale, float mag_scale, float mag_eps, int prec,
                    int backend, void* stream);
/* log(clamp(x, clip)) * out_scale over fp32 (audio.py:11-18 dynamic_range_compression) */
int fd_log_clamp(const float* x, float* y, long long n, float clip, float out_scale, void* stream);

/* ------------------------------------------------------------------ training step (a8): backward of the denoiser */
/* General linear tap-GEMM: up to two source tensors, explicit source strides (0 = canonical [2][B][T][C]), a K offset
 * on the W operand (w_kshift + b*w_bstride_k).  It expresses every gradient GEMM of the WaveNet backward:
 *   data gradients: transposed packed weights, mirrored tap shifts, two sources ([dx_next | d_skip]);
 *   weight gradients: src = folded transpose of the output gradient ("rows" = output channels, C = padded time),
 *                     W = folded transpose of the forward input, w_kshift = tap shift, w_bstride_k = Tp,
 *                     out_f32 [B][rows][cols] holds one partial per batch item (reduced by fd_reduce_batch).
 * Epilogue = the LINEAR epilogue of fd_conv_cl_fwd plus res_scale on the res_planes term. */
typedef struct fd_gemm_desc {
  const uint16_t* src[2];
  int src_C[2];
  long long src_rs[2], src_bs[2], src_ps[2];
  const uint16_t* w;
  int n_total, k_total, w_kshift;
  long long w_bstride_k;
  int B, T, num_seg;
  int seg_src[16], seg_shift[16], seg_coff[16], seg_klen[16];
  const float* bias;
  const float* addend;
  const float* res_f32;
  const uint16_t* res_planes;
  const uint8_t* row_mask;
  float* out_f32;
  uint16_t* out_planes;
  float w_inv_scale, res_scale, post_scale, planes_scale, act_slope;
  int out_accum, act, prec, backend;
  int bias_bstride;   /* 0: bias [n_total]; n_total: one bias vector per batch item, bias [B][n_total] (per-utterance
                         speaker / pitch-shift embeddings of DiffSinger.forward_features, diffsinger.py:95-121) */
  /* gate backward fused into the epilogue (training; tensor-core back end only): when gate_y != NULL the accumulator is
   * dz [B][T][n_total = C] and the epilogue writes dy = d(sigmoid(g) tanh(f)) (wavenet.py:113-115) for the saved
   * pre-activations gate_y [2][B][T][2C] (packed order of fd_wavenet_block_fwd_train) into out_planes [2][B][T][2C], and
   * adds gate_cs_scale * column sums of dy into gate_cs [B][2C] and -- over the first / last gate_dil steps of each item --
   * gate_cs_edge [2][B][2C] (both zeroed by the caller; may be NULL).  Replaces fd_gate_bwd + fd_colsum + fd_colsum_edges. */
  const uint16_t* gate_y;
  float* gate_cs;
  float* gate_cs_edge;
  float gate_cs_scale;
  int gate_tile, gate_dil;
} fd_gemm_desc;
int fd_gemm_cl_fwd(const fd_gemm_desc* d, void* stream);

/* fd_wavenet_block_fwd for training: the updated residual stream goes to x_out_planes (x_planes stays intact, it is
 * needed by the weight gradient) and the gate/filter pre-activations are kept in y_planes [2][B][T][2C] (packed order). */
int fd_wavenet_block_fwd_train(const uint16_t* x_planes, uint16_t* x_out_planes, const uint16_t* cond_planes,
                               uint16_t* z_planes, uint16_t* y_planes, const uint16_t* w1, const uint16_t* w2,
                               const float* gb_full, const float* gb_lo, const float* gb_hi, int gb_bstride,
                               const float* b2, float* skip_f32, uint16_t* skip_planes, float skip_scale, int B, int T,
                               int C, int E, int dilation, int gate_tile, float w1_inv_scale, float w2_inv_scale,
                               int flags, int prec, int backend, void* stream);
/* gate-bias tables from already projected step vectors d [Bs][L][C] (training: the embedding MLP and the
 * diffusion projections run under torch autograd on [Bs,C]-sized tensors) */
int fd_wavenet_gate_bias_from_d(const float* d, const float* w1p, const float* bias_sum, float* gb_full, float* gb_lo,
                                float* gb_hi, int L, int Bs, int C, int KT, void* stream);
/* planes [2][B][T][C] -> planes [2][C][B][Tp] (item b at columns [pad, pad+T) of its Tp span, zeros elsewhere).
 * mode 0: value*scale (+ addvec[b*add_bstride + c]); mode 1: src is a packed pre-activation tensor with 2C columns,
 * value = sigmoid(g)*tanh(f); mode 2: value = src_f32 * (aux_planes > 0) (ReLU backward).
 * The C rows may be written at row offset dst_row0 of a taller destination with dst_rows rows (stacked operands of the
 * weight-gradient GEMMs); dst_rows <= 0 means dst_rows = C, dst_row0 = 0. */
int fd_fold_transpose(const uint16_t* src_planes, const float* src_f32, const uint16_t* aux_planes, const float* addvec,
                      int add_bstride, uint16_t* dst, int B, int T, int C, int Tp, int pad, float scale, int mode,
                      int gate_tile, int prec, int dst_rows, int dst_row0, void* stream);
/* backward of z = sigmoid(g)*tanh(f) (wavenet.py:114-115): dz fp32 [rows][C], y planes [2][rows][2C] -> dy planes */
int fd_gate_bwd(const float* dz, const uint16_t* y_planes, uint16_t* dy_planes, long long rows, int C, int gate_tile,
                int prec, void* stream);
/* out planes = split(grad * (act_planes > 0) * scale) (ReLU backward, wavenet.py:212,230) */
int fd_relu_bwd(const float* grad, const uint16_t* act_planes, uint16_t* out_planes, long long n, float scale, int prec,
                void* stream);
/* LeakyReLU backward with an optional addend -- autograd of one ResBlock1 iteration `x + c2(lrelu(c1(lrelu(x))))`
 * (nsf_hifigan/models.py:103-110; vocoder training, tools/nsf_hifigan/train.py:114-231):
 *   v = grad * (act > 0 ? 1 : slope) * scale + addend,   act_planes = planes of lrelu(x) (same sign as x)
 * written to out_f32 and / or out_planes (one of them may be NULL); addend may be NULL; n a multiple of 4. */
int fd_lrelu_bwd(const float* grad, const uint16_t* act_planes, const float* addend, float* out_f32,
                 uint16_t* out_planes, long long n, float slope, float scale, int prec, void* stream);
/* out[b][n] += scale * sum_t in[b,t,n]  (bias / step-vector gradients); exactly one of planes / f32 is non-NULL;
 * out must be zero-initialised by the caller */
int fd_colsum(const uint16_t* planes, const float* f32, float* out, int B, int T, int N, float scale, int prec,
              void* stream);
/* out[edge][b][n] += scale * sum_t planes[b,t,n] over t in [0,e) (edge 0) and [T-e,T) (edge 1); out zero-initialised
 * by the caller.  Autograd of `conv_layer(x + diffusion_step)` (modules/wavenet.py:107-111): the step vector d is added
 * before the zero-padded conv, so d(W_tap)/ += (sum over the steps where that tap reads inside [0,T) of dy) (x) d; the
 * sums are the full column sums minus these edge sums. */
int fd_colsum_edges(const uint16_t* planes, float* out, int B, int T, int N, int e, float scale, int prec,
                    void* stream);

/* Weight gradient straight from channels-last split planes, no transposes (tcgen05 with MN-major operands):
 *   part[s][r][c] = acc_scale * sum_{b in split s} sum_t ROW[b,t,r] * COL[b,t+shift(c),c]
 * Rows r are the concatenation of 1..2 row segments, columns c of 1..8 column segments; a segment names a source
 * tensor (planes [2][B][T][C_src]), its first channel, its width (multiple of 64) and -- columns only -- a time shift
 * (rows outside [0,T) read as zero: the conv zero padding of that tap).  Items are divided over `splits` partials
 * (1 <= splits <= B; ceil(B/splits) consecutive items each) which the caller sums with fd_reduce_batch.
 * Replaces autograd's conv-weight gradient of modules/wavenet.py:106-120 (reference runs it through cuDNN wgrad).
 * `prec` may carry FD_PREC_SINGLE. */
typedef struct fd_wgrad_desc {
  const uint16_t* row_src[2];
  int row_C[2];
  const uint16_t* col_src[2];
  int col_C[2];
  int num_row_seg;
  int row_seg_src[2], row_seg_coff[2], row_seg_width[2];
  int num_col_seg;
  int col_seg_src[8], col_seg_shift[8], col_seg_coff[8], col_seg_width[8];
  int B, T, splits;
  float* part;        /* [splits][R][Cc] fp32, R / Cc = total row / column widths */
  float acc_scale;
  int prec;
} fd_wgrad_desc;
int fd_wgrad_cl(const fd_wgrad_desc* d, void* stream);

/* out[i] = scale * sum_b in[b][i]  (reduction of the per-item weight-gradient partials) */
int fd_reduce_batch(const float* in, float* out, int B, long long n, float scale, void* stream);

/* Backward of ONE ResidualBlock (autograd of modules/wavenet.py:106-120) as one native call: the 5 GEMM launches and the
 * elementwise / reduction kernels around them, issued back to back on `stream`:
 *   dz   = [dx_next/sqrt2 | d_skip] . W2            (fd_gemm_cl_fwd, two sources; skip half only above the last layer)
 *   dy   = gate backward of dz on the saved pre-activations (fd_gate_bwd)
 *   gw2  = [dx_next ; d_skip]^T . z                  (fd_wgrad_cl + fd_reduce_batch; the 1/sqrt2 of the residual rows is
 *                                                     applied by the caller to all layers at once)
 *   gw1  = dy^T . [x(t-d) | x(t) | x(t+d) | cond]   (one weight-gradient GEMM, packed row order)
 *   cs_dy / cs_edge = column sums of dy (bias gradient, rank-one step-vector term of gw1)
 *   dx   = conv^T(dy) + dx_next/sqrt2 -> planes (+ fp32 copy when dx_f32 != NULL);  d_cond += dy . Wc;  cs_dx = colsum(dx)
 * All gradients inside the chain carry the caller's power-of-two scale S; results that leave it are multiplied by
 * inv_S.  cs_dy [B][2C], cs_edge [2][B][2C], cs_dx [B][C] must be zero on entry.  part1 / part2: fp32 workspaces of
 * splits1*2C*(3C+E) and splits2*2C*C floats.  Needs C, E multiples of 64 (the direct weight-gradient kernel). */
typedef struct fd_wavenet_bwd_desc {
  const uint16_t* x_planes;    /* xs[l]   [2][B][T][C]  residual stream entering the layer */
  const uint16_t* y_planes;    /* ys[l]   [2][B][T][2C] gate/filter pre-activations, packed order */
  const uint16_t* z_planes;    /* zs[l]   [2][B][T][C]  gated activations */
  const uint16_t* cond_planes; /* [2][B][T][E] */
  const uint16_t* dx_next;     /* planes of d(x_{l+1}) or NULL above the last layer */
  const uint16_t* dskip;       /* planes of d(skip_l) (the same for every layer) */
  const uint16_t* w2t; const uint16_t* w1t; const uint16_t* wct;   /* transposed packs [2][C][2C], [2][C][6C], [2][E][2C] */
  float w2t_inv, w1t_inv, wct_inv;
  uint16_t* dx_out;            /* planes of d(x_l) */
  float* dx_f32;               /* fp32 copy of d(x_l) or NULL */
  float* d_cond;               /* fp32 [B][T][E], accumulated, or NULL */
  float* gw1; float* gw2;      /* [2C][3C+E], [2C][C] */
  float* cs_dy; float* cs_edge; float* cs_dx;
  float* dz; uint16_t* dy;     /* workspaces [B][T][C] fp32, [2][B][T][2C] planes */
  float* part1; float* part2;
  int splits1, splits2;
  int B, T, C, E, dilation, gate_tile;
  float inv_S;
  int prec, backend;
} fd_wavenet_bwd_desc;
int fd_wavenet_block_bwd(const fd_wavenet_bwd_desc* d, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FISHDIFF_B200_H */
