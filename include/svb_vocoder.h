/*
 * svb_vocoder.h -- C ABI of libsvb_vocoder.so, the B200 (sm_100a) implementation of the
 * NeuralSVB mel-to-waveform hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types, no C++ in the
 * signatures.  Every entry point names the reference interface it replaces.  The reference
 * is pure Python/PyTorch, so its "FFI" is ctypes: INTEGRATION.md shows the stub a
 * maintainer adds to vocoders/hifigan.py to bind these.
 *
 * Conventions
 *   - every function returns 0 on success and a negative svb_status otherwise; nothing
 *     throws across the ABI; svb_last_error() gives the message for the calling thread.
 *   - "dev" pointers are device pointers on the handle's device, "host" pointers are host
 *     memory; all buffers are caller-owned; scratch space is owned by the handle.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *     stream-ordered and do not synchronise unless documented (the *_host entry points
 *     synchronise before returning, like the reference's `.cpu()`).
 *   - one handle per (process, device); a handle is not thread-safe.
 *   - all floating-point tensors are fp32, dense, row-major in the stated shape.
 */
#ifndef SVB_VOCODER_H_
#define SVB_VOCODER_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVB_ABI_VERSION 1

typedef enum svb_status {
    SVB_OK = 0,
    SVB_ERR_INVALID = -1,      /* bad argument / shape / config */
    SVB_ERR_CUDA = -2,         /* a CUDA runtime call or kernel failed */
    SVB_ERR_STATE = -3,        /* call order violated (e.g. forward before finalize) */
    SVB_ERR_MISSING = -4,      /* a required weight tensor was never set */
    SVB_ERR_NOMEM = -5
} svb_status;

/* arithmetic used for the dense ResBlock / upsampler contractions */
typedef enum svb_precision {
    SVB_PREC_FP32 = 0,         /* CUDA-core FFMA, fp32 everywhere                              */
    SVB_PREC_TF32 = 1,         /* tcgen05 kind::tf32, operands rounded to nearest, fp32 accum   */
    SVB_PREC_TF32X3 = 2,       /* tcgen05 3xTF32 split (hi*hi + hi*lo + lo*hi), ~fp32 accuracy */
    SVB_PREC_BF16X3 = 3        /* tcgen05 kind::f16, operands split into bf16 hi + lo (16-bit mantissa),
                                  3 MMAs at twice the TF32 rate, fp32 accumulate -- the default      */
} svb_precision;

#define SVB_MAX_UPS 8
#define SVB_MAX_RBK 4
#define SVB_MAX_DIL 4

/* Mirrors the `h` dict given to HifiGanGenerator(h) -- modules/hifigan/hifigan.py:105-142;
 * values for the shipped model: egs/egs_bases/tts/vocoder/hifigan.yaml:3-12. */
typedef struct svb_gen_config {
    int32_t n_mel;                                 /* input channels of conv_pre (80, hifigan.py:118)   */
    int32_t upsample_initial_channel;              /* 512                                                */
    int32_t n_ups;                                 /* len(upsample_rates)                                */
    int32_t upsample_rates[SVB_MAX_UPS];           /* [8,8,2,2]                                          */
    int32_t upsample_kernel_sizes[SVB_MAX_UPS];    /* [16,16,4,4]                                        */
    int32_t resblock;                              /* 1 = ResBlock1 (:30-67), 2 = ResBlock2 (:70-91)     */
    int32_t n_resblock_kernels;                    /* len(resblock_kernel_sizes)                         */
    int32_t resblock_kernel_sizes[SVB_MAX_RBK];    /* [3,7,11]                                           */
    int32_t n_dilations;                           /* dilations per ResBlock (3 for '1', 2 for '2')      */
    int32_t resblock_dilation_sizes[SVB_MAX_RBK][SVB_MAX_DIL];
    int32_t use_pitch_embed;                       /* NSF source + noise_convs (:111-117,126-132)        */
    int32_t audio_sample_rate;                     /* 22050                                              */
    int32_t precision;                             /* svb_precision                                      */
} svb_gen_config;

typedef struct svb_gen svb_gen_t;                  /* opaque generator handle */

/* Message describing the last failure on the calling thread (never NULL). */
const char *svb_last_error(void);
int svb_abi_version(void);

/* ---- HiFi-GAN(-NSF) generator: replaces HifiGanGenerator (modules/hifigan/hifigan.py:104-178)
 *      as it is built and driven by vocoders/hifigan.py:17-33 (load_model) and :55-69 (spec2wav). */

/* HifiGanGenerator.__init__ (hifigan.py:105-142).  `device` is a CUDA ordinal. */
int svb_gen_create(const svb_gen_config *cfg, int device, svb_gen_t **out);
void svb_gen_destroy(svb_gen_t *g);

/* load_state_dict + remove_weight_norm (vocoders/hifigan.py:27-28, hifigan.py:171-178).
 * `name` is the reference state_dict key with weight norm already folded
 * ("conv_pre.weight", "ups.0.bias", "resblocks.4.convs2.1.weight", "noise_convs.2.weight",
 * "m_source.l_linear.weight", ...); `data` is a HOST fp32 tensor in the PyTorch layout
 * (Conv1d [Cout,Cin,K]; ConvTranspose1d [Cin,Cout,K]; Linear [out,in]; bias [C]). */
int svb_gen_set_weight(svb_gen_t *g, const char *name, const float *data, const int64_t *shape, int32_t ndim);
/* weight-norm folding on the device: w = g * v / ||v|| over all dims but 0
 * (torch.nn.utils.weight_norm dim=0; hifigan.py:35-50,118,124,140).  v_host [d0, inner], g_host [d0]. */
int svb_fold_weight_norm_host(const float *v_host, const float *g_host, int64_t d0, int64_t inner,
                              float *w_host, int device);
/* Packs the weights into kernel layouts and uploads them; checks every tensor is present. */
int svb_gen_finalize(svb_gen_t *g);
/* change svb_precision after finalize (repacks nothing; all layouts are kept resident) */
int svb_gen_set_precision(svb_gen_t *g, int32_t precision);

/* HifiGanGenerator.forward(x, f0) (hifigan.py:144-169), batched, device buffers.
 *   mel_dev      [B, n_mel, T]   log10-mel
 *   f0_dev       [B, T] Hz, 0 = unvoiced, or NULL for the non-NSF call model(c)
 *   rand_ini_dev [B, 9]   initial phases of SineGen (source.py:53-55; column 0 is forced to 0)
 *   noise_dev    [B, T*hop, 9] standard-normal draw of SineGen (source.py:132)
 *                both NULL -> drawn in-kernel from a Philox4x32-10 stream keyed by `seed`
 *   wav_dev      [B, T*hop]      output in (-1, 1)
 * Stream-ordered, no host synchronisation. */
int svb_gen_forward(svb_gen_t *g, const float *mel_dev, const float *f0_dev, const float *rand_ini_dev,
                    const float *noise_dev, uint64_t seed, int32_t B, int32_t T, float *wav_dev, void *stream);

/* HifiGAN.spec2wav(mel, f0=...) (vocoders/hifigan.py:55-69) end to end from HOST memory:
 *   mel_host [B, T, n_mel] (the reference's [T, 80] frame-major layout, B clips of equal T),
 *   f0_host [B, T] or NULL, wav_host [B, T*hop].  Copies in (pinned staging, H2D), runs the
 *   generator, copies out (D2H) and synchronises `stream` before returning. */
int svb_gen_spec2wav_host(svb_gen_t *g, const float *mel_host, const float *f0_host, uint64_t seed,
                          int32_t B, int32_t T, float *wav_host, void *stream);

/* spec2wav followed by save_wav's sample conversion (utils/audio.py:11-16: [norm: wav / max|wav| per clip,]
 * wav * 32767, float -> int16 truncation toward zero) ON THE DEVICE, so the D2H copy is 2 bytes per sample:
 * the reference moves the fp32 waveform to the host (vocoders/hifigan.py:63-66) and converts it in a CPU pool
 * (tasks/tts/tts.py:111, svb_vae_task.py:373-375).  wav_host int16 [B, T*hop]. */
int svb_gen_spec2wav_host_i16(svb_gen_t *g, const float *mel_host, const float *f0_host, uint64_t seed, int32_t B,
                              int32_t T, int32_t norm, int16_t *wav_host, void *stream);
/* the conversion alone on device buffers: wav_dev fp32 [B, n] -> out_dev int16 [B, n] (stream-ordered). */
int svb_wav_to_int16(const float *wav_dev, int32_t B, int64_t n, int32_t norm, int16_t *out_dev, void *stream);

/* HifiGanGenerator.forward over clips of different lengths (padded device layout, like MleSVBVAE's output):
 *   mel_dev [B, n_mel, T_max], f0_dev [B, T_max] or NULL, lengths_host int32 [B] in [1, T_max],
 *   rand_ini_dev [B, 9] / noise_dev [B, T_max*hop, 9] or both NULL (Philox keyed by (t, b, harmonic) as in svb_gen_forward),
 *   wav_dev [B, T_max*hop]: clip b's first lengths[b]*hop samples, zeros after.  Values past a clip's length in
 *   mel / f0 / noise are never read.  Clip b's samples are bit-identical to a forward of that clip alone (same
 *   injected noise); tiles wholly past a clip's end are not computed.  Inference only: a handle in training mode
 *   returns SVB_ERR_INVALID.  Stream-ordered, no host synchronisation. */
int svb_gen_forward_ragged(svb_gen_t *g, const float *mel_dev, const float *f0_dev, const int32_t *lengths_host,
                           const float *rand_ini_dev, const float *noise_dev, uint64_t seed, int32_t B, int32_t T_max,
                           float *wav_dev, void *stream);
/* spec2wav over a ragged batch from HOST memory: mel_host [sum T_b, n_mel] and f0_host [sum T_b] (or NULL) clip after clip,
 * wav_host [sum T_b * hop] clip after clip (svb_wav2spec_batch_host's convention).  Synchronises `stream`. */
int svb_gen_spec2wav_ragged_host(svb_gen_t *g, const float *mel_host, const float *f0_host, const int32_t *lengths_host,
                                 int32_t B, uint64_t seed, float *wav_host, void *stream);
/* the same with save_wav's int16 conversion on the device; `norm` takes each clip's peak over its own samples. */
int svb_gen_spec2wav_ragged_host_i16(svb_gen_t *g, const float *mel_host, const float *f0_host, const int32_t *lengths_host,
                                     int32_t B, uint64_t seed, int32_t norm, int16_t *wav_host, void *stream);

/* Intermediate tap for layer-level parity tests: copies a named activation of the LAST forward
 * ("har_source" [B,T*hop]; "conv_pre", "ups{i}", "stage{i}" as [B,C,T_i]) to out_dev. */
int svb_gen_get_tap(svb_gen_t *g, const char *name, float *out_dev, int64_t capacity_floats,
                    int64_t *shape3, void *stream);
int64_t svb_gen_hop(const svb_gen_t *g);
/* number of kernels launched by the last forward / their algorithmic FLOPs (for bench.py) */
int64_t svb_gen_last_launches(const svb_gen_t *g);
double svb_gen_last_flops(const svb_gen_t *g);
/* on = 1: CUDA events around the whole forward (svb_gen_last_ms, else -1).
 * on = 2: additionally CUDA events around EVERY launch of the forward, on the launching stream;
 *         svb_gen_profile_count / _get return, per launch of the last forward: the kernel family,
 *         its event time, its algorithmic HBM bytes (layer-streaming model: each conv reads its
 *         input once, writes its output once, reads the residual / running sum once) and FLOPs. */
int svb_gen_enable_timing(svb_gen_t *g, int32_t on);
float svb_gen_last_ms(svb_gen_t *g);
int32_t svb_gen_profile_count(svb_gen_t *g);
int svb_gen_profile_get(svb_gen_t *g, int32_t i, char *name, int32_t name_cap, float *ms, double *bytes, double *flops);

/* ---- training: backward of the discriminator-side operators ------------------------------------------------
 * Replaces torch autograd through the Conv1d / Conv2d((k,1)) + leaky_relu stacks of DiscriminatorP / DiscriminatorS
 * (modules/hifigan/hifigan.py:193-221, :262-286), AvgPool1d(4,2,1) (:304-306), the reflect pad (:209-212) and the
 * element-wise loss gradients of feature_loss / discriminator_loss / generator_loss (:328-365) and of
 * SpectralConvergengeLoss / LogSTFTMagnitudeLoss (modules/parallel_wavegan/losses/stft_loss.py:34-73).
 *   svb_conv_nct_backward: tensors as svb_conv_nct_forward; y = the forward's post-activation output (mask source,
 *     may be null when out_slope == 1), dy = gradient w.r.t. y.  dz_scratch [B,Cout,Tout,W] receives the masked
 *     gradient; dx (written), dw / db (ACCUMULATED with atomics; the caller zeroes them) may each be null.
 *   svb_loss_grad: da = (accumulate ? da : 0) + scale * f(a, b); kind 0 sign(a-b), 1 (a-1), 2 a, 3 (a-b),
 *     4 sign(ln a - ln b) / a. */
int svb_conv_nct_backward(const float *x_dev, const float *w_dev, const float *y_dev, const float *dy_dev, int32_t B,
                          int32_t Cin, int32_t Cout, int32_t Tin, int32_t W, int32_t K, int32_t stride, int32_t dil,
                          int32_t pad, int32_t groups, float out_slope, float *dz_scratch_dev, float *dx_dev,
                          float *dw_dev, float *db_dev, void *stream);
/* cond_net of the mel-conditioned ("use_cond") discriminators: ConvTranspose1d(C = 80, 1, K = 2*stride, stride,
 * padding = stride/2) (modules/hifigan/hifigan.py:185-189, :257-260).  mel [B, C, T] -> y [B, (T-1)*stride - 2*pad + K];
 * w [C, 1, K], bias [1] on the device.  backward ACCUMULATES dw / db (the mel is an input: no gradient). */
int svb_cond_net_forward(const float *mel_dev, const float *w_dev, const float *bias_dev, int32_t B, int32_t C, int32_t T,
                         int32_t K, int32_t stride, int32_t pad, float *y_dev, void *stream);
int svb_cond_net_backward(const float *mel_dev, const float *dy_dev, int32_t B, int32_t C, int32_t T, int32_t K, int32_t stride,
                          int32_t pad, float *dw_dev, float *db_dev, void *stream);
int svb_avgpool1d_4_2_1_backward(const float *dy_dev, float *dx_dev, int64_t rows, int32_t Tin, void *stream);
int svb_pad_reflect_right_backward(const float *dy_dev, float *dx_dev, int64_t rows, int32_t T, int32_t Tpad, void *stream);
int svb_loss_grad(const float *a_dev, const float *b_dev, int32_t kind, float scale, float *da_dev, int64_t n,
                  int32_t accumulate, void *stream);
/* same, with the factor scale * (*scale_dev) read on the device (the upstream gradient of an autograd node) */
int svb_loss_grad_dev(const float *a_dev, const float *b_dev, int32_t kind, float scale, const float *scale_dev,
                      float *da_dev, int64_t n, int32_t accumulate, void *stream);

/* ---- dense discriminator convolutions on the tensor-core kernel -------------------------------------------------
 * One handle per Conv1d / Conv2d((k,1)) layer with groups == 1 (modules/hifigan/hifigan.py:193-199, :262-271):
 * tensors are PyTorch-layout device buffers [B, C, T, W] (W = period columns, 1 for DiscriminatorS); weights
 * [Cout, Cin, K] and bias are device buffers re-packed by svb_tc_layer_set_weight_dev (cheap: call it whenever
 * they change).  forward: y = leaky_relu(conv(x) + bias, out_slope).  backward: dy is the gradient w.r.t. y;
 * dx is written, dw [Cout, Cin, K] / db [Cout] are ACCUMULATED (caller zeroes them); each may be null.
 * Shapes: stride 1 needs padding (K-1)/2; Cin*K (stride > 1) or Cin (stride 1) and Cout multiples of 32, Cout <= 1024. */
typedef struct svb_tc_layer svb_tc_layer_t;
int svb_tc_layer_create(int32_t Cin, int32_t Cout, int32_t K, int32_t stride, int32_t pad, int32_t precision, int device,
                        svb_tc_layer_t **out);
/* The GROUPED k = 41 layers of DiscriminatorS (Conv1d(128,128,41,2,groups=4) ... Conv1d(1024,1024,41,1,groups=16),
 * modules/hifigan/hifigan.py:263-267: 32 % of the discriminators' FLOPs) on the same tcgen05 kernel, in polyphase
 * form: a stride-s conv with K taps = a stride-1 conv with ceil(K/s) taps over Cin*s "space-to-depth" channels (a
 * permutation of the input, 1x traffic); every GEMM column block contracts only over the input channels of its own conv
 * groups.  forward / backward / set_weight_dev / out_len / destroy are the svb_tc_layer_* calls below; weights are
 * the natural [Cout, Cin/groups, K] tensor.  Needs ceil(K/stride) odd and (Cin/groups*stride, Cout/groups) to tile into
 * 32-channel chunks (pairs of narrow groups share a tile). */
int svb_tc_layer_create_grouped(int32_t Cin, int32_t Cout, int32_t K, int32_t stride, int32_t pad, int32_t groups,
                                int32_t precision, int device, svb_tc_layer_t **out);
void svb_tc_layer_destroy(svb_tc_layer_t *layer);
int svb_tc_layer_set_weight_dev(svb_tc_layer_t *layer, const float *w_dev, const float *bias_dev, void *stream);
int64_t svb_tc_layer_out_len(const svb_tc_layer_t *layer, int64_t T);
int svb_tc_layer_forward(svb_tc_layer_t *layer, const float *x_dev, int32_t B, int32_t T, int32_t W, float out_slope,
                         float *y_dev, void *stream);
int svb_tc_layer_backward(svb_tc_layer_t *layer, const float *x_dev, const float *y_dev, const float *dy_dev, int32_t B,
                          int32_t T, int32_t W, float out_slope, float *dx_dev, float *dw_dev, float *db_dev, void *stream);

/* ---- training: backward of the generator -------------------------------------------------------------
 * Replaces torch autograd through HifiGanGenerator.forward (modules/hifigan/hifigan.py:144-169; ResBlock1/2
 * :54-61 / :81-86; weight_norm :35-50,118,124; SourceModuleHnNSF.l_linear source.py:393-394) for the
 * vocoder training step (SURVEY 8(d) cfg 3).
 *   svb_gen_set_training(g, 1): forwards keep every conv input (the tape), the flipped / transposed weight
 *     packings of the data-gradient convs are built and one gradient buffer per folded tensor is allocated.
 *   svb_gen_backward(g, dwav [B, T*hop]): ACCUMULATES d(loss)/d(folded tensor) for the last forward into those
 *     buffers (svb_gen_zero_grad clears them), in the reference's tensor names and layouts
 *     ("conv_pre.weight" [Cout,Cin,K], "ups.0.weight" [Cin,Cout,K], "noise_convs.0.weight",
 *     "resblocks.3.convs1.0.bias", "conv_post.weight", "m_source.l_linear.weight", ...).
 *   svb_gen_get_grad copies one of them to a device buffer of exactly svb_gen_grad_numel floats.
 *   After an optimizer step: svb_gen_set_weight(...) for the changed tensors, then svb_gen_update_weights(g).
 *   svb_weight_norm_backward: (dv, dg) of w = g * v / ||v|| (norm over all dims but 0) from dw. */
int svb_gen_set_training(svb_gen_t *g, int32_t on);
int svb_gen_update_weights(svb_gen_t *g);
/* Device-side variant (no host round trip): the folded tensor `name` is copied from a device buffer, then ALL
 * kernel packings (forward, data-gradient twins, tcgen05 tiles) are rebuilt by gather / tile kernels on `stream`.
 * svb_fold_weight_norm_dev: w = g * v / ||v|| on device buffers (hifigan.py:35-50 weight_norm, dim 0). */
int svb_gen_set_weight_dev(svb_gen_t *g, const char *name, const float *src_dev, int64_t n, void *stream);
int svb_gen_update_weights_dev(svb_gen_t *g, void *stream);
int svb_fold_weight_norm_dev(const float *v_dev, const float *g_dev, int64_t d0, int64_t inner, float *w_dev, void *stream);
int svb_gen_zero_grad(svb_gen_t *g, void *stream);
int svb_gen_backward(svb_gen_t *g, const float *dwav_dev, void *stream);
int64_t svb_gen_grad_numel(svb_gen_t *g, const char *name);
int svb_gen_get_grad(svb_gen_t *g, const char *name, float *dst_dev, int64_t n, void *stream);
int64_t svb_gen_bwd_launches(const svb_gen_t *g);
int svb_weight_norm_backward(const float *v_dev, const float *g_dev, const float *dw_dev, int64_t rows, int64_t cols,
                             float *dv_dev, float *dg_dev, void *stream);

/* One convolution layer of the generator on PyTorch-layout device tensors, through the CUDA-core
 * (precision 0) or tcgen05 (1, 2) kernel -- for kernel-level parity tests and per-layer timing.
 *   y = out_scale * (conv(leaky_relu(x, in_slope)) + bias [+ res])
 *   transposed_stride = 0: Conv1d(Cin, Cout, K, dilation=dil, padding=dil*(K-1)/2), w_host [Cout,Cin,K]
 *                          (F.conv1d; hifigan.py:30-61)
 *   transposed_stride = u: ConvTranspose1d(Cin, Cout, K, stride=u, padding=(K-u)/2), w_host [Cin,Cout,K]
 *                          (F.conv_transpose1d; hifigan.py:122-125)
 * x [B,Cin,T], res / y [B,Cout,T or T*u].  Runs 1 warm-up + `iters` timed launches; *avg_ms = mean
 * CUDA-event time per launch.  Synchronises `stream`. */
int svb_conv1d_run(const float *x_nct_dev, const float *w_host, const float *bias_host, const float *res_nct_dev,
                   int32_t B, int32_t Cin, int32_t Cout, int32_t T, int32_t K, int32_t dil,
                   int32_t transposed_stride, float in_slope, float out_scale, int32_t precision, int32_t iters,
                   float *y_nct_dev, float *avg_ms, void *stream);

/* ---- discriminator-side operators of the vocoder losses (forward; fp32 CUDA cores) ------------ */

/* y = leaky_relu(conv(x) + bias, out_slope) on PyTorch-layout tensors [B, C, T, W] with W independent inner
 * columns: W = 1 is F.conv1d(stride, dilation, padding, groups) (DiscriminatorS, hifigan.py:262-271);
 * W = period is the (K,1)-kernel / (stride,1)-stride Conv2d of DiscriminatorP (hifigan.py:193-200).
 * w_dev [Cout, Cin/groups, K], bias_dev [Cout] or NULL; Tout = (Tin + 2*pad - dil*(K-1) - 1)/stride + 1. */
int svb_conv_nct_forward(const float *x_dev, const float *w_dev, const float *bias_dev, float *y_dev, int32_t B,
                         int32_t Cin, int32_t Cout, int32_t Tin, int32_t W, int32_t K, int32_t stride, int32_t dil,
                         int32_t pad, int32_t groups, float out_slope, void *stream);
/* AvgPool1d(4, 2, padding=1) over the last dim of [rows, Tin] (MultiScaleDiscriminator.meanpools, hifigan.py:304-307) */
int svb_avgpool1d_4_2_1(const float *x_dev, float *y_dev, int64_t rows, int32_t Tin, void *stream);
/* F.pad(x, (0, Tpad - T), 'reflect') over the last dim of [rows, T] (DiscriminatorP.forward, hifigan.py:209-212) */
int svb_pad_reflect_right(const float *x_dev, float *y_dev, int64_t rows, int32_t T, int32_t Tpad, void *stream);
/* out6_dev (double[6]) = { sum (a-b)^2, sum a^2, sum |ln a - ln b| (if want_log), sum |a-b|, sum (1-a)^2, sum b^2 }
 * -- the reductions behind feature_loss / discriminator_loss / generator_loss (hifigan.py:328-365) and the
 * spectral-convergence / log-magnitude STFT losses (losses/stft_loss.py:34-73).  b_dev may be NULL. */
int svb_pair_stats(const float *a_dev, const float *b_dev, int64_t n, int32_t want_log, double *out6_dev, void *stream);
/* sigma = u . (W v) of torch.nn.utils.spectral_norm in eval mode (no power iteration), W [rows, inner] */
int svb_spectral_sigma_host(const float *w_host, const float *u_host, const float *v_host, int64_t rows, int64_t inner,
                            int device, float *sigma);

/* ---- STFT / mel front end ------------------------------------------------------------------ */

typedef enum svb_pad_mode {
    SVB_PAD_CENTER_ZERO = 0,    /* librosa.stft(center=True, pad_mode='constant'): data_gen_utils.py:123-124 */
    SVB_PAD_CENTER_REFLECT = 1, /* torch.stft(center=True) default: losses/stft_loss.py:26                   */
    SVB_PAD_HALF_REFLECT = 2    /* reflect-pad (n_fft-hop)/2 then center=False: mel_utils.py:66-71           */
} svb_pad_mode;

typedef enum svb_spec_out {
    SVB_OUT_LOG10_MEL = 0,      /* log10(max(eps, mel_basis @ |X|))              data_gen_utils.py:125-134   */
    SVB_OUT_LN_MEL = 1,         /* ln(max(eps, mel_basis @ sqrt(|X|^2 + 1e-9)))  mel_utils.py:74-76,23-24     */
    SVB_OUT_MAG = 2,            /* sqrt(max(|X|^2, floor))                       losses/stft_loss.py:31       */
    SVB_OUT_MAG_RAW = 3,        /* |X|                                           data_gen_utils.py:125        */
    SVB_OUT_MEL_MAG = 4         /* mel_basis @ sqrt(max(|X|^2, floor)), no log   parallel_wavegan/stft_loss.py:40-47 (use_mel_loss) */
} svb_spec_out;

typedef struct svb_stft_config {
    int32_t n_fft;              /* power of two, 64..4096                         */
    int32_t hop;
    int32_t win;                /* periodic hann(win) centred in n_fft            */
    int32_t pad_mode;           /* svb_pad_mode                                   */
    int32_t out_kind;           /* svb_spec_out                                   */
    int32_t clamp_input;        /* clamp(y, -1, 1) first (mel_utils.py:59)        */
    int32_t n_mels;             /* rows of mel_basis (mel outputs only)           */
    int32_t frames_major;       /* 1: out [B, frames, n_out]; 0: out [B, n_out, frames] */
    float eps;                  /* log floor (1e-10 / 1e-5) or magnitude floor (1e-7) */
} svb_stft_config;

/* number of frames the reference produces for `n` samples under cfg (bit-exact frame indexing):
 *   CENTER_*: 1 + n / hop ; HALF_REFLECT: 1 + (n + 2*((n_fft-hop)/2) - n_fft) / hop */
int64_t svb_stft_num_frames(const svb_stft_config *cfg, int64_t n);

/* wav_dev [B, n]; mel_basis_dev [n_mels, n_fft/2+1] (NULL for magnitude outputs);
 * out_dev [B, frames, n_out] or [B, n_out, frames]  (n_out = n_mels or n_fft/2+1). */
int svb_stft_forward(const svb_stft_config *cfg, const float *wav_dev, int32_t B, int64_t n,
                     const float *mel_basis_dev, float *out_dev, void *stream);
/* Backward of svb_stft_forward (torch autograd through torch.stft + magnitude [+ mel + log] in
 * mel_spectrogram, modules/hifigan/mel_utils.py:59-76, and stft(), modules/parallel_wavegan/losses/stft_loss.py:26-31):
 * dout = gradient w.r.t. the forward's output (same layout); the gradient w.r.t. the waveform is ACCUMULATED into
 * dwav [B, n] (atomics; the caller zeroes it).  The spectrum is recomputed per frame, nothing is kept from forward. */
int svb_stft_backward(const svb_stft_config *cfg, const float *wav_dev, int32_t B, int64_t n, const float *mel_basis_dev,
                      const float *dout_dev, float *dwav_dev, void *stream);

/* Spectral-subtraction post-filter of the vocoder output (vocoders/vocoder_utils.py:7-15, applied by
 * vocoders/hifigan.py:66-69 when hparams['vocoder_denoise_c'] > 0):  librosa.stft(n_fft, hop, win, pad 'constant') ->
 * max(|X| - v, 0) with the phase kept -> librosa.istft(hop, win).  wav [B, n] -> out [B, hop * (n / hop)] (device).
 * Only n_fft / hop / win of cfg are read. */
int svb_denoise(const svb_stft_config *cfg, const float *wav_dev, int32_t B, int64_t n, float v, float *out_dev, void *stream);

/* PWG.wav2spec / process_utterance (vocoders/pwg.py:105-122, data_gen_utils.py:93-147) from HOST
 * memory: wav_host [n] -> mel_host [frames, n_mels] (log10), wav_out_host [frames*hop] (zero padded
 * on the right, audio.librosa_pad_lr, utils/audio.py:67-76).  mel_basis_host [n_mels, n_fft/2+1].
 * Returns the frame count (>= 0) or a negative status. */
int64_t svb_wav2spec_host(const svb_stft_config *cfg, const float *wav_host, int64_t n,
                          const float *mel_basis_host, float *mel_host, float *wav_out_host, int device,
                          void *stream);

/* The binarizer's call site (data_gen/tts/base_binarizer.py:168-178, data_gen/singing/binarize_para.py:116-217 call
 * wav2spec once per file from a CPU process pool) as ONE call over a ragged batch: `n_clips` waveforms concatenated in
 * wav_concat_host with their lengths; mel_concat_host receives the [frames_c, n_mels] log10-mels back to back and
 * frames_out[c] their frame counts (1 + lengths[c] / hop each).  One H2D, one kernel launch over all frames of all
 * clips, one D2H.  Returns the total frame count or a negative status. */
int64_t svb_wav2spec_batch_host(const svb_stft_config *cfg, const float *wav_concat_host, const int64_t *lengths,
                                int32_t n_clips, const float *mel_basis_host, float *mel_concat_host, int64_t *frames_out,
                                int device, void *stream);

/* ---- SVB acoustic step, first piece (SURVEY 8(f) N1): the WN gated dilated-conv stack of the GlobalFVAE
 * (modules/fastspeech/fs2_vae.py:19-91; built by modules/voice_conversion/vae_models.py:81-146 with hidden 192,
 * kernel 5, dilation_rate 1, 4 decoder / 8 encoder layers).  Inference (eval mode: dropout is the identity).
 * Weights are the FOLDED ones (WN.remove_weight_norm, fs2_vae.py:96-103), set by the reference's state_dict names:
 *   in_layers.{i}.weight [2H, H, K] / .bias [2H];  res_skip_layers.{i}.weight [2H (H on the last layer), H, 1] / .bias;
 *   cond_layer.weight [2*H*n_layers, gin, 1] / .bias  (when gin_channels > 0). */
typedef struct svb_wn svb_wn_t;
int svb_wn_create(int32_t hidden_channels, int32_t kernel_size, int32_t dilation_rate, int32_t n_layers, int32_t gin_channels,
                  int32_t precision, int32_t device, svb_wn_t **out);
void svb_wn_destroy(svb_wn_t *w);
int svb_wn_set_weight(svb_wn_t *w, const char *name, const float *data_host, const int64_t *shape, int32_t ndim);
int svb_wn_finalize(svb_wn_t *w);
/* WN.forward(x, x_mask, g) (fs2_vae.py:62-94) on device tensors in the reference's layout: x [B, H, T], mask [B, T]
 * (x_mask[:, 0, :], NULL = all ones), g [B, gin, T] (NULL = unconditioned) -> out [B, H, T]. */
int svb_wn_forward(svb_wn_t *w, const float *x_dev, const float *mask_dev, const float *g_dev, int32_t B, int32_t T, float *out_dev,
                   void *stream);
/* FVAEDecoder / GlobalFVAEDecoder (modules/fastspeech/fs2_vae.py:130-152, modules/voice_conversion/vae_models.py:108-128): the mel
 * decoder whose output `spec2wav` consumes -- pre_net ConvTranspose1d(latent, H, k = stride, stride) -> * mask -> WN(dilation_rate 1)
 * -> * mask -> out_proj Conv1d(H, out, 1).  Same handle type as WN; additional weights `pre_net.0.weight [latent, H, stride]`,
 * `pre_net.0.bias`, `out_proj.weight [out, H, 1]`, `out_proj.bias` (svb_wn_set_weight), WN weights under their plain names.
 * forward: z [B, latent, T / stride], mask [B, T] or NULL, g [B, gin, T] or NULL -> out [B, out_channels, T]. */
int svb_fvae_decoder_create(int32_t latent_channels, int32_t hidden_channels, int32_t out_channels, int32_t kernel_size, int32_t n_layers,
                            int32_t gin_channels, int32_t stride, int32_t precision, int32_t device, svb_wn_t **out);
int svb_fvae_decoder_forward(svb_wn_t *w, const float *z_dev, const float *mask_dev, const float *g_dev, int32_t B, int32_t T,
                             float *out_dev, void *stream);

/* ---- PPG extractor (VCASR, modules/voice_conversion/vc_modules.py:56-80) pieces that are not convolutions, on [B, C, T] tensors.
 * nn.LayerNorm(C) of EncoderLayer (modules/fastspeech/conformer/layers.py:167-178): statistics over the channel axis per (b, t). */
int svb_layer_norm_nct(const float *x_dev, const float *gamma_dev, const float *beta_dev, int32_t B, int32_t C, int32_t T, float eps,
                       float *y_dev, void *stream);
/* RelPositionMultiHeadedAttention.forward after its linear projections (modules/commons/espnet_transformer_attn.py:147-186, with
 * rel_shift :127-145 and forward_attention :59-88): q, k, v [B, C, T] (head h = channels [h*dk, (h+1)*dk)), p = linear_pos(pos_emb)
 * [C, T], pos_bias_u / pos_bias_v [n_head * dk], mask [B, T] (0 = padded key; NULL = none) -> context [B, C, T] (before linear_out). */
int svb_relpos_attention_nct(const float *q_dev, const float *k_dev, const float *v_dev, const float *p_dev, const float *bias_u_dev,
                             const float *bias_v_dev, const float *mask_dev, int32_t B, int32_t C, int32_t T, int32_t n_head,
                             float *out_dev, void *stream);

/* Host-only view of the schedule of a merged tensor-core launch (csrc/conv_tc.cu: tc_schedule; no CUDA call, usable without a GPU):
 * `n_layers` convolutions of one shape class (taps KS[l], residual / accumulate flags) over B clips x Tq rows, tiles of 128 rows in
 * items of up to MT tiles, `col_blocks` column blocks, `grid` CTAs.  items_out receives 5 ints per item (layer, column block, clip,
 * first row, tiles) in execution order, off_out [grid + 1] the item range of every CTA, balance_out the mean / max estimated load.
 * Returns the item count or a negative status. */
int64_t svb_tc_schedule_probe(int32_t n_layers, const int32_t *KS, const int32_t *has_res, const int32_t *accumulate, int32_t Cin, int32_t B,
                              int32_t Tq, int32_t MT, int32_t col_blocks, int32_t chain_ordered, int32_t grid, int32_t *items_out,
                              int64_t items_capacity, int32_t *off_out, double *balance_out);
/* svb_tc_schedule_probe for a ragged batch: clip b has rows_per_clip[b] >= 1 rows (and only its own tiles). */
int64_t svb_tc_schedule_probe_ragged(int32_t n_layers, const int32_t *KS, const int32_t *has_res, const int32_t *accumulate,
                                     int32_t Cin, int32_t B, const int32_t *rows_per_clip, int32_t MT, int32_t col_blocks,
                                     int32_t chain_ordered, int32_t grid, int32_t *items_out, int64_t items_capacity,
                                     int32_t *off_out, double *balance_out);

#ifdef __cplusplus
}
#endif
#endif /* SVB_VOCODER_H_ */
