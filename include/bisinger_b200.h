/* bisinger_b200 -- C-ABI of the B200-native synthesis hot path (libbisinger_b200.so).
 *
 * The reference (BiSinger-SVS/BiSinger) has no FFI: its "operator API" for this path is three Python
 * call sites.  Each entry point below replaces one of them; INTEGRATION.md shows the ctypes binding a
 * maintainer adds on the reference side.  Paths are relative to /root/reference/train_bisinger/.
 *
 *   bsg_diffusion_*  <->  GaussianDiffusion.forward(infer=True) sampler loop over DiffNet
 *                         usr/diff/shallow_diffusion_tts.py:245-272 (p_sample :149-166),
 *                         usr/diff/net.py:107-130 (DiffNet.forward), :58-78 (ResidualBlock)
 *   bsg_hifigan_*    <->  HifiGanGenerator.forward(mel, f0)   modules/hifigan/hifigan.py:144-173
 *                         + SourceModuleHnNSF / SineGen       modules/parallel_wavegan/models/source.py:45-138,386-399
 *                         (called from HifiGAN.spec2wav vocoders/hifigan.py:55-69 and
 *                          run_vocoder inference/m4singer/base_svs_infer.py:142-151)
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success, non-zero on error; the message of the
 *     last error on the calling thread is returned by bsg_last_error().  Nothing throws across the ABI.
 *   - "device pointer" arguments are CUDA device pointers on the plan's device, owned by the caller.
 *     `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are asynchronous
 *     with respect to the host unless stated otherwise.
 *   - a plan owns its packed weights, look-up tables, workspaces and captured CUDA graphs.  A plan is bound
 *     to one device and must not be used from two threads at once (one plan per replica process).
 *   - there is no CPU fallback: if no sm_100 device is present, plan creation fails.
 */
#ifndef BISINGER_B200_H_
#define BISINGER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSG_ABI_VERSION 1

/* contraction precision of the tensor-core GEMMs */
#define BSG_PRECISION_BF16 0   /* bf16 operands, fp32 accumulate                                   */
#define BSG_PRECISION_BF16X3 1 /* bf16 hi/lo split operands, 3 MMAs per product, fp32 accumulate   */
#define BSG_PRECISION_FP16X2 2 /* fp16 activations x fp16 hi/lo split weights, 2 MMAs per product, fp32 accumulate (per-layer
                                  GEMMs of the sampler; its once-per-step GEMMs run BF16X3)       */

typedef struct bsg_diffusion_plan bsg_diffusion_plan;
typedef struct bsg_hifigan_plan bsg_hifigan_plan;
typedef struct bsg_pe_plan bsg_pe_plan;

int bsg_abi_version(void);
const char* bsg_last_error(void);
/* number of kernels launched by this library on the calling process so far (eager launches + nodes of
 * replayed graphs); bench.py reports the difference over the timed region as "gpu_launches". */
unsigned long long bsg_kernel_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * DiffNet + shallow-diffusion sampler
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
    int in_dims;            /* mel bins M (80)                      hparams['audio_num_mel_bins']        */
    int hidden_size;        /* encoder hidden H (256)               hparams['hidden_size']               */
    int residual_channels;  /* C (256)                              hparams['residual_channels']         */
    int residual_layers;    /* L (20)                               hparams['residual_layers']           */
    int dilation_cycle;     /* 4                                    hparams['dilation_cycle_length']     */
    int timesteps;          /* length of the schedule buffers       GaussianDiffusion.num_timesteps      */
    int k_step;             /* number of reverse steps K            GaussianDiffusion.K_step             */
    int precision;          /* BSG_PRECISION_*                                                            */
} bsg_diffnet_config;

/* Schedule buffers of the GaussianDiffusion module (host pointers, each [timesteps] float32), read from the
 * module (they may come from a checkpoint), never recomputed: shallow_diffusion_tts.py:103-123. */
typedef struct {
    const float* sqrt_alphas_cumprod;
    const float* sqrt_one_minus_alphas_cumprod;
    const float* sqrt_recip_alphas_cumprod;
    const float* sqrt_recipm1_alphas_cumprod;
    const float* posterior_mean_coef1;
    const float* posterior_mean_coef2;
    const float* posterior_log_variance_clipped;
} bsg_schedule;

/* weights_host: the DiffNet state_dict flattened to float32 in registration order (usr/diff/net.py:91-104):
 *   input_projection.{weight[C][M][1],bias[C]}, mlp.0.{weight[4C][C],bias}, mlp.2.{weight[C][4C],bias},
 *   residual_layers.i.{dilated_conv.{weight[2C][C][3],bias[2C]}, diffusion_projection.{weight[C][C],bias},
 *                      conditioner_projection.{weight[2C][H][1],bias}, output_projection.{weight[2C][C][1],bias}} (i<L),
 *   skip_projection.{weight[C][C][1],bias}, output_projection.{weight[M][C][1],bias}
 * spec_min / spec_max: host float32 [M] (GaussianDiffusion.spec_min/max, shallow_diffusion_tts.py:125-126). */
int bsg_diffusion_plan_create(const bsg_diffnet_config* cfg, const float* weights_host, size_t n_weights,
                              const bsg_schedule* sched, const float* spec_min, const float* spec_max, int device,
                              bsg_diffusion_plan** out);
void bsg_diffusion_plan_destroy(bsg_diffusion_plan* plan);

/* Infer branch of GaussianDiffusion.forward (shallow_diffusion_tts.py:245-272) after the FastSpeech2 handoff.
 *   cond        device f32 [B][T][H]    ret['decoder_inp'] (the reference transposes a view of it, :235)
 *   fs2_mel     device f32 [B][T][M]    ret['mel_out'] of the FastSpeech2 decoder; NULL => Gaussian start
 *                                       (x_K = start_noise, hparams['gaussian_start'], :253-256)
 *   start_noise device f32 [B][1][M][T] noise of q_sample (:204) / gaussian start; NULL => drawn on device
 *   step_noise  device f32 [K][B][1][M][T], entry k is used at t = K-1-k (:266-267); NULL => drawn on device
 *                                       (Philox4x32-10 keyed by `seed`); the CUDA-graph path is used when NULL
 *   mel2ph      device i64 [B][T] or NULL; mel_out is multiplied by (mel2ph > 0) (:269-272)
 *   mel_out     device f32 [B][T][M]    de-normalised mel (denorm_spec, :278-279)
 *   x_final     device f32 [B][1][M][T] or NULL: the normalised x_0 before denorm (for tests)            */
int bsg_diffusion_sample(bsg_diffusion_plan* plan, const float* cond, const float* fs2_mel, const float* start_noise,
                         const float* step_noise, unsigned long long seed, const int64_t* mel2ph, int B, int T,
                         float* mel_out, float* x_final, void* stream);

/* The same infer branch with hparams['pndm_speedup'] = interval: the PLMS / PNDM sampler (shallow_diffusion_tts.py:168-201
 * p_sample_plms, :258-264 the loop over reversed(range(0, K_step, interval))).  Deterministic after the start: no per-step
 * noise.  alphas_cumprod_host: host f32 [timesteps] = GaussianDiffusion.alphas_cumprod (:104).  The diffusion step is a scalar
 * (the reference takes max() of a [B] tensor at :189 and therefore only runs for B = 1; any B is accepted here).
 * Other arguments as bsg_diffusion_sample.                                                                        */
int bsg_diffusion_sample_plms(bsg_diffusion_plan* plan, const float* cond, const float* fs2_mel, const float* start_noise,
                              unsigned long long seed, const int64_t* mel2ph, const float* alphas_cumprod_host, int interval, int B,
                              int T, float* mel_out, float* x_final, void* stream);

/* One DiffNet evaluation eps = denoise_fn(x, t, cond) (usr/diff/net.py:107-130) -- the drop-in for
 * DiffNet.forward used by B200DiffNet and by the parity tests.
 *   spec device f32 [B][1][M][T], t = diffusion step (same for the whole batch, as at :267),
 *   cond device f32 [B][T][H]  (NOTE: channels-last, i.e. the un-transposed decoder_inp),
 *   eps_out device f32 [B][1][M][T]                                                                    */
int bsg_diffnet_forward(bsg_diffusion_plan* plan, const float* spec, int t, const float* cond, int B, int T,
                        float* eps_out, void* stream);

/* Step calls: the public step methods of GaussianDiffusion for callers that drive their own loop, with one diffusion step per
 * batch item.  Common arguments:
 *   t         HOST int32 [B]: the step of each batch item (the reference's [B] long tensor).  0 <= t[b] < k_step (q_sample and
 *             plms_update: < timesteps); out-of-range steps are an error.  When all items share one step the kernels of
 *             bsg_diffusion_sample run; otherwise their per-item variants (each 128-/256-row tile belongs to one item and looks its
 *             step up once).
 *   x, x_out  device f32 [B][1][M][T] (may be the same buffer); cond device f32 [B][T][H] as in bsg_diffusion_sample.
 *   cond_tag  the conditioner projections of all residual layers (about a fifth of a step's FLOPs) are kept in the (B, T) workspace
 *             with the caller's tag.  A nonzero tag equal to the stored one reuses them, so a caller passes the same nonzero tag for
 *             as long as cond is unchanged and a new one when it changes.  0 always recomputes.  bsg_diffusion_sample,
 *             bsg_diffusion_sample_plms, bsg_diffnet_forward and workspace eviction clear the stored tag.
 *   noise     device f32 [B][1][M][T] or NULL: drawn on the device (Philox, keyed by `seed`) from the stream bsg_diffusion_sample uses
 *             at the same point, so that a loop of step calls with seed s reproduces bsg_diffusion_sample(seed = s) exactly. */

/* q_sample (shallow_diffusion_tts.py:203-208): x_out = sqrt_alphas_cumprod[t_b] x_start + sqrt_one_minus_alphas_cumprod[t_b] noise.
 * Device noise: the start noise of bsg_diffusion_sample, i.e. q_sample(norm_spec(fs2_mel)^T, t = K-1, seed = s) is its start. */
int bsg_diffusion_q_sample(bsg_diffusion_plan* plan, const float* x_start, const int* t, const float* noise, unsigned long long seed, int B,
                           int T, float* x_out, void* stream);

/* p_sample (:149-166): one ancestral step of every item from its own t_b: eps = DiffNet(x, t, cond), x0 = clamp(c0 x - c1 eps) (no clamp
 * when clip_denoised == 0), x_out = c2 x0 + c3 x + sigma_t noise, with no noise where t_b == 0 (:165).  Device noise of item b: the
 * stream bsg_diffusion_sample draws at its executed step K-1-t_b. */
int bsg_diffusion_p_sample(bsg_diffusion_plan* plan, const float* x, const int* t, const float* cond, unsigned long long cond_tag,
                           const float* noise, unsigned long long seed, int clip_denoised, int B, int T, float* x_out, void* stream);

/* DiffNet.forward(spec, t, cond) (usr/diff/net.py:107-130) with a step per item; eps_out device f32 [B][1][M][T]. */
int bsg_diffnet_forward_steps(bsg_diffusion_plan* plan, const float* spec, const int* t, const float* cond, unsigned long long cond_tag, int B,
                              int T, float* eps_out, void* stream);

/* get_x_pred of p_sample_plms (:174-183) on the Adams-Bashforth combination of noise predictions (:188-199), per item with
 * a_prev = alphas_cumprod[max(t_b - interval, 0)]; coefficients in fp32 on the host as bsg_diffusion_sample_plms computes them.
 *   n_eps = 0: predictor, eps0 = the current prediction (x_pred of the first iteration, :189)
 *           1: (eps0 + eps1) / 2, eps1 = the prediction at x_pred (:190-191)
 *           2: (3 eps0 - eps1) / 2;  3: (23 eps0 - 16 eps1 + 5 eps2) / 12;  4: (55 eps0 - 59 eps1 + 37 eps2 - 9 eps3) / 24,
 *              eps1..3 = noise_list[-1], [-2], [-3] (:192-197)
 *   eps0..eps3 device f32 [B][1][M][T] (unused ones may be NULL); alphas_cumprod_host: host f32 [timesteps]. */
int bsg_diffusion_plms_update(bsg_diffusion_plan* plan, const float* x, const int* t, const float* alphas_cumprod_host, int interval, int n_eps,
                              const float* eps0, const float* eps1, const float* eps2, const float* eps3, int B, int T, float* x_out,
                              void* stream);

/* Measurement hook for bench.py's roofline line: average duration (ms, CUDA events on `stream`) of `reps` back-to-back
 * launches of one hot kernel at batch shape (B, T), cycling through the residual layers.
 *   which = 0: dilated-conv + conditioner GEMM with the sigmoid*tanh gate epilogue (net.py:67-74)            [unfused path]
 *   which = 1: residual half of the output-projection GEMM with the residual epilogue (net.py:76-78)         [unfused path]
 *   which = 2: skip halves of all layers' output projections (+ skip_projection) as one K = L*C GEMM (net.py:77-78,126-128)
 *   which = 3: the fused ResidualBlock kernel, one launch per layer (fp16x2 plans only; diffnet_layer_kernel)
 *   which = 4: the fused ResidualBlock kernel with ALL layers of a step in one launch, as a sampling step runs it; the
 *              returned time is PER LAYER (launch time / residual_layers); `reps` counts layers, i.e. reps / L launches
 *              (fp16x2 plans only).  bench.py's roofline line uses this one.
 * The kernels run on the plan's workspace (whatever the last sample left there); results are discarded.       */
int bsg_diffusion_time_kernel(bsg_diffusion_plan* plan, int which, int B, int T, int reps, float* avg_ms, void* stream);

/* ------------------------------------------------------------------------------------------------
 * HiFi-GAN / NSF generator
 * ------------------------------------------------------------------------------------------------ */
#define BSG_MAX_UPSAMPLES 8
#define BSG_MAX_RESBLOCK_KERNELS 4
#define BSG_MAX_RESBLOCK_DILATIONS 4

typedef struct {
    int num_mels;                 /* 80 (conv_pre input channels, hifigan.py:117)                          */
    int upsample_initial_channel; /* h['upsample_initial_channel']                                         */
    int num_upsamples;            /* len(h['upsample_rates'])                                              */
    int upsample_rates[BSG_MAX_UPSAMPLES];
    int upsample_kernel_sizes[BSG_MAX_UPSAMPLES];
    int num_kernels;              /* len(h['resblock_kernel_sizes'])                                       */
    int resblock_kernel_sizes[BSG_MAX_RESBLOCK_KERNELS];
    int num_dilations;            /* len of each h['resblock_dilation_sizes'][j] (ResBlock1: 3)            */
    int resblock_dilation_sizes[BSG_MAX_RESBLOCK_KERNELS][BSG_MAX_RESBLOCK_DILATIONS];
    int use_pitch_embed;          /* 1 => NSF harmonic source + noise_convs (hifigan.py:110-116)           */
    int audio_sample_rate;        /* h['audio_sample_rate']                                                */
    int harmonic_num;             /* 8 (hifigan.py:112)                                                    */
    int precision;                /* BSG_PRECISION_BF16                                                    */
} bsg_hifigan_config;

/* weights_host: the generator state_dict AFTER remove_weight_norm() (hifigan.py:175-182), float32, in this order:
 *   m_source.l_linear.{weight[1][9],bias[1]}            (only if use_pitch_embed)
 *   conv_pre.{weight[C0][80][7],bias}
 *   for i < num_upsamples: ups.i.{weight[Cin][Cout][k],bias[Cout]}
 *   for i < num_upsamples: noise_convs.i.{weight[Cout][1][k],bias} (only if use_pitch_embed)
 *   for r < num_upsamples*num_kernels: for m < num_dilations: resblocks.r.convs1.m.{weight[C][C][k],bias}
 *                                      for m < num_dilations: resblocks.r.convs2.m.{weight[C][C][k],bias}
 *   conv_post.{weight[1][C][7],bias[1]}                                                                   */
int bsg_hifigan_plan_create(const bsg_hifigan_config* cfg, const float* weights_host, size_t n_weights, int device,
                            bsg_hifigan_plan** out);
void bsg_hifigan_plan_destroy(bsg_hifigan_plan* plan);

/* HifiGanGenerator.forward (hifigan.py:144-173).
 *   mel       device f32 [B][num_mels][T]
 *   f0        device f32 [B][T] in Hz (0 = unvoiced) or NULL (no NSF branch)
 *   rand_ini  device f32 [B][harmonic_num+1] initial phases (SineGen, source.py:54-57; column 0 is ignored) or NULL => drawn
 *             U[0,1) on device from `seed` for every harmonic h >= 1 (the fundamental gets none), as torch.rand does at :54
 *   src_noise device f32 [B][T*hop][harmonic_num+1] ~ N(0,1) (source.py:133) or NULL => drawn on device from `seed`
 *   Each of the two falls back to the device-side Philox4x32-10 stream independently; the captured-graph path is used when both
 *   are NULL.
 *   wav       device f32 [B][T*hop]                                                                        */
int bsg_hifigan_forward(bsg_hifigan_plan* plan, const float* mel, const float* f0, const float* rand_ini,
                        const float* src_noise, unsigned long long seed, int B, int T, float* wav, void* stream);

/* NSF harmonic source only (hifigan.py:147-149): har_source device f32 [B][T*hop].  Exposed for parity tests. */
int bsg_hifigan_source(bsg_hifigan_plan* plan, const float* f0, const float* rand_ini, const float* src_noise,
                       unsigned long long seed, int B, int T, float* har_source, void* stream);

/* ------------------------------------------------------------------------------------------------
 * PitchExtractor: mel -> f0 between the sampler and the vocoder (SURVEY.md section 8f-2).
 * Replaces  self.pe(mel_out)['f0_denorm_pred']   inference/m4singer/bisinger/a-lang-esm-style-ori-shift.py:629-630,
 *           usr/diffsinger_task.py:107-113;  module: modules/fastspeech/pe.py:120-150 (eval mode).
 * ------------------------------------------------------------------------------------------------ */
#define BSG_PITCH_NORM_LOG 0      /* hparams['pitch_norm'] == 'log':      f0 = 2 ** pred       (utils/pitch_utils.py:66-67) */
#define BSG_PITCH_NORM_STANDARD 1 /* 'standard':                          f0 = pred * f0_std + f0_mean          (:64-65)    */
#define BSG_PITCH_NORM_NONE 2

typedef struct {
    int n_mel_bins;       /* PitchExtractor(n_mel_bins=80)                                                         */
    int hidden_size;      /* 256 (pe.py:123)                                                                       */
    int prenet_layers;    /* 3  (Prenet n_layers, pe.py:9)                                                         */
    int conv_layers;      /* PitchExtractor(conv_layers=2): ConvStacks blocks, 0 = no mel_encoder (pe.py:128-130)  */
    int predictor_layers; /* 5  (pe.py:133)                                                                        */
    int kernel_size;      /* 5  (Prenet / ConvStacks kernel, pe.py:9,82)                                           */
    int predictor_kernel; /* hparams['predictor_kernel'] (5)                                                       */
    int predictor_hidden; /* hparams['predictor_hidden'] if > 0 else hidden_size                                   */
    int gn_group_size;    /* 16: GroupNorm(n_chans // 16, n_chans) (pe.py:54)                                      */
    int left_padding;     /* 0: hparams['ffn_padding'] == 'SAME'; 1: (k-1, 0) padding (tts_modules.py:212-214)     */
    int pitch_norm;       /* BSG_PITCH_NORM_*                                                                      */
    int use_uv;           /* hparams['pitch_type'] == 'frame' and hparams['use_uv'] (pe.py:146)                    */
    float f0_mean, f0_std;
} bsg_pe_config;

/* weights_host: float32, in this order (names of the reference state_dict; BatchNorm folded by the caller):
 *   for i < prenet_layers: mel_prenet.layers.i.0.{weight[C][Cin][k],bias[C]}, bn_scale[C], bn_shift[C]
 *                          (scale = layers.i.2.weight / sqrt(running_var + 1e-5), shift = layers.i.2.bias - running_mean * scale)
 *   mel_prenet.out_proj.{weight[C][C],bias[C]}
 *   if conv_layers > 0: mel_encoder.in_proj.{weight,bias};
 *                       for j < conv_layers: mel_encoder.conv.j.conv.conv.{weight[C][C][k],bias}, mel_encoder.conv.j.norm.{weight,bias};
 *                       mel_encoder.out_proj.{weight,bias}
 *   pitch_predictor.pos_embed_alpha[1], frequencies[C/2] = exp(arange(C/2) * -(ln 1e4 / (C/2 - 1)))  (common_layers.py:130-132)
 *   for i < predictor_layers: pitch_predictor.conv.i.1.{weight[C][C][k],bias}, pitch_predictor.conv.i.3.{weight,bias}
 *   pitch_predictor.linear.{weight[2][C],bias[2]}                                                                  */
int bsg_pe_plan_create(const bsg_pe_config* cfg, const float* weights_host, size_t n_weights, int device, bsg_pe_plan** out);
void bsg_pe_plan_destroy(bsg_pe_plan* plan);

/* PitchExtractor.forward(mel_input) (pe.py:138-150).
 *   mel        device f32 [B][T][n_mel_bins]  (the sampler's mel_out as it stands; all-zero frames are padding)
 *   pitch_pred device f32 [B][T][2]           ret['pitch_pred']
 *   f0         device f32 [B][T]              ret['f0_denorm_pred'] (Hz, 0 = unvoiced / padding)                   */
int bsg_pe_forward(bsg_pe_plan* plan, const float* mel, int B, int T, float* pitch_pred, float* f0, void* stream);

/* ------------------------------------------------------------------------------------------------
 * FastSpeech FFT blocks: the mel-rate decoder of FastSpeech2 / FastSpeech2MIDI and its mel_out projection -- the conditioner's
 * handoff to the sampler (SURVEY.md section 8f-3).
 * Replaces  x = self.decoder(decoder_inp); x = self.mel_out(x); return x * tgt_nonpadding   modules/fastspeech/fs2.py:236-240
 * modules: modules/fastspeech/tts_modules.py:253-310 (FFTBlocks), :340-347 (FastspeechDecoder), modules/commons/common_layers.py:664-731
 * (EncSALayer), :598-644 (TransformerFFNLayer), :199-420 (MultiheadAttention, bias=False); eval mode (no dropout).
 * ------------------------------------------------------------------------------------------------ */
typedef struct bsg_fft_plan bsg_fft_plan;
typedef struct {
    int hidden_size;    /* 256  hparams['hidden_size']                                                              */
    int num_layers;     /* 4    hparams['dec_layers']                                                               */
    int num_heads;      /* 2    hparams['num_heads'] (head width 128)                                               */
    int ffn_kernel;     /* 9    hparams['dec_ffn_kernel_size'], padding 'SAME'                                      */
    int ffn_act;        /* 0 = gelu (hparams['ffn_act'] default), 1 = relu                                          */
    int use_pos_embed;  /* 1    FFTBlocks(use_pos_embed=True): x + pos_embed_alpha * SinusoidalPositionalEmbedding  */
    int out_dims;       /* 80 = mel_out Linear present (fs2.py:60), 0 = FFT blocks only                             */
} bsg_fft_config;

/* weights_host: float32, in this order (names of the FastspeechDecoder / FastSpeech2 state_dict):
 *   pos_embed_alpha[1], frequencies[C/2] = exp(arange(C/2) * -(ln 1e4 / (C/2 - 1)))   (common_layers.py:130-132)
 *   for i < num_layers: layers.i.op.layer_norm1.{weight,bias}[C], layers.i.op.self_attn.in_proj_weight[3C][C],
 *                       layers.i.op.self_attn.out_proj.weight[C][C], layers.i.op.layer_norm2.{weight,bias}[C],
 *                       layers.i.op.ffn.ffn_1.{weight[4C][C][k],bias[4C]}, layers.i.op.ffn.ffn_2.{weight[C][4C],bias[C]}
 *   layer_norm.{weight,bias}[C]
 *   if out_dims > 0: mel_out.{weight[out_dims][C],bias[out_dims]}                                                   */
int bsg_fft_plan_create(const bsg_fft_config* cfg, const float* weights_host, size_t n_weights, int device, bsg_fft_plan** out);
void bsg_fft_plan_destroy(bsg_fft_plan* plan);

/* FastspeechDecoder.forward(x) [+ mel_out, * tgt_nonpadding].
 *   x           device f32 [B][T][C]   decoder_inp; all-zero frames are padding (tts_modules.py:291)
 *   tgt_nonpad  device f32 [B][T] (1 / 0) or NULL: mel_out is multiplied by it (fs2.py:240, (mel2ph > 0))
 *   hidden_out  device f32 [B][T][C] or NULL: the decoder's return value (layer_norm(x) * nonpadding)
 *   mel_out     device f32 [B][T][out_dims] or NULL                                                                 */
int bsg_fft_forward(bsg_fft_plan* plan, const float* x, const float* tgt_nonpad, int B, int T, float* hidden_out, float* mel_out,
                    void* stream);

/* FFTBlocks.forward(x, padding_mask) (tts_modules.py:286-310) with the caller's mask instead of the all-zero-frame rule: the call
 * FastspeechEncoder.forward / FastspeechMIDIEncoder.forward make after their embeddings (tts_modules.py:333-335,
 * modules/diffsinger_midi/fs2.py:53-62; plan built with use_pos_embed = 0, num_layers = enc_layers, ffn_kernel = enc_ffn_kernel_size).
 *   padding_mask  device u8 [B][T], 1 = padding (txt_tokens.eq(0)): those keys are not attended to and those rows are zeroed after
 *                 every residual add and in the result; every utterance needs at least one non-padding position (the reference
 *                 returns NaN otherwise).  Other arguments as bsg_fft_forward.                                           */
int bsg_fft_forward_masked(bsg_fft_plan* plan, const float* x, const unsigned char* padding_mask, const float* tgt_nonpad, int B, int T,
                           float* hidden_out, float* mel_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Kernel self-test: C[b][l][n] = bias[n] + sum_taps A[b][l+shift][:] . W[n][tap][:] through the same tcgen05
 * implicit-GEMM kernel the plans use.  Device pointers; A f32 [B][L][Cin], W f32 host [N][ntaps][Cin].
 * ------------------------------------------------------------------------------------------------ */
int bsg_selftest_conv(const float* a_dev, const float* w_host, const float* bias_host, int B, int L, int Cin, int N,
                      int ntaps, const int* shifts, int n_tile, int precision, float* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BISINGER_B200_H_ */
