// Plan objects behind the C-ABI handles of include/bisinger_b200.h
#pragma once
#include <map>
#include <memory>
#include <utility>
#include <vector>

#include "../../include/bisinger_b200.h"
#include "runtime.h"

namespace b200 {

extern unsigned long long g_launch_count;   // process-wide kernel-launch counter (bsg_kernel_launch_count)

class DiffusionPlan {
public:
    DiffusionPlan(const bsg_diffnet_config& cfg, const float* weights, size_t n_weights, const bsg_schedule& sched,
                  const float* spec_min, const float* spec_max, int device);
    ~DiffusionPlan();

    void sample(const float* cond, const float* fs2_mel, const float* start_noise, const float* step_noise,
                unsigned long long seed, const int64_t* mel2ph, int B, int T, float* mel_out, float* x_final, cudaStream_t st);
    void sample_plms(const float* cond, const float* fs2_mel, const float* start_noise, unsigned long long seed, const int64_t* mel2ph,
                     const float* alphas_cumprod, int interval, int B, int T, float* mel_out, float* x_final, cudaStream_t st);
    void denoise(const float* spec, int t, const float* cond, int B, int T, float* eps_out, cudaStream_t st);
    // step calls (include/bisinger_b200.h): t is a host int32 [B], one diffusion step per batch item
    void q_sample(const float* x_start, const int* t, const float* noise, unsigned long long seed, int B, int T, float* x_out, cudaStream_t st);
    void p_sample(const float* x, const int* t, const float* cond, unsigned long long cond_tag, const float* noise, unsigned long long seed,
                  bool clip_denoised, int B, int T, float* x_out, cudaStream_t st);
    void denoise_steps(const float* spec, const int* t, const float* cond, unsigned long long cond_tag, int B, int T, float* eps_out,
                       cudaStream_t st);
    void plms_update(const float* x, const int* t, const float* alphas_cumprod, int interval, int n_eps, const float* const* eps, int B, int T,
                     float* x_out, cudaStream_t st);
    float time_kernel(int which, int B, int T, int reps, cudaStream_t st);

    bsg_diffnet_config cfg;
    int device;
    int terms = 1;        // MMAs per product of the per-layer GEMMs: 1 bf16, 2 fp16x2, 3 bf16x3
    int terms_side = 1;   // same for the once-per-step GEMMs (bf16x3 in fp16x2 mode)
    bool use_graphs = true;
    bool use_pair = true;    // 2-CTA (cta_group::2) tiles for the tensor-bound GEMMs (gate GEMM, skip-sum GEMM)
    bool use_fused = false;  // one fused kernel per ResidualBlock (fp16x2 mode)
    bool skip_fp8 = false;   // skip-sum GEMM: fp16 MMA + fp8 correction MMA (needs the fused kernel's e4m3 copy of z)
    bool skip_x1 = false;    // skip-sum GEMM: one fp16 MMA per product (no weight-rounding correction term)
    bool fused_mc = false;   // ... on 4-CTA clusters with multicast weight tiles
    bool fused_stack = true;    // ... all layers of a step in one launch (row-tile dataflow between the layers); BSG_LAYER_STACK=0: one launch per layer
    int gate_mode = 1, skip_mode = 1;   // launch_conv_gemm cluster mode of those two GEMMs: 0 single CTA, 1 pair, 2 two pairs + multicast weights
    unsigned long long launches = 0;

private:
    struct Workspace;
    struct Layer {
        PackedW g1, g2, gc;   // dilated conv taps, output projection, conditioner projection
        DevBuf g1_bias, g2_bias;
        int dilation = 1;
    };
    struct StepCoef {
        float sqrt_ac, sqrt_1mac, c0, c1, c2, c3, sigma;
    };
    Workspace& workspace(int B, int T);
    void precompute_cond(Workspace& w, cudaStream_t st);
    ConvGemmArgs gate_args(Workspace& w, int l);
    ConvGemmArgs resskip_args(Workspace& w, int l, const float* lut_t);
    ConvGemmArgs skipsum_args(Workspace& w);
    struct LayerArgs fused_args(Workspace& w, int l0, int n, const float* lut_t, int epoch = 1);
    void reset_dataflow(Workspace& w, cudaStream_t st);
    // rows: per-item step variants of enqueue_step (kRowsNet: the DiffNet kernels read w.t_of_b; kRowsPost: the posterior update reads
    // w.step_coef [B][5]; kRowsNoClip: ... without the clamp of x0).  0: every item at step t, the kernels sample() runs.
    static constexpr int kRowsNet = 1, kRowsPost = 2, kRowsNoClip = 4;
    void enqueue_step(Workspace& w, int t, int k_exec, const float* noise_k, bool last, bool use_mask, int tail, cudaStream_t st,
                      float* eps_out = nullptr, int epoch = 1, int rows = 0);
    void stage_steps(Workspace& w, const int* t, const float* coef, int n_coef, cudaStream_t st);
    void prepare_cond(Workspace& w, const float* cond, unsigned long long tag, cudaStream_t st);
    void import_x(Workspace& w, const float* x, cudaStream_t st);

    std::vector<Layer> layers;
    PackedW inproj, outproj, skipall;   // skipall: skip_projection x the skip halves of all output projections, [C][L*C]
    DevBuf inproj_bias, outproj_bias, skipall_bias;
    DevBuf lut, d_spec_min, d_spec_max, d_seed;
    std::vector<StepCoef> sched;
    static constexpr int kMaxShapes = 6;   // cached (B, T) workspaces, least recently used evicted first
    DevPool pool;                          // large buffers of evicted workspaces (declared before ws: destroyed after it)
    std::map<std::pair<int, int>, std::unique_ptr<Workspace>> ws;
    unsigned long long use_clock = 0;
    unsigned long long graph_nodes = 0;
};

class HifiganPlan {
public:
    HifiganPlan(const bsg_hifigan_config& cfg, const float* weights, size_t n_weights, int device);
    ~HifiganPlan();
    void forward(const float* mel, const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed, int B,
                 int T, float* wav, cudaStream_t st);
    void source(const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed, int B, int T, float* har,
                cudaStream_t st);

    bsg_hifigan_config cfg;
    int device;
    int hop = 1;
    bool pair_mode = true;   // 2-CTA tiles for the >= 128-channel stages (BSG_VOC_PAIR=0: single-CTA tiles everywhere)
    bool use_graphs = true;  // forward without injected noise replays one captured CUDA graph per shape (BSG_VOC_GRAPH=0: plain launches)
    bool noise_v2 = true;    // row-group layout of the noise-branch kernel (BSG_VOC_NOISE_V2=0: one warp per row)
    bool rows_epi = true;    // row-per-thread write-only epilogue with 256-bit stores (BSG_ROWS_EPI=0: transposing epilogue everywhere)
    bool rows_rmw = true;    // ... also for the read-modify-write epilogues, with 256-bit loads (BSG_ROWS_RMW=0: transposing epilogue for those)
    bool fuse_resblocks = true;   // stages with <= 128 channels: one kernel per ResBlock iteration (BSG_VOC_FUSE=0: two conv launches, fp32 stream)
    unsigned long long launches = 0;

private:
    struct Workspace;
    struct Conv {            // one packed convolution
        PackedW w;
        DevBuf bias;
        int cin = 0, cout = 0, k = 1, dilation = 1;
    };
    struct HalfConv {        // one convolution of a fused ResBlock iteration: fp16 weights [Cout][k * Cin] K-major (taps packed densely)
        DevBuf w;
        CUtensorMap map;     // box = 64 K-columns x Cout rows
    };
    struct Stage {
        int cin = 0, cout = 0, rate = 1, ksize = 1;
        bool fused = false;                        // ResBlock iterations on resblock_iter_kernel (C <= 128), 16-bit single-tensor stream
        std::vector<HalfConv> h1, h2;              // fp16 copies of convs1 / convs2 for the fused kernel
        std::vector<Conv> up_phase;                // one 2-tap (generally ceil(k/u)-tap) conv per output phase
        std::vector<std::vector<int>> up_shifts;   // row shifts of each phase's taps
        DevBuf up_bias;
        DevBuf noise_w, noise_b;                   // noise_convs[i] (f32, CUDA-core kernel)
        int noise_k = 1, noise_stride = 1, noise_pad = 0;
        std::vector<Conv> convs1, convs2;          // [num_kernels * num_dilations]
    };
    Workspace& workspace(int B, int T);
    void run_source(Workspace& w, const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed, int B, int T,
                    cudaStream_t st);
    void enqueue(Workspace& w, const float* mel, const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed,
                 int B, int T, float* wav, cudaStream_t st);

    Conv conv_pre;
    std::vector<Stage> stages;
    DevBuf post_w, post_b, src_lin;   // conv_post weights [7][C] f32, bias; l_linear weight[9]+bias
    DevBuf d_seed;
    static constexpr int kMaxShapes = 3;   // cached (B, T) workspaces (several GB each at batch sizes), least recently used evicted first
    std::map<std::pair<int, int>, std::unique_ptr<Workspace>> ws;
    unsigned long long use_clock = 0;
};

class PitchExtractorPlan {
public:
    PitchExtractorPlan(const bsg_pe_config& cfg, const float* weights, size_t n_weights, int device);
    ~PitchExtractorPlan();
    void forward(const float* mel, int B, int T, float* pitch_pred, float* f0, cudaStream_t st);

    bsg_pe_config cfg;
    int device;
    bool pair_mode = true;   // 2-CTA tiles when the batch has >= 4096 rows (BSG_PE_PAIR=0: single-CTA tiles)
    bool use_graphs = true;  // forward replays one captured CUDA graph per shape (BSG_PE_GRAPH=0: plain launches)
    bool rows_epi = true;    // row-per-thread write-only epilogue (BSG_ROWS_EPI=0: transposing epilogue)
    unsigned long long launches = 0;

private:
    struct Workspace;
    struct Conv {
        PackedW w;
        DevBuf bias;
        int cin = 0, cout = 0, k = 1;
    };
    struct Layer {           // convolution + the per-channel pair of its normalisation (scale/shift or gamma/beta)
        Conv conv;
        DevBuf p0, p1;
    };
    Workspace& workspace(int B, int T);
    void enqueue(Workspace& w, const float* mel, int B, int T, float* pitch_pred, float* f0, cudaStream_t st);

    std::vector<Layer> prenet, encoder, predictor;
    Conv prenet_out, enc_in, enc_out;
    DevBuf pos_freq, lin;    // sinusoid frequencies [C/2]; final Linear weight [2][C] + bias [2]
    float pos_alpha = 1.0f;
    std::map<std::pair<int, int>, std::unique_ptr<Workspace>> ws;
};

// FastSpeech FFT blocks (FastspeechDecoder; the FastspeechEncoder's block stack with use_pos_embed = 0 and an explicit mask) + mel_out:
// SURVEY.md section 8f-3 (fft_decoder.cu)
class FftDecoderPlan {
public:
    FftDecoderPlan(const bsg_fft_config& cfg, const float* weights, size_t n_weights, int device);
    ~FftDecoderPlan();
    // padding_mask: device u8 [B][T] (1 = padding) = FFTBlocks.forward(x, padding_mask); null = derived from all-zero frames of x
    void forward(const float* x, const float* tgt_nonpad, int B, int T, float* hidden_out, float* mel_out, cudaStream_t st,
                 const uint8_t* padding_mask = nullptr);

    bsg_fft_config cfg;
    int device;
    unsigned long long launches = 0;

private:
    struct Workspace;
    struct Conv {
        PackedW w;
        DevBuf bias;
        int cin = 0, cout = 0, k = 1;
    };
    struct Layer {
        DevBuf ln1_g, ln1_b, ln2_g, ln2_b;
        Conv in_proj, out_proj, ffn1, ffn2;
    };
    Workspace& workspace(int B, int T);

    std::vector<Layer> layers;
    Conv mel_out;
    DevBuf ln_g, ln_b, pos_freq;
    float pos_alpha = 1.0f;
    std::map<std::pair<int, int>, std::unique_ptr<Workspace>> ws;
    unsigned long long use_clock = 0;
};

}  // namespace b200
