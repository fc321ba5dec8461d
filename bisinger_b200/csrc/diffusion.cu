// DiffNet denoiser + shallow-diffusion ancestral sampler on the conv_gemm kernel.
//
// Reference (relative to /root/reference/train_bisinger/):
//   usr/diff/net.py:107-130 (DiffNet.forward), :58-78 (ResidualBlock), :32-44 (SinusoidalPosEmb)
//   usr/diff/shallow_diffusion_tts.py:149-166 (p_sample), :245-272 (infer loop), :275-279 (spec norm)
//
// Data layout in HBM (rows = b*T + t, channels-last):
//   xt      f32  [B][M][T]      the sampler state x_t in the reference layout [B,1,M,T]
//   xin     bf16 [rows][M]      hi/lo copy of x_t as the A operand of the input projection
//   cond    bf16 [rows][H]      hi/lo copy of decoder_inp (step-invariant)
//   xres    f32  [rows][C]      residual stream x
//   xa      bf16 [rows][C]      hi/lo of (x + d_l): the zero-padded input of layer l's dilated conv
//   z       bf16 [rows][L*C]    hi/lo of the gated activations of ALL layers of the current step (layer l = columns
//                               [l*C, (l+1)*C)): A operand of layer l's output projection and, at the end of the step, of
//                               ONE K = L*C GEMM that produces the skip sum (instead of an fp32 read-modify-write per layer)
//   s, h    bf16 [rows][C]      head operands: sum(skip)/sqrt(L) and relu(skip_projection)
// Per step: 1 + 2L + 3 launches of conv_gemm_kernel; all K steps are captured in one CUDA graph when the
// noise is generated on the device.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <memory>

#include "plans.h"
#include "diffnet_layer.cuh"

namespace b200 {

// ---------------------------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------------------------

// d[t][l][:] = diffusion_projection_l( mlp( SinusoidalPosEmb(t) ) )   -- depends on t only => LUT
// net.py:32-44 (embedding), :94-98 + diffusion.py:68-70 (Linear, Mish, Linear), :62,67 (per-layer Linear)
__global__ void step_lut_kernel(const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ w2,
                                const float* __restrict__ b2, const float* __restrict__ wd, const float* __restrict__ bd,
                                int C, int L, float* __restrict__ lut) {
    extern __shared__ float sm[];
    float* emb = sm;          // [C]
    float* hid = sm + C;      // [4C]
    float* e = hid + 4 * C;   // [C]
    const int t = blockIdx.x;
    const int half = C / 2;
    for (int j = threadIdx.x; j < C; j += blockDim.x) {
        const int jj = j < half ? j : j - half;
        const float w = expf(static_cast<float>(jj) * -(logf(10000.0f) / static_cast<float>(half - 1)));
        const float a = static_cast<float>(t) * w;
        emb[j] = j < half ? sinf(a) : cosf(a);
    }
    __syncthreads();
    for (int o = threadIdx.x; o < 4 * C; o += blockDim.x) {
        float acc = b0[o];
        const float* wr = w0 + static_cast<size_t>(o) * C;
        for (int i = 0; i < C; ++i) acc = fmaf(wr[i], emb[i], acc);
        const float sp = acc > 20.0f ? acc : log1pf(expf(acc));   // F.softplus (threshold 20)
        hid[o] = acc * tanhf(sp);                                  // Mish
    }
    __syncthreads();
    for (int o = threadIdx.x; o < C; o += blockDim.x) {
        float acc = b2[o];
        const float* wr = w2 + static_cast<size_t>(o) * 4 * C;
        for (int i = 0; i < 4 * C; ++i) acc = fmaf(wr[i], hid[i], acc);
        e[o] = acc;
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < L * C; idx += blockDim.x) {
        const int l = idx / C, o = idx % C;
        float acc = bd[l * C + o];
        const float* wr = wd + (static_cast<size_t>(l) * C + o) * C;
        for (int i = 0; i < C; ++i) acc = fmaf(wr[i], e[i], acc);
        lut[(static_cast<size_t>(t) * L + l) * C + o] = acc;
    }
}

// f32 [n] -> bf16 hi/lo
__global__ void split_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, size_t n) {
    const size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n) {
        const float4 v = *reinterpret_cast<const float4*>(src + i);
        const float f[4] = {v.x, v.y, v.z, v.w};
        __nv_bfloat16 h[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { float hf; split_bf16(f[k], hf, h[k], l[k]); }
        *reinterpret_cast<uint2*>(hi + i) = *reinterpret_cast<uint2*>(h);
        if (lo) *reinterpret_cast<uint2*>(lo + i) = *reinterpret_cast<uint2*>(l);
    } else {
        for (size_t k = i; k < n; ++k) {
            float hf; __nv_bfloat16 h, l;
            split_bf16(src[k], hf, h, l);
            hi[k] = h;
            if (lo) lo[k] = l;
        }
    }
}

// x_K: q_sample(norm_spec(fs2_mel)^T, t=K-1) (shallow_diffusion_tts.py:246-252,203-208,275-276) or the Gaussian
// start (:253-256); also used to import a caller-provided x for bsg_diffnet_forward (mode 2).
// One thread per (b, t); writes xt [B][M][T] and the bf16 operand copy xin [rows][M].
__global__ void init_x_kernel(int mode, const float* __restrict__ fs2_mel, const float* __restrict__ noise,
                              const float* __restrict__ smin, const float* __restrict__ smax, float sa, float sb,
                              const unsigned long long* __restrict__ seed_ptr, int B, int T, int M, float* __restrict__ xt,
                              __nv_bfloat16* __restrict__ xin_hi, __nv_bfloat16* __restrict__ xin_lo) {
    const long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= static_cast<long long>(B) * T) return;
    const int b = static_cast<int>(r / T), t = static_cast<int>(r % T);
    for (int c = 0; c < M; ++c) {
        const long long xi = (static_cast<long long>(b) * M + c) * T + t;
        float x;
        if (mode == 2) {
            x = noise[xi];   // plain import of x
        } else {
            float z = noise ? noise[xi] : philox_normal(__ldg(seed_ptr), 0xFFFFFFFFu, static_cast<uint64_t>(xi));
            if (mode == 0) {
                const float mn = smin[c], mx = smax[c];
                const float xs = (fs2_mel[r * M + c] - mn) / (mx - mn) * 2.0f - 1.0f;
                x = sa * xs + sb * z;
            } else {
                x = z;
            }
            xt[xi] = x;
        }
        float hf; __nv_bfloat16 h, l;
        split_bf16(x, hf, h, l);
        xin_hi[r * M + c] = h;
        if (xin_lo) xin_lo[r * M + c] = l;
    }
}

// One PLMS update (usr/diff/shallow_diffusion_tts.py:168-201).  prime = combination of the current and earlier noise predictions
// (mode 0: e0; 1: (e0 + e1)/2 -- first iteration, e1 = prediction at the predictor point; 2: (3 e0 - e1)/2; 3: (23 e0 - 16 e1 + 5 e2)/12;
// 4: (55 e0 - 59 e1 + 37 e2 - 9 e3)/24), x' = x + da * (cx * x - ce * prime)   (get_x_pred, :174-183; da, cx, ce from alphas_cumprod
// in fp32 on the host, same operation order).  write_x = 0: predictor of the first iteration -- only the operand copy for the next
// denoiser evaluation is written, x itself stays.  mel_out != null (last iteration): denorm_spec(x') * (mel2ph > 0) (:268-272).
// One thread per (b, t); x, e* are [B][M][T].
// ROWS = true (bsg_diffusion_plms_update, a step per batch item): item b uses da, cx, ce = coef_b[3b .. 3b+2] instead of the scalars, and
// the operand copy is written only when xin_hi != null (the step call writes none: the next denoiser call imports x itself).
template <bool ROWS>
__global__ void plms_update_kernel(int mode, int write_x, float da, float cx, float ce, float* __restrict__ x, const float* __restrict__ e0,
                                   const float* __restrict__ e1, const float* __restrict__ e2, const float* __restrict__ e3, int B, int T, int M,
                                   __nv_bfloat16* __restrict__ xin_hi, __nv_bfloat16* __restrict__ xin_lo, float* __restrict__ mel_out,
                                   const float* __restrict__ smin, const float* __restrict__ smax, const int64_t* __restrict__ mel2ph,
                                   const float* __restrict__ coef_b) {
    const long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= static_cast<long long>(B) * T) return;
    const int b = static_cast<int>(r / T), t = static_cast<int>(r % T);
    if constexpr (ROWS) {
        da = coef_b[3 * b];
        cx = coef_b[3 * b + 1];
        ce = coef_b[3 * b + 2];
    }
    const float mask = (mel_out != nullptr && mel2ph != nullptr && !(mel2ph[r] > 0)) ? 0.0f : 1.0f;
    for (int c = 0; c < M; ++c) {
        const long long i = (static_cast<long long>(b) * M + c) * T + t;
        const float a = e0[i];
        float prime;
        if (mode == 0) prime = a;
        else if (mode == 1) prime = (a + e1[i]) / 2.0f;
        else if (mode == 2) prime = (3.0f * a - e1[i]) / 2.0f;
        else if (mode == 3) prime = (23.0f * a - 16.0f * e1[i] + 5.0f * e2[i]) / 12.0f;
        else prime = (55.0f * a - 59.0f * e1[i] + 37.0f * e2[i] - 9.0f * e3[i]) / 24.0f;
        const float xv = x[i];
        const float xn = xv + da * (cx * xv - ce * prime);
        if (write_x) x[i] = xn;
        if (!ROWS || xin_hi != nullptr) {
            float hf; __nv_bfloat16 h, l;
            split_bf16(xn, hf, h, l);
            xin_hi[r * M + c] = h;
            if (xin_lo) xin_lo[r * M + c] = l;
        }
        if (mel_out != nullptr) mel_out[r * M + c] = ((xn + 1.0f) / 2.0f * (smax[c] - smin[c]) + smin[c]) * mask;
    }
}

// q_sample (shallow_diffusion_tts.py:203-208) with a step per batch item: x = sa_b * x_start + sb_b * noise, coef = [B][2] (sa_b, sb_b) =
// (sqrt_alphas_cumprod[t_b], sqrt_one_minus_alphas_cumprod[t_b]).  noise == null: drawn from the stream of the sampler's start noise
// (init_x_kernel), so that q_sample(t = K-1) with seed s is the start sample(seed = s) uses.  One thread per element of [B][M][T].
__global__ void q_sample_kernel(const float* __restrict__ x_start, const float* __restrict__ noise, const float* __restrict__ coef,
                                const unsigned long long* __restrict__ seed_ptr, int B, int M, int T, float* __restrict__ x_out) {
    const long long xi = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (xi >= static_cast<long long>(B) * M * T) return;
    const int b = static_cast<int>(xi / (static_cast<long long>(M) * T));
    const float sa = coef[2 * b], sb = coef[2 * b + 1];
    const float z = noise ? noise[xi] : philox_normal(__ldg(seed_ptr), 0xFFFFFFFFu, static_cast<uint64_t>(xi));
    x_out[xi] = sa * x_start[xi] + sb * z;
}

// ---------------------------------------------------------------------------------------------
// plan
// ---------------------------------------------------------------------------------------------
static const int kOneTap[1] = {0};
static constexpr int kXaBoxRows = 144;   // 128 + 2 * max dilation (8)
static constexpr int kSkipTilePair = 256; // N tile of the skip-sum GEMM when run on 2-CTA tiles
static constexpr int kResTile = 128;     // N tile of the residual / skip-sum GEMMs (N = 256): 2x the tiles -> better wave balance
struct DiffusionPlan::Workspace {
    int B = 0, T = 0;
    DevBuf cp;   // f32 [L][rows][2C]: conditioner projection + biases of every layer (step-invariant)
    DevBuf xt, xin_hi, xin_lo, cond_hi, cond_lo, xres, xa_hi, xa_lo, z_hi, z_lo, s_hi, s_lo, h_hi, h_lo, mel, mel2ph, eps;
    // fused layer kernel: a layer writes the NEXT layer's conv input while neighbouring tiles still read halo rows of its own
    // input, so the conv input ping-pongs between two buffers (layer l reads [l & 1]: xa_hi / xa8 are [0], these are [1])
    DevBuf xa8, xa16_b, xa8_b;   // xa8: e4m3 copy of the conv input (A operand of the fp8 correction MMAs)
    CUtensorMap m_xa16_b, m_xa8_b;
    CUtensorMap m_xin[2], m_cond[2], m_xa[2], m_z[2], m_s[2], m_h[2];
    CUtensorMap m_xa8, m_xe[2];      // fused layer kernel: 8-bit conv input; the fp16 conv input buffers as the epilogue reads them
    DevBuf z8;                       // e4m3 copy of z: the skip-sum GEMM's fp8 correction operand
    CUtensorMap m_z8;
    DevBuf plms_eps[4];              // PLMS: the last four noise predictions [B][M][T]
    DevBuf layer_tab;                // fused layer kernel: LayerParams[L] (weight / conditioner-projection tensor maps, scales) in device memory
    DevBuf layer_flags;              // ... and the slab completion counters of a multi-layer launch [L][B * ceil(T / 128)]
    DevBuf t_of_b, step_coef;        // step calls: int32 [B] diffusion step of each batch item; f32 [B][5] posterior coefficients
    unsigned long long cond_tag = 0; // step calls: caller's tag of the cond whose projections cp holds (0: none / unknown)
    cudaGraphExec_t graph = nullptr;
    bool graph_has_mask = false;
    cudaGraphExec_t plms_graph = nullptr;   // the PLMS loop for (plms_interval, plms_has_mask, plms_ac)
    int plms_interval = 0;
    bool plms_has_mask = false;
    std::vector<float> plms_ac;
    unsigned long long plms_nodes = 0;
    unsigned long long last_use = 0;        // LRU stamp
    size_t bytes = 0;
    ~Workspace() {
        if (graph) cudaGraphExecDestroy(graph);
        if (plms_graph) cudaGraphExecDestroy(plms_graph);
    }
};

static std::vector<float> take(const float*& p, size_t n) {
    std::vector<float> v(p, p + n);
    p += n;
    return v;
}

DiffusionPlan::DiffusionPlan(const bsg_diffnet_config& c, const float* w, size_t n_w, const bsg_schedule& s, const float* spec_min,
                             const float* spec_max, int device)
    : cfg(c), device(device) {
    B200_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    B200_CUDA(cudaGetDeviceProperties(&prop, device));
    B200_CHECK(prop.major == 10, "bisinger_b200 requires an sm_100 (B200) device; found sm_" + std::to_string(prop.major) +
                                     std::to_string(prop.minor) + " -- there is no fallback path");
    const int M = c.in_dims, H = c.hidden_size, C = c.residual_channels, L = c.residual_layers;
    B200_CHECK(C == 256 && H == 256, "this build is specialised for residual_channels == hidden_size == 256");
    B200_CHECK(M == 80, "this build is specialised for 80 mel bins");
    B200_CHECK(L >= 1 && c.k_step >= 1 && c.k_step <= c.timesteps, "bad layer/step counts");
    B200_CHECK(c.dilation_cycle >= 1 && (1 << (c.dilation_cycle - 1)) * 2 + kTileM <= kXaBoxRows, "dilation cycle too long for the halo tile");
    // the fused layer kernel's slab dataflow waits only for the neighbouring 128-row slabs: the halo must not reach further
    B200_CHECK((1 << (c.dilation_cycle - 1)) <= kTileM, "dilation longer than a slab");
    B200_CHECK(c.precision == BSG_PRECISION_BF16 || c.precision == BSG_PRECISION_BF16X3 || c.precision == BSG_PRECISION_FP16X2,
               "bad precision");
    // terms: the per-layer GEMMs (gate, residual, skip sum); terms_side: the once-per-step / once-per-batch GEMMs
    // (conditioner projection, input projection, skip_projection, output_projection), which stay bf16x3 in fp16x2 mode
    terms = c.precision == BSG_PRECISION_BF16X3 ? 3 : (c.precision == BSG_PRECISION_FP16X2 ? 2 : 1);
    terms_side = terms == 2 ? 3 : terms;
    const bool f16 = terms == 2;
    const size_t expect = static_cast<size_t>(C) * M + C + 4 * C * C + 4 * C + 4 * C * C + C +
                          static_cast<size_t>(L) * (2 * C * C * 3 + 2 * C + C * C + C + 2 * C * H + 2 * C + 2 * C * C + 2 * C) +
                          static_cast<size_t>(C) * C + C + static_cast<size_t>(M) * C + M;
    B200_CHECK(n_w == expect, "weight blob has " + std::to_string(n_w) + " floats, expected " + std::to_string(expect));

    const float* p = w;
    auto w_in = take(p, static_cast<size_t>(C) * M);
    auto b_in = take(p, C);
    auto w0 = take(p, 4 * C * C);
    auto b0 = take(p, 4 * C);
    auto w2 = take(p, 4 * C * C);
    auto b2 = take(p, C);
    std::vector<float> wd_all, bd_all;
    std::vector<float> skip_w(static_cast<size_t>(C) * L * C), skip_b(C, 0.0f);   // skip halves of all layers, K-concatenated
    layers.resize(L);
    for (int l = 0; l < L; ++l) {
        auto wdil = take(p, static_cast<size_t>(2 * C) * C * 3);   // [2C][C][3]
        auto bdil = take(p, 2 * C);
        auto wdp = take(p, static_cast<size_t>(C) * C);
        auto bdp = take(p, C);
        auto wc = take(p, static_cast<size_t>(2 * C) * H);         // [2C][H][1]
        auto bc = take(p, 2 * C);
        auto wo = take(p, static_cast<size_t>(2 * C) * C);         // [2C][C][1]
        auto bo = take(p, 2 * C);
        wd_all.insert(wd_all.end(), wdp.begin(), wdp.end());
        bd_all.insert(bd_all.end(), bdp.begin(), bdp.end());
        // G1 weights: [2C rows][K = 3*C (taps) + H (cond)], rows permuted so that every 256-row N tile holds the
        // gate rows of 128 channels followed by the filter rows of the same channels (gate = first half of the
        // conv output, filter = second half: net.py:73).
        // The conditioner projection is step-invariant: it is evaluated once per utterance batch (precompute_cond) and
        // added in the gate epilogue, so the per-step gate GEMM only carries the three dilated taps (K = 3*C).
        const int K1 = 3 * C;
        std::vector<float> g1(static_cast<size_t>(2 * C) * K1), gc(static_cast<size_t>(2 * C) * H), gb(2 * C);
        for (int tile = 0; tile < 2; ++tile)
            for (int part = 0; part < 2; ++part)
                for (int j = 0; j < 128; ++j) {
                    const int dst = tile * 256 + part * 128 + j;
                    const int src = part * C + tile * 128 + j;
                    float* row = &g1[static_cast<size_t>(dst) * K1];
                    for (int tap = 0; tap < 3; ++tap)
                        for (int ci = 0; ci < C; ++ci) row[tap * C + ci] = wdil[(static_cast<size_t>(src) * C + ci) * 3 + tap];
                    for (int ci = 0; ci < H; ++ci) gc[static_cast<size_t>(dst) * H + ci] = wc[static_cast<size_t>(src) * H + ci];
                    gb[dst] = bdil[src] + bc[src];
                }
        layers[l].g1.pack(g1, 2 * C, K1, f16);
        layers[l].gc.pack(gc, 2 * C, H);
        upload(layers[l].g1_bias, gb);
        // output projection: first half of the output channels = residual, second half = skip (net.py:77)
        layers[l].g2.pack(std::vector<float>(wo.begin(), wo.begin() + static_cast<size_t>(C) * C), C, C, f16);
        upload(layers[l].g2_bias, std::vector<float>(bo.begin(), bo.begin() + C));
        for (int o = 0; o < C; ++o) {
            for (int ci = 0; ci < C; ++ci) skip_w[static_cast<size_t>(o) * L * C + static_cast<size_t>(l) * C + ci] = wo[static_cast<size_t>(C + o) * C + ci];
            skip_b[o] += bo[C + o];
        }
        layers[l].dilation = 1 << (l % c.dilation_cycle);
    }
    auto w_skip = take(p, static_cast<size_t>(C) * C);
    auto b_skip = take(p, C);
    auto w_out = take(p, static_cast<size_t>(M) * C);
    auto b_out = take(p, M);
    inproj.pack(w_in, C, M);
    upload(inproj_bias, b_in);
    {
        // skip_projection folded into the skip sum (no nonlinearity between them, net.py:126-128):
        //   relu(W_sp (sum_l W_skip,l z_l + b_skip) / sqrt(L) + b_sp) = relu(((W_sp W_skip) z + W_sp b_skip + sqrt(L) b_sp) / sqrt(L))
        // one K = L*C GEMM produces the head activation h directly; products in fp64 on the host
        std::vector<float> fold(static_cast<size_t>(C) * L * C);
        std::vector<float> fold_b(C);
        std::vector<double> acc(static_cast<size_t>(L) * C);
        const double sqrtL = std::sqrt(static_cast<double>(L));
        for (int o2 = 0; o2 < C; ++o2) {
            std::fill(acc.begin(), acc.end(), 0.0);
            double ab = 0.0;
            for (int o = 0; o < C; ++o) {
                const double ws = w_skip[static_cast<size_t>(o2) * C + o];
                const float* row = &skip_w[static_cast<size_t>(o) * L * C];
                for (int k = 0; k < L * C; ++k) acc[k] += ws * row[k];
                ab += ws * skip_b[o];
            }
            for (int k = 0; k < L * C; ++k) fold[static_cast<size_t>(o2) * L * C + k] = static_cast<float>(acc[k]);
            fold_b[o2] = static_cast<float>(ab + sqrtL * b_skip[o2]);
        }
        skipall.pack(fold, C, L * C, f16);
        upload(skipall_bias, fold_b);
    }
    outproj.pack(w_out, M, C);
    upload(outproj_bias, b_out);

    // step-embedding LUT on the device
    {
        DevBuf d_w0, d_b0, d_w2, d_b2, d_wd, d_bd;
        upload(d_w0, w0); upload(d_b0, b0); upload(d_w2, w2); upload(d_b2, b2); upload(d_wd, wd_all); upload(d_bd, bd_all);
        lut.alloc(static_cast<size_t>(c.k_step) * L * C * sizeof(float));
        step_lut_kernel<<<c.k_step, 256, 6 * C * sizeof(float)>>>(d_w0.as<float>(), d_b0.as<float>(), d_w2.as<float>(),
                                                                   d_b2.as<float>(), d_wd.as<float>(), d_bd.as<float>(), C, L,
                                                                   lut.as<float>());
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaDeviceSynchronize());
    }
    // schedule (host copies; baked into kernel parameters per step)
    sched.resize(c.timesteps);
    for (int t = 0; t < c.timesteps; ++t) {
        sched[t].sqrt_ac = s.sqrt_alphas_cumprod[t];
        sched[t].sqrt_1mac = s.sqrt_one_minus_alphas_cumprod[t];
        sched[t].c0 = s.sqrt_recip_alphas_cumprod[t];
        sched[t].c1 = s.sqrt_recipm1_alphas_cumprod[t];
        sched[t].c2 = s.posterior_mean_coef1[t];
        sched[t].c3 = s.posterior_mean_coef2[t];
        sched[t].sigma = t == 0 ? 0.0f : std::exp(0.5f * s.posterior_log_variance_clipped[t]);   // nonzero_mask (:165)
    }
    upload(d_spec_min, std::vector<float>(spec_min, spec_min + M));
    upload(d_spec_max, std::vector<float>(spec_max, spec_max + M));
    d_seed.alloc(sizeof(unsigned long long));

    // set the dynamic-smem attribute of every instantiation outside of any stream capture
    ConvGemmArgs none{};
    for (int epi : {EPI_F32, EPI_INPROJ, EPI_RELU_BF16}) launch_conv_gemm(256, terms_side, epi, none, nullptr);
    launch_conv_gemm(80, terms_side, EPI_POSTERIOR, none, nullptr);
    launch_conv_gemm(256, terms, EPI_GATE, none, nullptr);
    launch_conv_gemm(kResTile, terms, EPI_RES_SKIP, none, nullptr);
    launch_conv_gemm(kResTile, terms, EPI_RELU_BF16, none, nullptr);
    if (const char* np = std::getenv("BSG_NO_PAIR")) use_pair = !(np[0] == '1');
    if (const char* ng = std::getenv("BSG_DIFF_GRAPH")) use_graphs = ng[0] == '1';   // 0: plain launches instead of captured graphs
    gate_mode = skip_mode = use_pair ? 1 : 0;
    if (const char* mc = std::getenv("BSG_MC")) {   // bit 0: gate GEMM, bit 1: skip-sum GEMM on 4-CTA clusters with multicast weights
        const int bits = std::atoi(mc);
        if (use_pair && terms == 2 && (bits & 1)) gate_mode = 2;
        if (use_pair && terms >= 2 && (bits & 2)) skip_mode = 2;
    }
    launch_conv_gemm(256, terms, EPI_GATE, none, nullptr, 1);
    launch_conv_gemm(kSkipTilePair, terms, EPI_RELU_BF16, none, nullptr, 1);
    // one fused kernel per ResidualBlock (diffnet_layer.cuh) in the fp16x2 mode; BSG_NO_FUSE=1 keeps the two-launch path
    use_fused = use_pair && terms == 2;
    if (const char* nf = std::getenv("BSG_NO_FUSE")) use_fused = use_fused && !(nf[0] == '1');
    if (const char* mc = std::getenv("BSG_LAYER_MC")) fused_mc = mc[0] == '1';
    if (const char* sk = std::getenv("BSG_LAYER_STACK")) fused_stack = sk[0] == '1';
    if (use_fused) { LayerArgs la{}; launch_diffnet_layer(la, nullptr, fused_mc); }
    // Skip-sum GEMM with the fp8 correction term (BSG_SKIP_FP8=1; needs the e4m3 copy of z only the fused layer kernel writes).
    // Off by default: measured 295 us against 240 us with two fp16 MMAs -- the K = L*C GEMM streams z from HBM and is bound
    // by operand bytes, and the 8-bit copy adds half as many again.
    skip_fp8 = false;
    if (const char* e = std::getenv("BSG_SKIP_FP8")) skip_fp8 = use_fused && skip_mode == 1 && e[0] == '1';
    if (skip_fp8) launch_conv_gemm(kSkipTilePair, 4, EPI_RELU_BF16, none, nullptr, 1);
    // skip-sum GEMM with ONE fp16 MMA per product (BSG_SKIP_X1=1|0): see conv_gemm.cuh TERMS == 5
    skip_x1 = false;
    if (const char* e = std::getenv("BSG_SKIP_X1")) skip_x1 = use_pair && terms == 2 && skip_mode == 1 && !skip_fp8 && e[0] == '1';
    if (skip_x1) launch_conv_gemm(kSkipTilePair, 5, EPI_RELU_BF16, none, nullptr, 1);
    if (gate_mode == 2) launch_conv_gemm(256, terms, EPI_GATE, none, nullptr, 2);
    if (skip_mode == 2) launch_conv_gemm(kSkipTilePair, terms, EPI_RELU_BF16, none, nullptr, 2);
}

DiffusionPlan::~DiffusionPlan() = default;

DiffusionPlan::Workspace& DiffusionPlan::workspace(int B, int T) {
    const auto key = std::make_pair(B, T);
    auto it = ws.find(key);
    if (it != ws.end()) {
        it->second->last_use = ++use_clock;
        return *it->second;
    }
    // Keep a few shapes alive (buffers + captured graphs): utterance lengths vary from call to call, so evict ONE least-recently
    // used entry at a time -- when there are more than kMaxShapes, or while the cached workspaces plus the new one (~70 KB per mel
    // frame) would exceed the byte budget (BSG_WS_BUDGET_GB, default 48).
    // The large buffers are sized for a capacity class of rows (next multiple of max(256, 2^ceil(log2 rows) / 8): at most 12.5 % more than
    // needed) and come from / go back to the plan's pool: a new length of the same class reuses an evicted workspace's memory instead of
    // paying cudaFree + cudaMalloc (tools/varying_length_latency.py: up to 700 ms per new length before, ~6 ms -- the graph capture -- now).
    // Only sizes are quantised: every offset, tensor map and launch below uses the actual B and T.
    const size_t rows = static_cast<size_t>(B) * T;
    size_t p2 = 256;
    while (p2 < rows) p2 <<= 1;
    const size_t step = std::max<size_t>(256, p2 / 8);
    const size_t cap = (rows + step - 1) / step * step;
    static const double budget_gb = [] { const char* e = std::getenv("BSG_WS_BUDGET_GB"); return e ? std::atof(e) : 48.0; }();
    auto total = [&] { size_t n = 0; for (auto& kv : ws) n += kv.second->bytes; return n; };
    {
        const size_t need = cap * 72 * 1024;
        while (!ws.empty() && (ws.size() >= static_cast<size_t>(kMaxShapes) || static_cast<double>(total() + need) > budget_gb * 1e9)) {
            auto lru = ws.begin();
            for (auto jt = ws.begin(); jt != ws.end(); ++jt)
                if (jt->second->last_use < lru->second->last_use) lru = jt;
            // its buffers are about to be handed to another shape, possibly on another stream: wait for the work that may still use them
            // (cudaFree did the same implicitly before the pool existed)
            B200_CUDA(cudaDeviceSynchronize());
            ws.erase(lru);
        }
    }
    auto w = std::make_unique<Workspace>();
    w->last_use = ++use_clock;
    const int M = cfg.in_dims, H = cfg.hidden_size, C = cfg.residual_channels;
    size_t pooled_bytes = 0;
    auto take = [&](DevBuf& b, size_t n) { b.alloc(n, &pool); pooled_bytes += n; };
    w->B = B;
    w->T = T;
    const bool lo = terms == 3, lo_side = terms_side == 3;
    take(w->xt, cap * M * 4);
    take(w->eps, cap * M * 4);
    take(w->xin_hi, cap * M * 2);
    take(w->cond_hi, cap * H * 2);
    take(w->xres, cap * C * 4);
    take(w->xa_hi, cap * C * 2);
    take(w->z_hi, cap * cfg.residual_layers * C * 2);
    take(w->s_hi, cap * C * 2);
    take(w->h_hi, cap * C * 2);
    take(w->mel, cap * M * 4);
    take(w->mel2ph, cap * 8);
    take(w->cp, static_cast<size_t>(cfg.residual_layers) * cap * 2 * C * 4);
    if (lo) {
        take(w->xa_lo, cap * C * 2);
        take(w->z_lo, cap * cfg.residual_layers * C * 2);
    }
    if (lo_side) {
        take(w->xin_lo, cap * M * 2);
        take(w->cond_lo, cap * H * 2);
        take(w->s_lo, cap * C * 2);
        take(w->h_lo, cap * C * 2);
    }
    auto mk = [&](CUtensorMap (&m)[2], const DevBuf& hi, const DevBuf& lo_, int ch, int box_rows = kTileM) {
        m[0] = make_act_tmap(hi.p, B, T, ch, 0, box_rows);
        m[1] = lo_.p ? make_act_tmap(lo_.p, B, T, ch, 0, box_rows) : m[0];
    };
    mk(w->m_xin, w->xin_hi, w->xin_lo, M);
    mk(w->m_cond, w->cond_hi, w->cond_lo, H);
    mk(w->m_xa, w->xa_hi, w->xa_lo, C, kXaBoxRows);   // halo tile of the dilated conv (3 taps, dilation <= 8)
    mk(w->m_z, w->z_hi, w->z_lo, cfg.residual_layers * C);
    mk(w->m_s, w->s_hi, w->s_lo, C);
    mk(w->m_h, w->h_hi, w->h_lo, C);
    if (use_fused) {
        take(w->xa8, cap * C);
        w->m_xa8 = make_act8_tmap(w->xa8.p, B, T, C, kXaBoxRows);
        if (skip_fp8) {
            take(w->z8, cap * cfg.residual_layers * C);
            w->m_z8 = make_act8_tmap(w->z8.p, B, T, cfg.residual_layers * C, kTileM);
        }
        take(w->xa16_b, cap * C * 2);
        take(w->xa8_b, cap * C);
        w->m_xa16_b = make_act_tmap(w->xa16_b.p, B, T, C, 0, kXaBoxRows);
        w->m_xa8_b = make_act8_tmap(w->xa8_b.p, B, T, C, kXaBoxRows);
        w->m_xe[1] = make_epi16_tmap(w->xa16_b.p, B, T, C);
        w->m_xe[0] = make_epi16_tmap(w->xa_hi.p, B, T, C);
        const int wbox = fused_mc ? 64 : 128;   // weight rows one CTA loads per tile (multicast: half of its 128)
        std::vector<LayerParams> tab(cfg.residual_layers);
        for (int l = 0; l < cfg.residual_layers; ++l) {
            Layer& ly = layers[l];
            LayerParams& lp = tab[l];
            CUtensorMap unused;
            ly.g1.maps(wbox, lp.wg16, unused);
            lp.wg8 = ly.g1.map8(wbox);
            ly.g2.maps(wbox, lp.wr[0], lp.wr[1]);
            lp.cp = make_f32_tmap(w->cp.as<float>() + static_cast<size_t>(l) * rows * 2 * C, B, T, 2 * C);
            lp.bias_r = ly.g2_bias.as<float>();
            lp.gscale = ly.g1.acc_scale;
            lp.rscale = ly.g2.acc_scale;
            lp.dilation = ly.dilation;
            lp.pad_ = 0;
        }
        w->layer_tab.alloc(tab.size() * sizeof(LayerParams));
        B200_CUDA(cudaMemcpy(w->layer_tab.p, tab.data(), tab.size() * sizeof(LayerParams), cudaMemcpyHostToDevice));
        const int n_slabs = B * ((T + kTileM - 1) / kTileM);
        w->layer_flags.alloc(static_cast<size_t>(cfg.residual_layers) * n_slabs * sizeof(int));
    }
    w->bytes = pooled_bytes;
    {   // what the pool keeps beyond the live workspaces counts against the same budget
        const double live = static_cast<double>(total() + w->bytes);
        pool.trim(live < budget_gb * 1e9 ? static_cast<size_t>(budget_gb * 1e9 - live) : 0);
    }
    auto& ref = *w;
    ws[key] = std::move(w);
    return ref;
}

static void set_w(ConvGemmArgs& a, PackedW& w, int n_tile) {
    w.maps(n_tile, a.wmap[0], a.wmap[1]);
    a.epi.acc_scale = w.acc_scale;
}


// cp[l] = conditioner_projection_l(cond) + its bias + the dilated conv's bias (net.py:68,71), all layers, once per call
void DiffusionPlan::precompute_cond(Workspace& w, cudaStream_t st) {
    const int H = cfg.hidden_size, C = cfg.residual_channels, L = cfg.residual_layers;
    for (int l = 0; l < L; ++l) {
        Layer& ly = layers[l];
        ConvGemmArgs a{};
        set_geometry(a, w.B, w.T, 2 * C, 256);
        a.amap[0] = w.m_cond[0]; a.amap[1] = w.m_cond[1];
        set_w(a, ly.gc, 256);
        set_taps(a, 0, 0, H / kBlockK, kOneTap, 1, 0);
        a.epi.bias = ly.g1_bias.as<float>();
        a.epi.f32_a = w.cp.as<float>() + static_cast<size_t>(l) * w.B * w.T * 2 * C;
        a.epi.out_pitch = 2 * C;
        launch_conv_gemm(256, terms_side, EPI_F32, a, st);
        ++launches, ++g_launch_count;
    }
}

// dilated conv(x + d) [+ precomputed conditioner projection] -> sigmoid*tanh gate (net.py:67-74)
ConvGemmArgs DiffusionPlan::gate_args(Workspace& w, int l) {
    const int H = cfg.hidden_size, C = cfg.residual_channels;
    Layer& ly = layers[l];
    ConvGemmArgs a{};
    set_geometry(a, w.B, w.T, 2 * C, 256, gate_mode != 0);
    a.amap[0] = w.m_xa[0]; a.amap[1] = w.m_xa[1];
    set_w(a, ly.g1, 256 >> gate_mode);   // 2-CTA tiles: each CTA stages half of the 256 weight rows (multicast: loads a quarter)
    const int shifts[3] = {-ly.dilation, 0, ly.dilation};
    set_taps(a, 0, 0, C / kBlockK, shifts, 3, C);
    a.a_rows = kXaBoxRows;   // the xa tensor maps are encoded once with the box of the largest dilation
    a.epi.aux0 = w.cp.as<float>() + static_cast<size_t>(l) * w.B * w.T * 2 * C;   // + conditioner projection + biases
    (void)H;
    a.epi.out_hi = w.z_hi.as<__nv_bfloat16>();
    a.epi.out_lo = terms == 3 ? w.z_lo.as<__nv_bfloat16>() : nullptr;
    a.epi.out_fp16 = terms == 2;
    a.epi.out_pitch = 2 * C;                         // pitch of the conditioner-projection rows (aux0)
    a.epi.act_pitch = cfg.residual_layers * C;       // pitch of the all-layer z matrix
    a.epi.out_col0 = l * C;
    if (const char* ab = std::getenv("BSG_ABLATE")) a.epi.flags = std::atoi(ab);   // timing experiments only (wrong results)
    return a;
}

// residual half of the output projection (net.py:76-78): x <- (x + W_res z + b) / sqrt(2), xa <- split(x + d_{l+1})
ConvGemmArgs DiffusionPlan::resskip_args(Workspace& w, int l, const float* lut_t) {
    const int C = cfg.residual_channels, L = cfg.residual_layers;
    Layer& ly = layers[l];
    const bool lo = terms == 3;
    ConvGemmArgs a{};
    set_geometry(a, w.B, w.T, C, kResTile);
    a.amap[0] = w.m_z[0]; a.amap[1] = w.m_z[1];
    set_w(a, ly.g2, kResTile);
    set_taps(a, 0, l * C, C / kBlockK, kOneTap, 1, 0);
    a.epi.bias = ly.g2_bias.as<float>();
    a.epi.f32_a = w.xres.as<float>();
    a.epi.out_hi = w.xa_hi.as<__nv_bfloat16>(); a.epi.out_lo = lo ? w.xa_lo.as<__nv_bfloat16>() : nullptr;
    a.epi.out_fp16 = terms == 2;
    a.epi.dvec = (l + 1 < L) ? lut_t + static_cast<size_t>(l + 1) * C : nullptr;
    a.epi.out_pitch = C;
    return a;
}

// ResidualBlocks [l0, l0 + n) in one launch of the fused layer kernel (diffnet_layer.cuh): per pair tile (two 128-row slabs) the
// gate GEMM of both channel halves + the residual GEMM; n > 1: slab dataflow across the layers (zero w.layer_flags before the launch)
LayerArgs DiffusionPlan::fused_args(Workspace& w, int l0, int n, const float* lut_t, int epoch) {
    const int C = cfg.residual_channels, L = cfg.residual_layers;
    LayerArgs a{};
    a.xa16[0] = w.m_xa[0]; a.xa16[1] = w.m_xa16_b;
    a.xa8[0] = w.m_xa8; a.xa8[1] = w.m_xa8_b;
    a.xe[0] = w.m_xe[0]; a.xe[1] = w.m_xe[1];
    a.z = w.m_z[0];
    a.tab = w.layer_tab.as<LayerParams>();
    a.layer0 = l0;
    a.n_layers = n;
    a.total_layers = L;
    a.B = w.B;
    a.T = w.T;
    a.slabs_per_item = (w.T + kTileM - 1) / kTileM;
    a.n_slabs = a.B * a.slabs_per_item;
    a.a_rows = kXaBoxRows;
    a.z_pitch = L * C;
    a.z_out = w.z_hi.as<__half>();
    a.z8_out = skip_fp8 ? w.z8.as<uint8_t>() : nullptr;
    a.xa16_out[0] = w.xa_hi.as<__half>(); a.xa16_out[1] = w.xa16_b.as<__half>();
    a.xa8_out[0] = w.xa8.as<uint8_t>(); a.xa8_out[1] = w.xa8_b.as<uint8_t>();
    a.lut_t = lut_t;
    a.flags = n > 1 ? w.layer_flags.as<int>() : nullptr;
    a.epoch = epoch;
    if (const char* ab = std::getenv("BSG_ABLATE")) a.flags_ablate = std::atoi(ab);   // timing experiments only (wrong results)
    return a;
}

// skip sum of all layers + skip_projection + ReLU as one K = L*C GEMM over the step's z matrix (net.py:77-78,126-128; weights
// pre-multiplied in the constructor) -> h (bf16 hi/lo), the A operand of the output projection
ConvGemmArgs DiffusionPlan::skipsum_args(Workspace& w) {
    const int C = cfg.residual_channels, L = cfg.residual_layers;
    ConvGemmArgs a{};
    const int nt = use_pair ? kSkipTilePair : kResTile;
    set_geometry(a, w.B, w.T, C, nt, skip_mode != 0);
    a.amap[0] = w.m_z[0]; a.amap[1] = w.m_z[1];
    set_w(a, skipall, nt >> skip_mode);
    if (skip_fp8) {   // fp16 + fp8-correction contraction (launch with terms 4): e4m3 z x e5m2 weight remainders
        a.amap[1] = w.m_z8;
        a.wmap[1] = skipall.map8(nt / 2);
    }
    set_taps(a, 0, 0, L * C / kBlockK, kOneTap, 1, 0);
    a.epi.bias = skipall_bias.as<float>();
    a.epi.out_hi = w.h_hi.as<__nv_bfloat16>();
    a.epi.out_lo = w.h_lo.p ? w.h_lo.as<__nv_bfloat16>() : nullptr;
    a.epi.out_pitch = C;
    a.epi.flags = 0;                                        // ReLU (net.py:128)
    a.epi.c0 = 1.0f / std::sqrt(static_cast<float>(L));
    return a;
}

// Average duration of one hot kernel, measured with CUDA events on `st`: `reps` back-to-back launches cycling through
// the layers (so weights change from launch to launch as in a real step).  which: 0 = gate GEMM, 1 = residual GEMM,
// 2 = skip-sum GEMM.
float DiffusionPlan::time_kernel(int which, int B, int T, int reps, cudaStream_t st) {
    B200_CHECK(which >= 0 && which <= 4, "unknown kernel id");   // 3 = one fused layer, 4 = all layers in one launch (time per layer)
    B200_CHECK(which < 3 || use_fused, "the fused layer kernel is not enabled in this plan");
    B200_CHECK(reps > 0, "reps must be positive");
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    const int L = cfg.residual_layers;
    cudaEvent_t e0, e1;
    B200_CUDA(cudaEventCreate(&e0));
    B200_CUDA(cudaEventCreate(&e1));
    int epoch = 0;
    if (which == 4) B200_CUDA(cudaMemsetAsync(w.layer_flags.p, 0, w.layer_flags.bytes, st));
    auto run = [&](int n) {
        for (int i = 0; i < n; ++i) {
            const int l = i % L;
            if (which == 4) {
                if (l != 0) continue;
                launch_diffnet_layer(fused_args(w, 0, L, lut.as<float>(), ++epoch), st, fused_mc);
            } else if (which == 3) launch_diffnet_layer(fused_args(w, l, 1, lut.as<float>()), st, fused_mc);
            else if (which == 0) launch_conv_gemm(256, terms, EPI_GATE, gate_args(w, l), st, gate_mode);
            else if (which == 1) launch_conv_gemm(kResTile, terms, EPI_RES_SKIP, resskip_args(w, l, lut.as<float>()), st);
            else launch_conv_gemm(use_pair ? kSkipTilePair : kResTile, skip_fp8 ? 4 : (skip_x1 ? 5 : terms), EPI_RELU_BF16, skipsum_args(w), st, skip_mode);
            ++launches, ++g_launch_count;
        }
    };
    run(3);
    B200_CUDA(cudaEventRecord(e0, st));
    run(reps);
    B200_CUDA(cudaEventRecord(e1, st));
    B200_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    B200_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (std::getenv("BSG_TRACE")) {
        // one more launch with the per-role cycle counters (conv_gemm.cuh: ConvGemmArgs::trace), averaged over the CTAs
        const int grid = 2 * device_sm_count();
        DevBuf tb;
        tb.alloc(static_cast<size_t>(grid) * 16 * 8);
        B200_CUDA(cudaMemsetAsync(tb.p, 0, static_cast<size_t>(grid) * 16 * 8, st));
        ConvGemmArgs a = which == 0 ? gate_args(w, 1) : (which == 1 ? resskip_args(w, 1, lut.as<float>()) : skipsum_args(w));
        a.trace = tb.as<unsigned long long>();
        if (which >= 3) {
            LayerArgs la = which == 4 ? fused_args(w, 0, L, lut.as<float>(), ++epoch) : fused_args(w, 1, 1, lut.as<float>());
            la.trace = tb.as<unsigned long long>();
            launch_diffnet_layer(la, st, fused_mc);
        } else if (which == 0) launch_conv_gemm(256, terms, EPI_GATE, a, st, gate_mode);
        else if (which == 1) launch_conv_gemm(kResTile, terms, EPI_RES_SKIP, a, st);
        else launch_conv_gemm(use_pair ? kSkipTilePair : kResTile, skip_fp8 ? 4 : terms, EPI_RELU_BF16, a, st, skip_mode);
        std::vector<unsigned long long> h(static_cast<size_t>(grid) * 16);
        B200_CUDA(cudaMemcpyAsync(h.data(), tb.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        double s[16] = {0};
        int n_mma = 0, n_cta = 0;
        for (int c = 0; c < grid; ++c) {
            if (h[c * 16 + 4] == 0) continue;
            ++n_cta;
            if (h[c * 16 + 0]) ++n_mma;
            for (int i = 0; i < 16; ++i) s[i] += static_cast<double>(h[c * 16 + i]);
        }
        if (n_mma && n_cta)
            std::fprintf(stderr,
                         "TRACE kernel %d: MMA thread total %.0f clk (tiles %.2f) wait tmem-empty %.0f a-full %.0f b-full %.0f | producer total %.0f "
                         "wait a-empty %.0f b-empty %.0f | epilogue warp total %.0f wait t-full %.0f\n",
                         which, s[0] / n_mma, s[10] / n_mma, s[1] / n_mma, s[2] / n_mma, s[3] / n_mma, s[4] / n_cta, s[5] / n_cta, s[6] / n_cta,
                         s[7] / n_cta, s[8] / n_cta);
        if (which >= 3 && n_cta)
            std::fprintf(stderr, "TRACE fused layer (waits for other tiles' rows: %.0f clk): producer waits for z %.0f clk | epilogue warp busy in gate ops %.0f, in residual ops %.0f, of which waiting for cp/x boxes %.0f | box producer waits for consumers %.0f (row tiles %.2f)\n",
                         s[15] / n_cta, s[9] / n_cta, s[11] / n_cta, s[12] / n_cta, s[14] / n_cta, s[13] / n_cta, n_mma ? s[10] / n_mma : 0.0);
    }
    return ms / static_cast<float>(reps);
}

// One DiffNet evaluation at diffusion step t (net.py:107-130) followed by `tail`:
//   tail == 0: posterior update of xt (p_sample), tail == 1: write eps to ws.eps
// epoch: 1-based index of this evaluation since reset_dataflow() (the fused layer kernel's row-tile counters run on from launch to
// launch instead of being zeroed by a memset node per step, which cut the programmatic-dependent-launch chain twice per step)
void DiffusionPlan::reset_dataflow(Workspace& w, cudaStream_t st) {
    if (use_fused && fused_stack) B200_CUDA(cudaMemsetAsync(w.layer_flags.p, 0, w.layer_flags.bytes, st));
}

void DiffusionPlan::enqueue_step(Workspace& w, int t, int k_exec, const float* noise_k, bool last, bool use_mask, int tail,
                                 cudaStream_t st, float* eps_out, int epoch, int rows) {
    const int M = cfg.in_dims, H = cfg.hidden_size, C = cfg.residual_channels, L = cfg.residual_layers;
    const int B = w.B, T = w.T;
    // rows & kRowsNet: the DiffNet kernels look up each batch item's step in w.t_of_b (lut_t is then the whole table);
    // rows & kRowsPost: the posterior update takes each item's coefficients from w.step_coef
    const bool rows_net = (rows & kRowsNet) != 0;
    const float* lut_t = lut.as<float>() + (rows_net ? 0 : static_cast<size_t>(t) * L * C);
    StepRows sr{};
    sr.t_of_b = w.t_of_b.as<int>();
    sr.coef = w.step_coef.as<float>();
    sr.dvec_stride = L * C;
    sr.k_last = cfg.k_step - 1;
    sr.clip = (rows & kRowsNoClip) ? 0 : 1;
    auto nz = [&](const DevBuf& b) { return b.p ? b.as<__nv_bfloat16>() : nullptr; };

    {   // input projection + ReLU (net.py:116-118); writes x and (x + d_0)
        ConvGemmArgs a{};
        set_geometry(a, B, T, C, 256);
        a.amap[0] = w.m_xin[0]; a.amap[1] = w.m_xin[1];
        set_w(a, inproj, 256);
        set_taps(a, 0, 0, (M + kBlockK - 1) / kBlockK, kOneTap, 1, 0);
        a.epi.bias = inproj_bias.as<float>();
        a.epi.f32_a = use_fused ? nullptr : w.xres.as<float>();   // fused layers carry the stream as the fp16 conv input only
        a.epi.out_hi = w.xa_hi.as<__nv_bfloat16>(); a.epi.out_lo = nz(w.xa_lo);
        a.epi.out_fp16 = terms == 2;
        a.epi.dvec = lut_t;
        a.epi.out_pitch = C;
        a.epi.out8 = use_fused ? w.xa8.as<uint8_t>() : nullptr;
        a.steps = sr;
        launch_conv_gemm(256, terms_side, rows_net ? EPI_INPROJ_STEPS : EPI_INPROJ, a, st);
        ++launches, ++g_launch_count;
    }
    if (use_fused && fused_stack) {
        // all ResidualBlocks in ONE launch: row tiles flow from layer to layer as soon as their three input tiles are done
        static const bool memset_each = [] { const char* e = std::getenv("BSG_LAYER_MEMSET"); return e && e[0] == '1'; }();
        if (memset_each) {   // round-1 behaviour (A/B experiments): zero the counters before every launch
            B200_CUDA(cudaMemsetAsync(w.layer_flags.p, 0, w.layer_flags.bytes, st));
            epoch = 1;
        }
        LayerArgs la = fused_args(w, 0, L, lut_t, epoch);
        la.t_of_b = sr.t_of_b;
        launch_diffnet_layer(la, st, fused_mc, rows_net);
        ++launches, ++g_launch_count;
    } else {
        for (int l = 0; l < L; ++l) {
            if (use_fused) {
                LayerArgs la = fused_args(w, l, 1, lut_t);
                la.t_of_b = sr.t_of_b;
                launch_diffnet_layer(la, st, fused_mc, rows_net);
                ++launches, ++g_launch_count;
                continue;
            }
            launch_conv_gemm(256, terms, EPI_GATE, gate_args(w, l), st, gate_mode);
            ++launches, ++g_launch_count;
            ConvGemmArgs ra = resskip_args(w, l, lut_t);
            ra.steps = sr;
            launch_conv_gemm(kResTile, terms, rows_net ? EPI_RES_SKIP_STEPS : EPI_RES_SKIP, ra, st);
            ++launches, ++g_launch_count;
        }
    }
    {   // skip sum sum_l (W_skip,l z_l + b_skip,l) / sqrt(L) (net.py:77-78,126) and skip_projection + ReLU (:127-128): one K = L*C GEMM
        launch_conv_gemm(use_pair ? kSkipTilePair : kResTile, skip_fp8 ? 4 : (skip_x1 ? 5 : terms), EPI_RELU_BF16, skipsum_args(w), st, skip_mode);
        ++launches, ++g_launch_count;
    }
    {   // output_projection (net.py:129) fused with the DDPM posterior update (shallow_diffusion_tts.py:149-166)
        ConvGemmArgs a{};
        set_geometry(a, B, T, M, 80);
        a.amap[0] = w.m_h[0]; a.amap[1] = w.m_h[1];
        set_w(a, outproj, 80);
        set_taps(a, 0, 0, C / kBlockK, kOneTap, 1, 0);
        a.epi.bias = outproj_bias.as<float>();
        if (tail == 1) {
            a.epi.f32_a = eps_out ? eps_out : w.eps.as<float>();
            a.epi.flags = 1;
        } else {
            const StepCoef& sc = sched[t];
            a.epi.f32_a = w.xt.as<float>();
            a.epi.f32_b = last ? w.mel.as<float>() : nullptr;
            a.epi.out_hi = last ? nullptr : w.xin_hi.as<__nv_bfloat16>();
            a.epi.out_lo = last ? nullptr : nz(w.xin_lo);
            a.epi.aux0 = noise_k;
            a.epi.aux1 = d_spec_min.as<float>();
            a.epi.aux2 = d_spec_max.as<float>();
            a.epi.mel2ph = use_mask ? w.mel2ph.as<int64_t>() : nullptr;
            a.epi.c0 = sc.c0; a.epi.c1 = sc.c1; a.epi.c2 = sc.c2; a.epi.c3 = sc.c3; a.epi.c4 = sc.sigma;
            a.epi.seed_ptr = d_seed.as<unsigned long long>();
            a.epi.step = static_cast<unsigned>(k_exec);
        }
        a.epi.out_pitch = M;
        a.steps = sr;
        launch_conv_gemm(80, terms_side, (tail == 0 && (rows & kRowsPost)) ? EPI_POSTERIOR_STEPS : EPI_POSTERIOR, a, st);
        ++launches, ++g_launch_count;
    }
}

void DiffusionPlan::sample(const float* cond, const float* fs2_mel, const float* start_noise, const float* step_noise,
                           unsigned long long seed, const int64_t* mel2ph, int B, int T, float* mel_out, float* x_final,
                           cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CHECK(cond != nullptr && mel_out != nullptr, "cond and mel_out are required");
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    const int M = cfg.in_dims, H = cfg.hidden_size, K = cfg.k_step;
    const size_t rows = static_cast<size_t>(B) * T;
    const bool lo = terms_side == 3;

    B200_CUDA(cudaMemcpyAsync(d_seed.p, &seed, sizeof(seed), cudaMemcpyHostToDevice, st));
    {
        const size_t n = rows * H;
        split_kernel<<<static_cast<unsigned>((n / 4 + 255) / 256 + 1), 256, 0, st>>>(cond, w.cond_hi.as<__nv_bfloat16>(),
                                                                                    lo ? w.cond_lo.as<__nv_bfloat16>() : nullptr, n);
        ++launches, ++g_launch_count;
        precompute_cond(w, st);
        w.cond_tag = 0;
        const int mode = fs2_mel ? 0 : 1;
        init_x_kernel<<<static_cast<unsigned>((rows + 127) / 128), 128, 0, st>>>(
            mode, fs2_mel, start_noise, d_spec_min.as<float>(), d_spec_max.as<float>(), sched[K - 1].sqrt_ac, sched[K - 1].sqrt_1mac,
            d_seed.as<unsigned long long>(), B, T, M, w.xt.as<float>(), w.xin_hi.as<__nv_bfloat16>(),
            lo ? w.xin_lo.as<__nv_bfloat16>() : nullptr);
        ++launches, ++g_launch_count;
        B200_CUDA(cudaGetLastError());
    }
    const bool use_mask = mel2ph != nullptr;
    if (use_mask) B200_CUDA(cudaMemcpyAsync(w.mel2ph.p, mel2ph, rows * 8, cudaMemcpyDeviceToDevice, st));

    if (step_noise == nullptr && use_graphs) {
        if (w.graph && w.graph_has_mask != use_mask) {
            cudaGraphExecDestroy(w.graph);
            w.graph = nullptr;
        }
        if (!w.graph) {
            cudaStream_t cs;
            B200_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            cudaGraph_t g = nullptr;
            const unsigned long long before = launches;
            B200_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            try {
                reset_dataflow(w, cs);
                for (int k = 0; k < K; ++k) enqueue_step(w, K - 1 - k, k, nullptr, k == K - 1, use_mask, 0, cs, nullptr, k + 1);
            } catch (...) {
                cudaStreamEndCapture(cs, &g);
                if (g) cudaGraphDestroy(g);
                cudaStreamDestroy(cs);
                throw;
            }
            B200_CUDA(cudaStreamEndCapture(cs, &g));
            graph_nodes = launches - before;
            launches = before;
            g_launch_count -= graph_nodes;
            B200_CUDA(cudaGraphInstantiate(&w.graph, g, 0));
            cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            w.graph_has_mask = use_mask;
        }
        B200_CUDA(cudaGraphLaunch(w.graph, st));
        launches += graph_nodes, g_launch_count += graph_nodes;
    } else {
        const size_t per_step = rows * M;
        reset_dataflow(w, st);
        for (int k = 0; k < K; ++k)
            enqueue_step(w, K - 1 - k, k, step_noise ? step_noise + static_cast<size_t>(k) * per_step : nullptr, k == K - 1, use_mask, 0,
                         st, nullptr, k + 1);
    }
    B200_CUDA(cudaMemcpyAsync(mel_out, w.mel.p, rows * M * 4, cudaMemcpyDeviceToDevice, st));
    if (x_final) B200_CUDA(cudaMemcpyAsync(x_final, w.xt.p, rows * M * 4, cudaMemcpyDeviceToDevice, st));
}

// get_x_pred coefficients in fp32, same operation order as the reference (:175-180): x' = x + da * (cx * x - ce * eps')
static void plms_coef(const float* alphas_cumprod, int t, int interval, float& da, float& cx, float& ce) {
    const float a_t = alphas_cumprod[t], a_prev = alphas_cumprod[t - interval > 0 ? t - interval : 0];
    const float a_t_sq = std::sqrt(a_t), a_prev_sq = std::sqrt(a_prev);
    da = a_prev - a_t;
    cx = 1.0f / (a_t_sq * (a_t_sq + a_prev_sq));
    ce = 1.0f / (a_t_sq * (std::sqrt((1.0f - a_prev) * a_t) + std::sqrt((1.0f - a_t) * a_prev)));
}

// PLMS / PNDM sampler: the infer branch with hparams['pndm_speedup'] = interval (shallow_diffusion_tts.py:168-201,258-264).
// Deterministic after the start; K/interval iterations, one denoiser evaluation each plus one more in the first.
void DiffusionPlan::sample_plms(const float* cond, const float* fs2_mel, const float* start_noise, unsigned long long seed,
                                const int64_t* mel2ph, const float* alphas_cumprod, int interval, int B, int T, float* mel_out,
                                float* x_final, cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CHECK(cond != nullptr && mel_out != nullptr && alphas_cumprod != nullptr, "cond, mel_out and alphas_cumprod are required");
    B200_CHECK(interval >= 1 && interval <= cfg.k_step, "bad pndm_speedup interval");
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    const int M = cfg.in_dims, H = cfg.hidden_size, K = cfg.k_step;
    const size_t rows = static_cast<size_t>(B) * T;
    const bool lo = terms_side == 3;
    if (w.plms_eps[0].p == nullptr)
        for (auto& e : w.plms_eps) e.alloc(rows * M * 4);
    B200_CUDA(cudaMemcpyAsync(d_seed.p, &seed, sizeof(seed), cudaMemcpyHostToDevice, st));
    {
        const size_t n = rows * H;
        split_kernel<<<static_cast<unsigned>((n / 4 + 255) / 256 + 1), 256, 0, st>>>(cond, w.cond_hi.as<__nv_bfloat16>(),
                                                                                    lo ? w.cond_lo.as<__nv_bfloat16>() : nullptr, n);
        ++launches, ++g_launch_count;
        precompute_cond(w, st);
        w.cond_tag = 0;
        init_x_kernel<<<static_cast<unsigned>((rows + 127) / 128), 128, 0, st>>>(
            fs2_mel ? 0 : 1, fs2_mel, start_noise, d_spec_min.as<float>(), d_spec_max.as<float>(), sched[K - 1].sqrt_ac, sched[K - 1].sqrt_1mac,
            d_seed.as<unsigned long long>(), B, T, M, w.xt.as<float>(), w.xin_hi.as<__nv_bfloat16>(),
            lo ? w.xin_lo.as<__nv_bfloat16>() : nullptr);
        ++launches, ++g_launch_count;
        B200_CUDA(cudaGetLastError());
    }
    if (mel2ph) B200_CUDA(cudaMemcpyAsync(w.mel2ph.p, mel2ph, rows * 8, cudaMemcpyDeviceToDevice, st));
    auto update = [&](int mode, int write_x, int t, const float* e0, const float* e1, const float* e2, const float* e3, bool last) {
        float da, cx, ce;
        plms_coef(alphas_cumprod, t, interval, da, cx, ce);
        plms_update_kernel<false><<<static_cast<unsigned>((rows + 127) / 128), 128, 0, st>>>(
            mode, write_x, da, cx, ce, w.xt.as<float>(), e0, e1, e2, e3, B, T, M, w.xin_hi.as<__nv_bfloat16>(),
            lo ? w.xin_lo.as<__nv_bfloat16>() : nullptr, last ? w.mel.as<float>() : nullptr, d_spec_min.as<float>(), d_spec_max.as<float>(),
            mel2ph ? w.mel2ph.as<int64_t>() : nullptr, nullptr);
        ++launches, ++g_launch_count;
        B200_CUDA(cudaGetLastError());
    };
    // the iterations: deterministic after the start, so the whole loop (K/interval + 1 denoiser evaluations and as many updates) is
    // captured once per (shape, interval, mask, schedule) and replayed, like the ancestral sampler's K steps
    auto body = [&](cudaStream_t s) {
        cudaStream_t saved = st;
        st = s;
        reset_dataflow(w, s);
        int epoch = 0;
        int n_hist = 0, head = 0;   // ring of the last noise predictions: plms_eps[(head - j) & 3] = j-th most recent
        const int t_first = ((K - 1) / interval) * interval;
        for (int t = t_first, it = 0; t >= 0; t -= interval, ++it) {
            head = (head + 1) & 3;
            float* e0 = w.plms_eps[head].as<float>();
            enqueue_step(w, t, it, nullptr, false, false, 1, s, e0, ++epoch);
            const bool last = t - interval < 0;
            const float* e1 = w.plms_eps[(head + 3) & 3].as<float>();
            const float* e2 = w.plms_eps[(head + 2) & 3].as<float>();
            const float* e3 = w.plms_eps[(head + 1) & 3].as<float>();
            if (n_hist == 0) {
                // first iteration (:188-191): predictor step, a second evaluation at max(t - interval, 0), average
                update(0, 0, t, e0, nullptr, nullptr, nullptr, false);
                float* ep = w.eps.as<float>();
                enqueue_step(w, t - interval > 0 ? t - interval : 0, it, nullptr, false, false, 1, s, ep, ++epoch);
                update(1, 1, t, e0, ep, nullptr, nullptr, last);
            } else {
                update(n_hist + 1 > 4 ? 4 : n_hist + 1, 1, t, e0, e1, e2, e3, last);
            }
            if (n_hist < 3) ++n_hist;
        }
        st = saved;
    };
    if (use_graphs) {
        const std::vector<float> ac(alphas_cumprod, alphas_cumprod + cfg.timesteps);
        const bool has_mask = mel2ph != nullptr;
        if (w.plms_graph && (w.plms_interval != interval || w.plms_has_mask != has_mask || w.plms_ac != ac)) {
            cudaGraphExecDestroy(w.plms_graph);
            w.plms_graph = nullptr;
        }
        if (!w.plms_graph) {
            cudaStream_t cs;
            B200_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            cudaGraph_t g = nullptr;
            const unsigned long long before = launches;
            B200_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            try {
                body(cs);
            } catch (...) {
                cudaStreamEndCapture(cs, &g);
                if (g) cudaGraphDestroy(g);
                cudaStreamDestroy(cs);
                throw;
            }
            B200_CUDA(cudaStreamEndCapture(cs, &g));
            w.plms_nodes = launches - before;
            launches = before;
            g_launch_count -= w.plms_nodes;
            B200_CUDA(cudaGraphInstantiate(&w.plms_graph, g, 0));
            cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            w.plms_interval = interval;
            w.plms_has_mask = has_mask;
            w.plms_ac = ac;
        }
        B200_CUDA(cudaGraphLaunch(w.plms_graph, st));
        launches += w.plms_nodes, g_launch_count += w.plms_nodes;
    } else {
        body(st);
    }
    B200_CUDA(cudaMemcpyAsync(mel_out, w.mel.p, rows * M * 4, cudaMemcpyDeviceToDevice, st));
    if (x_final) B200_CUDA(cudaMemcpyAsync(x_final, w.xt.p, rows * M * 4, cudaMemcpyDeviceToDevice, st));
}

void DiffusionPlan::denoise(const float* spec, int t, const float* cond, int B, int T, float* eps_out, cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CHECK(t >= 0 && t < cfg.k_step, "diffusion step outside the plan's LUT (0 <= t < k_step)");
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    const int M = cfg.in_dims, H = cfg.hidden_size;
    const size_t rows = static_cast<size_t>(B) * T;
    const bool lo = terms_side == 3;
    const size_t n = rows * H;
    split_kernel<<<static_cast<unsigned>((n / 4 + 255) / 256 + 1), 256, 0, st>>>(cond, w.cond_hi.as<__nv_bfloat16>(),
                                                                                lo ? w.cond_lo.as<__nv_bfloat16>() : nullptr, n);
    init_x_kernel<<<static_cast<unsigned>((rows + 127) / 128), 128, 0, st>>>(2, nullptr, spec, nullptr, nullptr, 0.f, 0.f, nullptr, B, T, M,
                                                                             nullptr, w.xin_hi.as<__nv_bfloat16>(),
                                                                             lo ? w.xin_lo.as<__nv_bfloat16>() : nullptr);
    launches += 2, g_launch_count += 2;
    B200_CUDA(cudaGetLastError());
    precompute_cond(w, st);
    w.cond_tag = 0;
    reset_dataflow(w, st);
    enqueue_step(w, t, 0, nullptr, false, false, 1, st, nullptr, 1);
    B200_CUDA(cudaMemcpyAsync(eps_out, w.eps.p, rows * M * 4, cudaMemcpyDeviceToDevice, st));
}

// ---------------------------------------------------------------------------------------------
// step calls: q_sample / p_sample / DiffNet.forward / the PLMS update with a diffusion step per batch item
// ---------------------------------------------------------------------------------------------

// Checks 0 <= t[b] < limit; returns whether all items share one step
static bool check_steps(const int* t, int B, int limit) {
    B200_CHECK(t != nullptr, "t is required");
    bool uniform = true;
    for (int b = 0; b < B; ++b) {
        B200_CHECK(t[b] >= 0 && t[b] < limit, "diffusion step t[" + std::to_string(b) + "] = " + std::to_string(t[b]) +
                                                  " outside [0, " + std::to_string(limit) + ")");
        uniform = uniform && t[b] == t[0];
    }
    return uniform;
}

// t (host) -> w.t_of_b; coef (host, n_coef floats per item, or none) -> w.step_coef
void DiffusionPlan::stage_steps(Workspace& w, const int* t, const float* coef, int n_coef, cudaStream_t st) {
    const size_t B = static_cast<size_t>(w.B);
    if (w.t_of_b.p == nullptr) {
        w.t_of_b.alloc(B * sizeof(int));
        w.step_coef.alloc(B * 5 * sizeof(float));
    }
    B200_CUDA(cudaMemcpyAsync(w.t_of_b.p, t, B * sizeof(int), cudaMemcpyHostToDevice, st));
    if (coef) B200_CUDA(cudaMemcpyAsync(w.step_coef.p, coef, B * n_coef * sizeof(float), cudaMemcpyHostToDevice, st));
}

// Conditioner projections of all layers for `cond`, unless the workspace already holds those of the same nonzero tag
void DiffusionPlan::prepare_cond(Workspace& w, const float* cond, unsigned long long tag, cudaStream_t st) {
    if (tag != 0 && tag == w.cond_tag) return;
    const bool lo = terms_side == 3;
    const size_t n = static_cast<size_t>(w.B) * w.T * cfg.hidden_size;
    split_kernel<<<static_cast<unsigned>((n / 4 + 255) / 256 + 1), 256, 0, st>>>(cond, w.cond_hi.as<__nv_bfloat16>(),
                                                                                lo ? w.cond_lo.as<__nv_bfloat16>() : nullptr, n);
    ++launches, ++g_launch_count;
    B200_CUDA(cudaGetLastError());
    precompute_cond(w, st);
    w.cond_tag = tag;
}

// x [B][M][T] -> the sampler state w.xt and its operand copy w.xin
void DiffusionPlan::import_x(Workspace& w, const float* x, cudaStream_t st) {
    const size_t rows = static_cast<size_t>(w.B) * w.T;
    const int M = cfg.in_dims;
    if (x != w.xt.as<float>()) B200_CUDA(cudaMemcpyAsync(w.xt.p, x, rows * M * 4, cudaMemcpyDeviceToDevice, st));
    init_x_kernel<<<static_cast<unsigned>((rows + 127) / 128), 128, 0, st>>>(2, nullptr, x, nullptr, nullptr, 0.f, 0.f, nullptr, w.B, w.T, M,
                                                                             nullptr, w.xin_hi.as<__nv_bfloat16>(),
                                                                             terms_side == 3 ? w.xin_lo.as<__nv_bfloat16>() : nullptr);
    ++launches, ++g_launch_count;
    B200_CUDA(cudaGetLastError());
}

// A small host table copied to the device for the kernels of ONE call on `st`.  Stream-ordered allocation: another call on another stream
// gets its own copy, and the memory goes back to the pool when the call's work is done.
struct StreamTable {
    void* p = nullptr;
    cudaStream_t st;
    StreamTable(const std::vector<float>& host, cudaStream_t s) : st(s) {
        B200_CUDA(cudaMallocAsync(&p, host.size() * sizeof(float), st));
        B200_CUDA(cudaMemcpyAsync(p, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    ~StreamTable() { if (p) cudaFreeAsync(p, st); }
    const float* f() const { return static_cast<const float*>(p); }
};

void DiffusionPlan::q_sample(const float* x_start, const int* t, const float* noise, unsigned long long seed, int B, int T, float* x_out,
                             cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CHECK(x_start != nullptr && x_out != nullptr, "x_start and x_out are required");
    check_steps(t, B, cfg.timesteps);
    B200_CUDA(cudaSetDevice(device));
    std::vector<float> coef(static_cast<size_t>(B) * 2);
    for (int b = 0; b < B; ++b) {
        coef[2 * b] = sched[t[b]].sqrt_ac;
        coef[2 * b + 1] = sched[t[b]].sqrt_1mac;
    }
    const StreamTable tab(coef, st);
    if (noise == nullptr) B200_CUDA(cudaMemcpyAsync(d_seed.p, &seed, sizeof(seed), cudaMemcpyHostToDevice, st));
    const long long n = static_cast<long long>(B) * cfg.in_dims * T;
    q_sample_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(x_start, noise, tab.f(), d_seed.as<unsigned long long>(), B,
                                                                           cfg.in_dims, T, x_out);
    ++launches, ++g_launch_count;
    B200_CUDA(cudaGetLastError());
}

void DiffusionPlan::p_sample(const float* x, const int* t, const float* cond, unsigned long long cond_tag, const float* noise,
                             unsigned long long seed, bool clip_denoised, int B, int T, float* x_out, cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CHECK(x != nullptr && cond != nullptr && x_out != nullptr, "x, cond and x_out are required");
    const bool uniform = check_steps(t, B, cfg.k_step);
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    const int M = cfg.in_dims, K = cfg.k_step;
    // the existing uniform-step kernels unless the items' steps differ (or the clamp is to be skipped: only the per-item posterior has the flag)
    const int rows = (uniform ? 0 : kRowsNet) | ((uniform && clip_denoised) ? 0 : kRowsPost) | (clip_denoised ? 0 : kRowsNoClip);
    std::vector<float> coef(static_cast<size_t>(B) * 5);
    for (int b = 0; b < B; ++b) {
        const StepCoef& sc = sched[t[b]];
        const float c[5] = {sc.c0, sc.c1, sc.c2, sc.c3, sc.sigma};   // sigma = 0 at t == 0: no noise (nonzero_mask, :165)
        std::copy(c, c + 5, &coef[5 * static_cast<size_t>(b)]);
    }
    stage_steps(w, t, coef.data(), 5, st);
    if (noise == nullptr) B200_CUDA(cudaMemcpyAsync(d_seed.p, &seed, sizeof(seed), cudaMemcpyHostToDevice, st));
    prepare_cond(w, cond, cond_tag, st);
    import_x(w, x, st);
    reset_dataflow(w, st);
    // device noise of item b: the stream sample() uses at the executed step K-1-t_b
    enqueue_step(w, t[0], K - 1 - t[0], noise, false, false, 0, st, nullptr, 1, rows);
    B200_CUDA(cudaMemcpyAsync(x_out, w.xt.p, static_cast<size_t>(B) * T * M * 4, cudaMemcpyDeviceToDevice, st));
}

void DiffusionPlan::denoise_steps(const float* spec, const int* t, const float* cond, unsigned long long cond_tag, int B, int T, float* eps_out,
                                  cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CHECK(spec != nullptr && cond != nullptr && eps_out != nullptr, "spec, cond and eps_out are required");
    const bool uniform = check_steps(t, B, cfg.k_step);
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    stage_steps(w, t, nullptr, 0, st);
    prepare_cond(w, cond, cond_tag, st);
    import_x(w, spec, st);
    reset_dataflow(w, st);
    enqueue_step(w, t[0], 0, nullptr, false, false, 1, st, eps_out, 1, uniform ? 0 : kRowsNet);
}

void DiffusionPlan::plms_update(const float* x, const int* t, const float* alphas_cumprod, int interval, int n_eps, const float* const* eps,
                                int B, int T, float* x_out, cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CHECK(x != nullptr && x_out != nullptr && alphas_cumprod != nullptr, "x, alphas_cumprod and x_out are required");
    B200_CHECK(interval >= 1, "interval must be >= 1");
    B200_CHECK(n_eps >= 0 && n_eps <= 4, "n_eps must be 0 (predictor), 1 (two evaluations) or 2..4 (history terms)");
    const int n_needed = n_eps == 0 ? 1 : (n_eps == 1 ? 2 : n_eps);
    for (int j = 0; j < n_needed; ++j) B200_CHECK(eps[j] != nullptr, "eps" + std::to_string(j) + " is required for n_eps = " + std::to_string(n_eps));
    check_steps(t, B, cfg.timesteps);
    B200_CUDA(cudaSetDevice(device));
    const int M = cfg.in_dims;
    const size_t rows = static_cast<size_t>(B) * T;
    // get_x_pred coefficients in fp32, same operation order as the reference (:175-180) and sample_plms; a_prev at max(t_b - interval, 0).
    // An element-wise update: no workspace, no operand copy (the next denoiser call imports x itself).
    std::vector<float> coef(static_cast<size_t>(B) * 3);
    for (int b = 0; b < B; ++b) plms_coef(alphas_cumprod, t[b], interval, coef[3 * b], coef[3 * b + 1], coef[3 * b + 2]);
    const StreamTable tab(coef, st);
    if (x_out != x) B200_CUDA(cudaMemcpyAsync(x_out, x, rows * M * 4, cudaMemcpyDeviceToDevice, st));
    plms_update_kernel<true><<<static_cast<unsigned>((rows + 127) / 128), 128, 0, st>>>(
        n_eps, 1, 0.f, 0.f, 0.f, x_out, eps[0], eps[1], eps[2], eps[3], B, T, M, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, tab.f());
    ++launches, ++g_launch_count;
    B200_CUDA(cudaGetLastError());
}

}  // namespace b200
