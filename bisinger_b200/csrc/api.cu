// extern "C" boundary of libbisinger_b200.so (see include/bisinger_b200.h). Nothing throws across it.
#include <string>

#include "plans.h"

namespace b200 {
unsigned long long g_launch_count = 0;
}

namespace {
thread_local std::string g_last_error;

template <class F>
int guarded(F&& f) {
    try {
        f();
        return 0;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return 1;
    } catch (...) {
        g_last_error = "unknown error";
        return 2;
    }
}
}  // namespace

struct bsg_diffusion_plan {
    b200::DiffusionPlan impl;
    template <class... A> explicit bsg_diffusion_plan(A&&... a) : impl(std::forward<A>(a)...) {}
};
struct bsg_hifigan_plan {
    b200::HifiganPlan impl;
    template <class... A> explicit bsg_hifigan_plan(A&&... a) : impl(std::forward<A>(a)...) {}
};

struct bsg_pe_plan {
    b200::PitchExtractorPlan impl;
    template <class... A> explicit bsg_pe_plan(A&&... a) : impl(std::forward<A>(a)...) {}
};

struct bsg_fft_plan {
    b200::FftDecoderPlan impl;
    template <class... A> explicit bsg_fft_plan(A&&... a) : impl(std::forward<A>(a)...) {}
};

extern "C" {

int bsg_abi_version(void) { return BSG_ABI_VERSION; }
const char* bsg_last_error(void) { return g_last_error.c_str(); }
unsigned long long bsg_kernel_launch_count(void) { return b200::g_launch_count; }

int bsg_diffusion_plan_create(const bsg_diffnet_config* cfg, const float* weights_host, size_t n_weights, const bsg_schedule* sched,
                              const float* spec_min, const float* spec_max, int device, bsg_diffusion_plan** out) {
    return guarded([&] {
        B200_CHECK(cfg && weights_host && sched && spec_min && spec_max && out, "null argument");
        *out = new bsg_diffusion_plan(*cfg, weights_host, n_weights, *sched, spec_min, spec_max, device);
    });
}
void bsg_diffusion_plan_destroy(bsg_diffusion_plan* plan) { delete plan; }

int bsg_diffusion_sample(bsg_diffusion_plan* plan, const float* cond, const float* fs2_mel, const float* start_noise,
                         const float* step_noise, unsigned long long seed, const int64_t* mel2ph, int B, int T, float* mel_out,
                         float* x_final, void* stream) {
    return guarded([&] {
        B200_CHECK(plan, "null plan");
        plan->impl.sample(cond, fs2_mel, start_noise, step_noise, seed, mel2ph, B, T, mel_out, x_final, static_cast<cudaStream_t>(stream));
    });
}

int bsg_diffusion_sample_plms(bsg_diffusion_plan* plan, const float* cond, const float* fs2_mel, const float* start_noise,
                              unsigned long long seed, const int64_t* mel2ph, const float* alphas_cumprod_host, int interval, int B,
                              int T, float* mel_out, float* x_final, void* stream) {
    return guarded([&] {
        B200_CHECK(plan, "null plan");
        plan->impl.sample_plms(cond, fs2_mel, start_noise, seed, mel2ph, alphas_cumprod_host, interval, B, T, mel_out, x_final,
                               static_cast<cudaStream_t>(stream));
    });
}

int bsg_diffnet_forward(bsg_diffusion_plan* plan, const float* spec, int t, const float* cond, int B, int T, float* eps_out,
                        void* stream) {
    return guarded([&] {
        B200_CHECK(plan && spec && cond && eps_out, "null argument");
        plan->impl.denoise(spec, t, cond, B, T, eps_out, static_cast<cudaStream_t>(stream));
    });
}

int bsg_diffusion_q_sample(bsg_diffusion_plan* plan, const float* x_start, const int* t, const float* noise, unsigned long long seed, int B,
                           int T, float* x_out, void* stream) {
    return guarded([&] {
        B200_CHECK(plan, "null plan");
        plan->impl.q_sample(x_start, t, noise, seed, B, T, x_out, static_cast<cudaStream_t>(stream));
    });
}

int bsg_diffusion_p_sample(bsg_diffusion_plan* plan, const float* x, const int* t, const float* cond, unsigned long long cond_tag,
                           const float* noise, unsigned long long seed, int clip_denoised, int B, int T, float* x_out, void* stream) {
    return guarded([&] {
        B200_CHECK(plan, "null plan");
        plan->impl.p_sample(x, t, cond, cond_tag, noise, seed, clip_denoised != 0, B, T, x_out, static_cast<cudaStream_t>(stream));
    });
}

int bsg_diffnet_forward_steps(bsg_diffusion_plan* plan, const float* spec, const int* t, const float* cond, unsigned long long cond_tag, int B,
                              int T, float* eps_out, void* stream) {
    return guarded([&] {
        B200_CHECK(plan, "null plan");
        plan->impl.denoise_steps(spec, t, cond, cond_tag, B, T, eps_out, static_cast<cudaStream_t>(stream));
    });
}

int bsg_diffusion_plms_update(bsg_diffusion_plan* plan, const float* x, const int* t, const float* alphas_cumprod_host, int interval, int n_eps,
                              const float* eps0, const float* eps1, const float* eps2, const float* eps3, int B, int T, float* x_out,
                              void* stream) {
    return guarded([&] {
        B200_CHECK(plan, "null plan");
        const float* eps[4] = {eps0, eps1, eps2, eps3};
        plan->impl.plms_update(x, t, alphas_cumprod_host, interval, n_eps, eps, B, T, x_out, static_cast<cudaStream_t>(stream));
    });
}

int bsg_diffusion_time_kernel(bsg_diffusion_plan* plan, int which, int B, int T, int reps, float* avg_ms, void* stream) {
    return guarded([&] {
        B200_CHECK(plan && avg_ms, "null argument");
        *avg_ms = plan->impl.time_kernel(which, B, T, reps, static_cast<cudaStream_t>(stream));
    });
}

int bsg_hifigan_plan_create(const bsg_hifigan_config* cfg, const float* weights_host, size_t n_weights, int device,
                            bsg_hifigan_plan** out) {
    return guarded([&] {
        B200_CHECK(cfg && weights_host && out, "null argument");
        *out = new bsg_hifigan_plan(*cfg, weights_host, n_weights, device);
    });
}
void bsg_hifigan_plan_destroy(bsg_hifigan_plan* plan) { delete plan; }

int bsg_hifigan_forward(bsg_hifigan_plan* plan, const float* mel, const float* f0, const float* rand_ini, const float* src_noise,
                        unsigned long long seed, int B, int T, float* wav, void* stream) {
    return guarded([&] {
        B200_CHECK(plan && mel && wav, "null argument");
        plan->impl.forward(mel, f0, rand_ini, src_noise, seed, B, T, wav, static_cast<cudaStream_t>(stream));
    });
}

int bsg_hifigan_source(bsg_hifigan_plan* plan, const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed,
                       int B, int T, float* har_source, void* stream) {
    return guarded([&] {
        B200_CHECK(plan && f0 && har_source, "null argument");
        plan->impl.source(f0, rand_ini, src_noise, seed, B, T, har_source, static_cast<cudaStream_t>(stream));
    });
}

int bsg_pe_plan_create(const bsg_pe_config* cfg, const float* weights_host, size_t n_weights, int device, bsg_pe_plan** out) {
    return guarded([&] {
        B200_CHECK(cfg && weights_host && out, "null argument");
        *out = new bsg_pe_plan(*cfg, weights_host, n_weights, device);
    });
}
void bsg_pe_plan_destroy(bsg_pe_plan* plan) { delete plan; }

int bsg_pe_forward(bsg_pe_plan* plan, const float* mel, int B, int T, float* pitch_pred, float* f0, void* stream) {
    return guarded([&] {
        B200_CHECK(plan && mel && pitch_pred && f0, "null argument");
        plan->impl.forward(mel, B, T, pitch_pred, f0, static_cast<cudaStream_t>(stream));
    });
}

int bsg_fft_plan_create(const bsg_fft_config* cfg, const float* weights_host, size_t n_weights, int device, bsg_fft_plan** out) {
    return guarded([&] {
        B200_CHECK(cfg && weights_host && out, "null argument");
        *out = new bsg_fft_plan(*cfg, weights_host, n_weights, device);
    });
}
void bsg_fft_plan_destroy(bsg_fft_plan* plan) { delete plan; }

int bsg_fft_forward(bsg_fft_plan* plan, const float* x, const float* tgt_nonpad, int B, int T, float* hidden_out, float* mel_out,
                    void* stream) {
    return guarded([&] {
        B200_CHECK(plan && x, "null argument");
        plan->impl.forward(x, tgt_nonpad, B, T, hidden_out, mel_out, static_cast<cudaStream_t>(stream));
    });
}

int bsg_fft_forward_masked(bsg_fft_plan* plan, const float* x, const unsigned char* padding_mask, const float* tgt_nonpad, int B, int T,
                           float* hidden_out, float* mel_out, void* stream) {
    return guarded([&] {
        B200_CHECK(plan && x && padding_mask, "null argument");
        plan->impl.forward(x, tgt_nonpad, B, T, hidden_out, mel_out, static_cast<cudaStream_t>(stream), padding_mask);
    });
}

int bsg_selftest_conv(const float* a_dev, const float* w_host, const float* bias_host, int B, int L, int Cin, int N, int ntaps,
                      const int* shifts, int n_tile, int precision, float* out_dev, void* stream) {
    using namespace b200;
    return guarded([&] {
        B200_CHECK(a_dev && w_host && bias_host && shifts && out_dev, "null argument");
        B200_CHECK(Cin % 8 == 0 && N % n_tile == 0 && ntaps >= 1 && ntaps <= kMaxTaps, "bad shape");
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        // test hooks: 0x100 = the 2-CTA (cta_group::2) variant of the kernel, 0x200 = two pairs per cluster with multicast weights
        const int pair = (precision & 0x200) ? 2 : ((precision & 0x100) ? 1 : 0);
        const int prec = precision & 0xff;
        const int terms = prec == BSG_PRECISION_BF16X3 ? 3 : (prec == BSG_PRECISION_FP16X2 ? 2 : 1);
        const size_t rows = static_cast<size_t>(B) * L;
        // activations -> bf16 hi/lo (same split kernel the plans use is file-local; do it on the host here)
        std::vector<float> a_host(rows * Cin);
        B200_CUDA(cudaMemcpyAsync(a_host.data(), a_dev, a_host.size() * 4, cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        std::vector<uint16_t> ah(a_host.size()), al(a_host.size());
        for (size_t i = 0; i < a_host.size(); ++i) {
            if (terms == 2) { ah[i] = f32_to_f16_bits(a_host[i]); al[i] = 0; continue; }   // fp16x2: one fp16 activation operand
            ah[i] = f32_to_bf16_bits(a_host[i]);
            al[i] = f32_to_bf16_bits(a_host[i] - bf16_bits_to_f32(ah[i]));
        }
        DevBuf d_ah, d_al, d_bias;
        upload(d_ah, ah);
        upload(d_al, al);
        upload(d_bias, std::vector<float>(bias_host, bias_host + N));
        // weights [N][ntaps][Cin] -> K-major [N][ntaps * Cpad] (Cpad = Cin rounded up to a k-block)
        const int n_kb = (Cin + kBlockK - 1) / kBlockK;
        const int Cpad = n_kb * kBlockK;
        std::vector<float> wp(static_cast<size_t>(N) * ntaps * Cpad, 0.0f);
        for (int n = 0; n < N; ++n)
            for (int tp = 0; tp < ntaps; ++tp)
                for (int c = 0; c < Cin; ++c)
                    wp[(static_cast<size_t>(n) * ntaps + tp) * Cpad + c] = w_host[(static_cast<size_t>(n) * ntaps + tp) * Cin + c];
        PackedW pw;
        pw.pack(wp, N, ntaps * Cpad, terms == 2);
        ConvGemmArgs a{};
        set_geometry(a, B, L, N, n_tile, pair != 0);
        const int rows_box = set_taps(a, 0, 0, n_kb, shifts, ntaps, Cpad);
        a.amap[0] = make_act_tmap(d_ah.p, B, L, Cin, 0, rows_box);
        a.amap[1] = make_act_tmap(d_al.p, B, L, Cin, 0, rows_box);
        pw.maps(pair == 2 ? n_tile / 4 : (pair ? n_tile / 2 : n_tile), a.wmap[0], a.wmap[1]);
        a.epi.bias = d_bias.as<float>();
        a.epi.f32_a = out_dev;
        a.epi.out_pitch = N;
        a.epi.acc_scale = pw.acc_scale;
        launch_conv_gemm(n_tile, terms, EPI_F32, a, st, pair);
        ++g_launch_count;
        B200_CUDA(cudaStreamSynchronize(st));
    });
}

}  // extern "C"
