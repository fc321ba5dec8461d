// HiFi-GAN generator with NSF harmonic source on the conv_gemm kernel.
//
// Reference (relative to /root/reference/train_bisinger/):
//   modules/hifigan/hifigan.py:144-173 (HifiGanGenerator.forward), :54-61 (ResBlock1.forward), :104-142 (ctor)
//   modules/parallel_wavegan/models/source.py:45-74,105-138 (SineGen), :386-399 (SourceModuleHnNSF.forward)
//
// Layout: every activation is channels-last, rows = b*L_i + l.  Per up-sampling stage i (C_i channels, L_i samples):
//   X0  f32  [rows][C]   stage input x (transposed conv + noise branch), residual of the first ResBlock iteration
//   A0  bf16 [rows][C]   lrelu(X0): A operand shared by the three ResBlocks
//   Xr  f32  [rows][C]   running residual x of the current ResBlock
//   Ar  bf16 [rows][C]   lrelu(Xr)
//   Tb  bf16 [rows][C]   lrelu(convs1 output)
//   S   f32  [rows][C]   MRF accumulator sum_j ResBlock_j(x) / num_kernels
// For C < 64 the TMA box (64 channels) is wider than the tensor: the out-of-bounds half of every swizzle row is
// zero-filled by the TMA unit and the packed weights carry matching zero columns, so no padded copies are stored.
// ConvTranspose1d (stride u) is run as u independent convolutions, one per output phase p: rows of the input, taps
// delta with 0 <= delta*u + p + pad < k, written to columns [p*Cout, (p+1)*Cout) of the [rows_in][u*Cout] view of the
// output (which is the same memory as [rows_in*u][Cout]).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <memory>

#include "plans.h"
#include "resblock_fused.cuh"

namespace b200 {

namespace {
constexpr float kLrelu = 0.1f;   // LRELU_SLOPE, hifigan.py:11

// mel f32 [B][M][T] -> bf16 [B*T][M] (A operand of conv_pre)
__global__ void mel_prep_kernel(const float* __restrict__ mel, int B, int M, int T, __nv_bfloat16* __restrict__ out) {
    const long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= static_cast<long long>(B) * T) return;
    const int b = static_cast<int>(r / T), t = static_cast<int>(r % T);
    for (int c = 0; c < M; ++c) out[r * M + c] = __float2bfloat16_rn(mel[(static_cast<long long>(b) * M + c) * T + t]);
}

// Phase at the start of each frame.  source.py:51-74: rad = (f0*h/sr) % 1 per sample, rad[0] += rand_ini, phase = cumsum(rad)
// (the reference subtracts 1 at every wrap only to keep the fp32 running sum small; sin(2*pi*x) is invariant to it).
// f0 is constant over a frame (nearest up-sampling, hifigan.py:113,147), so the cumulative phase at sample i of frame t is
// P[t] + (i+1)*rad[t].  P is kept as a 64-bit FIXED-POINT fraction of a turn (2^64 = one turn): rad is an fp32 number in [0,1), so
// rad * 2^64 is an exact integer, the running sum is exact, and the "modulo 1" is the wrap of unsigned arithmetic -- no rounding
// accumulates over a 60 s segment, and the scan needs no fp64 (whose latency made the serial scan 330 us).
__device__ __forceinline__ unsigned long long turn_fixed(float r) {   // r in [0,1) -> r * 2^64, exact, integer only
    const unsigned int u = __float_as_uint(r);
    const int e = static_cast<int>((u >> 23) & 0xffu);
    const unsigned long long m = (u & 0x7fffffu) | (e ? 0x800000u : 0u);
    const int sh = (e ? e : 1) - 127 + 41;            // r = m * 2^(e-150)  =>  r * 2^64 = m * 2^(e-86); e <= 126 => sh <= 40
    return sh >= 0 ? (m << sh) : (sh > -64 ? (m >> -sh) : 0ull);
}
__device__ __forceinline__ float rad_of(float f0, int h, float sr) {
    const float r = f0 * static_cast<float>(h + 1) / sr;
    return r - floorf(r);
}
// One warp per (utterance, harmonic): 32 frames per iteration, inclusive shuffle scan of the 64-bit increments plus a running carry.
// Integer addition is associative, so the result is bit-identical to a serial scan.
// rand_ini == nullptr (production): the initial phase of every harmonic h >= 1 is drawn U[0,1) on the device from the Philox key
// (torch.rand(B, dim) at source.py:54; the fundamental gets none, :56) -- 24 random bits, so the value is exactly representable.
__global__ void nsf_phase_kernel(const float* __restrict__ f0, const float* __restrict__ rand_ini,
                                 const unsigned long long* __restrict__ seed_ptr, int B, int T, int hop, int dim, float sr,
                                 unsigned long long* __restrict__ phase0) {
    const int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (idx >= B * dim) return;
    const int b = idx / dim, h = idx % dim;
    float ri = 0.0f;                                                              // rand_ini[:,0] = 0 (:56)
    if (h != 0) {
        if (rand_ini != nullptr) {
            ri = rand_ini[b * dim + h];
        } else {
            const unsigned long long seed = __ldg(seed_ptr);
            const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(idx), 0u, 0x1417u, 0x5eedu),
                                          make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
            ri = static_cast<float>(r.x >> 8) * 5.9604644775390625e-08f;          // [0, 1)
        }
    }
    ri = ri - floorf(ri);
    unsigned long long carry = turn_fixed(ri);
    const float* f = f0 + static_cast<long long>(b) * T;
    unsigned long long* out = phase0 + static_cast<long long>(b) * T * dim + h;
    for (int t0 = 0; t0 < T; t0 += 32) {
        const int t = t0 + lane;
        const unsigned long long inc = t < T ? static_cast<unsigned long long>(hop) * turn_fixed(rad_of(__ldg(f + t), h, sr)) : 0ull;
        unsigned long long v = inc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += u;
        }
        if (t < T) out[static_cast<long long>(t) * dim] = carry + v - inc;   // phase at the START of frame t
        carry += __shfl_sync(0xffffffffu, v, 31);
    }
}

// har_source[b][l] = tanh( Linear_9->1( sine*uv + noise_amp*noise ) )   source.py:121-137,394-395
__global__ void nsf_source_kernel(const float* __restrict__ f0, const unsigned long long* __restrict__ phase0, const float* __restrict__ noise,
                                  const unsigned long long* __restrict__ seed_ptr, const float* __restrict__ lin, int B, int T, int hop,
                                  int dim, float sr, float* __restrict__ har) {
    const long long L = static_cast<long long>(T) * hop;
    const long long g = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (g >= static_cast<long long>(B) * L) return;
    const int b = static_cast<int>(g / L);
    const long long l = g % L;
    const int t = static_cast<int>(l / hop), i = static_cast<int>(l % hop);
    const float f = f0[static_cast<long long>(b) * T + t];
    const float uv = f > 0.0f ? 1.0f : 0.0f;                      // voiced_threshold = 0 (:38-43)
    const float namp = uv * 0.003f + (1.0f - uv) * 0.1f / 3.0f;   // noise_std, sine_amp/3 (:131)
    float acc = lin[dim];                                         // l_linear bias
    const unsigned long long seed = noise ? 0ull : __ldg(seed_ptr);
    float4 zq = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int h = 0; h < dim; ++h) {
        // phase of this sample: P[t] + (i+1)*rad, wrapping = modulo one turn; the top 24 bits are all an fp32 phase can hold
        const unsigned long long ph = phase0[(static_cast<long long>(b) * T + t) * dim + h] +
                                      static_cast<unsigned long long>(i + 1) * turn_fixed(rad_of(f, h, sr));
        const float phf = static_cast<float>(static_cast<unsigned int>(ph >> 40)) * 5.9604644775390625e-08f;   // 2^-24
        const float sine = sinf(phf * 2.0f * 3.14159265358979323846f) * 0.1f;   // sine_amp (:121)
        float z;
        if (noise) {
            z = noise[(static_cast<long long>(b) * L + l) * dim + h];
        } else {   // four normals per Philox call: counter = (sample, h / 4)
            if ((h & 3) == 0) zq = philox_normal4(seed, 0x4E5Fu + static_cast<unsigned>(h >> 2), static_cast<uint64_t>(g));
            z = (h & 3) == 0 ? zq.x : ((h & 3) == 1 ? zq.y : ((h & 3) == 2 ? zq.z : zq.w));
        }
        acc = fmaf(lin[h], sine * uv + namp * z, acc);
    }
    har[g] = tanhf(acc);
}

// x += layer_norm_C( relu( noise_conv(har) ) ); a = lrelu(x)     hifigan.py:155-160
// noise_conv: Conv1d(1 -> C, kernel ksz, stride s, padding pad).  One warp per output row (grid-stride): lane owns
// channels lane, lane+32, ...; the conv weights sit in shared memory as [k][c] (conflict-free), the <= 32 source
// samples of the row's window are held one per lane and broadcast with shuffles; LayerNorm statistics by warp
// shuffles (two-pass, as F.layer_norm); x is read-modified-written with 128-byte coalesced accesses.
template <int CPL>   // channels per lane = C / 32
__global__ void __launch_bounds__(256) noise_branch_kernel(const float* __restrict__ har, const float* __restrict__ w,
                                                           const float* __restrict__ bias, int B, long long Lout, long long Lhar, int ksz,
                                                           int stride, int pad, int has_source, float* __restrict__ x,
                                                           __nv_bfloat16* __restrict__ act, int act_pitch) {
    constexpr int C = CPL * 32;
    extern __shared__ float wsm[];   // [ksz][C] then bias [C]
    if (has_source) {
        for (int i = threadIdx.x; i < ksz * C; i += blockDim.x) wsm[(i % ksz) * C + i / ksz] = w[i];   // w is [C][ksz]
        for (int i = threadIdx.x; i < C; i += blockDim.x) wsm[ksz * C + i] = bias[i];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp_g = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    const long long rows = static_cast<long long>(B) * Lout;
    for (long long row = warp_g; row < rows; row += n_warps) {
        float v[CPL];
#pragma unroll
        for (int j = 0; j < CPL; ++j) v[j] = 0.0f;
        if (has_source) {
            const int b = static_cast<int>(row / Lout);
            const long long l = row % Lout;
            const long long h0 = l * stride - pad;
            float hs = 0.0f;
            if (lane < ksz) {
                const long long hl = h0 + lane;
                if (hl >= 0 && hl < Lhar) hs = har[static_cast<long long>(b) * Lhar + hl];
            }
#pragma unroll
            for (int j = 0; j < CPL; ++j) v[j] = wsm[ksz * C + lane + 32 * j];
            for (int k = 0; k < ksz; ++k) {
                const float hk = __shfl_sync(0xffffffffu, hs, k);
#pragma unroll
                for (int j = 0; j < CPL; ++j) v[j] = fmaf(wsm[k * C + lane + 32 * j], hk, v[j]);
            }
            float sum = 0.0f;
#pragma unroll
            for (int j = 0; j < CPL; ++j) { v[j] = fmaxf(v[j], 0.0f); sum += v[j]; }
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            const float mean = sum / static_cast<float>(C);
            float q = 0.0f;
#pragma unroll
            for (int j = 0; j < CPL; ++j) { v[j] -= mean; q += v[j] * v[j]; }
            for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
            const float rstd = rsqrtf(q / static_cast<float>(C) + 1e-5f);
#pragma unroll
            for (int j = 0; j < CPL; ++j) v[j] *= rstd;
        }
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
            const int c = lane + 32 * j;
            const float xv = x[row * C + c] + v[j];
            x[row * C + c] = xv;
            act[row * act_pitch + c] = __float2bfloat16_rn(xv > 0.0f ? xv : xv * kLrelu);
        }
    }
}

// Same operation, laid out for memory-level parallelism: a row's C channels are spread over LPR = min(32, C/4) lanes as float4s, so a warp
// works on 32/LPR rows at once (C = 32: four rows per warp), two such row groups per loop iteration with all their loads issued before
// the arithmetic; LayerNorm reductions are shuffles within the LPR lanes of a row.  Needs ksz <= LPR (true for every stage of the hop-128
// generator: k = 32, 8, 4, 1 at C = 256, 128, 64, 32); the host falls back to the kernel above otherwise.
template <int C>
__global__ void __launch_bounds__(256) noise_branch_v2_kernel(const float* __restrict__ har, const float* __restrict__ w,
                                                              const float* __restrict__ bias, int B, long long Lout, long long Lhar, int ksz,
                                                              int stride, int pad, int has_source, float* __restrict__ x,
                                                              __nv_bfloat16* __restrict__ act, int act_pitch, int out_f16) {
    // out_f16: the activation is stored as fp16 (the fused ResBlock kernel's 16-bit stream: the ONLY copy of x) and x is not written back
    constexpr int LPR = C >= 128 ? 32 : C / 4;   // lanes per row
    constexpr int RPW = 32 / LPR;                // rows per warp and group
    constexpr int V = C / (LPR * 4);             // float4s per lane
    constexpr int U = C >= 512 ? 2 : 4;          // row groups in flight; a weight float4 read from shared memory serves all of them
    extern __shared__ float wsm[];   // [ksz][C] then bias [C]
    if (has_source) {
        for (int i = threadIdx.x; i < ksz * C; i += blockDim.x) wsm[(i % ksz) * C + i / ksz] = w[i];   // w is [C][ksz]
        for (int i = threadIdx.x; i < C; i += blockDim.x) wsm[ksz * C + i] = bias[i];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, sub = lane % LPR, rsub = lane / LPR;
    const long long warp_g = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    const long long rows = static_cast<long long>(B) * Lout;
    for (long long base = warp_g * (RPW * U); base < rows; base += n_warps * (RPW * U)) {
        float4 xv[U][V];
        float hs[U];
        long long row[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            row[u] = base + u * RPW + rsub;
            const bool ok = row[u] < rows;
            hs[u] = 0.0f;
#pragma unroll
            for (int j = 0; j < V; ++j)
                xv[u][j] = ok ? *reinterpret_cast<const float4*>(x + row[u] * C + (j * LPR + sub) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (has_source && ok && sub < ksz) {
                const int b = static_cast<int>(row[u] / Lout);
                const long long hl = (row[u] % Lout) * stride - pad + sub;
                if (hl >= 0 && hl < Lhar) hs[u] = har[static_cast<long long>(b) * Lhar + hl];
            }
        }
        float v[U][V][4];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < V; ++j) v[u][j][0] = v[u][j][1] = v[u][j][2] = v[u][j][3] = 0.0f;
        if (has_source) {
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const float4 bb = *reinterpret_cast<const float4*>(wsm + ksz * C + (j * LPR + sub) * 4);
#pragma unroll
                for (int u = 0; u < U; ++u) { v[u][j][0] = bb.x; v[u][j][1] = bb.y; v[u][j][2] = bb.z; v[u][j][3] = bb.w; }
            }
            for (int k = 0; k < ksz; ++k) {
                float hk[U];
#pragma unroll
                for (int u = 0; u < U; ++u) hk[u] = __shfl_sync(0xffffffffu, hs[u], k, LPR);
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const float4 ww = *reinterpret_cast<const float4*>(wsm + k * C + (j * LPR + sub) * 4);
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        v[u][j][0] = fmaf(ww.x, hk[u], v[u][j][0]); v[u][j][1] = fmaf(ww.y, hk[u], v[u][j][1]);
                        v[u][j][2] = fmaf(ww.z, hk[u], v[u][j][2]); v[u][j][3] = fmaf(ww.w, hk[u], v[u][j][3]);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float sum = 0.0f;
#pragma unroll
                for (int j = 0; j < V; ++j)
#pragma unroll
                    for (int q = 0; q < 4; ++q) { v[u][j][q] = fmaxf(v[u][j][q], 0.0f); sum += v[u][j][q]; }
#pragma unroll
                for (int o = LPR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                const float mean = sum / static_cast<float>(C);
                float qq = 0.0f;
#pragma unroll
                for (int j = 0; j < V; ++j)
#pragma unroll
                    for (int q = 0; q < 4; ++q) { v[u][j][q] -= mean; qq += v[u][j][q] * v[u][j][q]; }
#pragma unroll
                for (int o = LPR / 2; o > 0; o >>= 1) qq += __shfl_xor_sync(0xffffffffu, qq, o);
                const float rstd = rsqrtf(qq / static_cast<float>(C) + 1e-5f);
#pragma unroll
                for (int j = 0; j < V; ++j)
#pragma unroll
                    for (int q = 0; q < 4; ++q) v[u][j][q] *= rstd;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (row[u] < rows) {
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int c = (j * LPR + sub) * 4;
                    const float4 o4 = make_float4(xv[u][j].x + v[u][j][0], xv[u][j].y + v[u][j][1], xv[u][j].z + v[u][j][2],
                                                  xv[u][j].w + v[u][j][3]);
                    uint2 pk;
                    if (out_f16) {
                        pk.x = pack_h2(lrelu_f(o4.x, kLrelu), lrelu_f(o4.y, kLrelu));
                        pk.y = pack_h2(lrelu_f(o4.z, kLrelu), lrelu_f(o4.w, kLrelu));
                    } else {
                        *reinterpret_cast<float4*>(x + row[u] * C + c) = o4;
                        const __nv_bfloat162 a0 = __floats2bfloat162_rn(o4.x > 0.0f ? o4.x : o4.x * kLrelu, o4.y > 0.0f ? o4.y : o4.y * kLrelu);
                        const __nv_bfloat162 a1 = __floats2bfloat162_rn(o4.z > 0.0f ? o4.z : o4.z * kLrelu, o4.w > 0.0f ? o4.w : o4.w * kLrelu);
                        pk.x = *reinterpret_cast<const uint32_t*>(&a0);
                        pk.y = *reinterpret_cast<const uint32_t*>(&a1);
                    }
                    *reinterpret_cast<uint2*>(act + row[u] * act_pitch + c) = pk;
                }
            }
        }
    }
}

// wav = tanh( conv_post( lrelu(x, 0.01) ) )   hifigan.py:169-171 ; conv_post: Conv1d(C -> 1, k, padding (k-1)/2), C == 32.
// A block stages blockDim + k - 1 rows of lrelu(x) in shared memory (pitch 33: conflict-free) with coalesced loads.
// HALF_IN: x is the fused path's fp16 tensor with leaky_relu(0.01) already applied by the producing epilogue.
template <bool HALF_IN>
__global__ void __launch_bounds__(256) conv_post_kernel(const void* __restrict__ xin, const float* __restrict__ w,
                                                        const float* __restrict__ bias, int B, long long L, int ksz,
                                                        float* __restrict__ wav) {
    constexpr int C = 32, P = 33;
    extern __shared__ float sm[];
    float* wsm = sm;                  // [ksz][C]
    float* xs = sm + ksz * C;         // [blockDim + ksz - 1][P]
    const int half = (ksz - 1) / 2;
    for (int i = threadIdx.x; i < ksz * C; i += blockDim.x) wsm[i] = w[i];
    const long long g0 = static_cast<long long>(blockIdx.x) * blockDim.x;   // first output sample (flattened b*L + l) of this block
    const long long total = static_cast<long long>(B) * L;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int nrows = blockDim.x + ksz - 1;
    for (int r = warp; r < nrows; r += nwarp) {
        const long long g = g0 + r - half;          // flattened source row
        float v = 0.0f;
        if (g >= 0 && g < total) {
            if (HALF_IN) {
                v = __half2float(reinterpret_cast<const __half*>(xin)[g * C + lane]);
            } else {
                v = reinterpret_cast<const float*>(xin)[g * C + lane];
                v = v > 0.0f ? v : v * 0.01f;
            }
        }
        xs[r * P + lane] = v;
    }
    __syncthreads();
    const long long g = g0 + threadIdx.x;
    if (g >= total) return;
    const long long l = g % L;
    float acc = bias[0];
    for (int k = 0; k < ksz; ++k) {
        const long long ll = l + k - half;
        if (ll < 0 || ll >= L) continue;              // zero padding at the ends of every batch item
        const float* xr = xs + (threadIdx.x + k) * P;
        const float* ww = wsm + k * C;
#pragma unroll
        for (int c = 0; c < C; ++c) acc = fmaf(ww[c], xr[c], acc);
    }
    wav[g] = tanhf(acc);
}

std::vector<float> take(const float*& p, size_t n) {
    std::vector<float> v(p, p + n);
    p += n;
    return v;
}
int ntile_for(int cout) { return cout >= 256 ? 256 : cout; }
}  // namespace

struct HifiganPlan::Workspace {
    int B = 0, T = 0;
    DevBuf mel16, har, phase0, upin[2], X0, Xr, S, A0, Ar, Tb;
    // graph path (no injected noise): plan-owned copies of the caller's buffers, so that the captured launches see fixed addresses
    DevBuf in_mel, in_f0, out_wav;
    cudaGraphExec_t graph[2] = {nullptr, nullptr};   // [has_src]
    unsigned long long graph_nodes[2] = {0, 0};
    unsigned long long last_use = 0;                 // LRU stamp
    size_t bytes = 0;
    ~Workspace() {
        for (auto& g : graph)
            if (g) cudaGraphExecDestroy(g);
    }
};

// ---------------------------------------------------------------------------------------------
HifiganPlan::HifiganPlan(const bsg_hifigan_config& c, const float* w, size_t n_w, int device) : cfg(c), device(device) {
    B200_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    B200_CUDA(cudaGetDeviceProperties(&prop, device));
    B200_CHECK(prop.major == 10, "bisinger_b200 requires an sm_100 (B200) device -- there is no fallback path");
    B200_CHECK(c.num_upsamples >= 1 && c.num_upsamples <= BSG_MAX_UPSAMPLES, "bad num_upsamples");
    B200_CHECK(c.num_kernels >= 1 && c.num_kernels <= BSG_MAX_RESBLOCK_KERNELS, "bad num_kernels");
    B200_CHECK(c.num_dilations >= 1 && c.num_dilations <= BSG_MAX_RESBLOCK_DILATIONS, "bad num_dilations");
    B200_CHECK(c.num_mels % 8 == 0, "num_mels must be a multiple of 8");
    const int C0 = c.upsample_initial_channel;
    const int dim = c.harmonic_num + 1;
    hop = 1;
    for (int i = 0; i < c.num_upsamples; ++i) hop *= c.upsample_rates[i];

    const float* p = w;
    const float* end = w + n_w;
    auto need = [&](size_t n) { B200_CHECK(p + n <= end, "weight blob too short"); };

    if (c.use_pitch_embed) {
        need(dim + 1);
        auto lw = take(p, dim);
        auto lb = take(p, 1);
        lw.push_back(lb[0]);
        upload(src_lin, lw);
    }
    // a [Cout][Cin][k] conv weight -> K-major [Cout][k * Cp]
    auto pack_conv = [&](Conv& cv, const std::vector<float>& wt, const std::vector<float>& bs, int cout, int cin, int k, int dil) {
        const int cp = ((cin + kBlockK - 1) / kBlockK) * kBlockK;
        std::vector<float> m(static_cast<size_t>(cout) * k * cp, 0.0f);
        for (int o = 0; o < cout; ++o)
            for (int ci = 0; ci < cin; ++ci)
                for (int kk = 0; kk < k; ++kk) m[(static_cast<size_t>(o) * k + kk) * cp + ci] = wt[(static_cast<size_t>(o) * cin + ci) * k + kk];
        cv.w.pack(m, cout, k * cp);
        upload(cv.bias, bs);
        cv.cin = cin; cv.cout = cout; cv.k = k; cv.dilation = dil;
    };
    {
        need(static_cast<size_t>(C0) * c.num_mels * 7 + C0);
        auto wt = take(p, static_cast<size_t>(C0) * c.num_mels * 7);
        auto bs = take(p, C0);
        pack_conv(conv_pre, wt, bs, C0, c.num_mels, 7, 1);
    }
    stages.resize(c.num_upsamples);
    for (int i = 0; i < c.num_upsamples; ++i) {
        Stage& s = stages[i];
        s.cin = C0 >> i;
        s.cout = C0 >> (i + 1);
        s.rate = c.upsample_rates[i];
        s.ksize = c.upsample_kernel_sizes[i];
        B200_CHECK(s.cin % kBlockK == 0, "transposed-conv input channels must be a multiple of 64");
        B200_CHECK(s.cout % 32 == 0 && s.cout >= 32 && (s.cout >= 256 ? s.cout % 256 == 0 : (s.cout & (s.cout - 1)) == 0), "unsupported channel count");
        need(static_cast<size_t>(s.cin) * s.cout * s.ksize + s.cout);
        auto wt = take(p, static_cast<size_t>(s.cin) * s.cout * s.ksize);   // [Cin][Cout][k]
        auto bs = take(p, s.cout);
        const int pad = (s.ksize - s.rate) / 2;
        s.up_phase.resize(s.rate);
        s.up_shifts.resize(s.rate);
        for (int ph = 0; ph < s.rate; ++ph) {
            // taps delta with kernel index kk = delta*u + ph + pad in [0, k); input row = q - delta
            std::vector<int> deltas;
            for (int d = -s.ksize; d <= s.ksize; ++d) {
                const int kk = d * s.rate + ph + pad;
                if (kk >= 0 && kk < s.ksize) deltas.push_back(d);
            }
            B200_CHECK(!deltas.empty() && static_cast<int>(deltas.size()) <= kMaxTaps, "unsupported transposed-conv geometry");
            const int nt = static_cast<int>(deltas.size());
            std::vector<float> wk(static_cast<size_t>(s.cout) * s.cin * nt);   // as a [Cout][Cin][nt] conv
            for (int o = 0; o < s.cout; ++o)
                for (int ci = 0; ci < s.cin; ++ci)
                    for (int j = 0; j < nt; ++j) {
                        const int kk = deltas[j] * s.rate + ph + pad;
                        wk[(static_cast<size_t>(o) * s.cin + ci) * nt + j] = wt[(static_cast<size_t>(ci) * s.cout + o) * s.ksize + kk];
                    }
            pack_conv(s.up_phase[ph], wk, bs, s.cout, s.cin, nt, 1);
            for (int d : deltas) s.up_shifts[ph].push_back(-d);
        }
    }
    if (c.use_pitch_embed) {
        for (int i = 0; i < c.num_upsamples; ++i) {
            Stage& s = stages[i];
            int stride = 1;
            for (int j = i + 1; j < c.num_upsamples; ++j) stride *= c.upsample_rates[j];
            if (i + 1 < c.num_upsamples) { s.noise_k = 2 * stride; s.noise_stride = stride; s.noise_pad = stride / 2; }
            else { s.noise_k = 1; s.noise_stride = 1; s.noise_pad = 0; }
            need(static_cast<size_t>(s.cout) * s.noise_k + s.cout);
            upload(s.noise_w, take(p, static_cast<size_t>(s.cout) * s.noise_k));
            upload(s.noise_b, take(p, s.cout));
        }
    }
    if (const char* nf = std::getenv("BSG_VOC_FUSE")) fuse_resblocks = nf[0] == '1';
    // a [C][C][k] conv weight -> fp16 K-major [C][k * C], taps packed densely (the fused ResBlock kernel's operand)
    auto pack_half = [&](HalfConv& hc, const std::vector<float>& wt, int C, int k) {
        std::vector<uint16_t> m(static_cast<size_t>(C) * k * C);
        for (int o = 0; o < C; ++o)
            for (int ci = 0; ci < C; ++ci)
                for (int kk = 0; kk < k; ++kk)
                    m[(static_cast<size_t>(o) * k + kk) * C + ci] = f32_to_f16_bits(wt[(static_cast<size_t>(o) * C + ci) * k + kk]);
        upload(hc.w, m);
        hc.map = make_w_tmap(hc.w.p, C, k * C, C);
    };
    for (int i = 0; i < c.num_upsamples; ++i) {
        Stage& s = stages[i];
        const int C = s.cout;
        s.convs1.resize(c.num_kernels * c.num_dilations);
        s.convs2.resize(c.num_kernels * c.num_dilations);
        // fused ResBlock iterations: channel counts the kernel is instantiated for, dilated halo within its shared-memory slab
        s.fused = fuse_resblocks && (C == 32 || C == 64 || C == 128);
        for (int j = 0; j < c.num_kernels && s.fused; ++j)
            for (int m = 0; m < c.num_dilations; ++m)
                if (128 + (c.resblock_kernel_sizes[j] - 1) * c.resblock_dilation_sizes[j][m] > 184) s.fused = false;
        if (s.fused) { s.h1.resize(s.convs1.size()); s.h2.resize(s.convs2.size()); }
        for (int j = 0; j < c.num_kernels; ++j) {
            const int k = c.resblock_kernel_sizes[j];
            B200_CHECK(k % 2 == 1 && k <= kMaxTaps, "resblock kernel size must be odd and <= 11");
            for (int m = 0; m < c.num_dilations; ++m) {
                need(static_cast<size_t>(C) * C * k + C);
                auto wt = take(p, static_cast<size_t>(C) * C * k);
                auto bs = take(p, C);
                pack_conv(s.convs1[j * c.num_dilations + m], wt, bs, C, C, k, c.resblock_dilation_sizes[j][m]);
                if (s.fused) pack_half(s.h1[j * c.num_dilations + m], wt, C, k);
            }
            for (int m = 0; m < c.num_dilations; ++m) {
                need(static_cast<size_t>(C) * C * k + C);
                auto wt = take(p, static_cast<size_t>(C) * C * k);
                auto bs = take(p, C);
                pack_conv(s.convs2[j * c.num_dilations + m], wt, bs, C, C, k, 1);
                if (s.fused) pack_half(s.h2[j * c.num_dilations + m], wt, C, k);
            }
        }
    }
    {
        const int C = stages.back().cout;
        need(static_cast<size_t>(C) * 7 + 1);
        auto wt = take(p, static_cast<size_t>(C) * 7);   // [1][C][7]
        auto bs = take(p, 1);
        std::vector<float> m(static_cast<size_t>(7) * C);
        for (int ci = 0; ci < C; ++ci)
            for (int kk = 0; kk < 7; ++kk) m[kk * C + ci] = wt[ci * 7 + kk];
        upload(post_w, m);
        upload(post_b, bs);
    }
    B200_CHECK(p == end, "weight blob has " + std::to_string(n_w) + " floats, consumed " + std::to_string(p - w));
    d_seed.alloc(sizeof(unsigned long long));
    ConvGemmArgs none{};
    for (int nt : {256, 128, 64, 32}) launch_conv_gemm(nt, 1, EPI_BIAS_ACT, none, nullptr);
    if (const char* np = std::getenv("BSG_VOC_PAIR")) pair_mode = np[0] == '1';
    if (const char* ng = std::getenv("BSG_VOC_GRAPH")) use_graphs = ng[0] == '1';
    if (const char* nv = std::getenv("BSG_VOC_NOISE_V2")) noise_v2 = nv[0] == '1';
    if (const char* nr = std::getenv("BSG_ROWS_EPI")) rows_epi = nr[0] == '1';
    if (const char* nm = std::getenv("BSG_ROWS_RMW")) rows_rmw = nm[0] == '1';
    if (pair_mode) for (int nt : {256, 128}) launch_conv_gemm(nt, 1, EPI_BIAS_ACT, none, nullptr, 1);
    ResblockArgs rnone{};
    for (const Stage& s : stages)
        if (s.fused) launch_resblock_iter(s.cout, rnone, nullptr);
}

HifiganPlan::~HifiganPlan() = default;

HifiganPlan::Workspace& HifiganPlan::workspace(int B, int T) {
    const auto key = std::make_pair(B, T);
    auto it = ws.find(key);
    if (it != ws.end()) {
        it->second->last_use = ++use_clock;
        return *it->second;
    }
    // the stage buffers are large (~20 KB per mel frame): keep a few shapes, evict the least recently used one at a time
    {
        static const double budget_gb = [] { const char* e = std::getenv("BSG_WS_BUDGET_GB"); return e ? std::atof(e) : 48.0; }();
        const size_t need = static_cast<size_t>(B) * T * 110 * 1024;
        auto total = [&] { size_t n = 0; for (auto& kv : ws) n += kv.second->bytes; return n; };
        while (!ws.empty() && (ws.size() >= static_cast<size_t>(kMaxShapes) || static_cast<double>(total() + need) > budget_gb * 1e9)) {
            auto lru = ws.begin();
            for (auto jt = ws.begin(); jt != ws.end(); ++jt)
                if (jt->second->last_use < lru->second->last_use) lru = jt;
            ws.erase(lru);
        }
    }
    size_t free_before = 0, free_after = 0, total_mem = 0;
    cudaMemGetInfo(&free_before, &total_mem);
    auto w = std::make_unique<Workspace>();
    w->last_use = ++use_clock;
    w->B = B;
    w->T = T;
    const size_t BT = static_cast<size_t>(B) * T;
    const int dim = cfg.harmonic_num + 1;
    w->mel16.alloc(BT * cfg.num_mels * 2);
    w->har.alloc(BT * hop * 4);
    w->phase0.alloc(BT * dim * 8);
    size_t max_f32 = 0, max_b16 = 0, max_up = BT * cfg.upsample_initial_channel * 2;
    size_t rows = BT;
    for (size_t i = 0; i < stages.size(); ++i) {
        rows *= stages[i].rate;
        const size_t C = stages[i].cout;
        max_f32 = std::max(max_f32, rows * C * 4);
        max_b16 = std::max(max_b16, rows * C * 2);
        if (i + 1 < stages.size()) max_up = std::max(max_up, rows * C * 2);
    }
    w->upin[0].alloc(max_up);
    w->upin[1].alloc(max_up);
    w->X0.alloc(max_f32);
    w->Xr.alloc(max_f32);
    w->S.alloc(max_f32);
    w->A0.alloc(max_b16);
    w->Ar.alloc(max_b16);
    w->Tb.alloc(max_b16);
    cudaMemGetInfo(&free_after, &total_mem);
    w->bytes = free_before > free_after ? free_before - free_after : 0;
    auto& ref = *w;
    ws[key] = std::move(w);
    return ref;
}

void HifiganPlan::run_source(Workspace& w, const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed, int B,
                             int T, cudaStream_t st) {
    const int dim = cfg.harmonic_num + 1;
    B200_CHECK(cfg.use_pitch_embed, "this generator was built without the NSF source (use_pitch_embed = 0)");
    nsf_phase_kernel<<<(B * dim * 32 + 255) / 256, 256, 0, st>>>(f0, rand_ini, d_seed.as<unsigned long long>(), B, T, hop, dim,
                                                                 static_cast<float>(cfg.audio_sample_rate), w.phase0.as<unsigned long long>());
    const long long n = static_cast<long long>(B) * T * hop;
    nsf_source_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(f0, w.phase0.as<unsigned long long>(), src_noise,
                                                                              d_seed.as<unsigned long long>(), src_lin.as<float>(), B, T,
                                                                              hop, dim, static_cast<float>(cfg.audio_sample_rate),
                                                                              w.har.as<float>());
    launches += 2, g_launch_count += 2;
    B200_CUDA(cudaGetLastError());
}

void HifiganPlan::source(const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed, int B, int T, float* har,
                         cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    B200_CUDA(cudaMemcpyAsync(d_seed.p, &seed, sizeof(seed), cudaMemcpyHostToDevice, st));
    run_source(w, f0, rand_ini, src_noise, seed, B, T, st);
    B200_CUDA(cudaMemcpyAsync(har, w.har.p, static_cast<size_t>(B) * T * hop * 4, cudaMemcpyDeviceToDevice, st));
}

void HifiganPlan::forward(const float* mel, const float* f0, const float* rand_ini, const float* src_noise, unsigned long long seed, int B,
                          int T, float* wav, cudaStream_t st) {
    B200_CHECK(B > 0 && T > 0, "empty batch");
    B200_CUDA(cudaSetDevice(device));
    Workspace& w = workspace(B, T);
    const size_t BT = static_cast<size_t>(B) * T;
    const int has_src = f0 != nullptr ? 1 : 0;
    B200_CUDA(cudaMemcpyAsync(d_seed.p, &seed, sizeof(seed), cudaMemcpyHostToDevice, st));
    if (!use_graphs || rand_ini != nullptr || src_noise != nullptr) {   // injected randomness (parity tests): plain launches
        enqueue(w, mel, f0, rand_ini, src_noise, seed, B, T, wav, st);
        return;
    }
    // production path: the ~110 launches of one forward are captured once per shape and replayed (no launch gaps at small batches)
    w.in_mel.ensure(BT * cfg.num_mels * 4);
    w.out_wav.ensure(BT * hop * 4);
    if (has_src) w.in_f0.ensure(BT * 4);
    B200_CUDA(cudaMemcpyAsync(w.in_mel.p, mel, BT * cfg.num_mels * 4, cudaMemcpyDeviceToDevice, st));
    if (has_src) B200_CUDA(cudaMemcpyAsync(w.in_f0.p, f0, BT * 4, cudaMemcpyDeviceToDevice, st));
    if (!w.graph[has_src]) {
        cudaStream_t cs;
        B200_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaGraph_t g = nullptr;
        const unsigned long long before = launches;
        B200_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
        try {
            enqueue(w, w.in_mel.as<float>(), has_src ? w.in_f0.as<float>() : nullptr, nullptr, nullptr, seed, B, T, w.out_wav.as<float>(), cs);
        } catch (...) {
            cudaStreamEndCapture(cs, &g);
            if (g) cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            throw;
        }
        B200_CUDA(cudaStreamEndCapture(cs, &g));
        w.graph_nodes[has_src] = launches - before;
        launches = before;
        g_launch_count -= w.graph_nodes[has_src];
        B200_CUDA(cudaGraphInstantiate(&w.graph[has_src], g, 0));
        cudaGraphDestroy(g);
        cudaStreamDestroy(cs);
    }
    B200_CUDA(cudaGraphLaunch(w.graph[has_src], st));
    launches += w.graph_nodes[has_src], g_launch_count += w.graph_nodes[has_src];
    B200_CUDA(cudaMemcpyAsync(wav, w.out_wav.p, BT * hop * 4, cudaMemcpyDeviceToDevice, st));
}

// the launches of one forward pass on stream st (everything but the seed upload)
void HifiganPlan::enqueue(Workspace& w, const float* mel, const float* f0, const float* rand_ini, const float* src_noise,
                          unsigned long long seed, int B, int T, float* wav, cudaStream_t st) {
    const size_t BT = static_cast<size_t>(B) * T;
    const bool has_src = f0 != nullptr;
    if (has_src) run_source(w, f0, rand_ini, src_noise, seed, B, T, st);

    mel_prep_kernel<<<static_cast<unsigned>((BT + 127) / 128), 128, 0, st>>>(mel, B, cfg.num_mels, T, w.mel16.as<__nv_bfloat16>());
    launches += 1, g_launch_count += 1;

    auto run_conv = [&](Conv& cv, const void* a_ptr, int a_pitch, int Lrows, const std::vector<int>& shifts, const EpiParams& epi) {
        ConvGemmArgs a{};
        const int nt = ntile_for(cv.cout);
        // wide stages on 2-CTA tiles (M = 256): a single CTA reads 12 KB (N = 256) / 8 KB (N = 128) of shared memory per MMA and is
        // bound by that (DESIGN.md 4.1); a pair reads 8 / 6 KB per SM
        const int pair = (pair_mode && nt >= 128 && static_cast<long long>(B) * Lrows >= 4096) ? 1 : 0;
        set_geometry(a, B, Lrows, cv.cout, nt, pair != 0);
        const int cp = ((cv.cin + kBlockK - 1) / kBlockK) * kBlockK;
        const int rows_box = set_taps(a, 0, 0, cp / kBlockK, shifts.data(), static_cast<int>(shifts.size()), cp);
        a.amap[0] = make_act_tmap(a_ptr, B, Lrows, cv.cin, a_pitch, rows_box);
        a.amap[1] = a.amap[0];
        cv.w.maps(pair ? nt / 2 : nt, a.wmap[0], a.wmap[1]);
        a.k_steps = cv.cin >= kBlockK ? 0 : (cv.cin + 15) / 16;
        a.w_resident = (!pair && a.n_tiles_n == 1 && static_cast<int>(shifts.size()) * (cp / kBlockK) <= conv_gemm_weight_slots(nt, 1)) ? 1 : 0;
        a.epi = epi;
        a.epi.bias = cv.bias.as<float>();
        // row-per-thread write-only epilogue: needs 32-byte aligned rows (channel counts that are multiples of 16 / 8)
        if (rows_epi && a.epi.act_pitch % 16 == 0 && a.epi.out_pitch % 8 == 0 && a.epi.out_col0 % 8 == 0)
            a.epi.flags |= BA_ROWS | (rows_rmw ? BA_ROWS_RMW : 0);
        launch_conv_gemm(nt, 1, EPI_BIAS_ACT, a, st, pair);
        launches += 1, g_launch_count += 1;
    };
    auto same_shifts = [](int k, int dil) {
        std::vector<int> s;
        for (int j = 0; j < k; ++j) s.push_back((j - (k - 1) / 2) * dil);   // padding (k*d - d)/2, hifigan.py:26-27
        return s;
    };

    {   // conv_pre (hifigan.py:151) + the lrelu of the first up-sampling stage (:153)
        EpiParams e{};
        e.flags = BA_WRITE_ACT;
        e.c1 = kLrelu;
        e.out_hi = w.upin[0].as<__nv_bfloat16>();
        e.act_pitch = conv_pre.cout;
        e.out_pitch = conv_pre.cout;
        run_conv(conv_pre, w.mel16.p, cfg.num_mels, T, same_shifts(7, 1), e);
    }
    int Lcur = T;
    int up_sel = 0;
    const int nk = cfg.num_kernels, nd = cfg.num_dilations;
    for (size_t i = 0; i < stages.size(); ++i) {
        Stage& s = stages[i];
        const int C = s.cout, Cp = C;
        const bool last_stage = i + 1 == stages.size();
        // ---- transposed convolution, one launch per output phase (hifigan.py:154)
        for (int ph = 0; ph < s.rate; ++ph) {
            EpiParams e{};
            e.flags = BA_WRITE_F32;
            e.f32_a = w.X0.as<float>();
            e.out_pitch = s.rate * C;
            e.out_col0 = ph * C;
            run_conv(s.up_phase[ph], w.upin[up_sel].p, s.cin, Lcur, s.up_shifts[ph], e);
        }
        const long long Lout = static_cast<long long>(Lcur) * s.rate;
        const long long rows = static_cast<long long>(B) * Lout;
        __nv_bfloat16* A0 = w.A0.as<__nv_bfloat16>();
        __nv_bfloat16* Ar = w.Ar.as<__nv_bfloat16>();
        __nv_bfloat16* Tb = w.Tb.as<__nv_bfloat16>();
        // ---- harmonic-source branch + lrelu (hifigan.py:155-160, ResBlock1's first leaky_relu :56)
        {
            B200_CHECK(s.noise_k <= 32, "noise branch kernel holds the source window in one warp (kernel size <= 32)");
            const int blocks = device_sm_count() * 8;
            const size_t sm_bytes = (static_cast<size_t>(s.noise_k) * C + C) * sizeof(float);
            const float* nw = has_src ? s.noise_w.as<float>() : nullptr;
            const float* nb = has_src ? s.noise_b.as<float>() : nullptr;
            const long long Lhar = static_cast<long long>(T) * hop;
            const int lpr = C >= 128 ? 32 : C / 4;
            const bool v2 = (noise_v2 || s.fused) && s.noise_k <= lpr && Cp % 4 == 0 && C <= 512;
            B200_CHECK(v2 || !s.fused, "the fused ResBlock path needs the row-group noise-branch kernel (kernel size <= lanes per row)");
#define B200_NOISE(CPL)                                                                                                                 \
    do {                                                                                                                                \
        if (v2)                                                                                                                         \
            noise_branch_v2_kernel<CPL * 32><<<blocks, 256, sm_bytes, st>>>(w.har.as<float>(), nw, nb, B, Lout, Lhar, s.noise_k,        \
                                                                           s.noise_stride, s.noise_pad, has_src ? 1 : 0, w.X0.as<float>(), A0, Cp, \
                                                                           s.fused ? 1 : 0);                                            \
        else                                                                                                                            \
            noise_branch_kernel<CPL><<<blocks, 256, sm_bytes, st>>>(w.har.as<float>(), nw, nb, B, Lout, Lhar, s.noise_k, s.noise_stride, \
                                                                   s.noise_pad, has_src ? 1 : 0, w.X0.as<float>(), A0, Cp);              \
    } while (0)
            switch (C / 32) {
                case 1: B200_NOISE(1); break;
                case 2: B200_NOISE(2); break;
                case 4: B200_NOISE(4); break;
                case 8: B200_NOISE(8); break;
                case 16: B200_NOISE(16); break;
                default: throw Error("noise branch: unsupported channel count");
            }
#undef B200_NOISE
            launches += 1, g_launch_count += 1;
            B200_CUDA(cudaGetLastError());
        }
        // ---- MRF: sum_j ResBlock1_j(x) / num_kernels (hifigan.py:161-168, :54-61)
        if (s.fused) {
            // One kernel per ResBlock iteration on the 16-bit single-tensor stream (resblock_fused.cuh): A0 = fp16 lrelu(x) is the stage
            // input of all three ResBlocks, Ar / Tb ping-pong between iterations, S (viewed as fp16) accumulates the MRF sum; the last
            // iteration of the last ResBlock writes the next stage's transposed-conv operand (bf16 lrelu 0.1) or conv_post's input
            // (fp16 lrelu 0.01, hifigan.py:169).
            __half* pp[2] = {reinterpret_cast<__half*>(Ar), reinterpret_cast<__half*>(Tb)};
            for (int j = 0; j < nk; ++j) {
                const int k = cfg.resblock_kernel_sizes[j];
                for (int m = 0; m < nd; ++m) {
                    const int d = s.convs1[j * nd + m].dilation;
                    ResblockArgs a{};
                    const __half* in = m == 0 ? reinterpret_cast<const __half*>(A0) : pp[(m - 1) & 1];
                    a.B = B; a.L = static_cast<int>(Lout);
                    a.ntaps = k; a.dil = d;
                    a.V = kTileM - (k - 1);
                    a.a_rows = ((kTileM + (k - 1) * d) + 7) / 8 * 8;
                    a.tiles_per_batch = (a.L + a.V - 1) / a.V;
                    a.num_tiles = B * a.tiles_per_batch;
                    a.amap = make_act_tmap(in, B, a.L, C, C, a.a_rows);
                    a.w1map = s.h1[j * nd + m].map;
                    a.w2map = s.h2[j * nd + m].map;
                    a.bias1 = s.convs1[j * nd + m].bias.as<float>();
                    a.bias2 = s.convs2[j * nd + m].bias.as<float>();
                    a.a_in = in;
                    a.sum = w.S.as<__half>();
                    a.c0 = 1.0f / static_cast<float>(nk);
                    if (m + 1 < nd) {
                        a.mode = 0;
                        a.out = pp[m & 1];
                    } else if (j + 1 < nk) {
                        a.mode = j == 0 ? 1 : 2;
                    } else {
                        a.mode = nk == 1 ? 4 : 3;   // a single ResBlock has no MRF sum to add to
                        a.out = last_stage ? static_cast<void*>(w.X0.p) : static_cast<void*>(w.upin[up_sel ^ 1].p);
                        a.out_bf16 = last_stage ? 0 : 1;
                        a.slope_out = last_stage ? 0.01f : kLrelu;
                    }
                    a.w_slots = resblock_weight_slots(C);
                    const int n_wt = C == 32 ? (k + 1) / 2 : k * (C / kBlockK);
                    a.w_resident = 2 * n_wt <= a.w_slots ? 2 : (n_wt + 3 <= a.w_slots ? 1 : 0);   // both convs resident / conv1 only / streaming
                    static const bool trace_on = std::getenv("BSG_TRACE") != nullptr;
                    DevBuf tb;
                    if (trace_on) {   // per-role cycle counters of this launch, averaged over the CTAs (measurement only: synchronises)
                        tb.alloc(static_cast<size_t>(device_sm_count()) * 16 * 8);
                        B200_CUDA(cudaMemsetAsync(tb.p, 0, tb.bytes, st));
                        a.trace = tb.as<unsigned long long>();
                    }
                    launch_resblock_iter(C, a, st);
                    launches += 1, g_launch_count += 1;
                    if (trace_on) {
                        const int grid = device_sm_count();
                        std::vector<unsigned long long> h(static_cast<size_t>(grid) * 16);
                        B200_CUDA(cudaMemcpyAsync(h.data(), tb.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
                        B200_CUDA(cudaStreamSynchronize(st));
                        double sm[16] = {0};
                        int n = 0;
                        for (int c = 0; c < grid; ++c) {
                            if (h[c * 16] == 0) continue;
                            ++n;
                            for (int i = 0; i < 16; ++i) sm[i] += static_cast<double>(h[c * 16 + i]);
                        }
                        if (n)
                            std::fprintf(stderr,
                                         "TRACE resblock C=%d k=%d d=%d mode %d resident %d: per tile (%.0f tiles/CTA): MMA warp %.0f clk [waits: acc1 free %.0f, "
                                         "A tile %.0f, weights %.0f, acc2 free %.0f, t tile %.0f] | epilogue-1 %.0f [waits: acc1 full %.0f, t free %.0f] | "
                                         "epilogue-2 %.0f [wait acc2 full %.0f]\n",
                                         C, k, d, a.mode, a.w_resident, sm[6] / n, sm[0] / sm[6], sm[1] / sm[6], sm[2] / sm[6], sm[3] / sm[6], sm[4] / sm[6],
                                         sm[5] / sm[6], sm[7] / sm[6], sm[8] / sm[6], sm[9] / sm[6], sm[10] / sm[6], sm[11] / sm[6]);
                    }
                }
            }
        } else
        for (int j = 0; j < nk; ++j) {
            const int k = cfg.resblock_kernel_sizes[j];
            for (int m = 0; m < nd; ++m) {
                Conv& c1 = s.convs1[j * nd + m];
                Conv& c2 = s.convs2[j * nd + m];
                {
                    EpiParams e{};
                    e.flags = BA_WRITE_ACT;
                    e.c1 = kLrelu;
                    e.out_hi = Tb;
                    e.act_pitch = Cp;
                    e.out_pitch = C;
                    run_conv(c1, m == 0 ? A0 : Ar, Cp, static_cast<int>(Lout), same_shifts(k, c1.dilation), e);
                }
                {
                    EpiParams e{};
                    e.flags = BA_ADD_RES;
                    e.aux0 = m == 0 ? w.X0.as<float>() : w.Xr.as<float>();
                    e.out_pitch = C;
                    e.act_pitch = Cp;
                    e.c1 = kLrelu;
                    if (m + 1 < nd) {
                        e.flags |= BA_WRITE_F32 | BA_WRITE_ACT;
                        e.f32_a = w.Xr.as<float>();
                        e.out_hi = Ar;
                    } else {
                        e.flags |= BA_ACCUM_F32B | (j == 0 ? BA_ACCUM_INIT : 0);
                        e.f32_b = w.S.as<float>();
                        e.c0 = 1.0f / static_cast<float>(nk);
                        if (j + 1 == nk && !last_stage) {   // stage output -> lrelu -> next transposed conv (:153)
                            e.flags |= BA_WRITE_ACT | BA_ACT_FROM_B;
                            e.out_hi = w.upin[up_sel ^ 1].as<__nv_bfloat16>();
                            e.act_pitch = C;
                        }
                    }
                    run_conv(c2, Tb, Cp, static_cast<int>(Lout), same_shifts(k, 1), e);
                }
            }
        }
        up_sel ^= 1;
        Lcur = static_cast<int>(Lout);
    }
    {   // lrelu(0.01) -> conv_post -> tanh (hifigan.py:169-171)
        const int C = stages.back().cout;
        const long long n = static_cast<long long>(B) * Lcur;
        B200_CHECK(C == 32, "conv_post kernel is specialised for 32 input channels");
        if (stages.back().fused)
            conv_post_kernel<true><<<static_cast<unsigned>((n + 255) / 256), 256, (7 * 32 + (256 + 6) * 33) * sizeof(float), st>>>(
                w.X0.p, post_w.as<float>(), post_b.as<float>(), B, Lcur, 7, wav);
        else
            conv_post_kernel<false><<<static_cast<unsigned>((n + 255) / 256), 256, (7 * 32 + (256 + 6) * 33) * sizeof(float), st>>>(
                w.S.p, post_w.as<float>(), post_b.as<float>(), B, Lcur, 7, wav);
        launches += 1, g_launch_count += 1;
        B200_CUDA(cudaGetLastError());
    }
}

}  // namespace b200
