// Persistent warp-specialised implicit-GEMM convolution for sm_100a (tcgen05 + TMEM + TMA).
//
// One kernel template serves every 1-D convolution on the hot path.  Activations are stored
// channels-last ([B][L][C] bf16), so a convolution tap is a *row shift* of the A operand:
//     Y[b, t, n] = sum_tap sum_c  A[b, t + shift_tap, c] * W[n, wcol_tap + c]
// For every 64-channel k-block ONE halo tile of A (rows t0+min_shift .. t0+127+max_shift, <= 192 rows) is fetched
// by 3-D TMA; rows that fall outside [0, L) are zero-filled by the TMA unit, which is exactly the reference's zero
// padding (nn.Conv1d padding=dilation, usr/diff/net.py:61; get_padding, modules/hifigan/hifigan.py:26-27).  The taps
// then read that tile through UMMA descriptors whose start address is advanced by shift*128 B: the SWIZZLE_128B
// pattern is a function of the absolute shared-memory address, so a descriptor may start on any row of a swizzle
// atom (verified on B200 with csrc/experiments.cu, profiles/r01_c).  A k=11 convolution therefore moves its
// activations from L2 to shared memory once instead of eleven times.
// Weights are packed K-major ([N][Ktot] bf16) and fetched by 2-D TMA.  tcgen05.mma (M=128, N=N_TILE,
// K=16) accumulates in TMEM (fp32); two accumulator buffers let the epilogue of tile i overlap the
// MMAs of tile i+1.
//
// TERMS == 3 is the "bf16x3" contraction: every operand is carried as hi = bf16(x), lo = bf16(x - hi)
// and each k-block issues A_hi*W_hi + A_lo*W_hi + A_hi*W_lo into the same fp32 accumulator (~16
// mantissa bits).  The 100-step sampler needs it to stay within the 1e-2 mel tolerance (DESIGN.md §5).
//
// TERMS == 2 is the "fp16x2" contraction: activations are ONE fp16 operand, weights are carried as fp16 hi/lo
// (pre-scaled by a power of two so that lo stays out of the subnormal range; EpiParams::acc_scale undoes it) and each
// k-block issues A*W_hi + A*W_lo.  Weight rounding is the systematic error of the 100-step sampler; activation rounding
// at 11 significant bits is not (tests/tools/precision_study.py, DESIGN.md §5), so this mode meets the tolerance with 2/3 of
// the MMAs and half the activation bytes of bf16x3.
//
// Warp roles (320 threads): warp 0 = TMA producer + TMEM allocator, warp 1 = MMA issuer (one thread),
// warps 2..9 = epilogue (TMEM lane quadrant = warp_id % 4; the two warps of a quadrant split the tile's columns --
// a single warp per scheduler was instruction-latency bound, profiles/r01_b).  Before working on tile i every
// epilogue warp L2-prefetches the fp32 operands it will read-modify-write for tile i+1 (residual stream / skip sum).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <cstdint>

#include "ptx.cuh"

namespace b200 {

constexpr int kTileM = 128;
constexpr int kBlockK = 64;           // bf16 elements per k-block = one 128-byte swizzle row
constexpr int kMaxTaps = 11;
constexpr int kGemmThreads = 32 * (2 + 8);   // producer, MMA, 8 epilogue warps
#ifndef B200_ASTAGES2
#define B200_ASTAGES2 3
#endif
constexpr int kSmemBudget = 200 * 1024;

// The taps of one convolution: all read the same A source / channel range, each with its own row shift and its own
// K-column block of the packed weight matrix.
struct TapSet {
    int a_src;               // index of the A tensor-map pair (hi = 2*a_src, lo = 2*a_src + 1)
    int a_col0;              // first channel of A
    int n_kb;                // number of 64-channel k-blocks
    int row_shift;           // row shift of the halo tile's first row (= smallest tap shift, may be negative)
    int n_taps;
    int row_off[kMaxTaps];   // tap shift - row_shift  (>= 0): row of the halo tile where the tap's 128 rows start
    int w_col0[kMaxTaps];    // first K column of the tap in the packed weight matrix
};

// Epilogue selector
enum : int {
    EPI_F32 = 0,        // out_f32[row][n] = acc + bias[n]                       (unit tests)
    EPI_INPROJ = 1,     // relu(acc+bias) -> xres f32 ; (+dvec) -> xa hi/lo      (net.py:116-118)
    EPI_GATE = 2,       // sigmoid(g+bg) * tanh(f+bf) -> z hi/lo                 (net.py:71-74)
    EPI_RES_SKIP = 3,   // x=(x+r+b)/sqrt2 -> xres f32, split(x + d_next) -> xa  (net.py:76-78; skip half: see EPI_RELU_BF16)
    EPI_RELU_BF16 = 4,  // (acc+bias)*c0 [ReLU] -> hi/lo                         (net.py:126-128)
    EPI_POSTERIOR = 5,  // eps=acc+bias -> DDPM posterior update of x_t          (shallow_diffusion_tts.py:149-166)
    EPI_BIAS_ACT = 6,   // HiFi-GAN: y = acc+bias (+res) ; writes f32 and/or lrelu(y) bf16
    // the same epilogues with a diffusion step per batch item (ConvGemmArgs::steps): a row tile never spans two batch items, so
    // each tile looks up its item's step once.  Separate instantiations: the uniform-step kernels stay exactly as they are.
    EPI_INPROJ_STEPS = 7,
    EPI_RES_SKIP_STEPS = 8,
    EPI_POSTERIOR_STEPS = 9,
};
__host__ __device__ constexpr int epi_base(int epi) {
    return epi == EPI_INPROJ_STEPS ? EPI_INPROJ : (epi == EPI_RES_SKIP_STEPS ? EPI_RES_SKIP : (epi == EPI_POSTERIOR_STEPS ? EPI_POSTERIOR : epi));
}

struct EpiParams {
    const float* bias;         // [N_total]
    float* f32_a;              // EPI_F32: out ; INPROJ/RES: residual stream x [rows][256] ; POSTERIOR: x_t [B][M][T]
    float* f32_b;              // RES_SKIP: skip accumulator [rows][256] ; POSTERIOR: mel_out [B][T][M] (last step) or null
    __nv_bfloat16* out_hi;     // bf16 operand written for the next GEMM
    __nv_bfloat16* out_lo;     // (TERMS==3 consumers) low part, may be null
    __nv_bfloat16* out2_hi;    // RES_SKIP: head input (last layer) ; BIAS_ACT: second bf16 output
    __nv_bfloat16* out2_lo;
    const float* dvec;         // step-embedding vector added before the bf16 split (next layer's d), or null
    const float* aux0;         // POSTERIOR: injected noise [B][M][T] or null ; BIAS_ACT: residual f32 in
    const float* aux1;         // POSTERIOR: spec_min[M]
    const float* aux2;         // POSTERIOR: spec_max[M]
    const int64_t* mel2ph;     // POSTERIOR: [B][T] or null
    int out_pitch;             // elements per row of out_hi/out_lo/f32 outputs
    int out_col0;              // column offset added to n (transposed-conv phases)
    int act_pitch;             // BIAS_ACT: elements per row of the bf16 activation output (channel-padded buffers)
    int flags;                 // RES_SKIP: bit0 = first layer (skip = ...), bit1 = last layer ; BIAS_ACT: see hifigan
    float c0, c1, c2, c3, c4;  // POSTERIOR: sqrt_recip, sqrt_recipm1, coef1, coef2, sigma (0 at t==0) ; BIAS_ACT: scale, slope
    const unsigned long long* seed_ptr;  // POSTERIOR: device-resident Philox seed (read when aux0 == null)
    unsigned int step;         // POSTERIOR: Philox stream offset (executed step index)
    float acc_scale;           // accumulators are multiplied by this on load (2^-p of the fp16x2 weight pre-scale; 0 => 1)
    int out_fp16;              // out_hi receives ONE fp16 operand (consumer runs fp16x2) instead of bf16 hi[/lo]
    uint8_t* out8;             // INPROJ: also write e4m3(x + d) [rows][out_pitch] (A operand of the fp8 correction MMAs), or null
};

// A diffusion step per batch item (the *_STEPS epilogues).  INPROJ / RES_SKIP: dvec points at the embedding of step 0 and
// item b reads dvec + t_of_b[b] * dvec_stride.  POSTERIOR: c0..c4 of item b are coef[5b .. 5b+4] (c4 = 0 where t_b == 0), the
// device noise of item b is Philox stream k_last - t_of_b[b] (the executed step at which the sampler reaches t_b), and
// clip = 0 skips the clamp of x0 (clip_denoised=False).
struct StepRows {
    const int* t_of_b;     // device int32 [B]
    const float* coef;     // device f32 [B][5]
    int dvec_stride;
    int k_last;
    int clip;
};

struct ConvGemmArgs {
    CUtensorMap amap[4];   // A sources: (hi, lo) pairs, box = 64 channels x a_rows rows
    CUtensorMap wmap[2];   // packed weights hi / lo
    int B, L;              // batches, rows per batch
    int tiles_per_batch;   // ceil(L / 128)
    int n_tiles_n;         // N tiles per row tile
    int num_tiles;
    int w_row0;            // first weight row of this launch
    int a_rows;            // rows of the A halo box (multiple of 8, 128 + max_shift - min_shift rounded up)
    TapSet taps;
    EpiParams epi;
    int k_steps;           // MMAs (16 channels each) per 64-channel k-block; 0 = 4.  Fewer when Cin < 64 (the rest of the block is zero)
    int w_resident;        // 1: all n_taps * n_kb weight tiles fit the weight ring: they are loaded ONCE per CTA and stay in shared
                           //    memory for all its tiles (single-CTA tiles only).  Small-channel convolutions issue so little MMA work
                           //    per weight tile that streaming the weights per tile left the kernel bound by TMA round trips
                           //    (~150 cycles per MMA whatever N: profiles/r01_i)
    unsigned long long* trace;   // optional [grid][16] cycle counters of the three roles (tests/tools/gpu_probe.py tracetarget), or null
    StepRows steps;        // the *_STEPS epilogues only (kept behind every other member so that their offsets do not move)
};

// mbar_wait that adds the cycles spent waiting to *acc when tracing
__device__ __forceinline__ void mbar_wait_tr(uint64_t* bar, uint32_t parity, bool tr, long long& acc) {
    if (!tr) { mbar_wait(bar, parity); return; }
    const long long t0 = clock64();
    mbar_wait(bar, parity);
    acc += clock64() - t0;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 counter RNG + Box-Muller (production noise path; parity tests inject noise)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return ctr;
}
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
    const float u = (static_cast<float>(a) + 0.5f) * 2.3283064365386963e-10f;   // (0,1)
    const float v = (static_cast<float>(b) + 0.5f) * 2.3283064365386963e-10f;
    const float r = sqrtf(-2.0f * __logf(u));
    float s, c;
    __sincosf(6.283185307179586f * v, &s, &c);
    return make_float2(r * c, r * s);
}
// standard normal for element `idx` of executed step `step`
__device__ __forceinline__ float philox_normal(unsigned long long seed, uint32_t step, uint64_t idx) {
    const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(idx >> 2), static_cast<uint32_t>(idx >> 34), step, 0x5eedu),
                                  make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
    const uint32_t w = static_cast<uint32_t>(idx & 3);
    const float2 n = (w < 2) ? box_muller(r.x, r.y) : box_muller(r.z, r.w);
    return (w & 1) ? n.y : n.x;
}

// four standard normals from one Philox call (counter = idx4)
__device__ __forceinline__ float4 philox_normal4(unsigned long long seed, uint32_t step, uint64_t idx4) {
    const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(idx4), static_cast<uint32_t>(idx4 >> 32), step, 0x5eed4u),
                                  make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
    const float2 a = box_muller(r.x, r.y), b = box_muller(r.z, r.w);
    return make_float4(a.x, a.y, b.x, b.y);
}

// ---------------------------------------------------------------------------------------------
// Epilogue helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float fast_tanh(float x) {
    // tanh(x) = 1 - 2/(1+e^{2x}); ex2/rcp approximations (rel err ~1e-6), saturates correctly.
    const float e = __expf(2.0f * x);
    return 1.0f - __fdividef(2.0f, 1.0f + e);
}
__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }


// ---- accumulator access -----------------------------------------------------------------------
__device__ __forceinline__ void ld_acc32(uint32_t taddr, float (&v)[32], float scale) {
    uint32_t r[32];
    __syncwarp();   // tcgen05.ld is .sync.aligned: reconverge after any divergent store path
    tmem_ld32(taddr, r);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) * scale;
}
__device__ __forceinline__ void ld_acc16(uint32_t taddr, float (&v)[16], float scale) {
    uint32_t r[16];
    __syncwarp();
    tmem_ld16(taddr, r);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]) * scale;
}

// ---- coalescing transpose ---------------------------------------------------------------------
// tcgen05.ld hands every thread one accumulator ROW (32 consecutive columns).  Row-per-thread global accesses
// touch 32 different 128-byte lines per instruction, which made the epilogue LSU-bound (profiles/r01_a).  Each
// warp therefore bounces its 32x32 fp32 chunk (16 rows at a time) through a private shared-memory tile (row pitch
// 36 floats: conflict-free for the float4 row writes and for the float2 reads below) and continues in a transposed
// ownership: lane l holds, for rp = 0..15, the two columns cc = 2*(l & 15), cc+1 of row 2*rp + (l >> 4).
// A warp instruction then covers two full 128-byte row segments -> fully coalesced loads and stores.
constexpr int kStagePitch = 36;
constexpr int kStageFloatsPerWarp = 16 * kStagePitch;
constexpr int kEpiWarps = 8;          // two column groups x four TMEM lane quadrants

struct LanePos {
    int r0;   // 0 / 1: which row of each row pair this lane owns
    int cc;   // first of the two columns (within the 32-column chunk) this lane owns
};
__device__ __forceinline__ LanePos lane_pos(int lane) { return LanePos{lane >> 4, (lane & 15) * 2}; }

__device__ __forceinline__ void sts128(uint32_t saddr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ float2 lds64(uint32_t saddr) {
    float2 r;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "r"(saddr) : "memory");
    return r;
}
__device__ __forceinline__ void chunk_transpose(float* stage, int lane, const float (&v)[32], float2 (&o)[16]) {
    const LanePos lp = lane_pos(lane);
    const uint32_t sbase = smem_u32(stage);   // explicit shared-space accesses (generic LD/ST showed up as stall_lg)
    const uint32_t wr = sbase + (lane & 15) * (kStagePitch * 4);
    const uint32_t rd = sbase + (lp.r0 * kStagePitch + lp.cc) * 4;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        if (lp.r0 == half) {
#pragma unroll
            for (int j = 0; j < 8; ++j) sts128(wr + j * 16, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        __syncwarp();
#pragma unroll
        for (int rp = 0; rp < 8; ++rp) o[half * 8 + rp] = lds64(rd + rp * (2 * kStagePitch * 4));
        __syncwarp();
    }
}
// load one accumulator chunk (32 rows x 32 columns starting at column c) in transposed ownership
__device__ __forceinline__ void ld_chunk_t(uint32_t tacc, int c, float* stage, int lane, float2 (&o)[16], float scale) {
    float v[32];
    ld_acc32(tacc + c, v, scale);
    chunk_transpose(stage, lane, v, o);
}
// bf16 hi/lo split of two neighbouring values, packed for 4-byte stores
// fp16 operand of the fp16x2 mode (saturating: an out-of-range activation must not become inf)
__device__ __forceinline__ void st_half2(float2 y, __nv_bfloat16* dst) {
    const __half2 h = __floats2half2_rn(fminf(fmaxf(y.x, -65504.0f), 65504.0f), fminf(fmaxf(y.y, -65504.0f), 65504.0f));
    *reinterpret_cast<uint32_t*>(dst) = *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void st_split2(float2 y, __nv_bfloat16* hi, __nv_bfloat16* lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(y.x, y.y);
    const uint32_t hu = *reinterpret_cast<const uint32_t*>(&h);
    *reinterpret_cast<uint32_t*>(hi) = hu;
    if (lo != nullptr) {
        const float hx = __uint_as_float(hu << 16), hy = __uint_as_float(hu & 0xffff0000u);
        const __nv_bfloat162 l = __floats2bfloat162_rn(y.x - hx, y.y - hy);
        *reinterpret_cast<uint32_t*>(lo) = *reinterpret_cast<const uint32_t*>(&l);
    }
}
// next GEMM's A operand at element offset `off`: one fp16 value (fp16x2 consumer) or bf16 hi[/lo]
// FMT: 0 = bf16 split, 1 = fp16, 2 = decided at run time by e.out_fp16
template <int FMT>
__device__ __forceinline__ void st_operand2(const EpiParams& e, float2 y, long long off) {
    if (FMT == 1 || (FMT == 2 && e.out_fp16)) st_half2(y, e.out_hi + off);
    else st_split2(y, e.out_hi + off, e.out_lo ? e.out_lo + off : nullptr);
}
__device__ __forceinline__ float2 ldg2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ float2 ld2(const float* p) { return *reinterpret_cast<const float2*>(p); }
__device__ __forceinline__ void st2(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }

// How the two groups of four epilogue warps share the work: 2 = they split the columns of every tile, 1 = each group takes whole tiles
// (every other tile; the posterior epilogue alternates 16-channel chunks instead).  Narrow tiles are bound by the latency chain of an
// epilogue, not by its width, so two tiles in flight beat two half-width passes over one -- for N = 32; for N = 64 the split is faster
// (vocoder at cfg3: 56.3 ms vs 58.0 ms with -DB200_ALT_MAX_N=64, profiles/r01_m_vocoder_small_kernels.txt).
#ifndef B200_ALT_MAX_N
#define B200_ALT_MAX_N 32
#endif
__host__ __device__ constexpr int epi_col_split(int n_tile) { return (n_tile % 64 == 0 && n_tile > B200_ALT_MAX_N) ? 2 : 1; }

// BIAS_ACT flags (HiFi-GAN epilogue)
enum : int {
    BA_ADD_RES = 1,      // y += aux0[row][n]            (ResBlock1 residual, hifigan.py:60)
    BA_WRITE_F32 = 2,    // f32_a[row][n] = y
    BA_ACCUM_F32B = 4,   // f32_b[row][n] (+)= y * c0    (MRF sum / num_kernels, hifigan.py:161-168)
    BA_ACCUM_INIT = 8,   // with BA_ACCUM_F32B: '=' instead of '+='
    BA_WRITE_ACT = 16,   // out_hi[row][n] = bf16(lrelu(y, c1))
    BA_ACT_FROM_B = 32,  // the bf16 activation is taken from the accumulated f32_b value instead of y
    BA_ROWS = 64,        // the epilogue keeps the accumulator's row-per-thread ownership and uses 256-bit global accesses (see below)
    BA_ROWS_RMW = 128,   // ... also when it reads (BA_ADD_RES / BA_ACCUM_F32B)
    BA_GELU = 256,       // write-only row epilogue: y = gelu((acc + bias) * c0) (exact erf form, F.gelu) before the activation output -- the FFT
                         //    blocks' conv-FFN (common_layers.py:630-637: ffn_1 -> * kernel_size^-0.5 -> gelu)
    BA_RELU_SCALED = 512,   // ... same with relu instead of gelu (hparams['ffn_act'] == 'relu')
    BA_ACT_F16 = 1024,   // write-only row epilogue: the activation output is ONE fp16 tensor (out_hi viewed as __half) instead of bf16 hi/lo
};

// b: batch index, t_warp: first row (within the batch) of this warp's 32 accumulator lanes, grp: column group of the
// warp (0/1: two warps share a TMEM lane quadrant and split the tile's columns), stage: the warp's transpose tile.
// FULL: all 32 rows of the warp are inside the batch (no row predicates).  Rows t >= L are never stored.
template <int N_TILE, int EPI, bool FULL, bool OUT16>
__device__ __forceinline__ void run_epilogue(const EpiParams& e, int Lrows, uint32_t tacc, int b, int t_warp, int n_tile, int grp,
                                             float* stage, int lane, const StepRows& sr) {
    constexpr int BASE = epi_base(EPI);
    constexpr bool kSteps = BASE != EPI;   // a diffusion step per batch item
    (void)sr;
    const LanePos lp = lane_pos(lane);
    const float sc = e.acc_scale != 0.0f ? e.acc_scale : 1.0f;
    const long long row_w = static_cast<long long>(b) * Lrows + t_warp;   // global row of the warp's lane 0
    const int rows_left = Lrows - t_warp - lp.r0;                          // row pair rp is valid iff 2*rp < rows_left
#define B200_ROW_OK(rp) (FULL || 2 * (rp) < rows_left)
    // column range of this warp
    constexpr int kSplit = epi_col_split(N_TILE);
    constexpr int kColsPerGrp = N_TILE / kSplit;
    // kSplit == 1 (narrow tiles): the two warp groups do not split the columns, they alternate TILES (see the kernel's
    // epilogue loop); the posterior epilogue alternates 16-channel chunks instead
    const int c_begin = kSplit == 1 ? 0 : grp * kColsPerGrp;
    (void)rows_left; (void)c_begin; (void)row_w; (void)lp; (void)sc;

    if constexpr (EPI == EPI_F32) {
#pragma unroll 1
        for (int c = c_begin; c < c_begin + kColsPerGrp; c += 32) {
            float2 o[16];
            ld_chunk_t(tacc, c, stage, lane, o, sc);
            const int n = n_tile * N_TILE + c + lp.cc;
            const float2 bias = ldg2(e.bias + n);
            float* p = e.f32_a + (row_w + lp.r0) * e.out_pitch + n;
            const long long st = 2LL * e.out_pitch;
#pragma unroll
            for (int rp = 0; rp < 16; ++rp)
                if (B200_ROW_OK(rp)) st2(p + rp * st, make_float2(o[rp].x + bias.x, o[rp].y + bias.y));
        }
    } else if constexpr (BASE == EPI_INPROJ) {
        const float* dv = e.dvec;
        if constexpr (kSteps) dv += static_cast<long long>(__ldg(sr.t_of_b + b)) * sr.dvec_stride;
#pragma unroll 1
        for (int c = c_begin; c < c_begin + kColsPerGrp; c += 32) {
            float2 o[16];
            ld_chunk_t(tacc, c, stage, lane, o, sc);
            const int n = n_tile * N_TILE + c + lp.cc;
            const float2 bias = ldg2(e.bias + n), d = ldg2(dv + n);
            const long long off0 = (row_w + lp.r0) * e.out_pitch + n, st = 2LL * e.out_pitch;
#pragma unroll
            for (int rp = 0; rp < 16; ++rp) {
                if (B200_ROW_OK(rp)) {
                    const long long off = off0 + rp * st;
                    const float2 x = make_float2(fmaxf(o[rp].x + bias.x, 0.0f), fmaxf(o[rp].y + bias.y, 0.0f));
                    if (e.f32_a != nullptr) st2(e.f32_a + off, x);   // the fp32 residual stream: not kept by the fused layer kernel
                    st_operand2<2>(e, make_float2(x.x + d.x, x.y + d.y), off);
                    if (e.out8 != nullptr)
                        *reinterpret_cast<uint16_t*>(e.out8 + off) = __nv_cvt_float2_to_fp8x2(make_float2(x.x + d.x, x.y + d.y), __NV_SATFINITE, __NV_E4M3);
                }
            }
        }
    } else if constexpr (EPI == EPI_GATE) {
        // tile columns [0, N_TILE/2) = gate pre-activations, [N_TILE/2, N_TILE) = filter pre-activations of
        // the same N_TILE/2 channels (weight rows permuted by the packer).
        constexpr int HALF = N_TILE / 2;
        static_assert(HALF % 64 == 0, "gate epilogue splits HALF over two warp groups");
        const int abl = e.flags;   // ablation bits (timing experiments only): 1 no cp loads, 2 no transposes, 4 no stores, 8 no MUFU math
#pragma unroll 1
        for (int c = grp * (HALF / 2); c < (grp + 1) * (HALF / 2); c += 32) {
            const int nb = n_tile * N_TILE + c + lp.cc;   // packed column of the gate pre-activation ; filter at +HALF
            const int ch = n_tile * HALF + c + lp.cc;     // output channel
            // aux0 = precomputed conditioner projection + biases, f32 [rows][out_pitch] in the packed column order;
            // z goes to out_hi/out_lo [rows][act_pitch] at column out_col0 + channel (the all-layer z matrix)
            const long long cp0 = (row_w + lp.r0) * static_cast<long long>(e.out_pitch) + nb, cst = 2LL * e.out_pitch;
            float2 g[16], f[16], cp[16];
#pragma unroll
            for (int rp = 0; rp < 16; ++rp) cp[rp] = make_float2(0.f, 0.f);
            if (!(abl & 1)) {
#pragma unroll
                for (int rp = 0; rp < 16; ++rp)
                    if (B200_ROW_OK(rp)) cp[rp] = ld2(e.aux0 + cp0 + rp * cst);
            }
            if (abl & 2) {
                float v[32];
                ld_acc32(tacc + c, v, sc);
#pragma unroll
                for (int rp = 0; rp < 16; ++rp) g[rp] = make_float2(v[2 * rp], v[2 * rp + 1]);
            } else {
                ld_chunk_t(tacc, c, stage, lane, g, sc);
            }
#pragma unroll
            for (int rp = 0; rp < 16; ++rp) { g[rp].x += cp[rp].x; g[rp].y += cp[rp].y; }
            if (!(abl & 1)) {
#pragma unroll
                for (int rp = 0; rp < 16; ++rp)
                    if (B200_ROW_OK(rp)) cp[rp] = ld2(e.aux0 + cp0 + HALF + rp * cst);
            }
            if (abl & 2) {
                float v[32];
                ld_acc32(tacc + HALF + c, v, sc);
#pragma unroll
                for (int rp = 0; rp < 16; ++rp) f[rp] = make_float2(v[2 * rp], v[2 * rp + 1]);
            } else {
                ld_chunk_t(tacc, HALF + c, stage, lane, f, sc);
            }
            const long long off0 = (row_w + lp.r0) * static_cast<long long>(e.act_pitch) + e.out_col0 + ch, st = 2LL * e.act_pitch;
#pragma unroll
            for (int rp = 0; rp < 16; ++rp) {
                if (B200_ROW_OK(rp)) {
                    float2 z;
                    if (abl & 8) z = make_float2(g[rp].x * (f[rp].x + cp[rp].x), g[rp].y * (f[rp].y + cp[rp].y));
                    else z = make_float2(fast_sigmoid(g[rp].x) * fast_tanh(f[rp].x + cp[rp].x),
                                         fast_sigmoid(g[rp].y) * fast_tanh(f[rp].y + cp[rp].y));
                    if (!(abl & 4) || z.x == 123.456f) st_operand2<OUT16 ? 1 : 0>(e, z, off0 + rp * st);
                }
            }
        }
    } else if constexpr (BASE == EPI_RES_SKIP) {
        // residual half of the output projection: x <- (x + r + b) / sqrt(2)  (net.py:76-78); also writes the next
        // layer's conv input split(x + d_{l+1}) (net.py:69).  The skip half is not computed per layer: the skip sum is one
        // K = L*C GEMM over all gated activations at the end of the step (DiffusionPlan::enqueue_step).
        [[maybe_unused]] const float* dv = nullptr;   // kSteps: d_{l+1} of this tile's batch item
        if constexpr (kSteps) {
            if (e.dvec != nullptr) dv = e.dvec + static_cast<long long>(__ldg(sr.t_of_b + b)) * sr.dvec_stride;
        }
        const float rs2 = 0.70710678118654752440f;
        const long long st = 2LL * e.out_pitch;
        const int c0g = n_tile * N_TILE;
        // software pipeline: the residual rows of chunk c+1 are in flight while chunk c is processed
        float2 xn[16];
        {
            const long long off0 = (row_w + lp.r0) * e.out_pitch + c0g + c_begin + lp.cc;
#pragma unroll
            for (int rp = 0; rp < 16; ++rp)
                if (B200_ROW_OK(rp)) xn[rp] = ld2(e.f32_a + off0 + rp * st);
        }
#pragma unroll 1
        for (int c = c_begin; c < c_begin + kColsPerGrp; c += 32) {
            const int cl = c0g + c + lp.cc;
            const long long off0 = (row_w + lp.r0) * e.out_pitch + cl;
            float2 x[16];
#pragma unroll
            for (int rp = 0; rp < 16; ++rp) x[rp] = xn[rp];
            if (c + 32 < c_begin + kColsPerGrp) {
#pragma unroll
                for (int rp = 0; rp < 16; ++rp)
                    if (B200_ROW_OK(rp)) xn[rp] = ld2(e.f32_a + off0 + 32 + rp * st);
            }
            float2 o[16];
            ld_chunk_t(tacc, c, stage, lane, o, sc);
            const float2 bias = ldg2(e.bias + cl);
            float2 d = make_float2(0.f, 0.f);
            if constexpr (kSteps) {
                if (e.dvec != nullptr) d = ldg2(dv + cl);
            } else {
                if (e.dvec != nullptr) d = ldg2(e.dvec + cl);
            }
#pragma unroll
            for (int rp = 0; rp < 16; ++rp) {
                if (B200_ROW_OK(rp)) {
                    const long long off = off0 + rp * st;
                    const float2 y = make_float2((x[rp].x + o[rp].x + bias.x) * rs2, (x[rp].y + o[rp].y + bias.y) * rs2);
                    st2(e.f32_a + off, y);
                    if (e.dvec != nullptr)   // not needed after the last layer
                        st_operand2<OUT16 ? 1 : 0>(e, make_float2(y.x + d.x, y.y + d.y), off);
                }
            }
        }
    } else if constexpr (EPI == EPI_RELU_BF16) {
        // y = (acc + bias) * c0, ReLU unless flags & 1  -> bf16 hi/lo      (skip sum / sqrt(L): net.py:126 ; skip_projection + ReLU: :127-128)
#pragma unroll 1
        for (int c = c_begin; c < c_begin + kColsPerGrp; c += 32) {
            float2 o[16];
            ld_chunk_t(tacc, c, stage, lane, o, sc);
            const int n = n_tile * N_TILE + c + lp.cc;
            const float2 bias = ldg2(e.bias + n);
            const long long off0 = (row_w + lp.r0) * e.out_pitch + n, st = 2LL * e.out_pitch;
            const float lo_clamp = (e.flags & 1) ? -3.0e38f : 0.0f;
#pragma unroll
            for (int rp = 0; rp < 16; ++rp)
                if (B200_ROW_OK(rp))
                    st_operand2<2>(e, make_float2(fmaxf((o[rp].x + bias.x) * e.c0, lo_clamp), fmaxf((o[rp].y + bias.y) * e.c0, lo_clamp)),
                                off0 + rp * st);
        }
    } else if constexpr (BASE == EPI_POSTERIOR) {
        // row-per-thread ownership: row t_warp + lane.  x_t lives in the reference layout [B][M][T] (T contiguous): lanes hold
        // consecutive t, so the per-channel accesses below are coalesced.  The channels are processed in chunks of 16 with all
        // loads of a chunk issued before the first use (one exposed DRAM latency per chunk instead of one per channel:
        // profiles/r01_d had this epilogue at 192 us per launch); the two warps of a TMEM lane quadrant alternate chunks.
        static_assert(N_TILE % 16 == 0 && N_TILE <= 96, "posterior epilogue expects <= 96 mel bins, a multiple of 16");
        constexpr int M = N_TILE;
        const int t = t_warp + lane;
        const bool row_ok = FULL || t < Lrows;
        const long long row = row_w + lane;
        const long long LL = Lrows;
        const bool eps_only = (e.flags & 1) != 0;     // bsg_diffnet_forward: write the denoiser output, reference layout
        // kSteps: posterior coefficients and noise stream of this tile's batch item (the uniform-step kernel reads e.c0..c4, e.step)
        [[maybe_unused]] float k0 = 0.f, k1 = 0.f, k2 = 0.f, k3 = 0.f, k4 = 0.f;
        [[maybe_unused]] unsigned int k_step = 0;
        if constexpr (kSteps) {
            const float* cf = sr.coef + 5 * b;
            k0 = __ldg(cf); k1 = __ldg(cf + 1); k2 = __ldg(cf + 2); k3 = __ldg(cf + 3); k4 = __ldg(cf + 4);
            k_step = static_cast<unsigned int>(sr.k_last - __ldg(sr.t_of_b + b));
        }
        float* xt = e.f32_a + (static_cast<long long>(b) * M) * LL + t;
        const float* nz = (!eps_only && e.aux0) ? e.aux0 + (static_cast<long long>(b) * M) * LL + t : nullptr;
        // the noise of the t == 0 step is multiplied by zero (:165)
        const bool draw = !eps_only && nz == nullptr && (kSteps ? k4 : e.c4) != 0.0f;
        const unsigned long long seed = draw ? __ldg(e.seed_ptr) : 0ull;
        const float mask = (e.f32_b != nullptr && row_ok && e.mel2ph != nullptr && !(e.mel2ph[row] > 0)) ? 0.0f : 1.0f;
#pragma unroll 1
        for (int c0 = grp * 16; c0 < N_TILE; c0 += 32) {
            float acc[16], xv[16], zv[16];
            if (row_ok && !eps_only) {
#pragma unroll
                for (int i = 0; i < 16; ++i) xv[i] = xt[static_cast<long long>(c0 + i) * LL];
                if (nz != nullptr) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) zv[i] = nz[static_cast<long long>(c0 + i) * LL];
                }
            }
            ld_acc16(tacc + c0, acc, sc);
            if (!row_ok) continue;
            if (eps_only) {
#pragma unroll
                for (int i = 0; i < 16; ++i) xt[static_cast<long long>(c0 + i) * LL] = acc[i] + __ldg(e.bias + c0 + i);
                continue;
            }
            if (nz == nullptr) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    // one Philox4x32-10 call yields the four normals of channels c0+4q .. c0+4q+3 at this (b, t)
                    float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (draw) z4 = philox_normal4(seed, kSteps ? k_step : e.step, (static_cast<uint64_t>(b) * (M / 4) + (c0 >> 2) + q) * LL + t);
                    zv[4 * q] = z4.x; zv[4 * q + 1] = z4.y; zv[4 * q + 2] = z4.z; zv[4 * q + 3] = z4.w;
                }
            }
            if constexpr (kSteps) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float eps = acc[i] + __ldg(e.bias + c0 + i);
                    const float x = xv[i];
                    float x0 = k0 * x - k1 * eps;
                    if (sr.clip) x0 = fminf(fmaxf(x0, -1.0f), 1.0f);   // clip_denoised=False skips the clamp
                    const float mean = k2 * x0 + k3 * x;
                    xv[i] = mean + k4 * zv[i];
                }
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float eps = acc[i] + __ldg(e.bias + c0 + i);
                    const float x = xv[i];
                    float x0 = e.c0 * x - e.c1 * eps;                       // predict_start_from_noise (:134-138)
                    x0 = fminf(fmaxf(x0, -1.0f), 1.0f);                      // clamp_ (:153-154)
                    const float mean = e.c2 * x0 + e.c3 * x;                 // q_posterior (:140-147)
                    xv[i] = mean + e.c4 * zv[i];                             // (:166), c4 = 0 at t == 0
                }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) xt[static_cast<long long>(c0 + i) * LL] = xv[i];
            // bf16 operand copy [B][T][M] for the next step's input projection
            if (e.out_hi != nullptr) {
                __nv_bfloat16* hrow = e.out_hi + row * e.out_pitch + c0;
                __nv_bfloat16* lrow = e.out_lo ? e.out_lo + row * e.out_pitch + c0 : nullptr;
#pragma unroll
                for (int c = 0; c < 16; c += 8) {
                    uint32_t ph[4], pl[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float h0, h1;
                        __nv_bfloat16 bh0, bl0, bh1, bl1;
                        split_bf16(xv[c + 2 * i], h0, bh0, bl0);
                        split_bf16(xv[c + 2 * i + 1], h1, bh1, bl1);
                        ph[i] = static_cast<uint32_t>(__bfloat16_as_ushort(bh0)) | (static_cast<uint32_t>(__bfloat16_as_ushort(bh1)) << 16);
                        pl[i] = static_cast<uint32_t>(__bfloat16_as_ushort(bl0)) | (static_cast<uint32_t>(__bfloat16_as_ushort(bl1)) << 16);
                    }
                    *reinterpret_cast<uint4*>(hrow + c) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                    if (lrow) *reinterpret_cast<uint4*>(lrow + c) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
                }
            }
            // last step: mel_out = denorm_spec(x) * (mel2ph > 0)   (shallow_diffusion_tts.py:268-272,278-279)
            if (e.f32_b != nullptr) {
                float* mo = e.f32_b + row * M + c0;
#pragma unroll
                for (int c = 0; c < 16; c += 4) {
                    float o[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float mn = __ldg(e.aux1 + c0 + c + i), mx = __ldg(e.aux2 + c0 + c + i);
                        o[i] = ((xv[c + i] + 1.0f) / 2.0f * (mx - mn) + mn) * mask;
                    }
                    *reinterpret_cast<float4*>(mo + c) = make_float4(o[0], o[1], o[2], o[3]);
                }
            }
        }
    } else if constexpr (EPI == EPI_BIAS_ACT) {
        if ((e.flags & BA_ROWS) && !(e.flags & (BA_ADD_RES | BA_ACCUM_F32B))) {
            // Write-only epilogue (first conv of every ResBlock iteration, conv_pre, transposed-conv phases, PitchExtractor GEMMs): nothing is
            // read from global memory, so the shared-memory transposition that buys coalesced READS is pure overhead (~30 thread instructions
            // per output element; the narrow vocoder stages were bound by it, profiles/r01_l).  Each thread keeps the accumulator row that
            // tcgen05.ld hands it (32 consecutive columns) and writes full 32-byte sectors with 256-bit stores: ~6 instructions per element.
            const bool ok = FULL || lane < Lrows - t_warp;
            const long long row = row_w + lane;
#pragma unroll 1
            for (int c = c_begin; c < c_begin + kColsPerGrp; c += 32) {
                float v[32];
                ld_acc32(tacc + c, v, sc);
                const int n = n_tile * N_TILE + c;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 bb = __ldg(reinterpret_cast<const float4*>(e.bias + n) + j);
                    v[4 * j] += bb.x; v[4 * j + 1] += bb.y; v[4 * j + 2] += bb.z; v[4 * j + 3] += bb.w;
                }
                if (e.flags & (BA_GELU | BA_RELU_SCALED)) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const float y = v[i] * e.c0;
                        v[i] = (e.flags & BA_GELU) ? 0.5f * y * (1.0f + erff(y * 0.70710678118654752440f)) : fmaxf(y, 0.0f);
                    }
                }
                if (e.flags & BA_WRITE_F32) {
                    float* dst = e.f32_a + row * e.out_pitch + e.out_col0 + n;
                    if (ok) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            uint32_t q[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) q[i] = __float_as_uint(v[8 * j + i]);
                            stg256(dst + 8 * j, q);
                        }
                    }
                }
                if ((e.flags & BA_WRITE_ACT) && (e.flags & BA_ACT_F16)) {
                    uint32_t q[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const __half2 hh = __floats2half2_rn(fminf(fmaxf(v[2 * i], -65504.0f), 65504.0f), fminf(fmaxf(v[2 * i + 1], -65504.0f), 65504.0f));
                        q[i] = *reinterpret_cast<const uint32_t*>(&hh);
                    }
                    if (ok) {
                        __nv_bfloat16* dh = e.out_hi + row * e.act_pitch + n;
                        stg256(dh, reinterpret_cast<const uint32_t(&)[8]>(q[0]));
                        stg256(dh + 16, reinterpret_cast<const uint32_t(&)[8]>(q[8]));
                    }
                } else if (e.flags & BA_WRITE_ACT) {
                    uint32_t hi[16], lo[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float a = v[2 * i] > 0.0f ? v[2 * i] : v[2 * i] * e.c1;
                        const float bq = v[2 * i + 1] > 0.0f ? v[2 * i + 1] : v[2 * i + 1] * e.c1;
                        const __nv_bfloat162 h = __floats2bfloat162_rn(a, bq);
                        hi[i] = *reinterpret_cast<const uint32_t*>(&h);
                        const __nv_bfloat162 l2 = __floats2bfloat162_rn(a - __uint_as_float(hi[i] << 16), bq - __uint_as_float(hi[i] & 0xffff0000u));
                        lo[i] = *reinterpret_cast<const uint32_t*>(&l2);
                    }
                    if (ok) {
                        __nv_bfloat16* dh = e.out_hi + row * e.act_pitch + n;
                        uint32_t q[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) q[i] = hi[i];
                        stg256(dh, q);
#pragma unroll
                        for (int i = 0; i < 8; ++i) q[i] = hi[8 + i];
                        stg256(dh + 16, q);
                        if (e.out_lo != nullptr) {
                            __nv_bfloat16* dl = e.out_lo + row * e.act_pitch + n;
#pragma unroll
                            for (int i = 0; i < 8; ++i) q[i] = lo[i];
                            stg256(dl, q);
#pragma unroll
                            for (int i = 0; i < 8; ++i) q[i] = lo[8 + i];
                            stg256(dl + 16, q);
                        }
                    }
                }
            }
            return;
        }
        if (e.flags & BA_ROWS_RMW) {
            // Read-modify-write epilogues (second conv of a ResBlock iteration: residual add, running residual / MRF accumulator) in the same
            // row-per-thread ownership: every lane reads and writes whole 32-byte sectors of its own row with 256-bit accesses, 16 columns per
            // pass (loads of the pass are issued before the accumulator is fetched from TMEM).
            const bool ok = FULL || lane < Lrows - t_warp;
            const long long row = row_w + lane;
            const bool add_res = (e.flags & BA_ADD_RES) != 0, accum = (e.flags & BA_ACCUM_F32B) != 0;
            const bool rd_b = accum && !(e.flags & BA_ACCUM_INIT);
#pragma unroll 1
            for (int c = c_begin; c < c_begin + kColsPerGrp; c += 16) {
                const int n = n_tile * N_TILE + c;
                const long long o32 = row * e.out_pitch + e.out_col0 + n;
                float r0[8], r1[8], s0[8], s1[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { r0[i] = r1[i] = s0[i] = s1[i] = 0.0f; }
                if (ok && add_res) {
                    ldg256(e.aux0 + o32, r0);
                    ldg256(e.aux0 + o32 + 8, r1);
                }
                if (ok && rd_b) {
                    ldg256(e.f32_b + o32, s0);
                    ldg256(e.f32_b + o32 + 8, s1);
                }
                float v[16];
                ld_acc16(tacc + c, v, sc);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 bb = __ldg(reinterpret_cast<const float4*>(e.bias + n) + j);
                    v[4 * j] += bb.x; v[4 * j + 1] += bb.y; v[4 * j + 2] += bb.z; v[4 * j + 3] += bb.w;
                }
                if (add_res) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) { v[i] = __fadd_rn(v[i], r0[i]); v[8 + i] = __fadd_rn(v[8 + i], r1[i]); }
                }
                uint32_t q[8];
                if ((e.flags & BA_WRITE_F32) && ok) {
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) q[i] = __float_as_uint(v[8 * j + i]);
                        stg256(e.f32_a + o32 + 8 * j, q);
                    }
                }
                if (accum) {
                    float a[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        a[i] = __fmul_rn(v[i], e.c0);
                        if (rd_b) a[i] = __fadd_rn(a[i], i < 8 ? s0[i & 7] : s1[i & 7]);
                    }
                    if (ok) {
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
#pragma unroll
                            for (int i = 0; i < 8; ++i) q[i] = __float_as_uint(a[8 * j + i]);
                            stg256(e.f32_b + o32 + 8 * j, q);
                        }
                    }
                    if (e.flags & BA_ACT_FROM_B) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = a[i];
                    }
                }
                if (e.flags & BA_WRITE_ACT) {
                    uint32_t lo[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float y0 = v[2 * i] > 0.0f ? v[2 * i] : v[2 * i] * e.c1;
                        const float y1 = v[2 * i + 1] > 0.0f ? v[2 * i + 1] : v[2 * i + 1] * e.c1;
                        const __nv_bfloat162 h = __floats2bfloat162_rn(y0, y1);
                        q[i] = *reinterpret_cast<const uint32_t*>(&h);
                        const __nv_bfloat162 l2 = __floats2bfloat162_rn(y0 - __uint_as_float(q[i] << 16), y1 - __uint_as_float(q[i] & 0xffff0000u));
                        lo[i] = *reinterpret_cast<const uint32_t*>(&l2);
                    }
                    if (ok) {
                        stg256(e.out_hi + row * e.act_pitch + n, q);
                        if (e.out_lo != nullptr) stg256(e.out_lo + row * e.act_pitch + n, lo);
                    }
                }
            }
            return;
        }
        const long long st = 2LL * e.out_pitch, sta = 2LL * e.act_pitch;
#pragma unroll 1
        for (int c = c_begin; c < c_begin + kColsPerGrp; c += 32) {
            const int n = n_tile * N_TILE + c + lp.cc;     // bias / logical channel index
            const long long o32 = (row_w + lp.r0) * e.out_pitch + e.out_col0 + n;
            const long long o16 = (row_w + lp.r0) * e.act_pitch + n;
            float2 r[16], s[16];
            if (e.flags & BA_ADD_RES) {
#pragma unroll
                for (int rp = 0; rp < 16; ++rp)
                    if (B200_ROW_OK(rp)) r[rp] = ld2(e.aux0 + o32 + rp * st);
            }
            if ((e.flags & BA_ACCUM_F32B) && !(e.flags & BA_ACCUM_INIT)) {
#pragma unroll
                for (int rp = 0; rp < 16; ++rp)
                    if (B200_ROW_OK(rp)) s[rp] = ld2(e.f32_b + o32 + rp * st);
            }
            float2 o[16];
            ld_chunk_t(tacc, c, stage, lane, o, sc);
            const float2 bias = ldg2(e.bias + n);
#pragma unroll
            for (int rp = 0; rp < 16; ++rp) {
                if (B200_ROW_OK(rp)) {
                    float2 y = make_float2(o[rp].x + bias.x, o[rp].y + bias.y);
                    if (e.flags & BA_ADD_RES) { y.x += r[rp].x; y.y += r[rp].y; }
                    if (e.flags & BA_WRITE_F32) st2(e.f32_a + o32 + rp * st, y);
                    if (e.flags & BA_ACCUM_F32B) {
                        float2 a = make_float2(y.x * e.c0, y.y * e.c0);
                        if (!(e.flags & BA_ACCUM_INIT)) { a.x += s[rp].x; a.y += s[rp].y; }
                        st2(e.f32_b + o32 + rp * st, a);
                        if (e.flags & BA_ACT_FROM_B) y = a;
                    }
                    if (e.flags & BA_WRITE_ACT) {
                        y.x = y.x > 0.0f ? y.x : y.x * e.c1;
                        y.y = y.y > 0.0f ? y.y : y.y * e.c1;
                        st_split2(y, e.out_hi + o16 + rp * sta, e.out_lo ? e.out_lo + o16 + rp * sta : nullptr);
                    }
                }
            }
        }
    }
#undef B200_ROW_OK
}

// L2 prefetch of the fp32 tiles the epilogue of `tile` will read (this warp's 32 rows x its column group).
template <int N_TILE, int EPI>
__device__ __forceinline__ void prefetch_rmw_tile(const ConvGemmArgs& args, int tile, int tile_rows, int row_in_tile, int grp, int lane) {
    const EpiParams& e = args.epi;
    const int n_tile = tile % args.n_tiles_n;
    const int m = tile / args.n_tiles_n;
    const int b = m / args.tiles_per_batch;
    const int t0 = (m % args.tiles_per_batch) * tile_rows + row_in_tile;
    constexpr int kSplit = epi_col_split(N_TILE);
    constexpr int kCols = N_TILE / kSplit;
    constexpr int kLinesPerRow = (kCols * 4 + 127) / 128;
    const float* src0 = nullptr;
    const float* src1 = nullptr;
    int col = kSplit == 1 ? 0 : grp * kCols;
    if constexpr (EPI == EPI_RES_SKIP) {
        src0 = e.f32_a;
        col += n_tile * N_TILE;
    } else {
        col += e.out_col0 + n_tile * N_TILE;
        if (e.flags & BA_ADD_RES) src0 = e.aux0;
        if ((e.flags & BA_ACCUM_F32B) && !(e.flags & BA_ACCUM_INIT)) src1 = e.f32_b;
    }
    const int rows = min(32, args.L - t0);
    const long long row0 = static_cast<long long>(b) * args.L + t0;
    if constexpr (EPI == EPI_GATE) {
        // conditioner projection tile: this group's 64 gate columns and 64 filter columns (2 x 256 B per row)
        constexpr int HALF = N_TILE / 2;
        for (int idx = lane; idx < rows * 4; idx += 32) {
            const int r = idx >> 2, q = idx & 3;
            const long long off = (row0 + r) * static_cast<long long>(e.out_pitch) + n_tile * N_TILE + grp * (HALF / 2) + (q >> 1) * HALF + (q & 1) * 32;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(e.aux0 + off));
        }
        return;
    }
    for (int idx = lane; idx < rows * kLinesPerRow; idx += 32) {
        const int r = idx / kLinesPerRow, ln = idx % kLinesPerRow;
        const long long off = (row0 + r) * e.out_pitch + col + ln * 32;
        if (src0) asm volatile("prefetch.global.L2 [%0];" ::"l"(src0 + off));
        if (src1) asm volatile("prefetch.global.L2 [%0];" ::"l"(src1 + off));
    }
}

// ---------------------------------------------------------------------------------------------
// The kernel
// ---------------------------------------------------------------------------------------------
template <int N_TILE, int TERMS, bool PAIR = false>
struct GemmSmem {
    static constexpr int kAParts = TERMS == 3 ? 2 : 1;                              // activations: hi/lo only in bf16x3
    static constexpr int kBParts = (TERMS == 2 || TERMS == 3) ? 2 : 1;              // weights: hi/lo in bf16x3 and fp16x2 (TERMS 4: fp16 tiles and e5m2
                                                                                    // correction tiles take turns in single-part slots)
    static constexpr int kASlotRows = TERMS == 1 ? 192 : 144;                       // halo tile capacity
    static constexpr int kAPartBytes = kASlotRows * kBlockK * 2;                    // one of hi / lo
    static constexpr int kBPartBytes = (PAIR ? N_TILE / 2 : N_TILE) * kBlockK * 2;       // PAIR: each CTA stages half of the N columns
    static constexpr int kASlotBytes = kAParts * kAPartBytes;
    static constexpr int kBSlotBytes = kBParts * kBPartBytes;
    static constexpr int kAStages = TERMS == 3 ? 2 : (TERMS == 2 ? B200_ASTAGES2 : 3);
    static constexpr int kBStagesRaw = (kSmemBudget - kAStages * kASlotBytes) / kBSlotBytes;
    static constexpr int kBStages = kBStagesRaw > 12 ? 12 : kBStagesRaw;   // deep enough to hold a small convolution's whole weight set
    static constexpr int kOperandBytes = kAStages * kASlotBytes + kBStages * kBSlotBytes;
    static constexpr int kBarBytes = 512;
    static constexpr int kXposeBytes = kEpiWarps * kStageFloatsPerWarp * 4;   // one 16x36 fp32 transpose tile per epilogue warp
    static constexpr int kTotal = kOperandBytes + kBarBytes + kXposeBytes + 1024;  // +1024 for manual alignment
    static_assert(kBStages >= 2, "need at least a double-buffered weight ring");
    static_assert(kAPartBytes % 1024 == 0 && kBPartBytes % 1024 == 0, "tiles must keep 1024-byte swizzle alignment");
    static_assert((2 * kAStages + 2 * kBStages + 4) * 8 + 8 <= kBarBytes, "barrier area too small");
    static_assert(kTotal <= 227 * 1024, "shared memory budget");
};

__host__ __device__ constexpr int tmem_cols_for(int n) {
    return n <= 32 ? 32 : (n <= 64 ? 64 : (n <= 128 ? 128 : (n <= 256 ? 256 : 512)));
}

// PAIR = true: the kernel is launched in clusters of two CTAs that cooperate on 256-row tiles with
// tcgen05.mma.cta_group::2: CTA rank r stages rows [128r, 128r+128) of A and columns [r*N/2, (r+1)*N/2) of the
// weights, the leader CTA (rank 0) issues every MMA (M = 256) and each CTA's TMEM receives the accumulators of its own
// 128 rows.  Per MMA every SM reads 8 KB of shared memory instead of 12 KB, which is what a single CTA could not
// sustain next to the TMA fill (profiles/r01_d: 1-CTA SS-mode MMAs were shared-memory-bandwidth bound).
//
// MC = true (needs PAIR): clusters of FOUR CTAs = two pairs that work on two different 256-row tiles with the SAME weight
// rows.  Every weight tile is fetched from L2 once per cluster: CTA r loads a quarter of the N rows and multicasts it to
// the CTA with the same rank-in-pair in the other pair (cp.async.bulk.tensor ... .multicast::cluster).  A weight slot is
// free when BOTH pairs' MMAs have retired (tcgen05.commit multicast to all four CTAs, barrier count 2).  L2->SM traffic
// per MMA drops by a third (weights are two thirds of it), which is what starves the MMA issuer in the 2-CTA kernel
// (profiles/r01_g: ~25 % of the issuer's cycles wait on operand barriers at 7.4 TB/s of L2->SM traffic).
template <int N_TILE, int TERMS, int EPI, bool PAIR, bool MC = false>
__global__ void __launch_bounds__(kGemmThreads, 1) conv_gemm_kernel(const __grid_constant__ ConvGemmArgs args) {
    static_assert(!MC || PAIR, "weight multicast is built on 2-CTA tiles");
    using S = GemmSmem<N_TILE, TERMS, PAIR>;
    static_assert(N_TILE % 16 == 0 && N_TILE >= 16 && N_TILE <= 256, "UMMA N constraint for M=128");
    constexpr int kTmemCols = tmem_cols_for(2 * N_TILE);
    // TERMS == 5: fp16 activations x ONE fp16 weight operand (hi only; the packing's 2^p scale still applies): the skip-sum GEMM, a
    // once-per-step linear read-out whose weight rounding does not compound through the layers (tests/tools/exp_skip_x1.py)
    constexpr uint32_t kIdesc = umma_idesc_f16(PAIR ? 2 * kTileM : kTileM, N_TILE, /*fp16=*/TERMS == 2 || TERMS == 4 || TERMS == 5);
    // TERMS == 4 ("fp16 + fp8 correction", PAIR only): amap[0] / wmap[0] = fp16 activations / fp16(W 2^p) as in TERMS 2; after every second
    // 64-channel k-block one 128-channel block of amap[1] = e4m3 activations x wmap[1] = e5m2(W 2^p - hi) on the fp8 pipe (K = 32 per
    // MMA, twice the rate) into the same accumulator -- see diffnet_layer.cuh
    constexpr uint32_t kIdesc8 = umma_idesc_f8(PAIR ? 2 * kTileM : kTileM, N_TILE, 0, 1);
    static_assert(TERMS != 4 || (PAIR && !MC), "the fp8-correction mode is built for 2-CTA tiles");
    constexpr int kTileRows = PAIR ? 2 * kTileM : kTileM;
    // Narrow tiles (N_TILE = 32: the last HiFi-GAN stage) are bound by the epilogue's latency chain, not by its width: instead of
    // idling, the second group of four epilogue warps takes every other tile (accumulator buffer = tile parity = group).
    constexpr bool kAltTiles = epi_col_split(N_TILE) == 1 && epi_base(EPI) != EPI_POSTERIOR;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + S::kAStages * S::kASlotBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kOperandBytes);
    uint64_t* afull_bar = bars;
    uint64_t* aempty_bar = afull_bar + S::kAStages;
    uint64_t* bfull_bar = aempty_bar + S::kAStages;
    uint64_t* bempty_bar = bfull_bar + S::kBStages;
    uint64_t* tfull_bar = bempty_bar + S::kBStages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* xpose = reinterpret_cast<float*>(smem + S::kOperandBytes + S::kBarBytes);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int crank = PAIR ? static_cast<int>(cluster_ctarank()) : 0;          // rank in the cluster
    const int rank = crank & 1;                                                // rank in the CTA pair, 0 = leader
    const int pidx = MC ? (crank >> 1) : 0;                                    // which pair of the cluster
    const uint16_t pair_mask = static_cast<uint16_t>(3u << (2 * pidx));        // the two CTAs of this pair
    constexpr int kClusterCtas = MC ? 4 : (PAIR ? 2 : 1);
    const int worker = static_cast<int>(blockIdx.x) / kClusterCtas;
    const int n_workers = static_cast<int>(gridDim.x) / kClusterCtas;
    // MC: a work unit is (pair of consecutive row tiles, n_tile); pair `pidx` takes row tile 2*mp + pidx (it may not exist:
    // then its loads are zero-filled by the TMA unit (batch index out of range) and its epilogue stores nothing)
    const int n_row_tiles = args.B * args.tiles_per_batch;
    const int n_units = MC ? ((n_row_tiles + 1) / 2) * args.n_tiles_n : args.num_tiles;
#define B200_UNIT_TO_TILE(unit) (MC ? ((2 * ((unit) / args.n_tiles_n) + pidx) * args.n_tiles_n + (unit) % args.n_tiles_n) : (unit))

    if (threadIdx.x == 32) {
        for (int s = 0; s < S::kAStages; ++s) { mbar_init(&afull_bar[s], 1); mbar_init(&aempty_bar[s], 1); }
        for (int s = 0; s < S::kBStages; ++s) { mbar_init(&bfull_bar[s], 1); mbar_init(&bempty_bar[s], MC ? 2 : 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], (PAIR ? 2 * kEpiWarps : kEpiWarps) / (kAltTiles ? 2 : 1)); }
        fence_barrier_init();
    }
    if (warp == 0) {
        if constexpr (PAIR) { tmem_alloc_pair(tmem_slot, kTmemCols); tmem_relinquish_pair(); }
        else { tmem_alloc(tmem_slot, kTmemCols); tmem_relinquish(); }
    }
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // Programmatic dependent launch: everything above (barrier init, TMEM allocation) may overlap the tail of the
    // previous kernel in the stream / graph; global memory written by it is only touched after this wait.  The
    // trigger right behind it lets the NEXT kernel's CTAs be scheduled as soon as SMs drain.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const TapSet& ts = args.taps;

    if (warp == 0 && lane == 0) {
        // ================= TMA producer (one per CTA) =================
        const uint32_t a_bytes = static_cast<uint32_t>(args.a_rows) * kBlockK * 2 * S::kAParts * (PAIR ? 2 : 1);
        const uint32_t b_bytes = S::kBSlotBytes * (PAIR ? 2 : 1);
        int as = 0, bs = 0;
        uint32_t aph = 0, bph = 0;
        const bool tr = args.trace != nullptr;
        long long w_a = 0, w_b = 0;
        const long long t_begin = tr ? clock64() : 0;
        const bool wres = !PAIR && args.w_resident != 0;
        if (wres) {
            // the whole weight set of the convolution, slot = kb * n_taps + tap (n_tiles_n == 1: checked on the host)
            for (int kb = 0; kb < ts.n_kb; ++kb)
                for (int tp = 0; tp < ts.n_taps; ++tp) {
                    const int slot = kb * ts.n_taps + tp;
                    mbar_arrive_expect_tx(&bfull_bar[slot], b_bytes);
                    tma_load_2d(smem_b + slot * S::kBSlotBytes, &args.wmap[0], &bfull_bar[slot], ts.w_col0[tp] + kb * kBlockK, args.w_row0);
                    if (TERMS == 2 || TERMS == 3) tma_load_2d(smem_b + slot * S::kBSlotBytes + S::kBPartBytes, &args.wmap[1], &bfull_bar[slot], ts.w_col0[tp] + kb * kBlockK, args.w_row0);
                }
        }
        for (int unit = worker; unit < n_units; unit += n_workers) {
            const int tile = B200_UNIT_TO_TILE(unit);
            const int n_tile = tile % args.n_tiles_n;
            const int m = tile / args.n_tiles_n;
            const int b = m / args.tiles_per_batch;
            const int t0 = (m % args.tiles_per_batch) * kTileRows + rank * kTileM;
            const int wrow = args.w_row0 + n_tile * N_TILE + rank * (N_TILE / 2) + (MC ? pidx * (N_TILE / 4) : 0);
            for (int kb = 0; kb < ts.n_kb; ++kb) {
                // one halo tile of activations per 64-channel k-block ...
                mbar_wait_tr(&aempty_bar[as], aph ^ 1, tr, w_a);
                uint8_t* sa = smem_a + as * S::kASlotBytes;
                const int ac = ts.a_col0 + kb * kBlockK, ar = t0 + ts.row_shift;
                if constexpr (PAIR) {
                    // both CTAs' bytes are credited to the leader's barrier; only the leader arms it
                    if (rank == 0) mbar_arrive_expect_tx(&afull_bar[as], a_bytes);
                    tma_load_3d_pair(sa, &args.amap[2 * ts.a_src], &afull_bar[as], ac, ar, b);
                    if (TERMS == 3) tma_load_3d_pair(sa + S::kAPartBytes, &args.amap[2 * ts.a_src + 1], &afull_bar[as], ac, ar, b);
                } else {
                    mbar_arrive_expect_tx(&afull_bar[as], a_bytes);
                    tma_load_3d(sa, &args.amap[2 * ts.a_src], &afull_bar[as], ac, ar, b);
                    if (TERMS == 3) tma_load_3d(sa + S::kAPartBytes, &args.amap[2 * ts.a_src + 1], &afull_bar[as], ac, ar, b);
                }
                if (++as == S::kAStages) { as = 0; aph ^= 1; }
                // ... and one weight tile per tap
                for (int tp = 0; tp < (wres ? 0 : ts.n_taps); ++tp) {
                    mbar_wait_tr(&bempty_bar[bs], bph ^ 1, tr, w_b);
                    uint8_t* sb = smem_b + bs * S::kBSlotBytes;
                    const int wc = ts.w_col0[tp] + kb * kBlockK;
                    if constexpr (MC) {
                        // this CTA's quarter of the N rows, written to the same slot of the CTA with the same rank-in-pair in both pairs
                        if (rank == 0) mbar_arrive_expect_tx(&bfull_bar[bs], b_bytes);
                        const uint16_t mc_mask = static_cast<uint16_t>(5u << rank);
                        uint8_t* dq = sb + pidx * (S::kBPartBytes / 2);
                        tma_load_2d_pair_mc(dq, &args.wmap[0], &bfull_bar[bs], wc, wrow, mc_mask);
                        if (TERMS == 2 || TERMS == 3) tma_load_2d_pair_mc(dq + S::kBPartBytes, &args.wmap[1], &bfull_bar[bs], wc, wrow, mc_mask);
                    } else if constexpr (PAIR) {
                        if (rank == 0) mbar_arrive_expect_tx(&bfull_bar[bs], b_bytes);
                        tma_load_2d_pair(sb, &args.wmap[0], &bfull_bar[bs], wc, wrow);
                        if (TERMS == 2 || TERMS == 3) tma_load_2d_pair(sb + S::kBPartBytes, &args.wmap[1], &bfull_bar[bs], wc, wrow);
                    } else {
                        mbar_arrive_expect_tx(&bfull_bar[bs], b_bytes);
                        tma_load_2d(sb, &args.wmap[0], &bfull_bar[bs], wc, wrow);
                        if (TERMS == 2 || TERMS == 3) tma_load_2d(sb + S::kBPartBytes, &args.wmap[1], &bfull_bar[bs], wc, wrow);
                    }
                    if (++bs == S::kBStages) { bs = 0; bph ^= 1; }
                }
                if constexpr (TERMS == 4) {
                    if (kb & 1) {
                        // the fp8 correction block of the 128 channels just covered: e4m3 activations (amap[1]) x e5m2 weight remainders (wmap[1])
                        const int c8 = (kb >> 1) * 128;
                        mbar_wait_tr(&aempty_bar[as], aph ^ 1, tr, w_a);
                        if (rank == 0) mbar_arrive_expect_tx(&afull_bar[as], a_bytes);
                        tma_load_3d_pair(smem_a + as * S::kASlotBytes, &args.amap[1], &afull_bar[as], ts.a_col0 + c8, ar, b);
                        if (++as == S::kAStages) { as = 0; aph ^= 1; }
                        for (int tp = 0; tp < ts.n_taps; ++tp) {
                            mbar_wait_tr(&bempty_bar[bs], bph ^ 1, tr, w_b);
                            if (rank == 0) mbar_arrive_expect_tx(&bfull_bar[bs], b_bytes);
                            tma_load_2d_pair(smem_b + bs * S::kBSlotBytes, &args.wmap[1], &bfull_bar[bs], ts.w_col0[tp] + c8, wrow);
                            if (++bs == S::kBStages) { bs = 0; bph ^= 1; }
                        }
                    }
                }
            }
        }
        if (tr) {
            unsigned long long* t = args.trace + blockIdx.x * 16;
            t[4] = clock64() - t_begin; t[5] = w_a; t[6] = w_b;
        }
    } else if (warp == 1 && lane == 0 && rank == 0) {
        // ================= MMA issuer (single thread; leader CTA only in PAIR mode) =================
        int as = 0, bs = 0;
        uint32_t aph = 0, bph = 0;
        int it = 0;
        const bool tr = args.trace != nullptr;
        long long w_t = 0, w_a = 0, w_b = 0;
        const long long t_begin = tr ? clock64() : 0;
        const bool wres = !PAIR && args.w_resident != 0;
        const int k_steps = args.k_steps > 0 ? args.k_steps : kBlockK / 16;
        if (wres) {
            for (int slot = 0; slot < ts.n_kb * ts.n_taps; ++slot) mbar_wait_tr(&bfull_bar[slot], 0, tr, w_b);
            tc_fence_after();
        }
        for (int unit = worker; unit < n_units; unit += n_workers, ++it) {
            const int acc = it & 1;
            mbar_wait_tr(&tempty_bar[acc], ((it >> 1) & 1) ^ 1, tr, w_t);
            tc_fence_after();
            const uint32_t tacc = tmem_base + acc * N_TILE;
            uint32_t accumulate = 0;
            for (int kb = 0; kb < ts.n_kb; ++kb) {
                mbar_wait_tr(&afull_bar[as], aph, tr, w_a);
                tc_fence_after();
                const uint32_t a_slot = smem_u32(smem_a + as * S::kASlotBytes);
                for (int tp = 0; tp < ts.n_taps; ++tp) {
                    if (!wres) {
                        mbar_wait_tr(&bfull_bar[bs], bph, tr, w_b);
                        tc_fence_after();
                    }
                    const uint32_t a_hi = a_slot + ts.row_off[tp] * (kBlockK * 2);   // tap = row offset into the halo tile
                    const uint32_t a_lo = a_hi + S::kAPartBytes;
                    const uint32_t b_hi = smem_u32(smem_b + (wres ? kb * ts.n_taps + tp : bs) * S::kBSlotBytes);
                    const uint32_t b_lo = b_hi + S::kBPartBytes;
#pragma unroll
                    for (int k = 0; k < kBlockK / 16; ++k) {
                        if (k >= k_steps) continue;   // (no break: the four steps stay unrolled, the skipped ones are predicated off)
                        const uint64_t da = umma_smem_desc<128>(a_hi + k * 32);
                        const uint64_t db = umma_smem_desc<128>(b_hi + k * 32);
                        if constexpr (PAIR) {
                            umma_f16_pair(tacc, da, db, kIdesc, accumulate);
                            if (TERMS == 3) umma_f16_pair(tacc, umma_smem_desc<128>(a_lo + k * 32), db, kIdesc, 1);
                            if (TERMS == 2 || TERMS == 3) umma_f16_pair(tacc, da, umma_smem_desc<128>(b_lo + k * 32), kIdesc, 1);
                        } else {
                            umma_f16(tacc, da, db, kIdesc, accumulate);
                            if (TERMS == 3) umma_f16(tacc, umma_smem_desc<128>(a_lo + k * 32), db, kIdesc, 1);
                            if (TERMS == 2 || TERMS == 3) umma_f16(tacc, da, umma_smem_desc<128>(b_lo + k * 32), kIdesc, 1);
                        }
                        accumulate = 1;
                    }
                    if (wres) continue;
                    // free the weight slot (in both CTAs; MC: one of the two arrivals in all four) when these MMAs retire
                    if constexpr (PAIR) umma_commit_pair(&bempty_bar[bs], MC ? static_cast<uint16_t>(0xF) : pair_mask); else umma_commit(&bempty_bar[bs]);
                    if (++bs == S::kBStages) { bs = 0; bph ^= 1; }
                }
                // free the halo tile after its last tap
                if constexpr (PAIR) umma_commit_pair(&aempty_bar[as], pair_mask); else umma_commit(&aempty_bar[as]);
                if (++as == S::kAStages) { as = 0; aph ^= 1; }
                if constexpr (TERMS == 4) {
                    if (kb & 1) {
                        mbar_wait_tr(&afull_bar[as], aph, tr, w_a);
                        tc_fence_after();
                        const uint32_t a8 = smem_u32(smem_a + as * S::kASlotBytes);
                        for (int tp = 0; tp < ts.n_taps; ++tp) {
                            mbar_wait_tr(&bfull_bar[bs], bph, tr, w_b);
                            tc_fence_after();
                            const uint32_t a_op = a8 + ts.row_off[tp] * 128, b_op = smem_u32(smem_b + bs * S::kBSlotBytes);
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                umma_f8_pair(tacc, umma_smem_desc<128>(a_op + k * 32), umma_smem_desc<128>(b_op + k * 32), kIdesc8, 1);
                            umma_commit_pair(&bempty_bar[bs], pair_mask);
                            if (++bs == S::kBStages) { bs = 0; bph ^= 1; }
                        }
                        umma_commit_pair(&aempty_bar[as], pair_mask);
                        if (++as == S::kAStages) { as = 0; aph ^= 1; }
                    }
                }
            }
            // accumulator complete -> epilogue (of both CTAs)
            if constexpr (PAIR) umma_commit_pair(&tfull_bar[acc], pair_mask); else umma_commit(&tfull_bar[acc]);
        }
        if (tr) {
            unsigned long long* t = args.trace + blockIdx.x * 16;
            t[0] = clock64() - t_begin; t[1] = w_t; t[2] = w_a; t[3] = w_b; t[10] = it;
        }
    } else if (warp >= 2 && warp < 2 + kEpiWarps) {
        // ================= Epilogue warps =================
        const int quad = warp & 3;
        int it = 0;
        // PAIR: the accumulator-free barrier lives in the leader CTA (its MMA thread waits on it)
        const uint32_t tempty_remote0 = PAIR ? map_to_cta(smem_u32(&tempty_bar[0]), static_cast<uint32_t>(crank & ~1)) : 0;
        const bool tr = args.trace != nullptr && warp == 2 && lane == 0;
        long long w_f = 0;
        const long long t_begin = tr ? clock64() : 0;
        for (int unit = worker; unit < n_units; unit += n_workers, ++it) {
            const int tile = B200_UNIT_TO_TILE(unit);
            const int acc = it & 1;
            if (kAltTiles && acc != ((warp - 2) >> 2)) continue;
            const int n_tile = tile % args.n_tiles_n;
            const int m = tile / args.n_tiles_n;
            const int b = m / args.tiles_per_batch;
            const int t_warp = (m % args.tiles_per_batch) * kTileRows + rank * kTileM + quad * 32;
            mbar_wait_tr(&tfull_bar[acc], (it >> 1) & 1, tr, w_f);
            tc_fence_after();
            const uint32_t tacc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * N_TILE;
            float* stage = xpose + (warp - 2) * kStageFloatsPerWarp;
            const int grp = (warp - 2) >> 2;
            if constexpr (epi_base(EPI) == EPI_RES_SKIP || EPI == EPI_BIAS_ACT || EPI == EPI_GATE) {
                const int nu = unit + (kAltTiles ? 2 : 1) * n_workers;   // this group's next tile
                if (nu < n_units && B200_UNIT_TO_TILE(nu) < args.num_tiles)
                    prefetch_rmw_tile<N_TILE, epi_base(EPI)>(args, B200_UNIT_TO_TILE(nu), kTileRows, rank * kTileM + quad * 32, grp, lane);
            }
            // the fp16x2 per-layer GEMMs (gate, residual) feed fp16x2 consumers: fp16 operand output decided at compile time
            if (MC && b >= args.B) { /* the odd row tile of the last unit does not exist */ }
            else if (args.L - t_warp >= 32) run_epilogue<N_TILE, EPI, true, TERMS == 2 || TERMS == 4>(args.epi, args.L, tacc, b, t_warp, n_tile, grp, stage, lane, args.steps);
            else run_epilogue<N_TILE, EPI, false, TERMS == 2 || TERMS == 4>(args.epi, args.L, tacc, b, t_warp, n_tile, grp, stage, lane, args.steps);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (PAIR) mbar_arrive_remote(tempty_remote0 + acc * 8);
                else mbar_arrive(&tempty_bar[acc]);
            }
        }
        if (tr) {
            unsigned long long* t = args.trace + blockIdx.x * 16;
            t[7] = clock64() - t_begin; t[8] = w_f;
        }
    }

    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all(); else __syncthreads();   // PAIR: no CTA may exit while its peer can still signal it
    if (warp == 0) {
        tc_fence_after();
        if constexpr (PAIR) tmem_dealloc_pair(tmem_base, kTmemCols); else tmem_dealloc(tmem_base, kTmemCols);
    }
#undef B200_UNIT_TO_TILE
}

}  // namespace b200
