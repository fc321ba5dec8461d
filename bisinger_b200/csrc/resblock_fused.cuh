// One iteration of HiFi-GAN's ResBlock1 as ONE persistent kernel (modules/hifigan/hifigan.py:54-61):
//
//     xt = conv2( lrelu( conv1( lrelu(x), dilation d ) ), dilation 1 ) + x
//
// for the stages with C <= 128 channels.  The vocoder's residual stream lives in HBM as ONE 16-bit tensor a = fp16(lrelu(x)) --
// leaky_relu is invertible (x = a > 0 ? a : a / slope), so the conv input and the residual are the same bytes -- and the
// intermediate activation lrelu(conv1(..)) never leaves the SM:
//
//   producer warp   TMA: halo tile of a (128 + (k-1)(d+1) rows, zero-filled outside the utterance = the reference's zero padding)
//   MMA warp        conv1: taps = row offsets into the halo tile (as conv_gemm.cuh) -> fp32 accumulator in TMEM
//   epilogue-1      TMEM -> + bias1 -> lrelu -> fp16 -> SHARED memory, written directly in the SWIZZLE_128B K-major layout
//                   the tensor core reads (rows outside [0, L) are written as zeros: conv2's zero padding)
//   MMA warp        conv2: taps = row offsets into that shared-memory tile -> second TMEM accumulator
//   epilogue-2      TMEM -> + bias2 + x (inverse lrelu of the a rows, re-read through L2) -> fp16 lrelu -> HBM, or the MRF
//                   sum  sum_j ResBlock_j(x) / num_kernels  (hifigan.py:161-168) in its last iteration
//
// A tile computes 128 rows of the intermediate activation and V = 128 - (k - 1) output rows (halo recompute: 1.6 % / 4.9 % / 8.5 %
// for k = 3 / 7 / 11).  HBM traffic per iteration: one read and one write of the 16-bit stream (round 1: eight such passes through
// fp32 + bf16 copies).  Both accumulators are double-buffered in TMEM (4 C <= 512 columns) and the two epilogues are separate warp
// groups, so conv1 of tile i+1, epilogue-1 of tile i+1, conv2 of tile i and epilogue-2 of tile i-1 overlap.
// The weights of both convolutions stay resident in shared memory when they fit (always for C = 32, k <= 7 for C = 64); otherwise
// they stream through a ring in the order the MMA warp consumes them.
// MMA issue: the WHOLE warp runs the issue loop convergently and elects one lane inside the asm block, so descriptors and the
// accumulator address stay in uniform registers (UIADD3 + UTCHMMA, no per-MMA ELECT / R2UR / branch: profiles/r01_p).
#pragma once
#include "conv_gemm.cuh"

namespace b200 {

struct ResblockArgs {
    CUtensorMap amap;            // a = fp16 lrelu(x) [B][L][C], box = 64 channels x a_rows rows
    CUtensorMap w1map, w2map;    // fp16 weights [C][ntaps * Cw] K-major (Cw = C, taps packed densely), box = 64 x C
    int B, L;
    int tiles_per_batch, num_tiles;
    int ntaps, dil;
    int a_rows;                  // rows of the halo box: 128 + (ntaps - 1) * dil, rounded up to a multiple of 8
    int V;                       // output rows per tile: 128 - (ntaps - 1)
    const float* bias1;
    const float* bias2;
    const __half* a_in;          // the tensor behind amap (residual rows)
    void* out;                   // mode 0: next a = fp16 lrelu(y, 0.1); modes 3-4: the fp16 or bf16 stage output (see mode)
    __half* sum;                 // modes 1-3: MRF accumulator (fp16, raw); not touched in modes 0 and 4
    int mode;                    // 0: a_out = lrelu(y) | 1: sum = y c0 | 2: sum += y c0 | 3: out = lrelu(sum + y c0, slope_out)
                                 // | 4: out = lrelu(y c0, slope_out) (the only ResBlock of a single-kernel MRF: no sum to read)
    int out_bf16;                // modes 3-4: out is bf16 (operand of the next stage's transposed convolution) instead of fp16
    float c0, slope_out;
    int w_slots;                 // weight tiles the shared-memory weight area holds
    int w_resident;              // 2: all weight tiles of both convolutions are loaded once per CTA (2 * n_wtiles <= w_slots); 1: conv1's tiles
                                 //    are resident and conv2's stream through the remaining slots (n_wtiles + 2 <= w_slots); 0: both stream
    unsigned long long* trace;   // optional [grid][16] cycle counters of the roles (tests/tools/gpu_probe.py), or null
};

template <int C>
struct ResblockSmem {
    static constexpr int kNKB = C >= 64 ? C / 64 : 1;
    static constexpr int kASlotBytes = 184 * 128;                 // halo slab of one k-block (k = 11, d = 5: 178 rows)
    static constexpr int kAStages = 3;
    static constexpr int kTSlabBytes = 144 * 128;                 // intermediate tile: 128 rows + (k - 1) rows of slack
    static constexpr int kTBytes = kNKB * kTSlabBytes;
    static constexpr int kWTileBytes = C * 128;                   // one weight tile: C rows (N) x 64 K-columns
    static constexpr int kWArea = C == 32 ? 49152 : (C == 64 ? 114688 : 65536);
    static constexpr int kWSlots = kWArea / kWTileBytes;
    static constexpr int kOffT = kAStages * kASlotBytes;
    static constexpr int kOffW = kOffT + 2 * kTBytes;
    static constexpr int kOffVec = kOffW + kWArea;                // bias1, bias2
    static constexpr int kOffBar = kOffVec + 2 * C * 4;
    static constexpr int kBarBytes = 512;
    static constexpr int kTotal = kOffBar + kBarBytes + 1024;
    static_assert(kOffT % 1024 == 0 && kOffW % 1024 == 0 && kTSlabBytes % 1024 == 0 && kWTileBytes % 1024 == 0, "swizzle alignment");
    static_assert((2 * kAStages + 2 * kWSlots + 12 + 1) * 8 + 8 <= kBarBytes, "barrier area too small");
    static_assert(kTotal <= 227 * 1024, "shared memory budget");
};

constexpr int kRbThreads = 32 * 10;   // producer, MMA, 4 x epilogue-1, 4 x epilogue-2

// ---- MMA issue helpers: called by ALL lanes of the issuing warp (convergent); one elected lane issues ----------------------------------
__device__ __forceinline__ void mma_f16_x4(uint32_t tacc, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p, q, e;\n\t.reg .b64 a1, b1;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.eq.b32 q, 0, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "add.s64 a1, %1, 2;\n\tadd.s64 b1, %2, 2;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t"
        "add.s64 a1, %1, 4;\n\tadd.s64 b1, %2, 4;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t"
        "add.s64 a1, %1, 6;\n\tadd.s64 b1, %2, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t}"
        ::"r"(tacc), "l"(da), "l"(db), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void mma_f16_x2(uint32_t tacc, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p, q, e;\n\t.reg .b64 a1, b1;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.eq.b32 q, 0, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "add.s64 a1, %1, 2;\n\tadd.s64 b1, %2, 2;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t}"
        ::"r"(tacc), "l"(da), "l"(db), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint64_t* bar) {   // whole warp; one lane commits
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void sts128u(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {   // saturating: an out-of-range activation must not become inf
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
__device__ __forceinline__ float lrelu_f(float v, float slope) { return v > 0.0f ? v : v * slope; }


// ---- warp-uniform mbarrier wait (all 32 lanes poll; the loop condition is a vote, so control flow stays convergent and the
//      compiler can keep the issue loop's state in uniform registers) ------------------------------------------------------------------
__device__ __forceinline__ bool mbar_try_wait_s(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_warp(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!__all_sync(0xffffffffu, mbar_try_wait_s(bar, parity))) {
        if (++spins > (1u << 26)) {   // ~seconds: a protocol bug must not hang the GPU box -- trap instead
            if ((threadIdx.x & 31) == 0) printf("resblock_iter_kernel: block %d waited too long on barrier %u parity %u\n", blockIdx.x, bar, parity);
            __trap();
        }
    }
}
__device__ __forceinline__ void umma_commit_elect_s(uint32_t bar) {   // whole warp; one lane commits
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(bar)
        : "memory");
}

// shared-memory addresses of everything the MMA warp touches (all warp-uniform)
struct RbMmaCtx {
    uint32_t smem_a, smem_t, smem_w;
    uint32_t afull, aempty, wfull, wempty, acc1_full, acc1_empty, acc2_full, acc2_empty, t_full, t_empty, wres_full;
    uint32_t tmem_base;
    int n_my, dil, w_slots, wres;
    unsigned long long* trace;   // this CTA's 16 counters or null
};

// The MMA warp's whole loop, specialised for the tap count so that the tap loops unroll with immediate descriptor offsets.
template <int C, int NT>
__device__ __forceinline__ void rb_mma_role(const RbMmaCtx& x) {
    using S = ResblockSmem<C>;
    constexpr int N = C, NKB = S::kNKB;
    constexpr uint32_t kIdesc = umma_idesc_f16(kTileM, N, /*fp16=*/true);
    constexpr int TILE16 = S::kWTileBytes >> 4;                       // weight tile size in descriptor units
    constexpr int NWT = C == 32 ? (NT + 1) / 2 : NT * NKB;            // weight tiles per convolution
    const int ring0 = x.wres == 1 ? NWT : 0;
    int as = 0, ws = ring0;
    uint32_t aph = 0, wph = 0;
    const bool tr = x.trace != nullptr;
    long long w_acc1 = 0, w_a = 0, w_w = 0, w_acc2 = 0, w_t = 0;
    const long long t_begin = tr ? clock64() : 0;
    auto wait_tr = [&](uint32_t bar, uint32_t parity, long long& acc) {
        if (!tr) { mbar_wait_warp(bar, parity); return; }
        const long long t0 = clock64();
        mbar_wait_warp(bar, parity);
        acc += clock64() - t0;
    };
    if (x.wres) { mbar_wait_warp(x.wres_full, 0); tc_fence_after(); }
    const uint64_t w_desc0 = umma_smem_desc<128>(x.smem_w);
    const uint64_t a_tap_step = static_cast<uint64_t>(x.dil) * 8;     // descriptor units of 16 bytes: dil rows x 128 B
    // all taps of k-block kb of convolution `conv` into tacc; A operand of tap tp at a_desc + tp * a_step
    auto conv_taps = [&](uint32_t tacc, uint64_t a_desc, uint64_t a_step, int conv, int kb, uint32_t first_acc) {
        if (x.wres == 2 || (x.wres == 1 && conv == 0)) {
            const uint64_t b0 = w_desc0 + static_cast<uint64_t>(conv * NWT * TILE16) + static_cast<uint64_t>(C == 32 ? 0 : kb * TILE16);
#pragma unroll
            for (int tp = 0; tp < NT; ++tp) {
                if (C == 32) mma_f16_x2(tacc, a_desc + tp * a_step, b0 + static_cast<uint64_t>((tp >> 1) * TILE16 + (tp & 1) * 4), kIdesc, tp == 0 ? first_acc : 1u);
                else mma_f16_x4(tacc, a_desc + tp * a_step, b0 + static_cast<uint64_t>(tp * NKB * TILE16), kIdesc, tp == 0 ? first_acc : 1u);
            }
        } else {
#pragma unroll
            for (int tp = 0; tp < NT; ++tp) {
                if (C != 32 || (tp & 1) == 0) { wait_tr(x.wfull + ws * 8, wph, w_w); tc_fence_after(); }
                const uint64_t b = w_desc0 + static_cast<uint64_t>(ws * TILE16 + (C == 32 ? (tp & 1) * 4 : 0));
                if (C == 32) mma_f16_x2(tacc, a_desc + tp * a_step, b, kIdesc, tp == 0 ? first_acc : 1u);
                else mma_f16_x4(tacc, a_desc + tp * a_step, b, kIdesc, tp == 0 ? first_acc : 1u);
                if (C != 32 || (tp & 1) || tp + 1 == NT) {
                    umma_commit_elect_s(x.wempty + ws * 8);
                    if (++ws == x.w_slots) { ws = ring0; wph ^= 1; }
                }
            }
        }
    };
    auto conv1 = [&](int it) {
        const int buf = it & 1;
        // acc1[buf] is free without a wait of its own: conv1(it) is issued after conv2(it - 2), which waited for t_full(it - 2), and
        // epilogue-1 signals that barrier only after it has read acc1[buf] out of TMEM
        (void)w_acc1;
#pragma unroll
        for (int kb = 0; kb < NKB; ++kb) {
            wait_tr(x.afull + as * 8, aph, w_a);
            tc_fence_after();
            conv_taps(x.tmem_base + buf * N, umma_smem_desc<128>(x.smem_a + as * S::kASlotBytes), a_tap_step, 0, kb, kb == 0 ? 0u : 1u);
            umma_commit_elect_s(x.aempty + as * 8);
            if (++as == S::kAStages) { as = 0; aph ^= 1; }
        }
        umma_commit_elect_s(x.acc1_full + buf * 8);
    };
    auto conv2 = [&](int it) {
        const int buf = it & 1;
        wait_tr(x.acc2_empty + buf * 8, ((it >> 1) & 1) ^ 1, w_acc2);
        wait_tr(x.t_full + buf * 8, (it >> 1) & 1, w_t);
        tc_fence_after();
#pragma unroll
        for (int kb = 0; kb < NKB; ++kb)
            conv_taps(x.tmem_base + (2 + buf) * N, umma_smem_desc<128>(x.smem_t + buf * S::kTBytes + kb * S::kTSlabBytes), 8, 1, kb, kb == 0 ? 0u : 1u);
        umma_commit_elect_s(x.acc2_full + buf * 8);
        umma_commit_elect_s(x.t_empty + buf * 8);
    };
    if (x.n_my > 0) conv1(0);
    for (int it = 0; it < x.n_my; ++it) {
        if (it + 1 < x.n_my) conv1(it + 1);
        conv2(it);
    }
    if (tr && (threadIdx.x & 31) == 0) {
        x.trace[0] = clock64() - t_begin; x.trace[1] = w_acc1; x.trace[2] = w_a; x.trace[3] = w_w; x.trace[4] = w_acc2; x.trace[5] = w_t;
        x.trace[6] = x.n_my;
    }
}

template <int C>
__global__ void __launch_bounds__(kRbThreads, 1) resblock_iter_kernel(const __grid_constant__ ResblockArgs args) {
    using S = ResblockSmem<C>;
    constexpr int N = C;
    constexpr int NKB = S::kNKB;
    constexpr int kTmemCols = 4 * N;   // acc1[2], acc2[2]
    constexpr float kSlope = 0.1f, kInvSlope = 10.0f;   // LRELU_SLOPE, hifigan.py:11

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    const uint32_t smem_a = smem_u32(smem);
    const uint32_t smem_t = smem_a + S::kOffT;
    const uint32_t smem_w = smem_a + S::kOffW;
    float* vec = reinterpret_cast<float*>(smem + S::kOffVec);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kOffBar);
    uint64_t* afull = bars;
    uint64_t* aempty = afull + S::kAStages;
    uint64_t* wfull = aempty + S::kAStages;
    uint64_t* wempty = wfull + S::kWSlots;
    uint64_t* acc1_full = wempty + S::kWSlots;
    uint64_t* acc1_empty = acc1_full + 2;
    uint64_t* acc2_full = acc1_empty + 2;
    uint64_t* acc2_empty = acc2_full + 2;
    uint64_t* t_full = acc2_empty + 2;
    uint64_t* t_empty = t_full + 2;
    uint64_t* wres_full = t_empty + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wres_full + 1);

    const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // warp-uniform for the compiler, too
    const int lane = threadIdx.x & 31;
    const int ntaps = args.ntaps;
    const int n_wt = C == 32 ? (ntaps + 1) / 2 : ntaps * NKB;   // weight tiles per convolution (C = 32: two taps share a 64-column tile)
    const int wres = args.w_resident;                      // 0 / 1 / 2, see ResblockArgs
    const int ring0 = wres == 1 ? n_wt : 0;                // first slot of the streaming ring
    const int w_slots = args.w_slots;

    if (threadIdx.x == 32) {
        for (int s = 0; s < S::kAStages; ++s) { mbar_init(&afull[s], 1); mbar_init(&aempty[s], 1); }
        for (int s = 0; s < S::kWSlots; ++s) { mbar_init(&wfull[s], 1); mbar_init(&wempty[s], 1); }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&acc1_full[a], 1); mbar_init(&acc1_empty[a], 4);
            mbar_init(&acc2_full[a], 1); mbar_init(&acc2_empty[a], 4);
            mbar_init(&t_full[a], 4); mbar_init(&t_empty[a], 1);
        }
        mbar_init(wres_full, 1);
        fence_barrier_init();
    }
    if (warp == 0) { tmem_alloc(tmem_slot, kTmemCols); tmem_relinquish(); }
    for (int i = threadIdx.x; i < 2 * C; i += kRbThreads) vec[i] = i < C ? args.bias1[i] : args.bias2[i - C];   // weights: not written by the previous kernel
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const int n_my = (args.num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
    auto tile_of = [&](int it) { return static_cast<int>(blockIdx.x) + it * static_cast<int>(gridDim.x); };
    const int h2 = (ntaps - 1) / 2;              // conv2: dilation 1
    const int halo = h2 + h2 * args.dil;         // rows of a before the first output row

    if (warp == 0 && lane == 0) {
        // ================= TMA producer =================
        const uint32_t a_bytes = static_cast<uint32_t>(args.a_rows) * 128;
        int as = 0;
        uint32_t aph = 0, wph = 0;
        int ws = ring0;
        auto load_w = [&](const CUtensorMap* map, int wt) {   // weight tile wt of one convolution, through the ring
            mbar_wait(&wempty[ws], wph ^ 1);
            mbar_arrive_expect_tx(&wfull[ws], S::kWTileBytes);
            tma_load_2d(smem + S::kOffW + ws * S::kWTileBytes, map, &wfull[ws], wt * 64, 0);
            if (++ws == w_slots) { ws = ring0; wph ^= 1; }
        };
        if (wres) {
            mbar_arrive_expect_tx(wres_full, static_cast<uint32_t>(wres * n_wt) * S::kWTileBytes);
            for (int wt = 0; wt < n_wt; ++wt) tma_load_2d(smem + S::kOffW + wt * S::kWTileBytes, &args.w1map, wres_full, wt * 64, 0);
            if (wres == 2)
                for (int wt = 0; wt < n_wt; ++wt) tma_load_2d(smem + S::kOffW + (n_wt + wt) * S::kWTileBytes, &args.w2map, wres_full, wt * 64, 0);
        }
        auto conv1_loads = [&](int it) {
            const int m = tile_of(it);
            const int b = m / args.tiles_per_batch;
            const int o0 = (m % args.tiles_per_batch) * args.V;
            for (int kb = 0; kb < NKB; ++kb) {
                mbar_wait(&aempty[as], aph ^ 1);
                mbar_arrive_expect_tx(&afull[as], a_bytes);
                tma_load_3d(smem + as * S::kASlotBytes, &args.amap, &afull[as], kb * 64, o0 - halo, b);
                if (++as == S::kAStages) { as = 0; aph ^= 1; }
                if (wres == 0) {
                    if (C == 32) { for (int wt = 0; wt < n_wt; ++wt) load_w(&args.w1map, wt); }
                    else { for (int tp = 0; tp < ntaps; ++tp) load_w(&args.w1map, tp * NKB + kb); }
                }
            }
        };
        auto conv2_loads = [&]() {
            if (wres == 2) return;
            for (int kb = 0; kb < NKB; ++kb) {
                if (C == 32) { for (int wt = 0; wt < n_wt; ++wt) load_w(&args.w2map, wt); }
                else { for (int tp = 0; tp < ntaps; ++tp) load_w(&args.w2map, tp * NKB + kb); }
            }
        };
        // same order as the MMA warp: conv1(0) | conv1(i+1), conv2(i) ...
        if (n_my > 0) conv1_loads(0);
        for (int it = 0; it < n_my; ++it) {
            if (it + 1 < n_my) conv1_loads(it + 1);
            conv2_loads();
        }
    } else if (warp == 1) {
        // ================= MMA issuer: the whole warp, convergent; one elected lane issues =================
        RbMmaCtx x;
        x.smem_a = smem_a; x.smem_t = smem_t; x.smem_w = smem_w;
        x.afull = smem_u32(afull); x.aempty = smem_u32(aempty); x.wfull = smem_u32(wfull); x.wempty = smem_u32(wempty);
        x.acc1_full = smem_u32(acc1_full); x.acc1_empty = smem_u32(acc1_empty); x.acc2_full = smem_u32(acc2_full);
        x.acc2_empty = smem_u32(acc2_empty); x.t_full = smem_u32(t_full); x.t_empty = smem_u32(t_empty); x.wres_full = smem_u32(wres_full);
        x.tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
        x.n_my = n_my; x.dil = args.dil; x.w_slots = w_slots; x.wres = wres;
        x.trace = args.trace ? args.trace + blockIdx.x * 16 : nullptr;
        switch (ntaps) {
            case 3: rb_mma_role<C, 3>(x); break;
            case 5: rb_mma_role<C, 5>(x); break;
            case 7: rb_mma_role<C, 7>(x); break;
            case 9: rb_mma_role<C, 9>(x); break;
            case 11: rb_mma_role<C, 11>(x); break;
            default: rb_mma_role<C, 1>(x); break;   // ntaps == 1
        }
    } else if (warp >= 2 && warp < 6) {
        // ================= epilogue-1: TMEM -> bias, lrelu -> fp16 -> swizzled shared-memory tile (conv2's A operand) =================
        const int quad = warp & 3;
        const int r = quad * 32 + lane;          // row of the intermediate tile
        const bool tr = args.trace != nullptr && warp == 2 && lane == 0;
        long long w_f = 0, w_te = 0;
        const long long t_begin = tr ? clock64() : 0;
        for (int it = 0; it < n_my; ++it) {
            const int buf = it & 1;
            const int m = tile_of(it);
            const int o0 = (m % args.tiles_per_batch) * args.V;
            const int g = o0 - h2 + r;           // row of this thread inside the utterance
            const bool inside = g >= 0 && g < args.L;
            mbar_wait_tr(&acc1_full[buf], (it >> 1) & 1, tr, w_f);
            mbar_wait_tr(&t_empty[buf], ((it >> 1) & 1) ^ 1, tr, w_te);
            tc_fence_after();
            const uint32_t tacc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * N;
            const uint32_t trow = smem_t + buf * S::kTBytes + r * 128;
            const uint32_t sw = static_cast<uint32_t>(r & 7);
#pragma unroll 1
            for (int c = 0; c < C; c += 32) {
                uint32_t v[32];
                __syncwarp();
                tmem_ld32(tacc + c, v);
                tmem_ld_wait32(v);
                uint32_t h[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float2 bb = *reinterpret_cast<const float2*>(vec + c + 2 * i);
                    const float y0 = lrelu_f(__uint_as_float(v[2 * i]) + bb.x, kSlope);
                    const float y1 = lrelu_f(__uint_as_float(v[2 * i + 1]) + bb.y, kSlope);
                    h[i] = inside ? pack_h2(y0, y1) : 0u;
                }
                // 32 channels = four 16-byte chunks of the row's 128-byte line in slab c / 64; chunk j sits at (j ^ (row & 7))
                const uint32_t slab = trow + (c >> 6) * S::kTSlabBytes;
                const uint32_t j0 = static_cast<uint32_t>((c & 63) >> 3);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    sts128u(slab + (((j0 + j) ^ sw) << 4), h[4 * j], h[4 * j + 1], h[4 * j + 2], h[4 * j + 3]);
            }
            tc_fence_before();
            fence_proxy_async_smem();            // the tensor core reads the tile through the async proxy
            __syncwarp();
            if (lane == 0) mbar_arrive(&t_full[buf]);   // also hands acc1[buf] back (see the MMA warp)
        }
        if (tr) { unsigned long long* t = args.trace + blockIdx.x * 16; t[7] = clock64() - t_begin; t[8] = w_f; t[9] = w_te; }
    } else if (warp >= 6) {
        // ================= epilogue-2: TMEM -> bias + residual -> HBM =================
        const int quad = warp & 3;
        const int q = quad * 32 + lane;          // output row of the tile
        const float* b2 = vec + C;
        const bool tr = args.trace != nullptr && warp == 6 && lane == 0;
        long long w_f = 0;
        const long long t_begin = tr ? clock64() : 0;
        for (int it = 0; it < n_my; ++it) {
            const int buf = it & 1;
            const int m = tile_of(it);
            const int b = m / args.tiles_per_batch;
            const int g = (m % args.tiles_per_batch) * args.V + q;
            const bool ok = q < args.V && g < args.L;
            const long long row = static_cast<long long>(b) * args.L + g;
            const __half* xrow = args.a_in + row * C;
            // (the residual rows were fetched by this tile's TMA a moment ago: the loads below are L2 hits)
            mbar_wait_tr(&acc2_full[buf], (it >> 1) & 1, tr, w_f);
            tc_fence_after();
            const uint32_t tacc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + (2 + buf) * N;
#pragma unroll 1
            for (int c = 0; c < C; c += 32) {
                float xa[8], xb[8], sa[8], sb[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { xa[i] = xb[i] = sa[i] = sb[i] = 0.0f; }
                if (ok) {
                    ldg256(xrow + c, xa);        // 16 fp16 each
                    ldg256(xrow + c + 16, xb);
                    if (args.mode == 2 || args.mode == 3) {
                        ldg256(args.sum + row * C + c, sa);
                        ldg256(args.sum + row * C + c + 16, sb);
                    }
                }
                uint32_t v[32];
                __syncwarp();
                tmem_ld32(tacc + c, v);
                tmem_ld_wait32(v);
                float y[32];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const uint32_t px = __float_as_uint(i < 8 ? xa[i] : xb[i - 8]);
                    const float2 a2 = __half22float2(*reinterpret_cast<const __half2*>(&px));
                    const float x0 = a2.x > 0.0f ? a2.x : a2.x * kInvSlope, x1 = a2.y > 0.0f ? a2.y : a2.y * kInvSlope;   // inverse lrelu
                    y[2 * i] = __uint_as_float(v[2 * i]) + b2[c + 2 * i] + x0;
                    y[2 * i + 1] = __uint_as_float(v[2 * i + 1]) + b2[c + 2 * i + 1] + x1;
                }
                uint32_t o[16];
                if (args.mode == 0) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) o[i] = pack_h2(lrelu_f(y[2 * i], kSlope), lrelu_f(y[2 * i + 1], kSlope));
                    if (ok) {
                        __half* dst = reinterpret_cast<__half*>(args.out) + row * C + c;
                        stg256(dst, reinterpret_cast<const uint32_t(&)[8]>(o[0]));
                        stg256(dst + 16, reinterpret_cast<const uint32_t(&)[8]>(o[8]));
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        float s0 = y[2 * i] * args.c0, s1 = y[2 * i + 1] * args.c0;
                        if (args.mode == 2 || args.mode == 3) {
                            const uint32_t ps = __float_as_uint(i < 8 ? sa[i] : sb[i - 8]);
                            const float2 s2 = __half22float2(*reinterpret_cast<const __half2*>(&ps));
                            s0 += s2.x; s1 += s2.y;
                        }
                        y[2 * i] = s0; y[2 * i + 1] = s1;
                    }
                    if (args.mode < 3) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) o[i] = pack_h2(y[2 * i], y[2 * i + 1]);
                        if (ok) {
                            __half* dst = args.sum + row * C + c;
                            stg256(dst, reinterpret_cast<const uint32_t(&)[8]>(o[0]));
                            stg256(dst + 16, reinterpret_cast<const uint32_t(&)[8]>(o[8]));
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const float z0 = lrelu_f(y[2 * i], args.slope_out), z1 = lrelu_f(y[2 * i + 1], args.slope_out);
                            o[i] = args.out_bf16 ? pack_bf16(z0, z1) : pack_h2(z0, z1);
                        }
                        if (ok) {
                            uint16_t* dst = reinterpret_cast<uint16_t*>(args.out) + row * C + c;
                            stg256(dst, reinterpret_cast<const uint32_t(&)[8]>(o[0]));
                            stg256(dst + 16, reinterpret_cast<const uint32_t(&)[8]>(o[8]));
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_relaxed(&acc2_empty[buf]);
        }
        if (tr) { unsigned long long* t = args.trace + blockIdx.x * 16; t[10] = clock64() - t_begin; t[11] = w_f; }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

}  // namespace b200
