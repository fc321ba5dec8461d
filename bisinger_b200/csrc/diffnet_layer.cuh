// The DiffNet ResidualBlocks (usr/diff/net.py:58-78) as ONE persistent 2-CTA kernel: one launch runs a range of layers
// (normally all 20 of a diffusion step), row tiles flowing from layer to layer as soon as their inputs are complete.
//
// Per pair tile n (256 rows: one 128-row slab per CTA of the pair, see "Slabs" below) three GEMM "ops" run on one producer /
// MMA / epilogue pipeline:
//     G(n,0)  G(n,1)   : acc[256 x 256] = conv_dilated(xa)[:, gate | filter rows of channel half h]            (K = 3 x 256)
//                        epilogue: + conditioner projection, sigmoid * tanh -> z (fp16, the all-layer z matrix)
//     R(n)             : acc[256 x 256] = z[rows, this layer's columns] * W_res^T                               (K = 256)
//                        epilogue: x = (x + acc + b) / sqrt2 with x = fp16 conv input - d_l (the residual stream is carried only
//                        as the conv input) ; fp16 / e4m3 of (x + d_next) -> next layer's conv input
// issued in the order  G(0,0) G(0,1) | G(1,0) G(1,1) R(0) | G(2,0) G(2,1) R(1) | ... | R(last)  so that the gate epilogues of
// tile n (which R(n) depends on) overlap the gate GEMMs of tile n+1.  TMEM holds two 256-column accumulators that
// alternate op by op.  R(n) reads the z rows the same CTA has just written: they go to global memory anyway (the skip sum
// of the step is one K = L*C GEMM over that matrix) and come back through L2 by TMA; the epilogue warps order their stores
// before the async-proxy reads with fence.proxy.async + an mbarrier the TMA producer waits on.
//
// Contraction (fp16x2 mode, tests/tools/precision_study.py): activations are ONE fp16 operand; the weights are fp16(W 2^p) plus a
// correction.  In the gate GEMM (3/4 of the FLOPs) the correction term runs on the fp8 pipe at twice the rate:
//     acc += fp16(A) * fp16(W_hi)  [kind::f16, K = 16]   +   e4m3(A) * e5m2(W 2^p - W_hi)  [kind::f8f6f4, K = 32]
// into the same fp32 accumulator (hardware-checked: csrc/experiments.cu bsg_experiment_f8).  The correction only has to be
// good to a few bits: what it removes is the SYSTEMATIC fp16 weight-rounding error that would add up over the 100 steps.
// The residual GEMM keeps two fp16 MMAs per product (its z operand has no 8-bit copy).
//
// Epilogue: the streams the epilogue consumes (conditioner projection cp in fp32; the fp16 conv input, which doubles as the
// residual stream) move by TMA through a ring of [128 rows x 16 columns] shared-memory boxes (SWIZZLE_64B) fed by a second producer warp,
// and every epilogue thread works on ONE accumulator row exactly as tcgen05.ld delivers it -- no shared-memory transposes,
// no global loads in the epilogue warps, 32-byte (full-sector) row stores for the 16-/8-bit outputs.  The register/LSU
// epilogue of conv_gemm.cuh needed 15-20k cycles per op here and paced the kernel (profiles/r01_g, r01_h).
//
// Warps: 0 = operand producer (TMA), 1 = MMA issuer (leader CTA), 2..9 = epilogue (TMEM lane quadrant = warp % 4, two
// column groups), 10 = epilogue-operand producer (TMA loads of the cp / conv-input boxes).
//
// Slabs: the rows of an item are cut into ceil(T / 128) slabs of 128 rows, numbered across the batch (g = b * slabs_per_item + s).
// Pair tile u runs slabs 2u and 2u + 1, one per CTA: each CTA stages its own A rows with its own TMA loads, so the two halves
// of an M = 256 MMA may belong to two items: an item's last pair tile leaves at most 127 rows idle, not 255 (T = 1875: 15 slabs
// per item, 240 pair tiles at B = 32 instead of 256 item-aligned 256-row tiles).  Only the last pair tile of an odd slab count
// has an empty half.  A CTA's 128 rows never span two items.
//
// Layers: slab g of layer l reads halo rows of slabs g-1, g, g+1 (of the same item) of layer l-1 (dilation <= 128); completion
// counters in global memory (wait_inputs below) order that, the conv input ping-pongs between two buffers, and the deal of
// pair tiles to CTA pairs rotates per layer so that the uneven split (240 pair tiles over 74 pairs) averages out.
#pragma once
#include "conv_gemm.cuh"

namespace b200 {

// per-layer parameters, in global memory (tensor maps must be 64-byte aligned)
struct alignas(128) LayerParams {
    CUtensorMap wg16;      // dilated-conv weights fp16(W 2^p) [2C (gate/filter permuted)][3C], box = 64 x 128 (64 with multicast)
    CUtensorMap wg8;       // e5m2 correction of the same, box = 128 x 128 (64)
    CUtensorMap wr[2];     // residual half of the output projection fp16 hi / lo [C][C], box = 64 x 128 (64)
    CUtensorMap cp;        // conditioner projection + biases f32 [B][T][2C] (packed column order), box = 16 x 128, SWIZZLE_64B
    const float* bias_r;   // [C] residual bias
    float gscale, rscale;  // 2^-p of the gate / residual weight packing
    int dilation;
    int pad_;
};

struct LayerArgs {
    CUtensorMap xa16[2];   // conv input fp16 [B][T][C], box = 64 channels x a_rows rows; layer l reads [l & 1] and writes the other
    CUtensorMap xa8[2];    // conv input e4m3 [B][T][C], box = 128 channels x a_rows rows
    CUtensorMap xe[2];     // the fp16 conv input once more, as the epilogue reads it: box = 32 channels x 128 rows, SWIZZLE_64B
    CUtensorMap z;         // all-layer gated activations fp16 [B][T][L*C], box = 64 x 128
    const LayerParams* tab;   // [total layers]
    int layer0, n_layers;  // layers [layer0, layer0 + n_layers) run in this launch; total_layers: the last one writes no conv input
    int total_layers;
    int B, T;
    int slabs_per_item;    // ceil(T / 128): slab g = b * slabs_per_item + s holds rows [128 s, 128 s + 128) of item b
    int n_slabs;           // B * slabs_per_item; pair tile u runs slabs 2u (leader CTA) and 2u + 1
    int a_rows;            // rows of the xa halo boxes (128 + 2 * max dilation, multiple of 8)
    int z_pitch;           // elements per row of the z matrix (layer l owns columns [l*C, (l+1)*C))
    __half* z_out;         // z matrix base
    uint8_t* z8_out;       // e4m3 copy of z (same shape): A operand of the skip-sum GEMM's fp8 correction term; may be null
    __half* xa16_out[2];   // conv input buffers as plain pointers (layer l writes [(l + 1) & 1])
    uint8_t* xa8_out[2];
    const float* lut_t;    // [total layers][C] step embeddings d_l of this diffusion step
    int* flags;            // n_layers > 1: [total layers][n_slabs] completion counters: every launch adds 8 (epilogue warps per CTA)
                           //    to each; they are zeroed ONCE per sampling call, not per launch
    int epoch;             // 1-based count of launches since the counters were zeroed: a slab is complete at 8 * epoch
    int flags_ablate;      // timing ablations (bit 1: no fp8 MMAs, bit 2: no fp16 MMAs)
    unsigned long long* trace;
    const int* t_of_b;     // diffnet_layer_kernel<MC, true>: device int32 [B] diffusion step of each batch item; lut_t is then the
                           //    embedding table of ALL steps [k_step][total layers][C] (kept last: the members above do not move)
};

// op j of a CTA pair that owns cnt pair tiles (3 * cnt ops): kind 0 = gate GEMM of channel half h, 1 = residual GEMM, of local pair tile n
struct LayerOp {
    int kind, n, h;
};
__device__ __forceinline__ LayerOp layer_op(int j, int cnt) {
    if (j < 2) return LayerOp{0, 0, j};
    const int q = (j - 2) / 3, r = (j - 2) % 3;
#ifdef B200_ORDER_GRG
    if (q == cnt - 1 || r == 1) return LayerOp{1, q, 0};
    return LayerOp{0, q + 1, r == 0 ? 0 : 1};
#else
    // G(q+1,0) G(q+1,1) R(q): the residual GEMM of a tile comes TWO gate GEMMs after the gate epilogue it depends on, so the
    // operand producer never waits for z (with G R G it stalled ~10k cycles per row tile and starved the MMA issuer)
    if (q == cnt - 1 || r == 2) return LayerOp{1, q, 0};
    return LayerOp{0, q + 1, r};
#endif
}

#ifndef B200_GATE_MATH
#define B200_GATE_MATH 2
#endif
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// sigmoid(g) * tanh(f)   (net.py:73-74)
__device__ __forceinline__ float gate_act(float g, float f) {
#if B200_GATE_MATH == 2
    // two MUFU ops: sigmoid(g) = 0.5 * tanh(g / 2) + 0.5 ; tanh.approx.f32 has a relative error of 2^-11, the size of the
    // fp16 rounding z gets anyway
    return fmaf(0.5f, tanh_approx(0.5f * g), 0.5f) * tanh_approx(f);
#elif B200_GATE_MATH == 1
    // three MUFU ops: a = e^-g, b = e^-2f, z = (1 - b) / ((1 + a)(1 + b)); arguments clamped so that nothing becomes inf/inf
    const float a = __expf(-fmaxf(g, -80.0f));
    const float b = __expf(-2.0f * fmaxf(f, -40.0f));
    return __fdividef(1.0f - b, (1.0f + a) * (1.0f + b));
#else
    return fast_sigmoid(g) * fast_tanh(f);
#endif
}

// Two gated activations at once in half2 arithmetic: t = tanh.approx.f16x2 (one MUFU op for two values),
// z = (0.5 t(g/2) + 0.5) * t(f).  gh = g / 2 (already halved), f: fp32 pre-activations.  The result is the fp16 pair that is
// stored; its error (fp16 rounding of the tanh arguments and results, ~2^-10 relative) is of the size of the fp16 rounding
// z gets in any case, and like it changes pseudo-randomly from step to step (no systematic part).
__device__ __forceinline__ uint32_t gate_act_h2(float gh0, float gh1, float f0, float f1) {
    const __half2 g = __floats2half2_rn(gh0, gh1), f = __floats2half2_rn(f0, f1);
    uint32_t tg, tf;
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(tg) : "r"(*reinterpret_cast<const uint32_t*>(&g)));
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(tf) : "r"(*reinterpret_cast<const uint32_t*>(&f)));
    const __half2 half = __float2half2_rn(0.5f);
    const __half2 sg = __hfma2(*reinterpret_cast<const __half2*>(&tg), half, half);
    const __half2 z = __hmul2(sg, *reinterpret_cast<const __half2*>(&tf));
    return *reinterpret_cast<const uint32_t*>(&z);
}

// ---------------------------------------------------------------------------------------------
// shared-memory plan
// ---------------------------------------------------------------------------------------------
struct LayerSmem {
    static constexpr int kASlotBytes = 144 * 128;              // halo tile: 144 rows x 128 B (64 fp16 or 128 e4m3 channels)
    static constexpr int kAStages = 3;
    static constexpr int kWSlotBytes = 128 * 128;              // weight tile: 128 N rows x 128 B
#ifndef B200_WSTAGES
#define B200_WSTAGES 6
#endif
    static constexpr int kWStages = B200_WSTAGES;
    static constexpr int kEBoxBytes = 128 * 16 * 4;            // epilogue box: 128 rows x 16 fp32
#ifndef B200_ESTAGES
#define B200_ESTAGES 9
#endif
    static constexpr int kEStages = B200_ESTAGES;
    static constexpr int kVecBytes = 2 * 256 * 4;              // residual bias + next step embedding
    static constexpr int kBarBytes = 512;
    static constexpr int kOffW = kAStages * kASlotBytes;
    static constexpr int kOffE = kOffW + kWStages * kWSlotBytes;
    static constexpr int kOffVec = kOffE + kEStages * kEBoxBytes;
    static constexpr int kOffBar = kOffVec + kVecBytes;
    static constexpr int kTotal = kOffBar + kBarBytes + 1024;  // + manual 1024-byte alignment
    static_assert(kTotal <= 227 * 1024, "shared memory budget");
    static_assert((2 * kAStages + 2 * kWStages + 2 * kEStages + 6) * 8 + 8 <= kBarBytes, "barrier area too small");
    static_assert(kOffW % 1024 == 0 && kOffE % 1024 == 0, "swizzled tiles need 1024-byte alignment");
};
constexpr int kLayerThreads = 32 * 11;
constexpr int kGateBoxes = 16, kResBoxes = 8;

// byte offset of 16-byte chunk k (4 fp32 columns) of row r in a SWIZZLE_64B box
__device__ __forceinline__ uint32_t ebox_off(int r, int k) { return static_cast<uint32_t>(r * 64 + ((k ^ ((r >> 1) & 3)) << 4)); }

__device__ __forceinline__ float4 lds128(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
    const __half2 h = __floats2half2_rn(fminf(fmaxf(a, -65504.0f), 65504.0f), fminf(fmaxf(b, -65504.0f), 65504.0f));
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_half2_nc(float a, float b) {   // values known to be far inside the fp16 range
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_half2_sat(float lo, float hi) {   // one instruction, out-of-range -> +-65504
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
// sigmoid(2 gh) * tanh(f) with two MUFU ops: sigmoid(g) = 0.5 tanh(g / 2) + 0.5; tanh.approx.f32 has a relative error of 2^-11,
// the size of the fp16 rounding z gets anyway (measured: 2.0e-3 max mel error after 100 steps against 1.3e-3 with exp/rcp)
__device__ __forceinline__ float gate_half(float gh, float f) { return fmaf(0.5f, tanh_approx(gh), 0.5f) * tanh_approx(f); }
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
    const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
    const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
    return lo | (hi << 16);
}
__device__ __forceinline__ void tma_load_3d_local(uint32_t smem_dst, const void* desc, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_dst), "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_store_3d(const void* desc, uint32_t smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(desc), "r"(smem_src), "r"(c0), "r"(c1),
                 "r"(c2)
                 : "memory");
}

// MC = 1: clusters of FOUR CTAs = two pairs working on two consecutive pair tiles with the same weights; every weight tile is
// read from L2 once per cluster (each CTA loads a quarter of the N rows and multicasts it to the CTA of the same rank in
// the other pair).  At ~1.3 MB of L2->SM traffic per pair tile and CTA, more than half of it weights, the 2-CTA kernel runs
// into the L2->SM throughput limit (profiles/r01_h); only 33 such clusters fit on a B200, but 120 units over 33 clusters
// are the same 4 rounds as 240 pair tiles over 74 pairs.
// STEPS = true: a diffusion step per batch item (args.t_of_b).  A CTA's slab never spans two batch items, so the residual epilogue
// of each CTA reads d_l and d_{l+1} of its slab's step from the embedding table through L1 instead of the per-layer shared-memory
// staging (the two CTAs of a pair tile may be at different steps).
template <int MC, bool STEPS = false>
__global__ void __launch_bounds__(kLayerThreads, 1) diffnet_layer_kernel(const __grid_constant__ LayerArgs args) {
    using S = LayerSmem;
    constexpr int C = 256;
    constexpr uint32_t kIdesc16 = umma_idesc_f16(2 * kTileM, 256, /*fp16=*/true);
    constexpr uint32_t kIdesc8 = umma_idesc_f8(2 * kTileM, 256, /*A e4m3*/ 0, /*B e5m2*/ 1);

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    const uint32_t smem_a = smem_u32(smem);
    const uint32_t smem_w = smem_a + S::kOffW;
    const uint32_t smem_e = smem_a + S::kOffE;
    float* vec = reinterpret_cast<float*>(smem + S::kOffVec);        // [0,256) residual bias - this layer's step embedding, [256,512) next step embedding
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kOffBar);
    uint64_t* afull_bar = bars;
    uint64_t* aempty_bar = afull_bar + S::kAStages;
    uint64_t* wfull_bar = aempty_bar + S::kAStages;
    uint64_t* wempty_bar = wfull_bar + S::kWStages;
    uint64_t* efull_bar = wempty_bar + S::kWStages;
    uint64_t* edone_bar = efull_bar + S::kEStages;
    uint64_t* tfull_bar = edone_bar + S::kEStages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* zfull_bar = tempty_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(zfull_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int crank = static_cast<int>(cluster_ctarank());
    const int rank = crank & 1;                      // rank in the CTA pair (0 = leader: issues the MMAs)
    const int pidx = MC ? (crank >> 1) : 0;          // which pair of the cluster
    const uint16_t pair_mask = static_cast<uint16_t>(3u << (2 * pidx));
    constexpr int kClusterCtas = MC ? 4 : 2;
    constexpr int kPairs = MC ? 2 : 1;
    const int cluster_id = static_cast<int>(blockIdx.x) / kClusterCtas;
    const int n_clusters = static_cast<int>(gridDim.x) / kClusterCtas;
    // local pair tile n of this pair is global pair tile kPairs * (cluster_id + n * n_clusters) + pidx.  A slab past the last one
    // (odd slab count; with MC also a missing pair tile of the last unit) gets batch index B: its loads are zero-filled by the TMA
    // unit and nothing is stored or counted
    const int n_pair_tiles = (args.n_slabs + 1) / 2;
    const int n_units = (n_pair_tiles + kPairs - 1) / kPairs;
    const int n_workers = kPairs * n_clusters;       // pair-tile stride
    // The units are dealt round-robin to the clusters, so n_units % n_clusters of them own one unit more than the rest (240 pair
    // tiles over 74 pairs: 18 pairs with 4, 56 with 3).  In a multi-layer launch the deal rotates from layer to layer, so that
    // over the layers every cluster gets the same share instead of the same clusters finishing last in every layer.
    const int rot = args.n_layers > 1 ? n_units % n_clusters : 0;
    auto layer_cluster = [&](int l) { return (cluster_id + (l - args.layer0) * rot) % n_clusters; };
    auto layer_cnt = [&](int l) { return (n_units - layer_cluster(l) + n_clusters - 1) / n_clusters; };       // pair tiles of this pair in layer l
    auto layer_worker = [&](int l) { return kPairs * layer_cluster(l) + pidx; };                              // ... the first of them
    // this CTA's slab of pair tile m: its index g, batch item b (B if the slab does not exist) and first row t0 in the item
    struct Slab { int g, b, t0; };
    auto slab_of = [&](int m) {
        const int g = 2 * m + rank;
        if (g >= args.n_slabs) return Slab{g, args.B, 0};
        return Slab{g, g / args.slabs_per_item, (g % args.slabs_per_item) * kTileM};
    };

    if (threadIdx.x == 32) {
        for (int s = 0; s < S::kAStages; ++s) { mbar_init(&afull_bar[s], 1); mbar_init(&aempty_bar[s], 1); }
        for (int s = 0; s < S::kWStages; ++s) { mbar_init(&wfull_bar[s], 1); mbar_init(&wempty_bar[s], MC ? 2 : 1); }
        for (int s = 0; s < S::kEStages; ++s) { mbar_init(&efull_bar[s], 1); mbar_init(&edone_bar[s], 4); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 2 * kEpiWarps); }
        // z rows of local row tile n published: both gate epilogues, every epilogue warp of THIS CTA.  Two barriers (n & 1):
        // a fast warp may publish tile n+1 before a slow one has published tile n, never tile n+2 (the accumulator hand-over
        // keeps the warps within two ops of each other)
        for (int a = 0; a < 2; ++a) mbar_init(&zfull_bar[a], 2 * kEpiWarps);
        fence_barrier_init();
    }
    if (warp == 0) { tmem_alloc_pair(tmem_slot, 512); tmem_relinquish_pair(); }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const bool tr_on = args.trace != nullptr;
    const int layer_end = args.layer0 + args.n_layers;
    // Several layers in one launch: slab g of layer l reads conv-input rows that the slabs g-1, g, g+1 (of the same batch item)
    // of layer l-1 wrote IN THIS LAUNCH, possibly on other SMs.  Each of the 8 epilogue warps of the CTA that ran a slab fences
    // its stores and bumps flags[l-1][slab]; a TMA-issuing thread of the reading CTA polls (acquire) and orders the generic-proxy
    // writes before its async-proxy reads.  Pairs therefore run ahead into the next layer wherever their inputs are ready: the
    // partial last round of a layer (240 pair tiles over 74 pairs) overlaps the next layer instead of idling.
    auto wait_inputs = [&](int l, const Slab& sl, long long& acc_wait) {
        if (args.flags == nullptr || l == args.layer0 || sl.b >= args.B) return;
        const long long t0w = tr_on ? clock64() : 0;
        const int g = sl.g, s = sl.t0 / kTileM;
        const int lo = s > 0 ? g - 1 : g, hi = (s + 1 < args.slabs_per_item) ? g + 1 : g;
        const int* f = args.flags + static_cast<size_t>(l - 1) * args.n_slabs;
        const int done = kEpiWarps * args.epoch;   // counters run on from launch to launch (no memset node between the kernels of a step)
        for (int mm = lo; mm <= hi; ++mm) {
            int v;
            unsigned spins = 0;
            long long t_start = 0;
            do {
                asm volatile("ld.acquire.gpu.global.b32 %0, [%1];" : "=r"(v) : "l"(f + mm) : "memory");
                if (v < done && (++spins & 15) == 0) {
                    __nanosleep(64);
                    // bounded: the dataflow needs every CTA of the grid resident (one per SM, sized from the device's SM count);
                    // if something else pins SMs for seconds, fail loudly instead of hanging the device
                    const long long now = clock64();
                    if (t_start == 0) t_start = now;
                    if (now - t_start > 8000000000LL) {
                        printf("diffnet_layer_kernel: block %d waited > 4 s for slab %d of layer %d\n", blockIdx.x, mm, l - 1);
                        __trap();
                    }
                }
            } while (v < done);
        }
        asm volatile("fence.proxy.async.global;" ::: "memory");
        if (tr_on) acc_wait += clock64() - t0w;
    };

    if (warp == 0 && lane == 0) {
        // ================= operand producer (one per CTA) =================
        int as = 0, ws = 0;
        uint32_t aph = 0, wph = 0;
        long long w_a = 0, w_b = 0, w_z = 0;
        const long long t_begin = tr_on ? clock64() : 0;
        auto load_a = [&](const CUtensorMap* map, uint32_t bytes, int c0, int row, int b) {
            mbar_wait_tr(&aempty_bar[as], aph ^ 1, tr_on, w_a);
            if (rank == 0) mbar_arrive_expect_tx(&afull_bar[as], bytes * 2);
            tma_load_3d_pair(reinterpret_cast<void*>(smem + as * S::kASlotBytes), map, &afull_bar[as], c0, row, b);
            if (++as == S::kAStages) { as = 0; aph ^= 1; }
        };
        auto load_w = [&](const CUtensorMap* map, int c0, int row) {   // row: first of this CTA's 128 weight rows
            mbar_wait_tr(&wempty_bar[ws], wph ^ 1, tr_on, w_b);
            if (rank == 0) mbar_arrive_expect_tx(&wfull_bar[ws], S::kWSlotBytes * 2);
            uint8_t* dst = smem + S::kOffW + ws * S::kWSlotBytes;
            if (MC)   // this CTA's half of those rows, into the same slot of the same-rank CTA of both pairs
                tma_load_2d_pair_mc(dst + pidx * (S::kWSlotBytes / 2), map, &wfull_bar[ws], c0, row + pidx * 64, static_cast<uint16_t>(5u << rank));
            else
                tma_load_2d_pair(dst, map, &wfull_bar[ws], c0, row);
            if (++ws == S::kWStages) { ws = 0; wph ^= 1; }
        };
        const uint32_t halo_bytes = static_cast<uint32_t>(args.a_rows) * 128;
        long long w_dep = 0;
        int ng0 = 0;   // local row tiles finished in earlier layers (z barrier parity runs on across layers)
        for (int l = args.layer0, cnt = 0; l < layer_end; ++l, ng0 += cnt) {
            const LayerParams& lp = args.tab[l];
            const int dil = lp.dilation;
            cnt = layer_cnt(l);
            const int worker = layer_worker(l), n_ops = 3 * cnt;
            for (int j = 0; j < n_ops; ++j) {
                const LayerOp op = layer_op(j, cnt);
                const Slab sl = slab_of(worker + op.n * n_workers);
                const int b = sl.b, t0 = sl.t0;
                if (op.kind == 0) {
                    if (op.h == 0) wait_inputs(l, sl, w_dep);
                    const int wrow = op.h * 256 + rank * 128;
                    for (int k8 = 0; k8 < 2; ++k8) {
                        for (int kk = 0; kk < 2; ++kk) {
                            const int kb = 2 * k8 + kk;
                            load_a(&args.xa16[l & 1], halo_bytes, kb * 64, t0 - dil, b);
                            for (int tp = 0; tp < 3; ++tp) load_w(&lp.wg16, tp * C + kb * 64, wrow);
                        }
                        load_a(&args.xa8[l & 1], halo_bytes, k8 * 128, t0 - dil, b);
                        for (int tp = 0; tp < 3; ++tp) load_w(&lp.wg8, tp * C + k8 * 128, wrow);
                    }
                } else {
                    const int ng = ng0 + op.n;
                    mbar_wait_tr(&zfull_bar[ng & 1], static_cast<uint32_t>((ng >> 1) & 1), tr_on, w_z);   // this CTA's z rows of the tile are in global memory
                    asm volatile("fence.proxy.async.global;" ::: "memory");   // reader side of the same hand-over
                    for (int kb = 0; kb < 4; ++kb) {
                        load_a(&args.z, kTileM * 128, l * C + kb * 64, t0, b);
                        load_w(&lp.wr[0], kb * 64, rank * 128);
                        load_w(&lp.wr[1], kb * 64, rank * 128);
                    }
                }
            }
        }
        if (tr_on) args.trace[blockIdx.x * 16 + 15] = w_dep;
        if (tr_on) {
            unsigned long long* t = args.trace + blockIdx.x * 16;
            t[4] = clock64() - t_begin; t[5] = w_a; t[6] = w_b; t[9] = w_z;
        }
    } else if (warp == 1 && lane == 0 && rank == 0) {
        // ================= MMA issuer (leader CTA) =================
        int as = 0, ws = 0;
        uint32_t aph = 0, wph = 0;
        long long w_t = 0, w_a = 0, w_b = 0;
        const long long t_begin = tr_on ? clock64() : 0;
        uint32_t accumulate = 0;
        uint32_t tacc = 0;
        // four MMAs of one weight slot against the A tile at a_op (16-bit: K = 16 each, 8-bit: K = 32 each; both advance 32 bytes)
        auto mma_slot = [&](uint32_t a_op, bool eight) {
            mbar_wait_tr(&wfull_bar[ws], wph, tr_on, w_b);
            tc_fence_after();
            const uint32_t b_op = smem_w + ws * S::kWSlotBytes;
            const bool skip = (eight && (args.flags_ablate & 2)) || (!eight && (args.flags_ablate & 4));   // timing ablations (wrong results)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint64_t da = umma_smem_desc<128>(a_op + k * 32), db = umma_smem_desc<128>(b_op + k * 32);
                if (skip && accumulate) continue;
                if (eight) umma_f8_pair(tacc, da, db, kIdesc8, accumulate);
                else umma_f16_pair(tacc, da, db, kIdesc16, accumulate);
                accumulate = 1;
            }
            umma_commit_pair(&wempty_bar[ws], MC ? static_cast<uint16_t>(0xF) : pair_mask);   // MC: one of two arrivals in all four CTAs
            if (++ws == S::kWStages) { ws = 0; wph ^= 1; }
        };
        auto wait_a = [&]() {
            mbar_wait_tr(&afull_bar[as], aph, tr_on, w_a);
            tc_fence_after();
            return smem_a + as * S::kASlotBytes;
        };
        auto free_a = [&]() {
            umma_commit_pair(&aempty_bar[as], pair_mask);
            if (++as == S::kAStages) { as = 0; aph ^= 1; }
        };
        int jg = 0;   // ops issued so far: accumulator buffer = jg & 1, across layers
        int cnt_total = 0;
        for (int l = args.layer0; l < layer_end; ++l) {
            const uint32_t tap_stride = static_cast<uint32_t>(args.tab[l].dilation) * 128;   // taps = rows 0, d, 2d of the halo tile
            const int cnt = layer_cnt(l), n_ops = 3 * cnt;
            cnt_total += cnt;
            for (int j = 0; j < n_ops; ++j, ++jg) {
                const int kind = layer_op(j, cnt).kind;
                const int acc = jg & 1;
                mbar_wait_tr(&tempty_bar[acc], ((jg >> 1) & 1) ^ 1, tr_on, w_t);
                tc_fence_after();
                tacc = tmem_base + acc * 256;
                accumulate = 0;
                if (kind == 0) {
                    for (int k8 = 0; k8 < 2; ++k8) {
                        for (int kk = 0; kk < 2; ++kk) {
                            const uint32_t a_slot = wait_a();
                            for (int tp = 0; tp < 3; ++tp) mma_slot(a_slot + tp * tap_stride, false);
                            free_a();
                        }
                        const uint32_t a_slot = wait_a();
                        for (int tp = 0; tp < 3; ++tp) mma_slot(a_slot + tp * tap_stride, true);
                        free_a();
                    }
                } else {
                    for (int kb = 0; kb < 4; ++kb) {
                        const uint32_t a_slot = wait_a();
                        mma_slot(a_slot, false);
                        mma_slot(a_slot, false);
                        free_a();
                    }
                }
                umma_commit_pair(&tfull_bar[acc], pair_mask);
            }
        }
        if (tr_on) {
            unsigned long long* t = args.trace + blockIdx.x * 16;
            t[0] = clock64() - t_begin; t[1] = w_t; t[2] = w_a; t[3] = w_b; t[10] = cnt_total;
        }
    } else if (warp == 10 && lane == 0) {
        // ================= epilogue-operand producer: cp boxes (gate ops) / conv-input boxes (residual ops) =================
        // gate op, 16 boxes of 16 fp32 columns of cp: box i -> chunk c = i / 4, column group g = (i / 2) % 2, i % 2 = gate / filter
        // columns.  residual op, 8 boxes of 32 fp16 channels of the conv input: box i -> chunk c = i / 2, group g = i % 2.
        long long w_e = 0, w_dep = 0;
        int q = 0;
        for (int l = args.layer0; l < layer_end; ++l) {
            const LayerParams& lp = args.tab[l];
            const int cnt = layer_cnt(l), worker = layer_worker(l), n_ops = 3 * cnt;
            for (int j = 0; j < n_ops; ++j) {
                const LayerOp op = layer_op(j, cnt);
                const Slab sl = slab_of(worker + op.n * n_workers);
                const int b = sl.b, row = sl.t0;
                const int nb = op.kind == 0 ? kGateBoxes : kResBoxes;
                if (op.kind == 1) wait_inputs(l, sl, w_dep);   // the boxes of a residual op are rows of this layer's conv input
                for (int i = 0; i < nb; ++i, ++q) {
                    const int s = q % S::kEStages;
                    if (q >= S::kEStages) mbar_wait_tr(&edone_bar[s], ((q / S::kEStages) - 1) & 1, tr_on, w_e);   // previous occupant consumed by its four warps
                    const int col = op.kind == 0 ? op.h * 256 + ((i >> 1) & 1) * 64 + (i >> 2) * 16 + (i & 1) * 128 : (i & 1) * 128 + (i >> 1) * 32;
                    mbar_arrive_expect_tx(&efull_bar[s], S::kEBoxBytes);
                    tma_load_3d_local(smem_e + s * S::kEBoxBytes, op.kind == 0 ? &lp.cp : &args.xe[l & 1], &efull_bar[s], col, row, b);
                }
            }
        }
        if (tr_on) args.trace[blockIdx.x * 16 + 13] = w_e;
    } else if (warp >= 2 && warp < 2 + kEpiWarps) {
        // ================= epilogue warps: thread = one accumulator row =================
        const int quad = warp & 3;
        const int grp = (warp - 2) >> 2;
        const int r_box = quad * 32 + lane;                 // row of this thread in the CTA's 128-row boxes
        const uint32_t tempty_remote0 = map_to_cta(smem_u32(&tempty_bar[0]), static_cast<uint32_t>(crank & ~1));
        const bool tr = tr_on && warp == 2 && lane == 0;
        long long w_f = 0, w_e = 0, t_gate = 0, t_res = 0;
        const long long t_begin = tr ? clock64() : 0;
        const float rs2 = 0.70710678118654752440f;
        const uint32_t vec_s = smem_u32(vec);
        uint32_t xo[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) xo[k] = ebox_off(r_box, k);

        int q_base = 0;           // first box of the current op in this CTA's box sequence
        bool z_pending = false;   // z rows stored by the previous gate op, not yet fenced / signalled
        int z_tile = 0;           // ... and the local row tile they belong to
        auto publish_z = [&]() {
            // the z rows are read back by this CTA's TMA loads of R(n).  The TMA unit reads L2, not this SM's store path: the
            // stores must be PERFORMED at device scope (fence.acq_rel.gpu waits for their acknowledgements) before they are
            // ordered against the async proxy and the producer is signalled -- an mbarrier arrive is a CTA-scope release and by
            // itself let a load overtake a store still on its way to L2 (profiles/r02_c: a stale z tile, i.e. the previous
            // diffusion step's values, in about one of three FIRST samplings on a new workspace inside the GPU test suite).  Deferred to the start of the next
            // op (the stores have drained by then and the fences return at once) unless that op is the residual GEMM that needs them.
            __threadfence();
            asm volatile("fence.proxy.async.global;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&zfull_bar[z_tile & 1]);
            z_pending = false;
        };
        int jg = 0, ng0 = 0;      // ops / local row tiles of earlier layers (accumulator and z-barrier parities run on across layers)
        for (int l = args.layer0, cnt = 0; l < layer_end; ++l, ng0 += cnt) {
          const LayerParams& lpar = args.tab[l];
          cnt = layer_cnt(l);
          const int worker = layer_worker(l), n_ops = 3 * cnt;
          const float gscale = lpar.gscale, rscale = lpar.rscale;
          const bool has_next = l + 1 < args.total_layers;
          __half* const xa16_out = args.xa16_out[(l + 1) & 1];
          uint8_t* const xa8_out = args.xa8_out[(l + 1) & 1];
          {   // per-column vectors of this layer's residual epilogue: vec[0,256) = residual bias - d_l (the residual stream is
              // fp16(x + d_l)), vec[256,512) = d_{l+1}.  All epilogue warps are past the previous layer's last use.
              asm volatile("bar.sync 1, 256;" ::: "memory");
              const int c = threadIdx.x - 64;
              if constexpr (STEPS) {   // the step embeddings are per batch item: subtracted / added per op below
                  vec[c] = lpar.bias_r[c];
              } else {
                  vec[c] = lpar.bias_r[c] - args.lut_t[static_cast<size_t>(l) * C + c];
                  vec[256 + c] = has_next ? args.lut_t[static_cast<size_t>(l + 1) * C + c] : 0.0f;
              }
              asm volatile("bar.sync 1, 256;" ::: "memory");
          }
          for (int j = 0; j < n_ops; ++j, ++jg) {
            const LayerOp op = layer_op(j, cnt);
            const int acc = jg & 1;
            const Slab sl = slab_of(worker + op.n * n_workers);
            const int b = sl.b;
            const int t = sl.t0 + r_box;   // this thread's row in the batch item
            const bool row_ok = t < args.T && b < args.B;
            const long long row = static_cast<long long>(b) * args.T + t;
            mbar_wait_tr(&tfull_bar[acc], (jg >> 1) & 1, tr, w_f);
            tc_fence_after();
            const long long t_op = tr ? clock64() : 0;
            const uint32_t tacc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * 256;
            const int q_op = q_base;
            q_base += op.kind == 0 ? kGateBoxes : kResBoxes;
            if (op.kind == 0) {
                // ---- gate: z = sigmoid(acc_g + cp_g) * tanh(acc_f + cp_f)   (net.py:71-74)
                // (loops kept rolled: with the four roles' code paths resident the unrolled epilogue stalled on instruction fetch)
                const float hs = 0.5f * gscale;
                __half* zrow = args.z_out + row * args.z_pitch + l * C + op.h * 128;
                uint8_t* z8row = args.z8_out ? args.z8_out + row * args.z_pitch + l * C + op.h * 128 : nullptr;
                // one 16-channel chunk; vg / vf: its gate / filter accumulator columns (already waited for)
                auto gate_chunk = [&](int c, const uint32_t (&vg)[16], const uint32_t (&vf)[16]) {
                    const int cg = grp * 64 + c * 16;          // gate columns [cg, cg+16), filter columns +128
                    const int q = q_op + 4 * c + 2 * grp;      // boxes q (cp of the gate columns), q + 1 (filter columns)
                    const int sg = q % S::kEStages, sf = (q + 1) % S::kEStages;
                    mbar_wait_tr(&efull_bar[sg], (q / S::kEStages) & 1, tr, w_e);
                    mbar_wait_tr(&efull_bar[sf], ((q + 1) / S::kEStages) & 1, tr, w_e);
                    float4 pg[4], pf[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        pg[k] = lds128(smem_e + sg * S::kEBoxBytes + xo[k]);
                        pf[k] = lds128(smem_e + sf * S::kEBoxBytes + xo[k]);
                    }
                    uint32_t zz[8], z8[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        // sigmoid(g) = 0.5 tanh(g/2) + 0.5: the gate pre-activations are formed already halved
                        const float g0 = fmaf(__uint_as_float(vg[4 * k]), hs, 0.5f * pg[k].x), g1 = fmaf(__uint_as_float(vg[4 * k + 1]), hs, 0.5f * pg[k].y);
                        const float g2 = fmaf(__uint_as_float(vg[4 * k + 2]), hs, 0.5f * pg[k].z), g3 = fmaf(__uint_as_float(vg[4 * k + 3]), hs, 0.5f * pg[k].w);
                        const float f0 = fmaf(__uint_as_float(vf[4 * k]), gscale, pf[k].x), f1 = fmaf(__uint_as_float(vf[4 * k + 1]), gscale, pf[k].y);
                        const float f2 = fmaf(__uint_as_float(vf[4 * k + 2]), gscale, pf[k].z), f3 = fmaf(__uint_as_float(vf[4 * k + 3]), gscale, pf[k].w);
                        const float z0 = gate_half(g0, f0), z1 = gate_half(g1, f1), z2 = gate_half(g2, f2), z3 = gate_half(g3, f3);
                        zz[2 * k] = pack_half2_nc(z0, z1);
                        zz[2 * k + 1] = pack_half2_nc(z2, z3);
                        z8[k] = pack_e4m3x4(z0, z1, z2, z3);
                    }
                    // hand the boxes back only now: the arithmetic above could not issue before the ld.shared data had arrived.
                    // (Signalling right behind the ld.shared instructions let the TMA refill overtake loads still queued
                    // behind this warp's stores -- a rare 32-row corruption.)
                    __syncwarp();
                    if (lane == 0) { mbar_arrive_relaxed(&edone_bar[sg]); mbar_arrive_relaxed(&edone_bar[sf]); }
                    if (row_ok) {
                        stg256(zrow + cg, zz);
                        if (z8row != nullptr) *reinterpret_cast<uint4*>(z8row + cg) = make_uint4(z8[0], z8[1], z8[2], z8[3]);
                    }
                };
                // the accumulator columns of chunk c+1 are read from TMEM while chunk c is processed (under MMA load a
                // tcgen05.ld round trip is ~1k cycles and was 40 % of this loop: profiles/r01_h)
                uint32_t ag[16], af[16], bg[16], bf[16];
                __syncwarp();
                tmem_ld16(tacc + grp * 64, ag);
                tmem_ld16(tacc + 128 + grp * 64, af);
#pragma unroll 1
                for (int c = 0; c < 4; c += 2) {
                    tmem_ld_wait16x2(ag, af);
                    __syncwarp();
                    tmem_ld16(tacc + grp * 64 + (c + 1) * 16, bg);
                    tmem_ld16(tacc + 128 + grp * 64 + (c + 1) * 16, bf);
                    if (c == 2 && z_pending) publish_z();   // the previous gate op's z rows (their stores have long drained)
                    gate_chunk(c, ag, af);
                    tmem_ld_wait16x2(bg, bf);
                    if (c + 2 < 4) {
                        __syncwarp();
                        tmem_ld16(tacc + grp * 64 + (c + 2) * 16, ag);
                        tmem_ld16(tacc + 128 + grp * 64 + (c + 2) * 16, af);
                    }
                    gate_chunk(c + 1, bg, bf);
                }
                z_pending = true;
                z_tile = ng0 + op.n;
#ifdef B200_PUBLISH_NOW
                publish_z();
#endif
                // R(n) directly follows the second gate op of the last row tile: it cannot wait for a deferred signal
                if (j + 1 < n_ops && layer_op(j + 1, cnt).kind == 1 && layer_op(j + 1, cnt).n == op.n) publish_z();
            } else {
                // ---- residual: x <- (x + W_res z + b) / sqrt(2)  (net.py:76-78); fp16 / e4m3 of (x + d_next) feed the next layer's conv
                // The residual stream is carried only as the fp16 conv input: x = fp16(x + d_cur) - d_cur (tests/tools/precision_study.py
                // "state fp16": 1.5-2.2e-3 vs 1.2-1.3e-3 max mel error).  No fp32 x is read or written: the epilogue streams the conv
                // input once more (32-channel boxes) and stores only the next layer's fp16 / e4m3 conv input.
                const float* d_cur = nullptr;   // STEPS: d_l of this tile's step (d_{l+1} follows at + C)
                if constexpr (STEPS) {
                    const int tb = b < args.B ? __ldg(args.t_of_b + b) : 0;
                    d_cur = args.lut_t + (static_cast<size_t>(tb) * args.total_layers + l) * C;
                }
                auto res_chunk = [&](int c, const uint32_t (&v)[32]) {   // 32 channels
                    const int cl = grp * 128 + c * 32;
                    const int q = q_op + 2 * c + grp;
                    const int sx = q % S::kEStages;
                    const uint32_t box = smem_e + sx * S::kEBoxBytes;
                    mbar_wait_tr(&efull_bar[sx], (q / S::kEStages) & 1, tr, w_e);
                    uint4 xh[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float4 t4 = lds128(box + xo[k]);   // 8 fp16 channels
                        xh[k] = make_uint4(__float_as_uint(t4.x), __float_as_uint(t4.y), __float_as_uint(t4.z), __float_as_uint(t4.w));
                    }
                    uint32_t h16[16], h8[8];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t pk[4] = {xh[k].x, xh[k].y, xh[k].z, xh[k].w};
                        float y[8];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 xf = __half22float2(*reinterpret_cast<const __half2*>(&pk[e]));
                            y[2 * e] = xf.x; y[2 * e + 1] = xf.y;
                        }
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            const int c4 = cl + 8 * k + 4 * hh;
                            float4 bb = lds128(vec_s + c4 * 4), dd;
                            if constexpr (STEPS) {
                                const float4 dl = __ldg(reinterpret_cast<const float4*>(d_cur + c4));
                                bb = make_float4(bb.x - dl.x, bb.y - dl.y, bb.z - dl.z, bb.w - dl.w);
                                dd = has_next ? __ldg(reinterpret_cast<const float4*>(d_cur + C + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                            } else {
                                dd = lds128(vec_s + (256 + c4) * 4);
                            }
                            const float y0 = (y[4 * hh] + fmaf(__uint_as_float(v[8 * k + 4 * hh]), rscale, bb.x)) * rs2 + dd.x;
                            const float y1 = (y[4 * hh + 1] + fmaf(__uint_as_float(v[8 * k + 4 * hh + 1]), rscale, bb.y)) * rs2 + dd.y;
                            const float y2 = (y[4 * hh + 2] + fmaf(__uint_as_float(v[8 * k + 4 * hh + 2]), rscale, bb.z)) * rs2 + dd.z;
                            const float y3 = (y[4 * hh + 3] + fmaf(__uint_as_float(v[8 * k + 4 * hh + 3]), rscale, bb.w)) * rs2 + dd.w;
                            h16[4 * k + 2 * hh] = pack_half2_sat(y0, y1);          // saturating: an out-of-range activation must not become inf
                            h16[4 * k + 2 * hh + 1] = pack_half2_sat(y2, y3);
                            h8[2 * k + hh] = pack_e4m3x4(y0, y1, y2, y3);
                        }
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive_relaxed(&edone_bar[sx]);   // after the arithmetic that consumed the box (see the gate loop)
                    if (row_ok && has_next) {
                        // one row = 64 contiguous bytes of the fp16 and 32 of the e4m3 conv input: full 32-byte sectors
                        stg256(xa16_out + row * C + cl, reinterpret_cast<const uint32_t(&)[8]>(h16[0]));
                        stg256(xa16_out + row * C + cl + 16, reinterpret_cast<const uint32_t(&)[8]>(h16[8]));
                        stg256(xa8_out + row * C + cl, h8);
                    }
                };
                uint32_t va[32], vb[32];
                __syncwarp();
                tmem_ld32(tacc + grp * 128, va);
#pragma unroll 1
                for (int c = 0; c < 4; c += 2) {
                    tmem_ld_wait32(va);
                    __syncwarp();
                    tmem_ld32(tacc + grp * 128 + (c + 1) * 32, vb);
                    if (c == 2 && z_pending) publish_z();
                    res_chunk(c, va);
                    tmem_ld_wait32(vb);
                    if (c + 2 < 4) {
                        __syncwarp();
                        tmem_ld32(tacc + grp * 128 + (c + 2) * 32, va);
                    }
                    res_chunk(c + 1, vb);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote_relaxed(tempty_remote0 + acc * 8);   // TMEM reads ordered by tcgen05.wait::ld + fence
            if (op.kind == 1 && args.flags != nullptr && l + 1 < layer_end && b < args.B) {
                // this warp's rows of the next layer's conv input are written: make them visible device-wide, then count the
                // warp in (8 warps per slab; readers: wait_inputs).  The readers are TMA loads (async proxy) issued by OTHER
                // CTAs: the generic-proxy stores are ordered against the async proxy HERE, by the threads that made them (as
                // publish_z does for the z rows), not only by the reader's fence after its acquire
                asm volatile("fence.proxy.async.global;" ::: "memory");
                __threadfence();
                __syncwarp();
                if (lane == 0) asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(args.flags + static_cast<size_t>(l) * args.n_slabs + sl.g) : "memory");
            }
            if (tr) { if (op.kind == 0) t_gate += clock64() - t_op; else t_res += clock64() - t_op; }
          }
        }
        if (z_pending) publish_z();
        if (tr) {
            unsigned long long* tt = args.trace + blockIdx.x * 16;
            tt[7] = clock64() - t_begin; tt[8] = w_f; tt[11] = t_gate; tt[12] = t_res; tt[14] = w_e;
        }
    }

    tc_fence_before();
    cluster_sync_all();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
}

}  // namespace b200
