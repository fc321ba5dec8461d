// Instantiations + host dispatcher of conv_gemm_kernel, and TMA tensor-map encoding.
#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>

#include "runtime.h"
#include "diffnet_layer.cuh"

namespace b200 {

EncodeTiledFn get_encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
        if (e == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    if (!fn) throw Error("cuTensorMapEncodeTiled not available from the CUDA driver");
    return fn;
}

CUtensorMap make_tmap_ex(const void* base, int kind, int swizzle, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                         const uint32_t* box) {
    CUtensorMap m;
    cuuint64_t gdim[5];
    cuuint64_t gstr[4];
    cuuint32_t bx[5], es[5];
    for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
    B200_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "tensor map base must be 16-byte aligned");
    for (int i = 0; i + 1 < rank; ++i) B200_CHECK(gstr[i] % 16 == 0, "tensor map strides must be multiples of 16 bytes");
    const CUtensorMapDataType dt = kind == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : (kind == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
    const CUtensorMapSwizzle sw = swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
    CUresult r = get_encode_tiled()(&m, dt, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim, gstr, bx, es,
                                    CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw Error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
    return m;
}
CUtensorMap make_tmap_bf16(const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box, bool bytes) {
    return make_tmap_ex(base, bytes ? 1 : 0, 128, rank, dims, strides_bytes, box);
}

// SM count of the current device (cached per device; plans of different devices may live in one process)
int device_sm_count() {
    static std::mutex mu;
    static int cache[64] = {0};
    int dev = 0;
    B200_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && cache[dev] > 0) return cache[dev];
    int n = 0;
    B200_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    if (dev >= 0 && dev < 64) cache[dev] = n;
    return n;
}

namespace {
// How many clusters of `cluster` CTAs of `kern` can be co-resident on the current device (cached per device and kernel): the
// persistent kernels size their grids from it.  On a whole B200 it is SMs / 2 for CTA pairs and 33 for 4-CTA clusters; it is
// smaller when the context only owns part of the device (MPS active-thread percentage, green contexts).
template <class K>
int max_active_clusters(K kern, int cluster, int threads, int smem_bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, int> cache;   // (device, kernel) -> clusters
    int dev = 0;
    B200_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_pair(dev, reinterpret_cast<const void*>(kern));
    const auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    cudaLaunchConfig_t q{};
    q.gridDim = dim3(cluster * 128);
    q.blockDim = dim3(threads);
    q.dynamicSmemBytes = smem_bytes;
    cudaLaunchAttribute qa;
    qa.id = cudaLaunchAttributeClusterDimension;
    qa.val.clusterDim.x = cluster; qa.val.clusterDim.y = 1; qa.val.clusterDim.z = 1;
    q.attrs = &qa;
    q.numAttrs = 1;
    int n = 0;
    B200_CUDA(cudaOccupancyMaxActiveClusters(&n, kern, &q));
    B200_CHECK(n > 0, "no cluster of this kernel fits on the device");
    cache[key] = n;
    return n;
}
}  // namespace

bool use_pdl() {
    static const bool on = [] { const char* e = std::getenv("BSG_NO_PDL"); return !(e && e[0] == '1'); }();
    return on;
}

namespace {

template <int N_TILE, int TERMS, int EPI, bool PAIR, bool MC = false>
void launch_inst(const ConvGemmArgs& args, cudaStream_t stream) {
    using S = GemmSmem<N_TILE, TERMS, PAIR>;
    auto kern = conv_gemm_kernel<N_TILE, TERMS, EPI, PAIR, MC>;
    static std::once_flag once;   // per instantiation
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal); });
    B200_CUDA(attr_err);
    const int sms = device_sm_count();
    if (args.num_tiles > 0)
        B200_CHECK(args.a_rows >= kTileM && args.a_rows <= S::kASlotRows && args.a_rows % 8 == 0, "A halo box does not fit the shared-memory slot");
    const int pairs = sms / 2;
    int grid = PAIR ? 2 * (args.num_tiles < pairs ? args.num_tiles : pairs) : (args.num_tiles < sms ? args.num_tiles : sms);
    if (MC) {
        // clusters of four CTAs: the GPCs cannot host sms/4 of them at once -- ask the driver (33 on B200)
        const int max_clusters = max_active_clusters(kern, 4, kGemmThreads, S::kTotal);
        const int units = ((args.B * args.tiles_per_batch + 1) / 2) * args.n_tiles_n;
        grid = 4 * (units < max_clusters ? units : max_clusters);
    }
    if (args.num_tiles <= 0) return;   // attribute / occupancy set-up call (outside of any stream capture)
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = S::kTotal;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (use_pdl()) {   // the kernel's prologue overlaps the previous kernel's tail (griddepcontrol.wait inside)
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    if (PAIR) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = MC ? 4 : 2;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = na;
    B200_CUDA(cudaLaunchKernelEx(&cfg, kern, args));
    B200_CUDA(cudaGetLastError());
}

}  // namespace

// One fused DiffNet layer (diffnet_layer.cuh): persistent CTA pairs over the 256-row tiles, or (mc) clusters of two pairs
// with multicast weight tiles (weight tensor maps must then have 64-row boxes).
template <int MC, bool STEPS>
static void launch_layer_inst(const LayerArgs& args, cudaStream_t stream) {
    auto kern = diffnet_layer_kernel<MC, STEPS>;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, LayerSmem::kTotal); });
    B200_CUDA(attr_err);
    constexpr int kCtas = MC ? 4 : 2;
    // The layer-to-layer dataflow of a multi-layer launch makes CTAs wait for rows other CTAs of the grid produce: every CTA of
    // the grid must be resident.  The grid is therefore sized from what the driver says fits on THIS context's share of the device
    // (see the co-residency notes at the launch below).
    const int max_clusters = max_active_clusters(kern, kCtas, kLayerThreads, LayerSmem::kTotal);
    if (args.n_row_tiles <= 0) return;
    B200_CHECK(args.n_layers == 1 || args.flags != nullptr, "a multi-layer launch needs the row-tile completion counters");
    B200_CHECK(!STEPS || args.t_of_b != nullptr, "the per-item step variant needs the step table");
    B200_CHECK(args.a_rows >= kTileM && args.a_rows * 128 <= LayerSmem::kASlotBytes && args.a_rows % 8 == 0, "A halo box does not fit the shared-memory slot");
    const int units = MC ? (args.n_row_tiles + 1) / 2 : args.n_row_tiles;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(kCtas * (units < max_clusters ? units : max_clusters));
    cfg.blockDim = dim3(kLayerThreads);
    cfg.dynamicSmemBytes = LayerSmem::kTotal;
    cfg.stream = stream;
    cudaLaunchAttribute attr[3];
    int na = 0;
    // Co-residency of the whole grid is what the cross-CTA waits need (ADVICE r1).  Three measures:
    //  (1) the grid is sized from cudaOccupancyMaxActiveClusters on this context (above), so a partitioned device (MPS active-thread
    //      percentage, green contexts) gets a grid that fits;
    //  (2) multi-layer launches of one process are serialised per device across streams (an event chain, below): two fused kernels of two
    //      plans / streams never overlap, so neither can strand half of the other's grid.  Inside a stream capture the chain cannot be
    //      recorded; captured graphs of different streams must not be replayed concurrently (INTEGRATION.md section 5);
    //  (3) BSG_LAYER_COOP=1 additionally launches cooperatively (the scheduler then places the whole grid or nothing).  Off by default:
    //      Nsight Compute cannot replay a cooperative cluster launch (the launch fails under ncu, profiles/r02_e), and profiling must work.
    // A kernel of ANOTHER process on the same SMs is outside our control: the bounded wait in wait_inputs traps after ~4 s instead of
    // hanging, and BSG_LAYER_STACK=0 (one launch per layer, no cross-CTA waits) is the mode for shared GPUs.
    static const bool coop = [] { const char* e = std::getenv("BSG_LAYER_COOP"); return e && e[0] == '1'; }();
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (args.n_layers > 1) cudaStreamIsCapturing(stream, &cap);
    const bool chain = args.n_layers > 1 && cap == cudaStreamCaptureStatusNone;
    static std::mutex chain_mu;
    static std::map<int, cudaEvent_t> chain_ev;     // device -> completion of the last eager multi-layer launch
    cudaEvent_t ev = nullptr;
    if (chain) {
        int dev = 0;
        B200_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> lock(chain_mu);
        auto it = chain_ev.find(dev);
        if (it == chain_ev.end()) {
            B200_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            chain_ev[dev] = ev;
        } else {
            ev = it->second;
            B200_CUDA(cudaStreamWaitEvent(stream, ev, 0));
        }
    }
    if (coop && args.n_layers > 1) {
        attr[na].id = cudaLaunchAttributeCooperative;
        attr[na].val.cooperative = 1;
        ++na;
    } else if (use_pdl()) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = kCtas;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
    cfg.attrs = attr;
    cfg.numAttrs = na;
    B200_CUDA(cudaLaunchKernelEx(&cfg, kern, args));
    B200_CUDA(cudaGetLastError());
    if (chain) B200_CUDA(cudaEventRecord(ev, stream));
}
void launch_diffnet_layer(const LayerArgs& args, cudaStream_t stream, bool mc, bool steps) {
    if (steps) {
        if (mc) launch_layer_inst<1, true>(args, stream);
        else launch_layer_inst<0, true>(args, stream);
    } else if (mc) launch_layer_inst<1, false>(args, stream);
    else launch_layer_inst<0, false>(args, stream);
}

int conv_gemm_weight_slots(int n_tile, int terms) {
    if (terms != 1) return 0;
    switch (n_tile) {
        case 32: return GemmSmem<32, 1, false>::kBStages;
        case 64: return GemmSmem<64, 1, false>::kBStages;
        case 128: return GemmSmem<128, 1, false>::kBStages;
        case 256: return GemmSmem<256, 1, false>::kBStages;
        default: return 0;
    }
}

#define B200_CASE(NT, TM, EP) \
    if (!pair && n_tile == NT && terms == TM && epi == EP) return launch_inst<NT, TM, EP, false>(args, stream);
#define B200_PAIR(NT, TM, EP) \
    if (pair == 1 && n_tile == NT && terms == TM && epi == EP) return launch_inst<NT, TM, EP, true>(args, stream);
#define B200_MC(NT, TM, EP) \
    if (pair == 2 && n_tile == NT && terms == TM && epi == EP) return launch_inst<NT, TM, EP, true, true>(args, stream);

void launch_conv_gemm(int n_tile, int terms, int epi, const ConvGemmArgs& args, cudaStream_t stream, int pair) {
    // unit-test GEMMs
    B200_CASE(256, 1, EPI_F32) B200_CASE(256, 3, EPI_F32) B200_CASE(128, 1, EPI_F32) B200_CASE(128, 3, EPI_F32)
    B200_CASE(64, 1, EPI_F32) B200_CASE(32, 1, EPI_F32)
    B200_PAIR(256, 1, EPI_F32) B200_PAIR(256, 3, EPI_F32) B200_PAIR(128, 3, EPI_F32)
    B200_CASE(256, 2, EPI_F32) B200_CASE(128, 2, EPI_F32) B200_PAIR(256, 2, EPI_F32) B200_PAIR(128, 2, EPI_F32)
    // DiffNet
    B200_CASE(256, 1, EPI_INPROJ) B200_CASE(256, 3, EPI_INPROJ)
    B200_CASE(256, 1, EPI_GATE) B200_CASE(256, 3, EPI_GATE) B200_PAIR(256, 1, EPI_GATE) B200_PAIR(256, 3, EPI_GATE)
    B200_CASE(256, 1, EPI_RES_SKIP) B200_CASE(256, 3, EPI_RES_SKIP) B200_CASE(128, 1, EPI_RES_SKIP) B200_CASE(128, 3, EPI_RES_SKIP)
    B200_CASE(256, 1, EPI_RELU_BF16) B200_CASE(256, 3, EPI_RELU_BF16) B200_CASE(128, 1, EPI_RELU_BF16) B200_CASE(128, 3, EPI_RELU_BF16)
    B200_PAIR(256, 1, EPI_RELU_BF16) B200_PAIR(256, 3, EPI_RELU_BF16) B200_PAIR(128, 1, EPI_RELU_BF16) B200_PAIR(128, 3, EPI_RELU_BF16)
    B200_CASE(80, 1, EPI_POSTERIOR) B200_CASE(80, 3, EPI_POSTERIOR)
    // DiffNet with a diffusion step per batch item (step calls whose items are at different steps)
    B200_CASE(256, 1, EPI_INPROJ_STEPS) B200_CASE(256, 3, EPI_INPROJ_STEPS)
    B200_CASE(128, 1, EPI_RES_SKIP_STEPS) B200_CASE(128, 2, EPI_RES_SKIP_STEPS) B200_CASE(128, 3, EPI_RES_SKIP_STEPS)
    B200_CASE(80, 1, EPI_POSTERIOR_STEPS) B200_CASE(80, 3, EPI_POSTERIOR_STEPS)
    // two CTA pairs per cluster with multicast weights
    B200_MC(256, 1, EPI_F32) B200_MC(256, 2, EPI_F32) B200_MC(256, 3, EPI_F32) B200_MC(128, 2, EPI_F32)
    B200_MC(256, 2, EPI_GATE) B200_MC(256, 2, EPI_RELU_BF16) B200_MC(256, 3, EPI_RELU_BF16)
    // DiffNet, fp16x2 per-layer GEMMs
    B200_CASE(256, 2, EPI_GATE) B200_PAIR(256, 2, EPI_GATE) B200_CASE(128, 2, EPI_RES_SKIP)
    B200_CASE(128, 2, EPI_RELU_BF16) B200_PAIR(256, 2, EPI_RELU_BF16) B200_PAIR(256, 4, EPI_RELU_BF16) B200_PAIR(256, 4, EPI_F32)
    B200_PAIR(256, 5, EPI_RELU_BF16)
    // HiFi-GAN
    B200_PAIR(256, 1, EPI_BIAS_ACT) B200_PAIR(128, 1, EPI_BIAS_ACT)
    B200_CASE(256, 1, EPI_BIAS_ACT) B200_CASE(128, 1, EPI_BIAS_ACT) B200_CASE(64, 1, EPI_BIAS_ACT) B200_CASE(32, 1, EPI_BIAS_ACT)
    // PitchExtractor (bf16x3)
    B200_CASE(256, 3, EPI_BIAS_ACT) B200_PAIR(256, 3, EPI_BIAS_ACT)
    throw Error("conv_gemm: no instantiation for n_tile=" + std::to_string(n_tile) + " terms=" + std::to_string(terms) +
                " epi=" + std::to_string(epi) + (pair == 2 ? " (pair, multicast)" : (pair ? " (pair)" : "")));
}

}  // namespace b200
