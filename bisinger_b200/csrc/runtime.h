// Host-side runtime helpers: error handling, device buffers, TMA tensor-map encoding, launch glue.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <iterator>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "conv_gemm.cuh"

namespace b200 {

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define B200_CUDA(expr)                                                                                  \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            throw ::b200::Error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " (" + __FILE__ + ":" + \
                                std::to_string(__LINE__) + ")");                                         \
    } while (0)

#define B200_CHECK(cond, msg)                                                                            \
    do {                                                                                                 \
        if (!(cond)) throw ::b200::Error(std::string("check failed: ") + #cond + ": " + (msg));          \
    } while (0)

// Free list of device buffers by exact size (plan-owned).  The per-shape workspaces of a plan draw their large buffers from it and hand them
// back when a shape is evicted: utterance lengths change from call to call, and cudaMalloc / cudaFree of gigabyte buffers cost up to
// hundreds of milliseconds each time (tools/varying_length_latency.py).  Workspace sizes are quantised (capacity classes of rows), so
// buffers of one class fit every shape of the class.  Must outlive every DevBuf that was allocated from it.
struct DevPool {
    std::multimap<size_t, void*> free_list;
    size_t pooled = 0;
    void* take(size_t n) {
        auto it = free_list.find(n);
        if (it == free_list.end()) return nullptr;
        void* p = it->second;
        free_list.erase(it);
        pooled -= n;
        return p;
    }
    void give(void* p, size_t n) {
        free_list.emplace(n, p);
        pooled += n;
    }
    void trim(size_t keep_bytes) {   // largest first
        while (pooled > keep_bytes && !free_list.empty()) {
            auto it = std::prev(free_list.end());
            cudaFree(it->second);
            pooled -= it->first;
            free_list.erase(it);
        }
    }
    ~DevPool() { trim(0); }
};

// RAII device allocation (plan-owned workspaces / packed weights)
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DevPool* pool = nullptr;   // where the buffer goes on release (null: cudaFree)
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes), pool(o.pool) { o.p = nullptr; o.bytes = 0; o.pool = nullptr; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { release(); p = o.p; bytes = o.bytes; pool = o.pool; o.p = nullptr; o.bytes = 0; o.pool = nullptr; }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() {
        if (p) {
            if (pool) pool->give(p, bytes);
            else cudaFree(p);
        }
        p = nullptr;
        bytes = 0;
        pool = nullptr;
    }
    // from != null: reuse a pooled buffer of exactly n bytes if there is one (contents are whatever its last user left), and return
    // the buffer to that pool on release
    void alloc(size_t n, DevPool* from = nullptr) {
        release();
        if (n == 0) n = 16;
        pool = from;
        if (from != nullptr && (p = from->take(n)) != nullptr) {
            bytes = n;
            return;
        }
        cudaError_t err = cudaMalloc(&p, n);
        if (err == cudaErrorMemoryAllocation && from != nullptr && from->pooled > 0) {   // the free list may be holding what is missing
            cudaGetLastError();
            from->trim(0);
            err = cudaMalloc(&p, n);
        }
        if (err != cudaSuccess) p = nullptr;
        B200_CUDA(err);
        bytes = n;
        // debugging aid (BSG_ALLOC_FILL=<hex byte>): fill every fresh device buffer, e.g. ff = NaN patterns in f32 / f16 / e4m3, so a
        // read of memory the path never wrote shows up in the results instead of depending on what the allocation held before
        static const int fill = [] { const char* e = getenv("BSG_ALLOC_FILL"); return e ? static_cast<int>(strtol(e, nullptr, 16)) : -1; }();
        if (fill >= 0) B200_CUDA(cudaMemset(p, fill, n));
    }
    void ensure(size_t n) {
        if (n > bytes) alloc(n);
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

template <class T>
inline void upload(DevBuf& d, const std::vector<T>& h) {
    d.alloc(h.size() * sizeof(T));
    B200_CUDA(cudaMemcpy(d.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
}

// round-to-nearest-even fp32 -> bf16 on the host (packer)
inline uint16_t f32_to_bf16_bits(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);  // NaN
    u += 0x7fffu + ((u >> 16) & 1u);
    return static_cast<uint16_t>(u >> 16);
}
inline float bf16_bits_to_f32(uint16_t b) {
    uint32_t u = static_cast<uint32_t>(b) << 16;
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency)
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_tiled();

// 16-bit (bf16 / fp16) tensor -- or 8-bit with bytes = true -- dims given innermost-first; strides (bytes) for dims 1..rank-1;
// SWIZZLE_128B, zero OOB fill.
CUtensorMap make_tmap_bf16(const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                           bool bytes = false);

// general form: kind 0 = 16-bit, 1 = 8-bit, 2 = fp32 elements; swizzle 128 or 64 (bytes)
CUtensorMap make_tmap_ex(const void* base, int kind, int swizzle, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box);
// 8-bit activations [B][L][C], box = 128 channels (128 bytes) x box_rows rows
inline CUtensorMap make_act8_tmap(const void* base, int B, int L, int C, int box_rows) {
    const uint64_t dims[3] = {static_cast<uint64_t>(C), static_cast<uint64_t>(L), static_cast<uint64_t>(B)};
    const uint64_t strides[2] = {static_cast<uint64_t>(C), static_cast<uint64_t>(C) * L};
    const uint32_t box[3] = {128, static_cast<uint32_t>(box_rows), 1};
    return make_tmap_ex(base, 1, 128, 3, dims, strides, box);
}
// fp32 rows [B][L][C] read / written by the epilogue through shared memory: box = 16 columns (64 bytes, SWIZZLE_64B) x 128 rows
inline CUtensorMap make_f32_tmap(const void* base, int B, int L, int C) {
    const uint64_t dims[3] = {static_cast<uint64_t>(C), static_cast<uint64_t>(L), static_cast<uint64_t>(B)};
    const uint64_t strides[2] = {static_cast<uint64_t>(C) * 4, static_cast<uint64_t>(C) * 4 * L};
    const uint32_t box[3] = {16, 128, 1};
    return make_tmap_ex(base, 2, 64, 3, dims, strides, box);
}
// 16-bit rows [B][L][C] as the fused layer kernel's epilogue reads them: box = 32 channels (64 bytes, SWIZZLE_64B) x 128 rows
inline CUtensorMap make_epi16_tmap(const void* base, int B, int L, int C) {
    const uint64_t dims[3] = {static_cast<uint64_t>(C), static_cast<uint64_t>(L), static_cast<uint64_t>(B)};
    const uint64_t strides[2] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(C) * 2 * L};
    const uint32_t box[3] = {32, 128, 1};
    return make_tmap_ex(base, 0, 64, 3, dims, strides, box);
}
// activations [B][L][C] (channels-last), box = 64 channels x box_rows rows (the halo tile of one k-block)
inline CUtensorMap make_act_tmap(const void* base, int B, int L, int C, int row_pitch_elems = 0, int box_rows = kTileM) {
    if (row_pitch_elems == 0) row_pitch_elems = C;
    const uint64_t dims[3] = {static_cast<uint64_t>(C), static_cast<uint64_t>(L), static_cast<uint64_t>(B)};
    const uint64_t strides[2] = {static_cast<uint64_t>(row_pitch_elems) * 2, static_cast<uint64_t>(row_pitch_elems) * 2 * L};
    const uint32_t box[3] = {static_cast<uint32_t>(kBlockK), static_cast<uint32_t>(box_rows), 1};
    return make_tmap_bf16(base, 3, dims, strides, box);
}
// packed weights [N][K] (K-major), box = 64 x n_tile
inline CUtensorMap make_w_tmap(const void* base, int N, int K, int n_tile, int row_pitch_elems = 0) {
    if (row_pitch_elems == 0) row_pitch_elems = K;
    const uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(N)};
    const uint64_t strides[1] = {static_cast<uint64_t>(row_pitch_elems) * 2};
    const uint32_t box[2] = {static_cast<uint32_t>(kBlockK), static_cast<uint32_t>(n_tile)};
    return make_tmap_bf16(base, 2, dims, strides, box);
}

int device_sm_count();
bool use_pdl();   // programmatic dependent launch attribute on the GEMM launches (BSG_NO_PDL=1: off)
// weight-ring slots of the single-CTA conv_gemm instantiation (n_tile, terms): a convolution with n_taps * n_kb <= this many
// weight tiles may keep them resident (ConvGemmArgs::w_resident)
int conv_gemm_weight_slots(int n_tile, int terms);

// Launch one instantiation of conv_gemm_kernel (defined in gemm_launch.cu)
// pair = 1: 2-CTA clusters on 256-row tiles (tcgen05 cta_group::2); the weight tensor map box must then be n_tile/2 rows
// pair = 2: clusters of two such pairs with multicast weight tiles; weight tensor map box = n_tile/4 rows
void launch_conv_gemm(int n_tile, int terms, int epi, const ConvGemmArgs& args, cudaStream_t stream, int pair = 0);

// One fused DiffNet layer (diffnet_layer.cuh); args.n_slabs == 0 only sets the kernel attributes up
struct LayerArgs;
void launch_diffnet_layer(const LayerArgs& args, cudaStream_t stream, bool mc = false, bool steps = false);   // steps: diffnet_layer_kernel<MC, true>

// One fused HiFi-GAN ResBlock1 iteration (resblock_fused.cuh) for channels in {32, 64, 128}; args.num_tiles == 0 only sets the kernel
// attributes up.  resblock_weight_slots: weight tiles (C rows x 64 K-columns) its shared-memory weight area holds.
struct ResblockArgs;
void launch_resblock_iter(int channels, const ResblockArgs& args, cudaStream_t stream);
int resblock_weight_slots(int channels);

// fills the tile-geometry fields of args from (B, L, N_total, n_tile)
inline void set_geometry(ConvGemmArgs& a, int B, int L, int n_total, int n_tile, bool pair = false) {
    a.B = B;
    a.L = L;
    const int rows = pair ? 2 * kTileM : kTileM;
    a.tiles_per_batch = (L + rows - 1) / rows;
    a.n_tiles_n = n_total / n_tile;
    a.num_tiles = B * a.tiles_per_batch * a.n_tiles_n;
    a.w_row0 = 0;
}

// Fills args.taps / args.a_rows for a convolution whose tap j reads rows shifted by shifts[j] and K columns
// [j * w_tap_stride, ...) of the packed weights.  Returns the rows the A halo box must have.
inline int set_taps(ConvGemmArgs& a, int a_src, int a_col0, int n_kb, const int* shifts, int n_taps, int w_tap_stride) {
    B200_CHECK(n_taps >= 1 && n_taps <= kMaxTaps, "too many taps");
    int lo = shifts[0], hi = shifts[0];
    for (int j = 1; j < n_taps; ++j) { lo = shifts[j] < lo ? shifts[j] : lo; hi = shifts[j] > hi ? shifts[j] : hi; }
    a.taps.a_src = a_src;
    a.taps.a_col0 = a_col0;
    a.taps.n_kb = n_kb;
    a.taps.row_shift = lo;
    a.taps.n_taps = n_taps;
    for (int j = 0; j < n_taps; ++j) { a.taps.row_off[j] = shifts[j] - lo; a.taps.w_col0[j] = j * w_tap_stride; }
    a.a_rows = ((kTileM + hi - lo) + 7) / 8 * 8;
    return a.a_rows;
}
inline int halo_rows(int span) { return ((kTileM + span) + 7) / 8 * 8; }

// round-to-nearest-even fp32 -> fp16 on the host (packer)
inline uint16_t f32_to_f16_bits(float f) {
    const __half_raw r = static_cast<__half_raw>(__float2half_rn(f));
    return r.x;
}
inline float f16_bits_to_f32(uint16_t b) {
    __half_raw r;
    r.x = b;
    return __half2float(__half(r));
}

// Packed (hi, lo) weight matrix on the device: bf16 pair (bf16 / bf16x3 modes) or fp16 pair pre-scaled by 2^p (fp16x2)
struct PackedW {
    DevBuf hi, lo;
    DevBuf lo8;            // fp16x2 packing only: e5m2(w * 2^p - hi), the weight-correction operand of the fp8 MMAs
    CUtensorMap tm8;       // box = 128 K-columns (bytes) x 128 rows
    bool tm8_ok = false;
    int tm8_rows = 0;
    const CUtensorMap& map8(int box_rows = 128) {
        if (!tm8_ok || tm8_rows != box_rows) {
            const uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(N)};
            const uint64_t strides[1] = {static_cast<uint64_t>(K)};
            const uint32_t box[2] = {128, static_cast<uint32_t>(box_rows)};
            tm8 = make_tmap_ex(lo8.p, 1, 128, 2, dims, strides, box);
            tm8_ok = true;
            tm8_rows = box_rows;
        }
        return tm8;
    }
    int N = 0, K = 0;
    float acc_scale = 1.0f;   // 2^-p: what the epilogue multiplies the accumulators with
    CUtensorMap tm[2];     // cached TMA descriptors (hi, lo) for box = 64 x tm_ntile
    int tm_ntile = 0;
    void maps(int n_tile, CUtensorMap& mhi, CUtensorMap& mlo) {
        if (tm_ntile != n_tile) {
            tm[0] = make_w_tmap(hi.p, N, K, n_tile);
            tm[1] = make_w_tmap(lo.p, N, K, n_tile);
            tm_ntile = n_tile;
        }
        mhi = tm[0];
        mlo = tm[1];
    }
    // w: row-major [N][K] fp32 on the host
    void pack(const std::vector<float>& w, int n, int k, bool fp16 = false) {
        N = n;
        K = k;
        tm_ntile = 0;
        std::vector<uint16_t> h(w.size()), l(w.size());
        if (!fp16) {
            acc_scale = 1.0f;
            for (size_t i = 0; i < w.size(); ++i) {
                h[i] = f32_to_bf16_bits(w[i]);
                l[i] = f32_to_bf16_bits(w[i] - bf16_bits_to_f32(h[i]));
            }
        } else {
            // hi = fp16(w * 2^p), lo = fp16(w * 2^p - hi) with the largest |w| * 2^p in [8192, 16384): the low parts of all but the
            // tiniest weights are normal fp16 numbers (a subnormal lo would lose its mantissa bits)
            float mx = 0.0f;
            for (float v : w) mx = std::fmax(mx, std::fabs(v));
            int p = 0;
            if (mx > 0.0f && std::isfinite(mx)) {
                p = 13 - static_cast<int>(std::floor(std::log2(mx)));
                p = p < -14 ? -14 : (p > 24 ? 24 : p);
            }
            const float up = std::ldexp(1.0f, p);
            acc_scale = std::ldexp(1.0f, -p);
            std::vector<uint8_t> l8(w.size());
            for (size_t i = 0; i < w.size(); ++i) {
                const float v = w[i] * up;
                h[i] = f32_to_f16_bits(v);
                const float rem = v - f16_bits_to_f32(h[i]);
                l[i] = f32_to_f16_bits(rem);
                l8[i] = static_cast<uint8_t>(__nv_cvt_float_to_fp8(rem, __NV_SATFINITE, __NV_E5M2));
            }
            upload(lo8, l8);
            tm8_ok = false;
        }
        upload(hi, h);
        upload(lo, l);
    }
};

}  // namespace b200
